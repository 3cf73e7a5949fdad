"""Geo re-ranking without a GPU: argument checks of nais_powerlaw_logmax / nais_fullrank_topk_geo_planned (returned
before any CUDA call), the declared symbols, and the sharded logic of ShardedRanker.topk(geo=...) on gloo with injected
local maximum / top-k callables."""
import ctypes as C
import os
import re
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _codes():
    hdr = open(os.path.join(ROOT, "include", "nais_b200.h")).read()
    return {n: int(v) for n, v in re.findall(r"#define NAIS_ERR_(\w+) (-?\d+)", hdr)}


NULL, MODE, SHAPE = (_codes()[n] for n in ("NULL", "MODE", "SHAPE"))


def _lib():
    from poi_recommendation_models_b200 import _lib
    if not os.path.isfile(_lib.LIB_PATH):
        pytest.skip("library not built")
    return _lib, _lib.load()


def test_new_symbols_are_declared_and_bound():
    from poi_recommendation_models_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "nais_b200.h")).read()
    for name in ("nais_powerlaw_logmax", "nais_fullrank_topk_geo_planned"):
        assert re.search(r"NAIS_API int " + name + r"\(", hdr)
        assert name in _lib.SYMBOLS
    assert "typedef struct NaisGeoMix" in hdr
    assert [f for f, _ in _lib.NaisGeoMix._fields_] == ["a", "b", "alpha", "user_logmax"]


def _structs(L, with_coords=True):
    cat = L.NaisCatalog()
    cat.row_base, cat.n_rows = 0, 1000
    users = L.NaisUsers()
    users.n_users = 3
    fake = 0x10000  # never dereferenced: every call below returns from its argument checks
    users.offsets, users.items = fake, fake
    if with_coords:
        cat.coords, users.coords = fake, fake
    return cat, users


def test_logmax_argument_errors():
    L, lib = _lib()
    cat, users = _structs(L)
    out = 0x20000
    assert lib.nais_powerlaw_logmax(C.byref(cat), C.byref(users), 0, 1000, 0.0, -1.0, 1, out, None) == MODE  # a <= 0 -> MODE
    assert lib.nais_powerlaw_logmax(C.byref(cat), C.byref(users), 0, 1000, float("nan"), -1.0, 1, out, None) == MODE
    assert lib.nais_powerlaw_logmax(C.byref(cat), C.byref(users), 0, 1001, 0.8, -1.0, 1, out, None) == SHAPE  # range -> SHAPE
    assert lib.nais_powerlaw_logmax(C.byref(cat), C.byref(users), 0, 1000, 0.8, -1.0, 1, None, None) == NULL  # NULL
    cat2, users2 = _structs(L, with_coords=False)
    assert lib.nais_powerlaw_logmax(C.byref(cat2), C.byref(users2), 0, 1000, 0.8, -1.0, 1, out, None) == NULL


def _params(L):
    p = L.NaisParams()
    p.n_branch, p.hid, p.item_num, p.region_num, p.dist_mode, p.beta = 1, 64, 1000, 1, L.DIST_NONE, 0.5
    br = p.branch[0]
    fake = 0x10000
    br.hist_poi = br.tgt_poi = br.w1 = br.b1 = br.w2 = fake
    br.w_poi, br.w_reg = 64, 0
    return p


def test_geo_planned_argument_errors():
    L, lib = _lib()
    p = _params(L)
    cat, users = _structs(L)
    fp32 = L.PRECISIONS["fp32"]
    out_s, out_i, ws = 0x30000, 0x40000, 0x50000

    def call(geo, lo=0, hi=1000, k=10, cat_=cat, users_=users):
        g = C.byref(geo) if geo is not None else None
        return lib.nais_fullrank_topk_geo_planned(C.byref(p), C.byref(cat_), C.byref(users_), lo, hi, k, 1, fp32, None, 0, g, None,
                                                  out_s, out_i, ws, 1 << 20, None)

    ok = 0x60000
    assert call(None) == NULL                                         # no NaisGeoMix -> NULL
    assert call(L.NaisGeoMix(0.0, -1.3, 0.2, ok)) == MODE             # a <= 0 -> MODE
    assert call(L.NaisGeoMix(-1.0, -1.3, 0.2, ok)) == MODE
    assert call(L.NaisGeoMix(0.8, -1.3, float("nan"), ok)) == MODE    # non-finite alpha -> MODE
    assert call(L.NaisGeoMix(0.8, -1.3, float("inf"), ok)) == MODE
    assert call(L.NaisGeoMix(0.8, -1.3, 0.2, None)) == NULL           # no user_logmax -> NULL
    cat2, users2 = _structs(L, with_coords=False)
    assert call(L.NaisGeoMix(0.8, -1.3, 0.2, ok), cat_=cat2, users_=users2) == NULL  # no coordinates -> NULL
    good = L.NaisGeoMix(0.8, -1.3, 0.2, ok)
    assert call(good, hi=1001) == SHAPE                                # range -> SHAPE, as the planned call
    assert call(good, k=0) == SHAPE and call(good, k=129) == SHAPE        # k -> SHAPE


# ---- sharded geo ranking on gloo -----------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q, min_shard, want_grid):
    try:
        _worker_body(rank, world, port, q, min_shard, want_grid)
    except Exception:
        import traceback
        q.put((rank, traceback.format_exc()))


def _mixed_table(U, N):
    rng = np.random.default_rng(0)
    score = rng.normal(size=(U, N)).astype(np.float32)
    logg = (rng.normal(size=(U, N)) * 3 - 50).astype(np.float32)
    hist = [rng.choice(N, 5, replace=False) for _ in range(U)]
    return score, logg, hist


def _ref_lists(score, logg, hist, alpha, k):
    U, N = score.shape
    out = []
    for u in range(U):
        cand = np.setdiff1d(np.arange(N), hist[u])
        M = logg[u, cand].max()
        mixed = np.float32(1 - alpha) / (1 + np.exp(-score[u].astype(np.float32))) + np.float32(alpha) * np.exp(logg[u] - M)
        mixed = mixed.astype(np.float32)
        mixed[hist[u]] = -np.inf
        order = np.lexsort((np.arange(N), -mixed))[:k]
        out.append((mixed[order], order.astype(np.int32)))
    return out


def _worker_body(rank, world, port, q, min_shard, want_grid):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from types import SimpleNamespace
    from poi_recommendation_models_b200 import ops
    from poi_recommendation_models_b200.distributed import ShardedRanker
    N, U, k, alpha = 1000, 7, 20, 0.3
    score, logg, hist = _mixed_table(U, N)
    calls = []

    def local_logmax(users, lo, hi, a, b):
        m = np.full(len(users.ids), -np.inf, np.float32)
        for j, u in enumerate(users.ids):
            keep = np.setdiff1d(np.arange(lo, hi), hist[u])
            if len(keep):
                m[j] = logg[u, keep].max()
        calls.append(("max", lo, hi))
        return torch.from_numpy(m)

    def local_topk(users, kk, lo, hi, precision, geo=None):
        assert geo is not None and geo.alpha == alpha and geo.logmax.shape == (len(users.ids),)
        out_s, out_i = torch.full((len(users.ids), kk), -float("inf")), torch.full((len(users.ids), kk), -1, dtype=torch.int32)
        for j, u in enumerate(users.ids):
            M = np.float32(geo.logmax[j].item())
            mixed = (np.float32(1 - alpha) / (1 + np.exp(-score[u, lo:hi])) + np.float32(alpha) * np.exp(logg[u, lo:hi] - M))
            mixed = mixed.astype(np.float32)
            h = hist[u][(hist[u] >= lo) & (hist[u] < hi)] - lo
            mixed[h] = -np.inf
            valid = np.isfinite(mixed)
            ids = np.arange(lo, hi)[valid]
            order = np.lexsort((ids, -mixed[valid]))[:kk]
            out_s[j, :len(order)] = torch.from_numpy(mixed[valid][order])
            out_i[j, :len(order)] = torch.from_numpy(ids[order].astype(np.int32))
        return out_s, out_i

    def slice_users(users, u0, u1):
        return SimpleNamespace(offsets=users.offsets, n_users=u1 - u0, ids=users.ids[u0:u1])

    def merge(keys):
        gs, gi = ops.keys_to_lists(keys)
        L_, U_, k_ = gs.shape
        s, i = gs.permute(1, 0, 2).reshape(U_, L_ * k_).numpy(), gi.permute(1, 0, 2).reshape(U_, L_ * k_).numpy()
        os_, oi = np.full((U_, k_), -np.inf, np.float32), np.full((U_, k_), -1, np.int32)
        for u in range(U_):
            v = i[u] >= 0
            o = np.lexsort((i[u][v], -s[u][v]))[:k_]
            os_[u, :len(o)], oi[u, :len(o)] = s[u][v][o], i[u][v][o]
        return torch.from_numpy(os_), torch.from_numpy(oi)

    r = ShardedRanker(SimpleNamespace(item_num=N), rank, world, local_topk=local_topk, merge=merge, min_shard_pois=min_shard,
                      slice_users=slice_users, local_logmax=local_logmax)
    users = SimpleNamespace(offsets=torch.zeros(1), n_users=U, ids=np.arange(U))
    s, i = r.topk(users, k, geo=(0.8, -1.3, alpha))
    ref = _ref_lists(score, logg, hist, alpha, k)  # one rank, the whole catalogue
    ok = (r.gc, r.gu) == want_grid and s.shape == (U, k)
    ok = ok and all(np.array_equal(i[u].numpy(), ref[u][1]) for u in range(U))
    ok = ok and all(np.array_equal(s[u].numpy(), ref[u][0]) for u in range(U))
    ok = ok and calls == [("max", r.lo, r.hi)]
    q.put((rank, bool(ok)))
    dist.destroy_process_group()


def _run(world, min_shard, want_grid):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q, min_shard, want_grid)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=180) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(r, True) for r in range(world)], res


def test_geo_sharded_catalogue_world2_gloo():
    """two catalogue ranges: the range maxima meet in one all_reduce(MAX), the lists equal one rank's"""
    _run(2, 0, (2, 1))


def test_geo_user_sliced_world2_gloo():
    """two user slices (ragged last slice): each rank's maximum covers the whole catalogue for its own users"""
    _run(2, 32768, (1, 2))
