"""CPU-side checks: the C-ABI library builds, loads and exports every symbol the header declares; host-side drop-ins
(batches, eval_metrics, synthetic data, shard ranges) against the reference / oracle.  No compute calls need a GPU."""
import os
import random
import re

import numpy as np
import pytest
import torch

from oracle import nais_oracle as orc
from oracle import ref_shim
from poi_recommendation_models_b200 import _lib, batches as PB, eval_metrics as PM, model as M, synthetic
from poi_recommendation_models_b200.distributed import shard_range

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_builds_and_exports_every_declared_symbol():
    import __graft_entry__
    __graft_entry__.build()
    lib = _lib.load()
    hdr = open(os.path.join(ROOT, "include", "nais_b200.h")).read()
    declared = set(re.findall(r"NAIS_API\s+[\w\s\*]+?\b(nais_\w+)\s*\(", hdr))
    assert declared and declared == set(_lib.SYMBOLS), (declared ^ set(_lib.SYMBOLS))
    for name in declared:
        assert getattr(lib, name) is not None
    assert lib.nais_abi_version() == 2
    assert b"workspace" in lib.nais_strerror(-4)
    assert lib.nais_launch_count() >= 0


def test_argument_errors_are_reported_before_any_launch():
    import ctypes as C
    lib = _lib.load()
    p = _lib.NaisParams()
    b = _lib.NaisPairs()
    assert lib.nais_pairs_forward(C.byref(p), C.byref(b), None, None, None, None, None) == -2  # n_branch = 0 -> shape error
    p.n_branch, p.hid, p.item_num = 1, 64, 10
    p.branch[0].w_poi = 64
    assert lib.nais_pairs_forward(C.byref(p), C.byref(b), None, None, None, None, None) == -1  # NULL tables
    assert lib.nais_fullrank_workspace_bytes(C.byref(p), 4, 100, 0, 10, 5, 0) == 0  # invalid params -> 0


def test_new_v2_entry_points_validate_before_launching():
    import ctypes as C
    lib = _lib.load()
    p = _lib.NaisParams()
    assert lib.nais_fullrank_plan_bytes(C.byref(p), 0, 100, _lib.PREC_TC_AUTO) == 0            # invalid params -> 0
    assert lib.nais_topk_merge_keys(None, 20, 20, 0, 1, 20, None, None, None, None) == 0        # no users: nothing to do
    assert lib.nais_topk_merge_keys(None, 20, 20, 4, 1, 20, None, None, None, None) == -1       # NULL input
    assert lib.nais_topk_merge_keys(None, 10, 20, 4, 1, 20, None, None, None, None) == -2       # stride shorter than a list
    assert lib.nais_poll_bad_index(None, None) == -1
    assert b"index" in lib.nais_strerror(_lib.ERR_INDEX)
    p.n_branch, p.hid, p.item_num, p.pairs_precision = 1, 64, 10, 7
    p.branch[0].w_poi = 64
    for f in ("hist_poi", "tgt_poi", "w1", "b1", "w2"):
        setattr(p.branch[0], f, 16)  # (never dereferenced: the argument checks run first)
    b = _lib.NaisPairs()
    assert lib.nais_pairs_forward(C.byref(p), C.byref(b), None, None, None, None, None) == -5         # unknown pairs_precision


def test_ranking_keys_pack_and_unpack_like_make_key():
    """ops.lists_to_keys / keys_to_lists mirror csrc/nais_common.cuh make_key / split_key: order = score desc, then id asc;
    NaN ranks as -inf; id < 0 is "no entry" (key 0)."""
    from poi_recommendation_models_b200 import ops
    s = torch.tensor([[1.5, -2.0, 0.0, float("-inf"), 3e38, -1e-30, float("nan"), 1.5]])
    i = torch.tensor([[5, 7, 0, 3, 2147483647, 9, 11, 4]], dtype=torch.int32)
    keys = ops.lists_to_keys(s, i)
    s2, i2 = ops.keys_to_lists(keys)
    assert torch.equal(i2, i) and torch.equal(s2[0, :6], s[0, :6]) and s2[0, 6] == float("-inf")
    ku = keys.numpy().astype(np.uint64)[0]
    order = np.argsort(ku)[::-1]
    assert order.tolist()[:3] == [4, 7, 0]  # 3e38, then the two 1.5s by ascending id (4 before 5)
    assert ku[3] > ku[6] or ku[6] > ku[3]   # -inf with different ids still totally ordered
    empty = ops.lists_to_keys(torch.zeros(1, 2), torch.tensor([[-1, 3]], dtype=torch.int32))
    assert int(empty[0, 0]) == 0 and int(empty[0, 1]) != 0
    e_s, e_i = ops.keys_to_lists(empty)
    assert e_s[0, 0] == float("-inf") and int(e_i[0, 0]) == -1


def test_ops_refuse_cpu_tensors():
    m = M.NAIS_basic(20, 16, 16, 0.5).eval()
    with pytest.raises(RuntimeError, match="CUDA"):
        m(torch.zeros(2, 3, dtype=torch.long), torch.zeros(2, dtype=torch.long))


def test_state_dict_keys_and_init_match_reference_classes(golden_dir):
    # tests/golden/scorer_<variant>.npz holds parameter sets the reference class of each of the five variants loaded with
    # strict=True (make_golden.py): the drop-in class must declare exactly those keys and shapes
    for variant in orc.VARIANTS:
        z = np.load(os.path.join(golden_dir, f"scorer_{variant}.npz"))
        sd = {k[len("reference_sd."):]: torch.from_numpy(z[k]) for k in z.files if k.startswith("reference_sd.")}
        N, D, hid, beta, R = int(z["N"]), int(z["D"]), int(z["hid"]), float(z["beta"]), int(z["R"])
        cls = M.CLASSES[variant]
        b = cls(N, D, hid, beta) if variant == "basic" else cls(N, D, hid, beta, R) if variant == "region" else cls(N, D, hid, beta, R, 1)
        assert {k: tuple(v.shape) for k, v in b.state_dict().items()} == {k: tuple(v.shape) for k, v in sd.items()}, variant
        b.load_state_dict(sd, strict=True)
        assert b.item_num == N and b.beta == beta
    if not ref_shim.reference_available():  # the key order and the seeded initial values need the reference classes themselves
        return
    ref = ref_shim.load_reference("model")
    cases = [("NAIS_basic", (50, 16, 8, 0.5)), ("NAIS_regionEmbedding", (50, 16, 8, 0.5, 7)),
             ("NAIS_region_distance_Embedding", (50, 16, 8, 0.5, 7, 1)), ("NAIS_distance_Embedding", (50, 16, 8, 0.5, 7, 1)),
             ("NAIS_region_distance_disentangled_Embedding", (50, 16, 8, 0.5, 7, 1))]
    for name, args in cases:
        torch.manual_seed(0)
        a = getattr(ref, name)(*args)
        torch.manual_seed(0)
        b = getattr(M, name)(*args)
        sa, sb = a.state_dict(), b.state_dict()
        assert list(sa.keys()) == list(sb.keys()), name
        for k in sa:
            assert torch.equal(sa[k], sb[k]), (name, k)  # same seed -> same initial weights
        b.load_state_dict(sa)  # reference checkpoints load
        for attr in ("embed_size", "item_num", "beta", "hidden_size"):
            assert getattr(a, attr) == getattr(b, attr)


def test_batches_match_reference_golden(golden_dir):
    z = np.load(os.path.join(golden_dir, "batches.npz"))
    import scipy.sparse as sp
    csr = sp.csr_matrix((np.ones(len(z["indices"])), z["indices"], z["indptr"]), shape=(4, int(z["N"])))
    for u in range(4):
        random.seed(123 + u)
        hist, tgt, label, hreg, treg = PB.get_NAIS_batch_region(csr, int(z["N"]), u, int(z["num_ng"]), z["region"])
        for name, got in (("hist", hist), ("tgt", tgt), ("label", label), ("hreg", hreg), ("treg", treg)):
            assert np.array_equal(got.cpu().numpy(), z[f"u{u}.{name}"]), (u, name)
        h2, t2, _, _, _ = PB.get_NAIS_batch_test_region(csr, u, z["region"])
        assert np.array_equal(t2.cpu().numpy(), z[f"u{u}.test_tgt"])
        assert np.array_equal(h2[0].cpu().numpy(), z[f"u{u}.test_hist0"])


def test_lat_lon_pairs_equals_latlon_mat_lookup():
    rng = np.random.default_rng(0)
    coords = np.stack([40.5 + rng.random(30), -74 + rng.random(30)], 1)
    mat = np.zeros((30, 30, 2))
    for i in range(30):  # run.py:47-54
        for j in range(30):
            mat[i][j][0] = abs(coords[i][0] - coords[j][0])
            mat[i][j][1] = abs(coords[i][1] - coords[j][1])
    tgt = rng.integers(0, 30, 7)
    hist = np.stack([rng.choice(30, 5, replace=False) for _ in range(7)])
    ref = torch.tensor(mat[np.repeat(tgt.reshape(-1, 1), 5, 1), hist], dtype=torch.float32)  # run.py:239-247
    assert torch.equal(PB.lat_lon_pairs(coords, tgt, hist, device="cpu"), ref)


def test_metrics_bit_identical_to_reference(golden_dir):
    # the values the reference's eval_metrics.py returned for its own recommended lists (tests/golden/validation_*.npz rows:
    # precision, recall, hit rate on the validation positives, then on the test positives, one column per k)
    for name in ("validation_rd.npz", "validation_basic.npz", "validation_region.npz"):
        z = np.load(os.path.join(golden_dir, name))
        rec = z["rec"].tolist()
        for j, part in enumerate(("val", "test")):
            flat, ptr = z[part + "_flat"], z[part + "_ptr"]
            positive = [flat[ptr[u]:ptr[u + 1]].tolist() for u in range(int(z["U"]))]
            for c, fn in enumerate((PM.precision_at_k, PM.recall_at_k, PM.hitrate_at_k)):
                assert [fn(positive, rec, k) for k in z["k_list"].tolist()] == z["metrics"][3 * j + c].tolist(), (name, part, c)
    rng = np.random.default_rng(3)
    U = 200
    actual = [rng.choice(500, rng.integers(0, 6), replace=False).tolist() for _ in range(U)]
    pred = [rng.choice(500, 50, replace=False).tolist() for _ in range(U)]
    for k in (5, 10, 15, 20, 25, 30):
        assert PM.precision_at_k(actual, pred, k) == orc.precision_at_k(actual, pred, k)
        assert PM.recall_at_k(actual, pred, k) == orc.recall_at_k(actual, pred, k)
        assert PM.hitrate_at_k(actual, pred, k) == orc.hitrate_at_k(actual, pred, k)
        assert PM.ndcg_at_k(actual, pred, k) == orc.ndcg_at_k(actual, pred, k)
    if ref_shim.reference_available():
        ref = ref_shim.load_reference("eval_metrics")
        for k in (5, 10, 30):
            assert PM.precision_at_k(actual, pred, k) == ref.precision_at_k(actual, pred, k)
            assert PM.recall_at_k(actual, pred, k) == ref.recall_at_k(actual, pred, k)
            assert PM.hitrate_at_k(actual, pred, k) == ref.hitrate_at_k(actual, pred, k)


def test_rank_metrics_bit_identical_to_reference(golden_dir):
    """apk / mapk / precision_at_k_per_sample drop-ins vs the golden written by the unmodified eval_metrics.py:29-34, 70-125
    (repeated ids in the ranked list, users without positives, lists shorter than k) and vs the live reference."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("mk_rank", os.path.join(golden_dir, "make_golden_rank_metrics.py"))
    mk = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mk)
    g = np.load(os.path.join(golden_dir, "rank_metrics.npz"))
    actual, predicted = mk.make_lists()
    for j, k in enumerate(g["ks"].tolist()):
        for u, (a, p) in enumerate(zip(actual, predicted)):
            assert PM.apk(a, p, k) == g["apk"][u, j] == orc.apk(a, p, k)
            assert PM.precision_at_k_per_sample(a, p, k) == g["pps"][u, j]
        assert PM.mapk(actual, predicted, k) == g["mapk"][j]
    assert PM.apk([1, 2], [2, 1]) == 1.0 and PM.apk([], [1, 2]) == 0.0
    if ref_shim.reference_available():
        ref = ref_shim.load_reference("eval_metrics")
        rng = np.random.default_rng(5)
        a2 = [rng.choice(60, rng.integers(0, 7), replace=False).tolist() for _ in range(100)]
        p2 = [rng.integers(0, 60, 25).tolist() for _ in range(100)]  # with repeats
        for k in (3, 10, 25, 40):
            assert PM.mapk(a2, p2, k) == ref.mapk(a2, p2, k)
            assert all(PM.precision_at_k_per_sample(a, p, k) == ref.precision_at_k_per_sample(a, p, k) for a, p in zip(a2, p2))


def test_synthetic_checkins_are_consistent():
    d = synthetic.make_checkins(20, 800, seed=1)
    assert d.indptr[-1] == len(d.indices) and d.region.max() + 1 == d.region_num
    for u in range(20):
        h = d.history(u)
        assert len(set(h.tolist())) == len(h) and (np.diff(h) > 0).all()
        assert not set(h.tolist()) & set(d.val_positive[u]) and not set(h.tolist()) & set(d.test_positive[u])
        assert len(d.val_positive[u]) >= 1
    d2 = synthetic.make_checkins(20, 800, seed=1)
    assert np.array_equal(d.indices, d2.indices) and np.array_equal(d.coords, d2.coords)  # seed-exact
    fixed = synthetic.make_checkins(5, 400, hist_len=32, seed=2)
    assert (np.diff(fixed.indptr) == 32).all()


@pytest.mark.parametrize("n,world", [(40000, 1), (40000, 8), (1000, 3), (100, 8), (5, 4), (1000000, 8)])
def test_shard_ranges_partition_the_catalogue(n, world):
    ranges = [shard_range(n, r, world) for r in range(world)]
    assert ranges[0][0] == 0 and ranges[-1][1] == n
    for (a0, a1), (b0, b1) in zip(ranges, ranges[1:]):
        assert a1 == b0 and a0 <= a1
    for lo, hi in ranges[:-1]:
        assert lo % 128 == 0 or lo == n


def test_whole_module_pickle_roundtrip(tmp_path):
    """run.py:266-268 checkpoints with torch.save(model): the drop-in modules must survive a whole-module pickle."""
    for name, args in (("NAIS_region_distance_Embedding", (40, 16, 16, 0.5, 5, 1)), ("NAIS_basic", (40, 16, 16, 0.5)),
                       ("NAIS_region_distance_disentangled_Embedding", (40, 16, 16, 0.5, 5, 1))):
        m = getattr(M, name)(*args)
        m.set_catalog(region=np.arange(40) % 5, coords=np.stack([40.5 + np.arange(40) * 1e-3, -74 + np.arange(40) * 1e-3], 1))
        path = tmp_path / (name + ".pt")
        torch.save(m, path)
        m2 = torch.load(path, weights_only=False)
        assert type(m2).__name__ == name and m2.beta == m.beta and m2.item_num == m.item_num
        for (k1, v1), (k2, v2) in zip(m.state_dict().items(), m2.state_dict().items()):
            assert k1 == k2 and torch.equal(v1, v2)
        assert m2._catalog.n_rows == 40 and torch.equal(m2._catalog.region, m._catalog.region)


def test_ctypes_mirrors_match_the_header_layout(tmp_path):
    """Every struct of include/nais_b200.h, compiled by gcc as plain C, has the size and field offsets of its ctypes mirror
    in _lib.py — a drifted mirror would make the library read garbage past the struct (no compute call involved)."""
    import ctypes as C
    import shutil
    import subprocess
    from poi_recommendation_models_b200 import _lib as L
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    structs = ["NaisBranch", "NaisParams", "NaisPairs", "NaisGrads", "NaisAdagrad", "NaisDenseAdagrad", "NaisCatalog", "NaisUsers"]
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "nais_b200.h"', 'int main(void) {']
    for s in structs:
        cls = getattr(L, s)
        lines.append(f'  printf("{s} %zu\\n", sizeof({s}));')
        for f, _ in cls._fields_:
            lines.append(f'  printf("{s}.{f} %zu\\n", offsetof({s}, {f}));')
    lines += ['  return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    inc = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include")
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", f"-I{inc}", str(src), "-o", str(exe)], check=True)
    got = dict(ln.split() for ln in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    for s in structs:
        cls = getattr(L, s)
        assert int(got[s]) == C.sizeof(cls), s
        for f, _ in cls._fields_:
            assert int(got[f"{s}.{f}"]) == getattr(cls, f).offset, (s, f)


def test_precision_flags_and_train_step_entry_validate():
    """The `precision` flag bits of the header equal the Python names; nais_pairs_train_step checks its arguments before it
    launches anything (no GPU here)."""
    import ctypes as C
    import re
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "nais_b200.h")).read()
    flags = dict((m.group(1), int(m.group(2), 16)) for m in re.finditer(r"#define (NAIS_PREC_FLAG_\w+) (0x[0-9a-fA-F]+)", hdr))
    assert flags == {"NAIS_PREC_FLAG_GENERIC": _lib.PREC_FLAG_GENERIC, "NAIS_PREC_FLAG_ONE_CTA": _lib.PREC_FLAG_ONE_CTA}
    assert _lib.PRECISIONS["tc_auto_onecta"] == _lib.PREC_TC_AUTO | _lib.PREC_FLAG_ONE_CTA
    lib = _lib.load()
    p, b = _lib.NaisParams(), _lib.NaisPairs()
    assert lib.nais_pairs_train_step_workspace_bytes(C.byref(p), C.byref(b)) == 0                      # invalid params -> 0
    assert lib.nais_pairs_train_step(C.byref(p), C.byref(b), None, None, None, None, None, None, None, 0, None) < 0
    p.n_branch, p.hid, p.item_num = 1, 64, 10
    p.branch[0].w_poi = 64
    for f in ("hist_poi", "tgt_poi", "w1", "b1", "w2"):
        setattr(p.branch[0], f, 16)  # (never dereferenced: the argument checks run first)
    b.H = 4
    assert lib.nais_pairs_train_step(C.byref(p), C.byref(b), None, None, None, None, None, None, None, 0, None) == -1  # NULL optimizer state
    ad, dn = _lib.NaisAdagrad(), _lib.NaisDenseAdagrad()
    for f in ("sum_w1", "sum_b1", "sum_w2"):
        setattr(dn, f, 16)
    indptr, users = np.array([0, 3, 5], dtype=np.int64), np.array([2], dtype=np.int64)  # user 2 of a 2-row matrix
    assert lib.nais_train_users(C.byref(p), indptr.ctypes.data, 2, 16, None, None, None, None, users.ctypes.data, 1, 4, 0, C.byref(ad),
                                C.byref(dn), 16, 16, 1 << 20, None) == -2                                     # user id outside the matrix
    assert lib.nais_train_users_workspace_bytes(C.byref(p), 100, 4) > 0


def test_segment_structure_rides_in_one_upload():
    """ops.segment_structure packs its index arrays (and the caller's extras) into one buffer: the views must equal the arrays."""
    import torch
    from poi_recommendation_models_b200 import ops
    H = np.array([3, 0, 130, 17, 1], dtype=np.int64)
    extra = np.arange(7, dtype=np.int64) * 11
    st = ops.segment_structure(H, 5 * H, torch.device("cpu"), extra=[(extra, np.int64), (np.array([5, 6, 7], dtype=np.int32), np.int32)])
    assert st["seg_offsets"].tolist() == [0, 3, 3, 133, 150, 151]
    assert st["row_offsets"].tolist() == [0, 15, 15, 665, 750, 755]
    assert st["seg_cell_offsets"].tolist() == np.concatenate([[0], np.cumsum(5 * H * H)]).tolist()
    assert st["tile_seg"].dtype == torch.int32 and st["tile_row0"].dtype == torch.int64
    assert st["n_tiles"] == len(st["tile_seg"]) == len(st["tile_row0"])
    # tiles: min(16, 128 // H) rows of one segment each (1 row when H > 128); a segment without history has none
    rows_per_tile = {0: 16, 2: 1, 3: 7, 4: 16}
    for t in range(st["n_tiles"]):
        s_ = int(st["tile_seg"][t])
        assert s_ != 1 and (int(st["tile_row0"][t]) - int(st["row_offsets"][s_])) % rows_per_tile[s_] == 0
    assert st["extra"][0].tolist() == extra.tolist() and st["extra"][1].tolist() == [5, 6, 7] and st["extra"][1].dtype == torch.int32
    assert st["B"] == 755 and st["n_cells"] == int((5 * H * H).sum()) and st["max_hist"] == 130


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver times next to ours): one JSON line with the contract's keys on
    rank 0; any other rank exits 0 without work or output."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--config", "tiny", "--steps", "1", "--warmup", "1",
           "--cpu-users", "1"]
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    out = subprocess.run(cmd, check=True, capture_output=True, text=True, env=env, timeout=300).stdout.strip().splitlines()
    line = json.loads(out[-1])
    assert line["impl"] == "reference" and line["metric"] == "fullrank_eval_users_per_sec" and line["unit"] == "users/s"
    assert line["value"] > 0 and line["higher_is_better"] is True and line["vs_baseline"] is None
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    if ref_shim.reference_available():  # the unmodified reference classes (or their oracle/_ref snapshot) are what is timed
        assert line["cpu_baseline"]["kind"] == "reference"
    assert line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": "users/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    env1 = dict(env, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run(cmd, check=True, capture_output=True, text=True, env=env1, timeout=300)
    assert r.stdout.strip() == ""


def test_presort_pair_validates_before_launching():
    """nais_pairs_forward_presort / nais_pairs_backward_presorted: one branch only, a NaisGrads skeleton and a workspace of at least
    nais_pairs_backward_workspace_bytes are required — all reported before anything is enqueued (no GPU here)."""
    import ctypes as C
    lib = _lib.load()
    p, b, g = _lib.NaisParams(), _lib.NaisPairs(), _lib.NaisGrads()
    assert lib.nais_pairs_forward_presort(C.byref(p), C.byref(b), C.byref(g), None, None, None, None, None, 0, None) == -2  # no branch
    p.n_branch, p.hid, p.item_num = 1, 64, 10
    p.branch[0].w_poi = 64
    for f in ("hist_poi", "tgt_poi", "w1", "b1", "w2"):
        setattr(p.branch[0], f, 16)  # (never dereferenced: the argument checks run first)
    b.H = 4
    assert lib.nais_pairs_forward_presort(C.byref(p), C.byref(b), None, None, None, None, None, None, 0, None) == -1        # no NaisGrads
    assert lib.nais_pairs_forward_presort(C.byref(p), C.byref(b), C.byref(g), None, None, None, None, None, 0, None) == 0    # B = 0: nothing to do
    b.B, b.hist, b.tgt = 8, 16, 16
    assert lib.nais_pairs_forward_presort(C.byref(p), C.byref(b), C.byref(g), None, None, None, None, 16, 1 << 30, None) == -1  # no score
    assert lib.nais_pairs_forward_presort(C.byref(p), C.byref(b), C.byref(g), 16, None, None, None, None, 0, None) == -1     # no workspace
    need = lib.nais_pairs_backward_workspace_bytes(C.byref(p), C.byref(b))
    assert need > 0
    assert lib.nais_pairs_forward_presort(C.byref(p), C.byref(b), C.byref(g), 16, None, None, None, 16, need - 1, None) == -4  # too small
    assert lib.nais_pairs_backward_presorted(C.byref(p), C.byref(b), 16, 16, None, 16, C.byref(g), 16, need - 1, None) == -4
    assert lib.nais_pairs_backward_presorted(C.byref(p), C.byref(b), 16, 16, None, 16, C.byref(g), 24, need, None) == -3     # misaligned
    p2 = _lib.NaisParams.from_buffer_copy(p)
    p2.n_branch = 2
    p2.branch[1] = p.branch[0]
    assert lib.nais_pairs_forward_presort(C.byref(p2), C.byref(b), C.byref(g), 16, None, None, None, 16, 1 << 30, None) == -5  # two branches
    assert lib.nais_pairs_backward_presorted(C.byref(p2), C.byref(b), 16, 16, None, 16, C.byref(g), 16, 1 << 30, None) == -5
    # the one-user-ahead pipeline of nais_train_users holds two users: its workspace is twice one user's
    assert lib.nais_train_users_workspace_bytes(C.byref(p), 100, 4) % 2 == 0
