"""Explanations of pair scores on the GPU (nais_pairs_explain, ops.pairs_explain, model.explain): the selected history items,
their contributions and attention shares against the float64 terms of tests/explain_terms.py, for every variant, both layouts,
the FP32 and the tcgen05 pair forward, short / two-chunk / long histories; the score bit for bit against the pair forward; the
padding, masking and tie order; and model.explain on predict_topk's lists."""
import numpy as np
import pytest
import torch

import explain_terms
from oracle import nais_oracle as orc
from poi_recommendation_models_b200 import model as M, ops, synthetic

pytestmark = pytest.mark.gpu
VARIANTS = ["basic", "region", "region_distance", "distance", "disentangled"]
HAS_REG = {"basic": False, "region": True, "region_distance": True, "distance": False, "disentangled": True}
DIST = {"basic": None, "region": None, "region_distance": "latlon", "distance": "latlon", "disentangled": "km"}
BETA = 0.5


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


class Case:
    """Parameters, a catalogue (centred float32 coordinates like set_catalog's) and rows: a list of users, each with a history
    and targets (every third target inside its own history: a masked cell)."""

    def __init__(self, variant, D, hid, hist_lens, rows_per_user, seed, N=900):
        rng = np.random.default_rng(seed)
        self.variant, self.N = variant, N
        coords, self.region, R = synthetic.make_catalog(N, seed=seed)
        c = np.asarray(coords, dtype=np.float64)
        self.center = (float((c[:, 0].min() + c[:, 0].max()) / 2), float((c[:, 1].min() + c[:, 1].max()) / 2))
        self.cc = (c - np.array(self.center)).astype(np.float32)  # centred, as the kernels see them
        self.sd = orc.init_state(variant, N, D, hid, R, 1, seed=seed + 1, style="trained")
        self.P = {n: self.sd[n].cuda().contiguous() for n in ops.VARIANT_PARAMS[variant]}
        self.hists = [rng.choice(N, H, replace=False).astype(np.int64) for H in hist_lens]
        self.tgts = []
        for h, r in zip(self.hists, rows_per_user):
            t = rng.integers(0, N, r).astype(np.int64)
            if len(h) > 1:
                t[::3] = h[(np.arange(len(t[::3])) * 7) % len(h)]
            self.tgts.append(t)

    def aux(self, hist, tgt):
        """aux of dense rows hist [B,H] / tgt [B] from the centred coordinates (float32 |dlat|,|dlon|, or haversine km)"""
        d = DIST[self.variant]
        if d == "latlon":
            return np.abs(self.cc[tgt][:, None, :] - self.cc[hist]).astype(np.float32)
        if d == "km":
            u = self.cc.astype(np.float64) + np.array(self.center)
            return orc.dist_km(u[tgt][:, None, 0], u[tgt][:, None, 1], u[hist][..., 0], u[hist][..., 1]).astype(np.float32)
        return None

    def dense_user(self, i):
        """(hist [B,H], tgt, hreg, treg, aux) numpy rows of user i in the dense layout"""
        hist = np.broadcast_to(self.hists[i], (len(self.tgts[i]), len(self.hists[i]))).copy()
        tgt = self.tgts[i]
        reg = HAS_REG[self.variant]
        return hist, tgt, self.region[hist] if reg else None, self.region[tgt] if reg else None, self.aux(hist, tgt)

    def dense_gpu(self, rows):
        hist, tgt, hreg, treg, aux = rows
        return tuple(None if a is None else _dev(a) for a in (hist, tgt, hreg, treg, aux))

    def segmented(self):
        st = ops.segment_structure([len(h) for h in self.hists], [len(t) for t in self.tgts], "cuda")
        hist, tgt = np.concatenate(self.hists), np.concatenate(self.tgts)
        reg, co = HAS_REG[self.variant], DIST[self.variant] is not None
        return ops.SegmentedPairs(
            hist=_dev(hist), hreg=_dev(self.region[hist].astype(np.int64)) if reg else None, hist_coords=_dev(self.cc[hist]) if co else None,
            tgt=_dev(tgt), treg=_dev(self.region[tgt].astype(np.int64)) if reg else None, tgt_coords=_dev(self.cc[tgt]) if co else None,
            label=None, seg_offsets=st["seg_offsets"], row_offsets=st["row_offsets"], seg_cell_offsets=st["seg_cell_offsets"],
            tile_seg=st["tile_seg"], tile_row0=st["tile_row0"], n_seg=st["n_seg"], B=st["B"], n_tiles=st["n_tiles"],
            n_cells=st["n_cells"], max_hist=st["max_hist"], host_row_offsets=st["host_row_offsets"], center=self.center)

    def terms(self, rows):
        t = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a))
        return explain_terms.attention_terms(self.sd, self.variant, BETA, *(t(a) for a in rows))


def check_rows(T, pos, contrib, attn, m):
    """The returned (pos, contrib, attn) of some rows [R, m] / [n_branch, R, m] against their float64 terms T."""
    c64, pi64, mask = T["contrib"].numpy(), T["attn"].numpy(), T["mask"].numpy()
    for r in range(c64.shape[0]):
        sel = mask[r]
        n = min(m, int(sel.sum()))
        scale = float(np.abs(c64[r][sel]).sum())
        tol = 1e-4 * scale
        p = pos[r]
        assert (p[n:] == -1).all() and np.isneginf(contrib[r][n:]).all() and (attn[:, r, n:] == 0).all(), "padding"
        q = p[:n]
        assert len(set(q.tolist())) == n and (q >= 0).all() and sel[q].all(), "selection: distinct, unmasked positions"
        assert np.abs(contrib[r][:n] - c64[r][q]).max(initial=0) <= tol, (r, contrib[r][:n], c64[r][q])
        assert np.abs(attn[:, r, :n] - pi64[:, r, q]).max(initial=0) <= 1e-4
        assert (np.diff(contrib[r][:n]) <= 0).all(), "descending"
        ties = np.diff(contrib[r][:n]) == 0
        assert (np.diff(q)[ties] > 0).all(), "ties by ascending position"
        rest = np.setdiff1d(np.flatnonzero(sel), q)
        if n and len(rest):
            assert c64[r][rest].max() <= c64[r][q].min() + 2 * tol, "a valid top-m outside the tie band"


def _cpu(*ts):
    return tuple(t.cpu().numpy() for t in ts)


SHAPES = [("fp32", 64, 64), ("tc", 64, 64), ("tc", 32, 48)]  # (pair precision, D, hid): two threads per cell, run-time shape


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("pp,D,hid", SHAPES)
@pytest.mark.parametrize("H,m", [(3, 5), (37, 8), (129, 8), (300, 6)])
def test_dense_rows_against_float64(variant, pp, D, hid, H, m):
    case = Case(variant, D, hid, [1], [1], seed=H + D)
    rng = np.random.default_rng(H)
    hist = np.stack([rng.choice(case.N, H, replace=False) for _ in range(23)]).astype(np.int64)  # every row its own history
    tgt = rng.integers(0, case.N, 23).astype(np.int64)
    tgt[::3] = hist[::3, H // 2]
    reg = HAS_REG[variant]
    rows = (hist, tgt, case.region[hist] if reg else None, case.region[tgt] if reg else None, case.aux(hist, tgt))
    score, pos, contrib, attn = ops.pairs_explain(variant, BETA, case.P, *case.dense_gpu(rows), m=m, precision=pp)
    check_rows(case.terms(rows), *_cpu(pos, contrib, attn), m)
    ops.check_indices(sync=True)


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("pp,D,hid", SHAPES)
def test_segmented_against_float64(variant, pp, D, hid):
    """Users of 3 (padding at m = 5), 37, 129 (two chunks) and 300 items, and one without history (no rows)."""
    case = Case(variant, D, hid, [3, 37, 0, 129, 300], [9, 20, 0, 5, 4], seed=D + hid)
    m = 5
    score, pos, contrib, attn = _cpu(*ops.pairs_explain(variant, BETA, case.P, case.segmented(), m=m, precision=pp))
    r0 = 0
    for i in range(len(case.hists)):
        R = len(case.tgts[i])
        if R == 0:
            continue
        sl = slice(r0, r0 + R)
        check_rows(case.terms(case.dense_user(i)), pos[sl], contrib[sl], attn[:, sl], m)
        r0 += R
    assert r0 == len(score)
    ops.check_indices(sync=True)


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("pp", ["fp32", "auto"])
@pytest.mark.parametrize("layout", ["dense", "segmented"])
def test_score_is_the_pair_forwards_bit_for_bit(variant, pp, layout):
    case = Case(variant, 64, 64, [37, 129, 5], [11, 3, 17], seed=7)
    if layout == "dense":
        batch = case.dense_gpu(case.dense_user(0))
    else:
        batch = (case.segmented(), None, None, None, None)
    score = ops.pairs_explain(variant, BETA, case.P, *batch, m=4, precision=pp)[0]
    ref = ops.pairs_forward_raw(variant, BETA, case.P, *batch, drop=(0.0, 0, pp))[0]
    assert torch.equal(score, ref)


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("pp", ["fp32", "auto"])
@pytest.mark.parametrize("H", [3, 20, 32])
def test_all_positions_sum_to_the_score(variant, pp, H):
    """m >= H: every unmasked position is returned, the contributions add up to the score and the attention to 1."""
    case = Case(variant, 64, 64, [H], [13], seed=H)
    rows = case.dense_user(0)
    score, pos, contrib, attn = _cpu(*ops.pairs_explain(variant, BETA, case.P, *case.dense_gpu(rows), m=32, precision=pp))
    T = case.terms(rows)
    mask = T["mask"].numpy()
    scale = np.abs(T["contrib"].numpy()).sum(-1)
    c = np.where(pos >= 0, contrib, 0.0).astype(np.float64)
    assert ((pos >= 0).sum(1) == mask.sum(1)).all()
    assert (np.abs(c.sum(1) - score) <= 1e-5 * scale).all()
    assert (np.abs(attn.astype(np.float64).sum(-1) - 1.0) <= 1e-5).all()


@pytest.mark.parametrize("pp", ["fp32", "tc"])
def test_masked_positions_and_ties(pp):
    """A training-style batch (the target inside its history) never selects the masked position; repeated history items (equal
    cells, equal contributions) come out in ascending position order."""
    case = Case("region", 64, 64, [6], [1], seed=2)
    hist = np.array([[5, 7, 5, 9, 7, 11, 5, 9], [4, 8, 15, 16, 23, 42, 8, 4], [1, 2, 3, 4, 5, 6, 7, 8]], dtype=np.int64)
    tgt = np.array([9, 8, 300], dtype=np.int64)
    rows = (hist, tgt, case.region[hist], case.region[tgt], None)
    score, pos, contrib, attn = _cpu(*ops.pairs_explain("region", BETA, case.P, *case.dense_gpu(rows), m=8, precision=pp))
    check_rows(case.terms(rows), pos, contrib, attn, 8)
    assert not np.isin(pos[0], [3, 7]).any() and not np.isin(pos[1], [1, 6]).any()
    assert (pos[0] >= 0).sum() == 6 and (pos[1] >= 0).sum() == 6 and (pos[2] >= 0).all()
    for r in range(2):
        for item in set(hist[r].tolist()) - {int(tgt[r])}:
            at = np.flatnonzero(hist[r][np.maximum(pos[r], 0)] == item)
            at = at[pos[r][at] >= 0]
            if len(at) > 1:  # equal items sit next to each other in the ranking, in ascending position
                assert (np.diff(at) == 1).all() and (np.diff(pos[r][at]) > 0).all()
                assert (contrib[r][at] == contrib[r][at[0]]).all()


def _catalogue_model(variant, D=32, hid=32, N=80, seed=0):
    coords, region, R = synthetic.make_catalog(N, seed=seed)
    sd = orc.init_state(variant, N, D, hid, R, 1, seed=seed + 1, style="trained")
    cls = M.CLASSES[variant]
    m = cls(N, D, hid, BETA) if variant == "basic" else (cls(N, D, hid, BETA, R) if variant == "region" else cls(N, D, hid, BETA, R, 1))
    m.load_state_dict(sd)
    m = m.cuda().eval()
    m.set_catalog(region=region, coords=coords)
    return m, sd, coords, region


@pytest.mark.parametrize("variant", VARIANTS)
def test_model_explain_on_predict_topk_lists(variant):
    """Every class: the explained POIs are the user's history items, sigmoid(score) is predict_topk's score, padded entries and a
    user without history are padding with a NaN score, and the result equals ops.pairs_explain on the dense batch of each user."""
    N, k, mm = 80, 12, 4
    m, sd, coords, region = _catalogue_model(variant, N=N)
    rng = np.random.default_rng(5)
    hists = [rng.choice(N, 9, replace=False), np.array([], dtype=np.int64), rng.choice(N, N - 5, replace=False),
             rng.choice(N, 40, replace=False), rng.choice(N, 2, replace=False)]  # user 2: 5 candidates < k -> -1 padding
    csr = lambda hs: (np.concatenate([[0], np.cumsum([len(h) for h in hs])]), np.concatenate(hs).astype(np.int64))
    s_top, ids = m.predict_topk(csr(hists[:1] + hists[2:]), k)  # (ranked for the users with a history)
    filler = torch.tensor([[3, 4, 5] + [-1] * (k - 3)], device="cuda")
    ids = torch.cat([ids[:1], filler, ids[1:]])  # user 1: no history, some ids
    s_top = torch.cat([s_top[:1], torch.full((1, k), float("nan"), device="cuda"), s_top[1:]])
    users = m.make_users(*csr(hists))
    ex = m.explain(users, ids, m=mm)
    ids_h, s_h = ids.cpu().numpy(), s_top.cpu().numpy()
    score, poi, pos, contrib, attn = _cpu(*ex)
    nb = 2 if variant == "disentangled" else 1
    assert score.shape == (5, k) and poi.shape == pos.shape == contrib.shape == (5, k, mm) and attn.shape == (nb, 5, k, mm)
    assert (ids_h[2] == -1).sum() == k - 5
    for u in range(5):
        for j in range(k):
            if ids_h[u, j] < 0 or len(hists[u]) == 0:
                assert np.isnan(score[u, j]) and (pos[u, j] == -1).all() and (poi[u, j] == -1).all()
                assert np.isneginf(contrib[u, j]).all() and (attn[:, u, j] == 0).all()
                continue
            assert abs(1 / (1 + np.exp(-float(score[u, j]))) - s_h[u, j]) <= 1e-4
            sel = pos[u, j] >= 0
            assert sel.sum() == min(mm, len(hists[u]))
            assert np.isin(poi[u, j][sel], hists[u]).all() and (poi[u, j][sel] == hists[u][pos[u, j][sel]]).all()
    # the same explanations from the dense layout, user by user
    cc = m._catalog.coords.cpu().numpy()
    center = m._catalog.center
    for u in (0, 2, 3, 4):
        v = ids_h[u][ids_h[u] >= 0]
        hist = np.broadcast_to(hists[u], (len(v), len(hists[u]))).astype(np.int64).copy()
        aux = None
        if DIST[variant] == "latlon":
            aux = np.abs(cc[v][:, None, :] - cc[hist]).astype(np.float32)
        elif DIST[variant] == "km":
            g = cc.astype(np.float64) + np.array(center)
            aux = orc.dist_km(g[v][:, None, 0], g[v][:, None, 1], g[hist][..., 0], g[hist][..., 1]).astype(np.float32)
        reg = HAS_REG[variant]
        rows = (hist, v, region[hist].astype(np.int64) if reg else None, region[v].astype(np.int64) if reg else None, aux)
        d_score, d_pos, d_contrib, d_attn = _cpu(*ops.pairs_explain(variant, BETA, m._params(), *(None if a is None else _dev(a) for a in rows),
                                                                     m=mm))
        n = len(v)
        scale = np.abs(case_terms(sd, variant, rows)["contrib"].numpy()).sum(-1)
        assert (np.abs(score[u, :n] - d_score) <= 1e-5 * scale).all()
        dv = d_pos >= 0
        assert np.array_equal(pos[u, :n] >= 0, dv) and np.isneginf(contrib[u, :n][~dv]).all()
        assert (np.abs(contrib[u, :n][dv] - d_contrib[dv]) <= 1e-5 * np.broadcast_to(scale[:, None], dv.shape)[dv]).all()
        assert np.abs(attn[:, u, :n] - d_attn).max() <= 1e-5
        for r in range(n):  # same positions wherever the contributions are not tied within that band
            for i in range(mm):
                if not dv[r, i]:
                    continue
                others = np.delete(d_contrib[r], i)
                if np.all(np.abs(others - d_contrib[r, i]) > 2e-5 * scale[r]):
                    assert pos[u, r, i] == d_pos[r, i], (u, r, i)
    ops.check_indices(sync=True)


def case_terms(sd, variant, rows):
    t = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a))
    return explain_terms.attention_terms(sd, variant, BETA, *(t(a) for a in rows))


def test_bad_ids_raise_index_error():
    case = Case("region", 32, 48, [10], [6], seed=1)
    hist, tgt, hreg, treg, aux = case.dense_user(0)
    tgt = tgt.copy()
    tgt[2] = case.N + 17
    ops.check_indices(sync=True)
    ops.pairs_explain("region", BETA, case.P, *case.dense_gpu((hist, tgt, hreg, treg, aux)), m=3)
    with pytest.raises(IndexError):
        ops.check_indices(sync=True)
    m, *_ = _catalogue_model("basic")
    ids = torch.tensor([[3, 1000, -1]], device="cuda")
    m.explain((np.array([0, 4]), np.array([1, 2, 5, 7])), ids, m=2)
    with pytest.raises(IndexError):
        ops.check_indices(sync=True)
