"""Fused power-law geo re-ranking on the GPU: nais_powerlaw_logmax and the geo mode of the full-rank kernels
(powerlaw.fused_rerank_topk, ops.fullrank_topk(geo=...)), against a float64 restatement of
    mixed(u, j) = (1 - alpha) * sigmoid(score(u, j)) + alpha * exp(logG(u, j) - M_u)
on the seeded catalogue of tests/golden/powerlaw.npz, with trained-style weights and a steep law (a = 0.8, b = -1.3)."""
import numpy as np
import pytest
import torch

import nais_testutil as util
from oracle import nais_oracle as orc
from poi_recommendation_models_b200 import ops
from poi_recommendation_models_b200 import powerlaw as PL

pytestmark = pytest.mark.gpu

A_, B_, ALPHA = 0.8, -1.3, 0.2


def _golden():
    z = util.load_golden("powerlaw.npz")
    return z, int(z["U"]), int(z["N"])


def _model(variant, N, region, coords, D=64, hid=64, seed=8):
    R = int(region.max()) + 1
    sd = orc.init_state(variant, N, D, hid, R, 1, seed=seed, style="trained")
    m = util.make_model(variant, sd, 0.5)
    m.set_catalog(region=region, coords=coords)
    return m, sd


def _long_catalogue():
    """700 POIs; users with a 600-item history (> HMETA = 512 staged items), none, one, and a short one."""
    rng = np.random.default_rng(5)
    N = 700
    coords = np.stack([40.7 + rng.normal(0, 0.05, N), -74.0 + rng.normal(0, 0.05, N)], 1)
    region = rng.integers(0, 6, N)
    hists = [rng.choice(N, 600, replace=False), np.array([], dtype=np.int64), np.array([17]), rng.choice(N, 40, replace=False)]
    indptr = np.concatenate([[0], np.cumsum([len(h) for h in hists])]).astype(np.int64)
    return N, coords, region, indptr, np.concatenate(hists).astype(np.int64)


def _logg64(coords, hist, cand, a, b):
    if len(hist) == 0:
        return np.zeros(len(cand))
    d = PL.dist((coords[hist][None, :, 0], coords[hist][None, :, 1]), (coords[cand][:, None, 0], coords[cand][:, None, 1]))
    return (np.log(a) + b * np.log(np.maximum(0.01, d))).sum(1)


def _ref_mixed(variant, sd, coords, region, hist, N, a, b, alpha, exclude):
    """{candidate id: float64 mixed value} over the ranked candidate set"""
    cand = np.setdiff1d(np.arange(N), hist) if exclude else np.arange(N)
    s, _ = util.oracle_user_scores(sd, variant, 0.5, coords, region, hist, cand)
    lg = _logg64(coords, hist, cand, a, b)
    mixed = (1 - alpha) / (1 + np.exp(-s)) + alpha * np.exp(lg - lg.max())
    # a history item whose own cell is the user's only one has the score 0 / 0: it ranks as -inf, as in the kernels' keys
    mixed = np.where(np.isnan(mixed), -np.inf, mixed)
    return dict(zip(cand.tolist(), mixed.tolist()))


def _check_lists(val, idx, ref, k, rtol=1e-4):
    """ids equal to the float64 top-k outside 1e-4 tie bands of `mixed`, values within rtol"""
    order = sorted(ref, key=lambda j: (-ref[j], j))[:k]
    got = [int(j) for j in idx if j >= 0]
    assert len(got) == min(k, len(ref))
    for r, j in enumerate(got):
        if ref[j] == ref[order[r]]:  # (equal, -inf included)
            continue
        assert abs(ref[j] - ref[order[r]]) <= rtol * abs(ref[order[r]]) + 1e-4, (r, j, order[r], ref[j], ref[order[r]])
    np.testing.assert_allclose(np.asarray(val[:len(got)], dtype=np.float64), [ref[j] for j in got], rtol=rtol, atol=1e-6)


def test_logmax_is_bit_identical_to_log_scores_max():
    for N, coords, region, indptr, indices in (_golden_arrays(), _long_catalogue()):
        m, _ = _model("region_distance", N, region, coords)
        users = m.make_users(indptr, indices)
        U = len(indptr) - 1
        for lo, hi in ((0, N), (0, 200), (130, N), (257, 300)):
            logg = PL.log_scores(m._catalog, users, A_, B_, lo, hi)
            for excl in (True, False):
                lm = ops.powerlaw_logmax(m._catalog, users, A_, B_, lo, hi, excl)
                want = logg.clone()
                if excl:
                    for u in range(U):
                        h = indices[indptr[u]:indptr[u + 1]]
                        h = h[(h >= lo) & (h < hi)] - lo
                        want[u, torch.as_tensor(h, device=want.device, dtype=torch.int64)] = float("-inf")
                want = want.max(1).values
                assert torch.equal(lm, want), (N, lo, hi, excl, lm, want)
    # a user whose every candidate is in the history: -inf
    m, _ = _model("basic", 300, np.zeros(300, np.int64), _golden()[0]["coords"])
    users = m.make_users(np.array([0, 3]), np.array([5, 6, 7]))
    lm = ops.powerlaw_logmax(m._catalog, users, A_, B_, 5, 8, True)
    assert lm.item() == float("-inf")


def _golden_arrays():
    z, U, N = _golden()
    return N, z["coords"], z["region"], z["indptr"], z["indices"]


@pytest.mark.parametrize("variant", ["region_distance", "distance", "basic", "region", "disentangled"])
@pytest.mark.parametrize("precision", ["fp32", "tc_auto", "tc_split"])
def test_fused_against_float64(variant, precision):
    N, coords, region, indptr, indices = _golden_arrays()
    m, sd = _model(variant, N, region, coords)
    U = len(indptr) - 1
    for k in (15, 40):  # the k <= 32 register top-k and the 512-key block sort
        val, idx = PL.fused_rerank_topk(m, (indptr, indices), k, A_, B_, ALPHA, precision=precision)
        assert val.dtype == torch.float32 and idx.dtype == torch.int64 and val.shape == (U, k)
        for u in range(U):
            hist = indices[indptr[u]:indptr[u + 1]]
            ref = _ref_mixed(variant, sd, coords, region, hist, N, A_, B_, ALPHA, True)
            assert not set(idx[u].tolist()) & set(hist.tolist())
            _check_lists(val[u].cpu().numpy(), idx[u].cpu().numpy(), ref, k)


@pytest.mark.parametrize("precision", ["fp32", "tc_split", "tc_auto"])
def test_fused_long_history_wide_model_and_no_exclusion(precision):
    """histories past HMETA (the __ldg fallback), a user without history, D = hid = 128 (the tensor kernel whose `comb`
    aliases A_ext), exclude_history=False (the h = j term at d = 0 counts).  A 600-term fp32 sum of log terms of ~|5| carries
    ~1e-3 absolute error into exp(logG - M): values of the 600-item user are held to 1e-3."""
    N, coords, region, indptr, indices = _long_catalogue()
    U = len(indptr) - 1
    for D in (64, 128):
        m, sd = _model("region_distance", N, region, coords, D=D, hid=D, seed=3)
        for excl in (True, False):
            val, idx = PL.fused_rerank_topk(m, (indptr, indices), 20, A_, B_, ALPHA, precision=precision, exclude_history=excl)
            for u in range(U):
                hist = indices[indptr[u]:indptr[u + 1]]
                if len(hist) == 0:  # the attention score is 0 / 0 (as in predict_topk): every candidate ranks as -inf
                    assert torch.isneginf(val[u]).all() and (idx[u] >= 0).all()
                    continue
                ref = _ref_mixed("region_distance", sd, coords, region, hist, N, A_, B_, ALPHA, excl)
                _check_lists(val[u].cpu().numpy(), idx[u].cpu().numpy(), ref, 20, rtol=1e-3 if len(hist) > 512 else 1e-4)


def test_fused_against_rerank_topk():
    N, coords, region, indptr, indices = _golden_arrays()
    m, _ = _model("region_distance", N, region, coords)
    users = m.make_users(indptr, indices)
    val, idx = PL.fused_rerank_topk(m, users, 15, A_, B_, ALPHA, precision="fp32")
    rv, ri = PL.rerank_topk(m, users, 15, A_, B_, ALPHA, precision="fp32")
    for u in range(len(indptr) - 1):
        for r in range(15):
            if int(idx[u, r]) != int(ri[u, r]):  # only inside a tie band
                assert abs(float(val[u, r]) - float(rv[u, r])) < 1e-4, (u, r)
        np.testing.assert_allclose(val[u].cpu().numpy(), rv[u].cpu().numpy(), rtol=1e-4, atol=1e-6)


@pytest.mark.parametrize("precision", ["fp32", "tc_split"])
def test_alpha_zero_is_predict_topk(precision):
    N, coords, region, indptr, indices = _golden_arrays()
    m, _ = _model("region_distance", N, region, coords)
    users = m.make_users(indptr, indices)
    val, idx = PL.fused_rerank_topk(m, users, 20, A_, B_, 0.0, precision=precision)
    pv, pi = m.predict_topk(users, 20, precision=precision + ("_generic" if precision != "fp32" else ""))
    np.testing.assert_allclose(val.cpu().numpy(), pv.cpu().numpy(), rtol=5e-7, atol=0)
    pvn = pv.cpu().numpy()
    for u in range(len(indptr) - 1):
        for r in range(20):
            distinct = (r == 0 or pvn[u, r - 1] != pvn[u, r]) and (r == 19 or pvn[u, r + 1] != pvn[u, r])
            if distinct:
                assert int(idx[u, r]) == int(pi[u, r]), (u, r)


@pytest.mark.parametrize("precision", ["fp32", "tc_auto"])
def test_simulated_sharding_is_bit_identical(precision):
    """two catalogue ranges, M = max of the two range maxima, per-range keys, topk_merge_keys == the whole-range call"""
    N, coords, region, indptr, indices = _golden_arrays()
    m, _ = _model("region_distance", N, region, coords)
    users = m.make_users(indptr, indices)
    cat, P = m._catalog, m._params()
    lm = ops.powerlaw_logmax(cat, users, A_, B_, 0, N)
    geo = ops.GeoMix(A_, B_, ALPHA, lm)
    plan = m.ranking_plan(precision)
    ws, wi = ops.fullrank_topk(m.variant, 0.5, P, cat, users, 20, 0, N, True, plan.precision, plan, geo=geo)
    keys, maxes = [], []
    for lo, hi in ((0, 128), (128, N)):
        maxes.append(ops.powerlaw_logmax(cat, users, A_, B_, lo, hi))
    M = torch.maximum(maxes[0], maxes[1])
    assert torch.equal(M, lm)
    for lo, hi in ((0, 128), (128, N)):
        pl = m.ranking_plan(precision, lo, hi)
        keys.append(ops.fullrank_topk(m.variant, 0.5, P, cat, users, 20, lo, hi, True, pl.precision, pl, return_keys=True,
                                      geo=ops.GeoMix(A_, B_, ALPHA, M)))
    ss, si = ops.topk_merge_keys(torch.stack(keys))
    assert torch.equal(ss, ws) and torch.equal(si, wi)


def test_repeated_planned_call_is_identical():
    N, coords, region, indptr, indices = _golden_arrays()
    m, _ = _model("disentangled", N, region, coords)
    users = m.make_users(indptr, indices)
    a = PL.fused_rerank_topk(m, users, 20, A_, B_, ALPHA, precision="tc_auto")
    b = PL.fused_rerank_topk(m, users, 20, A_, B_, ALPHA, precision="tc_auto")
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def test_no_users_by_catalogue_buffer():
    """C2-shaped call (40 000 POIs, H = 128): no allocation beyond the planned call's workspace + O(U k) (the plan is built by
    the warm-up call), so no [U, N] buffer"""
    rng = np.random.default_rng(1)
    N, U, H, k = 40000, 256, 128, 20
    coords = np.stack([40.7 + rng.normal(0, 0.1, N), -74.0 + rng.normal(0, 0.1, N)], 1)
    region = rng.integers(0, 50, N)
    m, _ = _model("region_distance", N, region, coords)
    indptr = np.arange(U + 1, dtype=np.int64) * H
    indices = rng.integers(0, N, U * H)
    users = m.make_users(indptr, indices)
    plan = m.ranking_plan("tc_auto")
    PL.fused_rerank_topk(m, users, k, A_, B_, ALPHA, precision="tc_auto")  # warm
    torch.cuda.synchronize()
    from poi_recommendation_models_b200 import _lib
    lib = _lib.load()
    p = ops.build_params(m.variant, m._params(), 0.5, [])
    ws = lib.nais_fullrank_planned_workspace_bytes(ops.C.byref(p), U, U * H, 0, N, k, ops.PRECISIONS[plan.precision])
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    PL.fused_rerank_topk(m, users, k, A_, B_, ALPHA, precision="tc_auto")
    torch.cuda.synchronize()
    extra = torch.cuda.max_memory_allocated() - base
    assert extra <= ws + U * k * 16 + U * 4 + (1 << 20), (extra, ws)  # < ws + one [U, N] fp32 matrix (41 MB)
