"""The two-branch NAIS_region_distance_disentangled_Embedding (model.py:410-541) on the tcgen05 pair kernels (csrc/nais_pairs_tc.cu,
csrc/nais_pairs_tc_bwd.cu: one launch per branch, the haversine-km logit term as the kKm instantiations): dispatch, forward and
backward against the float64 oracle with the bars of the one-branch classes, the per-branch ReLU pattern, and the fused training
paths against the FP32 kernels, dense autograd and the exact-order references."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

import nais_testutil as util
import test_gpu_disentangled_train as dtrain
import test_gpu_segment_reduce as sred
from oracle import nais_oracle as orc
from poi_recommendation_models_b200 import batches as PB, model as M, ops, synthetic

pytestmark = pytest.mark.gpu
V = "disentangled"


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _km(coords, tgt, hist):
    return orc.dist_km(coords[tgt][:, None, 0], coords[tgt][:, None, 1], coords[hist][..., 0], coords[hist][..., 1]).astype(np.float32)


def _case(N, D, hid, B, H, seed, n_dist=1):
    """Parameters and a dense batch whose every third row targets an item of its own history (a live mask)."""
    rng = np.random.default_rng(seed)
    coords, region, R = synthetic.make_catalog(N, seed=seed)
    sd = orc.init_state(V, N, D, hid, R, n_dist, seed=seed + 1, style="trained")
    hist = np.stack([rng.choice(N, H, replace=False) for _ in range(B)]).astype(np.int64)
    tgt = rng.integers(0, N, B).astype(np.int64)
    if H > 1:
        tgt[::3] = hist[::3, H // 2]
    return sd, hist, tgt, region, _km(coords, tgt, hist)


def _model(sd, beta=0.5):
    N, D = sd["embed_history.weight"].shape
    m = M.CLASSES[V](N, D, sd["attn_layer1.weight"].shape[0], beta, sd["embed_region.weight"].shape[0], sd["embed_distance.weight"].shape[0])
    m.load_state_dict(sd, strict=True)
    return m.cuda().eval()


def _ref(sd, beta, hist, tgt, region, km):
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    s, scale = orc.attention_network_with_scale(sd, V, beta, t(hist), t(tgt), t(region[hist]), t(region[tgt]), t(km), dtype=torch.float64)
    return s.numpy(), scale.numpy()


def _segmented(D, hid, seed, N=800):
    """Nine users: user 1 without history (a segment without tiles), user 4 with 140 items (one-row tiles, two chunks)."""
    data = synthetic.make_checkins(9, N, seed=seed, hist_len=None, max_hist=60, min_hist=2, median_hist=14)
    rows = [data.history(u) for u in range(9)]
    rows[1], rows[4] = rows[1][:0], np.random.default_rng(seed + 2).choice(N, 140, replace=False)
    csr = sp.csr_matrix((np.ones(sum(map(len, rows))), (np.repeat(np.arange(9), [len(r) for r in rows]), np.concatenate(rows))),
                        shape=(9, N))
    bt = PB.DeviceBatcher(csr, data.region, data.coords, device="cuda", seed=0)
    b = bt.multi_user_batch(np.arange(9), 4, seed=9)
    sd = orc.init_state(V, N, D, hid, data.region_num, 1, seed=seed + 1, style="trained")
    return data, csr, b, sd


def _per_user(data, csr, b):
    """(row slice, hist, tgt, km) of every segment with history, in the reference's dense form."""
    ro, tgt_all = b.host_row_offsets, b.tgt.cpu().numpy()
    for s in range(len(ro) - 1):
        hist = csr.getrow(s).indices.astype(np.int64)
        if ro[s + 1] == ro[s] or len(hist) == 0:
            continue
        tgt = tgt_all[ro[s]:ro[s + 1]]
        hh = np.broadcast_to(hist, (len(tgt), len(hist))).copy()
        yield slice(ro[s], ro[s + 1]), hh, tgt, _km(data.coords, tgt, hh)


def _params_struct(sd, batch, pp, dist):
    keep = []
    P = {n: sd[n].cuda().contiguous() for n in ops.VARIANT_PARAMS[V]}
    p = ops.build_params(V, P, 0.5, keep, pairs_precision=pp)
    if dist == "none":
        p.dist_mode = 0  # NAIS_DIST_NONE
    return p, ops._pairs_struct(*batch, keep), keep


# ---- 1. dispatch ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dist", ["km", "none"])
@pytest.mark.parametrize("layout", ["dense", "segmented"])
@pytest.mark.parametrize("D,hid", [(64, 64), (32, 64), (32, 32)])
def test_dispatch_picks_the_tensor_kernels(D, hid, layout, dist):
    """Both directions on tcgen05 wherever both have kernels; the backward's exist for hid = 64 only."""
    if layout == "dense":
        sd, hist, tgt, region, km = _case(300, D, hid, 8, 11, seed=D)
        batch = (_dev(hist), _dev(tgt), _dev(region[hist]), _dev(region[tgt]), _dev(km) if dist == "km" else None)
    else:
        _, _, b, sd = _segmented(D, hid, seed=D)
        batch = (b, None, None, None, None)
    for pp, want in (("auto", (True, hid == 64)), ("tc", (True, hid == 64)), ("fp32", (False, False))):
        p, b_, _keep = _params_struct(sd, batch, pp, dist)
        assert ops.pairs_dispatch(p, b_) == want, (pp, D, layout, dist)


def test_hid_128_forces_no_tensor_backward():
    sd, hist, tgt, region, km = _case(300, 64, 128, 8, 11, seed=5)
    batch = (_dev(hist), _dev(tgt), _dev(region[hist]), _dev(region[tgt]), _dev(km))
    p, b, _keep = _params_struct(sd, batch, "tc", "km")
    assert ops.pairs_dispatch(p, b) == (True, False)
    m = _model(sd)
    m.pairs_precision = "tc"
    s = m.attention_network(*batch)
    with pytest.raises(RuntimeError, match="unsupported or inconsistent dimension"):
        s.sum().backward()
        torch.cuda.synchronize()


# ---- 2. forward -------------------------------------------------------------------------------------------------------------
def _three(m, fn):
    out = {}
    with torch.no_grad():
        for pp in ("tc", "auto", "fp32"):
            m.pairs_precision = pp
            out[pp] = fn().cpu().numpy()
    assert np.array_equal(out["tc"], out["auto"]), "auto must pick the tensor-core kernels"
    return out


@pytest.mark.parametrize("H", [1, 3, 13, 100, 128, 129, 300])
def test_forward_history_lengths(H):
    sd, hist, tgt, region, km = _case(900, 64, 64, 37, H, seed=H)
    m = _model(sd)
    args = (_dev(hist), _dev(tgt), _dev(region[hist]), _dev(region[tgt]), _dev(km))
    out = _three(m, lambda: m.attention_network(*args))
    ref, scale = _ref(sd, 0.5, hist, tgt, region, km)
    assert not np.array_equal(out["tc"], out["fp32"]) or H == 1, "the tensor-core path did not run"
    e_tc, e_fp = util.cond_err(out["tc"], ref, scale), util.cond_err(out["fp32"], ref, scale)
    assert e_tc < util.TOL and e_tc <= max(4 * e_fp, 5e-6), (e_tc, e_fp)


@pytest.mark.parametrize("D,hid", [(32, 32), (16, 48), (48, 64), (64, 128)])
def test_forward_shapes(D, hid):
    sd, hist, tgt, region, km = _case(500, D, hid, 120, 21, seed=D + hid)
    m = _model(sd, beta=0.7)
    args = (_dev(hist), _dev(tgt), _dev(region[hist]), _dev(region[tgt]), _dev(km))
    out = _three(m, lambda: m.attention_network(*args))
    ref, scale = _ref(sd, 0.7, hist, tgt, region, km)
    e_tc, e_fp = util.cond_err(out["tc"], ref, scale), util.cond_err(out["fp32"], ref, scale)
    assert e_tc < util.TOL and e_tc <= max(4 * e_fp, 5e-6), (e_tc, e_fp)


@pytest.mark.parametrize("D", [32, 64])
def test_forward_segmented(D):
    data, csr, b, sd = _segmented(D, D, seed=3)
    m = _model(sd)
    out = _three(m, lambda: m.segmented_scores(b))
    assert not np.array_equal(out["tc"], out["fp32"])
    e_tc = e_fp = 0.0
    for sl, hh, tgt, km in _per_user(data, csr, b):
        ref, scale = _ref(sd, 0.5, hh, tgt, data.region, km)
        e_tc = max(e_tc, util.cond_err(out["tc"][sl], ref, scale))
        e_fp = max(e_fp, util.cond_err(out["fp32"][sl], ref, scale))
    assert e_tc < util.TOL and e_tc <= max(4 * e_fp, 5e-6), (e_tc, e_fp)


# ---- 3. backward ------------------------------------------------------------------------------------------------------------
def _grads(m, pp, fn, dscore):
    m.zero_grad(set_to_none=True)
    m.pairs_precision = pp
    (fn() * dscore).sum().backward()
    ops.check_indices(sync=True)
    return {n: p.grad.detach().cpu().double().numpy() for n, p in m.named_parameters()}


def _assert_grads(g, ref, what):
    for name, r in ref.items():
        r = np.asarray(r, dtype=np.float64)
        assert np.abs(r).max() > 0, (what, name)
        err = float(np.abs(g[name] - r).max() / np.abs(r).max())
        assert err <= 2e-4, (what, name, err)


@pytest.mark.parametrize("B,H,D", [(256, 128, 64), (150, 21, 64), (40, 300, 64), (100, 50, 32), (40, 129, 32), (40, 300, 32)])
def test_backward_dense_matches_the_oracle(B, H, D):
    sd, hist, tgt, region, km = _case(3000, D, 64, B, H, seed=B + H, n_dist=3)
    m = _model(sd)
    m.train()
    args = (_dev(hist), _dev(tgt), _dev(region[hist]), _dev(region[tgt]), _dev(km))
    dscore = np.random.default_rng(7).normal(size=B)
    g_tc = _grads(m, "tc", lambda: m.attention_network(*args), _dev(dscore).float())
    g_fp = _grads(m, "fp32", lambda: m.attention_network(*args), _dev(dscore).float())
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    _, ref = orc.grads(sd, V, 0.5, t(hist), t(tgt), t(region[hist]), t(region[tgt]), t(km), t(dscore))
    ref = {k: v.numpy() for k, v in ref.items()}
    for n in ("attn_layer1.weight", "region_attn_layer1.weight"):
        assert not np.array_equal(g_tc[n], g_fp[n]), "the tensor-core backward did not run"
    assert np.all(g_tc["embed_distance.weight"][1:] == 0), "rows 1.. of embed_distance are never read"
    ref["embed_distance.weight"] = ref["embed_distance.weight"][:1]
    g_tc["embed_distance.weight"] = g_tc["embed_distance.weight"][:1]
    _assert_grads(g_tc, ref, ("dense", B, H, D))


def _segmented_cells(b):
    """(history POI id, target POI id) of every cell of a segmented batch, in cell order (include/nais_b200.h)."""
    so, ro = b.seg_offsets.cpu().numpy(), b.host_row_offsets
    hflat, tgt = b.hist.cpu().numpy(), b.tgt.cpu().numpy()
    hc = [hflat[so[s]:so[s + 1]] for s in range(len(ro) - 1) for _ in range(ro[s], ro[s + 1])]
    tc = [np.full(so[s + 1] - so[s], tgt[r]) for s in range(len(ro) - 1) for r in range(ro[s], ro[s + 1])]
    hc, tc = (np.concatenate(v) if v else np.zeros(0, np.int64) for v in (hc, tc))
    assert len(hc) == b.n_cells
    return hc, tc


FWD_KINK = 2e-7  # the fp16-split forward's pre-activations are within ~2e-7 of sum_d |W_kd x_d| + |b_k| (DESIGN.md section 3)


@pytest.mark.parametrize("D", [32, 64])
def test_backward_segmented_matches_the_oracle(D):
    """Every gradient of a segmented batch (a user without history, one of 140 items: two-chunk tiles) against the float64
    oracle.  The backward takes the ReLU step from act_mask, so a unit whose pre-activation lies within the forward's own error
    of the kink may take the other side than float64 and move the gradients by that cell's whole contribution (at D = 32 on this
    batch: 2 of 6.9 M units, at |t| <= 5.3e-8 of their scale, give 4.5e-4 of max|d attn_layer1.weight|).  So: the forward's
    pattern must equal float64's sign outside that band; the backward, given float64's pattern, must meet the bar; and the whole
    path (forward pattern included) must meet it when no unit fell inside the band."""
    data, csr, b, sd = _segmented(D, 64, seed=4)
    P = {n: sd[n].cuda().contiguous() for n in ops.VARIANT_PARAMS[V]}
    batch = (b, None, None, None, None)
    dscore = torch.from_numpy(np.random.default_rng(2).normal(size=b.B).astype(np.float32)).cuda()
    G = None
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    for sl, hh, tgt, km in _per_user(data, csr, b):
        _, gu = orc.grads(sd, V, 0.5, t(hh), t(tgt), t(data.region[hh]), t(data.region[tgt]), t(km), dscore[sl].cpu())
        G = gu if G is None else {k: G[k] + gu[k] for k in G}
    G = {k: v.numpy() for k, v in G.items()}
    # the forward's saved pattern against float64's
    _, row_sum, parts, mask = ops.pairs_forward_raw(V, 0.5, P, *batch, (0.0, 0, "tc"))
    words = mask.cpu().numpy().view(np.uint64).reshape(2, -1)
    hc, tc = _segmented_cells(b)
    Eh, Et, Er = (sd[n].numpy() for n in ("embed_history.weight", "embed_target.weight", "embed_region.weight"))
    exact, in_band = [], 0
    for bi, (prefix, q, p) in enumerate([("", Eh[hc], Et[tc]), ("region_", Er[data.region[hc]], Er[data.region[tc]])]):
        t64, scale = _t64(sd, prefix, q, p)
        bits = ((words[bi][:, None] >> np.arange(64, dtype=np.uint64)) & np.uint64(1)).astype(bool)
        off = bits != (t64 > 0)
        assert np.all(np.abs(t64[off]) <= FWD_KINK * scale[off]), (bi, np.abs(t64[off]).max())
        in_band += int(off.sum())
        exact.append(((t64 > 0).astype(np.uint64) << np.arange(64, dtype=np.uint64)).sum(1).astype(np.uint64).view(np.int64))
    # the backward on float64's pattern
    am = torch.from_numpy(np.concatenate(exact)).cuda()
    g = ops.pairs_backward_raw(V, 0.5, P, *batch, row_sum, parts, dscore, (0.0, 0, "tc"), act_mask=am)
    _assert_grads({n: v.double().cpu().numpy() for n, v in g.items()}, G, ("segmented, float64 pattern", D))
    if in_band == 0:  # the whole path: the model's autograd step on the forward's own pattern
        m = _model(sd)
        _assert_grads(_grads(m, "tc", lambda: m.segmented_scores(b), dscore), G, ("segmented", D))


def _t64(sd, prefix, q, p):
    """float64 pre-activations W x + b of a branch for x = q (.) p: [cells, hid]"""
    x = q.astype(np.float64) * p.astype(np.float64)
    W, b1 = sd[prefix + "attn_layer1.weight"].double().numpy(), sd[prefix + "attn_layer1.bias"].double().numpy()
    return x @ W.T + b1, np.abs(x) @ np.abs(W).T + np.abs(b1)


def test_act_mask_holds_both_branches():
    B, H = 64, 40
    sd, hist, tgt, region, km = _case(2000, 64, 64, B, H, seed=17)
    P = {n: sd[n].cuda().contiguous() for n in ops.VARIANT_PARAMS[V]}
    batch = (_dev(hist), _dev(tgt), _dev(region[hist]), _dev(region[tgt]), _dev(km))
    _, _, _, mask = ops.pairs_forward_raw(V, 0.5, P, *batch, (0.0, 0, "tc"))
    assert mask is not None and mask.numel() == 2 * B * H
    words = mask.cpu().numpy().view(np.uint64).reshape(2, B * H)
    Eh, Et, Er = (sd[n].numpy() for n in ("embed_history.weight", "embed_target.weight", "embed_region.weight"))
    cases = [("", Eh[hist.reshape(-1)], np.repeat(Et[tgt], H, 0)), ("region_", Er[region[hist].reshape(-1)], np.repeat(Er[region[tgt]], H, 0))]
    for bi, (prefix, q, p) in enumerate(cases):
        t, scale = _t64(sd, prefix, q, p)
        bits = ((words[bi][:, None] >> np.arange(64, dtype=np.uint64)) & np.uint64(1)).astype(bool)
        far = np.abs(t) > 1e-5 * scale  # (units on the kink may go either way)
        assert np.array_equal(bits[far], (t > 0)[far]), bi
    assert not np.array_equal(words[0], words[1])
    # a one-branch model's pattern keeps its size
    _, h1, t1, r1, _ = _case(500, 64, 64, 16, 9, seed=2)
    coords, _, R1 = synthetic.make_catalog(500, seed=2)
    ll = orc.latlon_abs_diff(coords, t1, h1).astype(np.float32)
    sd1 = orc.init_state("region_distance", 500, 64, 64, R1, 1, seed=3, style="trained")
    P1 = {n: sd1[n].cuda().contiguous() for n in ops.VARIANT_PARAMS["region_distance"]}
    _, _, _, m1 = ops.pairs_forward_raw("region_distance", 0.5, P1, _dev(h1), _dev(t1), _dev(r1[h1]), _dev(r1[t1]), _dev(ll), (0.0, 0, "tc"))
    assert m1.numel() == 16 * 9


# ---- 4. the per-branch ReLU pattern -------------------------------------------------------------------------------------------
def _bf16(v):
    u = np.ascontiguousarray(v, dtype=np.float32).view(np.uint32).astype(np.uint64)
    u = (u + np.uint64(0x7FFF) + ((u >> np.uint64(16)) & np.uint64(1))) & np.uint64(0xFFFF0000)
    return u.astype(np.uint32).view(np.float32)


def _split(v, rnd):
    hi = rnd(v)
    return hi, rnd((v.astype(np.float32) - hi).astype(np.float32))


def _pow2(amax):  # pow2_scale(amax, 9) of the forward: amax * s in [256, 512)
    return 2.0 ** (9 - np.frexp(amax)[1])


def _three_term(W, x, rnd):
    (wh, wl), (xh, xl) = _split(W, rnd), _split(x, rnd)
    return wh.astype(np.float64) @ xh + wl.astype(np.float64) @ xh + wh.astype(np.float64) @ xl


def test_branch_1_takes_its_relu_pattern_from_the_forward():
    """Hidden units of branch 1 at one cell are put on the kink's far side from the error of a bf16 two-term recompute of W x
    (the tcgen05 backward's operands), at half that error — many times the error of the fp16-split forward, which therefore
    saves the exact pattern.  A backward that thresholded its own recompute (or read branch 0's words) would flip those units
    and move the region MLP's gradients by that cell's whole contribution."""
    B, H, cell_r, cell_h = 2, 6, 0, 2
    sd, hist, tgt, region, km = _case(200, 64, 64, B, H, seed=31)
    assert hist[cell_r, cell_h] != tgt[cell_r]  # a live cell
    Er = sd["embed_region.weight"].numpy()
    x = (Er[region[hist[cell_r, cell_h]]] * Er[region[tgt[cell_r]]]).astype(np.float32)  # the kernels' fp32 products
    W = sd["region_attn_layer1.weight"].numpy()
    exact = W.astype(np.float64) @ x.astype(np.float64)
    S = np.abs(W).astype(np.float64) @ np.abs(x)
    e_bwd = _three_term(W, x, _bf16) - exact
    sx, sw = _pow2(np.abs(x).max()), _pow2(np.abs(W).max())
    f16 = lambda v: v.astype(np.float16).astype(np.float32)
    e_fwd = _three_term((W * sw).astype(np.float32), (x * sx).astype(np.float32), f16) / (sx * sw) - exact
    sel = np.abs(e_bwd) / 2 > 4 * np.abs(e_fwd) + 5e-7 * S  # (5e-7 S: room for the forward's fp32 accumulation in TMEM)
    assert sel.sum() >= 4, sel.sum()
    b1 = sd["region_attn_layer1.bias"].numpy().astype(np.float64)
    b1 = np.where(sel, -np.sign(e_bwd) * np.abs(e_bwd) / 2 - exact, b1).astype(np.float32)
    sd = dict(sd)
    sd["region_attn_layer1.bias"] = torch.from_numpy(b1)
    t_exact = exact + b1.astype(np.float64)
    flips = sel & (np.sign(t_exact) != np.sign(exact + e_bwd + b1.astype(np.float64)))
    assert flips.sum() == sel.sum()
    m = _model(sd)
    args = (_dev(hist), _dev(tgt), _dev(region[hist]), _dev(region[tgt]), _dev(km))
    P = {n: sd[n].cuda().contiguous() for n in ops.VARIANT_PARAMS[V]}
    _, _, _, mask = ops.pairs_forward_raw(V, 0.5, P, *args, (0.0, 0, "tc"))
    w1 = int(mask.cpu().numpy().view(np.uint64)[B * H + cell_r * H + cell_h])
    sure = sel | (np.abs(t_exact) > 1e-5 * S)
    bits = np.array([(w1 >> k) & 1 for k in range(64)], dtype=bool)
    assert np.array_equal(bits[sure], (t_exact > 0)[sure]), "the forward's pattern is not the exact one"
    dscore = np.array([1.0, 0.1])
    g = _grads(m, "tc", lambda: m.attention_network(*args), _dev(dscore).float())
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    _, ref = orc.grads(sd, V, 0.5, t(hist), t(tgt), t(region[hist]), t(region[tgt]), t(km), t(dscore))
    _assert_grads(g, {k: v.numpy() for k, v in ref.items()}, "kink")


# ---- 5. fused paths -----------------------------------------------------------------------------------------------------------
def _models(N, R, n, seed=1):
    sd = orc.init_state(V, N, 64, 64, R, 1, seed=seed, style="trained")
    ms = [util.make_model(V, sd, 0.5).train() for _ in range(n)]
    # a warm accumulator: Adagrad's first step moves an element by +-lr whatever |g| is, so a rounding-level gradient difference
    # near 0 would flip it; with sum > 0 the step is continuous in g
    return ms, [torch.optim.Adagrad(m.parameters(), lr=0.05, initial_accumulator_value=0.1) for m in ms]


@pytest.mark.parametrize("loss", ["bce", "bpr"])
@pytest.mark.parametrize("layout", ["dense", "segmented"])
def test_one_call_step_on_the_tensor_kernels(layout, loss):
    N, num_ng = 900, 4
    data = dtrain._data(12, N, seed=3, max_hist=40, min_hist=3)
    (m_tc, m_fp, m_ref), (o_tc, o_fp, o_ref) = _models(N, data.region_num, 3)
    m_fp.pairs_precision = "fp32"
    m_ref.one_call = False  # autograd through the pair kernels + torch.optim.Adagrad (the op-by-op path)
    bt = PB.DeviceBatcher(data.train_csr(), data.region, data.coords, device="cuda", seed=0)
    for it in range(5):
        dtrain._sync_from(m_fp, o_fp, m_tc, o_tc)
        dtrain._sync_from(m_ref, o_ref, m_tc, o_tc)
        if layout == "dense":
            h, tg, lab, hr, tr, _ = bt.batch(it, num_ng)
            kmt = PB.dist_km_pairs(data.coords, tg.cpu().numpy(), h.cpu().numpy(), device="cuda")
            args = (h, tg, hr, tr, kmt)
            p, b, _keep = _params_struct({k: v.detach() for k, v in m_tc.state_dict().items()}, args, "auto", "km")
        else:
            b_ = bt.multi_user_batch(np.arange(3 * it, 3 * it + 3) % 12, num_ng, seed=it)
            args, lab = (b_,), b_.label
            p, b, _keep = _params_struct({k: v.detach() for k, v in m_tc.state_dict().items()}, (b_, None, None, None, None), "auto", "km")
        assert ops.pairs_dispatch(p, b) == (True, True)
        for m, o in ((m_tc, o_tc), (m_fp, o_fp), (m_ref, o_ref)):
            if loss == "bce":
                m.fused_adagrad_step(o, lab, *args)
            else:
                m.fused_bpr_step(o, *args, num_neg=num_ng)
        dtrain._close(m_tc, o_tc, m_fp, o_fp, 1e-4, f"{layout} {loss} step {it}: auto vs fp32")
        dtrain._close(m_tc, o_tc, m_ref, o_ref, 1e-4, f"{layout} {loss} step {it}: one call vs autograd")
    ops.check_indices(sync=True)


def test_fused_table_step_is_rows_adagrad_ref_of_the_dense_gradients():
    N = 700
    batch, R = sred._segmented_batch(V, N, seed=3)
    sred._fused_equals_dense_then_ref(V, 64, 64, batch, R, N, "tc", seed=3)
    sred._fused_equals_dense_then_ref(V, 32, 64, batch, R, N, "tc", seed=4)
    sd, hist, tgt, region, km = _case(N, 64, 64, 200, 33, seed=6)
    dense = (_dev(hist), _dev(tgt), _dev(region[hist]), _dev(region[tgt]), _dev(km))
    sred._fused_equals_dense_then_ref(V, 64, 64, dense, int(region.max()) + 1, N, "tc", seed=6)


def test_one_step_is_reproducible():
    N = 900
    data = dtrain._data(12, N, seed=5, max_hist=60, min_hist=3)
    (m1, m2), (o1, o2) = _models(N, data.region_num, 2)
    bt = PB.DeviceBatcher(data.train_csr(), data.region, data.coords, device="cuda", seed=0)
    b = bt.multi_user_batch(np.arange(12), 4, seed=1)
    l1, l2 = m1.fused_adagrad_step(o1, b.label, b), m2.fused_adagrad_step(o2, b.label, b)
    assert float(l1) == float(l2)
    for (n, a), (_, c) in zip(m1.named_parameters(), m2.named_parameters()):
        assert torch.equal(a, c), n
        assert torch.equal(o1.state[a]["sum"], o2.state[c]["sum"]), n


@pytest.mark.parametrize("loss", ["bce", "bpr"])
def test_train_users_is_the_per_user_loop_bit_for_bit(loss):
    N = 1500
    data = dtrain._data(30, N, seed=11, max_hist=140, min_hist=0)
    (m_all, m_loop), (o_all, o_loop) = _models(N, data.region_num, 2)
    bt = PB.DeviceBatcher(data.train_csr(), data.region, data.coords, device="cuda", seed=0)
    uids = np.array([3, 7, 0, 12, 29, 5, 5, 18, 21, 9])
    b0 = bt.multi_user_batch(np.array([3]), 4, seed=1)
    p, b, _keep = _params_struct({k: v.detach() for k, v in m_all.state_dict().items()}, (b0, None, None, None, None), "auto", "km")
    assert ops.pairs_dispatch(p, b) == (True, True)
    losses = m_all.train_users(o_all, bt, uids, 4, seed=77, loss=loss)
    ref = []
    for u in uids:
        if bt.indptr[u + 1] == bt.indptr[u]:
            ref.append(0.0)
            continue
        bu = bt.multi_user_batch(np.array([u]), 4, seed=77 + int(u))
        ref.append(float(m_loop.fused_adagrad_step(o_loop, bu.label, bu) if loss == "bce" else m_loop.fused_bpr_step(o_loop, bu, num_neg=4)))
    ops.check_indices(sync=True)
    assert np.array_equal(losses.cpu().numpy(), np.array(ref, dtype=np.float32)), (losses.cpu().numpy(), ref)
    for (n, pa), (_, pb) in zip(m_all.named_parameters(), m_loop.named_parameters()):
        assert torch.equal(pa, pb), n
        assert torch.equal(o_all.state[pa]["sum"], o_loop.state[pb]["sum"]), n


# ---- 6. ids -------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D", [32, 64])
def test_out_of_range_region_id_raises_and_moves_no_region_row(D):
    N = 600
    data = dtrain._data(6, N, seed=2, max_hist=30, min_hist=3)
    sd = orc.init_state(V, N, D, 64, data.region_num, 1, seed=1, style="trained")
    m = util.make_model(V, sd, 0.5).train()
    m.pairs_precision = "tc"
    o = torch.optim.Adagrad(m.parameters(), lr=0.05)
    bt = PB.DeviceBatcher(data.train_csr(), data.region, data.coords, device="cuda", seed=0)
    b = bt.multi_user_batch(np.arange(6), 4, seed=3)
    b.treg = b.treg.clone()
    b.treg[5] = data.region_num + 7
    ops.check_indices(sync=True)
    before = m.embed_region.weight.detach().clone()
    ok_rows = torch.cat([b.hreg, b.treg[b.treg < data.region_num]]).unique()
    m.fused_adagrad_step(o, b.label, b)
    with pytest.raises(IndexError):
        ops.check_indices(sync=True)
    untouched = torch.ones(data.region_num, dtype=torch.bool, device="cuda")
    untouched[ok_rows] = False
    assert torch.equal(m.embed_region.weight[untouched], before[untouched])
    assert torch.isfinite(m.embed_region.weight).all()
