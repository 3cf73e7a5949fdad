"""Train-mode dropout of NAIS_basic / NAIS_regionEmbedding (model.py:71,162) on the fast training paths: the tcgen05 pair kernels,
segmented multi-user batches and `train_users`.  Masks are replayed on the host (ops.dropout_keep_mask[_cells]) and handed to the
float64 oracle as `l1_scale`."""
import numpy as np
import pytest
import torch

import nais_testutil as util
from oracle import nais_oracle as orc
from poi_recommendation_models_b200 import _lib, batches as PB, ops, synthetic

pytestmark = pytest.mark.gpu

P_DROP = 0.5


def _setup(variant, D, hid, U=9, N=700, seed=3, max_hist=60):
    data = synthetic.make_checkins(U, N, seed=seed, hist_len=None, max_hist=max_hist, min_hist=2, median_hist=14)
    sd = orc.init_state(variant, N, D, hid, data.region_num, 1, seed=4, style="trained")
    bt = PB.DeviceBatcher(data.train_csr(), data.region, data.coords, device="cuda", seed=0)
    return data, sd, bt


def _dense_rows(data, csr_hist, tgt):
    hh = np.broadcast_to(csr_hist, (len(tgt), len(csr_hist))).copy()
    return hh, data.region[hh], data.region[tgt]


def _oracle(sd, variant, hist, tgt, hreg, treg, scale, P=None):
    P = P if P is not None else {k: v.double().requires_grad_(True) for k, v in sd.items()}
    s = orc.attention_network(P, variant, 0.5, torch.from_numpy(hist), torch.from_numpy(tgt), torch.from_numpy(hreg),
                              torch.from_numpy(treg), None, dtype=torch.float64, l1_scale=torch.from_numpy(scale))
    return s, P


def _t1(sd, variant, hist, tgt, hreg, treg):
    """float64 pre-activation of attn_layer1 [B,H,hid] (no distance lanes: basic / region)."""
    P = {k: v.double() for k, v in sd.items()}
    q, p = P["embed_history.weight"][torch.from_numpy(hist)], P["embed_target.weight"][torch.from_numpy(tgt)]
    if variant == "region":
        q = torch.cat((q, P["embed_region.weight"][torch.from_numpy(hreg)]), -1)
        p = torch.cat((p, P["embed_region.weight"][torch.from_numpy(treg)]), -1)
    return (q * p[:, None, :]) @ P["attn_layer1.weight"].T + P["attn_layer1.bias"]


def _check_grads(m, P, tol=2e-4):
    for n, p in m.named_parameters():
        ref = P[n].grad.numpy() if P[n].grad is not None else np.zeros(tuple(p.shape))
        got = p.grad.detach().cpu().double().numpy() if p.grad is not None else np.zeros_like(ref)
        scale = max(np.abs(ref).max(), 1e-30)
        assert np.abs(got - ref).max() <= tol * scale, (n, np.abs(got - ref).max() / scale)


def _args(variant, hist, tgt, hreg, treg):
    """the arguments of attention_network"""
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return (d(hist), d(tgt)) if variant == "basic" else (d(hist), d(tgt), d(hreg), d(treg))


def _pair_args(variant, hist, tgt, hreg, treg):
    """(hist, tgt, hreg, treg, aux) of the ops entry points"""
    a = _args(variant, hist, tgt, hreg, treg)
    return a + (None, None, None) if variant == "basic" else a + (None,)


def _params_struct(D, hid, pp="auto"):
    p = _lib.NaisParams()
    p.n_branch, p.hid, p.item_num, p.region_num, p.dist_mode, p.beta = 1, hid, 1000, 10, _lib.DIST_NONE, 0.5
    br = p.branch[0]
    br.w_poi, br.w_reg = D // 2, D // 2
    br.hist_poi = br.tgt_poi = br.hist_reg = br.tgt_reg = br.w1 = br.b1 = br.w2 = 256  # (aligned; nothing is launched)
    p.dropout_p, p.dropout_seed, p.pairs_precision = P_DROP, 1, _lib.PAIRS_PRECISIONS[pp]
    return p


def test_dispatch_takes_the_tensor_kernels_with_dropout():
    b = _lib.NaisPairs()
    b.B, b.H = 1, 5
    for D in (16, 32, 48, 64):
        for hid in (32, 64, 128):
            f, g = ops.pairs_dispatch(_params_struct(D, hid), b)
            assert f, (D, hid)
            assert g == (D in (32, 64) and hid == 64), (D, hid)
            f, g = ops.pairs_dispatch(_params_struct(D, hid, "fp32"), b)
            assert not f and not g


@pytest.mark.parametrize("variant,D", [("basic", 64), ("region", 64), ("basic", 32), ("region", 32)])
def test_tc_dense_scores_gradients_and_saved_mask(variant, D):
    """D = 64: the two-threads-per-cell kernels; D = 32: the run-time-shape forward and the 128-thread backward (hid = 64)."""
    hid = 64
    data, sd, bt = _setup(variant, D, hid)
    rng = np.random.default_rng(5)
    hist = data.history(0).astype(np.int64)
    tgt = rng.integers(0, 700, 3 * len(hist)).astype(np.int64)
    tgt[::5] = hist[0]
    hist, hreg, treg = _dense_rows(data, hist, tgt)
    B, H = hist.shape
    m = util.make_model(variant, sd, 0.5).train()
    m.pairs_precision = "tc"
    torch.manual_seed(11)
    s = m.attention_network(*_args(variant, hist, tgt, hreg, treg))
    dscore = rng.normal(size=B)
    (s * torch.from_numpy(dscore).cuda().float()).sum().backward()
    keep = ops.dropout_keep_mask(m.last_dropout_seed, B, H, hid, P_DROP)
    ref, P = _oracle(sd, variant, hist, tgt, hreg, treg, keep / (1 - P_DROP))
    (ref * torch.from_numpy(dscore)).sum().backward()
    np.testing.assert_allclose(s.detach().cpu().double().numpy(), ref.detach().numpy(), rtol=1e-4, atol=1e-6)
    _check_grads(m, P)
    # the saved pattern: active AND kept, bit k of word b*H + h
    P32 = m._params()
    _, _, _, mask = ops.pairs_forward_raw(variant, 0.5, P32, *_pair_args(variant, hist, tgt, hreg, treg),
                                          drop=(P_DROP, m.last_dropout_seed, "tc"))
    bits = (mask.cpu().numpy().view(np.uint64)[:, None] >> np.arange(hid, dtype=np.uint64)) & np.uint64(1)
    t1 = _t1(sd, variant, hist, tgt, hreg, treg).numpy().reshape(B * H, hid)
    want = (t1 > 0) & keep.reshape(B * H, hid)
    far = np.abs(t1) > 1e-5  # (units on the kink may go either way)
    assert np.array_equal(bits.astype(bool)[far], want[far])
    assert 0.4 < keep.mean() < 0.6 and want.mean() < keep.mean()


@pytest.mark.parametrize("variant", ["basic", "region"])
def test_backward_without_the_saved_mask(variant):
    """With dropout the tcgen05 backward takes the mask from act_mask: without one, "auto" runs the FP32 backward (it regenerates
    the mask) and "tc" refuses (NAIS_ERR_NULL)."""
    D = hid = 64
    data, sd, bt = _setup(variant, D, hid)
    rng = np.random.default_rng(6)
    hist = data.history(1).astype(np.int64)
    tgt = rng.integers(0, 700, 4 * len(hist)).astype(np.int64)
    hist, hreg, treg = _dense_rows(data, hist, tgt)
    B, H = hist.shape
    m = util.make_model(variant, sd, 0.5)
    P32 = m._params()
    a = _pair_args(variant, hist, tgt, hreg, treg)
    seed = 987654321
    score, row_sum, parts, mask = ops.pairs_forward_raw(variant, 0.5, P32, *a, drop=(P_DROP, seed, "tc"))
    assert mask is not None
    dscore = torch.from_numpy(rng.normal(size=B).astype(np.float32)).cuda()
    G = ops.pairs_backward_raw(variant, 0.5, P32, *a, row_sum, parts, dscore, (P_DROP, seed, "auto"), act_mask=None)
    G_tc = ops.pairs_backward_raw(variant, 0.5, P32, *a, row_sum, parts, dscore, (P_DROP, seed, "tc"), act_mask=mask)
    keep = ops.dropout_keep_mask(seed, B, H, hid, P_DROP)
    ref, P = _oracle(sd, variant, hist, tgt, hreg, treg, keep / (1 - P_DROP))
    (ref * dscore.cpu().double()).sum().backward()
    for n, g in G.items():
        r = P[n].grad.numpy()
        for got in (g, G_tc[n]):
            assert np.abs(got.cpu().double().numpy() - r).max() <= 2e-4 * np.abs(r).max(), n
    with pytest.raises(RuntimeError, match="NULL"):
        ops.pairs_backward_raw(variant, 0.5, P32, *a, row_sum, parts, dscore, (P_DROP, seed, "tc"), act_mask=None)


@pytest.mark.parametrize("variant,D,pp", [("basic", 64, "tc"), ("region", 64, "tc"), ("region", 32, "tc"), ("region", 64, "fp32")])
def test_segmented_scores_and_gradients(variant, D, pp):
    hid = 64
    data, sd, bt = _setup(variant, D, hid, U=11, max_hist=150)  # histories up to 150: one-row tiles with two chunks
    csr = data.train_csr()
    uids = np.arange(csr.shape[0])
    b = bt.multi_user_batch(uids, 4, seed=9)
    rng = np.random.default_rng(2)
    dscore = rng.normal(size=b.B)
    m = util.make_model(variant, sd, 0.5).train()
    m.pairs_precision = pp
    torch.manual_seed(3)
    s = m.segmented_scores(b)
    (s * torch.from_numpy(dscore).cuda().float()).sum().backward()
    keep = ops.dropout_keep_mask_cells(m.last_dropout_seed, b.n_cells, hid, P_DROP)
    ro, co, tgt_all = b.host_row_offsets, b.seg_cell_offsets.cpu().numpy(), b.tgt.cpu().numpy()
    P = {k: v.double().requires_grad_(True) for k, v in sd.items()}
    for si, u in enumerate(uids):
        h = csr.getrow(u).indices.astype(np.int64)
        if len(h) == 0:
            continue
        tgt = tgt_all[ro[si]:ro[si + 1]]
        hist, hreg, treg = _dense_rows(data, h, tgt)
        k = keep[co[si]:co[si + 1]].reshape(len(tgt), len(h), hid)
        ref, _ = _oracle(sd, variant, hist, tgt, hreg, treg, k / (1 - P_DROP), P)
        (ref * torch.from_numpy(dscore[ro[si]:ro[si + 1]])).sum().backward()
        np.testing.assert_allclose(s.detach()[ro[si]:ro[si + 1]].cpu().double().numpy(), ref.detach().numpy(), rtol=1e-4, atol=1e-6)
    _check_grads(m, P)
    ops.check_indices(sync=True)


@pytest.mark.parametrize("pp", ["fp32", "tc"])
def test_one_segment_batch_draws_the_dense_mask(pp):
    variant, D, hid = "region", 64, 64
    data, sd, bt = _setup(variant, D, hid)
    csr = data.train_csr()
    m = util.make_model(variant, sd, 0.5)
    P = tuple(m._params().values())
    for u in (0, 4):
        b = bt.multi_user_batch(np.array([u]), 4, seed=u)
        h = csr.getrow(u).indices.astype(np.int64)
        tgt = b.tgt.cpu().numpy()
        hist, hreg, treg = _dense_rows(data, h, tgt)
        with torch.no_grad():
            s_seg = ops.pairs_score(variant, 0.5, P, b, None, None, None, None, P_DROP, 4242, pp)
            s_dense = ops.pairs_score(variant, 0.5, P, *_pair_args(variant, hist, tgt, hreg, treg), P_DROP, 4242, pp)
            s_off = ops.pairs_score(variant, 0.5, P, *_pair_args(variant, hist, tgt, hreg, treg), 0.0, 0, pp)
        assert torch.allclose(s_seg, s_dense, rtol=1e-6, atol=0), float((s_seg - s_dense).abs().max())
        assert not torch.allclose(s_dense, s_off, rtol=1e-3)


@pytest.mark.parametrize("variant", ["basic", "region"])
def test_segmented_dropout_step(variant):
    """fused_adagrad_step on a multi-user segmented batch in train mode: the one-call step == the op-by-op step (same torch seed
    -> same mask) == autograd through segmented_scores + torch.optim.Adagrad, from a common start."""
    D = hid = 64
    data, sd, bt = _setup(variant, D, hid, U=12)
    b = bt.multi_user_batch(np.arange(12), 4, seed=1)
    ms = [util.make_model(variant, sd, 0.5).train() for _ in range(3)]
    os_ = [torch.optim.Adagrad(m.parameters(), lr=0.05) for m in ms]
    ms[1].one_call = False
    losses = []
    for i in range(2):
        torch.manual_seed(77)
        losses.append(float(ms[i].fused_adagrad_step(os_[i], b.label, b)))
    torch.manual_seed(77)
    os_[2].zero_grad()
    l3 = ms[2].loss_func(torch.sigmoid(ms[2].segmented_scores(b)), b.label)
    l3.backward()
    os_[2].step()
    assert ms[0].last_dropout_seed == ms[1].last_dropout_seed == ms[2].last_dropout_seed
    assert abs(losses[0] - losses[1]) <= 2e-6 * abs(losses[1]) and abs(losses[0] - float(l3)) <= 1e-5 * abs(float(l3))
    # one Adagrad step from a zero accumulator moves an element by lr * g / (|g| + eps): summation-order differences in a tiny g
    # show up at ~1e-5 of the tensor (the bounds of tests/test_gpu_train_step.py)
    for (n, pa), (_, pb), (_, pc) in zip(ms[0].named_parameters(), ms[1].named_parameters(), ms[2].named_parameters()):
        for other, tol in ((pb, 5e-5), (pc, 1e-4)):
            assert float((pa - other).abs().max()) <= tol * max(float(other.abs().max()), 1e-3), n


@pytest.mark.parametrize("variant,pp", [("basic", "auto"), ("region", "auto"), ("region", "fp32")])
def test_train_users_with_dropout_is_the_per_user_loop_bit_for_bit(variant, pp):
    N = 1500
    data = synthetic.make_checkins(30, N, seed=11, hist_len=None, max_hist=140, min_hist=0, median_hist=15)
    sd = orc.init_state(variant, N, 64, 64, data.region_num, 1, seed=1, style="trained")
    ms = [util.make_model(variant, sd, 0.5).train() for _ in range(3)]
    os_ = [torch.optim.Adagrad(m.parameters(), lr=0.05) for m in ms]
    for m in ms:
        m.pairs_precision = pp
        assert m.drop.p == P_DROP
    bt = PB.DeviceBatcher(data.train_csr(), data.region, data.coords, device="cuda", seed=0)
    uids = np.array([3, 7, 0, 12, 29, 5, 5, 18, 21, 9])
    torch.manual_seed(5)
    losses = ms[0].train_users(os_[0], bt, uids, 4, seed=77)
    last = ms[0].last_dropout_seed
    torch.manual_seed(5)
    ref = []
    for u in uids:
        if bt.indptr[u + 1] == bt.indptr[u]:
            ref.append(0.0)
            continue
        b = bt.multi_user_batch(np.array([u]), 4, seed=77 + int(u))
        ref.append(float(ms[1].fused_adagrad_step(os_[1], b.label, b)))
    assert ms[1].last_dropout_seed == last
    torch.manual_seed(6)
    ms[2].train_users(os_[2], bt, uids, 4, seed=77)
    ops.check_indices(sync=True)
    assert np.array_equal(losses.cpu().numpy(), np.array(ref, dtype=np.float32)), (losses.cpu().numpy(), ref)
    for (n, pa), (_, pb), (_, pc) in zip(ms[0].named_parameters(), ms[1].named_parameters(), ms[2].named_parameters()):
        assert torch.equal(pa, pb), n
        assert torch.equal(os_[0].state[pa]["sum"], os_[1].state[pb]["sum"]), n
    assert not torch.equal(ms[0].attn_layer1.weight, ms[2].attn_layer1.weight)  # another torch seed, another mask
