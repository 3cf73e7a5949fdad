"""BPR training: nais_pairs_train_step_bpr (one library call = zero_grad -> forward -> -logsigmoid(s+ - s-) -> backward ->
Adagrad.step) against the op-by-op path of `fused_bpr_step` (torch's own logsigmoid / autograd on the [n_groups, 1 + num_neg] view
of the scores, torch.optim.Adagrad on the MLP parameters) and against a plain dense step (autograd through the model +
`optimizer.step()`); the loss kernel against float64; and nais_train_users_bpr against the per-user Python loop, bit for bit."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

import nais_testutil as util
from oracle import nais_oracle as orc
from poi_recommendation_models_b200 import batches as PB, ops, synthetic
from test_bpr_train_cpu import bpr_reference

pytestmark = pytest.mark.gpu
VARIANTS = ["region_distance", "distance", "region", "basic", "disentangled"]


def _models(variant, N, R, n=3, seed=1, dropout=0.0):
    sd = orc.init_state(variant, N, 64, 64, R, 1, seed=seed, style="trained")
    ms = [util.make_model(variant, sd, 0.5).train() for _ in range(n)]
    for m in ms:
        if hasattr(m, "drop"):
            m.drop.p = dropout
    return ms, [torch.optim.Adagrad(m.parameters(), lr=0.05) for m in ms]


def _sync_from(dst_m, dst_o, src_m, src_o):  # teacher forcing: every path takes each step from the same point
    with torch.no_grad():
        for (_, pd), (_, ps_) in zip(dst_m.named_parameters(), src_m.named_parameters()):
            pd.copy_(ps_)
            dst_o.state[pd]["sum"].copy_(src_o.state[ps_]["sum"])


def _close(a, oa, b, ob, tol, what, mean_tol=None):
    """max |a - b| / max |b| <= tol for every parameter and its Adagrad sum (mean_tol: also the mean, see test_gpu_train_step)."""
    for (n, pa), (_, pb) in zip(a.named_parameters(), b.named_parameters()):
        err = (pa - pb).detach().abs()
        scale = max(float(pb.detach().abs().max()), 1e-6)
        assert torch.isfinite(pa).all(), (what, n)
        assert float(err.max()) / scale <= tol, (what, n, float(err.max()) / scale)
        if mean_tol is not None:
            assert float(err.mean()) / scale <= mean_tol, (what, n, float(err.mean()) / scale)
        sa, sb = oa.state[pa]["sum"], ob.state[pb]["sum"]
        assert float((sa - sb).abs().max()) <= tol * max(float(sb.abs().max()), 1e-12), (what, n, "sum")


def _dense_args(variant, data, h, t, hr, tr, ll):
    """(model-call args, fused-step kwargs) of a dense batch of DeviceBatcher.batch."""
    if variant == "disentangled":
        ll = PB.dist_km_pairs(data.coords, t.cpu().numpy(), h.cpu().numpy(), device="cuda")
    full = {"region_distance": (h, t, hr, tr, ll), "distance": (h, t, None, None, ll), "region": (h, t, hr, tr, None),
            "basic": (h, t, None, None, None), "disentangled": (h, t, hr, tr, ll)}[variant]
    args = {"region_distance": (h, t, hr, tr, ll), "distance": (h, t, hr, tr, ll), "region": (h, t, hr, tr), "basic": (h, t),
            "disentangled": (h, t, hr, tr, ll)}[variant]
    return args, dict(zip(("hist", "tgt", "hreg", "treg", "aux"), full))


def _bpr(s, num_neg, gw=None):
    v = s.view(-1, num_neg + 1)
    nll = -torch.nn.functional.logsigmoid(v[:, :1] - v[:, 1:])
    return nll.mean() if gw is None else (nll * gw[:, None]).sum()


@pytest.mark.parametrize("layout", ["dense", "segmented"])
@pytest.mark.parametrize("num_neg", [1, 4])
@pytest.mark.parametrize("variant", VARIANTS)
def test_one_call_bpr_step_equals_the_op_by_op_and_the_dense_step(variant, num_neg, layout):
    N = 900
    data = synthetic.make_checkins(12, N, seed=3, hist_len=None, max_hist=40, min_hist=3, median_hist=12)
    (m_one, m_ops, m_dense), (o_one, o_ops, o_dense) = _models(variant, N, data.region_num)
    m_ops.one_call = False
    bt = PB.DeviceBatcher(data.train_csr(), data.region, data.coords, device="cuda", seed=0)
    for it in range(4):
        _sync_from(m_one, o_one, m_ops, o_ops)
        _sync_from(m_dense, o_dense, m_ops, o_ops)
        o_dense.zero_grad()
        if layout == "dense":
            h, t, _, hr, tr, ll = bt.batch(it, num_neg)
            args, kw = _dense_args(variant, data, h, t, hr, tr, ll)
            l1 = m_one.fused_bpr_step(o_one, num_neg=num_neg, **kw)
            l2 = m_ops.fused_bpr_step(o_ops, num_neg=num_neg, **kw)
            l3 = _bpr(m_dense.attention_network(*(args if variant != "distance" else (h, t, ll))), num_neg)
        else:
            b = bt.multi_user_batch(np.arange(3 * it, 3 * it + 3) % 12, num_neg, seed=it)
            l1 = m_one.fused_bpr_step(o_one, b, num_neg=num_neg)
            l2 = m_ops.fused_bpr_step(o_ops, b, num_neg=num_neg)
            l3 = _bpr(m_dense.segmented_scores(b), num_neg)
        l3.backward()
        o_dense.step()
        assert abs(float(l1) - float(l2)) <= 2e-6 * abs(float(l2)), (it, float(l1), float(l2))
        assert abs(float(l1) - float(l3.detach())) <= 2e-5 * abs(float(l3.detach())), (it, float(l1), float(l3.detach()))
        _close(m_one, o_one, m_ops, o_ops, 5e-5, f"step {it} vs op-by-op")
        _close(m_one, o_one, m_dense, o_dense, 1e-4, f"step {it} vs dense")
    ops.check_indices(sync=True)
    for n, pa in m_one.named_parameters():
        if n in m_one._params():
            assert float(o_one.state[pa]["step"]) == 4.0, n


def test_multi_user_step_with_group_weights_is_the_sum_of_the_per_user_losses():
    """group_weight = 1 / pairs(user) makes one segmented step over many users carry the sum of their mean BPR losses; each user's
    loss is taken by a one-call step on that user's rows alone (dense layout), from the same parameters."""
    N, num_neg, V = 2000, 4, "region_distance"
    data = synthetic.make_checkins(40, N, seed=5, hist_len=None, max_hist=60, min_hist=3, median_hist=20)
    csr = data.train_csr()
    (m_one, m_ops, m_user), (o_one, o_ops, o_user) = _models(V, N, data.region_num)
    m_ops.one_call = False
    bt = PB.DeviceBatcher(csr, data.region, data.coords, device="cuda", seed=0)
    reg = torch.from_numpy(data.region).cuda()
    for it in range(3):
        uids = np.arange(10 * it, 10 * it + 10)
        b = bt.multi_user_batch(uids, num_neg, seed=it)
        ro = b.host_row_offsets
        groups = np.diff(ro) // (num_neg + 1)
        gw = torch.from_numpy(np.repeat(1.0 / np.maximum(groups * num_neg, 1), groups).astype(np.float32)).cuda()
        per_user = 0.0
        for s, u in enumerate(uids):
            _sync_from(m_user, o_user, m_one, o_one)
            hist = torch.from_numpy(csr.getrow(int(u)).indices.astype(np.int64)).cuda()
            tgt = b.tgt[ro[s]:ro[s + 1]]
            h = hist[None, :].expand(len(tgt), -1).contiguous()
            ll = PB.lat_lon_pairs(data.coords, tgt.cpu().numpy(), h.cpu().numpy(), device="cuda")
            per_user += float(m_user.fused_bpr_step(o_user, h, tgt, reg[h], reg[tgt], ll, num_neg=num_neg))
        _sync_from(m_ops, o_ops, m_one, o_one)
        l1 = m_one.fused_bpr_step(o_one, b, num_neg=num_neg, group_weight=gw)
        l2 = m_ops.fused_bpr_step(o_ops, b, num_neg=num_neg, group_weight=gw)
        assert abs(float(l1) - per_user) <= 1e-5 * abs(per_user), (it, float(l1), per_user)
        assert abs(float(l1) - float(l2)) <= 2e-6 * abs(float(l2)), (it, float(l1), float(l2))
        _close(m_one, o_one, m_ops, o_ops, 1e-5, f"multi-user step {it}")
    ops.check_indices(sync=True)


@pytest.mark.parametrize("scale", [1.0, 60.0])
def test_loss_kernel_against_float64(scale):
    """The loss of the one-call step on the scores it returns equals the float64 restatement of the contract; with embed_history
    x60 the scores are in the hundreds (sigmoid saturated in fp32): loss and parameters stay finite and agree with op-by-op.
    Parameters are held to the bound of several Adagrad steps from a zero accumulator (test_gpu_train_step._close): an element
    whose first gradient is ~eps moves by a rounding-dependent fraction of lr."""
    N, num_neg, V = 900, 4, "basic"
    data = synthetic.make_checkins(12, N, seed=8, hist_len=None, max_hist=40, min_hist=3, median_hist=12)
    (m_one, m_ops, _), (o_one, o_ops, _) = _models(V, N, data.region_num)
    m_ops.one_call = False
    with torch.no_grad():
        for m in (m_one, m_ops):
            m.embed_history.weight.mul_(scale)
    bt = PB.DeviceBatcher(data.train_csr(), data.region, data.coords, device="cuda", seed=0)
    saw_saturated = False
    for it in range(3):
        _sync_from(m_ops, o_ops, m_one, o_one)
        b = bt.multi_user_batch(np.arange(4 * it, 4 * it + 4), num_neg, seed=it)
        groups = b.B // (num_neg + 1)
        gw = None if it != 1 else torch.rand(groups, device="cuda") + 0.1
        P = m_one._params()
        dsum = {n: o_one.state[t]["sum"] for n, t in P.items() if n not in ops._TABLES}
        tsum = {n: o_one.state[t]["sum"] for n, t in P.items() if n in ops._TABLES}
        loss, score = ops.pairs_train_step_bpr(V, 0.5, P, tsum, dsum, 0.05, 1e-10, 0.05, 1e-10, num_neg, b, group_weight=gw,
                                               want_score=True)
        for t in P.values():
            o_one.state[t]["step"] += 1
        l2 = m_ops.fused_bpr_step(o_ops, b, num_neg=num_neg, group_weight=gw)
        s64 = score.double().cpu().numpy()
        d = s64.reshape(-1, num_neg + 1)
        saw_saturated |= bool(np.abs(d[:, :1] - d[:, 1:]).max() > 50)
        ref, _ = bpr_reference(s64, num_neg, None if gw is None else gw.double().cpu().numpy())
        assert np.isfinite(float(loss)) and abs(float(loss) - ref) <= 1e-6 * abs(ref), (it, float(loss), ref)
        assert abs(float(loss) - float(l2)) <= 2e-6 * abs(float(l2)), (it, float(loss), float(l2))
        _close(m_one, o_one, m_ops, o_ops, 2e-2, f"step {it}", mean_tol=5e-5)
    assert saw_saturated or scale == 1.0
    ops.check_indices(sync=True)


@pytest.mark.parametrize("layout", ["dense", "segmented"])
@pytest.mark.parametrize("variant", ["basic", "region"])
def test_dropout_classes_draw_the_same_mask_seed_in_both_paths(variant, layout):
    N, num_neg = 900, 4
    data = synthetic.make_checkins(12, N, seed=9, hist_len=None, max_hist=40, min_hist=3, median_hist=12)
    (m_one, m_ops, _), (o_one, o_ops, _) = _models(variant, N, data.region_num, dropout=0.5)
    m_ops.one_call = False
    bt = PB.DeviceBatcher(data.train_csr(), data.region, data.coords, device="cuda", seed=0)
    for it in range(3):
        _sync_from(m_ops, o_ops, m_one, o_one)
        if layout == "dense":
            h, t, _, hr, tr, ll = bt.batch(it, num_neg)
            kw = _dense_args(variant, data, h, t, hr, tr, ll)[1]
            batch = ()
        else:
            kw, batch = {}, (bt.multi_user_batch(np.arange(3 * it, 3 * it + 3), num_neg, seed=it),)
        torch.manual_seed(100 + it)
        l1 = m_one.fused_bpr_step(o_one, *batch, num_neg=num_neg, **kw)
        torch.manual_seed(100 + it)
        l2 = m_ops.fused_bpr_step(o_ops, *batch, num_neg=num_neg, **kw)
        assert m_one.last_dropout_seed == m_ops.last_dropout_seed
        assert abs(float(l1) - float(l2)) <= 2e-6 * abs(float(l2)), (it, float(l1), float(l2))
        _close(m_one, o_one, m_ops, o_ops, 5e-5, f"dropout step {it}")
    ops.check_indices(sync=True)


@pytest.mark.parametrize("variant", VARIANTS)
def test_train_users_bpr_is_the_per_user_loop_bit_for_bit(variant):
    """nais_train_users_bpr leaves exactly the parameters, optimizer sums, step counters and losses of the Python loop
    `for u: fused_bpr_step(opt, multi_user_batch([u], 4, seed + u), num_neg=4)` — dropout classes in train mode included (the same
    torch seed gives the same mask seeds)."""
    N, num_neg, U = 1500, 4, 30
    data = synthetic.make_checkins(U, N, seed=11, hist_len=None, max_hist=60, min_hist=2, median_hist=15)
    rows = [data.history(u) for u in range(U)]
    rows[2], rows[5] = rows[2][:0], np.random.default_rng(5).choice(N, 140, replace=False)  # no history; history > 128
    csr = sp.csr_matrix((np.ones(sum(map(len, rows))), (np.repeat(np.arange(U), [len(r) for r in rows]), np.concatenate(rows))),
                        shape=(U, N))
    (m_all, m_loop, _), (o_all, o_loop, _) = _models(variant, N, data.region_num, dropout=0.5)
    bt = PB.DeviceBatcher(csr, data.region, data.coords, device="cuda", seed=0)
    uids = np.array([3, 7, 2, 0, 12, 5, 29, 5, 18, 21, 9])  # user 5 twice
    torch.manual_seed(5)
    losses = m_all.train_users(o_all, bt, uids, num_neg, seed=77, loss="bpr")
    torch.manual_seed(5)
    ref = []
    for u in uids:
        if bt.indptr[u + 1] == bt.indptr[u]:
            ref.append(0.0)
            continue
        b = bt.multi_user_batch(np.array([u]), num_neg, seed=77 + int(u))
        ref.append(float(m_loop.fused_bpr_step(o_loop, b, num_neg=num_neg)))
    ops.check_indices(sync=True)
    assert losses.shape == (len(uids),) and float(losses[2]) == 0.0
    assert np.array_equal(losses.cpu().numpy(), np.array(ref, dtype=np.float32)), (losses.cpu().numpy(), ref)
    for (n, pa), (_, pb) in zip(m_all.named_parameters(), m_loop.named_parameters()):
        assert torch.equal(pa, pb), n
        assert torch.equal(o_all.state[pa]["sum"], o_loop.state[pb]["sum"]), n
        assert float(o_all.state[pa]["step"]) == float(o_loop.state[pb]["step"]), n
        if n in m_all._params():
            assert float(o_all.state[pa]["step"]) == 10.0, n


def test_a_bpr_trained_model_ranks():
    """A few epochs of train_users(loss="bpr") lower the loss, and predict_topk on the trained weights passes the full-rank parity
    check against the float64 oracle (a smoke test that the weights are usable, not a quality claim)."""
    U, N, k, V = 40, 1200, 10, "region_distance"
    data = synthetic.make_checkins(U, N, seed=13, hist_len=None, max_hist=40, min_hist=5, median_hist=15)
    (m,), (o,) = _models(V, N, data.region_num, n=1)
    bt = PB.DeviceBatcher(data.train_csr(), data.region, data.coords, device="cuda", seed=0)
    epochs = [float(m.train_users(o, bt, np.arange(U), 4, seed=100 * e, loss="bpr").mean()) for e in range(6)]
    assert all(np.isfinite(epochs)) and epochs[-1] < epochs[0], epochs
    m.eval()
    m.set_catalog(region=data.region, coords=data.coords)
    sd = {n: t.detach().cpu() for n, t in m.state_dict().items()}
    score, ids = m.predict_topk((data.indptr, data.indices), k, precision="fp32")
    ids = ids.cpu().numpy()
    cat = orc.Catalog(data.coords, data.region)
    for u in range(0, U, 4):
        hist = data.history(u)
        _, _, cand, pred = orc.fullrank_user(sd, V, 0.5, cat, hist, k, dtype=torch.float64, return_all=True)
        assert not set(ids[u].tolist()) & set(hist.tolist())
        util.lists_equal_outside_ties(ids[u], None, dict(zip(cand.tolist(), pred.tolist())), k)
