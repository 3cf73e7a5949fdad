"""Training of the two-branch NAIS_region_distance_disentangled_Embedding (model.py:410-541) on the fused paths: segmented batches
with the haversine km formed in the kernel, the one-call Adagrad step and `train_users` — against the float64 oracle, the op-by-op
step and autograd + torch.optim.Adagrad."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

import nais_testutil as util
from oracle import nais_oracle as orc
from poi_recommendation_models_b200 import batches as PB, ops, synthetic

pytestmark = pytest.mark.gpu
V = "disentangled"


def _data(U, N, seed, max_hist, min_hist=2):
    return synthetic.make_checkins(U, N, seed=seed, hist_len=None, max_hist=max_hist, min_hist=min_hist, median_hist=14)


def _user_rows(data, csr, b, s, u):
    """The rows of segment s of a segmented batch in the reference's dense form: (hist [R,H], tgt [R], hreg, treg, km float64)."""
    ro = b.host_row_offsets
    hist = csr.getrow(u).indices.astype(np.int64)
    tgt = b.tgt.cpu().numpy()[ro[s]:ro[s + 1]]
    hh = np.broadcast_to(hist, (len(tgt), len(hist))).copy()
    km = orc.dist_km(data.coords[tgt][:, None, 0], data.coords[tgt][:, None, 1], data.coords[hh][..., 0], data.coords[hh][..., 1])
    return hh, tgt, data.region[hh], data.region[tgt], km


def test_segmented_km_forward_and_backward_match_the_oracle():
    N, num_ng = 800, 4
    data = _data(9, N, seed=3, max_hist=60)
    # user 1 gets no history (a segment without tiles), user 4 gets 140 items (one-row tiles with two chunks)
    rows = [data.history(u) for u in range(9)]
    rows[1], rows[4] = rows[1][:0], np.random.default_rng(5).choice(N, 140, replace=False)
    csr = sp.csr_matrix((np.ones(sum(map(len, rows))), (np.repeat(np.arange(9), [len(r) for r in rows]), np.concatenate(rows))),
                        shape=(9, N))
    bt = PB.DeviceBatcher(csr, data.region, data.coords, device="cuda", seed=0)
    lens = np.diff(csr.indptr)
    assert lens.max() > 128 and (lens == 0).any()
    sd = orc.init_state(V, N, 64, 64, data.region_num, 1, seed=4, style="trained")
    m = util.make_model(V, sd, 0.5)
    uids = np.arange(len(lens))
    b = bt.multi_user_batch(uids, num_ng, seed=9)
    dscore = torch.from_numpy(np.random.default_rng(2).normal(size=b.B).astype(np.float32)).cuda()
    s = m.segmented_scores(b)
    (s * dscore).sum().backward()
    ops.check_indices(sync=True)
    ro = b.host_row_offsets
    worst, G = 0.0, None
    for si, u in enumerate(uids):
        if ro[si + 1] == ro[si]:
            continue
        hh, tgt, hr, tr, km = (torch.from_numpy(x) for x in _user_rows(data, csr, b, si, u))
        ref, scale = orc.attention_network_with_scale(sd, V, 0.5, hh, tgt, hr, tr, km, dtype=torch.float64)
        worst = max(worst, util.cond_err(s.detach()[ro[si]:ro[si + 1]].cpu().numpy(), ref.numpy(), scale.numpy()))
        _, g = orc.grads(sd, V, 0.5, hh, tgt, hr, tr, km, dscore[ro[si]:ro[si + 1]].cpu())
        G = g if G is None else {k: G[k] + g[k] for k in G}
    assert worst < util.TOL, worst
    for n, p in m.named_parameters():
        ref = G[n]
        err = float((p.grad.double().cpu() - ref).abs().max()) / max(float(ref.abs().max()), 1e-30)
        assert err <= 2e-4, (n, err)
    assert float(m.embed_distance.weight.grad[0].abs().max()) > 0


def _models(N, R, n=3, seed=1):
    sd = orc.init_state(V, N, 64, 64, R, 1, seed=seed, style="trained")
    ms = [util.make_model(V, sd, 0.5).train() for _ in range(n)]
    return ms, [torch.optim.Adagrad(m.parameters(), lr=0.05) for m in ms]


def _sync_from(dst_m, dst_o, src_m, src_o):  # teacher forcing: every path takes each step from the same point
    with torch.no_grad():
        for (_, pd), (_, ps_) in zip(dst_m.named_parameters(), src_m.named_parameters()):
            pd.copy_(ps_)
            dst_o.state[pd]["sum"].copy_(src_o.state[ps_]["sum"])


def _close(a, oa, b, ob, tol, what):
    for (n, pa), (_, pb) in zip(a.named_parameters(), b.named_parameters()):
        scale = max(float(pb.abs().max()), 1e-6)
        assert float((pa - pb).abs().max()) / scale <= tol, (what, n)
        sa, sb = oa.state[pa]["sum"], ob.state[pb]["sum"]
        assert float((sa - sb).abs().max()) <= tol * max(float(sb.abs().max()), 1e-12), (what, n, "sum")


@pytest.mark.parametrize("layout", ["dense", "segmented"])
def test_one_call_step_equals_the_op_by_op_and_the_dense_step(layout):
    N = 900
    data = _data(12, N, seed=3, max_hist=40, min_hist=3)
    (m_one, m_ops, m_dense), (o_one, o_ops, o_dense) = _models(N, data.region_num)
    m_ops.one_call = False
    bt = PB.DeviceBatcher(data.train_csr(), data.region, data.coords, device="cuda", seed=0)
    steps = 5
    for it in range(steps):
        _sync_from(m_one, o_one, m_ops, o_ops)
        _sync_from(m_dense, o_dense, m_ops, o_ops)
        before = {n: t.detach().clone() for n, t in m_one.named_parameters()}
        if layout == "dense":
            h, t, lab, hr, tr, _ = bt.batch(it, 4)
            km = PB.dist_km_pairs(data.coords, t.cpu().numpy(), h.cpu().numpy(), device="cuda")
            args = (h, t, hr, tr, km)
            l1 = m_one.fused_adagrad_step(o_one, lab, *args)
            l2 = m_ops.fused_adagrad_step(o_ops, lab, *args)
            o_dense.zero_grad()
            l3 = m_dense.loss_func(m_dense(*args), lab)
            touched = {"embed_history.weight": h.unique(), "embed_target.weight": t.unique(),
                       "embed_region.weight": torch.cat([hr.reshape(-1), tr]).unique()}
        else:
            b = bt.multi_user_batch(np.arange(3 * it, 3 * it + 3) % 12, 4, seed=it)
            lab = b.label
            l1 = m_one.fused_adagrad_step(o_one, lab, b)
            l2 = m_ops.fused_adagrad_step(o_ops, lab, b)
            o_dense.zero_grad()
            l3 = m_dense.loss_func(torch.sigmoid(m_dense.segmented_scores(b)), lab)
            touched = ops.touched_rows(b, None)
        l3.backward()
        o_dense.step()
        assert abs(float(l1) - float(l2)) <= 2e-6 * abs(float(l2)) + 1e-7, (it, float(l1), float(l2))
        assert abs(float(l1) - float(l3.detach())) <= 2e-5 * abs(float(l3.detach())) + 1e-6, (it, float(l1), float(l3))
        _close(m_one, o_one, m_ops, o_ops, 5e-5, f"{layout} step {it} vs op-by-op")
        _close(m_one, o_one, m_dense, o_dense, 1e-4, f"{layout} step {it} vs dense")
        # untouched table rows (and embed_distance rows the forward never reads) stay bit-identical
        after = dict(m_one.named_parameters())
        for n, ids in touched.items():
            keep = torch.ones(after[n].shape[0], dtype=torch.bool, device="cuda")
            keep[ids] = False
            assert torch.equal(after[n][keep], before[n][keep]), n
        assert torch.equal(after["embed_distance.weight"][1:], before["embed_distance.weight"][1:])
        assert not torch.equal(after["embed_distance.weight"][0], before["embed_distance.weight"][0])
    ops.check_indices(sync=True)
    for n, pa in m_one.named_parameters():
        assert float(o_one.state[pa]["step"]) == steps, n


def test_train_users_is_the_per_user_loop_bit_for_bit():
    N = 1500
    data = _data(30, N, seed=11, max_hist=140, min_hist=0)
    (m_all, m_loop), (o_all, o_loop) = _models(N, data.region_num, n=2)
    bt = PB.DeviceBatcher(data.train_csr(), data.region, data.coords, device="cuda", seed=0)
    uids = np.array([3, 7, 0, 12, 29, 5, 5, 18, 21, 9])
    losses = m_all.train_users(o_all, bt, uids, 4, seed=77)
    ref = []
    for u in uids:
        if bt.indptr[u + 1] == bt.indptr[u]:
            ref.append(0.0)
            continue
        b = bt.multi_user_batch(np.array([u]), 4, seed=77 + int(u))
        ref.append(float(m_loop.fused_adagrad_step(o_loop, b.label, b)))
    ops.check_indices(sync=True)
    assert np.array_equal(losses.cpu().numpy(), np.array(ref, dtype=np.float32)), (losses.cpu().numpy(), ref)
    for (n, pa), (_, pb) in zip(m_all.named_parameters(), m_loop.named_parameters()):
        assert torch.equal(pa, pb), n
        assert torch.equal(o_all.state[pa]["sum"], o_loop.state[pb]["sum"]), n
        assert float(o_all.state[pa]["step"]) == float(o_loop.state[pb]["step"]), n


def test_out_of_range_region_id_raises_and_moves_no_region_row():
    N = 600
    data = _data(6, N, seed=2, max_hist=30, min_hist=3)
    (m,), (o,) = _models(N, data.region_num, n=1)
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
