"""The sorted-segment reduce of csrc/nais_bwd.cu (every embedding-table gradient and every fused row-sparse Adagrad step goes
through it) held BIT FOR BIT to nais_testutil.segment_reduce_ref / rows_adagrad_ref, its float32 restatement in the documented
summation order, over every path the reduce has:

  pass 1   the lean kernel (dense gradients, and fused Adagrad on lists of more than 65 536 entries) and the kOpt kernel (fused
           Adagrad on lists of at most 65 536 entries: deferred, batched updates; 16 rows in flight for w <= 32);
  widths   NQ = 1, 2, 4 floats per lane (w <= 32, <= 64, <= 128), with column masks where w is not a multiple of 32;
  runs     inside a chunk of 64 entries, or crossing chunks (partial slots [2c] / [2c+1]; pass 2 finds the continuing chunks
           32 at a time);
  ids      outside [0, n_rows), negative ones included, are dropped.

nais_rows_adagrad is called directly (both output modes: sum == NULL writes the summed rows to grad_out) with its outputs inside
guarded buffers, and through the pair backward: the fused step (nais_pairs_backward_adagrad) must equal rows_adagrad_ref applied
to the dense table gradients of nais_pairs_backward, since both reduce the same rows in the same sorted order.

The step computes p - (lr * g) / (sqrt(s) + eps); torch.optim.Adagrad computes p + (-lr) * (g / (sqrt(s) + eps)).  The two can
differ by one ulp, which is why the fused step is compared with rows_adagrad_ref here and with torch at a tolerance elsewhere."""
import numpy as np
import pytest
import torch

import nais_testutil as util
from oracle import nais_oracle as orc
from poi_recommendation_models_b200 import _lib, batches as PB, ops, synthetic

pytestmark = pytest.mark.gpu
KOPT_MAX = 65536           # fused-Adagrad lists up to this length run the kOpt pass-1 kernel (launch_segment_reduce)
SENTINEL = 0x7FC0DEAD      # a NaN pattern no kernel produces: untouched rows and guards must keep it bit for bit
LR, EPS = 0.05, 1e-10


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _path(adagrad, n):
    return "kopt" if adagrad and n <= KOPT_MAX else "lean"


class Guarded:
    """A [n_rows, w] float32 table inside a device buffer with `guard` floats on each side, all sentinel unless `init` given."""

    def __init__(self, n_rows, w, init=None, guard=None):
        self.n_rows, self.w = n_rows, w
        self.guard = guard if guard is not None else 4 * w + 64
        host = np.full(self.guard * 2 + n_rows * w, SENTINEL, np.uint32).view(np.float32)
        if init is not None:
            host[self.guard:self.guard + n_rows * w] = np.asarray(init, np.float32).reshape(-1)
        self.host0 = host.copy()
        self.dev = torch.from_numpy(host).cuda()

    @property
    def ptr(self):
        return self.dev.data_ptr() + 4 * self.guard

    def get(self):
        return self.dev.cpu().numpy()

    def table(self, flat):
        return flat[self.guard:self.guard + self.n_rows * self.w].reshape(self.n_rows, self.w)

    def expect(self, ids, rows):
        """The buffer the call must leave: the start state with rows `ids` replaced."""
        e = self.host0.copy()
        self.table(e)[ids] = rows
        return e


def _launch(keys, rows, n_rows, grad_out=None, param=None, state=None, lr=LR, eps=EPS):
    lib = _lib.load()
    n, w = rows.shape
    k = torch.from_numpy(np.ascontiguousarray(keys, np.int32)).cuda()
    r = torch.from_numpy(np.ascontiguousarray(rows, np.float32)).cuda()
    ws_bytes = lib.nais_rows_adagrad_workspace_bytes(n, w)
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device="cuda")
    rc = lib.nais_rows_adagrad(k.data_ptr(), r.data_ptr(), n, w, n_rows, grad_out.ptr if grad_out else None,
                               param.ptr if param else None, state.ptr if state else None, lr, eps, ws.data_ptr(), ws_bytes,
                               torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "nais_rows_adagrad")
    torch.cuda.synchronize()


# ---- key layouts --------------------------------------------------------------------------------------------------------------

def _keys(layout, n, rng):
    """(ascending keys [n], n_rows) of a named layout."""
    if layout == "unique":
        n_rows = n + 17
        return np.sort(rng.choice(n_rows, n, replace=False)), n_rows
    if layout == "equal":                       # one run over every chunk of the list
        return np.full(n, 3), 5
    if layout == "runs40":                      # chunks whose first run comes from the chunk before and whose last run goes on
        return np.arange(n) // 40, n // 40 + 1
    if layout == "offsets":                     # runs of 63, 64 and 65 entries starting at every offset of a chunk
        out, key = [], 0
        for L in (63, 64, 65):
            for o in range(64):
                fill = (o - len(out)) % 64      # single-entry runs up to the wanted offset
                out.extend(range(key, key + fill))
                key += fill
                out.extend([key] * L)
                key += 1
        out = np.array(out)
        reps = -(-n // len(out))
        k = np.concatenate([out + i * (key + 1) for i in range(reps)])[:n]
        return k, int(k.max()) + 1
    if layout == "zipf":                        # a few hot keys and a long tail
        n_rows = max(n // 8, 4)
        return np.sort((rng.zipf(1.3, n) - 1) % n_rows), n_rows
    if layout == "out_of_range":                # negative head over a chunk edge, a tail == n_rows and > n_rows over chunks
        n_rows = max(n // 4, 2)
        body = np.sort(rng.integers(0, n_rows, n))
        h, t = min(n // 3, 70), min(n // 3, 150)
        body[:h] = np.where(np.arange(h) < (2 * h) // 3, -3, -1)
        if t:
            body[n - t:] = np.where(np.arange(t) < t // 2, n_rows, n_rows + 9)
        return np.sort(body), n_rows
    raise ValueError(layout)


def _rows(rng, n, w):
    # magnitudes over several binades so that rounding happens in every sum; a few signed zeros
    r = (rng.normal(size=(n, w)) * np.exp2(rng.integers(-6, 7, (n, 1)))).astype(np.float32)
    r[rng.random((n, w)) < 0.01] = -0.0
    return r


def _gamma_bound(keys, rows, ids, got):
    """|got - exact| <= gamma_k * sum|r| per run, k = run length + pieces (float64 np.add.at as the exact sum)."""
    u = 2.0 ** -24
    ok = np.isin(keys, ids)
    k_ok, r_ok = keys[ok], rows[ok].astype(np.float64)
    pos = np.searchsorted(ids, k_ok)
    exact = np.zeros((len(ids), rows.shape[1]))
    absum = np.zeros_like(exact)
    np.add.at(exact, pos, r_ok)
    np.add.at(absum, pos, np.abs(r_ok))
    length = np.bincount(pos, minlength=len(ids))
    idx = np.flatnonzero(ok)
    new_piece = np.ones(len(idx), bool)
    new_piece[1:] = (k_ok[1:] != k_ok[:-1]) | (idx[1:] % util.SEG_CHUNK == 0)
    pieces = np.bincount(pos[new_piece], minlength=len(ids))
    k = (length + pieces).astype(np.float64)[:, None]
    bound = k * u / (1 - k * u) * absum + 1e-300
    assert np.all(np.abs(got.astype(np.float64) - exact) <= bound)


WIDTHS = [1, 16, 31, 32, 33, 48, 64, 65, 96, 127, 128]
SIZES = [1, 63, 64, 65, 127, 128, 129, 64 * 32, 64 * 33, 64 * 33 + 1, 64 * 64, 64 * 65]  # one run over 1 .. 65 chunks
LAYOUTS = ["unique", "equal", "runs40", "offsets", "zipf", "out_of_range"]


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("w", WIDTHS)
def test_gradient_mode_is_the_documented_order_bit_for_bit(w, layout):
    """sum == NULL (the lean pass-1 kernel): grad_out rows of the listed ids == segment_reduce_ref, every other float of the
    guarded buffer untouched; the float64 error bound holds."""
    rng = np.random.default_rng(w * 100 + LAYOUTS.index(layout))
    for n in SIZES + ([20000] if layout == "offsets" else []):  # (the whole offsets pattern takes ~18 500 entries)
        keys, n_rows = _keys(layout, n, rng)
        rows = _rows(rng, n, w)
        ids, g = util.segment_reduce_ref(keys, rows, n_rows)
        out = Guarded(n_rows, w)
        _launch(keys, rows, n_rows, grad_out=out)
        got = out.get()
        want = out.expect(ids, g)
        bad = np.flatnonzero(_bits(got) != _bits(want))
        assert bad.size == 0, (layout, n, w, bad[:8], got[bad[:4]], want[bad[:4]])
        _gamma_bound(keys, rows, ids, out.table(got)[ids])


@pytest.mark.parametrize("zero_sum", [True, False], ids=["sum0", "sum"])
@pytest.mark.parametrize("n", [KOPT_MAX, KOPT_MAX + 1], ids=["kopt", "lean"])
@pytest.mark.parametrize("w", [16, 32, 64, 128])
def test_adagrad_mode_is_rows_adagrad_ref_bit_for_bit(w, n, zero_sum):
    """Fused Adagrad (param + sum) over a list with hot keys across many chunks, unique keys, a negative head and an
    out-of-range tail: every row of param and sum == rows_adagrad_ref(segment_reduce_ref(...)); untouched rows and the guards
    unchanged.  n = 65536 runs the kOpt pass-1 kernel, 65537 the lean one; w = 16 / 32 / 64 / 128 covers NQ = 1 (16 rows in
    flight in kOpt), 1, 2, 4."""
    assert _path(True, n) == ("kopt" if n == KOPT_MAX else "lean")
    rng = np.random.default_rng(w + n)
    n_rows = 6000
    body = np.concatenate([np.full(5000, 11), np.full(3000, 2500), rng.choice(np.arange(3000, 6000), 1500, replace=False),
                           np.sort(rng.zipf(1.2, n - 9500 - 300) % n_rows)])
    keys = np.sort(np.concatenate([np.full(70, -3), np.full(30, -1), body, np.full(100, n_rows), np.full(100, n_rows + 7)]))
    assert keys.size == n and keys[69] == -3 and keys[64] == -3 and keys[-1] == n_rows + 7
    rows = _rows(rng, n, w) * np.float32(0.01)
    p0 = rng.normal(size=(n_rows, w)).astype(np.float32)
    s0 = np.zeros((n_rows, w), np.float32) if zero_sum else np.abs(rng.normal(size=(n_rows, w))).astype(np.float32)
    ids, g = util.segment_reduce_ref(keys, rows, n_rows)
    p_ref, s_ref = util.rows_adagrad_ref(p0[ids], s0[ids], g, LR, EPS)
    P, S = Guarded(n_rows, w, p0), Guarded(n_rows, w, s0)
    _launch(keys, rows, n_rows, param=P, state=S)
    for buf, ref, what in ((P, p_ref, "param"), (S, s_ref, "sum")):
        got, want = buf.get(), buf.expect(ids, ref)
        bad = np.flatnonzero(_bits(got) != _bits(want))
        assert bad.size == 0, (what, _path(True, n), w, bad[:8])
    # the same call again from the same start: bit-identical
    P2, S2 = Guarded(n_rows, w, p0), Guarded(n_rows, w, s0)
    _launch(keys, rows, n_rows, param=P2, state=S2)
    assert np.array_equal(_bits(P2.get()), _bits(P.get())) and np.array_equal(_bits(S2.get()), _bits(S.get()))


@pytest.mark.parametrize("n", [KOPT_MAX, KOPT_MAX + 1], ids=["kopt", "lean"])
def test_one_row_table_with_one_run_over_every_chunk(n):
    """n_rows = 1 and n equal keys (1025 or 1026 chunks): one row in both modes."""
    rng = np.random.default_rng(n)
    w = 33
    keys = np.zeros(n, np.int64)
    rows = _rows(rng, n, w) * np.float32(0.01)
    ids, g = util.segment_reduce_ref(keys, rows, 1)
    out = Guarded(1, w)
    _launch(keys, rows, 1, grad_out=out)
    assert np.array_equal(_bits(out.get()), _bits(out.expect(ids, g)))
    p0, s0 = rng.normal(size=(1, w)).astype(np.float32), np.full((1, w), 0.5, np.float32)
    p_ref, s_ref = util.rows_adagrad_ref(p0, s0, g, LR, EPS)
    P, S = Guarded(1, w, p0), Guarded(1, w, s0)
    _launch(keys, rows, 1, param=P, state=S)
    assert np.array_equal(_bits(P.get()), _bits(P.expect(ids, p_ref)))
    assert np.array_equal(_bits(S.get()), _bits(S.expect(ids, s_ref)))


@pytest.mark.parametrize("n", [1000, KOPT_MAX + 1], ids=["kopt", "lean"])
def test_out_of_range_ids_move_nothing(n):
    """Only ids outside [0, n_rows) — negative, == n_rows, > n_rows — over several chunks: nothing moves, in either mode."""
    rng = np.random.default_rng(1)
    w, n_rows = 64, 50
    keys = np.sort(np.concatenate([np.full(n // 4, -3), np.full(n // 4, -1), np.full(n // 4, n_rows),
                                   np.full(n - 3 * (n // 4), n_rows + 1000)]))
    rows = _rows(rng, n, w)
    out = Guarded(n_rows, w)
    _launch(keys, rows, n_rows, grad_out=out)
    assert np.array_equal(_bits(out.get()), _bits(out.host0))
    P, S = Guarded(n_rows, w, rng.normal(size=(n_rows, w))), Guarded(n_rows, w, np.ones((n_rows, w)))
    _launch(keys, rows, n_rows, param=P, state=S)
    assert np.array_equal(_bits(P.get()), _bits(P.host0)) and np.array_equal(_bits(S.get()), _bits(S.host0))


def test_ops_rows_adagrad_does_not_wrap_int64_ids():
    """ops.rows_adagrad takes int64 ids: 2**32 + 5 must not alias row 5, 2**31 + 1 must not turn negative."""
    rng = np.random.default_rng(4)
    w, n_rows = 8, 10
    p0 = rng.normal(size=(n_rows, w)).astype(np.float32)
    s0 = np.full((n_rows, w), 0.25, np.float32)
    rows = rng.normal(size=(4, w)).astype(np.float32)
    keys = torch.tensor([-5, 5, 2 ** 31 + 1, 2 ** 32 + 5], dtype=torch.int64, device="cuda")
    P, S = torch.from_numpy(p0.copy()).cuda(), torch.from_numpy(s0.copy()).cuda()
    ops.rows_adagrad(keys, torch.from_numpy(rows).cuda(), P, S, LR, EPS)
    p_ref, s_ref = p0.copy(), s0.copy()
    p_ref[5], s_ref[5] = util.rows_adagrad_ref(p0[5], s0[5], rows[1], LR, EPS)
    assert np.array_equal(_bits(P.cpu().numpy()), _bits(p_ref)) and np.array_equal(_bits(S.cpu().numpy()), _bits(s_ref))
    with pytest.raises(RuntimeError, match="keys must be 1-D"):
        ops.rows_adagrad(keys[:3], torch.from_numpy(rows).cuda(), P, S, LR, EPS)


# ---- through the pair backward ------------------------------------------------------------------------------------------------

def _dense_batch(rng, N, R, B, H, one_user=False):
    if one_user:
        hist = np.broadcast_to(rng.choice(N, H, replace=False), (B, H)).copy()
    else:
        hist = rng.integers(0, N, (B, H))
        hist[:, :5] = 7                                  # a hot item: >= 5 B entries, a run over 40+ chunks
    tgt = rng.integers(0, N, B)
    region = rng.integers(0, R, N)
    aux = (rng.random((B, H, 2)) * 0.1).astype(np.float32)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return (dev(hist), dev(tgt), dev(region[hist]), dev(region[tgt]), dev(aux))


def _segmented_batch(variant, N, seed):
    data = synthetic.make_checkins(11, N, seed=seed, hist_len=None, max_hist=150, min_hist=2, median_hist=14)
    csr = data.train_csr()
    bt = PB.DeviceBatcher(csr, data.region, data.coords, device="cuda", seed=0)
    b = bt.multi_user_batch(np.arange(csr.shape[0]), 4, seed=seed)
    return (b, None, None, None, None), data.region_num


def _forward_backward(variant, D, hid, batch, R, N, pp, seed):
    """Parameters, one forward and one dscore, and the dense gradients of nais_pairs_backward."""
    rng = np.random.default_rng(seed)
    sd = orc.init_state(variant, N, D, hid, R, 1, seed=seed, style="trained")
    P = {n: sd[n].cuda().contiguous() for n in ops.VARIANT_PARAMS[variant]}
    drop = (0.0, 0, pp)
    _, row_sum, parts, mask = ops.pairs_forward_raw(variant, 0.5, P, *batch, drop)
    dscore = torch.from_numpy(rng.normal(size=int(row_sum.shape[1])).astype(np.float32)).cuda()
    G = ops.pairs_backward_raw(variant, 0.5, P, *batch, row_sum, parts, dscore, drop, act_mask=mask)
    return P, G, (row_sum, parts, dscore, drop, mask)


def _tables(variant):
    return [n for n in ops.VARIANT_PARAMS[variant] if n in ops._TABLES]


def _assert_rows_bitwise(got, ref, what):
    bad = np.flatnonzero((_bits(got) != _bits(ref)).any(1))
    assert bad.size == 0, (what, bad[:8])


def _fused_equals_dense_then_ref(variant, D, hid, batch, R, N, pp, seed):
    """nais_pairs_backward_adagrad == rows_adagrad_ref(dense gradients of nais_pairs_backward) on every row of every table and
    of its optimizer sum (the first table starts from a zero sum, the next from a non-zero one, ...)."""
    P, G, (row_sum, parts, dscore, drop, mask) = _forward_backward(variant, D, hid, batch, R, N, pp, seed)
    rng = np.random.default_rng(seed + 1)
    tables = _tables(variant)
    sums = {n: torch.from_numpy(np.abs(rng.normal(size=tuple(P[n].shape))).astype(np.float32) * (i % 2)).cuda()
            for i, n in enumerate(tables)}
    P2 = {n: t.clone() for n, t in P.items()}
    S2 = {n: t.clone() for n, t in sums.items()}
    ops.pairs_backward_adagrad(variant, 0.5, P2, S2, LR, EPS, *batch, row_sum, parts, dscore, drop, act_mask=mask)
    ops.check_indices(sync=True)
    for n in tables:
        g = G[n].cpu().numpy()
        assert np.count_nonzero(np.abs(g).sum(1)) > 1, n
        p_ref, s_ref = util.rows_adagrad_ref(P[n].cpu().numpy(), sums[n].cpu().numpy(), g, LR, EPS)
        _assert_rows_bitwise(P2[n].cpu().numpy(), p_ref, (variant, D, pp, n, "param"))
        _assert_rows_bitwise(S2[n].cpu().numpy(), s_ref, (variant, D, pp, n, "sum"))


# (variant, D, hid, B, H): list lengths and the pass-1 kernel each table's reduce runs
BWD_CASES = {
    # history 65 536 entries (kOpt, w = 32), regions 66 048 over 6 rows (lean, hot keys over ~170 chunks each), targets 512
    "rd64_B512": ("region_distance", 64, 64, 512, 128),
    # history 65 664, regions 66 177: both lean
    "rd64_B513": ("region_distance", 64, 64, 513, 128),
    "rd32_B512": ("region_distance", 32, 64, 512, 128),   # w = 16: kOpt with 16 rows in flight
    "rd128_B513": ("region_distance", 128, 64, 513, 128),  # w = 64, lean
    "rd128_B512": ("region_distance", 128, 64, 512, 128),  # w = 64, kOpt
    "basic128_B512": ("basic", 128, 64, 512, 128),         # w = 128, kOpt (FP32 backward)
    "basic96_B513": ("basic", 96, 64, 513, 128),           # w = 96, lean
}
TC_SHAPES = {(32, 64), (64, 64)}  # (D, hid) with a tcgen05 backward (csrc/nais_pairs_tc_bwd.cu)


@pytest.mark.parametrize("pp", ["tc", "fp32"])
@pytest.mark.parametrize("case", list(BWD_CASES))
def test_fused_backward_step_equals_dense_gradients_then_reference(case, pp):
    variant, D, hid, B, H = BWD_CASES[case]
    if pp == "tc" and (D, hid) not in TC_SHAPES:
        pytest.skip("no tcgen05 backward at this shape")
    rng = np.random.default_rng(B + D)
    N, R = 3000, 6
    batch = _dense_batch(rng, N, R, B, H)
    if variant == "basic":
        batch = batch[:2] + (None, None, None)
    n_hist = B * H
    assert _path(True, n_hist) == ("kopt" if B == 512 else "lean")
    _fused_equals_dense_then_ref(variant, D, hid, batch, R, N, pp, seed=B + D)


@pytest.mark.parametrize("pp", ["tc", "fp32"])
def test_fused_backward_step_one_user_batch(pp):
    """The reference's one-user batch: one history repeated over (1 + num_ng) * H rows."""
    rng = np.random.default_rng(8)
    H = 23
    batch = _dense_batch(rng, 500, 4, 5 * H, H, one_user=True)
    _fused_equals_dense_then_ref("region_distance", 64, 64, batch, 4, 500, pp, seed=8)


@pytest.mark.parametrize("variant,pp", [("region_distance", "tc"), ("region_distance", "fp32"), ("disentangled", "fp32")])
def test_fused_backward_step_segmented_batch(variant, pp):
    """A multi-user batch in the segmented layout; the two-branch disentangled model steps its region table through
    sum_reg[1]."""
    N = 700
    batch, R = _segmented_batch(variant, N, seed=3)
    _fused_equals_dense_then_ref(variant, 64, 64, batch, R, N, pp, seed=3)


@pytest.mark.parametrize("pp", ["tc", "fp32"])
def test_row_compacted_gradients_are_the_dense_rows(pp):
    """pairs_backward_compact: the touched rows of every table == the dense gradients at the returned ids, bit for bit."""
    rng = np.random.default_rng(12)
    N, R = 3000, 6
    batch = _dense_batch(rng, N, R, 512, 128)
    P, G, (row_sum, parts, dscore, drop, mask) = _forward_backward("region_distance", 64, 64, batch, R, N, pp, seed=12)
    remaps = {n: torch.zeros(P[n].shape[0], dtype=torch.int32, device="cuda") for n in _tables("region_distance")}
    _, sparse = ops.pairs_backward_compact("region_distance", 0.5, P, *batch, row_sum, parts, dscore, remaps, drop, act_mask=mask)
    assert set(sparse) == set(remaps)
    for n, (ids, rows) in sparse.items():
        g = G[n].cpu().numpy()
        i = ids.cpu().numpy()
        assert np.array_equal(_bits(rows.cpu().numpy()), _bits(g[i])), n
        rest = np.ones(len(g), bool)
        rest[i] = False
        assert not _bits(g[rest]).any(), n                 # the dense gradient has nothing outside the returned ids


@pytest.mark.parametrize("pp", ["tc", "fp32"])
def test_sparse_row_exchange_world_1_equals_the_fused_step(pp):
    """SparseRowExchange.step at world size 1 (row-compacted gradients -> nais_rows_adagrad, unique ids) moves every table row and
    optimizer sum exactly as the fused step (nais_pairs_backward_adagrad) does with the same dscore, bit for bit."""
    from poi_recommendation_models_b200.distributed import SparseRowExchange
    rng = np.random.default_rng(13)
    variant, N, R, B, H = "region_distance", 3000, 6, 512, 128
    batch = _dense_batch(rng, N, R, B, H)
    label = torch.from_numpy((rng.random(B) < 0.2).astype(np.float32)).cuda()
    sd = orc.init_state(variant, N, 64, 64, R, 1, seed=13, style="trained")
    m = util.make_model(variant, sd, 0.5)
    m.pairs_precision = pp
    opt = torch.optim.Adagrad(m.parameters(), lr=LR, eps=EPS)
    P = m._params()
    for n in _tables(variant):
        opt.state[P[n]]["sum"].copy_(torch.from_numpy(np.abs(rng.normal(size=tuple(P[n].shape))).astype(np.float32)))
    P0 = {n: t.detach().clone() for n, t in P.items()}
    S0 = {n: opt.state[P[n]]["sum"].clone() for n in _tables(variant)}
    SparseRowExchange(m, opt, world=1).step(label, *batch)
    # the fused step from the same start with the dscore the exchange's BCE loss gives
    drop = (0.0, 0, pp)
    score, row_sum, parts, mask = ops.pairs_forward_raw(variant, 0.5, P0, *batch, drop)
    s = score.detach().requires_grad_(True)
    m.loss_func(torch.sigmoid(s), label).backward()
    ops.pairs_backward_adagrad(variant, 0.5, P0, S0, LR, EPS, *batch, row_sum, parts, s.grad, drop, act_mask=mask)
    torch.cuda.synchronize()
    for n in _tables(variant):
        assert torch.equal(P[n].detach().view(torch.int32), P0[n].view(torch.int32)), n
        assert torch.equal(opt.state[P[n]]["sum"].view(torch.int32), S0[n].view(torch.int32)), n
