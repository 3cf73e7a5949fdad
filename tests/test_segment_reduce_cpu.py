"""CPU checks of the sorted-segment reduce's entry point and of its float32 restatement (nais_testutil.segment_reduce_ref /
rows_adagrad_ref), which tests/test_gpu_segment_reduce.py holds the kernels to bit for bit: nais_rows_adagrad rejects bad
arguments before any CUDA call, the vectorised reference equals a plain loop over the documented order, and its fmaf equals an
exact rational computation."""
import ctypes as C
from fractions import Fraction

import numpy as np
import pytest
import torch

import nais_testutil as util
from poi_recommendation_models_b200 import _lib, ops

ERR_NULL, ERR_SHAPE, ERR_ALIGN, ERR_WORKSPACE, ERR_MODE = -1, -2, -3, -4, -5
FAKE = 1 << 20  # a 256-aligned address that is never dereferenced: every check below returns before a CUDA call


def _call(keys=FAKE, rows=FAKE, n=100, w=32, n_rows=10, grad_out=FAKE, param=None, state=None, lr=0.01, eps=1e-10, ws=FAKE,
          ws_bytes=None):
    lib = _lib.load()
    if ws_bytes is None:
        ws_bytes = lib.nais_rows_adagrad_workspace_bytes(max(n, 0), w) if 1 <= w <= 128 else 1 << 30
    return lib.nais_rows_adagrad(keys, rows, n, w, n_rows, grad_out, param, state, lr, eps, ws, ws_bytes, None)


def test_rows_adagrad_workspace_bytes_rejects_bad_shapes():
    lib = _lib.load()
    assert lib.nais_rows_adagrad_workspace_bytes(-1, 32) == 0
    assert lib.nais_rows_adagrad_workspace_bytes(100, 0) == 0
    assert lib.nais_rows_adagrad_workspace_bytes(100, 129) == 0
    # two int slots and a w-wide row per 64-entry chunk, each region 256-aligned
    for n, w in ((1, 1), (64, 32), (65, 128), (65537, 64)):
        nch = (n + 63) // 64
        assert lib.nais_rows_adagrad_workspace_bytes(n, w) >= 2 * (2 * nch * 4) + 2 * nch * w * 4


def test_rows_adagrad_rejects_bad_arguments_before_any_cuda_call():
    for kw in (dict(n=-1), dict(w=0), dict(w=129), dict(n_rows=0), dict(n_rows=-5)):
        assert _call(**kw) == ERR_SHAPE, kw
    # an empty list is a no-op, whatever the pointers
    assert _call(n=0, keys=None, rows=None, grad_out=None, ws=None) == 0
    assert _call(n=0, keys=None, rows=None, grad_out=None, param=None, state=FAKE, ws=None) == 0
    for kw in (dict(keys=None), dict(rows=None), dict(ws=None), dict(grad_out=None), dict(grad_out=None, state=FAKE, param=None)):
        assert _call(**kw) == ERR_NULL, kw
    # gradient mode (sum == NULL) needs grad_out only; Adagrad mode needs param only
    for lr, eps in ((-0.01, 1e-10), (float("nan"), 1e-10), (0.01, -1e-10), (0.01, float("nan"))):
        assert _call(grad_out=None, param=FAKE, state=FAKE, lr=lr, eps=eps) == ERR_MODE, (lr, eps)
    assert _call(ws=FAKE + 4) == ERR_ALIGN
    for n, w in ((1, 1), (100, 32), (64 * 33 + 1, 65), (65537, 128)):
        need = _lib.load().nais_rows_adagrad_workspace_bytes(n, w)
        assert _call(n=n, w=w, ws_bytes=need - 1) == ERR_WORKSPACE, (n, w)
        assert _call(n=n, w=w, grad_out=None, param=FAKE, state=FAKE, ws_bytes=need - 1) == ERR_WORKSPACE, (n, w)


def test_ops_rows_adagrad_checks_shapes_before_the_device():
    p, s = torch.zeros(10, 8), torch.zeros(10, 8)
    with pytest.raises(RuntimeError, match="keys must be 1-D"):
        ops.rows_adagrad(torch.zeros(3, dtype=torch.int64), torch.zeros(4, 8), p, s, 0.1, 1e-10)
    with pytest.raises(RuntimeError, match="keys must be 1-D"):
        ops.rows_adagrad(torch.zeros(4, 1, dtype=torch.int64), torch.zeros(4, 8), p, s, 0.1, 1e-10)
    with pytest.raises(RuntimeError, match="param and its state"):
        ops.rows_adagrad(torch.zeros(4, dtype=torch.int64), torch.zeros(4, 4), p, s, 0.1, 1e-10)
    with pytest.raises(RuntimeError, match="param and its state"):
        ops.rows_adagrad(torch.zeros(4, dtype=torch.int64), torch.zeros(4, 8), p, torch.zeros(9, 8), 0.1, 1e-10)
    with pytest.raises(RuntimeError, match="CUDA device"):
        ops.rows_adagrad(torch.zeros(4, dtype=torch.int64), torch.zeros(4, 8), p, s, 0.1, 1e-10)


# ---- the references themselves ------------------------------------------------------------------------------------------------

def _segment_reduce_loop(keys, rows, n_rows):
    """The documented order, one entry at a time in plain Python over np.float32 scalars."""
    out = {}
    n, w = rows.shape
    i = 0
    while i < n:
        j = i
        while j < n and keys[j] == keys[i]:
            j += 1
        g = None
        a = i
        while a < j:                                   # pieces: [a, min(j, next multiple of 64))
            b = min(j, (a // 64 + 1) * 64)
            piece = [np.float32(0.0)] * w
            for e in range(a, b):
                piece = [np.float32(piece[c] + rows[e, c]) for c in range(w)]
            g = piece if g is None else [np.float32(g[c] + piece[c]) for c in range(w)]
            a = b
        if 0 <= keys[i] < n_rows:
            out[int(keys[i])] = np.array(g, dtype=np.float32)
        i = j
    return out


def _random_keys(rng, n, n_rows):
    layout = rng.integers(4)
    if layout == 0:
        k = rng.integers(-3, n_rows + 3, n)                 # anything, out-of-range ids included
    elif layout == 1:
        k = rng.zipf(1.3, n) % (n_rows + 2) - 1             # a few hot keys
    elif layout == 2:
        k = np.repeat(rng.integers(0, n_rows, 1), n)         # one run
    else:
        k = np.repeat(np.arange(n_rows), rng.integers(0, 70, n_rows))[:n]  # runs of up to 69 entries
        k = np.concatenate([k, np.full(n - len(k), n_rows)])
    return np.sort(k)


@pytest.mark.parametrize("seed", range(12))
def test_segment_reduce_ref_equals_a_plain_loop(seed):
    rng = np.random.default_rng(seed)
    n, w, n_rows = int(rng.integers(1, 300)), int(rng.choice([1, 3, 32, 33])), int(rng.integers(1, 20))
    keys = _random_keys(rng, n, n_rows)
    rows = (rng.normal(size=(n, w)) * np.exp2(rng.integers(-20, 20, (n, 1)))).astype(np.float32)
    rows[rng.random((n, w)) < 0.05] = -0.0
    ids, g = util.segment_reduce_ref(keys, rows, n_rows)
    ref = _segment_reduce_loop(keys, rows, n_rows)
    assert ids.tolist() == sorted(ref)
    for i, r in zip(ids, g):
        assert np.array_equal(r.view(np.uint32), ref[int(i)].view(np.uint32)), int(i)


@pytest.mark.parametrize("seed", range(6))
def test_segment_reduce_ref_on_exact_integers_equals_add_at(seed):
    """Small integers sum exactly in float32 in any order: the reference equals np.add.at on every kept row and drops the rest."""
    rng = np.random.default_rng(100 + seed)
    n, w, n_rows = int(rng.integers(1, 5000)), int(rng.integers(1, 129)), int(rng.integers(1, 50))
    keys = _random_keys(rng, n, n_rows)
    rows = rng.integers(-1000, 1000, (n, w)).astype(np.float32)
    ids, g = util.segment_reduce_ref(keys, rows, n_rows)
    ok = (keys >= 0) & (keys < n_rows)
    dense = np.zeros((n_rows, w), np.float64)
    np.add.at(dense, keys[ok], rows[ok].astype(np.float64))
    assert ids.tolist() == np.unique(keys[ok]).tolist()
    assert np.array_equal(g.astype(np.float64), dense[ids])


def _round_f32(q: Fraction) -> np.float32:
    """q rounded to the nearest float32, ties to even, by exact comparison with the neighbours."""
    r = np.float32(float(q))
    cands = {r, np.nextafter(r, np.float32(np.inf)), np.nextafter(r, np.float32(-np.inf))}
    best = min(cands, key=lambda c: (abs(Fraction(float(c)) - q), int(np.array(c, np.float32).view(np.uint32)) & 1))
    return np.float32(best)


def _check_fmaf(g, s):
    got = util.fmaf32(g, g, s)
    for gi, si, o in zip(g, s, got):
        ref = _round_f32(Fraction(float(gi)) ** 2 + Fraction(float(si)))
        assert np.array([o]).view(np.uint32)[0] == np.array([ref]).view(np.uint32)[0], (float(gi), float(si), float(o), float(ref))


def test_fmaf_reference_equals_exact_rounding_on_random_inputs():
    rng = np.random.default_rng(7)
    n = 4000
    g = (rng.normal(size=n) * np.exp2(rng.integers(-40, 20, n))).astype(np.float32)
    s = (np.abs(rng.normal(size=n)) * np.exp2(rng.integers(-80, 40, n))).astype(np.float32)
    s[::7] = 0.0
    g[::11] = np.float32(1e-45)  # subnormal squares vanish below the float32 range
    _check_fmaf(g, s)


def test_fmaf_reference_breaks_ties_by_the_residual():
    """g = 1 + j * 2^-12 gives g*g = (float32) + 2^-24 exactly for odd j: a float32 tie.  A tiny s on either side must round
    away from the tie toward its sign, and s = 0 to even — where rounding the float64 sum to float32 alone would go to even."""
    gs, ss = [], []
    for j in range(1, 200, 2):
        for e in (-6, 0, 5):
            g = np.float32(np.ldexp(1.0 + j * 2.0 ** -12, e))
            q = Fraction(float(g)) ** 2 / Fraction(2) ** (2 * e)   # in [1, 2): float32 spacing 2^-23
            assert (q * 2 ** 24).denominator == 1 and (q * 2 ** 24).numerator % 2 == 1
            for s in (np.ldexp(1.0, 2 * e - 60), -np.ldexp(1.0, 2 * e - 60), np.ldexp(3.0, 2 * e - 70), 0.0):
                gs.append(g)
                ss.append(np.float32(s))
    g, s = np.array(gs, np.float32), np.array(ss, np.float32)
    _check_fmaf(g, s)
    # the residual mattered: naive double rounding differs on some of these
    naive = (g.astype(np.float64) ** 2 + s.astype(np.float64)).astype(np.float32)
    assert (naive != util.fmaf32(g, g, s)).sum() > 20


def test_rows_adagrad_ref_is_the_documented_float32_formula():
    rng = np.random.default_rng(3)
    p, s, g = (rng.normal(size=500).astype(np.float32) for _ in range(3))
    s = np.abs(s)
    p2, s2 = util.rows_adagrad_ref(p, s, g, 0.05, 1e-10)
    assert p2.dtype == np.float32 and s2.dtype == np.float32
    assert np.array_equal(s2, util.fmaf32(g, g, s))
    want = p - (np.float32(0.05) * g) / (np.sqrt(s2) + np.float32(1e-10))
    assert np.array_equal(p2, want)
    # a zero gradient moves nothing
    p3, s3 = util.rows_adagrad_ref(p, s, np.zeros_like(g), 0.05, 1e-10)
    assert np.array_equal(p3, p) and np.array_equal(s3, s)
