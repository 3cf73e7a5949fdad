"""Shared helpers for the parity tests."""
import os

import numpy as np
import torch

from oracle import nais_oracle as orc

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TOL = 1e-4  # north_star: per-pair scores within 1e-4 relative (condition-aware, SURVEY.md §7)


def load_golden(name):
    return np.load(os.path.join(GOLDEN, name), allow_pickle=False)


def golden_sd(z, prefix):
    return {k[len(prefix):]: torch.from_numpy(z[k]) for k in z.files if k.startswith(prefix)}


def make_model(variant, sd, beta, device="cuda"):
    from poi_recommendation_models_b200 import model as M
    N = sd["embed_history.weight"].shape[0]
    hid = sd["attn_layer1.weight"].shape[0]
    lanes = 2 if orc.VARIANTS[variant]["dist"] == "latlon" else 0
    D = sd["attn_layer1.weight"].shape[1] - lanes
    R = sd["embed_region.weight"].shape[0] if "embed_region.weight" in sd else 1
    cls = M.CLASSES[variant]
    if variant == "basic":
        m = cls(N, D, hid, beta)
    elif variant == "region":
        m = cls(N, D, hid, beta, R)
    else:
        m = cls(N, D, hid, beta, R, 1)
    m.load_state_dict(sd, strict=True)
    return m.to(device).eval()


def call(m, variant, hist, tgt, hreg, treg, aux, pre_sigmoid=True):
    fn = m.attention_network if pre_sigmoid else m.forward
    if variant == "basic":
        return fn(hist, tgt)
    if variant == "region":
        return fn(hist, tgt, hreg, treg)
    if variant == "distance":
        return fn(hist, tgt, aux) if pre_sigmoid else fn(hist, tgt, hreg, treg, aux)
    return fn(hist, tgt, hreg, treg, aux)


def cond_err(got, ref64, scale):
    """max |got-ref| / max(|ref|, sum_h|w_h s_h|)"""
    got, ref64, scale = (np.asarray(t, dtype=np.float64) for t in (got, ref64, scale))
    return float(np.max(np.abs(got - ref64) / np.maximum(np.maximum(np.abs(ref64), scale), 1e-30)))


def oracle_user_scores(sd, variant, beta, coords, region, history, cand, dtype=torch.float64):
    """Oracle scores (and conditioning scale) of one user against explicit candidates, history items included
    (their own cell masked)."""
    history = np.asarray(history, dtype=np.int64)
    cand = np.asarray(cand, dtype=np.int64)
    B = len(cand)
    hist = torch.from_numpy(history)[None, :].expand(B, -1)
    hreg = torch.from_numpy(region[history])[None, :].expand(B, -1)
    treg = torch.from_numpy(region[cand])
    aux = None
    if orc.VARIANTS[variant]["dist"] == "latlon":
        aux = torch.from_numpy(orc.latlon_abs_diff(coords, cand, history[None, :].repeat(B, 0)))
    elif orc.VARIANTS[variant]["dist"] == "km":
        aux = torch.from_numpy(orc.dist_km(coords[cand][:, None, 0], coords[cand][:, None, 1], coords[history][None, :, 0],
                                           coords[history][None, :, 1]))  # float64 km, powerLaw.dist
    s, scale = orc.attention_network_with_scale(sd, variant, beta, hist, torch.from_numpy(cand), hreg, treg, aux, dtype=dtype)
    return s.numpy(), scale.numpy()


SEG_CHUNK = 64  # entries per pass-1 chunk of the sorted-segment reduce (csrc/nais_bwd.cu)


def segment_reduce_ref(keys, rows, n_rows):
    """The embedding-gradient segment reduce of csrc/nais_bwd.cu restated in float32, in its documented summation order, so
    it must equal the kernel bit for bit: every maximal run of equal keys is split at multiples of SEG_CHUNK into pieces; a
    piece is 0.f + r[a] + r[a+1] + ... in entry order; a run's gradient is its first piece plus the following pieces, added in
    chunk order.  Runs whose key is outside [0, n_rows) are dropped.  keys [n] ascending, rows [n, w] float32.
    Returns (ids int64 [runs], grads float32 [runs, w]) of the kept runs, ids ascending."""
    keys = np.asarray(keys, dtype=np.int64)
    rows = np.asarray(rows, dtype=np.float32)
    n, w = rows.shape
    assert keys.shape == (n,) and (n == 0 or np.all(np.diff(keys) >= 0)), "keys must be ascending, one per row"
    if n == 0:
        return np.zeros(0, np.int64), np.zeros((0, w), np.float32)
    idx = np.arange(n)
    run_start = np.ones(n, bool)
    run_start[1:] = keys[1:] != keys[:-1]
    piece_start = run_start | (idx % SEG_CHUNK == 0)
    piece = np.cumsum(piece_start) - 1                       # piece of each entry
    first = idx[piece_start]                                 # first entry of each piece
    pos = idx - first[piece]                                 # position inside the piece (< SEG_CHUNK)
    acc = np.zeros((len(first), w), np.float32)
    for p in range(int(pos.max()) + 1):                      # one entry per piece per step: no repeated index in a step
        sel = pos == p
        acc[piece[sel]] += rows[sel]
    run_of_piece = np.cumsum(run_start[first]) - 1
    run_first_piece = np.flatnonzero(run_start[first])
    k_in_run = np.arange(len(first)) - run_first_piece[run_of_piece]
    g = acc[run_first_piece].copy()
    for k in range(1, int(k_in_run.max()) + 1):
        sel = k_in_run == k
        g[run_of_piece[sel]] += acc[sel]
    ids = keys[run_start]
    keep = (ids >= 0) & (ids < n_rows)
    return ids[keep], g[keep]


def fmaf32(a, b, c):
    """fmaf(a, b, c) on float32 arrays, rounded once like the device instruction: a*b is exact in float64, the float64 two-sum
    of a*b and c is exact, and where rounding that sum to float32 falls on a tie the residual decides the direction."""
    a, b, c = (np.asarray(x, dtype=np.float32) for x in (a, b, c))
    ab = a.astype(np.float64) * b.astype(np.float64)
    cd = c.astype(np.float64)
    t = ab + cd
    bb = t - ab
    err = (ab - (t - bb)) + (cd - bb)
    r = t.astype(np.float32)
    rd = r.astype(np.float64)
    with np.errstate(invalid="ignore"):
        other = np.nextafter(r, np.where(t > rd, np.float32(np.inf), np.float32(-np.inf)).astype(np.float32))
        tie = (rd != t) & ((rd + other.astype(np.float64)) * 0.5 == t)
        # on a tie, the exact value t + err lies on err's side: take the float32 neighbour on that side
        flip = tie & (err != 0) & (np.sign(err) != np.sign(rd - t))
    return np.where(flip, other, r).astype(np.float32)


def rows_adagrad_ref(param, state_sum, g, lr, eps):
    """The row-sparse Adagrad step of the segment reduce (csrc/nais_bwd.cu seg_store) in float32:
    s2 = fmaf(g, g, s);  p - (lr * g) / (sqrt(s2) + eps).  Returns (param, sum).  (torch.optim.Adagrad computes
    p + (-lr) * (g / d), which can differ from this by one ulp.)"""
    g = np.asarray(g, dtype=np.float32)
    s2 = fmaf32(g, g, state_sum)
    lr, eps = np.float32(lr), np.float32(eps)
    p = np.asarray(param, dtype=np.float32) - (lr * g) / (np.sqrt(s2) + eps)
    return p.astype(np.float32), s2


def lists_equal_outside_ties(got_ids, got_scores, ref_scores_by_id, k, tol=TOL):
    """got list must be a valid top-k of ref scores: every listed id's ref score >= (k-th best ref score) - tie tol,
    and the ref order is respected outside tie groups."""
    ref_sorted = np.sort(np.asarray(list(ref_scores_by_id.values()), dtype=np.float64))[::-1]
    kth = ref_sorted[min(k, len(ref_sorted)) - 1]
    for pos, i in enumerate(got_ids[:k]):
        r = ref_scores_by_id[int(i)]
        band = tol * max(abs(r), abs(kth), 1e-30)
        assert r >= kth - band, f"id {i} at rank {pos} has ref score {r} < kth {kth}"
        # rank consistency: the ref score at this rank differs from r by at most the tie band
        assert abs(ref_sorted[pos] - r) <= tol * max(abs(r), abs(ref_sorted[pos]), 1e-30) + 0.0, (pos, r, ref_sorted[pos])
