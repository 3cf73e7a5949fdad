"""Power-law geographical weighting of the reference (`/root/reference/powerLaw.py`) — SURVEY.md §8 f4.

    dist(loc1, loc2)                                   powerLaw.py:7-21    great-circle km, law of cosines, R = 6371
    PowerLaw.fit_distance_distribution                 powerLaw.py:57-83   log-log least squares by 2000 GD steps
    PowerLaw.pr_d / PowerLaw.predict                   powerLaw.py:85-92   prod_h a * max(0.01, d)^b
    normalize + (1 - alpha) * prediction + alpha * G   run.py:55-59, 523-546 (the re-ranking the reference keeps commented out)

`PowerLaw` mirrors the reference class (same attributes, same random draws, same fitted a, b to ~1e-12; the pair loop
and the gradient sums are vectorised).  `fused_rerank_topk` is the device path: the per-user maximum of log G in one pass
(`nais_powerlaw_logmax`), then the mix and its top-k inside the full-rank kernel against the model's ranking plan
(`nais_fullrank_topk_geo_planned`) — no [users, N] buffer.  `rerank_topk` is the earlier composed path (whole-catalogue
scores, log G and the mix materialised per slice of users, torch.topk); it stays as the comparison path.  On one B200 the
composed path is the faster of the two today (profiles/r3_geo_rerank.json, DESIGN.md §4.1); the fused one needs no
[users, N] memory and range-shards (distributed.ShardedRanker.topk(geo=...)).
"""
from __future__ import annotations

import ctypes as C
import time
from typing import Optional, Tuple

import numpy as np
import torch

from . import _lib, ops


def dist(loc1, loc2):
    """km between (lat, lon) pairs; arrays broadcast.  powerLaw.py:7-21 incl. the 1e-6-degree short-circuit."""
    lat1, lon1 = np.asarray(loc1[0], dtype=np.float64), np.asarray(loc1[1], dtype=np.float64)
    lat2, lon2 = np.asarray(loc2[0], dtype=np.float64), np.asarray(loc2[1], dtype=np.float64)
    d2r = np.pi / 180.0
    phi1, phi2 = (90.0 - lat1) * d2r, (90.0 - lat2) * d2r
    c = np.sin(phi1) * np.sin(phi2) * np.cos(lon1 * d2r - lon2 * d2r) + np.cos(phi1) * np.cos(phi2)
    out = np.arccos(np.clip(c, -1.0, 1.0)) * 6371
    same = (np.abs(lat1 - lat2) < 1e-6) & (np.abs(lon1 - lon2) < 1e-6)
    return np.where(same, 0.0, out)


class PowerLaw(object):
    def __init__(self, a=None, b=None):
        self.a = a
        self.b = b
        self.check_in_matrix = None
        self.visited_lids = {}
        self.poi_coos = None

    @staticmethod
    def compute_distance_distribution(check_in_matrix, poi_coos):
        """(distances x, probabilities t): histogram of int(km) over every unordered pair of a user's visited POIs,
        normalised, without its first bin (powerLaw.py:41-55)."""
        coos = np.asarray(poi_coos, dtype=np.float64)
        m = check_in_matrix.tocsr()
        counts = np.zeros(1, dtype=np.int64)
        for uid in range(m.shape[0]):
            lids = m.indices[m.indptr[uid]:m.indptr[uid + 1]]
            if len(lids) < 2:
                continue
            i, j = np.triu_indices(len(lids), 1)
            d = dist((coos[lids[i], 0], coos[lids[i], 1]), (coos[lids[j], 0], coos[lids[j], 1])).astype(np.int64)
            c = np.bincount(d)
            if len(c) > len(counts):
                counts = np.concatenate([counts, np.zeros(len(c) - len(counts), dtype=np.int64)])
            counts[:len(c)] += c
        total = 1.0 * counts.sum()
        keys = np.nonzero(counts)[0]
        return keys[1:], (counts[keys] / total)[1:]

    def fit_distance_distribution(self, check_in_matrix, poi_coos):
        self.check_in_matrix = check_in_matrix
        m = check_in_matrix.tocsr()
        for uid in range(m.shape[0]):
            self.visited_lids[uid] = m.indices[m.indptr[uid]:m.indptr[uid + 1]]
        ctime = time.time()
        self.poi_coos = poi_coos
        x, t = self.compute_distance_distribution(check_in_matrix, poi_coos)
        x, t = np.log10(x), np.log10(t)
        w0, w1 = np.random.random(), np.random.random()  # the reference's two draws from numpy's global stream
        lambda_w, alpha = 0.1, 1e-5
        for _ in range(2000):
            r = w0 + w1 * x - t
            d_w0, d_w1 = r.sum(), (r * x).sum()
            w0 -= alpha * (d_w0 + lambda_w * w0)
            w1 -= alpha * (d_w1 + lambda_w * w1)
        self.fit_seconds = time.time() - ctime
        self.a, self.b = 10 ** w0, w1

    def pr_d(self, d):
        return self.a * (np.maximum(0.01, d) ** self.b)

    def predict(self, uid, lj):
        coos = np.asarray(self.poi_coos, dtype=np.float64)
        li = self.visited_lids[uid]
        return np.prod(self.pr_d(dist((coos[li, 0], coos[li, 1]), (coos[lj, 0], coos[lj, 1]))))


def normalize(scores):
    """run.py:55-59"""
    scores = np.asarray(scores, dtype=np.float64)
    mx = scores.max()
    return scores / mx if mx != 0 else scores


def log_scores(cat: ops.DeviceCatalog, users: ops.DeviceUsers, a: float, b: float, poi_begin: int = 0,
               poi_end: Optional[int] = None) -> torch.Tensor:
    """log G [U, poi_end - poi_begin] on the device (nais_powerlaw_logscore)."""
    lib = _lib.load()
    poi_end = cat.row_base + cat.n_rows if poi_end is None else poi_end
    dev = users.offsets.device
    if dev.type != "cuda":
        raise RuntimeError("power-law scoring runs on a CUDA device: there is no CPU path")
    out = torch.empty(users.n_users, poi_end - poi_begin, device=dev, dtype=torch.float32)
    with torch.cuda.device(dev):
        c, u = ops._structs(cat, users)
        _lib.check(lib.nais_powerlaw_logscore(C.byref(c), C.byref(u), poi_begin, poi_end, float(a), float(b), out.data_ptr(),
                                              ops._stream()), "nais_powerlaw_logscore")
    return out


@torch.no_grad()
def rerank_topk(model, users, k: int, a: float, b: float, alpha: float, precision: str = "auto",
                exclude_history: bool = True, max_slice_bytes: int = 1 << 30) -> Tuple[torch.Tensor, torch.Tensor]:
    """Top-k of (1 - alpha) * forward(...) + alpha * normalize(G) over the whole catalogue minus the history
    (run.py:523-546 with the candidate set of validation.py:87).  G is normalised by its maximum over the user's
    candidates, in log space: normalize(G)[j] = exp(log G[j] - max_j log G).  Returns (mixed score [U,k], ids [U,k]).

    The mix needs every candidate's score (the normaliser is a maximum over the catalogue), so this path does materialise
    [users, N] score / log-G tiles — but only for a SLICE of users at a time: at most `max_slice_bytes` of temporaries
    (3 float32 matrices), whatever the batch and the catalogue are (30k users x 1M POIs would be 360 GB at once)."""
    if not isinstance(users, ops.DeviceUsers):
        users = model.make_users(*users)
    N = model._catalog.n_rows
    per = max(1, int(max_slice_bytes // (3 * 4 * max(N, 1))))
    if users.n_users > per and users.host_offsets is not None:
        parts = [rerank_topk(model, users.slice(u0, min(users.n_users, u0 + per)), k, a, b, alpha, precision, exclude_history,
                             max_slice_bytes) for u0 in range(0, users.n_users, per)]
        return torch.cat([v for v, _ in parts]), torch.cat([i for _, i in parts])
    s = ops.fullrank_scores(model.variant, float(model.beta), model._params(), model._catalog, users, precision=precision)
    logg = log_scores(model._catalog, users, a, b)
    if exclude_history:
        rows = torch.repeat_interleave(torch.arange(users.n_users, device=s.device), users.offsets[1:] - users.offsets[:-1])
        hist = users.items.to(torch.int64)
        logg[rows, hist] = float("-inf")
    g = torch.exp(logg - logg.max(dim=1, keepdim=True).values)
    mixed = (1.0 - alpha) * torch.sigmoid(s) + alpha * g
    if exclude_history:
        mixed[rows, hist] = float("-inf")
    val, idx = torch.topk(mixed, k, dim=1)
    return val, idx


@torch.no_grad()
def fused_rerank_topk(model, users, k: int, a: float, b: float, alpha: float, precision: str = "auto",
                      exclude_history: bool = True) -> Tuple[torch.Tensor, torch.Tensor]:
    """`rerank_topk` in two device passes and no [users, N] buffer: M_u = max_j log G over the candidates
    (`ops.powerlaw_logmax`), then the full-rank kernel forms (1 - alpha) * sigmoid(score) + alpha * exp(log G - M_u) per
    candidate and keeps its block top-k by that value (score descending, then id ascending), against `model.ranking_plan`.
    Returns (mixed score [U,k] float32, ids [U,k] int64; -inf / -1 padding).  The model needs a catalogue with coordinates
    (`set_catalog(..., coords=...)`), whatever its own distance input is."""
    if not isinstance(users, ops.DeviceUsers):
        users = model.make_users(*users)
    cat = model._catalog
    if cat is None or cat.coords is None or users.coords is None:
        raise RuntimeError("geo re-ranking needs catalogue coordinates: call set_catalog(..., coords=...) first")
    plan = model.ranking_plan(precision)
    logmax = ops.powerlaw_logmax(cat, users, a, b, 0, model.item_num, exclude_history)
    s, i = ops.fullrank_topk(model.variant, float(model.beta), model._params(), cat, users, k, 0, model.item_num, exclude_history,
                             plan.precision, plan, geo=ops.GeoMix(float(a), float(b), float(alpha), logmax))
    return s, i.to(torch.int64)
