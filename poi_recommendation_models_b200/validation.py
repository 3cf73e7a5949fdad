"""Drop-in for the NAIS validators of the reference's `validation.py` (:7-131).

Same names, arguments and return value (precision_v, recall_v, hit_v, precision_t, recall_t, hit_t), but the per-user
Python loop — candidates = all POIs minus history, chunks of 1024/2048 through `model(...)`, `torch.cat`, `torch.topk`
and 50 `.item()` syncs per user (validation.py:84-127) — is ONE fused full-rank call, `model.predict_topk`.

One argument changes meaning: the reference passes `latlon_mat`, a dense float64 [N,N,2] table of |dlat|,|dlon|
(23.5 GB at N=38,333; run.py:47-54).  Here the same parameter takes `place_coords` [N,2]; the kernel forms the
differences itself.
"""
from __future__ import annotations

import numpy as np
import torch

from . import eval_metrics, powerlaw


def _recommend(model, args, train_matrix, num_users, precision="auto", user_batch=2048, geo=None):
    csr = train_matrix.tocsr()  # read as stored: the history order of getrow(u).indices (validation.py:86); the caller's
    k = int(args.topk)          # matrix is never reordered (the kernels compare ids item by item, sorted or not)
    rec = []
    for u0 in range(0, num_users, user_batch):
        u1 = min(num_users, u0 + user_batch)
        indptr = csr.indptr[u0:u1 + 1] - csr.indptr[u0]
        indices = csr.indices[csr.indptr[u0]:csr.indptr[u1]]
        if geo is None:
            _, ids = model.predict_topk((indptr, indices), k, exclude_history=True, precision=precision)
        else:  # the power-law fusion of run.py:523-546 (alpha = Args.powerlaw_weight), fused into the full-rank kernel
            _, ids = powerlaw.fused_rerank_topk(model, (indptr, indices), k, *geo, precision=precision, exclude_history=True)
        rec.extend(ids.cpu().tolist())
    return [[i for i in r if i >= 0] for r in rec]


def _finish(recommended_list, test_positive, val_positive, k_list):
    precision_v, recall_v, hit_v = eval_metrics.evaluate_mp(val_positive, recommended_list, k_list)
    precision_t, recall_t, hit_t = eval_metrics.evaluate_mp(test_positive, recommended_list, k_list)
    return precision_v, recall_v, hit_v, precision_t, recall_t, hit_t


def NAIS_validation(model, args, num_users, test_positive, val_positive, train_matrix, k_list, precision="auto"):
    """validation.py:7-31."""
    model.eval()
    if model._catalog is None:
        model.set_catalog()
    return _finish(_recommend(model, args, train_matrix, num_users, precision), test_positive, val_positive, k_list)


def NAIS_region_validation(model, args, num_users, test_positive, val_positive, train_matrix, businessRegionEmbedList,
                           k_list, precision="auto"):
    """validation.py:34-59."""
    model.eval()
    model.set_catalog(region=businessRegionEmbedList)
    return _finish(_recommend(model, args, train_matrix, num_users, precision), test_positive, val_positive, k_list)


def NAIS_region_distance_validation(model, args, num_users, test_positive, val_positive, train_matrix,
                                    businessRegionEmbedList, place_coords, k_list, precision="auto",
                                    return_recommended=False, geo=None):
    """validation.py:62-131.  `geo` = (a, b, alpha): rank by (1 - alpha) * prediction + alpha * normalize(G) of the fitted
    power law (`powerlaw.PowerLaw` a, b; alpha = Args.powerlaw_weight) — the fusion the reference keeps commented out
    (validation.py:66 reads alpha and ignores it).  None (the default) ranks by the prediction, as the reference does."""
    model.eval()
    coords = np.asarray(place_coords)
    if coords.ndim != 2 or coords.shape[1] != 2:
        raise ValueError("pass place_coords [N,2] (lat, lon) here; the reference's dense latlon_mat [N,N,2] is not "
                         "needed (and its signs cannot be recovered)")
    model.set_catalog(region=businessRegionEmbedList, coords=coords)
    rec = _recommend(model, args, train_matrix, num_users, precision, geo=geo)
    out = _finish(rec, test_positive, val_positive, k_list)
    return (out, rec) if return_recommended else out
