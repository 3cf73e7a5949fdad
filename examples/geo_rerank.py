"""Users per second of the power-law geo re-ranking paths on one GPU:

    rerank_topk        composed path: whole-catalogue scores (unplanned nais_fullrank_scores), log G (nais_powerlaw_logscore),
                       the mix and torch.topk, in slices of users of at most 1 GiB of [users, N] temporaries
    fused_rerank_topk  nais_powerlaw_logmax + the geo mode of the full-rank kernel against the model's ranking plan
    predict_topk       the plain full-rank top-k (no geo term), for the cost of the mix

Shapes: C2 (40 000 POIs, H = 128, k = 20, 2048 users) and the C4 catalogue (1 000 000 POIs, 256 users), for
NAIS_region_distance_Embedding, plus the two-branch disentangled model at C2.  Trained-style weights, a = 0.8, b = -1.3,
alpha = 0.2, precision "auto".  Times: CUDA events around each call (which ends in its own device work), after one warm-up
call per path and shape (the ranking plan is built then and reused, as in an evaluation); the median of `--reps` calls.
The fused path's lists are checked against rerank_topk's on the first 64 users (ids equal outside 1e-4 tie bands).

    python examples/geo_rerank.py --out profiles/r3_geo_rerank.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import nais_oracle as orc  # noqa: E402
from poi_recommendation_models_b200 import model as M  # noqa: E402
from poi_recommendation_models_b200 import powerlaw as PL  # noqa: E402

A_, B_, ALPHA = 0.8, -1.3, 0.2


def _gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (x.strip() for x in q.split(","))
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # noqa: BLE001
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unknown ({e})"}


def _model(variant, N, D, seed=0):
    rng = np.random.default_rng(seed)
    R = 64
    sd = orc.init_state(variant, N, D, D, R, 1, seed=seed, style="trained")
    cls = M.CLASSES[variant]
    m = cls(N, D, D, 0.5, R, 1)
    m.load_state_dict(sd)
    m = m.cuda().eval()
    coords = np.stack([40.7 + rng.normal(0, 0.1, N), -74.0 + rng.normal(0, 0.1, N)], 1)
    m.set_catalog(region=rng.integers(0, R, N), coords=coords)
    return m


def _users(m, N, U, H, seed=1):
    rng = np.random.default_rng(seed)
    indptr = np.arange(U + 1, dtype=np.int64) * H
    return m.make_users(indptr, rng.integers(0, N, U * H))


def _time(fn, reps):
    fn()  # warm-up: modules, plans
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), out


def _agree(fused, composed, n=64):
    fv, fi = (t[:n].cpu().numpy() for t in fused)
    rv, ri = (t[:n].cpu().numpy() for t in composed)
    bad = 0
    for u in range(fv.shape[0]):
        for r in range(fv.shape[1]):
            if fi[u, r] != ri[u, r] and abs(float(fv[u, r]) - float(rv[u, r])) >= 1e-4:
                bad += 1
    return bad == 0, float(np.max(np.abs(fv - rv)))


def run_case(name, variant, N, U, H, k, D, reps):
    m = _model(variant, N, D)
    users = _users(m, N, U, H)
    t_rr, rr = _time(lambda: PL.rerank_topk(m, users, k, A_, B_, ALPHA), reps)
    t_fu, fu = _time(lambda: PL.fused_rerank_topk(m, users, k, A_, B_, ALPHA), reps)
    t_pt, _ = _time(lambda: m.predict_topk(users, k), reps)
    same, maxdiff = _agree(fu, rr)
    res = {"case": name, "model": type(m).__name__, "N": N, "users": U, "H": H, "k": k, "D": D, "hid": D,
           "precision": m.ranking_plan("auto").precision,
           "ms": {"rerank_topk": t_rr, "fused_rerank_topk": t_fu, "predict_topk": t_pt},
           "users_per_s": {"rerank_topk": U / t_rr * 1e3, "fused_rerank_topk": U / t_fu * 1e3, "predict_topk": U / t_pt * 1e3},
           "fused_speedup_vs_rerank_topk": t_rr / t_fu, "fused_cost_vs_predict_topk": t_fu / t_pt,
           "fused_lists_match_rerank_topk_outside_1e-4_ties": same, "max_abs_value_diff_vs_rerank_topk": maxdiff}
    print(json.dumps(res), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--small", action="store_true", help="tiny shapes (a functional check, not a measurement)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("this measurement needs a CUDA device")
    torch.manual_seed(0)
    if args.small:
        cases = [("tiny", "region_distance", 2000, 64, 32, 20, 64)]
    else:
        cases = [("C2", "region_distance", 40000, 2048, 128, 20, 64),
                 ("C2_disentangled", "disentangled", 40000, 2048, 128, 20, 64),
                 ("C4", "region_distance", 1000000, 256, 128, 20, 64)]
    out = {"what": "users/s of rerank_topk vs fused_rerank_topk vs predict_topk (examples/geo_rerank.py)",
           "law": {"a": A_, "b": B_, "alpha": ALPHA}, "timing": f"CUDA events, median of {args.reps} after one warm-up call",
           **_gpu_info(), "results": [run_case(*c, reps=args.reps) for c in cases]}
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
