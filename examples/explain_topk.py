"""What explaining the ranked lists costs next to ranking them (model.explain vs model.predict_topk) on one GPU.

Shape C2: 40 000 POIs, H = 128, D = hid = 64, NAIS_region_distance_Embedding with trained-style weights, precision "auto",
user slices of 2 048, k = 20, m = 5.  Per slice: predict_topk (against the model's ranking plan, built in the warm-up), then
explain of its lists — 2 048 x 20 rows x 128 history items = 5.2 M pair cells through the pair forward with per-cell terms and
the selection kernel.  The two calls alternate in one run, each timed with CUDA events (each call ends in its own device work),
after one warm-up of each; the medians over `--slices` slices are reported with their ratio.  A second run of two slices under
torch.profiler gives the kernel split of explain (forward with cells, selection).  The card's name and power limit are read in
the same process.

    python examples/explain_topk.py --out profiles/r3_explain.json
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


def _gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (x.strip() for x in q.split(","))
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # noqa: BLE001
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unknown ({e})"}


def _model(N, D, seed=0):
    rng = np.random.default_rng(seed)
    R = 64
    sd = orc.init_state("region_distance", N, D, D, R, 1, seed=seed, style="trained")
    m = M.NAIS_region_distance_Embedding(N, D, D, 0.5, R, 1)
    m.load_state_dict(sd)
    m = m.cuda().eval()
    coords = np.stack([40.7 + rng.normal(0, 0.1, N), -74.0 + rng.normal(0, 0.1, N)], 1)
    m.set_catalog(region=rng.integers(0, R, N), coords=coords)
    return m


def _timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-poi", type=int, default=40_000)
    ap.add_argument("--hist", type=int, default=128)
    ap.add_argument("--dim", type=int, default=64)
    ap.add_argument("--users", type=int, default=2048, help="users per slice")
    ap.add_argument("--slices", type=int, default=8)
    ap.add_argument("--k", type=int, default=20)
    ap.add_argument("--m", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("explain_topk.py measures on a CUDA device; none is available")
    N, H, U = args.n_poi, args.hist, args.users
    m = _model(N, args.dim)
    rng = np.random.default_rng(1)
    slices = [m.make_users(np.arange(U + 1, dtype=np.int64) * H, rng.integers(0, N, U * H)) for _ in range(args.slices)]
    # warm-up of both calls (modules, the ranking plan)
    _, ids = m.predict_topk(slices[0], args.k)
    m.explain(slices[0], ids, m=args.m)
    torch.cuda.synchronize()
    t_rank, t_explain = [], []
    for users in slices:
        tr, (score, ids) = _timed(lambda: m.predict_topk(users, args.k))
        te, ex = _timed(lambda: m.explain(users, ids, m=args.m))
        t_rank.append(tr)
        t_explain.append(te)
    # consistency on the last slice: sigmoid(explained score) is the ranked score; every explained POI is a history item
    gap = float((torch.sigmoid(ex.score) - score).abs().max())
    # kernel split, in a run of its own
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for users in slices[:2]:
            _, ids = m.predict_topk(users, args.k)
            m.explain(users, ids, m=args.m)
        torch.cuda.synchronize()
    kern = {}
    for e in prof.key_averages():
        if e.device_type.name == "CUDA" and ("pairs_fwd" in e.key or "explain_select" in e.key or "fullrank" in e.key):
            kern[e.key[:120]] = {"calls": e.count, "total_ms": round(e.device_time_total / 1e3, 4)}
    cells = U * args.k * H
    res = {
        "what": "model.explain (pair forward with per-cell terms + selection) vs model.predict_topk on the same user slices",
        **_gpu_info(), "n_poi": N, "H": H, "D": args.dim, "hid": args.dim, "users_per_slice": U, "k": args.k, "m": args.m,
        "precision": "auto", "slices": args.slices, "cells_per_explain": cells,
        "predict_topk_ms": {"median": round(float(np.median(t_rank)), 4), "all": [round(x, 4) for x in t_rank]},
        "explain_ms": {"median": round(float(np.median(t_explain)), 4), "all": [round(x, 4) for x in t_explain]},
        "explain_over_predict_topk": round(float(np.median(t_explain) / np.median(t_rank)), 5),
        "max_abs_sigmoid_score_gap": gap,
        "kernels_two_slices": kern,
    }
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
