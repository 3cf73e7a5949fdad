#!/usr/bin/env python
"""Train-mode dropout (NAIS_basic / NAIS_regionEmbedding, model.py:71,162; D = hid = 64) on one GPU: pairs_precision "fp32" (the
FP32 CUDA-core pair kernels) against "auto" (the tcgen05 pair kernels), alternating in one process.  Prints one JSON line (with the
GPU's name and power limit) and writes it to profiles/.

  c3     C3-shaped dense step (8,192 rows, history 128, 40,000 POIs): the pair forward, the backward with the fused table Adagrad
         (ops.pairs_backward_adagrad) and the whole model.fused_adagrad_step, CUDA events, with and without dropout;
  c1     C1-shaped epoch (1,083 users x 38,333 POIs, 4 negatives per positive, one optimizer step per user, run.py:227-255): the
         Python loop of fused_adagrad_step on dense batches against model.train_users (one library call);
  seg64  fused_adagrad_step on 64-user segmented batches (DeviceBatcher.multi_user_batch).

    python examples/train_dropout.py [--users 1083] [--out profiles/r3_train_dropout.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from poi_recommendation_models_b200 import batches as PB, model as M, ops, synthetic  # noqa: E402

D = HID = 64
BETA, NUM_NG, LR, P_DROP = 0.5, 4, 0.01, 0.5
CLASSES = {"basic": M.NAIS_basic, "region": M.NAIS_regionEmbedding}
PRECISIONS = ("fp32", "auto")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or [","])[0].split(",", 1)
    return {"name": name.strip() or torch.cuda.get_device_name(0), "power_limit": power.strip()}


def new_model(variant, N, R, sd=None):
    torch.manual_seed(0)
    m = (M.NAIS_basic(N, D, HID, BETA) if variant == "basic" else M.NAIS_regionEmbedding(N, D, HID, BETA, R)).cuda().train()
    if sd is not None:
        m.load_state_dict(sd)
    return m, torch.optim.Adagrad(m.parameters(), lr=LR)


def event_ms(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def wall_s(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def c3_step(variant, reps=30, rounds=5):
    N, H, B = 40000, 128, 8192
    data = synthetic.make_checkins(B // (H * (NUM_NG + 1)) + 1, N, seed=1, hist_len=H)
    rng = np.random.default_rng(0)
    hist = torch.from_numpy(np.stack([data.history(int(u)) for u in rng.integers(0, data.num_users, B)])).cuda()
    tgt = torch.from_numpy(rng.integers(0, N, B)).cuda()
    reg = torch.from_numpy(data.region).cuda()
    label = torch.from_numpy((np.arange(B) % (NUM_NG + 1) == 0).astype(np.float32)).cuda()
    pair = (hist, tgt) if variant == "basic" else (hist, tgt, reg[hist], reg[tgt])
    pair5 = pair + (None,) * (5 - len(pair))
    m, o = new_model(variant, N, data.region_num)
    P = m._params()
    sums = {n: o.state[t]["sum"] for n, t in P.items()}
    out = {}
    for pdrop in (P_DROP, 0.0):
        m.drop.p = pdrop
        dscore = torch.randn(B, device="cuda") * 1e-3
        for pp in PRECISIONS:
            m.pairs_precision = pp
            drop = (pdrop, 12345, pp)
            fwd = lambda: ops.pairs_forward_raw(variant, BETA, P, *pair5, drop)
            score, row_sum, parts, mask = fwd()
            bwd = lambda: ops.pairs_backward_adagrad(variant, BETA, P, sums, LR, 1e-10, *pair5, row_sum, parts, dscore, drop, act_mask=mask)
            step = lambda: m.fused_adagrad_step(o, label, *pair)
            for fn in (fwd, bwd, step):
                for _ in range(3):
                    fn()
        res = {pp: {"fwd_ms": [], "bwd_ms": [], "step_ms": []} for pp in PRECISIONS}
        for _ in range(rounds):  # the two precisions alternate
            for pp in PRECISIONS:
                m.pairs_precision = pp
                drop = (pdrop, 12345, pp)
                fwd = lambda: ops.pairs_forward_raw(variant, BETA, P, *pair5, drop)
                score, row_sum, parts, mask = fwd()
                res[pp]["fwd_ms"].append(event_ms(fwd, reps))
                res[pp]["bwd_ms"].append(event_ms(lambda: ops.pairs_backward_adagrad(variant, BETA, P, sums, LR, 1e-10, *pair5, row_sum, parts,
                                                                                     dscore, drop, act_mask=mask), reps))
                res[pp]["step_ms"].append(event_ms(lambda: m.fused_adagrad_step(o, label, *pair), reps))
        key = "dropout" if pdrop > 0 else "no_dropout"
        out[key] = {pp: {k: round(float(np.median(v)), 4) for k, v in r.items()} | {k + "_spread": round(float(np.ptp(v)), 4) for k, v in r.items()}
                    for pp, r in res.items()}
    out["rows"], out["history"], out["pois"] = B, H, N
    return out


def c1_epoch(variant, users, pois):
    data = synthetic.make_checkins(users, pois, seed=0, hist_len=None, max_hist=100, min_hist=5, median_hist=30)
    bt = PB.DeviceBatcher(data.train_csr(), data.region, data.coords, device="cuda", seed=0)
    order = np.random.default_rng(0).permutation(users)
    out = {"users": users, "pois": pois}
    sd0 = new_model(variant, pois, data.region_num)[0].state_dict()
    for pp in PRECISIONS:
        m_loop, o_loop = new_model(variant, pois, data.region_num, sd0)
        m_all, o_all = new_model(variant, pois, data.region_num, sd0)
        for m in (m_loop, m_all):
            m.pairs_precision = pp

        def loop():
            for u in order:
                h, t, lab, hr, tr, _ = bt.batch(int(u), NUM_NG)
                m_loop.fused_adagrad_step(o_loop, lab, h, t) if variant == "basic" else m_loop.fused_adagrad_step(o_loop, lab, h, t, hr, tr)

        loop_s = wall_s(loop)
        losses = []
        users_s = wall_s(lambda: losses.append(m_all.train_users(o_all, bt, order, NUM_NG, seed=1)))
        out[pp] = {"loop_dense_s": round(loop_s, 4), "loop_users_per_s": round(users / loop_s, 1), "train_users_s": round(users_s, 4),
                   "train_users_users_per_s": round(users / users_s, 1), "train_users_mean_loss": float(losses[0].mean())}
    return out


def seg64(variant, reps=20, rounds=5):
    N, U = 38333, 64
    data = synthetic.make_checkins(U, N, seed=2, hist_len=None, max_hist=100, min_hist=5, median_hist=30)
    bt = PB.DeviceBatcher(data.train_csr(), data.region, data.coords, device="cuda", seed=0)
    b = bt.multi_user_batch(np.arange(U), NUM_NG, seed=0)
    m, o = new_model(variant, N, data.region_num)
    res = {pp: [] for pp in PRECISIONS}
    for pp in PRECISIONS:
        m.pairs_precision = pp
        for _ in range(3):
            m.fused_adagrad_step(o, b.label, b)
    for _ in range(rounds):
        for pp in PRECISIONS:
            m.pairs_precision = pp
            res[pp].append(event_ms(lambda: m.fused_adagrad_step(o, b.label, b), reps))
    return {"users": U, "rows": int(b.B), "cells": int(b.n_cells), "pois": N} | {
        pp: {"step_ms": round(float(np.median(v)), 4), "step_ms_spread": round(float(np.ptp(v)), 4)} for pp, v in res.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--users", type=int, default=1083)
    ap.add_argument("--pois", type=int, default=38333)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_train_dropout.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    line = {"gpu": gpu_info(), "dropout_p": P_DROP, "D": D, "hid": HID,
            "results": {v: {"c3": c3_step(v), "c1": c1_epoch(v, args.users, args.pois), "seg64": seg64(v)} for v in CLASSES}}
    s = json.dumps(line)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(args.out), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
