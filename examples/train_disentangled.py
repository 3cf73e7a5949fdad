#!/usr/bin/env python
"""Training throughput of NAIS_region_distance_disentangled_Embedding (model.py:410-541, D = hid = 64) on one GPU, today's path
against the fused one.  Prints one JSON line (with the GPU's name and power limit) and writes it to profiles/.

  epoch  C1-shaped (1,083 users x 38,333 POIs, 4 negatives per positive, one optimizer step per user, run.py:227-255):
         dense batch + host-built dist_km [B,H] (batches.dist_km_pairs) + autograd + torch.optim.Adagrad per user, vs
         model.train_users (one library call for the whole list);
  step   C3-sized multi-user step (13 users x 128 history items x 5 rows per item = 8,320 rows, 40,000 POIs): autograd on the
         dense layout + torch.optim.Adagrad, vs model.fused_adagrad_step on the segmented batch.

  --pairs-precision picks the pair kernels (model.pairs_precision: "auto" = tcgen05 where the shape has them, "fp32" = the FP32
  CUDA-core kernels); a comma list runs each in turn, --repeats times, alternating, and the line holds one entry per run.

    python examples/train_disentangled.py [--users 1083] [--pairs-precision fp32,auto --repeats 2] [--out profiles/....json]
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
from poi_recommendation_models_b200 import batches as PB, model as M, synthetic  # noqa: E402

D = HID = 64
BETA, NUM_NG, LR = 0.5, 4, 0.01


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or [","])[0].split(",", 1)
    return {"name": name.strip() or torch.cuda.get_device_name(0), "power_limit": power.strip()}


def new_model(N, R, pairs_precision, sd=None):
    torch.manual_seed(0)
    m = M.NAIS_region_distance_disentangled_Embedding(N, D, HID, BETA, R, 1).cuda().train()
    if sd is not None:
        m.load_state_dict(sd)
    m.pairs_precision = pairs_precision
    return m, torch.optim.Adagrad(m.parameters(), lr=LR)


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def epoch(users, pois, pairs_precision):
    data = synthetic.make_checkins(users, pois, seed=0, hist_len=None, max_hist=100, min_hist=5, median_hist=30)
    bt = PB.DeviceBatcher(data.train_csr(), data.region, data.coords, device="cuda", seed=0)
    order = np.random.default_rng(0).permutation(users)
    m_ref, o_ref = new_model(pois, data.region_num, pairs_precision)
    sd0 = {k: v.detach().clone() for k, v in m_ref.state_dict().items()}

    def today():
        for u in order:
            h, t, lab, hr, tr, _ = bt.batch(int(u), NUM_NG)
            km = PB.dist_km_pairs(data.coords, t.cpu().numpy(), h[0].cpu().numpy(), device="cuda")
            o_ref.zero_grad()
            m_ref.loss_func(m_ref(h, t, hr, tr, km), lab).backward()
            o_ref.step()

    m_new, o_new = new_model(pois, data.region_num, pairs_precision, sd0)
    losses = []
    t_today = timed(today)
    t_fused = timed(lambda: losses.append(m_new.train_users(o_new, bt, order, NUM_NG, seed=1)))
    return {"users": users, "pois": pois, "steps": users, "today_s": round(t_today, 4), "today_users_per_s": round(users / t_today, 1),
            "train_users_s": round(t_fused, 4), "train_users_users_per_s": round(users / t_fused, 1),
            "train_users_mean_loss": float(losses[0].mean())}


def multi_user_step(pairs_precision, reps=20, warmup=3):
    N, H, U = 40000, 128, 13
    data = synthetic.make_checkins(U, N, seed=1, hist_len=H)
    bt = PB.DeviceBatcher(data.train_csr(), data.region, data.coords, device="cuda", seed=0)
    b = bt.multi_user_batch(np.arange(U), NUM_NG, seed=0)
    ro, tgt = b.host_row_offsets, b.tgt.cpu().numpy()
    hist = np.concatenate([np.broadcast_to(data.history(u), (ro[u + 1] - ro[u], H)) for u in range(U)])
    h, t = torch.from_numpy(hist).cuda(), b.tgt
    reg = torch.from_numpy(data.region).cuda()
    km = PB.dist_km_pairs(data.coords, tgt, hist, device="cuda")
    m_dense, o_dense = new_model(N, data.region_num, pairs_precision)
    m_fused, o_fused = new_model(N, data.region_num, pairs_precision, m_dense.state_dict())

    def dense_step():
        o_dense.zero_grad()
        m_dense.loss_func(m_dense(h, t, reg[h], reg[t], km), b.label).backward()
        o_dense.step()

    def fused_step():
        m_fused.fused_adagrad_step(o_fused, b.label, b)

    out = {"rows": int(b.B), "users": U, "history": H, "pois": N}
    for name, fn in (("autograd_dense_ms", dense_step), ("fused_segmented_ms", fused_step)):
        for _ in range(warmup):
            fn()
        out[name] = round(1e3 * timed(lambda: [fn() for _ in range(reps)]) / reps, 3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--users", type=int, default=1083)
    ap.add_argument("--pois", type=int, default=38333)
    ap.add_argument("--pairs-precision", default="auto", help='"auto", "fp32", "tc", or a comma list run in turn')
    ap.add_argument("--repeats", type=int, default=1, help="rounds over the --pairs-precision list")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_train_disentangled.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    names = args.pairs_precision.split(",")
    line = {"gpu": gpu_info(), "model": "NAIS_region_distance_disentangled_Embedding D=hid=64"}
    runs = []
    for r in range(args.repeats):
        for pp in names:
            runs.append({"pairs_precision": pp, "round": r, "epoch_c1": epoch(args.users, args.pois, pp), "step_c3": multi_user_step(pp)})
    if len(runs) == 1:
        line.update(runs[0])
    else:
        line["runs"] = runs
    s = json.dumps(line)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(args.out), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
