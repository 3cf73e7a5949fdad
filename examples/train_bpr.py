#!/usr/bin/env python
"""BPR training (-log sigmoid(s+ - s-)) on one GPU, NAIS_region_distance_Embedding with D = hid = 64.  Prints one JSON line (with
the GPU's name and power limit) and writes it to profiles/.

  c3     C3-shaped whole optimizer step: 4,096 (user, pos, neg) triples as groups of two rows [pos, neg], each triple with its own
         history of 128, 40,000 POIs.  autograd (attention_network -> -logsigmoid(s+ - s-).mean() -> backward ->
         torch.optim.Adagrad.step) against model.fused_bpr_step (one library call), CUDA events, eager and — where capture
         succeeds — as CUDA-graph replay; library launches per step (nais_launch_count), all CUDA kernels per step (torch.profiler)
         and the first-step loss of both paths from the same weights;
  c1     C1-shaped BPR epoch (1,083 users x 38,333 POIs, 4 negatives per positive, one optimizer step per user): the Python loop of
         fused_bpr_step over DeviceBatcher.multi_user_batch([u]) against model.train_users(loss="bpr") (one library call);
  seg64  fused_bpr_step on 64-user segmented batches with group_weight = 1 / pairs(user).

    python examples/train_bpr.py [--users 1083] [--out profiles/r3_train_bpr.json]
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
from bench import synth_histories  # noqa: E402
from poi_recommendation_models_b200 import _lib, batches as PB, model as M, ops, synthetic  # noqa: E402

D = HID = 64
BETA, NUM_NG, LR = 0.5, 4, 0.01
N_C3, H_C3, T_C3 = 40000, 128, 4096


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or [","])[0].split(",", 1)
    return {"name": name.strip() or torch.cuda.get_device_name(0), "power_limit": power.strip()}


def event_ms(fn, reps):
    """(device ms per call between CUDA events, host ms per call to enqueue it)."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    h0 = time.perf_counter()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    host = (time.perf_counter() - h0) * 1e3 / reps
    b.synchronize()
    return a.elapsed_time(b) / reps, host


def wall_s(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def c3_problem():
    """4,096 triples interleaved [pos, neg]: rows 2g and 2g + 1 share triple g's history (positive in it, negative not)."""
    coords, region, R = synthetic.make_catalog(N_C3, seed=0)
    hist_np = synth_histories(T_C3, N_C3, H_C3, seed=3)
    rng = np.random.default_rng(4)
    pos = hist_np[np.arange(T_C3), rng.integers(0, H_C3, T_C3)]
    neg = rng.integers(0, N_C3, T_C3)
    clash = (hist_np == neg[:, None]).any(1)
    neg[clash] = (neg[clash] + 1) % N_C3
    hist = torch.from_numpy(np.repeat(hist_np, 2, axis=0)).cuda()
    tgt = torch.from_numpy(np.stack([pos, neg], 1).reshape(-1)).cuda()
    reg, c = torch.from_numpy(region).cuda(), torch.from_numpy(coords).cuda()
    ll = (c[tgt][:, None, :] - c[hist]).abs().float().contiguous()
    torch.manual_seed(1)
    m = M.NAIS_region_distance_Embedding(N_C3, D, HID, BETA, R, 1)
    with torch.no_grad():
        for name, p in m.named_parameters():
            if name.startswith("embed_"):
                p.normal_(0, 0.3)
    return m.state_dict(), R, (hist, tgt, reg[hist], reg[tgt], ll)


def c3_models(sd, R):
    m = M.NAIS_region_distance_Embedding(N_C3, D, HID, BETA, R, 1)
    m.load_state_dict(sd)
    m = m.cuda().train()
    return m, torch.optim.Adagrad(m.parameters(), lr=LR)


def autograd_step(m, o, batch):
    o.zero_grad(set_to_none=True)
    v = m.attention_network(*batch).view(-1, 2)
    loss = -torch.nn.functional.logsigmoid(v[:, :1] - v[:, 1:]).mean()
    loss.backward()
    o.step()
    return loss.detach()


def kernels_per_step(fn):
    """CUDA kernels (and memcpy / memset) one call of `fn` runs, from torch.profiler (a run of its own)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    try:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if e.device_type.name == "CUDA"]
    except Exception as e:  # the count is a diagnostic: report why it is missing
        return {"error": f"{type(e).__name__}: {str(e)[:120]}"}
    return {"device_ops": len(names), "kernels": sum(1 for n in names if not n.startswith(("Memcpy", "Memset")))}


def c3(reps, rounds):
    sd, R, batch = c3_problem()
    (m_a, o_a), (m_f, o_f) = c3_models(sd, R), c3_models(sd, R)
    paths = {"autograd": lambda: autograd_step(m_a, o_a, batch), "fused_bpr_step": lambda: m_f.fused_bpr_step(o_f, *batch, num_neg=1)}
    out = {"triples": T_C3, "rows": 2 * T_C3, "history": H_C3, "pois": N_C3, "first_step_loss": {k: float(fn()) for k, fn in paths.items()}}
    lib = _lib.load()
    launches = {}
    for k, fn in paths.items():
        for _ in range(3):
            fn()
        l0 = lib.nais_launch_count()
        fn()
        launches[k] = int(lib.nais_launch_count() - l0)
    res = {k: {"ms": [], "host_ms": []} for k in paths}
    for _ in range(rounds):  # the two paths alternate
        for k, fn in paths.items():
            ms, host = event_ms(fn, reps)
            res[k]["ms"].append(ms)
            res[k]["host_ms"].append(host)
    ops.check_indices(sync=True)
    for k in paths:
        out[k] = {"eager_ms": round(float(np.median(res[k]["ms"])), 4), "eager_ms_spread": round(float(np.ptp(res[k]["ms"])), 4),
                  "host_enqueue_ms": round(float(np.median(res[k]["host_ms"])), 4), "library_launches_per_step": launches[k],
                  "profiler": kernels_per_step(paths[k])}
    out["eager_speedup"] = round(out["autograd"]["eager_ms"] / out["fused_bpr_step"]["eager_ms"], 2)
    return out, paths


def c3_graphs(out, paths, reps, rounds):
    """Each path captured once into a CUDA graph (the shapes are static) and replayed; where capture fails the path stays eager."""
    graphs = {}
    for k, fn in paths.items():
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    fn()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                loss = fn()
            graphs[k] = (g, loss)
            out[k]["graph"] = "captured"
        except Exception as e:  # capture is an optimisation of the measurement, never a requirement
            torch.cuda.synchronize()
            out[k]["graph"] = f"capture failed: {type(e).__name__}: {str(e)[:160]}"
    res = {k: [] for k in graphs}
    for k, (g, _) in graphs.items():
        for _ in range(3):
            g.replay()
    for _ in range(rounds):
        for k, (g, _) in graphs.items():
            res[k].append(event_ms(g.replay, reps)[0])
    for k, (g, loss) in graphs.items():
        out[k]["graph_ms"] = round(float(np.median(res[k])), 4)
        out[k]["graph_ms_spread"] = round(float(np.ptp(res[k])), 4)
        out[k]["graph_last_loss"] = float(loss)
    for k in paths:  # the number each path is compared by, and which mode it is in
        if "graph_ms" in out[k]:
            out[k]["best_ms"], out[k]["best_mode"] = out[k]["graph_ms"], "CUDA graph replay"
        else:
            out[k]["best_ms"], out[k]["best_mode"] = out[k]["eager_ms"], "eager"


def new_model(N, R, sd=None):
    torch.manual_seed(0)
    m = M.NAIS_region_distance_Embedding(N, D, HID, BETA, R, 1).cuda().train()
    if sd is not None:
        m.load_state_dict(sd)
    return m, torch.optim.Adagrad(m.parameters(), lr=LR)


def c1_epoch(users, pois):
    data = synthetic.make_checkins(users, pois, seed=0, hist_len=None, max_hist=100, min_hist=5, median_hist=30)
    bt = PB.DeviceBatcher(data.train_csr(), data.region, data.coords, device="cuda", seed=0)
    order = np.random.default_rng(0).permutation(users)
    sd0 = new_model(pois, data.region_num)[0].state_dict()
    (m_loop, o_loop), (m_all, o_all) = new_model(pois, data.region_num, sd0), new_model(pois, data.region_num, sd0)
    loop_losses = []

    def loop():
        for u in order:
            b = bt.multi_user_batch(np.array([u]), NUM_NG, seed=1 + int(u))
            loop_losses.append(m_loop.fused_bpr_step(o_loop, b, num_neg=NUM_NG))

    loop_s = wall_s(loop)
    losses = []
    users_s = wall_s(lambda: losses.append(m_all.train_users(o_all, bt, order, NUM_NG, seed=1, loss="bpr")))
    ops.check_indices(sync=True)
    same = bool(np.array_equal(torch.stack(loop_losses).cpu().numpy(), losses[0].cpu().numpy()))
    return {"users": users, "pois": pois, "negatives": NUM_NG, "loop_s": round(loop_s, 4), "loop_users_per_s": round(users / loop_s, 1),
            "train_users_s": round(users_s, 4), "train_users_users_per_s": round(users / users_s, 1),
            "train_users_mean_loss": float(losses[0].mean()), "loop_mean_loss": float(torch.stack(loop_losses).mean()),
            "losses_bit_identical": same}


def seg64(reps=20, rounds=5):
    N, U = 38333, 64
    data = synthetic.make_checkins(U, N, seed=2, hist_len=None, max_hist=100, min_hist=5, median_hist=30)
    bt = PB.DeviceBatcher(data.train_csr(), data.region, data.coords, device="cuda", seed=0)
    b = bt.multi_user_batch(np.arange(U), NUM_NG, seed=0)
    groups = np.diff(b.host_row_offsets) // (NUM_NG + 1)
    gw = torch.from_numpy(np.repeat(1.0 / (groups * NUM_NG), groups).astype(np.float32)).cuda()
    m, o = new_model(N, data.region_num)
    step = lambda: m.fused_bpr_step(o, b, num_neg=NUM_NG, group_weight=gw)
    for _ in range(3):
        step()
    ms = [event_ms(step, reps)[0] for _ in range(rounds)]
    ops.check_indices(sync=True)
    med = float(np.median(ms))
    return {"users_per_step": U, "rows": int(b.B), "step_ms": round(med, 4), "step_ms_spread": round(float(np.ptp(ms)), 4),
            "users_per_s": round(U / med * 1e3, 1), "last_loss": float(step())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--users", type=int, default=1083)
    ap.add_argument("--pois", type=int, default=38333)
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_train_bpr.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("train_bpr.py measures on a CUDA device; none is available")
    res = {"gpu": gpu_info(), "model": "NAIS_region_distance_Embedding", "D": D, "hid": HID, "lr": LR}
    res["c1"] = c1_epoch(args.users, args.pois)
    res["seg64"] = seg64(rounds=args.rounds)
    res["c3"], paths = c3(args.reps, args.rounds)
    c3_graphs(res["c3"], paths, args.reps, args.rounds)  # last: a failed capture is reported, nothing after it depends on the stream
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
