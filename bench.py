#!/usr/bin/env python
"""Headline benchmark: full-rank evaluation throughput of the NAIS region/distance scorer (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--precision tc_auto|tc_split|tc_mix|fp32]
    torchrun --nproc-per-node N ... bench.py --gpus N ...        (one rank per GPU, NCCL)

One *step* = one fused full-rank pass (scoring + top-k) of a batch of `--users-per-step` users against the whole
synthetic catalogue of the workload:

    C2 (default)  Gowalla-shaped: 30,000 users x 40,000 POIs, history 128, D = hid = 64, top-20   [BASELINE configs[1]]
    C4            Yelp-scale:     100,000 users x 1,000,000 POIs, history 128, D = hid = 64, top-20

Successive steps take successive user batches (wrapping around).  With N > 1 GPUs the catalogue is range-sharded
across ranks as far as a shard keeps >= 32k POIs (C4: N shards, as north_star / SURVEY.md §8e prescribe) and the user
batch is sliced across the remaining factor (C2's 40k POIs: user slices only; `distributed.grid_shape`); the per-rank
top-k lists travel as packed 8-byte keys in ONE all-gather over NCCL and are merged on the device; total work per step is
fixed -> "scaling": "strong".

The top-level numbers of the JSON line are C2 (comparable round over round).  The same line carries:

value   users/s with inputs resident in HBM (pair-scores/s = users/s x POIs is reported alongside)
value_exact  the same with the fp32-grade three-pass split (`tc_split`) instead of the default precision gate
e2e     the same metric through the drop-in API (`ShardedRanker.topk_host` on pinned host CSR arrays): host -> device
        copy of the step's histories and device -> host copy of the top-k lists inside the timed region
roofline  tensor roofline of the dominant kernel: algorithmic FLOPs (SURVEY.md §8d: F = 2*hid*(D+2) + 4*hid + 3*D + 16
        per (history item, candidate) cell) / CUDA-event time, against MEASURED_PEAKS.json bf16 (sustained)
c4      BASELINE configs[3]: the 1M-POI catalogue, POI-range shards x 1 on every N (N = 1 included), the SAME 296 users per
        step at every N -> a true strong-scaling curve of the north_star sharding (all-gather + on-device merge)
parity_n  (N > 1) rank 0 re-scores users of the last step ALONE over the full range and compares the lists bit for bit
train_c3  BASELINE configs[2]: 4096 (user, pos, neg) triples, H = 128: pair forward + BPR loss + hand-written backward
c1      (N = 1) BASELINE configs[0]: one training epoch (one-user steps vs 64-user segmented steps) + full-rank eval of all users
cpu_baseline  the UNMODIFIED reference `model.py` class on the host cores (oracle/_ref snapshot; kind "reference"), driven by
        the validation.py:84-127 flow (chunks of 2048, torch.cat, torch.topk(50)), on a bounded sample of users
parity  the CPU arm's users + more users scored by a float64 evaluation of the oracle, against the CUDA path's lists

`--impl reference` times that CPU arm alone and prints the same JSON line with "impl": "reference".

`--dump-outputs DIR` writes what the timed path returned in its last timed step, so that two builds can be compared output for
output (the inputs are seeded: the same arguments give the same inputs): eval mode `scores.npy` (float32, raw pre-sigmoid scores)
and `ids.npy` (float64) of the headline step's top-k lists [users_per_step, k]; train mode `loss.npy` and `grad.<parameter>.npy`
(float32) of the C3 step, taken from the step mode the line reports as `step_mode`: the CUDA-graph replay when it gave the eager
step's loss, else the eager step.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "C2": dict(users=30000, pois=40000, hist=128, D=64, hid=64, k=20, desc="Gowalla-shaped 30k users x 40k POIs, H=128, D=hid=64, top-20"),
    "C4": dict(users=100000, pois=1000000, hist=128, D=64, hid=64, k=20, desc="Yelp-scale 100k users x 1M POIs, H=128, D=hid=64, top-20"),
    "tiny": dict(users=512, pois=4096, hist=32, D=64, hid=64, k=20, desc="tiny self-test"),
}
BETA = 0.5
C4_USERS_PER_STEP = 296  # the c4 block: the same users at every N (2 per SM of one B200)
DTYPES = {"fp32": "f32", "tc_split": "f16x2-split/f32-accum", "tc_mix": "f16+e5m2-corrections/f32-accum", "tc_fast": "f16/f32-accum"}


def flops_per_cell(D, hid):
    return 2 * hid * (D + 2) + 4 * hid + 3 * D + 16  # SURVEY.md §8(d)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm=d.get("hbm_gbs", 6650.0), tf_burst=d.get("bf16_tflops", 1590.0),
                    tf_sust=d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1590.0)), which="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, which="fallback")


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """`--dump-outputs`: one DIR/<name>.npy per array; floats of up to 32 bits as float32, everything else (float64, integers:
    exact up to 2^53) as float64."""
    import torch
    arrays = {k: v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v) for k, v in arrays.items()}
    arrays = {k: v.astype(np.float32 if v.dtype.kind == "f" and v.itemsize <= 4 else np.float64) for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def synth_histories(users, pois, hist, seed=0):
    """Fixed-length histories without replacement: popularity-skewed + local, cheap to generate for 100k users."""
    rng = np.random.default_rng(seed)
    homes = rng.integers(0, pois, users)
    out = np.empty((users, hist), dtype=np.int64)
    span = max(4 * hist, min(pois, 2000))
    for u0 in range(0, users, 4096):
        u1 = min(users, u0 + 4096)
        n = u1 - u0
        # local window around home (in id space, which the catalogue generator leaves spatially unordered -> mix)
        cand = (homes[u0:u1, None] + rng.integers(-span, span, (n, 3 * hist))) % pois
        glob = (rng.pareto(1.0, (n, 3 * hist)) * 50).astype(np.int64) % pois
        pick = np.where(rng.random((n, 3 * hist)) < 0.7, cand, glob)
        for i in range(n):
            _, first = np.unique(pick[i], return_index=True)
            sel = pick[i][np.sort(first)][:hist]
            if len(sel) < hist:  # top up
                extra = np.setdiff1d(rng.permutation(pois)[:4 * hist], sel)[:hist - len(sel)]
                sel = np.concatenate([sel, extra])
            out[u0 + i] = np.sort(sel)
    return out


class ClockSampler:
    """`nvidia-smi -lms 100` streamed for the duration of the timed region (the recipe's clocks line)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.proc = index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            time.sleep(0.3)  # first sample is in flight before the timed region starts
        except Exception:
            self.proc = None

    def stop(self):
        rows = []
        if self.proc is not None:
            try:
                time.sleep(0.15)
                self.proc.terminate()
                out, _ = self.proc.communicate(timeout=5)
                rows = [[x.strip() for x in ln.split(",")] for ln in out.splitlines() if ln.strip()]
            except Exception:
                pass
        sm, mx, pw, reasons = [], [], [], set()
        for r in rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                pw.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        # "under load" = samples drawing more than half of the maximum power seen
        load = [c for c, p_ in zip(sm, pw) if pw and p_ >= 0.5 * max(pw)] or sm
        return {"sm_mhz": float(np.median(load)) if load else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "samples_under_load": len(load),
                "power_w_max": max(pw) if pw else None}


# ----------------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own model.py class on the host cores (oracle/_ref), or the oracle port if no reference is reachable
# ----------------------------------------------------------------------------------------------------------------------
def trained_like_state(cfg, R, seed):
    from oracle import nais_oracle as orc  # CPU arm / checker only
    return orc.init_state("region_distance", cfg["pois"], cfg["D"], cfg["hid"], R, 1, seed=seed, style="trained")


def cpu_arm(cfg, n_users, seed=0, warm=1, keep=None):
    """validation.py:84-127 (chunks of 2048, torch.cat, torch.topk(50)) on the host, all threads, through the UNMODIFIED
    reference class when its snapshot is present (kind "reference"), else through the oracle port.  Returns users/s over
    `n_users` users after `warm` warm-up users.  `keep` (a dict) receives the weights, inputs and the lists / full score
    vectors of the timed users, for `parity_block`."""
    import torch
    from oracle import nais_oracle as orc  # CPU arm only
    from poi_recommendation_models_b200 import synthetic
    torch.set_num_threads(os.cpu_count())
    coords, region, R = synthetic.make_catalog(cfg["pois"], seed=seed)
    sd = trained_like_state(cfg, R, seed + 1)
    hist = synth_histories(warm + n_users, cfg["pois"], cfg["hist"], seed=seed + 2)
    cat = orc.Catalog(coords, region)
    ref_model = orc.reference_model("region_distance", sd, BETA)
    kind = "reference" if ref_model is not None else "port"
    with torch.no_grad():
        for u in range(warm):
            orc.fullrank_user(sd, "region_distance", BETA, cat, hist[u], 50, model=ref_model)
        outs = []
        t0 = time.perf_counter()
        for u in range(warm, warm + n_users):
            outs.append(orc.fullrank_user(sd, "region_distance", BETA, cat, hist[u], 50, return_all=keep is not None, model=ref_model))
        dt = time.perf_counter() - t0
    if keep is not None:
        keep.update(sd=sd, coords=coords, region=region, R=R, hist=hist[warm:warm + n_users], outs=outs)
    return n_users / dt, dt, torch.get_num_threads(), kind


CPU_SAMPLE = {"reference": "unmodified reference model.py class (oracle/_ref snapshot) under the validation.py:84-127 flow (chunk 2048, torch CPU, top-50)",
              "port": "oracle port of validation.py:84-127 (chunk 2048, torch CPU, top-50); no reference snapshot reachable"}


def parity_block(dev, cfg, kept, precision, extra_users=28):
    """SURVEY.md §8(d) 'results-parity checks reported with every throughput number': the CPU arm's users scored again by the
    CUDA path with the SAME weights — our top-50 lists against the reference's (validation.py:84-127 flow, fp32 torch CPU) —
    plus `extra_users` more users whose every candidate is scored by the oracle in float64 with its tensors on the GPU
    (untimed; the checker, not the product).  Never raises: a failure is reported in the block, the throughput line stands."""
    try:
        import torch
        from oracle import nais_oracle as orc  # checker only
        from poi_recommendation_models_b200 import model as M
        N, D, hid, H = cfg["pois"], cfg["D"], cfg["hid"], cfg["hist"]
        m = M.NAIS_region_distance_Embedding(N, D, hid, BETA, kept["R"], 1)
        m.load_state_dict(kept["sd"])
        m = m.to(dev).eval()
        m.set_catalog(region=kept["region"], coords=kept["coords"])
        hist = kept["hist"]
        n = len(hist)
        more = synth_histories(extra_users, N, H, seed=77) if extra_users else np.zeros((0, H), dtype=np.int64)
        allh = np.concatenate([hist, more])
        s, ids = m.predict_topk((np.arange(0, (len(allh) + 1) * H, H, dtype=np.int64), allh.reshape(-1)), 50, precision=precision)
        s, ids = s.cpu().numpy(), ids.cpu().numpy()
        exact, overlap, valid, rel = 0, 0, True, 0.0
        for u, (rec, val, cand, pred) in enumerate(kept["outs"]):
            exact += int([int(i) for i in rec] == ids[u].tolist())
            overlap += len(set(int(i) for i in rec) & set(ids[u].tolist()))
            by_id = dict(zip(cand.tolist(), pred.tolist()))
            mine = np.array([by_id[int(i)] for i in ids[u]], dtype=np.float64)  # the CPU arm's score of each POI we list
            kth = float(val[-1])
            valid = valid and bool((mine >= kth - 1e-4 * abs(kth)).all())
            rel = max(rel, float(np.max(np.abs(s[u].astype(np.float64) - val) / np.maximum(np.abs(val), 1e-30))))
        out = {"users": n, "k": 50, "lists_identical": exact, "id_overlap": overlap / (50.0 * n),
               "valid_topk_of_oracle_scores_within_1e-4": valid, "max_rel_err_of_ranked_scores": rel,
               "against": "the CPU arm's lists (same weights and histories)"}
        # ---- float64 oracle on the GPU for the extra users: every candidate, condition-aware 1e-4, list validity ----------------
        if extra_users:
            sd64 = {k: v.to(dev) for k, v in kept["sd"].items()}
            coords_t = torch.from_numpy(kept["coords"]).to(dev)
            reg_t = torch.from_numpy(kept["region"]).to(dev)
            worst, ok_lists, ident = 0.0, 0, 0
            allc = torch.arange(N, device=dev)
            for j in range(extra_users):
                h = torch.from_numpy(more[j]).to(dev)
                sc = []
                for c0 in range(0, N, 8192):
                    t = allc[c0:c0 + 8192]
                    hh = h[None, :].expand(len(t), -1)
                    aux = (coords_t[t][:, None, :] - coords_t[hh]).abs().float()
                    sc.append(orc.attention_network(sd64, "region_distance", BETA, hh, t, reg_t[hh], reg_t[t], aux, dtype=torch.float64))
                ref = torch.sigmoid(torch.cat(sc))
                ref[h] = -1.0  # history items are not candidates
                top = torch.topk(ref, 50)
                mine_ids = torch.from_numpy(ids[n + j]).to(dev)
                mine_ref = ref[mine_ids]
                kth = float(top.values[-1])
                ok_lists += int(bool((mine_ref >= kth - 1e-4 * abs(kth)).all()))
                ident += int(torch.equal(top.indices, mine_ids))
                worst = max(worst, float(((torch.from_numpy(s[n + j]).to(dev).double() - mine_ref).abs() / mine_ref.abs().clamp_min(1e-30)).max()))
            out["float64_oracle"] = {"users": extra_users, "lists_valid_topk_within_1e-4": ok_lists, "lists_identical": ident,
                                     "max_rel_err_of_ranked_scores": worst,
                                     "against": "oracle restatement in float64, evaluated with its tensors on the GPU, all 40k candidates per user"}
        return out
    except Exception as e:  # noqa: BLE001
        return {"error": f"{type(e).__name__}: {e}"}


def run_reference(args, cfg, rank, world):
    if rank != 0:
        return
    n = max(1, args.cpu_users)
    t_all, vals = 0.0, []
    for s in range(args.steps):  # (the CPU arm warms up inside cpu_arm: one untimed user per step)
        v, dt, threads, kind = cpu_arm(cfg, n, seed=s)
        vals.append(v)
        t_all += dt
    value = float(np.mean(vals))
    line = {"impl": "reference", "metric": "fullrank_eval_users_per_sec", "value": value, "unit": "users/s",
            "pair_scores_per_sec": value * (cfg["pois"] - cfg["hist"]), "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000.0 * t_all / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.config}: {cfg['desc']}", "users_per_step": n, "topk": 50},
            "cpu_baseline": {"value": value, "unit": "users/s", "cores": threads, "kind": kind,
                             "sample": f"{n} users x {cfg['pois']} POIs per step, {args.steps} steps, {CPU_SAMPLE[kind]}"},
            "e2e": {"value": value, "unit": "users/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------------
# evaluation workloads
# ----------------------------------------------------------------------------------------------------------------------
def make_eval(cfg, dev, n_users, seed_hist=2):
    """Synthetic catalogue + random-init ("trained-like") weights of the named architecture + histories, identical on every rank."""
    import torch
    from poi_recommendation_models_b200 import model as M, synthetic
    N, D, hid = cfg["pois"], cfg["D"], cfg["hid"]
    coords, region, R = synthetic.make_catalog(N, seed=0)
    g = torch.Generator().manual_seed(1)
    torch.manual_seed(1)
    m = M.NAIS_region_distance_Embedding(N, D, hid, BETA, R, 1)
    with torch.no_grad():
        for name, p in m.named_parameters():
            if name.startswith("embed_"):
                p.copy_(torch.randn(p.shape, generator=g) * 0.3)
            elif name.endswith(".bias"):
                p.copy_(torch.randn(p.shape, generator=g) * 0.1)
    m = m.to(dev).eval()
    m.set_catalog(region=region, coords=coords)
    return m, synth_histories(n_users, N, cfg["hist"], seed=seed_hist)


def time_eval(m, hist_np, cfg, ups, steps, warmup, precision, rank, world, local, dev, lib, sample_clocks=False, e2e=True,
              parity_users=64, keep_last=False):
    """Device-resident timing (+ e2e through topk_host) of `steps` steps of `ups` users; returns a dict of raw results
    (`keep_last`: "last" = host copies of the (score, id) lists the last timed step returned)."""
    import torch
    import torch.distributed as dist
    from poi_recommendation_models_b200.distributed import ShardedRanker
    H, k = cfg["hist"], cfg["k"]
    n_batches = max(1, len(hist_np) // ups)
    ranker = ShardedRanker(m, rank, world)
    batches_dev, batches_host = [], []
    indptr = np.arange(0, (ups + 1) * H, H, dtype=np.int64)
    for b in range(n_batches):
        h = hist_np[b * ups:(b + 1) * ups]
        batches_dev.append(m.make_users(indptr, h.reshape(-1)))
        batches_host.append((torch.from_numpy(indptr).pin_memory(), torch.from_numpy(h.reshape(-1).copy()).pin_memory()))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for i in range(warmup):  # (the first call builds the ranking plan of this rank's range; every later step reuses it)
        ranker.topk(batches_dev[i % n_batches], k, precision=precision)
    barrier()
    sampler = ClockSampler(local) if sample_clocks else None
    if sampler:
        sampler.start()
    l0 = lib.nais_launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    barrier()
    for i in range(steps):
        flush.zero_()  # L2 flush between timed iterations (untimed)
        ev[i][0].record()
        out = ranker.topk(batches_dev[(warmup + i) % n_batches], k, precision=precision)
        ev[i][1].record()
    barrier()
    launches = int(lib.nais_launch_count() - l0)
    clocks = sampler.stop() if sampler else None
    t_local = torch.tensor([sum(a.elapsed_time(b) for a, b in ev)], dtype=torch.float64, device=dev)
    kern_ms = ranker.last_kernel_ms  # CUDA-event time of this rank's scoring call (pack + passes + item merge) of the last step
    if world > 1:
        dist.all_reduce(t_local, op=dist.ReduceOp.MAX)
    total_ms = float(t_local.item())
    res = {"ranker": ranker, "users_per_s": ups * steps / (total_ms / 1000.0), "ms_per_step": total_ms / steps, "kern_ms": kern_ms,
           "launches": launches, "clocks": clocks, "ups": ups, "last": (out[0].cpu(), out[1].cpu()) if keep_last else None}
    # ---- N > 1: rank 0 re-scores users of the last step alone, over the whole catalogue, and compares bit for bit ------------
    if world > 1 and parity_users:
        pn = {"users": 0, "identical": 0}
        if rank == 0:
            try:
                last = batches_dev[(warmup + steps - 1) % n_batches]
                n_chk = min(parity_users, ups)
                sub = last.slice(0, n_chk)
                solo = ShardedRanker(m, 0, 1)
                s1, i1 = solo.topk(sub, k, precision=precision)
                same = [bool(torch.equal(i1[u], out[1][u]) and torch.equal(s1[u], out[0][u])) for u in range(n_chk)]
                pn = {"users": n_chk, "identical": int(sum(same)), "k": k,
                      "what": f"lists of the {ranker.parallelism} step vs rank 0 alone over [0, {m.item_num}): ids and scores bit for bit"}
            except Exception as e:  # noqa: BLE001
                pn = {"error": f"{type(e).__name__}: {e}"}
        res["parity_n"] = pn
        barrier()
    # ---- end to end through the drop-in API: host CSR in, host top-k out ------------------------------------------------
    if e2e:
        for i in range(min(warmup, 2)):
            ranker.topk_host(*batches_host[i % n_batches], k, precision=precision)
        barrier()
        t0 = time.perf_counter()
        for i in range(steps):
            ranker.topk_host(*batches_host[(warmup + i) % n_batches], k, precision=precision)
        barrier()
        t_e2e = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
        res["e2e"] = {"value": ups * steps / float(t_e2e.item()), "unit": "users/s",
                      "h2d_bytes_per_step": int(batches_host[0][0].numel() * 8 + batches_host[0][1].numel() * 8),
                      "d2h_bytes_per_step": int(ups * k * (4 + 8))}
    del flush
    return res


def roofline_of(res, cfg, peaks, eff):
    """Tensor roofline of rank 0's scoring call: algorithmic FLOPs of its (user slice x catalogue range) / CUDA-event time."""
    ranker, ups = res["ranker"], res["ups"]
    D, hid, H, k = cfg["D"], cfg["hid"], cfg["hist"], cfg["k"]
    u0_, u1_, _ = ranker.user_range(ups)
    cells = (u1_ - u0_) * H * (ranker.hi - ranker.lo)
    F = flops_per_cell(D, hid)
    kern_ms = res["kern_ms"]
    ach = cells * F / (kern_ms / 1000.0) / 1e12 if kern_ms else None
    peak = peaks["tf_sust"]
    alg_bytes = (ranker.hi - ranker.lo) * (D // 2 * 4 + 4 + 8) + (u1_ - u0_) * H * (4 + D // 2 * 4 + 4 + 8) + (u1_ - u0_) * k * 8
    rl = {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": (ach / peak) if ach else None,
          "traffic": None, "kernel": ranker.kernel_name(eff), "kernel_ms": kern_ms, "flops_per_cell": F, "cells_per_launch": cells,
          "peak_source": f"{peaks['which']} bf16 sustained (MEASURED_PEAKS.json)",
          "hbm_frac": (alg_bytes / (kern_ms / 1000.0) / 1e9 / peaks["hbm"]) if kern_ms else None, "algorithmic_bytes": alg_bytes}
    if eff != "fp32" and kern_ms:
        # FLOPs the tensor pipe actually executes per step of 256 cells (128 candidates x 2 history items):
        # SPLIT 3 passes x (D/16 + 1 ext) MMAs of 128 x nrow x 16; MIX: 1 fp16 pass (incl. ONE ext MMA) + 2 e5m2 passes of D/32
        # K=32 MMAs, each occupying the pipe like an fp16 K=16 MMA (tests/umma_probe_f8.cu) -> fp16-equivalent pipe FLOPs
        nrow = max((2 * hid + 4 + 15) // 16 * 16, 2 * hid + 16)
        ks = D // 16 + 1
        per_step = {"tc_split": 3 * ks * 2 * 128 * nrow * 16, "tc_mix": (ks + 2 * (D // 32)) * 2 * 128 * nrow * 16,
                    "tc_fast": ks * 2 * 128 * nrow * 16 + 2 * ks * 2 * 128 * 16 * 16}[eff]
        issued = cells / 256 * per_step / (kern_ms / 1000.0) / 1e12
        rl.update({"issued_tflops": issued, "issued_frac": issued / peak,
                   "issued_note": "tensor-pipe FLOPs executed (fp16-equivalent issue slots) incl. split/correction passes, ext K-step and S/L rows"})
    for fn in ("r2_ncu_traffic.json", "r1_ncu_traffic.json"):
        tr = os.path.join(ROOT, "profiles", fn)
        if os.path.isfile(tr) and eff in ("tc_split", "tc_mix"):
            with open(tr) as f:
                t = json.load(f)
            t = t.get(eff, t if "dram_bytes_per_user" in t else None)  # one entry per precision mode
            if t:
                rl["traffic"] = t["dram_bytes_per_user"] * (u1_ - u0_) + t.get("dram_bytes_const", 0)
                rl["traffic_source"] = t["source"]
                break
    return rl


# ----------------------------------------------------------------------------------------------------------------------
# C3: BPR-style training step
# ----------------------------------------------------------------------------------------------------------------------
C3_SHAPE = (40000, 128, 64, 64, 4096)  # POIs, history, D, hid, triples


def c3_problem(dev, rank=0):
    """C3's seeded model (in train mode) and this rank's 2 x 4,096 (history row, target) pairs: positives first, then
    negatives.  Returns (model, hist, tgt, hreg, treg, ll, region count)."""
    import torch
    from poi_recommendation_models_b200 import model as M, synthetic
    N, H, D, hid, T = C3_SHAPE
    coords, region, R = synthetic.make_catalog(N, seed=0)
    torch.manual_seed(1)
    m = M.NAIS_region_distance_Embedding(N, D, hid, BETA, R, 1)
    with torch.no_grad():
        for name, p in m.named_parameters():
            if name.startswith("embed_"):
                p.normal_(0, 0.3)
    m = m.to(dev).train()
    hist_np = synth_histories(T, N, H, seed=3 + rank)
    rng = np.random.default_rng(4 + rank)
    pos = hist_np[np.arange(T), rng.integers(0, H, T)]
    neg = rng.integers(0, N, T)
    clash = (hist_np == neg[:, None]).any(1)
    neg[clash] = (neg[clash] + 1) % N
    hist = torch.from_numpy(np.concatenate([hist_np, hist_np])).to(dev)
    tgt = torch.from_numpy(np.concatenate([pos, neg])).to(dev)
    reg = torch.from_numpy(region).to(dev)
    c = torch.from_numpy(coords).to(dev)
    ll = (c[tgt][:, None, :] - c[hist]).abs().float().contiguous()
    return m, hist, tgt, reg[hist], reg[tgt], ll, R


def train_c3(args, dev, lib, peaks, rank, world, steps, warmup, full=False, dump_dir=None):
    """BASELINE config C3: BPR-style training forward + backward on (user, pos, neg) triples — 4,096 triples = 8,192
    (history row, target) pairs, history 128, D = hid = 64; every row has its own history, positives are in the history
    (live mask), negatives are not.  Step = pair forward (tcgen05), -log sigmoid(s+ - s-), hand-written backward of every
    parameter (tcgen05 tile kernel + sorted-segment embedding-row reduce).  Data parallel over triples with N > 1 (+ gradient
    all-reduce): weak scaling.  Returns the block for the JSON line; `dump_dir`: rank 0 writes the loss and the gradients of
    the last timed step of the step mode the block reports (`dump_outputs`)."""
    import torch
    import torch.distributed as dist
    from poi_recommendation_models_b200 import ops
    from poi_recommendation_models_b200.distributed import allreduce_gradients
    N, H, D, hid, T = C3_SHAPE
    m, hist, tgt, hreg, treg, ll, R = c3_problem(dev, rank)

    def step():
        m.zero_grad(set_to_none=True)
        s = m.attention_network(hist, tgt, hreg, treg, ll)
        loss = -torch.nn.functional.logsigmoid(s[:T] - s[T:]).mean()
        loss.backward()
        allreduce_gradients(m, world)
        return loss.detach()  # (a kept autograd graph would keep the AccumulateGrad nodes of the default stream alive: no capture)

    host_ms = [0.0]

    def timed(fn, n_w, n_s):
        for _ in range(n_w):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        l0 = lib.nais_launch_count()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        h0 = time.perf_counter()
        a.record()
        for _ in range(n_s):
            r = fn()
        b.record()
        host_ms[0] = (time.perf_counter() - h0) * 1e3 / n_s  # time the host needs to ENQUEUE a step (>= the device time: host-bound)
        torch.cuda.synchronize()
        t = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / n_s, int(lib.nais_launch_count() - l0) // n_s, r

    def outputs(loss_):  # what a step hands its caller, copied before the next step overwrites it
        if not dump_dir:
            return None
        return {"loss": loss_.detach().clone(),
                **{"grad." + n: p.grad.detach().clone() for n, p in m.named_parameters() if p.grad is not None}}

    ms, launches, loss = timed(step, warmup, steps)
    last = outputs(loss)
    step_host_ms = host_ms[0]
    eager_ms, mode = ms, "eager (one Python-level call chain per step)"
    # The eager step is ~60 launches and the host needs about as long to enqueue them as the device to run them (host_enqueue_ms_
    # per_step): whenever the host is the slower one the number measures the box's CPU.  The shapes are static, so the whole step —
    # zero_grad, forward, loss, backward incl. the library's forked streams, gradient all-reduce — is captured ONCE into a CUDA
    # graph and replayed: same kernels, same results, one launch per step.
    graph_loss = None
    try:
        ops.check_indices(sync=True)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        m.zero_grad(set_to_none=True)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            s_ = m.attention_network(hist, tgt, hreg, treg, ll)
            graph_loss = -torch.nn.functional.logsigmoid(s_[:T] - s_[T:]).mean()
            graph_loss.backward()
            allreduce_gradients(m, world)

        graph_loss = graph_loss.detach()

        def replay():
            graph.replay()
            return graph_loss

        g_ms, _, g_loss = timed(replay, warmup, steps)
        same = abs(float(g_loss.detach()) - float(loss.detach())) <= 1e-6 * abs(float(loss.detach()))
        if same:
            ms, loss, mode = g_ms, g_loss, "CUDA graph replay of the captured step (torch.cuda.graph), one launch per step"
            last = outputs(g_loss)
        else:
            mode = f"eager (graph replay gave another loss: {float(g_loss.detach())})"
    except Exception as e:  # capture is an optimisation of the measurement loop, never a requirement
        mode = f"eager (CUDA graph capture failed: {type(e).__name__}: {str(e)[:120]})"
        torch.cuda.synchronize()
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, last)
    cells = 2 * T * H
    F = flops_per_cell(D, hid)
    blk = {"metric": "bpr_train_triples_per_sec", "value": T * world / (ms / 1000.0), "unit": "triples/s", "ms_per_step": ms,
           "n_gpus": world, "scaling": "weak", "triples_per_gpu": T, "gpu_launches_per_step": launches, "loss": float(loss.detach()),
           "host_enqueue_ms_per_step": step_host_ms, "eager_ms_per_step": eager_ms, "step_mode": mode,
           "dtype": "f16x2-split fwd / bf16x2-split bwd, f32 accumulate (tcgen05); f32 reduces",
           "config": {"workload": "C3: 4096 (user,pos,neg) triples = 8192 rows, own history per row, H=128, D=hid=64, 40k POIs; fwd + BPR loss + bwd of every parameter",
                      "parallelism": "single GPU" if world == 1 else f"data parallel x{world}, dense gradient all-reduce (one flat bucket)",
                      "api": "model.attention_network + loss.backward() (torch.autograd.Function over the C ABI)"}}
    # component times (untimed region; events around the raw ops): forward, backward, backward without the embedding tables
    with torch.no_grad():
        P = m._params()
        dsc = torch.randn(2 * T, device=dev) / T
        s_, rs_, pt_, am_ = ops.pairs_forward_raw(m.variant, BETA, P, hist, tgt, hreg, treg, ll)
        f_ms, _, _ = timed(lambda: ops.pairs_forward_raw(m.variant, BETA, P, hist, tgt, hreg, treg, ll), 2, max(3, steps))
        b_ms, _, _ = timed(lambda: ops.pairs_backward_raw(m.variant, BETA, P, hist, tgt, hreg, treg, ll, rs_, pt_, dsc, act_mask=am_), 2,
                           max(3, steps))
        bn_ms, _, _ = timed(lambda: ops.pairs_backward_raw(m.variant, BETA, P, hist, tgt, hreg, treg, ll, rs_, pt_, dsc, tables=False,
                                                           act_mask=am_), 2, max(3, steps))
    red_ms = max(b_ms - bn_ms, 1e-6)
    red_bytes = cells * D * 4 + (cells * 2 + 2 * T) * 8 * 2  # dq rows gathered once (both halves) + (key, source) lists read / written
    tf = cells * 4 * F / (ms / 1000.0) / 1e12  # fwd F + bwd ~3F (SURVEY.md §8d)
    blk["components_ms"] = {"forward": f_ms, "backward": b_ms, "backward_without_tables": bn_ms, "sort_and_segment_reduce": red_ms}
    blk["roofline"] = {"bound": "tensor", "achieved": tf, "peak": peaks["tf_sust"], "unit": "TFLOP/s", "frac": tf / peaks["tf_sust"],
                       "note": "algorithmic 4F per cell (fwd F + bwd 3F) over the whole step incl. loss, autograd glue and the embedding-row reduce",
                       "kernels_only_frac": cells * 4 * F / ((f_ms + bn_ms) / 1000.0) / 1e12 / peaks["tf_sust"],
                       "hbm_frac_of_segment_reduce": red_bytes / (red_ms / 1000.0) / 1e9 / peaks["hbm"],
                       "segment_reduce_bytes": red_bytes, "peak_source": f"{peaks['which']} (MEASURED_PEAKS.json)"}
    if full and world == 1:
        blk["full_step"] = full_step_block(args, dev, m, hist, tgt, hreg, treg, ll, R, T, N, H, D, hid)
    if full:
        blk["dp_1m"] = dp_large_catalogue_block(args, dev, rank, world, T, H, D, hid)
    return blk


def dp_large_catalogue_block(args, dev, rank, world, T, H, D, hid):
    """Data-parallel optimizer step at C4's catalogue (1M POIs: 2 x 128 MB embedding tables + 45 MB region table), 8192 rows per
    rank, BCE + Adagrad: dense gradients + ONE flat all-reduce (266 MB) + dense torch Adagrad, against the touched-row exchange
    (`distributed.SparseRowExchange`: row-compacted gradients, all-gather of (id, row) lists, row-sparse Adagrad on the union)."""
    import torch
    import torch.distributed as dist
    from poi_recommendation_models_b200 import model as M, synthetic
    from poi_recommendation_models_b200.distributed import SparseRowExchange, allreduce_gradients
    n_big = 1000000
    c2np, r2np, R2 = synthetic.make_catalog(n_big, seed=0)
    hn = synth_histories(T, n_big, H, seed=5 + rank)
    h2 = torch.from_numpy(np.concatenate([hn, hn])).to(dev)
    t2 = torch.from_numpy(np.concatenate([hn[:, 0], (hn[:, 1] + 1) % n_big])).to(dev)
    r2, c2 = torch.from_numpy(r2np).to(dev), torch.from_numpy(c2np).to(dev)
    ll2 = (c2[t2][:, None, :] - c2[h2]).abs().float().contiguous()
    hr2, tr2 = r2[h2], r2[t2]
    label = torch.cat([torch.ones(T), torch.zeros(T)]).to(dev)
    out = {"pois": n_big, "n_gpus": world,
           "shapes": {"c3_rows": "8192 rows per GPU, own history per row (H=128): ~1M cells touch a large part of the tables",
                      "multi_user_64": "64 users per GPU (H=128 each), 5 rows per positive, segmented layout: ~50k touched rows"}}
    # the realistic large-catalogue step: a multi-user batch touches thousands of rows, not hundreds of thousands
    from poi_recommendation_models_b200 import batches as PB
    import scipy.sparse as sp
    nu = 64
    hu = synth_histories(nu, n_big, H, seed=50 + rank)
    csr = sp.csr_matrix((np.ones(nu * H), hu.reshape(-1), np.arange(0, (nu + 1) * H, H)), shape=(nu, n_big))
    bt = PB.DeviceBatcher(csr, r2np, c2np, device=dev, seed=0)
    mb = bt.multi_user_batch(np.arange(nu), 4, seed=rank)
    for shape, kind in (("c3_rows", "dense_allreduce"), ("c3_rows", "sparse_row_exchange"), ("multi_user_64", "dense_allreduce"),
                        ("multi_user_64", "sparse_row_exchange")):
        torch.manual_seed(2)
        m2 = M.NAIS_region_distance_Embedding(n_big, D, hid, BETA, R2, 1).to(dev).train()
        opt = torch.optim.Adagrad(m2.parameters(), lr=0.01, weight_decay=0.0)
        ex = SparseRowExchange(m2, opt, world) if kind == "sparse_row_exchange" else None

        def one():
            if shape == "multi_user_64":
                if ex is not None:
                    return ex.step(mb.label, mb)
                opt.zero_grad()
                ls_ = m2.loss_func(torch.sigmoid(m2.segmented_scores(mb)), mb.label)
            else:
                if ex is not None:
                    return ex.step(label, h2, t2, hr2, tr2, ll2)
                opt.zero_grad()
                ls_ = m2.loss_func(m2(h2, t2, hr2, tr2, ll2), label)
            ls_.backward()
            allreduce_gradients(m2, world)
            opt.step()
            return ls_.detach()

        for _ in range(max(2, args.warmup)):
            one()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        a2, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a2.record()
        for _ in range(args.steps):
            ls = one()
        b2.record()
        torch.cuda.synchronize()
        t = torch.tensor([a2.elapsed_time(b2) / args.steps], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        rows_gpu = mb.B if shape == "multi_user_64" else 2 * T
        key = f"{shape}/{kind}"
        out[key] = {"ms_per_step": float(t.item()), "rows_per_s": rows_gpu * world / (float(t.item()) / 1000.0), "rows_per_gpu": rows_gpu,
                    "loss": float(ls)}
        if ex is not None:
            out[key]["bytes_received_per_step"] = int(ex.last_bytes)
        else:
            out[key]["bytes_allreduced_per_step"] = int(sum(p.numel() for p in m2.parameters()) * 4) if world > 1 else 0
        del m2, opt, ex
        torch.cuda.empty_cache()
    return out


def full_step_block(args, dev, m, hist, tgt, hreg, treg, ll, R, T, N, H, D, hid):
    """The whole reference step (run.py:248-254: zero_grad, forward, BCELoss, backward, Adagrad.step) on 8192 pairs: dense
    torch.optim.Adagrad over the [N, D/2] tables vs the row-sparse Adagrad fused into the segment reduce (f2), at C3's
    catalogue (40k POIs) and at C4's (1M POIs: 128 MB tables, where the dense step is HBM traffic)."""
    import torch
    from poi_recommendation_models_b200 import model as M, synthetic
    full = {"note": "8192 pairs, BCE, lr 0.01: whole optimizer step; the fused variant touches only the rows in the batch"}
    for n_big in (N, 1000000):
        if n_big == N:
            h2, t2, hr2, tr2, ll2, R2 = hist, tgt, hreg, treg, ll, R
        else:
            c2np, r2np, R2 = synthetic.make_catalog(n_big, seed=0)
            hn = synth_histories(T, n_big, H, seed=5)
            h2 = torch.from_numpy(np.concatenate([hn, hn])).to(dev)
            t2 = torch.from_numpy(np.concatenate([hn[:, 0], (hn[:, 1] + 1) % n_big])).to(dev)
            r2, c2 = torch.from_numpy(r2np).to(dev), torch.from_numpy(c2np).to(dev)
            ll2 = (c2[t2][:, None, :] - c2[h2]).abs().float().contiguous()
            hr2, tr2 = r2[h2], r2[t2]
        label = torch.cat([torch.ones(T), torch.zeros(T)]).to(dev)
        for kind in ("dense_adagrad", "fused_sparse_adagrad"):
            torch.manual_seed(2)
            m2 = M.NAIS_region_distance_Embedding(n_big, D, hid, BETA, R2, 1).to(dev).train()
            opt = torch.optim.Adagrad(m2.parameters(), lr=0.01, weight_decay=0.0)

            def full_step():
                if kind == "dense_adagrad":
                    opt.zero_grad()
                    ls_ = m2.loss_func(m2(h2, t2, hr2, tr2, ll2), label)
                    ls_.backward()
                    opt.step()
                    return ls_.detach()
                return m2.fused_adagrad_step(opt, label, h2, t2, hr2, tr2, ll2)

            for _ in range(args.warmup):
                full_step()
            torch.cuda.synchronize()
            a2, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a2.record()
            for _ in range(args.steps):
                ls = full_step()
            b2.record()
            torch.cuda.synchronize()
            full[f"{kind}_ms_N{n_big}"] = a2.elapsed_time(b2) / args.steps
            full[f"{kind}_loss_N{n_big}"] = float(ls)
            del m2, opt
    return full


def train_cpu_baseline(n_triples=32):
    """C3's step through the UNMODIFIED reference class on the host cores (autograd of model.py:246-297 + BPR loss), on a bounded
    sample of triples."""
    import torch
    from oracle import nais_oracle as orc  # CPU arm only
    from poi_recommendation_models_b200 import synthetic
    torch.set_num_threads(os.cpu_count())
    N, H, D, hid = 40000, 128, 64, 64
    coords, region, R = synthetic.make_catalog(N, seed=0)
    sd = orc.init_state("region_distance", N, D, hid, R, 1, seed=1, style="trained")
    m = orc.reference_model("region_distance", sd, BETA)
    if m is None:
        return None
    m.train()
    T = n_triples
    hist_np = synth_histories(T, N, H, seed=3)
    rng = np.random.default_rng(4)
    pos = hist_np[np.arange(T), rng.integers(0, H, T)]
    neg = (pos + 1 + rng.integers(0, N - 1, T)) % N
    hist = torch.from_numpy(np.concatenate([hist_np, hist_np]))
    tgt = torch.from_numpy(np.concatenate([pos, neg]))
    reg = torch.from_numpy(region)
    ll = torch.from_numpy(orc.latlon_abs_diff(coords, tgt.numpy(), hist.numpy()))

    def step():
        m.zero_grad(set_to_none=True)
        s = m.attention_network(hist, tgt, reg[hist], reg[tgt], ll)
        loss = -torch.nn.functional.logsigmoid(s[:T] - s[T:]).mean()
        loss.backward()

    step()
    t0 = time.perf_counter()
    n = 0
    while time.perf_counter() - t0 < 5.0 or n < 3:
        step()
        n += 1
    dt = time.perf_counter() - t0
    return {"value": n * T / dt, "unit": "triples/s", "cores": torch.get_num_threads(), "kind": "reference",
            "sample": f"{n} steps of {T} triples ({2 * T} rows, H={H}) in {dt:.1f} s: attention_network + BPR loss + autograd of the unmodified reference class, dense embedding gradients"}


def c1_block(dev, lib, no_cpu=False):
    """BASELINE configs[0] (C1): Foursquare-NYC-shaped 1,083 users x 38,333 POIs, D = hid = 64, history <= 100: ONE training epoch
    (BCE, 4 negatives per positive, Adagrad lr 0.01: run.py:227-255) + full-rank evaluation of every user (validation.py:62-131).
    The epoch is timed two ways: the reference's schedule — one user per optimizer step — on a 256-user sample, and multi-user
    steps (64 users per step, segmented layout, device sampler; loss = sum of the per-user mean BCE losses)."""
    import torch
    from poi_recommendation_models_b200 import batches as PB, eval_metrics as PM, model as M, ops, synthetic
    U, N, D, hid, num_ng, lr = 1083, 38333, 64, 64, 4, 0.01
    data = synthetic.make_checkins(U, N, seed=0, hist_len=None, max_hist=100, min_hist=5, median_hist=30)
    csr = data.train_csr()
    torch.manual_seed(0)
    order = np.random.default_rng(0).permutation(U)

    def fresh():
        torch.manual_seed(0)
        m_ = M.NAIS_region_distance_Embedding(N, D, hid, BETA, data.region_num, 1).to(dev).train()
        return m_, torch.optim.Adagrad(m_.parameters(), lr=lr, weight_decay=0.0)

    bt = PB.DeviceBatcher(csr, data.region, data.coords, device=dev, seed=0)
    blk = {"config": {"workload": "C1: 1083 users x 38333 POIs (synthetic Foursquare-NYC shape), D=hid=64, H<=100 (median 30), num_ng=4, Adagrad lr 0.01"}}
    # (a) the reference's schedule: one user per step (fused row-sparse Adagrad, batch built on the device)
    m1, o1 = fresh()
    sample = order[:256]
    def one_user(u):  # device sampler (one segment), then the whole optimizer step in one library call (nais_pairs_train_step)
        b_ = bt.multi_user_batch(np.array([u]), num_ng, seed=int(u))
        return m1.fused_adagrad_step(o1, b_.label, b_)

    for u in sample[:8]:  # warm-up
        one_user(int(u))
    m1.train_users(o1, bt, sample[:8], num_ng, seed=0)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for u in sample:
        one_user(int(u))
    torch.cuda.synchronize()
    dt_py = time.perf_counter() - t0
    # the same schedule with the user loop inside the library (nais_train_users): a whole epoch of one-user steps in one call
    l0 = lib.nais_launch_count()
    t0 = time.perf_counter()
    m1.train_users(o1, bt, order, num_ng, seed=1)
    torch.cuda.synchronize()
    dt1 = time.perf_counter() - t0
    blk["epoch_one_user_per_step"] = {"users_per_s": U / dt1, "epoch_s": dt1, "steps": int(U),
                                      "gpu_launches_per_step": int(lib.nais_launch_count() - l0) / U,
                                      "python_loop_users_per_s": len(sample) / dt_py,
                                      "note": "the reference's schedule (run.py:227-255), one user per optimizer step, all 1083 users: "
                                              "nais_train_users (per user: device sampler + forward, BCE, backward, Adagrad; the user loop "
                                              "runs inside the library); python_loop = the same steps driven from Python, 256 users"}
    del m1, o1
    # (b) multi-user steps: 64 users per optimizer step, segmented layout, device sampler
    m2, o2 = fresh()
    ups = 64

    def epoch(seed0):
        loss = None
        for i, s0 in enumerate(range(0, U, ups)):
            b = bt.multi_user_batch(order[s0:s0 + ups], num_ng, seed=seed0 + i)
            ro = b.host_row_offsets
            w = torch.from_numpy(np.repeat(1.0 / np.maximum(np.diff(ro), 1), np.diff(ro)).astype(np.float32)).to(dev, non_blocking=True)
            loss = m2.fused_adagrad_step(o2, b.label, b, row_weight=w)
        return loss

    epoch(0)  # warm-up epoch (also a second epoch of training: the timed one starts from those weights)
    torch.cuda.synchronize()
    l0 = lib.nais_launch_count()
    t0 = time.perf_counter()
    loss = epoch(1000)
    torch.cuda.synchronize()
    dt2 = time.perf_counter() - t0
    ops.check_indices(sync=True)
    cells = int(5 * (np.diff(csr.indptr).astype(np.int64) ** 2).sum())
    blk["epoch_multi_user"] = {"users_per_s": U / dt2, "epoch_s": dt2, "users_per_step": ups, "steps": (U + ups - 1) // ups,
                               "rows": int(5 * csr.nnz), "cells": cells, "gpu_launches": int(lib.nais_launch_count() - l0),
                               "loss_last_step": float(loss), "batch": "nais_sample_batch (device) + segmented NaisPairs: no [B,H] repeat, no [B,H,2] tensor",
                               "speedup_vs_one_user_per_step": (U / dt2) / (U / dt1)}
    # (c) full-rank evaluation of every user with the trained weights
    m2.eval()
    m2.set_catalog(region=data.region, coords=data.coords)
    users = m2.make_users(data.indptr, data.indices)
    m2.predict_topk(users, 50)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    _, ids = m2.predict_topk(users, 50)
    hits = ops.hits_at_k(ids, data.test_positive, [10])
    torch.cuda.synchronize()
    dt3 = time.perf_counter() - t0
    rec = ids.cpu().tolist()
    blk["eval"] = {"users_per_s": U / dt3, "eval_s": dt3, "topk": 50, "recall@10_test": PM.recall_at_k(data.test_positive, rec, 10),
                   "note": "one fused full-rank call for all 1083 users + nais_hits_at_k (weights after 2 synthetic epochs: metrics are not meaningful, parity is in tests/)"}
    if not no_cpu:
        from oracle import nais_oracle as orc  # CPU arm only
        sd = {k: v.detach().cpu() for k, v in m2.state_dict().items()}
        ref = orc.reference_model("region_distance", sd, BETA)
        if ref is not None:
            import random as _r
            ref.train()
            opt = torch.optim.Adagrad(ref.parameters(), lr=lr)
            _r.seed(0)
            n_cpu, t0 = 0, time.perf_counter()
            for u in order[:160]:  # ~10 s of host work
                hist = data.history(int(u))
                h_, t_, lab_, hr_, tr_ = orc.train_batch_region(hist.tolist(), N, num_ng, data.region, _r)
                ll_ = orc.latlon_abs_diff(data.coords, t_, h_)
                opt.zero_grad()
                pred = ref(torch.from_numpy(h_), torch.from_numpy(t_), torch.from_numpy(hr_), torch.from_numpy(tr_), torch.from_numpy(ll_))
                ref.loss_func(pred, torch.from_numpy(lab_)).backward()
                opt.step()
                n_cpu += 1
            dtc = time.perf_counter() - t0
            blk["cpu_baseline"] = {"value": n_cpu / dtc, "unit": "users/s (training)", "cores": torch.get_num_threads(), "kind": "reference",
                                   "sample": f"{n_cpu} user-steps of run.py:235-254 with the unmodified reference class + dense torch Adagrad on the host ({dtc:.1f} s); batch built by the oracle's restatement of batches.py:67-108"}
    return blk


def run_train(args, dev, lib, peaks, rank, world):
    blk = train_c3(args, dev, lib, peaks, rank, world, args.steps, args.warmup, full=True, dump_dir=args.dump_outputs)
    if rank == 0:
        line = {"metric": blk["metric"], "value": blk["value"], "unit": blk["unit"], "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": blk["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": blk["dtype"], "data": "synthetic", "config": blk["config"], "gpu_launches": blk["gpu_launches_per_step"] * args.steps,
                "loss": blk["loss"], "host_enqueue_ms_per_step": blk.get("host_enqueue_ms_per_step"), "eager_ms_per_step": blk.get("eager_ms_per_step"),
                "step_mode": blk.get("step_mode"), "components_ms": blk["components_ms"],
                "roofline": blk["roofline"], "full_step": blk.get("full_step"),
                "dp_1m": blk.get("dp_1m")}
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = train_cpu_baseline()
        print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C2", choices=list(WORKLOADS))
    ap.add_argument("--precision", default=os.environ.get("NAIS_BENCH_PRECISION", "tc_auto"),
                    choices=["fp32", "tc_auto", "tc_split", "tc_mix", "tc_fast", "tc_auto_onecta", "tc_mix_onecta", "tc_split_onecta"])
    ap.add_argument("--users-per-step", type=int, default=0)
    ap.add_argument("--mode", default="eval", choices=["eval", "train"], help="eval = headline full-rank metric; train = C3 BPR fwd+bwd (triples/s)")
    ap.add_argument("--cpu-users", type=int, default=4, help="users in the bounded CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-blocks", action="store_true", help="headline workload only: skip the value_exact / c4 / train_c3 blocks")
    ap.add_argument("--no-presort", action="store_true", help="train: keep the backward's id sorts inside the backward call (A/B of ops.PRESORT_IN_FORWARD)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy (impl ours)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    cfg = WORKLOADS[args.config]

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, cfg, rank, world)
        return

    import torch
    import torch.distributed as dist
    from poi_recommendation_models_b200 import _lib

    assert torch.cuda.is_available(), "bench.py (impl=ours) needs a CUDA device: there is no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    peaks = load_peaks()
    if args.no_presort:
        from poi_recommendation_models_b200 import ops as _ops
        _ops.PRESORT_IN_FORWARD = False
    if args.mode == "train":
        run_train(args, dev, lib, peaks, rank, world)
        if world > 1:
            dist.destroy_process_group()
        return

    U, N, H, D, hid, k = cfg["users"], cfg["pois"], cfg["hist"], cfg["D"], cfg["hid"], cfg["k"]
    ups = args.users_per_step or max(148, int({"fp32": 296, "tc_fast": 4736}.get(args.precision, 2368) * min(1.0, 40000 / N)))
    ups = min(ups, U)
    n_batches = min(args.steps + args.warmup, max(1, U // ups))
    m, hist_np = make_eval(cfg, dev, n_batches * ups)
    res = time_eval(m, hist_np, cfg, ups, args.steps, args.warmup, args.precision, rank, world, local, dev, lib, sample_clocks=True,
                    keep_last=bool(args.dump_outputs))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"scores": res["last"][0], "ids": res["last"][1]})
    prec_base = args.precision[:-7] if args.precision.endswith("_onecta") else args.precision  # "_onecta": one CTA per SM instead of CTA pairs, same math
    eff, choice = prec_base, None
    if prec_base == "tc_auto":  # the device-side gate picked MIX or SPLIT (no host sync inside the timed regions)
        plan = next(iter(m._plans.values()), None)
        choice = plan.tc_choice() if plan is not None else None
        eff = "tc_mix" if choice and choice["use_mix"] else "tc_split"
    ranker = res["ranker"]
    line = None
    if rank == 0:
        line = {"metric": "fullrank_eval_users_per_sec", "value": res["users_per_s"], "unit": "users/s",
                "pair_scores_per_sec": res["users_per_s"] * N, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": DTYPES[eff], "data": "synthetic",
                "config": {"workload": f"{args.config}: {cfg['desc']}", "users_per_step": ups, "precision": args.precision,
                           "precision_effective": eff, "tc_auto_gate": choice,
                           "plan": "nais_fullrank_prepare once per model (first warm-up step), reused by every step",
                           "l2": "flushed between timed steps (256 MiB write)", "weights": "random init, trained-like scale",
                           "parallelism": ranker.parallelism if world > 1 else "single GPU"},
                "clocks": res["clocks"], "gpu_launches": res["launches"], "e2e": res["e2e"],
                "roofline": roofline_of(res, cfg, peaks, eff)}
        if "parity_n" in res:
            line["parity_n"] = res["parity_n"]
    del res, ranker
    if not args.no_blocks and args.config == "C2":
        # ---- the fp32-grade path on the same workload ----------------------------------------------------------------------
        if prec_base == "tc_auto":
            r2 = time_eval(m, hist_np, cfg, ups, min(3, args.steps), 1, "tc_split", rank, world, local, dev, lib, e2e=False, parity_users=0)
            if rank == 0:
                line["value_exact"] = {"value": r2["users_per_s"], "unit": "users/s", "precision": "tc_split", "dtype": DTYPES["tc_split"],
                                       "ms_per_step": r2["ms_per_step"], "steps": min(3, args.steps),
                                       "roofline_frac": roofline_of(r2, cfg, peaks, "tc_split")["frac"]}
            del r2
        del m
        torch.cuda.empty_cache()
        # ---- C4: 1M POIs, POI-range shards x 1 (north_star), the same users at every N ------------------------------------
        c4 = WORKLOADS["C4"]
        c_steps, c_warm = min(3, args.steps), 1
        m4, h4 = make_eval(c4, dev, C4_USERS_PER_STEP * (c_steps + c_warm), seed_hist=12)
        r4 = time_eval(m4, h4, c4, C4_USERS_PER_STEP, c_steps, c_warm, args.precision, rank, world, local, dev, lib)
        if rank == 0:
            rk = r4["ranker"]
            plan4 = next(iter(m4._plans.values()), None)
            ch4 = plan4.tc_choice() if (plan4 is not None and prec_base == "tc_auto") else None
            eff4 = ("tc_mix" if ch4 and ch4["use_mix"] else "tc_split") if prec_base == "tc_auto" else prec_base
            line["c4"] = {"metric": "fullrank_eval_users_per_sec", "value": r4["users_per_s"], "unit": "users/s",
                          "pair_scores_per_sec": r4["users_per_s"] * c4["pois"], "ms_per_step": r4["ms_per_step"], "n_gpus": world,
                          "steps": c_steps, "warmup": c_warm, "scaling": "strong",
                          "config": {"workload": f"C4: {c4['desc']}", "users_per_step": C4_USERS_PER_STEP,
                                     "users": "the same 296-user batches at every N (subset of the 100k: per-user cost is constant)",
                                     "parallelism": f"{rk.gc} shards x {rk.gu}" + (": POI-range shards, one all-gather of packed keys + on-device merge" if world > 1 else " (single GPU)"),
                                     "precision_effective": eff4},
                          "e2e": r4.get("e2e"), "gpu_launches": r4["launches"], "roofline": roofline_of(r4, c4, peaks, eff4)}
            if "parity_n" in r4:
                line["c4"]["parity_n"] = r4["parity_n"]
        del r4, m4
        torch.cuda.empty_cache()
        # ---- C3: the training step ------------------------------------------------------------------------------------------
        t3 = train_c3(args, dev, lib, peaks, rank, world, max(10, args.steps), 3)
        if rank == 0:
            line["train_c3"] = t3
            if world == 1:
                try:
                    line["c1"] = c1_block(dev, lib, args.no_cpu_baseline)
                except Exception as e:  # noqa: BLE001  (the headline line stands)
                    line["c1"] = {"error": f"{type(e).__name__}: {e}"}
    if rank == 0:
        if not args.no_cpu_baseline and world == 1:
            kept = {}
            v, dt, threads, kind = cpu_arm(cfg, max(1, args.cpu_users), keep=kept)
            line["parity"] = parity_block(dev, cfg, kept, args.precision)
            line["cpu_baseline"] = {"value": v, "unit": "users/s", "cores": threads, "kind": kind,
                                    "sample": f"{args.cpu_users} users x {N} POIs (H={H}), {dt:.1f} s, {CPU_SAMPLE[kind]}"}
            if "train_c3" in line:
                line["train_c3"]["cpu_baseline"] = train_cpu_baseline()
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
