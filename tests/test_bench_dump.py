"""bench.py --dump-outputs: what the timed path returned in its last step, as float32 / float64 .npy files, so that two builds
can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")
ENV = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}


def test_dump_outputs_writes_float_arrays_within_the_limit(tmp_path):
    d = tmp_path / "d"
    bench.dump_outputs(str(d), {"scores": torch.tensor([[2.5, 1.0]]), "ids": torch.tensor([[7, 3]], dtype=torch.int32),
                                "loss": np.float64(0.25)})
    s, i, loss = (np.load(d / f"{n}.npy") for n in ("scores", "ids", "loss"))
    assert s.dtype == np.float32 and i.dtype == np.float64 and loss.dtype == np.float64
    assert s.tolist() == [[2.5, 1.0]] and i.tolist() == [[7.0, 3.0]] and loss == 0.25
    with pytest.raises(RuntimeError, match="limit"):
        bench.dump_outputs(str(tmp_path / "big"), {"x": np.zeros(bench.DUMP_LIMIT_BYTES // 4 + 1, dtype=np.float32)})
    assert not (tmp_path / "big").exists()


def test_dump_outputs_is_refused_for_the_cpu_arm(tmp_path):
    r = subprocess.run([sys.executable, BENCH, "--impl", "reference", "--dump-outputs", str(tmp_path / "d")], capture_output=True,
                       text=True, env=ENV, timeout=300)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr and not (tmp_path / "d").exists()


def _bench(*args):
    out = subprocess.run([sys.executable, BENCH, *args], check=True, capture_output=True, text=True, env=ENV, timeout=900).stdout
    return json.loads(out.strip().splitlines()[-1])


@pytest.mark.gpu
def test_bench_dumps_the_lists_of_its_last_timed_step(tmp_path):
    """The tiny workload in four batches of 128 users, 2 warm-up + 4 timed steps: the steps score batches 2, 3, 0, 1, so the dump
    must hold batch 1's lists — those of no other batch — and they must be valid top-k lists of the float64 oracle's scores."""
    import nais_testutil as util
    from poi_recommendation_models_b200 import synthetic
    from poi_recommendation_models_b200.distributed import ShardedRanker
    d = tmp_path / "d"
    line = _bench("--config", "tiny", "--users-per-step", "128", "--steps", "4", "--warmup", "2", "--no-cpu-baseline",
                  "--dump-outputs", str(d))
    assert line["steps"] == 4 and line["config"]["users_per_step"] == 128
    s, i = np.load(d / "scores.npy"), np.load(d / "ids.npy")
    cfg = bench.WORKLOADS["tiny"]
    N, H, k = cfg["pois"], cfg["hist"], cfg["k"]
    assert s.dtype == np.float32 and i.dtype == np.float64 and s.shape == i.shape == (128, k)
    m, hist = bench.make_eval(cfg, torch.device("cuda", 0), 512)
    ranker, indptr = ShardedRanker(m, 0, 1), np.arange(0, 129 * H, H, dtype=np.int64)
    same = []
    for b in range(4):
        s_b, i_b = ranker.topk(m.make_users(indptr, hist[b * 128:(b + 1) * 128].reshape(-1)), k, precision=line["config"]["precision"])
        same.append(np.array_equal(s, s_b.cpu().numpy()) and np.array_equal(i, i_b.cpu().numpy().astype(np.float64)))
    assert same == [False, True, False, False]
    coords, region, _ = synthetic.make_catalog(N, seed=0)
    sd = {name: v.detach().cpu() for name, v in m.state_dict().items()}
    for u in range(4):
        h = hist[128 + u]
        cand = np.setdiff1d(np.arange(N), h)
        o_s, o_scale = util.oracle_user_scores(sd, "region_distance", bench.BETA, coords, region, h, cand)
        ids = i[u].astype(np.int64)
        util.lists_equal_outside_ties(ids, None, dict(zip(cand.tolist(), o_s.tolist())), k)
        at = np.searchsorted(cand, ids)
        assert util.cond_err(s[u], o_s[at], o_scale[at]) < util.TOL


@pytest.mark.gpu
def test_bench_train_dump_is_the_loss_and_gradients_of_the_c3_step(tmp_path):
    """`--mode train`: the dumped loss is the one the line reports, and it and every gradient match float64 autograd of the
    oracle on the same C3 pairs (per tensor: max |got - ref| <= 2e-4 max |ref|, as tests/test_gpu_backward.py)."""
    from oracle import nais_oracle as orc
    d = tmp_path / "t"
    line = _bench("--mode", "train", "--steps", "2", "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(d))
    loss = np.load(d / "loss.npy")
    assert loss.dtype == np.float32 and float(loss) == line["loss"]
    m, hist, tgt, hreg, treg, ll, _ = bench.c3_problem(torch.device("cuda", 0))
    T = bench.C3_SHAPE[4]
    sd = {name: v.detach() for name, v in m.state_dict().items()}
    s = orc.attention_network(sd, "region_distance", bench.BETA, hist, tgt, hreg, treg, ll, dtype=torch.float64)
    margin = s[:T] - s[T:]
    ref_loss = float(-torch.nn.functional.logsigmoid(margin).mean())
    dloss = -torch.sigmoid(-margin) / T  # d loss / d margin
    _, ref = orc.grads(sd, "region_distance", bench.BETA, hist, tgt, hreg, treg, ll, torch.cat([dloss, -dloss]))
    assert abs(float(loss) - ref_loss) <= 1e-5 * abs(ref_loss)
    for name, r in ref.items():
        r = r.cpu().numpy()
        f = d / f"grad.{name}.npy"
        if f.exists():
            got = np.load(f)
            assert got.dtype == np.float32 and got.shape == r.shape, name
        else:  # a parameter the step never reaches has no gradient
            got = np.zeros_like(r)
        assert np.abs(got - r).max() <= 2e-4 * np.abs(r).max() + 1e-12, (name, np.abs(got - r).max(), np.abs(r).max())
