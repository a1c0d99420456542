"""bench.py's config-4 / config-5 legs and the in-line torch CUDA-graph baseline, at toy sizes: the functions the driver's
bench run depends on are exercised by the GPU test tier too (a broken leg would otherwise only show up at round end)."""
import sys
from pathlib import Path

import pytest
import torch

pytestmark = pytest.mark.gpu
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))


def test_population_leg_runs_and_reports():
    import bench
    r = bench.run_population_leg(0, 1, "cuda:0", n_total=6, iters=3, rb_rows=1024)
    assert r["outputs_finite"] and r["agents_total"] == 6 and r["agents_this_rank"] == 6
    assert r["ms_per_iteration"] > 0 and r["agent_updates_per_s"] == pytest.approx(6 / r["ms_per_iteration"] * 1e3)
    assert 0 < r["hbm_floor_frac"] < 1 and r["scaling"] == "strong"
    w = bench.run_population_leg(0, 1, "cuda:0", n_total=3, iters=3, rb_rows=1024, weak=True)
    assert w["scaling"] == "weak" and w["agents_total"] == 3


def test_dp_leg_runs_and_reports():
    import bench
    r = bench.run_dp_leg(0, 1, "cuda:0", B=2048, rows=8192, iters=6)
    assert r["outputs_finite"] and r["graph_replay"] and r["allreduce_us"] is None
    assert r["transitions_per_s"] == pytest.approx(2048 / r["ms_per_iteration"] * 1e3)
    assert r["allreduce_bucket_bytes"] > 500_000


def test_torch_cudagraph_baseline_runs():
    import bench
    bench.WORKLOADS["_toy"] = ("sac", 11, 3, 1.0, 4096)
    try:
        r = bench.time_reference_cuda("_toy", steps=9, warmup=3, device="cuda")
    finally:
        del bench.WORKLOADS["_toy"]
    assert r["value"] > 0 and r["replay_rows"] == 4096 and not r["tf32"]
    assert r["kernels_per_graph"]["q"] is None or r["kernels_per_graph"]["q"] > 50  # ~130-230 torch kernels per update graph


@pytest.mark.parametrize("algo", ["td3", "sac"])
def test_dumped_outputs_repeat_for_the_same_steps(algo, tmp_path):
    """--dump-outputs: the same seeded run gives the same arrays bit for bit; one step more gives other ones."""
    import numpy as np

    import bench
    bench.WORKLOADS["_toy"] = (algo, 11, 3, 1.0, 4096)
    dumps = []
    try:
        for run, steps in enumerate((7, 7, 8)):
            eng = bench.build_learner("_toy", "cuda:0", seed=1000)[2]
            for i in range(steps):
                eng.iteration(i)
            torch.cuda.synchronize()
            bench.write_outputs(tmp_path / str(run), bench.timed_outputs(eng))
            dumps.append({p.stem: np.load(p) for p in (tmp_path / str(run)).glob("*.npy")})
    finally:
        del bench.WORKLOADS["_toy"]
    a, b, c = dumps
    assert {"loss.qf_loss", "loss.actor_loss", "batch.observations", "batch.index", "actor.fc_stack.fc_block_1.fc.weight",
            "qnet_target.fc_stack.fc_block_1.fc.weight"} <= a.keys()
    assert ("actor_target.fc_stack.fc_block_1.fc.weight" in a) == (algo == "td3") and ("log_alpha" in a) == (algo == "sac")
    assert a.keys() == b.keys() == c.keys()
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert all(np.array_equal(a[k], b[k]) for k in a)
    assert not np.array_equal(a["qnet.fc_stack.fc_block_1.fc.weight"], c["qnet.fc_stack.fc_block_1.fc.weight"])
