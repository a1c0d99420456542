#!/usr/bin/env python
"""What training a population against environments costs on top of its update: Population.step_async (behaviour policy
on pinned observations, actions published to pinned memory, stacked replay write from pinned rows, the iteration, the
log block published) against Population.iteration graph replays alone, alternating in one process.

    python tools/bench_population_step.py N n_envs [--wide 3xtf32|tf32|row] [--algo sac|td3] [--env hopper|humanoid]
                                          [--steps K] [--rounds R] [--out FILE.json]

(a) iteration: K graph replays of Population.iteration, host clock around them ending in a device synchronise;
(b) step: K steps of the loop a trainer runs — the host copies n_envs transitions and observations per agent into the
    pinned staging slot, step_async, wait_actions (the environments need them), wait for the previous step's log block
    (one step in flight) — host clock, ending in the last wait and a synchronise.
Both use a replay larger than the 126 MB L2 (at least 1 GB over all agents). The policy + action publish, the stacked
replay write and the log publish are also timed on their own: CUDA events around R replays of a graph holding only
those nodes. Prints one JSON record; --out appends it to a JSON list in FILE.
"""
import argparse
import json
import math
import statistics
import subprocess
import sys
import time
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from oracle import make_synthetic_transitions  # noqa: E402  (synthetic data only)
from sac_td3_cudagraphs_pytorch_b200 import _lib as L, sac_hps, td3_hps  # noqa: E402
from sac_td3_cudagraphs_pytorch_b200.population import Population  # noqa: E402

ENVS = {"hopper": (11, 3), "humanoid": (376, 17)}


def gpu_info() -> dict:
    """Name, power limit and max SM clock of the card (read-only query)."""
    try:
        line = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in line.split(",")]
    except Exception as e:  # (the numbers below still stand; say that the card could not be queried)
        name, power, clock = torch.cuda.get_device_name(), f"unknown ({e})", "unknown"
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def graph_ms(g: torch.cuda.CUDAGraph, reps: int) -> float:
    for _ in range(3):
        g.replay()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("N", type=int)
    ap.add_argument("n_envs", type=int)
    ap.add_argument("--wide", default="3xtf32", choices=["3xtf32", "tf32", "row"])
    ap.add_argument("--algo", default="sac", choices=["sac", "td3"])
    ap.add_argument("--env", default="hopper", choices=list(ENVS))
    ap.add_argument("--steps", type=int, default=0, help="steps per timed window (default: 40 for N >= 256, else 200)")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_population_step needs a CUDA device")
    ob, ac = ENVS[a.env]
    N, n = a.N, a.n_envs
    K = a.steps or (40 if N >= 256 else 200)
    hps = sac_hps() if a.algo == "sac" else td3_hps()
    rs = (2 * ob + ac + 2 + 3) & ~3
    rb_rows = min(20_000, max(2_000, math.ceil(1e9 / (N * rs * 4))))  # >= 1 GB of replay over all agents (L2: 126 MB)
    t0 = time.time()
    pop = Population(range(N), ob, ac, [-1.0] * ac, [1.0] * ac, hps, "cuda", seed=1, rb_capacity=rb_rows,
                     wide=None if a.wide == "row" else a.wide)
    pop.fill_replay(make_synthetic_transitions(rb_rows - 64, ob, ac, [-1.0] * ac, [1.0] * ac))
    t_init = time.time() - t0
    gen = torch.Generator().manual_seed(0)
    src_rows = [torch.randn(N, n, rs, generator=gen) for _ in range(2)]
    src_obs = [torch.randn(N, n, ob, generator=gen) for _ in range(2)]

    def iterations(k):
        t = time.perf_counter()
        for _ in range(k):
            pop.iteration()
        torch.cuda.synchronize()
        return (time.perf_counter() - t) / k * 1e3

    def steps(k):
        acc, prev = 0.0, None
        t = time.perf_counter()
        for j in range(k):
            pop.host_rows(n).copy_(src_rows[j & 1])
            pop.host_obs(n).copy_(src_obs[j & 1])
            tk = pop.step_async(None, n, n_obs=n)
            acc += float(pop.wait_actions()[0, 0, 0])  # the environments step on these
            if prev is not None:
                acc += float(pop.wait(prev, as_numpy=True)[0, L.OUT_QF_LOSS])
            prev = tk
        acc += float(pop.wait(prev, as_numpy=True)[0, L.OUT_QF_LOSS])
        torch.cuda.synchronize()
        assert math.isfinite(acc)
        return (time.perf_counter() - t) / k * 1e3

    for _ in range(2):  # capture and warm every graph variant
        iterations(6)
        steps(6)
    it_ms, st_ms = [], []
    for _ in range(a.rounds):  # alternating: both see the same machine state
        it_ms.append(iterations(K))
        st_ms.append(steps(K))

    # the step's own nodes, each in a graph of its own (own publish buffers: the step's sequence numbers stay untouched)
    lib = pop._lib
    obs_h = src_obs[0].pin_memory()
    rows_h = src_rows[0].pin_memory()
    blocks = (N * n * ac + 7) // 8
    d_act = torch.zeros(blocks * 8, device="cuda")
    h_act = torch.zeros(blocks * 8).pin_memory()
    h_out = torch.zeros(N * 8).pin_memory()
    seq_d = torch.zeros(2, dtype=torch.int64, device="cuda")
    seq_h = torch.zeros(2, dtype=torch.int64).pin_memory()
    g_pol, g_ext, g_pub = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
    torch.cuda.synchronize()
    with torch.cuda.graph(g_pol):
        pop._launch_predict(pop.args, obs_h.data_ptr(), n, True, 2 ** 64 - 1, d_act.data_ptr())
        L.check(lib.b2rl_publish_logs(d_act.data_ptr(), blocks, h_act.data_ptr(), seq_d[0].data_ptr(), seq_h[0].data_ptr(),
                                      torch.cuda.current_stream().cuda_stream), "publish actions")
    with torch.cuda.graph(g_ext):
        pop._launch_extend(rows_h.data_ptr(), n)
    with torch.cuda.graph(g_pub):
        L.check(lib.b2rl_publish_logs(pop.out.data_ptr(), N, h_out.data_ptr(), seq_d[1].data_ptr(), seq_h[1].data_ptr(),
                                      torch.cuda.current_stream().cuda_stream), "publish logs")
    reps = 200
    pol_ms, ext_ms, pub_ms = graph_ms(g_pol, reps), graph_ms(g_ext, reps), graph_ms(g_pub, reps)

    it, stp = statistics.median(it_ms), statistics.median(st_ms)
    rec = {
        **gpu_info(), "N": N, "n_envs": n, "algo": a.algo, "env": a.env, "path": a.wide, "batch": pop.B,
        "replay_rows_per_agent": rb_rows, "replay_bytes": N * rb_rows * rs * 4, "steps_per_window": K, "rounds": a.rounds,
        "iteration_ms": round(it, 4), "step_ms": round(stp, 4),
        "added_ms": round(stp - it, 4), "added_pct": round(100.0 * (stp - it) / it, 2),
        "agent_env_steps_per_s": round(N * n / stp * 1e3), "agent_updates_per_s_step": round(N / stp * 1e3),
        "agent_updates_per_s_iteration": round(N / it * 1e3),
        "iteration_ms_rounds": [round(x, 4) for x in it_ms], "step_ms_rounds": [round(x, 4) for x in st_ms],
        "policy_plus_action_publish_ms": round(pol_ms, 4), "stacked_replay_write_ms": round(ext_ms, 4),
        "log_publish_ms": round(pub_ms, 4), "action_floats_published": blocks * 8, "log_floats_published": N * 8,
        "init_s": round(t_init, 1), "finite": bool(torch.isfinite(pop.out).all()),
    }
    print(json.dumps(rec), flush=True)
    if a.out:
        p = Path(a.out)
        recs = json.loads(p.read_text()) if p.exists() else []
        recs.append(rec)
        p.write_text(json.dumps(recs, indent=1) + "\n")


if __name__ == "__main__":
    main()
