#!/usr/bin/env python
"""What training the large-batch data-parallel learner against environments costs on top of its update:
DataParallelLearner.step_async (behaviour policy on pinned observations, actions published to pinned memory, replay
write from pinned rows, the iteration, the log block published) against DataParallelLearner.iteration graph replays
alone, alternating in one process, for each n_envs.

    python tools/bench_dp_step.py [--algo sac|td3] [--batch 65536] [--wide 3xtf32|tf32] [--policy row|wide]
                                  [--n-envs 256,1024,4096,16384] [--steps K] [--rounds R] [--out FILE.json]
    torchrun --nproc-per-node 2 tools/bench_dp_step.py ...   (one record per rank, all-reduces over NCCL)

(a) iteration: K graph replays of iteration(i), host clock around them ending in a device synchronise;
(b) step: K steps of the loop a trainer runs — the host copies n_envs transitions and observations into the pinned
    staging slot, step_async, wait_actions (the environments need them), wait for the previous step's log block (one step
    in flight) — host clock, ending in the last wait and a synchronise.
The replay holds 2 M transitions (224 MB for Hopper, more than the 126 MB L2). The step's own nodes are also timed on
their own — the row policy (b2rl_actor_predict) and the wide policy (copy + tc_first + tc_linear + b2rl_wide_actor_predict),
each with its action publish, the replay write and the log publish: CUDA events around R replays of a graph holding only
those nodes. Prints one JSON record per (algo, n_envs); --out appends them to a JSON list in FILE.
"""
import argparse
import ctypes as C
import json
import math
import os
import statistics
import sys
import time
from pathlib import Path

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from oracle import make_synthetic_transitions  # noqa: E402  (synthetic data only)
from sac_td3_cudagraphs_pytorch_b200 import _lib as L, sac_hps, td3_hps  # noqa: E402
from sac_td3_cudagraphs_pytorch_b200.agents.agent import Agent  # noqa: E402
from sac_td3_cudagraphs_pytorch_b200.dp import DataParallelLearner, GradComm  # noqa: E402
from sac_td3_cudagraphs_pytorch_b200.replay import ReplayBuffer, pack_rows  # noqa: E402
from sac_td3_cudagraphs_pytorch_b200.wide import WidePredictor  # noqa: E402
from tools.bench_population_step import gpu_info, graph_ms  # noqa: E402

OB, AC = 11, 3  # Hopper
RB_ROWS = 2_000_000


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--algo", default="sac,td3")
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--wide", default="3xtf32", choices=["3xtf32", "tf32"])
    ap.add_argument("--policy", default="row", choices=["wide", "row"])
    ap.add_argument("--n-envs", default="256,1024,4096,16384")
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_dp_step needs a CUDA device")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if world > 1:
        torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
        dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
    dev = torch.device("cuda", torch.cuda.current_device())
    info = gpu_info()
    recs = []
    for algo in a.algo.split(","):
        torch.manual_seed(0)
        hps = (sac_hps if algo == "sac" else td3_hps)(batch_size=a.batch)
        ag = Agent({"ob_shape": (OB,), "ac_shape": (AC,)}, np.full(AC, -1.0, np.float32), np.full(AC, 1.0, np.float32), dev, hps,
                   seed=1, agent_id=rank)
        rb = ReplayBuffer(RB_ROWS, dev, seed=2, agent_id=rank)
        block = pack_rows({k: v.to(dev) for k, v in make_synthetic_transitions(65536, OB, AC, [-1.0] * AC, [1.0] * AC,
                                                                               seed=3 + rank).items()}, ag.fmt)
        rb._ensure(OB, AC)
        for r0 in range(0, RB_ROWS - 65536 + 1, 65536):
            rb.extend_rows(block)
        dp = DataParallelLearner(ag, rb, a.batch, GradComm(), wide=a.wide, policy=a.policy)
        gen = torch.Generator().manual_seed(rank)
        for n in [int(x) for x in a.n_envs.split(",")]:
            src_rows = [pack_rows(make_synthetic_transitions(n, OB, AC, [-1.0] * AC, [1.0] * AC, seed=10 + j), ag.fmt) for j in range(2)]
            src_obs = [torch.randn(n, OB, generator=gen) for _ in range(2)]
            it_no = [0]

            def iterations(k):
                t = time.perf_counter()
                for _ in range(k):
                    dp.iteration(it_no[0])
                    it_no[0] += 1
                torch.cuda.synchronize()
                return (time.perf_counter() - t) / k * 1e3

            def steps(k):
                acc, prev = 0.0, None
                t = time.perf_counter()
                for j in range(k):
                    dp.host_rows(n).copy_(src_rows[j & 1])
                    dp.host_obs(n).copy_(src_obs[j & 1])
                    tk = dp.step_async(it_no[0], n, n)
                    it_no[0] += 1
                    acc += float(dp.wait_actions()[0, 0])  # the environments step on these
                    if prev is not None:
                        acc += float(dp.wait(prev, as_numpy=True)[L.OUT_QF_LOSS])
                    prev = tk
                acc += float(dp.wait(prev, as_numpy=True)[L.OUT_QF_LOSS])
                torch.cuda.synchronize()
                assert math.isfinite(acc)
                return (time.perf_counter() - t) / k * 1e3

            for _ in range(2):  # capture and warm every graph variant
                iterations(2 * (int(hps.actor_update_delay) + 1))
                steps(4 * (int(hps.actor_update_delay) + 1))
            it_ms, st_ms = [], []
            for _ in range(a.rounds):  # alternating: both see the same machine state
                it_ms.append(iterations(a.steps))
                st_ms.append(steps(a.steps))

            # the step's own nodes, each in a graph of its own (own publish buffers: the step's sequence numbers stay untouched)
            lib, st = ag._lib, lambda: torch.cuda.current_stream().cuda_stream
            obs_h, rows_h = src_obs[0].pin_memory(), src_rows[0].pin_memory()
            blocks = (n * AC + 7) // 8
            d_act = torch.zeros(blocks * 8, device=dev)
            h_act = torch.zeros(blocks * 8).pin_memory()
            h_out = torch.zeros(8).pin_memory()
            seq_d = torch.zeros(3, dtype=torch.int64, device=dev)
            seq_h = torch.zeros(3, dtype=torch.int64).pin_memory()
            store = rb.storage.clone()  # the replay write goes to a copy: the learner's replay and counters stay as they are
            ctr = ag.counters.clone()
            pa = L.UpdateArgs()
            pa.hp, pa.fmt, pa.actor = ag._hyper, ag.fmt, ag.layout.actor.c_struct()
            pa.arena, pa.region_stride, pa.agent_base = ag.arena.flat.data_ptr(), ag.layout.region, ag.agent_id
            pa.min_ac, pa.max_ac, pa.counters = ag.min_ac.data_ptr(), ag.max_ac.data_ptr(), ag.counters.data_ptr()
            wp = WidePredictor(ag, n, a.wide)

            def publish_actions():
                L.check(lib.b2rl_publish_logs(d_act.data_ptr(), blocks, h_act.data_ptr(), seq_d[0].data_ptr(), seq_h[0].data_ptr(),
                                              st()), "publish actions")

            graphs = {k: torch.cuda.CUDAGraph() for k in ("row", "wide", "extend", "publish")}
            torch.cuda.synchronize()
            with torch.cuda.graph(graphs["row"]):
                L.check(lib.b2rl_actor_predict(C.byref(pa), obs_h.data_ptr(), n, 1, float(hps.actor_noise_std) if ag.td3 else 0.0,
                                               C.c_uint64(2 ** 64 - 1), d_act.data_ptr(), st()), "actor_predict")
                publish_actions()
            with torch.cuda.graph(graphs["wide"]):
                wp.enqueue(obs_h.data_ptr(), True, d_act.data_ptr())
                publish_actions()
            with torch.cuda.graph(graphs["extend"]):
                L.check(lib.b2rl_replay_extend_dev(store.data_ptr(), rb.capacity, rb.fmt, rows_h.data_ptr(), n, ctr.data_ptr(), st()),
                        "replay_extend_dev")
            with torch.cuda.graph(graphs["publish"]):
                L.check(lib.b2rl_publish_logs(ag.out.data_ptr(), 1, h_out.data_ptr(), seq_d[1].data_ptr(), seq_h[1].data_ptr(), st()),
                        "publish logs")
            node_ms = {k: graph_ms(g, 200) for k, g in graphs.items()}
            del store

            it, stp = statistics.median(it_ms), statistics.median(st_ms)
            rec = {
                **info, "world": world, "rank": rank, "algo": algo, "env": "hopper", "batch": a.batch, "precision": a.wide,
                "step_policy": a.policy, "n_envs": n, "replay_rows": RB_ROWS, "replay_bytes": RB_ROWS * ag.fmt.row_stride * 4,
                "steps_per_window": a.steps, "rounds": a.rounds,
                "iteration_ms": round(it, 4), "step_ms": round(stp, 4),
                "added_ms": round(stp - it, 4), "added_pct": round(100.0 * (stp - it) / it, 2),
                "env_steps_per_s": round(n / stp * 1e3), "iteration_ms_rounds": [round(x, 4) for x in it_ms],
                "step_ms_rounds": [round(x, 4) for x in st_ms],
                "row_policy_plus_action_publish_ms": round(node_ms["row"], 4),
                "wide_policy_plus_action_publish_ms": round(node_ms["wide"], 4),
                "replay_write_ms": round(node_ms["extend"], 4), "log_publish_ms": round(node_ms["publish"], 4),
                "finite": bool(torch.isfinite(ag.out).all()),
            }
            print(json.dumps(rec), flush=True)
            recs.append(rec)
        del dp, rb, ag
        torch.cuda.empty_cache()
    if a.out:
        p = Path(a.out)
        p.parent.mkdir(parents=True, exist_ok=True)
        if world > 1:
            p = p.with_name(f"{p.stem}.rank{rank}{p.suffix}")
        old = json.loads(p.read_text()) if p.exists() else []
        p.write_text(json.dumps(old + recs, indent=1) + "\n")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
