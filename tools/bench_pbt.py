#!/usr/bin/env python
"""Cost of one population-based-training exploit round over a sharded population (Population.exploit_many).
    python tools/bench_pbt.py [--n 1024] [--pairs 256] [--rounds 5] [--backend nccl|gloo] [--out FILE]
    torchrun --nproc-per-node W tools/bench_pbt.py ...      (W ranks; --backend gloo lets W ranks share one GPU)
1 024 SAC Hopper agents on the 3xTF32 path, shard(n, W, rank) per rank. A round of 256 pairs: dst d for every d = 0 mod 4
(spread over every rank), src = (d + n/2 + 2) mod n — so no src is a dst, and at W > 1 every pair crosses ranks (src on rank
r + W/2). Reports per rank the bytes sent and received, the wall time of exploit_many from a barrier until this rank's
stream is synchronised (one warm-up round, then --rounds rounds: median and all), one iteration's time (CUDA events over
30 iterations) and the ratio, with the card's name and power limit read in the same run. One JSON line per rank."""
import argparse
import json
import os
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from oracle import make_synthetic_transitions  # noqa: E402  (synthetic data only)
from sac_td3_cudagraphs_pytorch_b200 import sac_hps  # noqa: E402
from sac_td3_cudagraphs_pytorch_b200.population import Population, plan_exploit, shard  # noqa: E402


def card() -> dict:
    q = subprocess.run(["nvidia-smi", f"--id={torch.cuda.current_device()}", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = ([x.strip() for x in q.stdout.strip().split(",")] + ["?"] * 3)[:3]
    return {"name": name or torch.cuda.get_device_name(), "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1024)
    ap.add_argument("--pairs", type=int, default=256)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--rb-rows", type=int, default=4000)
    ap.add_argument("--backend", default="nccl")
    ap.add_argument("--out", help="also append the JSON lines to this file")
    a = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    local = local % torch.cuda.device_count() if a.backend == "gloo" else local
    torch.cuda.set_device(local)
    if world > 1:
        if a.backend == "nccl":
            dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
        else:
            dist.init_process_group("gloo")
    n = a.n
    pairs = [(d, (d + n // 2 + 2) % n) for d in range(0, n, 4)][:a.pairs]
    ids = shard(n, world, rank)
    pop = Population(ids, 11, 3, [-1.0] * 3, [1.0] * 3, sac_hps(), "cuda", seed=1, rb_capacity=a.rb_rows, wide="3xtf32")
    pop.fill_replay(make_synthetic_transitions(a.rb_rows, 11, 3, [-1.0] * 3, [1.0] * 3))
    for _ in range(6):
        pop.iteration()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(30):
        pop.iteration()
    e1.record()
    torch.cuda.synchronize()
    it_ms = e0.elapsed_time(e1) / 30

    plan = plan_exploit(pairs, pop._ranks(None).owner, pop._ranks(None).rank)
    row = pop.arena.flat[0].numel() * 4
    aux = pop._aux([pop.base]).numel() * 4
    sent = len(plan.sends) * (row + aux)
    received = len(plan.recvs) * (row + aux)
    times = []
    for k in range(a.rounds + 1):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        pop.exploit_many(pairs)
        torch.cuda.synchronize()
        if k:
            times.append((time.perf_counter() - t0) * 1e3)
    if world > 1:
        dist.barrier()
    med = float(np.median(times))
    out = {"tool": "bench_pbt", "card": card(), "world": world, "rank": rank, "backend": a.backend if world > 1 else None,
           "n_agents": n, "local_agents": pop.N, "pairs": len(pairs), "local_copies": len(plan.copies),
           "sends": len(plan.sends), "recvs": len(plan.recvs), "bytes_sent": sent, "bytes_received": received,
           "exploit_ms_median": round(med, 3), "exploit_ms": [round(t, 3) for t in times], "iteration_ms": round(it_ms, 3),
           "exploit_over_iteration": round(med / it_ms, 3)}
    line = json.dumps(out)
    print(line, flush=True)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        with open(a.out, "a") as f:
            f.write(line + "\n")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
