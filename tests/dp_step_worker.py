"""torchrun worker for tests/test_gpu_dp_step.py: two NCCL ranks train from their own environments with
DataParallelLearner.step (policy, replay write, iteration with the all-reduces captured, log publish in one graph) against
the eager two-rank protocol on clones (row predict, rb.extend, iteration without graphs) fed the same rows."""
import os
import sys
from pathlib import Path

import torch
import torch.distributed as dist

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from tests.test_gpu_dp_step import _inputs, _learner, _row_predict, _state  # noqa: E402
from sac_td3_cudagraphs_pytorch_b200.dp import GradComm  # noqa: E402


def main():
    rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    dist.init_process_group("nccl", device_id=dev)
    world = dist.get_world_size()
    for kind, wide, policy in (("sac", "3xtf32", "wide"), ("td3", None, "row")):
        dp = _learner(kind, wide, policy, agent_id=rank, comm=GradComm())
        ref = _learner(kind, wide, "row", agent_id=rank, comm=GradComm(), graphs=False)
        assert dp.graphs and not ref.graphs
        T = 3 * (int(dp.agent.hps.actor_update_delay) + 1)
        for t in range(T):
            rows, _ = _inputs(t, 48, 0, dp.agent.fmt, salt=7919 * rank)  # this rank's transitions
            _, obs = _inputs(t, 0, 160, dp.agent.fmt)  # the same observations on every rank
            explore = t % 3 != 1
            dp.host_rows(48).copy_(rows)
            dp.host_obs(160).copy_(obs)
            logs = dp.step(t, 48, 160, explore).clone()
            acts = torch.from_numpy(dp.wait_actions().copy()).to(dev)
            want = _row_predict(ref.agent, obs.to(dev), int(explore))
            if policy == "row":
                assert torch.equal(acts, want), f"{kind} step {t}: actions differ from the eager predict"
            ref.rb.extend_rows(rows.to(dev))
            ref.iteration(t)
            torch.cuda.synchronize()
            assert torch.equal(logs, ref.agent.out.cpu()), f"{kind} step {t}: log block"
            # actions are keyed on the rank id: equal across ranks without exploration noise, different with it
            got = [torch.zeros_like(acts) for _ in range(world)]
            dist.all_gather(got, acts)
            if not explore:
                assert all(torch.equal(g, got[0]) for g in got), f"{kind} step {t}: exploit actions differ across ranks"
            if explore:
                assert not torch.equal(got[0], got[1]), f"{kind} step {t}: ranks explored with the same noise"
        a, b = _state(dp), _state(ref)
        for k in a:
            same = torch.equal(a[k], b[k]) if isinstance(a[k], torch.Tensor) else a[k] == b[k]
            assert same, f"{kind}: rank {rank} {k} differs from the eager protocol"
        arena = dp.agent.arena.flat[:, :4].contiguous()
        all_arenas = [torch.zeros_like(arena) for _ in range(world)]
        dist.all_gather(all_arenas, arena)
        assert all(torch.equal(x, all_arenas[0]) for x in all_arenas), f"{kind}: replicas diverged"
        if rank == 0:
            print(f"DP_STEP_RESULT {kind} wide={wide} policy={policy} world={world} steps={T} graphs={len(dp._step_graphs)}",
                  flush=True)
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("DP_STEP_OK", flush=True)


if __name__ == "__main__":
    main()
