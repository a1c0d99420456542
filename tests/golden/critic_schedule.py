"""What one critic step computes, recorded bit for bit (critic_schedule.npz), so that a change to the critic kernel's
schedule — which CTA computes which network pass, in which order — can be checked to leave every result unchanged.

    python -m tests.golden.critic_schedule       # on a GPU: (re)records tests/golden/critic_schedule.npz

For every golden case (RAGGED_CASES included): one critic step through the Agent API with the case's first batch and
noise — the TD target and the twin online Q values per row (dbg_targ_q, dbg_q), qf_loss, the critic gradients and the
workspace activations h1 / h2 / dz1 / dz2 of both critics. For ENGINE_CASES: three LearnerEngine.step calls, whose
critic step samples its batch in the kernel with the new rows folded in — the log blocks, the whole parameter arena
and the replay storage. The per-row vectors are stored as they are; every larger array as the sha256 of its bytes,
which keeps the file small and the comparison exact. Test infrastructure."""
from __future__ import annotations

import hashlib
from pathlib import Path

import numpy as np
import torch

from tests.golden.cases import CASES, RAGGED_CASES, case_inputs
from tests.helpers import batch_of, make_agent

NPZ = Path(__file__).resolve().parent / "critic_schedule.npz"
ALL_CASES = {**CASES, **RAGGED_CASES}
ENGINE_CASES = ("td3_hopper", "sac_hopper", "sac_humanoid")
HID = 256


def digest(t: torch.Tensor) -> np.ndarray:
    a = np.ascontiguousarray(t.detach().cpu().numpy())
    return np.frombuffer(hashlib.sha256(a.tobytes()).digest() + str((a.dtype.str, a.shape)).encode(), np.uint8)


def critic_step(name: str) -> dict[str, np.ndarray]:
    inp = case_inputs(ALL_CASES[name])
    B = inp["B"]
    ag = make_agent(inp)
    targ_q = torch.full((B,), float("nan"), device="cuda")
    q = torch.full((2 * B,), float("nan"), device="cuda")
    batch = {k: v.cuda() for k, v in batch_of(inp, 0).items()}
    out = ag.update_qnets(batch, eps=inp["eps_q"][0].cuda(), dbg_targ_q=targ_q, dbg_q=q)
    torch.cuda.synchronize()
    ws = ag.workspace(B)[: 8 * B * HID].view(4, 2, B, HID)  # [h1 h2 dz1 dz2][critic][row][unit]
    r = {"dbg_targ_q": targ_q.cpu().numpy(), "dbg_q": q.cpu().numpy(),
         "qf_loss": out["loss/qf_loss"].cpu().numpy().reshape(-1)}
    for i, what in enumerate(("h1", "h2", "dz1", "dz2")):
        r[f"#{what}"] = digest(ws[i])
    for n, p in ag.qnet_params.items():
        r[f"#grad/{n}"] = digest(p.grad)
    return r


def engine_steps(name: str, n_it: int = 3) -> dict[str, np.ndarray]:
    from sac_td3_cudagraphs_pytorch_b200.engine import LearnerEngine
    from sac_td3_cudagraphs_pytorch_b200.replay import ReplayBuffer
    inp = case_inputs(ALL_CASES[name])
    n0, cap, n_new = 200, 210, 4  # the third step's new rows wrap the cursor
    ag = make_agent(inp, seed=7)
    rb = ReplayBuffer(cap, "cuda", seed=7)
    rb.extend({k: v[:n0].cuda() for k, v in inp["storage"].items()})
    eng = LearnerEngine(ag, rb, use_graphs=True)
    g = torch.Generator().manual_seed(3)
    outs = []
    for i in range(n_it):
        eng.host_rows(n_new).copy_(torch.randn(n_new, rb.fmt.row_stride, generator=g))
        outs.append(eng.step(i, n_new).clone())
    torch.cuda.synchronize()
    return {"out": torch.stack(outs).cpu().numpy(), "#arena": digest(ag.arena.flat), "#storage": digest(rb.storage)}


def record_all() -> dict[str, np.ndarray]:
    r = {}
    for name in ALL_CASES:
        r.update({f"critic/{name}/{k}": v for k, v in critic_step(name).items()})
    for name in ENGINE_CASES:
        r.update({f"engine/{name}/{k}": v for k, v in engine_steps(name).items()})
    return r


if __name__ == "__main__":
    import sys
    path = Path(sys.argv[1]) if len(sys.argv) > 1 else NPZ
    np.savez_compressed(path, **record_all())
    print(f"wrote {path}")
