"""Timing-perturbation stress of the hand-rolled synchronisation (st.async + mbarrier DSMEM exchanges and the split cluster
barrier of mlp_cluster.cuh, the mbarrier rings of the tcgen05 kernels, the last-CTA tickets): the update is specified to be
bitwise reproducible, so a data race shows up as a result that depends on timing. Each learner is run several times from
identical state while a second stream floods the GPU with a different amount of unrelated work (copies that thrash L2 and
matmuls that take SMs away, so clusters get scheduled in different orders and at different times); every run must give the
same bits. (compute-sanitizer's racecheck is not available on the GPU pool: profiles/r2_compute_sanitizer_refused.log.)"""
import pytest
import torch

from tests.golden.cases import CASES, case_inputs
from tests.helpers import make_agent

pytestmark = pytest.mark.gpu


def _run(name, noise_level, iters=9, engine="row", batch=None):
    from sac_td3_cudagraphs_pytorch_b200.engine import LearnerEngine
    from sac_td3_cudagraphs_pytorch_b200.replay import ReplayBuffer
    inp = case_inputs(CASES[name])
    ag = make_agent(inp, seed=11)
    rb = ReplayBuffer(2048, "cuda", seed=11)
    rb.extend({k: v.cuda() for k, v in inp["storage"].items()})
    side = torch.cuda.Stream()
    big_a, big_b = torch.empty(48 << 20, device="cuda"), torch.empty(48 << 20, device="cuda")  # 192 MB each: larger than L2
    ma = torch.randn(2048, 2048, device="cuda")
    if engine == "row":
        eng = LearnerEngine(ag, rb, batch_size=batch or inp["B"], use_graphs=True)
        step = eng.iteration
    else:
        from sac_td3_cudagraphs_pytorch_b200.dp import DataParallelLearner, GradComm
        dp = DataParallelLearner(ag, rb, 1024, GradComm(), wide="3xtf32", graphs=True)
        step = dp.iteration
    torch.cuda.synchronize()
    for i in range(iters):
        with torch.cuda.stream(side):
            for _ in range(noise_level):
                big_b.copy_(big_a)
                torch.mm(ma, ma)
        step(i)
    torch.cuda.synchronize()
    return ag.arena.flat.clone(), ag.out.clone(), ag.counters.clone()


@pytest.mark.parametrize("name,engine,batch", [pytest.param(n, e, None, id=f"{n}-{e}") for n, e in (
    ("td3_hopper", "row"), ("sac_hopper", "row"), ("sac_humanoid_b256", "row"), ("sac_hopper", "wide"), ("td3_hopper", "wide"))]
    + [pytest.param("sac_hopper", "row", 8192, id="sac_hopper-row-8192")])
def test_results_do_not_depend_on_timing(name, engine, batch):
    """batch 8 192 on the row path: the temperature step's last-cluster ticket (alpha_kernel) sees 1 024 arrivals, and its
    last cluster sums 1 024 partials (32 per lane)."""
    ref = _run(name, 0, engine=engine, batch=batch)
    assert torch.isfinite(ref[1]).all()
    for level in (1, 3, 6):
        got = _run(name, level, engine=engine, batch=batch)
        for a, b, what in zip(ref, got, ("arena", "log block", "counters")):
            assert torch.equal(a, b), f"{name}/{engine}: {what} differs under background load level {level}"
