"""GPU tests for the replay sampler/gather (bit-exact), the whole-iteration engine (graph == eager ==
step-by-step API, bitwise) and size-independent properties at BASELINE.json's full sizes."""
import numpy as np
import pytest
import torch

from oracle import make_synthetic_transitions, philox_randint
from tests.golden.cases import case_inputs
from tests.helpers import make_agent

pytestmark = pytest.mark.gpu


def _rb(cap, td, seed=0):
    from sac_td3_cudagraphs_pytorch_b200.replay import ReplayBuffer
    rb = ReplayBuffer(cap, "cuda", seed=seed)
    rb.extend({k: v.cuda() for k, v in td.items()})
    return rb


@pytest.mark.parametrize("ob,ac", [(11, 3), (376, 17), (4, 1), (17, 6)])
def test_gather_is_bit_exact(ob, ac):
    n, B = 5000, 256
    td = make_synthetic_transitions(n, ob, ac, [-1.0] * ac, [1.0] * ac, seed=1234)
    rb = _rb(n, td)
    assert len(rb) == n
    idx = torch.randint(0, n, (B,), generator=torch.Generator().manual_seed(4321))
    batch = rb.sample(B, idx=idx)
    torch.cuda.synchronize()
    for k in ("observations", "next_observations", "actions", "rewards", "terminations", "dones"):
        want = td[k][idx]
        got = batch[k].cpu()
        assert got.dtype == want.dtype and got.shape == want.shape, k
        assert torch.equal(got, want), k  # storage[key][idx], torchrl LazyTensorStorage semantics
    assert torch.equal(batch["index"].cpu(), idx)
    again = rb.sample(B, idx=idx).rows.clone()  # idempotent
    assert torch.equal(again, batch.rows)


def test_device_sampler_matches_philox_twin():
    n, B, seed = 70001, 512, 0xDEADBEEF12345
    td = make_synthetic_transitions(n, 11, 3, [-1.0] * 3, [1.0] * 3)
    rb = _rb(n, td, seed=seed)
    for step in range(3):
        b = rb.sample(B)
        idx = b["index"].cpu()
        want = torch.from_numpy(philox_randint(seed, step, n, B))
        assert torch.equal(idx, want), f"draw {step}"  # integer Philox: bit-exact with the numpy twin
        assert torch.equal(b["observations"].cpu(), td["observations"][idx])
        assert 0 <= int(idx.min()) and int(idx.max()) < n
    assert int(rb.counters[3]) == 3


def test_extend_round_robin_wraps():
    td = make_synthetic_transitions(13, 5, 2, [-1.0, -1.0], [1.0, 1.0])
    from sac_td3_cudagraphs_pytorch_b200.replay import ReplayBuffer
    rb = ReplayBuffer(10, "cuda")
    first = {k: v[:7].cuda() for k, v in td.items()}
    second = {k: v[7:13].cuda() for k, v in td.items()}
    rb.extend(first)
    assert len(rb) == 7
    rb.extend(second)  # rows 7,8,9 then wraps onto 0,1,2
    assert len(rb) == 10
    got = rb.sample(10, idx=torch.arange(10))["observations"].cpu()
    want = torch.cat([td["observations"][10:13], td["observations"][3:10]])
    assert torch.equal(got, want)
    with pytest.raises(RuntimeError):
        ReplayBuffer(4, "cuda").sample(2)


def _arena_equal(a, b):
    return torch.equal(a.arena.flat, b.arena.flat) and torch.equal(a._alpha_state, b._alpha_state)


@pytest.mark.parametrize("name,batch", [pytest.param(n, None, id=n) for n in ("sac_hopper", "td3_hopper", "sac_clip_targfreq2")]
                         + [pytest.param("sac_hopper", 4097, id="sac_hopper-4097")])
def test_engine_graph_equals_eager_equals_api(name, batch):
    """batch 4 097: 513 rows per warp slice of the weight-gradient kernel (17 staged chunks), so wgrad_kernel<true> (the
    fused optimizer) is bitwise equal to wgrad_kernel<false> followed by Adam on the long form of every batch loop as well
    (test_gpu_row_kernels.py checks the plain kernel against float64 there)."""
    from sac_td3_cudagraphs_pytorch_b200.engine import LearnerEngine
    inp = case_inputs(name)
    td = inp["storage"]
    n_it = 7
    agents = [make_agent(inp, seed=99) for _ in range(3)]
    rbs = [_rb(td["observations"].shape[0], td, seed=99) for _ in range(3)]
    # the graph engine also takes the fused-optimizer path (Adam + Polyak inside the weight-gradient kernel),
    # the eager one the three-launch path: bitwise equality below covers b2rl_*_update_opt
    eng_graph = LearnerEngine(agents[0], rbs[0], batch_size=batch, use_graphs=True, fused_opt=True)
    eng_eager = LearnerEngine(agents[1], rbs[1], batch_size=batch, use_graphs=False, record_noise=True)
    api = agents[2]
    for i in range(n_it):
        eng_graph.iteration(i)
        eng_eager.iteration(i)
        # replay the same draws through the reference-shaped API (separate Polyak launch)
        torch.cuda.synchronize()
        rows = eng_eager.rows.clone()
        api.update_qnets(rows, eps=eng_eager.noise_q.clone())
        api.qnet_updates_so_far += 1
        if i % (inp["hps"]["actor_update_delay"] + 1) == 0:
            for j in range(inp["hps"]["actor_update_delay"]):
                api.update_actor(rows, eps=eng_eager.noise_pi[j].clone(), eps_alpha=eng_eager.noise_alpha[j].clone())
                api.actor_updates_so_far += 1
        api.update_targ_nets()
    torch.cuda.synchronize()
    assert _arena_equal(agents[0], agents[1]), "graph replay differs from eager launches"
    assert _arena_equal(agents[1], agents[2]), "fused-Polyak iteration differs from the step-by-step API"
    assert torch.equal(agents[0].counters[:3], agents[1].counters[:3])
    assert int(agents[0].counters[0]) == n_it
    assert agents[0].qnet_updates_so_far == n_it
    assert torch.isfinite(agents[0].out).all()


@pytest.mark.parametrize("name", ["sac_hopper", "td3_hopper"])
def test_engine_step_graph_equals_extend_plus_iteration(name):
    """LearnerEngine.step (H2D copy, device-cursor replay write, iteration, D2H copy in ONE graph) against the
    separate calls rb.extend_rows + iteration: bitwise-equal learner state and replay storage, wrap-around included."""
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    from sac_td3_cudagraphs_pytorch_b200.engine import LearnerEngine
    from sac_td3_cudagraphs_pytorch_b200.replay import ReplayBuffer
    inp = case_inputs(name)
    td = inp["storage"]
    n0, cap, n_new, n_it = 200, 230, 4, 12   # 200 rows + 12 x 4 new ones > 230: the cursor wraps
    agents = [make_agent(inp, seed=7) for _ in range(2)]
    rbs = []
    for _ in range(2):
        rb = ReplayBuffer(cap, "cuda", seed=7)
        rb.extend({k: v[:n0].cuda() for k, v in td.items()})
        rbs.append(rb)
    a_step, a_ref = LearnerEngine(agents[0], rbs[0], use_graphs=True), LearnerEngine(agents[1], rbs[1], use_graphs=True)
    g = torch.Generator().manual_seed(3)
    for i in range(n_it):
        rows = torch.randn(n_new, rbs[0].fmt.row_stride, generator=g)
        a_step.host_rows(n_new).copy_(rows)  # (two staging slots, alternating with the step's sequence number)
        out = a_step.step(i, n_new)
        rbs[1].extend_rows(rows.cuda())
        a_ref.iteration(i)
        torch.cuda.synchronize()
        assert torch.equal(out, agents[1].out.cpu()), f"log block differs at step {i}"
    assert _arena_equal(agents[0], agents[1])
    assert torch.equal(rbs[0].storage, rbs[1].storage)
    assert len(rbs[0]) == len(rbs[1]) == cap and rbs[0]._cursor == rbs[1]._cursor == (n0 + n_it * n_new) % cap
    assert int(agents[0].counters[L.CTR_SIZE]) == cap and int(agents[0].counters[L.CTR_CURSOR]) == rbs[0]._cursor
    assert int(agents[0].counters[L.CTR_XTICKET]) == 0


@pytest.mark.parametrize("name", ["td3_hopper", "sac_hopper", "sac_humanoid"])
def test_engine_in_kernel_sampling_equals_gather_launch(name):
    """The critic kernel sampling its own batch from the replay storage (engine default) = a gather launch in front of
    it: same indices, same batch rows, same parameters — bitwise — over iterations with and without actor updates;
    a batch size that leaves a ragged last row group included."""
    from sac_td3_cudagraphs_pytorch_b200.engine import LearnerEngine
    from sac_td3_cudagraphs_pytorch_b200.replay import ReplayBuffer
    inp = case_inputs(name)
    td = inp["storage"]
    for batch in (None, 28):
        agents = [make_agent(inp, seed=7) for _ in range(2)]
        rbs = []
        for _ in range(2):
            rb = ReplayBuffer(300, "cuda", seed=7)
            rb.extend({k: v[:250].cuda() for k, v in td.items()})
            rbs.append(rb)
        e_in = LearnerEngine(agents[0], rbs[0], batch_size=batch, use_graphs=True, fused_sample=True)
        e_ga = LearnerEngine(agents[1], rbs[1], batch_size=batch, use_graphs=True, fused_sample=False)
        for i in range(7):
            e_in.iteration(i)
            e_ga.iteration(i)
            torch.cuda.synchronize()
            assert torch.equal(e_in.idx, e_ga.idx), f"indices differ at iteration {i}"
            assert torch.equal(e_in.rows, e_ga.rows), f"batch rows differ at iteration {i}"
            assert torch.equal(agents[0].out, agents[1].out)
        assert _arena_equal(agents[0], agents[1])
        assert e_in.launches(0) == e_ga.launches(0) - 1


@pytest.mark.parametrize("name", ["td3_hopper", "sac_hopper"])
@pytest.mark.parametrize("explore", [False, True])
def test_engine_step_with_policy_in_the_graph(name, explore):
    """step_async(..., n_obs=) runs Agent.predict inside the step graph, on the parameters BEFORE the step's update
    (reference loop: predict, env step, extend, update), reading pinned observations and publishing pinned actions:
    equal, bitwise, to the eager predict of a twin agent at the same point, and the learner is unaffected."""
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    from sac_td3_cudagraphs_pytorch_b200.engine import LearnerEngine
    from sac_td3_cudagraphs_pytorch_b200.replay import ReplayBuffer
    inp = case_inputs(name)
    td = inp["storage"]
    n0, cap, n_new, n_obs, n_it = 200, 230, 4, 5, 8
    agents = [make_agent(inp, seed=7) for _ in range(2)]
    rbs = []
    for _ in range(2):
        rb = ReplayBuffer(cap, "cuda", seed=7)
        rb.extend({k: v[:n0].cuda() for k, v in td.items()})
        rbs.append(rb)
    e_pol, e_ref = LearnerEngine(agents[0], rbs[0], use_graphs=True), LearnerEngine(agents[1], rbs[1], use_graphs=True)
    g = torch.Generator().manual_seed(5)
    for i in range(n_it):
        rows = torch.randn(n_new, rbs[0].fmt.row_stride, generator=g)
        obs = torch.randn(n_obs, inp["ob"], generator=g)
        # the graph keys the exploration noise on the critic step counter, bit 31 set (host-counted draws stay below 2^31)
        draw = int(agents[1].counters[L.CTR_Q]) | 0x80000000
        want = agents[1].predict_device(obs, explore=explore, draw=draw).cpu().numpy()
        e_pol.host_rows(n_new).copy_(rows)
        e_pol.host_obs(n_obs).copy_(obs)
        tk = e_pol.step_async(i, n_new, n_obs=n_obs, explore=explore)
        got = e_pol.wait_actions().copy()
        out = e_pol.wait(tk).clone()
        e_ref.host_rows(n_new).copy_(rows)
        ref_out = e_ref.step(i, n_new)
        assert (got == want).all(), f"actions differ at step {i}"
        assert torch.equal(out, ref_out)
    torch.cuda.synchronize()
    assert _arena_equal(agents[0], agents[1])


@pytest.mark.parametrize("name", ["td3_hopper", "sac_hopper"])
def test_engine_pipelined_steps_equal_synchronous_steps(name):
    """step_async / wait with one step in flight (the host fills the other staging slot and launches step t before it
    reads step t - 1's log block) = the same steps run one at a time: every log block and the final state, bitwise."""
    from sac_td3_cudagraphs_pytorch_b200.engine import LearnerEngine
    from sac_td3_cudagraphs_pytorch_b200.replay import ReplayBuffer
    inp = case_inputs(name)
    td = inp["storage"]
    n0, cap, n_new, n_it = 200, 230, 4, 13
    agents = [make_agent(inp, seed=7) for _ in range(2)]
    rbs = []
    for _ in range(2):
        rb = ReplayBuffer(cap, "cuda", seed=7)
        rb.extend({k: v[:n0].cuda() for k, v in td.items()})
        rbs.append(rb)
    e_pipe, e_sync = LearnerEngine(agents[0], rbs[0], use_graphs=True), LearnerEngine(agents[1], rbs[1], use_graphs=True)
    g = torch.Generator().manual_seed(3)
    rows = [torch.randn(n_new, rbs[0].fmt.row_stride, generator=g) for _ in range(n_it)]
    want = []
    for i in range(n_it):
        e_sync.host_rows(n_new).copy_(rows[i])
        want.append(e_sync.step(i, n_new).clone())
    got, prev = [], None
    for i in range(n_it):
        e_pipe.host_rows(n_new).copy_(rows[i])
        t = e_pipe.step_async(i, n_new)
        if prev is not None:
            got.append(e_pipe.wait(prev).clone())
        prev = t
    got.append(e_pipe.wait(prev).clone())
    for i in range(n_it):
        assert torch.equal(got[i], want[i]), f"log block differs at step {i}"
    torch.cuda.synchronize()
    assert _arena_equal(agents[0], agents[1])
    assert torch.equal(rbs[0].storage, rbs[1].storage)


@pytest.mark.parametrize("algo,ob,ac,bound", [("sac", 11, 3, 1.0), ("td3", 11, 3, 1.0), ("sac", 376, 17, 0.4)])
def test_full_size_properties(algo, ob, ac, bound):
    """BASELINE.json sizes: batch 256, replay 1e6 (Hopper) / 2e5 (Humanoid, 618 MB), graphs on."""
    from sac_td3_cudagraphs_pytorch_b200 import sac_hps, td3_hps
    from sac_td3_cudagraphs_pytorch_b200.agents.agent import Agent
    from sac_td3_cudagraphs_pytorch_b200.engine import LearnerEngine
    hps = sac_hps() if algo == "sac" else td3_hps()
    cap = 1_000_000 if ob < 100 else 200_000
    td = make_synthetic_transitions(cap, ob, ac, [-bound] * ac, [bound] * ac, seed=1234)
    rb = _rb(cap, td, seed=5)
    torch.manual_seed(0)
    ag = Agent({"ob_shape": (4, ob), "ac_shape": (4, ac)}, np.full(ac, -bound, np.float32),
               np.full(ac, bound, np.float32), torch.device("cuda"), hps, rb=rb, seed=5)
    p0 = ag.arena.region(0).clone()
    eng = LearnerEngine(ag)
    n_it = 60
    qf = []
    for i in range(n_it):
        eng.iteration(i)
        if i % 10 == 9:
            qf.append(float(eng.logs()["loss/qf_loss"]))
    torch.cuda.synchronize()
    assert all(np.isfinite(qf)), qf
    assert torch.isfinite(ag.arena.flat).all()
    n_pi = 2 * ((n_it + 2) // 3)
    assert ag.counters[:3].tolist() == [n_it, n_pi, n_pi if algo == "sac" else 0]
    assert ag.qnet_updates_so_far == n_it and ag.actor_updates_so_far == n_pi
    # every online tensor moved; targets trail the online nets (Polyak) but moved too
    moved = (ag.arena.region(0) != p0)
    lay = ag.layout
    for net in (*lay.critic, lay.actor):
        for f in ("w1t", "w2t", "w3", "b1", "b2", "b3"):
            o = net.off[f]
            assert moved[o:o + net.numel(f)].any(), f
    t_gap = (ag.arena.region(1) - ag.arena.region(0))[lay.critic[0].begin:lay.critic[1].end].abs().max()
    assert 0 < float(t_gap) < 1.0
    # sampled indices stay inside the buffer and the gathered rows are the stored rows
    idx = eng.idx.cpu()
    assert 0 <= int(idx.min()) and int(idx.max()) < cap
    assert torch.equal(eng.last_batch()["observations"].cpu(), td["observations"][idx])
    # the fc2 shadow copies never drift from the primary weights
    for net, mod in ((lay.critic[0], ag.qnet1), (lay.critic[1], ag.qnet2), (lay.actor, ag.actor)):
        assert torch.equal(ag.arena.tensor(net, "w2n"), mod.fc_stack.fc_block_2.fc.weight.detach().contiguous())
    if algo == "sac":
        assert float(ag.alpha) > 0
    # drop-in inference policy: deterministic action within bounds
    a = ag.predict({"observations": td["observations"][:4]}, explore=False)
    assert a.shape == (4, ac) and np.all(np.abs(a) <= bound + 1e-6)


def test_errors_are_loud():
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L, sac_hps
    from sac_td3_cudagraphs_pytorch_b200.agents.agent import Agent
    with pytest.raises(L.B2rlError):
        Agent({"ob_shape": (11,), "ac_shape": (3,)}, np.full(3, -1.0, np.float32), np.full(3, 1.0, np.float32),
              torch.device("cpu"), sac_hps())
    inp = case_inputs("sac_hopper")
    ag = make_agent(inp)
    with pytest.raises(L.B2rlError, match=">= 1"):
        ag.update_qnets(torch.zeros(0, ag.fmt.row_stride, device="cuda"))


def test_bad_sampling_and_tensor_core_arguments_are_refused():
    """Error behaviour of the entry points added for in-kernel sampling / the folded replay write and of the tcgen05
    entry points: a negative return code with a message, nothing launched."""
    import ctypes as C
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    lib = L.load()
    inp = case_inputs("sac_hopper")
    ag = make_agent(inp)
    rows = torch.zeros(16, ag.fmt.row_stride, device="cuda")
    storage = torch.zeros(64, ag.fmt.row_stride, device="cuda")
    new = torch.zeros(4, ag.fmt.row_stride, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    # the replay write needs in-kernel sampling
    a = ag.update_args(rows)
    a.new_rows, a.n_new, a.capacity = new.data_ptr(), 4, 64
    assert lib.b2rl_critic_update_sac(C.byref(a), st) < 0 and b"storage" in lib.b2rl_last_error()
    # more new rows than the buffer holds
    a = ag.update_args(rows, storage=storage, new_rows=new, n_new=4)
    a.n_new = 100
    assert lib.b2rl_critic_update_sac(C.byref(a), st) < 0 and b"n_new" in lib.b2rl_last_error()
    # a misaligned replay storage
    a = ag.update_args(rows, storage=storage)
    a.storage = storage.data_ptr() + 4
    assert lib.b2rl_critic_update_sac(C.byref(a), st) < 0
    # tensor-core weight gradient: MA larger than the columns that exist / misaligned operand
    x = torch.zeros(256, 64, device="cuda")
    y = torch.zeros(256, 256, device="cuda")
    c = torch.zeros(64, 256, device="cuda")
    sc = torch.zeros(lib.b2rl_tc_wgrad_scratch_floats(64, 256, 0), device="cuda")
    assert lib.b2rl_tc_wgrad(x.data_ptr(), 64, 32, 64, y.data_ptr(), 256, c.data_ptr(), None, sc.data_ptr(), 0, None, None, st) < 0
    assert lib.b2rl_tc_wgrad(x.data_ptr() + 4, 64, 64, 64, y.data_ptr(), 256, c.data_ptr(), None, sc.data_ptr(), 0, None, None, st) < 0
    assert lib.b2rl_tc_wgrad_scratch_floats(0, 256, 0) < 0
    # fused critic head without a head
    assert lib.b2rl_tc_linear_q(y.data_ptr(), 256, 256, y.data_ptr(), None, y.data_ptr(), None, None, 0, None, None, None, None, None, st) < 0
    torch.cuda.synchronize()  # (nothing was launched: no sticky error)


@pytest.mark.parametrize("name", ["sac_hopper", "td3_hopper"])
def test_update_functions_can_be_wrapped_like_cudagraphmodule(name):
    """SURVEY §8(b): `update_*` must be wrappable by tensordict's CudaGraphModule (orchestrator.py:313-315) — warm-up calls
    run eagerly, then ONE call on a static six-key input dict is captured, and every later call copies the new batch
    into the static inputs and replays. Emulated with torch.cuda.CUDAGraph (tensordict is not in this image): the wrapped
    agent ends bitwise equal to an unwrapped twin fed the same batches, and the returned loss tensors are refreshed."""
    from tests.golden.cases import case_inputs
    from tests.helpers import batch_of, make_agent
    inp = case_inputs(name)
    wrapped, plain = make_agent(inp, seed=4), make_agent(inp, seed=4)
    dev = lambda d: {k: v.cuda() for k, v in d.items()}
    static = dev(batch_of(inp, 0))
    graphs, outs = {}, {}

    def call(fn_name, batch):
        for k in static:
            static[k].copy_(batch[k])                       # CudaGraphModule: tree-copy into the static inputs
        fn = getattr(wrapped, fn_name)
        n = call.count[fn_name] = call.count.get(fn_name, 0) + 1
        if n <= 2:                                          # warm-up calls
            return dict(fn(static))
        if fn_name not in graphs:
            g = torch.cuda.CUDAGraph()
            torch.cuda.synchronize()
            with torch.cuda.graph(g):
                outs[fn_name] = dict(fn(static))
            graphs[fn_name] = g
        graphs[fn_name].replay()
        return {k: v.clone() for k, v in outs[fn_name].items()}
    call.count = {}

    for i in range(6):
        b = dev(batch_of(inp, i))
        got = call("update_qnets", b)
        want = dict(plain.update_qnets(b))
        for a in (wrapped, plain):
            a.qnet_updates_so_far += 1
        assert torch.equal(got["loss/qf_loss"], want["loss/qf_loss"]), i
        for j in range(2):
            got = call("update_actor", b)
            want = dict(plain.update_actor(b))
            assert torch.equal(got["loss/actor_loss"], want["loss/actor_loss"]), (i, j)
        for a in (wrapped, plain):
            a.update_targ_nets()
    torch.cuda.synchronize()
    assert len(graphs) == 2
    assert torch.equal(wrapped.arena.flat[:, :4], plain.arena.flat[:, :4])
    assert torch.equal(wrapped.counters[:3], plain.counters[:3])
