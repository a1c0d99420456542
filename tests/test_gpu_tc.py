"""tcgen05 (TF32) large-batch hidden layer vs torch: Linear -> LayerNorm -> ReLU (agents/nets.py:66-82).
Tolerance: TF32 products (10-bit mantissa, truncated operands) — a per-tensor bar of 3e-3 of the output scale; the
LayerNorm statistics and everything after the product are fp32. The element-wise bound derived from the truncation and the
fp32 accumulation (a few 1e-5 of the output scale at TF32) is test_gpu_tc_kernels.py's.
M = 65 536 (BASELINE.json config 5) runs the forward, first-layer and backward pipelines at full grid — 148 CTAs with four
tiles each, every ring slot and both TMEM buffers reused — with the same bounds as the small sizes: each output row (and
each per-tile column sum) is one K = 256 (or K = O) accumulation whatever M is, so unlike the weight gradient's
batch-long contraction there is no longer chain to allow for."""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("x3", [False, True])
@pytest.mark.parametrize("M,ln,relu", [(128, True, True), (1000, True, True), (4096, False, True), (300, True, False),
                                       (65536, True, True)])
def test_tc_linear_matches_torch(M, ln, relu, x3):
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    lib = L.load()
    L.init_device(torch.device("cuda"))
    g = torch.Generator(device="cuda").manual_seed(M)
    X = torch.randn(M, 256, device="cuda", generator=g)
    W = torch.randn(256, 256, device="cuda", generator=g) / 16.0
    b = torch.randn(256, device="cuda", generator=g) * 0.1
    gam = 1.0 + 0.1 * torch.randn(256, device="cuda", generator=g)
    bet = 0.1 * torch.randn(256, device="cuda", generator=g)
    H = torch.full((M, 256), float("nan"), device="cuda")
    XH = torch.full((M, 256), float("nan"), device="cuda")
    stat = torch.zeros(M, 2, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    Wlo = torch.empty_like(W)
    if x3:
        L.check(lib.b2rl_tc_split_lo(W.data_ptr(), Wlo.data_ptr(), W.numel(), None, st), "split")
    L.check(lib.b2rl_tc_linear(X.data_ptr(), 256, M, W.data_ptr(), Wlo.data_ptr() if x3 else None, b.data_ptr(), gam.data_ptr(),
                               bet.data_ptr(), int(ln),
                               int(relu), H.data_ptr(), XH.data_ptr(), stat.data_ptr(), None, st), "tc_linear")
    torch.cuda.synchronize()
    z = X.double() @ W.double().T + b.double()
    if ln:
        mu, var = z.mean(1, keepdim=True), z.var(1, unbiased=False, keepdim=True)
        xh = (z - mu) / torch.sqrt(var + 1e-5)
        y = xh * gam.double() + bet.double()
    else:
        xh, y = z, z
    want = torch.relu(y) if relu else y
    assert torch.isfinite(H).all() and torch.isfinite(XH).all()
    tol = 4e-6 if x3 else 3e-3  # 3xTF32: fp32-level; TF32: 10-bit mantissas
    scale = float(want.abs().max())
    eh, ex = float((H.double() - want).abs().max()) / scale, float((XH.double() - xh).abs().max()) / float(xh.abs().max())
    print(f"\nM={M} ln={ln} 3xTF32={x3}: max rel err H {eh:.2e}, x-hat {ex:.2e}")
    assert eh <= tol and ex <= tol
    if ln:
        assert float((stat[:, 0].double() - mu[:, 0]).abs().max()) <= tol * 4


@pytest.mark.parametrize("x3", [False, True])
@pytest.mark.parametrize("Bn,MA,lda,transpose", [(4096, 256, 256, True), (1000, 14, 28, False), (300, 6, 64, False),
                                                 (65536, 256, 256, True), (250, 393, 772, False)])
def test_tc_wgrad_matches_torch(Bn, MA, lda, transpose, x3):
    """C = A[:, :MA]^T . Bm on the tensor cores (MN-major operands, split over the batch) vs float64."""
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    lib = L.load()
    L.init_device(torch.device("cuda"))
    g = torch.Generator(device="cuda").manual_seed(Bn + MA)
    A = torch.randn(Bn, lda, device="cuda", generator=g)
    Bm = torch.randn(Bn, 256, device="cuda", generator=g)
    Cc = torch.full((MA, 256), float("nan"), device="cuda")
    Ct = torch.full((256, MA), float("nan"), device="cuda") if transpose else None
    scratch = torch.empty(lib.b2rl_tc_wgrad_scratch_floats(MA, Bn, 0), device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    L.check(lib.b2rl_tc_wgrad(A.data_ptr(), lda, lda, MA, Bm.data_ptr(), Bn, Cc.data_ptr(), L.ptr(Ct), scratch.data_ptr(), int(x3), None, None, st),
            "tc_wgrad")
    torch.cuda.synchronize()
    want = A[:, :MA].double().T @ Bm.double()
    err = float((Cc.double() - want).abs().max()) / float(want.abs().max())
    print(f"\nBn={Bn} MA={MA} 3xTF32={x3}: max rel err {err:.2e}")
    # (the 65 536-row contraction chains 384 fp32 accumulations per TMEM element: fp32-class, not 4e-6)
    assert err <= ((4e-6 if Bn <= 4096 else 2e-5) if x3 else 3e-3)
    if transpose:
        assert torch.equal(Ct, Cc.T.contiguous())


# ---- stacked agents (include/b2rl.h b2rl_stack_t): per-agent weights through rank-3 TMA maps ---------------------------------
@pytest.mark.parametrize("x3", [False, True])
@pytest.mark.parametrize("n_agents,M", [(3, 256), (5, 200), (2, 640), (4, 72)])
def test_tc_linear_stacked_agents_match_torch(n_agents, M, x3):
    """Agent g's rows [g*M, g*M + M) are multiplied by agent g's own matrix / bias / LayerNorm affine (param_stride apart,
    as in the population arena); ragged per-agent batches (200, 72: the tail of an agent's last tile is zero-filled by TMA,
    never read from the next agent's rows) and the single-learner entry give the same bits per agent."""
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    lib = L.load()
    L.init_device(torch.device("cuda"))
    g = torch.Generator(device="cuda").manual_seed(100 * n_agents + M)
    ps = 4 * 256 * 256 + 1024  # floats between agents' parameter blocks: [W | bias | gamma | beta | pad]
    P = torch.zeros(n_agents, ps, device="cuda")
    P[:, :65536] = torch.randn(n_agents, 65536, device="cuda", generator=g) / 16.0
    P[:, 65536:65792] = torch.randn(n_agents, 256, device="cuda", generator=g) * 0.1
    P[:, 65792:66048] = 1.0 + 0.1 * torch.randn(n_agents, 256, device="cuda", generator=g)
    P[:, 66048:66304] = 0.1 * torch.randn(n_agents, 256, device="cuda", generator=g)
    Plo = torch.zeros_like(P)
    X = torch.randn(n_agents * M, 256, device="cuda", generator=g)
    H = torch.full((n_agents * M, 256), float("nan"), device="cuda")
    XH = torch.full((n_agents * M, 256), float("nan"), device="cuda")
    stat = torch.zeros(n_agents * M, 2, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    stk = L.Stack(n_agents, 0, ps, ps, 0, 0, 0)
    base = P.data_ptr()
    if x3:
        L.check(lib.b2rl_tc_split_lo(base, Plo.data_ptr(), 65536, C.byref(stk), st), "split")
    L.check(lib.b2rl_tc_linear(X.data_ptr(), 256, M, base, Plo.data_ptr() if x3 else None, base + 4 * 65536, base + 4 * 65792,
                               base + 4 * 66048, 1, 1, H.data_ptr(), XH.data_ptr(), stat.data_ptr(), C.byref(stk), st), "tc_linear")
    # the same through the single-learner entry, agent by agent
    H1, XH1 = torch.empty(M, 256, device="cuda"), torch.empty(M, 256, device="cuda")
    st1 = torch.zeros(M, 2, device="cuda")
    tol = 4e-6 if x3 else 3e-3
    for a in range(n_agents):
        Xa = X[a * M:(a + 1) * M]
        pa = base + 4 * a * ps
        L.check(lib.b2rl_tc_linear(Xa.data_ptr(), 256, M, pa, (Plo.data_ptr() + 4 * a * ps) if x3 else None, pa + 4 * 65536,
                                   pa + 4 * 65792, pa + 4 * 66048, 1, 1, H1.data_ptr(), XH1.data_ptr(), st1.data_ptr(), None, st), "tc1")
        torch.cuda.synchronize()
        assert torch.equal(H[a * M:(a + 1) * M], H1) and torch.equal(XH[a * M:(a + 1) * M], XH1), f"agent {a}"
        assert torch.equal(stat[a * M:(a + 1) * M], st1)
        W = P[a, :65536].view(256, 256).double()
        z = Xa.double() @ W.T + P[a, 65536:65792].double()
        xh = (z - z.mean(1, keepdim=True)) / torch.sqrt(z.var(1, unbiased=False, keepdim=True) + 1e-5)
        want = torch.relu(xh * P[a, 65792:66048].double() + P[a, 66048:66304].double())
        assert float((H1.double() - want).abs().max()) / float(want.abs().max()) <= tol


@pytest.mark.parametrize("x3", [False, True])
@pytest.mark.parametrize("n_agents,Bn,MA,lda", [(3, 256, 256, 256), (4, 200, 14, 28), (2, 256, 1, 64), (2, 2500, 256, 256)])
def test_tc_wgrad_stacked_agents_match_torch(n_agents, Bn, MA, lda, x3):
    """Per-agent C_g = A_g[:, :MA]^T . B_g over the agent's own Bn rows, written into per-agent gradient tensors
    param_stride apart (+ the transposed shadow); the per-agent update counters advance by one."""
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    lib = L.load()
    L.init_device(torch.device("cuda"))
    g = torch.Generator(device="cuda").manual_seed(Bn + MA + n_agents)
    A = torch.randn(n_agents * Bn, lda, device="cuda", generator=g)
    Bm = torch.randn(n_agents * Bn, 256, device="cuda", generator=g)
    ps = 2 * 256 * 256 + 64
    G = torch.full((n_agents, ps), float("nan"), device="cuda")
    ctr = torch.zeros(n_agents, 8, dtype=torch.int64, device="cuda")
    transpose = MA == 256
    scratch = torch.empty(lib.b2rl_tc_wgrad_scratch_floats(MA, Bn, n_agents), device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    stk = L.Stack(n_agents, 0, ps, 0, 0, 8, 0)
    L.check(lib.b2rl_tc_wgrad(A.data_ptr(), lda, lda, MA, Bm.data_ptr(), Bn, G.data_ptr(), (G.data_ptr() + 4 * 65536) if transpose else None,
                              scratch.data_ptr(), int(x3), ctr.data_ptr() + 8 * 1, C.byref(stk), st), "tc_wgrad")
    torch.cuda.synchronize()
    assert ctr[:, 1].tolist() == [1] * n_agents and int(ctr.sum()) == n_agents
    for a in range(n_agents):
        want = A[a * Bn:(a + 1) * Bn, :MA].double().T @ Bm[a * Bn:(a + 1) * Bn].double()
        got = G[a, :MA * 256].view(MA, 256)
        err = float((got.double() - want).abs().max()) / float(want.abs().max())
        # (a 1024-row slice chains 128 fp32 accumulations per TMEM element: 7e-6 measured at Bn = 2500)
        assert err <= ((4e-6 if Bn <= 1024 else 1.5e-5) if x3 else 3e-3), (a, err)
        if transpose:
            assert torch.equal(G[a, 65536:2 * 65536].view(256, 256), got.T.contiguous())
    # a shard holding one agent gives the same bits (the split never depends on the number of agents)
    G1 = torch.full((1, ps), float("nan"), device="cuda")
    stk1 = L.Stack(1, 0, ps, 0, 0, 8, 0)
    a = n_agents - 1
    L.check(lib.b2rl_tc_wgrad(A[a * Bn:].data_ptr(), lda, lda, MA, Bm[a * Bn:].data_ptr(), Bn, G1.data_ptr(), None, scratch.data_ptr(),
                              int(x3), None, C.byref(stk1), st), "tc_wgrad")
    torch.cuda.synchronize()
    assert torch.equal(G1[0, :MA * 256], G[a, :MA * 256])


@pytest.mark.parametrize("x3", [False, True])
@pytest.mark.parametrize("n_agents,M,K,ldx", [(1, 256, 14, 28), (3, 200, 14, 28), (1, 1000, 11, 16), (2, 256, 393, 396), (1, 128, 32, 32),
                                              (4, 72, 5, 8), (1, 65536, 14, 28)])
def test_tc_first_layer_matches_torch(n_agents, M, K, ldx, x3):
    """The first layer on the tensor cores (MODE 1): X [M][K] K-major, w1t [K][256] MN-major (the arena's forward layout),
    K not a multiple of 32 (tails zero-filled by TMA on both operands), stacked agents with their own weights, vs float64
    and vs the FFMA kernel b2rl_wide_first."""
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    lib = L.load()
    L.init_device(torch.device("cuda"))
    g = torch.Generator(device="cuda").manual_seed(7 * n_agents + M + K)
    ps = ((K * 256 + 3 * 256 + 3) // 4) * 4 + 64
    P = torch.zeros(n_agents, ps, device="cuda")
    P[:, :K * 256] = torch.randn(n_agents, K * 256, device="cuda", generator=g) / (K ** 0.5)
    ob, og, obe = K * 256, K * 256 + 256, K * 256 + 512
    P[:, ob:ob + 256] = torch.randn(n_agents, 256, device="cuda", generator=g) * 0.1
    P[:, og:og + 256] = 1.0 + 0.1 * torch.randn(n_agents, 256, device="cuda", generator=g)
    P[:, obe:obe + 256] = 0.1 * torch.randn(n_agents, 256, device="cuda", generator=g)
    X = torch.randn(n_agents * M, ldx, device="cuda", generator=g)
    st = torch.cuda.current_stream().cuda_stream
    stk = C.byref(L.Stack(n_agents, 0, ps, 0, 0, 0, 0)) if n_agents > 1 else None
    base = P.data_ptr()
    outs = []
    for fn in ("tc", "ffma"):
        H = torch.full((n_agents * M, 256), float("nan"), device="cuda")
        XH = torch.full((n_agents * M, 256), float("nan"), device="cuda")
        stat = torch.zeros(n_agents * M, 2, device="cuda")
        if fn == "tc":
            L.check(lib.b2rl_tc_first(X.data_ptr(), ldx, M, K, base, base + 4 * ob, base + 4 * og, base + 4 * obe, 1, H.data_ptr(),
                                      XH.data_ptr(), stat.data_ptr(), int(x3), stk, st), "tc_first")
        else:
            L.check(lib.b2rl_wide_first(X.data_ptr(), ldx, M, K, base, base + 4 * ob, base + 4 * og, base + 4 * obe, 1, H.data_ptr(),
                                        XH.data_ptr(), stat.data_ptr(), stk, st), "wide_first")
        torch.cuda.synchronize()
        outs.append((H, XH, stat))
    tol = 4e-6 if x3 else 3e-3
    for a in range(n_agents):
        W = P[a, :K * 256].view(K, 256).double()
        z = X[a * M:(a + 1) * M, :K].double() @ W + P[a, ob:ob + 256].double()
        mu, var = z.mean(1, keepdim=True), z.var(1, unbiased=False, keepdim=True)
        xh = (z - mu) / torch.sqrt(var + 1e-5)
        want = torch.relu(xh * P[a, og:og + 256].double() + P[a, obe:obe + 256].double())
        for (H, XH, stat), t in zip(outs, (tol, 2e-6)):
            sl = slice(a * M, (a + 1) * M)
            assert torch.isfinite(H[sl]).all()
            assert float((H[sl].double() - want).abs().max()) / float(want.abs().max()) <= t
            assert float((XH[sl].double() - xh).abs().max()) / float(xh.abs().max()) <= t
            assert float((stat[sl, 0].double() - mu[:, 0]).abs().max()) <= 4 * t * max(1.0, float(mu.abs().max()))


def _bwd_reference(DZ2, W2t, XH, rstd, gam, bet, ln):
    """float64 restatement of the dX product + ReLU mask + LayerNorm backward of layer 1 (agents/nets.py:66-82 differentiated):
    returns dz1 and the three column sums {sum dz, sum dn * x-hat, sum dn}."""
    dh = DZ2.double() @ W2t.double().T  # w2t [in][out]: dh[b][i] = sum_o dz2[b][o] * W2[o][i]
    x = XH.double()
    if ln:
        on = (x * gam.double() + bet.double()) > 0
        dn = torch.where(on, dh, torch.zeros_like(dh))
        dx = dn * gam.double()
        m1, m2 = dx.mean(1, keepdim=True), (dx * x).mean(1, keepdim=True)
        dz = rstd.double()[:, None] * (dx - m1 - x * m2)
    else:
        dn = torch.where(x > 0, dh, torch.zeros_like(dh))
        dz = dn
    return dz, torch.stack([dz.sum(0), (dn * x).sum(0), dn.sum(0)])


@pytest.mark.parametrize("x3", [False, True, "in-kernel"])  # in-kernel: W_lo == W, the weights' lo parts made in shared memory
@pytest.mark.parametrize("n_agents,M,ln", [(1, 1000, True), (1, 4096, True), (3, 200, True), (1, 300, False), (2, 72, True),
                                            (1, 65536, True)])
def test_tc_linear_bwd_matches_torch(n_agents, M, ln, x3):
    """b2rl_tc_linear_bwd against float64: dz1 and the per-tile column sums (ragged and stacked batches), and part = NULL
    (dX only, the actor step's pass through the critics) gives the same dz1 bit for bit."""
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    lib = L.load()
    L.init_device(torch.device("cuda"))
    g = torch.Generator(device="cuda").manual_seed(7 * n_agents + M)
    ps = 65536 + 1024  # [w2t | gamma | beta | pad] per agent
    P = torch.zeros(n_agents, ps, device="cuda")
    P[:, :65536] = torch.randn(n_agents, 65536, device="cuda", generator=g) / 16.0
    P[:, 65536:65792] = 1.0 + 0.1 * torch.randn(n_agents, 256, device="cuda", generator=g)
    P[:, 65792:66048] = 0.1 * torch.randn(n_agents, 256, device="cuda", generator=g)
    Plo = torch.zeros_like(P)
    R = n_agents * M
    DZ2 = torch.randn(R, 256, device="cuda", generator=g)
    XH = torch.randn(R, 256, device="cuda", generator=g)
    stat = torch.stack([torch.zeros(R, device="cuda"), 0.5 + torch.rand(R, device="cuda", generator=g)], 1).contiguous()
    n_tiles = (M + 127) // 128
    st = torch.cuda.current_stream().cuda_stream
    stk = L.Stack(n_agents, 0, ps, ps, 0, 0, 0)
    sp = C.byref(stk) if n_agents > 1 else None
    base = P.data_ptr()
    if x3 is True:
        L.check(lib.b2rl_tc_split_lo(base, Plo.data_ptr(), 65536, C.byref(stk), st), "split")
    lo_ptr = None if not x3 else (base if x3 == "in-kernel" else Plo.data_ptr())
    out = []
    for with_part in (True, False):
        DZ1 = torch.full((R, 256), float("nan"), device="cuda")
        part = torch.full((n_agents, n_tiles, 3, 256), float("nan"), device="cuda")
        L.check(lib.b2rl_tc_linear_bwd(DZ2.data_ptr(), M, base, lo_ptr, XH.data_ptr(), stat.data_ptr(),
                                       (base + 4 * 65536) if ln else None, (base + 4 * 65792) if ln else None, int(ln),
                                       DZ1.data_ptr(), part.data_ptr() if with_part else None, sp, st), "tc_linear_bwd")
        torch.cuda.synchronize()
        out.append((DZ1, part))
    (DZ1, part), (DZ1n, _) = out
    assert torch.isfinite(DZ1).all() and torch.equal(DZ1, DZ1n)
    tol = 6e-6 if x3 else 4e-3
    for a in range(n_agents):
        rows = slice(a * M, (a + 1) * M)
        dz, cs = _bwd_reference(DZ2[rows], P[a, :65536].view(256, 256), XH[rows], stat[rows, 1], P[a, 65536:65792],
                                P[a, 65792:66048], ln)
        e = float((DZ1[rows].double() - dz).abs().max()) / float(dz.abs().max())
        got = part[a].double().sum(0)
        nq = 3 if ln else 1  # (without LayerNorm only the bias gradient is defined)
        ec = float((got[:nq] - cs[:nq]).abs().max()) / float(cs[:nq].abs().max())
        print(f"\nagents={n_agents} M={M} ln={ln} 3xTF32={x3} agent {a}: dz1 {e:.2e}, column sums {ec:.2e}")
        assert e <= tol and ec <= tol


@pytest.mark.parametrize("M,n_out", [(1000, 1), (300, 6), (4096, 1)])
def test_wide_ln_bwd_matches_torch(M, n_out):
    """b2rl_wide_ln_bwd (head backward + ReLU mask + LayerNorm backward of layer 2) against float64, its column sums, the
    scalar head's weight gradient (dw3_part, n_out == 1), and part = NULL == the same dz."""
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    lib = L.load()
    L.init_device(torch.device("cuda"))
    g = torch.Generator(device="cuda").manual_seed(M + n_out)
    MO = L.MAX_OUT
    dz3 = torch.zeros(M, MO, device="cuda")
    dz3[:, :n_out] = torch.randn(M, n_out, device="cuda", generator=g)
    w3 = torch.randn(n_out, 256, device="cuda", generator=g) / 16.0
    XH = torch.randn(M, 256, device="cuda", generator=g)
    stat = torch.stack([torch.zeros(M, device="cuda"), 0.5 + torch.rand(M, device="cuda", generator=g)], 1).contiguous()
    gam = 1.0 + 0.1 * torch.randn(256, device="cuda", generator=g)
    bet = 0.1 * torch.randn(256, device="cuda", generator=g)
    P = (M + 127) // 128
    st = torch.cuda.current_stream().cuda_stream
    res = []
    for with_part in (True, False):
        dz = torch.full((M, 256), float("nan"), device="cuda")
        part = torch.full((P, 3, 256), float("nan"), device="cuda")
        dw3 = torch.full((P, 3, 256), float("nan"), device="cuda")
        L.check(lib.b2rl_wide_ln_bwd(dz3.data_ptr(), n_out, w3.data_ptr(), XH.data_ptr(), stat.data_ptr(), gam.data_ptr(),
                                     bet.data_ptr(), 1, M, dz.data_ptr(), part.data_ptr() if with_part else None,
                                     dw3.data_ptr() if (with_part and n_out == 1) else None, None, st), "wide_ln_bwd")
        torch.cuda.synchronize()
        res.append((dz, part, dw3))
    (dz, part, dw3), (dzn, _, _) = res
    assert torch.isfinite(dz).all() and torch.equal(dz, dzn)
    x = XH.double()
    dh = dz3[:, :n_out].double() @ w3.double()
    pre = x * gam.double() + bet.double()
    dn = torch.where(pre > 0, dh, torch.zeros_like(dh))
    dx = dn * gam.double()
    want = stat[:, 1].double()[:, None] * (dx - dx.mean(1, keepdim=True) - x * (dx * x).mean(1, keepdim=True))
    cs = torch.stack([want.sum(0), (dn * x).sum(0), dn.sum(0)])
    e = float((dz.double() - want).abs().max()) / float(want.abs().max())
    ec = float((part.double().sum(0) - cs).abs().max()) / float(cs.abs().max())
    print(f"\nM={M} n_out={n_out}: dz {e:.2e}, column sums {ec:.2e}")
    assert e <= 2e-6 and ec <= 2e-6
    if n_out == 1:
        w = (dz3[:, :1].double() * torch.relu(pre)).sum(0)
        assert float((dw3[:, 0].double().sum(0) - w).abs().max()) / float(w.abs().max()) <= 2e-6


def test_tc_kernels_are_reproducible_at_full_grid():
    """The 2-SM pipelines at a machine-filling size (65 536 rows: 148 CTAs, four tiles each, every ring slot and both TMEM
    buffers reused; cross-CTA mbarrier arrivals, TMA-fed and TMA-stored epilogues): 12 launches each of the 3xTF32 forward,
    backward and weight-gradient kernels, and of the plain-TF32 backward (the multicast pipeline, one CTA per MMA, whose
    epilogue runs ahead of it), from the same inputs must give the same bits — a race in the hand-rolled synchronisation
    would show up as a result that depends on timing. (The plain-TF32 backward once refilled an x-hat slot by TMA without
    ordering the lanes' reads of it first: a few rows per launch took the next chunk's x-hat into their LayerNorm sums.)"""
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    lib = L.load()
    L.init_device(torch.device("cuda"))
    g = torch.Generator(device="cuda").manual_seed(5)
    M = 65536
    X = torch.randn(M, 256, device="cuda", generator=g)
    DZ = torch.randn(M, 256, device="cuda", generator=g)
    W = torch.randn(256, 256, device="cuda", generator=g) / 16.0
    Wlo = torch.empty_like(W)
    b = 0.1 * torch.randn(256, device="cuda", generator=g)
    gam = 1.0 + 0.1 * torch.randn(256, device="cuda", generator=g)
    bet = 0.1 * torch.randn(256, device="cuda", generator=g)
    st = torch.cuda.current_stream().cuda_stream
    L.check(lib.b2rl_tc_split_lo(W.data_ptr(), Wlo.data_ptr(), W.numel(), None, st), "split")
    nt = (M + 127) // 128
    scratch = torch.empty(lib.b2rl_tc_wgrad_scratch_floats(256, M, 0), device="cuda")
    first = None
    for it in range(12):
        H, XH = torch.empty(M, 256, device="cuda"), torch.empty(M, 256, device="cuda")
        stat = torch.empty(M, 2, device="cuda")
        L.check(lib.b2rl_tc_linear(X.data_ptr(), 256, M, W.data_ptr(), Wlo.data_ptr(), b.data_ptr(), gam.data_ptr(), bet.data_ptr(),
                                   1, 1, H.data_ptr(), XH.data_ptr(), stat.data_ptr(), None, st), "tc_linear")
        DZ1, part = torch.empty(M, 256, device="cuda"), torch.empty(nt, 3, 256, device="cuda")
        L.check(lib.b2rl_tc_linear_bwd(DZ.data_ptr(), M, W.data_ptr(), Wlo.data_ptr(), XH.data_ptr(), stat.data_ptr(), gam.data_ptr(),
                                       bet.data_ptr(), 1, DZ1.data_ptr(), part.data_ptr(), None, st), "tc_linear_bwd")
        DZ1t = torch.empty(M, 256, device="cuda")
        L.check(lib.b2rl_tc_linear_bwd(DZ.data_ptr(), M, W.data_ptr(), None, XH.data_ptr(), stat.data_ptr(), gam.data_ptr(),
                                       bet.data_ptr(), 1, DZ1t.data_ptr(), None, None, st), "tc_linear_bwd (TF32)")
        G, Gt = torch.empty(256, 256, device="cuda"), torch.empty(256, 256, device="cuda")
        L.check(lib.b2rl_tc_wgrad(H.data_ptr(), 256, 256, 256, DZ1.data_ptr(), M, G.data_ptr(), Gt.data_ptr(), scratch.data_ptr(), 1,
                                  None, None, st), "tc_wgrad")
        torch.cuda.synchronize()
        cur = (H, XH, stat, DZ1, part, G, Gt, DZ1t)
        if first is None:
            first = cur
            assert all(torch.isfinite(t).all() for t in cur)
        else:
            for a, c, what in zip(first, cur, ("H", "x-hat", "stat", "dz1", "column sums", "dW", "dW^T", "dz1 (TF32)")):
                assert torch.equal(a, c), f"launch {it}: {what} differs from the first launch"
