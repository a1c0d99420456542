// critic.cu — fused critic step: next action -> twin target Q -> TD target -> twin online Q ->
// MSE -> backward (dX path), for 8 batch rows per 4-CTA CLUSTER. Replaces agents/agent.py:186-235
// (Agent.update_qnets up to qf_loss.backward()); the weight-gradient contraction over the batch
// is wgrad.cu, the optimizer step is adam.cu.
//
// Cluster rank = 2k + c: the twin critics are independent except for min(Q'_1, Q'_2) in the TD target, so
// group k (2 CTAs) takes critic k — target pass, online pass, backward — and CTA c of the group computes
// output columns [128c, 128c+128) of every layer (mlp_cluster.cuh). Both groups recompute the (cheap,
// identical) next-action pass; the two groups swap their 8 target Q values through distributed shared
// memory. Critical path: 4 network passes, each layer streaming 128 KB of weights per SM; 4 * B/8 = 128 CTAs.
#include "mlp_cluster.cuh"
#include "policy.cuh"
#include "rng.cuh"

namespace b2rl {

constexpr int MAX_A = MAX_OUT / 2;

struct CriticSmem {
  Work s;
  Acts a;                      // the online critic's pass (kept for its backward pass)
  NetStage nsA, nsT, nsQ;      // staged small tensors of the actor, of target critic k and of online critic k
  Net nA, nT, nQ;              // their descriptors
  float lo[MAX_A], hi[MAX_A], eps[RT][MAX_A];
  float rd[RT][2];             // (reward, done) of the 8 rows
  float logpi[RT], qn[2][RT], y[RT], dq[RT], sq[RT];  // per-row scalars
  // followed by two input tiles float4[RQ * (O + A)]: [next_obs | a'] and [obs | act], then CriticVals
};
// this agent's values (common.cuh agent_hp), behind the tiles so that the tiles keep their offset
struct CriticVals { float gamma, td3_std, td3_c, pad; };

__host__ __device__ inline size_t critic_smem_bytes(int in_dim) {
  return sizeof(CriticSmem) + (size_t)2 * RQ * in_dim * sizeof(float4) + sizeof(CriticVals);
}

template <bool WIDE>
__global__ void __launch_bounds__(NT, 1) critic_fused_kernel(const __grid_constant__ b2rl_update_args_t A) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  CriticSmem& M = *reinterpret_cast<CriticSmem*>(smem_raw);
  Work& S = M.s;
  exchange_init_arrive(S);  // (shared memory and the cluster barrier only: legal before the grid dependency)
  pdl_enter();
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const int k = rank >> 1;  // the critic this CTA's group owns
  const Group G{rank & 1, rank & ~1};
  const int t = threadIdx.x, w = t >> 5, l = t & 31;
  const int agent = blockIdx.y, rb = blockIdx.x >> 2, b0 = rb * RT;
  const int O = A.fmt.ob_dim, AD = A.fmt.ac_dim, rs = A.fmt.row_stride, B = A.batch;
  const int ldx = O + AD, nvalid = min(RT, B - b0);
  float4* XA = reinterpret_cast<float4*>(smem_raw + sizeof(CriticSmem));  // [next_obs | a']
  float4* XB = XA + RQ * ldx;                                             // [obs | act]
  CriticVals& V = *reinterpret_cast<CriticVals*>(XB + RQ * ldx);
  const uint32_t gid = (uint32_t)(A.agent_base + agent);  // global agent id: keys the Philox streams
  const bool td3 = A.hp.td3 != 0;

  const float* P = A.arena + (size_t)agent * A.arena_agent_stride;  // region 0: online
  const float* T = P + A.region_stride;                             // region 1: target
  const float* rows = A.rows + (size_t)agent * A.rows_agent_stride;
  const uint64_t step = A.counters[(size_t)agent * 8 + B2RL_CTR_Q];
  float* wsb = A.workspace + (size_t)agent * A.workspace_agent_stride;

  // ---- prologue: one asynchronous burst of both input tiles and every small tensor the kernel will touch. Each
  //      warp has its own job (the jobs are instruction-bound: side by side they cost the longest, not the sum).
  B2RL_TICK(0);
  B2RL_TICK(40);
  const Net &act = M.nA, &qt = M.nT, &qo = M.nQ;
  const float* PA = td3 ? T : P;  // SAC samples from the ONLINE actor (agent.py:205), TD3 uses the TARGET actor (:194-202)
  if (w == 0) {
    if (l < AD) {
      M.lo[l] = __ldg(A.min_ac + l);
      M.hi[l] = __ldg(A.max_ac + l);
    }
    if (l == 0) {
      V.gamma = agent_hp(A.agent_hp, agent, HP_GAMMA, A.hp.gamma);
      V.td3_std = agent_hp(A.agent_hp, agent, HP_TD3_STD, A.hp.td3_std);
      V.td3_c = agent_hp(A.agent_hp, agent, HP_TD3_C, A.hp.td3_c);
    }
    tile_noise<RT, MAX_A>(M.eps, A.eps, rank == 0 ? A.eps_out : nullptr, A.hp.seed, (int64_t)agent * B + b0, b0, nvalid, AD, step, gid,
                          STREAM_CRITIC_EPS, !td3 || A.hp.targ_smoothing, l);
  } else if (w == 1) {
    stage_net(PA, &A.actor, &M.nsA, &M.nA, G.c * CW);
  } else if (w == 2) {
    stage_net(T, &A.critic[k], &M.nsT, &M.nT, G.c * CW);
  } else if (w == 3) {
    stage_net(P, &A.critic[k], &M.nsQ, &M.nQ, G.c * CW);
  } else {
    // In-kernel sampling (A.storage): lane i draws the replay index of tile row i & 7 — the Philox key of
    // replay.cu::gather_kernel, so the batch is the one b2rl_replay_sample_gather would have gathered — and the tiles
    // are read straight from the replay storage; cluster rank 0 also writes the rows out for the kernels that follow.
    // With A.new_rows the replay write is folded in as well (include/b2rl.h): draw over the grown size, read a drawn
    // new row from new_rows itself; the spare CTA of the wgrad launch that follows writes the new rows into the storage
    // and advances cursor / size (a read of pinned host memory is a 2 us round trip: not in this kernel's prologue).
    const float* myrow = batch_row(rows, rs, b0, nvalid);
    int64_t myidx = -1, cursor = 0;
    if (A.storage) {
      const float* sto = A.storage + (size_t)agent * A.storage_agent_stride;
      uint64_t size = A.storage_size ? (uint64_t)A.storage_size : A.counters[(size_t)agent * 8 + B2RL_CTR_SIZE];
      if (A.new_rows) {
        cursor = (int64_t)A.counters[(size_t)agent * 8 + B2RL_CTR_CURSOR];
        size = min(size + (uint64_t)A.n_new, (uint64_t)A.capacity);
      }
      const int r = l & 7, rr = r < nvalid ? r : nvalid - 1;
      myidx = philox_index(A.hp.seed, (uint32_t)(b0 + rr), step, gid, size);
      myrow = sto + (size_t)myidx * rs;
      if (A.new_rows) {
        int64_t j = myidx - cursor;
        if (j < 0) j += A.capacity;
        if (j < A.n_new) myrow = A.new_rows + (size_t)j * rs;
      }
    }
    if (w < 6) {
      stage_tile(myrow, nvalid, O + AD + 2, O, XA, ldx, t - 128, 64);
    } else {
      stage_tile(myrow, nvalid, 0, O + AD, XB, ldx, t - 192, 64);  // [obs | act] is contiguous in the row
      if (w == 6) {
        const int i = l, r = (i >> 1) & 7, rr = r < nvalid ? r : nvalid - 1;
        const float* src = reinterpret_cast<const float*>(__shfl_sync(0xffffffffu, reinterpret_cast<unsigned long long>(myrow), rr));
        if (i < 2 * RT) cp_async4(&M.rd[r][i & 1], src + O + AD + (i & 1));
      }
    }
    if (A.storage && rank == 0) {  // the sampled rows (and their indices) for the kernels that follow: two rows per warp
      float* dst = const_cast<float*>(rows);
#pragma unroll 1
      for (int r = w - 4; r < nvalid; r += 4) {
        const float* src = reinterpret_cast<const float*>(__shfl_sync(0xffffffffu, reinterpret_cast<unsigned long long>(myrow), r));
        const int64_t si = __shfl_sync(0xffffffffu, myidx, r);
        for (int c = l; c < (rs >> 2); c += 32) st_stream4(dst + (size_t)(b0 + r) * rs + 4 * c, ld_stream4(src + 4 * c));
        if (l == 0 && A.idx_out) A.idx_out[(size_t)agent * B + b0 + r] = si;
      }
    }
  }
  B2RL_TICK(41);
#ifdef B2RL_TIMING
  if (blockIdx.x == 0 && blockIdx.y == 0 && l == 0) g_b2rl_timing[44 + w] = clock64();
#endif
  cp_async_wait_all();
#ifdef B2RL_TIMING
  if (blockIdx.x == 0 && blockIdx.y == 0 && l == 0) g_b2rl_timing[52 + w] = clock64();
#endif
  __syncthreads();
  int gi = 0;

  // ---- next action
  gi = trunk_fwd<WIDE>(G, &act, XA, ldx, nullptr, &S, gi, nullptr, nullptr, b0, nvalid, 2);
  rowdot(act.p[F_W3], act.p[F_B3], act.out_dim, S.h[1], S.u);
  __syncthreads();
  B2RL_TICK(10);
  for (int r = w; r < RT; r += NW) {  // warp <-> batch row, lane <-> action dim
    float lp = 0.f;
    if (l < AD) {
      const float lo = M.lo[l], hi = M.hi[l];
      const float scale = (hi - lo) * 0.5f, bias = (hi + lo) * 0.5f;  // agents/nets.py:200-204
      const float z = M.eps[r][l];
      const float u0 = uref(S.u, r, l);
      float act_v;
      if (td3) {
        float th;
        act_v = td3_action(u0, scale, bias, th);
        if (A.hp.targ_smoothing) {
          float n = __fmul_rn(z, V.td3_std);
          n = fminf(fmaxf(n, -V.td3_c), V.td3_c);
          act_v = fminf(fmaxf(__fadd_rn(act_v, n), lo), hi);
        }
      } else {
        const GaussSample g = gauss_sample(u0, uref(S.u, r, AD + l), z, scale, bias);
        act_v = g.action;
        lp = g.logp;
      }
      reinterpret_cast<float*>(&XA[(r >> 2) * ldx + O + l])[r & 3] = act_v;
    }
    lp = warp_sum(lp);
    if (l == 0) M.logpi[r] = lp;
  }
  __syncthreads();

  // ---- target Q_k on (next_obs, a')  (agent.py:208-210), then swap the 8 values with the peer group
  B2RL_TICK(11);
  gi = trunk_fwd<WIDE>(G, &qt, XA, ldx, nullptr, &S, gi, nullptr, nullptr, b0, nvalid, 12);
  rowdot(qt.p[F_W3], qt.p[F_B3], 1, S.h[1], S.u);
  __syncthreads();
  B2RL_TICK(21);
  if (t == 0) mbar_expect(&S.xbar[0], RT * sizeof(float));
  if (t < RT) {
    const float q = uref(S.u, t, 0);
    M.qn[k][t] = q;
    st_async_f32(map_peer(smem_u32(&M.qn[k][t]), rank ^ 2), q, map_peer(smem_u32(&S.xbar[0]), rank ^ 2));
  }
  __syncthreads();
  mbar_wait(&S.xbar[0], 0);
  B2RL_TICK(22);

  // ---- TD target (agent.py:212-228)
  if (t < RT) {
    const int r = t;
    const float q0 = M.qn[0][r], q1 = M.qn[1][r];
    const float qmin = fminf(q0, q1);
    float qp = A.hp.bcq_mix ? __fadd_rn(__fmul_rn(0.75f, qmin), __fmul_rn(0.25f, fmaxf(q0, q1))) : qmin;
    if (!td3) {
      const float alpha = expf(A.log_alpha[(size_t)agent * 5]);
      qp = __fsub_rn(qp, __fmul_rn(alpha, M.logpi[r]));
    }
    const float rew = M.rd[r][0], done = M.rd[r][1];
    const float y = __fadd_rn(rew, __fmul_rn(__fmul_rn(1.0f - done, V.gamma), qp));
    M.y[r] = y;
    if (A.dbg_targ_q && rank == 0 && r < nvalid) A.dbg_targ_q[(size_t)agent * B + b0 + r] = y;
  }
  // (M.y is read after the barriers inside trunk_fwd)

  // ---- online Q_k, loss, backward (agent.py:230-235)
  {
    const Workspace ws = ws_carve(wsb, B, k);
    float* part = ws.part + (size_t)rb * PART_LEN;
    B2RL_TICK(23);
    gi = trunk_fwd<WIDE>(G, &qo, XB, ldx, &M.a, &S, gi, ws.h1, ws.h2, b0, nvalid, 24);
    rowdot(qo.p[F_W3], qo.p[F_B3], 1, S.h[1], S.u);
    __syncthreads();
    B2RL_TICK(33);
    if (t < RT) {
      const int r = t;
      const bool valid = r < nvalid;
      const float qv = uref(S.u, r, 0);
      const float dlt = qv - M.y[r];
      const float dq = valid ? dlt * (2.0f / (float)B) : 0.f;  // d mean((q-y)^2) / dq
      M.dq[r] = dq;
      M.sq[r] = valid ? dlt * dlt : 0.f;
      if (valid && G.c == 0) {
        ws.dz3[(size_t)(b0 + r) * MAX_OUT] = dq;
        if (A.dbg_q) A.dbg_q[((size_t)agent * 2 + k) * B + b0 + r] = qv;
      }
    }
    __syncthreads();
    if (t == 0 && G.c == 0) {
      float sd = 0.f, ss = 0.f;
#pragma unroll
      for (int r = 0; r < RT; ++r) { sd += M.dq[r]; ss += M.sq[r]; }
      part[PART_DB3] = sd;
      part[PART_SCAL] = ss;
    }
    const float w3 = qo.p[F_W3][t];
#pragma unroll
    for (int r = 0; r < RT; ++r) S.red[DH_OFF + r * HID + t] = M.dq[r] * w3;  // dLoss/dh2, column t (read back by thread t)
    B2RL_TICK(34);
    gi = trunk_bwd(G, &qo, &M.a, &S, gi, ws.dz1, ws.dz2, part, b0, nvalid);
    B2RL_TICK(35);
  }
}

#ifdef B2RL_TIMING
extern "C" int b2rl_debug_timing(long long* host64) {  // critic_fused_kernel's phase timestamps (debug builds)
  return cudaMemcpyFromSymbol(host64, g_b2rl_timing, sizeof(long long) * 64) == cudaSuccess ? 0 : -2;
}
#endif

// loads the kernel (CUDA loads lazily; a first launch inside stream capture would fail) and opts in
// to > 48 KB of dynamic shared memory
int max_in_dim_critic() { return (int)((MAX_DYN_SMEM - critic_smem_bytes(0)) / (2 * RQ * sizeof(float4))); }

cudaError_t init_critic() {
  cudaError_t e = cudaFuncSetAttribute(critic_fused_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, MAX_DYN_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(critic_fused_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, MAX_DYN_SMEM);
  return e;
}

cudaError_t launch_critic_fused(const b2rl_update_args_t& a, cudaStream_t st) {
  const size_t smem = critic_smem_bytes(a.fmt.ob_dim + a.fmt.ac_dim);
  if (smem > (size_t)MAX_DYN_SMEM) return cudaErrorInvalidValue;
  // clusters of 4 along x: (row block, critic, column slice)
  const dim3 grid(4 * row_blocks(a.batch), a.n_agents);
  if (a.fmt.ob_dim + a.fmt.ac_dim > W1S_ROWS) return launch_cluster(critic_fused_kernel<true>, grid, 4, smem, st, a);
  return launch_cluster(critic_fused_kernel<false>, grid, 4, smem, st, a);
}

}  // namespace b2rl
