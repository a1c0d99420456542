// actor.cu — fused actor step (forward, twin-Q with constant critic parameters, loss, backward into the
// actor), the SAC temperature step, and the inference policy. Replaces agents/agent.py:247-283, :295-303,
// :172-181. Built from the cluster column-split blocks of mlp_cluster.cuh: 8 batch rows per cluster.
#include "mlp_cluster.cuh"
#include "policy.cuh"
#include "rng.cuh"

namespace b2rl {

constexpr int MAX_A = MAX_OUT / 2;

struct ActorSmem {
  Work s;
  Acts pi;         // the actor's pass (kept for its backward pass)
  Acts q;          // this group's critic pass
  NetStage nsA, nsQ;
  Net nA, nQ;
  float lo[MAX_A], hi[MAX_A];
  float eps[RT][MAX_A], sg[RT][MAX_A], yy[RT][MAX_A], th[RT][MAX_A];
  float4 da_peer[RQ * MAX_OUT];  // dLoss/da through the peer group's critic, same layout as Work::u
  float qv[2][RT], logpi[RT], dq[2][RT], lossr[RT], lpv[RT];
  // followed by the input tile float4[RQ * (O + A)]: [obs | a_pi]
};
__host__ __device__ inline size_t actor_smem_bytes(int in_dim) {
  return sizeof(ActorSmem) + (size_t)RQ * in_dim * sizeof(float4);
}

// SAC: cluster of 4, rank = 2k + c. Group k evaluates and differentiates critic k for the cluster's 8 rows (both
// groups recompute the identical actor forward), the groups swap Q_k (8 floats) to agree on the arg-min, group 1
// hands its dQ/da to group 0 through distributed shared memory and retires; group 0 runs the actor's backward
// pass. TD3's loss uses critic 0 only (agent.py:274-275): clusters of 2, one group.
template <bool WIDE>
__global__ void __launch_bounds__(NT, 1) actor_fused_kernel(const __grid_constant__ b2rl_update_args_t A) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  ActorSmem& M = *reinterpret_cast<ActorSmem*>(smem_raw);
  Work& S = M.s;
  exchange_init_arrive(S);  // (shared memory and the cluster barrier only: legal before the grid dependency)
  pdl_enter();
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank(), csize = (int)cluster.num_blocks();
  const int k = rank >> 1;
  const Group G{rank & 1, rank & ~1};
  const int t = threadIdx.x, w = t >> 5, l = t & 31;
  const int agent = blockIdx.y, rb = blockIdx.x / csize, b0 = rb * RT;
  const int O = A.fmt.ob_dim, AD = A.fmt.ac_dim, rs = A.fmt.row_stride, B = A.batch;
  const int ldx = O + AD, nvalid = min(RT, B - b0);
  float4* X = reinterpret_cast<float4*>(smem_raw + sizeof(ActorSmem));
  const uint32_t gid = (uint32_t)(A.agent_base + agent);  // global agent id: keys the Philox streams
  const bool td3 = A.hp.td3 != 0;

  const float* P = A.arena + (size_t)agent * A.arena_agent_stride;
  const float* rows = A.rows + (size_t)agent * A.rows_agent_stride;
  const uint64_t step = A.counters[(size_t)agent * 8 + B2RL_CTR_PI];
  float* wsb = A.workspace + (size_t)agent * A.workspace_agent_stride;
  const Workspace ws = ws_carve(wsb, B, 0);
  float* part = ws.part + (size_t)rb * PART_LEN;
  const float alpha = td3 ? 0.f : expf(A.log_alpha[(size_t)agent * 5]);
  const float invB = 1.0f / (float)B;

  // ---- prologue: the observation tile and the small tensors, one job per warp
  const Net &act = M.nA, &q = M.nQ;
  if (w == 0) {
    if (l < AD) {
      M.lo[l] = __ldg(A.min_ac + l);
      M.hi[l] = __ldg(A.max_ac + l);
    }
    if (!td3)
      tile_noise<RT, MAX_A>(M.eps, A.eps, rank == 0 ? A.eps_out : nullptr, A.hp.seed, (int64_t)agent * B + b0, b0, nvalid, AD, step, gid,
                            STREAM_ACTOR_EPS, true, l);
  } else if (w == 1) {
    stage_net(P, &A.actor, &M.nsA, &M.nA, G.c * CW);
  } else if (w == 2) {
    stage_net(P, &A.critic[k], &M.nsQ, &M.nQ, G.c * CW);
  } else if (w >= 4) {
    stage_tile(batch_row(rows, rs, b0, nvalid), nvalid, 0, O, X, ldx, t - 128, 128);
  }
  cp_async_wait_all();
  __syncthreads();
  int gi = 0;

  // ---- actor forward on obs (agent.py:251 / :254-255)
  gi = trunk_fwd<WIDE>(G, &act, X, ldx, &M.pi, &S, gi, k == 0 ? ws.h1 : nullptr, k == 0 ? ws.h2 : nullptr, b0, nvalid);
  rowdot(act.p[F_W3], act.p[F_B3], act.out_dim, S.h[1], S.u);
  __syncthreads();
  for (int r = w; r < RT; r += NW) {  // warp <-> batch row, lane <-> action dim
    float lp = 0.f;
    if (l < AD) {
      const float lo = M.lo[l], hi = M.hi[l];
      const float scale = (hi - lo) * 0.5f, bias = (hi + lo) * 0.5f;
      const float u0 = uref(S.u, r, l);
      float act_v;
      if (td3) {
        float th;
        act_v = td3_action(u0, scale, bias, th);
        M.th[r][l] = th;
      } else {
        const GaussSample g = gauss_sample(u0, uref(S.u, r, AD + l), M.eps[r][l], scale, bias);
        act_v = g.action;
        lp = g.logp;
        M.sg[r][l] = g.sigma; M.yy[r][l] = g.y; M.th[r][l] = g.th;
      }
      reinterpret_cast<float*>(&X[(r >> 2) * ldx + O + l])[r & 3] = act_v;
    }
    lp = warp_sum(lp);
    if (l == 0) M.logpi[r] = lp;
  }
  __syncthreads();

  // ---- Q_k(obs, a_pi) with the critic's parameters held constant (agent.py:272-278)
  gi = trunk_fwd<WIDE>(G, &q, X, ldx, &M.q, &S, gi, nullptr, nullptr, b0, nvalid);
  rowdot(q.p[F_W3], q.p[F_B3], 1, S.h[1], S.u);
  __syncthreads();
  if (!td3 && t == 0) mbar_expect(&S.xbar[0], RT * sizeof(float));
  if (t < RT) {
    const float qk = uref(S.u, t, 0);
    M.qv[k][t] = qk;
    if (!td3) st_async_f32(map_peer(smem_u32(&M.qv[k][t]), rank ^ 2), qk, map_peer(smem_u32(&S.xbar[0]), rank ^ 2));
  }
  __syncthreads();
  if (!td3) mbar_wait(&S.xbar[0], 0);

  // ---- loss and dLoss/dQ_k per row: SAC  mean(alpha*logpi - min_k Q_k), TD3  mean(-Q_0)
  if (t < RT) {
    const int r = t;
    const bool valid = r < nvalid;
    const float q0 = M.qv[0][r];
    float lossr, d0 = -invB, d1 = 0.f;
    if (td3) {
      lossr = -q0;
    } else {
      const float q1 = M.qv[1][r];
      const bool first = q0 <= q1;  // torch.min(0) returns the first minimal index on ties
      d0 = first ? -invB : 0.f;
      d1 = first ? 0.f : -invB;
      lossr = __fsub_rn(__fmul_rn(alpha, M.logpi[r]), first ? q0 : q1);
    }
    M.dq[0][r] = valid ? d0 : 0.f;
    M.dq[1][r] = valid ? d1 : 0.f;
    M.lossr[r] = valid ? lossr : 0.f;
    M.lpv[r] = valid ? M.logpi[r] : 0.f;
  }
  __syncthreads();
  if (t == 0 && rank == 0) {
    float sl = 0.f, sp = 0.f;
#pragma unroll
    for (int r = 0; r < RT; ++r) { sl += M.lossr[r]; sp += M.lpv[r]; }
    part[PART_SCAL] = sl;
    part[PART_SCAL + 1] = sp;
  }

  // ---- backward through critic k down to its action inputs
  {
    const float w3 = q.p[F_W3][t];
#pragma unroll
    for (int r = 0; r < RT; ++r) S.red[DH_OFF + r * HID + t] = M.dq[k][r] * w3;  // dLoss/dh2 of critic k, column t
    gi = trunk_bwd(G, &q, &M.q, &S, gi, nullptr, nullptr, nullptr, b0, nvalid);
    rowdot(q.p[F_W1T] + (size_t)O * HID, nullptr, AD, S.h[1], S.u);  // dQ/da_i = sum_j dz1_j * W1[j][O+i]
    __syncthreads();
  }
  if (!td3) {
    if (k == 1) {  // hand dQ/da to group 0 and retire
      for (int i = t; i < RQ * AD; i += NT) {
        const int qq = i / AD, a = i - qq * AD;
        st_async_v4(map_peer(smem_u32(&M.da_peer[qq * MAX_OUT + a]), rank ^ 2), S.u[qq * MAX_OUT + a],
                    map_peer(smem_u32(&S.xbar[1]), rank ^ 2));
      }
      return;
    }
    if (t == 0) mbar_expect(&S.xbar[1], RQ * AD * sizeof(float4));
    mbar_wait(&S.xbar[1], 0);
  }

  // ---- backward through the action head (group 0)
  for (int r = w; r < RT; r += NW) {
    if (l < AD) {
      const float scale = (M.hi[l] - M.lo[l]) * 0.5f;
      float ga = uref(S.u, r, l);                       // through critic 0
      if (!td3) ga += uref(M.da_peer, r, l);            // + through critic 1
      float g_a = 0.f, g_b = 0.f;
      if (td3) {
        const float th = M.th[r][l];
        g_a = ga * scale * (1.0f - th * th);
      } else if (r < nvalid) {
        GaussSample g;
        g.y = M.yy[r][l]; g.sigma = M.sg[r][l]; g.th = M.th[r][l];
        gauss_backward(g, M.eps[r][l], scale, ga, alpha * invB, g_a, g_b);
      }
      uref(S.du, r, l) = g_a;
      if (!td3) uref(S.du, r, AD + l) = g_b;
      if (G.c == 0 && r < nvalid) {
        ws.dz3[(size_t)(b0 + r) * MAX_OUT + l] = g_a;
        if (!td3) ws.dz3[(size_t)(b0 + r) * MAX_OUT + AD + l] = g_b;
      }
    }
  }
  __syncthreads();
  if (t < act.out_dim && G.c == 0) {
    const float4 d0 = S.du[t], d1 = S.du[MAX_OUT + t];
    part[PART_DB3 + t] = ((d0.x + d0.y) + (d0.z + d0.w)) + ((d1.x + d1.y) + (d1.z + d1.w));
  }
  {  // head backward: dLoss/dh2[r][t] = sum_o du[o][r] * W3[o][t]
    float dh[RT];
#pragma unroll
    for (int r = 0; r < RT; ++r) dh[r] = 0.f;
    const float* W3 = act.p[F_W3];
#pragma unroll 8  // (a head wider than the staged 8 rows is read from global memory: keep 8 loads in flight)
    for (int o = 0; o < act.out_dim; ++o) {
      const float wv = W3[(size_t)o * HID + t];
      const float4 d0 = S.du[o], d1 = S.du[MAX_OUT + o];
      dh[0] = fmaf(wv, d0.x, dh[0]); dh[1] = fmaf(wv, d0.y, dh[1]); dh[2] = fmaf(wv, d0.z, dh[2]); dh[3] = fmaf(wv, d0.w, dh[3]);
      dh[4] = fmaf(wv, d1.x, dh[4]); dh[5] = fmaf(wv, d1.y, dh[5]); dh[6] = fmaf(wv, d1.z, dh[6]); dh[7] = fmaf(wv, d1.w, dh[7]);
    }
#pragma unroll
    for (int r = 0; r < RT; ++r) S.red[DH_OFF + r * HID + t] = dh[r];
  }
  gi = trunk_bwd(G, &act, &M.pi, &S, gi, ws.dz1, ws.dz2, part, b0, nvalid);
}

// ---- SAC temperature step -------------------------------------------------------------------
// Every cluster of 2: log-prob of a fresh sample from the UPDATED actor for its 8 rows; the last cluster to
// finish (ticket in counters[4]) sums the per-cluster partials in a fixed order, forms
//   alpha_loss = mean(alpha * (-logpi - targ_ent)),  d/dlog_alpha = same value,
// and applies torch's capturable Adam step to the scalar.
struct AlphaSmem {
  Work s;
  NetStage ns;
  Net n;
  float logpi[RT];
  int last;
  // followed by the observation tile float4[RQ * O]
};
__host__ __device__ inline size_t alpha_smem_bytes(int ob_dim) {
  return sizeof(AlphaSmem) + (size_t)RQ * ob_dim * sizeof(float4) + 4 * sizeof(float);  // + {targ_ent, lr} behind the tile
}

__device__ __forceinline__ void adam_scalar(float* st /*{p,g,m,v}*/, float g, float lr, float t, float b1, float b2,
                                            float eps) {
  float p = st[0], m = st[2], v = st[3];
  m = m + (1.0f - b1) * (g - m);
  v = v * b2 + (1.0f - b2) * g * g;
  const float bc1 = 1.0f - powf(b1, t), bc2 = 1.0f - powf(b2, t);
  const float ssn = -(lr / bc1);
  const float denom = sqrtf(v) / (sqrtf(bc2) * ssn) + eps / ssn;
  p += m / denom;
  st[0] = p; st[1] = g; st[2] = m; st[3] = v;
}

template <bool WIDE>
__global__ void __launch_bounds__(NT, 1) alpha_kernel(const __grid_constant__ b2rl_update_args_t A, float lr) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  AlphaSmem& M = *reinterpret_cast<AlphaSmem*>(smem_raw);
  Work& S = M.s;
  exchange_init_arrive(S);  // (shared memory and the cluster barrier only: legal before the grid dependency)
  pdl_enter();
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const Group G{rank, 0};
  const int t = threadIdx.x, w = t >> 5, l = t & 31;
  const int agent = blockIdx.y, rb = blockIdx.x >> 1, b0 = rb * RT, nblk = gridDim.x >> 1;
  const int O = A.fmt.ob_dim, AD = A.fmt.ac_dim, rs = A.fmt.row_stride, B = A.batch;
  const int nvalid = min(RT, B - b0);
  float4* X = reinterpret_cast<float4*>(smem_raw + sizeof(AlphaSmem));
  float* hpv = reinterpret_cast<float*>(X + RQ * O);  // this agent's {targ_ent, lr} (common.cuh agent_hp)
  const uint32_t gid = (uint32_t)(A.agent_base + agent);
  const float* P = A.arena + (size_t)agent * A.arena_agent_stride;
  const float* rows = A.rows + (size_t)agent * A.rows_agent_stride;
  uint64_t* ctr = A.counters + (size_t)agent * 8;
  const uint64_t step = ctr[B2RL_CTR_PI];
  float* wsb = A.workspace + (size_t)agent * A.workspace_agent_stride;
  float* part = ws_carve(wsb, B, 0).part;

  if (w == 0) {
    stage_net(P, &A.actor, &M.ns, &M.n, G.c * CW);
    if (l == 0) {
      hpv[0] = agent_hp(A.agent_hp, agent, HP_TARG_ENT, A.hp.targ_ent);
      hpv[1] = agent_hp(A.agent_hp, agent, HP_LR + B2RL_CTR_ALPHA, lr);  // (lr > 0 decides whether to step at all)
    }
  } else {
    stage_tile(batch_row(rows, rs, b0, nvalid), nvalid, 0, O, X, O, t - 32, NT - 32);
  }
  const Net& act = M.n;
  cp_async_wait_all();
  __syncthreads();
  int gi = 0;
  gi = trunk_fwd<WIDE>(G, &act, X, O, nullptr, &S, gi, nullptr, nullptr, b0, nvalid);
  if (rank != 0) return;  // (no peer touches this CTA's shared memory after the last all-gather's barrier)
  rowdot(act.p[F_W3], act.p[F_B3], act.out_dim, S.h[1], S.u);
  __syncthreads();
  for (int r = w; r < RT; r += NW) {
    float lp = 0.f;
    if (l < AD && r < nvalid) {
      const float lo = __ldg(A.min_ac + l), hi = __ldg(A.max_ac + l);
      const int64_t e = ((int64_t)agent * B + b0 + r) * AD + l;
      const float z = noise_at(A.eps2, e, A.hp.seed, b0 + r, l, step, gid, STREAM_ALPHA_EPS);
      if (A.eps2_out) A.eps2_out[e] = z;
      lp = gauss_sample(uref(S.u, r, l), uref(S.u, r, AD + l), z,
                        (hi - lo) * 0.5f, (hi + lo) * 0.5f).logp;
    }
    lp = warp_sum(lp);
    if (l == 0) M.logpi[r] = lp;
  }
  __syncthreads();
  if (t == 0) {
    const float te = hpv[0];
    float s = 0.f;
    for (int r = 0; r < nvalid; ++r) s += (-M.logpi[r] - te);  // sum_r (-logpi_r - targ_ent), agent.py:300
    part[(size_t)rb * PART_LEN + PART_SCAL + 2] = s;
    __threadfence();
    const unsigned long long ticket = atomicAdd((unsigned long long*)&ctr[B2RL_CTR_TICKET], 1ULL);
    M.last = (ticket == (unsigned long long)nblk - 1);
  }
  __syncthreads();
  if (!M.last) return;
  if (w == 0) {  // the last cluster: lane-strided sum of the per-cluster partials, fixed shuffle tree
    __threadfence();
    float s = 0.f;
    for (int i = l; i < nblk; i += 32) s += __ldcg(&part[(size_t)i * PART_LEN + PART_SCAL + 2]);
    s = warp_sum(s);
    if (l == 0) {
      float* st = A.log_alpha + (size_t)agent * 5;
      const float alpha = expf(st[0]);
      const float loss = alpha * (s / (float)B);
      if (lr > 0.f) {
        const uint64_t tstep = ctr[B2RL_CTR_ALPHA] + 1;
        adam_scalar(st, loss, hpv[1], (float)tstep, 0.9f, 0.999f, 1e-8f);
        ctr[B2RL_CTR_ALPHA] = tstep;
      } else {
        st[1] = loss;  // data parallel: local gradient only; b2rl_alpha_adam finishes after the all-reduce
      }
      ctr[B2RL_CTR_TICKET] = 0;  // re-arm the ticket for the next launch / graph replay
      float* out = A.out + (size_t)agent * 8;
      out[B2RL_OUT_ALPHA_LOSS] = loss;
      out[B2RL_OUT_ALPHA] = expf(st[0]);
    }
  }
}

// hp: per-agent learning rates (b2rl_alpha_adam_hp) or NULL (b2rl_alpha_adam: lr for every agent)
__global__ void alpha_adam_kernel(float* log_alpha, uint64_t* counters, int n_agents, float lr, const b2rl_agent_hp_t* hp,
                                  float grad_scale, float* out) {
  pdl_enter();
  const int a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= n_agents) return;
  float* st = log_alpha + (size_t)a * 5;
  uint64_t* ctr = counters + (size_t)a * 8;
  const uint64_t tstep = ctr[B2RL_CTR_ALPHA] + 1;
  adam_scalar(st, st[1] * grad_scale, agent_hp(hp, a, HP_LR + B2RL_CTR_ALPHA, lr), (float)tstep, 0.9f, 0.999f, 1e-8f);
  ctr[B2RL_CTR_ALPHA] = tstep;
  if (out) {
    out[(size_t)a * 8 + B2RL_OUT_ALPHA_LOSS] = st[1];
    out[(size_t)a * 8 + B2RL_OUT_ALPHA] = expf(st[0]);
  }
}

cudaError_t launch_alpha_adam(float* log_alpha, uint64_t* counters, int n_agents, float lr, const b2rl_agent_hp_t* hp,
                              float grad_scale, float* out, cudaStream_t st) {
  return launch_k(alpha_adam_kernel, dim3((n_agents + 127) / 128), dim3(128), 1, 0, st, log_alpha, counters, n_agents, lr, hp,
                  grad_scale, out);
}

// ---- inference policy ----------------------------------------------------------------------------
struct PredictSmem {
  Work s;
  NetStage ns;
  Net n;
  // followed by the observation tile float4[RQ * O]
};
__host__ __device__ inline size_t predict_smem_bytes(int ob_dim) {
  return sizeof(PredictSmem) + (size_t)RQ * ob_dim * sizeof(float4) + 4 * sizeof(float);  // + explore_std behind the tile
}

template <bool WIDE>
__global__ void __launch_bounds__(NT, 1)
predict_kernel(const __grid_constant__ b2rl_update_args_t A, const float* __restrict__ obs, int n, int mode,
               float explore_std, uint64_t draw, float* __restrict__ actions) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  PredictSmem& M = *reinterpret_cast<PredictSmem*>(smem_raw);
  Work& S = M.s;
  exchange_init_arrive(S);  // (shared memory and the cluster barrier only: legal before the grid dependency)
  pdl_enter();
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const Group G{rank, 0};
  const int t = threadIdx.x, w = t >> 5, l = t & 31;
  const int b0 = (blockIdx.x >> 1) * RT;
  const int O = A.fmt.ob_dim, AD = A.fmt.ac_dim;
  const int nvalid = min(RT, n - b0);
  float4* X = reinterpret_cast<float4*>(smem_raw + sizeof(PredictSmem));
  float* xstd = reinterpret_cast<float*>(X + RQ * O);  // this agent's explore_std (common.cuh agent_hp)
  const bool td3 = A.hp.td3 != 0;
  // stacked agents (grid y = local agent g; one learner: g = 0): g's actor, counters, observations, noise and actions
  const int g = blockIdx.y;
  if (w == 0) {
    stage_net(A.arena + (size_t)g * A.arena_agent_stride, &A.actor, &M.ns, &M.n, G.c * CW);
    if (l == 0) *xstd = agent_hp(A.agent_hp, g, HP_EXPLORE, explore_std);
  } else {
    stage_tile(batch_row(obs + (size_t)g * n * O, O, b0, nvalid), nvalid, 0, O, X, O, t - 32, NT - 32);
  }
  const Net& act = M.n;
  cp_async_wait_all();
  __syncthreads();
  int gi = 0;
  gi = trunk_fwd<WIDE>(G, &act, X, O, nullptr, &S, gi, nullptr, nullptr, b0, nvalid);
  if (rank != 0) return;
  rowdot(act.p[F_W3], act.p[F_B3], act.out_dim, S.h[1], S.u);
  __syncthreads();
  // draw = ~0: key the exploration noise on the critic step counter (a captured step graph cannot take a new
  // host value per replay; the counter advances once per learner iteration). Bit 31 of the 32-bit step field separates
  // these draws from the host-counted ones (draw = 1, 2, ... < 2^31), and the GLOBAL agent id is part of the key, so learners
  // that share a seed (data-parallel ranks, population members) explore independently.
  const uint64_t step = (draw == ~0ull && A.counters) ? (A.counters[(size_t)g * 8 + B2RL_CTR_Q] | 0x80000000ull) : draw;
  const uint32_t agent = (uint32_t)(A.agent_base + g);
  for (int r = w; r < nvalid; r += NW) {
    if (l < AD) {
      const float lo = __ldg(A.min_ac + l), hi = __ldg(A.max_ac + l);
      const float scale = (hi - lo) * 0.5f, bias = (hi + lo) * 0.5f;
      const int64_t e = ((int64_t)g * n + b0 + r) * AD + l;  // [n_agents][n][AD]
      const float u0 = uref(S.u, r, l);
      float a;
      if (td3) {  // agents/nets.py:149-159
        float th;
        a = td3_action(u0, scale, bias, th);
        if (mode == 1) {
          const float z = noise_at(A.eps, e, ~A.hp.seed, b0 + r, l, step, agent, STREAM_ACTOR_EPS);
          if (A.eps_out) A.eps_out[e] = z;
          a += z * (scale * *xstd);
        }
      } else if (mode == 1) {  // sample
        const float z = noise_at(A.eps, e, ~A.hp.seed, b0 + r, l, step, agent, STREAM_ACTOR_EPS);  // key != learner's
        if (A.eps_out) A.eps_out[e] = z;
        a = gauss_sample(u0, uref(S.u, r, AD + l), z, scale, bias).action;
      } else {  // mode = tanh(mean)*scale + bias, agents/nets.py:233
        a = __fadd_rn(__fmul_rn(tanhf(u0), scale), bias);
      }
      actions[e] = a;
    }
  }
}

int max_in_dim_actor() { return (int)((MAX_DYN_SMEM - actor_smem_bytes(0)) / (1 * RQ * sizeof(float4))); }

template <typename K>
static cudaError_t opt_in_smem(K kernel) {
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, MAX_DYN_SMEM);
}
cudaError_t init_actor() {
  cudaError_t e = opt_in_smem(actor_fused_kernel<false>);
  if (e == cudaSuccess) e = opt_in_smem(actor_fused_kernel<true>);
  if (e == cudaSuccess) e = opt_in_smem(alpha_kernel<false>);
  if (e == cudaSuccess) e = opt_in_smem(alpha_kernel<true>);
  if (e == cudaSuccess) e = opt_in_smem(predict_kernel<false>);
  if (e == cudaSuccess) e = opt_in_smem(predict_kernel<true>);
  if (e == cudaSuccess) {
    cudaFuncAttributes fa;
    e = cudaFuncGetAttributes(&fa, alpha_adam_kernel);
  }
  return e;
}

cudaError_t launch_actor_fused(const b2rl_update_args_t& a, cudaStream_t st) {
  const size_t smem = actor_smem_bytes(a.fmt.ob_dim + a.fmt.ac_dim);
  if (smem > (size_t)MAX_DYN_SMEM) return cudaErrorInvalidValue;
  const int csize = a.hp.td3 ? 2 : 4;  // (row block, [critic,] column slice)
  const dim3 grid(csize * row_blocks(a.batch), a.n_agents);
  if (a.fmt.ob_dim + a.fmt.ac_dim > W1S_ROWS) return launch_cluster(actor_fused_kernel<true>, grid, csize, smem, st, a);
  return launch_cluster(actor_fused_kernel<false>, grid, csize, smem, st, a);
}

cudaError_t launch_alpha(const b2rl_update_args_t& a, float lr, cudaStream_t st) {
  const size_t smem = alpha_smem_bytes(a.fmt.ob_dim);
  if (smem > (size_t)MAX_DYN_SMEM) return cudaErrorInvalidValue;
  const dim3 grid(2 * row_blocks(a.batch), a.n_agents);
  if (a.fmt.ob_dim > W1S_ROWS) return launch_cluster(alpha_kernel<true>, grid, 2, smem, st, a, lr);
  return launch_cluster(alpha_kernel<false>, grid, 2, smem, st, a, lr);
}

cudaError_t launch_predict(const b2rl_update_args_t& a, const float* obs, int n, int mode, float explore_std,
                           uint64_t draw, float* actions, cudaStream_t st) {
  const size_t smem = predict_smem_bytes(a.fmt.ob_dim);
  if (smem > (size_t)MAX_DYN_SMEM) return cudaErrorInvalidValue;
  const dim3 grid(2 * row_blocks(n), a.n_agents > 1 ? a.n_agents : 1);  // n_agents 0 or 1: one learner, as before
  if (a.fmt.ob_dim > W1S_ROWS)
    return launch_cluster(predict_kernel<true>, grid, 2, smem, st, a, obs, n, mode, explore_std, draw, actions);
  return launch_cluster(predict_kernel<false>, grid, 2, smem, st, a, obs, n, mode, explore_std, draw, actions);
}

}  // namespace b2rl
