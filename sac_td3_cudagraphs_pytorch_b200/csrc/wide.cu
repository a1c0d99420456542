// wide.cu — the layer-by-layer ("wide") path of the update for LARGE batches (BASELINE.json config 5: batch 65 536;
// stacked populations later): every step of agents/agent.py:186-235 as its own batch-parallel kernel around the
// tensor-core hidden layers of tc_linear.cu, with all intermediates in HBM. The row-group kernels of
// mlp_cluster.cuh are latency-optimal at batch 256 but stream each layer's weights from L2 once per 8 rows
// (~10 TFLOP/s at any batch size); here the weights are read once per 128 rows by TMA and the products run on
// tcgen05. Same arithmetic as the row path outside the products (LayerNorm two-pass statistics, policy heads,
// TD target, losses); the Philox noise is keyed identically, so both paths draw the same samples.
//
// Kernels (all: grid over rows, no atomics, fixed summation order => bitwise reproducible):
//   wide_first       X[M][K] . w1t -> LayerNorm -> ReLU  (first layers: K = O or O + A, FFMA)
//   wide_policy_head h2 -> head -> tanh-Gaussian sample / TD3 smoothed action; writes [next_obs | a'] and log-prob
//   wide_q_head      h2 -> Q; online mode: TD target from the twin target Qs, dQ, squared-error partials
//   wide_ln_bwd      dLoss/dhead -> dh2 -> ReLU mask -> LayerNorm backward -> dz2, per-CTA column sums
//   (tc_linear mode 2: dz2 . W2 -> LayerNorm backward of layer 1 in the TMEM epilogue -> dz1, column sums)
//   wide_colsum      per-CTA column-sum partials -> bias / LayerNorm-affine gradients; loss scalar
#include "common.cuh"
#include "policy.cuh"
#include "rng.cuh"

namespace b2rl {

constexpr int WF_ROWS = 64;  // rows per CTA of wide_first: 8 per warp
constexpr int WF_KC = 32;    // k chunk of weights / inputs staged in shared memory

// ---- first layer -------------------------------------------------------------------------------------------------
// z[r][j] = b[j] + sum_k X[r][k] * w1t[k][j], then LayerNorm / ReLU. A WARP owns 8 rows and all 256 columns (lane l:
// columns 4l..4l+3 and 128+4l..+3), so a row's LayerNorm statistics are two warp reductions over registers — no staging
// of z in shared memory, no CTA barrier between the product and the row-wise part (the first version, thread <-> column
// over 32 rows with z staged through shared memory, ran at 1.4-2.9 TB/s: 187 us for 268-536 MB of output at
// n_agents x M = 262 144 rows) — and every store is a full 512-byte row segment per warp instruction. The weight chunk
// [k][256] and the rows' inputs are staged once per CTA; per four k a lane issues 8 LDS.128 of weights (16-byte lane
// stride: conflict-free) and 8 broadcast LDS.128 of inputs for 256 FMAs.
__global__ void __launch_bounds__(256)
wide_first_kernel(const float* __restrict__ X, int64_t ldx, int M, int K, const float* __restrict__ w1t,
                  const float* __restrict__ b, const float* __restrict__ g, const float* __restrict__ be, int ln,
                  float* __restrict__ H, float* __restrict__ XH, float2* __restrict__ stat, long long ps) {
  {  // stacked agents: blockIdx.y = agent; its rows are M further, its parameters ps floats further
    const size_t ag = blockIdx.y;
    X += ag * M * ldx, H += ag * M * HID, w1t += ag * ps, b += ag * ps;
    if (XH) XH += ag * M * HID;
    if (stat) stat += ag * M;
    if (ln) g += ag * ps, be += ag * ps;
  }
  __shared__ __align__(16) float ws[WF_KC][HID];      // weight chunk, forward layout [k][j]
  __shared__ __align__(16) float xs[WF_ROWS][WF_KC];  // the rows' inputs for the chunk
  const int t = threadIdx.x, w = t >> 5, l = t & 31;
  const int m0 = blockIdx.x * WF_ROWS, r0 = m0 + 8 * w;
  float acc[8][8];
#pragma unroll
  for (int r = 0; r < 8; ++r)
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[r][c] = 0.f;
  for (int k0 = 0; k0 < K; k0 += WF_KC) {
    const int kc = min(WF_KC, K - k0), kc4 = (kc + 3) & ~3;
    for (int i = t; i < kc4 * (HID / 4); i += 256) {  // (rows kc..kc4-1 are zero: they meet zero inputs, but must be finite)
      const int k = i >> 6, q = i & 63;
      reinterpret_cast<float4*>(ws[k])[q] = k < kc ? ldg4(w1t + (size_t)(k0 + k) * HID + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    for (int i = t; i < WF_ROWS * WF_KC; i += 256) {
      const int r = i >> 5, k = i & 31;
      const int row = min(m0 + r, M - 1);  // (rows beyond M repeat the last one; their outputs are not stored)
      xs[r][k] = k < kc ? __ldg(X + (size_t)row * ldx + k0 + k) : 0.f;
    }
    __syncthreads();
    for (int k = 0; k < kc4; k += 4) {
      float4 wa[4], wb[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        wa[u] = *reinterpret_cast<const float4*>(&ws[k + u][4 * l]);
        wb[u] = *reinterpret_cast<const float4*>(&ws[k + u][128 + 4 * l]);
      }
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const float4 x = *reinterpret_cast<const float4*>(&xs[8 * w + r][k]);
        const float xv[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          acc[r][0] = fmaf(xv[u], wa[u].x, acc[r][0]); acc[r][1] = fmaf(xv[u], wa[u].y, acc[r][1]);
          acc[r][2] = fmaf(xv[u], wa[u].z, acc[r][2]); acc[r][3] = fmaf(xv[u], wa[u].w, acc[r][3]);
          acc[r][4] = fmaf(xv[u], wb[u].x, acc[r][4]); acc[r][5] = fmaf(xv[u], wb[u].y, acc[r][5]);
          acc[r][6] = fmaf(xv[u], wb[u].z, acc[r][6]); acc[r][7] = fmaf(xv[u], wb[u].w, acc[r][7]);
        }
      }
    }
    __syncthreads();
  }
  const float4 ba = ldg4(b + 4 * l), bb = ldg4(b + 128 + 4 * l);
  const float bj[8] = {ba.x, ba.y, ba.z, ba.w, bb.x, bb.y, bb.z, bb.w};
  float gj[8], bej[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) gj[c] = 1.f, bej[c] = 0.f;
  if (ln) {
    const float4 ga = ldg4(g + 4 * l), gb = ldg4(g + 128 + 4 * l), ea = ldg4(be + 4 * l), eb = ldg4(be + 128 + 4 * l);
    gj[0] = ga.x, gj[1] = ga.y, gj[2] = ga.z, gj[3] = ga.w, gj[4] = gb.x, gj[5] = gb.y, gj[6] = gb.z, gj[7] = gb.w;
    bej[0] = ea.x, bej[1] = ea.y, bej[2] = ea.z, bej[3] = ea.w, bej[4] = eb.x, bej[5] = eb.y, bej[6] = eb.z, bej[7] = eb.w;
  }
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    const int row = r0 + r;
    if (row >= M) break;  // (warp-uniform)
    float z[8], h[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) z[c] = acc[r][c] + bj[c];
    if (ln) {  // two-pass mean / variance over the row's 256 values (8 per lane + shuffles)
      float s = ((z[0] + z[1]) + (z[2] + z[3])) + ((z[4] + z[5]) + (z[6] + z[7]));
      s = warp_sum(s);
      const float mean = s * (1.0f / HID);
      float q = 0.f;
#pragma unroll
      for (int c = 0; c < 8; ++c) { const float d = z[c] - mean; q = fmaf(d, d, q); }
      q = warp_sum(q);
      const float rstd = 1.0f / sqrtf(q * (1.0f / HID) + LN_EPS);
      if (stat && l == 0) stat[row] = make_float2(mean, rstd);
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        z[c] = (z[c] - mean) * rstd;  // x-hat
        h[c] = fmaxf(fmaf(z[c], gj[c], bej[c]), 0.f);
      }
    } else {
#pragma unroll
      for (int c = 0; c < 8; ++c) h[c] = fmaxf(z[c], 0.f);
    }
    float* hp = H + (size_t)row * HID;
    *reinterpret_cast<float4*>(hp + 4 * l) = make_float4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<float4*>(hp + 128 + 4 * l) = make_float4(h[4], h[5], h[6], h[7]);
    if (XH) {
      float* xp = XH + (size_t)row * HID;
      *reinterpret_cast<float4*>(xp + 4 * l) = make_float4(z[0], z[1], z[2], z[3]);
      *reinterpret_cast<float4*>(xp + 128 + 4 * l) = make_float4(z[4], z[5], z[6], z[7]);
    }
  }
}

// ---- policy head: warp per row ----------------------------------------------------------------------------------------
using WidePolicyArgs = b2rl_wide_policy_t;

constexpr int WP_ROWS = 64;  // rows per CTA (8 per warp): the head's weights are staged once per 64 rows, not once per 8
// Two phases per CTA of 64 rows. (1) WARP <-> row: the head's dot products (lanes over the 256 inputs), results to shared
// memory. (2) THREAD <-> (row, action dimension): noise, tanh-Gaussian sample / TD3 smoothing, log-prob terms — the
// transcendental part (Philox, Box-Muller, 2 tanh, exp, 2 log, a division: ~450 instructions) now runs once per 32
// (row, dimension) pairs instead of once per row with 3 lanes alive: the one-phase version issued 669 warp instructions
// per row and was issue-bound (74 % issue-slot utilisation, 1.5 TB/s of its 6.5: profiles/r2_ncu_full_pop256_summary.csv).
// (min 5 CTAs per SM: without it, the per-agent smoothing values pushed ptxas from 48 to 64 registers, 4 CTAs per SM)
// Phase (1) of the policy heads: us[rr][o] = w3s[o] . h2[grow0 + rr] + b3[o] for the CTA's nrows rows, a warp per row (rows
// w, w + 8, ...). per_row(grow) runs at the top of each row's turn (the training head copies the row's obs-part there).
template <class PerRow>
__device__ __forceinline__ void head_rows(const float* __restrict__ h2, size_t grow0, int nrows, int out_dim, const float* w3s,
                                          const float* __restrict__ b3g, float* us, int w, int l, PerRow per_row) {
  float hn[8];  // the next row's activations are requested before this row's head is computed (one round trip hidden)
  if (w < nrows) {
#pragma unroll
    for (int i = 0; i < 8; ++i) hn[i] = __ldg(h2 + (grow0 + w) * HID + l + 32 * i);
  }
  for (int rr = w; rr < nrows; rr += 8) {
    const size_t grow = grow0 + rr;   // row of the stacked arrays
    float h[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) h[i] = hn[i];
    if (rr + 8 < nrows) {
#pragma unroll
      for (int i = 0; i < 8; ++i) hn[i] = __ldg(h2 + (grow + 8) * HID + l + 32 * i);
    }
    per_row(grow);
    if (out_dim <= 8) {
      // Heads of up to 8 outputs (every task but Humanoid's SAC head): the dot products are reduced TOGETHER — a butterfly
      // that halves the number of live sums at each of its first three steps (9 shuffles instead of 5 per output; the same
      // pairs are added in the same order as warp_sum does). The per-output loop made the kernel issue-bound (ncu: 61 %
      // issue utilisation at 46 us per 65 536 rows, ~220 warp instructions per row).
      float s[8];
#pragma unroll
      for (int o = 0; o < 8; ++o) {
        s[o] = 0.f;
        if (o < out_dim) {
#pragma unroll
          for (int i = 0; i < 8; ++i) s[o] = fmaf(w3s[o * HID + l + 32 * i], h[i], s[o]);
        }
      }
      const bool b4 = l & 16, b3 = l & 8, b2 = l & 4;  // the output this lane ends up with: 4 b4 + 2 b3 + b2
      float a4[4], a2[2], a1;
#pragma unroll
      for (int j = 0; j < 4; ++j) a4[j] = (b4 ? s[4 + j] : s[j]) + __shfl_xor_sync(0xffffffffu, b4 ? s[j] : s[4 + j], 16);
#pragma unroll
      for (int j = 0; j < 2; ++j) a2[j] = (b3 ? a4[2 + j] : a4[j]) + __shfl_xor_sync(0xffffffffu, b3 ? a4[j] : a4[2 + j], 8);
      a1 = (b2 ? a2[1] : a2[0]) + __shfl_xor_sync(0xffffffffu, b2 ? a2[0] : a2[1], 4);
      a1 += __shfl_xor_sync(0xffffffffu, a1, 2);
      a1 += __shfl_xor_sync(0xffffffffu, a1, 1);
      const int o = (b4 ? 4 : 0) + (b3 ? 2 : 0) + (b2 ? 1 : 0);
      if ((l & 3) == 0 && o < out_dim) us[rr * out_dim + o] = a1 + __ldg(b3g + o);
    } else {
      for (int o = 0; o < out_dim; ++o) {
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) s = fmaf(w3s[o * HID + l + 32 * i], h[i], s);
        s = warp_sum(s);
        if (l == 0) us[rr * out_dim + o] = s + __ldg(b3g + o);
      }
    }
  }
}

__global__ void __launch_bounds__(256, 5) wide_policy_head_kernel(const __grid_constant__ WidePolicyArgs P, const Stk K) {
  extern __shared__ float w3s[];            // [out][256], then us [64][out] head outputs, then lps [64][A] log-prob terms
  float* us = w3s + P.out_dim * HID;
  float* lps = us + WP_ROWS * P.out_dim;
  const int t = threadIdx.x, w = t >> 5, l = t & 31;
  const size_t ag = blockIdx.y;                 // stacked agents: rows [ag * M, ag * M + M), parameters ps further
  const float* w3g = P.w3 + ag * K.ps;
  const float* b3g = P.b3 + ag * K.ps;
  for (int i = t; i < P.out_dim * HID; i += 256) w3s[i] = __ldg(w3g + i);
  __syncthreads();
  const int row0 = blockIdx.x * WP_ROWS;        // first row of this CTA inside the agent's batch
  const int nrows = min(WP_ROWS, P.M - row0);
  head_rows(P.h2, ag * P.M + row0, nrows, P.out_dim, w3s, b3g, us, w, l, [&](size_t grow) {
    // the obs-part of the next network's input
    const float* src = P.rows + grow * P.row_stride + P.src_off;
    float* xr = P.xn + grow * P.ldn;
    for (int k = l; k < P.O; k += 32) xr[k] = __ldg(src + k);
  });
  __syncthreads();
  const uint32_t agent = P.agent + (uint32_t)ag;
  const uint64_t step = P.counters[ag * K.cs + P.counter_idx];
  // this agent's target smoothing, loaded beside `step`; the actor and temperature steps run the head without smoothing
  const bool smooth = P.td3 && P.smoothing;
  const float td3_std = smooth ? agent_hp(K.hp, (int)ag, HP_TD3_STD, P.td3_std) : 0.f;
  const float td3_c = smooth ? agent_hp(K.hp, (int)ag, HP_TD3_C, P.td3_c) : 0.f;
  for (int i = t; i < nrows * P.A; i += 256) {
    const int rr = i / P.A, a = i - rr * P.A;
    const int row = row0 + rr;                  // row inside the agent's batch: the Philox key
    const size_t grow = ag * P.M + row;
    const float lo = __ldg(P.min_ac + a), hi = __ldg(P.max_ac + a);
    const float scale = (hi - lo) * 0.5f, bias = (hi + lo) * 0.5f;
    const float u_mu = us[rr * P.out_dim + a];
    const int64_t e = (int64_t)grow * P.A + a;
    float act_v, lp = 0.f;
    if (P.td3) {
      float th;
      act_v = td3_action(u_mu, scale, bias, th);
      if (P.save) P.save[grow * 4 * P.A + 3 * P.A + a] = th;
      if (P.smoothing) {
        const float z = noise_at(P.eps, e, P.seed, row, a, step, agent, P.stream_id);
        if (P.eps_out) P.eps_out[e] = z;
        float n = __fmul_rn(z, td3_std);
        n = fminf(fmaxf(n, -td3_c), td3_c);
        act_v = fminf(fmaxf(__fadd_rn(act_v, n), lo), hi);
      }
    } else {
      const float z = noise_at(P.eps, e, P.seed, row, a, step, agent, P.stream_id);
      if (P.eps_out) P.eps_out[e] = z;
      const GaussSample gs = gauss_sample(u_mu, us[rr * P.out_dim + P.A + a], z, scale, bias);
      act_v = gs.action;
      lp = gs.logp;
      if (P.save) {  // what the head's backward pass needs: [M][4][A] = eps, sigma, tanh(x), tanh(raw log-std)
        float* sv = P.save + grow * 4 * P.A;
        sv[a] = z; sv[P.A + a] = gs.sigma; sv[2 * P.A + a] = gs.y; sv[3 * P.A + a] = gs.th;
      }
    }
    P.xn[grow * P.ldn + P.O + a] = act_v;
    lps[i] = lp;
  }
  if (P.logp) {
    __syncthreads();
    if (t < nrows) {  // log pi(a|s) = sum over the action dimensions, in index order
      float s = 0.f;
      for (int a = 0; a < P.A; ++a) s += lps[t * P.A + a];
      P.logp[ag * P.M + row0 + t] = s;
    }
  }
}

// ---- behaviour policy: Agent.predict (agents/agent.py:172-181, nets.py:149-159, :222-234) on h2 of n observations --------
// Phase (1) as the training head; phase (2) thread <-> (row, action dimension) with exactly the formulas and Philox key of
// actor.cu predict_kernel (seed ~hp.seed, stream STREAM_ACTOR_EPS, row and dimension as there): the two policies draw the
// same noise and differ only by the arithmetic of the forward pass. TD3 mode 1 adds the noise without a clamp, as
// predict_kernel does (the reference's clamp result is dropped, SURVEY App. C.7).
__global__ void __launch_bounds__(256) wide_predict_kernel(const __grid_constant__ b2rl_wide_predict_t P) {
  extern __shared__ float w3s[];  // [out][256], then us [64][out]
  float* us = w3s + P.out_dim * HID;
  const int t = threadIdx.x, w = t >> 5, l = t & 31;
  for (int i = t; i < P.out_dim * HID; i += 256) w3s[i] = __ldg(P.w3 + i);
  __syncthreads();
  const int row0 = blockIdx.x * WP_ROWS;
  const int nrows = min(WP_ROWS, P.n - row0);
  head_rows(P.h2, (size_t)row0, nrows, P.out_dim, w3s, P.b3, us, w, l, [](size_t) {});
  __syncthreads();
  const uint64_t step = (P.draw == ~0ull && P.counters) ? (P.counters[B2RL_CTR_Q] | 0x80000000ull) : P.draw;
  const float xstd = agent_hp(P.agent_hp, 0, HP_EXPLORE, P.explore_std);
  for (int i = t; i < nrows * P.A; i += 256) {
    const int rr = i / P.A, a = i - rr * P.A;
    const int row = row0 + rr;
    const float lo = __ldg(P.min_ac + a), hi = __ldg(P.max_ac + a);
    const float scale = (hi - lo) * 0.5f, bias = (hi + lo) * 0.5f;
    const int64_t e = (int64_t)row * P.A + a;
    const float u0 = us[rr * P.out_dim + a];
    float act;
    if (P.td3) {
      float th;
      act = td3_action(u0, scale, bias, th);
      if (P.mode == 1) {
        const float z = noise_at(P.eps, e, ~P.seed, row, a, step, P.agent, STREAM_ACTOR_EPS);
        if (P.eps_out) P.eps_out[e] = z;
        act += z * (scale * xstd);
      }
    } else if (P.mode == 1) {
      const float z = noise_at(P.eps, e, ~P.seed, row, a, step, P.agent, STREAM_ACTOR_EPS);
      if (P.eps_out) P.eps_out[e] = z;
      act = gauss_sample(u0, us[rr * P.out_dim + P.A + a], z, scale, bias).action;
    } else {
      act = __fadd_rn(__fmul_rn(tanhf(u0), scale), bias);
    }
    P.actions[e] = act;
  }
}

// ---- critic head: warp per row ------------------------------------------------------------------------------------------
using WideQArgs = b2rl_wide_q_t;

__global__ void __launch_bounds__(256) wide_q_head_kernel(const __grid_constant__ WideQArgs Q, const Stk K) {
  __shared__ float sq_w[8], dq_w[8];
  const int t = threadIdx.x, w = t >> 5, l = t & 31;
  const size_t ag = blockIdx.y;
  const int lrow = blockIdx.x * 8 + w;
  const size_t row = ag * Q.M + lrow;
  const float* w3 = Q.w3 + ag * K.ps;
  const float gamma = agent_hp(K.hp, (int)ag, HP_GAMMA, Q.gamma);
  float sq = 0.f, dqv = 0.f;
  if (lrow < Q.M) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s = fmaf(__ldg(w3 + l + 32 * i), __ldg(Q.h2 + row * HID + l + 32 * i), s);
    const float q = warp_sum(s) + __ldg(Q.b3 + ag * K.ps);
    if (l == 0) {
      Q.q_out[row] = q;
      if (Q.mode == 1) {  // agents/agent.py:212-233
        const float q0 = Q.qn0[row], q1 = Q.qn1[row];
        const float qmin = fminf(q0, q1);
        float qp = Q.bcq_mix ? __fadd_rn(__fmul_rn(0.75f, qmin), __fmul_rn(0.25f, fmaxf(q0, q1))) : qmin;
        if (!Q.td3) qp = __fsub_rn(qp, __fmul_rn(expf(Q.log_alpha[ag * K.as]), Q.logp[row]));
        const float* rr = Q.rows + row * Q.row_stride + Q.rd_off;
        const float y = __fadd_rn(rr[0], __fmul_rn(__fmul_rn(1.0f - rr[1], gamma), qp));
        if (Q.targ_out) Q.targ_out[row] = y;
        const float dlt = q - y;
        dqv = dlt * (2.0f / (float)Q.M);
        Q.dz3[row * MAX_OUT] = dqv;
        sq = dlt * dlt;
      }
    }
  }
  if (Q.mode == 1) {
    if (l == 0) { sq_w[w] = sq; dq_w[w] = dqv; }
    __syncthreads();
    if (t == 0) {  // per-CTA partials {sum of squared errors, sum of dQ}: sq_part[2 * cta], [2 * cta + 1]
      float s = 0.f, d = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) { s += sq_w[i]; d += dq_w[i]; }
      const size_t pi = ag * gridDim.x + blockIdx.x;
      Q.sq_part[2 * pi] = s;
      Q.sq_part[2 * pi + 1] = d;
    }
  }
}

// ---- backward of the head and of layer 2's row-wise step: warp per row, 16 rows per warp, 128 per CTA -----------------
// dh2[j] = sum_o dz3[row][o] * w3[o][j]; ReLU mask (recomputed from x-hat), LayerNorm backward -> dz2; per-CTA column
// sums {sum dz, sum dn*xhat, sum dn} -> part[cta][3][256]. dw3_part (scalar heads only, n_out == 1: the critics): the
// head's weight gradient dW3[j] = sum_b dz3[b] * h2[b][j] rides along — h2 is recomputed from x-hat, which this kernel
// reads anyway — as a fourth column sum -> dw3_part[cta][3][256] (slot 0), so the critics need no tc_wgrad launch (a
// 268 MB re-read of h2 per critic at 1 024 agents, 34 + 15 us per critic at batch 65 536) for a 256-float gradient.
constexpr int WB_ROWS = 128;
__global__ void __launch_bounds__(256)
wide_ln_bwd_kernel(const float* __restrict__ dz3, int n_out, const float* __restrict__ w3, const float* __restrict__ xh,
                   const float2* __restrict__ stat, const float* __restrict__ g, const float* __restrict__ be, int ln, int M,
                   float* __restrict__ dz, float* __restrict__ part, float* __restrict__ dw3_part, long long ps) {
  {  // stacked agents: blockIdx.y = agent
    const size_t ag = blockIdx.y;
    dz3 += ag * M * MAX_OUT, xh += ag * M * HID, dz += ag * M * HID, w3 += ag * ps;
    if (part) part += ag * gridDim.x * 3 * HID;
    if (dw3_part) dw3_part += ag * gridDim.x * 3 * HID;
    if (ln) stat += ag * M, g += ag * ps, be += ag * ps;
  }
  extern __shared__ float wsm[];          // w3 [n_out][256], then the cross-warp reduction buffer [8][3][256]
  float* w3s = wsm;
  float* red = wsm + n_out * HID;
  const int t = threadIdx.x, w = t >> 5, l = t & 31;
  for (int i = t; i < n_out * HID; i += 256) w3s[i] = __ldg(w3 + i);
  __syncthreads();
  float gj[8], bj[8], sdz[8], sdx[8], sdn[8], sw3[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    gj[i] = ln ? __ldg(g + l + 32 * i) : 1.f;
    bj[i] = ln ? __ldg(be + l + 32 * i) : 0.f;
    sdz[i] = sdx[i] = sdn[i] = sw3[i] = 0.f;
  }
  const int r0 = blockIdx.x * WB_ROWS + w * (WB_ROWS / 8);
  // Everything a row needs from global memory — x-hat, its rstd, the head's first gradient — is requested one row ahead:
  // with the loads at their points of use a row was three dependent round trips (ncu: 39 % long-scoreboard samples).
  float xn[8], rstd_n = 1.f, d_n = 0.f;
  auto fetch = [&](int row) {
#pragma unroll
    for (int i = 0; i < 8; ++i) xn[i] = __ldg(xh + (size_t)row * HID + l + 32 * i);
    if (ln) rstd_n = __ldg(&stat[row].y);
    d_n = __ldg(dz3 + (size_t)row * MAX_OUT);
  };
  if (r0 < M) fetch(r0);
  for (int rr = 0; rr < WB_ROWS / 8; ++rr) {
    const int row = r0 + rr;
    if (row >= M) break;
    float dh[8], x[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      dh[i] = 0.f;
      x[i] = xn[i];
    }
    const float d0 = d_n, rstd_row = rstd_n;
    if (rr + 1 < WB_ROWS / 8 && row + 1 < M) fetch(row + 1);
    for (int o = 0; o < n_out; ++o) {
      const float d = o == 0 ? d0 : __ldg(dz3 + (size_t)row * MAX_OUT + o);
#pragma unroll
      for (int i = 0; i < 8; ++i) dh[i] = fmaf(d, w3s[o * HID + l + 32 * i], dh[i]);
    }
    float dn[8], dx[8], s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float pre = ln ? fmaf(x[i], gj[i], bj[i]) : x[i];  // the forward pre-ReLU value, recomputed bit-exactly
      const bool on = pre > 0.f;
      sw3[i] = fmaf(d0, on ? pre : 0.f, sw3[i]);
      dn[i] = on ? dh[i] : 0.f;
      dx[i] = dn[i] * gj[i];
      s1 += dx[i];
      s2 = fmaf(dx[i], x[i], s2);
    }
    float rstd = 1.f, m1 = 0.f, m2 = 0.f;
    if (ln) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        s1 += __shfl_xor_sync(0xffffffffu, s1, o);
        s2 += __shfl_xor_sync(0xffffffffu, s2, o);
      }
      m1 = s1 * (1.0f / HID);
      m2 = s2 * (1.0f / HID);
      rstd = rstd_row;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float z = ln ? rstd * (dx[i] - m1 - x[i] * m2) : dn[i];
      dz[(size_t)row * HID + l + 32 * i] = z;
      sdz[i] += z;
      sdx[i] = fmaf(dn[i], x[i], sdx[i]);
      sdn[i] += dn[i];
    }
  }
  if (part) {  // (uniform; NULL: the pass is after dz only — the actor step's way through the critics)
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      red[(w * 3 + 0) * HID + l + 32 * i] = sdz[i];
      red[(w * 3 + 1) * HID + l + 32 * i] = sdx[i];
      red[(w * 3 + 2) * HID + l + 32 * i] = sdn[i];
    }
    __syncthreads();
    for (int v = 0; v < 3; ++v) {
      float s = 0.f;
#pragma unroll
      for (int ww = 0; ww < 8; ++ww) s += red[(ww * 3 + v) * HID + t];
      part[((size_t)blockIdx.x * 3 + v) * HID + t] = s;
    }
  }
  if (dw3_part) {  // (uniform) one more cross-warp reduction through the same buffer
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 8; ++i) red[w * HID + l + 32 * i] = sw3[i];
    __syncthreads();
    float s = 0.f;
#pragma unroll
    for (int ww = 0; ww < 8; ++ww) s += red[ww * HID + t];
    dw3_part[(size_t)blockIdx.x * 3 * HID + t] = s;
  }
}

// ---- final reductions ----------------------------------------------------------------------------------------------------
// G[off[v] + j] = sum_p part[p][v][j], v < 3 (v >= 1 only when layer_norm). Grid (8 column chunks, 3 vectors); thread
// (c = t & 31, s = t >> 5) sums partials s, s + 32, ... of column 32 * chunk + c; fixed-order combine over s. 1 024 threads:
// the kernel is a chain of L2 round trips (512 partials per column at batch 65 536), so the slices are spread over 32 warps
// and each takes its partials eight loads at a time.
// Up to 8 jobs (partial-sum arrays of equal P) per launch: blockIdx.y = 3 * job + vector.
__global__ void __launch_bounds__(1024)
wide_colsum_kernel(const __grid_constant__ ColsumJobs J, int P, float* __restrict__ G, long long ps) {
  const int job = blockIdx.y / 3, v = blockIdx.y - 3 * job;
  const float* __restrict__ part = J.part[job] + (size_t)blockIdx.z * P * 3 * HID;  // stacked agents: blockIdx.z = agent
  const int64_t off_b = J.off[job][0], off_g = J.off[job][1], off_be = J.off[job][2];
  const int ln = J.ln[job];
  G += (size_t)blockIdx.z * ps;
  __shared__ float red[32][32];
  const int t = threadIdx.x, c = t & 31, sl = t >> 5, j = blockIdx.x * 32 + c;
  if (v > 0 && !ln) return;
  float s = 0.f;
  const int nsl = (int)blockDim.x >> 5;  // 32 warps for long lists (P >= 64), 8 otherwise: a function of P only
  for (int p0 = sl; p0 < P; p0 += 8 * nsl) {  // eight loads in flight, added in the order of the plain loop
    float u[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int p = p0 + nsl * i;
      u[i] = p < P ? __ldg(part + ((size_t)p * 3 + v) * HID + j) : 0.f;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) s += u[i];
  }
  red[sl][c] = s;
  __syncthreads();
  if (sl == 0) {
    float a = 0.f;
    for (int i = 0; i < nsl; ++i) a += red[i][c];
    G[(v == 0 ? off_b : v == 1 ? off_g : off_be) + j] = a;
  }
}
// qf_loss = sum_k mean_b (q_k - y)^2  (agents/agent.py:233); d b3_k = sum_b dQ_k. sq0 / sq1: the per-CTA partials
// {sum sq, sum dQ} written by wide_q_head (online mode), P of them per critic.
__global__ void __launch_bounds__(256)
wide_critic_scalars_kernel(const float* __restrict__ sq0, const float* __restrict__ sq1, int P, int M, float* __restrict__ G,
                           int64_t off_b3_0, int64_t off_b3_1, float* __restrict__ out, const Stk K) {
  sq0 += (size_t)blockIdx.x * P * 2, sq1 += (size_t)blockIdx.x * P * 2;  // stacked agents: blockIdx.x = agent
  G += (size_t)blockIdx.x * K.ps, out += (size_t)blockIdx.x * K.os;
  __shared__ float red[3][256];
  const int t = threadIdx.x;
  float a = 0.f, d0 = 0.f, d1 = 0.f;
  for (int p = t; p < P; p += 256) {
    a += sq0[2 * p] + sq1[2 * p];
    d0 += sq0[2 * p + 1];
    d1 += sq1[2 * p + 1];
  }
  red[0][t] = a; red[1][t] = d0; red[2][t] = d1;
  __syncthreads();
  if (t < 3) {
    float s = 0.f;
    for (int i = 0; i < 256; ++i) s += red[t][i];
    if (t == 0) out[B2RL_OUT_QF_LOSS] = s / (float)M;
    else G[t == 1 ? off_b3_0 : off_b3_1] = s;
  }
}

// ---- actor step: loss and dLoss/dQ per row (agents/agent.py:272-283); thread per row ------------------------------------
// SAC  mean(alpha * logpi - min_k Q_k): the gradient goes to the arg-min critic (first index on ties, torch.min);
// TD3  mean(-Q_0). dzq_k[row * MAX_OUT] <- dLoss/dQ_k; per-CTA partials {sum loss, sum logpi} -> part[cta][2].
__global__ void __launch_bounds__(256)
wide_actor_loss_kernel(const float* __restrict__ q0, const float* __restrict__ q1, const float* __restrict__ logp,
                       const float* __restrict__ log_alpha, int td3, int M, float* __restrict__ dzq0, float* __restrict__ dzq1,
                       float* __restrict__ part, long long as) {
  {  // stacked agents: blockIdx.y = agent
    const size_t ag = blockIdx.y;
    q0 += ag * M, dzq0 += ag * M * MAX_OUT, part += ag * gridDim.x * 2;
    if (!td3) q1 += ag * M, logp += ag * M, log_alpha += ag * as, dzq1 += ag * M * MAX_OUT;
  }
  __shared__ float red[2][8];
  const int t = threadIdx.x, row = blockIdx.x * 256 + t;
  float lossr = 0.f, lp = 0.f;
  if (row < M) {
    const float invM = 1.0f / (float)M;
    const float a0 = q0[row];
    float d0 = -invM, d1 = 0.f;
    if (td3) {
      lossr = -a0;
    } else {
      const float a1 = q1[row];
      const bool first = a0 <= a1;
      d0 = first ? -invM : 0.f;
      d1 = first ? 0.f : -invM;
      lp = logp[row];
      lossr = __fsub_rn(__fmul_rn(expf(log_alpha[0]), lp), first ? a0 : a1);
    }
    dzq0[(size_t)row * MAX_OUT] = d0;
    if (dzq1) dzq1[(size_t)row * MAX_OUT] = d1;
  }
  lossr = warp_sum(lossr);
  lp = warp_sum(lp);
  if ((t & 31) == 0) { red[0][t >> 5] = lossr; red[1][t >> 5] = lp; }
  __syncthreads();
  if (t < 2) {
    float a = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) a += red[t][i];
    part[2 * blockIdx.x + t] = a;
  }
}

// dQ/da[row][a] = sum_j dz1[row][j] * w1t[O + a][j]  (first-layer dX, action columns only); warp per row, 64 rows per CTA
// (the action rows of w1t are staged once per 64 rows — with 8 rows per CTA they were a third of the bytes the kernel read —
// and a warp requests its next row before it reduces the current one)
constexpr int WD_ROWS = 64;
__global__ void __launch_bounds__(256)
wide_dqda_kernel(const float* __restrict__ dz1, const float* __restrict__ w1a /* w1t + O * 256: [A][256] */, int A, int M,
                 float* __restrict__ dqda, long long ps) {
  dz1 += (size_t)blockIdx.y * M * HID, dqda += (size_t)blockIdx.y * M * A, w1a += (size_t)blockIdx.y * ps;  // blockIdx.y = agent
  extern __shared__ float was[];
  const int t = threadIdx.x, w = t >> 5, l = t & 31;
  for (int i = t; i < A * HID; i += 256) was[i] = __ldg(w1a + i);
  __syncthreads();
  const int row0 = blockIdx.x * WD_ROWS, nrows = min(WD_ROWS, M - row0);
  float dn[8];
  if (w < nrows) {
#pragma unroll
    for (int i = 0; i < 8; ++i) dn[i] = __ldg(dz1 + (size_t)(row0 + w) * HID + l + 32 * i);
  }
  for (int rr = w; rr < nrows; rr += 8) {
    const int row = row0 + rr;
    float d[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) d[i] = dn[i];
    if (rr + 8 < nrows) {
#pragma unroll
      for (int i = 0; i < 8; ++i) dn[i] = __ldg(dz1 + (size_t)(row + 8) * HID + l + 32 * i);
    }
    for (int a = 0; a < A; ++a) {
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) s = fmaf(d[i], was[a * HID + l + 32 * i], s);
      s = warp_sum(s);
      if (l == 0) dqda[(size_t)row * A + a] = s;
    }
  }
}

// backward through the action head (agents/nets.py:143-147, :214-234): du[row][o] = dLoss/d(head output o); thread per row.
// Per-CTA column sums of du (d head.bias) -> part_du[cta][MAX_OUT].
__global__ void __launch_bounds__(256)
wide_actor_head_bwd_kernel(const float* __restrict__ dqda0, const float* __restrict__ dqda1, const float* __restrict__ save,
                           const float* __restrict__ min_ac, const float* __restrict__ max_ac, const float* __restrict__ log_alpha,
                           int td3, int A, int M, float* __restrict__ du /* [M][MAX_OUT] */, float* __restrict__ part_du,
                           long long as) {
  {  // stacked agents: blockIdx.y = agent
    const size_t ag = blockIdx.y;
    dqda0 += ag * M * A, save += ag * M * 4 * A, du += ag * M * MAX_OUT, part_du += ag * gridDim.x * MAX_OUT;
    if (dqda1) dqda1 += ag * M * A;
    if (!td3) log_alpha += ag * as;
  }
  __shared__ float red[8][MAX_OUT];
  const int t = threadIdx.x, row = blockIdx.x * 256 + t, out = td3 ? A : 2 * A;
  const bool live = row < M;
  const float c_pi = td3 ? 0.f : expf(log_alpha[0]) / (float)M;
  for (int a = 0; a < A; ++a) {
    float g_a = 0.f, g_b = 0.f;
    if (live) {
      const float scale = (__ldg(max_ac + a) - __ldg(min_ac + a)) * 0.5f;
      float ga = dqda0[(size_t)row * A + a];
      if (dqda1) ga += dqda1[(size_t)row * A + a];
      const float* sv = save + (size_t)row * 4 * A;
      if (td3) {
        const float th = sv[3 * A + a];
        g_a = ga * scale * (1.0f - th * th);
      } else {
        GaussSample gs;
        gs.sigma = sv[A + a]; gs.y = sv[2 * A + a]; gs.th = sv[3 * A + a];
        gauss_backward(gs, sv[a], scale, ga, c_pi, g_a, g_b);
      }
      du[(size_t)row * MAX_OUT + a] = g_a;
      if (!td3) du[(size_t)row * MAX_OUT + A + a] = g_b;
    }
    const float sa = warp_sum(g_a), sb = warp_sum(g_b);
    if ((t & 31) == 0) {
      red[t >> 5][a] = sa;
      if (!td3) red[t >> 5][A + a] = sb;
    }
  }
  __syncthreads();
  if (t < out) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += red[i][t];
    part_du[(size_t)blockIdx.x * MAX_OUT + t] = s;
  }
}

// actor_loss, mean logpi, alpha -> out; d head.bias -> G. part_s [P][2], part_du [P][MAX_OUT] from the two kernels above.
__global__ void __launch_bounds__(256)
wide_actor_scalars_kernel(const float* __restrict__ part_s, const float* __restrict__ part_du, int P, int M, int out_dim, int td3,
                          const float* __restrict__ log_alpha, float* __restrict__ G, int64_t off_b3, float* __restrict__ out,
                          const Stk K) {
  {  // stacked agents: blockIdx.x = agent
    const size_t ag = blockIdx.x;
    part_s += ag * P * 2, part_du += ag * P * MAX_OUT, G += ag * K.ps, out += ag * K.os;
    if (!td3) log_alpha += ag * K.as;
  }
  const int t = threadIdx.x;
  if (t < out_dim) {
    float s = 0.f;
    for (int p = 0; p < P; ++p) s += part_du[(size_t)p * MAX_OUT + t];
    G[off_b3 + t] = s;
  } else if (t >= 64 && t < 66) {
    float s = 0.f;
    for (int p = 0; p < P; ++p) s += part_s[2 * p + (t - 64)];
    if (t == 64) out[B2RL_OUT_ACTOR_LOSS] = s / (float)M;
    else out[B2RL_OUT_LOGPI_MEAN] = s / (float)M;
  } else if (t == 66 && !td3) {
    out[B2RL_OUT_ALPHA] = expf(log_alpha[0]);
  }
}

// temperature gradient (agents/agent.py:295-303): log_alpha state slot 1 <- alpha * mean(-logpi'' - targ_ent); one CTA
__global__ void __launch_bounds__(256)
wide_alpha_grad_kernel(const float* __restrict__ logp2, int M, float targ_ent_arg, float* __restrict__ alpha_state, long long as,
                       const b2rl_agent_hp_t* __restrict__ hp) {
  const float targ_ent = agent_hp(hp, blockIdx.x, HP_TARG_ENT, targ_ent_arg);
  logp2 += (size_t)blockIdx.x * M, alpha_state += (size_t)blockIdx.x * as;  // stacked agents: blockIdx.x = agent
  __shared__ float red[256];
  const int t = threadIdx.x;
  float s = 0.f;
  for (int r0 = t; r0 < M; r0 += 16 * 256) {  // sixteen loads in flight, added in the order of the plain loop
    float v[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = r0 + 256 * i < M ? __ldg(logp2 + r0 + 256 * i) : 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i)
      if (r0 + 256 * i < M) s += (-v[i] - targ_ent);
  }
  red[t] = s;
  __syncthreads();
  if (t == 0) {
    float a = 0.f;
    for (int i = 0; i < 256; ++i) a += red[i];
    alpha_state[1] = expf(alpha_state[0]) * (a / (float)M);
  }
}

// ---- launches ----------------------------------------------------------------------------------------------------------------
cudaError_t init_wide() {
  cudaError_t e = cudaFuncSetAttribute(wide_policy_head_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (MAX_OUT * HID + WP_ROWS * (MAX_OUT + MAX_OUT / 2)) * 4);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(wide_predict_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (MAX_OUT * HID + WP_ROWS * MAX_OUT) * 4);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(wide_ln_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (MAX_OUT + 24) * HID * 4);
  cudaFuncAttributes fa;
  if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, wide_first_kernel);
  if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, wide_q_head_kernel);
  if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, wide_colsum_kernel);
  if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, wide_critic_scalars_kernel);
  if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, wide_actor_loss_kernel);
  if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, wide_dqda_kernel);
  if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, wide_actor_head_bwd_kernel);
  if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, wide_actor_scalars_kernel);
  if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, wide_alpha_grad_kernel);
  return e;
}
cudaError_t launch_wide_first(const float* X, int64_t ldx, int M, int K, const float* w1t, const float* b, const float* g,
                              const float* be, int ln, float* H, float* XH, float* stat, const Stk& k, cudaStream_t st) {
  wide_first_kernel<<<dim3((M + WF_ROWS - 1) / WF_ROWS, k.n), 256, 0, st>>>(X, ldx, M, K, w1t, b, g, be, ln, H, XH,
                                                                            reinterpret_cast<float2*>(stat), k.ps);
  return cudaGetLastError();
}
cudaError_t launch_wide_policy_head(const WidePolicyArgs& p, const Stk& k, cudaStream_t st) {
  const size_t smem = ((size_t)p.out_dim * HID + (size_t)WP_ROWS * (p.out_dim + p.A)) * sizeof(float);
  wide_policy_head_kernel<<<dim3((p.M + WP_ROWS - 1) / WP_ROWS, k.n), 256, smem, st>>>(p, k);
  return cudaGetLastError();
}
cudaError_t launch_wide_predict(const b2rl_wide_predict_t& p, cudaStream_t st) {
  const size_t smem = ((size_t)p.out_dim * HID + (size_t)WP_ROWS * p.out_dim) * sizeof(float);
  wide_predict_kernel<<<(p.n + WP_ROWS - 1) / WP_ROWS, 256, smem, st>>>(p);
  return cudaGetLastError();
}
cudaError_t launch_wide_q_head(const WideQArgs& q, const Stk& k, cudaStream_t st) {
  wide_q_head_kernel<<<dim3((q.M + 7) / 8, k.n), 256, 0, st>>>(q, k);
  return cudaGetLastError();
}
cudaError_t launch_wide_ln_bwd(const float* dz3, int n_out, const float* w3, const float* xh, const float* stat, const float* g,
                               const float* be, int ln, int M, float* dz, float* part, float* dw3_part, const Stk& k,
                               cudaStream_t st) {
  wide_ln_bwd_kernel<<<dim3((M + WB_ROWS - 1) / WB_ROWS, k.n), 256, (size_t)(n_out + 24) * HID * 4, st>>>(
      dz3, n_out, w3, xh, reinterpret_cast<const float2*>(stat), g, be, ln, M, dz, part, dw3_part, k.ps);
  return cudaGetLastError();
}
cudaError_t launch_wide_colsum_multi(const ColsumJobs& J, int P, float* G, const Stk& k, cudaStream_t st) {
  wide_colsum_kernel<<<dim3(HID / 32, 3 * J.n, k.n), P >= 64 ? 1024 : 256, 0, st>>>(J, P, G, k.ps);
  return cudaGetLastError();
}
cudaError_t launch_wide_colsum(const float* part, int P, float* G, int64_t off_b, int64_t off_g, int64_t off_be, int ln,
                               const Stk& k, cudaStream_t st) {
  ColsumJobs J = {};
  J.part[0] = part, J.off[0][0] = off_b, J.off[0][1] = off_g, J.off[0][2] = off_be, J.ln[0] = ln, J.n = 1;
  return launch_wide_colsum_multi(J, P, G, k, st);
}
cudaError_t launch_wide_critic_scalars(const float* sq0, const float* sq1, int P, const float*, const float*, int M, float* G,
                                       int64_t off0, int64_t off1, float* out, const Stk& k, cudaStream_t st) {
  wide_critic_scalars_kernel<<<k.n, 256, 0, st>>>(sq0, sq1, P, M, G, off0, off1, out, k);
  return cudaGetLastError();
}

cudaError_t launch_wide_actor_loss(const float* q0, const float* q1, const float* logp, const float* log_alpha, int td3, int M,
                                   float* dzq0, float* dzq1, float* part, const Stk& k, cudaStream_t st) {
  wide_actor_loss_kernel<<<dim3((M + 255) / 256, k.n), 256, 0, st>>>(q0, q1, logp, log_alpha, td3, M, dzq0, dzq1, part, k.as);
  return cudaGetLastError();
}
cudaError_t launch_wide_dqda(const float* dz1, const float* w1a, int A, int M, float* dqda, const Stk& k, cudaStream_t st) {
  wide_dqda_kernel<<<dim3((M + WD_ROWS - 1) / WD_ROWS, k.n), 256, (size_t)A * HID * 4, st>>>(dz1, w1a, A, M, dqda, k.ps);
  return cudaGetLastError();
}
cudaError_t launch_wide_actor_head_bwd(const float* dqda0, const float* dqda1, const float* save, const float* min_ac,
                                       const float* max_ac, const float* log_alpha, int td3, int A, int M, float* du,
                                       float* part_du, const Stk& k, cudaStream_t st) {
  wide_actor_head_bwd_kernel<<<dim3((M + 255) / 256, k.n), 256, 0, st>>>(dqda0, dqda1, save, min_ac, max_ac, log_alpha, td3, A, M, du,
                                                                         part_du, k.as);
  return cudaGetLastError();
}
cudaError_t launch_wide_actor_scalars(const float* part_s, const float* part_du, int P, int M, int out_dim, int td3,
                                      const float* log_alpha, float* G, int64_t off_b3, float* out, const Stk& k, cudaStream_t st) {
  wide_actor_scalars_kernel<<<k.n, 256, 0, st>>>(part_s, part_du, P, M, out_dim, td3, log_alpha, G, off_b3, out, k);
  return cudaGetLastError();
}
cudaError_t launch_wide_alpha_grad(const float* logp2, int M, float targ_ent, float* alpha_state, const Stk& k, cudaStream_t st) {
  wide_alpha_grad_kernel<<<k.n, 256, 0, st>>>(logp2, M, targ_ent, alpha_state, k.as, k.hp);
  return cudaGetLastError();
}

}  // namespace b2rl
