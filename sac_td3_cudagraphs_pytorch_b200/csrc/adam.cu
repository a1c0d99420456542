// adam.cu — one launch for "Adam step on some spans + Polyak averaging on some spans" of the flat
// parameter arena. Replaces torch's _multi_tensor_adam (~16 foreach launches per optimizer.step(),
// agents/agent.py:236,286) and tensordict's lerp_ (agents/agent.py:328-331).
//
// Arithmetic: torch/optim/adam.py `capturable` branch (:478-527) — the one the reference runs on the
// GPU (agents/agent.py:118):
//   m = m + (1-b1)(g-m);  v = v*b2 + (1-b2) g g;
//   ss = -(lr / (1-b1^t));  denom = sqrt(v) / (sqrt(1-b2^t) * ss) + eps/ss;  p += m/denom
// Polyak (torch.lerp, weight < 0.5):  targ = targ + polyak * (p_new - targ).
// HBM-bound: 28 B/param for Adam, +8 B/param when fused with Polyak (the new p is still in registers),
// 12 B/param for Polyak alone.
#include "adam_math.cuh"

namespace b2rl {

using SegScalars = AdamScalars;

// PS.seg[q]: the segment whose scalars (lr, step count, clip, Polyak) govern shadow pair q. launch_adam has already cut
// the pairs' spans out of the segment list, so the element-wise loop below never meets them.
struct PairSeg { int seg[3]; };
__global__ void __launch_bounds__(256) adam_polyak_kernel(const __grid_constant__ b2rl_adam_args_t A, const __grid_constant__ PairSeg PS) {
  pdl_enter();
  const int agent = blockIdx.y;
  float* P = A.arena + (size_t)agent * A.arena_agent_stride;
  float* T = P + A.region_stride;
  float* M1 = P + 2 * A.region_stride;
  float* V = P + 3 * A.region_stride;
  float* G = P + 4 * A.region_stride;
  const uint64_t* ctr = A.counters + (size_t)agent * 8;
  float* LO = A.lo ? A.lo + (size_t)agent * A.lo_agent_stride : nullptr;  // 3xTF32 mirror: lo parts of what is written here
  const float polyak = agent_hp(A.agent_hp, agent, HP_POLYAK, A.polyak);

  __shared__ SegScalars sc[B2RL_MAX_SEG];
  if (threadIdx.x < A.n_seg) {
    const b2rl_seg_t& s = A.seg[threadIdx.x];
    SegScalars v = {0.f, 1.f, 1.f, 1.f, 0.f};
    if (s.do_adam) {
      const float t = (float)ctr[s.counter];  // step count AFTER this step's bump (>= 1)
      v = adam_scalars(agent_hp(A.agent_hp, agent, HP_LR + s.counter, s.lr), A.beta1, A.beta2, t);
      adam_finish(v, A.eps);
      v.gscale = s.grad_scale;
      if (s.clip) {  // clip_grad_norm_: g *= min(1, max_norm / (norm + 1e-6))
        const float norm = sqrtf(A.grad_sumsq[agent]) * s.grad_scale;
        v.gscale *= fminf(1.0f, agent_hp(A.agent_hp, agent, HP_CLIP, A.clip_norm) / (norm + 1e-6f));
      }
    }
    sc[threadIdx.x] = v;
  }
  __syncthreads();

  const float omb1 = 1.0f - A.beta1, omb2 = 1.0f - A.beta2;
  const int main_ctas = (int)gridDim.x - 64 * A.n_shadow;
  if ((int)blockIdx.x >= main_ctas) {
    // ---- shadow pairs: one 32 x 32 tile of a net's w2t per CTA; the step is computed once, at the w2t position, and
    // the results go to w2t (as they are read: rows of 128 bytes) and, transposed through shared memory, to w2n.
    __shared__ float tr[6][32][33];  // p, m, v, lo(p), target, lo(target)
    const int tile = (int)blockIdx.x - main_ctas, pr = tile >> 6, tin = tile & 63;
    const int64_t src = A.shadow_src[pr], dst = A.shadow_dst[pr];
    const int si = PS.seg[pr];
    const b2rl_seg_t& s = A.seg[si];
    const SegScalars k = sc[si];
    const int k0 = (tin >> 3) * 32, j0 = (tin & 7) * 32, r = threadIdx.x >> 3, c4 = (threadIdx.x & 7) * 4;
    const int64_t i = src + (int64_t)(k0 + r) * HID + j0 + c4;        // w2t[k0 + r][j0 + c4 ..]
    const int64_t it = dst + (int64_t)(j0 + r) * HID + k0 + c4;       // w2n[j0 + r][k0 + c4 ..]
    auto stage = [&](int b, const float4& x) {  // x is held for w2t[k0 + r][j0 + c4 ..]
      tr[b][r][c4] = x.x, tr[b][r][c4 + 1] = x.y, tr[b][r][c4 + 2] = x.z, tr[b][r][c4 + 3] = x.w;
    };
    auto out_t = [&](int b, float* base) {      // -> base[w2n tile], transposed
      *reinterpret_cast<float4*>(base + it) = make_float4(tr[b][c4][r], tr[b][c4 + 1][r], tr[b][c4 + 2][r], tr[b][c4 + 3][r]);
    };
    const bool da = s.do_adam != 0, dp = s.do_polyak != 0;
    float4 p = *reinterpret_cast<const float4*>(P + i);
    float4 tg = make_float4(0.f, 0.f, 0.f, 0.f);
    if (dp) tg = *reinterpret_cast<const float4*>(T + i);  // (requested before the Adam arithmetic)
    if (da) {
      float4 g = *reinterpret_cast<const float4*>(G + i);
      float4 m = *reinterpret_cast<const float4*>(M1 + i);
      float4 v = *reinterpret_cast<const float4*>(V + i);
      float* pp = &p.x; float* gp = &g.x; float* mp = &m.x; float* vp = &v.x;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const float gg = __fmul_rn(gp[c], k.gscale);
        gp[c] = gg;
        adam_elem(pp[c], gg, mp[c], vp[c], k, A.beta2, omb1, omb2, A.eps);
      }
      if (s.clip) *reinterpret_cast<float4*>(G + i) = g;
      *reinterpret_cast<float4*>(P + i) = p;
      *reinterpret_cast<float4*>(M1 + i) = m;
      *reinterpret_cast<float4*>(V + i) = v;
      stage(0, p);
      stage(1, m);
      stage(2, v);
      if (LO) {
        const float4 l = tf32_lo4(p);
        *reinterpret_cast<float4*>(LO + i) = l;
        stage(3, l);
      }
    }
    if (dp) {
      tg.x = polyak_elem(tg.x, p.x, polyak);
      tg.y = polyak_elem(tg.y, p.y, polyak);
      tg.z = polyak_elem(tg.z, p.z, polyak);
      tg.w = polyak_elem(tg.w, p.w, polyak);
      *reinterpret_cast<float4*>(T + i) = tg;
      stage(4, tg);
      if (LO) {
        const float4 l = tf32_lo4(tg);
        *reinterpret_cast<float4*>(LO + A.region_stride + i) = l;
        stage(5, l);
      }
    }
    __syncthreads();
    if (da) {
      out_t(0, P);
      out_t(1, M1);
      out_t(2, V);
      if (LO) out_t(3, LO);
    }
    if (dp) {
      out_t(4, T);
      if (LO) out_t(5, LO + A.region_stride);
    }
    return;
  }
  // ---- everything else, element-wise: the segments (pieces between the pairs' spans) form ONE flat index space, so that
  // a thread's elements are independent loads in flight instead of one dependent round trip per segment
  __shared__ int64_t sbeg[B2RL_MAX_SEG], slen[B2RL_MAX_SEG];
  if (threadIdx.x < B2RL_MAX_SEG) {
    const bool on = (int)threadIdx.x < A.n_seg;
    sbeg[threadIdx.x] = on ? A.seg[threadIdx.x].begin : 0;
    slen[threadIdx.x] = on ? A.seg[threadIdx.x].end - A.seg[threadIdx.x].begin : 0;
  }
  __syncthreads();
  int64_t total = 0;
#pragma unroll
  for (int q = 0; q < B2RL_MAX_SEG; ++q) total += slen[q];
  const int64_t stride = (int64_t)main_ctas * blockDim.x * 4;
  for (int64_t f = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4; f < total; f += stride) {
    int si = 0;
    int64_t off = f;
#pragma unroll
    for (int q = 0; q < B2RL_MAX_SEG - 1; ++q)
      if (si == q && off >= slen[q]) { off -= slen[q]; si = q + 1; }
    const int64_t i = sbeg[si] + off;
    const b2rl_seg_t& s = A.seg[si];
    const SegScalars k = sc[si];
    {
      float4 p = *reinterpret_cast<const float4*>(P + i);
      if (s.do_adam) {
        float4 g = *reinterpret_cast<const float4*>(G + i);
        float4 m = *reinterpret_cast<const float4*>(M1 + i);
        float4 v = *reinterpret_cast<const float4*>(V + i);
        float* pp = &p.x; float* gp = &g.x; float* mp = &m.x; float* vp = &v.x;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const float gg = __fmul_rn(gp[c], k.gscale);
          gp[c] = gg;
          adam_elem(pp[c], gg, mp[c], vp[c], k, A.beta2, omb1, omb2, A.eps);
        }
        // clip_grad_norm_ scales .grad in place (agent.py:284-285): keep region 4 what torch would show
        if (s.clip) *reinterpret_cast<float4*>(G + i) = g;
        *reinterpret_cast<float4*>(P + i) = p;
        if (LO) *reinterpret_cast<float4*>(LO + i) = tf32_lo4(p);
        *reinterpret_cast<float4*>(M1 + i) = m;
        *reinterpret_cast<float4*>(V + i) = v;
      }
      if (s.do_polyak) {
        float4 tg = *reinterpret_cast<const float4*>(T + i);
        tg.x = polyak_elem(tg.x, p.x, polyak);
        tg.y = polyak_elem(tg.y, p.y, polyak);
        tg.z = polyak_elem(tg.z, p.z, polyak);
        tg.w = polyak_elem(tg.w, p.w, polyak);
        *reinterpret_cast<float4*>(T + i) = tg;
        if (LO) *reinterpret_cast<float4*>(LO + A.region_stride + i) = tf32_lo4(tg);
      }
    }
  }
}

// sum of squares of a gradient span: stage 1 (per-CTA partials) and stage 2 (fixed-order total)
__global__ void __launch_bounds__(256) sumsq_partial_kernel(const float* arena, int64_t region_stride,
                                                            int64_t agent_stride, int64_t begin, int64_t end,
                                                            float* scratch) {
  pdl_enter();
  const int agent = blockIdx.y;
  const float* G = arena + (size_t)agent * agent_stride + 4 * region_stride;
  float s = 0.f;
  for (int64_t i = begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < end; i += (int64_t)gridDim.x * blockDim.x) {
    const float g = G[i];
    s = fmaf(g, g, s);
  }
  __shared__ float ws[8];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tsum = 0.f;
    for (int w = 0; w < 8; ++w) tsum += ws[w];
    scratch[(size_t)agent * gridDim.x + blockIdx.x] = tsum;
  }
}
__global__ void sumsq_final_kernel(const float* scratch, int n_part, float* sumsq) {
  pdl_enter();
  const int agent = blockIdx.x;
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int i = 0; i < n_part; ++i) s += scratch[(size_t)agent * n_part + i];
    sumsq[agent] = s;
  }
}

__global__ void bump_kernel(uint64_t* counters, int which, int n_agents) {
  pdl_enter();
  const int a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a < n_agents) counters[(size_t)a * 8 + which] += 1ULL;
}

constexpr int SUMSQ_PARTS = 64;

cudaError_t init_adam() {
  cudaFuncAttributes fa;
  cudaError_t e = cudaFuncGetAttributes(&fa, adam_polyak_kernel);
  if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, sumsq_partial_kernel);
  if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, sumsq_final_kernel);
  if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, bump_kernel);
  return e;
}

cudaError_t launch_adam(const b2rl_adam_args_t& a_in, cudaStream_t st) {
  // Keep only the shadow pairs this launch touches (w2t inside one of its segments) and CUT their two spans out of the
  // segment list: the element-wise CTAs then walk plain spans (a per-element "is this a pair's span?" test made of
  // dependent constant-bank loads cost 8 us per launch), the pairs go to 64 tile CTAs each. A pair's tiles take their
  // scalars from any piece of the segment the pair was cut from (or from a zero-length piece if nothing is left of it).
  b2rl_adam_args_t a = a_in;
  PairSeg ps = {{0, 0, 0}};
  a.n_shadow = 0;
  a.n_seg = 0;
  const int64_t n = (int64_t)HID * HID;
  int64_t total = 0;
  for (int i = 0; i < a_in.n_seg; ++i) {
    const b2rl_seg_t& s = a_in.seg[i];
    int64_t cuts[6][2];
    int nc = 0;
    const int first_pair = a.n_shadow;
    for (int q = 0; q < a_in.n_shadow; ++q)
      if (a_in.shadow_src[q] >= s.begin && a_in.shadow_src[q] < s.end) {
        a.shadow_src[a.n_shadow] = a_in.shadow_src[q];
        a.shadow_dst[a.n_shadow++] = a_in.shadow_dst[q];
        cuts[nc][0] = a_in.shadow_src[q], cuts[nc++][1] = a_in.shadow_src[q] + n;
        cuts[nc][0] = a_in.shadow_dst[q], cuts[nc++][1] = a_in.shadow_dst[q] + n;
      }
    for (int x = 0; x < nc; ++x)  // sort the cuts by start
      for (int y = x + 1; y < nc; ++y)
        if (cuts[y][0] < cuts[x][0]) {
          const int64_t t0 = cuts[x][0], t1 = cuts[x][1];
          cuts[x][0] = cuts[y][0], cuts[x][1] = cuts[y][1], cuts[y][0] = t0, cuts[y][1] = t1;
        }
    const int first_piece = a.n_seg;
    int64_t cur = s.begin;
    for (int x = 0; x <= nc; ++x) {
      const int64_t stop = x < nc ? cuts[x][0] : s.end;
      if (stop > cur || (x == nc && a.n_seg == first_piece)) {  // (at least one piece per segment: it carries the scalars)
        if (a.n_seg >= B2RL_MAX_SEG) return cudaErrorInvalidValue;
        a.seg[a.n_seg] = s;
        a.seg[a.n_seg].begin = cur;
        a.seg[a.n_seg].end = stop > cur ? stop : cur;
        total += a.seg[a.n_seg].end - cur;
        ++a.n_seg;
      }
      if (x < nc) cur = cuts[x][1];
    }
    for (int q = first_pair; q < a.n_shadow; ++q) ps.seg[q] = first_piece;
  }
  int ctas = (int)((total / 4 + 255) / 256);
  if (ctas < 1) ctas = 1;
  if (ctas > 148 * 4) ctas = 148 * 4;  // grid-stride beyond four CTAs per SM
  // + 64 tile CTAs per shadow pair (blockIdx.x >= ctas)
  return launch_k(adam_polyak_kernel, dim3(ctas + 64 * a.n_shadow, a.n_agents), dim3(256), 1, 0, st, a, ps);
}

cudaError_t launch_sumsq(const float* arena, int64_t region_stride, int64_t agent_stride, int64_t begin, int64_t end,
                         int n_agents, float* sumsq, float* scratch, cudaStream_t st) {
  cudaError_t e = launch_k(sumsq_partial_kernel, dim3(SUMSQ_PARTS, n_agents), dim3(256), 1, 0, st, arena, region_stride, agent_stride,
                           begin, end, scratch);
  if (e != cudaSuccess) return e;
  return launch_k(sumsq_final_kernel, dim3(n_agents), dim3(32), 1, 0, st, (const float*)scratch, (int)SUMSQ_PARTS, sumsq);
}

cudaError_t launch_bump(uint64_t* counters, int which, int n_agents, cudaStream_t st) {
  return launch_k(bump_kernel, dim3((n_agents + 127) / 128), dim3(128), 1, 0, st, counters, which, n_agents);
}

}  // namespace b2rl
