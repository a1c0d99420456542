// mlp_cluster.cuh — building blocks of the fused SAC/TD3 kernels: a 2x256 MLP evaluated (and
// differentiated) for a tile of RT = 8 batch rows by a GROUP of CS = 2 CTAs of one thread-block cluster.
//
// Why this shape (DESIGN.md §3): at batch 256 the update is a chain of ~20 dependent [256x256]x[256xB]
// products. Batch rows are independent through the forward pass and through the dX half of the backward
// pass, so a group that owns 8 rows runs every layer of every network back to back with no grid-wide
// synchronisation; only the weight gradients (a contraction over the batch) need a second kernel (wgrad.cu).
// Inside a group the OUTPUT COLUMNS of every layer are split: CTA c computes columns [128c, 128c+128) for the 8
// rows, so it streams half of the layer's weights (128 KB of a 256x256 layer) from L2 — the first version, one
// CTA per 4 rows streaming whole layers, was bound by exactly that L2->SM traffic (profiles/r1_*). The 8x128
// slices are then exchanged through distributed shared memory (st.async into the peer's Z buffer, completion
// counted on the peer's mbarrier: no cluster barrier, no fence), and both CTAs run the cheap row-wise part
// (LayerNorm, ReLU) for the full 8x256 tile redundantly, which leaves each holding the full operand of the next
// layer. (Four-way splits with 16 rows need clusters of 8 for the twin critics, of which only 15 fit on a B200
// at one CTA per SM — one short of the 16 that batch 256 needs; tools/probes/cluster_occupancy.cu.)
// The products are fp32 FFMA2 (fma.rn.f32x2: two fused multiply-adds per lane per issue slot).
//
// CODE SIZE IS A FIRST-CLASS COST HERE. The kernels are one long dependent chain executed once by 8 warps in
// lockstep, so instruction fetch is not hidden by other warps: the first clustered version (everything unrolled
// and inlined, 140 KB of SASS per kernel against a 32 KB L1.5 instruction cache) spent 41 % of its issue slots
// waiting for instructions (profiles/r1f_*). Hence: rolled loops with register rotation instead of unrolled
// pipelines, ONE copy of every step shared by all passes (__noinline__ functions whose arguments are register
// values or pointers into shared memory), table-driven prologues.
//
// Arithmetic restated from agents/nets.py:66-92 (Linear -> LayerNorm -> ReLU twice, then head).
#pragma once
#include <cooperative_groups.h>

#include "common.cuh"

namespace b2rl {
namespace cg = cooperative_groups;

// ---- network descriptors -----------------------------------------------------------------------------------------
// Tensor pointers in the field order of b2rl_net_t (w1t b1 g1 be1 w2t b2 g2 be2 w3 b3 w2n), so that layer 1 / 2
// tensors are p[F_x1 + 4 * layer]. The small tensors may point into shared memory (NetStage). A Net lives in
// shared memory: the shared __noinline__ steps take it by pointer.
enum { F_W1T, F_B1, F_G1, F_BE1, F_W2T, F_B2, F_G2, F_BE2, F_W3, F_B3, F_W2N, F_N };
struct Net {
  const float* p[F_N];
  const float* w1s;  // this CTA's column slice of w1t staged in shared memory ([in_dim][128]), or null
  const float* w1s_hi;  // a full-width pass (trunk_fwd_full): columns [128, 256) of w1t, staged likewise, or null
  int in_dim, out_dim, ln, pad;
};

// ---- asynchronous copies (LDGSTS): fire-and-forget, so a whole burst costs one L2 round trip ------------------
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)),
               "l"(gsrc)
               : "memory");
}
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)),
               "l"(gsrc)
               : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
  asm volatile("cp.async.commit_group;\n cp.async.wait_group 0;" ::: "memory");
}

// Everything of a network that the row-wise steps and the head touch (biases, LayerNorm affine, head weights,
// and the first layer's weight slice when that layer is narrow), copied once into shared memory at kernel start.
constexpr int W3_ROWS = 8;    // head rows staged (a wider head is read from global memory)
constexpr int W1S_ROWS = 32;  // first layers up to this many inputs are staged
struct NetStage {
  float vec[6][HID];          // b1 g1 be1 b2 g2 be2
  float b3[MAX_OUT];
  float w3[W3_ROWS * HID];
  float w1s[W1S_ROWS * CW];   // [in_dim][128]
};
// One warp's prologue job (lane = threadIdx.x & 31): copy the network's small tensors into `st` (cp.async, waited for
// by the caller), leave the descriptor in `out`. __noinline__: one copy of this code serves every network of a kernel
// (different warps, different arguments).
// This job is the critical path of the prologue: every other warp's job is done ~2 000 cycles after kernel start and the
// whole CTA waits for this one at the staging barrier. Measured with the in-kernel clock (tools/phase_timing.py; cycles
// after kernel start at which the data had landed): rolled loops that index the offsets from the parameter block in
// every iteration (a dependent ~130-cycle parameter load each) 5 500; THIS version, every offset loaded once up front,
// 3 650; and, no better, so not kept: cp.async.bulk with one copy per lane 3 630 or all from one lane 4 080 (~190
// cycles per bulk copy: too many small pieces for the TMA engine), ~40 unrolled LDG.128 + STS.128 3 650, offsets
// passed by shuffle + fully rolled loops 3 500-4 300. The three networks' 45 KB per CTA (5.8 MB per launch) from L2 and
// ~90 LDGSTS per SM set the floor, not the mechanism.
// The first layer's slice [j0, j0 + 128) goes to st->w1s; with w1s_hi (j0 = 0, a network run at full width by one CTA)
// columns [128, 256) go there as well; j0 < 0 stages no first-layer weights (a network this CTA never runs forward).
static __device__ __noinline__ void stage_net(const float* region, const b2rl_net_t* d, NetStage* st, Net* out, int j0,
                                              float* w1s_hi = nullptr) {
  const int lane = threadIdx.x & 31;
  const int64_t* offs = &d->w1t;
  int64_t o[F_N];
#pragma unroll
  for (int f = 0; f < F_N; ++f) o[f] = offs[f];
  const int in_dim = d->in_dim, out_dim = d->out_dim;
  const bool ln = d->layer_norm != 0;
  const bool w3s = out_dim <= W3_ROWS, w1s = in_dim <= W1S_ROWS && j0 >= 0;
  if (lane < F_N) {
    const float* ptr = region + offs[lane];
    const int v = lane - 1 - (lane > 4);  // b1 g1 be1 -> 0 1 2, b2 g2 be2 -> 3 4 5
    if (lane >= F_B1 && lane <= F_BE2 && lane != F_W2T && (ln || lane == F_B1 || lane == F_B2)) ptr = st->vec[v];
    if (lane == F_B3) ptr = st->b3;
    if (lane == F_W3 && w3s) ptr = st->w3;
    out->p[lane] = ptr;
  }
  if (lane == F_N) {
    out->in_dim = in_dim; out->out_dim = out_dim; out->ln = d->layer_norm;
    out->w1s = w1s ? st->w1s : nullptr;
    out->w1s_hi = w1s ? w1s_hi : nullptr;
  }
  if (w1s) {  // the first layer's column slice first (the first product needs it): 512 contiguous bytes per input feature
    const float* w1 = region + o[F_W1T] + j0 + 4 * lane;
#pragma unroll 4
    for (int k = 0; k < in_dim; ++k) cp_async16(st->w1s + k * CW + 4 * lane, w1 + (size_t)k * HID);
    if (w1s_hi) {
#pragma unroll 4
      for (int k = 0; k < in_dim; ++k) cp_async16(w1s_hi + k * CW + 4 * lane, w1 + CW + (size_t)k * HID);
    }
  }
#pragma unroll
  for (int v = 0; v < 6; ++v) {  // 64 float4 per vector: two per lane
    if (ln || v == 0 || v == 3) {
      const float* src = region + o[v + 1 + (v > 2)] + 4 * lane;
      cp_async16(&st->vec[v][4 * lane], src);
      cp_async16(&st->vec[v][4 * lane + 128], src + 128);
    }
  }
  if (lane < (out_dim + 3) / 4) cp_async16(st->b3 + 4 * lane, region + o[F_B3] + 4 * lane);
  if (w3s) {
    const float* w3 = region + o[F_W3] + 4 * lane;
#pragma unroll 2
    for (int i = 0; i < out_dim * (HID / 128); ++i) cp_async16(st->w3 + 4 * lane + 128 * i, w3 + 128 * i);
  }
}

// ---- layouts in shared memory -------------------------------------------------------------------------------
// Operand tile ("T-layout"): float4 T[q * ld + k] holds feature k of rows 4q..4q+3 (q < RQ = 2). The product reads
// it as a broadcast, the row-wise steps write it with consecutive threads on consecutive k.
// Z-layout: float Z[r * HID + j], row-major: what the exchange fills and the row statistics read.
struct Acts {          // what one forward pass leaves behind for its backward pass, per layer
  float4 xh[2][RQ * HID];  // LayerNorm x-hat (or the pre-activation when layer_norm is off)
  float2 st[2][RT];        // per row (mean, rstd)
};
struct Work {          // per-CTA scratch shared by all passes
  float red[KS * RT * CW];    // split-K partial sums [k-slice][row][col] (32 KB); the backward pass also uses it as
                              // row-wise scratch: [0,8K) dx, [8K,16K) dx*xhat, [16K,24K) the incoming dh (Z-layout)
  float z[2][RT * HID];       // exchange targets (double buffered: the peer may run one layer ahead)
  float4 h[2][RQ * HID];      // operand tiles: h1 / h2 of the running pass, dz tiles of the backward pass
  float4 u[RQ * MAX_OUT];     // head outputs / small row-dot results: u[q * MAX_OUT + o]
  float4 du[RQ * MAX_OUT];
  float2 stat[RT];
  uint64_t mbar[2];           // one mbarrier per z buffer: the peer's slice has landed (st.async complete_tx)
  uint64_t xbar[2];           // cross-group exchanges of the kernels (twin Q values, dQ/da), each used once
};
constexpr int DH_OFF = 2 * RT * HID;  // float offset of the incoming-gradient tile inside Work::red

struct Group {  // the CS CTAs that share 8 rows of one network
  int c;        // this CTA's column slice
  int base;     // cluster rank of slice 0
};
constexpr int ALL_COLS = -1;  // Group::c of a CTA that runs a network alone (trunk_fwd_full): it owns every column

// ---- the products: red[w][r][j] = sum_{k in slice(w)} W[k][j0 + j] * X[r][k],  r < 8, j < 128 --------------------
// W is [K][256] row-major (w1t / w2t for the forward pass, w2n for dX). Warp w owns a contiguous slice of K;
// lane l owns columns j0+4l..+3 for all 8 rows: per k one 128-bit load of weights (512 contiguous bytes per warp),
// two broadcast LDS.128 of the rows' activations, 16 FFMA2.
__device__ __forceinline__ void ffma2(float2& d, float w, const float2 x) {
  float2 ww = make_float2(w, w);  // (ptxas folds the duplicate into FFMA2's scalar-broadcast operand form)
  asm("fma.rn.f32x2 %0, %1, %2, %0;"
      : "+l"(*reinterpret_cast<unsigned long long*>(&d))
      : "l"(*reinterpret_cast<unsigned long long*>(&ww)), "l"(*reinterpret_cast<const unsigned long long*>(&x)));
}
__device__ __forceinline__ void fma_k(float2 (&acc)[4][4], const float4 wv, const float4 x0, const float4 x1) {
  const float2 p0 = make_float2(x0.x, x0.y), p1 = make_float2(x0.z, x0.w);
  const float2 p2 = make_float2(x1.x, x1.y), p3 = make_float2(x1.z, x1.w);
  ffma2(acc[0][0], wv.x, p0); ffma2(acc[0][1], wv.x, p1); ffma2(acc[0][2], wv.x, p2); ffma2(acc[0][3], wv.x, p3);
  ffma2(acc[1][0], wv.y, p0); ffma2(acc[1][1], wv.y, p1); ffma2(acc[1][2], wv.y, p2); ffma2(acc[1][3], wv.y, p3);
  ffma2(acc[2][0], wv.z, p0); ffma2(acc[2][1], wv.z, p1); ffma2(acc[2][2], wv.z, p2); ffma2(acc[2][3], wv.z, p3);
  ffma2(acc[3][0], wv.w, p0); ffma2(acc[3][1], wv.w, p1); ffma2(acc[3][2], wv.w, p2); ffma2(acc[3][3], wv.w, p3);
}
__device__ __forceinline__ void zero_acc(float2 (&acc)[4][4]) {
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int p = 0; p < 4; ++p) acc[i][p] = make_float2(0.f, 0.f);
}
__device__ __forceinline__ void store_partials(const float2 (&acc)[4][4], float* __restrict__ red) {
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  float* rp = red + (size_t)(w * RT) * CW + 4 * l;
#pragma unroll
  for (int p = 0; p < 4; ++p) {
    *reinterpret_cast<float4*>(rp + (2 * p) * CW) = make_float4(acc[0][p].x, acc[1][p].x, acc[2][p].x, acc[3][p].x);
    *reinterpret_cast<float4*>(rp + (2 * p + 1) * CW) = make_float4(acc[0][p].y, acc[1][p].y, acc[2][p].y, acc[3][p].y);
  }
}

// Hidden (256-deep) layers: warp w multiplies k in [32w, 32w+32) as 8 groups of 4 k through four register sets
// that rotate WITHOUT register moves (a move of a register with a load in flight waits for the load, which would
// collapse the pipeline to one group): the loop body handles 4 groups, each set is reloaded right after its
// multiplies and used again 4 groups later, so 3 groups (12 k, ~190 FFMA2 per thread) are always in flight.
// hidden_prefetch requests groups 0..2; the caller puts independent work — the previous layer's exchange and
// row-wise step — between it and hidden_fma, hiding the first L2 round trip. hidden_fma's body is ~5 KB of SASS
// executed twice (it fits the 6 KB L0 instruction cache).
constexpr int KW = HID / KS;  // k per warp (32)
struct WPipe {
  float4 s[4][4];  // [set][k in group]
};
__device__ __forceinline__ const float* hidden_wptr(const float* __restrict__ W, int j0) {
  return W + (size_t)((threadIdx.x >> 5) * KW) * HID + j0 + 4 * (threadIdx.x & 31);
}
__device__ __forceinline__ void load_group(float4 (&set)[4], const float* wp, int g) {
  const int gc = min(g, KW / 4 - 1);  // (past the end: re-request the last group — no branch, no overrun)
#pragma unroll
  for (int u = 0; u < 4; ++u) set[u] = ldg4(wp + (size_t)(4 * gc + u) * HID);
}
__device__ __forceinline__ void hidden_prefetch(const float* __restrict__ W, int j0, WPipe& P) {
  const float* wp = hidden_wptr(W, j0);
  load_group(P.s[0], wp, 0);
  load_group(P.s[1], wp, 1);
  load_group(P.s[2], wp, 2);
}
__device__ __forceinline__ void fma_group(float2 (&acc)[4][4], const float4 (&set)[4], const float4* xa, const float4* xb, int g) {
#pragma unroll
  for (int u = 0; u < 4; ++u) fma_k(acc, set[u], xa[4 * g + u], xb[4 * g + u]);
}
__device__ __forceinline__ void hidden_fma(const float* __restrict__ W, int j0, WPipe& P, const float4* __restrict__ X,
                                           float* __restrict__ red) {
  const float* wp = hidden_wptr(W, j0);
  const float4* xa = X + (threadIdx.x >> 5) * KW;
  const float4* xb = xa + HID;
  float2 acc[4][4];  // [col][row pair]
  zero_acc(acc);
#pragma unroll 1
  for (int g = 0; g < KW / 4; g += 4) {
    load_group(P.s[3], wp, g + 3);
    fma_group(acc, P.s[0], xa, xb, g);
    load_group(P.s[0], wp, g + 4);
    fma_group(acc, P.s[1], xa, xb, g + 1);
    load_group(P.s[1], wp, g + 5);
    fma_group(acc, P.s[2], xa, xb, g + 2);
    load_group(P.s[2], wp, g + 6);
    fma_group(acc, P.s[3], xa, xb, g + 3);
  }
  store_partials(acc, red);
}

// First layers whose weight slice waits in shared memory (K = O or O + A <= 32): a rolled loop, 3 LDS + 16 FFMA2 per k.
__device__ __forceinline__ void first_smem(const float* __restrict__ Ws, int K, const float4* __restrict__ X, int ldx,
                                           float* __restrict__ red) {
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  const int ks = (K + KS - 1) / KS;
  const int k0 = min(K, w * ks), k1 = min(K, k0 + ks);
  float2 acc[4][4];
  zero_acc(acc);
#pragma unroll 1
  for (int k = k0; k < k1; ++k)
    fma_k(acc, *reinterpret_cast<const float4*>(Ws + k * CW + 4 * l), X[k], X[ldx + k]);
  store_partials(acc, red);
}
// First layers read from global memory (any K; Humanoid: 376 / 393): the hidden layers' four-set register rotation
// (three groups of 4 k always in flight, no register moves) over this warp's slice of K. The slice is padded to a whole
// number of 4-group trips: padded k re-request the slice's last weight row (an L1 hit) and multiply x = 0. (The first
// version — chunks of 8 k, two chunks in flight — ran the same bytes 1.3-1.6x slower than the hidden layers' pipeline:
// 8-10 k cycles per Humanoid first layer, 35 % of its critic kernel.)
static __device__ __noinline__ void first_global(const float* __restrict__ W, int K, const float4* __restrict__ X, int ldx,
                                                 int j0, float* __restrict__ red) {
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  float2 acc[4][4];
  zero_acc(acc);
  const int ks = (K + KS - 1) / KS;
  const int k0 = min(K, w * ks), n = min(K, k0 + ks) - k0;
  if (n > 0) {
    const float* wp = W + (size_t)k0 * HID + j0 + 4 * l;
    const float4* xa = X + k0;
    const float4* xb = xa + ldx;
    const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
    const int ng = (n + 3) >> 2;  // groups of 4 k
    float4 s0[4], s1[4], s2[4], s3[4];
#define B2RL_LOADG(set, g) \
  _Pragma("unroll") for (int u = 0; u < 4; ++u) set[u] = ldg4(wp + (size_t)min(4 * (g) + u, n - 1) * HID);
#define B2RL_FMAG(set, g)                                          \
  _Pragma("unroll") for (int u = 0; u < 4; ++u) {                  \
    const int kk = 4 * (g) + u;                                    \
    const int kc = min(kk, n - 1);                                 \
    const bool on = kk < n;                                        \
    fma_k(acc, set[u], on ? xa[kc] : zero, on ? xb[kc] : zero);    \
  }
    B2RL_LOADG(s0, 0)
    B2RL_LOADG(s1, 1)
    B2RL_LOADG(s2, 2)
#pragma unroll 1
    for (int g = 0; g < ng; g += 4) {
      B2RL_LOADG(s3, g + 3)
      B2RL_FMAG(s0, g)
      B2RL_LOADG(s0, g + 4)
      B2RL_FMAG(s1, g + 1)
      B2RL_LOADG(s1, g + 5)
      B2RL_FMAG(s2, g + 2)
      B2RL_LOADG(s2, g + 6)
      B2RL_FMAG(s3, g + 3)
    }
#undef B2RL_LOADG
#undef B2RL_FMAG
  }
  store_partials(acc, red);
}

// ---- mbarrier / st.async plumbing (PTX ISA: mbarrier, st.async; SASS: SYNCS.*, STAS) ------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* b, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect(uint64_t* b, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* b, uint32_t parity) {
  asm volatile(
      "{\n .reg .pred p;\n WAIT_%=:\n mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n @p bra DONE_%=;\n bra WAIT_%=;\n DONE_%=:\n}" ::"r"(
          smem_u32(b)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ uint32_t map_peer(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void st_async_v4(uint32_t raddr, float4 v, uint32_t rmbar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.f32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(raddr),
               "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "r"(rmbar)
               : "memory");
}
__device__ __forceinline__ void st_async_f32(uint32_t raddr, float v, uint32_t rmbar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.f32 [%0], %1, [%2];" ::"r"(raddr), "f"(v), "r"(rmbar)
               : "memory");
}
// Once per kernel, before the first exchange: the mbarriers armed for one arrival (thread 0's expect_tx) per
// phase, made visible to the peers, and one cluster barrier so that no st.async can reach an uninitialised
// barrier. The barrier is split: arrive first thing in the kernel, wait just before the first exchange (inside
// reduce_gather), by when every CTA of the cluster has long arrived.
__device__ __forceinline__ void exchange_init_arrive(Work& S) {
  if (threadIdx.x == 0) {
    mbar_init(&S.mbar[0], 1);
    mbar_init(&S.mbar[1], 1);
    mbar_init(&S.xbar[0], 1);
    mbar_init(&S.xbar[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory");  // (the init fence above is the release)
}
__device__ __forceinline__ void exchange_init_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }

// ---- split-K reduction (fixed order) + bias ----------------------------------------------------------------------
// Thread t: row t >> 5, columns j0 + 4 (t & 31)..+3, summed over the k-slices in a fixed order, plus the bias.
__device__ __forceinline__ float4 reduce_slice(const Work& S, int j0, const float* __restrict__ bias) {
  const int t = threadIdx.x, r = t >> 5, cq = t & 31;
  const float* rp = S.red + (size_t)r * CW + 4 * cq;
  float4 s = *reinterpret_cast<const float4*>(rp);
#pragma unroll
  for (int w = 1; w < KS; ++w) {
    const float4 v = *reinterpret_cast<const float4*>(rp + (size_t)w * RT * CW);
    s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
  }
  if (bias) {
    const float4 bv = *reinterpret_cast<const float4*>(bias + j0 + 4 * cq);
    s.x += bv.x; s.y += bv.y; s.z += bv.z; s.w += bv.w;
  }
  return s;
}

// ---- split-K reduction + exchange of this CTA's 8x128 slice with the peer ----------------------------------------
// Thread (r = t >> 5, cq = t & 31) owns row r, columns j0+4cq..+3. Its float4 goes to the local z buffer with a
// plain store and to the peer's with st.async, which also counts 16 bytes on the PEER's mbarrier; thread 0 has
// armed this CTA's mbarrier for the 4096 bytes the peer will send. No cluster barrier and no memory fence: each
// CTA waits for exactly the data it needs. Returns the buffer that then holds the full 8x256 tile. `gi` counts
// the exchanges (every thread of the cluster advances it in step): buffer gi & 1, mbarrier phase parity
// (gi >> 1) & 1. Two buffers are enough because the peer can run at most one layer ahead — it needs this CTA's
// slice for the layer after, and this CTA sends that only after it has finished reading the current buffer.
__device__ __forceinline__ const float* reduce_gather(const Group G, Work& S, int& gi, const float* __restrict__ bias) {
  const int t = threadIdx.x, r = t >> 5, cq = t & 31, j = G.c * CW + 4 * cq;
  const int b = gi & 1;
  if (t == 0) mbar_expect(&S.mbar[b], RT * CW * sizeof(float));
  const float4 s = reduce_slice(S, G.c * CW, bias);
  float* zl = S.z[b];
  float* dst = zl + (size_t)r * HID + j;
  *reinterpret_cast<float4*>(dst) = s;
  if (gi == 0) exchange_init_wait();  // first remote access of the kernel: the peers' mbarriers are initialised
  const uint32_t peer = (uint32_t)(G.base + (G.c ^ 1));
  st_async_v4(map_peer(smem_u32(dst), peer), s, map_peer(smem_u32(&S.mbar[b]), peer));
  __syncthreads();                           // this CTA's slice is visible to all its threads
  mbar_wait(&S.mbar[b], (gi >> 1) & 1);      // the peer's slice has landed
  ++gi;
  return zl;
}

// ---- row statistics: warp w reduces row w of a [8][256] buffer ---------------------------------------------------
__device__ __forceinline__ void row_stats(const float* za, const float* zb, float2* out, bool layernorm_stats) {
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  float v[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = za[w * HID + l + 32 * i];
  float s = ((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]));
  if (layernorm_stats) {  // (mean, rstd) with the biased variance taken around the mean (two-pass)
    s = warp_sum(s);
    const float mean = s * (1.0f / HID);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) { const float d = v[i] - mean; q = fmaf(d, d, q); }
    q = warp_sum(q);
    if (l == 0) out[w] = make_float2(mean, 1.0f / sqrtf(q * (1.0f / HID) + LN_EPS));
  } else {  // two plain means (LayerNorm backward: mean(dx), mean(dx * xhat))
    float u[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) u[i] = zb[w * HID + l + 32 * i];
    float s2 = ((u[0] + u[1]) + (u[2] + u[3])) + ((u[4] + u[5]) + (u[6] + u[7]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {  // the two reductions interleaved (independent shuffle chains)
      s += __shfl_xor_sync(0xffffffffu, s, o);
      s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    }
    if (l == 0) out[w] = make_float2(s * (1.0f / HID), s2 * (1.0f / HID));
  }
}

// ---- forward row-wise step of one layer: LayerNorm, ReLU on the gathered 8x256 tile (thread <-> column) ---------
// Writes the next operand tile hT, keeps x-hat in xhT (if non-null) and the statistics in stat_keep, and stores
// this CTA's column slice of h to the workspace (for wgrad.cu) when ws_h != NULL. Ends with __syncthreads.
__device__ __forceinline__ void layer_fwd_rows(const float* __restrict__ z, const float* __restrict__ g,
                                               const float* __restrict__ be, bool ln, Work& S, float4* hT, float4* xhT,
                                               float2* stat_keep, float* ws_h, int b0, int nvalid, const Group G, int tk) {
  const int t = threadIdx.x, j = t;
  float gj = 1.f, bej = 0.f;
  float zc[RT];  // this thread's column, requested before the statistics so that its latency hides behind them
#pragma unroll
  for (int r = 0; r < RT; ++r) zc[r] = z[r * HID + j];
  if (ln) {
    gj = g[j];
    bej = be[j];
    row_stats(z, z, S.stat, true);
    __syncthreads();
    B2RL_TICK(tk);
    if (stat_keep && t < RT) stat_keep[t] = S.stat[t];
  }
  const bool mine = ws_h && (G.c == ALL_COLS || (j >> 7) == G.c);
#pragma unroll
  for (int q = 0; q < RQ; ++q) {
    float xh[4], h[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = 4 * q + i;
      const float zv = zc[r];
      if (ln) {
        const float2 s = S.stat[r];
        xh[i] = (zv - s.x) * s.y;
        h[i] = fmaxf(fmaf(xh[i], gj, bej), 0.f);
      } else {
        xh[i] = zv;
        h[i] = fmaxf(zv, 0.f);
      }
      if (mine && r < nvalid) ws_h[(size_t)(b0 + r) * HID + j] = h[i];
    }
    hT[q * HID + j] = make_float4(h[0], h[1], h[2], h[3]);
    if (xhT) xhT[q * HID + j] = make_float4(xh[0], xh[1], xh[2], xh[3]);
  }
  __syncthreads();
}

// ---- backward row-wise step of one layer: ReLU mask, LayerNorm backward (thread <-> column, all 8 rows) ---------
// dh[r]: gradient w.r.t. the post-ReLU activation of column j. Leaves dz (w.r.t. the Linear output) in dh and
// writes this CTA's slice of the column sums {sum_r dz, sum_r dn*xhat, sum_r dn} (d bias, d ln.weight, d ln.bias)
// to part3[0..2][j]. Uses S.red[0, 16K) as scratch. Rows beyond the batch carry dh = 0 and stay 0.
__device__ __forceinline__ void layer_bwd_rows(float (&dh)[RT], const float4* xhT, const float2* stat,
                                               const float* __restrict__ g, const float* __restrict__ be, bool ln,
                                               Work& S, float* part3, const Group G) {
  const int t = threadIdx.x, j = t;
  float xh[RT], dn[RT];
  const float gj = ln ? g[j] : 1.f, bej = ln ? be[j] : 0.f;
  float* s1 = S.red;
  float* s2 = S.red + RT * HID;
#pragma unroll
  for (int q = 0; q < RQ; ++q) {
    const float4 x4 = xhT[q * HID + j];
    xh[4 * q] = x4.x; xh[4 * q + 1] = x4.y; xh[4 * q + 2] = x4.z; xh[4 * q + 3] = x4.w;
  }
#pragma unroll
  for (int r = 0; r < RT; ++r) {
    const bool on = ln ? (fmaf(xh[r], gj, bej) > 0.f) : (xh[r] > 0.f);  // the forward ReLU(h) > 0, recomputed bit-exactly
    dn[r] = on ? dh[r] : 0.f;
    if (ln) {
      const float dx = dn[r] * gj;
      s1[r * HID + j] = dx;
      s2[r * HID + j] = dx * xh[r];
    }
  }
  if (ln) {
    __syncthreads();
    row_stats(s1, s2, S.stat, false);
    __syncthreads();
#pragma unroll
    for (int r = 0; r < RT; ++r) {
      const float2 c = S.stat[r];
      dh[r] = stat[r].y * (dn[r] * gj - c.x - xh[r] * c.y);
    }
  } else {
#pragma unroll
    for (int r = 0; r < RT; ++r) dh[r] = dn[r];
  }
  if (part3 && (j >> 7) == G.c) {
    float a = 0.f, b = 0.f, c = 0.f;
#pragma unroll
    for (int r = 0; r < RT; ++r) {
      a += dh[r];
      b += dn[r] * xh[r];
      c += dn[r];
    }
    part3[0 * HID + j] = a;
    if (ln) {
      part3[1 * HID + j] = b;
      part3[2 * HID + j] = c;
    }
  }
}

// ---- small products against [n][256] row-major matrices (global or staged in shared memory) -----------------
// out[q * MAX_OUT + o] (8 rows) = bias[o] + sum_k W[o][k] * X[.][k]: warp w takes outputs w, w+NW, ...; lanes
// stride k. Used for the heads (n = 1, A or 2A) and for dQ/da = dz1 . w1t[O+a][:] in the actor step. Both CTAs of
// a group compute all outputs (each holds the full tile); no exchange.
static __device__ __noinline__ void rowdot(const float* __restrict__ W, const float* __restrict__ bias, int n,
                                           const float4* __restrict__ X, float4* __restrict__ out) {
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
#pragma unroll 1
  for (int o = w; o < n; o += NW) {
    float a[RT], wr[HID / 32];
#pragma unroll
    for (int r = 0; r < RT; ++r) a[r] = 0.f;
#pragma unroll
    for (int i = 0; i < HID / 32; ++i) wr[i] = W[(size_t)o * HID + l + 32 * i];  // one round trip per output row
#pragma unroll
    for (int i = 0; i < HID / 32; ++i) {
      const int k = l + 32 * i;
      const float wv = wr[i];
      const float4 x0 = X[k], x1 = X[HID + k];
      a[0] = fmaf(wv, x0.x, a[0]); a[1] = fmaf(wv, x0.y, a[1]); a[2] = fmaf(wv, x0.z, a[2]); a[3] = fmaf(wv, x0.w, a[3]);
      a[4] = fmaf(wv, x1.x, a[4]); a[5] = fmaf(wv, x1.y, a[5]); a[6] = fmaf(wv, x1.z, a[6]); a[7] = fmaf(wv, x1.w, a[7]);
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1)  // eight independent shuffle chains
#pragma unroll
      for (int r = 0; r < RT; ++r) a[r] += __shfl_xor_sync(0xffffffffu, a[r], s);
    if (l == 0) {
      const float bo = bias ? bias[o] : 0.f;
      out[o] = make_float4(a[0] + bo, a[1] + bo, a[2] + bo, a[3] + bo);
      out[MAX_OUT + o] = make_float4(a[4] + bo, a[5] + bo, a[6] + bo, a[7] + bo);
    }
  }
}

// scalar element (row r, slot o) of a u / du style array
__device__ __forceinline__ float& uref(float4* u, int r, int o) {
  return reinterpret_cast<float*>(&u[(r >> 2) * MAX_OUT + o])[r & 3];
}

// ---- input tiles: X[q * ld + k].(r & 3) = row r, feature off + k, copied asynchronously (cp.async) -----------------
// `myrow` is per LANE: lane i of every calling warp holds the global-memory base of tile row i & 7 (the batch row, or —
// in-kernel sampling — the sampled replay row); rows beyond the batch (r >= nvalid) repeat the last valid row: finite
// values whose results are masked later. Executed by the `nth` threads whose index among them is `tid` (a prologue
// job of some warps): rows over the job's warps, features over the lanes.
static __device__ __noinline__ void stage_tile(const float* myrow, int nvalid, int off, int len, float4* X, int ld, int tid,
                                               int nth) {
  const int lane = tid & 31, nw = nth >> 5;
#pragma unroll 1
  for (int r = tid >> 5; r < RT; r += nw) {
    const int rr = r < nvalid ? r : nvalid - 1;
    const float* src = reinterpret_cast<const float*>(__shfl_sync(0xffffffffu, reinterpret_cast<unsigned long long>(myrow), rr)) + off;
    float* d = reinterpret_cast<float*>(&X[(r >> 2) * ld]) + (r & 3);
#pragma unroll 1
    for (int k = lane; k < len; k += 32) cp_async4(d + 4 * k, src + k);
  }
}
// the per-lane row base for a batch held in rows[.][row_stride]
__device__ __forceinline__ const float* batch_row(const float* rows, int row_stride, int b0, int nvalid) {
  const int r = threadIdx.x & 7;
  return rows + (size_t)(b0 + (r < nvalid ? r : nvalid - 1)) * row_stride;
}

__device__ __forceinline__ void store_tile(float4* T, const float (&v)[RT]) {  // operand tile, column = threadIdx.x
  const int j = threadIdx.x;
#pragma unroll
  for (int q = 0; q < RQ; ++q) T[q * HID + j] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
}
__device__ __forceinline__ void store_slice(float* __restrict__ dst, int b0, int nvalid, const float (&v)[RT],
                                            const Group G) {  // dst [B][256]: this CTA's 128 columns
  const int j = threadIdx.x;
  if ((j >> 7) != G.c) return;
#pragma unroll
  for (int r = 0; r < RT; ++r)
    if (r < nvalid) dst[(size_t)(b0 + r) * HID + j] = v[r];
}

// ---- the two hidden layers, forward. Leaves h2 in S.h[1] (synchronised), x-hat / statistics in `A` if given. -----
// One copy per kernel (__noinline__, every argument a register value, Net and Work in shared memory); the two
// layers share one copy of the exchange and of the row-wise step (rolled loop). Returns the exchange counter.
// WIDE: first layers wider than W1S_ROWS inputs exist (read from global memory by first_global); the narrow
// instantiation does not carry that code (instruction footprint: see the header comment).
template <bool WIDE>
static __device__ __noinline__ int trunk_fwd(const Group G, const Net* np, const float4* __restrict__ X, int ldx,
                                             Acts* A, Work* Sp, int gi, float* ws_h1, float* ws_h2, int b0, int nvalid,
                                             int tk = 54) {
  const Net& n = *np;
  Work& S = *Sp;
  const int j0 = G.c * CW;
  B2RL_TICK(tk + 0);
  if (!WIDE || n.w1s) first_smem(n.w1s, n.in_dim, X, ldx, S.red);
  else first_global(n.p[F_W1T], n.in_dim, X, ldx, j0, S.red);
  WPipe P;  // the second layer's first weight groups: requested now, multiplied after the first layer's exchange
  hidden_prefetch(n.p[F_W2T], j0, P);  // and row-wise step, which hide their L2 latency
  __syncthreads();
  B2RL_TICK(tk + 1);
#pragma unroll 1
  for (int layer = 0; layer < 2; ++layer) {
    if (layer == 1) {
      hidden_fma(n.p[F_W2T], j0, P, S.h[0], S.red);
      __syncthreads();
      B2RL_TICK(tk + 4);
    }
    const float* z = reduce_gather(G, S, gi, n.p[F_B1 + 4 * layer]);
    B2RL_TICK(tk + 2 + 3 * layer);
    layer_fwd_rows(z, n.p[F_G1 + 4 * layer], n.p[F_BE1 + 4 * layer], n.ln != 0, S, S.h[layer], A ? A->xh[layer] : nullptr,
                   A ? A->st[layer] : nullptr, layer ? ws_h2 : ws_h1, b0, nvalid, G, tk + 7);
    B2RL_TICK(tk + 3 + 3 * layer);
  }
  return gi;
}

// ---- the two hidden layers, forward, all 256 columns by this CTA alone (no exchange) --------------------------------
// For a CTA that runs a whole network pass while its peer runs another one (critic.cu, first pass). Each layer's
// product is trunk_fwd's two column slices one after the other — the same calls with j0 = 0 and then j0 = 128, each
// followed by the same fixed-order reduction — so every element is bit-identical to the split pass; the local
// reduction fills the Z buffer that the exchange fills there. The next product's first weight groups are requested
// before each reduction (and before the row-wise step). Only S.z[1] is used: the peer's first exchange after this pass
// targets S.z[0] and may land while this pass still runs. Leaves h2 in S.h[1] (synchronised), x-hat / statistics in
// `A` if given, and stores all 256 columns of h1 / h2 to the workspace when ws_h1 / ws_h2 are given. Touches no
// mbarrier: the exchange counter of trunk_fwd / trunk_bwd is unaffected.
template <bool WIDE>
static __device__ __noinline__ void trunk_fwd_full(const Net* np, const float4* __restrict__ X, int ldx, Acts* A, Work* Sp,
                                                   float* ws_h1, float* ws_h2, int b0, int nvalid, int tk) {
  const Net& n = *np;
  Work& S = *Sp;
  float* z = S.z[1];
  WPipe P;
  B2RL_TICK2(tk + 0);
#pragma unroll 1
  for (int layer = 0; layer < 2; ++layer) {
#pragma unroll 1
    for (int h = 0; h < CS; ++h) {
      const int j0 = h * CW;
      if (layer == 0) {
        if (!WIDE || n.w1s) first_smem(h ? n.w1s_hi : n.w1s, n.in_dim, X, ldx, S.red);
        else first_global(n.p[F_W1T], n.in_dim, X, ldx, j0, S.red);
        if (h == CS - 1) hidden_prefetch(n.p[F_W2T], 0, P);  // (not before: first_global is a call)
      } else {
        hidden_fma(n.p[F_W2T], j0, P, S.h[0], S.red);
        if (h == 0) hidden_prefetch(n.p[F_W2T], CW, P);
      }
      __syncthreads();
      const float4 v = reduce_slice(S, j0, n.p[F_B1 + 4 * layer]);
      *reinterpret_cast<float4*>(z + (threadIdx.x >> 5) * HID + j0 + 4 * (threadIdx.x & 31)) = v;
      __syncthreads();  // S.red is free for the next product; after the last slice, z holds the full tile
    }
    B2RL_TICK2(tk + 2 + 3 * layer);
    layer_fwd_rows(z, n.p[F_G1 + 4 * layer], n.p[F_BE1 + 4 * layer], n.ln != 0, S, S.h[layer], A ? A->xh[layer] : nullptr,
                   A ? A->st[layer] : nullptr, layer ? ws_h2 : ws_h1, b0, nvalid, Group{ALL_COLS, 0}, tk + 7);
    B2RL_TICK2(tk + 3 + 3 * layer);
  }
}

// ---- the two hidden layers, backward (dX path) ----------------------------------------------------------------------
// In: the gradient w.r.t. h2 as a Z-layout tile at S.red + DH_OFF (written by the caller; thread j wrote column j).
// Writes this CTA's slices of dz2/dz1 to the workspace (for wgrad.cu) and of the column partial sums when the
// pointers are non-null. On return S.h[1] holds the dz1 tile (synchronised). Same conventions as trunk_fwd.
static __device__ __noinline__ int trunk_bwd(const Group G, const Net* np, const Acts* A, Work* Sp, int gi, float* ws_dz1,
                                             float* ws_dz2, float* part, int b0, int nvalid) {
  const Net& n = *np;
  Work& S = *Sp;
  const int j = threadIdx.x, j0 = G.c * CW;
  WPipe P;
  hidden_prefetch(n.p[F_W2N], j0, P);  // in flight during the row-wise step below
  const float* src = S.red + DH_OFF;
#pragma unroll 1
  for (int layer = 1; layer >= 0; --layer) {
    float dh[RT];
#pragma unroll
    for (int r = 0; r < RT; ++r) dh[r] = src[r * HID + j];
    layer_bwd_rows(dh, A->xh[layer], A->st[layer], n.p[F_G1 + 4 * layer], n.p[F_BE1 + 4 * layer], n.ln != 0, S,
                   part ? part + 3 * HID * layer : nullptr, G);
    store_tile(S.h[1 - layer], dh);
    float* ws = layer ? ws_dz2 : ws_dz1;
    if (ws) store_slice(ws, b0, nvalid, dh, G);
    __syncthreads();
    if (layer == 1) {
      hidden_fma(n.p[F_W2N], j0, P, S.h[0], S.red);
      __syncthreads();
      src = reduce_gather(G, S, gi, nullptr);
    }
  }
  return gi;
}

}  // namespace b2rl
