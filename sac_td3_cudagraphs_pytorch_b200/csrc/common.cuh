// common.cuh — shared device helpers for libb2rl (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "../../include/b2rl.h"

namespace b2rl {

constexpr int HID = B2RL_HID;    // 256
constexpr int RT = B2RL_ROWS;    // batch rows per CTA group of the fused kernels (8)
constexpr int RQ = RT / 4;       // row quads: row tiles are stored as float4 (one float per batch row of a quad)
constexpr int CS = 2;            // CTAs per group: each computes HID / CS output columns of every layer
constexpr int CW = HID / CS;     // 128
constexpr int NT = HID;          // threads per CTA in the fused kernels: thread t <-> hidden unit t in the row-wise steps
constexpr int NW = NT / 32;
constexpr int KS = NW;           // product k-slices: one per warp
constexpr int MAX_OUT = B2RL_MAX_OUT;
constexpr float LN_EPS = 1e-5f;  // torch.nn.LayerNorm default (agents/nets.py:70)

static_assert(RT == 8 && NT == 256 && CS == 2, "thread mappings of mlp_cluster.cuh");
__host__ __device__ inline int row_blocks(int B) { return (B + RT - 1) / RT; }

// workspace layout per agent (floats); `slot` = 0/1 for the twin critics, 0 for the actor
//   H1, H2, DZ1, DZ2 : [2][B][256]   DZ3 : [2][B][MAX_OUT]   PART : [2][ceil(B/8)][PART_LEN]
constexpr int PART_VEC = 6;                               // db1 dg1 dbe1 db2 dg2 dbe2
constexpr int PART_LEN = PART_VEC * HID + MAX_OUT + 8;    // + db3[MAX_OUT] + {loss terms}
constexpr int PART_DB3 = PART_VEC * HID;
constexpr int PART_SCAL = PART_VEC * HID + MAX_OUT;       // [0] sum sq err / actor loss, [1] logpi sum, ...

struct Workspace {
  float *h1, *h2, *dz1, *dz2, *dz3, *part;
};
__host__ __device__ inline int64_t ws_floats(int B) {
  return (int64_t)2 * B * HID * 4 + (int64_t)2 * B * MAX_OUT + (int64_t)2 * row_blocks(B) * PART_LEN;
}
__host__ __device__ inline Workspace ws_carve(float* base, int B, int slot) {
  Workspace w;
  const int64_t bh = (int64_t)B * HID;
  w.h1 = base + (0 * 2 + slot) * bh;
  w.h2 = base + (1 * 2 + slot) * bh;
  w.dz1 = base + (2 * 2 + slot) * bh;
  w.dz2 = base + (3 * 2 + slot) * bh;
  float* p = base + 8 * bh;
  w.dz3 = p + (int64_t)slot * B * MAX_OUT;
  p += (int64_t)2 * B * MAX_OUT;
  w.part = p + (int64_t)slot * row_blocks(B) * PART_LEN;
  return w;
}

// ---- optional in-kernel phase timing (build with B2RL_EXTRA_NVCC_FLAGS=-DB2RL_TIMING; tools/phase_timing.py)
#ifdef B2RL_TIMING
static __device__ long long g_b2rl_timing[64];  // one copy per translation unit
#define B2RL_TICK(slot)                                                                    \
  do {                                                                                     \
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) g_b2rl_timing[slot] = clock64(); \
  } while (0)
#else
#define B2RL_TICK(slot) do {} while (0)
#endif

// ---- cluster launches ----------------------------------------------------------------------------------------
constexpr int MAX_DYN_SMEM = 232448;  // 227 KB: the opt-in dynamic shared memory limit of sm_100

// Every kernel of the update is launched with programmatic stream serialisation (programmatic dependent launch):
// it calls pdl_enter() first thing, which (1) lets the NEXT kernel in the stream begin launching — its CTAs are
// then resident and parked when this grid drains, instead of paying the launch latency after it — and (2) waits
// until the PREVIOUS grid has completed and its writes are visible. Nothing is read or written before the wait,
// so the data dependences are exactly those of plain stream order; inside a captured graph the edges become
// programmatic dependencies. Measured (B200, batch 256): 0.3-1 us less per kernel, except the weight-gradient kernel
// (300 small CTAs), which loses 1.5 us when its successor's CTAs are parked beside it — so that one is launched
// plainly. B2RL_PDL=0 in the environment turns the attribute off everywhere (A/B measurements).
__device__ __forceinline__ void pdl_enter() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
}
bool pdl_enabled();  // api.cu

// cluster_x < 0: |cluster_x| CTAs per cluster (1 = none) and NO programmatic launch for this kernel
template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, int cluster_x, size_t smem, cudaStream_t st,
                            Args&&... args) {
  const bool pdl = cluster_x > 0 && pdl_enabled();
  if (cluster_x < 0) cluster_x = -cluster_x;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[2];
  int n = 0;
  if (cluster_x > 1) {
    at[n].id = cudaLaunchAttributeClusterDimension;
    at[n].val.clusterDim.x = cluster_x;
    at[n].val.clusterDim.y = 1;
    at[n].val.clusterDim.z = 1;
    ++n;
  }
  if (pdl) {
    at[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  cfg.attrs = at;
  cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<Args&&>(args)...);
}
template <typename... KArgs, typename... Args>
inline cudaError_t launch_cluster(void (*kernel)(KArgs...), dim3 grid, int cluster_x, size_t smem, cudaStream_t st,
                                  Args&&... args) {
  return launch_k(kernel, grid, dim3(NT), cluster_x, smem, st, static_cast<Args&&>(args)...);
}

// ---- per-agent hyperparameters (include/b2rl.h b2rl_agent_hp_t): float index of each field in a row
enum AgentHpField { HP_LR = 0 /* + B2RL_CTR_* */, HP_GAMMA = 3, HP_POLYAK, HP_TD3_STD, HP_TD3_C, HP_TARG_ENT, HP_CLIP, HP_EXPLORE };
static_assert(sizeof(b2rl_agent_hp_t) == 64, "one 64-byte row per agent");
static_assert(offsetof(b2rl_agent_hp_t, gamma) == 4 * HP_GAMMA && offsetof(b2rl_agent_hp_t, polyak) == 4 * HP_POLYAK &&
                  offsetof(b2rl_agent_hp_t, td3_std) == 4 * HP_TD3_STD && offsetof(b2rl_agent_hp_t, td3_c) == 4 * HP_TD3_C &&
                  offsetof(b2rl_agent_hp_t, targ_ent) == 4 * HP_TARG_ENT && offsetof(b2rl_agent_hp_t, clip_norm) == 4 * HP_CLIP &&
                  offsetof(b2rl_agent_hp_t, explore_std) == 4 * HP_EXPLORE,
              "AgentHpField follows b2rl_agent_hp_t");
// Agent g's value of one hyperparameter: row g of the launch's table, or — no table — the scalar the launch was given.
// Every kernel that reads a swept value goes through here, once per CTA and ahead of its dependent chain.
__device__ __forceinline__ float agent_hp(const b2rl_agent_hp_t* tab, int g, int field, float scalar) {
  return tab ? __ldg(reinterpret_cast<const float*>(tab + g) + field) : scalar;
}

// stacked agents on the wide path (include/b2rl.h b2rl_stack_t): the device-side copy, n = 1 and zero strides when NULL
struct Stk {
  int n;
  unsigned base;
  long long ps, ls, as, cs, os;  // param / lo / alpha / counters / out strides
  const b2rl_agent_hp_t* hp;     // per-agent hyperparameters or NULL
};
inline Stk make_stk(const b2rl_stack_t* s) {
  Stk k = {1, 0u, 0, 0, 0, 0, 0, nullptr};
  if (s) k = {s->n_agents, (unsigned)s->agent_base, s->param_stride, s->lo_stride, s->alpha_stride, s->counters_stride, s->out_stride,
              s->agent_hp};
  return k;
}

// the job table of wide.cu::wide_colsum_kernel (b2rl_wide_colsum_multi), passed by value
struct ColsumJobs {
  const float* part[8];
  long long off[8][3];
  int ln[8];
  int n;
};

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

// streaming 128-bit load/store that do not allocate in L1 (replay rows are touched once)
__device__ __forceinline__ float4 ld_stream4(const float* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void st_stream4(float* p, float4 v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y),
               "f"(v.z), "f"(v.w));
}

// "lo part" of an fp32 value for the 3xTF32 products: x - (x truncated to TF32's 10 mantissa bits, as the tensor core reads it)
__device__ __forceinline__ float tf32_lo(float x) { return x - __uint_as_float(__float_as_uint(x) & 0xFFFFE000u); }
__device__ __forceinline__ float4 tf32_lo4(float4 x) { return make_float4(tf32_lo(x.x), tf32_lo(x.y), tf32_lo(x.z), tf32_lo(x.w)); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ float f4get(const float4& v, int i) {
  return i == 0 ? v.x : (i == 1 ? v.y : (i == 2 ? v.z : v.w));
}

}  // namespace b2rl
