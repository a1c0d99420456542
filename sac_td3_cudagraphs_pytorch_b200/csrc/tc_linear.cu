// tc_linear.cu — the hidden-layer product for LARGE batches on the 5th-generation tensor cores:
//     Z = X · Wᵀ + b ;  H = ReLU(LayerNorm(Z))        X [M][256], W [256][256] (natural torch layout [out][in])
// agents/nets.py:66-82 (fc_block_2: Linear -> LayerNorm -> ReLU) for M in the tens of thousands (BASELINE.json
// config 5, batch 65 536; stacked populations), where the row-group kernels of mlp_cluster.cuh stream every layer's
// weights from L2 once per 8 rows and top out at ~10 TFLOP/s.
//
// Persistent CTAs (one per SM, clusters of 2) over 128-row tiles, warp-specialised; two TMEM accumulator buffers, so the
// epilogue of one tile overlaps the loads and MMAs of the next:
//   warp 0   TMA producer: cp.async.bulk.tensor loads of the A tile (128 x 32 fp32) and of this CTA's HALF of the weight
//            k-slab (128 x 32 fp32) into a shared-memory ring, 128-byte swizzle, completion on mbarriers. 3xTF32 hidden
//            layers (PAIR): the half stays in this CTA and the two CTAs run 2-SM MMAs; otherwise it is multicast to both
//            CTAs of the cluster (every tile needs the same weights) and a ring slot is reused when BOTH CTAs' MMAs have
//            released it (multicast tcgen05.commit);
//   warp 1   TMEM allocation (2 x 256 columns) and the MMA issuer: one elected thread issues tcgen05.mma kind::tf32
//            (cta_group::1 M=128, or cta_group::2 M=256 from cluster rank 0 on behalf of both SMs; rank 1's warp 1 then
//            relays "my slab has landed"), N=256 K=8, accumulating in TMEM; tcgen05.commit releases each ring slot back to
//            the producer and finally signals the epilogue;
//   warps 2-3 (3xTF32 only) split each arriving activation slab (stacked agents: and weight slab) into its lo part;
//   warps 4.. epilogue, 4 or 8 warps (TcCfg::EPW): thread <-> TMEM lane <-> one output ROW, so bias, the LayerNorm statistics
//            (one shifted pass over the row, no shuffles), affine and ReLU are thread-local; with 8 warps two warps share 32
//            rows, each taking half of the columns and swapping its row sums through shared memory. Per-column vectors sit
//            in shared memory (as global loads they were 1280 exposed L1 round trips per warp and tile: ncu, long
//            scoreboard); rows go to / come from global memory through swizzled 32x32 per-warp tiles that TMA fills
//            (x-hat for the backward epilogue) and TMA stores drain (outputs), or that the warp copies out itself where
//            it has one tile only.
// Operands are fp32 in memory and are read by the tensor core as TF32 (10-bit mantissa, truncated): products carry
// ~1e-3 relative error — the "looser stated bound" of the north star for tensor-core modes; the accumulation, the
// LayerNorm and everything downstream are fp32. Both operands are K-major: X rows and the natural-layout weight
// rows are contiguous along the contraction (the dX product uses the w2t copy the same way).
#include <cuda.h>

#include "common.cuh"

namespace b2rl {

constexpr int TCM = 128, TCN = 256, TCK = 32;
// PREC 0: TF32 products (operands truncated to 10 mantissa bits by the tensor core); ring depths: TcCfg below.
// PREC 1: "3xTF32": x = hi + lo with hi = the TF32 truncation the tensor core applies anyway and lo = x - hi (exact in
//         fp32, re-truncated to TF32: 2^-21 of x); a.b ~ hi.hi + lo.hi + hi.lo, three MMAs into the same accumulator —
//         fp32-level accuracy (~1e-6) from the tensor cores. The weights' lo parts are precomputed (tc_split_lo), the
//         activations' are made in shared memory by two split warps.
// PREC 2: 3xTF32 with the WEIGHTS' lo parts made in shared memory as well (by the same two warps, from the slab TMA has
//         just delivered) instead of being read from a precomputed mirror: for stacked agents every weight slab serves one
//         tile pair only, so a mirror costs as many HBM bytes as the weights themselves (268 MB per launch at 1 024 agents,
//         plus the optimizer's writes to keep it current) while the split costs ~2 us of two idle warps per 15 us tile.
// PAIR (the 3xTF32 hidden layers, forward and backward): the two CTAs of the cluster run ONE tensor-core instruction
// together — tcgen05.mma.cta_group::2, M = 256: CTA r supplies its own 128 rows of A and rows [128r, 128r + 128) of the
// weight slab (its half of N), and receives its own 128 x 256 accumulator tile in its own TMEM. Each CTA then holds (and,
// for stacked agents, splits) only HALF of every weight slab: a stage is 64 KB instead of 96, so the 192 KB ring has three
// stages, and each SM's tensor core reads 8 KB of operands per instruction from its shared memory instead of 12 (three
// products per k-step make the operand reads of the MMAs the largest shared-memory client of the kernel).
template <int MODE, int PREC>
struct TcCfg {
  static constexpr bool PAIR = MODE != 1 && PREC != 0;
  static constexpr int BN = PAIR ? TCN / 2 : TCN;            // weight rows per CTA and stage
  // (the backward kernel is bound by its epilogue: it gives a stage's worth of shared memory to the x-hat rings)
  // (the first layer is one or two k-slabs per tile and all epilogue: a short ring, two epilogue warps per 32 rows)
  static constexpr int STAGES = MODE == 2 ? 2 : MODE == 1 ? (PREC ? 1 : 2) : 3;
  // Epilogue warps: one per 32 accumulator rows (TMEM lanes 32 * (warp % 4) ..); the backward kernel, whose epilogue is
  // instruction-bound (~10 k warp instructions per tile on a lone warp per scheduler: 20 us against 7 us of MMAs), runs two
  // per 32 rows, each on one half of the columns.
  // The 3xTF32 hidden layer keeps one warp per 32 rows: its three 64 KB stages leave room for four staging tiles only,
  // and with a two-stage ring the MMA pipeline, not the epilogue, sets its pace (measured: 59.8 vs 54.3 us per 65 536 rows).
  static constexpr int EPW = (MODE == 0 && PREC != 0) ? 4 : 8;
  static constexpr int THREADS = 128 + 32 * EPW;  // warp 0 TMA, 1 MMA, 2-3 lo split, 4.. epilogue
  static constexpr int NXB = EPW == 8 ? 2 : 1;     // staging tiles per epilogue warp
};
template <int MODE, int PREC>
struct __align__(1024) TcSmemT {
  static constexpr int STAGES = TcCfg<MODE, PREC>::STAGES, BN = TcCfg<MODE, PREC>::BN, NXB = TcCfg<MODE, PREC>::NXB;
  static constexpr int EPW = TcCfg<MODE, PREC>::EPW;
  float a[STAGES][TCM * TCK];  // 16 KB per stage, 128-byte rows, swizzle-128B
  float b[STAGES][BN * TCK];   // 32 KB per stage (PAIR: 16 KB)
  float alo[PREC ? STAGES : 1][PREC ? TCM * TCK : 4];
  float blo[PREC ? STAGES : 1][PREC ? BN * TCK : 4];
  uint64_t full[STAGES], empty[STAGES], lo_ready[STAGES], peer_full[STAGES], acc_full[2], acc_empty[2], xfull[EPW][NXB];
  uint32_t tmem_base;
  // epilogue: per-warp 32x32 staging tile (128-byte rows, 16-byte units XOR-swizzled by row & 7), the per-column
  // vectors {bias, gamma, beta}, and (MODE 2) per-warp column-sum partials. MODE 2: four tiles per warp — the ring TMA
  // fills with the x-hat chunks the LayerNorm backward reads (and the staging tile of the chunk being worked on)
  alignas(1024) float tile[EPW][NXB][32 * 32];  // (TMA reads and writes them: the 128-byte swizzle follows absolute address bits)
  alignas(16) float cvec[4][HID];  // bias, gamma, beta, and (fused critic head) w3
  alignas(16) float wpart[MODE == 2 ? 4 : 1][MODE == 2 ? 3 : 4][HID];  // (forward: only the second vector set lives here, 4 KB)
  float qgamma[2];  // fused critic head: the discount of each vector set's agent (fetched with the vectors)
  float4 xch[EPW == 8 ? 2 * 2 * TCM : 1];  // [slot][half][row]: what the two column halves of a row swap (paired epilogue warps)
};

__device__ __forceinline__ uint32_t s32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init_(uint64_t* b, int n) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(s32(b)), "r"(n) : "memory"); }
__device__ __forceinline__ void mbar_expect_(uint64_t* b, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(s32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait_(uint64_t* b, uint32_t parity) {
  asm volatile(
      "{\n .reg .pred p;\n W_%=:\n mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n @p bra D_%=;\n bra W_%=;\n D_%=:\n}" ::"r"(s32(b)),
      "r"(parity)
      : "memory");
}
// (the maps are rank 3: {k, row, agent} — agent = 0 for a single learner — so that rows beyond an agent's batch are
// zero-filled by TMA instead of running on into the next agent's rows)
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, int c0, int c1, int c2, uint64_t* bar) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(s32(dst)),
               "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(s32(bar))
               : "memory");
}
// TMA store of one staging tile (32 rows x 32 columns, the box of the output's map); rows beyond the agent's batch are
// clipped by the map. Bulk-group completion: wait_group.read N = all but the N most recent groups have READ their source.
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, const void* src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(map), "r"(s32(src)), "r"(c0),
               "r"(c1), "r"(c2)
               : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
// K-major, 128-byte swizzle: rows of 128 bytes, 8-row groups 1024 bytes apart (cute::UMMA::SmemDescriptor fields:
// start address [0,14), stride byte offset [32,46), version = 1 [46,48), layout SWIZZLE_128B = 2 [61,64))
__device__ __forceinline__ uint64_t umma_desc(const void* smem, int byte_off) {
  const uint64_t addr = (uint64_t)((s32(smem) + (uint32_t)byte_off) & 0x3FFFFu) >> 4;
  return addr | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
// cute::UMMA::InstrDescriptor: c_format F32 = 1 [4,6), a/b format TF32 = 2 [7,10) [10,13), K-major both, N>>3 [17,23), M>>4 [24,29)
constexpr uint32_t TC_IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(TCN >> 3) << 17) | ((uint32_t)(TCM >> 4) << 24);

template <bool B_MN = false>
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t accumulate) {
  constexpr uint32_t idesc = TC_IDESC | (B_MN ? (1u << 16) : 0u);  // bit 16: b_major = MN
  asm volatile(
      "{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}" ::"r"(tmem_d),
      "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
      : "memory");
}
// MN-major B operand, SWIZZLE_128B_BASE32B (layout type 1): 32-column chunks 4 KB apart (LBO), 4-row atoms 512 B apart (SBO);
// one K = 8 instruction consumes two atoms (1 KB) of every chunk (tc_wgrad.cu)
__device__ __forceinline__ uint64_t umma_desc_mn(const void* smem, int byte_off) {
  const uint64_t addr = (uint64_t)((s32(smem) + (uint32_t)byte_off) & 0x3FFFFu) >> 4;
  return addr | ((uint64_t)(4096 >> 4) << 16) | ((uint64_t)(512 >> 4) << 32) | (1ull << 46) | (1ull << 61);
}
// multicast forms (2-CTA cluster): the load lands at the same shared-memory offset of every CTA in `mask` and counts its
// bytes on the mbarrier at the same offset there; the commit arrives on the mbarrier of every CTA in `mask`
__device__ __forceinline__ void tma_load_3d_mc(void* dst, const CUtensorMap* map, int c0, int c1, int c2, uint64_t* bar, uint16_t mask) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%2, %3, %4}], [%5], %6;" ::"r"(
          s32(dst)),
      "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(s32(bar)), "h"(mask)
      : "memory");
}
__device__ __forceinline__ void umma_commit_mc(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(s32(bar)),
               "h"(mask)
               : "memory");
}
// ---- cta_group::2 forms: issued by one thread of the cluster's rank-0 CTA on behalf of both SMs
__device__ __forceinline__ void umma_tf32_pair(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t accumulate) {
  constexpr uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(TCN >> 3) << 17) | ((uint32_t)((2 * TCM) >> 4) << 24);
  const uint32_t z = 0;
  asm volatile(
      "{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n"
      " tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n}" ::"r"(tmem_d),
      "l"(da), "l"(db), "r"(idesc), "r"(accumulate), "r"(z)
      : "memory");
}
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {  // arrives on `bar` of BOTH CTAs
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(s32(bar)),
               "h"((uint16_t)3)
               : "memory");
}
// arrive on the mbarrier at the same offset as `bar` in the cluster's rank-0 CTA. Plain (CTA-scope release) forms on both
// sides, as for every other cross-CTA mbarrier of these kernels: what the arrivals order is shared-memory traffic the
// issuing threads have already fenced towards the async proxy (split warps) or TMEM reads completed with
// tcgen05.wait::ld (epilogue). The .release.cluster / .acquire.cluster forms compile to MEMBAR.ALL.GPU + ERRBAR per
// arrival — which also waits for the epilogue's global stores — and CCTL.IVALL per wait: measured 68 instead of 55 us
// per 65 536-row launch (ncu SASS view).
__device__ __forceinline__ void mbar_arrive_rank0(uint64_t* bar) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, 0;" : "=r"(r) : "r"(s32(bar)));
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(r) : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(s32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}


// ---- the epilogue's staging tile: 32 rows x 32 fp32, 16-byte unit q of row r at unit q ^ (r & 7). Conflict-free for
// thread-per-row float4 access (TMEM side), for 8-lanes-per-row float4 access (global side: 4 full 128-byte row
// segments per warp instruction instead of 32 scattered 16-byte pieces) and for lane-per-column scalar reads.
__device__ __forceinline__ float4* tile_q(float* t, int r, int q) { return reinterpret_cast<float4*>(t + r * 32 + ((q ^ (r & 7)) << 2)); }
__device__ __forceinline__ void tile_put(float* t, int lane, const float (&v)[32]) {  // thread-per-row registers -> tile
#pragma unroll
  for (int q = 0; q < 8; ++q) *tile_q(t, lane, q) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
}
__device__ __forceinline__ void tile_get(float* t, int lane, float (&v)[32]) {  // tile -> thread-per-row registers
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const float4 x = *tile_q(t, lane, q);
    v[4 * q] = x.x, v[4 * q + 1] = x.y, v[4 * q + 2] = x.z, v[4 * q + 3] = x.w;
  }
}
// tile -> rows of a [.][256] matrix at G (= row 0 of the tile, first column of the chunk), rows < rows_valid only
__device__ __forceinline__ void tile_store(float* t, int lane, float* G, int rows_valid) {
#pragma unroll
  for (int it = 0; it < 8; ++it) {
    const int r = it * 4 + (lane >> 3), q = lane & 7;
    if (r < rows_valid) *reinterpret_cast<float4*>(G + (size_t)r * TCN + q * 4) = *tile_q(t, r, q);
  }
}
__device__ __forceinline__ float tile_colsum(const float* t, int lane) {  // sum over the 32 rows of column `lane`
  float cs = 0.f;
#pragma unroll
  for (int r = 0; r < 32; ++r) cs += t[r * 32 + (((lane >> 2) ^ (r & 7)) << 2) + (lane & 3)];
  return cs;
}

// MODE 0: forward  H = [ReLU](LayerNorm(A . B^T + bias)), optional x-hat / statistics outputs.
// MODE 1: the FIRST layer (agents/nets.py:66-72), same epilogue: A = the rows' inputs X [M][K] (any K: ceil(K/32) slabs,
//         columns beyond K zero-filled by TMA), B = w1t [K][256] in the arena's forward layout, i.e. an MN-MAJOR operand:
//         staged by TMA in the SWIZZLE_128B_BASE32B layout tc_wgrad.cu uses (boxes of 32 columns x 32 k) and described to
//         the tensor core with b_major = MN. The FFMA first layer (wide.cu) is issue/latency-bound at 152 us per 262 144
//         rows; on the tensor cores the layer costs its epilogue.
// MODE 2: backward dX: D = A . B^T with A = dz2 [M][256], B = w2t; epilogue = the ReLU mask and LayerNorm backward of
//         layer 1 (x-hat and rstd read per row), H <- dz1, and this CTA's column sums {sum dz, sum dn*xhat, sum dn}
//         -> part[cta][3][256] (bias / LayerNorm-affine gradients; deterministic: transposed through shared memory).
template <int MODE, int PREC>
__global__ void __launch_bounds__((TcCfg<MODE, PREC>::THREADS), 1)
tc_linear_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                 const __grid_constant__ CUtensorMap mapBlo, const __grid_constant__ CUtensorMap mapX,
                 const __grid_constant__ CUtensorMap mapH, const __grid_constant__ CUtensorMap mapXH, int M, int kb_first,
                 const float* __restrict__ bias, const float* __restrict__ g, const float* __restrict__ be, int ln, int relu,
                 float* __restrict__ H, float* __restrict__ XH, float2* __restrict__ stat, float* __restrict__ part,
                 const __grid_constant__ b2rl_wide_q_t Q, const Stk K) {
  extern __shared__ unsigned char tc_raw[];  // (the swizzle atoms need 1024-byte alignment: align by hand)
  using Smem = TcSmemT<MODE, PREC>;
  constexpr int TC_STAGES = Smem::STAGES;
  constexpr bool PAIR = TcCfg<MODE, PREC>::PAIR;
  constexpr int EPW = Smem::EPW, EPT = 32 * EPW;  // epilogue warps / threads
  // bytes TMA delivers into one stage of THIS CTA (multicast path: the whole weight slab, half of it sent by the peer)
  constexpr uint32_t TC_STAGE_BYTES = (TCM + Smem::BN * (PREC == 1 ? 2 : 1)) * TCK * sizeof(float);
  Smem& S = *reinterpret_cast<Smem*>(tc_raw + ((1024u - (s32(tc_raw) & 1023u)) & 1023u));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = (M + TCM - 1) / TCM;  // per agent (M = rows per agent)
  // Persistent, in clusters of 2: cluster ci works on tile pairs ci, ci + n_clusters, ...; CTA `crank` of the cluster takes
  // tile 2 * pair + crank (a ghost tile beyond the batch loads zeros and stores nothing, so that both CTAs run the same
  // number of k-slabs: each loads HALF of every weight slab and multicasts it to both). Local tile i accumulates in TMEM
  // buffer i & 1, so the epilogue of tile i runs while the ring and the tensor core work on tile i + 1.
  // Stacked agents: the pairs of all agents form one list, pair p belongs to agent p / pairs_per_agent — a pair never
  // straddles two agents, so both CTAs of a cluster always want the same agent's weight slab (the multicast stands).
  uint32_t crank;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(crank));
  const int ppa = (n_tiles + 1) >> 1;  // pairs per agent
  const int n_clusters = (int)gridDim.x >> 1, ci = (int)blockIdx.x >> 1, n_pairs = ppa * K.n;
  const int my_tiles = (n_pairs - ci + n_clusters - 1) / n_clusters;
  auto agent_of = [&](int i) { return (ci + i * n_clusters) / ppa; };
  auto tile_of = [&](int i) { return 2 * ((ci + i * n_clusters) % ppa) + (int)crank; };  // tile inside the agent's batch

  if (warp == 0 && lane == 0) {
    // multicast path: `empty` collects both CTAs' MMA commits. PAIR: one commit reaches both CTAs; the issuing CTA's
    // lo_ready / acc_empty collect the split warps / epilogue threads of BOTH CTAs.
    for (int s = 0; s < TC_STAGES; ++s) {
      mbar_init_(&S.full[s], 1);
      mbar_init_(&S.empty[s], PAIR ? 1 : 2);
      mbar_init_(&S.lo_ready[s], PAIR ? 128 : 64);
      mbar_init_(&S.peer_full[s], 1);  // (PAIR, rank 0) the peer CTA's slab has landed: relayed by the peer's idle MMA warp
    }
    for (int b = 0; b < 2; ++b) { mbar_init_(&S.acc_full[b], 1); mbar_init_(&S.acc_empty[b], PAIR ? 2 * EPT : EPT); }
    for (int e = 0; e < EPW; ++e)
      for (int j = 0; j < Smem::NXB; ++j) mbar_init_(&S.xfull[e][j], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {  // TMEM: two accumulator tiles of 256 fp32 columns x 128 lanes (all 512 columns: one CTA per SM)
    if constexpr (PAIR) {  // (the same warp of both CTAs, the same destination offset)
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s32(&S.tmem_base)), "n"(2 * TCN) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s32(&S.tmem_base)), "n"(2 * TCN) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  cluster_sync_all();  // the peer's barriers are initialised before anything of ours can land on them
  const uint32_t tmem = S.tmem_base;
  const int KB = MODE == 1 ? kb_first : HID / TCK;  // k-slabs: 8 for the hidden layers, ceil(K / 32) for a first layer
  constexpr bool BMN = MODE == 1;                   // the first layer's weights are MN-major (forward layout)
  auto bdesc = [&](const float* base, int k) { return BMN ? umma_desc_mn(base, k * 1024) : umma_desc(base, k * 32); };

  // 384-thread form: the first warpgroup (TMA, MMA, lo split) hands registers to the two epilogue warpgroups
  // (each warpgroup's setmaxnreg opens a branch that does not rejoin the other before the teardown)
  if (warp < 4) {
  if constexpr (MODE == 2) asm volatile("setmaxnreg.dec.sync.aligned.u32 72;" ::: "memory");
  if (warp == 0) {
    if (lane == 0) {  // ===== TMA producer: the ring runs on across tiles
      int it = 0;
      for (int i = 0; i < my_tiles; ++i) {
        const int m0 = tile_of(i) * TCM, ag = agent_of(i);
        const int half = (int)crank * (TCN / 2);  // this CTA's rows of the weight slab
        for (int kb = 0; kb < KB; ++kb, ++it) {
          const int s = it % TC_STAGES;
          if (it >= TC_STAGES) mbar_wait_(&S.empty[s], ((it / TC_STAGES) - 1) & 1);  // free in BOTH CTAs
          mbar_expect_(&S.full[s], TC_STAGE_BYTES);
          tma_load_3d(S.a[s], &mapA, kb * TCK, m0, ag, &S.full[s]);
          if constexpr (PAIR) {  // this CTA's half of the weight slab, into its own shared memory only
            tma_load_3d(S.b[s], &mapB, kb * TCK, half, ag, &S.full[s]);
            if constexpr (PREC == 1) tma_load_3d(S.blo[s], &mapBlo, kb * TCK, half, ag, &S.full[s]);
          } else if constexpr (BMN) {  // this CTA's four 32-column chunks of the [32 k][256] slab, multicast to both CTAs
#pragma unroll
            for (int c = 0; c < 4; ++c)
              tma_load_3d_mc(S.b[s] + (4 * (int)crank + c) * 1024, &mapB, 32 * (4 * (int)crank + c), kb * TCK, ag, &S.full[s], 3);
          } else
          tma_load_3d_mc(S.b[s] + half * TCK, &mapB, kb * TCK, half, ag, &S.full[s], 3);
          if constexpr (PREC == 1 && !PAIR) tma_load_3d_mc(S.blo[s] + half * TCK, &mapBlo, kb * TCK, half, ag, &S.full[s], 3);
          (void)mapBlo;
        }
      }
    }
  } else if (warp == 1) {
    if (PAIR && lane == 0 && crank == 0) {  // ===== MMA issuer of the pair: every instruction drives both SMs
      int it = 0;
      for (int i = 0; i < my_tiles; ++i) {
        const int buf = i & 1;
        const uint32_t acc = tmem + buf * TCN;
        if (i >= 2) {  // BOTH epilogues must have drained this buffer (tile i - 2)
          mbar_wait_(&S.acc_empty[buf], ((i >> 1) - 1) & 1);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        }
        for (int kb = 0; kb < KB; ++kb, ++it) {
          const int s = it % TC_STAGES;
          mbar_wait_(&S.full[s], (it / TC_STAGES) & 1);               // this CTA's slab has landed ...
          mbar_wait_(&S.peer_full[s], (it / TC_STAGES) & 1);  // ... and the peer's
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
          for (int k = 0; k < TCK / 8; ++k) {  // the product(s) whose operands TMA delivered run while the lo split is made
            umma_tf32_pair(acc, umma_desc(S.a[s], k * 32), umma_desc(S.b[s], k * 32), (kb | k) != 0);
            if constexpr (PREC == 1) umma_tf32_pair(acc, umma_desc(S.a[s], k * 32), umma_desc(S.blo[s], k * 32), 1);
          }
          mbar_wait_(&S.lo_ready[s], (it / TC_STAGES) & 1);  // both CTAs' split warps are done with this slab
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
          for (int k = 0; k < TCK / 8; ++k) {
            umma_tf32_pair(acc, umma_desc(S.alo[s], k * 32), umma_desc(S.b[s], k * 32), 1);
            if constexpr (PREC == 2) umma_tf32_pair(acc, umma_desc(S.a[s], k * 32), umma_desc(S.blo[s], k * 32), 1);
          }
          umma_commit_pair(&S.empty[s]);  // frees the slot in both CTAs
        }
        umma_commit_pair(&S.acc_full[buf]);
      }
    } else if (PAIR && lane == 0) {  // rank 1: tell the issuer when this CTA's slabs have landed
      for (int it = 0; it < my_tiles * KB; ++it) {
        const int s = it % TC_STAGES;
        mbar_wait_(&S.full[s], (it / TC_STAGES) & 1);
        mbar_arrive_rank0(&S.peer_full[s]);
      }
    } else if (!PAIR && lane == 0) {  // ===== MMA issuer
      int it = 0;
      for (int i = 0; i < my_tiles; ++i) {
        const int buf = i & 1;
        const uint32_t acc = tmem + buf * TCN;
        if (i >= 2) {  // the epilogue must have drained this buffer (tile i - 2)
          mbar_wait_(&S.acc_empty[buf], ((i >> 1) - 1) & 1);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        }
        for (int kb = 0; kb < KB; ++kb, ++it) {
          const int s = it % TC_STAGES;
          mbar_wait_(&S.full[s], (it / TC_STAGES) & 1);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
          for (int k = 0; k < TCK / 8; ++k) {  // UMMA K = 8 tf32 = 32 bytes: advance inside the 128-byte swizzle row
            umma_tf32<BMN>(acc, umma_desc(S.a[s], k * 32), bdesc(S.b[s], k), (kb | k) != 0);
            if constexpr (PREC == 1) umma_tf32<BMN>(acc, umma_desc(S.a[s], k * 32), bdesc(S.blo[s], k), 1);
          }
          if constexpr (PREC != 0) {  // the product(s) whose operands TMA delivered run while the lo split is made
            mbar_wait_(&S.lo_ready[s], (it / TC_STAGES) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
            for (int k = 0; k < TCK / 8; ++k) {
              umma_tf32<BMN>(acc, umma_desc(S.alo[s], k * 32), bdesc(S.b[s], k), 1);
              if constexpr (PREC == 2) umma_tf32<BMN>(acc, umma_desc(S.a[s], k * 32), bdesc(S.blo[s], k), 1);
            }
          }
          umma_commit_mc(&S.empty[s], 3);  // (implies tcgen05.fence::before_thread_sync) frees the slot in both CTAs
        }
        umma_commit(&S.acc_full[buf]);
      }
    }
  } else {  // ===== (3xTF32) the activations' lo parts, slab by slab as the ring fills
    if constexpr (PREC != 0) {
      const int lt = threadIdx.x - 64;  // 0..63
      for (int it = 0; it < my_tiles * KB; ++it) {
        const int s = it % TC_STAGES;
        mbar_wait_(&S.full[s], (it / TC_STAGES) & 1);
        const float4* src = reinterpret_cast<const float4*>(S.a[s]);
        float4* dst = reinterpret_cast<float4*>(S.alo[s]);
#pragma unroll 4
        for (int i = 0; i < TCM * TCK / 4 / 64; ++i)  // element-wise, so the swizzled layout carries over
          dst[lt + 64 * i] = tf32_lo4(src[lt + 64 * i]);
        if constexpr (PREC == 2) {  // the weight slab too (multicast path: both halves landed here; PAIR: this CTA's half)
          const float4* bs = reinterpret_cast<const float4*>(S.b[s]);
          float4* bd = reinterpret_cast<float4*>(S.blo[s]);
#pragma unroll 4
          for (int i = 0; i < Smem::BN * TCK / 4 / 64; ++i) bd[lt + 64 * i] = tf32_lo4(bs[lt + 64 * i]);
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> visible to the MMA's reads
        if constexpr (PAIR) mbar_arrive_rank0(&S.lo_ready[s]);
        else asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(s32(&S.lo_ready[s])) : "memory");
      }
    }
  }
  } else {  // ===== epilogue: warp w may touch TMEM lanes 32*(w % 4) .. +31
    if constexpr (MODE == 2) asm volatile("setmaxnreg.inc.sync.aligned.u32 208;" ::: "memory");
    const int lg = warp & 3, ew = warp - 4, et = threadIdx.x - 128;
    float* T = S.tile[ew][0];
    const bool head = MODE != 2 && Q.w3 != nullptr;  // the critic's scalar head rides in this epilogue (wide.cu::wide_q_head)
    // Per-column vectors {bias, gamma, beta, w3} of the tile's agent, in shared memory (broadcast reads). One learner: loaded
    // once. Stacked agents: every tile pair belongs to another agent, and loading its vectors at the top of the tile put a
    // dependent global round trip and two barriers on every tile (ncu: 18 % long-scoreboard + 15-20 % barrier stalls of a
    // first-layer launch) — so there are two sets, and the NEXT agent's set is fetched with cp.async while this tile is
    // worked on. Set 1 lives where the other mode's data would be: in wpart (forward: unused) or in the bias / w3 slots of
    // set 0 (backward: only gamma and beta are needed).
    auto vptr = [&](int set, int q) -> float* {  // vector q of set `set`
      if constexpr (MODE == 2) return S.cvec[set ? (q == 1 ? 0 : 3) : q];
      return (set ? &S.wpart[0][0][0] : &S.cvec[0][0]) + q * HID;
    };
    auto fetch_vectors = [&](int ag, int set) {  // 64 cp.async of 16 bytes per vector; constants where a vector is absent
      const size_t po = (size_t)ag * K.ps;
      for (int i = et; i < 4 * (HID / 4); i += EPT) {
        const int q = i / (HID / 4), u = i - q * (HID / 4);
        if (MODE == 2 && (q == 0 || q == 3)) continue;
        const float* src = q == 0 ? bias : q == 1 ? g : q == 2 ? be : Q.w3;
        float* dst = vptr(set, q) + 4 * u;
        if (src) {
          asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(s32(dst)), "l"(src + po + 4 * u) : "memory");
        } else {
          const float c = q == 1 ? 1.f : 0.f;
          *reinterpret_cast<float4*>(dst) = make_float4(c, c, c, c);
        }
      }
      if (head && et == 0) {  // the TD target's discount: agent_hp's choice, fetched like the vectors
        if (K.hp) asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(s32(&S.qgamma[set])), "l"(&K.hp[ag].gamma) : "memory");
        else S.qgamma[set] = Q.gamma;  // (no table: the scalar, as common.cuh agent_hp would return)
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
    };
    float v[32];
    int cset = 0, sti = 0, xc = 0;  // sti: this warp's TMA stores so far (the staging tiles rotate); xc: pair exchanges
    (void)sti, (void)xc;
    if (my_tiles > 0) fetch_vectors(agent_of(0), 0);
    for (int ti = 0; ti < my_tiles; ++ti) {
      const int tile = tile_of(ti), buf = ti & 1, ag = agent_of(ti);
      const bool next_differs = ti + 1 < my_tiles && agent_of(ti + 1) != ag;
      if (ti == 0 || agent_of(ti - 1) != ag) {  // this agent's set has landed, and everyone is done with the other set
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        asm volatile("bar.sync 1, %0;" ::"n"(EPT) : "memory");
      }
      if (next_differs) fetch_vectors(agent_of(ti + 1), cset ^ 1);
      const float *cb = vptr(cset, 0), *cg = vptr(cset, 1), *cbe = vptr(cset, 2), *cw3 = vptr(cset, 3);
      const size_t arow = (size_t)ag * M;           // first row of this agent in the stacked arrays
      const int row0 = tile * TCM + 32 * lg, row = row0 + lane;  // inside the agent's batch
      const uint32_t tl = tmem + buf * TCN + ((uint32_t)(32 * lg) << 16);
      if constexpr (MODE != 2) {
        // EPW == 8 (first layer): warp (eh, lg) owns column chunks 4 eh .. 4 eh + 3 of rows 32 lg ..; the LayerNorm sums are
        // the two halves' partial sums added in a fixed order (half 0 + half 1), swapped through shared memory
        constexpr int CPW = (TCN / 32) / (EPW / 4);
        const int eh = ew >> 2, c0 = CPW * eh;
        // what the two halves of a row exchange (one 64-thread named barrier; a slot is reused two exchanges later)
        auto pair_swap = [&](float4 mine) -> float4 {
          float4* xs = S.xch + (xc & 1) * 2 * TCM;
          ++xc;
          xs[eh * TCM + 32 * lg + lane] = mine;
          asm volatile("bar.sync %0, 64;" ::"r"(2 + lg) : "memory");
          return xs[(eh ^ 1) * TCM + 32 * lg + lane];
        };
        mbar_wait_(&S.acc_full[buf], (ti >> 1) & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        float mean = 0.f, rstd = 1.f;
        if (ln) {
          // LayerNorm statistics in ONE pass over the accumulator (the two-pass form read all of it twice before the output
          // pass): sums of d = z - shift and d^2 with shift = the mean of the row's first 32 columns (of this warp's half),
          // so |mean - shift| is a fraction of the row's standard deviation and the variance formula below cancels nothing
          // of significance (its terms are sigma^2 (1 + O(1/32)) and O(sigma^2 / 32)).
          tmem_ld32(tl + c0 * 32, v);
          float sh = 0.f;
#pragma unroll
          for (int i = 0; i < 32; ++i) sh += v[i] + cb[c0 * 32 + i];
          sh *= (1.0f / 32);
          float s1 = 0.f, s2 = 0.f;
          for (int c = c0; c < c0 + CPW; ++c) {
            if (c != c0) tmem_ld32(tl + c * 32, v);
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              const float d = v[i] + cb[c * 32 + i] - sh;
              s1 += d;
              s2 = fmaf(d, d, s2);
            }
          }
          float var;
          if constexpr (EPW == 8) {  // combine the halves in the order (half 0, half 1): both warps get the same bits
            const float4 o = pair_swap(make_float4(sh, s1, s2, 0.f));
            const float sh0 = eh ? o.x : sh, a0 = eh ? o.y : s1, q0 = eh ? o.z : s2;
            const float sh1 = eh ? sh : o.x, a1 = eh ? s1 : o.y, q1 = eh ? s2 : o.z;
            constexpr float NH = TCN / 2;
            mean = (fmaf(NH, sh0, a0) + fmaf(NH, sh1, a1)) * (1.0f / TCN);
            const float e0 = mean - sh0, e1 = mean - sh1;
            var = ((q0 - 2.f * e0 * a0 + NH * e0 * e0) + (q1 - 2.f * e1 * a1 + NH * e1 * e1)) * (1.0f / TCN);
          } else {
            const float m = s1 * (1.0f / TCN);
            mean = sh + m;
            var = fmaf(-m, m, s2 * (1.0f / TCN));
          }
          rstd = 1.0f / sqrtf(fmaxf(var, 0.f) + LN_EPS);
          if (stat && row < M && eh == 0) stat[arow + row] = make_float2(mean, rstd);
        }
        float qacc = 0.f;
        for (int c = c0; c < c0 + CPW; ++c) {
          tmem_ld32(tl + c * 32, v);
          if (c == c0 + CPW - 1) {  // last TMEM read of this tile: hand the buffer back to the MMA issuer
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            if constexpr (PAIR) mbar_arrive_rank0(&S.acc_empty[buf]);
            else asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(s32(&S.acc_empty[buf])) : "memory");
          }
          float h[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const int j = c * 32 + i;
            float x = v[i] + cb[j];
            if (ln) {
              x = (x - mean) * rstd;
              v[i] = x;  // x-hat
              x = fmaf(x, cg[j], cbe[j]);
            } else {
              v[i] = x;  // pre-activation
            }
            h[i] = relu ? fmaxf(x, 0.f) : x;
            if (head) qacc = fmaf(h[i], cw3[j], qacc);
          }
          // Outputs leave through TMA stores of the staging tile (one instruction of one lane instead of 8 LDS.128 + 8
          // STG.128 per lane: the staging was the epilogue's MIO bottleneck, ncu short-scoreboard / mio stalls) where the
          // warp has two tiles to alternate; with one (MODE 0: the ring takes the rest) a store's read latency would sit
          // between every two tiles written (measured 53 vs 46 us), so there the warp copies the tile out itself.
          if constexpr (Smem::NXB < 2) {
            const int rows_valid = M - row0;
            if (H) {
              tile_put(T, lane, h);
              __syncwarp();
              tile_store(T, lane, H + (arow + row0) * TCN + c * 32, rows_valid);
              __syncwarp();
            }
            if (XH) {
              tile_put(T, lane, v);
              __syncwarp();
              tile_store(T, lane, XH + (arow + row0) * TCN + c * 32, rows_valid);
              __syncwarp();
            }
          } else {
          if (H) {  // (a target critic with the fused head never needs its h2 in memory)
            float* Ts = S.tile[ew][sti % Smem::NXB];
            if (lane == 0) tma_store_wait_read<Smem::NXB - 1>();  // the store that last read this tile is done with it
            __syncwarp();
            tile_put(Ts, lane, h);
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) tma_store_3d(&mapH, Ts, c * 32, row0, ag);
            ++sti;
          }
          if (XH) {
            float* Ts = S.tile[ew][sti % Smem::NXB];
            if (lane == 0) tma_store_wait_read<Smem::NXB - 1>();
            __syncwarp();
            tile_put(Ts, lane, v);
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) tma_store_3d(&mapXH, Ts, c * 32, row0, ag);
            ++sti;
          }
          }
        }
        if constexpr (EPW == 8) {  // the two column halves' parts of w3 . h2, added in the order (half 0, half 1)
          if (head) {
            const float o = pair_swap(make_float4(qacc, 0.f, 0.f, 0.f)).x;
            qacc = eh ? o + qacc : qacc + o;
          }
        }
        if (head && eh == 0) {  // q = w3 . h2 + b3 per row (thread); online critics: TD target, dLoss/dQ, squared error (agent.py:212-233)
          float sq = 0.f, dqv = 0.f;
          const size_t grow = arow + row;
          if (row < M) {
            const float q = qacc + __ldg(Q.b3 + (size_t)ag * K.ps);
            Q.q_out[grow] = q;
            if (Q.mode == 1) {
              const float q0 = Q.qn0[grow], q1 = Q.qn1[grow];
              const float qmin = fminf(q0, q1);
              float qp = Q.bcq_mix ? __fadd_rn(__fmul_rn(0.75f, qmin), __fmul_rn(0.25f, fmaxf(q0, q1))) : qmin;
              if (!Q.td3) qp = __fsub_rn(qp, __fmul_rn(expf(Q.log_alpha[(size_t)ag * K.as]), Q.logp[grow]));
              const float* rr = Q.rows + grow * Q.row_stride + Q.rd_off;
              const float y = __fadd_rn(rr[0], __fmul_rn(__fmul_rn(1.0f - rr[1], S.qgamma[cset]), qp));
              if (Q.targ_out) Q.targ_out[grow] = y;
              const float dlt = q - y;
              dqv = dlt * (2.0f / (float)Q.M);
              Q.dz3[grow * MAX_OUT] = dqv;
              sq = dlt * dlt;
            }
          }
          if (Q.mode == 1) {  // {sum of squared errors, sum of dQ} per 8 rows: the layout wide_critic_scalars reduces
#pragma unroll
            for (int sft = 1; sft < 8; sft <<= 1) {
              sq += __shfl_xor_sync(0xffffffffu, sq, sft);
              dqv += __shfl_xor_sync(0xffffffffu, dqv, sft);
            }
            if ((lane & 7) == 0 && row < M) {
              const size_t pi = (size_t)ag * ((M + 7) >> 3) + (row >> 3);
              Q.sq_part[2 * pi] = sq;
              Q.sq_part[2 * pi + 1] = dqv;
            }
          }
        }
      } else {  // ===== backward epilogue: XH = x-hat of layer 1 (input), stat = its (mean, rstd), H <- dz1
        // x-hat reaches the warp through its own ring of NXB 32x32 tiles filled by TMA (boxes of 32 rows x 32 columns in
        // the 128-byte swizzle = exactly the staging-tile layout): lane 0 requests the chunk of visit v + NXB as soon as the
        // warp is done with the tile of visit v, so NXB - 1 chunks are always in flight — across the two passes and across
        // tiles (x-hat does not depend on this kernel's products). The first version fetched each chunk with the epilogue
        // threads' own loads one chunk ahead (all the registers allow): 16 KB in flight per SM, a third of the launch's
        // long-scoreboard stalls on the store that staged it (ncu), 24 us of epilogue per tile against 11 us of MMAs.
        // Two warps per 32 rows: warp (eh, lg) owns column chunks 4 * eh .. 4 * eh + 3; the row sums of the LayerNorm backward
        // are the two halves' partial sums added in a fixed order (half 0 + half 1), swapped through shared memory.
        const bool live = row < M;
        constexpr int NXB = Smem::NXB, CPW = TCN / 32 / 2;  // column chunks per warp
        const int eh = ew >> 2, c0 = CPW * eh;
        const int vpt = ln ? 2 * CPW : CPW;  // chunk visits per tile: two passes with LayerNorm, else one
        auto xissue = [&](int vj) {  // lane 0 only
          if (vj < my_tiles * vpt) {
            const int tj = vj / vpt, c = c0 + ((vj - tj * vpt) & (CPW - 1)), b = vj % NXB;
            mbar_expect_(&S.xfull[ew][b], 32 * 32 * sizeof(float));
            tma_load_3d(S.tile[ew][b], &mapX, c * 32, tile_of(tj) * TCM + 32 * lg, agent_of(tj), &S.xfull[ew][b]);
          }
        };
        if (ti == 0 && lane == 0)
          for (int j = 0; j < NXB; ++j) xissue(j);
        int vi = ti * vpt;
        float x[32];
        mbar_wait_(&S.acc_full[buf], (ti >> 1) & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        float s1 = 0.f, s2 = 0.f;
        if (ln) {
          for (int c = c0; c < c0 + CPW; ++c, ++vi) {
            mbar_wait_(&S.xfull[ew][vi % NXB], (vi / NXB) & 1);
            tile_get(S.tile[ew][vi % NXB], lane, x);
            // every lane's reads of the slot are ordered before TMA's refill of it (generic -> async proxy): without the
            // fence a refill could overwrite rows a lane had not read yet, and their row sums took the next chunk's x-hat
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) xissue(vi + NXB);
            tmem_ld32(tl + c * 32, v);
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              const int j = c * 32 + i;
              const float gj = cg[j];
              const float dx = (fmaf(x[i], gj, cbe[j]) > 0.f ? v[i] : 0.f) * gj;
              s1 += dx;
              s2 = fmaf(dx, x[i], s2);
            }
          }
          float4* xs = S.xch + (ti & 1) * 2 * TCM;  // [half][row of the tile]; a slot is reused two pair barriers later
          xs[eh * TCM + 32 * lg + lane] = make_float4(s1, s2, 0.f, 0.f);
          asm volatile("bar.sync %0, 64;" ::"r"(2 + lg) : "memory");
          const float4 o = xs[(eh ^ 1) * TCM + 32 * lg + lane];
          s1 = eh ? o.x + s1 : s1 + o.x;
          s2 = eh ? o.y + s2 : s2 + o.y;
        }
        const float m1 = s1 * (1.0f / TCN), m2 = s2 * (1.0f / TCN), rstd = (ln && live) ? stat[arow + row].y : 1.f;
        for (int c = c0; c < c0 + CPW; ++c, ++vi) {
          T = S.tile[ew][vi % NXB];  // the chunk's tile doubles as the staging tile once x-hat is in registers
          mbar_wait_(&S.xfull[ew][vi % NXB], (vi / NXB) & 1);
          tile_get(T, lane, x);
          __syncwarp();
          tmem_ld32(tl + c * 32, v);
          if (c == c0 + CPW - 1) {  // last TMEM read of this tile
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            if constexpr (PAIR) mbar_arrive_rank0(&S.acc_empty[buf]);
            else asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(s32(&S.acc_empty[buf])) : "memory");
          }
          float dz[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const int j = c * 32 + i;
            if (ln) {
              const float gj = cg[j];
              v[i] = fmaf(x[i], gj, cbe[j]) > 0.f ? v[i] : 0.f;  // dn: gradient at the LayerNorm output
              dz[i] = rstd * (v[i] * gj - m1 - x[i] * m2);
            } else {
              v[i] = x[i] > 0.f ? v[i] : 0.f;
              dz[i] = v[i];
            }
            if (!live) dz[i] = 0.f;
            x[i] *= v[i];  // dn * x-hat
          }
          // dz: to global (coalesced through the tile) and its column sums; then the two LayerNorm-affine sums.
          // Column sums over this warp's 32 rows: lane <-> column of the tile (deterministic, fixed order).
          tile_put(T, lane, dz);
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          __syncwarp();
          if (lane == 0) tma_store_3d(&mapH, T, c * 32, row0, ag);  // dz1 -> global, while the column sums read the tile
          if (part) {  // (uniform; NULL: dz1 only — the actor step's pass through the critics needs no parameter gradients)
            S.wpart[lg][0][c * 32 + lane] = tile_colsum(T, lane);
            if (lane == 0) tma_store_wait_read<0>();
            __syncwarp();
            tile_put(T, lane, x);
            __syncwarp();
            S.wpart[lg][1][c * 32 + lane] = tile_colsum(T, lane);
            __syncwarp();
            tile_put(T, lane, v);
            __syncwarp();
            S.wpart[lg][2][c * 32 + lane] = tile_colsum(T, lane);
          } else if (lane == 0) {
            tma_store_wait_read<0>();
          }
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // this warp's generic accesses before TMA's next write
          __syncwarp();
          if (lane == 0) xissue(vi + NXB);
        }
        if (part) {
          asm volatile("bar.sync 1, %0;" ::"n"(EPT) : "memory");  // all epilogue warps
          for (int i = et; i < 3 * HID && tile < n_tiles; i += EPT) {
            const int q = i / HID, j = i - q * HID;
            part[(((size_t)ag * n_tiles + tile) * 3 + q) * HID + j] = (S.wpart[0][q][j] + S.wpart[1][q][j]) + (S.wpart[2][q][j] + S.wpart[3][q][j]);
          }
          asm volatile("bar.sync 1, %0;" ::"n"(EPT) : "memory");  // (wpart is rewritten by the next tile)
        }
      }
      if (next_differs) cset ^= 1;
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // this warp's stores have left shared memory
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  cluster_sync_all();  // (the peer's last commits arrive on this CTA's barriers: do not exit under them)
  if (warp == 1) {
    if constexpr (PAIR) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(2 * TCN) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(2 * TCN) : "memory");
  }
}

static int tc_grid(int M, int n_agents) {  // persistent: one CTA per SM (or per tile when there are fewer)
  static int sms = [] {
    int dev = 0, n = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    return n;
  }();
  const int pairs = (((M + TCM - 1) / TCM + 1) / 2) * n_agents;  // clusters of 2 CTAs, one tile pair at a time
  const int clusters = pairs < sms / 2 ? pairs : sms / 2;
  return 2 * clusters;
}

// ---- host side: tensor maps (driver entry point fetched through the runtime: libb2rl links no libcuda) -------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return (EncodeTiledFn)p;
  }();
  return fn;
}
// [n_agents][rows][cols] fp32, row pitch `ld` floats, `agent_stride` floats between agents; box = 32 columns (128 bytes =
// the swizzle span) x box_rows rows x 1 agent
static bool make_map(CUtensorMap* m, const float* base, int64_t rows, int64_t cols, int64_t ld, int box_rows, int n_agents,
                     int64_t agent_stride) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return false;
  if (n_agents <= 1) agent_stride = rows * ld;  // (one agent: any legal stride)
  const cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)(n_agents < 1 ? 1 : n_agents)};
  const cuuint64_t strides[2] = {(cuuint64_t)ld * sizeof(float), (cuuint64_t)agent_stride * sizeof(float)};
  const cuuint32_t box[3] = {(cuuint32_t)TCK, (cuuint32_t)box_rows, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  return fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// MN-major operand [n_agents][rows = k][cols] fp32 (the arena's forward-layout w1t): boxes of 32 columns x 32 rows x 1 agent
// in the SWIZZLE_128B_ATOM_32B pattern (tc_wgrad.cu); rows beyond `rows` are zero-filled
static bool make_map_mn(CUtensorMap* m, const float* base, int64_t rows, int64_t cols, int64_t ld, int n_agents, int64_t agent_stride) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return false;
  if (n_agents <= 1) agent_stride = rows * ld;
  const cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)(n_agents < 1 ? 1 : n_agents)};
  const cuuint64_t strides[2] = {(cuuint64_t)ld * sizeof(float), (cuuint64_t)agent_stride * sizeof(float)};
  const cuuint32_t box[3] = {32, (cuuint32_t)TCK, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  return fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// lo part of a weight matrix for the 3xTF32 mode: lo = w - tf32_truncate(w)
__global__ void tc_split_lo_kernel(const float* __restrict__ w, float* __restrict__ lo, int n, long long ps, long long ls) {
  w += (size_t)blockIdx.y * ps, lo += (size_t)blockIdx.y * ls;  // stacked agents: blockIdx.y = agent
  const int n4 = n >> 2;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += gridDim.x * blockDim.x)
    reinterpret_cast<float4*>(lo)[i] = tf32_lo4(__ldg(reinterpret_cast<const float4*>(w) + i));
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) lo[4 * n4 + threadIdx.x] = tf32_lo(w[4 * n4 + threadIdx.x]);
}
cudaError_t launch_tc_split_lo(const float* w, float* lo, int n, const Stk& k, cudaStream_t st) {
  int ctas = (n / 4 + 255) / 256;
  ctas = ctas < 1 ? 1 : (ctas > 592 ? 592 : ctas);
  tc_split_lo_kernel<<<dim3(ctas, k.n), 256, 0, st>>>(w, lo, n, k.ps, k.ls);
  return cudaGetLastError();
}

template <typename K>
static cudaError_t tc_opt_in(K kernel, size_t bytes) {
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes + 1024);
}
cudaError_t init_tc() {
  cudaError_t e = tc_opt_in(tc_linear_kernel<0, 0>, sizeof(TcSmemT<0, 0>));
  if (e == cudaSuccess) e = tc_opt_in(tc_linear_kernel<2, 0>, sizeof(TcSmemT<2, 0>));
  if (e == cudaSuccess) e = tc_opt_in(tc_linear_kernel<0, 1>, sizeof(TcSmemT<0, 1>));
  if (e == cudaSuccess) e = tc_opt_in(tc_linear_kernel<2, 1>, sizeof(TcSmemT<2, 1>));
  if (e == cudaSuccess) e = tc_opt_in(tc_linear_kernel<0, 2>, sizeof(TcSmemT<0, 2>));
  if (e == cudaSuccess) e = tc_opt_in(tc_linear_kernel<2, 2>, sizeof(TcSmemT<2, 2>));
  if (e == cudaSuccess) e = tc_opt_in(tc_linear_kernel<1, 0>, sizeof(TcSmemT<1, 0>));
  if (e == cudaSuccess) e = tc_opt_in(tc_linear_kernel<1, 2>, sizeof(TcSmemT<1, 2>));
  cudaFuncAttributes fa;
  if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, tc_split_lo_kernel);
  return e;
}

// Wlo: the precomputed lo part of W (tc_split_lo) => 3xTF32; == W => 3xTF32 with the weights' lo parts made in the kernel;
// NULL => plain TF32
cudaError_t launch_tc_linear(const float* X, int64_t ldx, int M, const float* W, const float* Wlo, const float* bias,
                             const float* g, const float* be, int ln, int relu, float* H, float* XH, float* stat,
                             const b2rl_wide_q_t* head, const Stk& k, cudaStream_t st) {
  b2rl_wide_q_t q = {};
  if (head) q = *head;
  CUtensorMap ma, mb, ml;  // (the weight maps have boxes of HALF a slab: each CTA of a cluster loads one and multicasts it)
  if (!make_map(&ma, X, M, HID, ldx, TCM, k.n, (int64_t)M * ldx) || !make_map(&mb, W, HID, HID, HID, TCN / 2, k.n, k.ps))
    return cudaErrorInvalidValue;
  CUtensorMap mh = ma, mxh = ma;  // outputs: boxes of 32 rows x 32 columns (TMA stores of the epilogue's staging tiles)
  if ((H && !make_map(&mh, H, M, HID, HID, 32, k.n, (int64_t)M * HID)) || (XH && !make_map(&mxh, XH, M, HID, HID, 32, k.n, (int64_t)M * HID)))
    return cudaErrorInvalidValue;
  const dim3 grid(tc_grid(M, k.n)), block(TcCfg<0, 0>::THREADS);
  float2* st2 = reinterpret_cast<float2*>(stat);
  float* none = nullptr;
  if (Wlo == W)
    return launch_k(tc_linear_kernel<0, 2>, grid, dim3(TcCfg<0, 2>::THREADS), -2, sizeof(TcSmemT<0, 2>) + 1024, st, ma, mb, mb, ma, mh, mxh, M, 0, bias, g, be, ln, relu, H, XH,
                    st2, none, q, k);
  if (Wlo) {
    if (!make_map(&ml, Wlo, HID, HID, HID, TCN / 2, k.n, k.ls)) return cudaErrorInvalidValue;
    return launch_k(tc_linear_kernel<0, 1>, grid, dim3(TcCfg<0, 1>::THREADS), -2, sizeof(TcSmemT<0, 1>) + 1024, st, ma, mb, ml, ma, mh, mxh, M, 0, bias, g, be, ln, relu, H, XH,
                    st2, none, q, k);
  }
  return launch_k(tc_linear_kernel<0, 0>, grid, block, -2, sizeof(TcSmemT<0, 0>) + 1024, st, ma, mb, mb, ma, mh, mxh, M, 0, bias, g, be, ln, relu, H, XH, st2,
                  none, q, k);
}
// First layer on the tensor cores: X [M][K] (row pitch ldx), w1t [K][256] forward layout; x3: 3xTF32 with both lo parts made
// in the kernel, else plain TF32.
cudaError_t launch_tc_first(const float* X, int64_t ldx, int M, int K, const float* w1t, const float* bias, const float* g,
                            const float* be, int ln, float* H, float* XH, float* stat, int x3, const Stk& k, cudaStream_t st) {
  CUtensorMap ma, mb;
  if (!make_map(&ma, X, M, K, ldx, TCM, k.n, (int64_t)M * ldx) || !make_map_mn(&mb, w1t, K, HID, HID, k.n, k.ps))
    return cudaErrorInvalidValue;
  CUtensorMap mh = ma, mxh = ma;
  if ((H && !make_map(&mh, H, M, HID, HID, 32, k.n, (int64_t)M * HID)) || (XH && !make_map(&mxh, XH, M, HID, HID, 32, k.n, (int64_t)M * HID)))
    return cudaErrorInvalidValue;
  const dim3 grid(tc_grid(M, k.n)), block(TcCfg<1, 0>::THREADS);
  float2* st2 = reinterpret_cast<float2*>(stat);
  float* none = nullptr;
  const b2rl_wide_q_t q = {};
  const int kb = (K + TCK - 1) / TCK;
  if (x3)
    return launch_k(tc_linear_kernel<1, 2>, grid, block, -2, sizeof(TcSmemT<1, 2>) + 1024, st, ma, mb, mb, ma, mh, mxh, M, kb, bias, g, be, ln, 1, H, XH,
                    st2, none, q, k);
  return launch_k(tc_linear_kernel<1, 0>, grid, block, -2, sizeof(TcSmemT<1, 0>) + 1024, st, ma, mb, mb, ma, mh, mxh, M, kb, bias, g, be, ln, 1, H, XH, st2,
                  none, q, k);
}
cudaError_t launch_tc_linear_bwd(const float* DZ2, int M, const float* w2t, const float* w2t_lo, const float* xh1,
                                 const float* stat1, const float* g1, const float* be1, int ln, float* DZ1, float* part,
                                 const Stk& k, cudaStream_t st) {
  CUtensorMap ma, mb, ml, mx, mh;  // mx: x-hat in boxes of 32 rows x 32 columns (the epilogue warps' rings)
  if (!make_map(&ma, DZ2, M, HID, HID, TCM, k.n, (int64_t)M * HID) || !make_map(&mb, w2t, HID, HID, HID, TCN / 2, k.n, k.ps) ||
      !make_map(&mx, xh1, M, HID, HID, 32, k.n, (int64_t)M * HID) || !make_map(&mh, DZ1, M, HID, HID, 32, k.n, (int64_t)M * HID))
    return cudaErrorInvalidValue;
  const dim3 grid(tc_grid(M, k.n)), block(TcCfg<2, 0>::THREADS);
  float* xh = const_cast<float*>(xh1);
  float2* st1 = reinterpret_cast<float2*>(const_cast<float*>(stat1));
  const float* none = nullptr;
  const b2rl_wide_q_t q = {};
  if (w2t_lo == w2t)
    return launch_k(tc_linear_kernel<2, 2>, grid, block, -2, sizeof(TcSmemT<2, 2>) + 1024, st, ma, mb, mb, mx, mh, mh, M, 0, none, g1, be1, ln, 0, DZ1, xh, st1,
                    part, q, k);
  if (w2t_lo) {
    if (!make_map(&ml, w2t_lo, HID, HID, HID, TCN / 2, k.n, k.ls)) return cudaErrorInvalidValue;
    return launch_k(tc_linear_kernel<2, 1>, grid, block, -2, sizeof(TcSmemT<2, 1>) + 1024, st, ma, mb, ml, mx, mh, mh, M, 0, none, g1, be1, ln, 0, DZ1, xh, st1,
                    part, q, k);
  }
  return launch_k(tc_linear_kernel<2, 0>, grid, block, -2, sizeof(TcSmemT<2, 0>) + 1024, st, ma, mb, mb, mx, mh, mh, M, 0, none, g1, be1, ln, 0, DZ1, xh, st1, part, q, k);
}

}  // namespace b2rl
