// replay.cu — GPU-resident replay buffer: uniform index sample + transition gather, and the
// round-robin write. Replaces torchrl's TensorDictReplayBuffer(LazyTensorStorage) as the reference
// uses it (main.py:167-171; sample at orchestrator.py:338, extend at orchestrator.py:100-113):
// there, one randint kernel + one `index` kernel per key (6-7) on SoA tensors whose rows are not
// 16-byte aligned (11 floats), then 7 more copies into the CUDA graph's static inputs.
// Here a transition is ONE padded row (row_stride % 4 == 0 floats), so the whole gather is a
// stream of 128-bit loads/stores: the lanes of a warp move the 16-byte chunks of whole rows.
// HBM-bound: algorithmic bytes per sampled transition = 2 * row_stride * 4 (+ 8 for the index).
#include "common.cuh"
#include "rng.cuh"

namespace b2rl {

// Lanes <-> 16-byte chunks of whole rows: a warp takes 32 / chunks rows per group when a row has at most 32 chunks
// (Hopper: 7 chunks, 4 rows = 28 lanes), one row at a time otherwise (Humanoid: 193 chunks). The lane that owns chunk 0 of
// a row draws its index — ONE Philox-4x32-10 per row, not one per chunk — and the row's other lanes take it by shuffle.
// U groups per trip: every lane has U independent 16-byte loads in flight before the first store.
template <int U>
__global__ void __launch_bounds__(256)
gather_kernel(const float* __restrict__ storage, int64_t storage_agent_stride, int64_t size, int row_stride,
              int batch, const int64_t* __restrict__ idx_in, int64_t* __restrict__ idx_out,
              float* __restrict__ rows_out, uint64_t seed, const uint64_t* __restrict__ counters, int step_counter,
              int agent_base) {
  pdl_enter();
  const int agent = blockIdx.y;
  const int chunks = row_stride >> 2;
  const uint64_t step = counters ? counters[(size_t)agent * 8 + step_counter] : 0;
  if (size == 0) size = (int64_t)counters[(size_t)agent * 8 + B2RL_CTR_SIZE];  // buffer still filling under a graph
  const float* src = storage + (size_t)agent * storage_agent_stride;
  float* dst = rows_out + (size_t)agent * batch * row_stride;
  const int64_t* iin = idx_in ? idx_in + (size_t)agent * batch : nullptr;
  int64_t* iout = idx_out ? idx_out + (size_t)agent * batch : nullptr;
  const uint32_t gid = (uint32_t)(agent_base + agent);
  const int lane = threadIdx.x & 31;
  const int warp = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), n_warps = (int)((gridDim.x * blockDim.x) >> 5);
  auto draw = [&](int b) -> int64_t { return iin ? iin[b] : philox_index(seed, (uint32_t)b, step, gid, (uint64_t)size); };
  if (chunks <= 32) {
    const int rpw = 32 / chunks, my_r = lane / chunks, c = lane - my_r * chunks;
    const bool active = my_r < rpw;
    const int owner = active ? my_r * chunks : 0;  // the lane holding chunk 0 of this lane's row
    for (int b0 = warp * rpw * U; b0 < batch; b0 += n_warps * rpw * U) {
      float4 v[U];
      int64_t r[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int b = b0 + u * rpw + my_r;
        const bool ok = active && b < batch;
        int64_t mine = (ok && c == 0) ? draw(b) : 0;
        mine = __shfl_sync(0xffffffffu, mine, owner);
        r[u] = mine;
        if (ok) v[u] = ld_stream4(src + ((size_t)mine * row_stride + 4 * c));
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int b = b0 + u * rpw + my_r;
        if (active && b < batch) {
          st_stream4(dst + ((size_t)b * row_stride + 4 * c), v[u]);
          if (iout && c == 0) iout[b] = r[u];
        }
      }
    }
  } else {
    for (int b = warp; b < batch; b += n_warps) {
      int64_t r = lane == 0 ? draw(b) : 0;
      r = __shfl_sync(0xffffffffu, r, 0);
      if (iout && lane == 0) iout[b] = r;
      const float* s = src + (size_t)r * row_stride;
      float* d = dst + (size_t)b * row_stride;
      for (int c0 = lane; c0 < chunks; c0 += 32 * 4) {
        float4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (c0 + 32 * u < chunks) v[u] = ld_stream4(s + 4 * (c0 + 32 * u));
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (c0 + 32 * u < chunks) st_stream4(d + 4 * (c0 + 32 * u), v[u]);
      }
    }
  }
}

// a counter must advance only after every CTA of gather_kernel has read it: separate tiny launch,
// used when the sampler is driven on its own (inside the fused iteration the draw is keyed on the
// critic step counter, which wgrad.cu advances, so no extra launch is needed there)
__global__ void bump_sample_kernel(uint64_t* counters, int n_agents, int which) {
  pdl_enter();
  const int a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a < n_agents) counters[(size_t)a * 8 + which] += 1ULL;
}

__global__ void __launch_bounds__(256)
extend_kernel(float* __restrict__ storage, int64_t capacity, int64_t cursor, int row_stride,
              const float* __restrict__ new_rows, int n) {
  pdl_enter();
  const int chunks = row_stride >> 2;
  const int64_t total = (int64_t)n * chunks;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int b = (int)(i / chunks), c = (int)(i - (int64_t)b * chunks);
    const int64_t r = (cursor + b) % capacity;
    st_stream4(storage + ((size_t)r * row_stride + 4 * c), ld_stream4(new_rows + ((size_t)b * row_stride + 4 * c)));
  }
}

// graph-capturable write: cursor and size live in the device counters; the last CTA to finish advances them.
// Stacked agents: grid y = agent g, with its own storage slice, source rows [g][n][row_stride] and counters[g*8 + ..];
// the last CTA of agent g's grid row advances g's cursor and size and resets g's ticket.
__global__ void __launch_bounds__(256, 8)  // 8 resident CTAs per SM (launch_extend_dev's grid): <= 32 registers
extend_dev_kernel(float* __restrict__ storage, int64_t storage_agent_stride, int64_t capacity, int row_stride,
                  const float* __restrict__ new_rows, int n, uint64_t* __restrict__ counters) {
  pdl_enter();
  const int g = blockIdx.y;
  storage += (size_t)g * storage_agent_stride;
  new_rows += (size_t)g * n * row_stride;
  counters += (size_t)g * 8;
  const int chunks = row_stride >> 2;
  const int64_t total = (int64_t)n * chunks;
  const int64_t cursor = (int64_t)counters[B2RL_CTR_CURSOR];
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int b = (int)(i / chunks), c = (int)(i - (int64_t)b * chunks);
    const int64_t r = (cursor + b) % capacity;
    st_stream4(storage + ((size_t)r * row_stride + 4 * c), ld_stream4(new_rows + ((size_t)b * row_stride + 4 * c)));
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned long long ticket = atomicAdd((unsigned long long*)&counters[B2RL_CTR_XTICKET], 1ULL);
    if (ticket == (unsigned long long)gridDim.x - 1) {  // every CTA has read the cursor
      counters[B2RL_CTR_CURSOR] = (uint64_t)((cursor + n) % capacity);
      const uint64_t size = counters[B2RL_CTR_SIZE] + (uint64_t)n;
      counters[B2RL_CTR_SIZE] = size < (uint64_t)capacity ? size : (uint64_t)capacity;
      counters[B2RL_CTR_XTICKET] = 0;
    }
  }
}

cudaError_t launch_extend_dev(float* storage, int64_t storage_agent_stride, int64_t capacity, b2rl_rowfmt_t fmt,
                              const float* new_rows, int n, int n_agents, uint64_t* counters, cudaStream_t st) {
  const int64_t total = (int64_t)n * (fmt.row_stride >> 2);
  int ctas = (int)((total + 255) / 256);
  if (ctas > 148 * 8) ctas = 148 * 8;
  if (ctas < 1) ctas = 1;
  return launch_k(extend_dev_kernel, dim3(ctas, n_agents), dim3(256), 1, 0, st, storage, storage_agent_stride, capacity,
                  (int)fmt.row_stride, new_rows, n, counters);
}

// last node of a captured step: log block -> pinned host memory, then the sequence number the host polls
__global__ void publish_kernel(const float* __restrict__ out, int n, float* host_out, uint64_t* seq_dev,
                               volatile uint64_t* host_seq) {
  pdl_enter();
  for (int i = threadIdx.x; i < n; i += blockDim.x) host_out[i] = out[i];
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    const uint64_t s = *seq_dev + 1ULL;
    *seq_dev = s;
    *host_seq = s;
  }
}
cudaError_t launch_publish(const float* out, int n_agents, float* host_out, uint64_t* seq_dev, uint64_t* host_seq,
                           cudaStream_t st) {
  return launch_k(publish_kernel, dim3(1), dim3(64), 1, 0, st, out, n_agents * 8, host_out, seq_dev, (volatile uint64_t*)host_seq);
}

cudaError_t init_replay() {
  cudaFuncAttributes fa;
  cudaError_t e = cudaFuncGetAttributes(&fa, gather_kernel<1>);
  if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, gather_kernel<4>);
  if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, bump_sample_kernel);
  if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, extend_kernel);
  if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, extend_dev_kernel);
  if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, publish_kernel);
  return e;
}

cudaError_t launch_gather(const float* storage, int64_t storage_agent_stride, int64_t size, b2rl_rowfmt_t fmt,
                          int batch, int n_agents, const int64_t* idx_in, int64_t* idx_out, float* rows_out,
                          uint64_t seed, uint64_t* counters, int step_counter, int bump, int agent_base, cudaStream_t st) {
  // a warp moves 32 / chunks rows per group (or one row when a row is longer than a warp), U groups per trip: small
  // batches spread over as many warps as they have groups (latency), large ones keep 4 loads in flight per lane (bandwidth)
  const int chunks = fmt.row_stride >> 2, rpw = chunks <= 32 ? 32 / chunks : 1;
  const bool big = (int64_t)batch * n_agents * chunks >= (int64_t)148 * 8 * 256 * 4;
  const int64_t warps = ((int64_t)batch + rpw * (big && chunks <= 32 ? 4 : 1) - 1) / (rpw * (big && chunks <= 32 ? 4 : 1));
  int ctas = (int)((warps + 7) / 8);
  if (ctas > 148 * 8) ctas = 148 * 8;  // 8 resident CTAs of 256 threads per SM, grid-stride beyond
  if (ctas < 1) ctas = 1;
  cudaError_t e;
  if (big)
    e = launch_k(gather_kernel<4>, dim3(ctas, n_agents), dim3(256), 1, 0, st, storage, storage_agent_stride, size, (int)fmt.row_stride,
                 batch, idx_in, idx_out, rows_out, seed, (const uint64_t*)counters, step_counter, agent_base);
  else
    e = launch_k(gather_kernel<1>, dim3(ctas, n_agents), dim3(256), 1, 0, st, storage, storage_agent_stride, size, (int)fmt.row_stride,
                 batch, idx_in, idx_out, rows_out, seed, (const uint64_t*)counters, step_counter, agent_base);
  if (e != cudaSuccess || idx_in || !counters || !bump) return e;
  return launch_k(bump_sample_kernel, dim3((n_agents + 127) / 128), dim3(128), 1, 0, st, counters, n_agents, step_counter);
}

cudaError_t launch_extend(float* storage, int64_t capacity, int64_t cursor, b2rl_rowfmt_t fmt, const float* new_rows,
                          int n, cudaStream_t st) {
  const int64_t total = (int64_t)n * (fmt.row_stride >> 2);
  int ctas = (int)((total + 255) / 256);
  if (ctas > 148 * 8) ctas = 148 * 8;
  if (ctas < 1) ctas = 1;
  return launch_k(extend_kernel, dim3(ctas), dim3(256), 1, 0, st, storage, capacity, cursor, (int)fmt.row_stride, new_rows, n);
}

}  // namespace b2rl
