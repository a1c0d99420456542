// api.cu — the extern "C" surface declared in include/b2rl.h: argument validation, error text,
// kernel launches. No allocation, no synchronisation, no host read of device memory.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "common.cuh"

namespace b2rl {
cudaError_t launch_critic_fused(const b2rl_update_args_t&, cudaStream_t);
cudaError_t launch_actor_fused(const b2rl_update_args_t&, cudaStream_t);
cudaError_t launch_alpha(const b2rl_update_args_t&, float, cudaStream_t);
cudaError_t launch_alpha_adam(float*, uint64_t*, int, float, const b2rl_agent_hp_t*, float, float*, cudaStream_t);
cudaError_t launch_predict(const b2rl_update_args_t&, const float*, int, int, float, uint64_t, float*, cudaStream_t);
cudaError_t launch_wgrad(const b2rl_update_args_t&, int, int, const b2rl_adam_args_t*, cudaStream_t, int skip_vec = 0);
cudaError_t launch_adam(const b2rl_adam_args_t&, cudaStream_t);
cudaError_t launch_sumsq(const float*, int64_t, int64_t, int64_t, int64_t, int, float*, float*, cudaStream_t);
cudaError_t launch_bump(uint64_t*, int, int, cudaStream_t);
cudaError_t launch_gather(const float*, int64_t, int64_t, b2rl_rowfmt_t, int, int, const int64_t*, int64_t*, float*,
                          uint64_t, uint64_t*, int, int, int, cudaStream_t);
cudaError_t launch_extend(float*, int64_t, int64_t, b2rl_rowfmt_t, const float*, int, cudaStream_t);
cudaError_t launch_publish(const float*, int, float*, uint64_t*, uint64_t*, cudaStream_t);
cudaError_t launch_extend_dev(float*, int64_t, int64_t, b2rl_rowfmt_t, const float*, int, int, uint64_t*, cudaStream_t);
int max_in_dim_critic();
int max_in_dim_actor();
cudaError_t init_critic();
cudaError_t init_actor();
cudaError_t init_wgrad();
cudaError_t init_adam();
cudaError_t init_replay();
cudaError_t init_tc();
cudaError_t init_wide();
cudaError_t init_tc_wgrad();
int tc_wgrad_splits(int, int, int);
cudaError_t launch_tc_wgrad(const float*, int64_t, int, int, const float*, int, float*, float*, float*, int, unsigned long long*,
                            const Stk&, int, cudaStream_t);
cudaError_t launch_wide_first(const float*, int64_t, int, int, const float*, const float*, const float*, const float*, int, float*,
                              float*, float*, const Stk&, cudaStream_t);
cudaError_t launch_tc_linear_bwd(const float*, int, const float*, const float*, const float*, const float*, const float*,
                                 const float*, int, float*, float*, const Stk&, cudaStream_t);
cudaError_t launch_wide_policy_head(const b2rl_wide_policy_t&, const Stk&, cudaStream_t);
cudaError_t launch_wide_q_head(const b2rl_wide_q_t&, const Stk&, cudaStream_t);
cudaError_t launch_wide_ln_bwd(const float*, int, const float*, const float*, const float*, const float*, const float*, int, int,
                               float*, float*, float*, const Stk&, cudaStream_t);
cudaError_t launch_wide_actor_loss(const float*, const float*, const float*, const float*, int, int, float*, float*, float*,
                                   const Stk&, cudaStream_t);
cudaError_t launch_wide_dqda(const float*, const float*, int, int, float*, const Stk&, cudaStream_t);
cudaError_t launch_wide_actor_head_bwd(const float*, const float*, const float*, const float*, const float*, const float*, int, int,
                                       int, float*, float*, const Stk&, cudaStream_t);
cudaError_t launch_wide_actor_scalars(const float*, const float*, int, int, int, int, const float*, float*, int64_t, float*,
                                      const Stk&, cudaStream_t);
cudaError_t launch_wide_alpha_grad(const float*, int, float, float*, const Stk&, cudaStream_t);
cudaError_t launch_wide_colsum(const float*, int, float*, int64_t, int64_t, int64_t, int, const Stk&, cudaStream_t);
cudaError_t launch_wide_colsum_multi(const ColsumJobs&, int, float*, const Stk&, cudaStream_t);
cudaError_t launch_wide_critic_scalars(const float*, const float*, int, const float*, const float*, int, float*, int64_t, int64_t,
                                       float*, const Stk&, cudaStream_t);
cudaError_t launch_tc_linear(const float*, int64_t, int, const float*, const float*, const float*, const float*, const float*, int,
                             int, float*, float*, float*, const b2rl_wide_q_t*, const Stk&, cudaStream_t);
cudaError_t launch_tc_split_lo(const float*, float*, int, const Stk&, cudaStream_t);
cudaError_t launch_tc_first(const float*, int64_t, int, int, const float*, const float*, const float*, const float*, int, float*, float*,
                            float*, int, const Stk&, cudaStream_t);
}  // namespace b2rl

namespace b2rl {
bool pdl_enabled() {
  static const bool on = [] {
    const char* e = getenv("B2RL_PDL");
    return !(e && e[0] == '0');
  }();
  return on;
}
}  // namespace b2rl

static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
static int check_launch(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return B2RL_OK;
  return fail(B2RL_E_LAUNCH, "%s: %s", what, cudaGetErrorString(e));
}
static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
// a per-agent hyperparameter table (NULL = the scalars): float-aligned device rows
static int check_hp(const b2rl_agent_hp_t* hp, const char* what) {
  if (hp && (reinterpret_cast<uintptr_t>(hp) & 3u)) return fail(B2RL_E_INVALID, "%s: agent_hp must be 4-byte aligned", what);
  return B2RL_OK;
}
// the stacked-agents descriptor of the wide path (NULL = one learner)
static int check_stack(const b2rl_stack_t* s, const char* what) {
  if (!s) return B2RL_OK;
  if (s->n_agents < 1 || s->n_agents > 65535) return fail(B2RL_E_INVALID, "%s: stack.n_agents %d out of range", what, s->n_agents);
  if (s->agent_base < 0 || (int64_t)s->agent_base + s->n_agents > (1 << 30)) return fail(B2RL_E_INVALID, "%s: agent ids must stay below 2^30", what);
  if (s->param_stride < 0 || s->lo_stride < 0 || s->alpha_stride < 0 || s->counters_stride < 0 || s->out_stride < 0 ||
      (s->param_stride & 3) || (s->lo_stride & 3))
    return fail(B2RL_E_INVALID, "%s: stack strides must be >= 0 (param / lo strides multiples of 4 floats)", what);
  return check_hp(s->agent_hp, what);
}
using b2rl::make_stk;

static int check_fmt(const b2rl_rowfmt_t& f) {
  if (f.ob_dim < 1 || f.ac_dim < 1) return fail(B2RL_E_INVALID, "row format: ob_dim/ac_dim must be >= 1");
  if (f.ac_dim > B2RL_MAX_OUT / 2) return fail(B2RL_E_INVALID, "ac_dim %d > %d", f.ac_dim, B2RL_MAX_OUT / 2);
  const int max_in = b2rl::max_in_dim_critic() < b2rl::max_in_dim_actor() ? b2rl::max_in_dim_critic() : b2rl::max_in_dim_actor();
  if (f.ob_dim + f.ac_dim > max_in)  // the fused kernels keep their input tiles in shared memory
    return fail(B2RL_E_INVALID, "ob_dim + ac_dim %d > %d", f.ob_dim + f.ac_dim, max_in);
  if (f.row_stride % 4 != 0 || f.row_stride < 2 * f.ob_dim + f.ac_dim + 2)
    return fail(B2RL_E_INVALID, "row_stride %d must be a multiple of 4 and >= 2*ob+ac+2", f.row_stride);
  return B2RL_OK;
}

static int check_net(const b2rl_net_t& n, const char* name, bool need_w2n) {
  if (n.in_dim < 1 || n.in_dim > 1024 || n.out_dim < 1 || n.out_dim > B2RL_MAX_OUT)
    return fail(B2RL_E_INVALID, "%s: in_dim %d / out_dim %d out of range", name, n.in_dim, n.out_dim);
  const int64_t offs[] = {n.w1t, n.b1, n.w2t, n.b2, n.w3, n.b3, n.begin, n.end};
  for (int64_t o : offs)
    if (o < 0 || (o & 3)) return fail(B2RL_E_INVALID, "%s: tensor offsets must be >= 0 and multiples of 4 floats", name);
  if (n.layer_norm && ((n.g1 | n.be1 | n.g2 | n.be2) < 0 || ((n.g1 | n.be1 | n.g2 | n.be2) & 3)))
    return fail(B2RL_E_INVALID, "%s: LayerNorm offsets invalid", name);
  if (need_w2n && (n.w2n < 0 || (n.w2n & 3))) return fail(B2RL_E_INVALID, "%s: needs the w2n shadow", name);
  return B2RL_OK;
}

static int check_update(const b2rl_update_args_t* a, bool actor_step) {
  if (!a) return fail(B2RL_E_INVALID, "null args");
  if (int rc = check_fmt(a->fmt)) return rc;
  if (a->batch < 1 || a->batch > (1 << 24)) return fail(B2RL_E_INVALID, "batch %d out of range", a->batch);
  if (a->n_agents < 1 || a->n_agents > 65535) return fail(B2RL_E_INVALID, "n_agents %d out of range", a->n_agents);
  if (a->agent_base < 0 || (int64_t)a->agent_base + a->n_agents > (1 << 30)) return fail(B2RL_E_INVALID, "agent ids must stay below 2^30");
  if (!a->arena || !a->rows || !a->min_ac || !a->max_ac || !a->counters || !a->workspace || !a->out)
    return fail(B2RL_E_INVALID, "null device pointer in update args");
  if (!aligned16(a->arena) || !aligned16(a->workspace) || (a->region_stride & 3) || (a->arena_agent_stride & 3) ||
      (a->workspace_agent_stride & 3))
    return fail(B2RL_E_INVALID, "arena/workspace must be 16-byte aligned with strides that are multiples of 4 floats");
  if (!a->hp.td3 && !a->log_alpha) return fail(B2RL_E_INVALID, "SAC needs log_alpha");
  if (int rc = check_hp(a->agent_hp, "update args")) return rc;
  if (int rc = check_net(a->actor, "actor", actor_step)) return rc;
  if (int rc = check_net(a->critic[0], "critic[0]", true)) return rc;
  if (int rc = check_net(a->critic[1], "critic[1]", true)) return rc;
  const int want_out = a->hp.td3 ? a->fmt.ac_dim : 2 * a->fmt.ac_dim;
  if (a->actor.in_dim != a->fmt.ob_dim || a->actor.out_dim != want_out)
    return fail(B2RL_E_INVALID, "actor dims (%d -> %d) do not match the row format / algorithm", a->actor.in_dim, a->actor.out_dim);
  for (int k = 0; k < 2; ++k)
    if (a->critic[k].in_dim != a->fmt.ob_dim + a->fmt.ac_dim || a->critic[k].out_dim != 1)
      return fail(B2RL_E_INVALID, "critic[%d] dims (%d -> %d) do not match the row format", k, a->critic[k].in_dim, a->critic[k].out_dim);
  if (a->storage && (!aligned16(a->storage) || (a->storage_agent_stride & 3) || a->storage_size < 0))
    return fail(B2RL_E_INVALID, "storage must be 16-byte aligned, its agent stride a multiple of 4 floats");
  if (a->new_rows) {
    if (!a->storage || a->n_agents != 1) return fail(B2RL_E_INVALID, "new_rows needs in-kernel sampling (storage) and a single learner");
    if (!aligned16(a->new_rows) || a->capacity < 1 || a->n_new < 1 || a->n_new > a->capacity)
      return fail(B2RL_E_INVALID, "new_rows: 16-byte aligned, 1 <= n_new <= capacity");
  }
  return B2RL_OK;
}

// ---- FFMA probe ----------------------------------------------------------------------------------
namespace b2rl {
__global__ void __launch_bounds__(256) ffma_probe_kernel(float* sink, int iters) {
  float a[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) a[i] = 1.0f + 1e-3f * (threadIdx.x + i);
  const float m = 0.999f, c = 1e-3f;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 16; ++i) a[i] = fmaf(a[i], m, c);
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 16; ++i) s += a[i];
  if (s == 12345.678f) sink[0] = s;  // never true; keeps the chain alive
}
}  // namespace b2rl

extern "C" {

int b2rl_version(void) { return B2RL_VERSION; }
const char* b2rl_last_error(void) { return g_err; }

int b2rl_init(void) {
  cudaError_t e = b2rl::init_critic();
  if (e == cudaSuccess) e = b2rl::init_actor();
  if (e == cudaSuccess) e = b2rl::init_wgrad();
  if (e == cudaSuccess) e = b2rl::init_adam();
  if (e == cudaSuccess) e = b2rl::init_replay();
  if (e == cudaSuccess) e = b2rl::init_tc();
  if (e == cudaSuccess) e = b2rl::init_wide();
  if (e == cudaSuccess) e = b2rl::init_tc_wgrad();
  if (e == cudaSuccess) {
    cudaFuncAttributes fa;
    e = cudaFuncGetAttributes(&fa, b2rl::ffma_probe_kernel);
  }
  return check_launch(e, "b2rl_init");
}

int64_t b2rl_workspace_floats(int32_t batch) {
  if (batch < 1) return -1;
  return b2rl::ws_floats(batch);
}

int b2rl_replay_sample_gather(const float* storage, int64_t storage_agent_stride, int64_t size, b2rl_rowfmt_t fmt,
                              int32_t batch, int32_t n_agents, const int64_t* idx_in, int64_t* idx_out,
                              float* rows_out, uint64_t seed, uint64_t* counters, int32_t step_counter, int32_t bump,
                              int32_t agent_base, void* stream) {
  if (int rc = check_fmt(fmt)) return rc;
  if (!storage || !rows_out) return fail(B2RL_E_INVALID, "null storage / rows_out");
  if (!aligned16(storage) || !aligned16(rows_out)) return fail(B2RL_E_INVALID, "storage and rows_out must be 16-byte aligned");
  if (batch < 1 || n_agents < 1 || n_agents > 65535) return fail(B2RL_E_INVALID, "bad batch / n_agents");
  if (size < 0 || size >= (1LL << 32)) return fail(B2RL_E_INVALID, "size %lld must be in [0, 2^32)", (long long)size);
  if ((!idx_in || size == 0) && !counters) return fail(B2RL_E_INVALID, "device-side sampling needs the counters");
  if (step_counter < 0 || step_counter > 3) return fail(B2RL_E_INVALID, "bad step_counter");
  if (storage_agent_stride & 3) return fail(B2RL_E_INVALID, "storage_agent_stride must be a multiple of 4 floats");
  return check_launch(b2rl::launch_gather(storage, storage_agent_stride, size, fmt, batch, n_agents, idx_in, idx_out,
                                          rows_out, seed, counters, step_counter, bump, agent_base, (cudaStream_t)stream),
                      "replay_sample_gather");
}

int b2rl_replay_extend(float* storage, int64_t capacity, int64_t cursor, b2rl_rowfmt_t fmt, const float* new_rows,
                       int32_t n, void* stream) {
  if (int rc = check_fmt(fmt)) return rc;
  if (!storage || !new_rows || !aligned16(storage) || !aligned16(new_rows))
    return fail(B2RL_E_INVALID, "storage / new_rows must be non-null and 16-byte aligned");
  if (capacity < 1 || cursor < 0 || cursor >= capacity || n < 0 || n > capacity)
    return fail(B2RL_E_INVALID, "bad capacity / cursor / n");
  if (n == 0) return B2RL_OK;
  return check_launch(b2rl::launch_extend(storage, capacity, cursor, fmt, new_rows, n, (cudaStream_t)stream), "replay_extend");
}

int b2rl_replay_extend_dev_stack(float* storage, int64_t storage_agent_stride, int64_t capacity, b2rl_rowfmt_t fmt,
                                 const float* new_rows, int32_t n, int32_t n_agents, uint64_t* counters, void* stream) {
  if (int rc = check_fmt(fmt)) return rc;
  if (!storage || !new_rows || !counters || !aligned16(storage) || !aligned16(new_rows))
    return fail(B2RL_E_INVALID, "storage / new_rows / counters must be non-null, rows 16-byte aligned");
  if (capacity < 1 || n < 1 || n > capacity) return fail(B2RL_E_INVALID, "bad capacity / n");
  if (n_agents < 1 || n_agents > 65535) return fail(B2RL_E_INVALID, "n_agents %d out of range", n_agents);
  if (storage_agent_stride & 3) return fail(B2RL_E_INVALID, "storage_agent_stride must be a multiple of 4 floats");
  if (n_agents > 1 && storage_agent_stride < capacity * fmt.row_stride)
    return fail(B2RL_E_INVALID, "storage_agent_stride %lld is smaller than one agent's storage (capacity x row_stride)",
                (long long)storage_agent_stride);
  return check_launch(b2rl::launch_extend_dev(storage, storage_agent_stride, capacity, fmt, new_rows, n, n_agents, counters,
                                              (cudaStream_t)stream),
                      "replay_extend_dev");
}

int b2rl_replay_extend_dev(float* storage, int64_t capacity, b2rl_rowfmt_t fmt, const float* new_rows, int32_t n,
                           uint64_t* counters, void* stream) {
  return b2rl_replay_extend_dev_stack(storage, 0, capacity, fmt, new_rows, n, 1, counters, stream);
}

int b2rl_tc_split_lo(const float* W, float* W_lo, int32_t n, const b2rl_stack_t* stack, void* stream) {
  if (!W || !W_lo || n < 1 || !aligned16(W) || !aligned16(W_lo)) return fail(B2RL_E_INVALID, "tc_split_lo: bad arguments (16-byte aligned tensors)");
  if (int rc = check_stack(stack, "tc_split_lo")) return rc;
  return check_launch(b2rl::launch_tc_split_lo(W, W_lo, n, make_stk(stack), (cudaStream_t)stream), "tc_split_lo");
}
int b2rl_tc_linear(const float* X, int64_t ldx, int32_t M, const float* W, const float* W_lo, const float* bias, const float* g,
                   const float* be, int32_t layer_norm, int32_t relu, float* H, float* XH, float* stat, const b2rl_stack_t* stack,
                   void* stream) {
  if (!X || !W || !bias || !H || M < 1) return fail(B2RL_E_INVALID, "tc_linear: bad arguments");
  if (int rc = check_stack(stack, "tc_linear")) return rc;
  if (layer_norm && (!g || !be)) return fail(B2RL_E_INVALID, "tc_linear: LayerNorm needs weight and bias");
  if (!aligned16(X) || !aligned16(W) || !aligned16(H) || (XH && !aligned16(XH)) || ldx < B2RL_HID || (ldx & 3))
    return fail(B2RL_E_INVALID, "tc_linear: 16-byte aligned tensors, ldx >= 256 and a multiple of 4");
  if (W_lo && !aligned16(W_lo)) return fail(B2RL_E_INVALID, "tc_linear: W_lo must be 16-byte aligned");
  return check_launch(b2rl::launch_tc_linear(X, ldx, M, W, W_lo, bias, g, be, layer_norm, relu, H, XH, stat, nullptr, make_stk(stack),
                                             (cudaStream_t)stream), "tc_linear");
}
int b2rl_tc_linear_q(const float* X, int64_t ldx, int32_t M, const float* W, const float* W_lo, const float* bias, const float* g,
                     const float* be, int32_t layer_norm, float* H, float* XH, float* stat, const b2rl_wide_q_t* q,
                     const b2rl_stack_t* stack, void* stream) {
  if (!X || !W || !bias || !q || M < 1) return fail(B2RL_E_INVALID, "tc_linear_q: bad arguments");
  if (int rc = check_stack(stack, "tc_linear_q")) return rc;
  if (layer_norm && (!g || !be)) return fail(B2RL_E_INVALID, "tc_linear_q: LayerNorm needs weight and bias");
  if (!aligned16(X) || !aligned16(W) || (H && !aligned16(H)) || (XH && !aligned16(XH)) || ldx < B2RL_HID || (ldx & 3))
    return fail(B2RL_E_INVALID, "tc_linear_q: 16-byte aligned tensors, ldx >= 256 and a multiple of 4");
  if (W_lo && !aligned16(W_lo)) return fail(B2RL_E_INVALID, "tc_linear_q: W_lo must be 16-byte aligned");
  if (!q->w3 || !q->b3 || !q->q_out || q->M != M || (q->mode != 0 && q->mode != 1)) return fail(B2RL_E_INVALID, "tc_linear_q: bad head");
  if (q->mode == 1 && (!q->qn0 || !q->qn1 || !q->rows || !q->dz3 || !q->sq_part || (!q->td3 && (!q->logp || !q->log_alpha))))
    return fail(B2RL_E_INVALID, "tc_linear_q: mode 1 needs the target Q values, the batch rows, dz3 and sq_part");
  return check_launch(b2rl::launch_tc_linear(X, ldx, M, W, W_lo, bias, g, be, layer_norm, 1, H, XH, stat, q, make_stk(stack),
                                             (cudaStream_t)stream), "tc_linear_q");
}

int b2rl_wide_first(const float* X, int64_t ldx, int32_t M, int32_t K, const float* w1t, const float* b, const float* g,
                    const float* be, int32_t layer_norm, float* H, float* XH, float* stat, const b2rl_stack_t* stack, void* stream) {
  if (!X || !w1t || !b || !H || M < 1 || K < 1 || ldx < K) return fail(B2RL_E_INVALID, "wide_first: bad arguments");
  if (int rc = check_stack(stack, "wide_first")) return rc;
  if (layer_norm && (!g || !be)) return fail(B2RL_E_INVALID, "wide_first: LayerNorm needs weight and bias");
  return check_launch(b2rl::launch_wide_first(X, ldx, M, K, w1t, b, g, be, layer_norm, H, XH, stat, make_stk(stack), (cudaStream_t)stream), "wide_first");
}
int b2rl_tc_first(const float* X, int64_t ldx, int32_t M, int32_t K, const float* w1t, const float* b, const float* g,
                  const float* be, int32_t layer_norm, float* H, float* XH, float* stat, int32_t x3, const b2rl_stack_t* stack,
                  void* stream) {
  if (!X || !w1t || !b || !H || M < 1 || K < 1 || K > 1024 || ldx < K) return fail(B2RL_E_INVALID, "tc_first: bad arguments");
  if (layer_norm && (!g || !be)) return fail(B2RL_E_INVALID, "tc_first: LayerNorm needs weight and bias");
  if (!aligned16(X) || (ldx & 3) || !aligned16(w1t) || !aligned16(H) || (XH && !aligned16(XH)))
    return fail(B2RL_E_INVALID, "tc_first: X / w1t / H must be 16-byte aligned and ldx a multiple of 4 floats (use b2rl_wide_first otherwise)");
  if (int rc = check_stack(stack, "tc_first")) return rc;
  return check_launch(b2rl::launch_tc_first(X, ldx, M, K, w1t, b, g, be, layer_norm, H, XH, stat, x3, make_stk(stack), (cudaStream_t)stream),
                      "tc_first");
}
int b2rl_tc_linear_bwd(const float* DZ2, int32_t M, const float* w2t, const float* w2t_lo, const float* xh1, const float* stat1,
                       const float* g1, const float* be1, int32_t layer_norm, float* DZ1, float* part, const b2rl_stack_t* stack,
                       void* stream) {
  if (!DZ2 || !w2t || !xh1 || !DZ1 || M < 1) return fail(B2RL_E_INVALID, "tc_linear_bwd: bad arguments");
  if (int rc = check_stack(stack, "tc_linear_bwd")) return rc;
  if (layer_norm && (!g1 || !be1 || !stat1)) return fail(B2RL_E_INVALID, "tc_linear_bwd: LayerNorm needs weight, bias and statistics");
  if (!aligned16(DZ2) || !aligned16(w2t) || !aligned16(DZ1)) return fail(B2RL_E_INVALID, "tc_linear_bwd: 16-byte aligned tensors");
  return check_launch(b2rl::launch_tc_linear_bwd(DZ2, M, w2t, w2t_lo, xh1, stat1, g1, be1, layer_norm, DZ1, part, make_stk(stack), (cudaStream_t)stream),
                      "tc_linear_bwd");
}
int b2rl_wide_policy_head(const b2rl_wide_policy_t* p, const b2rl_stack_t* stack, void* stream) {
  if (int rc = check_stack(stack, "wide_policy_head")) return rc;
  if (!p || !p->h2 || !p->w3 || !p->b3 || !p->rows || !p->min_ac || !p->max_ac || !p->xn || !p->counters || p->M < 1 ||
      p->A < 1 || p->A > 32 || p->out_dim < p->A || p->out_dim > B2RL_MAX_OUT || p->ldn < p->O + p->A)
    return fail(B2RL_E_INVALID, "wide_policy_head: bad arguments");
  return check_launch(b2rl::launch_wide_policy_head(*p, make_stk(stack), (cudaStream_t)stream), "wide_policy_head");
}
int b2rl_wide_q_head(const b2rl_wide_q_t* q, const b2rl_stack_t* stack, void* stream) {
  if (int rc = check_stack(stack, "wide_q_head")) return rc;
  if (!q || !q->h2 || !q->w3 || !q->b3 || !q->q_out || q->M < 1) return fail(B2RL_E_INVALID, "wide_q_head: bad arguments");
  if (q->mode == 1 && (!q->qn0 || !q->qn1 || !q->rows || !q->dz3 || !q->sq_part || (!q->td3 && (!q->logp || !q->log_alpha))))
    return fail(B2RL_E_INVALID, "wide_q_head: online mode needs the target Qs, rows, dz3, sq_part (and logp / log_alpha for SAC)");
  return check_launch(b2rl::launch_wide_q_head(*q, make_stk(stack), (cudaStream_t)stream), "wide_q_head");
}
int b2rl_wide_ln_bwd(const float* dz3, int32_t n_out, const float* w3, const float* xh, const float* stat, const float* g,
                     const float* be, int32_t layer_norm, int32_t M, float* dz, float* part, float* dw3_part,
                     const b2rl_stack_t* stack, void* stream) {
  if (int rc = check_stack(stack, "wide_ln_bwd")) return rc;
  if (dw3_part && n_out != 1) return fail(B2RL_E_INVALID, "wide_ln_bwd: dw3_part is for scalar heads (n_out == 1)");
  if (!dz3 || !w3 || !xh || !dz || M < 1 || n_out < 1 || n_out > B2RL_MAX_OUT) return fail(B2RL_E_INVALID, "wide_ln_bwd: bad arguments");
  if (dw3_part && !part) return fail(B2RL_E_INVALID, "wide_ln_bwd: dw3_part without part");
  if (layer_norm && (!g || !be || !stat)) return fail(B2RL_E_INVALID, "wide_ln_bwd: LayerNorm needs weight, bias and statistics");
  return check_launch(b2rl::launch_wide_ln_bwd(dz3, n_out, w3, xh, stat, g, be, layer_norm, M, dz, part, dw3_part, make_stk(stack), (cudaStream_t)stream), "wide_ln_bwd");
}
int b2rl_wide_colsum_multi(const b2rl_colsum_job_t* jobs, int32_t n_jobs, int32_t P, float* G, const b2rl_stack_t* stack,
                           void* stream) {
  if (int rc = check_stack(stack, "wide_colsum_multi")) return rc;
  if (!jobs || !G || P < 1 || n_jobs < 1 || n_jobs > B2RL_MAX_COLSUM_JOBS) return fail(B2RL_E_INVALID, "wide_colsum_multi: bad arguments");
  b2rl::ColsumJobs J = {};
  for (int i = 0; i < n_jobs; ++i) {
    if (!jobs[i].part) return fail(B2RL_E_INVALID, "wide_colsum_multi: a job without partial sums");
    J.part[i] = jobs[i].part, J.off[i][0] = jobs[i].off_b, J.off[i][1] = jobs[i].off_g, J.off[i][2] = jobs[i].off_be;
    J.ln[i] = jobs[i].layer_norm;
  }
  J.n = n_jobs;
  return check_launch(b2rl::launch_wide_colsum_multi(J, P, G, make_stk(stack), (cudaStream_t)stream), "wide_colsum_multi");
}
int b2rl_wide_colsum(const float* part, int32_t P, float* G, int64_t off_b, int64_t off_g, int64_t off_be, int32_t layer_norm,
                     const b2rl_stack_t* stack, void* stream) {
  if (int rc = check_stack(stack, "wide_colsum")) return rc;
  if (!part || !G || P < 1) return fail(B2RL_E_INVALID, "wide_colsum: bad arguments");
  return check_launch(b2rl::launch_wide_colsum(part, P, G, off_b, off_g, off_be, layer_norm, make_stk(stack), (cudaStream_t)stream), "wide_colsum");
}
int b2rl_wide_critic_scalars(const float* sq0, const float* sq1, int32_t P, const float* dz3_0, const float* dz3_1, int32_t M,
                             float* G, int64_t off_b3_0, int64_t off_b3_1, float* out, const b2rl_stack_t* stack, void* stream) {
  if (int rc = check_stack(stack, "wide_critic_scalars")) return rc;
  if (!sq0 || !sq1 || !G || !out || P < 1 || M < 1) return fail(B2RL_E_INVALID, "wide_critic_scalars: bad arguments");
  return check_launch(b2rl::launch_wide_critic_scalars(sq0, sq1, P, dz3_0, dz3_1, M, G, off_b3_0, off_b3_1, out, make_stk(stack), (cudaStream_t)stream),
                      "wide_critic_scalars");
}
int b2rl_wide_actor_loss(const float* q0, const float* q1, const float* logp, const float* log_alpha, int32_t td3, int32_t M,
                         float* dzq0, float* dzq1, float* part, const b2rl_stack_t* stack, void* stream) {
  if (int rc = check_stack(stack, "wide_actor_loss")) return rc;
  if (!q0 || !dzq0 || !part || M < 1 || (!td3 && (!q1 || !dzq1 || !logp || !log_alpha)))
    return fail(B2RL_E_INVALID, "wide_actor_loss: bad arguments");
  return check_launch(b2rl::launch_wide_actor_loss(q0, q1, logp, log_alpha, td3, M, dzq0, dzq1, part, make_stk(stack), (cudaStream_t)stream), "wide_actor_loss");
}
int b2rl_wide_dqda(const float* dz1, const float* w1a, int32_t A, int32_t M, float* dqda, const b2rl_stack_t* stack, void* stream) {
  if (int rc = check_stack(stack, "wide_dqda")) return rc;
  if (!dz1 || !w1a || !dqda || A < 1 || A > 32 || M < 1) return fail(B2RL_E_INVALID, "wide_dqda: bad arguments");
  return check_launch(b2rl::launch_wide_dqda(dz1, w1a, A, M, dqda, make_stk(stack), (cudaStream_t)stream), "wide_dqda");
}
int b2rl_wide_actor_head_bwd(const float* dqda0, const float* dqda1, const float* save, const float* min_ac,
                             const float* max_ac, const float* log_alpha, int32_t td3, int32_t A, int32_t M, float* du,
                             float* part_du, const b2rl_stack_t* stack, void* stream) {
  if (int rc = check_stack(stack, "wide_actor_head_bwd")) return rc;
  if (!dqda0 || !save || !min_ac || !max_ac || !du || !part_du || A < 1 || A > 32 || M < 1 || (!td3 && !log_alpha))
    return fail(B2RL_E_INVALID, "wide_actor_head_bwd: bad arguments");
  return check_launch(b2rl::launch_wide_actor_head_bwd(dqda0, dqda1, save, min_ac, max_ac, log_alpha, td3, A, M, du, part_du,
                                                       make_stk(stack), (cudaStream_t)stream), "wide_actor_head_bwd");
}
int b2rl_wide_actor_scalars(const float* part_s, const float* part_du, int32_t P, int32_t M, int32_t out_dim, int32_t td3,
                            const float* log_alpha, float* G, int64_t off_b3, float* out, const b2rl_stack_t* stack, void* stream) {
  if (int rc = check_stack(stack, "wide_actor_scalars")) return rc;
  if (!part_s || !part_du || !G || !out || P < 1 || M < 1 || out_dim < 1 || out_dim > B2RL_MAX_OUT)
    return fail(B2RL_E_INVALID, "wide_actor_scalars: bad arguments");
  return check_launch(b2rl::launch_wide_actor_scalars(part_s, part_du, P, M, out_dim, td3, log_alpha, G, off_b3, out, make_stk(stack), (cudaStream_t)stream),
                      "wide_actor_scalars");
}
int b2rl_wide_alpha_grad(const float* logp2, int32_t M, float targ_ent, float* alpha_state, const b2rl_stack_t* stack, void* stream) {
  if (int rc = check_stack(stack, "wide_alpha_grad")) return rc;
  if (!logp2 || !alpha_state || M < 1) return fail(B2RL_E_INVALID, "wide_alpha_grad: bad arguments");
  return check_launch(b2rl::launch_wide_alpha_grad(logp2, M, targ_ent, alpha_state, make_stk(stack), (cudaStream_t)stream), "wide_alpha_grad");
}
int64_t b2rl_tc_wgrad_scratch_floats(int32_t MA, int32_t Bn, int32_t n_agents) {
  if (MA < 1 || Bn < 1 || n_agents < 0) return -1;
  const int64_t per_agent = (int64_t)b2rl::tc_wgrad_splits(Bn, MA, n_agents > 0) * ((MA + 127) / 128 * 128) * B2RL_HID;
  return per_agent * (n_agents > 0 ? n_agents : 1);
}
int b2rl_tc_wgrad(const float* A, int64_t lda, int32_t a_cols, int32_t MA, const float* Bm, int32_t Bn, float* C, float* Ct,
                  float* scratch, int32_t x3, uint64_t* bump, const b2rl_stack_t* stack, void* stream) {
  if (int rc = check_stack(stack, "tc_wgrad")) return rc;
  if (!A || !Bm || !C || !scratch || MA < 1 || a_cols < MA || lda < a_cols || (lda & 3) || Bn < 1)
    return fail(B2RL_E_INVALID, "tc_wgrad: bad arguments");
  if (!aligned16(A) || !aligned16(Bm) || !aligned16(C) || !aligned16(scratch)) return fail(B2RL_E_INVALID, "tc_wgrad: 16-byte aligned tensors");
  if (Ct && (MA & 3)) return fail(B2RL_E_INVALID, "tc_wgrad: the transposed copy needs MA % 4 == 0");
  return check_launch(b2rl::launch_tc_wgrad(A, lda, a_cols, MA, Bm, Bn, C, Ct, scratch, x3, (unsigned long long*)bump, make_stk(stack),
                                            stack != nullptr, (cudaStream_t)stream), "tc_wgrad");
}
int b2rl_wgrad(const b2rl_update_args_t* a, int32_t actor_step, int32_t bump_counter, int32_t skip_vectors, void* stream) {
  if (int rc = check_update(a, actor_step != 0)) return rc;
  if (bump_counter < -1 || bump_counter > 3) return fail(B2RL_E_INVALID, "wgrad: bad bump_counter");
  return check_launch(b2rl::launch_wgrad(*a, actor_step != 0, bump_counter, nullptr, (cudaStream_t)stream, skip_vectors != 0), "wgrad");
}

int b2rl_publish_logs(const float* out, int32_t n_agents, float* host_out, uint64_t* seq_dev, uint64_t* host_seq,
                      void* stream) {
  if (!out || !host_out || !seq_dev || !host_seq || n_agents < 1) return fail(B2RL_E_INVALID, "publish_logs: bad arguments");
  return check_launch(b2rl::launch_publish(out, n_agents, host_out, seq_dev, host_seq, (cudaStream_t)stream), "publish_logs");
}

// the fused optimizer's description: seg[0] = plain Adam (+ Polyak) on exactly the trained span, the rest Polyak-only
static int check_opt(const b2rl_update_args_t* a, const b2rl_adam_args_t* o, int64_t begin, int64_t end, int counter) {
  if (!o) return B2RL_OK;
  if (o->n_seg < 1 || o->n_seg > B2RL_MAX_SEG) return fail(B2RL_E_INVALID, "opt: n_seg %d out of range", o->n_seg);
  if (o->lo)  // (the weight-gradient kernel does not write the 3xTF32 mirror: it would go stale)
    return fail(B2RL_E_INVALID, "opt: the fused optimizer does not keep a lo mirror current; use the three-launch form");
  if (a->agent_hp || o->agent_hp)  // (the weight-gradient kernel takes its optimizer scalars from opt alone)
    return fail(B2RL_E_INVALID, "opt: the fused optimizer takes no per-agent hyperparameter table; use the three-launch form");
  const b2rl_seg_t& s0 = o->seg[0];
  if (!s0.do_adam || s0.clip || s0.grad_scale != 1.0f || s0.begin != begin || s0.end != end || s0.counter != counter)
    return fail(B2RL_E_INVALID, "opt: seg[0] must be an unclipped, unscaled Adam segment over the trained nets");
  for (int i = 1; i < o->n_seg; ++i) {
    const b2rl_seg_t& s = o->seg[i];
    if (s.do_adam || !s.do_polyak || s.begin < 0 || s.end < s.begin || (s.begin & 3) || (s.end & 3) || s.end > a->region_stride)
      return fail(B2RL_E_INVALID, "opt: extra segment %d must be a 4-float aligned Polyak-only span", i);
  }
  return B2RL_OK;
}

static int critic_update(const b2rl_update_args_t* a, int td3, const b2rl_adam_args_t* opt, void* stream) {
  if (int rc = check_update(a, false)) return rc;
  if (opt && a->new_rows) return fail(B2RL_E_INVALID, "new_rows is not supported by the fused-optimizer entry point");
  if (int rc = check_opt(a, opt, a->critic[0].begin, a->critic[1].end, B2RL_CTR_Q)) return rc;
  if ((a->hp.td3 != 0) != (td3 != 0)) return fail(B2RL_E_INVALID, "hp.td3 does not match the entry point");
  if (int rc = check_launch(b2rl::launch_critic_fused(*a, (cudaStream_t)stream), "critic_fused")) return rc;
  return check_launch(b2rl::launch_wgrad(*a, 0, B2RL_CTR_Q, opt, (cudaStream_t)stream), "critic wgrad");
}
int b2rl_critic_update_sac(const b2rl_update_args_t* a, void* stream) { return critic_update(a, 0, nullptr, stream); }
int b2rl_critic_update_td3(const b2rl_update_args_t* a, void* stream) { return critic_update(a, 1, nullptr, stream); }
int b2rl_critic_update_opt(const b2rl_update_args_t* a, const b2rl_adam_args_t* opt, void* stream) {
  if (!a || !opt) return fail(B2RL_E_INVALID, "null args");
  return critic_update(a, a->hp.td3 != 0, opt, stream);
}

static int actor_update(const b2rl_update_args_t* a, int td3, const b2rl_adam_args_t* opt, void* stream) {
  if (int rc = check_update(a, true)) return rc;
  if (int rc = check_opt(a, opt, a->actor.begin, a->actor.end, B2RL_CTR_PI)) return rc;
  if ((a->hp.td3 != 0) != (td3 != 0)) return fail(B2RL_E_INVALID, "hp.td3 does not match the entry point");
  if (int rc = check_launch(b2rl::launch_actor_fused(*a, (cudaStream_t)stream), "actor_fused")) return rc;
  return check_launch(b2rl::launch_wgrad(*a, 1, B2RL_CTR_PI, opt, (cudaStream_t)stream), "actor wgrad");
}
int b2rl_actor_update_sac(const b2rl_update_args_t* a, void* stream) { return actor_update(a, 0, nullptr, stream); }
int b2rl_actor_update_td3(const b2rl_update_args_t* a, void* stream) { return actor_update(a, 1, nullptr, stream); }
int b2rl_actor_update_opt(const b2rl_update_args_t* a, const b2rl_adam_args_t* opt, void* stream) {
  if (!a || !opt) return fail(B2RL_E_INVALID, "null args");
  return actor_update(a, a->hp.td3 != 0, opt, stream);
}

int b2rl_alpha_update(const b2rl_update_args_t* a, float log_alpha_lr, void* stream) {
  if (int rc = check_update(a, false)) return rc;
  if (a->hp.td3) return fail(B2RL_E_INVALID, "alpha_update is SAC-only");
  if (!(log_alpha_lr >= 0.f)) return fail(B2RL_E_INVALID, "log_alpha_lr must be >= 0");
  return check_launch(b2rl::launch_alpha(*a, log_alpha_lr, (cudaStream_t)stream), "alpha_update");
}

int b2rl_alpha_adam(float* log_alpha, uint64_t* counters, int32_t n_agents, float log_alpha_lr, float grad_scale,
                    float* out, void* stream) {
  if (!log_alpha || !counters || n_agents < 1 || !(log_alpha_lr > 0.f))
    return fail(B2RL_E_INVALID, "alpha_adam: bad arguments");
  return check_launch(b2rl::launch_alpha_adam(log_alpha, counters, n_agents, log_alpha_lr, nullptr, grad_scale, out,
                                              (cudaStream_t)stream),
                      "alpha_adam");
}

int b2rl_alpha_adam_hp(float* log_alpha, uint64_t* counters, int32_t n_agents, const b2rl_agent_hp_t* hp, float grad_scale,
                       float* out, void* stream) {
  if (!log_alpha || !counters || n_agents < 1 || !hp) return fail(B2RL_E_INVALID, "alpha_adam_hp: bad arguments");
  if (int rc = check_hp(hp, "alpha_adam_hp")) return rc;
  return check_launch(b2rl::launch_alpha_adam(log_alpha, counters, n_agents, 0.f, hp, grad_scale, out, (cudaStream_t)stream),
                      "alpha_adam_hp");
}

int b2rl_grad_sumsq(const float* arena, int64_t region_stride, int64_t arena_agent_stride, int64_t begin, int64_t end,
                    int32_t n_agents, float* sumsq, float* scratch, void* stream) {
  if (!arena || !sumsq || !scratch || begin < 0 || end < begin || n_agents < 1)
    return fail(B2RL_E_INVALID, "grad_sumsq: bad arguments");
  return check_launch(b2rl::launch_sumsq(arena, region_stride, arena_agent_stride, begin, end, n_agents, sumsq, scratch,
                                         (cudaStream_t)stream),
                      "grad_sumsq");
}

int b2rl_adam_polyak_multi(const b2rl_adam_args_t* a, void* stream) {
  if (!a || !a->arena || !a->counters) return fail(B2RL_E_INVALID, "adam: null args");
  if (a->n_seg < 1 || a->n_seg > B2RL_MAX_SEG) return fail(B2RL_E_INVALID, "adam: n_seg %d out of range", a->n_seg);
  if (a->n_agents < 1 || a->n_agents > 65535) return fail(B2RL_E_INVALID, "adam: bad n_agents");
  if (!aligned16(a->arena) || (a->region_stride & 3) || (a->arena_agent_stride & 3))
    return fail(B2RL_E_INVALID, "adam: arena must be 16-byte aligned, strides multiples of 4 floats");
  if (a->lo && (!aligned16(a->lo) || (a->lo_agent_stride & 3) || a->lo_agent_stride < 2 * a->region_stride))
    return fail(B2RL_E_INVALID, "adam: the lo mirror must be 16-byte aligned, its agent stride >= 2 regions and a multiple of 4 floats");
  if (a->n_shadow < 0 || a->n_shadow > 3) return fail(B2RL_E_INVALID, "adam: n_shadow %d out of range", a->n_shadow);
  if (int rc = check_hp(a->agent_hp, "adam")) return rc;
  for (int q = 0; q < a->n_shadow; ++q) {
    const int64_t src = a->shadow_src[q], dst = a->shadow_dst[q], n = (int64_t)B2RL_HID * B2RL_HID;
    if (src < 0 || dst < 0 || (src & 3) || (dst & 3) || src + n > a->region_stride || dst + n > a->region_stride ||
        (src < dst + n && dst < src + n))
      return fail(B2RL_E_INVALID, "adam: shadow pair %d must be two disjoint, 4-float aligned 256x256 spans of a region", q);
    for (int i = 0; i < a->n_seg; ++i) {  // a segment holds a pair's two spans entirely or not at all
      const b2rl_seg_t& s = a->seg[i];
      const bool in_src = src >= s.begin && src + n <= s.end, in_dst = dst >= s.begin && dst + n <= s.end;
      const bool cut = (src < s.end && src + n > s.begin && !in_src) || (dst < s.end && dst + n > s.begin && !in_dst);
      if (cut || in_src != in_dst) return fail(B2RL_E_INVALID, "adam: segment %d splits shadow pair %d", i, q);
    }
  }
  for (int i = 0; i < a->n_seg; ++i) {
    const b2rl_seg_t& s = a->seg[i];
    if (s.begin < 0 || s.end < s.begin || (s.begin & 3) || (s.end & 3) || s.end > a->region_stride)
      return fail(B2RL_E_INVALID, "adam: segment %d [%lld,%lld) must be 4-float aligned inside a region", i,
                  (long long)s.begin, (long long)s.end);
    if (s.do_adam && (s.counter < 0 || s.counter > 3)) return fail(B2RL_E_INVALID, "adam: segment %d bad counter", i);
    if (s.do_adam && a->agent_hp && s.counter > B2RL_CTR_ALPHA)  // (the table has a learning rate for counters 0..2)
      return fail(B2RL_E_INVALID, "adam: segment %d: with agent_hp the counter must be Q, PI or ALPHA", i);
    if (s.do_adam && s.clip && !a->grad_sumsq) return fail(B2RL_E_INVALID, "adam: clip needs grad_sumsq");
  }
  return check_launch(b2rl::launch_adam(*a, (cudaStream_t)stream), "adam_polyak_multi");
}

int b2rl_bump_counter(uint64_t* counters, int32_t which, int32_t n_agents, void* stream) {
  if (!counters || which < 0 || which > 7 || n_agents < 1) return fail(B2RL_E_INVALID, "bump_counter: bad arguments");
  return check_launch(b2rl::launch_bump(counters, which, n_agents, (cudaStream_t)stream), "bump_counter");
}

int b2rl_actor_predict(const b2rl_update_args_t* a, const float* obs, int32_t n, int32_t mode, float explore_std,
                       uint64_t draw, float* actions_out, void* stream) {
  if (!a || !obs || !actions_out || n < 1) return fail(B2RL_E_INVALID, "predict: bad arguments");
  if (int rc = check_fmt(a->fmt)) return rc;
  if (int rc = check_net(a->actor, "actor", false)) return rc;
  if (!a->arena || !a->min_ac || !a->max_ac) return fail(B2RL_E_INVALID, "predict: null device pointer");
  if (mode != 0 && mode != 1) return fail(B2RL_E_INVALID, "predict: mode must be 0 or 1");
  if (int rc = check_hp(a->agent_hp, "predict")) return rc;
  if (a->n_agents < 0 || a->n_agents > 65535) return fail(B2RL_E_INVALID, "predict: n_agents %d out of range", a->n_agents);
  if (a->n_agents > 1 && (a->agent_base < 0 || (int64_t)a->agent_base + a->n_agents > (1 << 30) || a->arena_agent_stride < 1 ||
                          (a->arena_agent_stride & 3)))
    return fail(B2RL_E_INVALID, "predict: stacked agents need ids below 2^30 and an arena agent stride that is a positive multiple of 4 floats");
  return check_launch(b2rl::launch_predict(*a, obs, n, mode, explore_std, draw, actions_out, (cudaStream_t)stream), "actor_predict");
}

int b2rl_launch_single(const b2rl_update_args_t* a, int32_t which, void* stream) {
  if (int rc = check_update(a, which >= 2)) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  switch (which) {
    case 0: return check_launch(b2rl::launch_critic_fused(*a, st), "critic_fused");
    case 1: return check_launch(b2rl::launch_wgrad(*a, 0, -1, nullptr, st), "critic wgrad");
    case 2: return check_launch(b2rl::launch_actor_fused(*a, st), "actor_fused");
    case 3: return check_launch(b2rl::launch_wgrad(*a, 1, -1, nullptr, st), "actor wgrad");
    case 4:
      if (a->hp.td3) return fail(B2RL_E_INVALID, "alpha kernel is SAC-only");
      return check_launch(b2rl::launch_alpha(*a, 1e-3f, st), "alpha");
    default: return fail(B2RL_E_INVALID, "launch_single: which must be 0..4");
  }
}

int b2rl_ffma_probe(float* sink, int32_t iters, double* flops, void* stream) {
  if (!sink || iters < 1) return fail(B2RL_E_INVALID, "ffma_probe: bad arguments");
  const int ctas = 148 * 8;
  b2rl::ffma_probe_kernel<<<ctas, 256, 0, (cudaStream_t)stream>>>(sink, iters);
  if (flops) *flops = 2.0 * 16.0 * (double)iters * 256.0 * (double)ctas;
  return check_launch(cudaGetLastError(), "ffma_probe");
}

}  // extern "C"
