/* b2rl.h — C ABI of libb2rl.so: the B200-native SAC/TD3 learner update.
 *
 * The reference (lionelblonde/sac-td3-cudagraphs-pytorch) has no FFI of its own: its
 * hot path is the Python object `Agent` (agents/agent.py) driven by orchestrator.py:337-352.
 * Each entry point below replaces one torch-op sequence of that path; the citation on
 * every function names the reference lines it stands in for. The host-side mirror
 * (sac_td3_cudagraphs_pytorch_b200/agents/agent.py) binds these with ctypes.
 *
 * Conventions
 *  - plain C: pointers, sizes, POD structs; no torch / C++ types.
 *  - every pointer marked `dev` is device memory owned by the caller (torch allocator).
 *  - every call only ENQUEUES work on `stream` (a cudaStream_t passed as void*): no
 *    allocation, no synchronisation, no host read of device memory => legal inside CUDA
 *    graph capture (the replacement for tensordict's CudaGraphModule, orchestrator.py:313-315).
 *  - return value: 0 on success, <0 on error (B2RL_E_*); text via b2rl_last_error().
 *  - all floating point is fp32; indices are int64 (as torchrl's sampler returns them).
 */
#ifndef B2RL_H
#define B2RL_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2RL_VERSION 111 /* 0.1.1 */
#define B2RL_HID 256     /* hidden width; agents/agent.py:56,101 hard-codes (256, 256) */
#define B2RL_ROWS 8      /* batch rows per CTA group of the fused kernels; a batch need not be a multiple (the tail is masked) */
#define B2RL_MAX_OUT 64  /* max head width (2*A for SAC) */
#define B2RL_MAX_SEG 8   /* max segments per adam_polyak_multi launch */

#define B2RL_OK 0
#define B2RL_E_INVALID (-1) /* bad argument (null pointer, unsupported size, misalignment) */
#define B2RL_E_LAUNCH (-2)  /* CUDA reported an error at launch */

/* ---- parameter arena -------------------------------------------------------------------
 * One agent owns one flat fp32 ARENA of 5 equally laid out REGIONS:
 *   0 online params | 1 target params | 2 Adam exp_avg | 3 Adam exp_avg_sq | 4 gradients
 * A net (actor or one critic) is a contiguous span [begin,end) of a region; b2rl_net_t gives
 * the float offsets of its tensors inside a region. Layouts:
 *   w1t [in_dim][256], w2t [256][256]  "forward layout": w?t[k*256+j] == fc.weight[j][k]
 *       (exposed to torch as a transposed view, so state_dict keys/shapes stay those of
 *        agents/nets.py:66-84);
 *   w3  [out_dim][256]                 natural torch layout (head.weight);
 *   w2n [256][256]                     natural-layout SHADOW of fc_block_2.fc.weight used by the
 *        backward dX pass; it is a parameter in its own right (own grad, exp_avg, exp_avg_sq,
 *        updated by the same Adam arithmetic), hence bit-identical to w2t transposed. -1 if absent.
 */
typedef struct b2rl_net {
  int32_t in_dim;     /* O (actor) or O+A (critic)            agents/nets.py:63-67,106-110 */
  int32_t out_dim;    /* 1 (critic), A (TD3 actor), 2A (SAC)  agents/nets.py:84,127,192   */
  int32_t layer_norm; /* hps.layer_norm                        agents/nets.py:69,75        */
  int32_t reserved;
  int64_t w1t, b1, g1, be1;
  int64_t w2t, b2, g2, be2;
  int64_t w3, b3;
  int64_t w2n;
  int64_t begin, end;
} b2rl_net_t;

/* ---- transition rows -------------------------------------------------------------------
 * Replay storage AND sampled batches use one padded array-of-structs row per transition:
 *   [ obs(O) | act(A) | reward | done(0/1) | next_obs(O) | pad ]   row_stride % 4 == 0 floats
 * so a row is a whole number of 128-bit words and [obs|act] (the critic input, agents/nets.py:89)
 * is already contiguous. The reference stores six separate [cap,d] tensors (main.py:167-171,
 * orchestrator.py:100-113). */
typedef struct b2rl_rowfmt {
  int32_t ob_dim, ac_dim;
  int32_t row_stride; /* floats, multiple of 4, >= 2*ob_dim + ac_dim + 2 */
  int32_t reserved;
} b2rl_rowfmt_t;

/* ---- device-side counters ----------------------------------------------------------------
 * uint64[8] in device memory, owned by the caller, zero-initialised:
 *   [0] critic Adam steps done  [1] actor Adam steps done  [2] alpha Adam steps done
 *   [3] replay samples drawn    [4] ticket (self-resetting)   [5] replay size
 *   [6] replay write cursor     [7] ticket of b2rl_replay_extend_dev (self-resetting)
 * They advance on the device so that a captured graph can be replayed without host patches. */
#define B2RL_CTR_Q 0
#define B2RL_CTR_PI 1
#define B2RL_CTR_ALPHA 2
#define B2RL_CTR_SAMPLE 3
#define B2RL_CTR_TICKET 4 /* alpha_update's last-CTA ticket */
#define B2RL_CTR_SIZE 5   /* replay rows filled: written by the host side of the replay buffer, or advanced on the
                             device by b2rl_replay_extend_dev */
#define B2RL_CTR_CURSOR 6 /* round-robin write position (b2rl_replay_extend_dev) */
#define B2RL_CTR_XTICKET 7

typedef struct b2rl_hyper {
  int32_t td3;                 /* hps.prefer_td3_over_sac */
  int32_t bcq_mix;             /* hps.bcq_style_targ_mix        agents/agent.py:213-219 */
  int32_t targ_smoothing;      /* hps.targ_actor_smoothing      agents/agent.py:197-202 */
  int32_t autotune;            /* hps.autotune                  agents/agent.py:130-139 */
  float gamma;                 /* agents/agent.py:228 */
  float td3_std, td3_c;        /* agents/agent.py:198-199 */
  float targ_ent;              /* -A                            agents/agent.py:134 */
  uint64_t seed;               /* Philox key when noise/indices are drawn on the device */
} b2rl_hyper_t;

/* ---- per-agent hyperparameters -------------------------------------------------------------
 * One 64-byte row per local agent of a launch, in device memory (row g = agent g, a local index like
 * arena_agent_stride). A captured graph freezes every by-value argument, so values that may differ between
 * stacked agents (a sweep) or change during training (population-based training) are read from this table
 * instead: rewriting a row with a stream-ordered copy changes what the next replay computes, with no recapture.
 * Where a struct or entry point takes `agent_hp`, NULL means its scalars as before; a table replaces exactly the
 * scalars listed here and only where the scalar path reads them (the flags — targ_smoothing, seg.do_adam /
 * do_polyak / clip, predict's mode — still decide whether a value is used). */
typedef struct b2rl_agent_hp {
  float lr[3];           /* Adam learning rate by the optimizer's counter: [B2RL_CTR_Q] critics (hps.qnets_lr),
                            [B2RL_CTR_PI] actor (hps.actor_lr), [B2RL_CTR_ALPHA] temperature (hps.log_alpha_lr);
                            replaces b2rl_seg_t.lr and the log_alpha_lr arguments */
  float gamma, polyak;   /* agents/agent.py:228, :328-331 */
  float td3_std, td3_c;  /* target smoothing (agents/agent.py:197-200) */
  float targ_ent;        /* SAC target entropy (-A in the reference, agents/agent.py:134) */
  float clip_norm;       /* used when seg.clip; +inf = this agent does not clip (min(1, inf / (norm + 1e-6)) is exactly 1) */
  float explore_std;     /* TD3 behaviour noise (hps.actor_noise_std, nets.py:155-159) */
  float reserved[6];
} b2rl_agent_hp_t;

/* Everything a fused update needs. Pointers are `dev`. Population stacking: agent g uses
 * base + g*<x>_agent_stride for every per-agent buffer (n_agents == 1 for a single learner). */
typedef struct b2rl_update_args {
  b2rl_hyper_t hp;
  b2rl_rowfmt_t fmt;
  b2rl_net_t actor;            /* online actor                                         */
  b2rl_net_t critic[2];        /* twin critics (reference stacks them on dim 0, agent.py:106) */
  int32_t batch;               /* B >= 1 (a tail that does not fill a group of B2RL_ROWS rows is masked) */
  int32_t n_agents;
  int32_t agent_base;          /* global id of local agent 0: Philox streams are keyed on the GLOBAL id, so a
                                  population gives the same results however it is sharded over GPUs */
  int32_t reserved;
  int64_t region_stride;       /* floats between regions of the arena */
  int64_t arena_agent_stride;  /* floats between agents' arenas */
  float* arena;                /* dev */
  const float* rows;           /* dev: the sampled batch, [n_agents][B][row_stride] */
  int64_t rows_agent_stride;
  const float* min_ac;         /* dev [A] */
  const float* max_ac;         /* dev [A] */
  float* log_alpha;            /* dev: 5 floats per agent {log_alpha, grad, exp_avg, exp_avg_sq, spare}; SAC only */
  const float* eps;            /* dev [n_agents][B][A] N(0,1) noise, or NULL => Philox on device */
  const float* eps2;           /* dev: second noise tensor (SAC alpha step), or NULL */
  float* eps_out;              /* dev or NULL: noise actually used (parity tests) */
  float* eps2_out;             /* dev or NULL */
  uint64_t* counters;          /* dev uint64[8] per agent */
  float* workspace;            /* dev, b2rl_workspace_floats() per agent */
  int64_t workspace_agent_stride;
  float* out;                  /* dev float[8] per agent: {qf_loss, actor_loss, alpha_loss, alpha, ...} */
  float* dbg_targ_q;           /* dev [n_agents][B] or NULL   (TD target y, agent.py:226-228) */
  float* dbg_q;                /* dev [n_agents][2][B] or NULL (online Q values) */
  /* In-kernel sampling (b2rl_critic_update_* only; agent.rb.sample(B), orchestrator.py:338, folded into the critic
   * step): storage != NULL => every row group draws its batch indices itself — Philox keyed exactly as
   * b2rl_replay_sample_gather keys them (hp.seed, batch row, counters[B2RL_CTR_Q], global agent id), so the batch is
   * the same — reads its transitions straight from the replay storage, and the step also WRITES them to `rows` (and
   * the indices to idx_out), which the kernels that follow (weight gradients, actor / alpha steps) read. */
  const float* storage;        /* dev [n_agents][capacity][row_stride] or NULL */
  int64_t storage_agent_stride;
  int64_t storage_size;        /* rows filled; 0 => read counters[B2RL_CTR_SIZE] (graph replays while the buffer fills) */
  int64_t* idx_out;            /* dev [n_agents][B] or NULL */
  /* Replay write folded into the same step (agent.rb.extend(td), orchestrator.py:100-113; single learner, with
   * `storage`): new_rows != NULL => the n_new transitions at new_rows (device or pinned host memory) are appended at
   * counters[B2RL_CTR_CURSOR] (round robin over `capacity` rows) BEFORE the batch is drawn: the draw uses the grown
   * size, a drawn index that falls on a new row is read from new_rows itself, one CTA writes the rows into the storage,
   * and the weight-gradient launch of the critic step (which runs after every CTA has read them) advances
   * counters[CURSOR] / counters[SIZE]. Same result as b2rl_replay_extend_dev followed by the critic step. */
  const float* new_rows;
  int64_t capacity;
  int32_t n_new;
  int32_t reserved2;
  /* dev [n_agents] or NULL: per-agent gamma, td3_std / td3_c, targ_ent, explore_std (b2rl_actor_predict) and the
   * temperature's learning rate (b2rl_alpha_update) in place of hp.* and the scalar arguments. Refused by the
   * fused-optimizer entry points (b2rl_*_update_opt). */
  const b2rl_agent_hp_t* agent_hp;
} b2rl_update_args_t;

#define B2RL_OUT_QF_LOSS 0
#define B2RL_OUT_ACTOR_LOSS 1
#define B2RL_OUT_ALPHA_LOSS 2
#define B2RL_OUT_ALPHA 3
#define B2RL_OUT_LOGPI_MEAN 4

/* segment of the arena handled by one adam_polyak_multi launch */
typedef struct b2rl_seg {
  int64_t begin, end;  /* float offsets inside a region */
  float lr;
  int32_t do_adam;     /* p,m,v <- Adam(p, g, m, v)           torch/optim/adam.py:347-551 */
  int32_t do_polyak;   /* target <- lerp(target, p, polyak)   agents/agent.py:328-331 */
  int32_t counter;     /* B2RL_CTR_* holding this optimizer's step count (read, not bumped) */
  float grad_scale;    /* multiplies g first (1/world for data parallel; 1 otherwise) */
  int32_t clip;        /* 1: scale g by min(1, clip_norm/(norm+1e-6)), norm = sqrt(b2rl_grad_sumsq) * grad_scale */
} b2rl_seg_t;

typedef struct b2rl_adam_args {
  b2rl_seg_t seg[B2RL_MAX_SEG];
  int32_t n_seg;
  int32_t n_agents;
  float polyak;
  float clip_norm;             /* hps.clip_norm (agents/agent.py:284-285), used when seg.clip */
  float beta1, beta2, eps;     /* 0.9, 0.999, 1e-8 (torch defaults, agents/agent.py:115-124) */
  int32_t reserved;
  int64_t region_stride, arena_agent_stride;
  float* arena;                /* dev */
  const uint64_t* counters;    /* dev uint64[8] per agent */
  const float* grad_sumsq;     /* dev float per agent (from b2rl_grad_sumsq) or NULL */
  /* 3xTF32 mirror (wide path): when not NULL, every parameter this launch writes also leaves its "lo part"
   * p - tf32_truncate(p) (what b2rl_tc_split_lo computes) at the same region offset of the mirror
   * lo[agent][0 = online | 1 = target][region_stride], so the tensor-core kernels never need a split pass over weights
   * that an optimizer step has just changed. */
  float* lo;                   /* dev or NULL */
  int64_t lo_agent_stride;     /* floats between agents' mirrors (>= 2 * region_stride) */
  /* Shadow pairs: shadow_src[i] / shadow_dst[i] are the region offsets of a net's w2t [256][256] and of its natural-layout
   * shadow w2n (= w2t transposed, see "parameter arena"). For a pair whose w2t lies inside one of the segments, the launch
   * steps w2t from ITS gradient and writes the new parameter / exp_avg / exp_avg_sq / target (and lo parts) to BOTH
   * layouts through a 32 x 32 transposing tile; the shadow's own gradient, exp_avg and exp_avg_sq are never read. Same
   * values as stepping the shadow with the transposed gradient (it stays bit-identical to w2t^T), 20 bytes per shadow
   * element less traffic, and no transposed gradient copy is needed (weight-gradient kernels, data-parallel all-reduce). */
  int64_t shadow_src[3], shadow_dst[3];
  int32_t n_shadow;            /* 0..3 */
  int32_t reserved2;
  /* dev [n_agents] or NULL: agent g steps with lr[seg.counter] (seg.lr is ignored), polyak and clip_norm of its row.
   * b2rl_grad_sumsq and seg.clip are needed when ANY agent clips; an agent that does not gets clip_norm = +inf. */
  const b2rl_agent_hp_t* agent_hp;
} b2rl_adam_args_t;

/* ---- entry points ---------------------------------------------------------------------- */

int b2rl_version(void);
const char* b2rl_last_error(void);

/* Load every kernel and opt in to large dynamic shared memory. Call once per process and device,
 * after the CUDA context exists and BEFORE any stream capture (CUDA loads kernels lazily and a
 * first launch inside a capture is illegal). The only entry point that is not capture-safe. */
int b2rl_init(void);

/* floats of workspace one agent needs for a batch of B rows */
int64_t b2rl_workspace_floats(int32_t batch);

/* Replaces `agent.rb.sample(B)` (orchestrator.py:338): torchrl RandomSampler
 * `randint(0, len, (B,))` + one advanced-index gather per key + the 7 copies CudaGraphModule makes
 * into its static inputs (orchestrator.py:313-315). Uniform with replacement.
 *   storage [n_agents][capacity][row_stride], size = filled rows (same for all agents), or 0 to
 *           read it from counters[B2RL_CTR_SIZE] on the device (a captured graph then follows a
 *           buffer that is still filling)
 *   idx_in  int64 [n_agents][B] or NULL => idx = (philox(seed, step, row) * size) >> 32 with
 *           step = counters[step_counter] (B2RL_CTR_SAMPLE when the sampler runs on its own with
 *           bump = 1; B2RL_CTR_Q with bump = 0 inside a fused iteration, where the critic step
 *           advances that counter)
 *   idx_out int64 [n_agents][B] or NULL;  rows_out [n_agents][B][row_stride] */
int b2rl_replay_sample_gather(const float* storage, int64_t storage_agent_stride, int64_t size,
                              b2rl_rowfmt_t fmt, int32_t batch, int32_t n_agents,
                              const int64_t* idx_in, int64_t* idx_out, float* rows_out,
                              uint64_t seed, uint64_t* counters, int32_t step_counter, int32_t bump,
                              int32_t agent_base, void* stream);

/* Replaces `rb.extend(td)` (orchestrator.py:100-113; torchrl round-robin writer): scatter n
 * freshly packed rows [n][row_stride] to storage rows (cursor + i) % capacity. */
int b2rl_replay_extend(float* storage, int64_t capacity, int64_t cursor, b2rl_rowfmt_t fmt,
                       const float* new_rows, int32_t n, void* stream);

/* Graph-capturable variant of b2rl_replay_extend (orchestrator.py:100-113): the write cursor and the fill count
 * live on the device (counters[B2RL_CTR_CURSOR], counters[B2RL_CTR_SIZE]) and advance there, so one captured
 * graph can hold "copy the new transitions in -> write them -> sample -> update" and be replayed without host
 * patches. The last CTA to finish advances the counters (self-resetting ticket in counters[B2RL_CTR_XTICKET]).
 * new_rows may be device memory or pinned host memory (device-addressable: the kernel then is the host->device copy).
 * Same kernel and results as b2rl_replay_extend_dev_stack with n_agents = 1. */
int b2rl_replay_extend_dev(float* storage, int64_t capacity, b2rl_rowfmt_t fmt, const float* new_rows, int32_t n,
                           uint64_t* counters, void* stream);

/* b2rl_replay_extend_dev for n_agents stacked learners (a population: every member appends n transitions per step).
 *   storage   [n_agents][..][row_stride], agent g's slice of `capacity` rows at storage + g * storage_agent_stride
 *             (>= capacity * row_stride floats, a multiple of 4; any value when n_agents == 1)
 *   new_rows  [n_agents][n][row_stride], contiguous, device or pinned host memory
 *   counters  uint64[n_agents][8]: agent g's cursor, fill count and ticket are counters[g*8 + B2RL_CTR_CURSOR / _SIZE /
 *             _XTICKET]; each agent's cursor and size advance on their own (the last CTA of agent g's grid row) */
int b2rl_replay_extend_dev_stack(float* storage, int64_t storage_agent_stride, int64_t capacity, b2rl_rowfmt_t fmt,
                                 const float* new_rows, int32_t n, int32_t n_agents, uint64_t* counters, void* stream);

/* ---- stacked agents on the wide path ------------------------------------------------------------------------------------
 * Every entry point of the wide (layer-by-layer, tensor-core) path below takes a trailing `const b2rl_stack_t* stack`.
 * NULL = one learner, M batch rows. Otherwise n_agents independent learners are processed by the same launches
 * (BASELINE.json config 4: a population of agents, the reference's one-process-per-seed scale-out, spawner.py:148-178):
 *   - M is the number of rows PER AGENT and every per-row array ([M][..]) is [n_agents][M][..], contiguous;
 *   - every parameter / gradient pointer (weights, biases, LayerNorm affine, the gradient region G) addresses agent 0's
 *     copy and agent g's is `param_stride` floats further (the arena's agent stride); lo parts: `lo_stride`;
 *   - per-agent scalars: log_alpha / alpha state (`alpha_stride` floats), step counters (`counters_stride` uint64), the
 *     log block `out` (`out_stride` floats); per-CTA partial-sum scratch arrays are [n_agents][P][..];
 *   - Philox streams are keyed on the GLOBAL agent id `agent_base + g` and on the row index inside the agent's batch,
 *     so the draws equal those of the single-learner path and do not depend on how a population is sharded.
 * No data is shared between agents and nothing is reduced across them. */
typedef struct b2rl_stack {
  int32_t n_agents;        /* >= 1 */
  int32_t agent_base;      /* global id of local agent 0 */
  int64_t param_stride;    /* floats between consecutive agents' copies of a parameter / gradient tensor */
  int64_t lo_stride;       /* floats between consecutive agents' lo-part tensors (b2rl_tc_split_lo) */
  int64_t alpha_stride;    /* floats between agents' log_alpha state blocks */
  int64_t counters_stride; /* uint64 between agents' counter blocks (8) */
  int64_t out_stride;      /* floats between agents' log blocks (8) */
  const b2rl_agent_hp_t* agent_hp; /* dev [n_agents] or NULL: per-agent gamma (critic heads), td3_std / td3_c (policy head
                                      with smoothing), targ_ent (b2rl_wide_alpha_grad) in place of the scalars */
} b2rl_stack_t;

/* Large-batch hidden layer on the tensor cores (tcgen05.mma kind::tf32, operands staged by TMA, accumulator in
 * TMEM): H = [ReLU](LayerNorm(X . W^T + bias)) for X [M][256] (row pitch ldx floats, 16-byte aligned rows) and W
 * [256][256] in torch's natural layout — agents/nets.py:66-82 (fc_block_2) for M in the tens of thousands
 * (BASELINE.json config 5 / stacked populations). Products are TF32 (~1e-3 relative), accumulation, LayerNorm and
 * outputs fp32. H [M][256]; XH (x-hat, or the pre-activation when ln = 0) and stat (mean, rstd per row) may be
 * NULL. Builds two TMA descriptors on the host, then enqueues one kernel. */
int b2rl_tc_linear(const float* X, int64_t ldx, int32_t M, const float* W, const float* W_lo, const float* bias, const float* g,
                   const float* be, int32_t layer_norm, int32_t relu, float* H, float* XH, float* stat, const b2rl_stack_t* stack,
                   void* stream);
/* W_lo (here, in b2rl_tc_linear_q and in b2rl_tc_linear_bwd): NULL => plain TF32 products (~1e-3); else 3xTF32: x = hi +
 * lo, a.b ~ hi.hi + lo.hi + hi.lo as three MMAs into the same TMEM accumulator — fp32-level accuracy (~1e-6) on the
 * tensor cores (the activations' lo parts are made in shared memory). The weights' lo parts come from W_lo, the mirror
 * b2rl_tc_split_lo / the optimizer launch (b2rl_adam_args_t.lo) keep — or, with W_lo == W, are made in shared memory as
 * well from each slab TMA delivers: no mirror to read or to keep current, the right trade when a weight slab serves one
 * tile pair only (stacked agents: per-agent weights). The same three products either way (their order in the
 * accumulation differs, so results agree to fp32 rounding, not bitwise). */
int b2rl_tc_split_lo(const float* W, float* W_lo, int32_t n, const b2rl_stack_t* stack, void* stream);

/* ---- the wide (layer-by-layer, tensor-core) path for large batches: csrc/wide.cu, csrc/tc_linear.cu ------------------
 * Each entry point is one batch-parallel kernel of agents/agent.py:186-235 / agents/nets.py; the host mirror
 * (sac_td3_cudagraphs_pytorch_b200/wide.py) strings them together. Intermediates are [M][256] fp32 arrays in HBM. */

/* First layer (agents/nets.py:66-72): H = ReLU(LayerNorm(X[:, :K] . w1t + b)); w1t [K][256] forward layout. */
int b2rl_wide_first(const float* X, int64_t ldx, int32_t M, int32_t K, const float* w1t, const float* b, const float* g,
                    const float* be, int32_t layer_norm, float* H, float* XH, float* stat, const b2rl_stack_t* stack, void* stream);

/* The same first layer on the tensor cores (tc_linear.cu, MODE 1): the rows' inputs are the K-major operand (columns beyond
 * K zero-filled by TMA), w1t — forward layout, i.e. MN-major — the other; LayerNorm / ReLU / outputs in the TMEM epilogue as
 * in b2rl_tc_linear. x3 != 0: 3xTF32 (both lo parts made in shared memory), else plain TF32. Needs X 16-byte aligned and
 * ldx a multiple of 4 floats (TMA); b2rl_wide_first is the fallback for other layouts. */
int b2rl_tc_first(const float* X, int64_t ldx, int32_t M, int32_t K, const float* w1t, const float* b, const float* g,
                  const float* be, int32_t layer_norm, float* H, float* XH, float* stat, int32_t x3, const b2rl_stack_t* stack,
                  void* stream);

/* Backward dX product of the hidden layer on the tensor cores with the LayerNorm / ReLU backward of layer 1 in the
 * epilogue: DZ1 = LNbwd(ReLU'(DZ2 . W2)); w2t = forward-layout copy of fc_block_2.fc.weight; part [ceil(M/128)][3][256]
 * receives per-CTA column sums {sum dz, sum dn*xhat, sum dn}, or is NULL when only DZ1 is wanted (the actor step's pass
 * through the critics, agents/agent.py:272-283: no critic parameter gradient is used there). */
int b2rl_tc_linear_bwd(const float* DZ2, int32_t M, const float* w2t, const float* w2t_lo, const float* xh1, const float* stat1,
                       const float* g1, const float* be1, int32_t layer_norm, float* DZ1, float* part, const b2rl_stack_t* stack,
                       void* stream);

typedef struct b2rl_wide_policy {  /* policy head + action sample (agents/nets.py:143-147, :214-234; agent.py:194-205) */
  const float* h2;      /* [M][256] */
  const float* w3;      /* [out][256] */
  const float* b3;
  const float* rows;    /* [M][row_stride]: the obs-part of xn is copied from column src_off */
  const float* min_ac;
  const float* max_ac;
  const float* eps;     /* [M][A] or NULL => Philox */
  float* eps_out;       /* or NULL */
  float* xn;            /* out [M][ldn]: [obs-part | action] */
  float* logp;          /* out [M] (SAC) or NULL */
  float* save;          /* out [M][4][A] or NULL: eps, sigma, tanh(x), tanh(raw log-std) for the head's backward pass */
  const uint64_t* counters;
  int32_t M, O, A, out_dim, row_stride, ldn, src_off;
  int32_t td3, smoothing, counter_idx, stream_id;
  float td3_std, td3_c;
  uint64_t seed;
  uint32_t agent;
  uint32_t reserved;
} b2rl_wide_policy_t;
int b2rl_wide_policy_head(const b2rl_wide_policy_t* p, const b2rl_stack_t* stack, void* stream);

/* Behaviour policy on the wide path: b2rl_actor_predict (Agent.predict, agents/agent.py:172-181, nets.py:149-159, :222-234)
 * for ONE learner on the h2 [n][256] of its actor — b2rl_tc_first and b2rl_tc_linear on the n observations — so that the
 * actor's weights are read once per 128 rows instead of once per 8. mode, explore_std, draw, eps and agent_hp mean what they
 * mean for b2rl_actor_predict, and the Philox noise is the same numbers (key ~seed, the global id `agent`, row and action
 * dimension as there; draw = UINT64_MAX: counters[B2RL_CTR_Q] | 2^31): the two policies differ only by the forward pass's
 * arithmetic. TD3 mode 1 adds the noise unclamped, as b2rl_actor_predict does. */
typedef struct b2rl_wide_predict {
  const float* h2;      /* [n][256] */
  const float* w3;      /* [out_dim][256] */
  const float* b3;
  const float* min_ac;
  const float* max_ac;
  const float* eps;     /* [n][A] or NULL => Philox */
  float* eps_out;       /* [n][A] or NULL: the noise used (mode 1) */
  float* actions;       /* out [n][A] */
  const uint64_t* counters;         /* the learner's (read when draw = UINT64_MAX) */
  const b2rl_agent_hp_t* agent_hp;  /* NULL, or a row whose explore_std replaces explore_std */
  int32_t n, A, out_dim, mode, td3;
  float explore_std;    /* TD3 mode 1 (hps.actor_noise_std) */
  uint64_t seed;        /* the learner's hp.seed */
  uint64_t draw;
  uint32_t agent;       /* global learner id */
  uint32_t reserved;
} b2rl_wide_predict_t;
int b2rl_wide_actor_predict(const b2rl_wide_predict_t* p, void* stream);
/* n rows of `width` floats from src (row pitch lds floats) to dst (pitch ldd): ONE memory-copy node (cudaMemcpy2DAsync),
 * either side device or pinned host memory. Puts pinned observations [n][O] into the [n][(O + 3) & ~3] device buffer whose
 * rows TMA can address (b2rl_tc_first). */
int b2rl_copy_rows(float* dst, int64_t ldd, const float* src, int64_t lds, int32_t n, int32_t width, void* stream);

typedef struct b2rl_wide_q {  /* critic head; mode 1 adds the TD target, dLoss/dQ and squared-error partials (agent.py:212-233) */
  const float* h2;
  const float* w3;
  const float* b3;
  float* q_out;         /* [M] */
  const float* qn0;     /* mode 1: twin target Q on (next_obs, a') */
  const float* qn1;
  const float* logp;    /* SAC */
  const float* rows;    /* reward at column rd_off, done at rd_off + 1 */
  const float* log_alpha;
  float* dz3;           /* [M][B2RL_MAX_OUT], column 0 */
  float* sq_part;       /* [ceil(M/8)][2]: per-CTA {sum of squared errors, sum of dQ} */
  float* targ_out;      /* [M] or NULL */
  int32_t M, mode, row_stride, rd_off, td3, bcq_mix;
  float gamma;
  uint32_t reserved;
} b2rl_wide_q_t;
int b2rl_wide_q_head(const b2rl_wide_q_t* q, const b2rl_stack_t* stack, void* stream);
/* The critic's second layer (b2rl_tc_linear with ReLU) with that head fused into its epilogue — the thread that owns a row
 * of h2 takes its dot product with w3 (q->h2 is ignored): no second pass over h2, and H may be NULL (target critics:
 * h2 never goes to memory). agents/nets.py:88-92 + agents/agent.py:208-233. */
int b2rl_tc_linear_q(const float* X, int64_t ldx, int32_t M, const float* W, const float* W_lo, const float* bias, const float* g,
                     const float* be, int32_t layer_norm, float* H, float* XH, float* stat, const b2rl_wide_q_t* q,
                     const b2rl_stack_t* stack, void* stream);

/* Head backward + ReLU mask + LayerNorm backward of layer 2: dz = LNbwd(ReLU'(dz3[:, :n_out] . w3)); part
 * [ceil(M/128)][3][256] per-CTA column sums (NULL: dz only). dw3_part (NULL, or [ceil(M/128)][3][256] with n_out == 1): per-CTA partials
 * (slot 0) of the scalar head's weight gradient dW3[j] = sum_b dz3[b] * h2[b][j], h2 recomputed from x-hat — finish with
 * b2rl_wide_colsum(dw3_part, P, G, off_w3, 0, 0, 0, ...): the critics then need no b2rl_tc_wgrad launch for w3. */
int b2rl_wide_ln_bwd(const float* dz3, int32_t n_out, const float* w3, const float* xh, const float* stat, const float* g,
                     const float* be, int32_t layer_norm, int32_t M, float* dz, float* part, float* dw3_part,
                     const b2rl_stack_t* stack, void* stream);
/* Column-sum partials -> gradients of bias / ln.weight / ln.bias at float offsets off_* of the gradient region G. */
typedef struct b2rl_colsum_job {
  const float* part;              /* [P][3][256] per-CTA partial column sums (agent g: P * 768 floats further) */
  int64_t off_b, off_g, off_be;   /* float offsets in the gradient region: column sums 0 / 1 / 2 (1, 2: layer_norm only) */
  int32_t layer_norm;
  int32_t reserved;
} b2rl_colsum_job_t;
#define B2RL_MAX_COLSUM_JOBS 8
/* The same for up to 8 partial-sum arrays of equal P in ONE launch (`jobs` is read on the host at call time): a step's
 * column sums have different producers but one consumer, the optimizer launch, so they can all be taken at the end of the
 * step. Per job bitwise equal to b2rl_wide_colsum. */
int b2rl_wide_colsum_multi(const b2rl_colsum_job_t* jobs, int32_t n_jobs, int32_t P, float* G, const b2rl_stack_t* stack,
                           void* stream);
int b2rl_wide_colsum(const float* part, int32_t P, float* G, int64_t off_b, int64_t off_g, int64_t off_be, int32_t layer_norm,
                     const b2rl_stack_t* stack, void* stream);
/* qf_loss -> out[B2RL_OUT_QF_LOSS] and the head-bias gradients of the twin critics, from wide_q_head's per-CTA partials
 * (sq0 / sq1 [P][2]; dz3_0 / dz3_1 are unused and may be NULL). */
int b2rl_wide_critic_scalars(const float* sq0, const float* sq1, int32_t P, const float* dz3_0, const float* dz3_1, int32_t M,
                             float* G, int64_t off_b3_0, int64_t off_b3_1, float* out, const b2rl_stack_t* stack, void* stream);
/* Actor step, wide path (agents/agent.py:247-303). actor_loss: per-row loss and dLoss/dQ_k (column 0 of dzq_k
 * [M][B2RL_MAX_OUT]; q1 / dzq1 NULL for TD3), per-CTA partials part [ceil(M/256)][2]. dqda: dQ/da = dz1 . w1t[O + a][:]
 * (w1a = w1t + O * 256). actor_head_bwd: du [M][B2RL_MAX_OUT] = dLoss/d(head outputs) from dQ/da (summed over the
 * critics) and the saved sampling intermediates; part_du [ceil(M/256)][B2RL_MAX_OUT]. actor_scalars: loss / mean
 * log-prob / alpha -> out, d head.bias -> G. alpha_grad: alpha_state[1] <- alpha * mean(-logpi'' - targ_ent); follow
 * with b2rl_alpha_adam. */
int b2rl_wide_actor_loss(const float* q0, const float* q1, const float* logp, const float* log_alpha, int32_t td3, int32_t M,
                         float* dzq0, float* dzq1, float* part, const b2rl_stack_t* stack, void* stream);
int b2rl_wide_dqda(const float* dz1, const float* w1a, int32_t A, int32_t M, float* dqda, const b2rl_stack_t* stack, void* stream);
int b2rl_wide_actor_head_bwd(const float* dqda0, const float* dqda1, const float* save, const float* min_ac,
                             const float* max_ac, const float* log_alpha, int32_t td3, int32_t A, int32_t M, float* du,
                             float* part_du, const b2rl_stack_t* stack, void* stream);
int b2rl_wide_actor_scalars(const float* part_s, const float* part_du, int32_t P, int32_t M, int32_t out_dim, int32_t td3,
                            const float* log_alpha, float* G, int64_t off_b3, float* out, const b2rl_stack_t* stack, void* stream);
int b2rl_wide_alpha_grad(const float* logp2, int32_t M, float targ_ent, float* alpha_state, const b2rl_stack_t* stack, void* stream);
/* (b2rl_wide_q_head / b2rl_tc_linear_q read gamma, b2rl_wide_policy_head td3_std / td3_c when smoothing, and
 * b2rl_wide_alpha_grad targ_ent from stack->agent_hp when it is set.) */

/* Weight gradient of one layer on the tensor cores (tc_wgrad.cu): C[m][n] = sum_b A[b][m] * Bm[b][n] for m < MA, with A
 * [Bn][lda] (a_cols >= MA columns exist; 16-byte aligned rows) and Bm [Bn][256]; Ct, if not NULL, receives the transpose
 * [256][MA]. Split over the batch, slices added in a fixed order. scratch: b2rl_tc_wgrad_scratch_floats(MA, Bn) floats.
 * x3: 3xTF32 (fp32-level accuracy) or plain TF32. bump, if not NULL: a device counter incremented once (the update
 * counter b2rl_wgrad advances: agents/agent.py:240 / :288 count optimizer steps; stacked: agent g's is bump +
 * g * counters_stride). Stacked: A, Bm are [n_agents][Bn][..], C / Ct are gradient tensors (param_stride apart), and the
 * number of batch splits depends on (MA, Bn) only — never on n_agents — so a population's gradients are bitwise the
 * same however it is sharded. Replaces, for large batches, what
 * loss.backward() does for the weights (agents/agent.py:235,283). */
int b2rl_tc_wgrad(const float* A, int64_t lda, int32_t a_cols, int32_t MA, const float* Bm, int32_t Bn, float* C, float* Ct,
                  float* scratch, int32_t x3, uint64_t* bump, const b2rl_stack_t* stack, void* stream);
int64_t b2rl_tc_wgrad_scratch_floats(int32_t MA, int32_t Bn, int32_t n_agents /* 0: the single-learner form (stack NULL) */);

/* The weight-gradient kernel on its own (wgrad.cu): reads rows, H1, H2, DZ1, DZ2, DZ3 of the workspace. skip_vectors:
 * the bias / LayerNorm / loss reductions were done elsewhere (wide path). bump_counter: B2RL_CTR_* or -1. */
int b2rl_wgrad(const b2rl_update_args_t* a, int32_t actor_step, int32_t bump_counter, int32_t skip_vectors, void* stream);

/* End of a captured learner step: copy the log block `out` (float[8] per agent, device) into `host_out` — pinned
 * host memory, written by the kernel itself over PCIe/NVLink-C2C, no copy-engine node — then advance the device
 * sequence number *seq_dev and publish it in *host_seq (system-scope fence in between): the host polls *host_seq
 * instead of synchronising the stream. Replaces the `.item()` / clone-and-sync reads of the losses in the
 * reference's logging path (orchestrator.py:341-352, :383). */
int b2rl_publish_logs(const float* out, int32_t n_agents, float* host_out, uint64_t* seq_dev, uint64_t* host_seq,
                      void* stream);

/* Replaces Agent.update_qnets up to and including `qf_loss.backward()` (agents/agent.py:186-235);
 * advances counters[Q] (the optimizer's step_t += 1) so that the Adam launch that follows sees t:
 * next action (SAC: online tanh-Gaussian sample + log-prob, nets.py:222-234; TD3: target actor +
 * clipped noise, agent.py:194-202), twin target Q (agent.py:208-210), min / BCQ mix (:212-219),
 * entropy term (:221-223), TD target (:226-228), twin online Q + per-critic MSE + sum (:230-233),
 * full backward into region 4 (gradients of both critics). Writes out[QF_LOSS]. Two launches. */
int b2rl_critic_update_sac(const b2rl_update_args_t* a, void* stream);
int b2rl_critic_update_td3(const b2rl_update_args_t* a, void* stream);

/* Replaces Agent.update_actor up to `actor_loss.backward()` (agents/agent.py:247-283): actor
 * forward (+ reparameterised sample and log-prob for SAC), twin Q with constant critic params
 * (:272-278), loss `alpha*logpi - min Q` (SAC) or `-Q_0` (TD3), backward through the critics'
 * inputs into the actor; gradients of the actor into region 4. Writes out[ACTOR_LOSS]; advances
 * counters[PI]. Two launches. */
int b2rl_actor_update_sac(const b2rl_update_args_t* a, void* stream);
int b2rl_actor_update_td3(const b2rl_update_args_t* a, void* stream);

/* b2rl_{critic,actor}_update_* FOLLOWED BY b2rl_adam_polyak_multi(opt), as two launches instead of three: the
 * weight-gradient kernel applies Adam (and the Polyak average) to each parameter whose gradient it has just
 * produced — `optimizer.step()` (agents/agent.py:236,286) and `update_targ_nets` (:320-331) without a launch of
 * their own. Same arithmetic as b2rl_adam_polyak_multi: results are bitwise equal. The algorithm is taken from
 * a->hp.td3. opt->seg[0] must be an Adam segment (clip = 0, grad_scale = 1) over exactly the trained nets
 * ([critic[0].begin, critic[1].end) / [actor.begin, actor.end)) with the matching counter; further segments must
 * be Polyak-only spans (e.g. TD3's actor target in an iteration without actor update). Gradient clipping and
 * data-parallel training need the gradients complete before the step: use the three-launch form there. The
 * 3xTF32 mirror is not written here: opt->lo must be NULL (B2RL_E_INVALID otherwise, before any launch), and a
 * learner that keeps a mirror uses the three-launch form. The same holds for per-agent hyperparameters: a->agent_hp
 * and opt->agent_hp must be NULL. */
int b2rl_critic_update_opt(const b2rl_update_args_t* a, const b2rl_adam_args_t* opt, void* stream);
int b2rl_actor_update_opt(const b2rl_update_args_t* a, const b2rl_adam_args_t* opt, void* stream);

/* Replaces the autotune tail of update_actor (agents/agent.py:295-303): second no-grad
 * get_action with the UPDATED actor and fresh noise (a->eps2), alpha_loss, its gradient, and the
 * scalar Adam step on log_alpha (lr = log_alpha_lr; 0 = gradient only, see b2rl_alpha_adam). Writes
 * out[ALPHA_LOSS], out[ALPHA]; bumps counters[ALPHA]. One launch. With a->agent_hp, agent g's target entropy is
 * its row's targ_ent, and a positive log_alpha_lr means "step with the row's lr[B2RL_CTR_ALPHA]". */
int b2rl_alpha_update(const b2rl_update_args_t* a, float log_alpha_lr, void* stream);

/* Data-parallel variant of the temperature step: b2rl_alpha_update with log_alpha_lr == 0 only
 * computes the LOCAL alpha_loss and its gradient (log_alpha state slot 1) and leaves log_alpha alone;
 * after the gradient has been summed over ranks, this applies the scalar Adam step with
 * g = grad_scale * state[1] (grad_scale = 1/world) and bumps counters[ALPHA]. */
int b2rl_alpha_adam(float* log_alpha, uint64_t* counters, int32_t n_agents, float log_alpha_lr,
                    float grad_scale, float* out, void* stream);
/* b2rl_alpha_adam with per-agent learning rates: agent g steps with hp[g].lr[B2RL_CTR_ALPHA] (hp: dev [n_agents]). */
int b2rl_alpha_adam_hp(float* log_alpha, uint64_t* counters, int32_t n_agents, const b2rl_agent_hp_t* hp,
                       float grad_scale, float* out, void* stream);

/* Sum of squares of the gradient span [begin,end) of region 4, per agent, into sumsq[agent]
 * (first half of clip_grad_norm_, agents/agent.py:284-285). Deterministic two-stage reduction. */
int b2rl_grad_sumsq(const float* arena, int64_t region_stride, int64_t arena_agent_stride,
                    int64_t begin, int64_t end, int32_t n_agents, float* sumsq, float* scratch,
                    void* stream);

/* Replaces `optimizer.step()` (agents/agent.py:236,286; torch _multi_tensor_adam, ~16 foreach
 * launches per step) and `update_targ_nets` (agents/agent.py:320-331; foreach lerp_) with ONE
 * launch over up to B2RL_MAX_SEG spans. Adam follows torch's `capturable` branch
 * (torch/optim/adam.py:478-527), which is what the reference runs on the GPU (agent.py:118). */
int b2rl_adam_polyak_multi(const b2rl_adam_args_t* a, void* stream);

/* counters[which] += 1 for every agent (the optimizer's `step_t += 1`, adam.py:413). Runs as a
 * 1-thread-per-agent kernel so the value the *next* launches see is stream-ordered. */
int b2rl_bump_counter(uint64_t* counters, int32_t which, int32_t n_agents, void* stream);

/* Replaces the policies behind Agent.predict (agents/agent.py:172-181, nets.py:149-159,222-234):
 * actor forward on n observation rows [n][ob_dim] -> actions [n][A].
 *   mode 0: SAC mode / TD3 exploit;  1: SAC sample / TD3 explore (noise from a->eps [n][A], or
 *   Philox keyed on (`draw`, a->agent_base = the learner's global id), `draw` < 2^31 advanced by the caller per call;
 *   draw = UINT64_MAX with a->counters set: keyed on counters[B2RL_CTR_Q] | 2^31, for use inside a captured step graph,
 *   a key space disjoint from the host-counted draws). `obs` and `actions_out` may be pinned host memory
 *   (device-addressable): the kernel then is the host<->device copy.
 * Stacked agents (a->n_agents > 1; 0 or 1 = one learner): agent g reads its actor at a->arena + g * a->arena_agent_stride,
 *   its counters at a->counters + g * 8 (draw = UINT64_MAX), keys its noise on the global id a->agent_base + g, and
 *   obs / a->eps / actions_out are [n_agents][n][..], contiguous. Each agent's actions equal those of a single call for it.
 *   a->agent_hp: agent g's TD3 noise std in mode 1 is its row's explore_std (explore_std is then ignored).
 *   a->eps_out [n_agents][n][A] or NULL: mode 1 records the noise it used there. */
int b2rl_actor_predict(const b2rl_update_args_t* a, const float* obs, int32_t n, int32_t mode,
                       float explore_std, uint64_t draw, float* actions_out, void* stream);

/* Measurement hook: enqueue exactly ONE kernel of the update so that bench.py / ncu can time it in
 * isolation. which: 0 critic_fused, 1 critic wgrad, 2 actor_fused, 3 actor wgrad, 4 alpha (SAC).
 * Step counters are NOT advanced (wgrad's bump is disabled), otherwise same work as in the update. */
int b2rl_launch_single(const b2rl_update_args_t* a, int32_t which, void* stream);

/* fp32 FFMA peak probe (roofline denominator for the fused MLP kernels): runs `iters` dependent
 * FFMA chains on every SM; the caller times it. flops = 2 * 148*? is returned through *flops. */
int b2rl_ffma_probe(float* sink, int32_t iters, double* flops, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B2RL_H */
