/* dppo.h — C ABI of libdppo.so, the sm_100a implementation of Diamond PPO's hot path.
 *
 * The reference (Auxeno/diamond-ppo) is pure Python/PyTorch and has no FFI layer; its "plugin
 * boundary" for this path is the Python API (PPO / ContinuousPPO / RecurrentPPO, the PPOConfig
 * family and the custom-network interface).  This header is the native boundary a maintainer
 * would bind from that Python code (ctypes, see INTEGRATION.md); every entry point names the
 * reference lines whose arithmetic it replaces (paths relative to the reference root).
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on error; dppo_last_error(ctx) has the text
 *   - all device pointers are caller-owned (PyTorch tensors); the library allocates nothing on
 *     the device.  Scratch memory is passed in as `ws` (size from the *_workspace_bytes calls)
 *   - every launch is asynchronous on the cudaStream_t passed as `stream` (void*); no entry
 *     point synchronises the device
 *   - only sm_100a SASS is embedded: creating a context on any other GPU is an error.  There
 *     is no CPU fallback
 *   - layouts: rollout tensors are time-major [T, N, ...] with the env index contiguous
 *     (flat sample index i = t*N + env, diamond/ppo.py:246-249); weights are row-major
 *     [out, in] like torch.nn.Linear
 */
#ifndef DPPO_H
#define DPPO_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DPPO_VERSION 100
#define DPPO_MAX_ACT 32          /* action count / action dims handled by the fused head kernels */
#define DPPO_GEMM_HEADS_MAX_HIDDEN 2048   /* bounds of the GEMM-head path (dppo_mlp_grad_minibatch_gemm_heads) */
#define DPPO_GEMM_HEADS_MAX_ACT 1024

typedef struct dppo_ctx dppo_ctx;

/* Default actor-critic MLP (diamond/ppo.py:40-71, diamond/continuous_ppo.py:50-82). */
typedef struct dppo_mlp_desc {
    int32_t obs_dim;      /* D */
    int32_t hidden;       /* H = cfg.network_hidden_dim */
    int32_t act_dim;      /* A: Discrete.n, or prod(Box.shape) when continuous */
    int32_t continuous;   /* 0: categorical logits head; 1: gaussian mean head + actor_log_std */
} dppo_mlp_desc;

/* Offsets (in floats) of each tensor inside the flat parameter / gradient / Adam buffers.
 * w3/b3 hold actor_head.0 (rows 0..H-1) and critic_head.0 (rows H..2H-1) back to back so both
 * first head layers run as one [2H, H] product.  Every offset is a multiple of 4 floats. */
typedef struct dppo_mlp_layout {
    int64_t w1, b1;       /* base.0  [H, D], [H] */
    int64_t w2, b2;       /* base.2  [H, H], [H] */
    int64_t w3, b3;       /* actor_head.0 | critic_head.0  [2H, H], [2H] */
    int64_t wa, ba;       /* actor_head.2 (actor_mean_head.2)  [A, H], [A] */
    int64_t wc, bc;       /* critic_head.2  [1, H], [1] */
    int64_t log_std;      /* actor_log_std [A] (continuous only, else -1) */
    int64_t total;        /* floats in the flat buffer (padded) */
} dppo_mlp_layout;

/* Hyper-parameters of one optimiser step (PPOConfig fields, diamond/ppo.py:17-37). */
typedef struct dppo_hyper {
    float ppo_clip;           /* cfg.ppo_clip */
    float value_loss_weight;  /* cfg.value_loss_weight */
    float entropy_beta;       /* cfg.entropy_beta */
    float grad_norm_clip;     /* cfg.grad_norm_clip */
    float adam_eps;           /* cfg.adam_eps */
    float pad0;
    double lr;                /* current learning rate (after LinearLR, ppo.py:137-142) */
    double beta1, beta2;      /* 0.9, 0.999 (torch.optim.Adam defaults, ppo.py:135) */
    int64_t step;             /* 1-based Adam step count of THIS update */
    int32_t advantage_norm;   /* cfg.advantage_norm: normalise with adv_stats while gathering */
    int32_t pad1;
    int64_t adv_count;        /* number of samples behind adv_stats (global batch T*N) */
    int64_t loss_denominator; /* rows the loss means divide by (global minibatch size) */
    const float* step_consts; /* optional DEVICE pointer to 16 bytes {f32 sqrt(1 - beta2^step), f32 -lr / (1 - beta1^step), u64 seq}:
                                 when set, the Adam kernel reads its two step-dependent constants (and the data-parallel exchange
                                 kernel the sequence number it publishes / waits for) from device memory instead of from lr / step,
                                 so a captured CUDA graph of an optimiser step can be replayed */
    double* grad_sumsq;       /* optional DEVICE buffer of dppo_grad_sumsq_bytes(): dppo_mlp_grad_minibatch and
                                 dppo_rnn_grad_minibatch leave the fp64 partial sums of squares of the gradient they assembled there
                                 and dppo_clip_adam_step reads them instead of launching its own norm kernel (single-GPU path; under
                                 DP the norm is taken after the exchange) */
} dppo_hyper;

/* ---- context -------------------------------------------------------------------------- */
int dppo_create(dppo_ctx** out, int device);
int dppo_destroy(dppo_ctx* ctx);
const char* dppo_last_error(dppo_ctx* ctx);          /* ctx may be NULL: last create() error */
int dppo_version(void);
int dppo_device_info(dppo_ctx* ctx, int* sm_count, int* cc_major, int* cc_minor);
int64_t dppo_launch_count(dppo_ctx* ctx);            /* kernels launched through this context so far */
int dppo_count_launches(dppo_ctx* ctx, int64_t n);   /* add n: launches replayed from a CUDA graph captured through this context */
/* Kernel-variant switches used by tests and bench.py for A/B measurements:
 *   "tensor_cores" 1 (default): CTA-pair (cta_group::2) persistent 3xTF32 tcgen05 GEMMs + tcgen05 weight gradients where
 *                  the shape allows (rows >= 1024, K % 16 == 0, N % 256 == 0 or N == 128); 0: FP32 FFMA GEMMs everywhere
 *   "row_sweep"    bit mask, default 31: L2 reuse along the layer chain of an optimiser step / the pre-update pass.  1: consecutive
 *                  GEMM launches alternate the direction of their row sweep (a launch starts with the rows its predecessor wrote
 *                  last, which are still in the L2); 2: the head kernels sweep against the GEMM before them; 4: the head kernel's
 *                  d3 stores are plain instead of streaming; 8: inputs that are dead after the launch are read with the L2
 *                  evict-first hint; 16: the same for the operands of the weight-gradient launch.  0 = every launch ascending,
 *                  no hints (A/B).  Forward outputs do not depend on the mask; masks 1 and 2 re-order fp32
 *                  partial sums of the gradient (deterministic for a fixed mask)
 *   "tc_prefetch"  bit mask, default 0: software L2 prefetch ahead of the TMA loads (kept for A/B).  1: forward GEMMs and 2: dgrad
 *                  GEMMs prefetch the next tile's activations while the current tile computes, 4: the weight-gradient kernel
 *                  prefetches its operand chunks 8 chunks ahead.  All three measured slower inside the optimiser step (the
 *                  in-situ DRAM counters show prefetched lines being fetched twice)
 *   "gae_variant"  0 (default): pipelined TMA-staged GAE kernel (T >= 128; chunked loads, stores overlap them) or the
 *                  single-barrier TMA kernel when the layout allows, 1: register-staged, 2: single-barrier TMA
 *   "gae_inputs_settled" 0 (default): plain launch -- the GAE kernel starts after its stream predecessor has completed and
 *                  requests nothing early (safe for any caller, e.g. a cast kernel writing a mask right before it);
 *                  1: promise that the kernel launched immediately before dppo_gae_f32 on the stream writes none of
 *                  rewards / terminations / truncations (rollout data): the launch uses programmatic stream serialization and
 *                  requests those three tiles before griddepcontrol.wait; 2: promise that it writes none of the five inputs:
 *                  all tiles are requested early and the wait only guards the kernel's global writes, so consecutive
 *                  launches overlap (PPO.learn(): the predecessor is the 32-byte statistics fill). */
int dppo_set_option(dppo_ctx* ctx, const char* name, int value);

/* ---- rollout buffer + batched action sampling (diamond/ppo.py:153-186, 73-82) ---------- */
/* Unpack one vectorised env step, staged as ONE packed record
 *   [obs f32 N*D | next_obs f32 N*D | rewards f64 N | actions (i64 N | f32 N*A) | term u8 N | trunc u8 N]
 * (the six arrays diamond/ppo.py:165-172 appends), into row t of the time-major device buffers
 * with the casts of ppo.py:229-232 (rewards/terminations/truncations -> f32; actions i64 -> i32). */
int dppo_buffer_store_step(dppo_ctx* ctx, const void* record, int t, int N, int D, int act_dim, int continuous,
                           float* obs, float* next_obs, void* actions, float* rewards,
                           float* terminations, float* truncations, void* stream);
int64_t dppo_step_record_bytes(int N, int D, int act_dim, int continuous);

/* Categorical(logits).sample() (ppo.py:81) with a counter-based generator keyed by
 * (seed, global env id, draw counter): results do not depend on the launch shape or GPU count.
 * Also emits log_prob(action) (recurrent_ppo.py:219-221).  actions: int64 [N]. */
int dppo_sample_categorical(dppo_ctx* ctx, const float* logits, int N, int A, uint64_t seed, uint64_t counter,
                            int64_t env_offset, int64_t* actions, float* log_probs, void* stream);
/* Greedy action of a categorical policy (evaluation): actions[e] = torch.argmax(logits[e], -1), the FIRST index of the row's
 * maximum; a NaN counts as the maximum, so a row holding a NaN selects its first NaN.  log_probs (optional) receives
 * log_softmax(logits[e])[actions[e]] with the arithmetic of dppo_sample_categorical.  No generator is involved.  The greedy action of
 * a Gaussian policy is its mean (heads bit 0 of dppo_mlp_forward / dppo_rnn_forward), which needs no kernel of its own. */
int dppo_select_greedy_categorical(dppo_ctx* ctx, const float* logits, int N, int A, int64_t* actions, float* log_probs, void* stream);
/* JointNormal(mean, exp(log_std)).sample() (continuous_ppo.py:92). actions: f32 [N, A]. */
int dppo_sample_gaussian(dppo_ctx* ctx, const float* mean, const float* log_std, int N, int A, uint64_t seed,
                         uint64_t counter, int64_t env_offset, float* actions, float* log_probs, void* stream);

/* counter_base_dev (device uint64, NULL to clear): while set, every dppo_sample_* launch adds *counter_base_dev to its draw
 * counter at run time -- a captured rollout (counters 0..T-1 baked into the CUDA graph) then draws fresh numbers on every replay. */
int dppo_set_draw_counter_base(dppo_ctx* ctx, const unsigned long long* counter_base_dev);

/* ---- GAE (diamond/ppo.py:188-222) + returns/normalisation (ppo.py:241-243) -------------- */
/* advantages[t,e], returns[t,e] = values + advantages (returns may be NULL).  If stats != NULL,
 * adds sum(A) and sum(A^2) (fp64) to stats[0..1] (caller zeroes them; under env-sharded data
 * parallelism the caller all-reduces the two doubles before normalising). */
int dppo_gae_f32(dppo_ctx* ctx, const float* rewards, const float* terminations, const float* truncations,
                 const float* values, const float* next_values, float* advantages, float* returns,
                 double* stats, int T, int N, double gamma, double gae_lambda, void* stream);
/* out = (adv - mean) / (std + 1e-6), unbiased std over `count` samples described by stats. */
int dppo_adv_normalize_f32(dppo_ctx* ctx, const float* adv, float* out, const double* stats, int64_t count,
                           int64_t n, void* stream);

/* ---- minibatch permutation + gather (diamond/ppo.py:252-255, 261-272) ------------------ */
/* HOST function (no device work): np.random.permutation(n) of the legacy global RandomState,
 * bit-exact: MT19937 state (key[624], *pos) is taken from / returned to np.random.get_state().
 * out: int32 [n].  Meant to run on a worker thread while the GPU processes the previous epoch. */
int dppo_permutation_mt19937(uint32_t* key, int32_t* pos, int64_t n, int32_t* out);
int dppo_mt19937_seed(uint32_t* key, int32_t* pos, uint32_t seed);      /* np.random.seed(int) */
/* Advances the stream exactly as dppo_permutation_mt19937(key, pos, n, .) would, without building the permutation. */
int dppo_permutation_mt19937_skip(uint32_t* key, int32_t* pos, int64_t n);
/* FAST (non-parity) generator, SURVEY.md 2.2 K4a: out[0..n) = a pseudo-random permutation of [0, n) that is a pure function of
 * (seed, counter) -- a keyed Feistel bijection over the next power of two with cycle walking, evaluated per element on the
 * device (no sort, no host work; every data-parallel rank computes the same permutation without communication).  It replaces
 * the reference's np.random.permutation draw (ppo.py:254) when the caller opts out of the bit-exact numpy stream. */
int dppo_permutation_device(dppo_ctx* ctx, uint64_t seed, uint64_t counter, int64_t n, int32_t* out, void* stream);
/* Env-sharded data parallelism (SURVEY.md 8e): perm is ONE global permutation of the concatenated buffer (flat index
 * t*n_global_envs + env, B_global entries, identical on every rank), cut into num_minibatches consecutive global minibatches
 * (ppo.py:255).  For every minibatch k the members whose env lies in [env_lo, env_lo + n_local) are kept in permutation order,
 * re-indexed to the rank-local buffer (t*n_local + env - env_lo) and written to idx_out[k*M_pad ..], padded with -1 up to M_pad
 * (rows with a negative index contribute nothing to dppo_mlp_grad_minibatch); counts[k] = members kept; *overflow |= 1 if a
 * minibatch had more than M_pad members (the surplus is dropped: the caller must treat that as an error). */
int dppo_perm_shard_filter(dppo_ctx* ctx, const int32_t* perm, int64_t B_global, int n_global_envs, int env_lo, int n_local,
                           int num_minibatches, int64_t M_pad, int32_t* idx_out, int32_t* counts, int32_t* overflow, void* stream);
/* dst[i, :] = src[idx[i], :]  (row_floats floats per row; a negative index reads row 0); the fused update gathers on the fly,
 * this standalone form serves the custom-network path. */
int dppo_gather_rows_f32(dppo_ctx* ctx, const float* src, const int32_t* idx, float* dst, int64_t rows,
                         int row_floats, void* stream);

/* ---- actor-critic MLP: forward, fused update (diamond/ppo.py:91-96, 235-238, 258-285) --- */
int dppo_mlp_layout_compute(const dppo_mlp_desc* desc, dppo_mlp_layout* out);
int64_t dppo_mlp_workspace_bytes(const dppo_mlp_desc* desc, int64_t rows, int training);

/* Forward only (pre-update pass ppo.py:235-238 and get_actions ppo.py:75-79).
 * heads bit0: actor output head_out [rows, A] (logits / means); bit1: values [rows].
 * idx (optional int32 [rows]) gathers input rows from obs. */
int dppo_mlp_forward(dppo_ctx* ctx, const dppo_mlp_desc* desc, const float* params, const float* obs,
                     const int32_t* idx, int64_t rows, int heads, float* head_out, float* values,
                     void* ws, int64_t ws_bytes, void* stream);
/* SURVEY.md 8f-2: next_values for GAE when the rollout already recorded values[t] = V(obs[t]) with the current parameters
 * (replaces the critic half of the pre-update pass, ppo.py:238).  Wherever the environment did not finish at step t,
 * next_obs[t] is obs[t+1] and next_values[t] = values[t+1]; the critic is evaluated only on the final observations of finished
 * steps and on the last row.  Which rows those are is decided ON THE DEVICE: every launch has a fixed shape and reads the row
 * count from device memory, so the call needs no host synchronisation between rollout and learn().  next_obs [T*N, D],
 * terminations / truncations / values / next_values [T, N]. */
int64_t dppo_mlp_next_values_workspace_bytes(const dppo_mlp_desc* desc, int T, int N);
int dppo_mlp_next_values(dppo_ctx* ctx, const dppo_mlp_desc* desc, const float* params, const float* next_obs,
                         const float* terminations, const float* truncations, const float* values, int T, int N,
                         float* next_values, void* ws, int64_t ws_bytes, void* stream);
int dppo_logprob_categorical(dppo_ctx* ctx, const float* logits, const int32_t* actions, float* log_probs,
                             int64_t rows, int A, void* stream);
int dppo_logprob_gaussian(dppo_ctx* ctx, const float* mean, const float* log_std, const float* actions,
                          float* log_probs, int64_t rows, int A, void* stream);

/* One minibatch of ppo.py:258-283: gather rows idx[0..M) of the flat rollout tensors, forward,
 * clipped-surrogate + value + entropy loss, full backward.  Writes the flat gradient (layout of
 * dppo_mlp_layout) to grads and (policy, value, entropy, total) to losses[0..3].
 * idx[i] < 0 marks a padding row: it enters no loss term and no gradient (fixed-shape steps under data parallelism).
 * actions: int32 [B] (discrete) or f32 [B, A] (continuous).  adv is the UN-normalised advantage
 * when hyper->advantage_norm is set (normalised on the fly from adv_stats), else used as is. */
int dppo_mlp_grad_minibatch(dppo_ctx* ctx, const dppo_mlp_desc* desc, const float* params, float* grads,
                            const float* obs, const void* actions, const float* old_log_probs, const float* adv,
                            const float* returns, const double* adv_stats, const int32_t* idx, int64_t M,
                            const dppo_hyper* hyper, float* losses, void* ws, int64_t ws_bytes, void* stream);
/* dppo_mlp_grad_minibatch runs its output heads in one fused kernel (one warp per row, lane a <-> action a, Wa and per-warp
 * [(A+1), H] weight-gradient accumulators in shared memory).  That kernel takes 1 <= act_dim <= 32, hidden <= 512 and
 * 9 (act_dim + 1) hidden floats within 200 KB; it refuses every other shape.  dppo_mlp_fused_heads_supported returns 1 exactly
 * for the shapes it takes (host only, no context needed).
 * dppo_mlp_grad_minibatch_gemm_heads computes the same gradient with GEMM heads: the head products, their backward and the head
 * weight gradients are GEMMs, and a row kernel evaluates the distribution, the loss and the critic head.  Same arguments, same
 * flat-gradient layout, losses and hyper->grad_sumsq partials as dppo_mlp_grad_minibatch (results agree to fp32 summation
 * order), no synchronisation, no allocation; ws of dppo_mlp_gemm_heads_workspace_bytes(desc, M) bytes.  It takes every shape
 * with hidden <= DPPO_GEMM_HEADS_MAX_HIDDEN and 1 <= act_dim <= DPPO_GEMM_HEADS_MAX_ACT, including those the fused kernel
 * takes, and refuses larger ones with an error naming the bound; the workspace size is 0 for them.
 * dppo_mlp_forward and dppo_mlp_next_values choose by themselves: the fused head evaluation up to 32 actions and hidden 512,
 * else the actor product as a GEMM and one warp per row for the critic. */
int dppo_mlp_fused_heads_supported(const dppo_mlp_desc* desc);
int64_t dppo_mlp_gemm_heads_workspace_bytes(const dppo_mlp_desc* desc, int64_t rows);
int dppo_mlp_grad_minibatch_gemm_heads(dppo_ctx* ctx, const dppo_mlp_desc* desc, const float* params, float* grads,
                                       const float* obs, const void* actions, const float* old_log_probs, const float* adv,
                                       const float* returns, const double* adv_stats, const int32_t* idx, int64_t M,
                                       const dppo_hyper* hyper, float* losses, void* ws, int64_t ws_bytes, void* stream);

/* The whole update loop of a learn() for the DEFAULT 64-wide network (ppo.py:258-285; BASELINE north_star item 4) in ONE launch:
 * `steps` consecutive optimiser steps (all epochs x minibatches), each on `rows` samples idx[step*rows .. +rows) (idx < 0: padding
 * row), run by one thread-block cluster of 8 CTAs (rows <= 256) or 16 CTAs (more rows) with the parameters, the gradient partials
 * and the sharded Adam state resident in (distributed) shared memory -- gather, forward, loss, backward, gradient reduce-scatter,
 * global-norm clip, Adam and parameter all-gather never leave the SMs.  1 <= rows <= 2048 and steps >= 1; anything else is refused
 * before launch.  Padding rows (idx < 0) and hyper->loss_denominator (0: rows) behave as in dppo_mlp_grad_minibatch: a padding
 * row enters no loss term and no gradient, and the loss means divide by the denominator.  step_consts: DEVICE float [steps][2] =
 * {sqrt(1 - beta2^t), -lr / (1 - beta1^t)} of each step (torch/optim/adam.py:531-547, computed by the caller in double).  params /
 * exp_avg / exp_avg_sq are updated in place, grads receives the clipped gradient of the last step, grad_norm_out (optional) its
 * pre-clip norm, losses [steps][4] = policy, value, entropy, total per step.  Supported (dppo_small_update_supported): hidden == 64,
 * 1 <= act_dim <= 8, and 1 <= obs_dim <= 64 with the kernel's shared memory within 220 KB, which bounds obs_dim at 30 (8 actions)
 * to 36 (1 action). */
int dppo_small_update_supported(const dppo_mlp_desc* desc);
int dppo_small_update(dppo_ctx* ctx, const dppo_mlp_desc* desc, float* params, float* grads, float* exp_avg, float* exp_avg_sq,
                      const float* obs, const void* actions, const float* old_log_probs, const float* adv, const float* returns,
                      const double* adv_stats, const int32_t* idx, int64_t rows, int steps, const dppo_hyper* hyper,
                      const float* step_consts, float* losses, float* grad_norm_out, void* stream);

/* clip_grad_norm_ (ppo.py:284) + Adam (ppo.py:285) over flat buffers of n floats.
 * grad_norm_out (optional, device float) receives the pre-clip global norm. */
int dppo_clip_adam_step(dppo_ctx* ctx, float* params, float* grads, float* exp_avg, float* exp_avg_sq, int64_t n,
                        const dppo_hyper* hyper, float* grad_norm_out, void* ws, int64_t ws_bytes, void* stream);
int64_t dppo_clip_adam_workspace_bytes(int64_t n);
int64_t dppo_grad_sumsq_bytes(dppo_ctx* ctx, int64_t n);

/* ---- env-sharded data parallelism: the per-minibatch exchange step (SURVEY.md 8e) -------- */
/* One process per GPU.  Each rank writes the gradient of its shard of the global minibatch (and its 4 loss sums) into the
 * slot dppo_dp_slot() returns for that optimiser step; dppo_dp_allreduce_clip_adam then performs, in ONE kernel per rank,
 * the cross-GPU sum over NVLink peer memory (every rank reads every rank's slot and adds them in rank order, so all
 * replicas obtain the bit-identical gradient) together with the partial sums of the global gradient norm, followed by the
 * clip + Adam kernel of dppo_clip_adam_step.  Set-up: dppo_dp_create (allocates the exchange buffer -- the one device
 * allocation libdppo makes, CUDA IPC needs a base allocation), all-gather the dppo_dp_handle bytes of every rank
 * (torch.distributed), dppo_dp_connect.  Exchanges are numbered by their own monotonic sequence `seq` = 1, 2, 3, ... (never
 * the Adam step, which a restored checkpoint may move backwards); all ranks must call dppo_dp_allreduce_clip_adam with the
 * same sequence.  A kernel that waits ~10 s for a peer in vain gives up and raises the flag dppo_dp_status() reports. */
#define DPPO_MAX_RANKS 16
typedef struct dppo_dp dppo_dp;
int dppo_dp_create(dppo_ctx* ctx, int world, int rank, int64_t n_floats, dppo_dp** out);
int dppo_dp_handle_bytes(void);
int dppo_dp_handle(dppo_dp* dp, void* handle_out);
int dppo_dp_connect(dppo_ctx* ctx, dppo_dp* dp, const void* all_handles);
int dppo_dp_destroy(dppo_dp* dp);
int dppo_dp_status(dppo_dp* dp);                     /* 0 ok; 1 + q: timed out waiting for rank q (host-mapped flag, no sync) */
float* dppo_dp_slot(dppo_dp* dp, int64_t seq);       /* [n_floats gradient | 4 loss sums] of exchange number `seq` */
int dppo_dp_zero_slot(dppo_ctx* ctx, dppo_dp* dp, int64_t seq, void* stream);   /* a rank with no rows contributes zeros */
int64_t dppo_dp_workspace_bytes(int64_t n_floats);
/* hyper->step_consts (optional): the exchange kernel then reads the sequence number it publishes / waits for from the u64 at
 * step_consts + 2 floats (CUDA-graph replay); `seq` must still carry its parity (it selects the slot). */
int dppo_dp_allreduce_clip_adam(dppo_ctx* ctx, dppo_dp* dp, int64_t seq, float* params, float* grads_out, float* exp_avg,
                                float* exp_avg_sq, const dppo_hyper* hyper, float* losses_out, float* grad_norm_out,
                                void* ws, int64_t ws_bytes, void* stream);

/* Standalone loss forward+backward for custom network_cls modules (readme.md:89-111): the user
 * module runs under PyTorch autograd, this provides loss values and d(loss)/d(outputs).
 * Rows are already gathered (M rows).  losses[0..3] = policy, value, entropy, total.
 * 1 <= A <= DPPO_GEMM_HEADS_MAX_ACT; above 32 actions the lanes of a row's warp stride over the actions (size ws with
 * dppo_ppo_loss_workspace_bytes(M, A)). */
int dppo_ppo_loss_discrete(dppo_ctx* ctx, const float* logits, const float* values, const int32_t* actions,
                           const float* old_log_probs, const float* adv, const float* returns, int64_t M, int A,
                           const dppo_hyper* hyper, float* losses, float* dlogits, float* dvalues,
                           void* ws, int64_t ws_bytes, void* stream);
/* log_std_row_stride == 0: log_std is one shared [A] vector (actor_log_std, continuous_ppo.py:76) and
 * dlog_std receives its summed gradient [A]; otherwise log_std is per-row ([M, stride]) and dlog_std
 * receives per-row gradients [M, A] (state-dependent std of a custom network). */
int dppo_ppo_loss_gaussian(dppo_ctx* ctx, const float* mean, const float* log_std, int64_t log_std_row_stride, const float* values,
                           const float* actions, const float* old_log_probs, const float* adv, const float* returns,
                           int64_t M, int A, const dppo_hyper* hyper, float* losses, float* dmean, float* dlog_std,
                           float* dvalues, void* ws, int64_t ws_bytes, void* stream);
int64_t dppo_ppo_loss_workspace_bytes(int64_t M, int A);

/* ---- recurrent actor-critic (RecurrentPPO, diamond/recurrent_ppo.py) --------------------------------- */
/* Default RecurrentActorCriticNetwork (recurrent_ppo.py:94-125): base Linear(D,H)+Tanh -> GRU(H,Hg) -> actor head
 * Linear(Hg,H)+Tanh+Linear(H,A) and critic head Linear(Hg,H)+Tanh+Linear(H,1).
 * continuous = 1: RecurrentContinuousActorCriticNetwork (RecurrentContinuousPPO), the same trunk with a Gaussian policy -- the actor
 * head (actor_mean_head) outputs the action means and a state-independent log-std vector actor_log_std [A] is a parameter. */
typedef struct dppo_rnn_desc {
    int32_t obs_dim;      /* D */
    int32_t hidden;       /* H  = cfg.network_hidden_dim (<= 512) */
    int32_t gru_hidden;   /* Hg = cfg.gru_hidden_dim (<= 512; 129-512 run on thread-block-cluster scans) */
    int32_t act_dim;      /* A  = Discrete.n, or the action dimensions of a Box (<= DPPO_MAX_ACT) */
    int32_t continuous;   /* 0: categorical policy (logits), 1: Gaussian policy (means + actor_log_std) */
} dppo_rnn_desc;
/* Offsets (floats, multiples of 4) in the flat parameter / gradient / Adam buffers; the GRU tensors are nn.GRU's
 * weight_ih_l0 [3Hg,H], weight_hh_l0 [3Hg,Hg], bias_ih_l0, bias_hh_l0 (gate order r,z,n); w3/b3 = actor_head.0 | critic_head.0
 * (continuous: actor_mean_head.0 | critic_head.0), wa/ba = actor_head.2 (continuous: actor_mean_head.2).  log_std = actor_log_std [A],
 * placed after bc when continuous, else -1; every other offset is the same for both kinds. */
typedef struct dppo_rnn_layout {
    int64_t w1, b1;
    int64_t wih, whh, bih, bhh;
    int64_t w3, b3;
    int64_t wa, ba;
    int64_t wc, bc;
    int64_t log_std;
    int64_t total;
} dppo_rnn_layout;
int dppo_rnn_layout_compute(const dppo_rnn_desc* desc, dppo_rnn_layout* out);
int64_t dppo_rnn_workspace_bytes(const dppo_rnn_desc* desc, int T, int N, int64_t M, int training);
/* get_logits_values_and_hx / get_values (recurrent_ppo.py:127-149) over a [T,N] sequence: obs [T,N,D]; prev_dones uint8 [T,N]
 * (NULL: no resets) zeroes the hidden state of an environment BEFORE step t (recurrent_ppo.py:84); hx0 [N,Hg] (NULL: zeros).
 * heads bit0: logits [T*N,A] (continuous: the action means [T*N,A]; the log-std is params + layout.log_std); bit1: values [T*N];
 * hx_out (optional) [N,Hg] final hidden state. */
int dppo_rnn_forward(dppo_ctx* ctx, const dppo_rnn_desc* desc, const float* params, const float* obs,
                     const unsigned char* prev_dones, const float* hx0, int T, int N, int heads, float* logits,
                     float* values, float* hx_out, void* ws, int64_t ws_bytes, void* stream);
/* One optimiser step's gradient (recurrent_ppo.py:335-362): full-sequence forward with the current parameters, the rows
 * idx[0..M) of the flattened [T*N] outputs enter the PPO loss (idx NULL: all rows in order, M = T*N), back-propagation
 * through all T steps.  The entries of idx must be distinct and in [0, T*N): d(loss)/d(h_t) is scattered back to row idx[i],
 * so there are no padding rows (unlike dppo_mlp_grad_minibatch) and a repeated row would lose a contribution.
 * actions: int32 [T*N] (discrete) or f32 [T*N, A] (continuous: the Gaussian loss of continuous_ppo.py, with the gradient of
 * actor_log_std at layout.log_std); old_log_probs / adv / returns f32 [T*N]; flat gradient -> grads, (policy, value, entropy,
 * total) -> losses[0..3].
 * Both calls refuse, before launching anything, hidden > 512, gru_hidden > 512, act_dim > DPPO_MAX_ACT; dppo_rnn_grad_minibatch
 * also refuses the (hidden, act_dim) pairs whose per-warp head-gradient accumulators exceed the head kernel's 200 KB of shared
 * memory (9 (act_dim + 1) hidden floats: e.g. act_dim <= 10 at hidden 512, <= 32 up to hidden 172). */
int dppo_rnn_grad_minibatch(dppo_ctx* ctx, const dppo_rnn_desc* desc, const float* params, float* grads, const float* obs,
                            const unsigned char* prev_dones, const float* hx0, int T, int N, const void* actions,
                            const float* old_log_probs, const float* adv, const float* returns, const double* adv_stats,
                            const int32_t* idx, int64_t M, const dppo_hyper* hyper, float* losses, void* ws,
                            int64_t ws_bytes, void* stream);

/* ---- device-resident vectorised environments (SURVEY.md 8f-1) ------------------------------------ */
/* Replaces the host `envs.step(actions)` + `envs.reset(options={"reset_mask": dones})` + list append of a rollout step
 * (diamond/ppo.py:160-182): one kernel steps all environments and writes row t of the time-major rollout buffers.
 * kind 0: CartPole-v1, 1: Pendulum-v1, 4: Acrobot-v1, 5: MountainCar-v0, 6: MountainCarContinuous-v0 (Gymnasium
 * classic-control dynamics, float64 state; MountainCarContinuous keeps Gymnasium's float32 state), 2 / 3: synthetic discrete /
 * continuous (i.i.d. normal observations; the scale benchmark's shape stand-in).  Autoreset-DISABLED contract: next_obs[t]
 * is the true final observation; with auto_reset != 0 finished environments are then reset inside the same kernel and
 * cur_obs holds the post-reset observation (ppo.py:174-179), else the caller resets them with dppo_env_reset(mask).
 *
 * Normalisation (normalize != 0): every environment e keeps its own float64 statistics, as one Gymnasium NormalizeObservation /
 * NormalizeReward(gamma) wrapper per sub-environment would; the kernel that steps e updates them in the same thread (warp).
 *   Observations: mean[e, D] (start 0), var[e, D] (start 1), count[e] (start 1e-4).  Every observation the environment emits
 *   updates them before it is normalised: each step's true final observation (next_obs[t]) and each post-reset observation (the
 *   in-kernel reset and dppo_env_reset).  The update is RunningMeanStd.update on a batch of one float32 observation x widened to
 *   double: delta = x - mean; tot = count + 1; mean += delta * 1 / tot; var = (var * count + 0 + delta^2 * count * 1 / tot) / tot;
 *   count = tot.  The environment emits float32((x - mean) / sqrt(var + epsilon)), then clipped to [-clip_observation,
 *   clip_observation] in float32.  Every operation is an explicitly rounded double intrinsic, so the statistics are bit-identical
 *   to a float64 NumPy restatement.  next_obs[t] and cur_obs of an environment that did not finish are the same float32 values.
 *   Rewards: per step acc = acc * gamma * (1 - terminated) + r (r: the float64 reward of the dynamics); a scalar RunningMeanStd
 *   (mean 0, var 1, count 1e-4) is updated with acc; rewards[t] receives r / sqrt(var + epsilon), clipped to [-clip_reward,
 *   clip_reward] in double, then cast to float32.  As in Gymnasium's NormalizeReward the accumulator is cut by termination
 *   only: not by truncation, and not by a reset.  Episode returns (ep_return, done_return) stay raw.
 *   *update == 0 (read by the kernel at run time, so replayed CUDA graphs follow it) freezes both sets of statistics
 *   (Gymnasium's update_running_mean); the reward accumulator keeps running.
 * Zero-initialised fields (normalize = 0) leave the environments exactly as without them. */
#define DPPO_ENV_NORMALIZE_OBS 1
#define DPPO_ENV_NORMALIZE_REWARD 2
typedef struct dppo_env_desc {
    int32_t kind;
    int32_t num_envs;
    int32_t obs_dim;        /* 4 (CartPole), 3 (Pendulum), 6 (Acrobot), 2 (MountainCar, MountainCarContinuous), any (synthetic) */
    int32_t act_dim;        /* Discrete.n, or action dims when continuous: 3 (Acrobot, MountainCar), 1 (MountainCarContinuous) */
    uint64_t seed;          /* reset / synthetic draws: Philox4x32-10 keyed by (seed, env_offset + env, episode or step) */
    int64_t env_offset;     /* global id of env 0 (env-sharded data parallelism) */
    float p_term, p_trunc;  /* synthetic kinds only */
    int32_t normalize;      /* DPPO_ENV_NORMALIZE_OBS | DPPO_ENV_NORMALIZE_REWARD; 0: off */
    int32_t pad0;
    double gamma;           /* reward discount of the return accumulator, in [0, 1] */
    double epsilon;         /* > 0 when normalising */
    double clip_observation;/* >= 0; 0: no clip */
    double clip_reward;     /* >= 0; 0: no clip */
} dppo_env_desc;
typedef struct dppo_env_state {  /* caller-allocated device buffers */
    double* state;          /* [N, 4] */
    int32_t* steps;         /* [N] steps taken in the current episode */
    int64_t* episode;       /* [N] episodes started */
    double* ep_return;      /* [N] running return of the current episode */
    float* cur_obs;         /* [N, D] observation the next sampling step reads */
    double* obs_mean;       /* [N, D] observation normalisation (may be NULL without DPPO_ENV_NORMALIZE_OBS) */
    double* obs_var;        /* [N, D] */
    double* obs_count;      /* [N] */
    double* ret_stats;      /* [N, 4] accumulated discounted return, its running mean, variance, count (DPPO_ENV_NORMALIZE_REWARD) */
    const int32_t* update;  /* device int32 [1]: nonzero updates the statistics (required when normalising) */
} dppo_env_state;
/* mask: uint8 [N] (NULL: reset every environment).  Refused before any launch: normalisation with a NULL statistics buffer or
 * update flag, gamma outside [0, 1], epsilon <= 0, a negative clip, unknown normalize bits.  With normalisation on, the synthetic
 * kinds keep the raw first observation feature (which their reward reads) in state[e, 0]. */
int dppo_env_reset(dppo_ctx* ctx, const dppo_env_desc* desc, const dppo_env_state* state, const unsigned char* mask, void* stream);
/* actions: int64 [N] (what dppo_sample_categorical writes) or f32 [N, A].  obs / next_obs / buf_actions / rewards /
 * terminations / truncations are the BASES of the [T, N, ...] buffers (obs and buf_actions may be NULL); row t is written with
 * the casts of ppo.py:229-232.  done_return (optional, f32 [N]) receives the return of every episode that ended at this step.
 * raw_rewards (optional) is the base of a [T, N] f32 buffer whose row t receives the rewards before normalisation (the same
 * values as rewards[t] when the descriptor does not normalise rewards). */
int dppo_env_step(dppo_ctx* ctx, const dppo_env_desc* desc, const dppo_env_state* state, const void* actions, int t, int auto_reset,
                  float* obs, float* next_obs, void* buf_actions, float* rewards, float* terminations, float* truncations,
                  float* done_return, float* raw_rewards, void* stream);

/* ---- device-side episode statistics (SURVEY.md 8 f4) ------------------------------------------- */
/* Replaces the per-step host Ticker.tick(rewards, dones) (diamond/utils.py:99-123, call site ppo.py:181-182) for rollouts that
 * live on the device: one pass over the [T, N] rewards / terminations / truncations of a rollout updates the per-environment
 * running return (fp64) and length in ep_return / ep_len (carried across rollouts; caller zeroes them when the environments
 * are reset), writes the number of episodes that finished to *finished and the last min(window, *finished) of them, in the
 * Ticker's order (step by step, environments in index order), to out_returns / out_lengths[0 .. *out_n). */
int64_t dppo_episode_stats_workspace_bytes(int T, int N);
int dppo_episode_stats(dppo_ctx* ctx, const float* rewards, const float* terminations, const float* truncations, int T, int N,
                       double* ep_return, int32_t* ep_len, int window, double* out_returns, int32_t* out_lengths, int32_t* out_n,
                       unsigned long long* finished, void* ws, int64_t ws_bytes, void* stream);
/* Episode bookkeeping of an evaluation, one launch per chunk of T steps of N environments ([T, N] rewards / terminations /
 * truncations).  The arithmetic of dppo_episode_stats: f32 rewards summed in fp64, length + 1 per step, done = termination |
 * truncation; the running return and length in ep_return / ep_len carry across chunks (caller zeroes them with the reset).
 * Environment e records only its first quota[e] finished episodes: the k-th (k counted by recorded[e], caller zeroes it) goes to
 * out_returns / out_lengths[slot_offset[e] + k].  When recorded[e] reaches quota[e], *remaining is decremented once (the caller
 * sets it to the number of environments with quota > 0, so it reads 0 when every quota is met).  Later episodes of e are ignored,
 * so an environment past its quota may keep stepping and every launch keeps its shape. */
int dppo_eval_episodes(dppo_ctx* ctx, const float* rewards, const float* terminations, const float* truncations, int T, int N,
                       const int32_t* quota, const int64_t* slot_offset, double* ep_return, int32_t* ep_len, int32_t* recorded,
                       double* out_returns, int32_t* out_lengths, int32_t* remaining, void* stream);

/* ---- tensor-core building blocks of the fused update (unit tests, A/B measurements) ---------- */
/* C[M,N] = epi(A[M,K] * op(W)) as an error-compensated 3xTF32 tcgen05 GEMM (fp32-accurate, SURVEY.md 0.6) on CTA pairs
 * (tcgen05 cta_group::2, 256-row tiles shared by the two SMs of a TPC; persistent, TMA-fed, warp-specialised).
 * transpose 0: W is [N,K] row-major (nn.Linear forward, ppo.py:91-96); 1: W is [K,N] (its backward, ppo.py:283).
 * epi 1: C = tanh(A W^T + bias); epi 2: C = (A W) * (1 - Hact^2) with Hact [M,N], and, if colsum != NULL,
 * partial column sums of C in colsum [dppo_tc_colsum_parts(ctx, M, N), N]: the first fifth of the rows are the per-CTA
 * partials, the rest per-quadrant working rows; sum only rows [0, parts/5) (bias-gradient partials).
 * ws (dppo_tc_linear_workspace_bytes) holds the split weight images; prepared != 0 re-uses the images an earlier call
 * with the same W left in ws (kernel-only timing). */
int dppo_tc_linear_f32(dppo_ctx* ctx, int epi, const float* A, int64_t M, int K, const float* W, int N, int transpose,
                       const float* bias, const float* Hact, float* C, float* colsum, void* ws, int64_t ws_bytes,
                       int prepared, void* stream);
int64_t dppo_tc_linear_workspace_bytes(int N, int K);
int dppo_tc_colsum_parts(dppo_ctx* ctx, int64_t M, int N);
/* dW[N1,N2] = sum_m D[m,N1] * H[m,N2]  (weight gradient of a Linear layer, ppo.py:283): split over row
 * ranges on tcgen05, partials summed in a fixed order (bit-reproducible). */
int dppo_tc_wgrad_f32(dppo_ctx* ctx, const float* D, const float* H, int64_t M, int N1, int N2, float* dW, void* ws,
                      int64_t ws_bytes, void* stream);
int64_t dppo_tc_wgrad_workspace_bytes(dppo_ctx* ctx, int64_t M, int N1, int N2);

/* ---- measurement helper ---------------------------------------------------------------- */
/* Runs a register-resident FFMA loop on every SM (iters FMAs per thread, 16 independent chains;
 * sink: >= 65 floats of finite values);
 * bench.py times it with CUDA events to obtain the FP32 FMA-pipe peak of this very GPU. */
int dppo_fma_peak_kernel(dppo_ctx* ctx, float* sink, int64_t iters, int* blocks_out, int* threads_out, void* stream);

/* Issue rate of tcgen05.mma with shared-memory operands: every CTA (pair != 0: every CTA pair, cta_group::2, M = 256;
 * else M = 128) issues iters back-to-back MMAs of N = n, K = 32 bytes (tf32, or bf16 if bf16 != 0) and writes the SM
 * cycles they took to out[blockIdx] (int64 [*grid_out]; only the leader of a pair writes).  bench.py derives the
 * tensor-pipe peak the 3xTF32 GEMMs are measured against from it. */
int dppo_tc_mma_probe(dppo_ctx* ctx, int pair, int bf16, int n, int iters, long long* out, int* grid_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DPPO_H */
