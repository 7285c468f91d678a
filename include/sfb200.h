/*
 * sfb200.h -- C ABI of libsfb200.so: the B200 (sm_100a) implementation of Sample Factory's APPO hot path
 *             (rollout sampler -> PPO / V-trace learner).
 *
 * The reference (alex-petrenko/sample-factory) has no FFI for this path: it is Python calling PyTorch ATen.  Each
 * entry point below therefore cites the reference Python site (paths relative to sample_factory/) whose arithmetic
 * it replaces; INTEGRATION.md shows the ctypes binding a maintainer adds at that site.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless the name ends in _host
 *   - all tensors are caller-owned ("borrowed"), dense in their last dimension, fp32 unless stated;
 *     bool tensors are 1 byte per element (torch.bool); ld* / *_stride arguments are element strides
 *   - `stream` is a cudaStream_t (CUstream) passed as void*; every call only ENQUEUES work on that stream,
 *     never allocates device memory and never synchronises the host
 *   - return value: 0 = ok, otherwise an error code; sfb200_last_error() returns the message (thread-local)
 *   - layouts are the reference trajectory layout (algo/utils/shared_buffers.py:79-117): [num_traj, T(+1), ...]
 */
#ifndef SFB200_H
#define SFB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default) /* everything declared here is exported; the rest of the library is hidden */
#endif

#define SFB200_ABI_VERSION 2

/* activation codes (model/model_utils.py:27-35) */
#define SFB200_ACT_NONE 0
#define SFB200_ACT_ELU 1
#define SFB200_ACT_RELU 2
#define SFB200_ACT_TANH 3

/* GEMM engine selection for sfb200_linear_* */
#define SFB200_GEMM_SIMT_FP32 0   /* CUDA-core fp32 FFMA tiles */
#define SFB200_GEMM_TC_3XTF32 1   /* tcgen05 kind::tf32, error-compensated 3-pass split, fp32 accumulate in TMEM */
#define SFB200_GEMM_TC_TF32 2     /* tcgen05 kind::tf32 single pass (fast, NOT parity grade) */

/* ---------------------------------------------------------------- library ---- */
int sfb200_abi_version(void);
const char* sfb200_last_error(void);
/* binds the calling thread to `device` (cudaSetDevice); call once per thread before anything else */
int sfb200_set_device(int device);
/* number of SMs of the bound device (grid sizing) */
int sfb200_sm_count(void);
/* 1 if the tcgen05/TMA GEMM engine is usable in this process (driver entry points resolved), else 0 */
int sfb200_tc_available(void);
/* Pre-split weights for the 3xTF32 engine.  register: from now on every tcgen05-3xTF32 GEMM whose WEIGHT operand lies
 * inside [base, base+n) reads the operand's low tf32 half from `lo` (same offsets) instead of deriving it in shared
 * memory for every output tile, and sfb200_clip_adam_step on a registered buffer keeps `lo` current.  Any other write
 * to the weights (checkpoint load, weight copy) must be followed by sfb200_refresh_tf32_lo(base).  With the
 * environment variable SFB200_CHECK_LO=1 every use verifies the pair on the device and traps on a stale `lo`. */
int sfb200_register_tf32_lo(const float* base, float* lo, int64_t n);
int sfb200_unregister_tf32_lo(const float* base);
int sfb200_refresh_tf32_lo(const float* base, void* stream);
/* The fp16-split form of the same 3-pass engine (fp32 accuracy class of 3xTF32 -- 22 significand bits per operand --
 * on the kind::f16 tensor-core path: twice the MMA rate, 2/3 of the operand bytes).  A 3xTF32 GEMM takes it when
 *   (1) its WEIGHT operand lies inside a buffer with registered fp16 twins: twins = [hi16[n] | lo16[n]],
 *       hi = fp16(w * 2^8), lo = fp16((w * 2^8 - hi) * 2^11) (|w| < 255); for dX = dz . W, where the weight matrix is read
 *       transposed, a per-matrix transposed copy [hiT[K][N] | loT[K][N]] registered with ..._f16_transposed; and
 *   (2) its ACTIVATION operand lies inside a buffer with a registered bound: a device float >= max|x| (fp16 has five
 *       exponent bits: the kernel scales the operand by the power of two that places the bound in [2^14, 2^15)).
 * sfb200_clip_adam_step keeps registered twins current; the transposed copies and the twins after any other write to
 * the weights are refreshed by the refresh_* calls.  sfb200_linear_out_bound derives the bound of a layer's output from
 * the bound of its input: max_n (in_bound * sum_k |W[n][k]| + |b[n]|) (tanh: at most 1); out_bound_dev is FOUR 32-bit words
 * [bound, scratch, counter, -], the middle two zero on entry and on return.  No counterpart in the reference (its
 * nn.Linear runs cuBLAS fp32 / CPU). */
int sfb200_register_f16_twins(const float* base, void* twins, int64_t n);
int sfb200_unregister_f16_twins(const float* base);
int sfb200_refresh_f16_twins(const float* base, void* stream);
int sfb200_register_f16_transposed(const float* W, int N, int K, void* twinsT);
int sfb200_unregister_f16_transposed(const float* W);
int sfb200_refresh_f16_transposed(const float* W, void* stream);
int sfb200_register_operand_bound(const void* base, int64_t bytes, const float* bound_dev);
int sfb200_unregister_operand_bound(const void* base);
int sfb200_linear_out_bound(const float* W, const float* b, int N, int K, const float* in_bound_dev, float* out_bound_dev,
                            int act, void* stream);
/* bound of the gradient sfb200_heads_backward writes for the last hidden layer (the activation operand of dX):
 * max_m (|dvalues[m]| + sum_a |dlogits[m][a]|) * max(|Wv|_inf, |Wa|_inf); act' <= 1 for every supported activation.
 * out_bound_dev: THREE 32-bit words [bound, scratch, counter], the last two zero on entry and on return. */
int sfb200_heads_dz_bound(const float* dlogits, const float* dvalues, int64_t rows, int A, const float* Wv, const float* Wa,
                          int H, float* out_bound_dev, void* stream);
/* total number of CUDA kernels this library has launched (or recorded into a stream capture) in this process */
uint64_t sfb200_launch_count(void);

/* ------------------------------------------------------------- normalizers ---- */
/* utils/normalize.py:51-70 + algo/utils/running_mean_std.py:96-110 (normalize branch), out of place:
 *   y = clamp(((x - sub_mean) * inv_scale - mean) * (1 / sqrt(var + eps)), -clip, clip)
 * mean/var are the float64 running buffers (running_mean_std.py:45-46); if mean == NULL only sub/scale apply.
 * x rows have element stride ldx, y rows ldy. */
int sfb200_normalize_obs(const float* x, int64_t ldx, float* y, int64_t ldy, int64_t rows, int dim,
                         const double* mean, const double* var, float sub_mean, float inv_scale, float eps,
                         float clip, void* stream);

/* running_mean_std.py:72-77: batch mean and UNBIASED variance over dim 0 of x[rows, dim] (fp64 accumulation,
 * results rounded to fp32 like the reference's fp32 tensors).  workspace: >= sfb200_moments_workspace_bytes(dim). */
int64_t sfb200_moments_workspace_bytes(int dim);
int sfb200_batch_moments(const float* x, int64_t ldx, int64_t rows, int dim, float* batch_mean, float* batch_var,
                         void* workspace, void* stream);

/* running_mean_std.py:49-62: in-place Welford merge of (batch_mean, batch_var, batch_count) into the float64
 * running buffers mean/var[dim] and count[1]. */
int sfb200_rms_merge(double* mean, double* var, double* count, const float* batch_mean, const float* batch_var,
                     double batch_count, int dim, void* stream);

/* running_mean_std.py:96-110 with input_shape (1,), in place on a flat vector (the returns normalizer,
 * learner.py:1018-1019 and :969-975): denormalize=0: x = clamp((x-mean)*(1/sigma), +-clip);
 * denormalize=1: x = clamp(x, +-clip)*sigma + mean.  mean/var: float64 [1]. */
int sfb200_rms_apply_scalar(float* x, int64_t n, const double* mean, const double* var, float eps, float clip,
                            int denormalize, void* stream);

/* ------------------------------------------------------------- model forward ---- */
/* model/model_utils.py:46-56 (create_mlp layer): y[M,N] = act(x[M,K] . W[N,K]^T + b[N]);  W in nn.Linear layout.
 * engine: SFB200_GEMM_*.  x row stride ldx (lets the learner feed obs[:, T] rows in place), y row stride ldy. */
int sfb200_linear_act_forward(const float* x, int64_t ldx, const float* W, const float* b, float* y, int64_t ldy,
                              int64_t M, int N, int K, int act, int engine, void* stream);

/* Sampling mode of the calling host thread, picked up by every heads entry below that samples actions (the
 * `action_mask=` argument of ActorCritic.forward, model/actor_critic.py:189-195, filled from the observation dict's
 * "action_mask" entry, algo/sampling/inference_worker.py:324-331; and enjoy.py:165-171 `eval_deterministic`).
 *   action_mask        uint8 [rows, mask_row_stride] on the device or NULL; 0 = action not allowed.  Plain Discrete
 *                      spaces only: p = masked_softmax(logits, mask), log_prob = masked_log_softmax(logits, mask)_a,
 *                      rows that allow nothing sample from a uniform 1e-6 vector (action_distributions.py:84-95,
 *                      135-143); the stored action_logits stay the raw logits.  The pointer is read at launch time
 *                      (a captured CUDA graph keeps reading the same buffer).
 *   deterministic      != 0: the action is argmax(p) (first index on ties) / the Gaussian mean, no noise is consumed.
 * Stays in force until changed; (NULL, 0, 0) is the default. */
int sfb200_set_sampling_mode(const uint8_t* action_mask, int64_t mask_row_stride, int deterministic);

/* critic_linear + distribution_linear + CategoricalActionDistribution (model/actor_critic.py:171-186,
 * model/action_parameterization.py:33-39, algo/utils/action_distributions.py:110-148):
 *   values[i]  = h[i] . Wv + bv                                   (written at values[i * values_stride])
 *   logits[i]  = h[i] . Wa^T + ba                                 (logits + i * logits_stride, A floats)
 * and, if actions_f32 != NULL (sampling mode, inference_worker.py:313-341):
 *   a = argmax_j softmax(logits)_j / q_j   (== torch.multinomial(p, 1, True); q = noise row if noise != NULL,
 *                                           else Exp(1) from Philox4x32-10(seed, subsequence=i*A+j,
 *                                           offset = philox_offset + (philox_offset_dev ? *philox_offset_dev : 0));
 *                                           the device-side term keeps a captured CUDA graph drawing fresh noise)
 *   actions_f32[i*actions_stride] = (float)a ; env_actions_i32[i] = a ; log_prob[i*log_prob_stride] = log_softmax_a
 *   policy_version_out[i*pv_stride] = *policy_version_scalar (inference_worker.py:332)
 * Any output pointer except values may be NULL.  A <= 32. */
int sfb200_heads_forward(const float* h, int64_t ldh, int64_t rows, int H, int A, const float* Wv, const float* bv,
                         const float* Wa, const float* ba, float* values, int64_t values_stride, float* logits,
                         int64_t logits_stride, const float* noise, uint64_t philox_seed, uint64_t philox_offset,
                         const int64_t* philox_offset_dev, float* actions_f32, int64_t actions_stride, int32_t* env_actions_i32, float* log_prob,
                         int64_t log_prob_stride, const float* policy_version_scalar, float* policy_version_out,
                         int64_t pv_stride, void* stream);

/* sfb200_heads_forward / sfb200_heads_from_partials for a Tuple of Discretes: every head softmaxes and samples over its own
 * logit segment (noise rows hold the heads' Exp(1) draws side by side, A floats); actions_f32[i*actions_stride + k] and
 * env_actions_i32[i*K + k] receive head k's index, log_prob the sum of the heads' log-probs. */
int sfb200_heads_forward_tuple(const float* h, int64_t ldh, int64_t rows, int H, int A, int num_heads,
                               const int32_t* head_sizes_host, const float* Wv, const float* bv, const float* Wa,
                               const float* ba, float* values, int64_t values_stride, float* logits,
                               int64_t logits_stride, const float* noise, uint64_t philox_seed, uint64_t philox_offset,
                               const int64_t* philox_offset_dev, float* actions_f32, int64_t actions_stride,
                               int32_t* env_actions_i32, float* log_prob, int64_t log_prob_stride,
                               const float* policy_version_scalar, float* policy_version_out, int64_t pv_stride,
                               void* stream);
int sfb200_heads_from_partials_tuple(const float* head_partials, int P, int64_t rows, int A, int num_heads,
                                     const int32_t* head_sizes_host, const float* bv, const float* ba, float* values,
                                     int64_t values_stride, float* logits, int64_t logits_stride, const float* noise,
                                     uint64_t philox_seed, uint64_t philox_offset, const int64_t* philox_offset_dev,
                                     float* actions_f32, int64_t actions_stride, int32_t* env_actions_i32,
                                     float* log_prob, int64_t log_prob_stride, const float* policy_version_scalar,
                                     float* policy_version_out, int64_t pv_stride, void* stream);

/* Continuous (Box) action spaces: critic_linear + distribution_linear + ContinuousActionDistribution
 * (algo/utils/action_distributions.py:290-323 = Independent(Normal(means, clamp(exp(log_std), 1e-4, 1e4)), 1);
 * model/action_parameterization.py:33-39 when adaptive_stddev -- distribution_linear has 2*act_dim rows [means|log_std]
 * -- and :42-78 when not -- act_dim rows, means = tanh(z/tanh_scale)*tanh_scale if tanh_scale > 0, log_std = the
 * learned vector).  params[i] (2*act_dim floats at params + i*params_stride) receives [means | log_std], the layout of
 * the reference's `action_logits`.  Sampling mode (actions_f32 != NULL): a = eps*std + mean (product and sum rounded
 * separately = Normal.sample()), eps = noise[i*act_dim + j] or N(0,1) from Philox4x32-10(seed, subsequence i*act_dim+j,
 * offset); actions_f32[i*actions_stride + j] = env_actions_f32[i*act_dim + j] = a_j; log_prob = sum_j Normal.log_prob.
 * The _from_partials variant finishes sfb200_linear_act_heads_forward exactly like sfb200_heads_from_partials. */
int sfb200_heads_forward_continuous(const float* h, int64_t ldh, int64_t rows, int H, int act_dim, int adaptive_stddev,
                                    const float* Wv, const float* bv, const float* Wa, const float* ba,
                                    const float* learned_log_std, float tanh_scale, float* values,
                                    int64_t values_stride, float* params, int64_t params_stride, const float* noise,
                                    uint64_t philox_seed, uint64_t philox_offset, const int64_t* philox_offset_dev,
                                    float* actions_f32, int64_t actions_stride, float* env_actions_f32, float* log_prob,
                                    int64_t log_prob_stride, const float* policy_version_scalar,
                                    float* policy_version_out, int64_t pv_stride, void* stream);
int sfb200_heads_from_partials_continuous(const float* head_partials, int P, int64_t rows, int act_dim,
                                          int adaptive_stddev, const float* bv, const float* ba,
                                          const float* learned_log_std, float tanh_scale, float* values,
                                          int64_t values_stride, float* params, int64_t params_stride,
                                          const float* noise, uint64_t philox_seed, uint64_t philox_offset,
                                          const int64_t* philox_offset_dev, float* actions_f32, int64_t actions_stride,
                                          float* env_actions_f32, float* log_prob, int64_t log_prob_stride,
                                          const float* policy_version_scalar, float* policy_version_out,
                                          int64_t pv_stride, void* stream);

/* The last hidden layer and the heads in ONE pass (same reference sites as sfb200_linear_act_forward +
 * sfb200_heads_forward): the tcgen05 epilogue forms y = act(x W^T + b) in registers and contracts it at once with
 * [Wv ; Wa], so y is not re-read by a heads kernel -- and not written at all when y == NULL (the sampler never needs
 * it).  Two calls:
 *   P = sfb200_linear_heads_partials(N, A, engine)          0 -> shape/engine not covered: use the two separate calls
 *   sfb200_linear_act_heads_forward(..., head_partials)      head_partials: P * M * 12 floats of scratch
 *   sfb200_heads_from_partials(head_partials, P, M, A, ...)  same outputs / sampling semantics as sfb200_heads_forward
 * The partial sums are combined in a fixed order (deterministic). */
int sfb200_linear_heads_partials(int N, int A, int engine);
int sfb200_linear_act_heads_forward(const float* x, int64_t ldx, const float* W, const float* b, float* y, int64_t ldy,
                                    int64_t M, int N, int K, int act, int engine, const float* Wv, const float* Wa,
                                    int A, float* head_partials, void* stream);
/* Everything of a sampler step that follows the policy GEMMs, for the synthetic tape env of BASELINE config 2
 * (sample_factory_b200.envs.TapeVecEnv), in ONE launch: sfb200_heads_from_partials (finish heads, sample, log-prob, version
 * stamp into traj[:, t]) -> the env step (sfb200_tape_env_step rules; the env's own obs / rew / terminated / truncated
 * buffers are kept current) -> sfb200_sampler_post_step for step t -> generate_policy_request + normalisation for step t+1
 * (sfb200_sampler_pre_step; x_norm == NULL at the last step of a rollout).  One warp walks one env through all stages.
 * sampler_step is the Philox offset counter (read, then advanced by one), env_step_counter the env's {step, ticket}. */
int sfb200_sampler_tail_tape_step(const float* head_partials, int P, int64_t n_envs, int A, const float* bv, const float* ba,
                                  float* values_t, int64_t values_stride, float* logits_t, int64_t logits_stride,
                                  const float* noise, uint64_t philox_seed, int64_t* sampler_step, float* actions_t,
                                  int64_t actions_stride, int32_t* env_actions, float* log_prob_t, int64_t log_prob_stride,
                                  const float* policy_version_scalar, float* policy_version_t, int64_t pv_stride,
                                  const float* tape, int64_t tape_len, int dim, int64_t env_index_offset, int term_period,
                                  int trunc_period, int64_t* env_step_counter, float* env_obs, float* env_rew,
                                  uint8_t* env_terminated, uint8_t* env_truncated, float reward_scale, float reward_clip,
                                  int32_t policy_id, float* traj_rewards_t, uint8_t* traj_dones_t, uint8_t* traj_time_outs_t,
                                  int32_t* traj_policy_id_t, int64_t traj_stride, float* ep_return, int32_t* ep_len,
                                  float* ep_min_raw, float* ep_max_raw, int32_t len_increment, double* stats,
                                  float* fin_return_t, int32_t* fin_len_t, float* traj_obs_next, int64_t traj_obs_stride,
                                  const float* rnn, int rnn_dim, float* traj_rnn_next, int64_t traj_rnn_stride, float* x_norm,
                                  const double* mean, const double* var, float sub_mean, float inv_scale, float eps,
                                  float clip, void* stream);
/* A WHOLE ROLLOUT of a two-layer MLP policy over the synthetic tape env as one persistent kernel (csrc/rollout_fused.cu):
 * T x { layer 1, layer 2 + head partials, sfb200_sampler_tail_tape_step } with thread-block clusters of H2/128 CTAs owning a
 * 128-env row block for all T steps (cluster barriers only; no kernel boundary inside the rollout).  Replaces, per rollout,
 * T x (sfb200_linear_act_forward + sfb200_linear_act_heads_forward + sfb200_sampler_tail_tape_step); the caller runs
 * sfb200_sampler_pre_step for step 0 first (x_norm holds the normalised step-0 observations).  Pointers with suffix _0 are
 * the trajectory slots of step 0 ([:, 0]); step t is at + t elements (x A for logits, x dim for traj_obs / rnn rows).
 *   P = sfb200_rollout_mlp2_partials(...)   0 -> not covered (3xTF32 engine, K1 in {32,64,96,128}, H1 == H2 in {128,256,512},
 *       A <= 8, both weight matrices inside a registered tf32-lo buffer); head_partials: P * n_envs * 12 floats,
 *       h1_scratch: n_envs * H1 floats. */
int sfb200_rollout_mlp2_partials(const float* W1, const float* W2, int K1, int H1, int H2, int A, int engine);
/* debug aid: device buffer of T x 16 uint64 that the following rollouts fill with %globaltimer stamps of one CTA's phases
 * (tools/rollout_trace.py); NULL switches it off */
int sfb200_rollout_set_trace(void* trace_dev);
int sfb200_rollout_mlp2_tape(int64_t n_envs, int T, int K1, const float* W1, const float* b1, int H1, const float* W2,
                             const float* b2, int H2, int act, int engine, const float* Wv, const float* bv, const float* Wa,
                             const float* ba, int A, float* h1_scratch, float* head_partials, float* x_norm,
                             float* values_0, int64_t values_stride, float* logits_0, int64_t logits_stride,
                             const float* noise, uint64_t philox_seed, int64_t* sampler_step, float* actions_0,
                             int64_t actions_stride, int32_t* env_actions, float* log_prob_0, int64_t log_prob_stride,
                             const float* policy_version_scalar, float* policy_version_0, int64_t pv_stride,
                             const float* tape, int64_t tape_len, int64_t env_index_offset, int term_period, int trunc_period,
                             int64_t* env_step_counter, float* env_obs, float* env_rew, uint8_t* env_terminated,
                             uint8_t* env_truncated, float reward_scale, float reward_clip, int32_t policy_id,
                             float* traj_rewards_0, uint8_t* traj_dones_0, uint8_t* traj_time_outs_0, int32_t* traj_policy_id_0,
                             int64_t traj_stride, float* ep_return, int32_t* ep_len, float* ep_min_raw, float* ep_max_raw,
                             int32_t len_increment, double* stats, float* fin_return_0, int32_t* fin_len_0, float* traj_obs_0,
                             int64_t traj_obs_stride, const float* rnn, int rnn_dim, float* traj_rnn_0, int64_t traj_rnn_stride,
                             const double* mean, const double* var, float sub_mean, float inv_scale, float eps, float clip,
                             void* stream);
int sfb200_heads_from_partials(const float* head_partials, int P, int64_t rows, int A, const float* bv, const float* ba,
                               float* values, int64_t values_stride, float* logits, int64_t logits_stride,
                               const float* noise, uint64_t philox_seed, uint64_t philox_offset,
                               const int64_t* philox_offset_dev, float* actions_f32, int64_t actions_stride,
                               int32_t* env_actions_i32, float* log_prob, int64_t log_prob_stride,
                               const float* policy_version_scalar, float* policy_version_out, int64_t pv_stride,
                               void* stream);

/* ------------------------------------------------------------- sampler steps ---- */
/* BatchedVectorEnvRunner.generate_policy_request (algo/sampling/batched_sampling.py:374-388) fused with the
 * inference-side normalisation (inference_worker.py:326):  traj_obs[:, t] = obs ; traj_rnn[:, t] = rnn ;
 * x_norm = normalize(obs).  traj_obs_t / traj_rnn_t point at element [0, t]; row strides in elements. */
int sfb200_sampler_pre_step(const float* obs, int64_t n_envs, int dim, float* traj_obs_t, int64_t traj_obs_stride,
                            const float* rnn, int rnn_dim, float* traj_rnn_t, int64_t traj_rnn_stride,
                            float* x_norm, const double* mean, const double* var, float sub_mean, float inv_scale,
                            float eps, float clip, void* stream);

/* advance_rollouts part 2 (batched_sampling.py:319-357, _process_rewards :208-213, _process_env_step :215-287):
 * dones = terminated | truncated ; r = clamp(rew*reward_scale, +-reward_clip) ; writes rewards/dones/time_outs/
 * policy_id at [.., t] (pointers at element [0,t], element stride traj_stride) ; device-side episode accounting:
 * per-env ep_return[n], ep_len[n] (int32), ep_min_raw[n], ep_max_raw[n] and, for episodes finishing this step, the
 * accumulators stats[0..4] = {count, sum_return, sum_len, sum_min_raw_reward, sum_max_raw_reward} (doubles) -- the
 * reference's per-episode report (:228-234) aggregated on device, no host sync.  step_counter (optional, device
 * int64) is incremented by one: the sampler's policy-step count, used as the Philox offset of the next step.
 * fin_return_t / fin_len_t (optional, element [0,t] of [N,T] buffers, same element stride): the per-episode report
 * itself -- return and length of the episode that finished at this step, NaN / -1 where none did (what the
 * reference sends as episodic stats messages; consumed by EvalSamplingAPI.eval_stats). */
int sfb200_sampler_post_step(const float* rew, const uint8_t* terminated, const uint8_t* truncated, int64_t n_envs,
                             float reward_scale, float reward_clip, int32_t policy_id, float* traj_rewards_t,
                             uint8_t* traj_dones_t, uint8_t* traj_time_outs_t, int32_t* traj_policy_id_t,
                             int64_t traj_stride, float* ep_return, int32_t* ep_len, float* ep_min_raw,
                             float* ep_max_raw, int32_t len_increment, double* stats, int64_t* step_counter,
                             float* fin_return_t, int32_t* fin_len_t, void* stream);

/* sfb200_sampler_post_step for step t and sfb200_sampler_pre_step for step t+1 in ONE launch (both only consume the
 * env's outputs of step t).  traj_obs_next / traj_rnn_next point at element [0, t+1]; x_norm may be NULL (last step of
 * the rollout: the observation is only recorded, batched_sampling.py:289-296).  With an RNN core, `rnn` must already
 * hold the done-masked state for t+1. */
int sfb200_sampler_post_pre_step(const float* rew, const uint8_t* terminated, const uint8_t* truncated, int64_t n_envs,
                                 float reward_scale, float reward_clip, int32_t policy_id, float* traj_rewards_t,
                                 uint8_t* traj_dones_t, uint8_t* traj_time_outs_t, int32_t* traj_policy_id_t,
                                 int64_t traj_stride, float* ep_return, int32_t* ep_len, float* ep_min_raw,
                                 float* ep_max_raw, int32_t len_increment, double* stats, int64_t* step_counter,
                                 float* fin_return_t, int32_t* fin_len_t,
                                 const float* obs, int dim, float* traj_obs_next, int64_t traj_obs_stride,
                                 const float* rnn, int rnn_dim, float* traj_rnn_next, int64_t traj_rnn_stride,
                                 float* x_norm, const double* mean, const double* var, float sub_mean, float inv_scale,
                                 float eps, float clip, void* stream);

/* Shuffled minibatches (learner.py:498-526: `buffer[indices]` with indices = a permutation of recurrence-length chunks):
 * dst[r, :] = src[idx[r], :] for `rows` rows of `row_bytes` bytes each (any element type; dense rows). */
/* strided row copy of any element type (bool masks, int32 ids): rows of row_bytes bytes, row strides in bytes */
int sfb200_copy_rows_bytes(const void* src, int64_t src_stride_bytes, void* dst, int64_t dst_stride_bytes, int64_t rows,
                           int64_t row_bytes, void* stream);
int sfb200_gather_rows(const void* src, int64_t row_bytes, const int32_t* idx, int64_t rows, void* dst, void* stream);
/* strided row copy dst[i*dst_stride + 0..dim) = src[i*src_stride + 0..dim) (_finalize_trajectories :289-296) */
int sfb200_copy_rows(const float* src, int64_t src_stride, float* dst, int64_t dst_stride, int64_t rows, int dim,
                     void* stream);

/* Synthetic "tape" vector env (ours, not the reference's; contract = algo/utils/make_env.py:147-237 step()):
 * step = step_counter ? *step_counter : step_host.  reward = action/num_actions; terminated = ((step*7 + env*13) %
 * term_period == 0); truncated = ((step + env) % trunc_period == 0) & !terminated, env = env_index_offset + i;
 * obs_out = tape[(step+1) % tape_len] (tape: [tape_len, n_envs, dim]).  step_counter, if not NULL, points to int64[2]
 * {step, ticket}: the last thread block to finish advances `step` (device-side counter keeps the call replayable
 * inside a CUDA graph without an extra launch). */
int sfb200_tape_env_step(const int32_t* actions, int64_t n_envs, int num_actions, int64_t env_index_offset,
                         int term_period, int trunc_period, int64_t* step_counter, int64_t step_host,
                         const float* tape, int64_t tape_len, int dim, float* obs_out, float* rew,
                         uint8_t* terminated, uint8_t* truncated, void* stream);
/* the same env with a Box(act_dim) action space: reward = clamp(actions[:, 0], -1, 1) */
int sfb200_tape_env_step_continuous(const float* actions_f32, int act_dim, int64_t n_envs, int64_t env_index_offset,
                                    int term_period, int trunc_period, int64_t* step_counter, int64_t step_host,
                                    const float* tape, int64_t tape_len, int dim, float* obs_out, float* rew,
                                    uint8_t* terminated, uint8_t* truncated, void* stream);

/* ------------------------------------------------------------- learner: batch prep ---- */
/* learner.py:950-955: valids[:, :T] = (policy_id == this_policy) & (train_step - policy_version < max_lag);
 * valids[:, T] = valids[:, T-1]. */
int sfb200_compute_valids(const int32_t* policy_id, const float* policy_version, int64_t n_traj, int T,
                          int32_t this_policy, float train_step, float max_policy_lag, uint8_t* valids,
                          void* stream);
/* the same with the train-step counter read from device memory (a CUDA-graph-captured learner replays the launch) */
int sfb200_compute_valids_dev(const int32_t* policy_id, const float* policy_version, int64_t n_traj, int T,
                              int32_t this_policy, const int64_t* train_step_dev, float max_policy_lag, uint8_t* valids,
                              void* stream);

/* learner.py:969-1003 fused, warp-scan over the time axis (algo/utils/rl_utils.py:51-94):
 *   dv = normalize_returns ? clamp(values, +-5)*sigma + mu : values            (:969-978)
 *   if value_bootstrap: rewards += gamma * dv[:, :-1] * time_outs * dones       (:990, IN PLACE like the reference)
 *   adv = GAE(rewards, dones, dv, valids, gamma, lambda)                        (:994-1001)
 *   returns = adv + valids[:, :-1] * dv[:, :-1]                                  (:1003)
 * values/valids: [n_traj, T+1]; rewards/dones/time_outs/adv/returns: [n_traj, T]. ret_mean/ret_var: float64[1]
 * or NULL when normalize_returns is off. */
int sfb200_gae_returns(float* rewards, const uint8_t* dones, const uint8_t* time_outs, const float* values,
                       const uint8_t* valids, int64_t n_traj, int T, float gamma, float lam, int value_bootstrap,
                       const double* ret_mean, const double* ret_var, float eps, float clip, float* adv,
                       float* returns, void* stream);

/* learner.py:602-640 (V-trace), on device: inputs flat [n*R] env-major.  Outputs vs (targets) and adv. */
int sfb200_vtrace(const float* ratio, const float* values, const float* rewards, const uint8_t* dones, int64_t n,
                  int R, float gamma, float rho_hat, float c_hat, float* vs, float* adv, void* stream);

/* ------------------------------------------------------------- learner: loss ---- */
/* Layout of the device-side loss statistics block (doubles), written by sfb200_ppo_loss_*: */
#define SFB200_LS_NUM_VALID 0
#define SFB200_LS_ADV_MEAN 1
#define SFB200_LS_ADV_STD 2
#define SFB200_LS_POLICY_LOSS 3
#define SFB200_LS_VALUE_LOSS 4      /* already multiplied by value_loss_coeff */
#define SFB200_LS_EXPLORATION_LOSS 5 /* -coeff * mean entropy */
#define SFB200_LS_KL_LOSS 6         /* kl_loss_coeff * mean KL(new||old) */
#define SFB200_LS_KL_OLD_MEAN 7
#define SFB200_LS_KL_OLD_MAX 8
#define SFB200_LS_ENTROPY_MEAN 9
#define SFB200_LS_RATIO_MEAN_ABS_DEV 10 /* mean |1 - ratio| over valid */
#define SFB200_LS_RATIO_MIN 11
#define SFB200_LS_RATIO_MAX 12
#define SFB200_LS_FRACTION_CLIPPED 13
#define SFB200_LS_VALUE_MEAN 14
#define SFB200_LS_TOTAL_LOSS 15
#define SFB200_LS_SIZE 16

int64_t sfb200_loss_workspace_bytes(int64_t batch);

/* learner.py:588-594: log_prob(actions) under new logits and ratio = clamp(exp(lp - lp_old), 0.05, 20)
 * (needed before V-trace; the GAE path does not call this). */
int sfb200_action_ratio(const float* logits, int A, const float* actions_f32, const float* log_prob_old,
                        int64_t batch, float* ratio, void* stream);

/* learner.py:646-647 statistics: masked (valids) count / mean / UNBIASED std of adv -> stats[NUM_VALID, ADV_MEAN,
 * ADV_STD].  dp_partials (optional, 3 doubles: count, sum, sumsq) exposes the raw sums so data-parallel ranks can
 * all-reduce them and call sfb200_adv_stats_finalize. */
int sfb200_adv_stats(const float* adv, const uint8_t* valids, int64_t batch, double* stats, double* dp_partials,
                     void* workspace, void* stream);
int sfb200_adv_stats_finalize(const double* dp_partials, double* stats, void* stream);

/* learner.py:586-657 + :431-477 forward AND backward in one pass over the minibatch:
 *   inputs: new logits [B,A], new values [B]; batch tensors actions (f32), log_prob_old, values_old, adv (raw),
 *           targets (returns or vs), valids, logits_old [B,A]
 *   uses stats[NUM_VALID, ADV_MEAN, ADV_STD] (from sfb200_adv_stats) for the per-minibatch advantage normalisation
 *   outputs: dlogits [B,A], dvalues [B] = d(total loss)/d(.) ; stats[POLICY_LOSS .. TOTAL_LOSS]
 * exploration_loss: 0 = entropy bonus (learner.py:473-477), 1 = symmetric KL to the uniform prior (:479-486,
 * action_distributions.py:168-177; stats[EXPLORATION_LOSS] = +coeff * min(mean, 30)).
 * All means are over valid entries only (algo/utils/torch_utils.py:50-55).  grad_scale multiplies every gradient
 * (1/world_size under data parallelism). */
int sfb200_ppo_loss_fwd_bwd(const float* logits, const float* values, int A, const float* actions_f32,
                            const float* log_prob_old, const float* values_old, const float* adv,
                            const float* targets, const uint8_t* valids, const float* logits_old, int64_t batch,
                            float clip_ratio, float clip_value, float exploration_coeff, int exploration_loss,
                            float value_coeff, float kl_coeff, float grad_scale, float* dlogits, float* dvalues,
                            double* stats, void* workspace, void* stream);

/* Tuple(Discrete(n_0), ..., Discrete(n_{K-1})) action spaces (TupleActionDistribution, action_distributions.py:197-286):
 * K <= 8 independent categorical heads over consecutive segments of the A = sum n_k logits (head_sizes_host: K int32 on
 * the HOST).  actions_f32 rows hold K floats (one index per head), log-prob / entropy / KL are sums over the heads. */
int sfb200_action_ratio_tuple(const float* logits, int A, int num_heads, const int32_t* head_sizes_host,
                              const float* actions_f32, const float* log_prob_old, int64_t batch, float* ratio,
                              void* stream);
int sfb200_ppo_loss_fwd_bwd_tuple(const float* logits, const float* values, int A, int num_heads,
                                  const int32_t* head_sizes_host, const float* actions_f32, const float* log_prob_old,
                                  const float* values_old, const float* adv, const float* targets, const uint8_t* valids,
                                  const float* logits_old, int64_t batch, float clip_ratio, float clip_value,
                                  float exploration_coeff, int exploration_loss, float value_coeff, float kl_coeff,
                                  float grad_scale, float* dlogits, float* dvalues, double* stats, void* workspace,
                                  void* stream);

/* The same for a Box action space (ContinuousActionDistribution, action_distributions.py:290-323): params / params_old
 * rows are [means | log_std] (2*act_dim floats, the `action_logits` layout), actions_f32 rows act_dim floats.
 * adaptive_stddev: dlogits [B, 2*act_dim] = [d means | d log_std]; otherwise dlogits [B, act_dim] = d(pre-tanh means)
 * and dlogstd [B, act_dim], whose column sum is the gradient of the learned log-stddev vector
 * (action_parameterization.py:56-62). */
int sfb200_action_ratio_continuous(const float* params, int act_dim, const float* actions_f32, const float* log_prob_old,
                                   int64_t batch, float* ratio, void* stream);
int sfb200_ppo_loss_fwd_bwd_continuous(const float* params, const float* values, int act_dim, int adaptive_stddev,
                                       float tanh_scale, const float* actions_f32, const float* log_prob_old,
                                       const float* values_old, const float* adv, const float* targets,
                                       const uint8_t* valids, const float* params_old, int64_t batch, float clip_ratio,
                                       float clip_value, float exploration_coeff, float value_coeff, float kl_coeff,
                                       float grad_scale, float* dlogits, float* dlogstd, float* dvalues, double* stats,
                                       void* workspace, void* stream);

/* uint8 observations (image envs: the reference converts with .float() before sub-mean / scale / running-mean-std,
 * utils/normalize.py:40-67): the same three entry points reading uint8 rows; the raw copy into the trajectory stays
 * uint8 (shared_buffers.py:88-96 keeps the observation space's dtype). */
int sfb200_normalize_obs_u8(const uint8_t* x, int64_t ldx, float* y, int64_t ldy, int64_t rows, int dim,
                            const double* mean, const double* var, float sub_mean, float inv_scale, float eps,
                            float clip, void* stream);
int sfb200_sampler_pre_step_u8(const uint8_t* obs, int64_t n_envs, int dim, uint8_t* traj_obs_t, int64_t traj_obs_stride,
                               const float* rnn, int rnn_dim, float* traj_rnn_t, int64_t traj_rnn_stride, float* x_norm,
                               const double* mean, const double* var, float sub_mean, float inv_scale, float eps,
                               float clip, void* stream);
int sfb200_sampler_post_pre_step_u8(const float* rew, const uint8_t* terminated, const uint8_t* truncated, int64_t n_envs,
                                    float reward_scale, float reward_clip, int32_t policy_id, float* traj_rewards_t,
                                    uint8_t* traj_dones_t, uint8_t* traj_time_outs_t, int32_t* traj_policy_id_t,
                                    int64_t traj_stride, float* ep_return, int32_t* ep_len, float* ep_min_raw,
                                    float* ep_max_raw, int32_t len_increment, double* stats, int64_t* step_counter,
                                    float* fin_return_t, int32_t* fin_len_t,
                                    const uint8_t* obs, int dim, uint8_t* traj_obs_next, int64_t traj_obs_stride,
                                    const float* rnn, int rnn_dim, float* traj_rnn_next, int64_t traj_rnn_stride,
                                    float* x_norm, const double* mean, const double* var, float sub_mean,
                                    float inv_scale, float eps, float clip, void* stream);

/* ------------------------------------------------------------- convolutional encoder ---- */
/* ConvEncoderImpl (model/encoder.py:88-118): Conv2d without padding = im2col + sfb200_linear_act_forward.
 *   col[(b,oh,ow), (ci,kh,kw)] = x[b, ci, oh*stride+kh, ow*stride+kw]      (column order == Conv2d weight flatten)
 * x is NCHW [B,C,H,W] (in_nchw = 1: the normalised observation) or NHWC [B,H,W,C] (the previous layer's GEMM output);
 * col is [B*OH*OW, C*kernel*kernel] with OH = (H-kernel)/stride+1. */
int sfb200_im2col(const float* x, int in_nchw, int64_t B, int C, int H, int W, int kernel, int stride, float* col,
                  void* stream);
/* backward of im2col fused with the activation derivative of the layer that produced x_act (NHWC, activated):
 *   dx[b,ih,iw,ci] = act'(x_act[b,ih,iw,ci]) * sum_{windows covering (ih,iw)} dcol[(b,oh,ow), (ci,kh,kw)]   (gather) */
int sfb200_col2im_act_backward(const float* dcol, const float* x_act, int64_t B, int C, int H, int W, int kernel,
                               int stride, int act, float* dx, void* stream);
/* [B, P, C] <-> [B, C, P]: NHWC rows of the last conv layer <-> the (C,H,W) flatten order of encoder.py:115 */
int sfb200_permute_bpc(const float* src, float* dst, int64_t B, int P, int C, int to_channel_major, void* stream);

/* ------------------------------------------------------------- learner: backward ---- */
int64_t sfb200_heads_backward_workspace_bytes(int H, int A);
/* backward of critic_linear + distribution_linear fused with the activation derivative of the layer that produced h:
 *   dz[i,j]   = (sum_a dlogits[i,a]*Wa[a,j] + dvalues[i]*Wv[j]) * act'(h[i,j])      (act' from the OUTPUT h)
 *   dWa, dWv, dba, dbv  (+= over rows)  and  db_prev[j] = sum_i dz[i,j]
 * Gradients are WRITTEN (not accumulated) to the given pointers. */
int sfb200_heads_backward(const float* h, int64_t ldh, int64_t rows, int H, int A, const float* Wv, const float* Wa,
                          const float* dlogits, const float* dvalues, int act, float* dz, int64_t lddz, float* dWv,
                          float* dbv, float* dWa, float* dba, float* db_prev, void* workspace, void* stream);

int64_t sfb200_linear_backward_workspace_bytes(int64_t M, int N, int K);
/* backward of y = act(x.W^T + b) given dz = dL/d(pre-activation) [M,N]:
 *   dW[N,K] = dz^T . x  (skipped if dW == NULL) ;  (db is produced by the kernel that made dz)
 *   if dx != NULL: dx[M,K] = (dz . W) * act_prev'(x)     (x is the previous layer's OUTPUT, act_prev its activation;
 *                                                       pass SFB200_ACT_NONE for the input layer)
 *   if db_prev != NULL: db_prev[k] = sum_i dx[i,k]  (bias gradient of the previous layer) */
int sfb200_linear_backward(const float* dz, int64_t lddz, const float* x, int64_t ldx, const float* W, int64_t M,
                           int N, int K, int act_prev, float* dW, float* dx, int64_t lddx, float* db_prev,
                           int engine, void* workspace, void* stream);

/* column sums out[n] = sum_m x[m, n] (bias gradients); workspace >= sfb200_colsum_workspace_bytes(N) */
int64_t sfb200_colsum_workspace_bytes(int N);
int sfb200_colsum(const float* x, int64_t ldx, int64_t M, int N, float* out, void* workspace, void* stream);

/* ------------------------------------------------------------- recurrent core ---- */
/* model/core.py:19-64 (ModelCoreRNN: nn.GRU / nn.LSTM, one layer).  The two gate GEMMs gi = x.W_ih^T + b_ih and
 * gh = h.W_hh^T + b_hh are sfb200_linear_act_forward calls (act NONE); these kernels do the cell math.
 * GRU (gates r,z,n):  r = s(gi_r+gh_r), z = s(gi_z+gh_z), n = tanh(gi_n + r*gh_n), h' = (1-z)*n + z*h
 *   h_out  [M,H]   the new state / core output
 *   h_next [M,H]   optional: h' with rows whose reset_next flag is set zeroed -- the next step's input state
 *                  (batched_sampling.py:332-335 in the sampler, rnn_utils.py:143-149 in the learner)
 *   gates  [M,3H]  optional save of (r,z,n) for the backward pass */
int sfb200_gru_cell_forward(const float* gi, int64_t ldgi, const float* gh, int64_t ldgh, const float* h_in, int64_t ldh,
                            float* h_out, int64_t ldo, float* h_next, int64_t ldn, const uint8_t* reset_next,
                            int64_t reset_stride, float* gates, int64_t ldg, int64_t M, int H, void* stream);
/* backward of one GRU step: dh = dh_out + (reset ? 0 : carry_a + carry_b)  (carry_* = gradient arriving from step t+1
 * through the state: the GEMM part dgh(t+1).W_hh and the direct part dh(t+1)*z(t+1); `reset` is the flag applied
 * between t and t+1).  Outputs dgi [M,3H], dgh [M,3H] and dh_direct = dh*z [M,H]. */
int sfb200_gru_cell_backward(const float* dh_out, int64_t lddo, const float* carry_a, const float* carry_b, int64_t ldc,
                             const uint8_t* reset, int64_t reset_stride, const float* gates, int64_t ldg, const float* gh,
                             int64_t ldgh, const float* h_in, int64_t ldh, float* dgi, int64_t lddgi, float* dgh,
                             int64_t lddgh, float* dh_direct, int64_t lddd, int64_t M, int H, void* stream);
/* LSTM (gates i,f,g,o over gi+gh), state layout [h || c] of width 2H as in the reference (core.py:51-53):
 *   c' = f*c + i*g ; h' = o*tanh(c') ; state_out = [h' || c'] ; state_next = state_out with reset rows zeroed ;
 *   gates [M,4H] optional save of the activated gates */
int sfb200_lstm_cell_forward(const float* gi, int64_t ldgi, const float* gh, int64_t ldgh, const float* state_in,
                             int64_t lds, float* state_out, int64_t ldo, float* state_next, int64_t ldn,
                             const uint8_t* reset_next, int64_t reset_stride, float* gates, int64_t ldg, int64_t M, int H,
                             void* stream);
/* backward of one LSTM step; dgates [M,4H] is the gradient of BOTH gi and gh; dc_in [M,H] is carried to step t-1 */
int sfb200_lstm_cell_backward(const float* dh_out, int64_t lddo, const float* dh_carry, const float* dc_carry, int64_t ldc,
                              const uint8_t* reset, int64_t reset_stride, const float* gates, int64_t ldg,
                              const float* state_in, int64_t lds, const float* state_out, int64_t ldo, float* dgates,
                              int64_t lddg, float* dc_in, int64_t lddc, int64_t M, int H, void* stream);
/* dst[i,:] = reset[i] ? 0 : src[i,:]   (last_rnn_state = new_rnn_states * (1 - done), batched_sampling.py:332-335) */
int sfb200_mask_rows(const float* src, int64_t src_stride, float* dst, int64_t dst_stride, const uint8_t* reset,
                     int64_t reset_stride, int64_t rows, int dim, void* stream);

/* ------------------------------------------------------------- optimizer ---- */
/* learner.py:782-797: global grad-norm clip (torch clip_grad_norm_: coef = min(max_norm/(norm+1e-6), 1), skipped
 * when max_norm <= 0) followed by torch.optim.Adam's update (no weight decay / amsgrad) on FLAT buffers:
 *   m = m + (1-b1)(g-m) ; v = b2 v + (1-b2) g^2 ; p -= (lr*lr_scale/(1-b1^t)) * m / (sqrt(v)/sqrt(1-b2^t) + eps)
 * lr_scale_num/lr_scale_den (device doubles or NULL): lr *= num/den  -- the valid-fraction scaling of :788-794
 * grad_norm_out (device float[1], optional) receives the pre-clip norm.  workspace >= 4096 bytes.
 * Scalars are doubles because the reference passes Python floats (torch converts them to fp32 op-math itself).
 * g is read, not rescaled in place (the reference's in-place clip of .grad is unobservable on this path). */
int sfb200_clip_adam_step(float* p, float* g, float* m, float* v, int64_t n, int64_t step, double lr, double beta1,
                          double beta2, double eps, double max_grad_norm, const double* lr_scale_num,
                          const double* lr_scale_den, float* grad_norm_out, void* workspace, void* stream);
/* Graph-replayable variant: the number of optimizer steps ALREADY taken and the learning rate are read from device
 * memory (bias corrections 1 - beta^(steps_done+1) are formed in the kernel, in double like the host path);
 * sfb200_advance_counters(a, b) adds 1 to up to two device counters (optimizer step, policy version) afterwards. */
int sfb200_clip_adam_step_dev(float* p, float* g, float* m, float* v, int64_t n, const int64_t* steps_done_dev,
                              const double* lr_dev, double beta1, double beta2, double eps, double max_grad_norm,
                              const double* lr_scale_num, const double* lr_scale_den, float* grad_norm_out,
                              void* workspace, void* stream);
int sfb200_advance_counters(int64_t* a, int64_t* b, void* stream);

/* The reference's other optimizer, cfg.optimizer = "lamb" (algo/utils/optimizers.py:13-175 as the learner constructs it,
 * learner.py:228-243: bias correction, weight_decay 1e-4, min_trust 0.01, no look-ahead), after the same global grad-norm
 * clip and valid-fraction lr scaling as sfb200_clip_adam_step.  The flat buffers are described per tensor by
 * seg_offsets / seg_numel (device int64[num_tensors]; padding between tensors is never touched) because the trust ratio
 *   clamp(min(|p_t|, 10) / |u_t|, min_trust, 1/min_trust),  u = m_hat / (sqrt(v_hat) + eps) + weight_decay * p
 * is per parameter tensor.  g is overwritten with u.  `step` starts at 1. */
int64_t sfb200_lamb_workspace_bytes(int num_tensors, int64_t max_numel);
int sfb200_clip_lamb_step(float* p, float* g, float* m, float* v, int64_t n, const int64_t* seg_offsets,
                          const int64_t* seg_numel, int num_tensors, int64_t max_numel, int64_t step, double lr,
                          double beta1, double beta2, double eps, double weight_decay, double min_trust,
                          double max_grad_norm, const double* lr_scale_num, const double* lr_scale_den,
                          float* grad_norm_out, void* workspace, void* stream);

/* ---------------------------------------------------------------- data parallel (NVLink peer memory) ----
 * New functionality (the reference has no collective, SURVEY 2a / 8e): G ranks x N envs == one process with G*N envs.
 * Equivalence target: learner.py:774-821 applied to the concatenated batch.  Every rank owns one comm buffer
 *   [16 KiB header | scratch_bytes of fp64 scratch | flat fp32 gradient]
 * that its peers map with CUDA IPC (sfb200_ipc_export on the owner, sfb200_ipc_import on each peer; the pointer may lie
 * anywhere inside a cudaMalloc allocation -- the handle names the allocation, `offset` the position inside it).  The
 * buffer must be zero-filled before the first collective.  sfb200_dp_create returns a communicator id (>= 0) or -1;
 * peer_ptrs_host[r] = device address of rank r's comm buffer as seen from THIS process (own buffer at [rank]).
 * All collectives only enqueue kernels; their sequence numbers live in device memory (CUDA-graph replayable).  Every
 * rank must issue the same sequence of dp_* calls. */
int sfb200_ipc_export(const void* ptr, void* handle_out_host, int64_t* offset_out_host);
int sfb200_ipc_import(const void* handle_host, int64_t offset, void** ptr_out_host);
int sfb200_ipc_close(void* ptr, int64_t offset);
int64_t sfb200_dp_header_bytes(void);
int sfb200_dp_create(int rank, int world, const uint64_t* peer_ptrs_host, int64_t scratch_bytes);
int sfb200_dp_destroy(int comm);
/* g_out[0..n) = sum over ranks (rank order 0..G-1) of the gradient regions of all comm buffers; workspace >= 4 KiB */
int sfb200_dp_grad_allreduce(int comm, float* g_out, int64_t n, void* workspace, void* stream);
/* the same all-reduce fused with sfb200_clip_adam_step(_dev) on the reduced gradient in ONE kernel (one-shot peer pull ->
 * device-wide barrier for the global norm -> clip -> Adam).  steps_done_dev / lr_dev non-NULL select the device-side
 * counters of sfb200_clip_adam_step_dev (then `step` / `lr` are ignored). */
int sfb200_dp_grad_allreduce_clip_adam(int comm, float* g_out, float* p, float* m, float* v, int64_t n, int64_t step,
                                       const int64_t* steps_done_dev, double lr, const double* lr_dev, double beta1,
                                       double beta2, double eps, double max_grad_norm, const double* lr_scale_num,
                                       const double* lr_scale_den, float* grad_norm_out, void* workspace, void* stream);
/* in-place all-reduce of n doubles; element i is column i % row_len (row_len <= 64; 0 = plain sum): columns in max_mask /
 * min_mask are combined with max / min, columns in keep_mask are left untouched, columns in avg_mask are averaged over
 * the ranks, all others are summed */
int sfb200_dp_allreduce_f64(int comm, double* buf, int n, int row_len, uint64_t max_mask, uint64_t min_mask,
                            uint64_t keep_mask, uint64_t avg_mask, void* stream);
/* per-rank (mean, UNBIASED var) over rows_per_rank rows -> moments of the concatenation of all ranks' rows, in place
 * (what makes G ranks update the running normalizers, running_mean_std.py:72-77, like one process with all rows) */
int sfb200_dp_pooled_moments(int comm, float* batch_mean, float* batch_var, int dim, double rows_per_rank, void* stream);
/* out[0] = sum_r src[r * stride + col] (global valid count from the all-reduced minibatch partials) */
int sfb200_colsum_f64(const double* src, int rows, int stride, int col, double* out, void* stream);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* SFB200_H */
