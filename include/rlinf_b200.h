/*
 * rlinf_b200.h - C ABI of librlinf_b200.so: the B200-native (sm_100a) drop-in for the
 * data-parallel hot path of RLinf's actor-learner (advantages, PPO/GRPO loss,
 * MLP policy forward/backward, grad-clip + AdamW, rollout sampling).
 *
 * Conventions (SURVEY.md §8b):
 *  - plain pointers and sizes; every pointer is a DEVICE pointer unless the name ends in `_host`;
 *  - every entry point takes a `stream` (a cudaStream_t passed as void*), never synchronises
 *    the device, allocates nothing the caller can see, and owns no state except a lazily
 *    created per-device scratch (a few KB of reduction slots, TMA descriptors);
 *  - outputs are caller-allocated; inputs are never mutated;
 *  - return value: 0 = ok, <0 = invalid argument (RB200_E_*), >0 = a cudaError_t;
 *  - bool tensors are 1 byte per element (torch.bool / uint8), fp tensors are float32
 *    (the reference asserts fp32: rlinf/algorithms/losses.py:232-240).
 *
 * Each entry point cites the reference interface it replaces (file:line under the
 * RLinf v0.4.0 tree).  The reference is 100 % Python; the binding a maintainer
 * would add is a ctypes stub, shown in INTEGRATION.md.
 */
#ifndef RLINF_B200_H
#define RLINF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RB200_ABI_VERSION 1

/* error codes (<0); >0 is a cudaError_t */
#define RB200_OK 0
#define RB200_E_NULL (-1)      /* required pointer is NULL */
#define RB200_E_SHAPE (-2)     /* non-positive / inconsistent dimension */
#define RB200_E_ARG (-3)       /* bad scalar argument (e.g. clip_ratio_c <= 1) */
#define RB200_E_ALIGN (-4)     /* pointer not aligned as required */
#define RB200_E_UNSUPPORTED (-5)

typedef void* rb200_stream_t; /* cudaStream_t */

int rb200_abi_version(void);
const char* rb200_strerror(int code);
/* sm count / compute capability of the current device (host-side query). */
int rb200_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* kernels launched by this library in this process so far (host counter; launches replayed from a
 * captured CUDA graph are counted once, at capture). */
uint64_t rb200_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * K0  loss mask            replaces compute_loss_mask, rlinf/utils/metric_utils.py:516-537
 *   dones     bool  [(nc+1), B, C]
 *   mask      bool  [nc, B, C]        step valid while no done seen in rows [0..t]
 *   mask_sum  int64 [B]               per-env valid-step count (the reference expands it
 *                                     to mask's shape as a view; the shim does the same)
 * ---------------------------------------------------------------------------------------- */
int rb200_loss_mask(const uint8_t* dones, uint8_t* mask, int64_t* mask_sum,
                    int nc, int B, int C, rb200_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K1  GAE scan (+ normalisation statistics)
 *   replaces compute_gae_advantages_and_returns, rlinf/algorithms/advantages.py:24-86
 *   (the T-iteration Python loop) and the statistics half of safe_normalize,
 *   rlinf/algorithms/utils.py:397-404.
 *   Step-major layout: rewards [T,B] f32, values [T+1,B] f32 (NULL = critic-free: gamma=lambda=1,
 *   delta=r), dones [T+1,B] bool, loss_mask [T,B] bool or NULL.
 *   adv, ret [T,B] f32 are the UN-normalised outputs, bit-identical to the reference's fp32
 *   sequential recurrence (each op rounded separately, no FMA contraction).
 *   stats (may be NULL): double[6] = {n, sum, sumsq} of adv over valid entries, then of ret.
 *   The caller zeroes nothing: the call resets stats itself.
 *   gamma / gae_lambda are doubles because the reference rounds fl32(gamma) for gamma*V but
 *   fl32(gamma*gae_lambda) (product taken in Python double) for the recurrence coefficient.
 * ---------------------------------------------------------------------------------------- */
int rb200_gae(const float* rewards, const float* values, const uint8_t* dones,
              const uint8_t* loss_mask, float* adv, float* ret, double* stats,
              int T, int B, double gamma, double gae_lambda, rb200_stream_t stream);

/* x <- (x - mean) / (std_unbiased + eps) with {n,sum,sumsq} = stats[0..2]; no-op if n == 0.
 * The apply half of safe_normalize (eps=1e-5, rlinf/algorithms/utils.py:397-404). In place. */
int rb200_normalize(float* x, const double* stats, int64_t n_elems, float eps,
                    rb200_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K1' GRPO: first-episode scores + group normalisation + broadcast over T
 *   replaces calculate_scores, rlinf/algorithms/utils.py:134-152 (CPU-only reverse loop) and
 *   compute_grpo_advantages, rlinf/algorithms/advantages.py:89-121.
 *   rewards [T,B] f32, dones [T+1,B] bool -> scores [B] f32 (bit-identical reverse accumulation)
 *   scores [B] (groups of G consecutive envs), loss_mask [T,B] bool -> adv [T,B] f32
 * ---------------------------------------------------------------------------------------- */
int rb200_grpo_scores(const float* rewards, const uint8_t* dones, float* scores,
                      int T, int B, rb200_stream_t stream);
int rb200_grpo_advantages(const float* scores, const uint8_t* loss_mask, float* adv,
                          int T, int B, int G, float eps, rb200_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * a12 trajectory gather    replaces process_nested_dict_for_train's
 *   `value.reshape(-1, ...)[shuffle_id]`, rlinf/utils/nested_dict_process.py:272-285.
 *   dst[i, :] = src[idx[i], :] for rows of `row_bytes` bytes (any dtype). idx is int64.
 * ---------------------------------------------------------------------------------------- */
int rb200_gather_rows(const void* src, const int64_t* idx, void* dst, int64_t n_rows_out,
                      int64_t n_rows_src, int64_t row_bytes, rb200_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K2  fused (gather +) PPO actor[-critic] loss, forward + backward in one pass
 *   replaces policy_loss, rlinf/algorithms/registry.py:77-92, preprocess_loss_inputs
 *   (algorithms/utils.py:280-376), compute_ppo_actor_loss (losses.py:170-312),
 *   compute_ppo_critic_loss (losses.py:315-380), the entropy term and 1/grad_accum scaling of
 *   embodied_fsdp_actor_worker.py:678-695, and autograd's backward of all of it.
 * ---------------------------------------------------------------------------------------- */
enum { RB200_LOGPROB_TOKEN = 0, RB200_LOGPROB_ACTION = 1, RB200_LOGPROB_CHUNK = 2 };

/* indices into the metrics vector written by rb200_ppo_loss */
enum {
  RB200_M_POLICY_LOSS = 0,      /* actor/policy_loss        */
  RB200_M_POLICY_LOSS_ABS = 1,  /* actor/policy_loss_abs    */
  RB200_M_RATIO = 2,            /* actor/ratio              */
  RB200_M_RATIO_ABS = 3,        /* actor/ratio_abs          */
  RB200_M_CLIPPED_RATIO = 4,    /* actor/clipped_ratio      */
  RB200_M_DUAL_CLIPPED_RATIO = 5, /* actor/dual_cliped_ratio (sic, reference spelling) */
  RB200_M_APPROX_KL = 6,        /* actor/approx_kl          */
  RB200_M_CLIP_FRACTION = 7,    /* actor/clip_fraction      */
  RB200_M_VALUE_LOSS = 8,       /* critic/value_loss        */
  RB200_M_VALUE_CLIP_RATIO = 9, /* critic/value_clip_ratio  */
  RB200_M_EV_COUNT = 10,        /* __sum__/_critic_explained_variance/count          */
  RB200_M_EV_RET_SUM = 11,      /*   .../returns_sum     */
  RB200_M_EV_RET_SQ_SUM = 12,   /*   .../returns_sq_sum  */
  RB200_M_EV_ERR_SUM = 13,      /*   .../errors_sum      */
  RB200_M_EV_ERR_SQ_SUM = 14,   /*   .../errors_sq_sum   */
  RB200_M_ENTROPY = 15,         /* actor/entropy_loss (masked mean entropy, before the bonus) */
  RB200_M_TOTAL_LOSS = 16,      /* actor/total_loss  (after entropy bonus and loss_scale)     */
  RB200_M_TOKEN_NUM = 17,       /* number of valid loss entries (count_nonzero of the mask)    */
  RB200_NUM_METRICS = 24
};

typedef struct rb200_ppo_args {
  /* shapes: bsz samples x C chunks x A action dims. A "unit" is one (sample, chunk) for
   * token/action level and one sample for chunk level; U = units per sample (C or 1). */
  int64_t bsz;
  int32_t C, A;
  int32_t logprob_type; /* RB200_LOGPROB_* */
  int32_t with_critic;  /* 1: actor_critic, 0: actor only */
  /* current policy outputs for this micro-batch (NOT gathered) */
  const float* logprobs; /* [bsz, C*A] */
  const float* values;   /* [bsz, U] or NULL */
  const float* entropy;  /* [bsz, C*A] or NULL (entropy bonus term, action-level reduction) */
  /* rollout data; row i of the micro-batch lives at row (idx ? idx[i] : i) */
  const int64_t* idx;          /* [bsz] or NULL */
  const float* old_logprobs;   /* [rows, C*A] */
  const float* advantages;     /* [rows, U] */
  const float* returns;        /* [rows, U] or NULL */
  const float* prev_values;    /* [rows, U] or NULL */
  const uint8_t* loss_mask;    /* [rows, U] or NULL */
  const int64_t* loss_mask_sum; /* [rows or mask_sum_rows, U] or NULL */
  int64_t mask_sum_row_mod;    /* >0: loss_mask_sum row = row % mask_sum_row_mod (per-env table) */
  /* deferred advantage normalisation: if non-NULL, advantages are normalised on the fly with
   * {n,sum,sumsq} = adv_stats[0..2] and eps adv_norm_eps (fusion of safe_normalize) */
  const double* adv_stats;
  float adv_norm_eps;
  /* hyper-parameters (losses.py:170-186, 315-325). Doubles: the reference holds them as Python
   * floats and rounds derived bounds (e.g. 1.0 - clip_ratio_low) once, from double. */
  double clip_ratio_low, clip_ratio_high;
  double clip_ratio_c;      /* <= 0: no dual clip; else must be > 1 */
  int32_t has_clip_log_ratio_min, has_clip_log_ratio_max;
  double clip_log_ratio_min, clip_log_ratio_max;
  double value_clip, huber_delta;
  int32_t max_episode_steps; /* >0 with mask+mask_sum: masked_mean_ratio aggregation */
  int32_t critic_warmup;     /* 1: policy loss := 0 (no actor grads) */
  double entropy_bonus;      /* 0: none */
  double loss_scale;         /* 1/gradient_accumulation */
  /* scratch: caller-provided, 32 doubles, ZERO before its first use; every call leaves it zeroed again (the last CTA
   * clears it), so one zero-initialised buffer per stream is reused without memset nodes. Calls sharing a workspace
   * must be stream-ordered. */
  double* workspace;
  /* outputs */
  float* loss;        /* [1] total loss (after entropy bonus and loss_scale) */
  float* metrics;     /* [RB200_NUM_METRICS] */
  float* d_logprobs;  /* [bsz, C*A] or NULL */
  float* d_values;    /* [bsz, U] or NULL */
  float* d_entropy;   /* [bsz, C*A] or NULL */
} rb200_ppo_args;

int rb200_ppo_loss(const rb200_ppo_args* args, rb200_stream_t stream);

/* "decoupled_actor_critic" (losses.py:27-167 + :315-380, registered :383-394): PPO clipped around a proximal policy.
 * `base` carries everything shared with rb200_ppo_loss (entropy / log-ratio clamps / adv_stats must be unset);
 * metrics use the RB200_DM_* layout. */
enum {
  RB200_DM_POLICY_LOSS = 0,            /* actor/policy_loss            */
  RB200_DM_PROXIMAL_RATIO = 1,         /* actor/proximal_ratio         */
  RB200_DM_CLIPPED_PROXIMAL_RATIO = 2, /* actor/clipped_proximal_ratio */
  RB200_DM_CLIP_FRACTION = 3,          /* actor/clip_fraction          */
  RB200_DM_DUAL_CLIP_FRACTION = 4,     /* actor/dual_clip_fraction     */
  RB200_DM_BEHAV_CLIP_FRACTION = 5,    /* actor/behav_clip_fraction    */
  RB200_DM_PROXIMAL_APPROX_KL = 6,     /* actor/proximal_approx_kl     */
  RB200_DM_BEHAV_APPROX_KL = 7,        /* actor/behav_approx_kl        */
  RB200_DM_VALUE_LOSS = 8,             /* critic/value_loss            */
  RB200_DM_VALUE_CLIP_RATIO = 9,       /* critic/value_clip_ratio      */
  RB200_DM_EV_COUNT = 10,              /* 10..14: explained-variance sufficient statistics, as RB200_M_EV_* */
  RB200_DM_AVERAGE_VERSION = 15,       /* actor/average_version (valid iff slot 19 != 0) */
  RB200_DM_TOTAL_LOSS = 16,
  RB200_DM_TOKEN_NUM = 17,
  RB200_DM_CURRENT_VERSION = 18,       /* actor/current_version */
  RB200_DM_HAS_VERSION_METRICS = 19
};
typedef struct rb200_dppo_args {
  rb200_ppo_args base;
  const float* proximal_logprobs; /* [rows, C*A] or NULL: anchor = old_logprobs, or the version interpolation */
  const float* versions;          /* [rows, C*A] fp32 weight version that generated each token, or NULL */
  int32_t has_current_version;
  double current_version;
  int32_t has_behave_weight_threshold;
  double behave_weight_threshold;
} rb200_dppo_args;
int rb200_decoupled_ppo_loss(const rb200_dppo_args* args, rb200_stream_t stream);

/* "opd" (losses.py:427-505): loss = agg(-logprobs * stop_grad(advantages)) with the mask / mask_sum broadcast over the
 * tokens of a unit. logprobs, advantages: [n_units, tokens_per_unit]; loss_mask (uint8), loss_mask_sum: [n_units].
 * max_episode_steps > 0 selects masked_mean_ratio. workspace: as rb200_ppo_args.workspace. */
enum { RB200_OM_POLICY_LOSS = 0, RB200_OM_OPD_REWARD = 1, RB200_OM_OPD_REVERSE_KL = 2, RB200_OM_TOTAL_LOSS = 16 };
int rb200_opd_loss(const float* logprobs, const float* advantages, const uint8_t* loss_mask,
                   const int64_t* loss_mask_sum, int64_t n_units, int tokens_per_unit, int max_episode_steps,
                   double loss_scale, double* workspace, float* loss /*[1] or NULL*/,
                   float* metrics /*[RB200_NUM_METRICS]*/, float* d_logprobs /*or NULL*/, rb200_stream_t stream);

/* x[i] *= s (device scalar-free helper for autograd's upstream scalar). */
int rb200_scale(float* x, int64_t n, float s, rb200_stream_t stream);
/* x[i] *= *s_dev  (the scalar lives on the device: no host sync in autograd's backward). */
int rb200_scale_by(float* x, int64_t n, const float* s_dev, rb200_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K4  grad-norm clip + AdamW on one flat fp32 buffer
 *   replaces FSDPModelManager.optimizer_step, hybrid_engines/fsdp/fsdp_model_manager.py:429-463
 *   (clip_grad_norm_ of the no_shard path strategy/fsdp.py:363-369 = torch.nn.utils.clip_grad_norm_:
 *   coef = min(1, max_norm/(norm+1e-6)); non-finite norm => step skipped) and torch.optim.AdamW
 *   with the two lr groups of build_optimizer :501-590.
 *   group_end[k] = exclusive end offset of lr group k in the flat buffer (ascending).
 *   state: double[4] device = {step_count, last_grad_norm, last_clip_coef, skipped_flag}.
 * ---------------------------------------------------------------------------------------- */
int rb200_grad_sqnorm(const float* grads, int64_t n, double* out_sq /*[1], reset by kernel*/,
                      rb200_stream_t stream);
int rb200_adamw_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                     int64_t n, const int64_t* group_end_host, const double* group_lr_host,
                     int n_groups, double beta1, double beta2, double eps, double weight_decay,
                     float max_grad_norm, float grad_scale, const double* grad_sq /*[1]*/,
                     double* state /*[4]*/, rb200_stream_t stream);
/* Same step with the per-group learning rates read from DEVICE memory (double[n_groups]) at execution time, so a
 * captured CUDA graph follows an LR schedule (LambdaLR stepped once per run_training,
 * workers/actor/embodied_fsdp_actor_worker.py:571, hybrid_engines/fsdp/utils.py:522) without re-capture.
 * In both entries lr < 0 marks a FROZEN group: its parameters and moments are left untouched - what
 * torch.optim.AdamW does for parameters outside its param groups (the actor during critic warm-up,
 * fsdp_model_manager.py:523-531) or whose grad is None. */
int rb200_adamw_step_dev(float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                         int64_t n, const int64_t* group_end_host, const double* group_lr_dev,
                         int n_groups, double beta1, double beta2, double eps, double weight_decay,
                         float max_grad_norm, float grad_scale, const double* grad_sq /*[1]*/,
                         double* state /*[4]*/, rb200_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K3/K5  MLP policy (3x256 tanh backbone + mean head, state-independent log-std, 3x256 value
 *   MLP).  replaces MLPPolicy.default_forward, models/embodiment/mlp_policy/mlp_policy.py:202-236,
 *   ValueHead.forward, models/embodiment/modules/value_head.py:66, _generate_actions :256-293,
 *   and autograd's backward through them.  Declared in the second half of this header
 *   (rb200_mlp_*), see below.
 * ---------------------------------------------------------------------------------------- */

/* flat parameter layout, in the reference's named_parameters() order */
typedef struct rb200_mlp_layout {
  int32_t obs_dim, act_dim /* C*A outputs of the mean head */, value_dim, hidden /* 256 */;
  int64_t logstd;                         /* [act_dim] */
  int64_t vw0, vb0, vw1, vb1, vw2, vb2, vw3; /* value head: [H,obs],[H],[H,H],[H],[H,H],[H],[value_dim,H] */
  int64_t bw0, bb0, bw1, bb1, bw2, bb2;   /* backbone */
  int64_t mw, mb;                         /* actor_mean [act_dim,H],[act_dim] */
  int64_t total;                          /* number of floats */
} rb200_mlp_layout;

int rb200_mlp_layout_init(rb200_mlp_layout* L, int obs_dim, int act_dim, int value_dim, int hidden);

/* scratch sizes (floats) for n rows: `acts` and `work` of forward/backward/sample/value each need this many */
int64_t rb200_mlp_fwd_scratch_floats(const rb200_mlp_layout* L, int64_t n);

/* Tensor-core weight cache (`wsplit`, required by the calls below): the hidden-layer weights as packed fp16 (hi, lo)
 * tiles of w * 2^10, a forward pack per matrix and a dgrad pack per square matrix, in the layout the fp16-split GEMMs
 * read.  rb200_mlp_wsplit_floats() floats, 16-byte aligned; refresh with rb200_mlp_prepare_weights() after every
 * parameter update. */
int64_t rb200_mlp_wsplit_floats(const rb200_mlp_layout* L);
int rb200_mlp_prepare_weights(const rb200_mlp_layout* L, const float* params, float* wsplit,
                              rb200_stream_t stream);

/* Forward for training: states [n,obs] (row i at idx?idx[i]:i), action [n,act] (same gather).
 * Writes logprobs [n,act], entropy [n,act] (NULL ok), values [n,value_dim] (NULL ok) and keeps
 * the activations needed by backward in `acts`. Hidden layers run on tcgen05 (kind::f16, 2-way fp16 split, fp32-level
 * accuracy); the first layer falls back to an fp32 SIMT GEMM when obs_dim % 32 != 0 or idx is given.  Activations are
 * plain fp32; the tensor-core kernels split them into fp16 (hi, lo) operands in shared memory. */
int rb200_mlp_forward(const rb200_mlp_layout* L, const float* params, const float* wsplit,
                      const float* states, const float* action, const int64_t* idx, int64_t n,
                      float* logprobs, float* entropy, float* values, float* acts, float* work,
                      rb200_stream_t stream);

/* Backward: given d_logprobs [n,act], d_entropy [n,act] or NULL, d_values [n,value_dim] or NULL,
 * ACCUMULATES (+=) parameter gradients into grads (flat, same layout). `acts` from forward.
 * The sums over rows are stored per block / sample chunk in `work` and added in a fixed order, so the gradients are
 * bit-identical from run to run; the exception is the first layer's weight gradient on the fp32 SIMT GEMM (obs_dim % 32
 * != 0, obs_dim > 256 or idx given), which adds float partial sums with atomics.  Calls sharing a `work` buffer must be
 * stream-ordered. */
int rb200_mlp_backward(const rb200_mlp_layout* L, const float* params, const float* wsplit,
                       const float* states, const float* action, const int64_t* idx, int64_t n,
                       const float* d_logprobs, const float* d_entropy, const float* d_values,
                       const float* acts, float* work, float* grads, rb200_stream_t stream);

/* Rollout step (inference): mean/value forward, action = mean + exp(logstd)*noise where noise is
 * either supplied ([n,act], parity mode) or drawn from Philox(seed, offset + *counter_dev) (noise == NULL;
 * counter_dev may be NULL); writes action [n,act], logprobs [n,act], values [n,value_dim]. */
int rb200_mlp_sample(const rb200_mlp_layout* L, const float* params, const float* wsplit,
                     const float* states, const float* noise, uint64_t seed, uint64_t offset,
                     const uint64_t* counter_dev, int64_t n, float* action, float* logprobs, float* values,
                     float* work, rb200_stream_t stream);

/* Unit-test entries of the fp16-split kind::f16 GEMMs of the MLP towers (csrc/tc_gemm_h.cu), fp32 in/out.
 * rb200_tc_gemm_h: mode 0: C = A[M,K] . B[256,K]^T; mode 1 (dgrad form, K = 256): C = A[M,256] . B[256,256]; K % 32 == 0;
 * work: >= 512*K floats (packed fp16 weight tiles: forward + dgrad pack).
 * rb200_tc_wgrad_h: dW[256,IN] += Z[n,256]^T . H[n,IN], IN % 32 == 0, IN <= 256.
 * amax: device float holding max|A| (or max|Z|), NULL = no operand scaling. */
int rb200_tc_gemm_h(const float* A, const float* B, float* C, int64_t M, int K, int mode, const float* amax,
                    float* work, rb200_stream_t stream);
int rb200_tc_wgrad_h(const float* Z, const float* H, float* dW, int64_t n, int IN, const float* amax,
                     rb200_stream_t stream);

/* probe hook of the fp16-split GEMM (csrc/tc_gemm_h.cu): 16 int64 per-role wait / work cycle counters of CTA 0 */
int rb200_tc_h_debug(void* prof16);

/* Persistent fused rollout (csrc/rollout_fused.cu): the whole T-step loop of one rank - MLP actor/critic inference,
 * Normal sampling, synthetic-env dynamics with auto-reset and the truncation bootstrap of rewards - in ONE kernel;
 * CTA c owns environments [c*E, c*E+E) for all T steps.  Replaces EnvWorker.interact / MultiStepRolloutWorker.generate
 * (rlinf/workers/env/env_worker.py:1059-1349, rlinf/workers/rollout/hf/huggingface_worker.py:678-781) for the
 * MLP-policy + device-resident env case; same buffers, row alignment and random streams as the per-kernel path
 * (rb200_mlp_sample + rb200_synth_env_step + rb200_mlp_value + rb200_bootstrap_rewards per step).
 * rb200_rollout_fused_supported() == 0 iff hidden == 256, obs_dim % 4 == 0, obs_dim <= 256, value_dim <= 1 and
 * B <= 32 * #SM.  `wt` (rb200_rollout_fused_wt_floats floats) holds the transposed hidden weights; refresh it with
 * rb200_rollout_fused_prepare() after every parameter update.  states row 0 is the current observation (input);
 * the device counters are read once (step t uses counter + t): add T to both afterwards (rb200_counter_add). */
int64_t rb200_rollout_fused_wt_floats(const rb200_mlp_layout* L);
int rb200_rollout_fused_supported(const rb200_mlp_layout* L, int B);
int rb200_rollout_fused_prepare(const rb200_mlp_layout* L, const float* params, float* wt, rb200_stream_t stream);
int rb200_rollout_fused(const rb200_mlp_layout* L, const float* params, const float* wt, const float* w_s,
                        const float* w_a, float* states, float* actions, float* logprobs, float* values,
                        float* rewards, uint8_t* terminations, uint8_t* truncations, uint8_t* dones,
                        float* final_obs, float* final_values, int32_t* elapsed, const float* policy_noise,
                        const float* env_noise, const uint64_t* counter_policy, const uint64_t* counter_env,
                        uint64_t seed_policy, uint64_t seed_env, uint64_t offset_policy, int T, int B,
                        int max_episode_steps, int auto_reset, int bootstrap_on_done, double gamma, double p_term,
                        double noise_std, double reward_noise_std, rb200_stream_t stream);

/* Persistent TENSOR-CORE rollout (csrc/rollout_tc.cu): same loop, buffers, row alignment and random streams as
 * rb200_rollout_fused, but every hidden layer of both towers and the env's s.W_s product run on tcgen05 (kind::f16,
 * 2-way fp16 split with fp32 accumulation, computed transposed: D[hidden unit, env] = W . X^T, 32 environments per CTA,
 * activations handed from TMEM to the next layer's operand tile in shared memory); the truncation bootstrap
 * V(final_obs) rides in 32 extra MMA columns of the next step's value tower.  The weights are streamed from a packed,
 * pre-split, pre-swizzled copy (rb200_rollout_tc_pack_bytes bytes, 16-byte aligned) that rb200_rollout_tc_prepare()
 * rebuilds from the flat parameters and the env's w_s [obs,obs] after every parameter update.
 * rb200_rollout_tc_supported() == 0 iff hidden == 256, value_dim == 1, act_dim <= 8, obs_dim % 32 == 0, obs_dim <= 128.
 * Replaces the same reference loop as rb200_rollout_fused (env_worker.py:1059-1349, huggingface_worker.py:678-781). */
int rb200_rollout_tc_supported(const rb200_mlp_layout* L, int B);
/* probe hook: ablation switches + 16 int64 wait-cycle counters of CTA 0 (flags = 0, prof16 = NULL: production kernel) */
int rb200_rollout_tc_debug(int flags, void* prof16);
int64_t rb200_rollout_tc_pack_bytes(const rb200_mlp_layout* L);
int rb200_rollout_tc_prepare(const rb200_mlp_layout* L, const float* params, const float* w_s, void* pack,
                             rb200_stream_t stream);
int rb200_rollout_tc(const rb200_mlp_layout* L, const float* params, const void* pack, const float* w_a,
                     float* states, float* actions, float* logprobs, float* values, float* rewards,
                     uint8_t* terminations, uint8_t* truncations, uint8_t* dones, float* final_obs,
                     float* final_values, int32_t* elapsed, const float* policy_noise, const float* env_noise,
                     const uint64_t* counter_policy, const uint64_t* counter_env, uint64_t seed_policy,
                     uint64_t seed_env, uint64_t offset_policy, int T, int B, int max_episode_steps, int auto_reset,
                     int bootstrap_on_done, double gamma, double p_term, double noise_std, double reward_noise_std,
                     rb200_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * SURVEY 8(f)3: token log-probabilities and entropies straight from the logits (csrc/logits.cu).
 * Replaces compute_logprobs_from_logits (rlinf/utils/utils.py:454-492, = -cross_entropy) and
 * compute_entropy_from_logits (:495-512, = -sum p log p over log_softmax) together with what their callers do first:
 * logits.div_(temperature) (workers/actor/fsdp_actor_worker.py:478) and the OpenVLA action-bin window, every logit
 * outside [v_lo, v_hi) treated as -inf (models/embodiment/openvla_oft/rlinf/openvla_oft_action_model.py:546-551).
 * logits: dtype 0 = fp32, 1 = bf16; row r lives at logits + (r / L) * batch_stride + (r % L) * row_stride (elements),
 * so the `[:, -L-1:-1, :]` slice of a [bsz, S, V] tensor needs no copy.  Forward reads every logit once and writes
 * logprob / entropy / lse [N] fp32 (entropy, lse nullable); backward reads the logits once more and writes
 *   dlogits_i = inv_T * (g_lp * (1[i = target] - p_i) - g_H * p_i * (log p_i + H)),  0 outside the window,
 * in the logits' dtype with its own strides d_batch_stride / d_row_stride (grad_logprob / grad_entropy nullable = zero). */
int rb200_logits_logprob_entropy_fwd(const void* logits, int dtype, const int64_t* target, int64_t N, int64_t L,
                                     int64_t batch_stride, int64_t row_stride, int V, int v_lo, int v_hi,
                                     double inv_temperature, float* logprob, float* entropy, float* lse,
                                     rb200_stream_t stream);
int rb200_logits_logprob_entropy_bwd(const void* logits, int dtype, const int64_t* target, int64_t N, int64_t L,
                                     int64_t batch_stride, int64_t row_stride, int V, int v_lo, int v_hi,
                                     double inv_temperature, const float* lse, const float* entropy,
                                     const float* grad_logprob, const float* grad_entropy, void* dlogits,
                                     int64_t d_batch_stride, int64_t d_row_stride, rb200_stream_t stream);

/* Value tower only: values [n,value_dim] = ValueHead(states). Used for the bootstrap value of
 * final observations (get_bootstrap_values, workers/rollout/hf/huggingface_worker.py:612-627). */
int rb200_mlp_value(const rb200_mlp_layout* L, const float* params, const float* wsplit,
                    const float* states, int64_t n, float* values, float* work, rb200_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Rollout-side helpers (device-resident rollout loop; replaces the per-chunk-step Channel hops with
 * CPU staging of env_worker.py:1087-1202 / huggingface_worker.py:678-704).
 * ---------------------------------------------------------------------------------------- */
/* Synthetic vector env step implementing the chunk_step contract (C = 1):
 *   s' = tanh(s.W_s + a.W_a + noise_std*eps), r = -|s'|^2/obs + reward_noise_std*eps_r,
 *   term ~ Bernoulli(p_term), trunc at max_episode_steps, auto-reset to N(0,I).
 * w_s [obs,obs] (in,out), w_a [act,obs]; noise: optional pre-drawn [B, 2*obs+2] (parity mode), else
 * Philox(seed, *counter_dev). final_obs = observation before the reset. */
int rb200_synth_env_step(const float* w_s, const float* w_a, const float* state, const float* action,
                         const float* noise, float* next_state, float* final_obs, float* reward,
                         uint8_t* term, uint8_t* trunc, uint8_t* done, int32_t* elapsed, float* z_scratch,
                         int B, int obs, int act, int max_episode_steps, int auto_reset, float p_term,
                         float noise_std, float reward_noise_std, uint64_t seed,
                         const uint64_t* counter_dev, rb200_stream_t stream);
/* env.chunk_step for num_action_chunks = C > 1 (rlinf/envs/maniskill/maniskill_env.py:327-375): C sub-steps of the
 * synthetic env WITHOUT auto-reset (sub-step c takes columns [c*act, (c+1)*act) of chunk_actions [B, C*act]), rewards
 * [B,C] of every sub-step, terminations / truncations / dones [B,C] all-zero except the last column = any over the
 * chunk, ONE auto-reset after the chunk (final_obs = observation before it).  noise: optional pre-drawn
 * [B, C*(obs+2) + obs] = per sub-step eps[obs] | eps_r | u_term, then the reset state; else Philox(seed, counter).
 * scratch: 3*B*obs floats. */
int rb200_synth_env_chunk_step(const float* w_s, const float* w_a, const float* state, const float* chunk_actions,
                               const float* noise, float* next_state, float* final_obs, float* rewards,
                               uint8_t* term, uint8_t* trunc, uint8_t* done, int32_t* elapsed, float* scratch,
                               int B, int obs, int act, int C, int max_episode_steps, int auto_reset, float p_term,
                               float noise_std, float reward_noise_std, uint64_t seed, const uint64_t* counter_dev,
                               rb200_stream_t stream);
/* strided form of rb200_bootstrap_rewards for the last sub-step of a chunk:
 * rewards[b*ld_rewards] += gamma * final_values[b*value_dim] where flag[b*ld_flag]  (env_worker.py:736-758) */
int rb200_bootstrap_rewards_ld(float* rewards, int ld_rewards, const float* final_values, int value_dim,
                               const uint8_t* flag, int ld_flag, int B, double gamma, rb200_stream_t stream);
/* rewards[b] += gamma * final_values[b*value_dim] where flag[b]  (compute_bootstrap_rewards,
 * workers/env/env_worker.py:736-758; flag = truncations ("standard") or dones ("always")). */
int rb200_bootstrap_rewards(float* rewards, const float* final_values, const uint8_t* flag, int B,
                            int value_dim, double gamma, rb200_stream_t stream);
/* counter_dev[0] += inc (device-side RNG step counter so captured CUDA graphs replay fresh noise). */
int rb200_counter_add(uint64_t* counter_dev, uint64_t inc, rb200_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Policy evaluation (EnvWorker.evaluate / env_evaluate_step, workers/env/env_worker.py:1374-1460, 557-620; episode
 * bookkeeping of ManiskillEnv, envs/maniskill/maniskill_env.py:232-391; compute_evaluate_metrics,
 * utils/metric_utils.py:372-420).
 * ---------------------------------------------------------------------------------------- */
/* Mean action only: mean [n,act_dim] = actor_mean(backbone(states)) (mode="eval", mlp_policy.py:268-271); no value
 * tower, no sampling, no log-prob.  Bit-identical to the mean the training head computes.  work: 3*n*256 floats
 * (rb200_mlp_fwd_scratch_floats(L, n) is enough). */
int rb200_mlp_mean(const rb200_mlp_layout* L, const float* params, const float* wsplit, const float* states, int64_t n,
                   float* mean, float* work, rb200_stream_t stream);
/* One chunk step of the synthetic eval env with per-episode bookkeeping.  Dynamics, noise layout [B, C*(obs+2) + obs]
 * and Philox streams of rb200_synth_env_step (C = 1) / rb200_synth_env_chunk_step (C > 1), the chunk counter being
 * `step`; success = the termination draw (u < p_term).  Per sub-step and env: ep_return += r (fp32), success_once |=
 * success, episode_len = elapsed; ignore_terminations drops the termination after recording.  After the chunk's last
 * sub-step one record row is written (rec_flags bit 0 = reported: done with auto_reset, else first done since the last
 * reset; bit 1 = success_once, bit 2 = success_at_end = success of the last sub-step; rec_return, rec_len), then done envs
 * auto-reset (state from the noise / Philox, elapsed, ep_return and success_once cleared).
 * state [B,obs] in/out; ep_flags [B] u8 bookkeeping (zero it with elapsed / ep_return at a full reset); scratch 3*B*obs. */
int rb200_synth_env_eval_step(const float* w_s, const float* w_a, float* state, const float* chunk_actions,
                              const float* noise, int32_t* elapsed, float* ep_return, uint8_t* ep_flags,
                              uint8_t* rec_flags, float* rec_return, int32_t* rec_len, float* scratch, int B, int obs,
                              int act, int C, int max_episode_steps, int auto_reset, int ignore_terminations,
                              float p_term, float noise_std, float reward_noise_std, uint64_t seed, uint64_t step,
                              rb200_stream_t stream);
/* out6 = {sum return, sum episode_len, sum return/episode_len (fp32 quotient), sum success_once, sum success_at_end,
 * count} over the n records with rec_flags bit 0, accumulated in fp64 in an order that depends on n only (identical
 * from run to run).  part: RB200_EVAL_MAX_PARTS * 6 doubles of scratch. */
#define RB200_EVAL_MAX_PARTS 512
int rb200_eval_metrics(const uint8_t* rec_flags, const float* rec_return, const int32_t* rec_len, int64_t n,
                       double* part, double* out6, rb200_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * a10 reward filter: replaces the filter_rewards block of EmbodiedFSDPActor._process_received_rollout_batch,
 *   workers/actor/embodied_fsdp_actor_worker.py:236-282 (= preprocess_embodied_batch, rlinf/utils/utils.py:803-830).
 *   rewards f32 [nc,B,C]; loss_mask bool [nc,B,C] or NULL; keep_env bool [B] (scratch/out);
 *   out_mask bool [nc,B,C] (= keep & loss_mask) or [nc,B,1] when loss_mask is NULL.
 * ---------------------------------------------------------------------------------------- */
int rb200_reward_filter(const float* rewards, const uint8_t* loss_mask, uint8_t* out_mask, uint8_t* keep_env,
                        int nc, int B, int C, int group_size, float lower, float upper,
                        rb200_stream_t stream);

/* a18 kl_penalty (rlinf/algorithms/utils.py:26-64): mode 0 k1/kl, 1 abs, 2 k2/mse, 3 k3/low_var_kl.
 * out[n] = penalty, d_logprob[n] (NULL ok) = d penalty / d logprob. */
int rb200_kl_penalty(const float* logprob, const float* ref_logprob, float* out, float* d_logprob, int64_t n,
                     int mode, rb200_stream_t stream);

/* a24 masked statistics for compute_rollout_metrics (rlinf/utils/metric_utils.py:422-506):
 * out4 = {count, sum, min, max} of x[i] over entries with mask[i / mask_div] != 0 (mask NULL = all). */
int rb200_masked_stats(const float* x, const uint8_t* mask, int64_t n, int64_t mask_div, double* out4,
                       rb200_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * SURVEY 8(f) rank 4 - the remaining advantage estimators of ADV_REGISTRY (rlinf/algorithms/advantages.py) and the
 * fp64 masked normalisations of rlinf/utils/distributed.py (a24).  Step-major [L,B] tensors, uint8 0/1 masks.
 * ---------------------------------------------------------------------------------------- */
/* masked_stats (distributed.py:942-954) and the three sums masked_normalization all-reduces (:903-933):
 * out3 = {count, sum x, sum x^2} over entries with mask != 0 (mask NULL = all), accumulated in fp64. */
int rb200_masked_moments(const float* x, const uint8_t* mask, int64_t n, double* out3 /*reset by the call*/,
                         rb200_stream_t stream);
/* Apply half, stats3 = (all-reduced) {count, sum, sumsq}:
 *  mode 0  masked_normalization(dim=None) :935-939  out = (x*mask - mean)/(sqrt(var[*n/(n-1)]) + eps), fp64 -> fp32
 *  mode 1  normalize_from_stats :957-965            out = (x - mean) * rsqrt(max(var,0) + 1e-5)
 *  mode 2  reinforce++ whitening, advantages.py:355-362   out = (x - mean) * rsqrt(max(var, eps)), biased var */
int rb200_masked_normalize(const float* x, const uint8_t* mask, float* out, int64_t n, const double* stats3,
                           int mode, double eps, int unbiased, rb200_stream_t stream);
/* "raw", advantages.py:410-438: adv[l,b] = scores[b] * mask[l,b]; stats3 (nullable) = {n, sum, sumsq} of the valid
 * entries for the optional safe_normalize-style normalisation (rb200_normalize, eps 1e-5). */
int rb200_raw_advantages(const float* scores /*[B]*/, const uint8_t* loss_mask /*[L,B]*/, float* adv /*[L,B]*/,
                         int L, int B, double* stats3, rb200_stream_t stream);
/* "reinpp", advantages.py:302-364: reward at the reference's eos index (its fliplr quirk reproduced), optional
 * -kl_beta * kl_penalty(logprob, ref_logprob) per token (kl_mode as rb200_kl_penalty), reverse cumulative sum over L
 * (fp64 accumulation as torch's CPU cumsum); stats3 = masked {n, sum, sumsq} of the returns for mode-2 whitening. */
int rb200_reinpp_returns(const float* rewards /*[B]*/, const uint8_t* loss_mask /*[L,B]*/, const float* logprob,
                         const float* ref_logprob, float* ret /*[L,B]*/, int L, int B, double kl_beta, int kl_mode,
                         double* stats3, rb200_stream_t stream);
/* "grpo_video", advantages.py:124-164: mode 0 = "frame", 1 = "video"; the mask is float in the reference (plain
 * product): pass it as mask_f32, or a 0/1 byte mask as mask_u8 (both NULL = no mask). */
int rb200_grpo_video_advantages(const float* rewards /*[S,B]*/, const float* mask_f32, const uint8_t* mask_u8,
                                float* adv /*[S,B]*/, int S, int B, int G, int mode, float eps, rb200_stream_t stream);
/* "grpo_dynamic", advantages.py:167-299: per-turn advantages [n] from per-turn rewards and the turn -> trajectory map
 * (int32, device); mode 0 = "trajectory", 1 = "turn".  The caller broadcasts over the sequence with the loss mask. */
int rb200_grpo_dynamic_turn_advantages(const float* rewards /*[n]*/, const int32_t* idx_to_traj /*[n]*/,
                                       float* turn_adv /*[n]*/, int n, int num_trajectories, int G, int mode,
                                       float eps, rb200_stream_t stream);
/* out = a - b, fp32 ("opd" advantages = teacher_logprobs - prev_logprobs, advantages.py:393). */
int rb200_sub(const float* a, const float* b, float* out, int64_t n, rb200_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* RLINF_B200_H */
