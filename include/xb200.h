/*
 * xb200.h — C ABI of the B200-native PPO hot path (libxb200.so, hand-written sm_100a CUDA kernels).
 *
 * This is the drop-in boundary.  The reference (fanliaoooo/xuanpolicy, a XuanCe 1.0.5 fork) is pure Python;
 * its own native-boundary idiom is a ctypes-loaded C library (xuance/environment/magent2/c_lib.py:10-23),
 * and that is how this library is bound (xuanpolicy_b200/_lib.py; INTEGRATION.md shows the reference-side stub).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the comment says "host";
 *   - every call only ENQUEUES work on `stream` (a cudaStream_t): no allocation, no synchronisation, so every
 *     call is CUDA-graph capturable;
 *   - return value: 0 = ok, > 0 = a cudaError_t, < 0 = an XB_E_* argument error.  Nothing throws.
 *   - rollout storage is TIME-MAJOR: element (step t, env e) of a per-transition scalar lives at [t*N + e];
 *     the reference's flat sample index k means (env = k / T, step = k % T)  (memory_tools.py:234).
 *   - observations are stored in rows of `XB_OBS_STRIDE` floats (16 B) so every row is one float4.
 *
 * Each entry point cites the reference code it replaces (paths relative to the reference root).
 */
#ifndef XB200_H
#define XB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define XB_VERSION 100
#define XB_OBS_STRIDE 4

#define XB_ENV_CARTPOLE 0 /* CartPole-v1: state (x, x_dot, theta, theta_dot), action int64 {0,1}, limit 500 */
#define XB_ENV_PENDULUM 1 /* Pendulum-v1: state (theta, theta_dot), action float32 torque, limit 200 */
#define XB_ENV_MOUNTAINCAR 2 /* MountainCar-v0: state (position, velocity), action int64 {0,1,2}, limit 200 */
#define XB_ENV_ACROBOT 3 /* Acrobot-v1: state (theta1, theta2, dtheta1, dtheta2), action int64 {0,1,2}, limit 500; obs 6 floats = TWO float4 per row */
/* MountainCar-v0 as the reference's make_envs builds it: MountainCar(Gym_Env), xuance/environment/gym/gym_env.py:50-83 —
 * observation = the last 4 frames (oldest first), 8 floats = TWO float4 per row; state fp64 [8][N] = (position, velocity,
 * frame t-3, frame t-2, frame t-1); same physics, action int64 {0,1,2}, limit 200 */
#define XB_ENV_MOUNTAINCAR_STACK4 4

#define XB_E_BADARG (-1)
#define XB_E_UNSUPPORTED (-2)
#define XB_E_DRIVER (-3)

#define XB_GAE_AUTO 0
#define XB_GAE_LDG 1 /* register-prefetch variant */
#define XB_GAE_TMA 2 /* cp.async.bulk.tensor + mbarrier ring variant */

typedef void* xb_stream_t; /* cudaStream_t */

int xb_version(void);
/* static string for a code returned by any entry point */
const char* xb_error_string(int code);

/* ------------------------------------------------------------------------------------------------------------
 * (1) Batched classic-control environments.  One thread per env, fp64 state in registers, every fp64 operation
 * individually rounded (__dadd_rn/__dmul_rn/__ddiv_rn, TU built with -fmad=false), correctly-rounded sin/cos.
 * Replaces  DummyVecEnv_Gym.reset / step_wait   xuance/environment/gym/gym_vec_env.py:177-212
 *           Gym_Env.reset / step                xuance/environment/gym/gym_env.py:36-49
 *           gym 0.26.2 CartPoleEnv / PendulumEnv / TimeLimit / np_random (third party, restated: SURVEY.md App. A/B)
 *
 * state     fp64 [S][N] (SoA; S = 4 CartPole / Acrobot, 2 Pendulum / MountainCar, 8 MountainCar 4-frame stack)
 * obs       f32 [N][4] rows (one float4 per env); Acrobot-v1: [N][8] (two float4: cos t1, sin t1, cos t2, sin t2 | dt1, dt2, 0, 0);
 *           MountainCar 4-frame stack: [N][8] (p, v of frames t-3, t-2 | t-1, t)
 * rng       u64  [4][N] (SoA) numpy PCG64: state_hi, state_lo, inc_hi, inc_lo
 * elapsed   i32  [N]    TimeLimit._elapsed_steps == Gym_Env._episode_step
 * ep_score  fp64 [N]    Gym_Env._episode_score
 * ---------------------------------------------------------------------------------------------------------- */

/* n_draws consecutive env.reset() calls per env (xuance does 2 before the first step: gym_env.py:19 and
 * runner_basic.py:12); zeroes elapsed/ep_score; writes the observation of the last draw to obs [N][4]. */
int xb_env_reset(int env_kind, double* state, uint64_t* rng, int32_t* elapsed, double* ep_score, float* obs,
                 int n_draws, int64_t N, xb_stream_t stream);

/* One vector step with auto-reset.
 * actions      int64 [N] (CartPole) or float32 [N] (Pendulum)
 * obs          f32 [N][4]  observation after the step: the TERMINAL observation for finished envs (buf_obs, :210)
 * next_obs     f32 [N][4]  nullable; obs with finished envs replaced by their reset observation (what the policy sees next)
 * rew          f32 [N];  term, trunc  u8 [N]
 * reset_obs    f32 [N][4]  written only where term|trunc (infos[e]["reset_obs"], :207-209)
 * ep_step_out  i32 [N], ep_score_out fp64 [N]   infos[e]["episode_step"/"episode_score"] of this step (gym_env.py:45-48)
 * ep_stats     fp64 [3] nullable: running (finished episodes, sum of their scores, sum of their lengths), the
 *              totals behind the per-episode log lines of ppoclip_agent.py:102-109 (atomically accumulated).
 */
int xb_env_step(int env_kind, double* state, uint64_t* rng, int32_t* elapsed, double* ep_score, const void* actions,
                float* obs, float* next_obs, float* rew, uint8_t* term, uint8_t* trunc, float* reset_obs,
                int32_t* ep_step_out, double* ep_score_out, double* ep_stats, int max_episode_steps, int64_t N,
                xb_stream_t stream);

/* Test hook: the kernel's correctly-rounded sin/cos on an array (fp64 [n] each). */
int xb_sincos_f64(const double* x, double* s, double* c, int64_t n, xb_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * (2) Device-resident rollout buffer.  Replaces DummyOnPolicyBuffer.store / store_element
 *     xuance/common/memory_tools.py:39-54,196-204  (memory[:, ptr] = data).
 * Writes row t of the time-major arrays (the *_row pointers already point at row t).  float4 stores for obs.
 * act: int64 [N] (act_is_i64=1, stored as float32 like the reference, memory_tools.py:173) or float32 [N][act_dim].
 * term/trunc are u8 in, term is stored as float32 0/1 (memory_tools.py:177), trunc as u8 (segment-end flag).
 * rew_std: nullable device scalar; when given, rewards are stored as clip(rew / *rew_std, +-rew_clip)
 *          (Agent._process_reward, xuance/torch/agents/agent.py:118-123).
 * obs_vec: float4s per observation row: 1 (obs_dim <= 4, XB_OBS_STRIDE floats) or 2 (wide rows of 8 floats for
 *          obs_dim 5..8, e.g. Acrobot-v1's 6); the gathers below infer the same width from obs_dim.
 * ---------------------------------------------------------------------------------------------------------- */
int xb_store(const float* obs, const void* act, int act_is_i64, int act_dim, const float* rew, const float* val,
             const uint8_t* term, const uint8_t* trunc, const float* logp, float* obs_row, float* act_row,
             float* rew_row, float* val_row, float* term_row, uint8_t* trunc_row, float* logp_row,
             const float* rew_std, float rew_clip, int obs_vec, int64_t N, xb_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * (3) GAE / discounted-return reverse scan over T, parallel over envs, + advantage statistics.
 * Replaces DummyOnPolicyBuffer.finish_path (memory_tools.py:206-229) for ALL envs and ALL path segments of a
 * rollout at once (batched form, SURVEY.md App. D) and discount_cumsum (common_tools.py:199-200).
 *   rew, val, term   f32 [T][N]        trunc  u8 [T][N] nullable (segment ends that are not terminals)
 *   boot             f32 [T][N] nullable: V(terminal obs) where trunc is set (read only there)
 *   boot_last        f32 [N]           V(next obs) after the last step
 *   adv, ret         f32 [T][N] out    stats fp64 [2] nullable: (sum adv, sum adv^2) over the whole rollout
 * The recurrence is carried in fp64 registers and rounded once on store.
 * ---------------------------------------------------------------------------------------------------------- */
int xb_gae(const float* rew, const float* val, const float* term, const uint8_t* trunc, const float* boot,
           const float* boot_last, float* adv, float* ret, double* stats, int64_t T, int64_t N, double gamma,
           double lam, int use_gae, int variant, xb_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * (4a) Minibatch gather.  Replaces DummyOnPolicyBuffer.sample / sample_batch (memory_tools.py:57-72,231-245).
 * idx int64 [B] are the reference's flat indices (env = k / T, step = k % T).
 * xb_gather_obs: obs rows -> obs_out [B][obs_dim] (the MLP input) and, if stats != NULL, the minibatch
 *   advantage statistics stats fp64 [2] = (sum, sum of squares) (np.mean/np.std at memory_tools.py:241-242).
 * xb_gather_batch: every field sample() returns, densely (compat path); any output may be NULL.
 * xb_normalize_adv: adv[i] = (adv[i] - mean) / (std + 1e-8) from stats over `count` samples, in place.
 * ---------------------------------------------------------------------------------------------------------- */
int xb_gather_obs(const int64_t* idx, int64_t B, int64_t T, int64_t N, const float* b_obs, int obs_dim,
                  const float* b_adv, float* obs_out, double* stats, xb_stream_t stream);
int xb_gather_batch(const int64_t* idx, int64_t B, int64_t T, int64_t N, const float* b_obs, int obs_dim,
                    const float* b_act, int act_dim, const float* b_ret, const float* b_val, const float* b_adv,
                    const float* b_logp, float* obs_out, float* act_out, float* ret_out, float* val_out,
                    float* adv_out, float* logp_out, double* stats, xb_stream_t stream);
int xb_normalize_adv(float* adv, const double* stats, int64_t count, int64_t B, xb_stream_t stream);
/* Packed transition records (act_dim == 1): once per rollout, after xb_gae, xb_pack_records builds one 32-byte,
 * sector-aligned record {obs[4], act, old_logp, adv, ret} per transition (rec f32 [T*N][8]); xb_gather_records then
 * reads ONE DRAM sector per sample instead of one per field and emits obs_out [B][obs_dim], scal_out f32 [B][4] =
 * {act, old_logp, adv, ret} and the minibatch advantage statistics.  Same replaced code as xb_gather_batch. */
int xb_pack_records(const float* b_obs, const float* b_act, const float* b_logp, const float* b_adv,
                    const float* b_ret, float* rec, int64_t TN, xb_stream_t stream);
int xb_gather_records(const int64_t* idx, int64_t B, int64_t T, int64_t N, const float* rec, int obs_dim,
                      float* obs_out, float* scal_out, double* stats, xb_stream_t stream);
/* xb_gather_records fused with the MLP's first layer (Basic_MLP: Linear(obs_dim, H) + LeakyReLU,
 * xuance/torch/representations/mlp.py:40-51; same arithmetic as xb_mlp_trunk_fwd, bit-identical output):
 * additionally writes h1 f32 [B][H] = leaky_relu(obs W0^T + b0), so the gathered rows feed the layer from registers and the
 * latency-bound gather hides behind the store-bound layer — one launch instead of two per update. */
int xb_gather_trunk_fwd(const int64_t* idx, int64_t B, int64_t T, int64_t N, const float* rec, int obs_dim, const float* W0,
                        const float* b0, float slope, int H, float* obs_out, float* scal_out, double* stats, float* h1,
                        uint32_t* h1_signs, xb_stream_t stream);
/*   h1_signs (nullable, xb_gather_trunk_fwd and xb_mlp_trunk_fwd; H a multiple of 128): u32 [B][H / 32] sign words of h1, four
 *   per 128-feature slice s — bit l of word 4 s + e = (h1[b][128 s + 4 l + e] > 0), the order the warp ballots produce them —
 *   for xb_dense_dgrad's epilogue mask. */

/* ------------------------------------------------------------------------------------------------------------
 * (4b) PPO-Clip loss forward + backward, fused with the gather of the per-transition scalars.
 * Replaces the loss arithmetic and its autograd backward in PPOCLIP_Learner.update
 *   xuance/torch/learners/policy_gradient/ppoclip_learner.py:33-44, and Categorical/Normal log_prob+entropy
 *   xuance/torch/utils/distributions.py:51-55,83-87  (closed forms: SURVEY.md App. C).
 * If idx != NULL, act/ret/adv/old_logp/val_old are the rollout arrays ([T][N], act [T][N][A]) read through idx;
 * if idx == NULL they are dense [B] minibatch arrays (compat path: update(obs, act, ret, value, adv, old_logp)).
 *   adv_stats fp64[2] nullable: (sum, sumsq) of the advantages of the (global) minibatch of adv_count samples;
 *             when given, advantages are normalised on the fly (x-mean)/(std+1e-8).
 *   value_clip <= 0 : plain MSE value loss (the reference).  > 0: max((v-R)^2, (v_old+clip(v-v_old,+-c)-R)^2)
 *             (opt-in, formula of xuance/torch/learners/multi_agent_rl/mappo_learner.py:78-87; needs val_old).
 *   clip_range <= 0 selects the A2C / PG surrogate instead: a_loss = -(adv * log_prob).mean() (old_logp unused, may be
 *             NULL) — A2C_Learner.update a2c_learner.py:24-35; PG_Learner.update pg_learner.py:19-27 (adv = returns, vf_coef = 0).
 *   inv_batch = 1 / (global minibatch size): the mean() of the reference.
 *   stride: element stride (in floats) of the dense act/ret/adv/old_logp/val_old arrays when idx == NULL — 1 for
 *             plain [B] arrays, 4 for the packed float4 {act, old_logp, adv, ret} rows xb_gather_records emits
 *             (pass base+0, base+3, base+2, base+1); must be 1 with idx, and with act_dim > 1.
 * Outputs: gradients of  L = a_loss - ent_coef*entropy + vf_coef*c_loss  w.r.t. the network outputs, and
 *   scalars fp64 [8] = sums over THIS call's samples of {min-surrogate, value loss term, entropy, v_pred,
 *   clipped-ratio count, 0, 0, 0} (overwritten; summed in a fixed order, so bit-reproducible run to run).
 * Gaussian: logstd f32 [A] is shared by the batch; dlogstd_acc fp64 [A] (overwritten) receives its gradient.
 * ---------------------------------------------------------------------------------------------------------- */
int xb_ppo_loss_categorical(const int64_t* idx, int64_t B, int64_t T, int64_t N, const float* logits, int A,
                            const float* v_pred, const float* act, const float* ret, const float* adv,
                            const float* old_logp, const float* val_old, const double* adv_stats, int64_t adv_count,
                            float clip_range, float vf_coef, float ent_coef, float value_clip, float inv_batch,
                            int64_t stride, float* dlogits, float* dv, double* scalars, xb_stream_t stream);
int xb_ppo_loss_gaussian(const int64_t* idx, int64_t B, int64_t T, int64_t N, const float* mu, const float* logstd,
                         int A, const float* v_pred, const float* act, const float* ret, const float* adv,
                         const float* old_logp, const float* val_old, const double* adv_stats, int64_t adv_count,
                         float clip_range, float vf_coef, float ent_coef, float value_clip, float inv_batch,
                         int64_t stride, float* dmu, double* dlogstd_acc, float* dv, double* scalars, xb_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * (4b) Losses that carry the OLD ACTION DISTRIBUTION (SURVEY.md §8 row f3: PPO-KL, PPG).  Forward + backward
 * w.r.t. the network outputs of
 *     L = surr_coef*a_loss + kl_w*mean KL(new||old) - ent_coef*mean H + vf_coef*mean (v-R)^2
 *         + aux_coef*mean (aux_v - stopgrad(v))^2
 * with  ratio = exp(log_prob(act) - old_dist.log_prob(act)),  a_loss = -mean(ratio*adv) (clip_range <= 0) or the
 * clipped surrogate (clip_range > 0), kl_w = kl_coef * (*kl_coef_dev if given).  Replaces
 *   PPOKL_Learner.update          xuance/torch/learners/policy_gradient/ppokl_learner.py:26-37
 *   PPG_Learner.update_policy     xuance/torch/learners/policy_gradient/ppg_learner.py:27-39   (surr 1, ent)
 *   PPG_Learner.update_critic     ppg_learner.py:58-60                                        (vf 1 only)
 *   PPG_Learner.update_auxiliary  ppg_learner.py:75-80                                        (kl_beta, vf 1, aux 1)
 *   CategoricalDistribution / DiagGaussianDistribution.kl_divergence   xuance/torch/utils/distributions.py:63-66,97-100
 *   merge_distributions           xuance/torch/utils/operations.py:75-92 (the caller passes the merged parameters)
 * All per-sample inputs are dense [B] minibatch arrays.  aux_v / daux are nullable (required when aux_coef != 0).
 * Gaussian: KL is averaged over B*A elements like the reference's `.mean()` of the element-wise Normal KL;
 *   old_std is [B][A] (old_std_per_sample = 1) or one shared row [A] (0).
 * scalars fp64 [8] (zeroed by the call) = sums of {surrogate, (v-R)^2, entropy, v_pred, clipped-ratio count,
 *   KL (summed over A), (aux_v-v)^2, 0}.
 * xb_kl_coef_adapt: the adaptive coefficient of ppokl_learner.py:39-43 on the device, from scalars[5]/count
 *   (count = B for Categorical, B*A for Gaussian): > 1.5*target -> x2, < 0.5*target -> /2, clip to [0.1, 20].
 * ---------------------------------------------------------------------------------------------------------- */
int xb_dist_loss_categorical(int64_t B, const float* logits, const float* old_logits, int A, const float* v_pred,
                             const float* aux_v, const float* act, const float* ret, const float* adv,
                             float clip_range, float surr_coef, float kl_coef, const float* kl_coef_dev, float vf_coef,
                             float ent_coef, float aux_coef, float inv_batch, float* dlogits, float* dv, float* daux,
                             double* scalars, xb_stream_t stream);
int xb_dist_loss_gaussian(int64_t B, const float* mu, const float* logstd, const float* old_mu, const float* old_std,
                          int old_std_per_sample, int A, const float* v_pred, const float* aux_v, const float* act,
                          const float* ret, const float* adv, float clip_range, float surr_coef, float kl_coef,
                          const float* kl_coef_dev, float vf_coef, float ent_coef, float aux_coef, float inv_batch,
                          float* dmu, double* dlogstd_acc, float* dv, float* daux, double* scalars, xb_stream_t stream);
int xb_kl_coef_adapt(const double* scalars, float* kl_coef_dev, float target_kl, int64_t count, xb_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Action sampling fused with log-prob (after the actor GEMM).  Replaces dists.stochastic_sample()+log_prob in
 * PPOCLIP_Agent._action (ppoclip_agent.py:50-57; distributions.py:57-58,89-90).  Philox4x32-10, counter-based:
 * stream position = (*counter_dev + offset, env index), so a captured graph replays with fresh numbers once
 * xb_counter_add has advanced the device counter.
 * ---------------------------------------------------------------------------------------------------------- */
int xb_sample_categorical(const float* logits, int A, uint64_t seed, const uint64_t* counter_dev, uint64_t offset,
                          int64_t* act_out, float* logp_out, int64_t N, xb_stream_t stream);
int xb_sample_gaussian(const float* mu, const float* logstd, int A, uint64_t seed, const uint64_t* counter_dev,
                       uint64_t offset, float* act_out, float* logp_out, int64_t N, xb_stream_t stream);
int xb_counter_add(uint64_t* counter_dev, uint64_t inc, xb_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Optimiser tail of PPOCLIP_Learner.update (ppoclip_learner.py:45-51) over ONE flat fp32 parameter/gradient
 * buffer: global-L2-norm clip (torch.nn.utils.clip_grad_norm_: scale = min(1, max_norm/(norm+1e-6))), Adam
 * (torch.optim.Adam semantics, eps inside the sqrt denominator, bias correction from *step_dev) and the
 * LinearLR factor  lr = lr0 * (1 + (end-1) * min(it, total)/total), all on device so it is graph-replayable.
 *   state: step_dev i64[1] (number of updates done so far; incremented by the call)
 *   grad_scale multiplies the gradient first (1/world_size after a sum-allreduce).
 *   workspace fp64 [8 + 1024] scratch, ZERO-INITIALISED once by the caller.  lr_out / gnorm_out f32[1] nullable:
 *   the lr used by this step and the pre-clip gradient norm.
 * ---------------------------------------------------------------------------------------------------------- */
int xb_clip_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                      int64_t* step_dev, float lr0, float lr_end_factor, int64_t lr_total_iters, float beta1,
                      float beta2, float eps, float max_norm /* <=0: no clip */, float grad_scale,
                      double* workspace, float* lr_out, float* gnorm_out, xb_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Device-side RunningMeanStd + observation / reward normalisation (per-step path when use_obsnorm / use_rewnorm).
 * Replaces RunningMeanStd.update/update_from_moments (xuance/common/statistic_tools.py:63-112),
 * Agent._process_observation/_process_reward (xuance/torch/agents/agent.py:104-123) and the per-env discounted
 * return tracker (ppoclip_agent.py:87,91-92).
 *   obs normaliser state: fp64 [9] = mean[4], var[4], count (mean/var hold float32-rounded values)
 *   xb_moments4      sums fp64 [2D + 1] = column sums (D), column sums of squares (D), N of x f32 [N][D], D = row_floats
 *                    (4, or 8 for wide rows: the first observations of an env-sharded agent, `obs_rms.update(obs)` of
 *                    ppoclip_agent.py:62 with the sums exchanged across ranks in between: the analogue of mpi_mean :6-17);
 *                    xb_rms_normalize takes the 4-float form
 *   xb_rms_normalize merges `sums` into state_in (Chan), writes the merged state to state_out (!= state_in) and
 *                    out = clip((x - mean) / (sqrt(var) + 1e-8), +-clip)     f32 [N][4]; lanes >= dim give 0.
 *                    Rows [0, n_merged_rows) use the merged statistics, rows beyond use state_in unchanged (the
 *                    previous step's terminal observations, normalised as ppoclip_agent.py:99 saw them);
 *                    n_merged_rows == 0 normalises without updating (sums may be NULL).
 *   xb_returns_track returns[i] = (1-term)*gamma*returns[i] + rew[i] (fp64 [N]; mask_terminal = 0 drops the (1-term) factor:
 *                    the A2C agent's tracker, a2c_agent.py:85); finished envs add (R, R^2, 1) to sums fp64 [3]
 *                    and restart at 0
 *   xb_rms_merge_scalar merges those sums into the return normaliser state fp64 [3] = (mean, var, count) and
 *                    publishes rew_std = clip(sqrt(var), 0.1, 100), the divisor xb_store applies to rewards
 * workspace: fp64 [8 + 8*1184], word 0 ZERO-INITIALISED once by the caller (one workspace per call site).
 * ---------------------------------------------------------------------------------------------------------- */
int xb_moments4(const float* x, int row_floats, double* sums, double* workspace, int64_t N, xb_stream_t stream);
int xb_rms_normalize(const float* x, int dim, const double* sums, const double* state_in, double* state_out,
                     float clip, float* out, int64_t N, int64_t n_merged_rows, xb_stream_t stream);
int xb_returns_track(double* returns, const float* rew, const uint8_t* term, const uint8_t* trunc, double gamma, int mask_terminal,
                     double* sums, double* workspace, int64_t N, xb_stream_t stream);
int xb_rms_merge_scalar(const double* sums, double* state, float* rew_std, xb_stream_t stream);
/* The same statistics for the fused path, where xb_rollout_step carries the merges (see there): observation rows of
 * row_floats = 4 or 8 floats, state fp64 [2*row_floats + 1] = mean, var, count.
 *   xb_rms_apply        out = normalise(x) with state_new for rows [0, n_new_rows) and state_old for the rest (no merge):
 *                       the policy input when the MLP runs in torch (xb_mlp_fwd_from_obs normalises by itself)
 *   xb_rms_update_rows  state_out = state_in merged with the batch moments of x [N rows] (`obs_rms.update(obs)`): used once,
 *                       for the very first observations.  partials fp64 [148 * 20], ticket u32 [1] zero-initialised. */
int xb_rms_apply(const float* x, int row_floats, int dim, const double* state_new, const double* state_old, int64_t n_new_rows,
                 float clip, float* out, int64_t N, xb_stream_t stream);
int xb_rms_update_rows(const float* x, int row_floats, int dim, int64_t N, const double* state_in, double* state_out,
                       double* partials, uint32_t* ticket, xb_stream_t stream);
/*   xb_rms_merge_sums   env-sharded form (mpi_moments + update_from_moments, statistic_tools.py:6-32,101-112): sums fp64 [n]
 *                       = the cross-rank totals of one step, n = 2D + 4 = 12 or 20 for D = 4 or 8 floats per row (layout of
 *                       xb_moments4 + the three return sums); obs_state_out = obs_state_in merged with them (nullable pair,
 *                       state fp64 [2D + 1], dim <= D), ret_state merged in place and rew_std republished (nullable pair). */
int xb_rms_merge_sums(const double* sums, int n, const double* obs_state_in, double* obs_state_out, int dim, double* ret_state,
                      float* rew_std, xb_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Non-GEMM half of the MLP backward (the GEMMs stay in torch/cuBLAS): LeakyReLU' fused with the bias gradient.
 *   dz[b,h] = dy[b,h] * (y[b,h] > 0 ? 1 : slope);   dbias[h] = sum_b dz[b,h]        (dz may alias dy)
 * Replaces torch autograd's leaky_relu_backward + sum(0) pair in every Linear+LeakyReLU block
 * (xuance/torch/utils/layers.py:15-21).  H % 4 == 0, H <= 1024.
 * workspace: fp32 [4 + 592*H], word 0 ZERO-INITIALISED once by the caller.
 * ---------------------------------------------------------------------------------------------------------- */
int xb_act_bias_bwd(const float* dy, const float* y, float slope, float* dz, float* dbias, float* workspace,
                    int64_t B, int H, xb_stream_t stream);
/* Narrow output heads (A <= 4 columns; bandwidth-bound matrix-vector work): the last Linear of the actor / critic.
 *   xb_head_fwd      out[b,a] = h[b,:] . W[a,:] + bias[a]                                       h f32 [B][H], W f32 [A][H]
 *   xb_head_bwd_act  the head's backward fused with the hidden layer's LeakyReLU backward and bias gradient:
 *                    dz[b,:] = (sum_a dout[b,a] W2[a,:]) * lrelu'(y[b,:]),  db1 = colsum(dz),
 *                    dW2[a,:] = sum_b dout[b,a] y[b,:],  db2[a] = sum_b dout[b,a]
 * Replace F.linear + its autograd (outer product, gemv, three reductions) for categorical.py:31,54 / gaussian.py:23,47.
 * workspace: fp32 [4 + 148*((1+A)*H + 4)], word 0 ZERO-INITIALISED once by the caller. */
int xb_head_fwd(const float* h, const float* W, const float* bias, float* out, int64_t B, int H, int A,
                xb_stream_t stream);
int xb_head_bwd_act(const float* dout, const float* y, const float* W2, float slope, float* dz, float* db1, float* dW2,
                    float* db2, float* workspace, int64_t B, int H, int A, xb_stream_t stream);
/* Forward epilogue of the same block: y[b,h] = leaky_relu(y[b,h] + bias[h]) in place, after a bias-free cuBLAS mm. */
int xb_bias_act_fwd(float* y, const float* bias, float slope, int64_t B, int H, xb_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * One vector step of the device-resident rollout in ONE launch: xb_sample_* + xb_env_step + xb_store fused per env
 * (PPOCLIP_Agent._action ppoclip_agent.py:50-57; DummyVecEnv_Gym.step_wait gym_vec_env.py:200-212;
 * DummyOnPolicyBuffer.store memory_tools.py:196-204).  CartPole-v1 / MountainCar-v0 (both forms) / Acrobot-v1: act_param = logits
 * [N][2] / [N][3] / [N][3], act_out int64 [N]; wide-row envs (Acrobot, MountainCar stack): x_in / obs / obs_row are [N][8];
 * Pendulum-v1: act_param = mu [N][1], logstd [1], act_out f32 [N].  x_in = the observations the action was computed
 * from (stored as the transition's obs); all other arguments as in xb_env_step / xb_store.  Physics and store are
 * bit-identical to the three separate calls; the sampled action may differ from xb_sample_* in the last ulp of the
 * transcendental functions (this translation unit is built without FMA contraction).
 * boot_src / boot_row (nullable pair, f32 [N]): V(terminal observation of the PREVIOUS step) copied into the previous
 * rollout row's bootstrap values — the value the reference obtains with a full-batch forward per finished env
 * (ppoclip_agent.py:98-100) — so the step needs no separate copy launch.
 * trig_cache (nullable, fp64 [3][N], initialise the first row to NaN): Pendulum's observation (cos, sin of the new theta)
 * is the next step's dynamics input; the row (theta, sin, cos) is reused when its key equals the current theta bit for
 * bit, recomputed otherwise — the values are identical either way (correctly-rounded pure functions of theta).
 * Running statistics carried by the same launch (stat_partials != NULL; csrc/normalize.cuh StepStats) — replaces, per step,
 * `obs_rms.update(obs)` of the next loop iteration, the per-env return tracker and `ret_rms.update` (ppoclip_agent.py:62,
 * 87-92; statistic_tools.py:63-112) and their four launches (xb_moments4, xb_rms_normalize, xb_returns_track,
 * xb_rms_merge_scalar):
 *   obs_state_in / obs_state_out (nullable pair, fp64 [2D+1], D = floats per obs row, DIFFERENT buffers): x_in holds RAW
 *     observations, the stored row is normalise(x_in, obs_state_in); obs_state_out = obs_state_in merged (Chan, float32) with
 *     the batch moments of next_obs; obs_dim real floats per row, obs_clip the clipping range;
 *   ret_state (nullable, fp64 [3]) with rew_std_io (f32 [1]: read as this step's reward divisor — pass the same pointer as
 *     rew_scale — and rewritten for the next step) and returns (fp64 [N] tracker), gamma, mask_terminal (1 = PPO, 0 = A2C);
 *   stat_partials fp64 [grid * 20] / stat_ticket u32 [1] (zero-initialised once): per-CTA sums, added in CTA order by the
 *     last CTA (deterministic);
 *   stat_sums_out (nullable, fp64 [2D + 4], env-sharded form): this rank's totals (sum x[D], sum x^2[D], N, sum R, sum R^2,
 *     n finished) are written there INSTEAD of being merged (obs_state_out / ret_state unused); exchange them across ranks
 *     (xb_peer_allreduce_merge, or xb_peer_allreduce_f64 and xb_rms_merge_sums).
 * ---------------------------------------------------------------------------------------------------------- */
int xb_rollout_step(int env_kind, const float* act_param, const float* logstd, const float* val, uint64_t seed,
                    const uint64_t* counter_dev, uint64_t offset, double* state, uint64_t* rng, int32_t* elapsed,
                    double* ep_score, float* obs, float* next_obs, float* rew, uint8_t* term, uint8_t* trunc,
                    float* reset_obs, int32_t* ep_step_out, double* ep_score_out, double* ep_stats,
                    int max_episode_steps, const float* x_in, void* act_out, float* logp_out, float* obs_row,
                    float* act_row, float* rew_row, float* val_row, float* term_row, uint8_t* trunc_row, float* logp_row,
                    const float* rew_scale, float rew_clip, const float* boot_src, float* boot_row, double* trig_cache,
                    const double* obs_state_in, double* obs_state_out, int obs_dim, float obs_clip, double* ret_state,
                    float* rew_std_io, double* returns, double gamma, int mask_terminal, double* stat_partials,
                    uint32_t* stat_ticket, double* stat_sums_out, int64_t N, xb_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * One vector step of the evaluation loop in ONE launch.  Replaces the body of PPOCLIP_Agent.test (ppoclip_agent.py:113-165):
 * `dist.stochastic_sample()`, `envs.step(acts)` with auto-reset (gym_vec_env.py:200-212), `scores.append(infos[i]
 * ["episode_score"])` for every finished env, and the `obs_rms.update(obs)` of the next loop iteration (:126).
 *   act_param / logstd  policy outputs as in xb_rollout_step; the action is drawn with Philox keyed by *key (u64 [1]) at
 *                       counter (env, *step); the launch adds 1 to *step (u64 [1]).  act_tape (nullable): the actions are also
 *                       written to row *step of [tape_steps][N] (int64, Pendulum float32) while *step < tape_steps.
 *   state .. ep_score   env state as in xb_env_step; next_obs f32 [N][4] or [N][8] receives the observation the policy acts
 *                       on next (reset observation for finished envs); trig_cache as in xb_rollout_step.
 *   scores / count      episode queue fp64 [cap] and its length (int64 [1]): the final ep_score of every env that finished in
 *                       this step is appended in env order (an ordered multi-CTA compaction, independent of CTA scheduling).
 *                       cap >= test_episode + N - 1 holds every score the loop can produce.
 *   test_episode        int64 [1].  Stop rule: a launch that finds *count >= *test_episode changes nothing.
 *   obs_state           nullable, fp64 [2D+1] (D = floats per obs row): merged IN PLACE with the moments of next_obs when
 *                       the new count is still below *test_episode (the loop goes round again); obs_state_cand fp64 [2D+1] is
 *                       the merge's scratch.  obs_dim real floats per row.
 *   partials fp64 [20 * ceil(N / 32)], workspace u64 [2 + ceil(N / 32)]: scratch, zero-initialised once, reset by every launch.
 * Physics bit-identical to xb_env_step.
 * ---------------------------------------------------------------------------------------------------------- */
int xb_eval_step(int env_kind, const float* act_param, const float* logstd, const uint64_t* key, uint64_t* step, double* state,
                 uint64_t* rng, int32_t* elapsed, double* ep_score, float* next_obs, double* trig_cache, int max_episode_steps,
                 void* act_tape, int64_t tape_steps, double* scores, int64_t* count, const int64_t* test_episode, int64_t cap,
                 double* obs_state, double* obs_state_cand, int obs_dim, double* partials, uint64_t* workspace, int64_t N,
                 xb_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Dense layers of the policy/value MLP at large batch on the tcgen05 tensor cores with fp32-level accuracy
 * ("3xTF32": x = hi + lo split, three kind::tf32 MMAs per k-step, fp32 accumulation in TMEM; csrc/dense_tc.cu).
 * Replace the cuBLAS SIMT sgemm calls torch issues for Basic_MLP / ActorNet / CriticNet forward
 * (xuance/torch/representations/mlp.py:49-51, policies/categorical.py:26-32,48-54, policies/gaussian.py:17-24,41-48)
 * and for their autograd backward under PPOCLIP_Learner.update (ppoclip_learner.py:47).
 * All matrices fp32 row-major, 16-byte aligned.  N (layer width) in {64, 128, 256}; K % 32 == 0, 32 <= K <= 256.
 *   xb_dense_split_weights  W [N][K] -> hi, lo [N][K] (TF32-representable hi, exact remainder lo) and, when thi != NULL,
 *                           their transposes into thi/tlo [K][ldt] at column offset toff (the dgrad operand; actor and
 *                           critic layers are concatenated along the reduction dimension).
 *   xb_dense_fwd            Y[M][N] = leaky_relu(X[M][K] . W^T + bias);  optionally the narrow head that follows it:
 *                           head_out[M][n_head] = Y . head_w[n_head][N]^T + head_b   (n_head in {0, 1, 2}).
 *                           b_resident != 0 keeps the whole weight operand in shared memory when it fits.
 *                           Y == NULL (with n_head > 0): only the head outputs are produced (no activation store).
 *   xb_dense_dgrad          dZ1[M][N] = ([dz0 | dz1] . [W0 ; W1]) * leaky'(H1)   with the A operand generated on the fly:
 *                           dz_s[r][k] = (sum_j dout_s[r][j] w2_s[j][k]) * leaky'(Y_s[r][k])   (s = actor, critic),
 *                           i.e. the backward of  H1 -> {Linear+LeakyReLU -> head}_s  without materialising dz_s.
 *                           Wthi/Wtlo: [N][K0+K1] from xb_dense_split_weights.  Y1 == NULL drops the second source.
 * ---------------------------------------------------------------------------------------------------------- */
int xb_dense_split_weights(const float* W, int N, int K, float* hi, float* lo, float* thi, float* tlo, int ldt,
                           int toff, xb_stream_t stream);
/*   xb_dense_split_weights2 both hidden layers (actor W0, critic W1, each [N][K]) in one launch; thi/tlo [K][2N] receive the
 *                           transposes side by side (W0^T | W1^T). */
int xb_dense_split_weights2(const float* W0, float* hi0, float* lo0, const float* W1, float* hi1, float* lo1, int N, int K,
                            float* thi, float* tlo, xb_stream_t stream);
int xb_dense_fwd(const float* X, int64_t M, int K, const float* Whi, const float* Wlo, int N, const float* bias,
                 float slope, float* Y, const float* head_w, const float* head_b, int n_head, float* head_out,
                 int b_resident, xb_stream_t stream);
/*   xb_dense_wgrad          weight gradients of {Linear(H_in,H_out)+LeakyReLU -> head}_s for s = actor, critic in one launch:
 *                           dW_s = dz_s^T X, db_s = colsum(dz_s) (dz_s generated on the fly as in xb_dense_dgrad),
 *                           dw2_s[j] = sum_b dout_s[b][j] Y_s[b][:], db2_s[j] = sum_b dout_s[b][j].
 *                           The reduction runs over the batch (MN-major tcgen05 operands straight from the row-major
 *                           activations); per-CTA partials are summed in a fixed order (deterministic).
 *                           H_out, H_in in {128, 256}.  workspace: xb_dense_wgrad_workspace_floats(H_in) floats. */
int xb_dense_wgrad_workspace_floats(int H_in);
/*   xb_mlp_backward_tail    ONE launch that finishes a backward pass: sums xb_dense_wgrad's partials (called with dW0 == NULL)
 *                           into the eight hidden/head gradients, xb_mlp_trunk_wgrad's partials (called with dW0 == NULL)
 *                           into dWt/dbt, and converts the loss kernel's fp64 log-std gradient to the fp32 parameter
 *                           gradient (dls64 / trunk_ws may be NULL). */
int xb_mlp_backward_tail(const float* wgrad_ws, int H_out, int H_in, int n_sources, int nh0, int nh1, float* dW0, float* db0,
                         float* dw2_0, float* db2_0, float* dW1, float* db1, float* dw2_1, float* db2_1,
                         const float* trunk_ws, int trunk_parts, int obs_dim, float* dWt, float* dbt, const double* dls64,
                         float* dls32, int A, xb_stream_t stream);
/* The same launch, additionally taking the global norm of the gradients it finishes (it finishes EVERY gradient of the
 * policy, so trunk_ws is required) and deriving the clipped-Adam step scalars into norm_workspace exactly like the first
 * kernel of xb_clip_adam_step (clip_grad_norm_ + LinearLR + bias corrections, ppoclip_learner.py:48-51): follow it with
 * xb_adam_apply.  Saves the separate gradient-norm launch of every update. */
int xb_mlp_backward_tail_norm(const float* wgrad_ws, int H_out, int H_in, int n_sources, int nh0, int nh1, float* dW0,
                              float* db0, float* dw2_0, float* db2_0, float* dW1, float* db1, float* dw2_1, float* db2_1,
                              const float* trunk_ws, int trunk_parts, int obs_dim, float* dWt, float* dbt,
                              const double* dls64, float* dls32, int A, double* norm_workspace, int64_t* step_dev,
                              float lr0, float lr_end_factor, int64_t lr_total_iters, float beta1, float beta2,
                              float max_norm, float grad_scale, float* lr_out, float* gnorm_out, xb_stream_t stream);
int xb_dense_wgrad(const float* Y0, const float* dout0, const float* w2_0, int nh0, const float* Y1, const float* dout1,
                   const float* w2_1, int nh1, const float* X, int64_t B, int H_out, int H_in, float slope,
                   float* workspace, float* dW0, float* db0, float* dw2_0, float* db2_0, float* dW1, float* db1,
                   float* dw2_1, float* db2_1, xb_stream_t stream);
/*   xb_dense_wgrad_bin      BINARY form of xb_dense_wgrad for rank-1 head gradients (nh = 1, or nh = 2 = the two opposite logit
 *                           gradients of a softmax pair: only dout[:, 0] is read).  leaky' = slope + (1 - slope) [y > 0] turns the
 *                           weight gradient into  w2'[m] ((1 - slope) sum_b [y > 0][b][m] (e[b] x[b][n]) + slope sum_b e[b] x[b][n]):
 *                           the MMA's A operand is the 0/1 matrix read from the forward's activation SIGN WORDS (xb_dense_fwd2's
 *                           sign_out; exact in TF32: 2 MMAs per k-step instead of 3) and the activations Y are not read at all.
 *                           Leaves partial sums in `workspace` (same size as xb_dense_wgrad's); xb_mlp_backward_tail_bin finishes
 *                           them, including the head-weight gradient dw2[m] = sum_n W[m][n] Gm[m][n] + b[m] gm[m]  (= sum_b e y).
 *   xb_mlp_backward_tail_bin  xb_mlp_backward_tail(_norm) for those partials: W_s [H_out][H_in], b_s [H_out], w2_s [nh_s][H_out] are
 *                           the hidden layer's master weights / bias and the head weights; norm_workspace == NULL: no norm pass. */
int xb_dense_wgrad_bin(const uint32_t* signs, int sign_ld, const float* dout0, int nh0, const float* dout1, int nh1,
                       const float* X, int64_t B, int H_out, int H_in, float* workspace, xb_stream_t stream);
int xb_mlp_backward_tail_bin(const float* wgrad_ws, int H_out, int H_in, int n_sources, int nh0, int nh1, float* dW0,
                             float* db0, float* dw2_0, float* db2_0, float* dW1, float* db1, float* dw2_1, float* db2_1,
                             const float* trunk_ws, int trunk_parts, int obs_dim, float* dWt, float* dbt, const double* dls64,
                             float* dls32, int A, double* norm_workspace, int64_t* step_dev, float lr0, float lr_end_factor,
                             int64_t lr_total_iters, float beta1, float beta2, float max_norm, float grad_scale, float* lr_out,
                             float* gnorm_out, const float* W0, const float* b0, const float* w2_0, const float* W1,
                             const float* b1, const float* w2_1, float slope, xb_stream_t stream);
/*   xb_dense_fwd2           two layers that share the input X in ONE launch (actor and critic hidden layers + their heads):
 *                           even CTAs evaluate layer 0, odd CTAs layer 1, each with its weights resident in shared memory. */
int xb_dense_fwd2(const float* X, int64_t M, int K, int N, float slope, const float* Whi0, const float* Wlo0,
                  const float* bias0, float* Y0, const float* head_w0, const float* head_b0, int n_head0, float* head_out0,
                  const float* Whi1, const float* Wlo1, const float* bias1, float* Y1, const float* head_w1,
                  const float* head_b1, int n_head1, float* head_out1, int b_resident, const float* prep_W0,
                  const float* prep_W1, float* prep_thi, float* prep_tlo, uint32_t* sign_out, xb_stream_t stream);
/*   sign_out (nullable, xb_dense_fwd2 and xb_dense_fwd2_loss): u32 [M][2 * N / 32] activation SIGN WORDS — bit j of word
 *   [row][layer * N / 32 + c] = (Y_layer[row][32 c + j] > 0).  The backward pass needs the hidden activations only through
 *   leaky_relu' = (y > 0 ? 1 : slope): xb_dense_dgrad reads these words (32 B per row) instead of the two activation tiles. */
/*   prep_W0 / prep_W1 / prep_thi / prep_tlo (nullable group, xb_dense_fwd2 and xb_dense_fwd2_loss): the fp32 master weights
 *   [N][N] of the two layers; the launch then also writes the weight operand of the MASK-FORM dgrad that follows:
 *   Wt'[n][s * N + k] = tf32 hi/lo split of w2'_s[k] * W_s[k][n], w2'_s = head_w_s[0] (- head_w_s[1] for a 2-logit head),
 *   f32 [N][2N] each — see wt_form of xb_dense_dgrad. */
/*   xb_mlp_fwd_from_obs     the whole actor-critic forward in ONE launch (rollout / inference): the trunk layer
 *                           h1 = leaky_relu(W0 obs + b0) is generated by the operand warps straight into tensor memory
 *                           (obs_dim <= 4, H in {64, 128}), then both hidden layers + heads as in xb_dense_fwd2.
 *                           Y0 / Y1 may both be NULL: only the head outputs are produced.
 *                           norm_new / norm_old (nullable pair, fp64 [9] observation-normaliser states): obs holds RAW
 *                           observations; rows [0, norm_rows) are normalised with norm_new, the rest with norm_old
 *                           (clip((obs - mean) / (sqrt(var) + 1e-8), +-norm_clip), agent.py:112-113) before the trunk layer.
 *                           The launch carries the programmatic-serialization attribute (it may become resident while the
 *                           launch before it still runs, and waits for it by itself).  flags: XB_FWD_WEIGHTS_STABLE = the
 *                           caller vouches that the launch immediately before this one on the stream writes none of the
 *                           weight / bias arrays: set-up and the resident-weight loads then overlap that launch (the
 *                           rollout loop: every forward after the first follows xb_rollout_step). */
#define XB_FWD_WEIGHTS_STABLE 1
/* xb_dense_fwd2 (actor | critic hidden layers + heads) with xb_ppo_loss_* fused into its epilogue: the epilogue thread that
 * holds a row's head outputs turns them straight into dL/d(mu | logits) (actor CTA) and dL/dv (critic CTA) with the formulas of
 * ppoclip_learner.py:33-44 (SURVEY.md App. C) — no loss launch, no round trip of the head outputs.
 *   scal        f32 [M][4] = {act, old_logp, adv, ret} per row (xb_gather_records / xb_gather_trunk_fwd); 16-byte aligned
 *   adv_stats   nullable (sum, sumsq) over adv_count samples -> on-the-fly advantage normalisation
 *   logstd      Gaussian actor (n_head0 = 1): f32 [1] shared log-std, dlogstd fp64 [1] receives its gradient;
 *               NULL: Categorical actor with n_head0 = 2 logits.  clip_range <= 0 selects the A2C / PG surrogate.
 *   dact f32 [M][n_head0], dv f32 [M]: gradients w.r.t. the head outputs (inputs of xb_dense_dgrad / xb_dense_wgrad)
 *   loss_partials fp64 [148 * 8], loss_ticket u32 [1] (zero once): scratch; scalars fp64 [8] as xb_ppo_loss_* (deterministic). */
int xb_dense_fwd2_loss(const float* X, int64_t M, int K, int N, float slope, const float* Whi0, const float* Wlo0,
                       const float* bias0, float* Y0, const float* head_w0, const float* head_b0, int n_head0,
                       float* head_out0, const float* Whi1, const float* Wlo1, const float* bias1, float* Y1,
                       const float* head_w1, const float* head_b1, int n_head1, float* head_out1, int b_resident,
                       const float* scal, const double* adv_stats, int64_t adv_count, float clip_range, float vf_coef,
                       float ent_coef, float inv_batch, const float* logstd, float* dact, float* dv, double* loss_partials,
                       uint32_t* loss_ticket, double* scalars, double* dlogstd, const float* prep_W0, const float* prep_W1,
                       float* prep_thi, float* prep_tlo, uint32_t* sign_out, xb_stream_t stream);
/* xb_mlp_fwd_from_obs for TRAINING: the trunk layer generated in the kernel plus everything xb_dense_fwd2_loss adds (Y0 / Y1,
 * sign_out, prep_*, and — with scal != NULL — the fused PPO loss).  h1_out f32 [M][H] receives the trunk activations
 * leaky_relu(W0 obs + b0) (stored by the operand warps of the layer-0 CTAs): the backward kernels read them, this launch does not.
 * Replaces xb_mlp_trunk_fwd / the first-layer half of xb_gather_trunk_fwd + the h1 read of xb_dense_fwd2_loss. */
int xb_mlp_fwd_from_obs_train(const float* obs, int ld, int obs_dim, const float* W0, const float* b0, int64_t M, int H,
                              float slope, const float* Whi0, const float* Wlo0, const float* bias0, float* Y0,
                              const float* head_w0, const float* head_b0, int n_head0, float* head_out0, const float* Whi1,
                              const float* Wlo1, const float* bias1, float* Y1, const float* head_w1, const float* head_b1,
                              int n_head1, float* head_out1, float* h1_out, const float* scal, const double* adv_stats,
                              int64_t adv_count, float clip_range, float vf_coef, float ent_coef, float inv_batch,
                              const float* logstd, float* dact, float* dv, double* loss_partials, uint32_t* loss_ticket,
                              double* scalars, double* dlogstd, const float* prep_W0, const float* prep_W1, float* prep_thi,
                              float* prep_tlo, uint32_t* sign_out, xb_stream_t stream);
int xb_mlp_fwd_from_obs(const float* obs, int ld, int obs_dim, const float* W0, const float* b0, int64_t M, int H,
                        float slope, const float* Whi0, const float* Wlo0, const float* bias0, float* Y0,
                        const float* head_w0, const float* head_b0, int n_head0, float* head_out0, const float* Whi1,
                        const float* Wlo1, const float* bias1, float* Y1, const float* head_w1, const float* head_b1,
                        int n_head1, float* head_out1, const double* norm_new, const double* norm_old, int64_t norm_rows,
                        float norm_clip, int flags, xb_stream_t stream);
int xb_dense_dgrad(const float* Y0, const float* dout0, const float* w2_0, int nh0, int K0, const float* Y1,
                   const float* dout1, const float* w2_1, int nh1, int K1, int64_t M, const float* Wthi,
                   const float* Wtlo, int N, const float* H1, float slope, float* dZ1, int wt_form, const uint32_t* signs,
                   const uint32_t* h1_signs, xb_stream_t stream);
/*   wt_form 0: Wthi / Wtlo = the plain transposed weights (xb_dense_split_weights*), any head gradients (nh <= 2).
 *   wt_form 1 ("mask form"): Wthi / Wtlo = the w2-scaled operand written by xb_dense_fwd2(_loss) (prep_*).  Valid when every
 *   source's head gradient is rank-1: one head, or two logits of a softmax head (whose gradients are opposite: dout[:, 1] is
 *   then NOT read, -dout[:, 0] is implied).  The operand warps then select per element between two per-row constants
 *   instead of multiplying and splitting — same 3xTF32 accuracy.
 *   signs (nullable): u32 [M][(K0 + K1) / 32] sign words of [Y0 | Y1] as written by xb_dense_fwd2(_loss) (sign_out); used by the
 *   tensor-memory (N <= 128, K0 + K1 <= 256) kernel in place of Y0 / Y1 (which are then not read) — bit-identical results.
 *   h1_signs (nullable, with signs, N = 128): u32 [M][4] sign words of H1 (xb_gather_trunk_fwd / xb_mlp_trunk_fwd): the
 *   epilogue mask leaky'(H1) without loading the H1 tiles (H1 is then not read; 16-byte aligned). */

/* ------------------------------------------------------------------------------------------------------------
 * First (narrow-input) layer of the MLP, Linear(obs_dim, H) + LeakyReLU — Basic_MLP
 * (xuance/torch/representations/mlp.py:40-51) — and its weight gradient; bandwidth-bound SIMT kernels (csrc/mlp_trunk.cu).
 *   xb_mlp_trunk_fwd    h1[b][n] = leaky_relu(b0[n] + sum_i obs[b*ld + i] W0[n][i])     obs_dim <= 8, H % 4 == 0
 *   xb_mlp_trunk_wgrad  dW0[n][i] = sum_b dz1[b][n] obs[b*ld + i],  db0[n] = sum_b dz1[b][n]   (deterministic two-stage sum)
 * workspace: xb_mlp_trunk_wgrad_workspace_floats(obs_dim, H) floats.  dW0 == NULL: leave the partial sums in the
 * workspace (xb_mlp_backward_tail finishes them together with the hidden layers' partials in one launch).
 * ---------------------------------------------------------------------------------------------------------- */
int xb_mlp_trunk_fwd(const float* obs, int ld, int obs_dim, const float* W0, const float* b0, float slope, float* h1,
                     int64_t B, int H, uint32_t* h1_signs, xb_stream_t stream);
int xb_mlp_trunk_wgrad_workspace_floats(int obs_dim, int H);
int xb_mlp_trunk_wgrad_parts(void);     /* number of partial sums per output in the workspace */
int xb_mlp_trunk_wgrad(const float* dz1, const float* obs, int ld, int obs_dim, float* workspace, float* dW0, float* db0,
                       int64_t B, int H, xb_stream_t stream);
/* Discrete(3) actor heads on the two-head dense kernels (MountainCar-v0 / Acrobot-v1; categorical.py:26-32 is generic in
 * action_dim): softmax(z0, z1, z2) == softmax(z0 - z2, z1 - z2, 0), so the kernels run with FOLDED head parameters
 *   xb_head3_fold           w2[j] = w3[j] - w3[2], b2[j] = b3[j] - b3[2] (j = 0, 1);  w3 f32 [3][H], w2 f32 [2][H]
 *   xb_head3_unfold_grads   rows 0, 1 of gw3 [3][H] / gb3 [3] hold the two-head gradients; row 2 = -(row 0 + row 1)
 * (dL/dz2 = -(dL/dz0 + dL/dz1) for any loss of the softmax).  The third logit is reported as 0. */
int xb_head3_fold(const float* w3, const float* b3, float* w2, float* b2, int H, xb_stream_t stream);
int xb_head3_unfold_grads(float* gw3, float* gb3, int H, xb_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * (5b) Env-sharded data parallelism over NVLink / NVSwitch PEER MEMORY (SURVEY.md §8(e)): the two exchanges of an
 * update — the (sum adv, sum adv^2) behind the global-minibatch advantage normalisation (memory_tools.py:241-242)
 * and the flat-gradient sum in front of clip_grad_norm_ + Adam (ppoclip_learner.py:47-49) — as kernels that read the
 * peers' buffers directly, fused with the computation that consumes the result.  The reference is single-process
 * (its only collective is the disabled mpi4py Allreduce of xuance/common/statistic_tools.py:6-32).
 *
 * Every rank owns one "comm block" (xb_peer_alloc: cudaMalloc, zeroed) of xb_peer_block_bytes(n) bytes, laid out
 *   [ barrier flags | stats fp64 [xb_peer_stats_max()] at xb_peer_stats_offset() | gradient inbox fp32 [2][8][n] at xb_peer_grad_offset() ]
 * exported / imported through CUDA IPC (xb_peer_export -> 64-byte handle -> xb_peer_import in the peer process).
 * peer_bases is a HOST array of the W device pointers (index = rank; own block at [rank]).
 * tickets: u32 [64] device, zero-initialised once, private to the rank (per-CTA barrier counters; never reset).
 * Every rank must issue the same sequence of xb_peer_* launches with the same n.  A barrier wait that exceeds 60 s gives up
 * and sets tickets[62] (the host checks it) instead of spinning forever when a peer process has died.
 *
 * xb_peer_allreduce_grad_norm: every CTA pushes its slice of grad_in (local, fp32 [n]) into inbox[launch parity][rank] of
 *   every peer with P2P stores; ONE barrier; grad_out[i] = sum_r inbox[parity][r][i] in rank order (bit-identical on every
 *   rank) read from local memory; squared norm of grad_out * grad_scale; then exactly the scalars xb_clip_adam_step's
 *   first kernel derives (workspace layout identical), so xb_adam_apply can follow.  n must be a multiple of 4.
 * xb_adam_apply: the second kernel of xb_clip_adam_step alone (clip + Adam from the scalars in workspace).
 * xb_peer_allreduce_mean: the push / barrier / rank-order sum of xb_peer_allreduce_grad_norm without the optimiser scalars:
 *   grad_out = (sum_r grad_in_r) * (1 / W), written to local memory, bit-identical on every rank (W = 1: grad_out = grad_in bit
 *   for bit).  The sharded form of the gradient a torch optimiser steps on (ppg_learner.py:44-46,59-63,80-84 `loss.backward();
 *   optimizer.step()` over a minibatch split across ranks).  Shares the inbox, the per-CTA tickets and the grid of
 *   xb_peer_allreduce_grad_norm: every launch on one comm block must pass the same n (a multiple of 4).
 * xb_peer_allreduce_f64: out[j] = sum_r stats_r[offset + j], j < n, offset + n <= xb_peer_stats_max().  Used once per epoch for
 *   the minibatch advantage statistics and, with use_obsnorm / use_rewnorm, once per vector step for the observation /
 *   return moments (the analogue of mpi_moments, xuance/common/statistic_tools.py:6-32).
 * xb_adv_stats_minibatches: stats[m] = (sum, sumsq) of adv over minibatch m = idx[m*B, (m+1)*B) for every minibatch
 *   of an epoch in one launch (adv element stride `stride` floats per transition row; zeroes stats first).
 * ---------------------------------------------------------------------------------------------------------- */
int64_t xb_peer_block_bytes(int64_t n_grad_floats);
int64_t xb_peer_stats_offset(void);
int64_t xb_peer_grad_offset(void);
int xb_peer_stats_max(void);
int xb_peer_alloc(void** ptr_out /* host */, int64_t bytes);
int xb_peer_free(void* ptr);
int xb_peer_export(void* ptr, void* handle_out /* host, 64 bytes */);
int xb_peer_import(const void* handle /* host, 64 bytes */, void** ptr_out /* host */);
int xb_peer_close(void* ptr);
int xb_peer_allreduce_grad_norm(const void* const* peer_bases /* host [W] */, int rank, int W, int64_t n,
                                const float* grad_in, float* grad_out, uint32_t* tickets, int64_t* step_dev, float lr0, float lr_end_factor,
                                int64_t lr_total_iters, float beta1, float beta2, float eps, float max_norm,
                                float grad_scale, double* workspace, float* lr_out, float* gnorm_out, xb_stream_t stream);
int xb_adam_apply(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float beta1, float beta2,
                  float eps, float grad_scale, const double* workspace, xb_stream_t stream);
/* xb_adam_apply fused with xb_dense_split_weights2: the two H x H hidden-layer weights W_s = param + w_off_s ([N][K]) get
 * their tf32 hi/lo operand copies (and the transposed, concatenated dgrad operand thi/tlo [K][2N]) rewritten by the same
 * threads that update them, so no separate split launch is needed before the next forward. */
int xb_adam_apply_split(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float beta1,
                        float beta2, float eps, float grad_scale, const double* workspace, int64_t w_off0, float* hi0,
                        float* lo0, int64_t w_off1, float* hi1, float* lo1, int N, int K, float* thi, float* tlo,
                        xb_stream_t stream);
int xb_peer_allreduce_mean(const void* const* peer_bases /* host [W] */, int rank, int W, int64_t n, const float* grad_in,
                           float* grad_out, uint32_t* tickets, xb_stream_t stream);
int xb_peer_allreduce_f64(const void* const* peer_bases /* host [W] */, int rank, int W, int offset, int n, double* out,
                          uint32_t* tickets, xb_stream_t stream);
/*   xb_peer_allreduce_merge   the per-vector-step statistics exchange of the env-sharded normalisers as ONE kernel with ONE
 *                             cross-GPU barrier + the merge of xb_rms_merge_sums: every rank pushes src[0..n) (n <= 20) into a
 *                             parity double-buffered inbox at doubles [inbox_offset, inbox_offset + 320) of every peer's
 *                             statistics area, out[0..n) = the totals (rank order, bit-identical on every rank); with
 *                             obs_state_in / ret_state (n = 2D + 4 = 12 or 20: sum x[D], sum x^2[D], N, sum R, sum R^2,
 *                             n finished, for D = 4 or 8 floats per observation row, dim <= D) the normaliser states are
 *                             merged in the same launch (mpi_moments, statistic_tools.py:6-32). */
int xb_peer_allreduce_merge(const void* const* peer_bases, int rank, int W, const double* src, int n, int inbox_offset,
                            double* out, uint32_t* tickets, const double* obs_state_in, double* obs_state_out, int dim,
                            double* ret_state, float* rew_std, xb_stream_t stream);
int xb_adv_stats_minibatches(const int64_t* idx, int64_t n_minibatches, int64_t B, int64_t T, int64_t N, const float* adv,
                             int64_t stride, double* stats, xb_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Device-side minibatch permutation: out[i] = P(i), a keyed pseudo-random bijection of [0, n) (swap-free Feistel
 * network on ceil(log2 n) bits + cycle walking), evaluated independently per index: one launch, no sort, no scratch.
 * Replaces np.random.shuffle(indexes) in PPOCLIP_Agent.train (ppoclip_agent.py:76-78).  The key is derived from
 * (seed, *counter_dev + offset), so a captured graph draws a fresh permutation on every replay once xb_counter_add
 * has advanced the device counter (counter_dev may be NULL).  The permutation itself is not a parity target (the
 * reference uses numpy's global MT19937 stream); being a permutation, and varying with the key, are tested.
 * ---------------------------------------------------------------------------------------------------------- */
int xb_random_permutation(int64_t* out, int64_t n, uint64_t seed, const uint64_t* counter_dev, uint64_t offset,
                          xb_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * HOST helper (host pointers, runs on the calling CPU thread; releases nothing on the device).
 * Uniform random permutation of 0..n-1 into out[n] (a pinned staging buffer): the host side of the minibatch
 * index feed, replacing np.random.shuffle(indexes) in PPOCLIP_Agent.train (ppoclip_agent.py:76-78).
 * ---------------------------------------------------------------------------------------------------------- */
int xb_host_permutation(int64_t* out /* host */, int64_t n, uint64_t seed);
/* 32-bit flavour (n < 2^31): half the pinned-memory / H2D bytes; above 2^16 indices a cache-friendly two-pass shuffle
 * (Rao-Sandelius bucket scatter + in-bucket Fisher-Yates), still a uniform random permutation. */
int xb_host_permutation32(int32_t* out, int64_t n, uint64_t seed);

#ifdef __cplusplus
}
#endif
#endif /* XB200_H */
