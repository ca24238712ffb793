/* omnisafe_b200 -- C ABI of the B200-native on-policy SafeRL hot path.
 *
 * The reference (PKU-Alignment/omnisafe) is pure Python: its seam for this path is the set of
 * Python methods listed below, not an FFI.  Each entry point here is what a ctypes binding of the
 * corresponding reference method body would call (see INTEGRATION.md for the stub).  All pointers
 * are DEVICE pointers to contiguous row-major arrays the caller owns; `stream` is a cudaStream_t
 * (NULL = default stream).  Every function returns 0 on success, non-zero on failure;
 * osb_last_error() returns the reason.  No function synchronises the host unless stated.
 * Host-side state (kernel attributes set once, the FOCOPS / P3O scratch scalar, the P2P step counter, the
 * last-error string) is per process: call the entry points from ONE host thread per device, one
 * process per GPU -- the way the reference's `distributed.fork` runs it.
 *
 * Slab layout ("time-major"): per-step scalars are [T][N] (env index contiguous), observations
 * [T][N][O], actions [T][N][A].  Sample k of the reference's env-major order
 * (vector_onpolicy_buffer.py:L125-129, k = i*T + t) lives at slab row t*N + i.
 *
 * Flat parameter vector theta = [actor | reward_critic | cost_critic], each in the reference's
 * named_parameters() order (utils/tools.py:L35-129): actor = log_std[A], W1[64][O], b1[64],
 * W2[64][64], b2[64], W3[A][64], b3[A]; critic = W1, b1, W2, b2, W3[1][64], b3[1].
 */
#ifndef OMNISAFE_B200_H
#define OMNISAFE_B200_H

#ifdef __cplusplus
extern "C" {
#endif

/* ---- plumbing ---------------------------------------------------------------------------- */
const char* osb_last_error(void);
int osb_abi_version(void);
/* kernels launched by this library in this process so far (bench.py counts its timed region with it) */
long long osb_launch_count(void);
int osb_device_info(int device, int* sm_count, int* cc_major, int* cc_minor);

/* ---- dual GAE (segmented reverse scan) ----------------------------------------------------
 * replaces OnPolicyBuffer.finish_path            omnisafe/common/buffer/onpolicy_buffer.py:L148-203
 *          _calculate_adv_and_value_targets('gae')                                     :L299-303
 *          discount_cumsum (fp64 carry)           omnisafe/utils/math.py:L59-82
 * flags bit0 = terminated, bit1 = truncated; a path also ends at t == T-1.  At a path end the
 * bootstrap value is 0 if terminated, else boot_{r,c}[t][i].  disc_ret may be NULL.
 * workspace: osb_gae_workspace_doubles(N) doubles.  sums[4] <- {sum adv_r, sum adv_r^2,
 * sum adv_c, count} over this rank's samples (fp64; all-reduce them across ranks, then call
 * osb_adv_moments). */
int osb_gae_workspace_doubles(int n_envs);
int osb_gae_dual(const float* rew, const float* cost, const float* val_r, const float* val_c,
                 const unsigned char* flags, const float* boot_r, const float* boot_c, int T, int N,
                 double gamma, double lam, double lam_c, double penalty_coef, float* adv_r,
                 float* adv_c, float* tv_r, float* tv_c, float* disc_ret, double* workspace,
                 double* sums, void* stream);
/* osb_gae_dual with the reference's other advantage estimators (onpolicy_buffer.py:L299-331):
 * estimator 0 = 'gae', 1 = 'gae-rtg' (targets = discounted reward-to-go of the penalised path incl.
 * its bootstrap slot), 2 = 'plain' (advantage = one-step delta, targets = reward-to-go), 3 = 'vtrace'
 * (on-policy V-trace, rho = c = 1: targets v_t = V_t + delta_t + gamma (v_{t+1} - V_{t+1}), advantage
 * r_t + gamma v_{t+1} - V_t; fp32 replay of the reference recurrence from an fp64 scan carry).
 * For 1 / 2 disc_ret shares the reward-to-go scan: pass NULL unless penalty_coef == 0. */
int osb_adv_estimate(const float* rew, const float* cost, const float* val_r, const float* val_c,
                     const uint8_t* flags, const float* boot_r, const float* boot_c, int T, int N,
                     double gamma, double lam, double lam_c, double penalty_coef, int estimator,
                     float* adv_r, float* adv_c, float* tv_r, float* tv_c, float* disc_ret,
                     double* workspace, double* sums, void* stream);
/* moments[4] <- {mean_r, std_r + 1e-8, mean_c, 1}: the statistics VectorOnPolicyBuffer.get()
 * standardises with (vector_onpolicy_buffer.py:L131-136, utils/distributed.py:L382-388). */
int osb_adv_moments(const double* sums, int standardize_r, int standardize_c, float* moments,
                    void* stream);
/* out_r = (adv_r - mean_r) / (std_r + 1e-8), out_c = adv_c - mean_c  (what get() returns). */
int osb_adv_standardize(const float* adv_r, const float* adv_c, const float* moments, long long n,
                        float* out_r, float* out_c, void* stream);
/* discount_cumsum over `rows` independent vectors of length `len` (utils/math.py:L59-82);
 * x is fp32 (x_is_f64 = 0) or fp64, out is fp64. */
int osb_discount_cumsum(const void* x, int x_is_f64, int rows, int len, double discount,
                        double* out, void* stream);

/* ---- rollout: fused env step + 3 MLP forwards + sample + slab append ------------------------
 * replaces, per step, ConstraintActorCritic.step  models/actor_critic/constraint_actor_critic.py:L84-109
 *          ActionScale.step / ObsNormalize.step    envs/wrapper.py:L510-514, L231-241
 *          Normalizer.normalize / _push            common/normalizer.py:L88-139
 *          VectorOnPolicyBuffer.store              common/buffer/vector_onpolicy_buffer.py:L96-99
 *          the per-env done loop                   adapter/onpolicy_adapter.py:L114-136
 * Env state arrays: s_raw[2][N][O], final_raw[2][N][O], ep_step[N], episode[N], gstep[N],
 * ep_ret[N], ep_cost[N], ep_len[N], bias[O].  Normaliser state: mean/sumsq/std/mean1/std1 [O],
 * count[2], acc_all[2][O], acc_fin[2][O] (int64 fixed point), fin_count[1], had_fin[1], ticket[1]
 * (all zero-initialised by the caller).  osb_env_reset = OnPolicyAdapter.reset() at epoch start
 * (onpolicy_adapter.py:L80).  osb_rollout_step with t in [0, T) performs step t; t == T is the
 * epoch-end bootstrap launch (critics only).  eps = [N][A] standard-normal draws of this step
 * (parity mode) or NULL (in-kernel Philox keyed by noise_seed / global_step).  precision: 0 = exact
 * fp32 FMA tiles (parity), 1 = tcgen05 TF32 tiles of 128 envs (O <= 64; falls back to 0 otherwise). */
int osb_env_reset(int O, int A, int max_episode_steps, unsigned seed, unsigned term_threshold,
                  unsigned env_id_offset, float cost_threshold, int obs_normalize, int N,
                  float* s_raw, float* final_raw, int* ep_step, unsigned* episode, unsigned* gstep,
                  float* ep_ret, float* ep_cost, int* ep_len, const float* bias,
                  float* norm_mean, float* norm_sumsq, float* norm_std, float* norm_mean1,
                  float* norm_std1, long long* norm_count, long long* acc_all, long long* acc_fin,
                  int* fin_count, int* had_fin, unsigned* ticket, void* stream);
int osb_rollout_step(int O, int A, int max_episode_steps, unsigned seed, unsigned term_threshold,
                     unsigned env_id_offset, float cost_threshold, int obs_normalize, int N, int T,
                     int t, float* s_raw, float* final_raw, int* ep_step, unsigned* episode,
                     unsigned* gstep, float* ep_ret, float* ep_cost, int* ep_len, const float* bias,
                     float* norm_mean, float* norm_sumsq, float* norm_std, float* norm_mean1,
                     float* norm_std1, long long* norm_count, long long* acc_all,
                     long long* acc_fin, int* fin_count, int* had_fin, unsigned* ticket,
                     float* obs, float* act, float* logp, float* rew, float* cost, float* val_r,
                     float* val_c, float* boot_r, float* boot_c, unsigned char* flags, float* epfin,
                     const float* theta, const float* eps, unsigned noise_seed,
                     unsigned global_step, int precision, void* stream);
/* Whole-epoch rollout in one call: reset, T step launches (eps_all = [T][N][A] or NULL), the
 * epoch-end bootstrap launch and the episode window (= OnPolicyAdapter.rollout,
 * adapter/onpolicy_adapter.py:L58-136).  Philox counter = epoch_index * T + t. */
int osb_rollout_epoch(int O, int A, int max_episode_steps, unsigned seed, unsigned term_threshold,
                      unsigned env_id_offset, float cost_threshold, int obs_normalize, int N, int T,
                      float* s_raw, float* final_raw, int* ep_step, unsigned* episode,
                      unsigned* gstep, float* ep_ret, float* ep_cost, int* ep_len, const float* bias,
                      float* norm_mean, float* norm_sumsq, float* norm_std, float* norm_mean1,
                      float* norm_std1, long long* norm_count, long long* acc_all,
                      long long* acc_fin, int* fin_count, int* had_fin, unsigned* ticket,
                      float* obs, float* act, float* logp, float* rew, float* cost, float* val_r,
                      float* val_c, float* boot_r, float* boot_c, unsigned char* flags, float* epfin,
                      const float* theta, const float* eps_all, unsigned noise_seed,
                      unsigned epoch_index, int W, float* ring, int* meta, double* window_sums,
                      int precision, void* stream);
/* Saute / Simmer mode of the following osb_env_reset / osb_rollout_* calls (SauteAdapter.step / reset,
 * adapter/saute_adapter.py:L135-217; SimmerAdapter.reset, simmer_adapter.py:L97-111): safety = [2][N] device floats (the
 * safety state z by step parity) or NULL for the plain OnPolicyAdapter.  The networks then take O + 1 inputs
 * ([normalised obs | z], theta sized accordingly) and the obs slab rows are O + 1 wide; z starts an epoch at safety_init,
 * z <- (z - cost / safety_budget) / saute_gamma per step, the stored reward is unsafe_reward once z <= 0, z <- 1 at
 * episode ends.  Process-wide until changed. */
int osb_rollout_set_saute(float* safety, float safety_budget, float saute_gamma, float unsafe_reward, float safety_init);
/* EarlyTerminated mode of the following osb_rollout_* calls (EarlyTerminatedAdapter.step,
 * adapter/early_terminated_adapter.py:L56-98, per env): cost_acc = [N] device floats holding the accumulated cost (not cleared
 * by ordinary episode ends) or NULL; once it exceeds cost_limit the step stores reward 0 and terminated = 1, the env is reset
 * and the accumulator cleared.  Process-wide until changed. */
int osb_rollout_set_early_termination(float* cost_acc, float cost_limit);
/* Logger window of the last <= W finished episodes in (step, env) order
 * (common/logger.py:L253-282, adapter/onpolicy_adapter.py:L159-175).  ring[3][W], meta[2] persist
 * across epochs; window_sums[4] <- {sum EpRet, sum EpCost, sum EpLen, count} (fp64). */
int osb_episode_window(const unsigned char* flags, const float* epfin, int T, int N, int W,
                       float* ring, int* meta, double* window_sums, void* stream);
/* RewardNormalize / CostNormalize (envs/wrapper.py:L280-423; Normalizer(shape=(), clip=5),
 * common/normalizer.py:L88-139) applied to one epoch's slab x[T][N] in place, after the rollout: row t
 * is pushed into the running statistics (batch of N) and normalised with the statistics valid right
 * after that push, exactly the reference's per-step sequence.  state: {mean, sumsq, std} (3 floats) and
 * count[1] persist across epochs; workspace: 4 * T floats. */
int osb_scalar_normalize_rows(float* x, int T, int N, float clip, float* state, long long* count,
                              float* workspace, void* stream);

/* ---- learner: fused minibatch forward + loss + backward ------------------------------------
 * replaces PolicyGradient._update minibatch body  algorithms/on_policy/base/policy_gradient.py:L369-381
 *          _update_reward_critic/_update_cost_critic/_update_actor                       :L407-524
 *          PPO._loss_pi  base/ppo.py:L35-87;  PPOLag._compute_adv_surrogate  naive_lagrange/ppo_lag.py:L82-102
 *          PolicyGradient._loss_pi  base/policy_gradient.py:L551-588;  CPO._loss_pi_cost  second_order/cpo.py:L182-212
 *          FOCOPS._loss_pi  first_order/focops.py:L62-108
 * Batch tensors are the slabs ([rows] / [rows][O] / [rows][A], row = t*N + i); advantages are the
 * RAW GAE outputs and are standardised on the fly with moments[4] (osb_adv_moments).  A minibatch is
 * the window [mb_start, mb_start+mb_count) of a permutation of [0,total): perm (slab rows, parity
 * mode) or NULL (in-kernel keyed Feistel bijection).  loss_kind: 0 PPO-clip, 1 plain ratio*adv,
 * 2 FOCOPS, 3 cost surrogate, 5 P3O (PPO-clip + kappa * relu(mean(ratio*adv_c) + Jc - limit),
 * penalty_function/p3o.py:L48-125; kappa is passed as focops_lam, Jc - limit as focops_eta; like
 * FOCOPS it runs a forward-only pass first for the minibatch mean).  lagrange: device scalar lambda or NULL (0).  net_mask bit0 actor,
 * bit1 reward critic, bit2 cost critic.  gpart: osb_update_grid_blocks(mb_count) * P floats;
 * stats_part: that many * 3 * 8 floats.  stop_flag (device int, may be NULL): non-zero = no-op. */
int osb_update_grid_blocks(int mb_count);
int osb_minibatch_grad(const float* theta, int O, int A, const float* obs, const float* act,
                       const float* logp, const float* adv_r, const float* adv_c,
                       const float* tv_r, const float* tv_c, const float* mu_old,
                       const float* moments, const int* perm, long long total, unsigned perm_seed,
                       long long mb_start, int mb_count, int loss_kind, float clip,
                       float entropy_coef, float focops_lam, float focops_eta,
                       const float* lagrange, const float* logstd_old, int net_mask, float* gpart,
                       float* stats_part, const int* stop_flag, void* stream);
/* Tensor-core variant of osb_minibatch_grad: the tile GEMMs run as tcgen05.mma kind::tf32 with TMEM
 * accumulators (operands fp32 in 128B-swizzled smem tiles; transposed activations produced by
 * role-swapped MMAs).  Same arguments and outputs; O <= 64, A <= 16.  This is arithmetic mode
 * `precision = 1` of osb_ppo_update_epoch; mode 0 is the exact-fp32 FMA parity path.
 * gpart / stats_part rows: osb_tc_grid_blocks(mb_count, net_mask) -- 49 CTAs per network when
 * several networks share the launch, up to 148 when net_mask names a single network. */
int osb_tc_grid_blocks(long long rows, int net_mask);
int osb_minibatch_grad_tc(const float* theta, int O, int A, const float* obs, const float* act,
                          const float* logp, const float* adv_r, const float* adv_c,
                          const float* tv_r, const float* tv_c, const float* mu_old,
                          const float* moments, const int* perm, long long total, unsigned perm_seed,
                          long long mb_start, int mb_count, int loss_kind, float clip,
                          float entropy_coef, float focops_lam, float focops_eta,
                          const float* lagrange, const float* logstd_old, int net_mask, float* gpart,
                          float* stats_part, const int* stop_flag, void* stream);
/* Split-bf16 ("bf16x3") parity-grade tensor-core variant (csrc/update_x3.cu): every GEMM = six kind::f16
 * MMAs over the three bf16 pieces of its fp32 operands, fp32 accumulate; O <= 64, loss kinds 0 / 1 / 3. */
int osb_minibatch_grad_x3(const float* theta, int O, int A, const float* obs, const float* act,
                          const float* logp, const float* adv_r, const float* adv_c,
                          const float* tv_r, const float* tv_c, const float* mu_old,
                          const float* moments, const int* perm, long long total, unsigned perm_seed,
                          long long mb_start, int mb_count, int loss_kind, float clip,
                          float entropy_coef, float focops_lam, float focops_eta,
                          const float* lagrange, const float* logstd_old, int net_mask, float* gpart,
                          float* stats_part, const int* stop_flag, void* stream);
/* Full-batch actor pass (KL early stop policy_gradient.py:L383-397; TRPO/CPO line-search
 * evaluations trpo.py:L102-138, cpo.py:L114-171).  mu_store != NULL: write mu(theta) per row.
 * Otherwise out[8] <- {sum_s sum_a KL(old||new), sum ratio*adv, sum ratio*adv_c, sum ratio, count,
 * sum ratio*adv_r, 0, 0} in fp64; rows 0, stride, 2*stride, ...; workspace: 296*8 doubles. */
int osb_actor_eval(const float* theta_actor, int O, int A, const float* obs, const float* act,
                   const float* logp, const float* adv_r, const float* adv_c, const float* mu_old,
                   const float* logstd_old, const float* moments, const float* lagrange,
                   long long total, int stride, float* mu_store, double* workspace, double* out,
                   void* stream);
/* Tensor-core (tcgen05 TF32) variant of osb_actor_eval: same arguments / outputs, O <= 64. */
int osb_actor_eval_tc(const float* theta_actor, int O, int A, const float* obs, const float* act,
                      const float* logp, const float* adv_r, const float* adv_c, const float* mu_old,
                      const float* logstd_old, const float* moments, const float* lagrange,
                      long long total, int stride, float* mu_store, double* workspace, double* out,
                      void* stream);
/* One update iteration of PolicyGradient._update (policy_gradient.py:L369-381) as ONE persistent cooperative
 * kernel on bf16x3 tiles (csrc/update_x3.cu): every minibatch = fused forward + loss + backward, fixed-order
 * partial reduction, per-network clip_grad_norm_, clipped-gradient exchange over NVLink peer memory when
 * world > 1 (clip -> average -> step: policy_gradient.py:L437-443, distributed.py:L193-198) and torch-Adam,
 * parameters re-staged in shared memory between minibatches.  perm = slab rows of this iteration or NULL. */
int osb_ppo_update_iter_x3(float* theta, float* grad, float* adam_m, float* adam_v, int* adam_step, int O, int A,
                           const float* obs, const float* act, const float* logp, const float* adv_r,
                           const float* adv_c, const float* tv_r, const float* tv_c, const float* moments,
                           const int* perm, long long total, unsigned perm_seed, int batch_size, int loss_kind,
                           float clip, float entropy_coef, const float* lagrange, int net_mask,
                           float critic_norm_coef, float max_grad_norm, float lr_actor, float lr_critic_r,
                           float lr_critic_c, float* gpart, float* stats_part, float* train_stats,
                           const int* stop_flag, void* peer_buf, void* peer_flag, int world, int rank,
                           int* p2p_error, void* stream);
/* Split-bf16 (parity-grade tensor-core) variant, O <= 64 (csrc/eval_x3.cu). */
int osb_actor_eval_x3(const float* theta_actor, int O, int A, const float* obs, const float* act,
                      const float* logp, const float* adv_r, const float* adv_c, const float* mu_old,
                      const float* logstd_old, const float* moments, const float* lagrange,
                      long long total, int stride, float* mu_store, double* workspace, double* out,
                      void* stream);
/* Fisher-vector product partials (NaturalPG._fvp, base/natural_pg.py:L74-119, analytic
 * Gauss-Newton form; damping is added by osb_reduce_partials).  gpart: blocks * P_actor floats. */
int osb_fvp_grid_blocks(long long total, int stride);
int osb_fvp_partials(const float* theta_actor, const float* vec, int O, int A, const float* obs,
                     long long total, int stride, float* gpart, void* stream);
/* Tensor-core Fisher-vector product (O <= 64): forward-mode tangent pass with stacked [W;V] weight
 * tiles (dmu scratch [total][A]) + the actor backward of the tensor-core gradient kernel.
 * gpart: osb_tc_grid_blocks(rows, 1) rows of P_actor floats, rows = ceil(total / stride);
 * stats_scratch: that many * 24 floats.  Reduce with osb_reduce_partials. */
int osb_fvp_partials_tc(const float* theta_actor, const float* vec, int O, int A, const float* obs,
                        long long total, int stride, float* dmu, float* gpart, float* stats_scratch,
                        void* stream);
/* Split-bf16 ("bf16x3") variant of osb_fvp_partials_tc (O <= 64): forward-mode tangent kernel on bf16x3 tiles
 * (csrc/fvp_x3.cu) + the bf16x3 actor backward with the tangent as output gradient: fp32-level F v on the tensor
 * cores.  NaturalPG._fvp, natural_pg.py:L74-119. */
int osb_fvp_partials_x3(const float* theta_actor, const float* vec, int O, int A, const float* obs,
                        long long total, int stride, float* dmu, float* gpart, float* stats_scratch,
                        void* stream);

/* ---- optimiser side --------------------------------------------------------------------------
 * osb_grad_reduce: grad <- sum of CTA partials (+ 2*critic_norm_coef*theta for critics,
 * policy_gradient.py:L431-433); advances adam_step[net]; accumulates train_stats[3][8]
 * ({sum of minibatch mean loss, mean ratio, mean kl, #minibatches}).  sumsq_part: 6*osb_optim_blocks.
 * osb_clip_adam: clip_grad_norm_ per network (do_clip) and torch.optim.Adam step (do_adam);
 * multi-rank order = clip -> all-reduce SUM -> grad_scale = 1/world -> Adam (policy_gradient.py:L437-443). */
int osb_optim_blocks(int O, int A);
int osb_grad_reduce(const float* gpart, const float* stats_part, int nblocks, int O, int A,
                    const float* theta, float* grad, float critic_norm_coef, int net_mask,
                    float* sumsq_part, int* adam_step, float* train_stats, const int* stop_flag,
                    void* stream);
int osb_clip_adam(float* grad, float* theta, float* adam_m, float* adam_v, const int* adam_step,
                  const float* sumsq_part, int O, int A, float max_grad_norm, float lr_actor,
                  float lr_critic_r, float lr_critic_c, float grad_scale, float critic_norm_coef,
                  float* train_stats, int do_clip, int do_adam, int net_mask, const int* stop_flag,
                  void* stream);
/* Single-rank fusion of osb_grad_reduce + osb_clip_adam (clip and step) in one cooperative launch. */
int osb_optim_fused(const float* gpart, const float* stats_part, int nblocks, int O, int A,
                    float* theta, float* grad, float* adam_m, float* adam_v, int* adam_step,
                    float critic_norm_coef, float max_grad_norm, float lr_actor, float lr_critic_r,
                    float lr_critic_c, int net_mask, float* sumsq_part, float* train_stats,
                    const int* stop_flag, void* stream);
/* Multi-rank fusion: reduce + clip + one-shot all-reduce over NVLink peer memory + Adam in one
 * cooperative kernel (reference order clip -> average -> step, policy_gradient.py:L437-443,
 * utils/distributed.py:L193-198).  Exchange buffers: every rank osb_p2p_alloc()s [2][P] floats and
 * [2][world] uint32 flags, the 64-byte cudaIpc handles are exchanged by the host, peers
 * osb_p2p_open() them; peer_buf / peer_flag are DEVICE arrays of `world` pointers.  step_id must
 * increase by one per call identically on every rank.  error_flag <- 1 on a peer timeout. */
int osb_p2p_alloc(long long bytes, void** ptr, unsigned char* handle64);
int osb_p2p_open(const unsigned char* handle64, void** ptr);
int osb_optim_fused_p2p(const float* gpart, const float* stats_part, int nblocks, int O, int A,
                        float* theta, float* grad, float* adam_m, float* adam_v, int* adam_step,
                        float critic_norm_coef, float max_grad_norm, float lr_actor,
                        float lr_critic_r, float lr_critic_c, int net_mask, float* sumsq_part,
                        float* train_stats, const int* stop_flag, void* peer_buf, void* peer_flag,
                        int world, int rank, unsigned step_id, int* error_flag, void* stream);
/* Lagrange.update_lagrange_multiplier (common/lagrange.py:L114-136) on the device: Adam step on
 * lambda with grad -(Jc - cost_limit), Jc = window_sums[1]/window_sums[3], clamp to
 * [0, upper_bound] (upper_bound < 0 = none).  state[4] = {lambda, m, v, t}.  nan_flag <- 1 when no
 * episode has finished yet (the reference asserts, naive_lagrange/ppo_lag.py:L74). */
int osb_lagrange_update(const double* window_sums, float cost_limit, float lambda_lr,
                        float upper_bound, float* state, int* nan_flag, void* stream);
/* PID-Lagrangian controller step (PIDLagrangian.pid_update, common/pid_lagrange.py:L95-125) in the
 * reference's Python-float (fp64) arithmetic.  pid_state: 64 doubles {integral, EMA(delta), EMA(Jc),
 * penalty, deque length, deque head, -, -, ring[pid_d_delay]}, initialised by the host to
 * {lagrangian_multiplier_init, 0, 0, 0, 1, 0, ..., ring[0] = 0}.  lagrange_state[0] <- (float) penalty.
 * Jc = window_sums[1] / window_sums[3]; an empty window sets *nan_flag. */
int osb_pid_lagrange_update(const double* window_sums, double pid_kp, double pid_ki, double pid_kd,
                            int pid_d_delay, double pid_delta_p_ema_alpha, double pid_delta_d_ema_alpha,
                            int sum_norm, int diff_norm, double penalty_max, double cost_limit,
                            double* pid_state, float* lagrange_state, int* nan_flag, void* stream);
/* kl = (float)(eval_out[0]/eval_out[4]); stops when (double)kl > target_kl, the reference's fp32 `kl.item() > target_kl`;
 * kl_state[4] = {last kl, passes done, stopped, 0}. */
int osb_kl_check(const double* eval_out, double target_kl, int early_stop, int* stop_flag,
                 float* kl_state, void* stream);
/* out[q] = scale * sum_b gpart[b*stride + q] + add_scale * add[q], q < n  (add may be NULL). */
int osb_reduce_partials(const float* gpart, int nblocks, int stride, int n, float scale,
                        const float* add, float add_scale, float* out, void* stream);
/* conjugate_gradients (utils/math.py:L86-132) as device-resident state: x, r, p [n],
 * cg_scalars[4] = {rdotr, converged, iterations, 0}; the caller computes z = F p between steps. */
int osb_cg_init(const float* b, int n, float* x, float* r, float* p, float* cg_scalars, void* stream);
int osb_cg_step(const float* z, int n, float* x, float* r, float* p, float* cg_scalars,
                float residual_tol, float eps, void* stream);
int osb_dot(const float* a, const float* b, int n, float* out, void* stream);
int osb_axpy(const float* x, const float* y, float alpha, int n, float* out, void* stream);

/* ---- epoch driver + NCCL -------------------------------------------------------------------
 * One epoch of PolicyGradient._update (policy_gradient.py:L345-405) issued from C: old-policy
 * snapshot, update_iters passes of minibatch steps (grad -> reduce -> clip -> [all-reduce] ->
 * Adam), full-batch KL after each pass, device-side early stop.  comm = handle from osb_nccl_init
 * (or NULL for a single rank).  With peer_buf / peer_flag (device arrays of `world_size` cudaIpc-mapped
 * pointers, see osb_p2p_alloc) the per-step gradient exchange is the fused one-shot NVLink kernel
 * osb_optim_fused_p2p instead of NCCL; NCCL then only carries the per-pass KL scalar. */
int osb_ppo_update_epoch(float* theta, float* grad, float* adam_m, float* adam_v, int* adam_step,
                         int O, int A, const float* obs, const float* act, const float* logp,
                         const float* adv_r, const float* adv_c, const float* tv_r,
                         const float* tv_c, float* mu_old, float* logstd_old, const float* moments,
                         const int* perm, long long total, unsigned perm_seed, int batch_size,
                         int update_iters, int loss_kind, float clip, float entropy_coef,
                         float focops_lam, float focops_eta, const float* lagrange, int net_mask,
                         float critic_norm_coef, float max_grad_norm, float lr_actor,
                         float lr_critic, double target_kl, int kl_early_stop, float* gpart,
                         float* stats_part, float* sumsq_part, float* train_stats, double* eval_ws,
                         double* eval_out, int* stop_flag, float* kl_state, int precision,
                         void* comm, int world_size, void* peer_buf, void* peer_flag, int rank,
                         int* p2p_error, void* stream);
/* NCCL via dlopen(libpath) of the libnccl.so.2 torch already loaded (distributed.py:L142-228). */
int osb_nccl_unique_id(const char* libpath, unsigned char* id128);
int osb_nccl_init(const char* libpath, const unsigned char* id128, int nranks, int rank,
                  void** comm_out);
int osb_nccl_allreduce(void* comm, void* buf, long long count, int is_f64, void* stream);
int osb_nccl_destroy(void* comm);

/* ---- diagnostics ---------------------------------------------------------------------------
 * One tcgen05 (kind::tf32, TMEM accumulator) GEMM D = A * B^T on a single CTA with every operand
 * major combination; out[128][N] is the raw TMEM dump.  Pins the descriptor / swizzle conventions
 * the tensor-core MLP tiles rely on (tests/test_umma_gpu.py). */
/* cycles for `reps` back-to-back M x N x 8 tf32 MMAs: out[0] issue->completion, out[1] issue loop. */
int osb_umma_timing(int M, int N, int reps, long long* out, void* stream);
int osb_umma_selftest(const float* A, const float* B, int M, int N, int K, int a_mn, int b_mn,
                      float* out, void* stream);

/* Split-bf16 ("bf16x3", kind::f16) building blocks of the parity-grade tensor-core mode (csrc/x3.cuh):
 * one single-CTA GEMM D = A * B^T with A [M][K], B [N][K] (row-major fp32 in global memory), each operand
 * staged as three bf16 tiles (SW128 or SW32) consumed K-major or MN-major; out[128][N] = raw TMEM dump
 * (tests/test_x3_gpu.py).  The timing / epilogue probes report clock64 cycles. */
int osb_x3_selftest(const float* A, const float* B, int M, int N, int K, int a_mn, int b_mn, int a_sw,
                    int b_sw, int b_ones, float* out, void* stream);
int osb_x3_debug_buffer(long long* buf);
/* development aid: clock64 stamps of CTA 0 of the streaming GAE kernel (tools/gae_stage_times.py); NULL turns it off */
int osb_gae_debug_buffer(long long* buf);
/* same for the persistent rollout kernel (tools/rollout_stage_times.py) */
int osb_rollout_debug_buffer(long long* buf);
int osb_x3_selftest_dbg(const float* A, const float* B, int M, int N, int K, int a_mn, int b_mn, int a_sw,
                        int b_sw, int b_ones, int a_lbo, int a_sbo, int b_lbo, int b_sbo, float* out, void* stream);
int osb_x3_timing(int M, int N, int reps, int style, long long* out, void* stream);
int osb_x3_epilogue_probe(int cols, int reps, int mode, long long* out, float* sink, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* OMNISAFE_B200_H */
