/* jorldy_b200 — C ABI of the B200-native rollout-collect -> buffer -> learn() core.
 *
 * The reference (kakaoenterprise/JORLDY) is pure Python and has no FFI of its own; its plugin
 * boundary is the Python classes Agent / Env / Buffer / Network / Optimizer.  This header is the
 * boundary a maintainer would bind from those classes (ctypes stub in INTEGRATION.md): plain
 * pointers and sizes, no torch types.  Each entry point names the reference code it replaces.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name says host; buffers are caller-owned
 *     (the Python host allocates them as torch tensors) and must stay alive until the stream
 *     has drained;
 *   - `stream` is a cudaStream_t passed as void*; calls only enqueue work (async w.r.t. host);
 *   - return value: 0 = ok, negative errno-style code otherwise (-22 bad argument, -5 CUDA
 *     launch/runtime failure).  Nothing throws;
 *   - one learner thread per handle/stream, as in the reference (run_mode.py:327).
 */
#ifndef JORLDY_B200_H
#define JORLDY_B200_H

#include <stdint.h>

#ifdef __cplusplus
#define JB_API extern "C"
#else
#define JB_API
#endif

/* ---------------------------------------------------------------------------------------------
 * Environments — jorldy/core/env/gym_env.py:61-83 (Cartpole.step / _Gym.reset :32-36),
 * :86-95 (Pendulum, MountainCar) + run_mode.py:91 auto-reset line; gym 0.23.0 physics.
 * kind: 0 cartpole (phys[n,4], obs[n,4]), 1 pendulum (phys[n,2], obs[n,3]),
 *       2 mountain_car (phys[n,2], obs[n,2]).
 * action_kind: 0 int64, 1 int32, 2 float32.
 * stats (may be NULL): [2] floats, += {episodes finished, sum of their scores}.
 * ------------------------------------------------------------------------------------------- */
JB_API int jb_env_classic_reset(int kind, double* phys, float* obs, int32_t* elapsed, int64_t* episode,
                                float* score, const uint8_t* mask, uint64_t seed, uint64_t stream_base,
                                int n, void* stream);
JB_API int jb_env_classic_step(int kind, double* phys, float* obs, int32_t* elapsed, int64_t* episode,
                               float* score, const void* action, int action_kind, float* next_obs,
                               float* reward, float* done, float* stats, int auto_reset, int max_steps,
                               uint64_t seed, uint64_t stream_base, int n, void* stream);

/* ---------------------------------------------------------------------------------------------
 * GAE — jorldy/core/agent/ppo.py:95-110.  Arrays are [N,T] row-major f32.
 * next_value may be NULL: then V(s'_t) = value[:,t+1] and last_value[N] closes the row.
 * ------------------------------------------------------------------------------------------- */
JB_API int jb_gae(const float* reward, const float* done, const float* value, const float* next_value,
                  const float* last_value, int N, int T, float gamma, float lambda, int standardize,
                  float* adv, float* ret, void* stream);

/* Synthetic continuous-control env with MuJoCo-task dimensions (replaces gym + mujoco_py behind
 * jorldy/core/env/mujoco.py:25-58; BASELINE configs[4]: obs 11 / act 3).  s' = tanh(Ws s + Wa a) + 0.01 N(0,I),
 * reward = -|s'|^2 / D, done ~ Bernoulli(p_done) or TimeLimit; obs f32 [n,D], action f32 [n,A]. */
JB_API int
jb_env_synth_reset(float* obs, int32_t* elapsed, int64_t* episode, float* score, uint64_t seed,
                   uint64_t stream_base, int n, int D, void* stream);
JB_API int
jb_env_synth_step(float* obs, int32_t* elapsed, int64_t* episode, int64_t* tcount, float* score,
                  const float* action, const float* Ws, const float* Wa, float* next_obs, float* reward,
                  float* done, float* stats, int auto_reset, int max_steps, float p_done, uint64_t seed,
                  uint64_t stream_base, int n, int D, int A, void* stream);

/* Replay ring rows (jorldy/core/buffer/replay_buffer.py:16-31, base.py:42-56 stack_transition): a field is a
 * [capacity, row_bytes] byte matrix; store scatters n batch rows to ring positions, gather collects a minibatch. */
JB_API int
jb_replay_store(void* ring, const void* batch, const int64_t* pos, int n, long long row_bytes, void* stream);
JB_API int
jb_replay_gather(const void* ring, const int64_t* idx, int n, long long row_bytes, void* batch, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Frame-deduplicated replay (csrc/frame_replay.cu) — replay_buffer.py:16-31 (ring write / sample), base.py:42-56
 * (stack_transition), per_buffer.py:95-96 (PER gather) for uint8 frame-stack fields [S, H, W], H*W % 16 == 0.
 * Each distinct frame is stored once: frames [F, frame_bytes] holds frame id i at row i % F; ref [nf, capacity, S] int64
 * the ids of each slot's stacks, min_ref [capacity] the oldest of them (INT64_MAX when empty);
 * ctl int64[4] = {next id, first id of the last store, its new frames, sticky overflow flag}.
 * host_fields is a HOST array of nf (<= 4) device pointers, field f = [n, S, frame_bytes]; row t*N + r is actor r at step t.
 *   jb_frame_plan    hashes u64[n*nf*S] (scratch); per actor, in row order: reuse a frame of hist_id/hist_h [N,16] (most
 *                    recently used first, byte-compared, id >= next id - F) or take the actor's next new frame.
 *                    codes [n*nf*S] = pool id or -(j+1), newsrc [n*nf*S] = batch frame of new frame j of actor r at r*(n/N)*nf*S + j, counts [N]
 *   jb_frame_assign  offs [N] = exclusive scan of counts (ids actor-major), ctl update, and the overflow check over the
 *                    min_ref of the slots outside [start, start+n) (mod capacity) and the n_codes reused ids in codes
 *   jb_frame_commit  new frames -> frames (not while the flag is set), ref / min_ref of the rows written, history -> ids
 *   jb_frame_gather  out [B, S, frame_bytes] = frames[ref[idx[b], s] % F] for one field's ref table
 * ------------------------------------------------------------------------------------------- */
JB_API int jb_frame_plan(const void* host_fields, int nf, int n, int N, int S, long long frame_bytes, const uint8_t* frames,
                         int64_t F, uint64_t* hashes, const int64_t* ctl, int64_t* hist_id, uint64_t* hist_h, int64_t* codes,
                         int64_t* newsrc, int64_t* counts, void* stream);
JB_API int jb_frame_assign(const int64_t* counts, int N, int64_t F, const int64_t* min_ref, int64_t capacity, int64_t start,
                           int64_t n, const int64_t* codes, int64_t n_codes, int64_t* offs, int64_t* ctl, void* stream);
JB_API int jb_frame_commit(const void* host_fields, int nf, int n, int N, int S, long long frame_bytes, uint8_t* frames,
                           int64_t F, const int64_t* ctl, const int64_t* counts, const int64_t* offs, const int64_t* newsrc,
                           const int64_t* codes, int64_t* ref, int64_t* min_ref, int64_t capacity, int64_t start,
                           int64_t* hist_id, void* stream);
JB_API int jb_frame_gather(const uint8_t* frames, int64_t F, long long frame_bytes, const int64_t* ref, int S,
                           const int64_t* idx, int B, uint8_t* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * PER sum-tree — jorldy/core/buffer/per_buffer.py:19-101.  tree is f64[2*capacity-1].
 * ------------------------------------------------------------------------------------------- */
JB_API int jb_per_update(double* tree, int64_t capacity, const int64_t* tree_idx, int64_t first_idx,
                         const double* new_p, const double* fill_p, double* max_priority, int B,
                         void* stream);
JB_API int jb_per_sample(const double* tree, int64_t capacity, int64_t counter, int B, double beta,
                         double uniform_sample_prob, const double* u_a, const double* u_b, uint64_t seed,
                         uint64_t rng_ctr, const double* shard_prob, const int64_t* global_counter,
                         int64_t* out_idx, double* out_w, double* out_p, double* out_stats, int normalize,
                         void* stream);
JB_API int jb_per_scale_weights(double* w, const double* wmax, int B, void* stream);
JB_API int jb_per_rebuild(double* tree, int64_t capacity, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Dense layers — jorldy/core/network/head.py:6-18, q_network.py, policy_value.py, dueling.py
 * (torch.nn.Linear: weight [out,in]) and network/utils.py:55-86 (NoisyNet: weight [in,out]).
 * ------------------------------------------------------------------------------------------- */
JB_API int jb_gemm(const float* A, int lda, int a_kc, const float* B, int ldb, int b_kc, float* C, int ldc,
                   int M, int N, int K, const float* bias, int relu, const float* mask, int ldmask,
                   float* rowsum_a, int accumulate, void* stream);
JB_API int jb_linear_fwd(const float* x, const float* w, const float* b, float* y, int M, int in_f, int out_f,
                         int relu, void* stream);
/* tcgen05 / TMEM 3xTF32 forward for large M (M % 128 == 0, out_f % 128 == 0, in_f % 32 == 0); -22 otherwise */
JB_API int jb_linear_fwd_tc(const float* x, const float* w, const float* b, float* y, int M, int in_f, int out_f,
                            int relu, void* stream);
JB_API int jb_linear_bwd_dx(const float* dy, const float* w, float* dx, int M, int in_f, int out_f,
                            const float* relu_act, void* stream);
JB_API int jb_linear_bwd_dw(const float* dy, const float* x, float* dw, float* db, int M, int in_f, int out_f,
                            void* stream);
JB_API int
jb_linear_bwd_dw_splitk(const float* dy, const float* x, float* dw, float* db, int M, int in_f, int out_f,
                        float* workspace, int splits, void* stream);
JB_API int jb_linear_io_fwd(const float* x, const float* w, const float* b, float* y, int M, int in_f, int out_f,
                            int relu, void* stream);
JB_API int jb_linear_io_bwd_dx(const float* dy, const float* w, float* dx, int M, int in_f, int out_f,
                               const float* relu_act, void* stream);
JB_API int jb_linear_io_bwd_dw(const float* dy, const float* x, float* dw, int M, int in_f, int out_f, void* stream);
JB_API int jb_colsum(const float* x, int M, int N, float* out, int accumulate, void* stream);
JB_API int jb_mlp_in_fwd(const float* x, const int32_t* idx, const float* w1, const float* b1, int M, int D, int H,
                         float* h1, float* xg, void* stream);
JB_API int jb_heads_fwd(const float* h, int M, int H, const float* w0, const float* b0, int n0, const float* w1,
                        const float* b1, int n1, const float* w2, const float* b2, int n2, float* out, void* stream);
JB_API int jb_heads_bwd_dx(const float* dout, const float* h, int M, int H, const float* w0, int n0, const float* w1,
                           int n1, const float* w2, int n2, float* dh, void* stream);
JB_API int jb_heads_bwd_dw(const float* dout, const float* h, int M, int H, float* dw0, float* db0, int n0, float* dw1,
                           float* db1, int n1, float* dw2, float* db2, int n2, void* stream);

/* ---------------------------------------------------------------------------------------------
 * PPO — jorldy/core/agent/ppo.py:54-69 (act), :83-93 (value / log_prob_old), :127-162 (loss).
 * `out` is the [M,nout] pre-activation head output: discrete [logits(A)|v], continuous
 * [mu(A)|log_std(A)|v].
 * ------------------------------------------------------------------------------------------- */
JB_API int jb_ppo_act_discrete(const float* out, int M, int A, int nout, const float* u, uint64_t seed,
                               uint64_t stream_base, uint64_t ctr, long long* row_ctr, int greedy, int64_t* action,
                               void* stream);
JB_API int jb_ppo_act_continuous(const float* out, int M, int A, int nout, const float* normal, uint64_t seed,
                                 uint64_t stream_base, uint64_t ctr, long long* row_ctr, int greedy, float* action,
                                 void* stream);
JB_API int jb_ppo_prepass_discrete(const float* out, const int32_t* action, int M, int A, int nout, float* value,
                                   float* logp_old, void* stream);
JB_API int jb_ppo_prepass_continuous(const float* out, const float* action, int M, int A, int nout, float* value,
                                     float* logp_old, void* stream);
JB_API int jb_take_minibatch(const int32_t* perm, long long* cursor, int B, int32_t* cur_idx, void* stream);
JB_API int jb_ppo_loss(int continuous, const float* out, const int32_t* idx, const void* action, const float* adv,
                       const float* ret, const float* value_old, const float* logp_old, int B, int A, int nout,
                       float eps_clip, float vf_coef, float ent_coef, float* dout, float* stats, float* acc,
                       void* stream);

/* ---------------------------------------------------------------------------------------------
 * Synthetic Atari-shaped env — observation contract of jorldy/core/env/atari.py:56-61,112,145-160.
 * ------------------------------------------------------------------------------------------- */
JB_API int jb_env_frames_reset(uint8_t* obs, int64_t* fcount, float* score, uint64_t seed, uint64_t stream_base, int n,
                               void* stream);
JB_API int jb_env_frames_step(uint8_t* obs, int64_t* fcount, float* score, uint8_t* next_obs, float* reward, float* done,
                              float* stats, int auto_reset, uint64_t seed, uint64_t stream_base, int n, void* stream);

/* ---------------------------------------------------------------------------------------------
 * CNN head lowering — jorldy/core/network/head.py:21-61 (im2col / col2im around jb_gemm).
 * ------------------------------------------------------------------------------------------- */
JB_API int jb_im2col_u8(const uint8_t* x, int B, int C, int H, int W, int KH, int KW, int S, float* col, void* stream);
/* Same, with output row b read from input row idx[b] (int32, < rows of x; NULL: row b): gathers a minibatch of
 * uint8 [rows, C, H, W] stacks inside conv1's im2col.  jb_im2col_u8 is this call with idx = NULL. */
JB_API int jb_im2col_u8_rows(const uint8_t* x, const int32_t* idx, int B, int C, int H, int W, int KH, int KW, int S,
                             float* col, void* stream);
JB_API int jb_im2col_nhwc(const float* x, int B, int C, int H, int W, int KH, int KW, int S, float* col, void* stream);
JB_API int jb_col2im_nhwc(const float* dcol, int B, int C, int H, int W, int KH, int KW, int S, const float* relu_act,
                          float* dx, void* stream);
JB_API int jb_nhwc_to_nchw(const float* x, int B, int P, int C, float* y, void* stream);
JB_API int jb_nchw_to_nhwc(const float* x, int B, int P, int C, const float* relu_act, float* y, void* stream);

/* Persistent minibatch-loop kernel (csrc/ppo_fused.cu); `host_args` points to a jb_ppo_fused_args
 * (include/jorldy_b200_fused.h) in HOST memory. */
JB_API int jb_ppo_fused_args_size(void);
JB_API int jb_ppo_fused_max_ctas(void);
JB_API int jb_ppo_fused_run(const void* host_args, void* stream);
/* Debug aid: clock64 stamps of the last step of the previous run made with JB_FUSED_SKIP=256 in the
 * environment; host_out receives 256 x 32 long longs. */
JB_API int jb_ppo_fused_trace(long long* host_out);

/* ---------------------------------------------------------------------------------------------
 * Value-based learners — jorldy/core/agent/dqn.py:99-138, double.py:25-41, multistep.py:41-50,
 * per.py:50-77, ape_x.py:63-116; dueling combine network/dueling.py:21-35, rainbow.py net :66-94.
 * ------------------------------------------------------------------------------------------- */
JB_API int jb_q_act(const float* q, int M, int A, float eps, const float* eps_rows, const float* u, uint64_t seed,
                    uint64_t stream_base, long long* row_ctr, int64_t* action, float* q_sel, void* stream);
JB_API int jb_dueling_fwd(const float* adv, const float* val, int B, int A, int K, float* out, void* stream);
JB_API int jb_dueling_bwd(const float* dout, int B, int A, int K, float* dadv, float* dval, void* stream);
JB_API int jb_td_loss(const float* q, const float* q_next, const float* qt_next, const void* action, int action_kind,
                      const float* reward, const float* done, const double* weights, int B, int A, float gamma,
                      float alpha, int n_step, int double_q, int loss_kind, int order, float* dq, double* prio,
                      float* stats, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Distributional learners — jorldy/core/agent/c51.py:62-135, rainbow.py:167-235, :285-292.
 * ------------------------------------------------------------------------------------------- */
JB_API int jb_c51_loss(const float* logits, const float* next_online, const float* next_target, const void* action,
                       int action_kind, const float* reward, const float* done, const double* weights, const float* z,
                       int B, int A, int K, float gamma, float v_min, float v_max, float alpha, int n_step, int variant,
                       float* dlogits, float* kl, double* prio, float* stats, float* scratch, void* stream);
JB_API int jb_c51_q(const float* logits, const float* z, int M, int A, int K, float* q, void* stream);

/* ---------------------------------------------------------------------------------------------
 * NoisyNet — jorldy/core/network/utils.py:55-86 (noisy_l), factorised noise.
 * ------------------------------------------------------------------------------------------- */
JB_API int jb_noisy_make(const float* mu_w, const float* sig_w, const float* mu_b, const float* sig_b, int in_f,
                         int out_f, const float* eps_i, const float* eps_j, uint64_t seed, uint64_t stream_id,
                         long long* draw_ctr, int is_train, float* f_i, float* f_j, float* w_eff, float* b_eff,
                         void* stream);
JB_API int jb_noisy_grad(const float* dw_eff, const float* db_eff, const float* f_i, const float* f_j, int in_f,
                         int out_f, float* dmu_w, float* dsig_w, float* dmu_b, float* dsig_b, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Optimisers — torch.optim.Adam / RMSprop(centered) via jorldy/core/optimizer/__init__.py:31,
 * torch.nn.utils.clip_grad_norm_ (ppo.py:166-168, ape_x.py:119), target copy dqn.py:153-154.
 * ------------------------------------------------------------------------------------------- */
JB_API int jb_grad_partials_count(long long P);
JB_API int jb_grad_sumsq(const float* g, long long P, float* partials, long long* step, void* stream);
JB_API int jb_adam_step(float* p, const float* g, float* m, float* v, long long P, const float* lr, float beta1,
                        float beta2, float eps, const long long* step, const float* partials, int n_partials,
                        float max_norm, float* norm_out, void* stream);
JB_API int jb_rmsprop_centered_step(float* p, const float* g, float* square_avg, float* grad_avg, long long P,
                                    const float* lr, float alpha, float eps, const float* partials, int n_partials,
                                    float max_norm, float* norm_out, void* stream);
JB_API int jb_copy_f32(float* dst, const float* src, long long P, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Continuous off-policy family (SURVEY.md 8f-4) — jorldy/core/agent/ddpg.py, td3.py, sac.py; the row / element-wise
 * steps between the dense layers (csrc/actor_critic.cu).
 *   jb_soft_update     t := tau p + (1 - tau) t over a flat buffer            ddpg.py:160-164, td3.py:190-196, sac.py:262-266
 *   jb_tanh_act        out = clip(tanh(pre) + clip(noise*scale, +-noise_clip), +-out_clip); noise NULL: plain tanh head
 *                      (network/policy.py:19-20; td3.py:141-142 act noise; td3.py:153-156 target smoothing)
 *   jb_tanh_bwd        dpre = da (1 - a^2)
 *   jb_ou_act          action = tanh(pre) + clip(X, +-1) with one Ornstein-Uhlenbeck process X[M,A] (f64) per env row and
 *                      ONE normal per row and step (agent/utils.py:8-26, ddpg.py:113-118); greedy: tanh(pre)
 *   jb_philox_fill     standard normals (kind 0) / uniforms in [lo,hi) (kind 1) from the device Philox stream
 *   jb_ac_critic_loss  y = r + ((1-d) gamma)(min(nq1,nq2) + alpha(-next_logp)); dq_i = 2(q_i - y)/B;
 *                      stats = {mse1, mse2, max y}; q2/nq2/alpha/next_logp may be NULL    ddpg.py:131-136, td3.py:150-168, sac.py:172-204
 *   jb_ac_neg_mean     stat = -mean(q), dq = -1/B                              ddpg.py:143-144, td3.py:176-177
 *   jb_sac_sample      a = tanh(mu + std eps), logp with the tanh correction  sac.py:151-160, network/policy.py:50-56
 *   jb_sac_minq        dq_i of L = mean(alpha logp - min(q1,q2)); stats = {L, mean min q, mean entropy, mean entropy - target}
 *   jb_sac_actor_bwd   d L / d (raw mu | raw log_std) [B,2A] from d L / d action and the alpha logp term   sac.py:222-236
 *   jb_sac_alpha       alpha_loss = log_alpha * stats4[3]; alpha := exp(log_alpha); grad := stats4[3]     sac.py:238-246
 * ------------------------------------------------------------------------------------------- */
JB_API int jb_soft_update(float* target, const float* online, int64_t n, double tau, void* stream);
JB_API int jb_tanh_act(const float* pre, const float* noise, int64_t n, float scale, float noise_clip, float out_clip,
                       float* out, void* stream);
JB_API int jb_tanh_bwd(const float* da, const float* a, int64_t n, float* dpre, void* stream);
JB_API int jb_ou_act(const float* pre, int M, int A, double* X, const double* normal, uint64_t seed, uint64_t stream_base,
                     long long* row_ctr, double theta, double mu, double sigma, int greedy, float* action, void* stream);
JB_API int jb_philox_fill(float* out, int64_t n, int kind, float lo, float hi, uint64_t seed, uint64_t stream_base,
                          uint64_t ctr, long long* ctr_dev, void* stream);
JB_API int jb_ac_critic_loss(const float* q1, const float* q2, const float* nq1, const float* nq2, const float* alpha,
                             const float* next_logp, const float* reward, const float* done, int B, float gamma,
                             float* dq1, float* dq2, float* stats, void* stream);
JB_API int jb_ac_neg_mean(const float* q, int B, float* dq, float* stat, void* stream);
JB_API int jb_sac_sample(const float* raw, int nout, const float* eps, int M, int A, float* action, float* logp,
                         void* stream);
JB_API int jb_sac_minq(const float* q1, const float* q2, const float* logp, const float* alpha, float target_entropy,
                       int B, float* dq1, float* dq2, float* stats, void* stream);
JB_API int jb_sac_actor_bwd(const float* raw, int nout, const float* eps, const float* action, const float* da,
                            const float* alpha, int B, int A, float* dout, void* stream);
JB_API int jb_sac_alpha(const float* log_alpha, const float* stats4, float* alpha, float* grad, float* alpha_loss,
                        void* stream);

#endif /* JORLDY_B200_H */
