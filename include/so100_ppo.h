/*
 * so100_ppo.h — C ABI of the fused PPO learner kernels in libso100_b200.so (SURVEY.md §8 f, rank 1).
 *
 * The reference trains with stable_baselines3.PPO("MlpPolicy", env, device='cpu') (src/so100_mujoco_rl/main.py:56-64,
 * 234-238).  These entry points are the hand-written sm_100a replacement of what SB3 runs per rollout step and per
 * minibatch for that exact policy: ActorCriticPolicy with net_arch dict(pi=[64,64], vf=[64,64]), tanh, a
 * state-independent log_std (DiagGaussianDistribution), clipped-surrogate + MSE value loss, per-minibatch advantage
 * normalisation, global-norm gradient clipping and Adam — SB3 2.6.0 defaults.
 *
 *   so100_ppo_act        <- ActorCriticPolicy.forward (collect_rollouts): actions, values, log-probs
 *   so100_ppo_post_step  <- OnPolicyAlgorithm.collect_rollouts bookkeeping: TimeLimit bootstrap
 *                           reward += gamma * V(terminal_observation), done flags, Monitor statistics
 *   so100_ppo_gae        <- RolloutBuffer.compute_returns_and_advantage
 *   so100_ppo_permutation <- RolloutBuffer.get: the per-epoch shuffle of the sample indices
 *   so100_ppo_grad       <- PPO.train: policy.evaluate_actions + losses + loss.backward() for one minibatch
 *   so100_ppo_adam       <- clip_grad_norm_ + Adam.step
 *   so100_ppo_sde_act, so100_ppo_sde_grad <- the same two with use_sde=True (gSDE, at the end of this header)
 *
 * All pointers are DEVICE pointers owned by the caller (torch tensors); nothing is allocated, nothing synchronises;
 * work is enqueued on `stream`.  Return value: SO100_OK or a negative SO100_ERR_* code (so100_last_error()).
 *
 * Parameter vector (float32, so100_ppo_param_count(obs_dim) entries), all matrices row-major [out][in]:
 *   pi: W1[64][od] b1[64] W2[64][64] b2[64] W3[6][64] b3[6]   vf: W1[64][od] b1[64] W2[64][64] b2[64] W3[1][64] b3[1]
 *   log_std[6]
 * = SB3's mlp_extractor.policy_net.{0,2}, action_net, mlp_extractor.value_net.{0,2}, value_net, log_std.
 */
#ifndef SO100_PPO_H
#define SO100_PPO_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SO100_PPO_HIDDEN 64
#define SO100_PPO_ACT 6
#define SO100_PPO_TILE 64       /* envs per CTA tile of the inference kernel (the gradient kernel uses 32-sample tiles) */
#define SO100_PPO_MAX_CTAS 1024 /* upper bound of the gradient kernel's grid (workspace sizing) */

int so100_ppo_param_count(int obs_dim); /* 10829 for obs_dim 15, 9933 for obs_dim 8; <0 if unsupported (obs_dim must be 1..16) */
/* floats of workspace so100_ppo_grad needs: per-CTA partial gradients + loss partial sums */
int64_t so100_ppo_workspace_floats(int obs_dim);

/*
 * Rollout inference for n envs: mean = pi(obs), value = vf(obs), action = mean + exp(log_std) * N(0,1) (Philox keyed by
 * (seed, env_offset + env, tick)), log_prob of the unclipped action.  act_clip = clip(action, -1, 1) is what SB3 hands
 * to env.step for a Box space.  Optional outputs may be NULL; obs_copy receives obs (the rollout buffer slot).
 */
int so100_ppo_act(int obs_dim, const float *params, const float *obs, int n, uint64_t seed, int64_t env_offset,
                  uint32_t tick, int deterministic, float *act_raw, float *act_clip, float *logp, float *value,
                  float *obs_copy, void *stream);

/*
 * After env.step: reward_out = reward + (truncated ? gamma * V(terminal_obs) : 0), done_out = terminated | truncated
 * (as float), and acc[4] (double) += {sum reward, sum ep_return over done, sum ep_len over done, done count}.
 */
int so100_ppo_post_step(int obs_dim, const float *params, int n, const float *reward, const uint8_t *terminated,
                        const uint8_t *truncated, const float *terminal_obs, const float *ep_return,
                        const int32_t *ep_len, float gamma, float *reward_out, float *done_out, double *acc,
                        void *stream);

/* GAE(lambda) over [T][N] buffers; done[t] = the episode ended AT step t.  adv, ret: [T][N]. */
int so100_ppo_gae(const float *rew, const float *val, const float *done, const float *last_val, int T, int N,
                  float gamma, float lam, float *adv, float *ret, void *stream);

/*
 * idx_out[0..n) = a keyed pseudo-random permutation of 0..n-1 (what np.random.permutation gives SB3's RolloutBuffer.get
 * once per epoch): 6-round Feistel network with cycle walking, one launch, every index exactly once for any key.
 */
int so100_ppo_permutation(int n, uint64_t key, int64_t *idx_out, void *stream);

/*
 * Gradient of  pg_loss + vf_coef * v_loss - ent_coef * entropy  over the minibatch idx[0..mb) of the flattened rollout
 * buffers (obs [S][od], act [S][6], logp_old [S], adv [S], ret [S]); advantages are normalised over the minibatch
 * ((a - mean) / (std_unbiased + 1e-8)) when normalize != 0 and mb > 1; a one-sample minibatch keeps its raw advantage,
 * as SB3 2.x does (normalising one sample would zero the policy gradient).  grad [param_count] is overwritten; loss_out[3] =
 * {pg_loss, v_loss, approx_kl}.  workspace: so100_ppo_workspace_floats() floats.  Deterministic (fixed tile order).
 */
int so100_ppo_grad(int obs_dim, const float *params, const float *obs, const float *act, const float *logp_old,
                   const float *adv, const float *ret, const int64_t *idx, int mb, float clip_range, float vf_coef,
                   float ent_coef, int normalize, float *workspace, float *grad, float *loss_out, void *stream);

/*
 * torch.nn.utils.clip_grad_norm_(max_norm) followed by one torch.optim.Adam step (no amsgrad, no weight decay).
 * step_count (device int32) is incremented; grad_scale multiplies grad first (1/world after an all-reduce sum), and the
 * norm that is clipped is that of the scaled gradient.  max_grad_norm <= 0 disables clipping.
 */
int so100_ppo_adam(int n_params, float *params, const float *grad, float *exp_avg, float *exp_avg_sq,
                   int32_t *step_count, float grad_scale, float max_grad_norm, float lr, float beta1, float beta2,
                   float eps, void *stream);

/*
 * Generalized State-Dependent Exploration (gSDE): SB3's PPO(use_sde=True) with StateDependentNoiseDistribution
 * (full_std, no expln, learn_features=False, epsilon 1e-6).  h = the policy tower's second hidden layer (64 tanh outputs).
 *
 * Parameter vector (so100_ppo_sde_param_count(obs_dim) entries): the layout above with log_std[6] replaced by
 * log_std[64][6] (row-major, SB3's tensor shape), still last.  Every offset before log_std is the same in both layouts,
 * which is why so100_ppo_post_step (value tower only), so100_ppo_gae, so100_ppo_permutation and so100_ppo_adam (with
 * n_params = the gSDE count) serve both unchanged.
 *
 * Distribution:  std = exp(log_std), S = exp(2 log_std);  E[k][j] = std[k][j] z[k][j] per env;
 *   action = mean + h E,  var_j = sum_k h_k^2 S[k][j],  scale_j = sqrt(var_j + 1e-6),  log_prob = log N(action; mean, scale),
 *   entropy = sum_j (0.5 + log sqrt(2 pi) + log scale_j).  The variance sends gradient to log_std only, never to the tower.
 *
 * Draw layout of E (not stored: regenerated in registers at every call): normal number i = 64 j + k of env e is position
 * i % 4 of the Philox-4x32-10 block keyed (seed_lo, seed_hi) with counter (env_offset + e, noise_key, 0x5D00 + i / 4, 0);
 * words (0, 1) and (2, 3) of a block give positions (0, 1) and (2, 3) through the Box-Muller transform of so100_ppo_act:
 *   u1 = ((w0 >> 8) + 0.5) 2^-24,  u2 = (w1 >> 8) 2^-24,  r = sqrt(-2 log u1),  z0 = r cos(2 pi u2),  z1 = r sin(2 pi u2).
 * The same (seed, env, noise_key) and log_std give the same E, whatever the call's n, env_offset split or tick.
 */
int so100_ppo_sde_param_count(int obs_dim);           /* 11207 for obs_dim 15, 10311 for obs_dim 8; <0 if unsupported */
int64_t so100_ppo_sde_workspace_floats(int obs_dim);  /* workspace of so100_ppo_sde_grad */

/* so100_ppo_act's contract with the gSDE distribution; noise_key (in place of tick) selects the exploration matrices.
 * deterministic != 0: act_raw = mean, and logp is the log-prob of the mean. */
int so100_ppo_sde_act(int obs_dim, const float *params, const float *obs, int n, uint64_t seed, int64_t env_offset,
                      uint32_t noise_key, int deterministic, float *act_raw, float *act_clip, float *logp, float *value,
                      float *obs_copy, void *stream);

/* so100_ppo_grad's signature and contract with the gSDE log-prob and entropy; grad [so100_ppo_sde_param_count],
 * workspace so100_ppo_sde_workspace_floats() floats. */
int so100_ppo_sde_grad(int obs_dim, const float *params, const float *obs, const float *act, const float *logp_old,
                       const float *adv, const float *ret, const int64_t *idx, int mb, float clip_range, float vf_coef,
                       float ent_coef, int normalize, float *workspace, float *grad, float *loss_out, void *stream);

#ifdef __cplusplus
}
#endif
#endif
