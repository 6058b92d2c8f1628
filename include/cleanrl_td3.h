/*
 * cleanrl_td3.h — C ABI of the TD3 part of libcleanrl_cuda.so
 *
 * Same library, same conventions as cleanrl_ddpg.h (included below): every function returns int (0 = CRL_OK), all
 * indices are 0-based, host pointers are borrowed for the call only, and there is no CPU fallback (CRL_ERR_CUDA without
 * an sm_100 device).
 *
 * ---- TD3 (an extension: the reference has no TD3) ----------------------------------------------------------------
 * CleanRL-Python's td3_continuous_action.py on Pendulum with the 64-wide nets of cleanrl_ddpg.h. Everything not listed
 * here is exactly the DDPG definition of cleanrl_ddpg.h: env and observation, the actor mu (4,481 floats), the critic
 * architecture, now used twice as qf1 and qf2 (4,545 floats each), the acting rule (warm-up uniform or
 * clamp(mu + 2 exploration_noise z, -2, 2), Philox stream 5), ring order, the learning gate and batch sampling (keyed
 * permutation, Philox stream 6, counter = learning-step index). With the same seed and config, TD3 and DDPG act alike
 * up to the first learning step, so their replay buffers are bit-identical until then.
 * What TD3 adds, at learning step t (0-based index) on the sampled batch:
 *  - target smoothing: for sample b (its position in the batch, not its ring row) r = Philox(seed, word = b,
 *    counter = t, stream 7); z_b = Box-Muller of u1 = ((r0 >> 8) + 1) 2^-24 and u2 = (r1 >> 8) 2^-24;
 *    eps_b = clamp(policy_noise z_b, -noise_clip, noise_clip) * 2; a'_b = clamp(mu'(s'_b) + eps_b, -2, 2); all in
 *    Float32, in this order.
 *  - target: y = r + gamma (1 - d) min(qf1'(s', a'), qf2'(s', a')) in Float64, with DDPG's expression.
 *  - critic step: loss mean((qf1(s,a) - y)^2) + mean((qf2(s,a) - y)^2), one Adam step of both critics. CleanRL's single
 *    q_optimizer over both parameter lists is element-wise, so it is two Adams that share a step count; the two losses
 *    are reported separately.
 *  - actor step on every policy_frequency-th learning step (learn_steps % policy_frequency == 0 after counting it;
 *    CleanRL gates on global_step % policy_frequency, the same steps when one env learns on every step and
 *    learning_starts is a multiple of policy_frequency): -mean qf1(s, mu(s)) against
 *    the qf1 just updated, Adam, then actor', qf1' and qf2' <- tau theta + (1 - tau) theta', in Float64 and rounded once.
 *  - defaults (CleanRL): policy_noise 0.2, noise_clip 0.5, exploration_noise 0.1, learning_starts 25,000, batch_size
 *    256, tau 0.005, lr 3e-4, buffer_size 1,000,000, gamma 0.99, policy_frequency 2.
 *  - one GPU.
 * The actor step is DDPG's: crl_ddpg_actor_loss_raw with qf1 gives TD3's actor loss and gradient, and
 * crl_ddpg_forward_raw evaluates the nets of both algorithms. */
#ifndef CLEANRL_TD3_H
#define CLEANRL_TD3_H

#include "cleanrl_ddpg.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct crl_td3_ctx crl_td3_ctx;
typedef struct crl_td3_config {
  int32_t struct_size;       /* = sizeof(crl_td3_config) */
  int32_t num_envs;          /* N */
  int32_t buffer_size;       /* replay capacity in transitions (>= num_envs) */
  int32_t learning_starts;   /* in global steps */
  int32_t batch_size;        /* 1..256 */
  int32_t train_freq;        /* in iterations */
  int32_t policy_frequency;  /* actor step + target update on every policy_frequency-th learning step */
  int32_t max_episode_steps; /* PendulumEnv() default: 200 */
  int32_t device;
  int32_t _pad;
  double gamma;
  double tau;                /* (0, 1] */
  double lr;                 /* Adam step size of all three nets */
  double exploration_noise;  /* noise scale, times the torque limit 2 */
  uint64_t seed;
  double policy_noise;       /* target smoothing noise scale (>= 0), before the clip */
  double noise_clip;         /* clip of the smoothing noise (>= 0), times the torque limit 2 after the clip */
} crl_td3_config;
typedef struct crl_td3_stats {
  double qf1_loss;      /* of the most recent learning step */
  double qf2_loss;
  double actor_loss;    /* of the most recent actor step (0 before the first) */
  double sum_return;    /* episodes finished during the call */
  double sum_length;
  int64_t episodes;
  int64_t learn_steps;  /* learning (critic) steps so far */
  int64_t actor_steps;  /* actor steps (= target updates) so far: learn_steps / policy_frequency */
  int64_t iterations;   /* iterations so far; global_step = iterations * num_envs */
  int64_t kernel_launches; /* kernels launched so far: acting launches + 2 per learning step + 4 per actor step */
} crl_td3_stats;

/* validates the configuration (CRL_ERR_INVALID with a message) before any device work */
CRL_API int crl_td3_create(const crl_td3_config* cfg, crl_td3_ctx** out);
CRL_API int crl_td3_destroy(crl_td3_ctx* ctx);
/* actor, qf1 and qf2 parameters; the three targets become copies; Adam state reset */
CRL_API int crl_td3_set_params(crl_td3_ctx* ctx, const float* actor, int32_t n_actor, const float* qf1, int32_t n_qf1,
                               const float* qf2, int32_t n_qf2);
/* each pointer may be NULL */
CRL_API int crl_td3_get_params(crl_td3_ctx* ctx, float* actor, float* qf1, float* qf2, float* actor_target,
                               float* qf1_target, float* qf2_target);
/* Adam moments (each may be NULL); beta_pow (may be NULL) = 4 doubles: actor beta1^t, beta2^t, critics beta1^t, beta2^t
 * (both critics share their step count) with t = steps taken + 1: the powers the next step of each optimiser uses */
CRL_API int crl_td3_get_adam_state(crl_td3_ctx* ctx, float* actor_m, float* actor_v, float* qf1_m, float* qf1_v,
                                   float* qf2_m, float* qf2_v, double* beta_pow);
CRL_API int crl_td3_reset(crl_td3_ctx* ctx);   /* reset every env, empty buffer, iteration and step counters 0 */
/* `iterations` vector steps with the learning steps that fall on them; stats may be NULL */
CRL_API int crl_td3_run(crl_td3_ctx* ctx, int64_t iterations, crl_td3_stats* stats);
/* replay buffer contents, as crl_ddpg_read_buffer */
CRL_API int crl_td3_read_buffer(crl_td3_ctx* ctx, float* obs, float* action, float* reward, float* next_obs,
                                uint8_t* terminal, int32_t* size, int32_t* ptr);
/* Raw TD3 critic step (DEVICE pointers; stream = cudaStream_t or NULL), the kernels crl_td3_run launches, on rows the
 * caller passes in (sample b = row b) and with the gradients written out instead of an Adam step. Parameter vectors
 * 16-byte aligned. The smoothing noise of sample b is drawn as crl_td3_run draws it at learning step learn_step.
 * obs, next_obs float [B][3], action, reward float [B], terminal uint8 [B]; 1 <= B <= 256, rows >= B are not read;
 * qf1_grads_out, qf2_grads_out float [4545]; qf1_loss_out, qf2_loss_out 1 double each. Allocates and frees scratch:
 * synchronises `stream`. */
CRL_API int crl_td3_critic_loss_raw(const float* actor_target, const float* qf1, const float* qf2, const float* qf1_target,
                                    const float* qf2_target, int32_t B, const float* obs, const float* action,
                                    const float* reward, const float* next_obs, const uint8_t* terminal, double gamma,
                                    double policy_noise, double noise_clip, uint64_t seed, uint64_t learn_step,
                                    float* qf1_grads_out, float* qf2_grads_out, double* qf1_loss_out,
                                    double* qf2_loss_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CLEANRL_TD3_H */
