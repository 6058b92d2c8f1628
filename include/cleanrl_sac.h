/*
 * cleanrl_sac.h — C ABI of the SAC part of libcleanrl_cuda.so
 *
 * Same library, same conventions as cleanrl_ddpg.h (included below): every function returns int (0 = CRL_OK), all
 * indices are 0-based, host pointers are borrowed for the call only, and there is no CPU fallback (CRL_ERR_CUDA without
 * an sm_100 device).
 *
 * ---- SAC (an extension: the reference has no SAC) ----------------------------------------------------------------
 * CleanRL-Python's sac_continuous_action.py on Pendulum with the 64-wide nets of cleanrl_ddpg.h. Everything not listed
 * here is exactly the DDPG definition of cleanrl_ddpg.h: env, observation and episode truncation, the warm-up rule
 * (uniform in [-2, 2) while global_step <= learning_starts, Philox stream 5), ring order, the learning gate and batch
 * sampling (keyed permutation, Philox stream 6, counter = learning-step index). With the same seed and config, SAC, DDPG
 * and TD3 therefore fill bit-identical replay buffers through the warm-up, up to the first iteration that acts from the
 * policy.
 *  - actor (CRL_SAC_ACTOR_PARAMS = 4,546 floats): Dense(3,64,relu) -> Dense(64,64,relu), then two heads fc_mean
 *    Dense(64,1) and fc_logstd Dense(64,1). Flat order W1, b1, W2, b2, W_mean, b_mean, W_logstd, b_logstd, each W
 *    (out,in) column-major. log_std = -5 + 3.5 (tanh(l) + 1) with l the fc_logstd output, std = exp(log_std),
 *    x = mean + std z, a = 2 tanh(x), log_pi = log N(x; mean, std) - log(2 (1 - tanh^2 x) + 1e-6).
 *  - critics qf1 and qf2: DDPG's critic architecture (4,545 floats each). Only the critics have targets; there is no
 *    target actor.
 *  - acting after warm-up: a = 2 tanh(mean + std z) with z the Box-Muller normal of DDPG's acting noise (Philox stream
 *    5, word = env id, counter = iteration, u1 = ((r0 >> 8) + 1) 2^-24, u2 = (r1 >> 8) 2^-24), in Float32.
 *  - every other draw is the same Box-Muller normal of Philox(seed, word = b, counter, stream) with b the sample's
 *    position in the batch (not its ring row), evaluated in Float64.
 *  - learning step t (0-based index) on the sampled batch; alpha is the temperature before this learning step:
 *     1. critic target: z'_b from stream 8, counter = t; a' and log_pi' from the CURRENT actor at s';
 *        y = r + gamma (1 - d) (min(qf1'(s', a'), qf2'(s', a')) - alpha log_pi') in Float64 with DDPG's expression.
 *        Loss mean((qf_k(s, a) - y)^2) for each critic, one Adam step of both with q_lr and a shared step count,
 *        exactly as TD3 does; the two losses are reported separately.
 *     2. count the learning step. If learn_steps % policy_frequency == 0, run policy_frequency actor iterations on the
 *        same batch (CleanRL's delayed-update loop). With u the 0-based count of actor iterations so far, iteration u:
 *        - z from stream 9, counter = u; actor_loss = mean(alpha log_pi - min(qf1(s, a), qf2(s, a))) against the
 *          critics just updated. Where qf1 = qf2 the gradient splits in halves between the two critics (torch.minimum).
 *          Adam on the actor with policy_lr.
 *        - if autotune: a fresh draw, z from stream 10, counter = u, through the actor just updated; alpha_loss =
 *          mean(-exp(log_alpha) (log_pi + target_entropy)) = -exp(log_alpha) (mean log_pi + target_entropy) with
 *          target_entropy = -1, evaluated in Float64 from the Float32 log_alpha. It is also its own gradient with
 *          respect to log_alpha, which is rounded to Float32 for one Adam step of log_alpha (Float32, as a torch
 *          parameter) with q_lr and the actor's step count; then alpha = exp(log_alpha) in Float64.
 *     3. if learn_steps % target_network_frequency == 0: qf1', qf2' <- tau theta + (1 - tau) theta', in Float64 and
 *        rounded once.
 *    Both gates count learning steps where CleanRL counts global_step: the same steps when one env learns on every
 *    step and learning_starts is a multiple of both frequencies.
 *  - temperature: with autotune, log_alpha starts at 0 (alpha = 1); without it alpha is the configured constant and
 *    log_alpha stays 0. alpha, log_alpha and its Adam moments live on the device, so a run is a plain launch sequence
 *    without a device-to-host read.
 *  - Adam: beta (0.9, 0.999), eps 1e-8, Float64 scalars, Float32 state.
 *  - defaults (CleanRL): learning_starts 5,000, batch_size 256, tau 0.005, gamma 0.99, policy_lr 3e-4, q_lr 1e-3,
 *    policy_frequency 2, target_network_frequency 1, alpha 0.2, autotune on, buffer_size 1,000,000.
 *  - one GPU. */
#ifndef CLEANRL_SAC_H
#define CLEANRL_SAC_H

#include "cleanrl_ddpg.h"

#ifdef __cplusplus
extern "C" {
#endif

#define CRL_SAC_ACTOR_PARAMS 4546

typedef struct crl_sac_ctx crl_sac_ctx;
typedef struct crl_sac_config {
  int32_t struct_size;              /* = sizeof(crl_sac_config) */
  int32_t num_envs;                 /* N */
  int32_t buffer_size;              /* replay capacity in transitions (>= num_envs) */
  int32_t learning_starts;          /* in global steps */
  int32_t batch_size;               /* 1..256 */
  int32_t train_freq;               /* in iterations */
  int32_t policy_frequency;         /* policy_frequency actor iterations on every policy_frequency-th learning step */
  int32_t target_network_frequency; /* target update on every target_network_frequency-th learning step (>= 1) */
  int32_t max_episode_steps;        /* PendulumEnv() default: 200 */
  int32_t device;
  int32_t autotune;                 /* 0 or 1: learn alpha */
  int32_t _pad;
  double gamma;
  double tau;                       /* (0, 1] */
  double policy_lr;                 /* Adam step size of the actor (finite, > 0) */
  double q_lr;                      /* Adam step size of both critics and of log_alpha (finite, > 0) */
  double alpha;                     /* the temperature when autotune is 0 (finite, >= 0) */
  uint64_t seed;
} crl_sac_config;
typedef struct crl_sac_stats {
  double qf1_loss;      /* of the most recent learning step */
  double qf2_loss;
  double actor_loss;    /* of the most recent actor iteration (0 before the first) */
  double alpha_loss;    /* of the most recent temperature step (0 before the first, and without autotune) */
  double alpha;         /* the temperature now */
  double sum_return;    /* episodes finished during the call */
  double sum_length;
  int64_t episodes;
  int64_t learn_steps;  /* learning (critic) steps so far */
  int64_t actor_steps;  /* actor iterations so far: policy_frequency * (learn_steps / policy_frequency) */
  int64_t iterations;   /* iterations so far; global_step = iterations * num_envs */
  int64_t kernel_launches; /* kernels launched so far: acting launches + 2 learn_steps + (2 + 2 autotune) actor_steps
                              + learn_steps / target_network_frequency */
} crl_sac_stats;

/* validates the configuration (CRL_ERR_INVALID with a message) before any device work */
CRL_API int crl_sac_create(const crl_sac_config* cfg, crl_sac_ctx** out);
CRL_API int crl_sac_destroy(crl_sac_ctx* ctx);
/* actor (4,546 floats), qf1 and qf2 (4,545 each); both targets become copies; Adam state reset; log_alpha 0 and alpha
 * 1 (autotune) or the configured alpha */
CRL_API int crl_sac_set_params(crl_sac_ctx* ctx, const float* actor, int32_t n_actor, const float* qf1, int32_t n_qf1,
                               const float* qf2, int32_t n_qf2);
/* each pointer may be NULL; log_alpha is 1 float */
CRL_API int crl_sac_get_params(crl_sac_ctx* ctx, float* actor, float* qf1, float* qf2, float* qf1_target, float* qf2_target,
                               float* log_alpha);
/* Adam moments (each may be NULL); log_alpha_mv (may be NULL) = 2 floats, log_alpha's m and v; beta_pow (may be NULL) =
 * 4 doubles: actor (and log_alpha) beta1^t, beta2^t, critics beta1^t, beta2^t with t = steps taken + 1 */
CRL_API int crl_sac_get_adam_state(crl_sac_ctx* ctx, float* actor_m, float* actor_v, float* qf1_m, float* qf1_v, float* qf2_m,
                                   float* qf2_v, float* log_alpha_mv, double* beta_pow);
CRL_API int crl_sac_reset(crl_sac_ctx* ctx);   /* reset every env, empty buffer, iteration and step counters 0 */
/* `iterations` vector steps with the learning steps that fall on them; stats may be NULL */
CRL_API int crl_sac_run(crl_sac_ctx* ctx, int64_t iterations, crl_sac_stats* stats);
/* replay buffer contents, as crl_ddpg_read_buffer */
CRL_API int crl_sac_read_buffer(crl_sac_ctx* ctx, float* obs, float* action, float* reward, float* next_obs,
                                uint8_t* terminal, int32_t* size, int32_t* ptr);
/* Raw entry points (DEVICE pointers; stream = cudaStream_t or NULL): the kernels crl_sac_run launches, on rows the
 * caller passes in (sample b = row b) and with gradients written out instead of an Adam step. Parameter vectors 16-byte
 * aligned. obs, next_obs float [B][3], action, reward float [B], terminal uint8 [B]; 1 <= B <= 256 and rows >= B are
 * not read. The noise of sample b is drawn as crl_sac_run draws it, from `seed` and the given counter. alpha is finite
 * and >= 0. The loss entry points allocate and free scratch: they synchronise `stream`.
 * forward: the acting kernel's actor forward and a critic on n rows: mean_out, log_std_out (after its squash to
 * [-5, 2]) and q_out = qf(obs, action), float [n] each. */
CRL_API int crl_sac_forward_raw(const float* actor, const float* qf, const float* obs, const float* action, float* mean_out,
                                float* log_std_out, float* q_out, int64_t n, void* stream);
/* the critic step at learning step learn_step (stream 8): both losses (1 double each) and both gradients (4,545 floats) */
CRL_API int crl_sac_critic_loss_raw(const float* actor, const float* qf1, const float* qf2, const float* qf1_target,
                                    const float* qf2_target, int32_t B, const float* obs, const float* action,
                                    const float* reward, const float* next_obs, const uint8_t* terminal, double gamma,
                                    double alpha, uint64_t seed, uint64_t learn_step, float* qf1_grads_out,
                                    float* qf2_grads_out, double* qf1_loss_out, double* qf2_loss_out, void* stream);
/* actor iteration actor_step (stream 9): actor_loss (1 double), its gradient (4,546 floats) and the batch's mean log_pi
 * (1 double) */
CRL_API int crl_sac_actor_loss_raw(const float* actor, const float* qf1, const float* qf2, int32_t B, const float* obs,
                                   double alpha, uint64_t seed, uint64_t actor_step, float* grads_out, double* loss_out,
                                   double* mean_log_pi_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CLEANRL_SAC_H */
