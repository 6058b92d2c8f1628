/*
 * cleanrl_ddpg.h — C ABI of the DDPG part of libcleanrl_cuda.so
 *
 * Same library, same conventions as cleanrl_cuda.h (included below for CRL_API, the error codes and
 * crl_last_error): every function returns int (0 = CRL_OK), all indices are 0-based, host pointers are
 * borrowed for the call only, and there is no CPU fallback (CRL_ERR_CUDA without an sm_100 device).
 *
 * ---- DDPG (src/algorithms/ddpg.jl) ---------------------------------------------------------------------
 * The reference trains DDPG on MuJoCo HalfCheetah through PyCall (ddpg.jl:50), which this library does not
 * have, and its source is not part of this checkout beyond what SURVEY §2.1 cites: the config struct
 * (ddpg.jl:1-15) and Polyak-averaged targets (ddpg.jl:39-43,128-129). Parity is therefore pinned to the
 * definition below (CleanRL-Python's ddpg_continuous_action.py, the project the reference follows, on
 * Pendulum with 64-wide nets), NOT to ddpg.jl:
 *  - env: Pendulum (CRL_ENV_PENDULUM), observation [cos th, sin th, thdot], episodes truncated at
 *    max_episode_steps; the stored terminal flag is the env's done flag (the time limit counts as done) and
 *    next_obs is the observation right after the step, before any reset.
 *  - actor mu: Dense(3,64,relu) -> Dense(64,64,relu) -> Dense(64,1) -> tanh -> x 2 (4,481 floats);
 *    critic Q([obs; action]): Dense(4,64,relu) -> Dense(64,64,relu) -> Dense(64,1) (4,545 floats). Flat
 *    parameters in Flux.params order, each W stored (out,in) column-major.
 *  - iteration it (1-based) = one vector step of N envs, global_step = it * N. While global_step <=
 *    learning_starts the action is uniform in [-2, 2); after that clamp(mu(obs) + 2 exploration_noise z, -2, 2)
 *    with z standard normal. Both draws come from Philox stream 5, counter = it, word = env id: the uniform is
 *    (r0 >> 8) 2^-24, the normal Box-Muller of u1 = ((r0 >> 8) + 1) 2^-24 and u2 = (r1 >> 8) 2^-24.
 *    Transitions go to the ring in env order; resets use the reset stream as everywhere else.
 *  - learning step when global_step > learning_starts, it % train_freq == 0 and size >= batch_size:
 *    batch_size rows WITHOUT replacement from [0, size) (keyed permutation, Philox stream 6, counter =
 *    learning-step index); critic: y = r + gamma (1 - d) Q'(s', mu'(s')) in Float64, loss mean((Q(s,a) - y)^2),
 *    Adam. On every policy_frequency-th learning step (learn_steps % policy_frequency == 0 after counting it),
 *    on the same batch and against the critic just updated: actor loss -mean Q(s, mu(s)), Adam, then both
 *    targets theta' <- tau theta + (1 - tau) theta'. Adam: beta (0.9, 0.999), eps 1e-8, Float64 scalars.
 *  - one GPU. */
#ifndef CLEANRL_DDPG_H
#define CLEANRL_DDPG_H

#include "cleanrl_cuda.h"

#ifdef __cplusplus
extern "C" {
#endif

#define CRL_DDPG_ACTOR_PARAMS 4481
#define CRL_DDPG_CRITIC_PARAMS 4545

typedef struct crl_ddpg_ctx crl_ddpg_ctx;
typedef struct crl_ddpg_config {
  int32_t struct_size;       /* = sizeof(crl_ddpg_config) */
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
  double lr;                 /* Adam step size of both nets */
  double exploration_noise;  /* noise scale, times the torque limit 2 */
  uint64_t seed;
} crl_ddpg_config;
typedef struct crl_ddpg_stats {
  double critic_loss;   /* of the most recent learning step */
  double actor_loss;    /* of the most recent actor step (0 before the first) */
  double sum_return;    /* episodes finished during the call */
  double sum_length;
  int64_t episodes;
  int64_t learn_steps;  /* learning (critic) steps so far */
  int64_t actor_steps;  /* actor steps (= target updates) so far: learn_steps / policy_frequency */
  int64_t iterations;   /* iterations so far; global_step = iterations * num_envs */
  int64_t kernel_launches; /* kernels launched so far (one acting launch covers the iterations up to the next learning step) */
} crl_ddpg_stats;

/* validates the configuration (CRL_ERR_INVALID with a message) before any device work */
CRL_API int crl_ddpg_create(const crl_ddpg_config* cfg, crl_ddpg_ctx** out);
CRL_API int crl_ddpg_destroy(crl_ddpg_ctx* ctx);
/* actor and critic parameters; both targets become copies; Adam state reset */
CRL_API int crl_ddpg_set_params(crl_ddpg_ctx* ctx, const float* actor, int32_t n_actor, const float* critic, int32_t n_critic);
/* each pointer may be NULL */
CRL_API int crl_ddpg_get_params(crl_ddpg_ctx* ctx, float* actor, float* critic, float* actor_target, float* critic_target);
/* Adam moments (each may be NULL); beta_pow (may be NULL) = 4 doubles: actor beta1^t, beta2^t, critic beta1^t, beta2^t with
 * t = steps taken + 1: the powers the next step of each optimiser uses */
CRL_API int crl_ddpg_get_adam_state(crl_ddpg_ctx* ctx, float* actor_m, float* actor_v, float* critic_m, float* critic_v,
                                    double* beta_pow);
CRL_API int crl_ddpg_reset(crl_ddpg_ctx* ctx);   /* reset every env, empty buffer, iteration and step counters 0 */
/* `iterations` vector steps with the learning steps that fall on them; stats may be NULL */
CRL_API int crl_ddpg_run(crl_ddpg_ctx* ctx, int64_t iterations, crl_ddpg_stats* stats);
/* replay buffer contents (host pointers, each may be NULL): obs/next_obs float [capacity][3], action, reward float
 * [capacity], terminal uint8 [capacity]; size and ptr (0-based next slot) */
CRL_API int crl_ddpg_read_buffer(crl_ddpg_ctx* ctx, float* obs, float* action, float* reward, float* next_obs,
                                 uint8_t* terminal, int32_t* size, int32_t* ptr);
/* Raw DDPG kernels (DEVICE pointers; stream = cudaStream_t or NULL), the ones crl_ddpg_run launches. Parameter vectors
 * 16-byte aligned.
 * crl_ddpg_forward_raw: mu(obs) by the acting kernel's forward pass and Q(obs, action) with the same tiling.
 * obs float [n][3], action float [n], mu_out, q_out float [n].
 * crl_ddpg_critic_loss_raw: critic loss and un-stepped critic gradient (float [4545]) of one batch, sample b = row b.
 * crl_ddpg_actor_loss_raw: actor loss -mean Q(obs, mu(obs)) and un-stepped actor gradient (float [4481]).
 * 1 <= B <= 256; rows >= B are not read; loss_out = 1 double. Both allocate and free scratch: they synchronise `stream`. */
CRL_API int crl_ddpg_forward_raw(const float* actor, const float* critic, const float* obs, const float* action,
                                 float* mu_out, float* q_out, int64_t n, void* stream);
CRL_API int crl_ddpg_critic_loss_raw(const float* actor_target, const float* critic, const float* critic_target, int32_t B,
                                     const float* obs, const float* action, const float* reward, const float* next_obs,
                                     const uint8_t* terminal, double gamma, float* grads_out, double* loss_out, void* stream);
CRL_API int crl_ddpg_actor_loss_raw(const float* actor, const float* critic, int32_t B, const float* obs, float* grads_out,
                                    double* loss_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CLEANRL_DDPG_H */
