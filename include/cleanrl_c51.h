/*
 * cleanrl_c51.h — C ABI of the C51 part of libcleanrl_cuda.so
 *
 * Same library, same conventions as cleanrl_cuda.h (included below): every function returns int (0 = CRL_OK), all
 * indices are 0-based, host pointers are borrowed for the call only, and there is no CPU fallback (CRL_ERR_CUDA without
 * an sm_100 device).
 *
 * ---- C51 (an extension: the reference has no C51) ----------------------------------------------------------------
 * CleanRL-Python's c51.py on the library's CartPole: a distributional Q-network over CRL_C51_ATOMS = 101 fixed atoms.
 *  - env and ring: exactly the DQN part's (crl_dqn_*): N CartPole envs step in lockstep, iteration it (1-based) is one
 *    vector step and global_step = it * N; the N transitions go to the ring in env order; RLEnvs' reward 0 on the
 *    terminating step; an episode truncated at max_episode_steps is stored as terminal.
 *  - acting: epsilon-greedy exactly as DQN: Philox stream 3 (word = env, counter = it), u < epsilon, the random action
 *    bit. The greedy action is argmax_a sum_j p_aj z_j, the first maximum (torch.argmax), the sum accumulated in Float32
 *    in ascending j. epsilon = linear_schedule(start_e, end_e, epsilon_duration, global_step), DQN's function; c51()
 *    passes epsilon_duration = exploration_fraction * total_timesteps, as CleanRL does. With epsilon pinned to 1, C51
 *    and DQN therefore fill bit-identical rings for the same seed and config.
 *  - schedule: a learning step runs when global_step > learning_starts, it % train_frequency == 0 and
 *    size >= batch_size. The target net is copied on every iteration with global_step > learning_starts and
 *    it % target_network_frequency == 0 (not only on learning iterations, as CleanRL), after that iteration's learning
 *    step if it has one. With N = 1 every rule is CleanRL's.
 *  - network: Linear(4,120) -> ReLU -> Linear(120,84) -> ReLU -> Linear(84, 2 * 101). Flat parameters W1, b1, W2, b2,
 *    W3, b3, each W (out,in) column-major, as the DQN part: the first 10,764 floats have DQN's layout. Head output
 *    o = a * 101 + j (CleanRL's view(n, 2, 101)). CRL_C51_PARAMS = 27,934 floats. pmf p_a = softmax over the 101 logits
 *    of action a.
 *  - atoms: z_j = (float)(v_min + j * ((v_max - v_min) / 100)), evaluated in Float64 and rounded once;
 *    dz = z_1 - z_0 in Float32 (CleanRL's atoms[1] - atoms[0]).
 *  - projection, all in Float32 in CleanRL's order without contraction, with gamma_f = (float)gamma and
 *    v_min, v_max rounded to Float32:
 *      tz_j = clamp(r + ((gamma_f z_j) (1 - d)), v_min, v_max);  b_j = (tz_j - v_min) / dz;
 *      l_j = clamp(floor b_j, 0, 100);  u_j = clamp(ceil b_j, 0, 100);
 *      d_m_l_j = (u_j + [l_j == u_j] - b_j) p'_j;  d_m_u_j = (b_j - l_j) p'_j
 *    where p' is the target net's pmf of the target net's own greedy action at s'. The target masses start at zero; the
 *    d_m_l terms are added to m[l_j] for ascending j, then the d_m_u terms to m[u_j] for ascending j (CPU index_add_).
 *  - loss: -mean_b sum_j m_bj log(clamp(p_{b,a_b,j}, 1e-5, 1 - 1e-5)), summed in Float64. Its gradient with respect to
 *    the taken action's logit i is (p_i sum_j m_j k_j - m_i k_i) / B with k_j = 1 where 1e-5 <= p_j <= 1 - 1e-5
 *    (torch's clamp passes the gradient at its bounds); the other action's logits get zero gradient. Every gradient is
 *    summed over the batch in ascending sample order.
 *  - Adam: beta (0.9, 0.999), eps = 0.01 / batch_size (c51.py), Float64 scalars on Float32 state (the DQN step).
 *  - defaults (CleanRL): lr 2.5e-4, buffer_size 10,000, gamma 0.99, target_network_frequency 500, batch_size 128,
 *    start_e 1, end_e 0.05, exploration_fraction 0.5, learning_starts 10,000, train_frequency 10, v_min -100,
 *    v_max 100, total_timesteps 500,000; max_episode_steps 500 (CartPole-v1).
 *  - deviations from CleanRL: the batch is sampled without replacement, as in DQN (keyed permutation, Philox stream 4,
 *    counter = learning-step index; SB3's buffer samples with replacement); truncation is stored as terminal; RLEnvs'
 *    reward rule; global_step counts env steps, which is CleanRL's count at N = 1.
 *  - batch_size 1..128; one GPU. */
#ifndef CLEANRL_C51_H
#define CLEANRL_C51_H

#include "cleanrl_cuda.h"

#ifdef __cplusplus
extern "C" {
#endif

#define CRL_C51_ATOMS 101
#define CRL_C51_PARAMS 27934

typedef struct crl_c51_ctx crl_c51_ctx;
typedef struct crl_c51_config {
  int32_t struct_size;              /* = sizeof(crl_c51_config) */
  int32_t num_envs;                 /* N */
  int32_t buffer_size;              /* replay capacity in transitions (>= num_envs) */
  int32_t learning_starts;          /* in global steps */
  int32_t batch_size;               /* 1..128 */
  int32_t train_frequency;          /* in iterations (>= 1) */
  int32_t target_network_frequency; /* in iterations (>= 1) */
  int32_t max_episode_steps;        /* CartPole-v1: 500 */
  int32_t device;
  int32_t _pad;
  double lr;                        /* finite, > 0 */
  double gamma;                     /* in [0, 1] */
  double start_e, end_e, epsilon_duration; /* epsilon_duration > 0, in global steps */
  double v_min, v_max;              /* finite, v_min < v_max */
  uint64_t seed;
} crl_c51_config;
typedef struct crl_c51_stats {
  double loss;          /* of the most recent learning step */
  double q_values;      /* batch mean of the taken action's expected Q at that step (CleanRL's losses/q_values) */
  double sum_return;    /* episodes finished during the call */
  double sum_length;
  double epsilon;       /* at the last iteration */
  int64_t episodes;
  int64_t learn_steps;  /* learning steps so far */
  int64_t target_copies; /* target copies so far */
  int64_t iterations;   /* iterations so far; global_step = iterations * num_envs */
  int64_t kernel_launches; /* kernels launched so far: acting launches + 3 learn_steps. One acting launch covers the
                              iterations up to and including the next learning iteration, at most 16 of them and at most
                              floor(buffer_size / num_envs). A target copy off a learning iteration is a device-to-device
                              copy, not a kernel. */
} crl_c51_stats;

/* validates the configuration (CRL_ERR_INVALID with a message) before any device work */
CRL_API int crl_c51_create(const crl_c51_config* cfg, crl_c51_ctx** out);
CRL_API int crl_c51_destroy(crl_c51_ctx* ctx);
/* q_network parameters (27,934 floats); the target becomes a copy; Adam state reset */
CRL_API int crl_c51_set_params(crl_c51_ctx* ctx, const float* params, int32_t n);
/* q_network and target parameters (target may be NULL) */
CRL_API int crl_c51_get_params(crl_c51_ctx* ctx, float* q_params, float* target_params, int32_t n);
/* Adam moments m, v (27,934 floats each, each may be NULL); beta_pow (may be NULL) = 2 doubles beta1^t, beta2^t with
 * t = steps taken + 1 */
CRL_API int crl_c51_get_adam_state(crl_c51_ctx* ctx, float* m, float* v, double* beta_pow);
CRL_API int crl_c51_reset(crl_c51_ctx* ctx);   /* reset every env, empty buffer, iteration and step counters 0 */
/* `iterations` vector steps with the learning steps and target copies that fall on them; stats may be NULL */
CRL_API int crl_c51_run(crl_c51_ctx* ctx, int64_t iterations, crl_c51_stats* stats);
/* replay buffer contents, as crl_dqn_read_buffer */
CRL_API int crl_c51_read_buffer(crl_c51_ctx* ctx, float* state, int32_t* action, float* reward, float* next_state,
                                uint8_t* terminal, int32_t* size, int32_t* ptr);
/* Raw entry points (DEVICE pointers; stream = cudaStream_t or NULL): the kernels crl_c51_run launches, on rows the
 * caller passes in. Parameter vectors and state rows 16-byte aligned.
 * forward: the acting kernel's forward pass, softmax, expectation and argmax on n rows of obs float [n][4]:
 * q_out float [n][2] (8-byte aligned), action_out int32 [n], pmf_out float [n][2][101] or NULL. */
CRL_API int crl_c51_forward_raw(const float* params, const float* obs, double v_min, double v_max, float* q_out,
                                int32_t* action_out, float* pmf_out, int64_t n, void* stream);
/* the learning step's three kernels with sample b taken from row b of state / action / reward / next_state / terminal
 * (nothing sampled; rows >= B are not read), 1 <= B <= 128, and the gradient written out instead of an Adam step:
 * target_pmf_out float [B][101] (the projected masses m), grads_out float [27934], loss_out 1 double. Allocates and
 * frees its scratch: synchronises `stream`. */
CRL_API int crl_c51_loss_raw(const float* q, const float* tgt, int32_t B, const float* state, const int32_t* action,
                             const float* reward, const float* next_state, const uint8_t* terminal, double gamma,
                             double v_min, double v_max, float* target_pmf_out, float* grads_out, double* loss_out,
                             void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CLEANRL_C51_H */
