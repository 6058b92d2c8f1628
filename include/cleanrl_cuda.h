/*
 * cleanrl_cuda.h — C ABI of libcleanrl_cuda.so
 *
 * B200 (sm_100a) implementation of the PPO training hot path of sash-a/CleanRL.jl:
 * rollout over vectorised environments, GAE, clipped-surrogate minibatch update.
 * The reference has no FFI boundary of its own (it is pure Julia); each entry point
 * below cites the reference lines (relative to the reference repo root) whose work
 * it replaces. The Julia `ccall` binding that uses this header is in
 * cleanrl.jl_b200/julia/CleanRLCuda.jl and is shown in INTEGRATION.md.
 *
 * Conventions
 *  - every function returns int: 0 = CRL_OK, negative = error code; the message is
 *    available from crl_last_error() (thread-local). No C++ exception crosses the ABI.
 *  - all indices are 0-BASED at this boundary. Julia is 1-based (actions, ppo.jl:26;
 *    minibatch indices, ppo.jl:191): the Julia shim subtracts/adds 1.
 *  - array layouts are the reference's column-major arrays read in C order:
 *      state   Float32 (D,N,T) -> [T][N][D]      (ppo.jl:96, replay_buffer.jl:16)
 *      action  Int32   (N,T)   -> [T][N]         (ppo.jl:97)  (float [T][N][A] for Gaussian)
 *      logprob/reward/value Float32 (N,T) -> [T][N]   (ppo.jl:98-101)
 *      terminal Bool (N,T) -> uint8 [T][N]       (ppo.jl:100)
 *    flat sample index b = n + N*t  (ppo.jl:184-189, env fastest).
 *  - parameters are one flat float32 vector in Flux.params(actor, critic) order
 *    (ppo.jl:196): actor W1,b1,W2,b2,W3,b3, critic W1,b1,W2,b2,W3,b3, each W stored
 *    (out,in) column-major exactly as Flux holds it; a Gaussian policy (Pendulum)
 *    appends a 13th array logstd[A].
 *  - "host" pointers are borrowed for the duration of the call only. The library owns
 *    all device memory behind the opaque handle. A handle is not thread-safe; use one
 *    handle per GPU. Work is enqueued on the handle's stream; calls that return data to
 *    the host synchronise that stream.
 *  - there is NO CPU fallback: every compute entry point fails with CRL_ERR_CUDA when no
 *    sm_100 device is usable.
 */
#ifndef CLEANRL_CUDA_H
#define CLEANRL_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CRL_VERSION 100

#if defined(__GNUC__)
#define CRL_API __attribute__((visibility("default")))
#else
#define CRL_API
#endif

/* error codes */
#define CRL_OK 0
#define CRL_ERR_INVALID (-1)  /* bad argument / unsupported configuration          */
#define CRL_ERR_CUDA (-2)     /* a CUDA runtime call failed (message has details)  */
#define CRL_ERR_NCCL (-3)     /* NCCL missing or a collective failed               */
#define CRL_ERR_STATE (-4)    /* call order violated (e.g. gae before rollout)     */

/* environments (the reference hard-codes CartPole, ppo.jl:79-83) */
#define CRL_ENV_CARTPOLE 0 /* discrete, D=4, A=2, categorical policy */
#define CRL_ENV_PENDULUM 1 /* continuous, D=3, A=1, Gaussian policy  */

/* GAE scan variants (SURVEY §8a-Q1) */
#define CRL_GAE_REF_COMPAT 0 /* ppo.jl:66 as written: scan starts at T-1 with zero carry; adv[T] := 0 */
#define CRL_GAE_FIXED 1      /* scan starts at T and uses the bootstrap value/flag */
#define CRL_GAE_A2C_RETURNS 2 /* discounted_future_rewards of a2c.jl:13-24: ret[t] = term[t] ? 0 : r[t] + γ ret[t+1], bootstrap
                                 final_value; adv = ret - value (a2c.jl:83). term[t] = is_terminated AFTER step t. */

/* crl_config.flags */
#define CRL_FLAG_LOCAL_STATS 1u /* multi-GPU: per-shard minibatch statistics (no pre-backward exchange) */
#define CRL_FLAG_A2C 2u         /* A2C losses (a2c.jl:78-97) instead of the PPO clipped surrogate: critic mean((ret-v)^2),
                                   actor -mean(logp * (ret - v)); use with CRL_GAE_A2C_RETURNS, 1 epoch x 1 minibatch */
#define CRL_FLAG_NO_VCLIP 4u    /* PPOConfig.clip_value_loss = false (ppo.jl:16,239-241): v_loss = 0.5 mean((newvalue - R)^2) */

/* buffer fields for crl_read_field / crl_write_field */
#define CRL_F_STATE 0       /* float  [T][N][D]                                    */
#define CRL_F_ACTION 1      /* int32  [T][N]  (categorical) | float [T][N][A]      */
#define CRL_F_LOGPROB 2     /* float  [T][N]                                       */
#define CRL_F_REWARD 3      /* float  [T][N]                                       */
#define CRL_F_TERMINAL 4    /* uint8  [T][N]                                       */
#define CRL_F_VALUE 5       /* float  [T][N]                                       */
#define CRL_F_ADVANTAGE 6   /* float  [T][N]                                       */
#define CRL_F_RETURN 7      /* float  [T][N]                                       */
#define CRL_F_NEXT_OBS 8    /* float  [N][D]   obs the next policy step will read  */
#define CRL_F_NEXT_DONE 9   /* uint8  [N]                                          */
#define CRL_F_NEXT_VALUE 10 /* float  [N]      bootstrap value written by crl_gae  */
#define CRL_F_ENV_STATE 11  /* float  [N][S]   S=4 CartPole, 2 Pendulum            */
#define CRL_F_ENV_T 12      /* int32  [N]      steps since reset                   */
#define CRL_F_EP_RETURN 13  /* double [N]      ppo.jl:108                          */
#define CRL_F_EP_LENGTH 14  /* int32  [N]      ppo.jl:109                          */
#define CRL_F_RESET_COUNT 15 /* uint32 [N]     resets so far (Philox reset stream) */
#define CRL_F_VNEW 16       /* float  [M]      scratch: critic values of the last minibatch */
#define CRL_NUM_FIELDS 17

typedef struct crl_ctx crl_ctx; /* opaque */

/* Hyper-parameters and sharding. Mirrors PPOConfig (ppo.jl:1-19) plus what the
 * reference hard-codes (env ppo.jl:82, clip threshold ppo.jl:93). */
typedef struct crl_config {
  int32_t struct_size; /* = sizeof(crl_config); ABI check */
  int32_t env_kind;    /* CRL_ENV_* */
  int32_t num_envs;    /* envs owned by THIS handle (local shard), ppo.jl:4 */
  int32_t num_steps;   /* T, ppo.jl:3 */
  int32_t num_minibatches; /* ppo.jl:5 */
  int32_t update_epochs;   /* ppo.jl:6 */
  int32_t max_episode_steps; /* CartPole max_steps=500 (ppo.jl:82); Pendulum 200 */
  int32_t gae_mode;    /* CRL_GAE_* */
  int32_t device;      /* CUDA device ordinal */
  int32_t world_size;  /* number of shards (GPUs); 1 = single GPU */
  int32_t rank;        /* this shard */
  int32_t env_id_base; /* global index of local env 0 (Philox counter word) */
  int32_t episode_capacity; /* per-rollout episode record capacity; 0 = default */
  uint32_t flags;      /* CRL_FLAG_* */
  float gamma;         /* ppo.jl:9 */
  float gae_lambda;    /* ppo.jl:10 */
  float clip_coef;     /* ppo.jl:12 */
  float ent_coeff;     /* ppo.jl:13 */
  float v_coef;        /* ppo.jl:14 */
  float clip_norm;     /* per-array gradient clip threshold, 0.5 at ppo.jl:93 */
  uint64_t seed;       /* Philox key */
} crl_config;

/* "Training Statistics" record, ppo.jl:247 (all Float64 in the reference) */
typedef struct crl_loss_stats {
  double loss;
  double pg_loss;
  double v_loss;
  double entropy_loss;
} crl_loss_stats;

/* one "Episode Statistics" record, ppo.jl:152-157. step = 0-based rollout step at which
 * the episode ended; global_step = base + (step+1)*N_global is formed by the host. */
typedef struct crl_episode {
  int32_t step;
  int32_t env; /* local env index */
  int32_t length;
  int32_t _pad;
  double episode_return;
} crl_episode;

/* per-rollout aggregate of the same records (throughput mode logging) */
typedef struct crl_episode_agg {
  int64_t count;
  double sum_return;
  double sum_length;
  double max_return;
  int64_t dropped; /* records that did not fit episode_capacity */
} crl_episode_agg;

/* per-kernel device time, accumulated with CUDA events on the handle's stream while
 * profiling is enabled (crl_profile). Index with CRL_K_*. */
#define CRL_K_ROLLOUT 0
#define CRL_K_GAE 1
#define CRL_K_MB_STATS 2
#define CRL_K_MB_COUNT 3
#define CRL_K_LOSS_GRAD 4
#define CRL_K_GRAD_REDUCE 5
#define CRL_K_CLIP_ADAM 6
#define CRL_K_ALLREDUCE 7
#define CRL_K_OTHER 8
#define CRL_NUM_KERNELS 9
typedef struct crl_kernel_times {
  double ms[CRL_NUM_KERNELS];
  int64_t launches[CRL_NUM_KERNELS];
} crl_kernel_times;

/* ---- library ------------------------------------------------------------------ */
CRL_API int crl_version(void);
CRL_API const char* crl_last_error(void);
CRL_API int crl_device_count(int32_t* count);

/* ---- handle ------------------------------------------------------------------- */
/* replaces the set-up block of ppo(), ppo.jl:76-115 (env vector, buffer, optimiser state) */
CRL_API int crl_create(const crl_config* cfg, crl_ctx** out);
CRL_API int crl_destroy(crl_ctx* ctx);
CRL_API int crl_sync(crl_ctx* ctx);
/* dimensions: D obs dim, A action dim, S env-state dim, P param floats, n_arrays */
CRL_API int crl_dims(const crl_ctx* ctx, int32_t* D, int32_t* A, int32_t* S, int32_t* P, int32_t* n_arrays);
/* offsets/sizes (in floats) of the parameter arrays inside the flat vector */
CRL_API int crl_param_layout(const crl_ctx* ctx, int32_t* offsets, int32_t* sizes, int32_t max_arrays);

/* ---- parameters / optimiser state (Flux.params order, ppo.jl:196; Adam state ppo.jl:93) */
CRL_API int crl_set_params(crl_ctx* ctx, const float* host, int32_t n);
CRL_API int crl_get_params(crl_ctx* ctx, float* host, int32_t n);
CRL_API int crl_get_grads(crl_ctx* ctx, float* host, int32_t n); /* un-clipped grads of the last minibatch */
/* m, v: P floats each; beta_pow: n_arrays*2 doubles (Flux keeps (β1^t, β2^t) per array) */
CRL_API int crl_get_adam_state(crl_ctx* ctx, float* m, float* v, double* beta_pow);
CRL_API int crl_set_adam_state(crl_ctx* ctx, const float* m, const float* v, const double* beta_pow);

/* ---- environments (replace MultiThreadEnv, multi_thread_env.jl:86-133) ------------ */
/* force-reset every env from the Philox reset stream and refresh next_obs/next_done
 * (ppo.jl:112-115). Zeroes the episode counters (ppo.jl:108-109). */
CRL_API int crl_env_reset(crl_ctx* ctx);
/* parity hook: overwrite env states ([N][S]) and step counters ([N], may be NULL = 0);
 * next_obs is refreshed from them, next_done cleared. */
CRL_API int crl_env_set_state(crl_ctx* ctx, const float* state, const int32_t* t);

/* ---- rollout (replaces the loop ppo.jl:123-166) ---------------------------------- */
/* Runs num_steps policy+env steps for every env in one launch and fills the rollout
 * buffer. action_noise / reset_noise are optional HOST arrays that replace the Philox
 * draws (parity mode):
 *   action_noise: categorical: double [T][N] uniforms in [0,1) (the rand() of
 *                 StatsBase.sample, ppo.jl:26); Gaussian: double [T][N][A] standard normals.
 *   reset_noise : float [T][N][4] raw U[0,1) draws used if env n terminates at step t. */
CRL_API int crl_rollout(crl_ctx* ctx, const double* action_noise, const float* reset_noise);

/* ---- GAE (replaces ppo.jl:169-181 and gae(), ppo.jl:48-73) ------------------------ */
CRL_API int crl_gae(crl_ctx* ctx);

/* ---- update (replaces ppo.jl:191-252) -------------------------------------------- */
/* one minibatch: loss + backward + per-array clip + Adam (+ allreduce when world>1).
 * idx: HOST int32[M] 0-based flat sample indices (local to this shard). lr = opt.eta
 * (ppo.jl:120). stats may be NULL. */
CRL_API int crl_update_minibatch(crl_ctx* ctx, const int32_t* idx, int32_t M, double lr, crl_loss_stats* stats);
/* all epochs. perms: HOST int32[update_epochs][B] permutations of 0..B-1 (shuffle,
 * ppo.jl:194), or NULL to use the device permutation (Philox-keyed Feistel bijection).
 * stats: update_epochs*num_minibatches records, may be NULL. */
CRL_API int crl_update_epochs(crl_ctx* ctx, const int32_t* perms, double lr, crl_loss_stats* stats);
/* the device permutation crl_update_epochs(NULL) uses for (update_index, epoch): HOST out int32[B] */
CRL_API int crl_device_permutation(crl_ctx* ctx, int64_t update_index, int32_t epoch, int32_t* out);

/* one whole PPO update = rollout + GAE + all epochs, device RNG, enqueued asynchronously
 * (CUDA graph). Results of the most recent update are fetched with crl_fetch_update. */
CRL_API int crl_train_update(crl_ctx* ctx, double lr);
CRL_API int crl_fetch_update(crl_ctx* ctx, crl_loss_stats* stats /* epochs*minibatches, may be NULL */,
                     crl_episode_agg* agg /* may be NULL */);
/* same, for the update enqueued `lag` calls before the latest (0 or 1). With lag = 1 the host can log
 * update u-1 (waits only for that update) while update u is running: the results are double-buffered. */
CRL_API int crl_fetch_update_at(crl_ctx* ctx, int32_t lag, crl_loss_stats* stats, crl_episode_agg* agg);

/* ---- data access ----------------------------------------------------------------- */
CRL_API int crl_read_field(crl_ctx* ctx, int32_t field, void* host, size_t bytes);
CRL_API int crl_write_field(crl_ctx* ctx, int32_t field, const void* host, size_t bytes);
/* episode records of the most recent rollout, sorted (step, env) = the reference's
 * logging order (ppo.jl:149). */
CRL_API int crl_pop_episodes(crl_ctx* ctx, crl_episode* out, int32_t max_records, int32_t* n_out, crl_episode_agg* agg);

/* ---- multi-GPU (the reference has none; SURVEY §8e) ------------------------------- */
CRL_API int crl_comm_unique_id(void* out128);                 /* 128 bytes, rank 0 */
CRL_API int crl_comm_init(crl_ctx* ctx, const void* id128);   /* all ranks, collective */

/* ---- instrumentation -------------------------------------------------------------- */
CRL_API int crl_kernel_launches(const crl_ctx* ctx, uint64_t* count); /* kernels launched so far */
/* multi-GPU: number of speculative updates whose on-device verification failed and that were replayed with the
 * exact statistics-exchange sequence (results are exact either way; this is a performance counter) */
CRL_API int crl_spec_replays(const crl_ctx* ctx, uint64_t* count);
CRL_API int crl_profile(crl_ctx* ctx, int32_t enable);  /* per-kernel CUDA-event timing on/off (disables graphs) */
CRL_API int crl_profile_read(crl_ctx* ctx, crl_kernel_times* out, int32_t reset);
CRL_API int crl_stream(const crl_ctx* ctx, void** cuda_stream);

/* ---- raw-pointer kernel entry points (DEVICE pointers; stream = cudaStream_t or NULL) -- */
/* gae(), ppo.jl:48-73 + returns ppo.jl:181. values/rewards/adv/ret float [T][N];
 * dones uint8 [T][N]; next_value float [N]; next_done uint8 [N]. */
CRL_API int crl_gae_raw(const float* values, const float* rewards, const uint8_t* dones,
                const float* next_value, const uint8_t* next_done, float* adv, float* ret,
                int32_t T, int64_t N, float gamma, float lambda, int32_t mode, void* stream);
/* one env step for n envs (upstream CartPoleEnv/PendulumEnv called at multi_thread_env.jl:91).
 * state float [n][S] in/out, t int32 [n] in/out, action int32 [n] (CartPole) or float [n]
 * (Pendulum); reward float [n], done uint8 [n]. No auto-reset. */
CRL_API int crl_env_step_raw(int32_t env_kind, float* state, int32_t* t, const void* action,
                     float* reward, uint8_t* done, int64_t n, int32_t max_episode_steps, void* stream);
/* actor+critic forward (get_action without sampling, ppo.jl:22-24,128). obs float [n][D];
 * out_policy float [n][A] (logits | mean); logp float [n][A] (log-softmax; Gaussian: unused);
 * value float [n]. params = flat device vector. */
CRL_API int crl_policy_forward_raw(int32_t env_kind, const float* params, const float* obs,
                           float* out_policy, float* logp, float* value, int64_t n, void* stream);
/* loss + gradient of one minibatch (ppo.jl:202-244). All device pointers; idx int32[M].
 * grads_out float [P] (un-clipped, summed over the minibatch), stats_out 4 doubles. */
CRL_API int crl_ppo_loss_raw(int32_t env_kind, const float* params, const int32_t* idx, int32_t M,
                     const float* states, const void* actions, const float* logprobs,
                     const float* advantages, const float* returns, const float* values,
                     float clip_coef, float ent_coeff, float v_coef, float* grads_out,
                     double* stats_out, void* stream);
/* Flux.Optimiser(ClipNorm, Adam) step, ppo.jl:93,250. beta_pow double [n_arrays][2]. */
CRL_API int crl_clip_adam_raw(int32_t env_kind, float* params, const float* grads, float* m, float* v,
                      double* beta_pow, double lr, float clip_norm, void* stream);

/* ---- DQN (SURVEY 8f-2; src/algorithms/dqn.jl) ---------------------------------------
 * The reference runs ONE CartPole env (dqn.jl:38) and counts everything in env steps. Here N envs step in
 * lockstep; iteration it (1-based) = one vector step, global_step = it * N. With N = 1 every rule below is the
 * reference's: epsilon = linear_schedule(global_step) (dqn.jl:28-31,52); greedy action = argmax q (first maximum,
 * dqn.jl:56-57); the N transitions are added to the ring buffer in env order (replay_buffer.jl:23-37); a learning
 * step runs when global_step > min_buff_size and it % train_freq == 0 (dqn.jl:94): batch_size indices WITHOUT
 * replacement from [0, size) (replay_buffer.jl:40-45), TD target r + gamma * max_a Q_target(s') * (1 - terminal)
 * in Float64 (dqn.jl:99-100), Flux.mse on the taken action's Q (dqn.jl:104-108), plain Adam (dqn.jl:41); the target
 * net is copied when it % target_net_freq == 0, checked on learning iterations only (dqn.jl:111-113).
 * Network: Dense(4,120,relu), Dense(120,84,relu), Dense(84,2) (dqn.jl:22-26); flat parameters in Flux.params order,
 * each W (out,in) column-major: 10,934 floats. Random draws are Philox streams 3 (epsilon test + random action,
 * counter = it, word = env) and 4 (batch permutation keys, counter = learning step index). Single GPU. */
typedef struct crl_dqn_ctx crl_dqn_ctx;
typedef struct crl_dqn_config {
  int32_t struct_size;       /* = sizeof(crl_dqn_config) */
  int32_t num_envs;          /* N */
  int32_t buffer_size;       /* replay capacity in transitions, dqn.jl:8 (>= num_envs) */
  int32_t min_buff_size;     /* dqn.jl:9 */
  int32_t batch_size;        /* dqn.jl:14, <= 128 */
  int32_t train_freq;        /* dqn.jl:12, in iterations */
  int32_t target_net_freq;   /* dqn.jl:13, in iterations */
  int32_t max_episode_steps; /* CartPoleEnv() default: 200 */
  int32_t device;
  int32_t _pad;
  double lr;                 /* dqn.jl:11 */
  double gamma;              /* dqn.jl:15 */
  double epsilon_start, epsilon_end, epsilon_duration; /* dqn.jl:17-19 */
  uint64_t seed;
} crl_dqn_config;
#define CRL_DQN_PARAMS 10934
typedef struct crl_dqn_stats {
  double last_loss;     /* Flux.mse of the most recent learning step (dqn.jl:116) */
  double sum_return;    /* episodes finished during the call (dqn.jl:80-86) */
  double sum_length;
  double epsilon;       /* at the last iteration */
  int64_t episodes;
  int64_t learn_steps;  /* learning steps so far */
  int64_t iterations;   /* iterations so far; global_step = iterations * num_envs */
  int64_t kernel_launches; /* kernels launched so far (one acting launch covers the iterations up to the next learning step) */
} crl_dqn_stats;
CRL_API int crl_dqn_create(const crl_dqn_config* cfg, crl_dqn_ctx** out);
CRL_API int crl_dqn_destroy(crl_dqn_ctx* ctx);
/* q_net parameters; target_net = deepcopy(q_net) (dqn.jl:40); Adam state reset */
CRL_API int crl_dqn_set_params(crl_dqn_ctx* ctx, const float* params, int32_t n);
CRL_API int crl_dqn_get_params(crl_dqn_ctx* ctx, float* q_params, float* target_params /* may be NULL */, int32_t n);
CRL_API int crl_dqn_reset(crl_dqn_ctx* ctx);   /* reset!(env) for every env, empty buffer, iteration counter 0 */
/* `iterations` vector steps with the learning steps that fall on them; stats may be NULL */
CRL_API int crl_dqn_run(crl_dqn_ctx* ctx, int64_t iterations, crl_dqn_stats* stats);
/* Data-parallel DQN over the GPUs of one box (an extension: dqn.jl has one env and one buffer; BASELINE configs[4]).
 * One handle per GPU and rank; call after crl_dqn_create / crl_dqn_set_params (same parameters on every rank) and
 * BEFORE crl_dqn_reset, on all ranks (collective), with the 128 bytes of crl_comm_unique_id from rank 0. Rank r then
 * owns the envs env_id_base .. env_id_base + num_envs - 1 (Philox is keyed by the global env id; the epsilon schedule
 * and the learning gate count world_size * num_envs steps per iteration), keeps its own ring of buffer_size
 * transitions and contributes batch_size samples of it to a global batch of world_size * batch_size; the gradient is
 * summed with ONE allreduce per learning step and Adam is applied identically on every rank. */
CRL_API int crl_dqn_comm_init(crl_dqn_ctx* ctx, const void* id128, int32_t world_size, int32_t rank, int32_t env_id_base);
/* replay buffer contents (host pointers, each may be NULL): state/next_state float [capacity][4], action int32,
 * reward float, terminal uint8; size/ptr as in replay_buffer.jl:11-12 (ptr 0-based) */
CRL_API int crl_dqn_read_buffer(crl_dqn_ctx* ctx, float* state, int32_t* action, float* reward, float* next_state,
                        uint8_t* terminal, int32_t* size, int32_t* ptr);
/* Raw DQN kernels (DEVICE pointers; stream = cudaStream_t or NULL), the ones crl_dqn_run launches:
 * crl_dqn_forward_raw: q_net(obs) (dqn.jl:56) by the acting kernel's forward pass. params float [10934] and
 * obs float [n][4] 16-byte aligned, q_out float [n][2] 8-byte aligned.
 * crl_dqn_loss_raw: loss and gradient of one batch (dqn.jl:96-108) by the learning step's two kernels, with sample b
 * taken from row b of state / action / reward / next_state / terminal (nothing sampled; rows >= B are not read).
 * q, tgt float [10934]; 1 <= B <= 128; grads_out float [10934] (the un-stepped gradient of Flux.mse, flat order);
 * loss_out 1 double = mean squared TD error. Allocates and frees its scratch: synchronises `stream`. */
CRL_API int crl_dqn_forward_raw(const float* params, const float* obs, float* q_out, int64_t n, void* stream);
CRL_API int crl_dqn_loss_raw(const float* q, const float* tgt, int32_t B, const float* state, const int32_t* action,
                     const float* reward, const float* next_state, const uint8_t* terminal, double gamma,
                     float* grads_out, double* loss_out, void* stream);

/* ---- logger hook: TensorBoard event files (logger.jl:7-29, TBLogger; records of ppo.jl:157,247) -------------------
 * Native writer for the "<message>/<key>" scalars the @info records become in TensorBoardLogger.jl. One call = one
 * record = one Event holding n scalars at `step`. tags: n NUL-terminated strings back to back. Host-only (no GPU). */
typedef struct crl_tb crl_tb;
CRL_API int crl_tb_open(const char* logdir /* existing directory */, crl_tb** out);
CRL_API int crl_tb_scalars(crl_tb* tb, double wall_time, int64_t step, int32_t n, const char* tags, const double* values);
CRL_API int crl_tb_flush(crl_tb* tb);
CRL_API int crl_tb_close(crl_tb* tb);

#ifdef __cplusplus
}
#endif
#endif /* CLEANRL_CUDA_H */
