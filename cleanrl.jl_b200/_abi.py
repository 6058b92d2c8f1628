"""ctypes mirror of include/cleanrl_cuda.h (structs and constants only; loads nothing)."""
import ctypes as C

CRL_VERSION = 100
CRL_OK, CRL_ERR_INVALID, CRL_ERR_CUDA, CRL_ERR_NCCL, CRL_ERR_STATE = 0, -1, -2, -3, -4
CRL_ENV_CARTPOLE, CRL_ENV_PENDULUM = 0, 1
CRL_GAE_REF_COMPAT, CRL_GAE_FIXED, CRL_GAE_A2C_RETURNS = 0, 1, 2
CRL_FLAG_LOCAL_STATS = 1
CRL_FLAG_A2C = 2
CRL_FLAG_NO_VCLIP = 4

(CRL_F_STATE, CRL_F_ACTION, CRL_F_LOGPROB, CRL_F_REWARD, CRL_F_TERMINAL, CRL_F_VALUE,
 CRL_F_ADVANTAGE, CRL_F_RETURN, CRL_F_NEXT_OBS, CRL_F_NEXT_DONE, CRL_F_NEXT_VALUE,
 CRL_F_ENV_STATE, CRL_F_ENV_T, CRL_F_EP_RETURN, CRL_F_EP_LENGTH, CRL_F_RESET_COUNT,
 CRL_F_VNEW) = range(17)

KERNEL_NAMES = ["rollout", "gae", "mb_stats", "mb_count", "loss_grad", "grad_reduce",
                "clip_adam", "allreduce", "other"]
CRL_NUM_KERNELS = len(KERNEL_NAMES)


class crl_config(C.Structure):
    _fields_ = [
        ("struct_size", C.c_int32), ("env_kind", C.c_int32), ("num_envs", C.c_int32),
        ("num_steps", C.c_int32), ("num_minibatches", C.c_int32), ("update_epochs", C.c_int32),
        ("max_episode_steps", C.c_int32), ("gae_mode", C.c_int32), ("device", C.c_int32),
        ("world_size", C.c_int32), ("rank", C.c_int32), ("env_id_base", C.c_int32),
        ("episode_capacity", C.c_int32), ("flags", C.c_uint32),
        ("gamma", C.c_float), ("gae_lambda", C.c_float), ("clip_coef", C.c_float),
        ("ent_coeff", C.c_float), ("v_coef", C.c_float), ("clip_norm", C.c_float),
        ("seed", C.c_uint64),
    ]


class crl_loss_stats(C.Structure):
    _fields_ = [("loss", C.c_double), ("pg_loss", C.c_double), ("v_loss", C.c_double),
                ("entropy_loss", C.c_double)]


class crl_episode(C.Structure):
    _fields_ = [("step", C.c_int32), ("env", C.c_int32), ("length", C.c_int32), ("_pad", C.c_int32),
                ("episode_return", C.c_double)]


class crl_episode_agg(C.Structure):
    _fields_ = [("count", C.c_int64), ("sum_return", C.c_double), ("sum_length", C.c_double),
                ("max_return", C.c_double), ("dropped", C.c_int64)]


class crl_kernel_times(C.Structure):
    _fields_ = [("ms", C.c_double * CRL_NUM_KERNELS), ("launches", C.c_int64 * CRL_NUM_KERNELS)]


def make_config(env_kind=CRL_ENV_CARTPOLE, num_envs=4, num_steps=32, num_minibatches=4, update_epochs=4,
                max_episode_steps=None, gae_mode=CRL_GAE_REF_COMPAT, device=0, world_size=1, rank=0,
                env_id_base=0, episode_capacity=0, flags=0, gamma=0.99, gae_lambda=0.95, clip_coef=0.2,
                ent_coeff=0.01, v_coef=0.5, clip_norm=0.5, seed=1):
    """crl_config with the reference defaults (ppo.jl:1-19, :82, :93)."""
    if max_episode_steps is None:
        max_episode_steps = 500 if env_kind == CRL_ENV_CARTPOLE else 200
    return crl_config(C.sizeof(crl_config), env_kind, num_envs, num_steps, num_minibatches, update_epochs,
                      max_episode_steps, gae_mode, device, world_size, rank, env_id_base, episode_capacity,
                      flags, gamma, gae_lambda, clip_coef, ent_coeff, v_coef, clip_norm, seed)


# ---- DQN (include/cleanrl_cuda.h, "DQN" section) -------------------------------------------------------------
CRL_DQN_PARAMS = 10934


class crl_dqn_config(C.Structure):
    _fields_ = [
        ("struct_size", C.c_int32), ("num_envs", C.c_int32), ("buffer_size", C.c_int32), ("min_buff_size", C.c_int32),
        ("batch_size", C.c_int32), ("train_freq", C.c_int32), ("target_net_freq", C.c_int32),
        ("max_episode_steps", C.c_int32), ("device", C.c_int32), ("_pad", C.c_int32),
        ("lr", C.c_double), ("gamma", C.c_double), ("epsilon_start", C.c_double), ("epsilon_end", C.c_double),
        ("epsilon_duration", C.c_double), ("seed", C.c_uint64),
    ]


class crl_dqn_stats(C.Structure):
    _fields_ = [("last_loss", C.c_double), ("sum_return", C.c_double), ("sum_length", C.c_double), ("epsilon", C.c_double),
                ("episodes", C.c_int64), ("learn_steps", C.c_int64), ("iterations", C.c_int64), ("kernel_launches", C.c_int64)]


def make_dqn_config(num_envs=1, buffer_size=10_000, min_buff_size=200, batch_size=120, train_freq=10, target_net_freq=100,
                    max_episode_steps=200, device=0, lr=1e-4, gamma=0.99, epsilon_start=1.0, epsilon_end=0.05,
                    epsilon_duration=10_000.0, seed=1):
    """crl_dqn_config with the reference defaults (dqn.jl:1-20; CartPoleEnv() max_steps = 200)."""
    return crl_dqn_config(C.sizeof(crl_dqn_config), num_envs, buffer_size, min_buff_size, batch_size, train_freq,
                          target_net_freq, max_episode_steps, device, 0, lr, gamma, epsilon_start, epsilon_end,
                          epsilon_duration, seed)


# ---- DDPG (include/cleanrl_ddpg.h) ----------------------------------------------------------------------------
CRL_DDPG_ACTOR_PARAMS = 4481
CRL_DDPG_CRITIC_PARAMS = 4545


class crl_ddpg_config(C.Structure):
    _fields_ = [
        ("struct_size", C.c_int32), ("num_envs", C.c_int32), ("buffer_size", C.c_int32), ("learning_starts", C.c_int32),
        ("batch_size", C.c_int32), ("train_freq", C.c_int32), ("policy_frequency", C.c_int32),
        ("max_episode_steps", C.c_int32), ("device", C.c_int32), ("_pad", C.c_int32),
        ("gamma", C.c_double), ("tau", C.c_double), ("lr", C.c_double), ("exploration_noise", C.c_double), ("seed", C.c_uint64),
    ]


class crl_ddpg_stats(C.Structure):
    _fields_ = [("critic_loss", C.c_double), ("actor_loss", C.c_double), ("sum_return", C.c_double), ("sum_length", C.c_double),
                ("episodes", C.c_int64), ("learn_steps", C.c_int64), ("actor_steps", C.c_int64), ("iterations", C.c_int64),
                ("kernel_launches", C.c_int64)]


def make_ddpg_config(num_envs=1, buffer_size=1_000_000, learning_starts=25_000, batch_size=256, train_freq=1, policy_frequency=2,
                     max_episode_steps=200, device=0, gamma=0.99, tau=0.005, lr=3e-4, exploration_noise=0.1, seed=1):
    """crl_ddpg_config with CleanRL's ddpg_continuous_action.py defaults (PendulumEnv() max_steps = 200)."""
    return crl_ddpg_config(C.sizeof(crl_ddpg_config), num_envs, buffer_size, learning_starts, batch_size, train_freq,
                           policy_frequency, max_episode_steps, device, 0, gamma, tau, lr, exploration_noise, seed)


# ---- TD3 (include/cleanrl_td3.h) -----------------------------------------------------------------------------
class crl_td3_config(C.Structure):
    _fields_ = crl_ddpg_config._fields_ + [("policy_noise", C.c_double), ("noise_clip", C.c_double)]


class crl_td3_stats(C.Structure):
    _fields_ = [("qf1_loss", C.c_double), ("qf2_loss", C.c_double), ("actor_loss", C.c_double), ("sum_return", C.c_double),
                ("sum_length", C.c_double), ("episodes", C.c_int64), ("learn_steps", C.c_int64), ("actor_steps", C.c_int64),
                ("iterations", C.c_int64), ("kernel_launches", C.c_int64)]


def make_td3_config(num_envs=1, buffer_size=1_000_000, learning_starts=25_000, batch_size=256, train_freq=1, policy_frequency=2,
                    max_episode_steps=200, device=0, gamma=0.99, tau=0.005, lr=3e-4, exploration_noise=0.1, seed=1,
                    policy_noise=0.2, noise_clip=0.5):
    """crl_td3_config with CleanRL's td3_continuous_action.py defaults (PendulumEnv() max_steps = 200)."""
    return crl_td3_config(C.sizeof(crl_td3_config), num_envs, buffer_size, learning_starts, batch_size, train_freq,
                          policy_frequency, max_episode_steps, device, 0, gamma, tau, lr, exploration_noise, seed,
                          policy_noise, noise_clip)


# ---- SAC (include/cleanrl_sac.h) -----------------------------------------------------------------------------
CRL_SAC_ACTOR_PARAMS = 4546


class crl_sac_config(C.Structure):
    _fields_ = [
        ("struct_size", C.c_int32), ("num_envs", C.c_int32), ("buffer_size", C.c_int32), ("learning_starts", C.c_int32),
        ("batch_size", C.c_int32), ("train_freq", C.c_int32), ("policy_frequency", C.c_int32),
        ("target_network_frequency", C.c_int32), ("max_episode_steps", C.c_int32), ("device", C.c_int32),
        ("autotune", C.c_int32), ("_pad", C.c_int32),
        ("gamma", C.c_double), ("tau", C.c_double), ("policy_lr", C.c_double), ("q_lr", C.c_double), ("alpha", C.c_double),
        ("seed", C.c_uint64),
    ]


class crl_sac_stats(C.Structure):
    _fields_ = [("qf1_loss", C.c_double), ("qf2_loss", C.c_double), ("actor_loss", C.c_double), ("alpha_loss", C.c_double),
                ("alpha", C.c_double), ("sum_return", C.c_double), ("sum_length", C.c_double), ("episodes", C.c_int64),
                ("learn_steps", C.c_int64), ("actor_steps", C.c_int64), ("iterations", C.c_int64), ("kernel_launches", C.c_int64)]


def make_sac_config(num_envs=1, buffer_size=1_000_000, learning_starts=5_000, batch_size=256, train_freq=1, policy_frequency=2,
                    target_network_frequency=1, max_episode_steps=200, device=0, autotune=1, gamma=0.99, tau=0.005,
                    policy_lr=3e-4, q_lr=1e-3, alpha=0.2, seed=1):
    """crl_sac_config with CleanRL's sac_continuous_action.py defaults (PendulumEnv() max_steps = 200)."""
    return crl_sac_config(C.sizeof(crl_sac_config), num_envs, buffer_size, learning_starts, batch_size, train_freq,
                          policy_frequency, target_network_frequency, max_episode_steps, device, autotune, 0, gamma, tau,
                          policy_lr, q_lr, alpha, seed)


# ---- C51 (include/cleanrl_c51.h) -----------------------------------------------------------------------------
CRL_C51_ATOMS = 101
CRL_C51_PARAMS = 27934


class crl_c51_config(C.Structure):
    _fields_ = [
        ("struct_size", C.c_int32), ("num_envs", C.c_int32), ("buffer_size", C.c_int32), ("learning_starts", C.c_int32),
        ("batch_size", C.c_int32), ("train_frequency", C.c_int32), ("target_network_frequency", C.c_int32),
        ("max_episode_steps", C.c_int32), ("device", C.c_int32), ("_pad", C.c_int32),
        ("lr", C.c_double), ("gamma", C.c_double), ("start_e", C.c_double), ("end_e", C.c_double),
        ("epsilon_duration", C.c_double), ("v_min", C.c_double), ("v_max", C.c_double), ("seed", C.c_uint64),
    ]


class crl_c51_stats(C.Structure):
    _fields_ = [("loss", C.c_double), ("q_values", C.c_double), ("sum_return", C.c_double), ("sum_length", C.c_double),
                ("epsilon", C.c_double), ("episodes", C.c_int64), ("learn_steps", C.c_int64), ("target_copies", C.c_int64),
                ("iterations", C.c_int64), ("kernel_launches", C.c_int64)]


def make_c51_config(num_envs=1, buffer_size=10_000, learning_starts=10_000, batch_size=128, train_frequency=10,
                    target_network_frequency=500, max_episode_steps=500, device=0, lr=2.5e-4, gamma=0.99, start_e=1.0,
                    end_e=0.05, epsilon_duration=250_000.0, v_min=-100.0, v_max=100.0, seed=1):
    """crl_c51_config with CleanRL's c51.py defaults (epsilon_duration = exploration_fraction 0.5 x total_timesteps
    500,000; CartPole-v1's 500-step limit)."""
    return crl_c51_config(C.sizeof(crl_c51_config), num_envs, buffer_size, learning_starts, batch_size, train_frequency,
                          target_network_frequency, max_episode_steps, device, 0, lr, gamma, start_e, end_e,
                          epsilon_duration, v_min, v_max, seed)
