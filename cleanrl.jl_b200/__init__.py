"""cleanrl.jl_b200 — B200-native PPO hot path of sash-a/CleanRL.jl behind a C ABI.

Host-side mirror of the reference's Julia interface (Python stands in for Julia, which is not
available in this image): PPOConfig / ppo() (ppo.jl), ConfigParser.argparse_struct
(config_parser.jl), Logger.make_logger (logger.jl), Networks.make_actor_critic (networks.jl).
All compute happens in libcleanrl_cuda.so (csrc/, sm_100a); importing this package loads
nothing — the library is dlopen'ed on first use and there is no CPU fallback.
"""
from . import _abi  # noqa: F401
from .config import PPOConfig, argparse_struct  # noqa: F401

__all__ = ["PPOConfig", "A2CConfig", "DQNConfig", "DDPGConfig", "TD3Config", "SACConfig", "C51Config", "argparse_struct", "ppo", "a2c", "dqn", "ddpg", "td3",
           "sac", "c51",
           "PPOHandle", "Networks", "Logger",
           "ConfigParser"]


def ppo(*args, **kwargs):
    """Drop-in for CleanRL.ppo(config) (ppo.jl:75); see ppo_algo.py."""
    from .ppo_algo import ppo as _ppo
    return _ppo(*args, **kwargs)


def a2c(*args, **kwargs):
    """Vectorised A2C on the same kernels (a2c.jl:30); see a2c_algo.py."""
    from .a2c_algo import a2c as _a2c
    return _a2c(*args, **kwargs)


def dqn(*args, **kwargs):
    """CleanRL.dqn(config) (dqn.jl:34), vectorised on the GPU: see dqn_algo.py"""
    from .dqn_algo import dqn as _dqn
    return _dqn(*args, **kwargs)


def ddpg(*args, **kwargs):
    """Vectorised DDPG on Pendulum (pinned to include/cleanrl_ddpg.h, not ddpg.jl); see ddpg_algo.py"""
    from .ddpg_algo import ddpg as _ddpg
    return _ddpg(*args, **kwargs)


def td3(*args, **kwargs):
    """Vectorised TD3 on Pendulum (pinned to include/cleanrl_td3.h; the reference has no TD3); see td3_algo.py"""
    from .td3_algo import td3 as _td3
    return _td3(*args, **kwargs)


def sac(*args, **kwargs):
    """Vectorised SAC on Pendulum (pinned to include/cleanrl_sac.h; the reference has no SAC); see sac_algo.py"""
    from .sac_algo import sac as _sac
    return _sac(*args, **kwargs)


def c51(*args, **kwargs):
    """Vectorised C51 on CartPole (pinned to include/cleanrl_c51.h; the reference has no C51); see c51_algo.py"""
    from .c51_algo import c51 as _c51
    return _c51(*args, **kwargs)


def __getattr__(name):
    if name == "C51Config":
        from .c51_algo import C51Config
        return C51Config
    if name == "SACConfig":
        from .sac_algo import SACConfig
        return SACConfig
    if name == "TD3Config":
        from .td3_algo import TD3Config
        return TD3Config
    if name == "DDPGConfig":
        from .ddpg_algo import DDPGConfig
        return DDPGConfig
    if name == "DQNConfig":
        from .dqn_algo import DQNConfig
        return DQNConfig
    # lazy: keep `import cleanrl_jl_b200` free of ctypes/torch side effects
    if name == "A2CConfig":
        from .a2c_algo import A2CConfig
        return A2CConfig
    if name == "PPOHandle":
        from .handle import PPOHandle
        return PPOHandle
    if name == "Networks":
        from . import networks
        return networks
    if name == "Logger":
        from . import logger
        return logger
    if name == "ConfigParser":
        from . import config
        return config
    raise AttributeError(name)
