"""ddpg(config) — vectorised DDPG on Pendulum over the crl_ddpg_* entry points (include/cleanrl_ddpg.h).

The reference's ddpg.jl trains on MuJoCo HalfCheetah through PyCall, which this library does not have, and its source is
not part of this checkout. DDPG parity is therefore pinned to the definition in include/cleanrl_ddpg.h (CleanRL-Python's
ddpg_continuous_action.py on Pendulum, with 64-wide nets), not to ddpg.jl. `DDPGConfig` keeps CleanRL's field names and
defaults and adds `train_freq`, `num_envs`, `seed` and `max_steps`. `num_envs` envs step in lockstep on the GPU;
`num_envs = 1` is CleanRL's update-to-data ratio of one learning step per env step."""
import ctypes as C
import dataclasses
import datetime
import time

import numpy as np

from . import _abi
from . import _lib as L
from . import logger as Logger


@dataclasses.dataclass
class DDPGConfig:
    run_name: str = dataclasses.field(default_factory=lambda: datetime.datetime.now().strftime("%y-%m-%d|%H:%M:%S"))
    log_frequency: int = 1000           # global steps between log records
    total_timesteps: int = 1_000_000
    buffer_size: int = 1_000_000
    learning_starts: int = 25_000
    batch_size: int = 256               # at most 256
    gamma: float = 0.99
    tau: float = 0.005
    lr: float = 3e-4                    # both nets
    exploration_noise: float = 0.1      # times the torque limit 2
    policy_frequency: int = 2
    # ---- not in CleanRL
    train_freq: int = 1                 # iterations between learning steps
    num_envs: int = 1
    seed: int = 1
    max_steps: int = 200                # PendulumEnv() default


def init_ddpg_params(seed=0):
    """(actor, critic): Chain(Dense(3,64,relu), Dense(64,64,relu), Dense(64,1)) and Chain(Dense(4,64,relu), Dense(64,64,relu),
    Dense(64,1)) with Flux's default glorot_uniform weights and zero biases, each flattened in Flux.params order with W
    (out,in) column-major (as init_q_params of dqn_algo.py)."""
    rng = np.random.default_rng(seed)
    nets = []
    for d_in, size in ((3, _abi.CRL_DDPG_ACTOR_PARAMS), (4, _abi.CRL_DDPG_CRITIC_PARAMS)):
        out = []
        for fan_in, fan_out in ((d_in, 64), (64, 64), (64, 1)):
            lim = np.sqrt(6.0 / (fan_in + fan_out))
            w = rng.uniform(-lim, lim, size=(fan_out, fan_in)).astype(np.float32)
            out.append(w.ravel(order="F"))
            out.append(np.zeros(fan_out, np.float32))
        p = np.concatenate(out)
        assert p.size == size
        nets.append(p)
    return nets[0], nets[1]


class DDPGHandle:
    """object wrapper over crl_ddpg_ctx"""

    def __init__(self, cfg):
        self.lib = L.load()
        self.cfg = cfg
        h = C.c_void_p()
        L.check(self.lib.crl_ddpg_create(C.byref(cfg), C.byref(h)))
        self.h = h

    def close(self):
        if self.h:
            L.check(self.lib.crl_ddpg_destroy(self.h))
            self.h = None

    def set_params(self, actor, critic):
        a = np.ascontiguousarray(actor, np.float32)
        c = np.ascontiguousarray(critic, np.float32)
        L.check(self.lib.crl_ddpg_set_params(self.h, L.ptr(a), a.size, L.ptr(c), c.size))

    def get_params(self):
        """dict of actor, critic, actor_target, critic_target"""
        out = {k: np.zeros(n, np.float32) for k, n in (("actor", _abi.CRL_DDPG_ACTOR_PARAMS), ("critic", _abi.CRL_DDPG_CRITIC_PARAMS),
                                                     ("actor_target", _abi.CRL_DDPG_ACTOR_PARAMS),
                                                     ("critic_target", _abi.CRL_DDPG_CRITIC_PARAMS))}
        L.check(self.lib.crl_ddpg_get_params(self.h, *[L.ptr(out[k]) for k in ("actor", "critic", "actor_target", "critic_target")]))
        return out

    def get_adam_state(self):
        """dict of actor_m, actor_v, critic_m, critic_v and beta_pow (actor b1^t, b2^t, critic b1^t, b2^t)"""
        out = {k: np.zeros(n, np.float32) for k, n in (("actor_m", _abi.CRL_DDPG_ACTOR_PARAMS), ("actor_v", _abi.CRL_DDPG_ACTOR_PARAMS),
                                                     ("critic_m", _abi.CRL_DDPG_CRITIC_PARAMS), ("critic_v", _abi.CRL_DDPG_CRITIC_PARAMS))}
        out["beta_pow"] = np.zeros(4, np.float64)
        L.check(self.lib.crl_ddpg_get_adam_state(self.h, *[L.ptr(out[k]) for k in ("actor_m", "actor_v", "critic_m", "critic_v", "beta_pow")]))
        return out

    def reset(self):
        L.check(self.lib.crl_ddpg_reset(self.h))

    def run(self, iterations):
        st = _abi.crl_ddpg_stats()
        L.check(self.lib.crl_ddpg_run(self.h, int(iterations), C.byref(st)))
        return st

    def read_buffer(self):
        cap = self.cfg.buffer_size
        out = {"obs": np.zeros((cap, 3), np.float32), "action": np.zeros(cap, np.float32), "reward": np.zeros(cap, np.float32),
               "next_obs": np.zeros((cap, 3), np.float32), "terminal": np.zeros(cap, np.uint8)}
        size, ptr = C.c_int32(), C.c_int32()
        L.check(self.lib.crl_ddpg_read_buffer(self.h, L.ptr(out["obs"]), L.ptr(out["action"]), L.ptr(out["reward"]),
                                              L.ptr(out["next_obs"]), L.ptr(out["terminal"]), C.byref(size), C.byref(ptr)))
        out["size"], out["ptr"] = size.value, ptr.value
        return out


def make_crl_ddpg_config(config, device=0):
    return _abi.make_ddpg_config(num_envs=config.num_envs, buffer_size=config.buffer_size, learning_starts=config.learning_starts,
                                 batch_size=config.batch_size, train_freq=config.train_freq,
                                 policy_frequency=config.policy_frequency, max_episode_steps=config.max_steps, device=device,
                                 gamma=config.gamma, tau=config.tau, lr=config.lr, exploration_noise=config.exploration_noise,
                                 seed=config.seed)


def ddpg(config=None, logger=None, params=None, device=0):
    """Runs `total_timesteps` env steps and returns a summary dict. Logs "Episode Statistics" (episode_return,
    episode_length, global_step, steps_per_sec) over the episodes that ended since the last record, and "Training
    Statistics" (critic_loss, actor_loss) every `log_frequency` steps. `params` = (actor, critic) or None."""
    config = config or DDPGConfig()
    own_logger = logger is None
    if own_logger:
        logger = Logger.make_logger("ddpg|%s" % config.run_name, to_terminal=False)
    h = DDPGHandle(make_crl_ddpg_config(config, device))
    try:
        h.set_params(*(init_ddpg_params(config.seed) if params is None else params))
        h.reset()
        n_iter = config.total_timesteps // config.num_envs
        chunk = max(1, config.log_frequency // config.num_envs)
        start = time.time()
        done_iter, episodes, last = 0, 0, None
        returns = []                     # mean return of each record, in order
        while done_iter < n_iter:
            k = min(chunk, n_iter - done_iter)
            last = h.run(k)
            done_iter += k
            global_step = done_iter * config.num_envs
            if last.episodes > 0:
                episodes += last.episodes
                returns.append(last.sum_return / last.episodes)
                logger.info("Episode Statistics", episode_return=returns[-1], episode_length=last.sum_length / last.episodes,
                            global_step=global_step, steps_per_sec=int(global_step / max(time.time() - start, 1e-9)))
            if last.learn_steps > 0:
                logger.info("Training Statistics", critic_loss=last.critic_loss,
                            actor_loss=last.actor_loss if last.actor_steps > 0 else float("nan"))
        wall = time.time() - start
        p = h.get_params()
    finally:
        h.close()
        if own_logger:
            logger.close()
    return {"global_step": n_iter * config.num_envs, "episodes": episodes,
            "learn_steps": int(last.learn_steps) if last else 0, "actor_steps": int(last.actor_steps) if last else 0,
            "critic_loss": float(last.critic_loss) if last else float("nan"),
            "actor_loss": float(last.actor_loss) if last and last.actor_steps else float("nan"),
            "steps_per_sec": n_iter * config.num_envs / max(wall, 1e-9), "episode_returns": returns,
            "last_mean_return": returns[-1] if returns else float("nan"), **p}
