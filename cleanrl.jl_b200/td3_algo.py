"""td3(config) — vectorised TD3 on Pendulum over the crl_td3_* entry points (include/cleanrl_td3.h).

The reference has no TD3; this is an extension next to DDPG. Its semantics are pinned to the definition in
include/cleanrl_td3.h: CleanRL-Python's td3_continuous_action.py on Pendulum, with the 64-wide nets of the DDPG part.
`TD3Config` keeps CleanRL's field names and defaults and adds `train_freq`, `num_envs`, `seed` and `max_steps`, as
`DDPGConfig` does. `num_envs = 1` is CleanRL's update-to-data ratio of one learning step per env step."""
import ctypes as C
import dataclasses
import datetime
import time

import numpy as np

from . import _abi
from . import _lib as L
from . import logger as Logger
from .ddpg_algo import init_ddpg_params


@dataclasses.dataclass
class TD3Config:
    run_name: str = dataclasses.field(default_factory=lambda: datetime.datetime.now().strftime("%y-%m-%d|%H:%M:%S"))
    log_frequency: int = 1000           # global steps between log records
    total_timesteps: int = 1_000_000
    buffer_size: int = 1_000_000
    learning_starts: int = 25_000
    batch_size: int = 256               # at most 256
    gamma: float = 0.99
    tau: float = 0.005
    lr: float = 3e-4                    # all three nets
    exploration_noise: float = 0.1      # times the torque limit 2
    policy_frequency: int = 2
    policy_noise: float = 0.2           # target smoothing noise, before the clip
    noise_clip: float = 0.5             # times the torque limit 2 after the clip
    # ---- not in CleanRL
    train_freq: int = 1                 # iterations between learning steps
    num_envs: int = 1
    seed: int = 1
    max_steps: int = 200                # PendulumEnv() default


def init_td3_params(seed=0):
    """(actor, qf1, qf2): actor and qf1 are init_ddpg_params(seed); qf2 is the critic init_ddpg_params draws for
    seed + 2^32, a generator of its own, so it never equals the qf1 of another 32-bit seed."""
    actor, qf1 = init_ddpg_params(seed)
    return actor, qf1, init_ddpg_params(seed + (1 << 32))[1]


class TD3Handle:
    """object wrapper over crl_td3_ctx"""

    NETS = (("actor", _abi.CRL_DDPG_ACTOR_PARAMS), ("qf1", _abi.CRL_DDPG_CRITIC_PARAMS), ("qf2", _abi.CRL_DDPG_CRITIC_PARAMS))

    def __init__(self, cfg):
        self.lib = L.load()
        self.cfg = cfg
        h = C.c_void_p()
        L.check(self.lib.crl_td3_create(C.byref(cfg), C.byref(h)))
        self.h = h

    def close(self):
        if self.h:
            L.check(self.lib.crl_td3_destroy(self.h))
            self.h = None

    def set_params(self, actor, qf1, qf2):
        a, q1, q2 = (np.ascontiguousarray(x, np.float32) for x in (actor, qf1, qf2))
        L.check(self.lib.crl_td3_set_params(self.h, L.ptr(a), a.size, L.ptr(q1), q1.size, L.ptr(q2), q2.size))

    def get_params(self):
        """dict of actor, qf1, qf2, actor_target, qf1_target, qf2_target"""
        keys = [k for k, _ in self.NETS] + [k + "_target" for k, _ in self.NETS]
        out = {k: np.zeros(n, np.float32) for k, n in self.NETS}
        out.update({k + "_target": np.zeros(n, np.float32) for k, n in self.NETS})
        L.check(self.lib.crl_td3_get_params(self.h, *[L.ptr(out[k]) for k in keys]))
        return out

    def get_adam_state(self):
        """dict of actor_m, actor_v, qf1_m, qf1_v, qf2_m, qf2_v and beta_pow (actor b1^t, b2^t, critics b1^t, b2^t)"""
        keys = [k + s for k, _ in self.NETS for s in ("_m", "_v")]
        out = {k + s: np.zeros(n, np.float32) for k, n in self.NETS for s in ("_m", "_v")}
        out["beta_pow"] = np.zeros(4, np.float64)
        L.check(self.lib.crl_td3_get_adam_state(self.h, *[L.ptr(out[k]) for k in keys + ["beta_pow"]]))
        return out

    def reset(self):
        L.check(self.lib.crl_td3_reset(self.h))

    def run(self, iterations):
        st = _abi.crl_td3_stats()
        L.check(self.lib.crl_td3_run(self.h, int(iterations), C.byref(st)))
        return st

    def read_buffer(self):
        cap = self.cfg.buffer_size
        out = {"obs": np.zeros((cap, 3), np.float32), "action": np.zeros(cap, np.float32), "reward": np.zeros(cap, np.float32),
               "next_obs": np.zeros((cap, 3), np.float32), "terminal": np.zeros(cap, np.uint8)}
        size, ptr = C.c_int32(), C.c_int32()
        L.check(self.lib.crl_td3_read_buffer(self.h, L.ptr(out["obs"]), L.ptr(out["action"]), L.ptr(out["reward"]),
                                             L.ptr(out["next_obs"]), L.ptr(out["terminal"]), C.byref(size), C.byref(ptr)))
        out["size"], out["ptr"] = size.value, ptr.value
        return out


def make_crl_td3_config(config, device=0):
    return _abi.make_td3_config(num_envs=config.num_envs, buffer_size=config.buffer_size, learning_starts=config.learning_starts,
                                batch_size=config.batch_size, train_freq=config.train_freq,
                                policy_frequency=config.policy_frequency, max_episode_steps=config.max_steps, device=device,
                                gamma=config.gamma, tau=config.tau, lr=config.lr, exploration_noise=config.exploration_noise,
                                seed=config.seed, policy_noise=config.policy_noise, noise_clip=config.noise_clip)


def td3(config=None, logger=None, params=None, device=0):
    """Runs `total_timesteps` env steps and returns a summary dict. Logs "Episode Statistics" (episode_return,
    episode_length, global_step, steps_per_sec) over the episodes that ended since the last record, and "Training
    Statistics" (qf1_loss, qf2_loss, actor_loss) every `log_frequency` steps. `params` = (actor, qf1, qf2) or None."""
    config = config or TD3Config()
    own_logger = logger is None
    if own_logger:
        logger = Logger.make_logger("td3|%s" % config.run_name, to_terminal=False)
    h = TD3Handle(make_crl_td3_config(config, device))
    try:
        h.set_params(*(init_td3_params(config.seed) if params is None else params))
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
                logger.info("Training Statistics", qf1_loss=last.qf1_loss, qf2_loss=last.qf2_loss,
                            actor_loss=last.actor_loss if last.actor_steps > 0 else float("nan"))
        wall = time.time() - start
        p = h.get_params()
    finally:
        h.close()
        if own_logger:
            logger.close()
    return {"global_step": n_iter * config.num_envs, "episodes": episodes,
            "learn_steps": int(last.learn_steps) if last else 0, "actor_steps": int(last.actor_steps) if last else 0,
            "qf1_loss": float(last.qf1_loss) if last else float("nan"),
            "qf2_loss": float(last.qf2_loss) if last else float("nan"),
            "actor_loss": float(last.actor_loss) if last and last.actor_steps else float("nan"),
            "steps_per_sec": n_iter * config.num_envs / max(wall, 1e-9), "episode_returns": returns,
            "last_mean_return": returns[-1] if returns else float("nan"), **p}
