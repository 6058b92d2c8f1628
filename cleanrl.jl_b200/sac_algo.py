"""sac(config) — vectorised SAC on Pendulum over the crl_sac_* entry points (include/cleanrl_sac.h).

The reference has no SAC; this is an extension next to DDPG and TD3. Its semantics are pinned to the definition in
include/cleanrl_sac.h: CleanRL-Python's sac_continuous_action.py on Pendulum, with the 64-wide nets of the DDPG part.
`SACConfig` keeps CleanRL's field names and defaults and adds `train_freq`, `num_envs`, `seed`, `max_steps` and
`log_frequency`, as `TD3Config` does. `num_envs = 1` is CleanRL's update-to-data ratio of one learning step per env
step."""
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
class SACConfig:
    run_name: str = dataclasses.field(default_factory=lambda: datetime.datetime.now().strftime("%y-%m-%d|%H:%M:%S"))
    log_frequency: int = 1000           # global steps between log records
    total_timesteps: int = 1_000_000
    buffer_size: int = 1_000_000
    learning_starts: int = 5_000
    batch_size: int = 256               # at most 256
    gamma: float = 0.99
    tau: float = 0.005
    policy_lr: float = 3e-4
    q_lr: float = 1e-3                  # both critics and the temperature
    policy_frequency: int = 2
    target_network_frequency: int = 1
    alpha: float = 0.2                  # the temperature when autotune is off
    autotune: bool = True
    # ---- not in CleanRL
    train_freq: int = 1                 # iterations between learning steps
    num_envs: int = 1
    seed: int = 1
    max_steps: int = 200                # PendulumEnv() default


def init_sac_params(seed=0):
    """(actor, qf1, qf2). The actor is Dense(3,64,relu) -> Dense(64,64,relu) with the heads fc_mean and fc_logstd
    Dense(64,1), with glorot_uniform weights and zero biases as init_ddpg_params, flattened W1, b1, W2, b2, W_mean, b_mean,
    W_logstd, b_logstd with W (out,in) column-major; qf1 and qf2 are the critics init_td3_params draws."""
    rng = np.random.default_rng(seed)
    out = []
    for fan_in, fan_out in ((3, 64), (64, 64), (64, 1), (64, 1)):
        lim = np.sqrt(6.0 / (fan_in + fan_out))
        out.append(rng.uniform(-lim, lim, size=(fan_out, fan_in)).astype(np.float32).ravel(order="F"))
        out.append(np.zeros(fan_out, np.float32))
    actor = np.concatenate(out)
    assert actor.size == _abi.CRL_SAC_ACTOR_PARAMS
    return actor, init_ddpg_params(seed)[1], init_ddpg_params(seed + (1 << 32))[1]


class SACHandle:
    """object wrapper over crl_sac_ctx"""

    NETS = (("actor", _abi.CRL_SAC_ACTOR_PARAMS), ("qf1", _abi.CRL_DDPG_CRITIC_PARAMS), ("qf2", _abi.CRL_DDPG_CRITIC_PARAMS))

    def __init__(self, cfg):
        self.lib = L.load()
        self.cfg = cfg
        h = C.c_void_p()
        L.check(self.lib.crl_sac_create(C.byref(cfg), C.byref(h)))
        self.h = h

    def close(self):
        if self.h:
            L.check(self.lib.crl_sac_destroy(self.h))
            self.h = None

    def set_params(self, actor, qf1, qf2):
        a, q1, q2 = (np.ascontiguousarray(x, np.float32) for x in (actor, qf1, qf2))
        L.check(self.lib.crl_sac_set_params(self.h, L.ptr(a), a.size, L.ptr(q1), q1.size, L.ptr(q2), q2.size))

    def get_params(self):
        """dict of actor, qf1, qf2, qf1_target, qf2_target and log_alpha (a float)"""
        keys = ["actor", "qf1", "qf2", "qf1_target", "qf2_target"]
        out = {k: np.zeros(n, np.float32) for k, n in self.NETS}
        out.update({k + "_target": np.zeros(n, np.float32) for k, n in self.NETS[1:]})
        la = np.zeros(1, np.float32)
        L.check(self.lib.crl_sac_get_params(self.h, *[L.ptr(out[k]) for k in keys], L.ptr(la)))
        out["log_alpha"] = float(la[0])
        return out

    def get_adam_state(self):
        """dict of actor_m, actor_v, qf1_m, qf1_v, qf2_m, qf2_v, log_alpha_mv (m, v) and beta_pow (actor and log_alpha
        b1^t, b2^t, critics b1^t, b2^t)"""
        keys = [k + s for k, _ in self.NETS for s in ("_m", "_v")]
        out = {k + s: np.zeros(n, np.float32) for k, n in self.NETS for s in ("_m", "_v")}
        out["log_alpha_mv"] = np.zeros(2, np.float32)
        out["beta_pow"] = np.zeros(4, np.float64)
        L.check(self.lib.crl_sac_get_adam_state(self.h, *[L.ptr(out[k]) for k in keys + ["log_alpha_mv", "beta_pow"]]))
        return out

    def reset(self):
        L.check(self.lib.crl_sac_reset(self.h))

    def run(self, iterations):
        st = _abi.crl_sac_stats()
        L.check(self.lib.crl_sac_run(self.h, int(iterations), C.byref(st)))
        return st

    def read_buffer(self):
        cap = self.cfg.buffer_size
        out = {"obs": np.zeros((cap, 3), np.float32), "action": np.zeros(cap, np.float32), "reward": np.zeros(cap, np.float32),
               "next_obs": np.zeros((cap, 3), np.float32), "terminal": np.zeros(cap, np.uint8)}
        size, ptr = C.c_int32(), C.c_int32()
        L.check(self.lib.crl_sac_read_buffer(self.h, L.ptr(out["obs"]), L.ptr(out["action"]), L.ptr(out["reward"]),
                                             L.ptr(out["next_obs"]), L.ptr(out["terminal"]), C.byref(size), C.byref(ptr)))
        out["size"], out["ptr"] = size.value, ptr.value
        return out


def make_crl_sac_config(config, device=0):
    return _abi.make_sac_config(num_envs=config.num_envs, buffer_size=config.buffer_size, learning_starts=config.learning_starts,
                                batch_size=config.batch_size, train_freq=config.train_freq,
                                policy_frequency=config.policy_frequency,
                                target_network_frequency=config.target_network_frequency, max_episode_steps=config.max_steps,
                                device=device, autotune=int(bool(config.autotune)), gamma=config.gamma, tau=config.tau,
                                policy_lr=config.policy_lr, q_lr=config.q_lr, alpha=config.alpha, seed=config.seed)


def sac(config=None, logger=None, params=None, device=0):
    """Runs `total_timesteps` env steps and returns a summary dict. Logs "Episode Statistics" (episode_return,
    episode_length, global_step, steps_per_sec) over the episodes that ended since the last record, and "Training
    Statistics" (qf1_loss, qf2_loss, actor_loss, alpha_loss, alpha) every `log_frequency` steps. `params` = (actor, qf1,
    qf2) or None."""
    config = config or SACConfig()
    own_logger = logger is None
    if own_logger:
        logger = Logger.make_logger("sac|%s" % config.run_name, to_terminal=False)
    h = SACHandle(make_crl_sac_config(config, device))
    try:
        h.set_params(*(init_sac_params(config.seed) if params is None else params))
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
                acted = last.actor_steps > 0
                logger.info("Training Statistics", qf1_loss=last.qf1_loss, qf2_loss=last.qf2_loss,
                            actor_loss=last.actor_loss if acted else float("nan"),
                            alpha_loss=last.alpha_loss if acted and config.autotune else float("nan"), alpha=last.alpha)
        wall = time.time() - start
        p = h.get_params()
    finally:
        h.close()
        if own_logger:
            logger.close()
    acted = bool(last and last.actor_steps)
    return {"global_step": n_iter * config.num_envs, "episodes": episodes,
            "learn_steps": int(last.learn_steps) if last else 0, "actor_steps": int(last.actor_steps) if last else 0,
            "qf1_loss": float(last.qf1_loss) if last else float("nan"),
            "qf2_loss": float(last.qf2_loss) if last else float("nan"),
            "actor_loss": float(last.actor_loss) if acted else float("nan"),
            "alpha_loss": float(last.alpha_loss) if acted and config.autotune else float("nan"),
            "alpha": float(last.alpha) if last else float("nan"),
            "steps_per_sec": n_iter * config.num_envs / max(wall, 1e-9), "episode_returns": returns,
            "last_mean_return": returns[-1] if returns else float("nan"), **p}
