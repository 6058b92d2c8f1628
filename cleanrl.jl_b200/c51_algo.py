"""c51(config) — vectorised C51 on CartPole over the crl_c51_* entry points (include/cleanrl_c51.h).

The reference has no C51; this is an extension next to DQN. Its semantics are pinned to the definition in
include/cleanrl_c51.h: CleanRL-Python's c51.py on the library's CartPole, with DQN's env, ring, epsilon-greedy acting and
batch sampling. `C51Config` keeps CleanRL's field names and defaults and adds `num_envs`, `seed`, `max_steps`,
`log_frequency` and `run_name`. `num_envs = 1` is CleanRL's schedule exactly."""
import ctypes as C
import dataclasses
import datetime
import time

import numpy as np

from . import _abi
from . import _lib as L
from . import logger as Logger


@dataclasses.dataclass
class C51Config:
    run_name: str = dataclasses.field(default_factory=lambda: datetime.datetime.now().strftime("%y-%m-%d|%H:%M:%S"))
    log_frequency: int = 1000           # global steps between log records
    total_timesteps: int = 500_000
    learning_rate: float = 2.5e-4
    n_atoms: int = 101                  # fixed: the kernels are specialised for 101 atoms
    v_min: float = -100.0
    v_max: float = 100.0
    buffer_size: int = 10_000
    gamma: float = 0.99
    target_network_frequency: int = 500
    batch_size: int = 128               # at most 128
    start_e: float = 1.0
    end_e: float = 0.05
    exploration_fraction: float = 0.5
    learning_starts: int = 10_000
    train_frequency: int = 10
    # ---- not in CleanRL
    num_envs: int = 1
    seed: int = 1
    max_steps: int = 500                # CartPole-v1's episode limit


def init_c51_params(seed=0):
    """QNetwork of c51.py: Linear(4,120) -> ReLU -> Linear(120,84) -> ReLU -> Linear(84, 2 * 101) with torch nn.Linear's
    default init, U(-1/sqrt(fan_in), 1/sqrt(fan_in)) for weights and biases, flattened W1, b1, W2, b2, W3, b3 with each
    W (out,in) column-major."""
    rng = np.random.default_rng(seed)
    out = []
    for fan_in, fan_out in ((4, 120), (120, 84), (84, 2 * _abi.CRL_C51_ATOMS)):
        lim = 1.0 / np.sqrt(fan_in)
        out.append(rng.uniform(-lim, lim, size=(fan_out, fan_in)).astype(np.float32).ravel(order="F"))
        out.append(rng.uniform(-lim, lim, size=fan_out).astype(np.float32))
    p = np.concatenate(out)
    assert p.size == _abi.CRL_C51_PARAMS
    return p


class C51Handle:
    """object wrapper over crl_c51_ctx"""

    def __init__(self, cfg):
        self.lib = L.load()
        self.cfg = cfg
        h = C.c_void_p()
        L.check(self.lib.crl_c51_create(C.byref(cfg), C.byref(h)))
        self.h = h

    def close(self):
        if self.h:
            L.check(self.lib.crl_c51_destroy(self.h))
            self.h = None

    def set_params(self, p):
        p = np.ascontiguousarray(p, np.float32)
        L.check(self.lib.crl_c51_set_params(self.h, L.ptr(p), p.size))

    def get_params(self):
        q = np.zeros(_abi.CRL_C51_PARAMS, np.float32)
        t = np.zeros(_abi.CRL_C51_PARAMS, np.float32)
        L.check(self.lib.crl_c51_get_params(self.h, L.ptr(q), L.ptr(t), q.size))
        return q, t

    def get_adam_state(self):
        m = np.zeros(_abi.CRL_C51_PARAMS, np.float32)
        v = np.zeros(_abi.CRL_C51_PARAMS, np.float32)
        bp = np.zeros(2, np.float64)
        L.check(self.lib.crl_c51_get_adam_state(self.h, L.ptr(m), L.ptr(v), L.ptr(bp)))
        return m, v, bp

    def reset(self):
        L.check(self.lib.crl_c51_reset(self.h))

    def run(self, iterations):
        st = _abi.crl_c51_stats()
        L.check(self.lib.crl_c51_run(self.h, int(iterations), C.byref(st)))
        return st

    def read_buffer(self):
        cap = self.cfg.buffer_size
        out = {"state": np.zeros((cap, 4), np.float32), "action": np.zeros(cap, np.int32), "reward": np.zeros(cap, np.float32),
               "next_state": np.zeros((cap, 4), np.float32), "terminal": np.zeros(cap, np.uint8)}
        size, ptr = C.c_int32(), C.c_int32()
        L.check(self.lib.crl_c51_read_buffer(self.h, L.ptr(out["state"]), L.ptr(out["action"]), L.ptr(out["reward"]),
                                             L.ptr(out["next_state"]), L.ptr(out["terminal"]), C.byref(size), C.byref(ptr)))
        out["size"], out["ptr"] = size.value, ptr.value
        return out


def make_crl_c51_config(config, device=0):
    if config.n_atoms != _abi.CRL_C51_ATOMS:
        raise ValueError("n_atoms must be %d: the kernels are specialised for it" % _abi.CRL_C51_ATOMS)
    return _abi.make_c51_config(num_envs=config.num_envs, buffer_size=config.buffer_size,
                                learning_starts=config.learning_starts, batch_size=config.batch_size,
                                train_frequency=config.train_frequency,
                                target_network_frequency=config.target_network_frequency, max_episode_steps=config.max_steps,
                                device=device, lr=config.learning_rate, gamma=config.gamma, start_e=config.start_e,
                                end_e=config.end_e, epsilon_duration=config.exploration_fraction * config.total_timesteps,
                                v_min=config.v_min, v_max=config.v_max, seed=config.seed)


def c51(config=None, logger=None, params=None, device=0):
    """Runs `total_timesteps` env steps and returns a summary dict. Logs "Episode Statistics" (episode_return,
    episode_length, global_step, epsilon, steps_per_sec) aggregated over the episodes that ended since the last record,
    and "Training Statistics" (loss, q_values: CleanRL's losses/loss and losses/q_values) every `log_frequency` steps."""
    config = config or C51Config()
    cfg = make_crl_c51_config(config, device)
    own_logger = logger is None
    if logger is None:
        logger = Logger.make_logger("c51|%s" % config.run_name, to_terminal=False)
    h = C51Handle(cfg)
    h.set_params(init_c51_params(config.seed) if params is None else params)
    h.reset()
    n_iter = config.total_timesteps // config.num_envs
    chunk = max(1, config.log_frequency // config.num_envs)
    start = time.time()
    done_iter, episodes, last = 0, 0, None
    returns = []
    while done_iter < n_iter:
        k = min(chunk, n_iter - done_iter)
        last = h.run(k)
        done_iter += k
        global_step = done_iter * config.num_envs
        if last.episodes > 0:
            episodes += last.episodes
            returns.append(last.sum_return / last.episodes)
            logger.info("Episode Statistics", episode_return=last.sum_return / last.episodes,
                        episode_length=last.sum_length / last.episodes, global_step=global_step, epsilon=last.epsilon,
                        steps_per_sec=int(global_step / max(time.time() - start, 1e-9)))
        if last.learn_steps > 0:
            logger.info("Training Statistics", loss=last.loss, q_values=last.q_values)
    wall = time.time() - start
    q, tgt = h.get_params()
    h.close()
    if own_logger:
        logger.close()
    return {"global_step": n_iter * config.num_envs, "episodes": episodes, "learn_steps": int(last.learn_steps) if last else 0,
            "target_copies": int(last.target_copies) if last else 0,
            "loss": float(last.loss) if last else float("nan"), "q_values": float(last.q_values) if last else float("nan"),
            "steps_per_sec": n_iter * config.num_envs / max(wall, 1e-9), "params": q, "target_params": tgt,
            "last_mean_return": (last.sum_return / last.episodes) if last and last.episodes else float("nan"),
            "recent_returns": returns[-10:]}
