"""Float64 NumPy restatement of DDPG as include/cleanrl_ddpg.h pins it: the nets, both losses and their gradients,
Adam, Polyak averaging and the run loop. The run loop takes its random draws from the oracle's Philox (olib.philox; the
per-env acting draws from philox_draw_many, a NumPy Philox that tests/test_ddpg.py pins to olib.philox bit for bit) and
its env steps and resets from the oracle's Float32 Pendulum (olib.env_step_raw, olib.reset_uniforms, olib.env_reset_raw),
so it needs nothing but those stateless helpers."""
import numpy as np

H = 64
ACTOR_P, CRITIC_P = 4481, 4545
STREAM_ACT, STREAM_BATCH = 5, 6
CRL_ENV_PENDULUM = 1


def net_offsets(d_in):
    """(name, start, end) of W1, b1, W2, b2, W3, b3 in the flat vector"""
    sizes = [("W1", H * d_in), ("b1", H), ("W2", H * H), ("b2", H), ("W3", H), ("b3", 1)]
    out, o = [], 0
    for name, n in sizes:
        out.append((name, o, o + n))
        o += n
    return out


ACTOR_ARRAYS, CRITIC_ARRAYS = net_offsets(3), net_offsets(4)


def unpack(p, d_in):
    p = np.asarray(p, np.float64)
    a = {n: p[s:e] for n, s, e in net_offsets(d_in)}
    return (a["W1"].reshape(d_in, H).T, a["b1"], a["W2"].reshape(H, H).T, a["b2"], a["W3"].reshape(1, H), a["b3"])


def mlp(p, x, d_in):
    """head pre-activation [n] and the intermediates (z1, h1, z2, h2) of Dense(d_in,64,relu) -> Dense(64,64,relu) -> Dense(64,1)"""
    W1, b1, W2, b2, W3, b3 = unpack(p, d_in)
    z1 = x @ W1.T + b1; h1 = np.maximum(z1, 0)
    z2 = h1 @ W2.T + b2; h2 = np.maximum(z2, 0)
    return (h2 @ W3.T + b3)[:, 0], (z1, h1, z2, h2)


def mu(actor, obs):
    u, _ = mlp(actor, np.asarray(obs, np.float64), 3)
    return 2.0 * np.tanh(u)


def q(critic, obs, act):
    x = np.concatenate([np.asarray(obs, np.float64), np.asarray(act, np.float64)[:, None]], axis=1)
    v, _ = mlp(critic, x, 4)
    return v


def mlp_backward(p, x, cache, dout, d_in):
    """flat gradient of sum_b dout[b] * head(x_b), and the gradient with respect to the input rows"""
    W1, _, W2, _, W3, _ = unpack(p, d_in)
    z1, h1, z2, h2 = cache
    gW3 = dout @ h2; gb3 = np.array([dout.sum()])
    dz2 = np.outer(dout, W3[0]) * (z2 > 0)
    gW2 = dz2.T @ h1; gb2 = dz2.sum(0)
    dz1 = (dz2 @ W2) * (z1 > 0)
    gW1 = dz1.T @ x; gb1 = dz1.sum(0)
    g = np.concatenate([gW1.T.ravel(), gb1, gW2.T.ravel(), gb2, gW3, gb3])   # (out,in) column-major
    return g, dz1 @ W1


def critic_loss_grad(actor_tgt, critic, critic_tgt, obs, act, rew, next_obs, term, gamma):
    """mean((Q(s,a) - y)^2) with y = r + gamma (1 - d) Q'(s', mu'(s')), and its gradient with respect to the critic"""
    obs, next_obs = np.asarray(obs, np.float64), np.asarray(next_obs, np.float64)
    B = len(obs)
    y = np.asarray(rew, np.float64) + gamma * (1.0 - np.asarray(term, np.float64)) * q(critic_tgt, next_obs, mu(actor_tgt, next_obs))
    x = np.concatenate([obs, np.asarray(act, np.float64)[:, None]], axis=1)
    v, cache = mlp(critic, x, 4)
    diff = v - y
    g, _ = mlp_backward(critic, x, cache, 2.0 * diff / B, 4)
    return np.mean(diff ** 2), g


def actor_loss_grad(actor, critic, obs):
    """-mean Q(s, mu(s)) and its gradient with respect to the actor, through the critic's action input"""
    obs = np.asarray(obs, np.float64)
    B = len(obs)
    u, acache = mlp(actor, obs, 3)
    a = 2.0 * np.tanh(u)
    x = np.concatenate([obs, a[:, None]], axis=1)
    v, ccache = mlp(critic, x, 4)
    _, dx = mlp_backward(critic, x, ccache, np.full(B, -1.0 / B), 4)
    du = dx[:, 3] * 2.0 / np.cosh(u) ** 2
    g, _ = mlp_backward(actor, obs, acache, du, 3)
    return -np.mean(v), g


def adam(p, m, v, g, t, lr, b1=0.9, b2=0.999, eps=1e-8):
    """one Adam step (t = 1-based step count); returns new (p, m, v)"""
    m = b1 * m + (1 - b1) * g
    v = b2 * v + (1 - b2) * g * g
    return p - lr * (m / (1 - b1 ** t)) / (np.sqrt(v / (1 - b2 ** t)) + eps), m, v


def polyak(p, t, tau):
    return tau * p + (1.0 - tau) * t


# ---------------------------------------------------------------------------------------------------- sampling
def _feistel_round(x, k, mask):
    x = (x ^ np.uint32(k)).astype(np.uint64)
    x = (x * 0x9E3779B1) & 0xFFFFFFFF
    x ^= x >> 15
    x = (x * 0x85EBCA77) & 0xFFFFFFFF
    x ^= x >> 13
    return x & mask


def perm_index(i, size, keys):
    """perm_index of device_math.cuh: the Philox-keyed Feistel bijection on [0, size) with cycle walking"""
    bits = 1
    while (1 << bits) < size:
        bits += 1
    half = (bits + 1) // 2
    mask = (1 << half) - 1
    x = np.asarray(i, np.uint64)
    todo = np.ones(x.shape, bool)
    while True:
        l, r = x >> half, x & mask
        for k in range(6):
            l, r = r, l ^ _feistel_round(r, int(keys[k]), mask)
        nx = (l << half) | r
        x = np.where(todo, nx, x)
        todo = x >= size
        if not todo.any():
            return x.astype(np.int64)


def philox_draw(olib, seed, word, counter, stream):
    return olib.philox([word, counter & 0xFFFFFFFF, counter >> 32, stream], [seed & 0xFFFFFFFF, seed >> 32]).astype(np.uint64)


def philox_draw_many(seed, words, counter, stream):
    """philox_draw of device_math.cuh (Philox4x32-10, ctr = (word, counter lo, counter hi, stream), key = seed) for every
    entry of `words` at once: [len(words), 4] uint64, bit for bit philox_draw's. Every product of two 32-bit words fits
    in uint64, so the rounds need no wider type."""
    m32 = np.uint64(0xFFFFFFFF)
    c0 = np.asarray(words, np.uint64).ravel()
    n = len(c0)
    c1 = np.full(n, counter & 0xFFFFFFFF, np.uint64)
    c2 = np.full(n, counter >> 32, np.uint64)
    c3 = np.full(n, stream, np.uint64)
    k0, k1 = seed & 0xFFFFFFFF, seed >> 32
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ np.uint64(k0), p1 & m32, (p0 >> np.uint64(32)) ^ c3 ^ np.uint64(k1), p0 & m32
        k0, k1 = (k0 + 0x9E3779B9) & 0xFFFFFFFF, (k1 + 0xBB67AE85) & 0xFFFFFFFF
    return np.stack([c0, c1, c2, c3], axis=1)


def batch_indices(olib, seed, learn_step, size, B):
    keys = np.concatenate([philox_draw(olib, seed, 0, learn_step, STREAM_BATCH), philox_draw(olib, seed, 0x80000000, learn_step, STREAM_BATCH)])
    return perm_index(np.arange(B), size, keys)


# ---------------------------------------------------------------------------------------------------- run loop
def obs_of(state):
    th, thd = state[:, 0], state[:, 1]
    return np.stack([np.cos(th), np.sin(th), thd], axis=1).astype(np.float32)


class RefDDPG:
    """crl_ddpg_run restated: N envs, the ring, the learning gate, the critic step, every policy_frequency-th actor step
    and the Polyak update, with Float64 nets and the oracle's Float32 Pendulum"""

    def __init__(self, olib, cfg, actor, critic):
        self.o, self.cfg = olib, cfg
        N, C = cfg.num_envs, cfg.buffer_size
        self.actor = np.asarray(actor, np.float64).copy(); self.critic = np.asarray(critic, np.float64).copy()
        self.actor_tgt, self.critic_tgt = self.actor.copy(), self.critic.copy()
        self.am, self.av = np.zeros(ACTOR_P), np.zeros(ACTOR_P)
        self.cm, self.cv = np.zeros(CRITIC_P), np.zeros(CRITIC_P)
        self.b_obs, self.b_next = np.zeros((C, 3), np.float32), np.zeros((C, 3), np.float32)
        self.b_act, self.b_rew, self.b_term = np.zeros(C, np.float32), np.zeros(C, np.float32), np.zeros(C, np.uint8)
        self.size = self.ptr = self.it = self.learn_steps = self.actor_steps = 0
        self.critic_loss = self.actor_loss = 0.0
        self.episodes, self.sum_return, self.sum_length = 0, 0.0, 0.0
        u = np.stack([olib.reset_uniforms(cfg.seed, n, 0) for n in range(N)])
        self.state, self.t = olib.env_reset_raw(CRL_ENV_PENDULUM, u)
        self.resets = np.ones(N, np.int64)
        self.ep_ret, self.ep_len = np.zeros(N), np.zeros(N, np.int64)

    def _actions(self, obs):
        cfg, N = self.cfg, self.cfg.num_envs
        gs = self.it * N
        r = philox_draw_many(cfg.seed, np.arange(N), self.it, STREAM_ACT)
        if gs <= cfg.learning_starts:
            u = (r[:, 0] >> 8).astype(np.float32) * np.float32(1.0 / 16777216.0)
            return (np.float32(4.0) * u - np.float32(2.0)).astype(np.float32)
        u1 = ((r[:, 0] >> 8) + 1).astype(np.float64) / 16777216.0
        u2 = (r[:, 1] >> 8).astype(np.float64) / 16777216.0
        z = np.sqrt(-2.0 * np.log(u1)) * np.cos(2.0 * np.pi * u2)
        return np.clip(mu(self.actor, obs) + cfg.exploration_noise * 2.0 * z, -2.0, 2.0).astype(np.float32)

    def step(self):
        cfg, N, C = self.cfg, self.cfg.num_envs, self.cfg.buffer_size
        self.it += 1
        obs = obs_of(self.state)
        act = self._actions(obs)
        self.state, self.t, rew, done = self.o.env_step_raw(CRL_ENV_PENDULUM, self.state, self.t, act, cfg.max_episode_steps)
        nobs = obs_of(self.state)
        slots = (self.ptr + np.arange(N)) % C
        self.b_obs[slots], self.b_next[slots], self.b_act[slots], self.b_rew[slots], self.b_term[slots] = obs, nobs, act, rew, done
        self.ep_ret += rew; self.ep_len += 1
        for n in np.nonzero(done)[0]:
            self.episodes += 1; self.sum_return += self.ep_ret[n]; self.sum_length += self.ep_len[n]
            self.ep_ret[n] = 0.0; self.ep_len[n] = 0
            s, t = self.o.env_reset_raw(CRL_ENV_PENDULUM, self.o.reset_uniforms(cfg.seed, int(n), int(self.resets[n]))[None])
            self.state[n], self.t[n] = s[0], t[0]
            self.resets[n] += 1
        self.ptr = (self.ptr + N) % C
        self.size = min(self.size + N, C)
        if self.it * N > cfg.learning_starts and self.it % cfg.train_freq == 0 and self.size >= cfg.batch_size:
            self.learn()

    def learn(self):
        cfg = self.cfg
        idx = batch_indices(self.o, cfg.seed, self.learn_steps, self.size, cfg.batch_size)
        self.critic_loss, g = critic_loss_grad(self.actor_tgt, self.critic, self.critic_tgt, self.b_obs[idx], self.b_act[idx],
                                               self.b_rew[idx], self.b_next[idx], self.b_term[idx], cfg.gamma)
        self.learn_steps += 1
        self.critic, self.cm, self.cv = adam(self.critic, self.cm, self.cv, g, self.learn_steps, cfg.lr)
        if self.learn_steps % cfg.policy_frequency == 0:
            self.actor_loss, g = actor_loss_grad(self.actor, self.critic, self.b_obs[idx])
            self.actor_steps += 1
            self.actor, self.am, self.av = adam(self.actor, self.am, self.av, g, self.actor_steps, cfg.lr)
            self.actor_tgt = polyak(self.actor, self.actor_tgt, cfg.tau)
            self.critic_tgt = polyak(self.critic, self.critic_tgt, cfg.tau)

    def run(self, iterations):
        for _ in range(iterations):
            self.step()
