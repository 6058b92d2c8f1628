"""NumPy restatement of C51 as include/cleanrl_c51.h pins it: the atoms, the network, the categorical projection, the
clamp-log loss and its gradient, Adam, and the run loop.

The projection's index arithmetic (tz, b, l, u and the coefficients of p') is Float32 in the header's order, so its bins
are the kernel's bit for bit; the pmfs, masses, loss, gradients and Adam are Float64. The run loop takes its random draws
from the same Philox streams as the kernels (philox_draw_many, pinned to the oracle's Philox in test_ddpg.py) and its env
steps and resets from the oracle's Float32 CartPole (olib.env_step_raw, olib.reset_uniforms, olib.env_reset_raw)."""
import numpy as np

from ddpg_reference import perm_index, philox_draw_many

F = np.float32
ATOMS, P = 101, 27934
D, H1, H2, O = 4, 120, 84, 2 * 101
STREAM_ACT, STREAM_BATCH = 3, 4
CRL_ENV_CARTPOLE = 0
ACT_MAX_STEPS = 16
LO, HI = 1e-5, 1.0 - 1e-5   # the clamp's bounds (the kernels compare Float32 pmfs with their Float32 roundings)


def net_offsets():
    """(name, start, end) of W1, b1, W2, b2, W3, b3 in the flat vector"""
    out, o = [], 0
    for name, n in (("W1", H1 * D), ("b1", H1), ("W2", H2 * H1), ("b2", H2), ("W3", O * H2), ("b3", O)):
        out.append((name, o, o + n))
        o += n
    return out


ARRAYS = net_offsets()
assert ARRAYS[-1][2] == P


def unpack(p):
    p = np.asarray(p, np.float64)
    a = {n: p[s:e] for n, s, e in ARRAYS}
    return a["W1"].reshape(D, H1).T, a["b1"], a["W2"].reshape(H1, H2).T, a["b2"], a["W3"].reshape(H2, O).T, a["b3"]


def pack(W1, b1, W2, b2, W3, b3):
    return np.concatenate([W1.T.ravel(), b1, W2.T.ravel(), b2, W3.T.ravel(), b3])


def atoms(v_min, v_max):
    """z_j = (float)(v_min + j ((v_max - v_min) / 100)) in Float64, rounded once"""
    return (v_min + np.arange(ATOMS, dtype=np.float64) * ((v_max - v_min) / (ATOMS - 1))).astype(F)


def forward(p, x):
    """logits [n, 2, 101] and the intermediates (x, z1, h1, z2, h2) in Float64"""
    W1, b1, W2, b2, W3, b3 = unpack(p)
    x = np.asarray(x, np.float64)
    z1 = x @ W1.T + b1; h1 = np.maximum(z1, 0)
    z2 = h1 @ W2.T + b2; h2 = np.maximum(z2, 0)
    # one product per action: equal weights give bit-equal logits (one product over all 202 outputs may round the two
    # halves differently)
    logits = np.stack([h2 @ W3[a * ATOMS:(a + 1) * ATOMS].T + b3[a * ATOMS:(a + 1) * ATOMS] for a in range(2)], axis=1)
    return logits, (x, z1, h1, z2, h2)


def softmax(l):
    e = np.exp(l - l.max(axis=-1, keepdims=True))
    return e / e.sum(axis=-1, keepdims=True)


def get_action(p, x, z):
    """pmfs [n, 2, 101], expected Q [n, 2], greedy action (first maximum) in Float64"""
    pm = softmax(forward(p, x)[0])
    q = (pm * z.astype(np.float64)).sum(axis=2)
    return pm, q, np.argmax(q, axis=1)


def project_bins(r, d, gamma, v_min, v_max):
    """the Float32 index arithmetic of the projection: b, l, u [n, 101] and the coefficients of p' for m[l] and m[u]"""
    z = atoms(v_min, v_max)
    r = np.asarray(r, F)[:, None]
    nd = F(1) - np.asarray(d, F)[:, None]
    with np.errstate(over="ignore"):
        tz = r + (F(gamma) * z) * nd
    tz = np.minimum(np.maximum(tz, F(v_min)), F(v_max))
    dz = z[1] - z[0]
    b = (tz - F(v_min)) / dz
    l = np.minimum(np.maximum(np.floor(b), F(0)), F(ATOMS - 1))
    u = np.minimum(np.maximum(np.ceil(b), F(0)), F(ATOMS - 1))
    cl = (u + (l == u).astype(F)) - b
    cu = b - l
    return b, l.astype(np.int64), u.astype(np.int64), cl, cu


def project(r, d, pn, gamma, v_min, v_max):
    """target masses [n, 101]: d_m_l = cl p' added at l for ascending j, then d_m_u = cu p' at u, as index_add_. With
    pn Float32 every operation is Float32 (CleanRL's code); with pn Float64 the masses are Float64 on Float32 bins."""
    _, l, u, cl, cu = project_bins(r, d, gamma, v_min, v_max)
    dt = pn.dtype
    m = np.zeros(pn.shape, dt)
    dml, dmu = cl.astype(dt) * pn, cu.astype(dt) * pn
    for i in range(len(pn)):
        np.add.at(m[i], l[i], dml[i])   # unbuffered, in index order
        np.add.at(m[i], u[i], dmu[i])
    return m


def loss_grad(q, tgt, s, a, r, s2, term, gamma, v_min, v_max):
    """one learning step on the rows given: (loss, gradient [27934], masses [B, 101], mean expected Q of the taken
    action, the smallest |Q_1 - Q_0| of the target net at s') in Float64"""
    z = atoms(v_min, v_max)
    B = len(a)
    pmn, qn, an = get_action(tgt, s2, z)
    pn = pmn[np.arange(B), an]
    m = project(r, term, pn, gamma, v_min, v_max)
    logits, (x, z1, h1, z2, h2) = forward(q, s)
    pm = softmax(logits)
    pa = pm[np.arange(B), a]
    loss = -(m * np.log(np.clip(pa, LO, HI))).sum(axis=1).mean()
    qv = (pa * z.astype(np.float64)).sum(axis=1).mean()
    kap = (pa >= LO) & (pa <= HI)
    mk = m * kap
    dla = (pa * mk.sum(axis=1, keepdims=True) - mk) / B
    dl = np.zeros((B, 2, ATOMS))
    dl[np.arange(B), a] = dla
    dl = dl.reshape(B, O)
    W1, b1, W2, b2, W3, b3 = unpack(q)
    dW3, db3 = dl.T @ h2, dl.sum(0)
    dz2 = (dl @ W3) * (z2 > 0)
    dW2, db2 = dz2.T @ h1, dz2.sum(0)
    dz1 = (dz2 @ W2) * (z1 > 0)
    dW1, db1 = dz1.T @ x, dz1.sum(0)
    return loss, pack(dW1, db1, dW2, db2, dW3, db3), m, qv, np.abs(qn[:, 1] - qn[:, 0]).min()


def adam(p, m, v, g, t, lr, eps, b1=0.9, b2=0.999):
    m = b1 * m + (1 - b1) * g
    v = b2 * v + (1 - b2) * g * g
    return p - lr * (m / (1 - b1 ** t)) / (np.sqrt(v / (1 - b2 ** t)) + eps), m, v


def linear_schedule(start_e, end_e, duration, t):
    return max((end_e - start_e) / duration * t + start_e, end_e)


def batch_indices(seed, learn_step, size, B):
    keys = np.concatenate([philox_draw_many(seed, [0], learn_step, STREAM_BATCH)[0],
                           philox_draw_many(seed, [0x80000000], learn_step, STREAM_BATCH)[0]])
    return perm_index(np.arange(B), size, keys)


def closed_form_counts(cfg, chunks):
    """(learn_steps, target_copies, acting launches) after run calls of `chunks` iterations: the learning iterations
    are the multiples of train_frequency from max(learning_starts // N + 1, ceil(batch_size / N)) on (none when the
    batch exceeds the ring), the copies the multiples of target_network_frequency from learning_starts // N + 1 on; an
    acting launch ends at a learning iteration, after ACT_MAX_STEPS iterations, before a step that would reuse a ring
    slot, and at the end of a call"""
    N, T = cfg.num_envs, sum(chunks)
    first = cfg.learning_starts // N + 1
    first_learn = max(first, -(-cfg.batch_size // N)) if cfg.batch_size <= cfg.buffer_size else T + 1

    def multiples(k, lo):
        return max(0, T // k - (lo - 1) // k) if lo <= T else 0
    learn, copies = multiples(cfg.train_frequency, first_learn), multiples(cfg.target_network_frequency, first)
    per_launch = min(ACT_MAX_STEPS, cfg.buffer_size // N)
    launches, it = 0, 0
    for c in chunks:
        end = it + c
        while it < end:
            nxt = -(-(max(it + 1, first_learn)) // cfg.train_frequency) * cfg.train_frequency   # next learning iteration
            it = min(end, it + per_launch, nxt)
            launches += 1
    return learn, copies, launches


class RefC51:
    """crl_c51_run restated: N CartPole envs, epsilon-greedy acting, the ring, the learning gate, the learning step with
    Float64 nets and Adam, and the target copies. `tie_tol`: where the Float64 gap between the two expected Qs of the
    online net is below it, the kernel's Float32 chains may pick either action, and the reference adopts the library's
    action from its ring (counted in `adopted`); the same gap for the target net at s' is recorded in `target_gap`."""

    def __init__(self, olib, cfg, params, tie_tol=1e-3):
        self.o, self.cfg, self.tie_tol = olib, cfg, tie_tol
        N, C = cfg.num_envs, cfg.buffer_size
        self.z = atoms(cfg.v_min, cfg.v_max)
        self.q = np.asarray(params, np.float64).copy()
        self.tgt = self.q.copy()
        self.m, self.v = np.zeros(P), np.zeros(P)
        self.b_state, self.b_next = np.zeros((C, 4), F), np.zeros((C, 4), F)
        self.b_action, self.b_reward, self.b_term = np.zeros(C, np.int32), np.zeros(C, F), np.zeros(C, np.uint8)
        self.size = self.ptr = self.it = self.learn_steps = self.target_copies = self.launches = self.adopted = 0
        self.greedy_decisions = 0
        self.target_gap = np.inf
        self.loss = self.q_values = 0.0
        self.eps = 0.0
        u = np.stack([olib.reset_uniforms(cfg.seed, n, 0) for n in range(N)])
        self.state, self.t = olib.env_reset_raw(CRL_ENV_CARTPOLE, u)
        self.resets = np.ones(N, np.int64)
        self.ep_ret, self.ep_len = np.zeros(N), np.zeros(N, np.int64)
        self.episodes, self.sum_return, self.sum_length = 0, 0.0, 0.0

    def step(self, lib_actions=None):
        cfg, N, C = self.cfg, self.cfg.num_envs, self.cfg.buffer_size
        self.it += 1
        gs = self.it * N
        self.eps = linear_schedule(cfg.start_e, cfg.end_e, cfg.epsilon_duration, float(gs))
        obs = self.state.copy()
        r = philox_draw_many(cfg.seed, np.arange(N), self.it, STREAM_ACT)
        u = (((r[:, 0] << np.uint64(32)) | r[:, 1]) >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)
        act = (r[:, 2] & np.uint64(1)).astype(np.int32)
        greedy = u >= self.eps
        slots = (self.ptr + np.arange(N)) % C
        if greedy.any():
            _, qv, ga = get_action(self.q, obs[greedy], self.z)
            near = np.abs(qv[:, 1] - qv[:, 0]) < self.tie_tol
            if near.any():
                assert lib_actions is not None, "a near-tie needs the library's ring"
                ga[near] = lib_actions[slots[greedy][near]]
                self.adopted += int(near.sum())
            act[greedy] = ga
            self.greedy_decisions += int(greedy.sum())
        self.state, self.t, rew, done = self.o.env_step_raw(CRL_ENV_CARTPOLE, self.state, self.t, act, cfg.max_episode_steps)
        self.b_state[slots], self.b_next[slots], self.b_action[slots] = obs, self.state, act
        self.b_reward[slots], self.b_term[slots] = rew, done
        self.ep_ret += rew; self.ep_len += 1
        for n in np.nonzero(done)[0]:
            self.episodes += 1; self.sum_return += self.ep_ret[n]; self.sum_length += self.ep_len[n]
            self.ep_ret[n] = 0.0; self.ep_len[n] = 0
            s, t = self.o.env_reset_raw(CRL_ENV_CARTPOLE, self.o.reset_uniforms(cfg.seed, int(n), int(self.resets[n]))[None])
            self.state[n], self.t[n] = s[0], t[0]
            self.resets[n] += 1
        self.ptr = (self.ptr + N) % C
        self.size = min(self.size + N, C)
        learn = gs > cfg.learning_starts and self.it % cfg.train_frequency == 0 and self.size >= cfg.batch_size
        if learn:
            self.learn()
        if gs > cfg.learning_starts and self.it % cfg.target_network_frequency == 0:
            self.tgt = self.q.copy()
            self.target_copies += 1
        return learn

    def learn(self):
        cfg = self.cfg
        idx = batch_indices(cfg.seed, self.learn_steps, self.size, cfg.batch_size)
        self.loss, g, _, self.q_values, gap = loss_grad(self.q, self.tgt, self.b_state[idx], self.b_action[idx],
                                                        self.b_reward[idx], self.b_next[idx], self.b_term[idx], cfg.gamma,
                                                        cfg.v_min, cfg.v_max)
        self.target_gap = min(self.target_gap, gap)
        self.learn_steps += 1
        self.q, self.m, self.v = adam(self.q, self.m, self.v, g, self.learn_steps, cfg.lr, 0.01 / cfg.batch_size)

    def run(self, iterations, lib_actions=None):
        """`iterations` steps, counting acting launches as crl_c51_run packs them; lib_actions: the library's ring of
        actions after the same iterations (read for near-ties only)"""
        self.episodes, self.sum_return, self.sum_length = 0, 0.0, 0.0
        per_launch = min(ACT_MAX_STEPS, self.cfg.buffer_size // self.cfg.num_envs)
        ns = 0
        for _ in range(iterations):
            if ns == 0:
                self.launches += 1
            ns += 1
            if self.step(lib_actions):
                self.launches += 3
                ns = 0
            elif ns == per_launch:
                ns = 0
