"""Float64 NumPy restatement of SAC as include/cleanrl_sac.h pins it, on top of tests/ddpg_reference.py: the three noise
draws (Philox streams 8, 9 and 10), the two-headed actor, the squashed sample and its log-prob, the critic, actor and
temperature losses with their hand-derived gradients, and the run loop (RefSAC: RefDDPG's envs, ring, warm-up and
batches, with SAC's acting and learning step)."""
import numpy as np

import ddpg_reference as R

STREAM_TARGET, STREAM_ACTOR, STREAM_ALPHA = 8, 9, 10
ACTOR_P = 4546
TARGET_ENTROPY = -1.0
HALF_LOG_2PI = 0.5 * np.log(2.0 * np.pi)


def _actor_offsets():
    out, o = [], 0
    for name, n in (("W1", 64 * 3), ("b1", 64), ("W2", 64 * 64), ("b2", 64), ("W_mean", 64), ("b_mean", 1), ("W_logstd", 64),
                    ("b_logstd", 1)):
        out.append((name, o, o + n))
        o += n
    return out


ACTOR_ARRAYS = _actor_offsets()
_OFF = {n: (s, e) for n, s, e in ACTOR_ARRAYS}


def normals(seed, counter, B, stream):
    """z_b of sample b = 0..B-1: Box-Muller of the first two words of Philox(seed, word = b, counter, stream), in Float64"""
    r = R.philox_draw_many(seed, np.arange(B), counter, stream)
    u1 = ((r[:, 0] >> 8) + 1).astype(np.float64) / 16777216.0
    u2 = (r[:, 1] >> 8).astype(np.float64) / 16777216.0
    return np.sqrt(-2.0 * np.log(u1)) * np.cos(2.0 * np.pi * u2)


def heads(actor, obs):
    """(mean, l, cache): the fc_mean and fc_logstd outputs (l before its squash) and the trunk's intermediates"""
    p = np.asarray(actor, np.float64)
    x = np.asarray(obs, np.float64)
    g = lambda n: p[_OFF[n][0]:_OFF[n][1]]
    W1, W2 = g("W1").reshape(3, 64).T, g("W2").reshape(64, 64).T
    z1 = x @ W1.T + g("b1"); h1 = np.maximum(z1, 0)
    z2 = h1 @ W2.T + g("b2"); h2 = np.maximum(z2, 0)
    return h2 @ g("W_mean") + g("b_mean")[0], h2 @ g("W_logstd") + g("b_logstd")[0], (x, z1, h1, z2, h2)


def actor_backward(actor, cache, dmean, dl):
    """flat gradient of sum_b dmean[b] mean_b + dl[b] l_b with respect to the actor"""
    p = np.asarray(actor, np.float64)
    g = lambda n: p[_OFF[n][0]:_OFF[n][1]]
    x, z1, h1, z2, h2 = cache
    W2 = g("W2").reshape(64, 64).T
    dz2 = (np.outer(dmean, g("W_mean")) + np.outer(dl, g("W_logstd"))) * (z2 > 0)
    dz1 = (dz2 @ W2) * (z1 > 0)
    return np.concatenate([(dz1.T @ x).T.ravel(), dz1.sum(0), (dz2.T @ h1).T.ravel(), dz2.sum(0), dmean @ h2, [dmean.sum()],
                           dl @ h2, [dl.sum()]])


def squash(mean, l, z):
    """dict: log_std = -5 + 3.5 (tanh(l) + 1), std, x = mean + std z, t = tanh x, s2 = 1 - t^2 (as 1/cosh^2 x),
    sq = 2 s2 + 1e-6, a = 2 t, log_pi = -z^2/2 - log_std - log(2 pi)/2 - log(sq), dls = d log_std / dl"""
    z = np.asarray(z, np.float64)
    log_std = -5.0 + 3.5 * (np.tanh(l) + 1.0)
    std = np.exp(log_std)
    x = mean + std * z
    with np.errstate(over="ignore"):
        s2 = 1.0 / np.cosh(x) ** 2
        dls = 3.5 / np.cosh(l) ** 2
    sq = 2.0 * s2 + 1e-6
    return dict(log_std=log_std, std=std, x=x, t=np.tanh(x), s2=s2, sq=sq, a=2.0 * np.tanh(x), z=z, dls=dls,
                log_pi=-0.5 * z * z - log_std - HALF_LOG_2PI - np.log(sq))


def sample(actor, obs, z):
    """(a, log_pi) of the current actor at obs with the noise z"""
    mean, l, _ = heads(actor, obs)
    s = squash(mean, l, z)
    return s["a"], s["log_pi"]


def critic_loss_grad(actor, qf1, qf2, qf1_tgt, qf2_tgt, obs, act, rew, next_obs, term, gamma, alpha, z):
    """(qf1_loss, qf2_loss, qf1 gradient, qf2 gradient) of mean((qf_k(s,a) - y)^2) with
    y = r + gamma (1 - d) (min(qf1'(s', a'), qf2'(s', a')) - alpha log_pi') and a', log_pi' from the actor at s'"""
    obs, next_obs = np.asarray(obs, np.float64), np.asarray(next_obs, np.float64)
    B = len(obs)
    a2, lp2 = sample(actor, next_obs, z)
    qn = np.minimum(R.q(qf1_tgt, next_obs, a2), R.q(qf2_tgt, next_obs, a2)) - alpha * lp2
    y = np.asarray(rew, np.float64) + gamma * (1.0 - np.asarray(term, np.float64)) * qn
    x = np.concatenate([obs, np.asarray(act, np.float64)[:, None]], axis=1)
    out = []
    for qf in (qf1, qf2):
        v, cache = R.mlp(qf, x, 4)
        diff = v - y
        g, _ = R.mlp_backward(qf, x, cache, 2.0 * diff / B, 4)
        out.append((np.mean(diff ** 2), g))
    return out[0][0], out[1][0], out[0][1], out[1][1]


def actor_loss_grad(actor, qf1, qf2, obs, alpha, z):
    """(actor_loss, gradient, mean log_pi) of mean(alpha log_pi - min(qf1(s, a), qf2(s, a))). d min/da is the smaller
    critic's dQ/da, and half of each on a tie (torch.minimum's backward)"""
    obs = np.asarray(obs, np.float64)
    B = len(obs)
    mean, l, cache = heads(actor, obs)
    s = squash(mean, l, z)
    x = np.concatenate([obs, s["a"][:, None]], axis=1)
    qs, dq = [], []
    for qf in (qf1, qf2):
        v, cc = R.mlp(qf, x, 4)
        _, dx = R.mlp_backward(qf, x, cc, np.ones(B), 4)
        qs.append(v); dq.append(dx[:, 3])
    c1 = np.where(qs[0] < qs[1], 1.0, np.where(qs[1] < qs[0], 0.0, 0.5))
    dqda = c1 * dq[0] + (1.0 - c1) * dq[1]
    gx = alpha * 4.0 * s["t"] * s["s2"] / s["sq"] - dqda * 2.0 * s["s2"]   # d(alpha log_pi - min Q)/dx
    dmean = gx / B
    dl = (gx * s["std"] * s["z"] - alpha) * s["dls"] / B
    loss = np.mean(alpha * s["log_pi"] - np.minimum(qs[0], qs[1]))
    return loss, actor_backward(actor, cache, dmean, dl), np.mean(s["log_pi"])


def alpha_loss(log_alpha, log_pi):
    """mean(-exp(log_alpha) (log_pi + target_entropy)), which is also its derivative with respect to log_alpha"""
    return -np.exp(log_alpha) * (np.mean(log_pi) + TARGET_ENTROPY)


class RefSAC(R.RefDDPG):
    """crl_sac_run restated: RefDDPG's envs, ring, warm-up and batches (qf1 is RefDDPG's critic), SAC's acting, the
    critic step, policy_frequency actor (and temperature) iterations on every policy_frequency-th learning step and the
    Polyak update of both critics' targets on every target_network_frequency-th"""

    def __init__(self, olib, cfg, actor, qf1, qf2):
        super().__init__(olib, cfg, np.zeros(R.ACTOR_P), qf1)
        self.actor = np.asarray(actor, np.float64).copy()
        self.actor_tgt = None
        self.am, self.av = np.zeros(ACTOR_P), np.zeros(ACTOR_P)
        self.qf2 = np.asarray(qf2, np.float64).copy()
        self.qf2_tgt = self.qf2.copy()
        self.q2m, self.q2v = np.zeros(R.CRITIC_P), np.zeros(R.CRITIC_P)
        self.log_alpha, self.la_m, self.la_v = 0.0, 0.0, 0.0
        self.alpha = 1.0 if cfg.autotune else cfg.alpha
        self.qf2_loss = self.alpha_loss = 0.0

    def _actions(self, obs):
        cfg, N = self.cfg, self.cfg.num_envs
        if self.it * N <= cfg.learning_starts:
            return super()._actions(obs)                       # the uniform warm-up draw
        r = R.philox_draw_many(cfg.seed, np.arange(N), self.it, R.STREAM_ACT)
        u1 = ((r[:, 0] >> 8) + 1).astype(np.float64) / 16777216.0
        u2 = (r[:, 1] >> 8).astype(np.float64) / 16777216.0
        z = np.sqrt(-2.0 * np.log(u1)) * np.cos(2.0 * np.pi * u2)
        mean, l, _ = heads(self.actor, obs)
        return squash(mean, l, z)["a"].astype(np.float32)

    def learn(self):
        cfg, B = self.cfg, self.cfg.batch_size
        idx = R.batch_indices(self.o, cfg.seed, self.learn_steps, self.size, B)
        obs = self.b_obs[idx]
        z = normals(cfg.seed, self.learn_steps, B, STREAM_TARGET)
        self.critic_loss, self.qf2_loss, g1, g2 = critic_loss_grad(
            self.actor, self.critic, self.qf2, self.critic_tgt, self.qf2_tgt, obs, self.b_act[idx], self.b_rew[idx],
            self.b_next[idx], self.b_term[idx], cfg.gamma, self.alpha, z)
        self.learn_steps += 1
        self.critic, self.cm, self.cv = R.adam(self.critic, self.cm, self.cv, g1, self.learn_steps, cfg.q_lr)
        self.qf2, self.q2m, self.q2v = R.adam(self.qf2, self.q2m, self.q2v, g2, self.learn_steps, cfg.q_lr)
        if self.learn_steps % cfg.policy_frequency == 0:
            for _ in range(cfg.policy_frequency):
                u = self.actor_steps
                self.actor_loss, g, _ = actor_loss_grad(self.actor, self.critic, self.qf2, obs, self.alpha,
                                                        normals(cfg.seed, u, B, STREAM_ACTOR))
                self.actor_steps += 1
                self.actor, self.am, self.av = R.adam(self.actor, self.am, self.av, g, self.actor_steps, cfg.policy_lr)
                if cfg.autotune:
                    _, lp = sample(self.actor, obs, normals(cfg.seed, u, B, STREAM_ALPHA))
                    self.alpha_loss = alpha_loss(self.log_alpha, lp)
                    self.log_alpha, self.la_m, self.la_v = R.adam(self.log_alpha, self.la_m, self.la_v, self.alpha_loss,
                                                                  self.actor_steps, cfg.q_lr)
                    self.alpha = np.exp(self.log_alpha)
        if self.learn_steps % cfg.target_network_frequency == 0:
            self.critic_tgt = R.polyak(self.critic, self.critic_tgt, cfg.tau)
            self.qf2_tgt = R.polyak(self.qf2, self.qf2_tgt, cfg.tau)


def closed_form_counts(cfg, iters):
    """(learn_steps, actor_steps, target updates) after `iters` iterations from a reset"""
    learn = 0
    for it in range(1, iters + 1):
        size = min(it * cfg.num_envs, cfg.buffer_size)
        learn += it * cfg.num_envs > cfg.learning_starts and it % cfg.train_freq == 0 and size >= cfg.batch_size
    return learn, cfg.policy_frequency * (learn // cfg.policy_frequency), learn // cfg.target_network_frequency


def kernel_launches(cfg, acting, learn, actor, targets):
    """include/cleanrl_sac.h's closed form: acting launches + 2 per learning step + (2 + 2 autotune) per actor iteration
    + 1 per target update"""
    return acting + 2 * learn + (2 + 2 * int(cfg.autotune)) * actor + targets
