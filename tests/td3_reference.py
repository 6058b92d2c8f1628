"""Float64 NumPy restatement of TD3 as include/cleanrl_td3.h pins it, on top of tests/ddpg_reference.py: the target
smoothing (Philox stream 7), the twin-critic loss and its gradients, and the run loop (RefTD3: RefDDPG's envs, ring,
acting and batches, with TD3's learning step)."""
import numpy as np

import ddpg_reference as R

STREAM_SMOOTH = 7


def smoothing_normals(seed, learn_step, B):
    """z_b of sample b = 0..B-1 at learning step `learn_step`: Box-Muller of the first two words of
    Philox(seed, word = b, counter = learn_step, stream 7), as the acting kernel forms its noise"""
    r = R.philox_draw_many(seed, np.arange(B), learn_step, STREAM_SMOOTH)
    u1 = ((r[:, 0] >> 8) + 1).astype(np.float64) / 16777216.0
    u2 = (r[:, 1] >> 8).astype(np.float64) / 16777216.0
    return np.sqrt(-2.0 * np.log(u1)) * np.cos(2.0 * np.pi * u2)


def target_actions(actor_tgt, next_obs, z, policy_noise, noise_clip):
    """a' = clamp(mu'(s') + clamp(policy_noise z, -noise_clip, noise_clip) * 2, -2, 2)"""
    eps = np.clip(policy_noise * np.asarray(z, np.float64), -noise_clip, noise_clip) * 2.0
    return np.clip(R.mu(actor_tgt, next_obs) + eps, -2.0, 2.0)


def twin_critic_loss_grad(actor_tgt, qf1, qf2, qf1_tgt, qf2_tgt, obs, act, rew, next_obs, term, gamma, z, policy_noise,
                          noise_clip):
    """(qf1_loss, qf2_loss, qf1 gradient, qf2 gradient) of mean((qf_k(s,a) - y)^2) with
    y = r + gamma (1 - d) min(qf1'(s', a'), qf2'(s', a')) and a' from target_actions"""
    obs, next_obs = np.asarray(obs, np.float64), np.asarray(next_obs, np.float64)
    B = len(obs)
    a2 = target_actions(actor_tgt, next_obs, z, policy_noise, noise_clip)
    qn = np.minimum(R.q(qf1_tgt, next_obs, a2), R.q(qf2_tgt, next_obs, a2))
    y = np.asarray(rew, np.float64) + gamma * (1.0 - np.asarray(term, np.float64)) * qn
    x = np.concatenate([obs, np.asarray(act, np.float64)[:, None]], axis=1)
    out = []
    for qf in (qf1, qf2):
        v, cache = R.mlp(qf, x, 4)
        diff = v - y
        g, _ = R.mlp_backward(qf, x, cache, 2.0 * diff / B, 4)
        out.append((np.mean(diff ** 2), g))
    return out[0][0], out[1][0], out[0][1], out[1][1]


class RefTD3(R.RefDDPG):
    """crl_td3_run restated: RefDDPG's envs, ring, acting and batches (qf1 is RefDDPG's critic), with the twin-critic
    step, the actor step against qf1 and the Polyak update of all three targets"""

    def __init__(self, olib, cfg, actor, qf1, qf2):
        super().__init__(olib, cfg, actor, qf1)
        self.qf2 = np.asarray(qf2, np.float64).copy()
        self.qf2_tgt = self.qf2.copy()
        self.q2m, self.q2v = np.zeros(R.CRITIC_P), np.zeros(R.CRITIC_P)
        self.qf2_loss = 0.0

    def learn(self):
        cfg = self.cfg
        idx = R.batch_indices(self.o, cfg.seed, self.learn_steps, self.size, cfg.batch_size)
        z = smoothing_normals(cfg.seed, self.learn_steps, cfg.batch_size)
        self.critic_loss, self.qf2_loss, g1, g2 = twin_critic_loss_grad(
            self.actor_tgt, self.critic, self.qf2, self.critic_tgt, self.qf2_tgt, self.b_obs[idx], self.b_act[idx],
            self.b_rew[idx], self.b_next[idx], self.b_term[idx], cfg.gamma, z, cfg.policy_noise, cfg.noise_clip)
        self.learn_steps += 1
        self.critic, self.cm, self.cv = R.adam(self.critic, self.cm, self.cv, g1, self.learn_steps, cfg.lr)
        self.qf2, self.q2m, self.q2v = R.adam(self.qf2, self.q2m, self.q2v, g2, self.learn_steps, cfg.lr)
        if self.learn_steps % cfg.policy_frequency == 0:
            self.actor_loss, g = R.actor_loss_grad(self.actor, self.critic, self.b_obs[idx])
            self.actor_steps += 1
            self.actor, self.am, self.av = R.adam(self.actor, self.am, self.av, g, self.actor_steps, cfg.lr)
            self.actor_tgt = R.polyak(self.actor, self.actor_tgt, cfg.tau)
            self.critic_tgt = R.polyak(self.critic, self.critic_tgt, cfg.tau)
            self.qf2_tgt = R.polyak(self.qf2, self.qf2_tgt, cfg.tau)


def acting_launches(cfg, calls, act_max_steps=1024):
    """acting launches of crl_td3_run (and crl_ddpg_run) over run calls of `calls` iterations each, from a reset: one
    launch runs up to and including the next learning iteration, at most act_max_steps iterations, no more than
    capacity // num_envs, and never past the end of its call"""
    N, C = cfg.num_envs, cfg.buffer_size
    launches, it, size = 0, 0, 0
    for n in calls:
        end = it + n
        while it < end:
            ns, learn = 0, False
            while it < end and ns < act_max_steps and (ns + 1) * N <= C and not learn:
                it += 1; ns += 1
                size = min(size + N, C)
                learn = it * N > cfg.learning_starts and it % cfg.train_freq == 0 and size >= cfg.batch_size
            launches += 1
    return launches
