"""DDPG on the GPU (include/cleanrl_ddpg.h) against the float64 reference of tests/ddpg_reference.py.

* crl_ddpg_forward_raw (the acting kernel's actor forward pass and the critic with the same tiling) at every 32-sample
  CTA boundary, with large observations and zero rows.
* crl_ddpg_critic_loss_raw / crl_ddpg_actor_loss_raw (the learning step's forward and update kernels, gradient out) per
  parameter array at every 16-sample CTA boundary of the batch and at edge batches.
* crl_ddpg_run against the reference's run loop on shared Philox streams, the closed-form step counts, determinism, a
  learning run of ddpg() and the CLI.
Run with `pytest -m gpu` on a B200."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import ddpg_reference as R
from test_ddpg import rand_nets

pytestmark = pytest.mark.gpu
F = np.float32
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def gpu_forward(crl, torch, actor, critic, obs, act):
    n = len(obs)
    mu = torch.full((n,), float("nan"), dtype=torch.float32, device="cuda")
    q = torch.full((n,), float("nan"), dtype=torch.float32, device="cuda")
    t = [dev(torch, x) for x in (actor, critic, obs, act)]
    crl.check(crl.load().crl_ddpg_forward_raw(*[crl.ptr(x) for x in t], crl.ptr(mu), crl.ptr(q), n, None))
    torch.cuda.synchronize()
    return mu.cpu().numpy(), q.cpu().numpy()


def gpu_critic(crl, torch, at, c, ct, obs, act, rew, nobs, term, gamma, B=None):
    B = len(act) if B is None else B
    g = torch.full((R.CRITIC_P,), float("nan"), dtype=torch.float32, device="cuda")
    loss = torch.full((1,), float("nan"), dtype=torch.float64, device="cuda")
    t = [dev(torch, x) for x in (at, c, ct, obs, act, rew, nobs, term)]
    crl.check(crl.load().crl_ddpg_critic_loss_raw(crl.ptr(t[0]), crl.ptr(t[1]), crl.ptr(t[2]), B, *[crl.ptr(x) for x in t[3:]],
                                                  gamma, crl.ptr(g), crl.ptr(loss), None))
    torch.cuda.synchronize()
    return g.cpu().numpy(), float(loss.cpu().numpy()[0])


def gpu_actor(crl, torch, a, c, obs, B=None):
    B = len(obs) if B is None else B
    g = torch.full((R.ACTOR_P,), float("nan"), dtype=torch.float32, device="cuda")
    loss = torch.full((1,), float("nan"), dtype=torch.float64, device="cuda")
    t = [dev(torch, x) for x in (a, c, obs)]
    crl.check(crl.load().crl_ddpg_actor_loss_raw(crl.ptr(t[0]), crl.ptr(t[1]), B, crl.ptr(t[2]), crl.ptr(g), crl.ptr(loss), None))
    torch.cuda.synchronize()
    return g.cpu().numpy(), float(loss.cpu().numpy()[0])


def assert_grad_close(g, ref, arrays, what=""):
    """per parameter array: |g - ref| <= 1e-4 |ref| + 2e-6 max|ref of that array| (the suite's gradient convention)"""
    for name, s, e in arrays:
        np.testing.assert_allclose(g[s:e], ref[s:e], rtol=1e-4, atol=2e-6 * np.abs(ref[s:e]).max(), err_msg=what + name)


# ------------------------------------------------------------------ forward
@pytest.mark.parametrize("n", [1, 31, 32, 33, 4097, 100_003])
def test_ddpg_forward_raw_matches_float64(crl, torch_cuda, n):
    """mu and Q at rtol 1e-5 with an atol of 1e-6 of the summed |summands| of the head"""
    rng = np.random.default_rng(n)
    a, c = rand_nets(n)
    obs = rng.uniform(-10, 10, (n, 3)).astype(F)
    act = rng.uniform(-2, 2, n).astype(F)
    obs[::7] = 0.0
    act[::7] = 0.0
    mu, q = gpu_forward(crl, torch_cuda, a, c, obs, act)
    ua, (_, _, _, h2a) = R.mlp(a, obs.astype(np.float64), 3)
    x = np.concatenate([obs, act[:, None]], 1).astype(np.float64)
    qr, (_, _, _, h2c) = R.mlp(c, x, 4)
    mag_a = np.abs(h2a) @ np.abs(a[R.ACTOR_ARRAYS[4][1]:R.ACTOR_ARRAYS[4][2]].astype(np.float64)) + abs(float(a[-1]))
    mag_c = np.abs(h2c) @ np.abs(c[R.CRITIC_ARRAYS[4][1]:R.CRITIC_ARRAYS[4][2]].astype(np.float64)) + abs(float(c[-1]))
    # d(2 tanh u) <= 2 du: the head's atol carries over to mu
    assert np.all(np.abs(mu - 2 * np.tanh(ua)) <= 1e-5 * np.abs(2 * np.tanh(ua)) + 2e-6 * mag_a + 1e-7)
    assert np.all(np.abs(q - qr) <= 1e-5 * np.abs(qr) + 1e-6 * mag_c)


def test_ddpg_forward_raw_zero_and_saturated_heads(crl, torch_cuda):
    rng = np.random.default_rng(5)
    a, c = rand_nets(5)
    obs = rng.uniform(-3, 3, (100, 3)).astype(F)
    act = rng.uniform(-2, 2, 100).astype(F)
    z = a.copy()
    z[R.ACTOR_ARRAYS[4][1]:] = 0.0                  # W3 and b3 of the actor
    mu, _ = gpu_forward(crl, torch_cuda, z, c, obs, act)
    assert np.all(mu == 0.0)
    for sign in (1.0, -1.0):
        s = z.copy()
        s[-1] = sign * 100.0                         # b3: tanh(+-100) = +-1
        mu, _ = gpu_forward(crl, torch_cuda, s, c, obs, act)
        assert np.all(mu == sign * 2.0)


# ------------------------------------------------------------------ loss and gradient
KINDS = ["mixed", "terminal", "open", "gamma0", "relu0"]
BATCHES = [1, 2, 15, 16, 17, 31, 32, 33, 64, 100, 128, 200, 255, 256]


def edge_batch(kind, B, seed):
    """(actor, critic, actor_tgt, critic_tgt, obs, act, rew, next_obs, term, gamma, zero_actor, zero_critic); the targets
    always differ from the online nets. Rewards are -1.5, 1 or 2 so that no TD error is close to 0.
      mixed     random batch, 20 % terminal, gamma 0.99
      terminal  every sample terminal (the targets drop out), gamma 0.99
      open      no sample terminal, gamma 1
      gamma0    no sample terminal, gamma 0
      relu0     every obs row and action 0 and every other first-layer bias 0: those pre-activations are exactly 0 and
                relu'(0) = 0, so the gradients of their W1 rows, b1 entries and W2 columns are exactly 0"""
    rng = np.random.default_rng(seed)
    a, c = rand_nets(seed)
    at, ct = rand_nets(seed + 1000)
    obs = rng.uniform(-1, 1, (B, 3)).astype(F); nobs = rng.uniform(-1, 1, (B, 3)).astype(F)
    act = rng.uniform(-2, 2, B).astype(F)
    rew = rng.choice(np.array([-1.5, 1.0, 2.0], F), B)
    term = (rng.random(B) < 0.2).astype(np.uint8)
    gamma = 0.99
    za, zc = np.zeros(0, int), np.zeros(0, int)
    if kind == "terminal":
        term[:] = 1
    elif kind == "open":
        term[:] = 0; gamma = 1.0
    elif kind == "gamma0":
        term[:] = 0; gamma = 0.0
    elif kind == "relu0":
        obs[:] = 0.0; act[:] = 0.0
        dead = np.arange(0, 64, 2)
        for p, arrays in ((a, R.ACTOR_ARRAYS), (c, R.CRITIC_ARRAYS)):
            p[arrays[1][1] + dead] = 0.0
        idx = []
        for arrays, d_in, out in ((R.ACTOR_ARRAYS, 3, "a"), (R.CRITIC_ARRAYS, 4, "c")):
            w1, b1, w2 = arrays[0][1], arrays[1][1], arrays[2][1]
            z = [w1 + j + 64 * k for j in dead for k in range(d_in)] + [b1 + j for j in dead] + [w2 + i + 64 * j for j in dead for i in range(64)]
            idx.append(np.array(z))
        za, zc = idx
    return a, c, at, ct, obs, act, rew, nobs, term, gamma, za, zc


@pytest.mark.parametrize("B", BATCHES)
@pytest.mark.parametrize("kind", KINDS)
def test_ddpg_critic_loss_raw_matches_float64(crl, torch_cuda, kind, B):
    a, c, at, ct, obs, act, rew, nobs, term, gamma, _, zc = edge_batch(kind, B, 11 * B + KINDS.index(kind))
    g, loss = gpu_critic(crl, torch_cuda, at, c, ct, obs, act, rew, nobs, term, gamma)
    lr, gr = R.critic_loss_grad(at, c, ct, obs, act, rew, nobs, term, gamma)
    np.testing.assert_allclose(loss, lr, rtol=1e-6)
    assert_grad_close(g, gr, R.CRITIC_ARRAYS, "critic %s B=%d " % (kind, B))
    if len(zc):
        assert np.all(g[zc] == 0.0)


@pytest.mark.parametrize("B", BATCHES)
@pytest.mark.parametrize("kind", ["mixed", "relu0"])
def test_ddpg_actor_loss_raw_matches_float64(crl, torch_cuda, kind, B):
    a, c, _, _, obs, _, _, _, _, _, za, _ = edge_batch(kind, B, 13 * B + 7 + KINDS.index(kind))
    g, loss = gpu_actor(crl, torch_cuda, a, c, obs)
    lr, gr = R.actor_loss_grad(a, c, obs)
    # -mean Q may cancel: the atol is 1e-6 of mean |Q|
    np.testing.assert_allclose(loss, lr, rtol=1e-6, atol=1e-6 * np.mean(np.abs(R.q(c, obs, R.mu(a, obs)))))
    assert_grad_close(g, gr, R.ACTOR_ARRAYS, "actor %s B=%d " % (kind, B))
    if len(za):
        assert np.all(g[za] == 0.0)


@pytest.mark.parametrize("B", [1, 17, 100, 255])
def test_ddpg_loss_raw_reads_nothing_past_row_B(crl, torch_cuda, B):
    a, c, at, ct, obs, act, rew, nobs, term, gamma, _, _ = edge_batch("mixed", B, B)
    g0, l0 = gpu_critic(crl, torch_cuda, at, c, ct, obs, act, rew, nobs, term, gamma)
    ga0, la0 = gpu_actor(crl, torch_cuda, a, c, obs)
    pad = lambda x, v: np.concatenate([x, np.full((7,) + x.shape[1:], v, x.dtype)])
    g1, l1 = gpu_critic(crl, torch_cuda, at, c, ct, pad(obs, np.nan), pad(act, np.nan), pad(rew, np.nan), pad(nobs, np.nan),
                        pad(term, 1), gamma, B=B)
    ga1, la1 = gpu_actor(crl, torch_cuda, a, c, pad(obs, np.nan), B=B)
    assert np.array_equal(g0, g1) and l0 == l1 and np.array_equal(ga0, ga1) and la0 == la1


# ------------------------------------------------------------------ run loop
RUNS = {   # name: (config overrides, iterations)
    "warmup_only": (dict(num_envs=16, buffer_size=256, learning_starts=10 ** 6), 20),
    "learn_every_iteration": (dict(num_envs=4, buffer_size=512, learning_starts=64, batch_size=32), 60),
    "train_freq_3": (dict(num_envs=4, buffer_size=512, learning_starts=64, batch_size=32, train_freq=3), 90),
    "policy_frequency_1": (dict(num_envs=4, buffer_size=512, learning_starts=64, batch_size=32, policy_frequency=1), 50),
    "policy_frequency_3": (dict(num_envs=4, buffer_size=512, learning_starts=64, batch_size=32, policy_frequency=3), 60),
    "truncated_at_10": (dict(num_envs=8, buffer_size=512, learning_starts=64, batch_size=32, max_episode_steps=10), 50),
    "ring_below_2N": (dict(num_envs=8, buffer_size=12, learning_starts=16, batch_size=8), 40),
    "ring_equal_N": (dict(num_envs=8, buffer_size=8, learning_starts=16, batch_size=8), 40),
    "learning_starts_below_batch": (dict(num_envs=2, buffer_size=256, learning_starts=4, batch_size=32), 60),
}


def closed_form_counts(cfg, iters):
    learn = 0
    for it in range(1, iters + 1):
        size = min(it * cfg.num_envs, cfg.buffer_size)
        learn += it * cfg.num_envs > cfg.learning_starts and it % cfg.train_freq == 0 and size >= cfg.batch_size
    return learn, learn // cfg.policy_frequency


def assert_run_close(got, ref, arrays, lr, steps, what):
    """rtol 1e-4 with an atol of 1e-6 max|ref| per array. Float32 and Float64 sums can give a gradient that cancels to
    within rounding opposite signs, and Adam's first steps move a parameter by about lr in the direction of that sign, so
    at most 0.1 % of an array (and at least 1 element) may instead differ by at most 2 lr per step taken"""
    for name, s, e in arrays:
        d = np.abs(got[s:e] - ref[s:e])
        tol = 1e-4 * np.abs(ref[s:e]) + 1e-6 * np.abs(ref[s:e]).max()
        bad = d > tol
        assert bad.sum() <= max(1, (e - s) // 1000) and np.all(d[bad] <= 2 * lr * steps), \
            "%s%s: %d elements off, worst %g" % (what, name, bad.sum(), d.max())


@pytest.mark.parametrize("name", list(RUNS))
def test_ddpg_run_loop_matches_the_reference(crl, olib, abi, torch_cuda, name):
    from cleanrl_jl_b200.ddpg_algo import DDPGHandle
    kw, iters = RUNS[name]
    cfg = abi.make_ddpg_config(**{**dict(exploration_noise=0.1, lr=1e-3, tau=0.05, seed=3), **kw})
    a, c = rand_nets(17)
    h = DDPGHandle(cfg)
    h.set_params(a, c)
    h.reset()
    ref = R.RefDDPG(olib, cfg, a, c)
    learn, actor = closed_form_counts(cfg, iters)
    first_actor_it = None
    for it in range(1, iters + 1):
        if first_actor_it is None and closed_form_counts(cfg, it)[1] > 0:
            first_actor_it = it
    try:
        if first_actor_it is not None and first_actor_it > 1:   # targets are the initial copies until the first actor step
            st = h.run(first_actor_it - 1)
            p = h.get_params()
            assert np.array_equal(p["actor_target"], a) and np.array_equal(p["critic_target"], c)
            ref.run(first_actor_it - 1)
            h.run(iters - first_actor_it + 1)
            ref.run(iters - first_actor_it + 1)
        else:
            h.run(iters)
            ref.run(iters)
        st = h.run(0)
        assert (st.learn_steps, st.actor_steps, st.iterations) == (learn, actor, iters)
        assert (ref.learn_steps, ref.actor_steps) == (learn, actor)
        buf = h.read_buffer()
        assert (buf["size"], buf["ptr"]) == (ref.size, ref.ptr)
        ring_rtol = 1e-5 if learn == 0 else 1e-4
        for k, r in (("obs", ref.b_obs), ("next_obs", ref.b_next), ("action", ref.b_act), ("reward", ref.b_rew)):
            np.testing.assert_allclose(buf[k], r, rtol=ring_rtol, atol=ring_rtol * 0.1, err_msg=k)
        np.testing.assert_array_equal(buf["terminal"], ref.b_term)
        p, m = h.get_params(), h.get_adam_state()
        for key, arrays, steps in (("critic", R.CRITIC_ARRAYS, learn), ("critic_target", R.CRITIC_ARRAYS, learn),
                                   ("actor", R.ACTOR_ARRAYS, actor), ("actor_target", R.ACTOR_ARRAYS, actor)):
            assert_run_close(p[key], getattr(ref, key.replace("_target", "_tgt")), arrays, cfg.lr, steps, key + " ")
        # Adam's moments: a gradient element that cancels to near 0 has a large relative error in Float32 (and may flip
        # sign), so up to 0.1 % of an array may be off; the rest agree at rtol 1e-3
        for key, r, arrays in (("critic_m", ref.cm, R.CRITIC_ARRAYS), ("actor_m", ref.am, R.ACTOR_ARRAYS),
                               ("critic_v", ref.cv, R.CRITIC_ARRAYS), ("actor_v", ref.av, R.ACTOR_ARRAYS)):
            for nm, s, e in arrays:
                d = np.abs(m[key][s:e] - r[s:e])
                bad = d > 1e-3 * np.abs(r[s:e]) + 1e-6 * np.abs(r[s:e]).max()
                assert bad.sum() <= max(1, (e - s) // 1000), "%s%s: %d elements off" % (key, nm, bad.sum())
        # the powers the next step of each Adam will use: beta^(steps + 1)
        np.testing.assert_allclose(m["beta_pow"], [0.9 ** (actor + 1), 0.999 ** (actor + 1), 0.9 ** (learn + 1), 0.999 ** (learn + 1)],
                                   rtol=1e-12)
        if learn:
            np.testing.assert_allclose(st.critic_loss, ref.critic_loss, rtol=1e-4)
        if actor:
            np.testing.assert_allclose(st.actor_loss, ref.actor_loss, rtol=1e-4)
        if name == "truncated_at_10":
            assert ref.b_term.sum() > 0 and np.all(ref.episodes >= cfg.num_envs * (iters // 10))
    finally:
        h.close()


def test_ddpg_run_is_deterministic(crl, abi, torch_cuda):
    from cleanrl_jl_b200.ddpg_algo import DDPGHandle
    cfg = abi.make_ddpg_config(num_envs=300, buffer_size=20_000, learning_starts=1000, batch_size=256, seed=9)
    a, c = rand_nets(2)
    out = []
    for _ in range(2):
        h = DDPGHandle(cfg)
        h.set_params(a, c)
        h.reset()
        st = h.run(40)
        out.append((h.get_params(), st.critic_loss, st.actor_loss))
        h.close()
    for k in out[0][0]:
        assert np.array_equal(out[0][0][k], out[1][0][k]), k
    assert out[0][1:] == out[1][1:]


# ------------------------------------------------------------------ learning and CLI
def test_ddpg_learns_pendulum(torch_cuda, tmp_path):
    """CleanRL's settings with one env and learning from step 5,000: mean episode return over the last 5,000 steps
    against the first 5,000 (uniform random torques). On one B200 (1000 W, seed 1) this run went from -1248.2 to -184.1;
    the thresholds below leave a wide margin under that."""
    from cleanrl_jl_b200 import DDPGConfig, ddpg
    from cleanrl_jl_b200 import logger as Logger
    lg = Logger.make_logger("ddpg", to_terminal=False, to_tensorboard=False, to_json=True, log_dir=str(tmp_path))
    cfg = DDPGConfig(total_timesteps=LEARN_STEPS, learning_starts=5_000, buffer_size=LEARN_STEPS, log_frequency=1000, seed=1)
    try:
        res = ddpg(cfg, logger=lg)
    finally:
        lg.close()
    recs = [json.loads(l) for l in open(tmp_path / "ddpg.json")]
    ep = [r["kwargs"] for r in recs if r["msg"] == "Episode Statistics"]
    tr = [r["kwargs"] for r in recs if r["msg"] == "Training Statistics"]
    assert ep and tr and {"episode_return", "episode_length", "global_step", "steps_per_sec"} <= set(ep[0]) \
        and {"critic_loss", "actor_loss"} <= set(tr[-1])
    r = np.array(res["episode_returns"])
    assert res["learn_steps"] == LEARN_STEPS - 5_000 and res["actor_steps"] == (LEARN_STEPS - 5_000) // 2
    first, last = r[:5].mean(), r[-5:].mean()
    print("ddpg learning: first 5k steps %.1f, last 5k steps %.1f" % (first, last))
    assert last > LEARN_MIN_RETURN and last - first > LEARN_MIN_GAIN, (first, last)


LEARN_STEPS = 30_000
LEARN_MIN_RETURN = -700.0
LEARN_MIN_GAIN = 400.0


def test_cli_runs_ddpg(torch_cuda, tmp_path):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "cleanrl_jl_b200.py"), "ddpg", "--num_envs", "64", "--total_timesteps",
                        "12800", "--learning_starts", "2000", "--buffer_size", "8192"], cwd=str(tmp_path), capture_output=True,
                       text=True, timeout=300)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    res = json.loads(p.stdout.strip().splitlines()[-1])
    assert res["algorithm"] == "ddpg" and res["global_step"] == 12800 and res["learn_steps"] > 0 and res["steps_per_sec"] > 0
