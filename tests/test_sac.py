"""SAC (include/cleanrl_sac.h) without a GPU: the float64 reference of tests/sac_reference.py against torch autograd of
CleanRL's expressions, the three noise draws, the run loop's counts and its acting before the first learning step, the C
header and its ctypes mirror, configuration validation before any device work, the host config and the CLI."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import ddpg_reference as R
import sac_reference as S
from test_ddpg import _torch_nets, rand_nets

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADERS = {k: os.path.join(ROOT, "include", "cleanrl_%s.h" % k) for k in ("cuda", "ddpg", "td3", "sac")}
F = np.float32


def _symbols(path):
    return set(re.findall(r"CRL_API\s+(?:int|const char\*)\s+(crl_\w+)\s*\(", open(path).read()))


def rand_actor(seed):
    """init_sac_params' actor with small random biases (a nonzero log_std head)"""
    from cleanrl_jl_b200.sac_algo import init_sac_params
    rng = np.random.default_rng(seed + 77)
    a = init_sac_params(seed)[0]
    for name, s, e in S.ACTOR_ARRAYS:
        if name.startswith("b"):
            a[s:e] = rng.normal(0, 0.1, e - s)
    return a


# ------------------------------------------------------------------ batches shared with tests/test_gpu_sac.py
KINDS = ["mixed", "terminal", "gamma0", "relu0", "q1_wins", "q2_wins", "ties", "logstd_low", "logstd_high", "squash", "alpha0"]


def sac_batch(kind, B, seed):
    """dict of the nets (actor, qf1, qf2, qf1_tgt, qf2_tgt), the batch, gamma, alpha, the noise counters and `zero_q` /
    `zero_a`, the critic and actor gradient entries that must be exactly 0. Rewards are -1.5, 1 or 2.
      mixed        random batch, 20 % terminal, gamma 0.99, alpha 0.2
      terminal     every sample terminal (the targets drop out)
      gamma0       no sample terminal, gamma 0
      relu0        every obs row and action 0 and every other first-layer bias of the actor, qf1 and qf2 0: those
                   pre-activations are exactly 0 and relu'(0) = 0, so their W1 rows, b1 entries and W2 columns get 0
                   (the actor's and, in the critic step, the critics')
      q1_wins      qf2 = qf1 + 5 and qf2' = qf1' + 5 (output bias): the minimum is qf1 (and qf1') everywhere
      q2_wins      the same with -5: the minimum is qf2 everywhere
      ties         qf2 = qf1 and qf2' = qf1': every minimum is a tie, and the halves of the gradient sum to one critic's
      logstd_low   fc_logstd bias -30: log_std saturates at -5
      logstd_high  fc_logstd bias +30: log_std saturates at 2 (std = e^2)
      squash       fc_mean bias 8 and log_std at -5: |x| is about 8, 2 (1 - tanh^2 x) is of the order of the 1e-6 guard
      alpha0       alpha 0: the entropy terms drop out"""
    rng = np.random.default_rng(seed)
    _, q1 = rand_nets(seed)
    _, q1t = rand_nets(seed + 1000)
    _, q2 = rand_nets(seed + 2000)
    _, q2t = rand_nets(seed + 3000)
    actor = rand_actor(seed)
    obs = rng.uniform(-1, 1, (B, 3)).astype(F); nobs = rng.uniform(-1, 1, (B, 3)).astype(F)
    act = rng.uniform(-2, 2, B).astype(F)
    rew = rng.choice(np.array([-1.5, 1.0, 2.0], F), B)
    term = (rng.random(B) < 0.2).astype(np.uint8)
    gamma, alpha, zero_q, zero_a = 0.99, 0.2, np.zeros(0, int), np.zeros(0, int)
    b_mean, b_logstd = S._OFF["b_mean"][0], S._OFF["b_logstd"][0]
    if kind == "terminal":
        term[:] = 1
    elif kind == "gamma0":
        term[:] = 0; gamma = 0.0
    elif kind == "relu0":
        obs[:] = 0.0; act[:] = 0.0; nobs[:] = 0.0
        dead = np.arange(0, 64, 2)
        w1, b1, w2 = (R.CRITIC_ARRAYS[i][1] for i in range(3))
        for p in (q1, q2):
            p[b1 + dead] = 0.0
        zero_q = np.array([w1 + j + 64 * k for j in dead for k in range(4)] + [b1 + j for j in dead] +
                          [w2 + i + 64 * j for j in dead for i in range(64)])
        w1, b1, w2 = (S.ACTOR_ARRAYS[i][1] for i in range(3))
        actor[b1 + dead] = 0.0
        zero_a = np.array([w1 + j + 64 * k for j in dead for k in range(3)] + [b1 + j for j in dead] +
                          [w2 + i + 64 * j for j in dead for i in range(64)])
    elif kind in ("q1_wins", "q2_wins"):
        d = 5.0 if kind == "q1_wins" else -5.0
        q2, q2t = q1.copy(), q1t.copy()
        q2[-1] += d; q2t[-1] += d
    elif kind == "ties":
        q2, q2t = q1.copy(), q1t.copy()
    elif kind == "logstd_low":
        actor[b_logstd] = -30.0
    elif kind == "logstd_high":
        actor[b_logstd] = 30.0
    elif kind == "squash":
        actor[b_mean] = 8.0; actor[b_logstd] = -30.0
    elif kind == "alpha0":
        alpha = 0.0
    return dict(actor=actor, q1=q1, q2=q2, q1t=q1t, q2t=q2t, obs=obs, act=act, rew=rew, nobs=nobs, term=term, gamma=gamma,
                alpha=alpha, learn_step=7 * B + KINDS.index(kind), actor_step=5 * B + KINDS.index(kind), zero_q=zero_q,
                zero_a=zero_a)


def ref_critic(d, z):
    return S.critic_loss_grad(d["actor"], d["q1"], d["q2"], d["q1t"], d["q2t"], d["obs"], d["act"], d["rew"], d["nobs"],
                              d["term"], d["gamma"], d["alpha"], z)


# ------------------------------------------------------------------ reference vs autograd
def _torch_actor(torch, p):
    t = torch.tensor(np.asarray(p, np.float64), requires_grad=True)
    part = {n: t[s:e] for n, s, e in S.ACTOR_ARRAYS}
    W1, W2 = part["W1"].reshape(3, 64).T, part["W2"].reshape(64, 64).T

    def get_action(x, z):
        """CleanRL's Actor.get_action with the rsample noise injected"""
        h = torch.relu(torch.relu(x @ W1.T + part["b1"]) @ W2.T + part["b2"])
        mean = h @ part["W_mean"] + part["b_mean"][0]
        log_std = torch.tanh(h @ part["W_logstd"] + part["b_logstd"][0])
        log_std = -5.0 + 0.5 * (2.0 - (-5.0)) * (log_std + 1)
        std = log_std.exp()
        normal = torch.distributions.Normal(mean, std)
        x_t = mean + std * z
        y_t = torch.tanh(x_t)
        action = y_t * 2.0
        log_prob = normal.log_prob(x_t)
        log_prob = log_prob - torch.log(2.0 * (1 - y_t.pow(2)) + 1e-6)
        return action, log_prob, x_t, log_std
    return t, get_action


# 1 - tanh^2 x cancels in CleanRL's expression where |x| is large: the reference takes it as 1/cosh^2 x, so where the
# squash saturates the two agree to the cancellation error of torch's form (about 1e-8 at |x| = 10), not to 1e-10
AUTOGRAD_RTOL = {"squash": 1e-6, "logstd_high": 1e-6}


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("B", [1, 17, 256])
def test_reference_matches_torch_autograd_of_cleanrl(kind, B):
    """CleanRL's sac_continuous_action.py critic, actor and temperature steps with the rsample noise injected"""
    torch = pytest.importorskip("torch")
    d = sac_batch(kind, B, 5 * B + KINDS.index(kind))
    rng = np.random.default_rng(B + 3)
    z8, z9, z10 = rng.standard_normal(B), rng.standard_normal(B), rng.standard_normal(B)
    rtol = AUTOGRAD_RTOL.get(kind, 1e-10)
    T = lambda x: torch.tensor(np.asarray(x, np.float64))
    alpha = d["alpha"]
    # critic step
    l1, l2, g1, g2 = ref_critic(d, z8)
    _, actor_f = _torch_actor(torch, d["actor"])
    t1, f1 = _torch_nets(torch, d["q1"], 4)
    t2, f2 = _torch_nets(torch, d["q2"], 4)
    _, f1t = _torch_nets(torch, d["q1t"], 4)
    _, f2t = _torch_nets(torch, d["q2t"], 4)
    tn = T(d["nobs"])
    with torch.no_grad():
        next_actions, next_log_pi, x_next, ls_next = actor_f(tn, T(z8))
        xn = torch.cat([tn, next_actions[:, None]], 1)
        q1n, q2n = f1t(xn), f2t(xn)
        min_qf_next_target = torch.min(q1n, q2n) - alpha * next_log_pi
        next_q_value = T(d["rew"]) + (1 - T(d["term"])) * d["gamma"] * min_qf_next_target
    x = torch.cat([T(d["obs"]), T(d["act"])[:, None]], 1)
    qf1_loss = torch.nn.functional.mse_loss(f1(x), next_q_value)
    qf2_loss = torch.nn.functional.mse_loss(f2(x), next_q_value)
    (qf1_loss + qf2_loss).backward()
    np.testing.assert_allclose([l1, l2], [qf1_loss.item(), qf2_loss.item()], rtol=rtol)
    np.testing.assert_allclose(g1, t1.grad.numpy(), rtol=rtol, atol=1e-14)
    np.testing.assert_allclose(g2, t2.grad.numpy(), rtol=rtol, atol=1e-14)
    if len(d["zero_q"]):
        assert np.all(g1[d["zero_q"]] == 0.0) and np.all(g2[d["zero_q"]] == 0.0)
    # actor step
    la, ga, mlp = S.actor_loss_grad(d["actor"], d["q1"], d["q2"], d["obs"], alpha, z9)
    ta, actor_f = _torch_actor(torch, d["actor"])
    _, f1 = _torch_nets(torch, d["q1"], 4)
    _, f2 = _torch_nets(torch, d["q2"], 4)
    to = T(d["obs"])
    pi, log_pi, x_t, log_std = actor_f(to, T(z9))
    qf1_pi, qf2_pi = f1(torch.cat([to, pi[:, None]], 1)), f2(torch.cat([to, pi[:, None]], 1))
    min_qf_pi = torch.min(qf1_pi, qf2_pi)
    actor_loss = ((alpha * log_pi) - min_qf_pi).mean()
    actor_loss.backward()
    np.testing.assert_allclose(la, actor_loss.item(), rtol=rtol, atol=1e-12)
    np.testing.assert_allclose(mlp, log_pi.mean().item(), rtol=rtol)
    scale = np.abs(ta.grad.numpy()).max()
    np.testing.assert_allclose(ga, ta.grad.numpy(), rtol=rtol, atol=1e-2 * rtol * scale)
    if len(d["zero_a"]):
        assert np.all(ga[d["zero_a"]] == 0.0)
    # temperature step
    log_alpha = torch.tensor(0.3, dtype=torch.float64, requires_grad=True)
    with torch.no_grad():
        _, lp10, _, _ = actor_f(to, T(z10))
    loss = (-log_alpha.exp() * (lp10 + S.TARGET_ENTROPY)).mean()
    loss.backward()
    _, lp = S.sample(d["actor"], d["obs"], z10)
    np.testing.assert_allclose([S.alpha_loss(0.3, lp)] * 2, [loss.item(), log_alpha.grad.item()], rtol=rtol)
    # each batch kind reaches the case it is named for
    with torch.no_grad():
        q1s, q2s = qf1_pi.numpy(), qf2_pi.numpy()
    if kind == "q1_wins":
        assert bool((q1n < q2n).all()) and np.all(q1s < q2s)
    if kind == "q2_wins":
        assert bool((q2n < q1n).all()) and np.all(q2s < q1s)
    if kind == "ties":
        assert bool((q1n == q2n).all()) and np.all(q1s == q2s)
        # the halves of torch.minimum's gradient sum to the gradient through one critic
        far = d["q1"].copy()
        far[-1] += 1e3                         # qf2 = qf1 + 1000: the minimum is qf1 alone
        _, g_one, _ = S.actor_loss_grad(d["actor"], d["q1"], far, d["obs"], alpha, z9)
        np.testing.assert_allclose(ga, g_one, rtol=1e-12, atol=1e-15)
    if kind == "logstd_low":
        assert np.all(log_std.detach().numpy() == -5.0) and np.all(ls_next.numpy() == -5.0)
    if kind == "logstd_high":
        assert np.all(log_std.detach().numpy() == 2.0)
    if kind == "squash":
        s2 = 2.0 / np.cosh(x_t.detach().numpy()) ** 2
        assert np.all(np.abs(x_t.detach().numpy()) > 5.0) and s2.max() < 1e-4 and s2.min() < 1e-5
    if kind == "alpha0":
        assert alpha == 0.0


# ------------------------------------------------------------------ draws
@pytest.mark.parametrize("stream", [8, 9, 10])
def test_draws_are_philox_keyed_by_batch_position_and_counter(olib, stream):
    seed, counter, B = 0x1234_5678_9ABC, (1 << 32) + 5, 40
    z = S.normals(seed, counter, B, stream)
    for b in (0, 1, B - 1):
        r = olib.philox([b, counter & 0xFFFFFFFF, counter >> 32, stream], [seed & 0xFFFFFFFF, seed >> 32])
        u1 = ((int(r[0]) >> 8) + 1) / 16777216.0
        u2 = (int(r[1]) >> 8) / 16777216.0
        assert z[b] == np.sqrt(-2.0 * np.log(u1)) * np.cos(2.0 * np.pi * u2)
    assert not np.array_equal(z, S.normals(seed, counter + 1, B, stream))
    assert not np.array_equal(z, S.normals(seed + 1, counter, B, stream))
    others = {5, 6, 7, 8, 9, 10} - {stream}
    for o in others:
        assert not np.array_equal(z, S.normals(seed, counter, B, o))
    z = S.normals(3, 0, 4000, stream)
    assert abs(z.mean()) < 0.1 and abs(z.std() - 1.0) < 0.1


def test_log_pi_is_the_squashed_gaussian_density():
    """log_pi integrates the density of a = 2 tanh(x) with the 1e-6 guard: without the guard it is the change of
    variables of N(mean, std) under a = 2 tanh x"""
    mean, l = np.array([0.3, -1.2]), np.array([0.1, -0.4])
    z = np.array([0.7, -1.1])
    s = S.squash(mean, l, z)
    std = np.exp(-5.0 + 3.5 * (np.tanh(l) + 1.0))
    x = mean + std * z
    exact = -0.5 * ((x - mean) / std) ** 2 - np.log(std) - 0.5 * np.log(2 * np.pi) - np.log(2 * (1 - np.tanh(x) ** 2))
    np.testing.assert_allclose(s["log_pi"], exact, rtol=1e-5)
    np.testing.assert_allclose(s["a"], 2 * np.tanh(x), rtol=1e-15)


# ------------------------------------------------------------------ run loop
def test_reference_run_loop_counts_and_acting_like_ddpg(olib, abi):
    kw = dict(num_envs=3, buffer_size=40, learning_starts=30, batch_size=8, train_freq=2, policy_frequency=3, max_episode_steps=7)
    from cleanrl_jl_b200.sac_algo import init_sac_params
    a, q1, q2 = init_sac_params(1)
    ref = S.RefSAC(olib, abi.make_sac_config(target_network_frequency=2, **kw), a, q1, q2)
    dd = R.RefDDPG(olib, abi.make_ddpg_config(**kw), rand_nets(1)[0], q1)
    ref.run(10); dd.run(10)
    assert ref.learn_steps == 0 and ref.size == 30
    for k in ("b_obs", "b_next", "b_act", "b_rew", "b_term"):
        assert np.array_equal(getattr(ref, k), getattr(dd, k)), k
    ref.run(20)
    # iterations 11..30 with gs = 3 it > 30, it even, size >= 8: 10 learning steps, 3 rounds of 3 actor iterations, 5
    # target updates
    assert (ref.learn_steps, ref.actor_steps, ref.size) == (10, 9, 40)
    assert S.closed_form_counts(ref.cfg, 30) == (10, 9, 5)
    assert ref.alpha != 1.0 and ref.log_alpha != 0.0
    assert not np.array_equal(ref.qf2_tgt, q2) and not np.array_equal(ref.actor, a)
    # without autotune alpha stays the configured constant
    ref = S.RefSAC(olib, abi.make_sac_config(autotune=0, alpha=0.3, **kw), a, q1, q2)
    ref.run(30)
    assert ref.alpha == 0.3 and ref.log_alpha == 0.0 and ref.alpha_loss == 0.0 and ref.actor_steps == 9


def test_kernel_launch_closed_form(abi):
    cfg = abi.make_sac_config(num_envs=4, buffer_size=512, learning_starts=64, batch_size=32, policy_frequency=3,
                              target_network_frequency=2)
    learn, actor, tgt = S.closed_form_counts(cfg, 60)
    assert (learn, actor, tgt) == (44, 42, 22)
    assert S.kernel_launches(cfg, 7, learn, actor, tgt) == 7 + 88 + 4 * 42 + 22
    cfg.autotune = 0
    assert S.kernel_launches(cfg, 7, learn, actor, tgt) == 7 + 88 + 2 * 42 + 22


# ------------------------------------------------------------------ C header and ctypes mirror
def test_sac_header_symbols_are_exported_bound_and_disjoint_from_the_other_headers(crl):
    syms = _symbols(HEADERS["sac"])
    assert syms == {"crl_sac_create", "crl_sac_destroy", "crl_sac_set_params", "crl_sac_get_params", "crl_sac_get_adam_state",
                    "crl_sac_reset", "crl_sac_run", "crl_sac_read_buffer", "crl_sac_forward_raw", "crl_sac_critic_loss_raw",
                    "crl_sac_actor_loss_raw"}
    for k in ("cuda", "ddpg", "td3"):
        assert not syms & _symbols(HEADERS[k]), k
    assert set(crl.SAC_SIGNATURES) == syms
    assert not set(crl.SAC_SIGNATURES) & (set(crl.SIGNATURES) | set(crl.DDPG_SIGNATURES) | set(crl.TD3_SIGNATURES))
    lib = crl.load()
    for s in syms:
        assert hasattr(lib, s), s
    nm = subprocess.check_output(["nm", "-D", os.path.join(ROOT, "cleanrl.jl_b200", "libcleanrl_cuda.so")], text=True)
    for s in syms:
        assert re.search(r"\bT %s\b" % s, nm), s


def test_sac_header_defines_the_actor_size_and_the_launch_count():
    src = open(HEADERS["sac"]).read()
    assert re.search(r"#define CRL_SAC_ACTOR_PARAMS 4546\b", src)
    assert "acting launches + 2 learn_steps + (2 + 2 autotune) actor_steps" in src
    assert S.ACTOR_ARRAYS[-1][2] == 4546


def test_pure_c_file_including_the_sac_header_compiles_with_warnings_as_errors(tmp_path):
    src = tmp_path / "sac_c.c"
    src.write_text('#include "cleanrl_sac.h"\n#include <stdio.h>\n'
                   'int main(void) { crl_sac_config c = {0}; crl_sac_stats s = {0}; c.struct_size = (int32_t)sizeof(c);\n'
                   '  int (*f)(const crl_sac_config*, crl_sac_ctx**) = crl_sac_create; (void)f; (void)s;\n'
                   '  int (*g)(const crl_ddpg_config*, crl_ddpg_ctx**) = crl_ddpg_create; (void)g;\n'
                   '  printf("%d %d %d\\n", c.struct_size, CRL_SAC_ACTOR_PARAMS, CRL_OK); return 0; }\n')
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), "-c", str(src),
                           "-o", str(tmp_path / "sac_c.o")])


def test_sac_struct_layout_matches_ctypes(tmp_path, abi):
    fields_c = [f for f, _ in abi.crl_sac_config._fields_]
    fields_s = [f for f, _ in abi.crl_sac_stats._fields_]
    expr = ["sizeof(crl_sac_config)"] + ["offsetof(crl_sac_config,%s)" % f for f in fields_c] + \
           ["sizeof(crl_sac_stats)"] + ["offsetof(crl_sac_stats,%s)" % f for f in fields_s]
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "cleanrl_sac.h"\nint main(){%s return 0;}\n'
                   % "".join('printf("%%zu\\n", (size_t)%s);' % e for e in expr))
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    want = [C.sizeof(abi.crl_sac_config)] + [getattr(abi.crl_sac_config, f).offset for f in fields_c] + \
           [C.sizeof(abi.crl_sac_stats)] + [getattr(abi.crl_sac_stats, f).offset for f in fields_s]
    assert got == want


# ------------------------------------------------------------------ validation and the no-GPU path
BAD_CONFIGS = [
    (dict(policy_lr=0.0), b"policy_lr"), (dict(policy_lr=-1e-3), b"policy_lr"), (dict(policy_lr=float("nan")), b"policy_lr"),
    (dict(policy_lr=float("inf")), b"policy_lr"), (dict(q_lr=0.0), b"q_lr"), (dict(q_lr=float("nan")), b"q_lr"),
    (dict(q_lr=float("inf")), b"q_lr"), (dict(alpha=-0.1), b"alpha"), (dict(alpha=float("nan")), b"alpha"),
    (dict(alpha=float("inf")), b"alpha"), (dict(target_network_frequency=0), b"target_network_frequency"),
    (dict(autotune=2), b"autotune"), (dict(autotune=-1), b"autotune"),
    (dict(batch_size=0), b"batch_size"), (dict(batch_size=257), b"batch_size"),
    (dict(num_envs=8, buffer_size=7), b"buffer_size"), (dict(train_freq=0), b"train_freq"),
    (dict(policy_frequency=0), b"policy_frequency"), (dict(tau=0.0), b"tau"), (dict(learning_starts=-1), b"learning_starts"),
]


@pytest.mark.parametrize("kw,msg", BAD_CONFIGS)
def test_invalid_sac_config_is_rejected_before_device_work(crl, abi, kw, msg):
    lib = crl.load()
    h = C.c_void_p()
    cfg = abi.make_sac_config(**kw)
    assert lib.crl_sac_create(C.byref(cfg), C.byref(h)) == abi.CRL_ERR_INVALID
    assert not h.value and msg in lib.crl_last_error()
    cfg = abi.make_sac_config()
    cfg.struct_size = C.sizeof(abi.crl_ddpg_config)
    assert lib.crl_sac_create(C.byref(cfg), C.byref(h)) == abi.CRL_ERR_INVALID
    assert b"struct_size" in lib.crl_last_error()


def test_sac_has_no_cpu_fallback_without_a_gpu(crl, abi):
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a GPU is visible")
    except ImportError:
        pass
    lib = crl.load()
    h = C.c_void_p()
    cfg = abi.make_sac_config()
    assert lib.crl_sac_create(C.byref(cfg), C.byref(h)) == abi.CRL_ERR_CUDA
    assert not h.value and len(lib.crl_last_error()) > 0
    from cleanrl_jl_b200.sac_algo import SACHandle
    with pytest.raises(crl.CleanRLCudaError):
        SACHandle(cfg)
    buf = np.zeros(S.ACTOR_P, np.float32)   # numpy's allocations are 16-byte aligned
    p = crl.ptr(buf)
    assert lib.crl_sac_critic_loss_raw(*[p] * 5, 1, *[p] * 5, 0.99, 0.2, 1, 0, *[p] * 4, None) == abi.CRL_ERR_CUDA
    assert lib.crl_sac_actor_loss_raw(*[p] * 3, 1, p, 0.2, 1, 0, p, p, p, None) == abi.CRL_ERR_CUDA
    assert lib.crl_sac_forward_raw(*[p] * 7, 1, None) == abi.CRL_ERR_CUDA
    # a bad alpha or B is rejected before the device check
    assert lib.crl_sac_actor_loss_raw(*[p] * 3, 1, p, -1.0, 1, 0, p, p, p, None) == abi.CRL_ERR_INVALID
    assert lib.crl_sac_critic_loss_raw(*[p] * 5, 0, *[p] * 5, 0.99, 0.2, 1, 0, *[p] * 4, None) == abi.CRL_ERR_INVALID


# ------------------------------------------------------------------ host config and CLI
def test_sac_config_defaults_are_cleanrls_and_argparse_works():
    from cleanrl_jl_b200 import SACConfig, argparse_struct
    c = SACConfig()
    assert (c.buffer_size, c.learning_starts, c.batch_size, c.gamma, c.tau, c.policy_lr, c.q_lr, c.policy_frequency,
            c.target_network_frequency, c.alpha, c.autotune, c.train_freq, c.num_envs, c.seed, c.max_steps) == \
        (1_000_000, 5_000, 256, 0.99, 0.005, 3e-4, 1e-3, 2, 1, 0.2, True, 1, 1, 1, 200)
    c = argparse_struct(SACConfig(), ["--num_envs", "64", "--autotune", "false", "--alpha", "0.1", "--q_lr", "2e-3"])
    assert isinstance(c, SACConfig) and (c.num_envs, c.autotune, c.alpha, c.q_lr) == (64, False, 0.1, 2e-3)
    assert c.batch_size == 256
    from cleanrl_jl_b200.sac_algo import make_crl_sac_config
    cc = make_crl_sac_config(c)
    assert (cc.num_envs, cc.autotune, cc.alpha, cc.q_lr, cc.policy_lr, cc.max_episode_steps) == (64, 0, 0.1, 2e-3, 3e-4, 200)
    assert make_crl_sac_config(SACConfig()).autotune == 1


def test_sac_init_params():
    from cleanrl_jl_b200.ddpg_algo import init_ddpg_params
    from cleanrl_jl_b200.sac_algo import init_sac_params
    from cleanrl_jl_b200.td3_algo import init_td3_params
    a, q1, q2 = init_sac_params(3)
    _, t1, t2 = init_td3_params(3)
    assert a.size == S.ACTOR_P and np.array_equal(q1, t1) and np.array_equal(q2, t2)
    for name, s, e in S.ACTOR_ARRAYS:
        if name.startswith("b"):
            assert np.all(a[s:e] == 0.0), name
        else:
            fan_in = {"W1": 3}.get(name, 64)
            fan_out = 1 if name in ("W_mean", "W_logstd") else 64
            lim = np.sqrt(6.0 / (fan_in + fan_out))
            assert np.all(np.abs(a[s:e]) <= lim) and np.abs(a[s:e]).max() > 0.5 * lim, name
    assert not np.array_equal(a[S._OFF["W_mean"][0]:S._OFF["W_mean"][1]], a[S._OFF["W_logstd"][0]:S._OFF["W_logstd"][1]])
    assert not np.array_equal(a, init_sac_params(4)[0])
    assert init_ddpg_params(3)[1].size == q1.size


def test_product_package_does_not_import_the_oracle():
    src = open(os.path.join(ROOT, "cleanrl.jl_b200", "sac_algo.py")).read()
    assert "oracle" not in src


def test_cli_lists_sac_on_a_line_of_its_own():
    run = lambda *a: subprocess.run([sys.executable, "-m", "cleanrl_jl_b200", *a], cwd=ROOT, capture_output=True, text=True, timeout=300)
    p = run()
    assert p.returncode == 2 and "{sac}" in p.stderr and "{td3}" in p.stderr and "{ddpg}" in p.stderr
    p = run("sac", "--help")
    assert p.returncode == 0
    for field in ("--buffer_size", "--learning_starts", "--batch_size", "--tau", "--policy_lr", "--q_lr", "--policy_frequency",
                  "--target_network_frequency", "--alpha", "--autotune", "--train_freq", "--num_envs", "--log_frequency"):
        assert field in p.stdout, field
