"""TD3 (include/cleanrl_td3.h) without a GPU: the float64 reference of tests/td3_reference.py against torch autograd of
CleanRL's expression, the smoothing draw, the run loop's counts, the C header and its ctypes mirror, configuration
validation before any device work, the host config and the CLI."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import ddpg_reference as R
import td3_reference as T
from test_ddpg import _torch_nets, rand_nets

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TD3_HEADER = os.path.join(ROOT, "include", "cleanrl_td3.h")
DDPG_HEADER = os.path.join(ROOT, "include", "cleanrl_ddpg.h")
MAIN_HEADER = os.path.join(ROOT, "include", "cleanrl_cuda.h")
F = np.float32


def _symbols(path):
    return set(re.findall(r"CRL_API\s+(?:int|const char\*)\s+(crl_\w+)\s*\(", open(path).read()))


# ------------------------------------------------------------------ batches shared with tests/test_gpu_td3.py
KINDS = ["mixed", "terminal", "gamma0", "relu0", "noise_clamp", "action_clamp", "q1_wins", "q2_wins"]


def td3_batch(kind, B, seed):
    """dict of the five nets (actor_tgt, qf1, qf2, qf1_tgt, qf2_tgt, all different), the batch, gamma, policy_noise,
    noise_clip, learn_step and `zero`, the gradient entries that must be exactly 0 in both critics. Rewards are -1.5, 1
    or 2 so that no TD error is close to 0.
      mixed         random batch, 20 % terminal, gamma 0.99, CleanRL's noise (0.2, clip 0.5)
      terminal      every sample terminal (the targets drop out)
      gamma0        no sample terminal, gamma 0
      relu0         every obs row and action 0 and every other first-layer bias of qf1 and qf2 0: those
                    pre-activations are exactly 0 and relu'(0) = 0, so their W1 rows, b1 entries and W2 columns get 0
      noise_clamp   policy_noise 5: most draws are clipped, to +noise_clip and to -noise_clip
      action_clamp  policy_noise 1 and a target actor near +2: mu' + eps is clipped at 2 for many samples
      q1_wins       qf2' = qf1' + 5: the minimum is qf1' everywhere
      q2_wins       qf2' = qf1' - 5: the minimum is qf2' everywhere"""
    rng = np.random.default_rng(seed)
    _, q1 = rand_nets(seed)
    at, q1t = rand_nets(seed + 1000)
    _, q2 = rand_nets(seed + 2000)
    _, q2t = rand_nets(seed + 3000)
    obs = rng.uniform(-1, 1, (B, 3)).astype(F); nobs = rng.uniform(-1, 1, (B, 3)).astype(F)
    act = rng.uniform(-2, 2, B).astype(F)
    rew = rng.choice(np.array([-1.5, 1.0, 2.0], F), B)
    term = (rng.random(B) < 0.2).astype(np.uint8)
    gamma, pn, nc, zero = 0.99, 0.2, 0.5, np.zeros(0, int)
    if kind == "terminal":
        term[:] = 1
    elif kind == "gamma0":
        term[:] = 0; gamma = 0.0
    elif kind == "relu0":
        obs[:] = 0.0; act[:] = 0.0
        dead = np.arange(0, 64, 2)
        w1, b1, w2 = (R.CRITIC_ARRAYS[i][1] for i in range(3))
        for p in (q1, q2):
            p[b1 + dead] = 0.0
        zero = np.array([w1 + j + 64 * k for j in dead for k in range(4)] + [b1 + j for j in dead] +
                        [w2 + i + 64 * j for j in dead for i in range(64)])
    elif kind == "noise_clamp":
        pn = 5.0
    elif kind == "action_clamp":
        pn = 1.0
        at[-1] = 3.0
    elif kind == "q1_wins":
        q2t = q1t.copy(); q2t[-1] += 5.0
    elif kind == "q2_wins":
        q2t = q1t.copy(); q2t[-1] -= 5.0
    return dict(at=at, q1=q1, q2=q2, q1t=q1t, q2t=q2t, obs=obs, act=act, rew=rew, nobs=nobs, term=term, gamma=gamma,
                pn=pn, nc=nc, learn_step=7 * B + KINDS.index(kind), zero=zero)


def ref_twin(d, z):
    return T.twin_critic_loss_grad(d["at"], d["q1"], d["q2"], d["q1t"], d["q2t"], d["obs"], d["act"], d["rew"], d["nobs"],
                                   d["term"], d["gamma"], z, d["pn"], d["nc"])


# ------------------------------------------------------------------ reference vs autograd
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("B", [1, 17, 256])
def test_reference_twin_critic_matches_torch_autograd_of_cleanrl(kind, B):
    """CleanRL's td3_continuous_action.py critic step with torch.randn_like replaced by the injected z"""
    torch = pytest.importorskip("torch")
    d = td3_batch(kind, B, 5 * B + KINDS.index(kind))
    z = np.random.default_rng(B).standard_normal(B)
    l1, l2, g1, g2 = ref_twin(d, z)
    t1, f1 = _torch_nets(torch, d["q1"], 4)
    t2, f2 = _torch_nets(torch, d["q2"], 4)
    _, fat = _torch_nets(torch, d["at"], 3)
    _, f1t = _torch_nets(torch, d["q1t"], 4)
    _, f2t = _torch_nets(torch, d["q2t"], 4)
    tn = torch.tensor(d["nobs"], dtype=torch.float64)
    with torch.no_grad():
        clipped_noise = (torch.tensor(z) * d["pn"]).clamp(-d["nc"], d["nc"]) * 2.0
        mu_t = 2.0 * torch.tanh(fat(tn))
        next_actions = (mu_t + clipped_noise).clamp(-2.0, 2.0)
        xn = torch.cat([tn, next_actions[:, None]], 1)
        q1n, q2n = f1t(xn), f2t(xn)
        y = torch.tensor(d["rew"], dtype=torch.float64) + d["gamma"] * (1 - torch.tensor(d["term"], dtype=torch.float64)) * torch.min(q1n, q2n)
    x = torch.cat([torch.tensor(d["obs"], dtype=torch.float64), torch.tensor(d["act"], dtype=torch.float64)[:, None]], 1)
    qf1_loss = torch.nn.functional.mse_loss(f1(x), y)
    qf2_loss = torch.nn.functional.mse_loss(f2(x), y)
    (qf1_loss + qf2_loss).backward()
    np.testing.assert_allclose([l1, l2], [qf1_loss.item(), qf2_loss.item()], rtol=1e-12)
    np.testing.assert_allclose(g1, t1.grad.numpy(), rtol=1e-10, atol=1e-14)
    np.testing.assert_allclose(g2, t2.grad.numpy(), rtol=1e-10, atol=1e-14)
    if len(d["zero"]):
        assert np.all(g1[d["zero"]] == 0.0) and np.all(g2[d["zero"]] == 0.0)
    # each batch kind reaches the case it is named for
    raw = d["pn"] * z
    if kind == "noise_clamp" and B > 1:
        assert (raw > d["nc"]).any() and (raw < -d["nc"]).any()
    if kind == "action_clamp" and B > 1:
        assert (mu_t.numpy() + clipped_noise.numpy() > 2.0).any()
    if kind == "q1_wins":
        assert bool((q1n < q2n).all())
    if kind == "q2_wins":
        assert bool((q2n < q1n).all())


def test_smoothing_draw_is_philox_stream_7_keyed_by_batch_position_and_learning_step(olib):
    seed, step, B = 0x1234_5678_9ABC, (1 << 32) + 5, 40
    z = T.smoothing_normals(seed, step, B)
    for b in (0, 1, B - 1):
        r = olib.philox([b, step & 0xFFFFFFFF, step >> 32, 7], [seed & 0xFFFFFFFF, seed >> 32])
        u1 = ((int(r[0]) >> 8) + 1) / 16777216.0
        u2 = (int(r[1]) >> 8) / 16777216.0
        assert z[b] == np.sqrt(-2.0 * np.log(u1)) * np.cos(2.0 * np.pi * u2)
    # the draw depends on the step (counter) and on the seed, and differs from DDPG's acting stream 5
    assert not np.array_equal(z, T.smoothing_normals(seed, step + 1, B))
    assert not np.array_equal(z, T.smoothing_normals(seed + 1, step, B))
    r5 = olib.philox([0, step & 0xFFFFFFFF, step >> 32, 5], [seed & 0xFFFFFFFF, seed >> 32])
    r7 = olib.philox([0, step & 0xFFFFFFFF, step >> 32, 7], [seed & 0xFFFFFFFF, seed >> 32])
    assert not np.array_equal(r5, r7)
    z = T.smoothing_normals(3, 0, 4000)
    assert abs(z.mean()) < 0.1 and abs(z.std() - 1.0) < 0.1


def test_noise_clip_zero_gives_the_ddpg_target():
    d = td3_batch("mixed", 33, 4)
    z = np.random.default_rng(0).standard_normal(33)
    d["q2"], d["q2t"], d["nc"] = d["q1"], d["q1t"], 0.0
    l1, l2, g1, g2 = ref_twin(d, z)
    ld, gd = R.critic_loss_grad(d["at"], d["q1"], d["q1t"], d["obs"], d["act"], d["rew"], d["nobs"], d["term"], d["gamma"])
    assert l1 == l2 == ld and np.array_equal(g1, gd) and np.array_equal(g2, gd)


# ------------------------------------------------------------------ run loop
def test_reference_run_loop_counts_and_acting_like_ddpg(olib, abi):
    cfg = abi.make_td3_config(num_envs=3, buffer_size=40, learning_starts=30, batch_size=8, train_freq=2, policy_frequency=3,
                              max_episode_steps=7)
    a, q1 = rand_nets(1)
    _, q2 = rand_nets(2)
    ref = T.RefTD3(olib, cfg, a, q1, q2)
    dd = R.RefDDPG(olib, abi.make_ddpg_config(num_envs=3, buffer_size=40, learning_starts=30, batch_size=8, train_freq=2,
                                              policy_frequency=3, max_episode_steps=7), a, q1)
    ref.run(10); dd.run(10)
    assert ref.learn_steps == 0 and ref.size == 30
    for k in ("b_obs", "b_next", "b_act", "b_rew", "b_term"):
        assert np.array_equal(getattr(ref, k), getattr(dd, k)), k
    ref.run(20)
    # iterations 11..30 with gs = 3 it > 30, it even, size >= 8: 10 learning steps, 3 actor steps
    assert ref.learn_steps == 10 and ref.actor_steps == 3 and ref.size == 40
    assert not np.array_equal(ref.qf2_tgt, q2) and not np.array_equal(ref.qf2, ref.critic)


def test_acting_launch_count():
    class Cfg:
        num_envs, buffer_size, learning_starts, batch_size, train_freq = 4, 1 << 20, 10 ** 9, 1, 1
    # warm-up only: one launch per 1,024 iterations, split at each call
    assert T.acting_launches(Cfg, [3000]) == 3 and T.acting_launches(Cfg, [1000, 1000, 1000]) == 3
    assert T.acting_launches(Cfg, [1025]) == 2 and T.acting_launches(Cfg, [0]) == 0
    Cfg.buffer_size = 40                   # ring of 10 iterations
    assert T.acting_launches(Cfg, [25]) == 3
    Cfg.buffer_size, Cfg.learning_starts, Cfg.train_freq = 1 << 20, 20, 3
    # it = 1..5 warm (gs <= 20); learning at it = 6, 9, 12, ...: launches end at 6, 9, 12, 15 and 17
    assert T.acting_launches(Cfg, [17]) == 5


# ------------------------------------------------------------------ C header and ctypes mirror
def test_td3_header_symbols_are_exported_bound_and_disjoint_from_both_headers(crl):
    syms = _symbols(TD3_HEADER)
    assert syms == {"crl_td3_create", "crl_td3_destroy", "crl_td3_set_params", "crl_td3_get_params", "crl_td3_get_adam_state",
                    "crl_td3_reset", "crl_td3_run", "crl_td3_read_buffer", "crl_td3_critic_loss_raw"}
    assert not syms & _symbols(MAIN_HEADER) and not syms & _symbols(DDPG_HEADER)
    assert set(crl.TD3_SIGNATURES) == syms
    assert not set(crl.TD3_SIGNATURES) & (set(crl.SIGNATURES) | set(crl.DDPG_SIGNATURES))
    lib = crl.load()
    for s in syms:
        assert hasattr(lib, s), s
    nm = subprocess.check_output(["nm", "-D", os.path.join(ROOT, "cleanrl.jl_b200", "libcleanrl_cuda.so")], text=True)
    for s in syms:
        assert re.search(r"\bT %s\b" % s, nm), s


def test_pure_c_file_including_the_td3_header_compiles_with_warnings_as_errors(tmp_path):
    src = tmp_path / "td3_c.c"
    src.write_text('#include "cleanrl_td3.h"\n#include <stdio.h>\n'
                   'int main(void) { crl_td3_config c = {0}; crl_td3_stats s = {0}; c.struct_size = (int32_t)sizeof(c);\n'
                   '  int (*f)(const crl_td3_config*, crl_td3_ctx**) = crl_td3_create; (void)f; (void)s;\n'
                   '  int (*g)(const crl_ddpg_config*, crl_ddpg_ctx**) = crl_ddpg_create; (void)g;\n'
                   '  printf("%d %d %d\\n", c.struct_size, CRL_DDPG_CRITIC_PARAMS, CRL_OK); return 0; }\n')
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), "-c", str(src),
                           "-o", str(tmp_path / "td3_c.o")])


def test_td3_struct_layout_matches_ctypes(tmp_path, abi):
    fields_c = [f for f, _ in abi.crl_td3_config._fields_]
    fields_s = [f for f, _ in abi.crl_td3_stats._fields_]
    expr = ["sizeof(crl_td3_config)"] + ["offsetof(crl_td3_config,%s)" % f for f in fields_c] + \
           ["sizeof(crl_td3_stats)"] + ["offsetof(crl_td3_stats,%s)" % f for f in fields_s]
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "cleanrl_td3.h"\nint main(){%s return 0;}\n'
                   % "".join('printf("%%zu\\n", (size_t)%s);' % e for e in expr))
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    want = [C.sizeof(abi.crl_td3_config)] + [getattr(abi.crl_td3_config, f).offset for f in fields_c] + \
           [C.sizeof(abi.crl_td3_stats)] + [getattr(abi.crl_td3_stats, f).offset for f in fields_s]
    assert got == want


# ------------------------------------------------------------------ validation and the no-GPU path
BAD_CONFIGS = [
    (dict(policy_noise=-0.1), b"policy_noise"), (dict(policy_noise=float("nan")), b"policy_noise"),
    (dict(policy_noise=float("inf")), b"policy_noise"), (dict(noise_clip=-0.5), b"noise_clip"),
    (dict(noise_clip=float("nan")), b"noise_clip"), (dict(noise_clip=float("inf")), b"noise_clip"),
    (dict(batch_size=0), b"batch_size"), (dict(batch_size=257), b"batch_size"),
    (dict(num_envs=8, buffer_size=7), b"buffer_size"), (dict(train_freq=0), b"train_freq"),
    (dict(policy_frequency=0), b"policy_frequency"), (dict(tau=0.0), b"tau"), (dict(lr=0.0), b"lr"),
]


@pytest.mark.parametrize("kw,msg", BAD_CONFIGS)
def test_invalid_td3_config_is_rejected_before_device_work(crl, abi, kw, msg):
    lib = crl.load()
    h = C.c_void_p()
    cfg = abi.make_td3_config(**kw)
    assert lib.crl_td3_create(C.byref(cfg), C.byref(h)) == abi.CRL_ERR_INVALID
    assert not h.value and msg in lib.crl_last_error()
    cfg = abi.make_td3_config()
    cfg.struct_size = C.sizeof(abi.crl_ddpg_config)
    assert lib.crl_td3_create(C.byref(cfg), C.byref(h)) == abi.CRL_ERR_INVALID
    assert b"struct_size" in lib.crl_last_error()


def test_td3_has_no_cpu_fallback_without_a_gpu(crl, abi):
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a GPU is visible")
    except ImportError:
        pass
    lib = crl.load()
    h = C.c_void_p()
    cfg = abi.make_td3_config()
    assert lib.crl_td3_create(C.byref(cfg), C.byref(h)) == abi.CRL_ERR_CUDA
    assert not h.value and len(lib.crl_last_error()) > 0
    from cleanrl_jl_b200.td3_algo import TD3Handle
    with pytest.raises(crl.CleanRLCudaError):
        TD3Handle(cfg)
    buf = np.zeros(R.CRITIC_P, np.float32)   # numpy's allocations are 16-byte aligned
    p = crl.ptr(buf)
    rc = lib.crl_td3_critic_loss_raw(*[p] * 5, 1, *[p] * 5, 0.99, 0.2, 0.5, 1, 0, *[p] * 4, None)
    assert rc == abi.CRL_ERR_CUDA and len(lib.crl_last_error()) > 0


# ------------------------------------------------------------------ host config and CLI
def test_td3_config_defaults_are_cleanrls_and_argparse_works():
    from cleanrl_jl_b200 import TD3Config, argparse_struct
    c = TD3Config()
    assert (c.buffer_size, c.learning_starts, c.batch_size, c.gamma, c.tau, c.lr, c.exploration_noise, c.policy_frequency,
            c.policy_noise, c.noise_clip, c.train_freq, c.num_envs, c.seed, c.max_steps) == \
        (1_000_000, 25_000, 256, 0.99, 0.005, 3e-4, 0.1, 2, 0.2, 0.5, 1, 1, 1, 200)
    c = argparse_struct(TD3Config(), ["--num_envs", "64", "--policy_noise", "0.3", "--noise_clip", "0.25"])
    assert isinstance(c, TD3Config) and (c.num_envs, c.policy_noise, c.noise_clip) == (64, 0.3, 0.25)
    assert c.batch_size == 256
    from cleanrl_jl_b200.td3_algo import make_crl_td3_config
    cc = make_crl_td3_config(c)
    assert (cc.num_envs, cc.policy_noise, cc.noise_clip, cc.max_episode_steps) == (64, 0.3, 0.25, 200)


def test_td3_init_params_reuse_ddpgs_and_draw_a_separate_qf2():
    from cleanrl_jl_b200.ddpg_algo import init_ddpg_params
    from cleanrl_jl_b200.td3_algo import init_td3_params
    a, q1, q2 = init_td3_params(3)
    da, dc = init_ddpg_params(3)
    assert np.array_equal(a, da) and np.array_equal(q1, dc) and q2.size == R.CRITIC_P and not np.array_equal(q1, q2)
    assert not any(np.array_equal(q2, init_ddpg_params(s)[1]) for s in range(8))


def test_cli_lists_td3_and_its_options():
    run = lambda *a: subprocess.run([sys.executable, "-m", "cleanrl_jl_b200", *a], cwd=ROOT, capture_output=True, text=True, timeout=300)
    p = run()
    assert p.returncode == 2 and "{td3}" in p.stderr and "{ddpg}" in p.stderr
    p = run("td3", "--help")
    assert p.returncode == 0
    for field in ("--buffer_size", "--learning_starts", "--batch_size", "--tau", "--exploration_noise", "--policy_frequency",
                  "--policy_noise", "--noise_clip", "--train_freq", "--num_envs"):
        assert field in p.stdout, field
