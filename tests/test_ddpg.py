"""DDPG (include/cleanrl_ddpg.h) without a GPU: the float64 NumPy reference against torch autograd, the C header and
its ctypes mirror, configuration validation before any device work, the host config and the CLI."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import ddpg_reference as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DDPG_HEADER = os.path.join(ROOT, "include", "cleanrl_ddpg.h")
MAIN_HEADER = os.path.join(ROOT, "include", "cleanrl_cuda.h")


def _symbols(path):
    return set(re.findall(r"CRL_API\s+(?:int|const char\*)\s+(crl_\w+)\s*\(", open(path).read()))


def rand_nets(seed):
    from cleanrl_jl_b200.ddpg_algo import init_ddpg_params
    rng = np.random.default_rng(seed)
    a, c = init_ddpg_params(seed)
    for p, arrays in ((a, R.ACTOR_ARRAYS), (c, R.CRITIC_ARRAYS)):
        for name, s, e in arrays:
            if name.startswith("b"):
                p[s:e] = rng.normal(0, 0.1, e - s)
    return a, c


# ------------------------------------------------------------------ reference vs autograd
def _torch_nets(torch, p, d_in):
    t = torch.tensor(np.asarray(p, np.float64), requires_grad=True)
    o, parts = 0, []
    for n in (64 * d_in, 64, 64 * 64, 64, 64, 1):
        parts.append(t[o:o + n]); o += n
    W1, b1, W2, b2, W3, b3 = parts
    W1 = W1.reshape(d_in, 64).T; W2 = W2.reshape(64, 64).T; W3 = W3.reshape(1, 64)

    def f(x):
        h1 = torch.relu(x @ W1.T + b1)
        h2 = torch.relu(h1 @ W2.T + b2)
        return (h2 @ W3.T + b3)[:, 0]
    return t, f


@pytest.mark.parametrize("B", [1, 7, 64])
def test_reference_gradients_match_torch_autograd(B):
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(B)
    a, c = rand_nets(B)
    at, ct = rand_nets(B + 100)
    obs = rng.uniform(-1, 1, (B, 3)); nobs = rng.uniform(-1, 1, (B, 3)); act = rng.uniform(-2, 2, B)
    rew = rng.normal(size=B); term = (rng.random(B) < 0.3).astype(np.uint8); gamma = 0.99
    loss, g = R.critic_loss_grad(at, c, ct, obs, act, rew, nobs, term, gamma)
    tc, fc = _torch_nets(torch, c, 4)
    _, fat = _torch_nets(torch, at, 3)
    _, fct = _torch_nets(torch, ct, 4)
    with torch.no_grad():
        tn = torch.tensor(nobs)
        y = torch.tensor(rew) + gamma * (1 - torch.tensor(term, dtype=torch.float64)) * fct(torch.cat([tn, 2 * torch.tanh(fat(tn))[:, None]], 1))
    tl = torch.mean((fc(torch.cat([torch.tensor(obs), torch.tensor(act)[:, None]], 1)) - y) ** 2)
    tl.backward()
    np.testing.assert_allclose(loss, tl.item(), rtol=1e-12)
    np.testing.assert_allclose(g, tc.grad.numpy(), rtol=1e-10, atol=1e-14)
    loss, g = R.actor_loss_grad(a, c, obs)
    ta, fa = _torch_nets(torch, a, 3)
    _, fc2 = _torch_nets(torch, c, 4)
    to = torch.tensor(obs)
    tl = -torch.mean(fc2(torch.cat([to, 2 * torch.tanh(fa(to))[:, None]], 1)))
    tl.backward()
    np.testing.assert_allclose(loss, tl.item(), rtol=1e-12)
    np.testing.assert_allclose(g, ta.grad.numpy(), rtol=1e-10, atol=1e-14)


def test_reference_adam_and_polyak_match_torch():
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(3)
    p = rng.normal(size=50); g1, g2 = rng.normal(size=50), rng.normal(size=50)
    tp = torch.tensor(p.copy(), requires_grad=True)
    opt = torch.optim.Adam([tp], lr=3e-4, betas=(0.9, 0.999), eps=1e-8)
    m = v = np.zeros(50)
    for t, g in ((1, g1), (2, g2)):
        p, m, v = R.adam(p, m, v, g, t, 3e-4)
        tp.grad = torch.tensor(g); opt.step()
    np.testing.assert_allclose(p, tp.detach().numpy(), rtol=1e-10)
    np.testing.assert_allclose(R.polyak(np.ones(3), np.zeros(3), 0.005), 0.005)
    np.testing.assert_array_equal(R.polyak(np.arange(3.0), np.zeros(3), 1.0), np.arange(3.0))


def test_reference_batch_is_a_sample_without_replacement_matching_the_oracle_permutation(olib):
    """perm_index restated in Python agrees with the oracle's C perm_index on its own keys, and a batch has no repeats"""
    keys = olib.perm_index_keys(7, 3, 1, 0)
    for size in (1, 2, 5, 256, 1000, 65537):
        got = R.perm_index(np.arange(min(size, 300)), size, keys)
        want = [olib.lib.orc_perm_index(C.c_uint32(i), C.c_uint32(size), keys.ctypes.data_as(C.c_void_p)) for i in range(min(size, 300))]
        assert list(got) == want, size
        assert len(set(got)) == len(got) and got.max() < size
    idx = R.batch_indices(olib, 1, 0, 1000, 256)
    assert len(set(idx.tolist())) == 256 and idx.max() < 1000


def test_numpy_philox_matches_the_oracle_bit_for_bit(olib):
    """philox_draw_many, the reference's vectorised Philox4x32-10 for the acting and smoothing draws, against olib.philox:
    random and extreme words, counters below, at and above 2^32, seeds below, at and above 2^32, and every stream the
    DDPG kernels use"""
    rng = np.random.default_rng(12)
    words = np.concatenate([[0, 1, 0x7FFFFFFF, 0x80000000, 0xFFFFFFFF], rng.integers(0, 1 << 32, 27)]).astype(np.uint64)
    seeds = [0, 1, 0xFFFFFFFF, 1 << 32, 0x5EED_0001_0002, (1 << 64) - 1] + [int(x) for x in rng.integers(1 << 32, 1 << 63, 2)]
    counters = [0, 9, 0xFFFFFFFF, 1 << 32, (1 << 40) + 3, (1 << 64) - 1] + [int(x) for x in rng.integers(1 << 32, 1 << 63, 2)]
    for seed in seeds:
        for counter in counters:
            for stream in (R.STREAM_ACT, R.STREAM_BATCH, 7):
                got = R.philox_draw_many(seed, words, counter, stream)
                want = np.stack([R.philox_draw(olib, seed, int(w), counter, stream) for w in words])
                assert got.dtype == np.uint64 and np.array_equal(got, want), (seed, counter, stream)


def test_reference_run_loop_counts_and_warmup_ring(olib, abi):
    cfg = abi.make_ddpg_config(num_envs=3, buffer_size=40, learning_starts=30, batch_size=8, train_freq=2, policy_frequency=3,
                               max_episode_steps=7)
    a, c = rand_nets(1)
    ref = R.RefDDPG(olib, cfg, a, c)
    ref.run(10)
    assert ref.learn_steps == 0 and ref.size == 30 and ref.ptr == 30
    assert np.all(np.abs(ref.b_act[:30]) <= 2.0) and ref.b_term[:30].sum() == 3 * (10 // 7)
    np.testing.assert_allclose(np.hypot(ref.b_obs[:30, 0], ref.b_obs[:30, 1]), 1.0, rtol=1e-6)
    ref.run(20)
    # iterations 11..30 with gs = 3 it > 30, it even, size >= 8: 10 learning steps, 3 actor steps
    assert ref.learn_steps == 10 and ref.actor_steps == 3 and ref.size == 40


# ------------------------------------------------------------------ C header and ctypes mirror
def test_ddpg_header_symbols_are_exported_bound_and_disjoint_from_the_main_header(crl):
    syms = _symbols(DDPG_HEADER)
    assert len(syms) == 11 and {"crl_ddpg_create", "crl_ddpg_run", "crl_ddpg_forward_raw", "crl_ddpg_critic_loss_raw",
                                "crl_ddpg_actor_loss_raw"} <= syms
    assert not syms & _symbols(MAIN_HEADER)
    assert set(crl.DDPG_SIGNATURES) == syms
    lib = crl.load()
    for s in syms:
        assert hasattr(lib, s), s
    nm = subprocess.check_output(["nm", "-D", os.path.join(ROOT, "cleanrl.jl_b200", "libcleanrl_cuda.so")], text=True)
    for s in syms:
        assert re.search(r"\bT %s\b" % s, nm), s


def test_pure_c_file_including_the_ddpg_header_compiles_with_warnings_as_errors(tmp_path):
    src = tmp_path / "ddpg_c.c"
    src.write_text('#include "cleanrl_ddpg.h"\n#include <stdio.h>\n'
                   'int main(void) { crl_ddpg_config c = {0}; crl_ddpg_stats s = {0}; c.struct_size = (int32_t)sizeof(c);\n'
                   '  int (*f)(const crl_ddpg_config*, crl_ddpg_ctx**) = crl_ddpg_create; (void)f; (void)s;\n'
                   '  printf("%d %d %d\\n", c.struct_size, CRL_DDPG_ACTOR_PARAMS, CRL_OK); return 0; }\n')
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-c", str(src),
                           "-o", str(tmp_path / "ddpg_c.o")])


def test_ddpg_struct_layout_matches_ctypes(tmp_path, abi):
    fields_c = [f for f, _ in abi.crl_ddpg_config._fields_]
    fields_s = [f for f, _ in abi.crl_ddpg_stats._fields_]
    expr = ["sizeof(crl_ddpg_config)"] + ["offsetof(crl_ddpg_config,%s)" % f for f in fields_c] + \
           ["sizeof(crl_ddpg_stats)"] + ["offsetof(crl_ddpg_stats,%s)" % f for f in fields_s]
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "cleanrl_ddpg.h"\nint main(){%s return 0;}\n'
                   % "".join('printf("%%zu\\n", (size_t)%s);' % e for e in expr))
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    want = [C.sizeof(abi.crl_ddpg_config)] + [getattr(abi.crl_ddpg_config, f).offset for f in fields_c] + \
           [C.sizeof(abi.crl_ddpg_stats)] + [getattr(abi.crl_ddpg_stats, f).offset for f in fields_s]
    assert got == want


# ------------------------------------------------------------------ validation and the no-GPU path
BAD_CONFIGS = [
    (dict(batch_size=0), b"batch_size"), (dict(batch_size=257), b"batch_size"),
    (dict(num_envs=8, buffer_size=7), b"buffer_size"), (dict(num_envs=0), b"num_envs"),
    (dict(train_freq=0), b"train_freq"), (dict(policy_frequency=0), b"policy_frequency"),
    (dict(max_episode_steps=0), b"max_episode_steps"),
    (dict(tau=0.0), b"tau"), (dict(tau=1.5), b"tau"), (dict(tau=float("nan")), b"tau"),
]


@pytest.mark.parametrize("kw,msg", BAD_CONFIGS)
def test_invalid_ddpg_config_is_rejected_before_device_work(crl, abi, kw, msg):
    lib = crl.load()
    h = C.c_void_p()
    cfg = abi.make_ddpg_config(**kw)
    assert lib.crl_ddpg_create(C.byref(cfg), C.byref(h)) == abi.CRL_ERR_INVALID
    assert not h.value and msg in lib.crl_last_error()
    cfg = abi.make_ddpg_config()
    cfg.struct_size -= 8
    assert lib.crl_ddpg_create(C.byref(cfg), C.byref(h)) == abi.CRL_ERR_INVALID


def test_ddpg_has_no_cpu_fallback_without_a_gpu(crl, abi):
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a GPU is visible")
    except ImportError:
        pass
    lib = crl.load()
    h = C.c_void_p()
    cfg = abi.make_ddpg_config()
    assert lib.crl_ddpg_create(C.byref(cfg), C.byref(h)) == abi.CRL_ERR_CUDA
    assert not h.value and len(lib.crl_last_error()) > 0
    from cleanrl_jl_b200.ddpg_algo import DDPGHandle
    with pytest.raises(crl.CleanRLCudaError):
        DDPGHandle(cfg)


# ------------------------------------------------------------------ host config and CLI
def test_ddpg_config_defaults_and_argparse():
    from cleanrl_jl_b200 import DDPGConfig, argparse_struct
    c = DDPGConfig()
    assert (c.buffer_size, c.learning_starts, c.batch_size, c.gamma, c.tau, c.lr, c.exploration_noise, c.policy_frequency,
            c.train_freq, c.num_envs, c.seed, c.max_steps) == (1_000_000, 25_000, 256, 0.99, 0.005, 3e-4, 0.1, 2, 1, 1, 1, 200)
    c = argparse_struct(DDPGConfig(), ["--num_envs", "64", "--tau", "0.01", "--policy_frequency", "3"])
    assert isinstance(c, DDPGConfig) and (c.num_envs, c.tau, c.policy_frequency) == (64, 0.01, 3)
    assert c.batch_size == 256


def test_ddpg_init_params_are_glorot_with_zero_biases():
    from cleanrl_jl_b200.ddpg_algo import init_ddpg_params
    a, c = init_ddpg_params(3)
    assert a.size == R.ACTOR_P and c.size == R.CRITIC_P and a.dtype == np.float32
    for p, arrays, d_in in ((a, R.ACTOR_ARRAYS, 3), (c, R.CRITIC_ARRAYS, 4)):
        for (name, s, e), (fi, fo) in zip(arrays[::2], ((d_in, 64), (64, 64), (64, 1))):
            assert np.abs(p[s:e]).max() <= np.sqrt(6.0 / (fi + fo)) and np.abs(p[s:e]).max() > 0
        for name, s, e in arrays[1::2]:
            assert not p[s:e].any()


def test_cli_lists_ddpg_and_its_options():
    run = lambda *a: subprocess.run([sys.executable, "-m", "cleanrl_jl_b200", *a], cwd=ROOT, capture_output=True, text=True, timeout=300)
    p = run()
    assert p.returncode == 2 and "{a2c,dqn,ppo}" in p.stderr and "{ddpg}" in p.stderr
    p = run("ddpg", "--help")
    assert p.returncode == 0
    for field in ("--buffer_size", "--learning_starts", "--batch_size", "--tau", "--exploration_noise", "--policy_frequency",
                  "--train_freq", "--num_envs"):
        assert field in p.stdout, field
