"""C51 (include/cleanrl_c51.h) without a GPU: the Float64 reference against torch autograd of CleanRL's c51.py expressions
on edge batches, the atoms against torch.linspace, the run-loop counts, the header, the ctypes mirror, the config and
the CLI."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import c51_reference as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "cleanrl_c51.h")
F = np.float32
KINDS = ("mixed", "terminal", "clamped", "integral", "saturated", "tie", "gamma0", "gamma1")


def edge_batch(kind, B, seed):
    """(q, tgt, state, action, reward, next_state, terminal, gamma) of one batch kind:
      mixed      random actions and rewards in {0, 1}, 20 % terminal, gamma 0.99
      terminal   every sample terminal: tz = r for every atom
      clamped    rewards of +-150 and +-99: tz beyond v_max and below v_min
      integral   reward 0 or 2 with gamma 1 and no terminal, or reward 0 and terminal: every b_j is an integer, with b = 0
                 and b = 100 among them (the l == u rule)
      saturated  the head scaled by 40: pmfs far below 1e-5 (the clamp is active) and none within 5 % of either bound
      tie        the head's rows of action 1 equal those of action 0 in both nets: equal pmfs, argmax -> action 0
      gamma0     gamma 0 (tz = r), gamma1 gamma 1 without terminals"""
    from cleanrl_jl_b200.c51_algo import init_c51_params
    rng = np.random.default_rng(seed)
    q, tgt = init_c51_params(seed), init_c51_params(seed + 1000)
    for p in (q, tgt):
        p[R.ARRAYS[4][1]:] *= 8.0                      # a head with some spread: pmfs away from uniform
    s = rng.uniform(-2, 2, (B, 4)).astype(F)
    s2 = rng.uniform(-2, 2, (B, 4)).astype(F)
    a = rng.integers(0, 2, B).astype(np.int32)
    r = rng.integers(0, 2, B).astype(F)
    term = (rng.random(B) < 0.2).astype(np.uint8)
    gamma = 0.99
    if kind == "terminal":
        term[:] = 1
    elif kind == "clamped":
        r = rng.choice(np.array([150.0, -150.0, 99.0, -99.0], F), B)
    elif kind == "integral":
        gamma = 1.0
        r = rng.choice(np.array([0.0, 2.0], F), B)
        term = (rng.random(B) < 0.3).astype(np.uint8)
        r[term == 1] = 0.0
    elif kind == "saturated":
        for p in (q, tgt):
            p[R.ARRAYS[4][1]:] *= 40.0
    elif kind == "tie":
        for p in (q, tgt):
            W3 = p[R.ARRAYS[4][1]:R.ARRAYS[4][2]].reshape(R.H2, R.O)      # column-major (202 x 84): row k = column k
            W3[:, R.ATOMS:] = W3[:, :R.ATOMS]
            b3 = p[R.ARRAYS[5][1]:]
            b3[R.ATOMS:] = b3[:R.ATOMS]
    elif kind == "gamma0":
        gamma = 0.0
    elif kind == "gamma1":
        gamma, term[:] = 1.0, 0
    else:
        assert kind == "mixed", kind
    return q, tgt, s, a, r, s2, term, gamma


def torch_c51(torch, q, tgt, s, a, r, s2, term, gamma, v_min=-100.0, v_max=100.0, dtype=None):
    """CleanRL's c51.py learning step on these rows: the target pmfs in Float32 exactly as c51.py computes them, then
    the loss and its gradient by autograd in `dtype` (Float64 by default) from those target pmfs"""
    import torch.nn as nn
    dtype = dtype or torch.float64
    n_atoms = 101

    def qnet(p, dt):
        net = nn.Sequential(nn.Linear(4, 120), nn.ReLU(), nn.Linear(120, 84), nn.ReLU(), nn.Linear(84, 2 * n_atoms)).to(dt)
        W1, b1, W2, b2, W3, b3 = R.unpack(p)
        with torch.no_grad():
            for lin, W, b in zip((net[0], net[2], net[4]), (W1, W2, W3), (b1, b2, b3)):
                lin.weight.copy_(torch.from_numpy(W)); lin.bias.copy_(torch.from_numpy(b))
        return net

    def get_action(net, x, atoms_, action=None):
        logits = net(x)
        pmfs = torch.softmax(logits.view(len(x), 2, n_atoms), dim=2)
        q_values = (pmfs * atoms_).sum(2)
        if action is None:
            action = torch.argmax(q_values, 1)
        return action, pmfs[torch.arange(len(x)), action]

    atoms32 = torch.from_numpy(R.atoms(v_min, v_max))
    target_network = qnet(tgt, torch.float32)
    rewards, dones = torch.from_numpy(r)[:, None], torch.from_numpy(term.astype(F))[:, None]
    with torch.no_grad():
        _, next_pmfs = get_action(target_network, torch.from_numpy(s2), atoms32)
        next_atoms = rewards + gamma * atoms32 * (1 - dones)
        delta_z = atoms32[1] - atoms32[0]
        tz = next_atoms.clamp(v_min, v_max)
        b = (tz - v_min) / delta_z
        l = b.floor().clamp(0, n_atoms - 1)
        u = b.ceil().clamp(0, n_atoms - 1)
        d_m_l = (u + (l == u).float() - b) * next_pmfs
        d_m_u = (b - l) * next_pmfs
        target_pmfs = torch.zeros_like(next_pmfs)
        for i in range(target_pmfs.size(0)):
            target_pmfs[i].index_add_(0, l[i].long(), d_m_l[i])
            target_pmfs[i].index_add_(0, u[i].long(), d_m_u[i])
    q_network = qnet(q, dtype)
    _, old_pmfs = get_action(q_network, torch.from_numpy(s).to(dtype), atoms32.to(dtype), torch.from_numpy(a.astype(np.int64)))
    loss = (-(target_pmfs.to(dtype) * old_pmfs.clamp(min=1e-5, max=1 - 1e-5).log()).sum(-1)).mean()
    q_network.zero_grad()
    loss.backward()
    g = R.pack(*[x.grad.detach().numpy().astype(np.float64) for lin in (q_network[0], q_network[2], q_network[4])
                 for x in (lin.weight, lin.bias)])
    return (float(loss.detach()), g, next_pmfs.numpy(), target_pmfs.numpy(), (b.numpy(), l.numpy(), u.numpy()), q_network,
            old_pmfs.detach().numpy())


@pytest.mark.parametrize("kind", KINDS)
def test_reference_matches_cleanrl_c51_in_torch(kind):
    """the projection bit for bit against c51.py in Float32 (same inputs: the target pmfs torch computed), the loss and
    the gradient against torch autograd in Float64 at rtol 1e-9, on every batch kind"""
    torch = pytest.importorskip("torch")
    B = 37
    q, tgt, s, a, r, s2, term, gamma = edge_batch(kind, B, 5)
    loss_t, g_t, pn32, m32, (b_t, l_t, u_t), _, old = torch_c51(torch, q, tgt, s, a, r, s2, term, gamma)
    b, l, u, _, _ = R.project_bins(r, term, gamma, -100.0, 100.0)
    np.testing.assert_array_equal(b, b_t)
    np.testing.assert_array_equal(l, l_t.astype(np.int64))
    np.testing.assert_array_equal(u, u_t.astype(np.int64))
    np.testing.assert_array_equal(R.project(r, term, pn32, gamma, -100.0, 100.0), m32)
    # the reference's Float64 masses, from its own Float64 target pmfs, against torch's Float32 ones
    loss, g, m, _, gap = R.loss_grad(q, tgt, s, a, r, s2, term, gamma, -100.0, 100.0)
    np.testing.assert_allclose(m, m32, rtol=1e-5, atol=1e-7)
    # loss and gradient from the same masses
    loss_m, g_m = torch_loss_from_masses(torch, q, s, a, m)
    _, g_ref = loss_grad_from_masses(q, s, a, m)
    assert abs(loss_m - loss) <= 1e-9 * abs(loss)
    np.testing.assert_allclose(g_ref, g_m, rtol=1e-9, atol=1e-12 * np.abs(g_m).max())
    np.testing.assert_allclose(g, g_m, rtol=1e-9, atol=1e-12 * np.abs(g_m).max())
    if kind == "integral":
        assert (b == np.round(b)).all() and (l == u).any() and (b == 0).any() and (b == 100).any()
    if kind == "clamped":
        tz_over = r[:, None] + F(gamma) * R.atoms(-100, 100) * (1 - term[:, None].astype(F))
        assert (tz_over > 100).any() and (tz_over < -100).any()
    if kind == "saturated":
        assert (old < 1e-5).any()
        ratio = old / 1e-5
        assert not ((ratio > 0.95) & (ratio < 1.05)).any() and not (np.abs(old - (1 - 1e-5)) < 5e-7).any()
    if kind == "tie":
        assert gap == 0.0
        pm, qv, ga = R.get_action(tgt, s2, R.atoms(-100, 100))
        assert (ga == 0).all() and np.array_equal(pm[:, 0], pm[:, 1])
    if kind == "terminal":
        assert (l == l[:, :1]).all() and (u == u[:, :1]).all()


def loss_grad_from_masses(q, s, a, m):
    """the reference's loss and gradient with the masses given (R.loss_grad's second half)"""
    B = len(a)
    logits, (x, z1, h1, z2, h2) = R.forward(q, s)
    pa = R.softmax(logits)[np.arange(B), a]
    loss = -(m * np.log(np.clip(pa, R.LO, R.HI))).sum(axis=1).mean()
    kap = (pa >= R.LO) & (pa <= R.HI)
    mk = m * kap
    dl = np.zeros((B, 2, R.ATOMS))
    dl[np.arange(B), a] = (pa * mk.sum(axis=1, keepdims=True) - mk) / B
    dl = dl.reshape(B, R.O)
    W1, b1, W2, b2, W3, b3 = R.unpack(q)
    dz2 = (dl @ W3) * (z2 > 0)
    dz1 = (dz2 @ W2) * (z1 > 0)
    return loss, R.pack(dz1.T @ x, dz1.sum(0), dz2.T @ h1, dz2.sum(0), dl.T @ h2, dl.sum(0))


def torch_loss_from_masses(torch, q, s, a, m):
    import torch.nn as nn
    net = nn.Sequential(nn.Linear(4, 120), nn.ReLU(), nn.Linear(120, 84), nn.ReLU(), nn.Linear(84, 202)).double()
    W1, b1, W2, b2, W3, b3 = R.unpack(q)
    with torch.no_grad():
        for lin, W, b in zip((net[0], net[2], net[4]), (W1, W2, W3), (b1, b2, b3)):
            lin.weight.copy_(torch.from_numpy(W)); lin.bias.copy_(torch.from_numpy(b))
    pmfs = torch.softmax(net(torch.from_numpy(s).double()).view(len(s), 2, 101), dim=2)
    old = pmfs[torch.arange(len(s)), torch.from_numpy(a.astype(np.int64))]
    loss = (-(torch.from_numpy(m) * old.clamp(min=1e-5, max=1 - 1e-5).log()).sum(-1)).mean()
    loss.backward()
    return float(loss), R.pack(*[x.grad.numpy() for lin in (net[0], net[2], net[4]) for x in (lin.weight, lin.bias)])


def test_reference_adam_matches_torch_adam_with_cleanrl_eps():
    """two steps of optim.Adam(lr, eps=0.01 / B) in Float64"""
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(3)
    p0 = rng.normal(size=50)
    g1, g2 = rng.normal(size=50) * 1e-3, rng.normal(size=50) * 1e-2
    B, lr = 128, 2.5e-4
    w = torch.tensor(p0.copy(), requires_grad=True)
    opt = torch.optim.Adam([w], lr=lr, eps=0.01 / B)
    for g in (g1, g2):
        w.grad = torch.from_numpy(g.copy())
        opt.step()
    p, m, v = p0.copy(), np.zeros(50), np.zeros(50)
    p, m, v = R.adam(p, m, v, g1, 1, lr, 0.01 / B)
    p, m, v = R.adam(p, m, v, g2, 2, lr, 0.01 / B)
    np.testing.assert_allclose(p, w.detach().numpy(), rtol=1e-13, atol=1e-15)


def test_atoms_against_torch_linspace():
    """bit for bit at the defaults. torch.linspace's Float32 arithmetic differs from the Float64 formula elsewhere: on
    the ranges below by at most one ulp of max(|v_min|, |v_max|) (half an ulp on all but one)"""
    torch = pytest.importorskip("torch")
    assert np.array_equal(R.atoms(-100.0, 100.0), torch.linspace(-100.0, 100.0, 101).numpy())
    worst = {}
    for lo, hi in ((-10.0, 10.0), (0.0, 500.0), (-1.0, 0.3), (-7.3, 123.4), (-0.5, 0.5)):
        z, t = R.atoms(lo, hi).astype(np.float64), torch.linspace(lo, hi, 101).numpy().astype(np.float64)
        worst[(lo, hi)] = np.abs(z - t).max() / np.spacing(np.float32(max(abs(lo), abs(hi))))
    assert max(worst.values()) <= 1.0 and sorted(worst.values())[-2] <= 0.5, worst


def test_closed_form_counts_match_the_reference_loop(olib, abi):
    """learn steps, target copies (off the learning grid too) and acting launches after three run calls"""
    cases = [dict(num_envs=3, buffer_size=60, learning_starts=20, batch_size=8, train_frequency=4, target_network_frequency=6),
             dict(num_envs=5, buffer_size=8, learning_starts=4, batch_size=8, train_frequency=3, target_network_frequency=2),
             dict(num_envs=2, buffer_size=400, learning_starts=10, batch_size=64, train_frequency=1, target_network_frequency=5),
             dict(num_envs=1, buffer_size=100, learning_starts=0, batch_size=4, train_frequency=37, target_network_frequency=7)]
    from cleanrl_jl_b200.c51_algo import init_c51_params
    for kw in cases:
        cfg = abi.make_c51_config(epsilon_duration=50.0, seed=2, max_episode_steps=9, **kw)
        ref = R.RefC51(olib, cfg, init_c51_params(1), tie_tol=0.0)
        chunks = (17, 40, 23)
        for c in chunks:
            ref.run(c)
        assert R.closed_form_counts(cfg, chunks) == (ref.learn_steps, ref.target_copies, ref.launches - 3 * ref.learn_steps), kw
        assert ref.learn_steps > 0 and ref.target_copies > 0
    # the first case learns on iterations 8, 12, ..., 80 (global step 3 it > 20) and copies on 12, 18, ..., 78: six
    # copies on the learning grid and six off it; every acting launch ends on a learning iteration
    assert R.closed_form_counts(abi.make_c51_config(**cases[0]), (80,)) == (19, 12, 19)


def test_epsilon_one_fills_dqns_ring(olib, abi):
    """with epsilon pinned to 1 every action is stream 3's random bit, as in DQN: the reference fills the oracle's DQN ring"""
    from oracle.oracle import OracleDQN
    from cleanrl_jl_b200.c51_algo import init_c51_params
    from cleanrl_jl_b200.dqn_algo import init_q_params
    kw = dict(num_envs=4, buffer_size=64, batch_size=16, seed=7)
    cfg = abi.make_c51_config(learning_starts=1000, start_e=1.0, end_e=1.0, max_episode_steps=20, **kw)
    ref = R.RefC51(olib, cfg, init_c51_params(1))
    o = OracleDQN(olib, abi.make_dqn_config(min_buff_size=1000, epsilon_start=1.0, epsilon_end=1.0, max_episode_steps=20, **kw))
    o.set_params(init_q_params(1)); o.reset()
    ref.run(50); o.run(50)
    b = o.read_buffer()
    for k, mine in (("state", ref.b_state), ("action", ref.b_action), ("reward", ref.b_reward), ("next_state", ref.b_next),
                    ("terminal", ref.b_term)):
        np.testing.assert_array_equal(mine, b[k], err_msg=k)
    o.close()


# ------------------------------------------------------------------ C header and ctypes mirror
def _symbols(path):
    return set(re.findall(r"CRL_API\s+int\s+(crl_\w+)\s*\(", open(path).read()))


def test_c51_header_symbols_are_bound_and_disjoint_from_the_other_tables():
    from cleanrl_jl_b200 import _lib as crl
    syms = _symbols(HEADER)
    assert syms == {"crl_c51_create", "crl_c51_destroy", "crl_c51_set_params", "crl_c51_get_params", "crl_c51_get_adam_state",
                    "crl_c51_reset", "crl_c51_run", "crl_c51_read_buffer", "crl_c51_forward_raw", "crl_c51_loss_raw"}
    assert set(crl.C51_SIGNATURES) == syms
    others = set(crl.SIGNATURES) | set(crl.DDPG_SIGNATURES) | set(crl.TD3_SIGNATURES) | set(crl.SAC_SIGNATURES)
    assert not syms & others
    for h in ("cleanrl_cuda.h", "cleanrl_ddpg.h", "cleanrl_td3.h", "cleanrl_sac.h"):
        assert not syms & _symbols(os.path.join(ROOT, "include", h)), h


def test_c51_header_constants_and_launch_count():
    from cleanrl_jl_b200 import _abi
    src = open(HEADER).read()
    assert re.search(r"#define CRL_C51_ATOMS 101\b", src) and re.search(r"#define CRL_C51_PARAMS 27934\b", src)
    assert "acting launches + 3 learn_steps" in src
    assert _abi.CRL_C51_ATOMS == 101 and _abi.CRL_C51_PARAMS == 27934 == R.P
    assert re.search(r"#define CRL_VERSION 100\b", open(os.path.join(ROOT, "include", "cleanrl_cuda.h")).read())


def test_pure_c_file_including_the_c51_header_compiles_with_warnings_as_errors(tmp_path):
    src = tmp_path / "c51_c.c"
    src.write_text('#include "cleanrl_c51.h"\n#include <stdio.h>\n'
                   'int main(void) { crl_c51_config c = {0}; crl_c51_stats s = {0}; c.struct_size = (int32_t)sizeof(c);\n'
                   '  int (*f)(const crl_c51_config*, crl_c51_ctx**) = crl_c51_create; (void)f; (void)s;\n'
                   '  printf("%d %d %d\\n", c.struct_size, CRL_C51_PARAMS, CRL_OK); return 0; }\n')
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), "-c", str(src),
                           "-o", str(tmp_path / "c51_c.o")])


def test_c51_struct_layout_matches_ctypes(tmp_path, abi):
    import ctypes as C
    fields_c = [f for f, _ in abi.crl_c51_config._fields_]
    fields_s = [f for f, _ in abi.crl_c51_stats._fields_]
    expr = ["sizeof(crl_c51_config)"] + ["offsetof(crl_c51_config,%s)" % f for f in fields_c] + \
           ["sizeof(crl_c51_stats)"] + ["offsetof(crl_c51_stats,%s)" % f for f in fields_s]
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "cleanrl_c51.h"\nint main(){%s return 0;}\n'
                   % "".join('printf("%%zu\\n", (size_t)%s);' % e for e in expr))
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    want = [C.sizeof(abi.crl_c51_config)] + [getattr(abi.crl_c51_config, f).offset for f in fields_c] + \
           [C.sizeof(abi.crl_c51_stats)] + [getattr(abi.crl_c51_stats, f).offset for f in fields_s]
    assert got == want


# ------------------------------------------------------------------ config and CLI
def test_c51_config_has_cleanrls_fields_and_defaults(abi):
    from cleanrl_jl_b200 import C51Config
    from cleanrl_jl_b200.c51_algo import make_crl_c51_config
    c = C51Config()
    want = dict(total_timesteps=500_000, learning_rate=2.5e-4, n_atoms=101, v_min=-100.0, v_max=100.0, buffer_size=10_000,
                gamma=0.99, target_network_frequency=500, batch_size=128, start_e=1.0, end_e=0.05, exploration_fraction=0.5,
                learning_starts=10_000, train_frequency=10, num_envs=1, seed=1, max_steps=500)
    for k, v in want.items():
        assert getattr(c, k) == v, k
    assert hasattr(c, "log_frequency") and hasattr(c, "run_name")
    cfg = make_crl_c51_config(c)
    assert (cfg.epsilon_duration, cfg.lr, cfg.train_frequency, cfg.max_episode_steps) == (250_000.0, 2.5e-4, 10, 500)
    d = abi.make_c51_config()
    for f, _ in abi.crl_c51_config._fields_:
        if f not in ("struct_size", "device"):
            assert getattr(d, f) == getattr(cfg, f), f
    with pytest.raises(ValueError):
        make_crl_c51_config(C51Config(n_atoms=51))


def test_c51_usage_line_and_field_options():
    run = lambda *a: subprocess.run([sys.executable, "-m", "cleanrl_jl_b200", *a], cwd=ROOT, capture_output=True, text=True,
                                    timeout=300)
    p = run()
    assert p.returncode == 2
    lines = p.stderr.splitlines()
    assert any("{c51}" in l for l in lines)
    for s in ("{a2c,dqn,ppo}", "{ddpg}", "{td3}", "{sac}"):
        assert any(s in l for l in lines), s
    p = run("c51", "--help")
    assert p.returncode == 0
    for field in ("--learning_rate", "--n_atoms", "--v_min", "--v_max", "--buffer_size", "--gamma", "--target_network_frequency",
                  "--batch_size", "--start_e", "--end_e", "--exploration_fraction", "--learning_starts", "--train_frequency"):
        assert field in p.stdout, field
    from cleanrl_jl_b200 import C51Config, argparse_struct
    c = argparse_struct(C51Config(), ["--v_min", "-10", "--batch_size", "64"])
    assert (c.v_min, c.batch_size, c.learning_rate) == (-10.0, 64, 2.5e-4)
