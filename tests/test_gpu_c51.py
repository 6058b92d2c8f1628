"""C51 on the GPU (include/cleanrl_c51.h): the acting kernel's forward and the learning step's three kernels against
Float64 on their own, crl_c51_run against the NumPy reference, the ring shared with DQN, determinism, the benchmark shape,
learning, and the CLI. Run with `pytest -m gpu` on a B200."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import c51_reference as R
from test_c51 import KINDS, edge_batch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F = np.float32


def dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def gpu_forward(crl, torch, params, obs, v_min=-100.0, v_max=100.0):
    n = obs.shape[0]
    q = torch.full((n, 2), float("nan"), dtype=torch.float32, device="cuda")
    act = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    pmf = torch.full((n, 2, R.ATOMS), float("nan"), dtype=torch.float32, device="cuda")
    tp, tobs = dev(torch, params), dev(torch, obs)
    crl.check(crl.load().crl_c51_forward_raw(crl.ptr(tp), crl.ptr(tobs), v_min, v_max, crl.ptr(q), crl.ptr(act), crl.ptr(pmf), n,
                                             None))
    torch.cuda.synchronize()
    return q.cpu().numpy(), act.cpu().numpy(), pmf.cpu().numpy()


def gpu_loss(crl, torch, q, tgt, s, a, r, s2, term, gamma, B=None, v_min=-100.0, v_max=100.0):
    B = len(a) if B is None else B
    g = torch.full((R.P,), float("nan"), dtype=torch.float32, device="cuda")
    m = torch.full((B, R.ATOMS), float("nan"), dtype=torch.float32, device="cuda")
    loss = torch.full((1,), float("nan"), dtype=torch.float64, device="cuda")
    t = [dev(torch, x) for x in (q, tgt, s, a, r, s2, term)]
    crl.check(crl.load().crl_c51_loss_raw(crl.ptr(t[0]), crl.ptr(t[1]), B, *[crl.ptr(x) for x in t[2:]], gamma, v_min, v_max,
                                          crl.ptr(m), crl.ptr(g), crl.ptr(loss), None))
    torch.cuda.synchronize()
    return g.cpu().numpy(), m.cpu().numpy(), float(loss.cpu().numpy()[0])


# ------------------------------------------------------------------ forward
@pytest.mark.parametrize("n", [1, 31, 32, 33, 148 * 32 + 5, 100_003])
def test_c51_forward_raw_matches_float64(crl, torch_cuda, n):
    """pmfs at rtol 2e-4 and atol 1e-6 (logits are 84-term Float32 chains after two Float32 layers; a pmf's relative
    error is about its logit's absolute one), Q at 1e-4 of sum_j p_j |z_j| plus 1e-5, and the action of every row whose
    Float64 gap |Q_1 - Q_0| is at least 1e-3 equal to the Float64 argmax"""
    from cleanrl_jl_b200.c51_algo import init_c51_params
    rng = np.random.default_rng(n)
    p = init_c51_params(7)
    p[R.ARRAYS[4][1]:] *= 8.0
    obs = rng.uniform(-2, 2, (n, 4)).astype(F)
    q, act, pmf = gpu_forward(crl, torch_cuda, p, obs)
    z = R.atoms(-100.0, 100.0)
    pm, q64, a64 = R.get_action(p, obs, z)
    np.testing.assert_allclose(pmf, pm, rtol=2e-4, atol=1e-6)
    scale = (pm * np.abs(z.astype(np.float64))).sum(axis=2)
    assert (np.abs(q - q64) <= 1e-4 * scale + 1e-5).all()
    far = np.abs(q64[:, 1] - q64[:, 0]) >= 1e-3
    assert far.mean() > 0.99
    np.testing.assert_array_equal(act[far], a64[far])
    # the kernel's own argmax of its own Q values: first maximum
    np.testing.assert_array_equal(act, (q[:, 1] > q[:, 0]).astype(np.int32))


def test_c51_forward_raw_ties_and_other_atom_ranges(crl, torch_cuda):
    """equal action heads give equal Q and action 0; the atoms follow v_min and v_max"""
    p = edge_batch("tie", 4, 3)[0]
    obs = np.random.default_rng(0).uniform(-2, 2, (97, 4)).astype(F)
    q, act, _ = gpu_forward(crl, torch_cuda, p, obs)
    assert np.array_equal(q[:, 0], q[:, 1]) and not act.any()
    q, _, pmf = gpu_forward(crl, torch_cuda, p, obs, -7.3, 123.4)
    z = R.atoms(-7.3, 123.4).astype(np.float64)
    np.testing.assert_allclose(q, (pmf.astype(np.float64) * z).sum(axis=2), rtol=1e-5, atol=1e-5)


# ------------------------------------------------------------------ learning step
def assert_close_per_array(g, ref, rtol, atol_frac, what):
    for name, s, e in R.ARRAYS:
        a, b = g[s:e], ref[s:e]
        np.testing.assert_allclose(a, b, rtol=rtol, atol=atol_frac * max(np.abs(b).max(), 1e-30), err_msg="%s %s" % (what, name))


@pytest.mark.parametrize("B", [1, 15, 16, 17, 120, 127, 128])
@pytest.mark.parametrize("kind", KINDS)
def test_c51_loss_raw_matches_float64(crl, torch_cuda, kind, B):
    """masses with the same bins (the index arithmetic is the header's Float32 in both) at rtol 1e-4 and atol 1e-6
    (p' is a Float32 pmf); every gradient array at rtol 1e-3 and an atol of 1e-4 of its largest entry (the logit
    gradient p_i sum m - m_i cancels where the pmf is close to the masses); the loss at rtol 1e-5"""
    q, tgt, s, a, r, s2, term, gamma = edge_batch(kind, B, 11 + B)
    g, m, loss = gpu_loss(crl, torch_cuda, q, tgt, s, a, r, s2, term, gamma)
    loss64, g64, m64, _, gap = R.loss_grad(q, tgt, s, a, r, s2, term, gamma, -100.0, 100.0)
    assert gap == 0.0 if kind == "tie" else gap > 1e-3, gap       # the target's greedy action is determined
    _, l, u, _, _ = R.project_bins(r, term, gamma, -100.0, 100.0)
    support = np.zeros((B, R.ATOMS), bool)
    for i in range(B):
        support[i, l[i]] = support[i, u[i]] = True
    np.testing.assert_array_equal(m[~support], 0.0)
    np.testing.assert_allclose(m, m64, rtol=1e-4, atol=1e-6)
    assert abs(loss - loss64) <= 1e-5 * abs(loss64)
    assert_close_per_array(g, g64, 1e-3, 1e-4, kind)


@pytest.mark.parametrize("B", [1, 17, 128])
def test_c51_loss_raw_reads_nothing_past_row_B(crl, torch_cuda, B):
    q, tgt, s, a, r, s2, term, gamma = edge_batch("mixed", B, 2)
    ref = gpu_loss(crl, torch_cuda, q, tgt, s, a, r, s2, term, gamma)
    pad = 128 + 16 - B

    def poison(x, v):
        return np.concatenate([x, np.full((pad,) + x.shape[1:], v, x.dtype)])
    got = gpu_loss(crl, torch_cuda, q, tgt, poison(s, np.nan), poison(a, 1 << 20), poison(r, np.nan), poison(s2, np.nan),
                   poison(term, 255), gamma, B=B)
    np.testing.assert_array_equal(got[0], ref[0])
    np.testing.assert_array_equal(got[1], ref[1])
    assert got[2] == ref[2]


# ------------------------------------------------------------------ run loop against the reference
def compare_run(olib, abi, cfg, params, chunks):
    """crl_c51_run and RefC51 over the same calls. Exact: counters, epsilon, launches, per-call episode statistics, ring
    actions, rewards and terminals. Env states: rtol 1e-4 and atol 2e-6 (chained CartPole steps, as the DQN tests).
    Parameters and target: every entry within 2 lr per learning step of the Float64 one (an Adam step moves an entry by
    at most about lr), and 99 % of each array within rtol 1e-3 and 1e-4 of its largest entry: Adam normalises small
    gradients, so an entry whose gradient is rounding noise may take a different step. Loss and q_values at rtol 1e-3
    plus 1e-4. Near-ties (Float64 gap below 1e-3) adopt the library's action; they stay below 2 % of the greedy choices
    (the most is 5 of 332, in the batch-size-gate run, whose untrained net's two Qs are close).
    The target net's greedy choice at s' cannot be adopted (the kernels do not report it): the smallest Float64 gap
    between its two expected Qs over every sampled s' must stay above 1e-5, where the Float32 Q's rounding (an ulp of
    100 is 7.6e-6) could flip it. The smallest such gaps of these runs are 1.4e-5 to 7.7e-4."""
    from cleanrl_jl_b200.c51_algo import C51Handle
    h = C51Handle(cfg)
    h.set_params(params); h.reset()
    ref = R.RefC51(olib, cfg, params)
    N, C, lr = cfg.num_envs, cfg.buffer_size, cfg.lr
    for chunk in chunks:
        assert chunk * N <= C, "the adopted actions are read from the ring"
        st = h.run(chunk)
        b = h.read_buffer()
        ref.run(chunk, b["action"])
        assert (st.iterations, st.learn_steps, st.target_copies) == (ref.it, ref.learn_steps, ref.target_copies)
        assert st.kernel_launches == ref.launches
        assert st.epsilon == ref.eps
        assert (st.episodes, st.sum_return, st.sum_length) == (ref.episodes, ref.sum_return, ref.sum_length)
        assert (b["size"], b["ptr"]) == (ref.size, ref.ptr)
        n = b["size"]
        np.testing.assert_array_equal(b["action"][:n], ref.b_action[:n])
        np.testing.assert_array_equal(b["reward"][:n], ref.b_reward[:n])
        np.testing.assert_array_equal(b["terminal"][:n], ref.b_term[:n])
        np.testing.assert_allclose(b["state"][:n], ref.b_state[:n], rtol=1e-4, atol=2e-6)
        np.testing.assert_allclose(b["next_state"][:n], ref.b_next[:n], rtol=1e-4, atol=2e-6)
        qh, th = h.get_params()
        for got, want in ((qh, ref.q), (th, ref.tgt)):
            assert np.abs(got - want).max() <= 2 * lr * max(ref.learn_steps, 1) + 1e-6
            for name, s, e in R.ARRAYS:
                bad = ~np.isclose(got[s:e], want[s:e], rtol=1e-3, atol=1e-4 * np.abs(want[s:e]).max())
                assert bad.mean() <= 0.01, (name, int(bad.sum()), e - s)
        if ref.learn_steps:
            assert abs(st.loss - ref.loss) <= 1e-3 * abs(ref.loss) + 1e-4
            assert abs(st.q_values - ref.q_values) <= 1e-3 * abs(ref.q_values) + 1e-4
            assert ref.target_gap > 1e-5, ref.target_gap
    assert ref.adopted <= 0.02 * max(ref.greedy_decisions, 1), (ref.adopted, ref.greedy_decisions)
    learn, copies, acting = R.closed_form_counts(cfg, chunks)
    assert (learn, copies, acting + 3 * learn) == (ref.learn_steps, ref.target_copies, ref.launches)
    m, v, bp = h.get_adam_state()
    np.testing.assert_allclose(bp, (0.9 ** (ref.learn_steps + 1), 0.999 ** (ref.learn_steps + 1)), rtol=1e-12)
    h.close()
    return ref


RUNS = {   # name: (config fields, iteration chunks)
    "one_env": (dict(num_envs=1, buffer_size=2000, learning_starts=200, batch_size=32, train_frequency=4, target_network_frequency=50), (200, 250, 150)),
    "33_envs": (dict(num_envs=33, buffer_size=4096, learning_starts=330, batch_size=64, train_frequency=2, target_network_frequency=10), (30, 40, 30)),
    "ragged_last_cta": (dict(num_envs=100, buffer_size=8192, learning_starts=1000, batch_size=128, train_frequency=3, target_network_frequency=9), (20, 30, 30)),
    "copies_off_the_grid": (dict(num_envs=8, buffer_size=512, learning_starts=64, batch_size=32, train_frequency=4, target_network_frequency=6), (48, 52, 50)),
    "ring_below_two_vector_steps": (dict(num_envs=100, buffer_size=150, learning_starts=100, batch_size=128, train_frequency=3, target_network_frequency=9), (1,) * 60),
    "batch_size_gate": (dict(num_envs=4, buffer_size=512, learning_starts=8, batch_size=100, train_frequency=2, target_network_frequency=10), (20, 30, 96)),
    "wrapped_1M_ring": (dict(num_envs=4096, buffer_size=1_000_000, learning_starts=900_000, batch_size=128, train_frequency=10, target_network_frequency=30), (120, 130, 50)),
}


@pytest.mark.parametrize("name", sorted(RUNS))
def test_c51_run_matches_reference(olib, abi, crl, torch_cuda, name):
    from cleanrl_jl_b200.c51_algo import init_c51_params
    kw, chunks = RUNS[name]
    cfg = abi.make_c51_config(epsilon_duration=40.0 * kw["num_envs"] * sum(chunks) / 50, end_e=0.05, seed=9,
                              max_episode_steps=60, **kw)
    ref = compare_run(olib, abi, cfg, init_c51_params(4), chunks)
    assert ref.learn_steps >= 3 and ref.target_copies >= 2
    if name == "wrapped_1M_ring":
        assert ref.it * cfg.num_envs > cfg.buffer_size and ref.size == cfg.buffer_size


# ------------------------------------------------------------------ ring, determinism, benchmark shape
def test_c51_fills_dqns_ring_with_epsilon_one(abi, crl, torch_cuda):
    """with epsilon pinned to 1, C51 and DQN fill bit-identical rings, learning steps included"""
    from cleanrl_jl_b200.c51_algo import C51Handle, init_c51_params
    from cleanrl_jl_b200.dqn_algo import DQNHandle, init_q_params
    kw = dict(num_envs=64, buffer_size=4096, batch_size=64, seed=5, max_episode_steps=500)
    c = C51Handle(abi.make_c51_config(learning_starts=640, train_frequency=4, target_network_frequency=8, start_e=1.0, end_e=1.0, **kw))
    d = DQNHandle(abi.make_dqn_config(min_buff_size=640, train_freq=4, target_net_freq=8, epsilon_start=1.0, epsilon_end=1.0, **kw))
    c.set_params(init_c51_params(1)); d.set_params(init_q_params(1))
    c.reset(); d.reset()
    sc, sd = c.run(150), d.run(150)
    assert sc.learn_steps == sd.learn_steps > 0
    bc, bd = c.read_buffer(), d.read_buffer()
    for k in ("state", "action", "reward", "next_state", "terminal", "size", "ptr"):
        assert np.array_equal(bc[k], bd[k]), k
    assert (sc.episodes, sc.sum_return, sc.sum_length) == (sd.episodes, sd.sum_return, sd.sum_length)
    c.close(); d.close()


def snapshot(h, stats):
    q, t = h.get_params()
    m, v, bp = h.get_adam_state()
    b = h.read_buffer()
    return [q, t, m, v, bp] + [b[k] for k in ("state", "action", "reward", "next_state", "terminal")] + \
           [np.array([stats.loss, stats.q_values, stats.learn_steps, stats.target_copies, stats.kernel_launches, b["size"], b["ptr"]])]


def test_c51_runs_are_deterministic(abi, crl, torch_cuda):
    from cleanrl_jl_b200.c51_algo import C51Handle, init_c51_params
    cfg = abi.make_c51_config(num_envs=256, buffer_size=20_000, learning_starts=2000, batch_size=128, train_frequency=2,
                              target_network_frequency=6, epsilon_duration=20_000.0, seed=3)
    snaps = []
    for _ in range(2):
        h = C51Handle(cfg)
        h.set_params(init_c51_params(2)); h.reset()
        snaps.append(snapshot(h, h.run(60)))
        h.close()
    for a, b in zip(*snaps):
        np.testing.assert_array_equal(a, b)


def test_c51_benchmark_shape_one_call_equals_split_calls(abi, crl, torch_cuda):
    """4,096 envs, a 2^20 ring, batch 128, learning every 10 iterations after 10,000 global steps: one call of 300
    iterations and the same split into three calls give the same bits, launch count and summed episode statistics. The
    calls end on learning iterations, where an acting launch ends anyway; a call ending elsewhere ends a launch early,
    which the closed form counts."""
    from cleanrl_jl_b200.c51_algo import C51Handle, init_c51_params
    cfg = abi.make_c51_config(num_envs=4096, buffer_size=1 << 20, learning_starts=10_000, batch_size=128, train_frequency=10,
                              target_network_frequency=500, epsilon_duration=250_000.0, seed=1)
    out = []
    for chunks in ((300,), (100, 20, 180)):
        h = C51Handle(cfg)
        h.set_params(init_c51_params(1)); h.reset()
        ep = [0, 0.0, 0.0]
        for c in chunks:
            st = h.run(c)
            ep[0] += st.episodes; ep[1] += st.sum_return; ep[2] += st.sum_length
        out.append((snapshot(h, st), ep))
        h.close()
    (a, ea), (b, eb) = out
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y)
    assert ea == eb and ea[0] > 0
    assert a[-1][2] == len(range(10, 301, 10)) and a[-1][3] == 0      # 30 learning steps; no copy before iteration 500
    learn, _, acting = R.closed_form_counts(cfg, (300,))
    assert a[-1][4] == acting + 3 * learn == 30 + 90
    assert R.closed_form_counts(cfg, (101, 17, 182))[2] == acting + 2


def test_c51_config_errors(abi, crl, torch_cuda):
    from cleanrl_jl_b200 import _lib as L
    from cleanrl_jl_b200.c51_algo import C51Handle
    bad = [dict(v_min=1.0, v_max=1.0), dict(v_max=float("inf")), dict(gamma=1.5), dict(lr=0.0), dict(lr=float("nan")),
           dict(batch_size=129), dict(batch_size=0), dict(train_frequency=0), dict(target_network_frequency=0),
           dict(buffer_size=3, num_envs=4), dict(epsilon_duration=0.0)]
    for kw in bad:
        with pytest.raises(L.CleanRLCudaError):
            C51Handle(abi.make_c51_config(**kw))


# ------------------------------------------------------------------ learning and the CLI
def test_c51_learns_cartpole(torch_cuda, tmp_path):
    """c51() with CleanRL's defaults and one env for CleanRL's 500,000 steps. Random play returns about 22; the mean of
    the last ten logged episode means must exceed 150. Measured with seed 1 on one NVIDIA B200 (1000 W power limit):
    500.0, CartPole-v1's limit, in 13.6 s."""
    from cleanrl_jl_b200 import C51Config, c51
    from cleanrl_jl_b200 import logger as Logger
    lg = Logger.make_logger("c51", to_terminal=False, to_tensorboard=False, to_json=True, log_dir=str(tmp_path))
    res = c51(C51Config(seed=1), logger=lg)
    lg.close()
    assert res["global_step"] == 500_000 and res["learn_steps"] == (500_000 - 10_000) // 10
    mean = float(np.mean(res["recent_returns"]))
    print("c51 CartPole: mean of the last ten logged episode returns %.1f" % mean)
    assert mean > 150.0, res["recent_returns"]


def test_c51_cli_runs(torch_cuda, tmp_path):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "cleanrl_jl_b200.py"), "c51", "--num_envs", "16", "--total_timesteps",
                        "8000", "--learning_starts", "500", "--buffer_size", "4096"], cwd=str(tmp_path), capture_output=True,
                       text=True, timeout=300)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    res = json.loads(p.stdout.strip().splitlines()[-1])
    assert res["algorithm"] == "c51" and res["global_step"] == 8000 and res["learn_steps"] > 0 and res["steps_per_sec"] > 0
