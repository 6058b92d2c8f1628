"""DQN kernels on their own and the DQN run loop at its schedule edges (GPU).

* The acting kernel's forward pass (crl_dqn_forward_raw) against float64 NumPy and the oracle, and its greedy choice
  against the argmax of those Q-values.
* The learning step's loss and gradient (crl_dqn_loss_raw: dqn_learn_fwd_kernel + dqn_learn_upd_kernel) per parameter
  array against float64 NumPy and orc_dqn_loss_raw, at every 16-sample CTA boundary of the batch and at edge batches.
* crl_dqn_run against the oracle on shared Philox streams where the host loop packs its launches differently: learning
  every iteration, several acting launches per learning step, a target copy off the learning grid, truncated episodes,
  rings smaller than two vector steps, the batch-size gate and greedy acting with exact ties.
Run with `pytest -m gpu` on a B200."""
import numpy as np
import pytest

from oracle.oracle import OracleDQN
from test_dqn import _np_forward, _np_loss_grad, assert_grad_close, edge_batch, relu0_zero_indices

pytestmark = pytest.mark.gpu
F = np.float32
P = 10934


def dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def gpu_forward(crl, torch, params, obs):
    q = torch.full((obs.shape[0], 2), float("nan"), dtype=torch.float32, device="cuda")
    tp, tobs = dev(torch, params), dev(torch, obs)      # held until the kernel has run
    crl.check(crl.load().crl_dqn_forward_raw(crl.ptr(tp), crl.ptr(tobs), crl.ptr(q), obs.shape[0], None))
    torch.cuda.synchronize()
    return q.cpu().numpy()


def gpu_loss(crl, torch, q, tgt, s, a, r, s2, term, gamma, B=None):
    B = len(a) if B is None else B
    g = torch.full((P,), float("nan"), dtype=torch.float32, device="cuda")
    loss = torch.full((1,), float("nan"), dtype=torch.float64, device="cuda")
    t = [dev(torch, x) for x in (q, tgt, s, a, r, s2, term)]
    crl.check(crl.load().crl_dqn_loss_raw(crl.ptr(t[0]), crl.ptr(t[1]), B, *[crl.ptr(x) for x in t[2:]], gamma,
                                          crl.ptr(g), crl.ptr(loss), None))
    torch.cuda.synchronize()
    return g.cpu().numpy(), float(loss.cpu().numpy()[0])


def head_magnitude(params, obs):
    """per (sample, output): sum of |summands| of the head, |W3| |h2| + |b3|, in float64 (the atol scale of a Q-value)"""
    _, (_, _, W3, _, h2, _, _) = _np_forward(params, obs.astype(np.float64))
    return np.abs(h2) @ np.abs(W3).T + np.abs(params[10932:].astype(np.float64))


# ------------------------------------------------------------------ forward
@pytest.mark.parametrize("n", [1, 31, 32, 33, 148 * 32 + 5, 100_003])
def test_dqn_forward_raw_matches_float64_and_oracle(crl, olib, abi, torch_cuda, n):
    """Q-values of the acting kernel's forward pass (32 samples per CTA, a partial last CTA) at rtol 1e-5 and an atol of
    1e-6 of the summed magnitudes of the head's summands (an 84-term fp32 chain after two fp32 layers; the oracle
    reaches 0.16 of this bound at n = 100,003)"""
    from cleanrl_jl_b200.dqn_algo import init_q_params
    rng = np.random.default_rng(n)
    p = init_q_params(7)
    p[480:600] = rng.normal(0, 0.2, 120); p[10680:10764] = rng.normal(0, 0.2, 84); p[10932:] = (0.3, -0.2)
    obs = (rng.uniform(-1, 1, (n, 4)) * 10 * rng.random((n, 1))).astype(F)      # |x| up to 10
    obs[::7] = 0.0
    qg = gpu_forward(crl, torch_cuda, p, obs)
    ref, _ = _np_forward(p, obs.astype(np.float64))
    atol = 1e-6 * head_magnitude(p, obs)
    assert np.all(np.abs(qg - ref) <= 1e-5 * np.abs(ref) + atol), np.abs(qg - ref).max()
    o = OracleDQN(olib, abi.make_dqn_config())
    qo = o.forward(p, obs)
    o.close()
    assert np.all(np.abs(qg - qo) <= 1e-5 * np.abs(qo) + atol), np.abs(qg - qo).max()
    if n > 1000:
        assert np.ptp(qg[:, 1] - qg[:, 0]) > 0.1       # both actions win somewhere


def test_dqn_forward_raw_errors(crl, torch_cuda):
    lib = crl.load()
    t = torch_cuda.zeros(P + 6, device="cuda")
    assert lib.crl_dqn_forward_raw(crl.ptr(t), crl.ptr(t), crl.ptr(t), 0, None) == 0
    assert lib.crl_dqn_forward_raw(crl.ptr(t), crl.ptr(t), crl.ptr(t), -1, None) == -1
    assert lib.crl_dqn_forward_raw(None, crl.ptr(t), crl.ptr(t), 1, None) == -1
    assert lib.crl_dqn_forward_raw(crl.ptr(t), crl.ptr(t[1:]), crl.ptr(t), 1, None) == -1       # obs not 16-byte aligned
    for B in (0, 129):
        assert lib.crl_dqn_loss_raw(*[crl.ptr(t)] * 2, B, *[crl.ptr(t)] * 5, 0.99, crl.ptr(t), crl.ptr(t), None) == -1
    assert b"B must be" in lib.crl_last_error()


def test_greedy_actions_are_the_argmax_of_the_forward_pass(crl, abi, torch_cuda):
    """epsilon = 0 and no learning step: every action the acting kernel recorded is the first maximum of the Q-values
    crl_dqn_forward_raw computes for the recorded state"""
    from cleanrl_jl_b200.dqn_algo import DQNHandle, init_q_params
    N, iters = 300, 40
    cfg = abi.make_dqn_config(num_envs=N, buffer_size=N * iters, min_buff_size=10 ** 8, batch_size=32, epsilon_start=0.0,
                              epsilon_end=0.0, seed=3)
    p = init_q_params(11)
    p[10932:] = (0.02, 0.0)       # keep both actions in play around the upright state
    h = DQNHandle(cfg)
    h.set_params(p); h.reset()
    h.run(iters)
    b = h.read_buffer()
    h.close()
    q = gpu_forward(crl, torch_cuda, p, b["state"])
    np.testing.assert_array_equal(b["action"], (q[:, 1] > q[:, 0]).astype(np.int32))
    assert 0.05 < b["action"].mean() < 0.95


# ------------------------------------------------------------------ loss and gradient
BATCHES = [1, 2, 15, 16, 17, 31, 32, 33, 64, 100, 120, 127, 128]


@pytest.mark.parametrize("kind", ["mixed", "action0", "terminal", "open", "gamma0", "relu0"])
@pytest.mark.parametrize("B", BATCHES)
def test_dqn_loss_raw_matches_float64_and_oracle(crl, olib, abi, torch_cuda, kind, B):
    """gradient per parameter array at rtol 1e-4, atol 2e-6 max|g| of the array, against float64 NumPy and the oracle;
    loss at rtol 1e-6 against float64 (achieved: 3.1e-7 over these batches; the Q-values are fp32, the TD errors
    float64) and 2e-6 against the oracle (itself up to 5.4e-7 off); the gradient reaches 0.06 of its bound against
    float64, 0.09 against the oracle; the exact zeros of the single-action and ReLU-at-0 batches"""
    q, tgt, s, a, r, s2, term, gamma = edge_batch(kind, B, seed=B)
    g, loss = gpu_loss(crl, torch_cuda, q, tgt, s, a, r, s2, term, gamma)
    gn, lossn = _np_loss_grad(q, tgt, s, a, r, s2, term, gamma)
    o = OracleDQN(olib, abi.make_dqn_config())
    go, losso = o.loss_raw(q, tgt, s, a, r, s2, term, gamma)
    o.close()
    assert np.isfinite(g).all()
    assert_grad_close(g, gn, what="vs float64 ")
    assert_grad_close(g, go, what="vs oracle ")
    assert abs(loss - lossn) <= 1e-6 * lossn and abs(loss - losso) <= 2e-6 * losso
    if kind == "action0":
        assert np.all(g[10765:10932:2] == 0) and g[10933] == 0
    if kind == "relu0":
        z = relu0_zero_indices()
        assert np.all(g[z] == 0), np.flatnonzero(g[z])[:8]


@pytest.mark.parametrize("B", [1, 17, 100])
def test_dqn_loss_raw_reads_nothing_past_row_B(crl, torch_cuda, B):
    """the same batch with 128 - B rows of NaN (and out-of-range actions / terminal flags) behind it: bit-identical"""
    q, tgt, s, a, r, s2, term, gamma = edge_batch("mixed", B, seed=B + 7)
    ref = gpu_loss(crl, torch_cuda, q, tgt, s, a, r, s2, term, gamma)
    pad = 128 - B + 3

    def poison(x, v):
        return np.concatenate([x, np.full((pad,) + x.shape[1:], v, x.dtype)])
    got = gpu_loss(crl, torch_cuda, q, tgt, poison(s, np.nan), poison(a, 1 << 20), poison(r, np.nan), poison(s2, np.nan),
                   poison(term, 255), gamma, B=B)
    np.testing.assert_array_equal(got[0], ref[0])
    assert got[1] == ref[1]


# ------------------------------------------------------------------ run loop vs the oracle
def compare_with_oracle(h, o, chunks):
    """test_dqn_cuda_matches_oracle's comparisons after every chunk (env states at the trajectory tolerance); yields the
    handle's stats and parameters"""
    for chunk in chunks:
        sh, so = h.run(chunk), o.run(chunk)
        assert (sh.iterations, sh.learn_steps, sh.episodes) == (so.iterations, so.learn_steps, so.episodes)
        assert sh.epsilon == so.epsilon
        assert sh.sum_return == so.sum_return and sh.sum_length == so.sum_length
        bh, bo = h.read_buffer(), o.read_buffer()
        assert (bh["size"], bh["ptr"]) == (bo["size"], bo["ptr"])
        n = bh["size"]
        np.testing.assert_array_equal(bh["action"][:n], bo["action"][:n])
        np.testing.assert_array_equal(bh["terminal"][:n], bo["terminal"][:n])
        np.testing.assert_array_equal(bh["reward"][:n], bo["reward"][:n])
        # env states are trajectories: rtol 1e-4, the suite's tolerance for chained CartPole steps (rounding grows
        # ~e^0.08 per step, and a learning policy keeps episodes going for a hundred steps and more)
        np.testing.assert_allclose(bh["state"][:n], bo["state"][:n], rtol=1e-4, atol=2e-6)
        np.testing.assert_allclose(bh["next_state"][:n], bo["next_state"][:n], rtol=1e-4, atol=2e-6)
        qh, th = h.get_params(); qo, to = o.get_params()
        np.testing.assert_allclose(qh, qo, rtol=1e-4, atol=2e-6)
        np.testing.assert_allclose(th, to, rtol=1e-4, atol=2e-6)
        if so.learn_steps:
            assert abs(sh.last_loss - so.last_loss) <= 1e-4 * abs(so.last_loss) + 1e-7
        yield sh, (qh, th)


def learn_iterations(cfg, iters):
    """the iterations (1-based) with a learning step (dqn.jl:94): global step it * N past min_buff_size, it a multiple
    of train_freq, min(it * N, capacity) >= batch_size"""
    N, tf = cfg.num_envs, cfg.train_freq
    first = max(cfg.min_buff_size // N + 1, -(-cfg.batch_size // N) if cfg.batch_size <= cfg.buffer_size else iters + 1)
    start = -(-first // tf) * tf
    return list(range(start, iters + 1, tf))


RUNS = {   # name: (config fields, iteration chunks)
    "learn_every_iteration": (dict(num_envs=8, buffer_size=512, min_buff_size=64, batch_size=32, train_freq=1, target_net_freq=5), (47, 53, 50)),
    "two_launches_per_learning_step": (dict(num_envs=8, buffer_size=512, min_buff_size=64, batch_size=32, train_freq=17, target_net_freq=34), (68, 17, 65)),
    "three_launches_per_learning_step": (dict(num_envs=8, buffer_size=2048, min_buff_size=64, batch_size=32, train_freq=37, target_net_freq=74), (74, 37, 39)),
    "target_copy_off_the_learning_grid": (dict(num_envs=8, buffer_size=512, min_buff_size=64, batch_size=32, train_freq=4, target_net_freq=6), (48, 52, 50)),
    "truncated_episodes": (dict(num_envs=16, buffer_size=4096, min_buff_size=64, batch_size=32, train_freq=4, target_net_freq=12, max_episode_steps=10), (48, 50, 52)),
    "ring_below_two_vector_steps": (dict(num_envs=100, buffer_size=150, min_buff_size=100, batch_size=128, train_freq=3, target_net_freq=9), (45, 55, 50)),
    "ring_of_one_vector_step": (dict(num_envs=64, buffer_size=64, min_buff_size=10, batch_size=64, train_freq=2, target_net_freq=4), (48, 51, 51)),
    "batch_size_gate": (dict(num_envs=4, buffer_size=512, min_buff_size=8, batch_size=100, train_freq=2, target_net_freq=10), (20, 30, 96)),
    "greedy_with_ties": (dict(num_envs=32, buffer_size=1024, min_buff_size=320, batch_size=64, train_freq=4, target_net_freq=12, epsilon_start=0.0, epsilon_end=0.0), (8, 40, 52, 50)),
}


@pytest.mark.parametrize("name", sorted(RUNS))
def test_dqn_run_loop_edges_match_oracle(crl, olib, abi, torch_cuda, name):
    from cleanrl_jl_b200.dqn_algo import DQNHandle, init_q_params
    kw, chunks = RUNS[name]
    cfg = abi.make_dqn_config(epsilon_duration=2000.0, seed=9, **kw)
    h, o = DQNHandle(cfg), OracleDQN(olib, cfg)
    p = init_q_params(3)
    if name == "greedy_with_ties":
        p[10764:] = 0.0           # zero head: Q = (0, 0) for every state, and the first maximum is action 0
    for x in (h, o):
        x.set_params(p); x.reset()
    learn_at = learn_iterations(cfg, sum(chunks))
    assert len(learn_at) >= 3
    done, copy_seen, nocopy_seen = 0, False, False
    for (st, (qh, th)), chunk in zip(compare_with_oracle(h, o, chunks), chunks):
        done += chunk
        past = [i for i in learn_at if i <= done]
        assert st.learn_steps == len(past)
        if not past or past[-1] % cfg.target_net_freq == 0:
            np.testing.assert_array_equal(qh, th)        # the last learning step copied the target (or none ran yet)
            copy_seen |= bool(past)
        else:
            assert not np.array_equal(qh, th)
            nocopy_seen = True
        if name == "greedy_with_ties" and done * cfg.num_envs <= cfg.min_buff_size:
            b = h.read_buffer()
            assert b["size"] == done * cfg.num_envs and not b["action"][:b["size"]].any()
    assert copy_seen and nocopy_seen, "every run ends one chunk on a copy and one off it"
    if name == "truncated_episodes":
        b = h.read_buffer()
        T, N, M = done, cfg.num_envs, cfg.max_episode_steps
        term = b["terminal"][:T * N].reshape(T, N).astype(bool)           # the ring has not wrapped: row t = iteration t + 1
        lengths = []
        for n in range(N):
            ends = np.flatnonzero(term[:, n])
            lengths += list(np.diff(np.concatenate([[-1], ends])))
        lengths = np.array(lengths)
        # done when t > max_episode_steps: a truncated episode has max_episode_steps + 1 transitions
        assert lengths.max() == M + 1 and np.mean(lengths == M + 1) > 0.5
    h.close(); o.close()
