"""DQN (SURVEY 8f-2; src/algorithms/dqn.jl): the CPU oracle against hand-derived values and a float64 NumPy
restatement (no GPU), and the CUDA path against the oracle on shared Philox streams (GPU)."""
import numpy as np
import pytest

from oracle.oracle import OracleDQN

F = np.float32


def _np_forward(p, x):
    """float64 NumPy restatement of Chain(Dense(4,120,relu), Dense(120,84,relu), Dense(84,2)), dqn.jl:25"""
    p = p.astype(np.float64)
    o = 0
    W1 = p[o:o + 480].reshape(4, 120).T; o += 480
    b1 = p[o:o + 120]; o += 120
    W2 = p[o:o + 10080].reshape(120, 84).T; o += 10080
    b2 = p[o:o + 84]; o += 84
    W3 = p[o:o + 168].reshape(84, 2).T; o += 168
    b3 = p[o:o + 2]
    z1 = x @ W1.T + b1; h1 = np.maximum(z1, 0)
    z2 = h1 @ W2.T + b2; h2 = np.maximum(z2, 0)
    return h2 @ W3.T + b3, (W1, W2, W3, h1, h2, z1, z2)


def _np_loss_grad(q, tgt, s, a, r, s2, term, gamma):
    B = len(a)
    qn, _ = _np_forward(tgt, s2.astype(np.float64))
    td = r.astype(np.float64) + gamma * qn.max(axis=1) * (1.0 - term.astype(np.float64))        # dqn.jl:99-100
    qv, (W1, W2, W3, h1, h2, z1, z2) = _np_forward(q, s.astype(np.float64))
    diff = td - qv[np.arange(B), a]
    loss = np.mean(diff ** 2)                                                                   # Flux.mse, dqn.jl:107
    dq = np.zeros((B, 2)); dq[np.arange(B), a] = -2.0 * diff / B
    gW3 = dq.T @ h2; gb3 = dq.sum(0)
    dz2 = (dq @ W3) * (z2 > 0)
    gW2 = dz2.T @ h1; gb2 = dz2.sum(0)
    dz1 = (dz2 @ W2) * (z1 > 0)
    gW1 = dz1.T @ s.astype(np.float64); gb1 = dz1.sum(0)
    g = np.concatenate([gW1.T.ravel(), gb1, gW2.T.ravel(), gb2, gW3.T.ravel(), gb3])            # (out,in) column-major
    return g, loss


def _rand_batch(rng, B):
    s = rng.uniform(-1, 1, (B, 4)).astype(F); s2 = rng.uniform(-1, 1, (B, 4)).astype(F)
    a = rng.integers(0, 2, B).astype(np.int32); r = rng.integers(0, 2, B).astype(F)
    term = (rng.random(B) < 0.2).astype(np.uint8)
    return s, a, r, s2, term


# flat parameter arrays of the Q-network (Flux.params order) and the per-array gradient tolerance of the suite
DQN_ARRAYS = (("W1", 0, 480), ("b1", 480, 600), ("W2", 600, 10680), ("b2", 10680, 10764), ("W3", 10764, 10932), ("b3", 10932, 10934))


def assert_grad_close(g, ref, rtol=1e-4, atol_frac=2e-6, what=""):
    """per parameter array: |g - ref| <= rtol |ref| + atol_frac * max|ref of that array|"""
    for name, a, b in DQN_ARRAYS:
        np.testing.assert_allclose(g[a:b], ref[a:b], rtol=rtol, atol=atol_frac * np.abs(ref[a:b]).max(), err_msg=what + name)


def edge_batch(kind, B, seed):
    """(q, tgt, state, action, reward, next_state, terminal, gamma) of one of the edge batches the DQN loss is tested at.
    tgt != q everywhere; rewards are -1.5, 1 or 2 so that no TD error is close to 0 (a float32 Q-value then decides the
    relative error of the whole gradient, which would make the per-array tolerance depend on luck rather than on the
    kernel). Kinds:
      mixed     random actions, 20 % terminal, gamma 0.99
      action0   every action 0: column 1 of dq is 0, so dW3 row 1 and db3[1] are exactly 0
      terminal  every sample terminal (the target net drops out), gamma 0.99
      open      no sample terminal, gamma 1
      gamma0    no sample terminal, gamma 0
      relu0     every state row 0, every other b1 entry 0 and the second-layer units 0, 7, 14, ... with zero weights and
                bias: those first- and second-layer pre-activations are exactly 0, and relu'(0) = 0 (Flux) makes their
                gradients exactly 0"""
    from cleanrl_jl_b200.dqn_algo import init_q_params
    rng = np.random.default_rng(seed)
    q = init_q_params(seed)
    q[480:600] = rng.normal(0, 0.2, 120)
    q[10680:10764] = rng.normal(0, 0.1, 84)
    q[10932:] = rng.normal(0, 0.1, 2)
    tgt = init_q_params(seed + 1000)
    tgt[480:600] = rng.normal(0, 0.2, 120)
    s = rng.uniform(-2, 2, (B, 4)).astype(F)
    s2 = rng.uniform(-2, 2, (B, 4)).astype(F)
    a = rng.integers(0, 2, B).astype(np.int32)
    r = rng.choice(np.array([-1.5, 1.0, 2.0], F), B)
    term = (rng.random(B) < 0.2).astype(np.uint8)
    gamma = 0.99
    if kind == "action0":
        a[:] = 0
    elif kind == "terminal":
        term[:] = 1
    elif kind == "open":
        term[:] = 0
        gamma = 1.0
    elif kind == "gamma0":
        term[:] = 0
        gamma = 0.0
    elif kind == "relu0":
        s[:] = 0.0
        q[480:600:2] = 0.0
        q[600:10680].reshape(120, 84)[:, ::7] = 0.0      # W2 (84 x 120) column-major: rows 0, 7, ... of W2
        q[10680:10764:7] = 0.0
    else:
        assert kind == "mixed", kind
    return q, tgt, s, a, r, s2, term, gamma


def relu0_zero_indices():
    """gradient entries that must be exactly 0 in the relu0 batch: all of dW1 (the states are 0), db1 of the zero-bias
    first-layer units, and dW2 row / db2 / dW3 column of the dead second-layer units"""
    w2 = np.zeros((84, 120), bool)
    w2[::7, :] = True
    dead = np.arange(0, 84, 7)
    return np.concatenate([np.arange(0, 480), 480 + np.arange(0, 120, 2), 600 + np.flatnonzero(w2.ravel(order="F")),
                           10680 + dead, 10764 + 2 * dead, 10764 + 2 * dead + 1])


def test_oracle_linear_schedule_matches_dqn_jl(olib, abi):
    o = OracleDQN(olib, abi.make_dqn_config())
    # dqn.jl:28-31 with the defaults 1.0 -> 0.05 over 10,000 steps
    assert o.linear_schedule(1.0, 0.05, 10000.0, 0.0) == 1.0
    assert abs(o.linear_schedule(1.0, 0.05, 10000.0, 5000.0) - 0.525) < 1e-15
    assert o.linear_schedule(1.0, 0.05, 10000.0, 10000.0) == pytest.approx(0.05, abs=1e-15)
    assert o.linear_schedule(1.0, 0.05, 10000.0, 123456.0) == 0.05
    from cleanrl_jl_b200.dqn_algo import linear_schedule
    for t in (0, 1, 777, 9999, 10001):
        assert linear_schedule(1.0, 0.05, 10000.0, t) == o.linear_schedule(1.0, 0.05, 10000.0, float(t))
    o.close()


def test_oracle_forward_and_gradient_match_float64_numpy(olib, abi):
    from cleanrl_jl_b200.dqn_algo import init_q_params
    o = OracleDQN(olib, abi.make_dqn_config())
    rng = np.random.default_rng(3)
    q = init_q_params(1); q[480:600] = rng.normal(0, 0.1, 120)      # non-zero biases
    tgt = init_q_params(2)
    s, a, r, s2, term = _rand_batch(rng, 120)
    qo = o.forward(q, s)
    qn, _ = _np_forward(q, s.astype(np.float64))
    np.testing.assert_allclose(qo, qn, rtol=2e-5, atol=2e-6)
    g, loss = o.loss_raw(q, tgt, s, a, r, s2, term, 0.99)
    gn, lossn = _np_loss_grad(q, tgt, s, a, r, s2, term, 0.99)
    # achieved here: loss 1e-8 relative; per array at most 3.5e-7 of the array's max|g| away, 0.11 of the bound below
    assert abs(loss - lossn) < 1e-7 * abs(lossn)
    assert_grad_close(g, gn, rtol=1e-5, atol_frac=1e-6)
    o.close()


@pytest.mark.parametrize("kind", ["mixed", "action0", "terminal", "open", "gamma0", "relu0"])
@pytest.mark.parametrize("B", [1, 2, 16, 17, 33, 100, 128])
def test_oracle_dqn_loss_at_the_edges_matches_float64_numpy(olib, abi, kind, B):
    """the reference the GPU loss kernels are compared with, pinned at the same edge batches: per array rtol 1e-4, atol
    2e-6 max|g| (achieved: at most 0.07 of that bound at every batch size of the GPU tests), loss rtol 1e-6 (achieved:
    5.4e-7), and the entries that must be exactly 0 are exactly 0"""
    o = OracleDQN(olib, abi.make_dqn_config())
    q, tgt, s, a, r, s2, term, gamma = edge_batch(kind, B, seed=B)
    g, loss = o.loss_raw(q, tgt, s, a, r, s2, term, gamma)
    gn, lossn = _np_loss_grad(q, tgt, s, a, r, s2, term, gamma)
    assert abs(loss - lossn) <= 1e-6 * lossn
    assert_grad_close(g, gn)
    if kind == "action0":
        assert np.all(g[10765:10932:2] == 0) and g[10933] == 0 and np.all(gn[10765:10932:2] == 0)
        assert np.abs(g[10764:10932:2]).max() > 0 and g[10932] != 0
    if kind == "relu0":
        z = relu0_zero_indices()
        assert np.all(g[z] == 0) and np.all(gn[z] == 0)
        assert np.count_nonzero(g[480:600]) >= 20 and np.count_nonzero(g[10680:10764]) >= 20   # the live units learn
    o.close()


def test_oracle_run_schedule_matches_reference_counters(olib, abi):
    """N = 1: learning steps at global_step in {210, 220, ...} (dqn.jl:94), target copies every 100 (dqn.jl:111)"""
    from cleanrl_jl_b200.dqn_algo import init_q_params
    cfg = abi.make_dqn_config(num_envs=1, buffer_size=500, min_buff_size=200, batch_size=32, seed=4)
    o = OracleDQN(olib, cfg)
    p0 = init_q_params(0)
    o.set_params(p0); o.reset()
    st = o.run(200)
    assert st.learn_steps == 0 and st.iterations == 200          # global_step > min_buff_size is strict
    q, t = o.get_params()
    np.testing.assert_array_equal(q, p0); np.testing.assert_array_equal(t, p0)
    st = o.run(95)                                               # up to 295: learn at 210..290
    assert st.learn_steps == 9
    q, t = o.get_params()
    assert not np.array_equal(q, p0) and np.array_equal(t, p0)   # target untouched before step 300
    st = o.run(5)                                                # step 300: learn, then copy
    assert st.learn_steps == 10
    q, t = o.get_params()
    np.testing.assert_array_equal(q, t)
    b = o.read_buffer()
    assert b["size"] == 300 and b["ptr"] == 300 and b["terminal"][:300].sum() >= 5
    st = o.run(300)                                              # ring wraps at 500
    b = o.read_buffer()
    assert b["size"] == 500 and b["ptr"] == 100
    o.close()


def _dqn_shards(olib, abi, world, n_local, **kw):
    shards = []
    for r in range(world):
        o = OracleDQN(olib, abi.make_dqn_config(num_envs=n_local, **kw))
        o.set_shard(world, r, r * n_local)
        shards.append(o)
    return shards


def test_sharded_dqn_acts_like_one_process_until_the_first_learning_step(olib, abi):
    """data-parallel extension: Philox is keyed by the GLOBAL env id and epsilon by the global step, so with equal
    parameters the union of the shards' transitions is the single-process run over all envs, env for env"""
    from cleanrl_jl_b200.dqn_algo import init_q_params
    kw = dict(buffer_size=4096, min_buff_size=10 ** 6, batch_size=16, train_freq=4, target_net_freq=12, epsilon_duration=500.0, seed=4)
    world, n_local, iters = 4, 6, 40
    single = OracleDQN(olib, abi.make_dqn_config(num_envs=world * n_local, **kw))
    shards = _dqn_shards(olib, abi, world, n_local, **kw)
    p = init_q_params(2)
    for o in [single] + shards:
        o.set_params(p); o.reset()
    s1 = single.run(iters)
    ss = OracleDQN.group_run(shards, iters)
    b1 = single.read_buffer()
    assert s1.learn_steps == 0 and all(s.learn_steps == 0 for s in ss)
    assert s1.episodes == sum(s.episodes for s in ss) and s1.sum_return == sum(s.sum_return for s in ss)
    assert all(s.epsilon == s1.epsilon for s in ss)
    N = world * n_local
    for r, o in enumerate(shards):
        b = o.read_buffer()
        assert b["size"] == iters * n_local
        for f in ("state", "action", "reward", "next_state", "terminal"):
            glob = b1[f][:iters * N].reshape((iters, N) + b1[f].shape[1:])[:, r * n_local:(r + 1) * n_local]
            np.testing.assert_array_equal(b[f][:iters * n_local].reshape(glob.shape), glob)
    for o in [single] + shards:
        o.close()


def test_sharded_dqn_learning_keeps_the_replicas_identical(olib, abi):
    """every shard applies Adam to the same rank-ordered gradient sum: parameters, target copies and losses agree bit for
    bit across the shards; world = 1 through the group entry point is the plain run"""
    from cleanrl_jl_b200.dqn_algo import init_q_params
    kw = dict(buffer_size=512, min_buff_size=64, batch_size=16, train_freq=4, target_net_freq=12, epsilon_duration=2000.0, seed=6)
    shards = _dqn_shards(olib, abi, 2, 8, **kw)
    p = init_q_params(5)
    for o in shards:
        o.set_params(p); o.reset()
    st = OracleDQN.group_run(shards, 60) and OracleDQN.group_run(shards, 40)      # two calls: state carries over
    assert st[0].learn_steps == st[1].learn_steps > 10 and st[0].iterations == 100
    assert st[0].last_loss == st[1].last_loss and np.isfinite(st[0].last_loss)
    (q0, t0), (q1, t1) = shards[0].get_params(), shards[1].get_params()
    np.testing.assert_array_equal(q0, q1)
    np.testing.assert_array_equal(t0, t1)
    assert np.abs(q0 - p).max() > 1e-4 and not np.array_equal(q0, t0)
    with pytest.raises(AssertionError):
        shards[0].run(1)                      # a shard of a larger world cannot step alone
    a, b = OracleDQN(olib, abi.make_dqn_config(num_envs=8, **kw)), OracleDQN(olib, abi.make_dqn_config(num_envs=8, **kw))
    for o in (a, b):
        o.set_params(p); o.reset()
    sa, sb = a.run(100), OracleDQN.group_run([b], 100)[0]
    assert (sa.last_loss, sa.learn_steps, sa.episodes) == (sb.last_loss, sb.learn_steps, sb.episodes)
    np.testing.assert_array_equal(a.get_params()[0], b.get_params()[0])
    for o in shards + [a, b]:
        o.close()


def test_dqn_config_has_the_reference_fields():
    from cleanrl_jl_b200 import DQNConfig
    c = DQNConfig()
    ref = dict(log_frequencey=1000, total_timesteps=500_000, buffer_size=10_000, min_buff_size=200, lr=0.0001, train_freq=10,
               target_net_freq=100, batch_size=120, gamma=0.99, epsilon_start=1.0, epsilon_end=0.05, epsilon_duration=10_000)
    for k, v in ref.items():
        assert getattr(c, k) == v, k


def test_dqn_config_through_the_cli_parser(monkeypatch):
    """ConfigParser.argparse_struct (config_parser.jl:18-40) works on DQNConfig like on PPOConfig"""
    import sys
    from cleanrl_jl_b200 import DQNConfig, argparse_struct
    monkeypatch.setattr(sys, "argv", ["dqn", "--num_envs", "64", "--lr", "0.001", "--epsilon_duration", "5000.5",
                                      "--batch_size", "64"])
    c = argparse_struct(DQNConfig())
    assert (c.num_envs, c.lr, c.epsilon_duration, c.batch_size) == (64, 0.001, 5000.5, 64)
    assert c.buffer_size == 10_000 and c.train_freq == 10      # untouched fields keep the reference defaults


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("N,iters,batch", [(1, 400, 32), (8, 120, 32), (64, 60, 32),
                                           # batch sizes that leave the last 16-sample CTA of the learning step partly
                                           # filled (120 = dqn.jl default, 33), fill all eight (128), or hold one sample
                                           (16, 80, 120), (16, 80, 33), (32, 40, 128), (8, 60, 1)])
def test_dqn_cuda_matches_oracle(crl, olib, abi, torch_cuda, N, iters, batch):
    from cleanrl_jl_b200.dqn_algo import DQNHandle, init_q_params
    cfg = abi.make_dqn_config(num_envs=N, buffer_size=max(512, 4 * N), min_buff_size=max(64, batch), batch_size=batch, train_freq=4,
                              target_net_freq=12, epsilon_duration=float(iters * N), seed=9)
    h, o = DQNHandle(cfg), OracleDQN(olib, cfg)
    p = init_q_params(3)
    for x in (h, o):
        x.set_params(p); x.reset()
    done = 0
    for chunk in (iters // 3, iters // 3, iters - 2 * (iters // 3)):
        sh, so = h.run(chunk), o.run(chunk)
        done += chunk
        assert (sh.iterations, sh.learn_steps, sh.episodes) == (so.iterations, so.learn_steps, so.episodes)
        assert sh.epsilon == so.epsilon
        assert sh.sum_return == so.sum_return and sh.sum_length == so.sum_length
        bh, bo = h.read_buffer(), o.read_buffer()
        assert (bh["size"], bh["ptr"]) == (bo["size"], bo["ptr"])
        n = bh["size"]
        np.testing.assert_array_equal(bh["action"][:n], bo["action"][:n])      # epsilon draws, argmax, ring order
        np.testing.assert_array_equal(bh["terminal"][:n], bo["terminal"][:n])
        np.testing.assert_array_equal(bh["reward"][:n], bo["reward"][:n])
        np.testing.assert_allclose(bh["state"][:n], bo["state"][:n], rtol=1e-5, atol=2e-6)
        np.testing.assert_allclose(bh["next_state"][:n], bo["next_state"][:n], rtol=1e-5, atol=2e-6)
        qh, th = h.get_params(); qo, to = o.get_params()
        np.testing.assert_allclose(qh, qo, rtol=1e-4, atol=2e-6)
        np.testing.assert_allclose(th, to, rtol=1e-4, atol=2e-6)
        if so.learn_steps:
            assert abs(sh.last_loss - so.last_loss) <= 1e-4 * abs(so.last_loss) + 1e-7
    assert so.learn_steps > 5 and so.episodes > 0
    h.close(); o.close()


@pytest.mark.gpu
def test_dqn_public_api_runs_and_learns_something(tmp_path, torch_cuda):
    from cleanrl_jl_b200 import DQNConfig, dqn
    from cleanrl_jl_b200 import logger as Logger
    lg = Logger.make_logger("dqn", to_terminal=False, to_tensorboard=False, to_json=True, log_dir=str(tmp_path))
    cfg = DQNConfig(num_envs=64, total_timesteps=64 * 3000, buffer_size=50_000, min_buff_size=1000, train_freq=1,
                    target_net_freq=50, lr=5e-4, epsilon_duration=64 * 1500, log_frequencey=64 * 250, seed=2)
    res = dqn(cfg, logger=lg)
    lg.close()
    assert res["global_step"] == 64 * 3000 and res["learn_steps"] > 2000 and np.isfinite(res["last_loss"])
    assert np.isfinite(res["params"]).all() and res["episodes"] > 100
    assert res["last_mean_return"] > 30          # random policy: ~22
    import json
    recs = [json.loads(l) for l in open(tmp_path / "dqn.json")]
    assert {r["msg"] for r in recs} == {"Episode Statistics", "Training Statistics"}


@pytest.mark.gpu
def test_dqn_argument_errors(crl, abi, torch_cuda):
    from cleanrl_jl_b200.dqn_algo import DQNHandle
    with pytest.raises(crl.CleanRLCudaError):
        DQNHandle(abi.make_dqn_config(batch_size=500))
    with pytest.raises(crl.CleanRLCudaError):
        DQNHandle(abi.make_dqn_config(num_envs=64, buffer_size=32))
    h = DQNHandle(abi.make_dqn_config())
    with pytest.raises(crl.CleanRLCudaError):
        h.run(1)                                  # before set_params / reset
    h.close()


def test_float32_env_substitute_for_the_float64_cartpole_of_dqn_and_a2c(olib, abi):
    """dqn.jl:37 `CartPoleEnv()` and a2c.jl:33 `CartPoleEnv(max_steps=500)` default to T = Float64 states, while the
    kernels (and the oracle) step the Float32 env of the PPO path (ppo.jl:82 `T=Float32`). The substitute is exact in
    everything discrete and within Float32 rounding per step in the state:
      * per step, from the same Float32-representable state: |s32 - s64| <= 4e-7 + 3e-7 |s64| per component
        (the Float32 step already evaluates the accelerations in Float64, SURVEY 8a row 5u, so only the stores round);
      * the termination test agrees unless the Float64 state lies within that distance of a threshold;
      * over a whole episode under a fixed action sequence the two trajectories stay within 1e-4 (chaotic growth
        ~e^0.08 per step of the per-step rounding) and end at the same step in >= 99 % of the episodes.
    Rewards (0/1), actions and the episode bookkeeping are integers in both."""
    rng = np.random.default_rng(11)
    n = 20000

    def step64(s, a):
        g, mc, mp, l, fm, dt = 9.8, 1.0, 0.1, 0.5, 10.0, 0.02
        x, xd, th, thd = s.T
        force = np.where(a == 1, fm, -fm)
        tmp = (force + mp * l * thd ** 2 * np.sin(th)) / (mc + mp)
        thacc = (g * np.sin(th) - np.cos(th) * tmp) / (l * (4.0 / 3.0 - mp * np.cos(th) ** 2 / (mc + mp)))
        xacc = tmp - mp * l * thacc * np.cos(th) / (mc + mp)
        return np.stack([x + dt * xd, xd + dt * xacc, th + dt * thd, thd + dt * thacc], 1)

    s0 = (rng.random((n, 4)) * np.array([4.0, 4.0, 0.4, 4.0]) - np.array([2.0, 2.0, 0.2, 2.0])).astype(F)
    a = rng.integers(0, 2, n).astype(np.int32)
    s32, _, r32, d32 = olib.env_step_raw(0, s0, np.zeros(n, np.int32), a, 200)
    s64 = step64(s0.astype(np.float64), a)
    assert np.all(np.abs(s32 - s64) <= 4e-7 + 3e-7 * np.abs(s64))
    d64 = (np.abs(s64[:, 0]) > 2.4) | (np.abs(s64[:, 2]) > 12 * 2 * np.pi / 360)
    near = (np.abs(np.abs(s64[:, 0]) - 2.4) < 1e-6) | (np.abs(np.abs(s64[:, 2]) - 12 * 2 * np.pi / 360) < 1e-6)
    assert np.array_equal(d32[~near].astype(bool), d64[~near]) and near.sum() < 5
    assert np.array_equal(r32[~near], np.where(d64[~near], 0.0, 1.0).astype(F))
    # whole episodes, fixed action sequences
    m, T = 2000, 200
    s = (rng.random((m, 4)) * 0.1 - 0.05).astype(F)
    sf, sd = s.copy(), s.astype(np.float64)
    acts = rng.integers(0, 2, (T, m)).astype(np.int32)
    alive32, alive64 = np.ones(m, bool), np.ones(m, bool)
    end32, end64 = np.full(m, T), np.full(m, T)
    worst = 0.0
    for t in range(T):
        nf, _, _, df = olib.env_step_raw(0, sf, np.zeros(m, np.int32), acts[t], 10 ** 6)
        nd = step64(sd, acts[t])
        dd = (np.abs(nd[:, 0]) > 2.4) | (np.abs(nd[:, 2]) > 12 * 2 * np.pi / 360)
        both = alive32 & alive64
        worst = max(worst, float(np.max(np.abs(nf[both] - nd[both]), initial=0.0)))
        end32[alive32 & df.astype(bool)] = t
        end64[alive64 & dd] = t
        alive32 &= ~df.astype(bool)
        alive64 &= ~dd
        sf, sd = nf, nd
    assert worst < 1e-4
    assert np.mean(end32 == end64) >= 0.99 and np.max(np.abs(end32 - end64)) <= 1
