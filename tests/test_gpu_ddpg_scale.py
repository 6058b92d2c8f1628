"""DDPG and TD3 run loops at the shapes they are benchmarked at (tools/ddpg_bench.py: 4,096 envs, a 1M ring, batch 256),
where the other run-loop tests (tests/test_gpu_ddpg.py, tests/test_gpu_td3.py, num_envs <= 16) do not reach: many acting
CTAs and a ragged last one, acting launches split at ACT_MAX_STEPS and at the ring capacity, a ring that wraps in the
middle of an iteration, batch 256 through the keyed permutation over a large ring, and the per-call episode statistics.

* Acting does not depend on the env count: env n is keyed by (seed, n, iteration) and every neuron is one fmaf chain, so
  before the first learning step env n's transitions are bit-identical for every num_envs > n.
* A run does not depend on how its iterations are split across calls: ring, parameters, targets, Adam state, losses and
  counters bit for bit, and the episode statistics summed over the calls.
* The run loop against the float64 reference (RefDDPG, RefTD3) at scale, in several calls, with the per-call episode
  statistics and the launch count.
Run with `pytest -m gpu` on a B200."""
import numpy as np
import pytest

import ddpg_reference as R
import td3_reference as T
from test_ddpg import rand_nets
from test_gpu_ddpg import assert_run_close, closed_form_counts
from test_gpu_td3 import make_handle

pytestmark = pytest.mark.gpu
ALGOS = ["ddpg", "td3"]
LAUNCHES_PER_ACTOR_STEP = {"ddpg": 3, "td3": 4}   # actor fwd + update + Polyak (+ TD3's qf2 Polyak)
# (GPU key, RefDDPG attribute, Adam moment attributes) of each critic; targets are key + "_target" and attribute + "_tgt"
CRITICS = {"ddpg": [("critic", "critic", "cm", "cv")], "td3": [("qf1", "critic", "cm", "cv"), ("qf2", "qf2", "q2m", "q2v")]}
LOSSES = {"ddpg": [("critic_loss", "critic_loss")], "td3": [("qf1_loss", "critic_loss"), ("qf2_loss", "qf2_loss")]}


def make(abi, algo, kw):
    """(cfg, handle, nets) of a fresh, reset run with the parameters of the other run-loop tests"""
    a, q1 = rand_nets(17)
    if algo == "td3":
        q2 = rand_nets(18)[1]
        cfg, h = make_handle(abi, kw, a, q1, q2)
        return cfg, h, (a, q1, q2)
    from cleanrl_jl_b200.ddpg_algo import DDPGHandle
    cfg = abi.make_ddpg_config(**{**dict(exploration_noise=0.1, lr=1e-3, tau=0.05, seed=3), **kw})
    h = DDPGHandle(cfg)
    h.set_params(a, q1)
    h.reset()
    return cfg, h, (a, q1)


def reference(olib, algo, cfg, nets):
    return R.RefDDPG(olib, cfg, *nets) if algo == "ddpg" else T.RefTD3(olib, cfg, *nets)


def expected_launches(algo, cfg, calls):
    learn, actor = closed_form_counts(cfg, sum(calls))
    return T.acting_launches(cfg, calls) + 2 * learn + LAUNCHES_PER_ACTOR_STEP[algo] * actor


def assert_ring_close(buf, ref):
    """TD3's run-loop rule for the ring once the actor acts: rtol 1e-4 / atol 1e-5, except at most 0.1 % of an array
    (at least 1 element) at rtol 1e-3 / atol 1e-4 (Pendulum carries the actor's Float32 rounding into later states);
    terminal exactly"""
    for k, r in (("obs", ref.b_obs), ("next_obs", ref.b_next), ("action", ref.b_act), ("reward", ref.b_rew)):
        d, ar = np.abs(buf[k] - r), np.abs(r)
        bad = d > 1e-4 * ar + 1e-5
        assert bad.sum() <= max(1, r.size // 1000) and np.all(d[bad] <= 1e-3 * ar[bad] + 1e-4), \
            "%s: %d of %d elements off, worst %g" % (k, bad.sum(), r.size, d.max())
    np.testing.assert_array_equal(buf["terminal"], ref.b_term)


def run_against_reference(olib, abi, algo, kw, calls):
    """runs `calls` on the GPU and in the reference, checking each call's episode statistics (episodes and sum_length
    exactly, sum_return at rtol 1e-4) against the reference's cumulative counters; returns (cfg, handle, ref, last stats)"""
    cfg, h, nets = make(abi, algo, kw)
    ref = reference(olib, algo, cfg, nets)
    try:
        for i, n in enumerate(calls):
            e0, r0, l0 = ref.episodes, ref.sum_return, ref.sum_length
            st = h.run(n)
            ref.run(n)
            what = "call %d of %s: " % (i, calls)
            assert st.episodes == ref.episodes - e0 and st.sum_length == ref.sum_length - l0, \
                what + "episodes %d sum_length %g, reference %d %g" % (st.episodes, st.sum_length, ref.episodes - e0, ref.sum_length - l0)
            np.testing.assert_allclose(st.sum_return, ref.sum_return - r0, rtol=1e-4, err_msg=what + "sum_return")
    except BaseException:
        h.close()
        raise
    return cfg, h, ref, st


# ------------------------------------------------------------------ acting across env counts
# learning_starts = N k with k = 4 makes every N act from the policy from iteration 5 on; the first learning step is at
# iteration 8 (train_freq 8), after that iteration's acting. Episodes of 3 steps end at iterations 3 (warm-up) and 6
# (policy), and the reset of iteration 3 is observed from iteration 4 on, that of iteration 6 from iteration 7 on.
INV_K, INV_T = 4, 8
INV_NS = [1, 31, 32, 33, 100, 4096, 4097]
INV_BASE = 4097


def invariance_kw(N):
    return dict(num_envs=N, buffer_size=INV_T * N, learning_starts=INV_K * N, train_freq=INV_T, max_episode_steps=3)


_acting_cache = {}


def acting_run(abi, algo, N):
    """(ring, stats) of INV_T iterations at N envs; nothing wraps (the ring holds exactly INV_T N transitions)"""
    if (algo, N) not in _acting_cache:
        _, h, _ = make(abi, algo, invariance_kw(N))
        try:
            st = h.run(INV_T)
            _acting_cache[(algo, N)] = (h.read_buffer(), st)
        finally:
            h.close()
    return _acting_cache[(algo, N)]


@pytest.mark.parametrize("N", INV_NS)
@pytest.mark.parametrize("algo", ALGOS)
def test_acting_is_bit_identical_across_env_counts(crl, abi, torch_cuda, algo, N):
    """ring slot (i-1) N + n of the N-env run equals slot (i-1) 4097 + n of the 4097-env run bit for bit, for every
    env n < N and iteration i, in warm-up and policy acting alike"""
    buf, st = acting_run(abi, algo, N)
    base, _ = acting_run(abi, algo, INV_BASE)
    assert (buf["size"], buf["ptr"]) == (INV_T * N, 0)
    for k in ("obs", "next_obs", "action", "reward", "terminal"):
        got = buf[k].reshape((INV_T, N) + buf[k].shape[1:])
        want = base[k].reshape((INV_T, INV_BASE) + base[k].shape[1:])[:, :N]
        bad = np.argwhere(got != want)
        assert len(bad) == 0, "%s: %d elements differ, first at (iteration, env) %s" % (k, len(bad), tuple(bad[0][:2] + [1, 0]))
    # every env truncates at iterations 3 and 6: 2 episodes of 3 steps each
    assert (st.episodes, st.sum_length, st.iterations) == (2 * N, 6.0 * N, INV_T)


@pytest.mark.parametrize("algo", ALGOS)
def test_acting_at_4097_envs_matches_the_reference(crl, olib, abi, torch_cuda, algo):
    """the 4097-env run the invariance test compares with: its ring and episode statistics against the float64
    reference (129 acting CTAs, the last with one env)"""
    cfg, h, ref, st = run_against_reference(olib, abi, algo, invariance_kw(INV_BASE), [INV_T])
    try:
        buf = h.read_buffer()
        assert (buf["size"], buf["ptr"]) == (ref.size, ref.ptr)
        assert_ring_close(buf, ref)
        assert (st.learn_steps, ref.learn_steps) == (1, 1)   # after the acting of iteration 8
        assert st.kernel_launches == expected_launches(algo, cfg, [INV_T]) == 1 + 2
    finally:
        h.close()


# ------------------------------------------------------------------ splitting a run across calls
SPLITS = {   # name: (config overrides, iterations, calls of the split run)
    # warm-up spans three launches (1024 + 1024 + 53 iterations); the first policy step and the first learning step are
    # the last iteration of the third launch
    "warmup_over_three_launches": (dict(num_envs=1, buffer_size=4096, learning_starts=2100, batch_size=64), 2300,
                                   [1, 1023, 1, 1024, 0, 251]),
    # policy acting from iteration 101, learning every 1100 iterations: acting launches are split at ACT_MAX_STEPS,
    # not by a learning step; the ring of 4000 wraps at iteration 1334 and is sampled at a non-power-of-two size
    "policy_over_act_max_steps": (dict(num_envs=3, buffer_size=4000, learning_starts=300, batch_size=64, train_freq=1100,
                                       policy_frequency=1), 3300, [1, 1023, 1, 1024, 1025, 226]),
    # every launch is bounded by the ring: at most 2 iterations of 5 envs in a ring of 12
    "ring_bounded_launches": (dict(num_envs=5, buffer_size=12, learning_starts=40, batch_size=8, train_freq=3), 200,
                              [1, 2, 1, 3, 50, 143]),
    # the benchmark's ring: launches of at most 256 iterations, learning from iteration 251 at batch 256
    "bench_ring": (dict(num_envs=4096, buffer_size=1 << 20, learning_starts=250 * 4096, batch_size=256), 300,
                   [1, 127, 1, 128, 43]),
}


def run_in_calls(abi, algo, kw, calls):
    cfg, h, _ = make(abi, algo, kw)
    try:
        stats = [h.run(n) for n in calls]
        return cfg, stats, h.read_buffer(), h.get_params(), h.get_adam_state()
    finally:
        h.close()


@pytest.mark.parametrize("name", list(SPLITS))
@pytest.mark.parametrize("algo", ALGOS)
def test_a_run_split_across_calls_is_bit_identical(crl, abi, torch_cuda, algo, name):
    kw, iters, calls = SPLITS[name]
    assert sum(calls) == iters
    cfg, (one,), buf1, p1, m1 = run_in_calls(abi, algo, kw, [iters])
    _, split, buf2, p2, m2 = run_in_calls(abi, algo, kw, calls)
    learn, actor = closed_form_counts(cfg, iters)
    assert learn > 0 and actor > 0
    for st, c in ((one, [iters]), (split[-1], calls)):
        assert (st.learn_steps, st.actor_steps, st.iterations) == (learn, actor, iters)
        assert st.kernel_launches == expected_launches(algo, cfg, c)
    assert T.acting_launches(cfg, calls) > T.acting_launches(cfg, [iters])
    for k in buf1:
        assert np.array_equal(buf1[k], buf2[k]), "ring " + k
    for k in p1:
        assert np.array_equal(p1[k], p2[k]), k
    for k in m1:
        assert np.array_equal(m1[k], m2[k]), k
    for key, _ in LOSSES[algo] + [("actor_loss", None)]:
        assert getattr(one, key) == getattr(split[-1], key), key
    assert one.episodes > 0
    assert (one.episodes, one.sum_length) == (sum(s.episodes for s in split), sum(s.sum_length for s in split))
    np.testing.assert_allclose(sum(s.sum_return for s in split), one.sum_return, rtol=1e-12)


# ------------------------------------------------------------------ the run loop against float64 at scale
# Episodes of at most 25 steps keep the ring comparable: Pendulum spreads a one-ulp difference of the state (GPU and
# oracle sinf/cosf, or the Float32 actor) over 0.02 % of the observations after 30 steps and 5.5 % after 200, while resets
# are exact. Every case runs in two calls, the boundary inside an episode.
SCALE_RUNS = {   # name: (config overrides, calls)
    "bench_shape": (dict(num_envs=4096, buffer_size=1 << 20, learning_starts=10_000, batch_size=256, max_episode_steps=5),
                    [6, 6]),
    # the ring of 1,000,000 (not a multiple of 4096) wraps inside iteration 245; learning from iteration 246 samples
    # batches of 256 from all 1,000,000 rows
    "wrapped_ring": (dict(num_envs=4096, buffer_size=1_000_000, learning_starts=245 * 4096, batch_size=256,
                          max_episode_steps=25), [130, 123]),
    "ragged_multi_cta": (dict(num_envs=100, buffer_size=5000, learning_starts=1000, batch_size=256, policy_frequency=3,
                              max_episode_steps=20), [27, 33]),
    "warmup_over_three_launches": (dict(num_envs=1, buffer_size=4096, learning_starts=2100, batch_size=64,
                                        max_episode_steps=25), [1090, 1050]),
    "policy_over_act_max_steps": (dict(num_envs=3, buffer_size=4000, learning_starts=300, batch_size=64, train_freq=1100,
                                       policy_frequency=1, max_episode_steps=25), [1510, 790]),
}


@pytest.mark.parametrize("name", list(SCALE_RUNS))
@pytest.mark.parametrize("algo", ALGOS)
def test_run_loop_at_scale_matches_the_reference(crl, olib, abi, torch_cuda, algo, name):
    """the assertions of the other run-loop tests (counts, launches, size and ptr, parameters by assert_run_close, Adam
    moments, beta powers, losses) plus TD3's ring rule and each call's episode statistics"""
    kw, calls = SCALE_RUNS[name]
    iters = sum(calls)
    cfg, h, ref, st = run_against_reference(olib, abi, algo, kw, calls)
    try:
        learn, actor = closed_form_counts(cfg, iters)
        assert learn > 0 and actor > 0
        assert (st.learn_steps, st.actor_steps, st.iterations) == (learn, actor, iters)
        assert (ref.learn_steps, ref.actor_steps) == (learn, actor)
        assert st.kernel_launches == expected_launches(algo, cfg, calls)
        buf = h.read_buffer()
        assert (buf["size"], buf["ptr"]) == (ref.size, ref.ptr)
        assert_ring_close(buf, ref)
        p, m = h.get_params(), h.get_adam_state()
        nets = [("actor", "actor", "am", "av", R.ACTOR_ARRAYS, actor)] + \
               [(k, a, mm, mv, R.CRITIC_ARRAYS, learn) for k, a, mm, mv in CRITICS[algo]]
        for key, attr, mm, mv, arrays, steps in nets:
            assert_run_close(p[key], getattr(ref, attr), arrays, cfg.lr, steps, key + " ")
            assert_run_close(p[key + "_target"], getattr(ref, attr + "_tgt"), arrays, cfg.lr, steps, key + "_target ")
            # a gradient element that cancels to near 0 has a large relative error in Float32 (and may flip sign), so
            # up to 0.1 % of an array may be off; the rest agree at rtol 1e-3
            for suffix, r in (("_m", getattr(ref, mm)), ("_v", getattr(ref, mv))):
                for nm, s, e in arrays:
                    d = np.abs(m[key + suffix][s:e] - r[s:e])
                    bad = d > 1e-3 * np.abs(r[s:e]) + 1e-6 * np.abs(r[s:e]).max()
                    assert bad.sum() <= max(1, (e - s) // 1000), "%s%s%s: %d elements off" % (key, suffix, nm, bad.sum())
        np.testing.assert_allclose(m["beta_pow"], [0.9 ** (actor + 1), 0.999 ** (actor + 1), 0.9 ** (learn + 1), 0.999 ** (learn + 1)],
                                   rtol=1e-12)
        for key, attr in LOSSES[algo] + [("actor_loss", "actor_loss")]:
            np.testing.assert_allclose(getattr(st, key), getattr(ref, attr), rtol=1e-4, err_msg=key)
    finally:
        h.close()
