"""TD3 on the GPU (include/cleanrl_td3.h) against the float64 reference of tests/td3_reference.py.

* crl_td3_critic_loss_raw (the twin-critic forward kernel and the twin reduction, gradients out) for both critics per
  parameter array, at every 16-sample CTA boundary of the batch and on edge batches, with the smoothing draw inside the
  kernel under test; its agreement with crl_ddpg_critic_loss_raw bit for bit when the noise is off.
* crl_td3_run against RefTD3 on shared Philox streams, the closed-form counts, acting identical to DDPG before the first
  learning step, determinism, a learning run of td3() and the CLI.
Run with `pytest -m gpu` on a B200."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import ddpg_reference as R
import td3_reference as T
from test_ddpg import rand_nets
from test_gpu_ddpg import RUNS, assert_grad_close, assert_run_close, closed_form_counts, dev, gpu_critic
from test_td3 import KINDS, td3_batch

pytestmark = pytest.mark.gpu
F = np.float32
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def gpu_twin(crl, torch, d, B=None, learn_step=None, seed=None, nc=None):
    B = len(d["act"]) if B is None else B
    g1 = torch.full((R.CRITIC_P,), float("nan"), dtype=torch.float32, device="cuda")
    g2 = torch.full((R.CRITIC_P,), float("nan"), dtype=torch.float32, device="cuda")
    l1 = torch.full((1,), float("nan"), dtype=torch.float64, device="cuda")
    l2 = torch.full((1,), float("nan"), dtype=torch.float64, device="cuda")
    t = [dev(torch, d[k]) for k in ("at", "q1", "q2", "q1t", "q2t", "obs", "act", "rew", "nobs", "term")]
    crl.check(crl.load().crl_td3_critic_loss_raw(
        *[crl.ptr(x) for x in t[:5]], B, *[crl.ptr(x) for x in t[5:]], d["gamma"], d["pn"], d["nc"] if nc is None else nc,
        SEED if seed is None else seed, d["learn_step"] if learn_step is None else learn_step,
        crl.ptr(g1), crl.ptr(g2), crl.ptr(l1), crl.ptr(l2), None))
    torch.cuda.synchronize()
    return g1.cpu().numpy(), g2.cpu().numpy(), float(l1.cpu().numpy()[0]), float(l2.cpu().numpy()[0])


SEED = 0x5EED_0001_0002
BATCHES = [1, 15, 16, 17, 31, 32, 33, 100, 255, 256]


# ------------------------------------------------------------------ loss and gradient
@pytest.mark.parametrize("B", BATCHES)
@pytest.mark.parametrize("kind", KINDS)
def test_td3_critic_loss_raw_matches_float64(crl, olib, torch_cuda, kind, B):
    """both gradients per parameter array at rtol 1e-4 with atol 2e-6 max|g| (DDPG's tolerance), the losses at rtol 1e-6;
    the smoothing noise is drawn inside the kernel and by the reference from Philox stream 7 (philox_draw_many)"""
    d = td3_batch(kind, B, 9 * B + KINDS.index(kind))
    g1, g2, l1, l2 = gpu_twin(crl, torch_cuda, d)
    z = T.smoothing_normals(SEED, d["learn_step"], B)
    r1, r2, rg1, rg2 = T.twin_critic_loss_grad(d["at"], d["q1"], d["q2"], d["q1t"], d["q2t"], d["obs"], d["act"], d["rew"],
                                               d["nobs"], d["term"], d["gamma"], z, d["pn"], d["nc"])
    np.testing.assert_allclose([l1, l2], [r1, r2], rtol=1e-6)
    assert_grad_close(g1, rg1, R.CRITIC_ARRAYS, "qf1 %s B=%d " % (kind, B))
    assert_grad_close(g2, rg2, R.CRITIC_ARRAYS, "qf2 %s B=%d " % (kind, B))
    if len(d["zero"]):
        assert np.all(g1[d["zero"]] == 0.0) and np.all(g2[d["zero"]] == 0.0)


@pytest.mark.parametrize("B", [1, 17, 100, 255])
def test_td3_critic_loss_raw_reads_nothing_past_row_B(crl, torch_cuda, B):
    d = td3_batch("mixed", B, B)
    r0 = gpu_twin(crl, torch_cuda, d)
    pad = lambda x, v: np.concatenate([x, np.full((7,) + x.shape[1:], v, x.dtype)])
    p = dict(d, obs=pad(d["obs"], np.nan), act=pad(d["act"], np.nan), rew=pad(d["rew"], np.nan), nobs=pad(d["nobs"], np.nan),
             term=pad(d["term"], 1))
    r1 = gpu_twin(crl, torch_cuda, p, B=B)
    assert np.array_equal(r0[0], r1[0]) and np.array_equal(r0[1], r1[1]) and r0[2:] == r1[2:]


def test_td3_smoothing_noise_depends_on_the_learning_step_only_through_the_clip(crl, torch_cuda):
    d = td3_batch("mixed", 64, 3)
    a = gpu_twin(crl, torch_cuda, d, learn_step=10)
    b = gpu_twin(crl, torch_cuda, d, learn_step=11)
    c = gpu_twin(crl, torch_cuda, d, learn_step=10, seed=SEED + 1)
    assert not np.array_equal(a[0], b[0]) and a[2] != b[2] and not np.array_equal(a[0], c[0])
    a = gpu_twin(crl, torch_cuda, d, learn_step=10, nc=0.0)
    b = gpu_twin(crl, torch_cuda, d, learn_step=(1 << 40) + 3, nc=0.0)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and a[2:] == b[2:]


@pytest.mark.parametrize("B", [1, 16, 33, 256])
@pytest.mark.parametrize("kind", ["mixed", "terminal", "relu0"])
def test_td3_with_the_noise_off_and_equal_twins_is_ddpg_bit_for_bit(crl, torch_cuda, kind, B):
    """noise_clip 0, qf1 = qf2 and qf1' = qf2': mu' is inside [-2, 2], so y is DDPG's target exactly, and both TD3
    gradients and losses equal crl_ddpg_critic_loss_raw's"""
    d = td3_batch(kind, B, 21 * B + KINDS.index(kind))
    d.update(q2=d["q1"], q2t=d["q1t"], nc=0.0, pn=0.7)
    g1, g2, l1, l2 = gpu_twin(crl, torch_cuda, d)
    gd, ld = gpu_critic(crl, torch_cuda, d["at"], d["q1"], d["q1t"], d["obs"], d["act"], d["rew"], d["nobs"], d["term"], d["gamma"])
    assert np.array_equal(g1, gd) and np.array_equal(g2, gd) and l1 == ld and l2 == ld


@pytest.mark.parametrize("kind", ["mixed", "noise_clamp", "action_clamp"])
def test_td3_equal_twins_give_bit_identical_gradients(crl, torch_cuda, kind):
    d = td3_batch(kind, 100, 31 + KINDS.index(kind))
    d.update(q2=d["q1"])
    g1, g2, l1, l2 = gpu_twin(crl, torch_cuda, d)
    assert np.array_equal(g1, g2) and l1 == l2


# ------------------------------------------------------------------ run loop
def make_handle(abi, kw, a, q1, q2, seed=3):
    from cleanrl_jl_b200.td3_algo import TD3Handle
    cfg = abi.make_td3_config(**{**dict(exploration_noise=0.1, lr=1e-3, tau=0.05, seed=seed, policy_noise=0.2, noise_clip=0.5), **kw})
    h = TD3Handle(cfg)
    h.set_params(a, q1, q2)
    h.reset()
    return cfg, h


@pytest.mark.parametrize("name", list(RUNS))
def test_td3_run_loop_matches_the_reference(crl, olib, abi, torch_cuda, name):
    """DDPG's run-loop tolerance: rtol 1e-4 with an atol of 1e-6 max|ref| per array, except that at most 0.1 % of an
    array (and at least 1 element) may differ by at most 2 lr per step taken: a gradient element that cancels to within
    Float32 rounding can flip sign, and Adam's first steps then move it by about lr the other way"""
    kw, iters = RUNS[name]
    a, q1 = rand_nets(17)
    _, q2 = rand_nets(18)
    cfg, h = make_handle(abi, kw, a, q1, q2)
    ref = T.RefTD3(olib, cfg, a, q1, q2)
    learn, actor = closed_form_counts(cfg, iters)
    first_actor_it = next((it for it in range(1, iters + 1) if closed_form_counts(cfg, it)[1] > 0), None)
    try:
        if first_actor_it is not None and first_actor_it > 1:   # the targets are the initial copies until the first actor step
            calls = [first_actor_it - 1, iters - first_actor_it + 1]
            h.run(calls[0])
            p = h.get_params()
            assert np.array_equal(p["actor_target"], a) and np.array_equal(p["qf1_target"], q1) and np.array_equal(p["qf2_target"], q2)
            ref.run(calls[0])
            h.run(calls[1])
            ref.run(calls[1])
        else:
            calls = [iters]
            h.run(iters)
            ref.run(iters)
        st = h.run(0)
        assert (st.learn_steps, st.actor_steps, st.iterations) == (learn, actor, iters)
        assert (ref.learn_steps, ref.actor_steps) == (learn, actor)
        assert st.kernel_launches == T.acting_launches(cfg, calls) + 2 * learn + 4 * actor
        buf = h.read_buffer()
        assert (buf["size"], buf["ptr"]) == (ref.size, ref.ptr)
        # the ring: rtol 1e-5 during warm-up. Once the actor acts, it may differ from the reference's as assert_run_close
        # allows, and Pendulum carries that into the states, so then rtol 1e-4 with up to 0.1 % of an array (at least 1
        # element) at rtol 1e-3
        for k, r in (("obs", ref.b_obs), ("next_obs", ref.b_next), ("action", ref.b_act), ("reward", ref.b_rew)):
            if learn == 0:
                np.testing.assert_allclose(buf[k], r, rtol=1e-5, atol=1e-6, err_msg=k)
                continue
            d, ar = np.abs(buf[k] - r), np.abs(r)
            bad = d > 1e-4 * ar + 1e-5
            assert bad.sum() <= max(1, r.size // 1000) and np.all(d[bad] <= 1e-3 * ar[bad] + 1e-4), \
                "%s: %d elements off, worst %g" % (k, bad.sum(), d.max())
        np.testing.assert_array_equal(buf["terminal"], ref.b_term)
        p, m = h.get_params(), h.get_adam_state()
        for key, r, arrays, steps in (("qf1", ref.critic, R.CRITIC_ARRAYS, learn), ("qf1_target", ref.critic_tgt, R.CRITIC_ARRAYS, learn),
                                      ("qf2", ref.qf2, R.CRITIC_ARRAYS, learn), ("qf2_target", ref.qf2_tgt, R.CRITIC_ARRAYS, learn),
                                      ("actor", ref.actor, R.ACTOR_ARRAYS, actor), ("actor_target", ref.actor_tgt, R.ACTOR_ARRAYS, actor)):
            assert_run_close(p[key], r, arrays, cfg.lr, steps, key + " ")
        for key, r, arrays in (("qf1_m", ref.cm, R.CRITIC_ARRAYS), ("qf2_m", ref.q2m, R.CRITIC_ARRAYS), ("actor_m", ref.am, R.ACTOR_ARRAYS),
                               ("qf1_v", ref.cv, R.CRITIC_ARRAYS), ("qf2_v", ref.q2v, R.CRITIC_ARRAYS), ("actor_v", ref.av, R.ACTOR_ARRAYS)):
            for nm, s, e in arrays:
                d = np.abs(m[key][s:e] - r[s:e])
                bad = d > 1e-3 * np.abs(r[s:e]) + 1e-6 * np.abs(r[s:e]).max()
                assert bad.sum() <= max(1, (e - s) // 1000), "%s%s: %d elements off" % (key, nm, bad.sum())
        np.testing.assert_allclose(m["beta_pow"], [0.9 ** (actor + 1), 0.999 ** (actor + 1), 0.9 ** (learn + 1), 0.999 ** (learn + 1)],
                                   rtol=1e-12)
        if learn:
            np.testing.assert_allclose([st.qf1_loss, st.qf2_loss], [ref.critic_loss, ref.qf2_loss], rtol=1e-4)
        if actor:
            np.testing.assert_allclose(st.actor_loss, ref.actor_loss, rtol=1e-4)
        if name == "truncated_at_10":
            assert ref.b_term.sum() > 0
    finally:
        h.close()


def test_td3_and_ddpg_act_alike_until_the_first_learning_step(crl, abi, torch_cuda):
    from cleanrl_jl_b200.ddpg_algo import DDPGHandle
    kw = dict(num_envs=64, buffer_size=4096, learning_starts=1000, batch_size=64, seed=11)
    a, q1 = rand_nets(4)
    _, q2 = rand_nets(5)
    cfg, h = make_handle(abi, kw, a, q1, q2, seed=11)
    dd = DDPGHandle(abi.make_ddpg_config(**{**dict(exploration_noise=0.1, lr=1e-3, tau=0.05), **kw}))
    try:
        dd.set_params(a, q1)
        dd.reset()
        first_learn = 1000 // 64 + 1                     # gs = 64 it > 1000 from it = 16
        for x in (h, dd):
            x.run(first_learn)
        bt, bd = h.read_buffer(), dd.read_buffer()
        for k in ("obs", "next_obs", "action", "reward", "terminal", "size", "ptr"):
            assert np.array_equal(bt[k], bd[k]), k
        assert h.run(0).learn_steps == 1 and dd.run(0).learn_steps == 1
        # the second learning step (iteration 17) is the first actor step, against different critics: from iteration
        # 18 on the two actors differ
        for x in (h, dd):
            x.run(2)
        assert not np.array_equal(h.read_buffer()["action"], dd.read_buffer()["action"])
    finally:
        h.close()
        dd.close()


def test_td3_run_is_deterministic(crl, abi, torch_cuda):
    a, q1 = rand_nets(2)
    _, q2 = rand_nets(3)
    out = []
    for _ in range(2):
        _, h = make_handle(abi, dict(num_envs=300, buffer_size=20_000, learning_starts=1000, batch_size=256), a, q1, q2, seed=9)
        st = h.run(40)
        out.append((h.get_params(), st.qf1_loss, st.qf2_loss, st.actor_loss))
        h.close()
    for k in out[0][0]:
        assert np.array_equal(out[0][0][k], out[1][0][k]), k
    assert out[0][1:] == out[1][1:]


# ------------------------------------------------------------------ learning and CLI
LEARN_STEPS = 30_000
LEARN_MIN_RETURN = -700.0
LEARN_MIN_GAIN = 400.0


def test_td3_learns_pendulum(torch_cuda, tmp_path):
    """CleanRL's settings with one env and learning from step 5,000: mean episode return over the last 5,000 steps
    against the first 5,000 (uniform random torques), with DDPG's bar. On one B200 (1000 W, seed 1) this run went from
    -1248.2 to -170.7; the thresholds below leave a wide margin under that."""
    from cleanrl_jl_b200 import TD3Config, td3
    from cleanrl_jl_b200 import logger as Logger
    lg = Logger.make_logger("td3", to_terminal=False, to_tensorboard=False, to_json=True, log_dir=str(tmp_path))
    cfg = TD3Config(total_timesteps=LEARN_STEPS, learning_starts=5_000, buffer_size=LEARN_STEPS, log_frequency=1000, seed=1)
    try:
        res = td3(cfg, logger=lg)
    finally:
        lg.close()
    recs = [json.loads(l) for l in open(tmp_path / "td3.json")]
    ep = [r["kwargs"] for r in recs if r["msg"] == "Episode Statistics"]
    tr = [r["kwargs"] for r in recs if r["msg"] == "Training Statistics"]
    assert ep and tr and {"episode_return", "episode_length", "global_step", "steps_per_sec"} <= set(ep[0]) \
        and {"qf1_loss", "qf2_loss", "actor_loss"} <= set(tr[-1])
    r = np.array(res["episode_returns"])
    assert res["learn_steps"] == LEARN_STEPS - 5_000 and res["actor_steps"] == (LEARN_STEPS - 5_000) // 2
    first, last = r[:5].mean(), r[-5:].mean()
    print("td3 learning: first 5k steps %.1f, last 5k steps %.1f" % (first, last))
    assert last > LEARN_MIN_RETURN and last - first > LEARN_MIN_GAIN, (first, last)


def test_cli_runs_td3(torch_cuda, tmp_path):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "cleanrl_jl_b200.py"), "td3", "--num_envs", "64", "--total_timesteps",
                        "12800", "--learning_starts", "2000", "--buffer_size", "8192", "--policy_noise", "0.3"], cwd=str(tmp_path),
                       capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    res = json.loads(p.stdout.strip().splitlines()[-1])
    assert res["algorithm"] == "td3" and res["global_step"] == 12800 and res["learn_steps"] > 0 and res["steps_per_sec"] > 0
    assert np.isfinite(res["qf1_loss"]) and np.isfinite(res["qf2_loss"])
