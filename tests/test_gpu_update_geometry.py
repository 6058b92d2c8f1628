"""The tcgen05 3xTF32 update (csrc/update_tc.cu), which runs every production minibatch, against the CPU oracle at
minibatch sizes that end mid-tile on both sides of each launch-geometry boundary of loss_grad_tc_plan: in its exact form
(crl_update_minibatch: TC kernel, then the reduce and clip+Adam kernels) and with the fused reduce / ClipNorm / Adam
tail (crl_train_update). The other GPU tests run minibatches of 32, 256, 1920 or a whole number of 1024 tiles and the
default loss coefficients only. Here the loss, GAE and optimiser also run at the two coefficient sets of
test_oracle_coefficients.py, and DQN acts at env counts that leave its last CTA partly filled, with a replay ring that
wraps in the middle of an iteration. Tolerances are those of the existing comparisons they extend (named per check)."""
import numpy as np
import pytest
import torch

from conftest import rand_params
from oracle.oracle import OracleDQN
from test_gpu_parity import BUF_FIELDS, dev, make_pair
from test_oracle_coefficients import SETS, assert_clip_branch, config_kw, loss_coefs
from test_oracle_grad import make_batch, torch_loss

pytestmark = pytest.mark.gpu
F = np.float32
RTOL = 1e-5
TC_S = 128                              # samples per tile of the tcgen05 kernel
SWEEP_N, SWEEP_T = 1024, 64             # one 65,536-sample rollout; num_minibatches = 1 admits any M in [2, 65536]
SWEEP_B = SWEEP_N * SWEEP_T
LR = float(F(2.5e-4))
UPDATE_FIELDS = ["STATE", "ACTION", "LOGPROB", "ADVANTAGE", "RETURN", "VALUE"]


def sweep_sizes(sm):
    """Minibatch sizes around every boundary of loss_grad_tc_plan (grid = 2 * n_tiles below the SM count, the whole
    GPU from there on; actor and critic CTAs each run ceil(n_tiles / CTAs) tiles): 2 and 3 samples, one tile and its
    ragged neighbours, two tiles; the last grid of 2 * n_tiles CTAs and the first full one; one tile per CTA more or
    less, 1-2 and 3-5 tiles per CTA with a ragged tail; the handle's whole rollout and one sample less."""
    half = sm // 2
    ms = [2, 3, 33, 127, 128, 129, 255, 257,
          TC_S * (half - 1), TC_S * (half - 1) + 1, TC_S * half + 1,
          TC_S * sm - 1, TC_S * sm, TC_S * sm + 1, TC_S * 2 * sm + 77, SWEEP_B - 1, SWEEP_B]
    return sorted({m for m in ms if 2 <= m <= SWEEP_B})


def ragged_points(sm):
    """two sizes that end mid-tile: a small grid, and a full grid with CTAs that run one or two tiles"""
    return [129, TC_S * sm + 1]


def stats_of(s):
    return np.array([s.loss, s.pg_loss, s.v_loss, s.entropy_loss])


CRITIC_SHIFT = 0.15   # new value - recorded value for every sample: 0.05 or more from every clip_coef used here


def update_params(olib, kind, p_roll):
    """The parameters the update runs with. With the rollout's own parameters every probability ratio is 1 and every
    new value equals the recorded one, so neither the ratio clip nor the value clip (both clip_coef) would be active.
    The actor moves (CartPole: perturbed weights; Pendulum: a larger log-std, since a mean moved by many standard
    deviations leaves the recorded actions deep in the tails, where d logp / d mean = (a - mean) / var multiplies the
    rounding error of the mean tenfold). Only the critic's output bias moves, so that every new value sits
    CRITIC_SHIFT above the recorded one: a sample within rounding distance of the value-clip boundary would switch
    branch between two correct implementations and change the gradient by |v - R| / M."""
    off, size = olib.param_layout(kind)
    p = p_roll.copy()
    if kind == 0:
        p[:off[6]] += (0.03 * np.random.default_rng(77).standard_normal(off[6])).astype(F)
    else:
        p[-1] = p_roll[-1] + 0.1
    p[off[11]] += CRITIC_SHIFT
    return p


def warm_adam(olib, kind):
    """Second moments ten steps into training, set identically on both sides before every point. From zero moments the
    first step is lr * g / (|g| + eps), i.e. lr * sign(g): a parameter comparison would check signs only and would be
    ill-conditioned wherever g is near zero. Second moments of the order of a squared gradient element make the step a
    smooth function of the gradient. First moments start at zero, so that m' = 0.1 * clipped gradient."""
    d = olib.dims(kind)
    m = np.zeros(d["P"], F)
    v = (np.random.default_rng(41 + kind).uniform(0.5, 1.5, d["P"]) * 1e-6).astype(F)
    bp = np.tile(np.array([0.9 ** 10, 0.999 ** 10]), (d["n_arrays"], 1))
    return m, v, bp


def sweep_pair(crl, olib, abi, kind, **kw):
    """handle + oracle on identical rollout buffers: device-RNG rollout and GAE on the GPU, GAE checked bit-exact
    against the oracle's recurrence on the GPU's own inputs (so cfg.gamma / cfg.gae_lambda reach the kernel), then the
    GPU's buffers copied into the oracle"""
    h, o = make_pair(crl, olib, abi, kind, N=SWEEP_N, T=SWEEP_T, mb=1, epochs=1, seed=31, **kw)
    if kind == 1:
        # the Gaussian mean head at its initial scale instead of rand_params' 30x (means of +-20 for actions in
        # [-2, 2]): the 3xTF32 bound of test_gpu_tc is stated for network outputs of that order; with the 30x head the
        # tensor-core actor W1 gradient is 2-7e-6 of the array's largest element away from float64 autograd
        off, size = olib.param_layout(kind)
        p = h.get_params()
        p[off[4]:off[4] + size[4]] /= 30.0
        h.set_params(p)
        o.set_params(p)
    t0 = spread_episode_clocks(abi, h)
    h.rollout()
    assert_truncated(h.pop_episodes()[0], t0, h.cfg.max_episode_steps)
    h.gae()
    rd = lambda name: h.read_field(getattr(abi, "CRL_F_" + name))
    cfg = h.cfg
    adv_o, ret_o = olib.gae_raw(rd("VALUE"), rd("REWARD"), rd("TERMINAL"), rd("NEXT_VALUE"), rd("NEXT_DONE"),
                                F(cfg.gamma), F(cfg.gae_lambda), cfg.gae_mode)
    np.testing.assert_array_equal(rd("ADVANTAGE"), adv_o)
    np.testing.assert_array_equal(rd("RETURN"), ret_o)
    for name in BUF_FIELDS + ["ADVANTAGE", "RETURN"]:
        o.write_field(getattr(abi, "CRL_F_" + name), rd(name))
    return h, o


def spread_episode_clocks(abi, *xs):
    """reset, then start the episode clocks spread over [0, max_episode_steps), every tenth env one step before the cap,
    so that episodes are truncated inside the rollouts"""
    h = xs[0]
    h.env_reset()
    st = h.read_field(abi.CRL_F_ENV_STATE)
    t0 = np.random.default_rng(h.N).integers(0, h.cfg.max_episode_steps, h.N).astype(np.int32)
    t0[::10] = h.cfg.max_episode_steps - 1
    for x in xs:
        x.env_set_state(st, t0)
    return t0


def assert_truncated(recs, t0, cap):
    """every env started one step before the cap ended its episode within the first two steps of the rollout"""
    assert np.any(t0 == cap - 1)
    assert set(np.nonzero(t0 == cap - 1)[0]) <= {r[1] for r in recs if r[0] <= 1}


def flat_inputs(h, abi):
    """the update's inputs as flat [B, ...] arrays (flat index n + N t)"""
    B = h.B
    out = {}
    for name in UPDATE_FIELDS:
        a = h.read_field(getattr(abi, "CRL_F_" + name))
        out[name] = a.reshape(B, -1) if name == "STATE" or (name == "ACTION" and h.continuous) else a.reshape(B)
    return out


def random_idx(B, M, seed, ends=False):
    idx = np.random.default_rng(seed).permutation(B)[:M].astype(np.int32)
    if ends:  # contains buffer entries 0 and B-1 (at the first and the last lane)
        idx = np.concatenate([[0], idx[(idx != 0) & (idx != B - 1)][:M - 2], [B - 1]]).astype(np.int32)
    return idx


def compare_point(h, o, olib, abi, kind, p, adam, idx, label):
    """one crl_update_minibatch on both sides from identical parameters and Adam state; returns the oracle's raw
    gradient and the GPU's (stats, gradient)"""
    M = len(idx)
    for x in (h, o):
        x.set_params(p)
        x.set_adam_state(*adam)
    sh, so = stats_of(h.update_minibatch(idx, LR)), stats_of(o.update_minibatch(idx, LR))
    np.testing.assert_allclose(sh, so, rtol=1e-5, atol=1e-6, err_msg=label)
    gh, go = h.get_grads(), o.get_grads()
    off, size = olib.param_layout(kind)
    mh, _, bph = h.get_adam_state()
    mo, _, bpo = o.get_adam_state()
    for i in range(len(off)):
        sl = slice(off[i], off[i] + size[i])
        # the 3xTF32 bound of test_gpu_tf32x3 / test_gpu_tc: within ~1e-6 of the largest element of the array
        np.testing.assert_allclose(gh[sl], go[sl], rtol=1e-4, atol=3e-6 * np.abs(go[sl]).max() + 1e-12,
                                   err_msg="%s: gradient array %d" % (label, i))
        # m' = 0.1 * clipped gradient: the same bound on the gradient the optimiser saw
        np.testing.assert_allclose(mh[sl], mo[sl], rtol=1e-4, atol=3e-6 * np.abs(mo[sl]).max() + 1e-12,
                                   err_msg="%s: Adam m array %d" % (label, i))
    np.testing.assert_allclose(bph, bpo, rtol=1e-14, err_msg=label)
    np.testing.assert_allclose(h.read_field(abi.CRL_F_VNEW)[:M], o.read_field(abi.CRL_F_VNEW)[:M], rtol=RTOL, atol=2e-6,
                               err_msg=label + ": VNEW")
    np.testing.assert_allclose(h.get_params(), o.get_params(), rtol=RTOL, atol=1e-6, err_msg=label + ": parameters")
    return go, sh, gh


def compare_autograd(olib, kind, h, abi, p, idx, st, g, coefs):
    """the GPU's raw gradient and loss statistics against float64 autograd, at the tolerance of test_oracle_grad"""
    d = olib.dims(kind)
    x = flat_inputs(h, abi)
    c, ent_c, v_c = coefs
    pt = torch.tensor(p.astype(np.float64), requires_grad=True)
    loss, pg, vl, en = torch_loss(pt, olib.param_layout(kind), d, idx.astype(np.int64), x["STATE"], x["ACTION"],
                                  x["LOGPROB"], x["ADVANTAGE"], x["RETURN"], x["VALUE"], c, ent_c, v_c, kind == 1)
    loss.backward()
    gt = pt.grad.numpy()
    np.testing.assert_allclose(st, [loss.item(), pg.item(), vl.item(), en.item()], rtol=2e-5, atol=1e-6)
    np.testing.assert_allclose(g, gt, rtol=2e-3, atol=2e-5 * np.abs(gt).max())


# ------------------------------------------------------------------ A. exact path, M sweep
@pytest.mark.parametrize("kind", [0, 1])
def test_exact_update_matches_oracle_across_the_tile_geometry(crl, olib, abi, torch_cuda, kind):
    sm = torch_cuda.cuda.get_device_properties(0).multi_processor_count
    olib.set_threads(8)
    try:
        h, o = sweep_pair(crl, olib, abi, kind)
        p = update_params(olib, kind, h.get_params())
        adam = warm_adam(olib, kind)
        sizes = sweep_sizes(sm)
        assert TC_S * (sm // 2 - 1) in sizes and TC_S * sm + 1 in sizes
        for M in sizes:
            idx = random_idx(SWEEP_B, M, seed=1000 + M, ends=(M == 2 or M == TC_S * sm + 1))
            go, st, gh = compare_point(h, o, olib, abi, kind, p, adam, idx, "M=%d" % M)
            if M in (2, 129, TC_S * sm + 1):
                compare_autograd(olib, kind, h, abi, p, idx, st, gh, (h.cfg.clip_coef, h.cfg.ent_coeff, h.cfg.v_coef))
        # Poisoned tail: NaN in every entry the minibatch does not select (a read of an unselected sample, or of a lane
        # past M, even one multiplied by zero, makes an output NaN); the oracle runs on the clean buffers
        clean = {name: h.read_field(getattr(abi, "CRL_F_" + name)) for name in UPDATE_FIELDS}
        poison = ["STATE", "ADVANTAGE", "LOGPROB", "RETURN", "VALUE"] + (["ACTION"] if kind == 1 else [])
        for M in ragged_points(sm):
            idx = random_idx(SWEEP_B, M, seed=2000 + M)
            keep = np.zeros(SWEEP_B, bool)
            keep[idx] = True
            for name in poison:
                a = clean[name].copy()
                a.reshape(SWEEP_B, -1)[~keep] = np.nan
                h.write_field(getattr(abi, "CRL_F_" + name), a)
            compare_point(h, o, olib, abi, kind, p, adam, idx, "poisoned M=%d" % M)
            for name in poison:
                h.write_field(getattr(abi, "CRL_F_" + name), clean[name])
        h.close()
    finally:
        olib.set_threads(1)


@pytest.mark.parametrize("kind", [0, 1])
@pytest.mark.parametrize("name", sorted(SETS))
def test_exact_update_matches_oracle_at_other_coefficients(crl, olib, abi, torch_cuda, kind, name):
    """two ragged points of the sweep on a handle configured with another coefficient set: the clip coefficient, loss
    weights, ClipNorm threshold, GAE gamma / lambda and the episode cap all reach the kernels"""
    sm = torch_cuda.cuda.get_device_properties(0).multi_processor_count
    olib.set_threads(8)
    try:
        h, o = sweep_pair(crl, olib, abi, kind, **config_kw(name, kind))
        p = update_params(olib, kind, h.get_params())
        adam = warm_adam(olib, kind)
        x = flat_inputs(h, abi)
        c = loss_coefs(name)[0]
        for M in ragged_points(sm):
            idx = random_idx(SWEEP_B, M, seed=3000 + M)
            go, _, _ = compare_point(h, o, olib, abi, kind, p, adam, idx, "%s M=%d" % (name, M))
            assert_clip_branch(name, go, olib.param_layout(kind))
            # some ratios fall outside [1 - clip_coef, 1 + clip_coef] and some inside
            _, logp_new, vnew = olib.policy_forward_raw(kind, p, x["STATE"][idx])
            if kind == 0:
                ratio = np.exp(logp_new[np.arange(M), x["ACTION"][idx]] - x["LOGPROB"][idx])
                assert 0 < np.sum(np.abs(ratio - 1) > c) < M
            # no sample near the value-clip boundary; the clip is active for every sample under set 1, for none under set 2
            dv = np.abs(vnew - x["VALUE"][idx])
            assert np.all(np.abs(dv - c) > 0.02)
            assert np.all(dv > c) == (c < CRITIC_SHIFT)
        h.close()
    finally:
        olib.set_threads(1)


# ------------------------------------------------------------------ B. fused tail at ragged M
SMALL = {  # name -> (kind, N, T, num_minibatches, A2C)
    "ppo_cartpole_175": (0, 100, 7, 4, False),      # 2 tiles, the second with 47 samples
    "ppo_pendulum_650": (1, 100, 13, 2, False),
    "a2c_cartpole_1300": (0, 100, 13, 1, True),
    "a2c_pendulum_18992": (1, 1187, 16, 1, True),   # 149 tiles, the last with 48 samples
}
SMALL_CASES = [(c, None) for c in SMALL] + [(c, s) for c in SMALL if not SMALL[c][4] for s in sorted(SETS)]


@pytest.mark.parametrize("case,coefs", SMALL_CASES)
def test_fused_update_matches_oracle_at_ragged_sizes(crl, olib, abi, torch_cuda, case, coefs):
    """crl_train_update (rollout, GAE and every minibatch through the fused tcgen05 kernel) for 3 updates against the
    oracle on the same Philox streams, as test_train_update_graph_matches_oracle; T <= 16 keeps fp32 divergence of the
    trajectories below the tolerance. Episode clocks start spread over [0, cap) so that episodes are truncated inside
    the rollouts. The first update runs with profiling on, which shows the fused kernel really ran."""
    kind, N, T, mb, a2c = SMALL[case]
    kw = config_kw(coefs, kind) if coefs else {}
    if a2c:
        kw.update(gae_mode=abi.CRL_GAE_A2C_RETURNS, flags=abi.CRL_FLAG_A2C, gae_lambda=1.0)
    epochs = 1 if a2c else 2
    h, o = make_pair(crl, olib, abi, kind, N=N, T=T, mb=mb, epochs=epochs, seed=37, **kw)
    o.env_reset()
    t0 = spread_episode_clocks(abi, h, o)
    h.profile(True)
    for u in range(3):
        lr = LR * (1 - u / 10)
        h.train_update(lr)
        sh, agg = h.fetch_update()
        if u == 0:
            prof = h.profile_read()
            assert prof["loss_grad"]["launches"] == epochs * mb, prof
            assert prof["grad_reduce"]["launches"] == 0 and prof["clip_adam"]["launches"] == 0, prof
            h.profile(False)
        so = o.train_update(lr)
        np.testing.assert_allclose(sh, so, rtol=5e-4, atol=1e-5, err_msg="update %d" % u)
        np.testing.assert_array_equal(h.read_field(abi.CRL_F_TERMINAL), o.read_field(abi.CRL_F_TERMINAL))
        if kind == 0:
            np.testing.assert_array_equal(h.read_field(abi.CRL_F_ACTION), o.read_field(abi.CRL_F_ACTION))
        np.testing.assert_allclose(h.get_params(), o.get_params(), rtol=1e-4, atol=2e-6, err_msg="update %d" % u)
        recs, ao = o.pop_episodes()
        assert agg.count == ao.count
        if u == 0:
            assert_truncated(recs, t0, h.cfg.max_episode_steps)
    assert h.spec_replays() == 0
    h.close()


@pytest.mark.parametrize("kind,N", [(0, 1187), (1, 2399)])
def test_fused_update_matches_exact_chain_at_large_ragged_sizes(abi, olib, torch_cuda, monkeypatch, kind, N):
    """minibatches of 18,992 (149 tiles, the last with 48 samples) and 38,384 samples (300 tiles, the last with 112):
    one update with the fused kernel against the same update through the exact 3-kernel chain (CRL_EXACT=1), which the
    sweep above pins to the oracle. Same seed: the rollouts are bit-identical. Tolerances of test_gpu_tc."""
    from cleanrl_jl_b200.handle import PPOHandle
    T = 16
    p = rand_params(olib, kind, seed=8)
    if kind == 1:
        p[-1] = -0.5
    res = []
    for exact in (False, True):
        if exact:
            monkeypatch.setenv("CRL_EXACT", "1")
        else:
            monkeypatch.delenv("CRL_EXACT", raising=False)
        h = PPOHandle(abi.make_config(env_kind=kind, num_envs=N, num_steps=T, num_minibatches=1, update_epochs=4, seed=43))
        h.set_params(p)
        h.env_reset()
        h.train_update(LR)
        st, _ = h.fetch_update()
        r = {name: h.read_field(getattr(abi, "CRL_F_" + name)) for name in ("STATE", "ACTION", "ADVANTAGE")}
        r.update(stats=st, params=h.get_params(), replays=h.spec_replays())
        h.close()
        res.append(r)
    monkeypatch.delenv("CRL_EXACT", raising=False)
    fused, exact = res
    for name in ("STATE", "ACTION", "ADVANTAGE"):
        np.testing.assert_array_equal(fused[name], exact[name], err_msg=name)
    np.testing.assert_allclose(fused["stats"], exact["stats"], rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(fused["params"], exact["params"], rtol=2e-5, atol=2e-6)
    assert fused["replays"] == 0


# ------------------------------------------------------------------ C. raw kernels at other coefficients
@pytest.mark.parametrize("kind", [0, 1])
@pytest.mark.parametrize("name", sorted(SETS))
@pytest.mark.parametrize("M", [129, 20000])
def test_ppo_loss_raw_at_other_coefficients(crl, olib, torch_cuda, kind, name, M):
    """the FFMA loss kernel (crl_ppo_loss_raw) at the tolerances of test_gpu_parity.test_ppo_loss_raw"""
    torch = torch_cuda
    d = olib.dims(kind)
    B = 2 * M
    p = rand_params(olib, kind, seed=9)
    if kind == 1:
        p[-1] = -0.3
    states, actions, logprobs, adv, ret, val = make_batch(olib, kind, B, 51 + M)
    idx = np.random.default_rng(M + 1).permutation(B)[:M].astype(np.int32)
    c, ent_c, v_c = loss_coefs(name)
    olib.set_threads(8)
    try:
        g_o, st_o, _ = olib.ppo_loss_raw(kind, p, idx, states, actions, logprobs, adv, ret, val, c, ent_c, v_c)
    finally:
        olib.set_threads(1)
    t = [dev(torch, a) for a in (p, idx, states, actions, logprobs, adv, ret, val)]
    g = torch.zeros(d["P"], dtype=torch.float32, device="cuda")
    st = torch.zeros(4, dtype=torch.float64, device="cuda")
    crl.check(crl.load().crl_ppo_loss_raw(kind, crl.ptr(t[0]), crl.ptr(t[1]), M, *[crl.ptr(x) for x in t[2:]],
                                          c, ent_c, v_c, crl.ptr(g), crl.ptr(st), None))
    torch.cuda.synchronize()
    np.testing.assert_allclose(st.cpu().numpy(), st_o, rtol=RTOL, atol=1e-7)
    gg = g.cpu().numpy()
    off, size = olib.param_layout(kind)
    for i in range(d["n_arrays"]):
        sl = slice(off[i], off[i] + size[i])
        np.testing.assert_allclose(gg[sl], g_o[sl], rtol=1e-4, atol=2e-6 * np.abs(g_o[sl]).max() + 1e-12,
                                   err_msg="array %d" % i)


@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("gamma,lam", [(0.9, 0.8), (1.0, 1.0), (0.0, 0.5)])
@pytest.mark.parametrize("T,N", [(37, 1001), (16, 148 * 1024 * 4 + 3)])
def test_gae_raw_bit_exact_at_other_coefficients(crl, olib, torch_cuda, mode, gamma, lam, T, N):
    torch = torch_cuda
    rng = np.random.default_rng(77 + T + N + mode)
    v = rng.standard_normal((T, N)).astype(F)
    r = rng.standard_normal((T, N)).astype(F)
    d = (rng.random((T, N)) < 0.05).astype(np.uint8)
    nv = rng.standard_normal(N).astype(F)
    nd = (rng.random(N) < 0.05).astype(np.uint8)
    adv_o, ret_o = olib.gae_raw(v, r, d, nv, nd, F(gamma), F(lam), mode)
    tv, tr, td, tnv, tnd = [dev(torch, a) for a in (v, r, d, nv, nd)]
    adv = torch.full((T, N), float("nan"), dtype=torch.float32, device="cuda")
    ret = torch.full((T, N), float("nan"), dtype=torch.float32, device="cuda")
    crl.check(crl.load().crl_gae_raw(crl.ptr(tv), crl.ptr(tr), crl.ptr(td), crl.ptr(tnv), crl.ptr(tnd), crl.ptr(adv),
                                     crl.ptr(ret), T, N, gamma, lam, mode, None))
    torch.cuda.synchronize()
    np.testing.assert_array_equal(adv.cpu().numpy(), adv_o)
    np.testing.assert_array_equal(ret.cpu().numpy(), ret_o)


# ------------------------------------------------------------------ D. DQN at ragged env counts
@pytest.mark.parametrize("N,buffer_size,iters", [(100, 1030, 30), (1007, 4500, 21)])
def test_dqn_ragged_env_counts_match_oracle(crl, olib, abi, torch_cuda, N, buffer_size, iters):
    """env counts that leave the last 32-env acting CTA partly filled (100: 4 CTAs, the last with 4 envs; 1007: the
    last with 15), a ring capacity that is not a multiple of N (it wraps in the middle of an iteration, more than twice
    in the run), and non-default learning settings; compared as test_dqn.test_dqn_cuda_matches_oracle. The episode cap
    of 40 steps bounds chaotic divergence of the trajectories."""
    from cleanrl_jl_b200.dqn_algo import DQNHandle, init_q_params
    cfg = abi.make_dqn_config(num_envs=N, buffer_size=buffer_size, min_buff_size=77, batch_size=77, train_freq=3,
                              target_net_freq=7, max_episode_steps=40, gamma=0.9, epsilon_start=0.6, epsilon_end=0.1,
                              epsilon_duration=float(iters * N * 2 // 3), seed=17)
    h, o = DQNHandle(cfg), OracleDQN(olib, cfg)
    p = init_q_params(5)
    for x in (h, o):
        x.set_params(p); x.reset()
    for chunk in (iters // 3, iters // 3, iters - 2 * (iters // 3)):
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
        np.testing.assert_allclose(bh["state"][:n], bo["state"][:n], rtol=1e-5, atol=2e-6)
        np.testing.assert_allclose(bh["next_state"][:n], bo["next_state"][:n], rtol=1e-5, atol=2e-6)
        qh, th = h.get_params(); qo, to = o.get_params()
        np.testing.assert_allclose(qh, qo, rtol=1e-4, atol=2e-6)
        np.testing.assert_allclose(th, to, rtol=1e-4, atol=2e-6)
        if so.learn_steps:
            assert abs(sh.last_loss - so.last_loss) <= 1e-4 * abs(so.last_loss) + 1e-7
    assert so.iterations * N >= 2 * buffer_size + N and buffer_size % N != 0
    assert so.learn_steps > 5 and so.episodes > 0 and so.epsilon == 0.1
    h.close(); o.close()
