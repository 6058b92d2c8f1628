"""The oracle's loss and optimiser away from the reference defaults (clip_coef 0.2, ent_coeff 0.01, v_coef 0.5,
clip_norm 0.5, gamma 0.99, gae_lambda 0.95). Every other oracle pin runs those defaults, so an oracle that hard-wired
one of them would still pass; here float64 autograd of the restated loss (test_oracle_grad.torch_loss) and
torch.optim.Adam pin the oracle at two other coefficient sets, which the GPU tests (test_gpu_update_geometry.py)
then hold the CUDA kernels to. CPU only."""
import numpy as np
import pytest
import torch

from conftest import rand_params
from test_oracle_grad import make_batch, torch_loss

F = np.float32

# Set 1 clips a lot: a tight ratio clip, a large entropy bonus, ClipNorm 0.05 (below the gradient norm of most
# parameter arrays), short discounting and episode caps that truncate several times within a few rollouts.
# Set 2 is the opposite corner: a wide ratio clip, no entropy term, ClipNorm 1e3 (never clips), long discounting and
# lambda = 1 (Monte-Carlo advantages).
SETS = {
    "set1": dict(clip_coef=0.1, ent_coeff=0.05, v_coef=1.0, clip_norm=0.05, gamma=0.9, gae_lambda=0.8,
                 max_episode_steps=(50, 30)),
    "set2": dict(clip_coef=0.3, ent_coeff=0.0, v_coef=0.25, clip_norm=1e3, gamma=0.995, gae_lambda=1.0),
}


def config_kw(name, kind):
    """make_config keyword arguments of coefficient set `name` for env kind `kind` (0 CartPole, 1 Pendulum)"""
    kw = dict(SETS[name])
    if "max_episode_steps" in kw:
        kw["max_episode_steps"] = kw["max_episode_steps"][kind]
    return kw


def loss_coefs(name):
    """(clip_coef, ent_coeff, v_coef) as the Float32 values the C ABI passes"""
    s = SETS[name]
    return tuple(float(F(s[k])) for k in ("clip_coef", "ent_coeff", "v_coef"))


def array_norms(g, layout):
    off, size = layout
    return np.array([np.linalg.norm(g[o:o + n].astype(np.float64)) for o, n in zip(off, size)])


def assert_clip_branch(name, g, layout):
    """ClipNorm branches differently from the default threshold 0.5 under each set: set 1 rescales some parameter
    arrays that 0.5 would leave alone, set 2 leaves alone some that 0.5 would rescale (and rescales none)"""
    nrm = array_norms(g, layout)
    thresh = SETS[name]["clip_norm"]
    if thresh < 0.5:
        assert np.any((nrm > thresh) & (nrm < 0.5)), nrm
    else:
        assert np.all(nrm < thresh) and np.any(nrm > 0.5), nrm


@pytest.mark.parametrize("kind", [0, 1])
@pytest.mark.parametrize("name", sorted(SETS))
@pytest.mark.parametrize("no_vclip", [False, True])
def test_oracle_loss_matches_float64_autograd(olib, kind, name, no_vclip):
    d = olib.dims(kind)
    layout = olib.param_layout(kind)
    B, M = 300, 96
    p = rand_params(olib, kind, seed=7 + kind)
    if kind == 1:
        p[-1] = -0.3
    states, actions, logprobs, adv, ret, val = make_batch(olib, kind, B, 19)
    idx = np.random.default_rng(6).permutation(B)[:M].astype(np.int32)
    c, ent_c, v_c = loss_coefs(name)
    olib.lib.orc_set_no_vclip(1 if no_vclip else 0)
    try:
        g, stats, vnew = olib.ppo_loss_raw(kind, p, idx, states, actions, logprobs, adv, ret, val, c, ent_c, v_c)
    finally:
        olib.lib.orc_set_no_vclip(0)
    pt = torch.tensor(p.astype(np.float64), requires_grad=True)
    loss, pg, vl, en = torch_loss(pt, layout, d, idx, states, actions, logprobs, adv, ret, val, c, ent_c, v_c, kind == 1,
                                  clip_vloss=not no_vclip)
    loss.backward()
    gt = pt.grad.numpy()
    np.testing.assert_allclose(stats, [loss.item(), pg.item(), vl.item(), en.item()], rtol=2e-5, atol=1e-6)
    np.testing.assert_allclose(g, gt, rtol=2e-3, atol=2e-5 * np.abs(gt).max())
    # the ratio clip is active for some samples and not for others, so clip_coef reaches the gradient
    ratio = np.exp(_new_logprob(olib, kind, p, states[idx], actions[idx]) - logprobs[idx])
    inside = np.abs(ratio - 1.0) <= c
    assert 0 < inside.sum() < M


def _new_logprob(olib, kind, p, states, actions):
    pol, logp, _ = olib.policy_forward_raw(kind, p, states)
    if kind == 0:
        return logp[np.arange(len(actions)), actions].astype(np.float64)
    logstd = float(p[-1])
    a = np.asarray(actions, np.float64)[:, 0]
    return -(a - pol[:, 0]) ** 2 / (2 * np.exp(2 * logstd)) - logstd - 0.9189385332046727


@pytest.mark.parametrize("kind", [0, 1])
@pytest.mark.parametrize("clip_norm", [0.05, 1e3])
def test_clip_adam_matches_torch_optim_adam(olib, kind, clip_norm):
    """Flux.Optimiser(ClipNorm(clip_norm), Adam) of the oracle against torch.optim.Adam in float64 with the per-array
    clip applied by hand (as test_oracle_torch_pins does at the default 0.5). Gradient elements of magnitude 0.06-0.1
    put every array's norm above 0.05, and the big arrays' norms above the default 0.5 but far below 1e3."""
    d = olib.dims(kind)
    layout = olib.param_layout(kind)
    off, size = layout
    rng = np.random.default_rng(23 + kind)
    p0 = rng.standard_normal(d["P"]).astype(F)
    tp = [torch.nn.Parameter(torch.tensor(p0[off[i]:off[i] + size[i]].astype(np.float64))) for i in range(d["n_arrays"])]
    lr = float(F(2.5e-4))
    opt = torch.optim.Adam(tp, lr=lr, betas=(0.9, 0.999), eps=1e-8)
    p, m, v = p0.copy(), np.zeros(d["P"], F), np.zeros(d["P"], F)
    bp = np.tile(np.array([0.9, 0.999]), (d["n_arrays"], 1))
    for it in range(6):
        g = (rng.choice([-1.0, 1.0], d["P"]) * rng.uniform(0.06, 0.1, d["P"])).astype(F)
        nrm = array_norms(g, layout)
        if clip_norm < 1.0:
            assert np.all(nrm > clip_norm)
        else:
            assert np.all(nrm < clip_norm) and np.any(nrm > 0.5)
        p, m, v, bp = olib.clip_adam_raw(kind, p, g, m, v, bp, lr, clip_norm)
        for i, q in enumerate(tp):
            gi = torch.tensor(g[off[i]:off[i] + size[i]].astype(np.float64))
            n = gi.norm()
            q.grad = gi * (clip_norm / n) if n > clip_norm else gi
        opt.step()
        ref = np.concatenate([q.detach().numpy() for q in tp])
        np.testing.assert_allclose(p, ref, rtol=0, atol=2e-7 * (it + 1) + 1.2e-7 * np.abs(ref).max())
    for i in range(d["n_arrays"]):
        st = opt.state[tp[i]]
        sl = slice(off[i], off[i] + size[i])
        # the first moment carries the clip scale: clip_norm / norm on every array for 0.05, 1 for 1e3
        np.testing.assert_allclose(m[sl], st["exp_avg"].numpy(), rtol=1e-5, atol=1e-9, err_msg="array %d" % i)
        np.testing.assert_allclose(v[sl], st["exp_avg_sq"].numpy(), rtol=1e-5, atol=1e-12, err_msg="array %d" % i)
