"""bench.py plumbing that needs no GPU: both arms describe the same workload, the roofline `traffic` figures come from
the newest committed ncu summary that holds the kernel (profiles/), and --dump-outputs writes float arrays within its
size limit."""
import argparse
import importlib.util
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _args(**kw):
    d = dict(gpus=1, steps=20, warmup=5, impl="ours", envs_per_gpu=4096, env="CartPole", no_cpu_baseline=False,
             no_secondary=False, gae_n=1 << 20, local_stats=False, dqn_mode="replicas", algo="ppo")
    d.update(kw)
    return argparse.Namespace(**d)


def test_both_arms_state_the_same_config():
    b = _bench()
    for gpus in (1, 8):
        ours = b.workload_config(_args(gpus=gpus, impl="ours"), gpus)
        ref = b.workload_config(_args(gpus=gpus, impl="reference"), gpus)
        assert ours == ref
        assert "workload" in ours and "model" not in ours
        assert ours["num_envs_global"] == 4096 * gpus


def test_roofline_traffic_comes_from_the_committed_ncu_summaries():
    b = _bench()
    tc, tc_file = b.ncu_traffic("loss_grad_tc_kernel")
    assert tc_file and tc_file.startswith("profiles/") and "ncu" in tc_file
    assert 5e6 < tc < 5e7          # the 16.5 MB rollout buffer read once under ncu (cold L2), per launch
    gae, gae_file = b.ncu_traffic("gae_kernel<0, 4, 4>")
    assert gae_file and 2.0e9 < gae < 2.4e9   # 2.29 GB algorithmic at T=128, N=2^20
    assert b.ncu_traffic("no_such_kernel") == (None, None)


def _dump(b, out, T, N):
    rng = np.random.default_rng(3)
    whole = {"params": rng.standard_normal(4610).astype(np.float32), "loss_stats": rng.standard_normal((16, 4))}
    per_env = {"obs": (rng.standard_normal((T, N, 4)).astype(np.float32), 1),
               "action": (rng.integers(0, 2, (T, N)).astype(np.int32), 1),
               "terminal": (rng.integers(0, 2, (T, N)).astype(np.uint8), 1),
               "next_obs": (rng.standard_normal((N, 4)).astype(np.float32), 0)}
    b.dump_outputs(str(out), whole, per_env, N)
    return whole, per_env, {f[:-4]: np.load(str(out / f)) for f in os.listdir(str(out))}


def test_dump_outputs_are_float_arrays_whole_when_they_fit(tmp_path):
    b = _bench()
    whole, per_env, got = _dump(b, tmp_path, 8, 16)
    assert set(got) == set(whole) | set(per_env)
    assert got["loss_stats"].dtype == np.float64 and got["action"].dtype == np.float32 and got["terminal"].dtype == np.float32
    for k, a in whole.items():
        np.testing.assert_array_equal(got[k], a)
    for k, (a, _) in per_env.items():
        np.testing.assert_array_equal(got[k], a.astype(np.float32))


def test_dump_outputs_sample_a_fixed_set_of_envs_beyond_the_size_limit(tmp_path, monkeypatch):
    b = _bench()
    monkeypatch.setattr(b, "DUMP_BYTES", 1 << 20)
    T, N = 128, 4096                                   # 12.6 MB of per-env data
    whole, per_env, got = _dump(b, tmp_path / "a", T, N)
    _, _, again = _dump(b, tmp_path / "b", T, N)
    assert sum(a.nbytes for a in got.values()) <= 1 << 20
    idx = got["env_index"].astype(np.int64)
    assert 0 < len(idx) < N and np.all(np.diff(idx) > 0)
    for k, (a, axis) in per_env.items():
        np.testing.assert_array_equal(got[k], np.take(a, idx, axis=axis).astype(np.float32))
    np.testing.assert_array_equal(got["params"], whole["params"])
    assert set(again) == set(got) and all(np.array_equal(again[k], got[k]) for k in got)
