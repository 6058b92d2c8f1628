"""bench.py --dump-outputs on the B200: what the last timed update computed is written as float arrays, and two runs
with the same arguments write the same bytes, so that two builds can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = {"params", "loss_stats", "episode_agg", "obs", "action", "logprob", "reward", "terminal", "value", "advantage",
         "return", "next_obs"}


def _bench(out, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "3",
           "--no-secondary", "--no-cpu-baseline", "--gae-n", "4096", "--dump-outputs", str(out)]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    return line, {f[:-4]: np.load(str(out / f)) for f in os.listdir(str(out))}


def test_bench_dumps_identical_outputs_for_identical_arguments(tmp_path, torch_cuda):
    line, a = _bench(tmp_path / "a", 2)
    _, b = _bench(tmp_path / "b", 2)
    assert line["steps"] == 2
    assert set(a) == NAMES and set(b) == NAMES
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    assert all(x.dtype in (np.float32, np.float64) for x in a.values())
    T, N = 128, 4096
    assert a["obs"].shape == (T, N, 4) and a["advantage"].shape == (T, N) and a["loss_stats"].shape == (16, 4)
    assert a["loss_stats"][-1, 0] == line["last_loss"]
    for k in NAMES:
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
