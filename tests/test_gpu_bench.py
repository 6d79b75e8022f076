"""GPU: bench.py --dump-outputs writes what the last timed step returned, the same from run to run, so that two builds
can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import c_oracle

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = {"obs", "reward", "done", "num_snakes", "episode_return", "episode_length"}


def _bench(out_dir, warmup, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup),
           "--no-configs", "--no-cpu-baseline", "--e2e-steps", "3", "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-4000:]
    return json.loads(r.stdout)


def test_dump_outputs_are_the_last_timed_step(tmp_path):
    """Two runs dump identical arrays, and they are what the C oracle computes after the bench's schedule: reset, the 16
    steps of the parity check (action stream steps 0..15), then the W warm-up and the K timed steps, both cycling through
    the min(K, 32) resident batches (action stream steps 100, 101, ...)."""
    import bench
    W, K = 2, 7
    a, b = _bench(tmp_path / "a", W, K), _bench(tmp_path / "b", W, K)
    assert a["parity"]["ranks_ok"] == 1
    assert sorted(os.listdir(tmp_path / "a")) == sorted(n + ".npy" for n in NAMES)
    got, total = {}, 0
    for name in NAMES:
        x, y = np.load(tmp_path / "a" / (name + ".npy")), np.load(tmp_path / "b" / (name + ".npy"))
        assert x.dtype == np.float32 and np.array_equal(x, y), name
        got[name] = x
        total += os.path.getsize(tmp_path / "a" / (name + ".npy"))
    assert total <= 64 << 20

    n = a["config"]["envs_total"]
    co = c_oracle.COracle(n, size=bench.SIZE, n_snakes=bench.N_SNAKES, rules=bench.RULES, seed=0)
    co.reset(want_obs=False)
    batches = min(K, 32)
    for s in list(range(16)) + [100 + t % batches for t in range(W)] + [100 + t % batches for t in range(K)]:
        _, rew, done, info = co.step(c_oracle.gen_actions(co.cfg, s, 1), want_obs=False)
    want = {"reward": rew, "done": done, "num_snakes": info["num_snakes"], "episode_return": info["episode_r"],
            "episode_length": info["episode_l"], "obs": co.observe()[bench.dump_obs_envs(n)]}
    for name in NAMES:
        assert np.array_equal(got[name], want[name].astype(np.float32)), name
