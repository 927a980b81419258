"""bench.py --dump-outputs on the GPU arm: the files hold bit for bit what the same rollouts return when they are run directly (warm-up
plus timed steps on the bench's seeded inputs), so two builds run with the same arguments can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_rollout(cuda_backend, tmp_path):
    import bench
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3", "--no-secondary", "--no-cpu-baseline",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 2 and line["warmup"] == 3

    be, spec = cuda_backend, bench.workload_spec("kuka")
    n, T, D = spec["n"], spec["T"], spec["obs_dim"]
    sim = be.make_sim(spec["env_id"], n, seed=0, model_blob=bench.model_blob("kuka"), global_env_offset=0, **spec["cfg"])
    st = be.stream()
    sim.reset(stream=st)
    acts_h, noise_h = bench.make_inputs("kuka", n, T, 0)
    acts, noise = be.from_host(acts_h), be.from_host(noise_h)
    want = {"obs": be.zeros((T, n, D), np.float32), "reward": be.zeros((T, n), np.float32), "done": be.zeros((T, n), np.uint8),
            "episode_return": be.zeros((T, n), np.float32), "episode_length": be.zeros((T, n), np.int32)}
    for _ in range(line["warmup"] + line["steps"]):
        sim.rollout(T, acts, noise, want["obs"], want["reward"], want["done"], want["episode_return"], want["episode_length"], stream=st)
    sim.close()
    for name, buf in want.items():
        got = np.load(str(tmp_path / (name + ".npy")))
        assert got.dtype == (np.float32 if name in ("obs", "reward", "episode_return") else np.float64), name
        np.testing.assert_array_equal(got, be.to_host(buf), err_msg=name)
