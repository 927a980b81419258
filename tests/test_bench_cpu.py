"""bench.py contract checks that need no GPU: the reference arm (`--impl reference`, the CPU oracle on the host cores) prints ONE
JSON line with the keys the driver reads, for the same metric / unit / config as the b200 arm."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("workload", ["mobile", "kuka"])
def test_reference_arm_json_line(workload, oracle_lib):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", workload, "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "env-steps/s" and d["higher_is_better"] is True and d["scaling"] == "weak"
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["steps"] == 1 and d["n_gpus"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert ("Kuka" if workload == "kuka" else "MobileRobot") in d["metric"] and "workload" in d["config"]


def test_reference_arm_other_ranks_exit_quietly(oracle_lib):
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and not [l for l in out.stdout.splitlines() if l.startswith("{")]


def _dump(tmp_path, tag, *args):
    d = tmp_path / tag
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(args) + ["--dump-outputs", str(d)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    return {f[:-len(".npy")]: np.load(str(d / f)) for f in os.listdir(str(d))}


def test_reference_arm_dumps_the_last_timed_rollout(oracle_lib, tmp_path):
    """--dump-outputs: the oracle pool's outputs of the last timed step, the same bytes on a rerun with the same arguments, other
    bytes when --steps adds a timed step."""
    args = ["--impl", "reference", "--workload", "mobile", "--warmup", "0", "--no-secondary"]
    a, b, c = _dump(tmp_path, "a", "--steps", "1", *args), _dump(tmp_path, "b", "--steps", "1", *args), _dump(tmp_path, "c", "--steps", "2", *args)
    assert sorted(a) == ["done", "obs", "reward"]
    n, T = 8192, 256
    assert a["obs"].shape == (T, n, 2) and a["reward"].shape == a["done"].shape == (T, n)
    assert a["obs"].dtype == a["reward"].dtype == np.float32 and a["done"].dtype == np.float64
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    for k in a:
        np.testing.assert_array_equal(a[k], b[k])
    assert not np.array_equal(a["obs"], c["obs"])


def test_dump_outputs_keeps_a_seeded_env_sample_within_the_budget(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_BUDGET_BYTES", 40000)
    T, n = 8, 1000
    obs = np.random.default_rng(0).random((T, n, 3), dtype=np.float32)
    arrays = {"obs": obs, "done": (obs[..., 0] > 0.5).astype(np.uint8),
              "episode_length": np.broadcast_to(np.arange(n, dtype=np.int32), (T, n))}   # every row holds the env index
    for tag in ("a", "b"):
        bench.dump_outputs(str(tmp_path / tag), arrays)
    a, b = [{k: np.load(str(tmp_path / tag / (k + ".npy"))) for k in arrays} for tag in ("a", "b")]
    assert a["obs"].dtype == np.float32 and a["done"].dtype == a["episode_length"].dtype == np.float64
    assert 0.9 * 40000 < sum(x.nbytes for x in a.values()) <= 40000
    cols = a["episode_length"][0].astype(np.int64)
    assert np.all(np.diff(cols) > 0) and np.all(a["episode_length"] == cols)
    np.testing.assert_array_equal(a["obs"], obs[:, cols])
    np.testing.assert_array_equal(a["done"], arrays["done"][:, cols])
    for k in arrays:
        np.testing.assert_array_equal(a[k], b[k])
