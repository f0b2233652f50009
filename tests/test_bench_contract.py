"""bench.py's output contract: exactly one line on stdout, and it is the JSON line; --dump-outputs writes what the last
timed step returned."""
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ, NCCL_DEBUG="VERSION")  # library banners must not reach stdout either
    res = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--cpu-sample-envs", "4096"], capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.split("\n") if l.strip()]
    assert len(lines) == 1, res.stdout[:2000]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "env-steps/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["steps"] == 1 and d["warmup"] == 1 and d["n_gpus"] == 1
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_reference_arm_nonzero_rank_is_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    res = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert res.returncode == 0 and res.stdout.strip() == ""


def _bench(args, out_dir):
    res = subprocess.run([sys.executable, str(ROOT / "bench.py"), *args, "--dump-outputs", str(out_dir)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    return json.loads(res.stdout), {p.stem: np.load(p) for p in sorted(out_dir.glob("*.npy"))}


def test_reference_arm_dumps_its_last_step(tmp_path):
    """Two runs with the same arguments write the same outputs of the same (last) step: here the 26th, which ends every
    SwingRacket episode."""
    args = ["--impl", "reference", "--steps", "2", "--warmup", "1", "--cpu-sample-envs", "300"]
    _, a = _bench(args, tmp_path / "a")
    _, b = _bench(args, tmp_path / "b")
    assert sorted(a) == ["done", "events", "obs", "reward", "terminal_obs"]
    for k in a:
        assert a[k].dtype == np.float32 and len(a[k]) == 300, k
        np.testing.assert_array_equal(a[k], b[k])
    assert a["obs"].shape == (300, 6) and (a["done"] == 1).all()


def test_dump_outputs_samples_within_the_limit(tmp_path, monkeypatch):
    import bench

    n = 1000
    arrays = {"obs": np.arange(n * 6, dtype=np.float32).reshape(n, 6), "done": np.ones(n, np.uint8),
              "value": np.arange(n, dtype=np.float64)}
    bench.dump_outputs(tmp_path / "full", arrays)
    full = {p.stem: np.load(p) for p in (tmp_path / "full").glob("*.npy")}
    assert sorted(full) == ["done", "obs", "value"] and full["done"].dtype == np.float32 and full["value"].dtype == np.float64
    np.testing.assert_array_equal(full["obs"], arrays["obs"])

    monkeypatch.setattr(bench, "DUMP_LIMIT", 4096 + 10000)
    for d in ("s1", "s2"):
        bench.dump_outputs(tmp_path / d, arrays)
    files = sorted((tmp_path / "s1").glob("*.npy"))
    assert sum(p.stat().st_size for p in files) <= bench.DUMP_LIMIT
    s = {p.stem: np.load(p) for p in files}
    idx = s["env_index"].astype(np.int64)
    assert 0 < len(idx) < n and (np.diff(idx) > 0).all()
    for k in arrays:
        np.testing.assert_array_equal(s[k], arrays[k][idx].astype(s[k].dtype))
        np.testing.assert_array_equal(s[k], np.load(tmp_path / "s2" / f"{k}.npy"))  # the sample is seeded


@pytest.mark.gpu
def test_b200_arm_dumps_its_last_timed_step(tmp_path):
    """--steps sets the number of timed env steps (the library's own env-step count says so), and the dumped outputs are
    those of the last timed step - in lock step a fast-forward step, which ends every episode - the same in every run."""
    n, steps = 4096, 30
    args = ["--envs-per-gpu", str(n), "--steps", str(steps), "--warmup", "3", "--extras", "off", "--skip-cpu-baseline"]
    line, a = _bench(args, tmp_path / "a")
    _, b = _bench(args, tmp_path / "b")
    assert line["steps"] == steps and line["episode_stats"]["env_steps"] == n * steps
    assert line["episode_stats"]["episodes"] == 2 * n  # the region ends on a fast-forward step: ceil(30 / 26) of them
    assert sorted(a) == ["done", "events", "obs", "reward", "terminal_obs"]
    for k in a:
        assert a[k].dtype == np.float32 and len(a[k]) == n, k
        np.testing.assert_array_equal(a[k], b[k])
    assert (a["done"] == 1).all() and np.isfinite(a["terminal_obs"]).all()
