"""bench.py contract, CPU side: the reference arm prints ONE JSON line with the keys the driver reads; the helper
formulas behind `roofline` are the ones DESIGN.md states."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--ref-envs", "16"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-500:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "env-steps/s" and d["dtype"] == "f64" and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["value"] > 0
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "1"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_roofline_helpers():
    sys.path.insert(0, ROOT)
    import bench
    assert bench.algorithmic_bytes(45) == 1553          # DESIGN.md section 3: 71 doubles each way + ctrl + obs + reward + done
    assert bench.algorithmic_bytes(48) == 1577          # SURVEY 8(d): tr_env 48-obs figure
    assert bench.flops_per_env_step(3, 2) == 20 * (3000 + 1350 + 2 * (1500 + 2700))


def test_dump_outputs_layout_and_sampling(tmp_path, monkeypatch):
    import torch
    sys.path.insert(0, ROOT)
    import bench
    n = 50
    obs = torch.arange(n * 45, dtype=torch.float64).reshape(n, 45)
    rew, done = torch.arange(n, dtype=torch.float64) * 0.5, (torch.arange(n) % 3 == 0).to(torch.uint8)
    bench.dump_outputs(str(tmp_path / "all"), obs, rew, done)
    got = {f[:-4]: np.load(tmp_path / "all" / f) for f in os.listdir(tmp_path / "all")}
    assert sorted(got) == ["done", "env_index", "obs", "reward"]
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert np.array_equal(got["obs"], obs.numpy()) and np.array_equal(got["reward"], rew.numpy())
    assert np.array_equal(got["done"], done.numpy()) and np.array_equal(got["env_index"], np.arange(n))
    # above the size budget: a fixed sample of envs, the same on every call
    row_bytes = 47 * 8 + 4
    monkeypatch.setattr(bench, "DUMP_BYTES", 20 * row_bytes)
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), obs, rew, done)
    idx = np.load(tmp_path / "s1" / "env_index.npy")
    assert len(idx) == 20 and np.all(np.diff(idx) > 0) and np.array_equal(idx, np.load(tmp_path / "s2" / "env_index.npy"))
    assert np.array_equal(np.load(tmp_path / "s1" / "obs.npy"), obs.numpy()[idx.astype(int)])
    assert sum(os.path.getsize(tmp_path / "s1" / f) for f in os.listdir(tmp_path / "s1")) <= 20 * row_bytes + 4 * 128   # + one npy header each


@pytest.mark.gpu
def test_dump_outputs_identical_across_runs(tmp_path):
    """two bench runs with the same arguments compute the same last timed step, bit for bit"""
    args = ["--envs", "4096", "--steps", "3", "--warmup", "1", "--settle", "20", "--no-cpu-baseline", "--no-e2e",
            "--no-workloads", "--sweep", ""]
    for d in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args, "--dump-outputs", str(tmp_path / d)],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 3
    for name in ("obs", "reward", "done", "env_index"):
        a, b = np.load(tmp_path / "a" / (name + ".npy")), np.load(tmp_path / "b" / (name + ".npy"))
        assert a.shape[0] == 4096 and np.array_equal(a, b), name
    assert np.isfinite(np.load(tmp_path / "a" / "obs.npy")).all()
