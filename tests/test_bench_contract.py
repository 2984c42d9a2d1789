"""bench.py's JSON contract (the reference arm runs on the CPU, so this needs no GPU): one JSON line on stdout
with the keys the driver reads, the CPU restatement as the timed implementation, bounded sample."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                          "--warmup", "1", "--envs", "2048"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "env-steps/s" and d["higher_is_better"] is True
    assert d["steps"] == 2 and d["warmup"] == 1 and d["value"] > 0 and d["scaling"] == "weak"
    assert d["metric"].startswith("batched env-steps/s") and "PredatorCapturePrey-v0" in d["config"]["workload"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "envs per step" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and d["vs_baseline"] is None and d["dtype"] == "f64" and d["data"] == "synthetic"


def test_dump_outputs_is_float_and_a_fixed_sample_under_64_mb(tmp_path):
    """bench.dump_outputs on a Warehouse-sized step (262,144 envs x 6 robots x 18 obs: 113 MB of obs alone): every
    file float32 / float64, 64 MB at most in all, the same envs from run to run, rows taken from the envs named."""
    import numpy as np
    import torch
    import bench
    B, N, D = 262144, 6, 18
    g = torch.Generator().manual_seed(0)
    outputs = {"obs": torch.rand((B, N, D), generator=g), "reward": torch.rand((B, N), generator=g),
               "done": torch.randint(0, 2, (B,), generator=g, dtype=torch.uint8),
               "message": torch.randint(0, 4, (B,), generator=g, dtype=torch.uint8)}
    runs = [tmp_path / "a", tmp_path / "b"]
    for d in runs:
        bench.dump_outputs(str(d), outputs)
    files = sorted(os.listdir(runs[0]))
    assert files == ["done.npy", "env_index.npy", "message.npy", "obs.npy", "reward.npy"]
    assert sum(os.path.getsize(runs[0] / f) for f in files) <= bench.DUMP_LIMIT_BYTES
    for f in files:
        a, b = np.load(runs[0] / f), np.load(runs[1] / f)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b), f
    index = np.load(runs[0] / "env_index.npy").astype(np.int64)
    assert B // 2 < len(index) < B and (np.diff(index) > 0).all()
    for name, t in outputs.items():
        assert np.array_equal(np.load(runs[0] / (name + ".npy")), t.numpy()[index].astype(np.float32)), name


def test_steps_below_one_are_refused():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True,
                         text=True, timeout=120, cwd=ROOT)
    assert out.returncode == 2 and "--steps" in out.stderr


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
