"""bench.py contract pieces that run without a GPU: the reference arm prints one JSON line with the agreed keys
(driver contract), and the CPU sample is bounded and uses only the threads the process may really use."""
import json
import os
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def test_usable_cores_is_bounded_by_affinity():
    sys.path.insert(0, str(ROOT))
    import bench

    n = bench.usable_cores()
    assert 1 <= n <= (os.cpu_count() or 1)
    if hasattr(os, "sched_getaffinity"):
        assert n <= len(os.sched_getaffinity(0))


def test_cpu_sample_is_time_boxed():
    sys.path.insert(0, str(ROOT))
    import bench

    tf, dt, sample, cores = bench.cpu_naive_sample(rows=512, seconds=0.0)   # stops after the first 256-row block
    assert tf > 0 and dt > 0 and cores >= 1
    assert "256 query rows" in sample


def test_dump_outputs_writes_a_fixed_float32_row_sample(tmp_path):
    sys.path.insert(0, str(ROOT))
    import bench
    import numpy as np
    import torch

    o = torch.randn(1, 2, bench.S, 4, generator=torch.Generator().manual_seed(3)).bfloat16()
    bench.dump_outputs(tmp_path / "a", o)
    bench.dump_outputs(tmp_path / "b", o)
    a, b = np.load(tmp_path / "a" / "out.npy"), np.load(tmp_path / "b" / "out.npy")
    assert a.dtype == np.float32 and a.shape == (2, bench.DUMP_ROWS, 4) and np.array_equal(a, b)
    rows = [int(np.flatnonzero((o[0, 0].float().numpy() == a[0, i]).all(-1))[0]) for i in (0, -1)]
    assert rows[0] < rows[1] and np.array_equal(a[:, -1], o[0, :, rows[1]].float().numpy())


def test_steps_must_be_positive():
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode != 0 and "--steps" in out.stderr


def test_reference_arm_prints_the_contract_line():
    env = dict(os.environ, RANK="0")
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, env=env, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["unit"] == "TFLOP/s" and line["higher_is_better"] is True
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    # other ranks of a torchrun launch exit 0 without printing
    out1 = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                          capture_output=True, text=True, env=dict(os.environ, RANK="1"), timeout=120, cwd=ROOT)
    assert out1.returncode == 0 and out1.stdout.strip() == ""
