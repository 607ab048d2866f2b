"""bench.py's contract pieces that can be checked without a GPU: the reference arm prints one JSON line with the
agreed keys, the GPU arm refuses to run without CUDA (no CPU fallback), and the core count honours the container."""
import json
import os
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


def run_bench(*args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], capture_output=True, text=True, cwd=ROOT,
                          env=e, timeout=600)


def test_reference_arm_prints_the_contract_line():
    p = run_bench("--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-sample", "4",
                  "--width", "320", "--height", "240")
    assert p.returncode == 0, p.stderr
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "frames/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["gpu_launches"] == 0
    assert line["e2e"] == {"value": line["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == line["value"] and 1 <= cb["cores"] <= cb["host_cpu_count"]
    assert line["config"]["workload"] == "detect_track30" and line["config"]["track_calls_per_frame"] == 30


def test_reference_arm_other_ranks_exit_quietly():
    p = run_bench("--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0", env={"RANK": "1", "WORLD_SIZE": "2"})
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_gpu_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is visible: the refusal path cannot be exercised")
    p = run_bench("--steps", "1", "--warmup", "0", "--batch", "2")
    assert p.returncode != 0
    assert "no CUDA device" in (p.stderr + p.stdout)


def test_bad_step_counts_are_refused():
    for args in (("--steps", "0"), ("--warmup", "-1")):
        p = run_bench("--impl", "reference", *args)
        assert p.returncode == 2 and "--steps must be at least 1" in p.stderr


def test_dump_outputs_above_the_limit_is_a_fixed_sample(tmp_path):
    sys.path.insert(0, str(ROOT))
    import bench
    import numpy as np
    arrays = {"rects": np.arange(1000 * 16, dtype=np.float64).reshape(1000, 16), "counts": np.arange(1000.0)}
    for d in ("a", "b"):
        bench.write_outputs(tmp_path / d, arrays, limit=40_000)
    idx = np.load(tmp_path / "a" / "frame_index.npy")
    assert 0 < len(idx) < 1000 and np.all(np.diff(idx) > 0)
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= 40_000
    for name, a in arrays.items():
        got = np.load(tmp_path / "a" / f"{name}.npy")
        assert np.array_equal(got, a[idx.astype(int)]) and np.array_equal(got, np.load(tmp_path / "b" / f"{name}.npy"))


def test_usable_cores_is_bounded_by_the_affinity_mask():
    sys.path.insert(0, str(ROOT))
    import bench
    n = bench.usable_cores()
    assert 1 <= n <= (os.cpu_count() or 1)
    if hasattr(os, "sched_getaffinity"):
        assert n <= len(os.sched_getaffinity(0))
