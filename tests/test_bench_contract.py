"""bench.py contract checks: without a GPU, the reference arm (the CPU path timed on host cores) prints exactly one
JSON line with the keys the driver reads, and the workload table names real model files; on the GPU, --dump-outputs
records the last timed step reproducibly."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.conftest import ROOT


def test_workloads_point_at_bundled_models():
    sys.path.insert(0, ROOT)
    import bench
    for name, wl in bench.WORKLOADS.items():
        assert os.path.exists(os.path.join(ROOT, "models", wl["model"])), name
        if wl.get("animated"):
            assert os.path.exists(os.path.join(ROOT, "backgrounds", wl["animated"])), name
    assert "meet720" in bench.WORKLOADS and bench.METRIC.startswith("composited frames")


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "mlkit480",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["value"] > 0 and d["cpu_baseline"]["kind"] == "port"
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["cpu_baseline"]["cores"] >= 1 and "workload" in d["config"]


def test_non_zero_rank_of_reference_arm_exits_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_is_refused_for_the_reference_arm(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode == 2 and "--dump-outputs" in out.stderr and not os.listdir(tmp_path)


@pytest.mark.gpu
def test_dump_outputs_of_the_last_timed_step(tmp_path):
    """--dump-outputs writes the sampled composite / YUYV / mask of the last timed step as float32, within 64 MB, and
    two runs with the same arguments write the same values."""
    S, B, W, H, steps = 2, 4, 640, 480, 3
    dumps = []
    for run in range(2):
        d = tmp_path / f"run{run}"
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "mlkit480", "--streams", str(S),
                              "--batch", str(B), "--steps", str(steps), "--warmup", "1", "--launches-per-step", "1",
                              "--no-e2e", "--no-configs", "--no-cpu-baseline", "--dump-outputs", str(d)],
                             capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads(out.stdout.strip().splitlines()[-1])
        assert line["steps"] == steps and line["config"]["frames_per_step"] == S * B
        assert line["gpu_launches"] == steps * S * line["roofline"]["cnn"]["launches_per_call"]
        files = sorted(os.listdir(d))
        assert files == ["composite.npy", "mask.npy", "pixel_index.npy", "yuyv.npy"]
        assert sum(os.path.getsize(d / f) for f in files) <= 64 << 20
        dumps.append({f[:-4]: np.load(d / f) for f in files})
    a, b = dumps
    idx = a["pixel_index"]
    assert idx.dtype == np.float64 and np.all(np.diff(idx) > 0) and 0 <= idx[0] and idx[-1] < S * B * W * H
    n = idx.size
    assert a["composite"].shape == (n, 3) and a["yuyv"].shape == (n, 2) and a["mask"].shape == (n,)
    for k in a:
        assert a[k].dtype in (np.float32, np.float64)
        assert np.array_equal(a[k], b[k]), k
    person = (a["mask"] < 128).mean()
    assert 0.05 < person < 0.6, person
