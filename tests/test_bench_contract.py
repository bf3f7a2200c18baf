"""bench.py prints ONE JSON line with the keys the driver reads; the reference arm runs without a GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches"}


def _run(args, timeout=900):
    env = dict(os.environ, GP_BENCH_CPU_THREADS="8")          # skip the thread-count probe of the CPU arm
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=timeout,
                       cwd=ROOT, env=env)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, p.stdout
    return json.loads(lines[0])


def test_reference_arm_line_on_cpu():
    j = _run(["--impl", "reference", "--steps", "1", "--warmup", "0", "--ref-res", "64"])
    assert BASE_KEYS <= set(j) and j["impl"] == "reference"
    assert j["metric"] == "images/sec at 768x768 depth" and j["unit"] == "images/s" and j["higher_is_better"] is True
    assert j["value"] > 0 and j["e2e"]["value"] == j["value"]
    assert j["e2e"]["h2d_bytes_per_step"] == 0 and j["e2e"]["d2h_bytes_per_step"] == 0
    cb = j["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == j["value"] and "sample" in cb


@pytest.mark.gpu
def test_engine_arm_line_on_gpu(tmp_path):
    j = _run(["--steps", "3", "--warmup", "3", "--batch", "1", "--res", "128", "--ref-res", "64", "--dump-outputs", str(tmp_path)])
    assert BASE_KEYS <= set(j) and "impl" not in j or j.get("impl") == "ours"
    assert j["n_gpus"] == 1 and j["steps"] == 3 and j["warmup"] >= 3 and j["scaling"] == "weak" and j["dtype"] == "f16"
    assert j["value"] > 0 and j["e2e"]["value"] > 0 and j["gpu_launches"] > 0
    assert j["e2e"]["h2d_bytes_per_step"] == 3 * 128 * 128 and j["e2e"]["d2h_bytes_per_step"] == 4 * 128 * 128
    r = j["roofline"]
    assert r["bound"] == "tensor" and r["unit"] == "TFLOP/s" and 0 < r["frac"] and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert {"value", "unit", "cores", "kind", "sample"} <= set(j["cpu_baseline"])
    assert "workload" in j["config"] and "sm_mhz" in j["clocks"]
    pred = np.load(tmp_path / "prediction.npy")             # the maps of the last timed step
    assert pred.shape == (1, 1, 128, 128) and pred.dtype == np.float32 and 0 <= pred.min() and pred.max() <= 1


def test_dump_outputs_stays_under_the_size_limit(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setattr(bench, "DUMP_LIMIT", 4096)
    small, big = np.arange(512, dtype=np.float32), np.arange(2048, dtype=np.float64)
    bench.dump_outputs(str(tmp_path / "a"), {"small": small})
    assert np.array_equal(np.load(tmp_path / "a" / "small.npy"), small)
    bench.dump_outputs(str(tmp_path / "b"), {"small": small, "big": big})      # 2048 + 16384 bytes: every 5th element
    got = {n: np.load(tmp_path / "b" / f"{n}.npy") for n in ("small", "big")}
    assert np.array_equal(got["small"], small[::5]) and np.array_equal(got["big"], big[::5])
    assert sum(v.nbytes for v in got.values()) <= 4096


def test_steps_must_be_positive():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                       timeout=300, cwd=ROOT)
    assert p.returncode != 0 and "--steps" in p.stderr


def test_reference_arm_under_torchrun_prints_one_line():
    """N > 1: the driver launches the reference arm like the engine arm; rank 0 alone works and prints."""
    env = dict(os.environ, GP_BENCH_CPU_THREADS="8")
    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29571", os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                        "--steps", "1", "--warmup", "0", "--ref-res", "64"], capture_output=True, text=True, timeout=900, cwd=ROOT,
                       env=env)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, p.stdout
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["n_gpus"] == 2 and j["value"] > 0
