"""CPU: the bench.py contract that can be exercised without a GPU — the reference arm (`--impl reference`: the oracle
port on the host cores) prints exactly one JSON line with the keys the driver reads, and the product arm refuses to
run without a CUDA device instead of falling back."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    # B200SVD_BENCH_CONTRACT_TEST: same code path on the reduced-width network (the real arm needs minutes of host time)
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=900, cwd=ROOT,
                       env=dict(os.environ, B200SVD_BENCH_CONTRACT_TEST="1"))
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "denoise_steps_per_sec" and d["unit"] == "steps/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["n_gpus"] == 1 and d["gpu_launches"] == 0
    assert d["value"] > 0 and abs(d["ms_per_step"] - 1e3 / d["value"]) < 1e-6 * d["ms_per_step"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_product_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "3",
                        "--no-cpu-baseline"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert p.returncode != 0 and "no CPU path" in (p.stderr + p.stdout)


@pytest.mark.gpu
def test_product_arm_dumps_its_last_step(cuda_dev, tmp_path):
    """--dump-outputs writes what the last timed step returned (the sampler's next latent) as float32."""
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--settle", "0",
                        "--no-cpu-baseline", "--no-gpu-reference", "--no-chunk", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    d = json.loads([ln for ln in p.stdout.splitlines() if ln.strip()][-1])
    assert d["steps"] == 2 and d["finite"]
    z = np.load(tmp_path / "latent.npy")
    assert z.dtype == np.float32 and z.shape == (25, 4, 72, 128) and np.isfinite(z).all()


def test_usable_cores_respects_affinity():
    sys.path.insert(0, ROOT)
    import bench
    n = bench._usable_cores()
    assert 1 <= n <= 32 and n <= (os.cpu_count() or 1)
    assert bench._usable_cores(cap=2) <= 2
