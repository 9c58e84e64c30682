"""bench.py contract: the reference arm runs without a GPU and prints ONE JSON line with the keys a consumer of the
line reads, the b200 arm refuses to run without a CUDA device (no CPU fallback), and on the GPU --dump-outputs writes
the same outputs on every run with the same arguments."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.timeout(300)
def test_reference_arm_json_line():
    env = dict(os.environ, OMP_NUM_THREADS="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--cpu-sample-envs", "512", "--cpu-sample-steps", "4"], capture_output=True, text=True, env=env,
                         timeout=280)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "6dof_env_steps_per_sec" and d["unit"] == "env-steps/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["gpu_launches"] == 0 and d["vs_baseline"] is None
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_b200_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA device present")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=200)
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_dump_outputs_repeat_exactly(tmp_path):
    """--dump-outputs writes obs / reward / done / flags of the last timed step as float32 / float64 .npy files, and two
    runs with the same arguments (seeded inputs) write the same values, so that two builds can be compared output for
    output."""
    import numpy as np
    n, dumps = 4096, []
    for r in range(2):
        d = tmp_path / f"run{r}"
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "1",
                              "--envs", str(n), "--preroll", "200", "--no-cpu-baseline", "--dump-outputs", str(d)],
                             capture_output=True, text=True, timeout=800)
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
        assert line["steps"] == 3
        dumps.append({p.stem: np.load(p) for p in d.glob("*.npy")})
    a, b = dumps
    assert sorted(a) == ["done", "env_index", "flags", "obs", "reward"]
    assert a["obs"].shape == (n, 14) and a["obs"].dtype == np.float32 and a["reward"].dtype == np.float64
    assert np.array_equal(a["env_index"], np.arange(n))
    for k in a:
        assert a[k].dtype in (np.float32, np.float64) and a[k].shape[0] == n, k
        assert np.array_equal(a[k], b[k]), k
    assert np.isfinite(a["obs"]).all() and a["done"].any()
