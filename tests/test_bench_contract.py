"""bench.py contract (CPU side): the reference arm runs without a GPU and prints ONE JSON line with the keys the
driver reads; the product arm must refuse to run without a CUDA device instead of falling back to the CPU.  On the
GPU: --dump-outputs writes what the last timed step computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args):
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT, env=env, capture_output=True,
                          text=True, timeout=600)


def test_reference_arm_json_line():
    out = run_bench("--impl", "reference", "--steps", "3", "--warmup", "1")
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip().startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    with open(os.path.join(ROOT, "BASELINE.json")) as fh:
        base = json.load(fh)
    assert d["impl"] == "reference" and "unavailable" not in d
    assert d["steps"] == 3 and d["warmup"] >= 1 and d["n_gpus"] == 1
    assert d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["unit"] == "iter/s" and d["dtype"] == "f64"
    if isinstance(base.get("metric"), str):
        assert "iter" in base["metric"].lower() or "rtr" in d["metric"]
    assert d["value"] > 0 and abs(d["ms_per_step"] * d["value"] - 1e3) <= 1e-6 * 1e3
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_product_arm_fails_loudly_without_gpu():
    out = run_bench("--steps", "1", "--warmup", "1", "--no-cpu", "--no-spmv")
    assert out.returncode != 0
    assert "{\"metric\"" not in out.stdout                   # no bench line from a CPU fallback


def test_steps_must_be_positive():
    out = run_bench("--impl", "reference", "--steps", "0", "--warmup", "1")
    assert out.returncode != 0 and "--steps" in out.stderr


@pytest.mark.gpu
def test_dump_outputs_is_the_last_timed_step(tmp_path):
    """--steps 2: the last timed step is step 1 of the cycle from the initial point, the same step as trajectory[1]."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--no-cpu",
                          "--no-spmv", "--no-multi", "--dump-outputs", str(tmp_path)], cwd=ROOT, capture_output=True,
                         text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([ln for ln in out.stdout.splitlines() if ln.strip().startswith("{")][-1])
    assert d["steps"] == 2
    assert sorted(os.listdir(tmp_path)) == ["X.npy", "f_opt.npy", "gradnorm_opt.npy"]
    X = np.load(os.path.join(tmp_path, "X.npy"))
    assert X.dtype == np.float64 and X.shape == (5, 4 * 2500) and np.all(np.isfinite(X))
    f = np.load(os.path.join(tmp_path, "f_opt.npy"))
    g = np.load(os.path.join(tmp_path, "gradnorm_opt.npy"))
    assert abs(f[0] - d["trajectory"][1]["f"]) <= 1e-12 * abs(f[0])
    assert abs(g[0] - d["trajectory"][1]["gradnorm"]) <= 1e-9 * abs(g[0])
