"""bench.py contract pieces that run without a GPU: the reference arm (CPU restatement timed on the host cores) prints one
JSON line with the agreed keys, and the product arm refuses to run without a CUDA device instead of falling back."""
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--ref-rows", "8"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "GSamples/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["dtype"] == "f64" and line["vs_baseline"] is None
    assert line["config"]["workload"] == "batch4096x4096_db4_J4"
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and "sample" in cb
    assert line["e2e"] == {"value": line["value"], "unit": "GSamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_do_nothing():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "1"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_steps_below_one_are_refused():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                       timeout=120, cwd=ROOT)
    assert p.returncode != 0 and "--steps must be at least 1" in p.stderr


@pytest.mark.gpu
def test_dump_outputs_is_the_same_from_run_to_run(tmp_path):
    import numpy as np
    runs = []
    for k in range(2):
        out = tmp_path / f"run{k}"
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "batch16x4096_db4_J4", "--steps", "2",
                            "--warmup", "1", "--no-cpu-baseline", "--no-e2e", "--no-extra", "--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert p.returncode == 0, p.stderr[-2000:]
        assert json.loads(p.stdout.strip().splitlines()[-1])["steps"] == 2
        runs.append({n: np.load(out / f"{n}.npy") for n in ("w", "v", "xr")})
    a, b = runs
    assert a["w"].shape == (4, 16 * 4096) and a["v"].shape == a["xr"].shape == (16 * 4096,)
    for n in a:
        assert a[n].dtype == np.float64 and np.array_equal(a[n], b[n]), n
    assert sum(x.nbytes for x in a.values()) <= 64 << 20


@pytest.mark.skipif(torch.cuda.is_available(), reason="needs a machine without CUDA")
def test_product_arm_has_no_cpu_fallback():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"], capture_output=True,
                       text=True, timeout=300, cwd=ROOT)
    assert p.returncode != 0 and "no CPU path" in (p.stderr + p.stdout)
