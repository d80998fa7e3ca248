"""bench.py's command line -- the reference arm (the oracle port on the host cores) prints the contract's JSON line,
the product arm refuses to run without a GPU instead of falling back to the CPU, and on a GPU the same arguments give the
same inputs and the same dumped outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "A", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["unit"] == "POI/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert d["config"]["workload"].startswith("A:")
    # BASELINE.md section 3: the CPU arm names its CPU, its core and thread counts, and reports best-of-N next to the mean
    cb = d["cpu_baseline"]
    assert cb["cpu_model"] and cb["logical_cpus"] >= cb["cores"] and cb["value"] >= cb["value_mean"] > 0
    assert "OMP_PROC_BIND=close" in cb["sample"] and "best of" in cb["sample"]
    assert set(d["config"]) == {"workload", "pois_per_gpu", "conv", "stop", "parallelism", "l2"}  # the GPU arm's keys


def test_reference_arm_dumps_outputs(tmp_path):
    """--dump-outputs writes the POI records of the last timed step; the same arguments give the same records."""
    sys.path.insert(0, ROOT)
    from opencorr_b200 import synth
    dumps = []
    for run in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "A", "--steps", "2",
                              "--warmup", "0", "--dump-outputs", str(tmp_path / run)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr
        assert os.listdir(tmp_path / run) == ["pois.npy"]
        dumps.append(np.load(tmp_path / run / "pois.npy"))
    q = dumps[0]
    assert q.dtype == np.float32 and q.shape == (200, 25)
    assert np.array_equal(q[:, 0:2], synth.grid_2d(*synth.CONFIGS["A"]["grid"]))
    assert (q[:, 16] > 0.9).mean() > 0.9  # the records hold converged IC-GN results
    assert np.array_equal(dumps[0], dumps[1])


def test_product_arm_needs_a_gpu():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "A", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert out.returncode != 0
    assert "no CPU fallback" in out.stdout + out.stderr


@pytest.mark.gpu
def test_gpu_rendered_inputs_are_reproducible():
    """The bench renders its pairs on the GPU (synth._render_torch): the same arguments give bit-identical images, and the same
    images as the numpy renderer."""
    import torch
    sys.path.insert(0, ROOT)
    from opencorr_b200 import synth
    dev = torch.device("cuda", 0)
    for f, size in ((synth.speckle_pair_2d, (512, 384)), (synth.speckle_pair_3d, (64, 56, 48))):
        a, b, c = f(*size, device=dev), f(*size, device=dev), f(*size)
        for x, y, z in zip(a, b, c):
            assert np.array_equal(x, y)
            assert np.array_equal(x, z)


@pytest.mark.gpu
def test_product_arm_dumps_outputs(tmp_path):
    """--dump-outputs on the timed GPU path: the records of the last timed step, identical from run to run."""
    sys.path.insert(0, ROOT)
    from opencorr_b200 import synth
    dumps = []
    for run in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "A", "--steps", "1", "--warmup", "3",
                              "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / run)],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr
        assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 1
        assert os.listdir(tmp_path / run) == ["pois.npy"]
        dumps.append(np.load(tmp_path / run / "pois.npy"))
    q = dumps[0]
    assert q.dtype == np.float32 and q.shape == (200, 25)
    assert np.array_equal(q[:, 0:2], synth.grid_2d(*synth.CONFIGS["A"]["grid"]))
    assert (q[:, 16] > 0.9).mean() > 0.9
    assert np.array_equal(dumps[0], dumps[1])
