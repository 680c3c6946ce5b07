"""bench.py contract checks that need no GPU: the reference arm runs on CPU and prints one JSON line
with the agreed keys; the default arm refuses to run without a CUDA device (no CPU fallback)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"].startswith("ECDSA-P256 verifies/sec")
    for k in ("value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "config", "cpu_baseline", "e2e"):
        assert k in line
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["value"] > 1000


def test_default_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode != 0  # fails loudly: there is no CPU fallback for the product path


def test_steps_must_be_positive():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode != 0 and "--steps" in out.stderr


def _workload():
    import oracle
    from oracle import corpus
    return corpus.make_batch(oracle.P256, n=65536, K=1024, seed=1)   # bench.py's rank-0 workload


def _dumped_verdicts_equal(out_dir, want):
    import numpy as np
    got = np.load(os.path.join(out_dir, "verdicts.npy"))
    assert got.dtype == np.float32 and got.shape == (65536,)
    assert np.array_equal(got, want.astype(np.float32))
    assert 0 < want.sum() < want.size


def test_reference_arm_dumps_the_last_step_outputs(tmp_path):
    import oracle
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert sorted(os.listdir(tmp_path)) == ["verdicts.npy"]
    # the reference arm verifies against the pre-built key of each item (key_idx), not the per-item qx / qy
    b = _workload()
    _, want = oracle.bench_verify(oracle.P256, b["r"], b["s"], b["keys"], b["key_idx"], b["digest"])
    _dumped_verdicts_equal(tmp_path, want)


@pytest.mark.gpu
def test_default_arm_dumps_the_last_step_outputs(tmp_path):
    import oracle
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--no-extras",
                          "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 2
    assert sorted(os.listdir(tmp_path)) == ["verdicts.npy"]
    b = _workload()
    _dumped_verdicts_equal(tmp_path, oracle.verify_batch(oracle.P256, b["r"], b["s"], b["qx"], b["qy"], b["digest"]))
