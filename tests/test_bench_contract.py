"""CPU: the reference arm of bench.py (`--impl reference`: the reference's arithmetic on the host cores) prints ONE JSON
line with the contract's keys; and `bench.py` without a GPU refuses to run the B200 arm instead of falling back.
GPU: `--dump-outputs` writes the same arrays for the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "mc_inference_image_samples_per_sec_N64_bayesian_resnet18"
    assert d["unit"] == "image-samples/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["steps"] == 1 and d["n_gpus"] == 1 and d["data"] == "synthetic"
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    # same step shape as the B200 arm: the full N=64 evaluate() loop per step; the real reference package when
    # baseline/_ref is installed (it is in the build container and travels to the GPU box)
    assert d["config"]["mc_samples_per_step"] == 64 and d["config"]["global_batch"] == 128
    if os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "bayesian_torch")):
        assert cb["kind"] == "reference"
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_b200_arm_refuses_to_run_without_a_gpu():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0 and "no CUDA device" in (r.stderr + r.stdout)
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")]


@pytest.mark.parametrize("args", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"],
                                  ["--profile", "--dump-outputs", "out"]])
def test_bench_rejects_bad_arguments(args, tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                       timeout=600, cwd=tmp_path)
    assert r.returncode == 2 and "error:" in r.stderr
    assert not list(tmp_path.iterdir())


@pytest.mark.gpu
def test_dump_outputs_repeat_for_the_same_arguments(tmp_path):
    """--dump-outputs writes the last timed step's mean / var; two runs with the same arguments agree bit for bit"""
    dumps = []
    for run in ("a", "b"):
        d = tmp_path / run
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--dtype", "fp32",
                            "--no-cpu-baseline", "--dump-outputs", str(d)], capture_output=True, text=True, timeout=900,
                           cwd=tmp_path)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])["steps"] == 2
        dumps.append({f.name: np.load(f) for f in sorted(d.iterdir())})
    a, b = dumps
    assert sorted(a) == ["fp32_mean.npy", "fp32_var.npy"]
    for name in a:
        assert a[name].dtype == np.float32 and a[name].shape == (128, 10), name
        assert np.array_equal(a[name], b[name]), name
    assert np.allclose(a["fp32_mean.npy"].sum(-1), 1.0, atol=1e-5) and (a["fp32_var.npy"] >= 0).all()
