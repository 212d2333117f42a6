"""bench.py --impl reference (the reference's CPU path, oracle/reference_step.py) prints ONE JSON line with the
contract's keys; the GPU arm refuses to run without a CUDA device (there is no CPU fallback)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    env = dict(os.environ, OMP_NUM_THREADS="1")          # what torchrun exports: the arm must still use the cores
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1", "--workload", "fb15k237"], capture_output=True, text=True, env=env, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "triples/s" and d["value"] > 0 and d["higher_is_better"] is True
    assert d["e2e"] == {"value": d["value"], "unit": "triples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == d["value"] and cb["cores"] >= 1 and "sample" in cb
    assert "workload" in d["config"] and d["vs_baseline"] is None and d["data"] == "synthetic"


def test_gpu_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True,
                         text=True, timeout=600)
    assert out.returncode != 0 and "no CPU path" in (out.stderr + out.stdout)


def test_reference_arm_refuses_dump_outputs(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--dump-outputs", str(tmp_path / "d")], capture_output=True, text=True, timeout=600)
    assert out.returncode != 0 and "--dump-outputs" in out.stderr and not (tmp_path / "d").exists()


@pytest.mark.gpu
def test_gpu_arm_dumps_last_step_outputs(cuda_device, tmp_path):
    """--dump-outputs writes the state after the LAST timed step, the same in every run: warmup 3 + 2 timed steps and
    warmup 4 + 1 timed step take the same five steps on the same batches and must dump the same bits; one more step
    must change them."""
    def dump(warmup, steps):
        d = tmp_path / f"w{warmup}s{steps}"
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", str(warmup),
                              "--no-strict", "--no-c5", "--no-large-kernel", "--cpu-steps", "0", "--torch-gpu-steps", "0",
                              "--eval-batches", "1", "--dump-outputs", str(d)], capture_output=True, text=True, timeout=900)
        assert out.returncode == 0, out.stderr[-2000:]
        lines = [l for l in out.stdout.splitlines() if l.strip()]
        assert len(lines) == 1 and json.loads(lines[0])["steps"] == steps
        return {f[:-len(".npy")]: np.load(d / f) for f in os.listdir(d)}
    arrays = dump(3, 2)
    assert sorted(arrays) == ["O", "R", "S", "core", "loss", "rgrad_norm"]
    assert all(a.dtype in (np.float32, np.float64) and np.isfinite(a).all() for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    assert arrays["core"].shape == (10, 200, 200) and arrays["R"].shape == (22, 10)
    assert arrays["S"].shape == arrays["O"].shape == (8192, 200)
    assert np.abs(arrays["S"]).sum(1).min() > 0 and np.abs(arrays["O"]).sum(1).min() > 0     # every sampled row filled
    assert float(arrays["loss"]) > 0 and float(arrays["rgrad_norm"]) > 0
    same = dump(4, 1)
    for k, a in arrays.items():
        assert np.array_equal(a, same[k]), k
    later = dump(3, 3)
    for k in ("loss", "rgrad_norm", "core", "S", "O"):
        assert not np.array_equal(arrays[k], later[k]), k
