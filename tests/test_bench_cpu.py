"""bench.py contract checks that need no GPU: the reference arm (CPU oracle) prints one JSON line with the agreed keys, and the
CUDA arm refuses to run -- loudly, non-zero -- when there is no device (no CPU fallback for the product path)."""
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT, capture_output=True, text=True, timeout=900)


def test_reference_arm_json_contract():
    r = _run("--impl", "reference", "--gpus", "1", "--steps", "6", "--warmup", "1", "--cpu-batch", "2")
    assert r.returncode == 0, r.stderr[-2000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
    d = json.loads(line)
    assert d["impl"] == "reference" and d["unit"] == "crops/s" and d["higher_is_better"] is True and d["n_gpus"] == 1
    assert d["steps"] == 6  # --steps is the number of timed steps
    assert d["value"] > 0 and d["vs_baseline"] is None and d["data"] == "synthetic"
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    # same metric / unit as the CUDA arm (BASELINE.json's metric)
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert isinstance(base, dict)
    assert "crops" in d["metric"]


def test_cuda_arm_fails_loudly_without_a_gpu():
    if torch.cuda.is_available():
        import pytest

        pytest.skip("a GPU is present")
    r = _run("--steps", "1", "--warmup", "1")
    assert r.returncode != 0
    assert "no CPU fallback" in (r.stdout + r.stderr)


def test_dump_outputs_are_a_fixed_sample_under_64mb(tmp_path):
    """--dump-outputs: the last timed step's losses, poses, head maps and gradient as float32 / float64 .npy files, the large
    two sampled at the same rows / entries on every run, 64 MB at most."""
    import numpy as np

    import bench

    g = torch.Generator().manual_seed(1)
    B = 64
    last = dict(losses=torch.rand(8, generator=g), logits=torch.randn(B * 4096, 72, generator=g),
                rot=torch.randn(B, 3, 3, generator=g), trans=torch.randn(B, 3, generator=g))
    flat_grad = torch.randn(3 * bench.DUMP_GRAD_ELEMS, generator=g)  # the model's is ~35M entries; the sample size is fixed
    a, b = bench.train_step_outputs(last, flat_grad), bench.train_step_outputs(last, flat_grad)
    assert sorted(a) == sorted(b) and all(np.array_equal(a[k], b[k]) for k in a)
    rows, idx = a["head_sample_rows"].astype(np.int64), a["grad_sample_index"].astype(np.int64)
    assert len(np.unique(rows)) == bench.DUMP_HEAD_ROWS and len(np.unique(idx)) == bench.DUMP_GRAD_ELEMS
    assert np.array_equal(a["head_sample"], last["logits"].numpy()[rows, :69])
    assert np.array_equal(a["grad_sample"], flat_grad.numpy()[idx])
    assert np.array_equal(a["losses"], last["losses"].numpy()) and np.array_equal(a["rot"], last["rot"].numpy())
    out = tmp_path / "out"
    bench.dump_outputs(str(out), a)
    files = sorted(out.iterdir())
    assert [f.name for f in files] == sorted(k + ".npy" for k in a)
    assert sum(f.stat().st_size for f in files) <= 64 << 20
    for f in files:
        assert np.load(f).dtype in (np.float32, np.float64)
