"""bench.py --dump-outputs on the GPU: two runs with the same arguments write the same outputs of the last timed step (the train
steps then use the engine's ordered reductions instead of fp32 atomics), for the headline train workload and for the
stand-alone Patch-PnP."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(1200)]

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, *args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--dump-outputs", str(out_dir), *args],
                       cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    return line, {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


def test_dump_outputs_of_train_step_are_reproducible(tmp_path):
    (la, a), (lb, b) = (_bench(tmp_path / r, "--quick", "--steps", "3", "--warmup", "3") for r in "ab")
    for line in (la, lb):
        assert line["steps"] == 3 and line["config"]["deterministic"] is True
    assert sorted(a) == sorted(b) == ["grad_sample", "grad_sample_index", "head_sample", "head_sample_rows", "losses", "rot", "trans"]
    for k in a:
        assert a[k].dtype in (np.float32, np.float64), k
        if k == "grad_sample":  # the bias-gradient column sums and the GroupNorm backward still add partials with atomics
            assert np.linalg.norm(a[k] - b[k]) <= 1e-6 * np.linalg.norm(b[k])
        else:
            assert np.array_equal(a[k], b[k]), k
    assert a["losses"].shape == (8,) and np.isfinite(a["losses"]).all() and (a["losses"] > 0).all()
    rot = a["rot"].astype(np.float64)
    assert rot.shape == (64, 3, 3) and np.abs(rot @ rot.transpose(0, 2, 1) - np.eye(3)).max() < 1e-4  # decoded rotations
    assert a["head_sample"].shape == (1 << 16, 69) and (a["grad_sample"] != 0).mean() > 0.5


def test_dump_outputs_of_patch_pnp_are_reproducible(tmp_path):
    (la, a), (lb, b) = (_bench(tmp_path / r, "--config", "pnp", "--steps", "2", "--warmup", "3") for r in "ab")
    assert la["steps"] == lb["steps"] == 2
    assert sorted(a) == ["rot", "t"] and a["rot"].shape[0] == a["t"].shape[0] == 512
    for k in a:
        assert np.array_equal(a[k], b[k]), k
