"""bench.py end to end on the tiny Llama: --dump-outputs writes the output of every forward of the last timed step, the
same from run to run, and the result line reports the --steps it was given."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from gbx_lm_b200 import workloads as W

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
           "--model", "tiny-llama", "--no-also", "--no-cpu-baseline", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, cwd=str(out.parent), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_bench_dump_outputs(cuda_device, tmp_path):
    dims = W.MODELS["tiny-llama"]
    plan = W.layer_plan(dims, W.STRATEGIES["bpw-4.0"](dims.layers), 4, 64)
    a, b = tmp_path / "a", tmp_path / "b"
    assert _bench(a, 2)["steps"] == 2
    assert _bench(b, 5)["steps"] == 5
    names = sorted(f"layer{i:02d}_{p}.npy" for (i, p, *_) in plan)
    assert sorted(os.listdir(a)) == names and sorted(os.listdir(b)) == names
    for (i, p, n, *_) in plan:
        ya, yb = np.load(a / f"layer{i:02d}_{p}.npy"), np.load(b / f"layer{i:02d}_{p}.npy")
        assert ya.dtype == np.float32 and ya.shape == (1, n)
        assert np.isfinite(ya).all() and np.abs(ya).max() > 0
        assert np.array_equal(ya, yb), (i, p)  # seeded inputs: every run computes the same outputs
