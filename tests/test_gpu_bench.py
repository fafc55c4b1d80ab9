"""bench.py --dump-outputs: the last timed step's quadrature rule lands in DIR as float64 .npy files."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_writes_the_timed_rule(tmp_path):
    N, n = 200_000, 100
    out_dir = tmp_path / "dump"
    args = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
            "--N", str(N), "--M", "2000", "--n", str(n), "--no-extra", "--no-cpu-baseline", "--no-e2e",
            "--dump-outputs", str(out_dir)]
    out = subprocess.run(args, capture_output=True, text=True, timeout=600, cwd=tmp_path)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2
    assert sorted(os.listdir(out_dir)) == ["indices.npy", "weights.npy"]
    idx, w = np.load(out_dir / "indices.npy"), np.load(out_dir / "weights.npy")
    assert idx.dtype == np.float64 and w.dtype == np.float64 and idx.shape == w.shape
    assert 1 <= len(idx) <= n and np.array_equal(idx, np.round(idx))
    assert idx.min() >= 0 and idx.max() < N and bool((np.diff(idx) > 0).all())
    assert bool((w > 0).all()) and abs(w.sum() - 1.0) < 1e-9
