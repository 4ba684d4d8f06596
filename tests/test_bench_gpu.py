"""bench.py on the GPU at a small size: one JSON line, and --dump-outputs saves what the last timed step returned (the
transform, the fitness and the iteration counts the line also reports)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_dump_outputs_holds_the_last_timed_step(tmp_path):
    out = tmp_path / "outputs"
    run = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
                          "--points", "200000", "--quick", "--no-cpu-baseline", "--dump-outputs", str(out)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert run.returncode == 0, run.stderr[-2000:]
    d = json.loads(run.stdout)
    assert d["steps"] == 2 and d["warmup"] == 1
    arrays = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert set(arrays) == {"transform", "fitness", "converged", "outer_iterations", "inner_iterations",
                           "cost_evaluations", "corr_queries", "corr_pairs_last"}
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    T = arrays["transform"]
    assert T.shape == (4, 4) and np.allclose(T[:3, :3] @ T[:3, :3].T, np.eye(3), atol=1e-5)
    assert float(arrays["fitness"]) == d["fitness"]
    assert float(arrays["converged"]) == 1.0
    assert float(arrays["outer_iterations"]) == d["config"]["outer_iterations"]
    assert float(arrays["cost_evaluations"]) == d["config"]["cost_evaluations"]
