"""bench.py's reference arm (the CPU port of the reference's path) runs without a GPU: its stdout must be exactly one JSON
line with the contract's keys, also under torchrun (rank 0 prints, the other rank prints nothing and exits 0, and the
oracle gets the host's threads back although torchrun exports OMP_NUM_THREADS=1)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
        "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"}


def _check(stdout, gpus):
    lines = [l for l in stdout.splitlines() if l.strip()]
    assert len(lines) == 1, stdout          # nothing but the JSON line on stdout
    d = json.loads(lines[0])
    assert KEYS <= set(d), KEYS - set(d)
    assert d["impl"] == "reference" and d["metric"] == "gicp_correspondences_per_s" and d["n_gpus"] == gpus
    assert d["value"] > 0 and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]
    return d


def test_reference_arm_prints_one_json_line():
    run = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--ref-points", "20000"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert run.returncode == 0, run.stderr[-2000:]
    _check(run.stdout, 1)


def test_bad_arguments_are_rejected():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        run = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True,
                             timeout=600, cwd=ROOT)
        assert run.returncode == 2 and run.stdout == "", (extra, run.stderr[-2000:])


def test_reference_arm_under_torchrun_rank0_only():
    run = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29611", os.path.join(ROOT, "bench.py"), "--impl",
                          "reference", "--gpus", "2", "--steps", "1", "--warmup", "0", "--ref-points", "20000"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert run.returncode == 0, run.stderr[-2000:]
    d = _check(run.stdout, 2)
    assert d["cpu_baseline"]["cores"] == (os.cpu_count() or 1)
