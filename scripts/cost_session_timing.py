"""Wall time of one cost / gradient evaluation as the BFGS loop sees it: the resident kernel of an inner solve
(cost_persistent=1, bench hook 4) against one launch per evaluation (hook 5), the bare kernel (hook 1), and the whole job
both ways, with the block shape (threads x ring stages) the resident kernel took.
Usage: python scripts/cost_session_timing.py [points ...]"""
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

from leica_point_cloud_processing_b200 import Engine, synth  # noqa: E402

sizes = [int(a) for a in sys.argv[1:]] or [100_000, 1_000_000, 4_000_000]
eng = Engine(0)
for n in sizes:
    s = (n / 1e6) ** 0.5
    src, tgt, _ = synth.make_pair(n, n, length=4.0 * s, width=2.0 * s)
    out = {}
    for mode in (0, 1):
        eng.set_params(max_corr_distance=1.0, cost_persistent=mode)
        for rep in range(3):
            t0 = time.perf_counter()
            eng.set_clouds(tgt, src)
            res = eng.align()
            fit = eng.fitness(res["transform"])
            dt = (time.perf_counter() - t0) * 1e3
        out[mode] = (dt, res)
    T = out[1][1]["transform"]
    ms_res, _ = eng.bench_kernel(4, T, iters=200)
    ms_one, _ = eng.bench_kernel(5, T, iters=200)
    ms_k, _ = eng.bench_kernel(1, T, iters=50)
    _, _, info = eng.cost_session(np.zeros((1, 6)))
    same = np.array_equal(out[0][1]["transform"], out[1][1]["transform"])
    print(f"n={n} shape={info['threads']}x{info['stages']} eval wall us: resident {1e3 * ms_res:.2f}  per-launch {1e3 * ms_one:.2f}  "
          f"kernel-only {1e3 * ms_k:.2f} | job ms (host arrays, wall): per-launch {out[0][0]:.3f} resident {out[1][0]:.3f} "
          f"evals {out[1][1]['cost_evaluations']} ms_cost {out[0][1]['ms_cost']:.3f} -> {out[1][1]['ms_cost']:.3f} "
          f"ms_corr {out[1][1]['ms_corr']:.3f} identical={same}", flush=True)
eng.close()
