"""Config 4 (10 M scan + FOD blobs minus the 10 M CAD cloud) through one context and through EngineGroup(devices).

    python scripts/group_difference_timing.py --devices 0,1,2,3,4,5,6,7 [--n 10000000] [--reps 7]

Both clouds come from pageable 32-byte rows (pcl::PointXYZRGB as the reference holds them) and from pinned packed xyz.  Every
call is warmed up, timed on the host clock around the whole call (it returns after its last copy to the host mask), and its
mask is compared with the single context's; the median of --reps runs is printed, with the subtract points each member
indexed.  Members that share one GPU (--devices 0,0) run one after another on it: that is a correctness run, not a speed
number."""
import argparse
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from leica_point_cloud_processing_b200 import Engine, EngineGroup, synth  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--devices", default="0")
    ap.add_argument("--n", type=int, default=10_000_000)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--threshold", type=float, default=4e-4)
    a = ap.parse_args()
    devices = [int(d) for d in a.devices.split(",")]
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True,
                         text=True).stdout.strip(), flush=True)
    src, tgt, T_star = synth.make_pair(a.n, a.n, length=12.0, width=4.0)
    inp, _ = synth.add_fod_blobs(synth.apply_rigid(T_star, src), n_blobs=20, length=12.0, width=4.0)

    def rows32(xyz):
        r = np.zeros((len(xyz), 8), np.float32)
        r[:, :3] = xyz
        r[:, 3] = 1.0
        return r

    layouts = {"pageable 32-byte rows": (rows32(inp), rows32(tgt)),
               "pinned packed xyz": (torch.from_numpy(inp).pin_memory(), torch.from_numpy(tgt).pin_memory())}
    eng = Engine(devices[0])
    want, kept = eng.cloud_difference(inp, tgt, a.threshold)
    print(f"{len(inp)} input points, {len(tgt)} subtract points, thr {a.threshold}: kept {kept}", flush=True)
    grp = EngineGroup(devices)

    def timed(label, fn):
        fn()
        fn()
        ms = []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            mask, k = fn()
            ms.append((time.perf_counter() - t0) * 1e3)
            assert k == kept and np.array_equal(mask, want), label
        print(f"{label}: median {np.median(ms):.2f} ms (min {min(ms):.2f}, max {max(ms):.2f}, {a.reps} runs)", flush=True)

    for name, (i_cloud, s_cloud) in layouts.items():
        timed(f"one context       {name}", lambda: eng.cloud_difference(i_cloud, s_cloud, a.threshold))
        timed(f"group {devices} {name}", lambda: grp.cloud_difference(i_cloud, s_cloud, a.threshold))
    print("subtract points indexed per member:", [grp.member(r).grid_info(2)["n_indexed"] for r in range(grp.size)])
    grp.close()
    eng.close()


if __name__ == "__main__":
    main()
