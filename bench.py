#!/usr/bin/env python
"""bench.py - GICP hot path benchmark (BASELINE.json metric: GICP correspondences/s and align ms).

    python bench.py --gpus N --steps K --warmup W          # this repo's CUDA engine (N > 1: under torchrun)
    python bench.py --impl reference --gpus N ...           # the reference's CPU algorithm (oracle, all host threads)
    python bench.py ... --dump-outputs DIR                  # also save the last timed step's results as DIR/*.npy

A step = one complete registration job on one synthetic pair (SURVEY section 8d config 2 at N = 1: 1 M-point noisy
scan vs 1 M-point CAD cloud of the aircraft-panel surface, 5 deg / 2 cm initial offset, gate 1 m): index both clouds,
kNN-20 covariances, the GICP outer loop to convergence, fitness score.  `value` is measured with the raw clouds
already resident in HBM; `e2e` goes through the same C-ABI calls with pinned HOST buffers, so the host->device copy
of both clouds and the read-back of the transform and fitness are inside the timed region.
value = (source queries answered by the correspondence kernel over all outer iterations, all ranks) / step time.
N > 1: weak scaling, 1 M source AND target points per GPU on a panel whose AREA grows with the point count (the same
8 m^2 per million points at every N); source sharded by rank, target replicated; the 14 partial sums of a cost
evaluation are added across the GPUs inside the cost kernel over NVLink peer memory (ncclAllReduce when the ranks
cannot map each other's memory).

Besides the headline the line carries, under `detail` (measured outside the timed steps of the headline):
  parity_vs_oracle       the job against the CPU oracle (N = 1: the benchmark workload itself; N > 1: a 1 M / 1 M pair of
                         the same generator solved by the SHARDED engine).  A miss of the north_star tolerance ends the
                         run with exit code 3.
  parity_vs_single_gpu   N > 1: the benchmark workload solved once more by an unsharded engine on rank 0's GPU.
  config3                BASELINE config 3: 10 M vs 10 M points, strong-scaled over the run's N GPUs (ms per job with
                         the clouds resident and end to end from pinned host clouds).
  sweep                  BASELINE config 5: 100 k ... 10 M points per cloud, strong-scaled over the run's N GPUs.
  issue_roofline         the instruction-issue bound of the search kernels (they are not HBM-bound).
  per-kernel times, the opt-in moments objective and the FOD pipeline rows either side of the registration (N = 1).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GATE_M = 1.0  # config 2: the only integer gate reachable through setMaxCorrespondenceDistance(int) that holds 20 cm
ROT_TOL, TRANS_TOL_REL, FIT_TOL_REL = 1e-4, 1e-5, 1e-4   # north_star parity bars
SWEEP_POINTS = (100_000, 300_000, 1_000_000, 3_000_000, 10_000_000)
CONFIG3_POINTS = 10_000_000


def workload_points(n_gpus, override):
    return override if override else 1_000_000 * n_gpus


def panel_dims(n):
    """Iso-density panels: 8 m^2 of surface per million points (4 m x 2 m at 1 M, 12.6 m x 6.3 m at 10 M), so that
    weak-scaling efficiency and the sweep compare like with like (~2.8 mm between neighbouring samples everywhere)."""
    s = (n / 1_000_000) ** 0.5
    return 4.0 * s, 2.0 * s


def make_clouds(n):
    from leica_point_cloud_processing_b200 import synth
    length, width = panel_dims(n)
    src, tgt, T_star = synth.make_pair(n, n, length=length, width=width)
    return src, tgt, T_star, (length, width)


def bbox_diag(a, b):
    lo = np.minimum(a.min(0), b.min(0))
    hi = np.maximum(a.max(0), b.max(0))
    return float(np.linalg.norm(hi - lo))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            parts = [p.strip() for p in l.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_hbm_peak():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_counters():
    """Per-launch counters of the main kernels from the committed `ncu --set full` capture (profiles/ncu_counters.json
    names the capture and the commit it was taken on)."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "ncu_counters.json")))
    except Exception:
        return {}


# ---------------------------------------------------------------------------------------------------------------
def run_reference(args):
    """The reference's own CPU algorithm for this path (oracle restatement of PCL 1.8.1 GICP; PCL itself cannot be
    built in this image), all host threads, same workload generator, bounded in size."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # torchrun exports OMP_NUM_THREADS=1 to every rank; this arm is the CPU implementation "with all the host threads it
    # can use", so the OpenMP runtime of the oracle library (loaded below, not before) gets the whole host back
    if os.environ.get("OMP_NUM_THREADS") == "1" and "TORCHELASTIC_RUN_ID" in os.environ:
        os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)
    from oracle.oracle import Oracle, default_params
    orc = Oracle(fast=True)
    n_full = workload_points(args.gpus, args.points)
    n = min(n_full, args.ref_points)
    # the bounded sample keeps the workload's sampling DENSITY (a patch of the same panel family, 8 m^2 per million points)
    src, tgt, T_star, dims = make_clouds(n)
    prm = default_params(max_corr_distance=GATE_M)
    times, queries, outer = [], 0, 0
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        r = orc.align(src, tgt, prm)
        orc.fitness(src, tgt, r["T"])
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
            queries += r["n_corr_queries"]
            outer = r["outer_iterations"]
    total = sum(times)
    value = queries / total
    sample = (f"full workload: {n} source x {n} target points" if n == n_full else
              f"{n} source x {n} target points of the same generator at the same density (workload is {n_full}); "
              f"whole job per step")
    line = {
        "impl": "reference", "metric": "gicp_correspondences_per_s", "value": value, "unit": "correspondences/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 search / f64 accumulate",
        "data": "synthetic",
        "config": {"workload": workload_name(n_full, args.gpus), "outer_iterations": outer},
        "cpu_baseline": {"value": value, "unit": "correspondences/s", "cores": orc.num_threads(), "kind": "port",
                         "sample": sample},
        "e2e": {"value": value, "unit": "correspondences/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


def workload_name(n, world):
    l, w = panel_dims(n)
    return (f"aircraft-panel {n} src vs {n} tgt ({l:.2f} m x {w:.2f} m, 8 m^2 per M points), 5deg/2cm offset, gate {GATE_M} m "
            f"(SURVEY 8d config 2{' x N, weak' if world > 1 else ''})")


# ---------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    from leica_point_cloud_processing_b200 import Engine, synth
    from leica_point_cloud_processing_b200.distributed import env_rank_world, init_engine_comm

    rank, world, local_rank = env_rank_world()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    peak, peak_src = measured_hbm_peak()
    counters = ncu_counters()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    eng = Engine(local_rank)
    fused_peer = init_engine_comm(eng, rank, world)
    job_params = dict(max_corr_distance=GATE_M, mahalanobis_fp32=args.maha_fp32, cost_moments=args.cost_moments,
                      use_previous_match=args.seed_previous)
    eng.set_params(**job_params)
    estream = torch.cuda.ExternalStream(eng.stream_handle(), device=torch.device("cuda", local_rank))

    def step(e, tgt_buf, src_buf):
        # host clouds: both uploads are queued on the copy stream, target first, so that the source uploads while the
        # target is being indexed (no-op on device clouds)
        e.prefetch(0, tgt_buf)
        e.prefetch(1, src_buf)
        e.set_clouds(tgt_buf, src_buf)   # index target; its covariances overlap the source's index; source covariances
        res = e.align()
        fit = e.fitness(res["transform"])
        return res, fit

    def timed(tgt_buf, src_buf, steps, warmup):
        for _ in range(warmup):
            flush.zero_()
            step(eng, tgt_buf, src_buf)
        times, last, queries, ms_corr, n_corr_launch = [], None, 0, 0.0, 0
        for _ in range(steps):
            flush.zero_()
            barrier()
            # device time of the step: CUDA events on the stream the engine launches on (the step also contains the
            # host BFGS loop, which the events bracket as idle gaps between launches)
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record(estream)
            res, fit = step(eng, tgt_buf, src_buf)
            ev1.record(estream)
            torch.cuda.synchronize()
            dt = ev0.elapsed_time(ev1) * 1e-3
            barrier()
            times.append(max_over_ranks(dt))
            queries += res["corr_queries"]
            ms_corr += res["ms_corr"]
            n_corr_launch += res["outer_iterations"]
            last = (res, fit)
        return times, last, queries, ms_corr, n_corr_launch

    class Clouds:
        """One synthetic pair: numpy arrays, pinned host tensors and device copies (every rank holds both full clouds,
        as a caller of the sharded engine does: each rank passes the same arrays and the engine picks its shard)."""

        def __init__(self, n):
            self.n = n
            self.src, self.tgt, self.T_star, self.dims = make_clouds(n)
            self.h_src = torch.from_numpy(self.src).pin_memory()
            self.h_tgt = torch.from_numpy(self.tgt).pin_memory()
            self.d_src = self.h_src.cuda()
            self.d_tgt = self.h_tgt.cuda()
            self.diag = bbox_diag(self.src, self.tgt)

    def job_series(c, steps, warmup, e2e=True):
        """ms per job / corr per s of the (possibly sharded) engine on pair `c`, clouds resident and end to end."""
        t, (r, f), q, msc, nl = timed(c.d_tgt, c.d_src, steps, warmup)
        n_shard = c.n // world
        corr_bytes = 96.0 * n_shard + 16.0 * c.n
        out = {"points_per_cloud": c.n, "panel_m": [round(c.dims[0], 3), round(c.dims[1], 3)],
               "ms_per_job": 1e3 * sum(t) / len(t), "corr_per_s": q / sum(t), "outer_iterations": r["outer_iterations"],
               "cost_evaluations": r["cost_evaluations"], "fitness": f,
               "corr_pass_ms": msc / max(nl, 1), "corr_pass_frac_of_hbm": corr_bytes / (msc / max(nl, 1) * 1e-3) / 1e9 / peak,
               "rot_err_vs_truth_rad": synth.rotation_error_rad(r["transform"], c.T_star),
               "trans_err_vs_truth_m": synth.translation_error(r["transform"], c.T_star)}
        if e2e:
            te, (re_, fe), qe, _, _ = timed(c.h_tgt, c.h_src, steps, max(1, warmup))
            out["ms_per_job_e2e"] = 1e3 * sum(te) / len(te)
            out["corr_per_s_e2e"] = qe / sum(te)
        return out, r, f

    # ---- the headline: config 2 (x N, weak) ----------------------------------------------------------------------
    n = workload_points(world, args.points)
    main = Clouds(n)
    src, tgt, T_star, dims = main.src, main.tgt, main.T_star, main.dims
    d_src, d_tgt = main.d_src, main.d_tgt

    sampler = ClockSampler(local_rank)
    launches0 = eng.launch_count()
    if rank == 0:
        sampler.start()
    times, (res, fit), queries, ms_corr, n_corr_launch = timed(d_tgt, d_src, args.steps, args.warmup)
    launches = eng.launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res, fit)
    e_times, (e_res, e_fit), e_queries, _, _ = timed(main.h_tgt, main.h_src, args.steps, max(1, args.warmup // 2))
    clocks = sampler.stop() if rank == 0 else None

    # the same job from PAGEABLE host clouds in the reference's own layout (pcl::PointCloud<PointXYZRGB>: 32-byte rows):
    # what a caller of the C++ drop-in gets; the library gathers xyz through its pinned ring (csrc/upload.hpp)
    pageable = None
    if world == 1:
        def rows32(xyz):
            r = np.zeros((len(xyz), 8), np.float32)
            r[:, :3] = xyz
            r[:, 3] = 1.0
            return r
        p_tgt, p_src = rows32(tgt), rows32(src)
        for _ in range(2):
            step(eng, p_tgt, p_src)
        t_pg = []
        for _ in range(3):
            flush.zero_()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            step(eng, p_tgt, p_src)
            t_pg.append((time.perf_counter() - t0) * 1e3)
        pageable = {"ms_per_step": float(np.median(t_pg)), "host_bytes_per_step": int(p_tgt.nbytes + p_src.nbytes),
                    "h2d_bytes_per_step": int(12 * (len(tgt) + len(src))) if p_tgt.nbytes >= (8 << 20) else int(p_tgt.nbytes + p_src.nbytes),
                    "note": "wall clock around one job from pageable numpy arrays of 32-byte PointXYZRGB rows"}

    # per-phase view of one more (untimed) step, for the roofline objects
    flush.zero_()
    torch.cuda.synchronize()
    t0 = time.perf_counter(); eng.set_target(d_tgt); t_tgt = time.perf_counter() - t0
    t0 = time.perf_counter(); eng.set_source(d_src); t_src = time.perf_counter() - t0
    t0 = time.perf_counter(); eng.compute_covariances(); t_cov = time.perf_counter() - t0
    t0 = time.perf_counter(); pres = eng.align(); t_align = time.perf_counter() - t0
    t0 = time.perf_counter(); eng.fitness(pres["transform"]); t_fit = time.perf_counter() - t0
    T_fin = pres["transform"]
    ms_corr_k, _ = eng.bench_kernel(0, T_fin, iters=10)   # correspondence pass at the converged pose (no seeding)
    ms_nn_k, _ = eng.bench_kernel(2, T_fin, iters=10)     # NN-1 only
    ms_cost_k, _ = eng.bench_kernel(1, T_fin, iters=20)   # cost/gradient evaluation
    ms_first_k, _ = eng.bench_kernel(3, np.eye(4, dtype=np.float32), iters=5)  # first pass of a job (initial pose)
    ginfo = eng.grid_info(0)

    n_shard = n // world
    total = sum(times)
    value = queries / total
    e_total = sum(e_times)
    e2e_value = e_queries / e_total
    # Dominant kernel of the step by total time: the correspondence pass (near + far instance = one pass).
    # Algorithmic bytes per pass (SURVEY 8d): 96 B per source point of this rank + 16 B per target point.  Its mean
    # duration is measured live: CUDA events on the engine stream around every pass of the timed steps.
    kc = counters.get("kernels", {})
    corr_bytes = 96.0 * n_shard + 16.0 * n
    corr_ms_live = ms_corr / max(n_corr_launch, 1)
    achieved = corr_bytes / (corr_ms_live * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "correspondence pass: correspondence_kernel near + far instances (transform, "
                "exact NN-1, gate, Mahalanobis)", "achieved": achieved,
                "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": kc.get("correspondence_pass_first", {}).get("dram_bytes"),
                "traffic_capture": counters.get("_capture"), "peak_source": peak_src,
                "algorithmic_bytes_per_launch": corr_bytes, "ms_per_launch": corr_ms_live,
                "launches_timed": n_corr_launch,
                "note": "mean over all passes of the timed steps; DRAM traffic equals the algorithmic bytes, so the pass is "
                        "not HBM-bound: detail.issue_roofline gives the instruction-issue bound that does apply; traffic = "
                        "dram read+write of the first pass from the committed ncu capture named in traffic_capture"}
    cost_bytes = (56.0 if args.maha_fp32 else 80.0) * n_shard
    knn_bytes = 40.0 * (n + n_shard)

    def kern(ms, nbytes, key=None):
        return {"ms": ms, "algorithmic_bytes": nbytes, "GBps": nbytes / (ms * 1e-3) / 1e9,
                "frac_of_measured_hbm": nbytes / (ms * 1e-3) / 1e9 / peak, "ncu_dram_bytes": kc.get(key, {}).get("dram_bytes")}

    # Instruction-issue roofline of the search kernels: an SM issues at most 4 warp instructions per clock (one per
    # scheduler), i.e. 4 x 32 thread instructions when every lane is active.  thread_inst is ncu's
    # smsp__thread_inst_executed.sum for one launch of the kernel on this workload (committed capture); the bound is
    # the time those instructions need at full issue rate with full warps.  achieved = bound / measured time.
    sm_clock_hz = 1e6 * float((clocks or {}).get("sm_mhz") or 1965.0)
    issue_rate = 148 * 4 * 32 * sm_clock_hz

    def issue(key, ms, queries_):
        c = kc.get(key)
        if not c or not c.get("thread_inst"):
            return None
        ti = float(c["thread_inst"])
        return {"thread_inst_per_launch": ti, "thread_inst_per_query": ti / max(c.get("queries", queries_), 1),
                "avg_active_lanes": c.get("lanes"), "issue_active": c.get("issue_active"),
                "bound_ms_full_warps_full_issue": 1e3 * ti / issue_rate, "measured_ms": ms,
                "frac_of_issue_roofline": (1e3 * ti / issue_rate) / ms if ms else None}

    extra = {
        "phases_ms": {"index_target": 1e3 * t_tgt, "index_source": 1e3 * t_src, "covariances": 1e3 * t_cov,
                      "align": 1e3 * t_align, "fitness": 1e3 * t_fit, "align_corr_kernel_total": pres["ms_corr"],
                      "align_cost_evals_total": pres["ms_cost"], "cost_evaluations": pres["cost_evaluations"],
                      "outer_iterations": pres["outer_iterations"], "corr_far_queries": pres["corr_far_queries"]},
        "kernels": {
            "correspondence_pass_first_of_job": kern(ms_first_k, corr_bytes, "correspondence_pass_first"),
            "correspondence_pass_converged_pose_unseeded": kern(ms_corr_k, corr_bytes, "correspondence_pass_steady"),
            "nn1_only_converged_pose": kern(ms_nn_k, 24.0 * n_shard + 16.0 * n),
            "cost_eval": kern(ms_cost_k, cost_bytes, "cost_eval"),
            "knn_covariances_both_clouds": kern(1e3 * t_cov, knn_bytes, "knn_cov"),
            "grid_build_both_clouds": kern(1e3 * (t_tgt + t_src), 36.0 * 2 * n),
        },
        "issue_roofline": {
            "peak_thread_inst_per_s": issue_rate, "sm_clock_hz": sm_clock_hz, "capture": counters.get("_capture"),
            "correspondence_pass_first_of_job": issue("correspondence_pass_first", ms_first_k, n_shard),
            "correspondence_pass_converged_pose": issue("correspondence_pass_steady", ms_corr_k, n_shard),
            "knn_covariances_one_cloud": issue("knn_cov", 0.5 * 1e3 * t_cov, n),
            "note": "frac_of_issue_roofline = what the kernel reaches of the bound set by the instructions it executes; the "
                    "remaining factor is lanes idling in divergent loops (avg_active_lanes of 32) and issue slots lost to "
                    "latency (issue_active).  An exact search costs >= 14 non-fused float instructions per candidate "
                    "(FMA contraction would change FLANN's d2 bits), so the HBM roofline is out of reach by construction."},
        "grid": {"cell_size_m": ginfo["cell_size"], "dims": ginfo["dims"], "bricks": ginfo["n_bricks_occupied"],
                 "cells_occupied": ginfo["n_cells_occupied"],
                 "points_per_cell": ginfo["n_indexed"] / max(ginfo["n_cells_occupied"], 1)},
    }

    # ---- secondary measurements (not part of the timed steps above) ----------------------------------------------
    def dev_ms(fn, iters=3):
        best = None
        for _ in range(iters):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record(estream)
            out = fn()
            e1.record(estream)
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            best = ms if best is None else min(best, ms)
        return best, out

    if world == 1 and not args.quick:
        # the opt-in moments mode: same objective from 74 moments per outer iteration (include/gicp_b200.h cost_moments)
        if not args.cost_moments:
            eng.set_params(cost_moments=1)
            m_times, (m_res, m_fit), m_queries, _, _ = timed(d_tgt, d_src, max(2, args.steps // 2), 1)
            eng.set_params(cost_moments=0)
            extra["cost_moments_mode"] = {
                "ms_per_step": 1e3 * sum(m_times) / len(m_times), "value": m_queries / sum(m_times),
                "outer_iterations": m_res["outer_iterations"], "cost_evaluations_on_host": m_res["cost_evaluations"],
                "vs_default_rot_rad": synth.rotation_error_rad(m_res["transform"], res["transform"]),
                "vs_default_trans_m": synth.translation_error(m_res["transform"], res["transform"]),
                "note": "opt-in: exact instead of float-rounded T*p; PCL's line search amplifies the 1e-8 relative "
                        "difference, so the result agrees with the default to the stopping slack, not to the parity bar"}
        # SURVEY 8a row a13 and 8f rows 1, 3 on the same data: difference of the aligned scan (+ 20 FOD blobs) against
        # the CAD cloud, clusters of the difference cloud, voxel-grid downsample of the scan as PointXYZRGB rows
        aligned = synth.apply_rigid(T_star, src)
        with_fod, _ = synth.add_fod_blobs(aligned.astype(np.float32), n_blobs=20, seed=999, length=dims[0], width=dims[1])
        d_fod = torch.from_numpy(np.ascontiguousarray(with_fod, dtype=np.float32)).cuda()
        thr = 4e-3 * 0.1
        ms_diff, (mask, kept) = dev_ms(lambda: eng.cloud_difference(d_fod, d_tgt, thr))
        diff_cloud = d_fod[mask.bool()].contiguous()
        ms_clu, (labels, n_clu) = dev_ms(lambda: eng.euclidean_clusters(diff_cloud, thr * 100, 3, 0))
        rgb = torch.zeros((n, 8), dtype=torch.float32, device="cuda")
        rgb[:, :3] = d_src
        rgb[:, 3] = 1.0
        eng.set_target(d_src)
        leaf = 10.0 * eng.cloud_resolution(0)          # src/LeicaStateMachine.cpp:61-65: leaf_size_factor 10
        eng.set_target(d_tgt)
        ms_vox, vox = dev_ms(lambda: eng.voxel_grid(rgb, leaf))
        n_fod = int(d_fod.shape[0])
        # the node's input (src/node.cpp:37): a PointCloud2 payload as pcl::toROSMsg lays it out, gathered into rows
        msg = rgb.view(torch.uint8).reshape(-1)
        ms_pc2, _ = dev_ms(lambda: eng.pointcloud2_to_xyzrgb(msg, n, 1, 32, 32 * n, 0, 4, 8, 16, device_out=True))
        extra["pointcloud2_unpack"] = dict(kern(ms_pc2, 64.0 * n), points=n,
                                           includes="output allocation by torch + the gather kernel; 32 B in + 32 B out per point")
        extra["fod_pipeline"] = {
            "cloud_difference": dict(kern(ms_diff, 16.0 * n_fod + 16.0 * n + n_fod), points_in=n_fod, kept=int(kept),
                                     includes="index build of the subtract cloud + difference kernels"),
            "euclidean_clusters": {"ms": ms_clu, "points": int(diff_cloud.shape[0]), "clusters": int(n_clu),
                                   "includes": "index build, union-find kernels, labels to the host, host grouping"},
            "voxel_grid": dict(kern(ms_vox, 32.0 * n + 32.0 * int(vox.shape[0])), points_in=n, points_out=int(vox.shape[0]),
                               leaf_m=float(leaf), includes="min/max, keys, radix sort, heads/scan, centroids"),
        }
        del d_fod, rgb, msg

    # ---- parity, in the driver-run record ------------------------------------------------------------------------
    parity_ok = True

    def transform_gap(Ta, Tb, diag):
        rot, tr = synth.rotation_error_rad(Ta, Tb), synth.translation_error(Ta, Tb)
        return {"rot_rad": rot, "trans_m": tr, "trans_tol_m": TRANS_TOL_REL * diag, "rot_tol_rad": ROT_TOL,
                "bit_equal": bool(np.array_equal(np.asarray(Ta, np.float32), np.asarray(Tb, np.float32))),
                "ok": bool(rot <= ROT_TOL and tr <= TRANS_TOL_REL * diag)}

    cpu_baseline = None
    if not args.no_cpu_baseline:
        # the pair the oracle solves: the benchmark workload itself at N = 1; at N > 1 a 1 M / 1 M pair of the same
        # generator, solved by the SHARDED engine on all ranks (so N > 1 correctness is in this record, not in a log)
        nb = min(n, args.cpu_points)
        if nb == n:
            par, p_res, p_fit = main, res, fit
        else:
            par = Clouds(nb)
            p_res, p_fit = step(eng, par.h_tgt, par.h_src)
        if rank == 0:
            from oracle.oracle import Oracle, default_params
            orc = Oracle(fast=True)
            t0 = time.perf_counter()
            r = orc.align(par.src, par.tgt, default_params(max_corr_distance=GATE_M))
            o_fit = orc.fitness(par.src, par.tgt, r["T"])
            dt = time.perf_counter() - t0
            if world == 1:
                cpu_baseline = {"value": r["n_corr_queries"] / dt, "unit": "correspondences/s", "cores": orc.num_threads(),
                                "kind": "port", "seconds": dt,
                                "sample": (f"one whole job on {nb} src x {nb} tgt points of the same generator"
                                           + ("" if nb == n else f" (workload is {n})")),
                                "outer_iterations": r["outer_iterations"]}
            gap = transform_gap(p_res["transform"], r["T"], par.diag)
            fit_rel = abs(p_fit - o_fit) / max(abs(o_fit), 1e-300)
            gap.update({"points_per_cloud": nb, "gpus": world, "outer_gpu": p_res["outer_iterations"],
                        "outer_cpu": r["outer_iterations"], "fitness_gpu": p_fit, "fitness_cpu": o_fit,
                        "fitness_rel": fit_rel, "fitness_tol_rel": FIT_TOL_REL})
            gap["ok"] = bool(gap["ok"] and fit_rel <= FIT_TOL_REL and p_res["outer_iterations"] == r["outer_iterations"])
            extra["parity_vs_oracle"] = gap
            parity_ok = parity_ok and gap["ok"]
        if nb != n:
            del par

    if world > 1:
        # the benchmark workload once more, UNSHARDED, on rank 0's GPU (a second engine without a communicator)
        if rank == 0:
            solo = Engine(local_rank)
            solo.set_params(**job_params)
            s_res, s_fit = step(solo, d_tgt, d_src)
            solo.close()
            gap = transform_gap(res["transform"], s_res["transform"], main.diag)
            fit_rel = abs(fit - s_fit) / max(abs(s_fit), 1e-300)
            gap.update({"points_per_cloud": n, "gpus": world, "outer_sharded": res["outer_iterations"],
                        "outer_single": s_res["outer_iterations"], "evals_sharded": res["cost_evaluations"],
                        "evals_single": s_res["cost_evaluations"], "fitness_sharded": fit, "fitness_single": s_fit,
                        "fitness_rel": fit_rel, "pairs_sharded": res["corr_pairs_last"], "pairs_single": s_res["corr_pairs_last"]})
            gap["ok"] = bool(gap["ok"] and fit_rel <= FIT_TOL_REL and res["outer_iterations"] == s_res["outer_iterations"]
                             and res["corr_pairs_last"] == s_res["corr_pairs_last"])
            extra["parity_vs_single_gpu"] = gap
            parity_ok = parity_ok and gap["ok"]
        barrier()

    # ---- BASELINE configs 3 and 5 at this N (strong scaling: the source of ONE job is sharded over the N GPUs) -------------
    del main, d_src, d_tgt
    torch.cuda.empty_cache()
    if not args.quick:
        sweep = []
        for m in SWEEP_POINTS:
            if m > args.max_sweep_points:
                continue
            c = Clouds(m)
            big = m >= 3_000_000
            entry, c_res, c_fit = job_series(c, 2 if big else 3, 1 if big else 2, e2e=(m == CONFIG3_POINTS))
            sweep.append(entry)
            if m == CONFIG3_POINTS:
                extra["config3"] = dict(entry, gpus=world, scaling="strong",
                                        what="BASELINE config 3: 10 M-point scan vs 10 M-point CAD cloud, one job sharded "
                                             "over the run's GPUs; e2e = from pinned host clouds, copies inside the timed region",
                                        under_1s_end_to_end=bool(entry["ms_per_job_e2e"] < 1000.0))
            del c
            torch.cuda.empty_cache()
        extra["sweep"] = {"gpus": world, "scaling": "strong", "what": "BASELINE config 5: one job per size on the run's GPUs, "
                          "clouds resident; corr_pass_frac_of_hbm = (96 B x shard + 16 B x target) / mean pass time / measured HBM peak",
                          "rows": sweep}

    if rank == 0:
        # sharded uploads (csrc/engine.cu do_prefetch): every rank uploads its 1 / world of the rows of both clouds and the
        # slices are exchanged between the GPUs, so the whole job moves each cloud over PCIe once
        shard_up = world > 1 and os.environ.get("GICPB_SHARD_UPLOAD", "1") != "0"
        h2d = int(src.nbytes + tgt.nbytes) * (1 if (world == 1 or shard_up) else world)
        line = {
            "metric": "gicp_correspondences_per_s", "value": value, "unit": "correspondences/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 search / f64 accumulate", "data": "synthetic",
            "config": {"workload": workload_name(n, world),
                       "points_source": n, "points_target": n, "sharding": f"source/{world}, target replicated",
                       "l2": "256 MiB flush write between timed steps", "timing": "CUDA events on the engine's stream around "
                       "each step, barrier + synchronize on both sides, max over ranks; kernels by CUDA events on the same stream",
                       "mahalanobis": "fp32" if args.maha_fp32 else "fp64",
                       "objective": "74 moments per outer iteration (cost_moments=1)" if args.cost_moments else
                                    "one cost-kernel pass per evaluation (PCL's float T*p arithmetic)",
                       "cross_gpu_sum": ("fused into the cost kernel over NVLink peer memory" if fused_peer else
                                         "ncclAllReduce per evaluation") if world > 1 else "none (one GPU)",
                       "outer_iterations": res["outer_iterations"], "cost_evaluations": res["cost_evaluations"]},
            "align_ms": res["ms_total"], "fitness": fit,
            "e2e": {"value": e2e_value, "unit": "correspondences/s", "ms_per_step": 1e3 * e_total / len(e_times),
                    "h2d_bytes_per_step": h2d, "h2d_bytes_per_rank": h2d // world if (world == 1 or shard_up) else h2d // world,
                    "d2h_bytes_per_step": 16 * 4 + 8 + 14 * 8 * int(e_res["cost_evaluations"])},
            "gpu_launches": int(launches),
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
            "clocks": clocks,
            "e2e_pageable_xyzrgb": pageable,
            "parity_ok": bool(parity_ok),
            "detail": extra,
        }
        emit(line)
    eng.close()
    ok_all = parity_ok
    if dist is not None:
        flag = torch.tensor([1.0 if parity_ok else 0.0], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        ok_all = bool(flag.item() > 0.5)
        dist.destroy_process_group()
    if not ok_all:
        sys.stderr.write("bench.py: PARITY FAILED (see parity_vs_oracle / parity_vs_single_gpu in the JSON line)\n")
        sys.exit(3)


def dump_outputs(out_dir, res, fit):
    """What the caller of the timed step receives from its last run, one .npy per value, so that two builds can be
    compared output for output on the same seeded clouds.  The timings in the result are left out: they differ from
    run to run."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"transform": np.asarray(res["transform"], np.float32), "fitness": np.float64(fit)}
    for key in ("converged", "outer_iterations", "inner_iterations", "cost_evaluations", "corr_queries",
                "corr_pairs_last"):
        arrays[key] = np.float64(res[key])
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


_JSON_FD = None


def emit(line):
    """The ONE JSON line goes to the process's real stdout; everything else this process or its libraries print
    (NCCL's version banner, torchrun notes) has been sent to stderr by main()."""
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)  # fd 1 now points at stderr: stdout carries nothing but the JSON line
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--points", type=int, default=0, help="points per cloud (default 1M x gpus)")
    ap.add_argument("--cpu-points", type=int, default=1_000_000, help="cpu_baseline / oracle parity sample size")
    ap.add_argument("--ref-points", type=int, default=2_000_000, help="--impl reference sample cap")
    ap.add_argument("--maha-fp32", type=int, default=0)
    ap.add_argument("--cost-moments", type=int, default=0, help="1: the opt-in moments objective (see gicp_b200.h)")
    ap.add_argument("--seed-previous", type=int, default=1, help="0: do not seed a pass with the previous pass's matches")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the oracle leg (cpu_baseline and parity_vs_oracle)")
    ap.add_argument("--quick", action="store_true", help="headline + parity only: no config 3 / sweep / FOD rows")
    ap.add_argument("--max-sweep-points", type=int, default=CONFIG3_POINTS)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's transform, fitness and iteration counts as "
                         "DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of this repo's engine (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
