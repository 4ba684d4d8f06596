"""GPU parity tests: the CUDA path, called through the C ABI (ctypes), against the CPU oracle on identical inputs.

Acceptance bars (BASELINE.json north_star): NN / kNN index sets bit-exact (ties -> lowest index); final transform
within 1e-4 rad and 1e-5 x bounding-box diagonal of the oracle's; fitness within 1e-4 relative; difference masks
bit-exact.
"""
import numpy as np
import pytest

from leica_point_cloud_processing_b200 import synth

pytestmark = pytest.mark.gpu

ROT_TOL = 1e-4          # rad
TRANS_TOL_REL = 1e-5    # x bounding-box diagonal
FIT_TOL_REL = 1e-4


def reset(engine, **kw):
    base = dict(max_iterations=100, transformation_epsilon=4e-3, rotation_epsilon=2e-3, max_corr_distance=4e-2,
                k_correspondences=20, gicp_epsilon=1e-3, max_inner_iterations=20, cell_size=0.0, points_per_cell=3.0,
                mahalanobis_fp32=0, use_previous_match=1, cost_moments=0, cost_persistent=1)
    base.update(kw)
    engine.set_params(**base)


def bbox_diag(*clouds):
    allp = np.concatenate([c[:, :3] for c in clouds])
    return float(np.linalg.norm(allp.max(0) - allp.min(0)))


def assert_transform_close(T_gpu, T_ref, diag):
    rot = synth.rotation_error_rad(T_gpu, T_ref)
    tr = synth.translation_error(T_gpu, T_ref)
    assert rot <= ROT_TOL, f"rotation differs by {rot} rad"
    assert tr <= TRANS_TOL_REL * diag, f"translation differs by {tr} m (diag {diag})"


# ---- NN-1 -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cell_size", [0.0, 0.05, 0.31, 1.7])
def test_nn1_cube_bit_exact(engine, oracle, cube_pair, cell_size):
    src, tgt, _ = cube_pair
    reset(engine, cell_size=cell_size)
    engine.set_target(tgt)
    idx, d2 = engine.nn1(src)
    oi, od = oracle.nn1(tgt, src)
    assert np.array_equal(idx, oi)
    assert np.array_equal(d2, od)
    # gated (reference default gate 0.04 m): 1473 of 5000 source points have a neighbour (SURVEY section 4)
    gi, gd = engine.nn1(src, max_dist=0.04)
    inside = od < np.float32(0.04) ** 2
    assert int(inside.sum()) == 1473
    assert np.array_equal(gi, np.where(inside, oi, -1))
    assert np.array_equal(gd[inside], od[inside])


def test_nn1_under_transform(engine, oracle, cube_pair):
    src, tgt, _ = cube_pair
    reset(engine)
    engine.set_target(tgt)
    T = oracle.apply_state([0.03, -0.02, 0.05, 0.02, -0.04, 0.1])
    idx, d2 = engine.nn1(src, T=T)
    oi, od = oracle.nn1(tgt, oracle.transform(T, src))
    assert np.array_equal(idx, oi)
    assert np.array_equal(d2, od)


@pytest.mark.parametrize("seed,cell_size", [(0, 0.0), (1, 0.02), (2, 0.4)])
def test_nn1_volume_and_far_queries(engine, oracle, seed, cell_size):
    rng = np.random.default_rng(seed)
    tgt = rng.random((20000, 3)).astype(np.float32)
    tgt[:2000] *= 0.05  # a dense clump
    q_in = rng.random((3000, 3)).astype(np.float32)
    q_far = (rng.random((600, 3)).astype(np.float32) - 0.5) * 30.0  # far outside the bounding box
    q_dup = tgt[rng.integers(0, len(tgt), 400)]                     # exact hits
    qry = np.concatenate([q_in, q_far, q_dup])
    reset(engine, cell_size=cell_size)
    engine.set_target(tgt)
    idx, d2 = engine.nn1(qry)
    oi, od = oracle.nn1(tgt, qry, use_tree=False)
    assert np.array_equal(idx, oi)
    assert np.array_equal(d2, od)


def test_nn1_ties_duplicates_and_nan(engine, oracle):
    rng = np.random.default_rng(5)
    base = rng.random((500, 3)).astype(np.float32)
    tgt = np.concatenate([base, base, base[:100]])  # every point duplicated: ties must resolve to the lowest index
    tgt[7] = np.nan                                  # non-finite target points are not indexed
    tgt[900, 1] = np.inf
    lattice = np.stack(np.meshgrid(*[np.arange(6, dtype=np.float32)] * 3, indexing="ij"), -1).reshape(-1, 3)
    tgt = np.concatenate([tgt, lattice])             # exact equidistant ties at lattice cell centres
    qry = np.concatenate([base[:200], lattice + 0.5, np.array([[np.nan, 0, 0]], np.float32)])
    reset(engine)
    engine.set_target(tgt)
    idx, d2 = engine.nn1(qry)
    oi, od = oracle.nn1(tgt, qry, use_tree=False)
    assert np.array_equal(idx, oi)
    assert np.array_equal(d2, od)
    assert idx[-1] == -1


# ---- kNN + covariances ------------------------------------------------------------------------------------
@pytest.mark.parametrize("cell_size", [0.0, 0.08, 0.9])
def test_knn_cube_bit_exact(engine, oracle, cube_pair, cell_size):
    src, tgt, _ = cube_pair
    reset(engine, cell_size=cell_size)
    engine.set_target(tgt)
    engine.set_source(src)
    for which, cloud in ((0, tgt), (1, src)):
        idx, d2 = engine.knn(which)
        oi, od = oracle.knn(cloud, 20)
        assert np.array_equal(idx, oi)
        assert np.array_equal(d2, od)


def test_knn_small_k_and_sparse_cloud(engine, oracle):
    rng = np.random.default_rng(11)
    cloud = np.concatenate([rng.random((3000, 3)) * 0.2, rng.random((300, 3)) * 25.0]).astype(np.float32)
    reset(engine, k_correspondences=7)
    engine.set_target(cloud)
    engine.set_source(cloud[:50])
    idx, d2 = engine.knn(0)
    oi, od = oracle.knn(cloud, 7)
    assert np.array_equal(idx, oi)
    assert np.array_equal(d2, od)
    reset(engine)


def test_covariances_match_oracle(engine, oracle, cube_pair):
    """Every point, no outlier allowance: the kernel's Jacobi eigen-solve and the oracle's SVD work on the same matrix
    (the kNN sets are bit-identical), so their regularised covariances may differ by at most what the conditioning of
    the smallest singular direction allows (tests/_cov_util.py normal_error_bound, also checked against numpy's SVD)."""
    from _cov_util import normal_error_bound, raw_covariances, regularised_from_svd
    src, tgt, _ = cube_pair
    panel = synth.panel_points(30000, 3, noise_sigma=5e-4)
    reset(engine)
    for tcloud, scloud in ((tgt, src), (panel, src)):
        engine.set_target(tcloud)
        engine.set_source(scloud)
        for which, cloud in ((0, tcloud), (1, scloud)):
            cov = engine.covariances(which)
            ref = oracle.covariances(cloud)
            w = np.linalg.eigvalsh(cov)
            assert np.allclose(w[:, 0], 1e-3, atol=1e-12) and np.allclose(w[:, 1:], 1.0, atol=1e-12)
            ki, _ = oracle.knn(cloud, 20)
            np_ref, sv = regularised_from_svd(raw_covariances(cloud, ki), 1e-3)
            bound = normal_error_bound(sv)
            err = np.abs(cov - ref).max(axis=(1, 2))
            assert (err <= 2.0 * bound).all(), float((err / bound).max())
            assert (np.abs(cov - np_ref).max(axis=(1, 2)) <= 2.0 * bound).all()
            well = (sv[:, 1] - sv[:, 2]) > 1e-3 * sv[:, 0]
            assert err[well].max() < 1e-9


# ---- correspondences, Mahalanobis, cost ------------------------------------------------------------------
def test_correspondences_and_cost(engine, oracle, cube_pair):
    src, tgt, _ = cube_pair
    reset(engine, max_corr_distance=5.0)
    engine.set_target(tgt)
    engine.set_source(src)
    cov_s, cov_t = engine.covariances(1), engine.covariances(0)
    T = oracle.apply_state([0.01, 0.02, -0.01, 0.01, 0.02, 0.05])
    pairs, idx, d2, maha = engine.correspondences(T)
    cnt, oi, od, omaha = oracle.correspondences(src, tgt, cov_s, cov_t, T, 5.0)
    assert pairs == cnt == 5000
    assert np.array_equal(idx, oi)
    assert np.array_equal(d2, od)
    assert np.allclose(maha, omaha, rtol=1e-9, atol=1e-9)
    x = np.array([0.012, 0.018, -0.008, 0.012, 0.018, 0.055])
    f, g = engine.cost(x)
    valid = np.nonzero(oi >= 0)[0].astype(np.int32)
    fo, go = oracle.cost(src, tgt, valid, oi[valid], omaha, x)
    assert abs(f - fo) <= 1e-10 * abs(fo)
    assert np.allclose(g, go, rtol=1e-9, atol=1e-12)
    # the same evaluations from the 74 second-order moments taken around T (no pass over the pairs): identical
    # up to the float rounding of T*p that PCL's functor carries (1e-7 relative per residual, averaged over pairs)
    reset(engine, max_corr_distance=5.0, cost_moments=1)
    engine.correspondences(T)
    for xx in (x, np.array([0.01, 0.02, -0.01, 0.01, 0.02, 0.05]), np.array([0.05, -0.03, 0.02, -0.04, 0.03, 0.12])):
        fm, gm = engine.cost(xx)
        fo, go = oracle.cost(src, tgt, valid, oi[valid], omaha, xx)
        assert abs(fm - fo) <= 2e-6 * abs(fo)
        assert np.allclose(gm, go, rtol=0, atol=2e-6 * np.abs(go).max())
    # at the expansion point itself (identity: the state reproduces the matrix exactly) the two modes agree to the last bits
    x0 = np.zeros(6)
    engine.correspondences(np.eye(4, dtype=np.float32))
    fm, gm = engine.cost(x0)
    reset(engine, max_corr_distance=5.0)
    engine.correspondences(np.eye(4, dtype=np.float32))
    fk, gk = engine.cost(x0)
    assert abs(fm - fk) <= 1e-13 * abs(fk) and np.allclose(gm, gk, rtol=0, atol=1e-12 * np.abs(gk).max())
    # gated: the reference's default 0.04 m
    reset(engine, max_corr_distance=0.04)
    pairs, idx, d2, maha = engine.correspondences(np.eye(4, dtype=np.float32))
    cnt, oi, od, omaha = oracle.correspondences(src, tgt, cov_s, cov_t, np.eye(4), 0.04)
    assert pairs == cnt == 1473
    assert np.array_equal(idx, oi)


# ---- whole alignment -------------------------------------------------------------------------------------
@pytest.mark.parametrize("params", [
    dict(),                                                         # reference defaults (gate 0.04, tf_eps 4e-3)
    dict(max_corr_distance=5.0, transformation_epsilon=5e-4),       # test_gicp_alignment.cpp testRun
    dict(max_corr_distance=5.0, transformation_epsilon=5e-4, use_previous_match=0),
])
def test_align_cube_matches_oracle(engine, oracle, cube_pair, params):
    from oracle.oracle import default_params
    src, tgt, T_true = cube_pair
    reset(engine, **params)
    engine.set_target(tgt)
    engine.set_source(src)
    res = engine.align()
    op = {k: v for k, v in params.items() if k in ("max_corr_distance", "transformation_epsilon")}
    ref = oracle.align(src, tgt, default_params(**op))
    assert res["converged"] == ref["converged"] == 1
    diag = bbox_diag(src, tgt)
    assert_transform_close(res["transform"], ref["T"], diag)
    assert res["outer_iterations"] == ref["outer_iterations"]
    assert synth.rotation_error_rad(res["transform"], T_true) < 2e-3
    fit = engine.fitness(res["transform"])
    fit_ref = oracle.fitness(src, tgt, ref["T"])
    fit_same_T = oracle.fitness(src, tgt, res["transform"])
    assert abs(fit - fit_same_T) <= 1e-9 * max(fit_same_T, 1e-30)  # the kernel itself
    assert abs(fit - fit_ref) <= FIT_TOL_REL * fit_ref + 1e-12      # end to end, incl. the transform difference


def test_align_panel_100k_matches_oracle(engine, oracle):
    from oracle.oracle import default_params
    src, tgt, T_star = synth.make_pair(100_000, 100_000)
    reset(engine, max_corr_distance=1.0)
    engine.set_target(tgt)
    engine.set_source(src)
    res = engine.align()
    ref = oracle.align(src, tgt, default_params(max_corr_distance=1.0))
    assert res["converged"] == ref["converged"] == 1
    diag = bbox_diag(src, tgt)
    assert_transform_close(res["transform"], ref["T"], diag)
    # and the known answer, within what 1 mm noise allows
    assert synth.rotation_error_rad(res["transform"], T_star) < 2e-3
    assert synth.translation_error(res["transform"], T_star) < 5e-3
    fit = engine.fitness(res["transform"])
    fit_ref = oracle.fitness(src, tgt, ref["T"])
    assert abs(fit - fit_ref) <= FIT_TOL_REL * fit_ref


@pytest.mark.parametrize("n,fp32", [(5000, 0), (3001, 1), (120_000, 0), (400_001, 1), (400_001, 0)])
def test_resident_cost_kernel_is_bit_identical(engine, n, fp32):
    """cost_persistent=1 (one resident kernel per inner solve, commands through mapped memory, a part of the pairs parked
    in shared memory) against cost_persistent=0 (one launch per evaluation): the same terms summed in another order, which
    the float32 transforms absorb, so the trajectory and the final transform are bit-identical - for pair counts below, at
    and above what the
    resident blocks hold, odd counts, and both Mahalanobis widths."""
    src, tgt, _ = synth.make_pair(n, n)
    out = {}
    for mode in (0, 1):
        reset(engine, max_corr_distance=1.0, cost_persistent=mode, mahalanobis_fp32=fp32)
        engine.set_clouds(tgt, src)
        res = engine.align()
        out[mode] = res
        x = np.array([0.01, -0.02, 0.015, 0.02, -0.01, 0.03])
        f, g = engine.cost(x)            # the single-evaluation hook (always one launch) on the final pairs
        out[mode, "fg"] = (f, g)
    assert out[0]["converged"] == 1
    assert np.array_equal(out[0]["transform"], out[1]["transform"])
    assert out[0]["cost_evaluations"] == out[1]["cost_evaluations"]
    assert out[0]["outer_iterations"] == out[1]["outer_iterations"]
    assert out[0, "fg"][0] == out[1, "fg"][0] and np.array_equal(out[0, "fg"][1], out[1, "fg"][1])
    # the resident session's own evaluations against the per-launch kernel at the same x
    T = out[1]["transform"]
    ms_res, _ = engine.bench_kernel(4, T, iters=5)
    ms_one, _ = engine.bench_kernel(5, T, iters=5)
    assert ms_res > 0 and ms_one > 0
    reset(engine)


def test_resident_cost_kernel_survives_an_idle_host(engine):
    """The resident kernel ends itself when no command arrives for GICPB_COST_IDLE_MS; an evaluation that finds it gone
    launches it again.  With the host stalled longer than that before EVERY command (test knob) each evaluation takes the
    relaunch path, and the result is still bit-identical."""
    import os
    from leica_point_cloud_processing_b200 import Engine
    src, tgt, _ = synth.make_pair(50_000, 50_000)
    reset(engine, max_corr_distance=1.0, max_iterations=2)
    engine.set_clouds(tgt, src)
    ref = engine.align()
    os.environ["GICPB_COST_IDLE_MS"] = "2"
    os.environ["GICPB_COST_TEST_STALL_MS"] = "8"
    try:
        e = Engine(0)
    finally:
        del os.environ["GICPB_COST_IDLE_MS"], os.environ["GICPB_COST_TEST_STALL_MS"]
    e.set_params(max_corr_distance=1.0, max_iterations=2, points_per_cell=3.0)
    e.set_clouds(tgt, src)
    launches0 = e.launch_count()
    r = e.align()
    relaunched = e.launch_count() - launches0
    e.close()
    assert np.array_equal(r["transform"], ref["transform"]) and r["cost_evaluations"] == ref["cost_evaluations"]
    assert relaunched >= r["cost_evaluations"]   # (nearly) one launch of the resident kernel per evaluation
    reset(engine)


def test_align_cost_moments_mode(engine, oracle):
    """cost_moments=1 evaluates the same objective from 74 moments per outer iteration, with exact instead of
    float-rounded T*p.  PCL's line search compares objective values that differ by less than that rounding, so the
    BFGS path is not reproduced step for step: the result agrees with the PCL-faithful default to the slack the
    reference's stopping rule (tf_eps 4e-3, 20 inner steps) leaves, not to the 1e-4 rad parity bar."""
    from oracle.oracle import default_params
    src, tgt, T_star = synth.make_pair(100_000, 100_000)
    reset(engine, max_corr_distance=1.0, cost_moments=1)
    engine.set_target(tgt)
    engine.set_source(src)
    res = engine.align()
    ref = oracle.align(src, tgt, default_params(max_corr_distance=1.0))
    assert res["converged"] == 1
    assert synth.rotation_error_rad(res["transform"], ref["T"]) < 5e-4
    assert synth.translation_error(res["transform"], ref["T"]) < 5e-4
    # as good a registration as the faithful path: same distance to the known answer, same fitness
    assert synth.rotation_error_rad(res["transform"], T_star) < 2e-3
    assert synth.translation_error(res["transform"], T_star) < 5e-3
    assert abs(engine.fitness(res["transform"]) - oracle.fitness(src, tgt, ref["T"])) <= 1e-2 * oracle.fitness(src, tgt, ref["T"])


def test_align_fp32_mahalanobis_within_tolerance(engine, oracle, cube_pair):
    from oracle.oracle import default_params
    src, tgt, _ = cube_pair
    reset(engine, max_corr_distance=5.0, mahalanobis_fp32=1)
    engine.set_target(tgt)
    engine.set_source(src)
    res = engine.align()
    ref = oracle.align(src, tgt, default_params(max_corr_distance=5.0))
    assert_transform_close(res["transform"], ref["T"], bbox_diag(src, tgt))


def test_prefetched_uploads_give_the_same_result(engine, oracle, cube_pair):
    """gicpb_prefetch_cloud only moves the upload to a copy stream: same index, same transform; a prefetch that the
    following set call does not match (another array) is ignored."""
    src, tgt, _ = cube_pair
    reset(engine, max_corr_distance=5.0, transformation_epsilon=5e-4)
    engine.set_target(tgt)
    engine.set_source(src)
    plain = engine.align()
    engine.prefetch(0, tgt)
    engine.prefetch(1, src)
    engine.set_target(tgt)
    engine.set_source(src)
    pre = engine.align()
    assert np.array_equal(plain["transform"], pre["transform"])
    engine.prefetch(1, tgt)                 # stale hint: a different cloud is then set as the source
    other = src.copy()
    engine.set_source(other)
    engine.set_target(tgt)
    again = engine.align()
    assert np.array_equal(plain["transform"], again["transform"])
    idx, d2 = engine.nn1(src)
    oi, od = oracle.nn1(tgt, src)
    assert np.array_equal(idx, oi) and np.array_equal(d2, od)


def test_set_clouds_equals_the_separate_calls(engine, oracle, cube_pair):
    """gicpb_set_clouds = set_target + set_source + compute_covariances with the target's covariance pass on a second
    stream beside the source's index build: covariances bit-identical, same transform and fitness; host, prefetched host
    and device clouds; a cloud smaller than k leaves the error to align, as before."""
    import torch
    from leica_point_cloud_processing_b200 import synth
    src, tgt, _ = cube_pair
    big_s, big_t, _ = synth.make_pair(60_000, 80_000)
    for s_, t_, gate in ((src, tgt, 5.0), (big_s, big_t, 1.0)):
        reset(engine, max_corr_distance=gate, transformation_epsilon=5e-4)
        engine.set_target(t_)
        engine.set_source(s_)
        engine.compute_covariances()
        c0t, c0s = engine.covariances(0), engine.covariances(1)
        plain = engine.align()
        f0 = engine.fitness(plain["transform"])
        for mode in ("host", "prefetched", "device"):
            if mode == "prefetched":
                engine.prefetch(0, t_)
                engine.prefetch(1, s_)
            a, b = (torch.from_numpy(t_).cuda(), torch.from_numpy(s_).cuda()) if mode == "device" else (t_, s_)
            engine.set_clouds(a, b)
            assert np.array_equal(engine.covariances(0), c0t) and np.array_equal(engine.covariances(1), c0s), mode
            both = engine.align()
            assert np.array_equal(plain["transform"], both["transform"]), mode
            assert both["outer_iterations"] == plain["outer_iterations"]
            assert engine.fitness(both["transform"]) == f0
    idx, d2 = engine.nn1(big_s)
    oi, od = oracle.nn1(big_t, big_s)
    assert np.array_equal(idx, oi) and np.array_equal(d2, od)
    # fewer points than k_correspondences in either cloud: set_clouds succeeds, align reports -7 (PCL: error + return)
    reset(engine, max_corr_distance=5.0)
    engine.set_clouds(tgt[:10], src)
    assert engine.align(raise_on_failure=False)["rc"] == -7
    engine.set_clouds(tgt, src[:10])
    assert engine.align(raise_on_failure=False)["rc"] == -7
    engine.set_clouds(tgt, src)
    assert engine.align()["converged"] == 1
    with pytest.raises(Exception):
        engine.set_clouds(tgt, src[:0])


def test_pageable_host_clouds_take_the_staged_upload(engine, oracle):
    """Large pageable host clouds (pcl::PointCloud memory: 32-byte rows) are gathered into packed xyz rows through a ring
    of pinned chunks (csrc/upload.hpp) instead of one pageable cudaMemcpy: same index, same answers as device clouds,
    for set_clouds (with and without prefetch), set_target / set_source, the difference input and NN-1 queries."""
    import torch
    from leica_point_cloud_processing_b200 import synth
    n = 700_000                                   # 22 MB per cloud at 32 bytes per point: three 8 MB chunks
    src3, tgt3, _ = synth.make_pair(n, n)
    def rows32(xyz):
        r = np.full((len(xyz), 8), 7.5, np.float32)  # the other 20 bytes must not matter
        r[:, :3] = xyz
        return r
    src, tgt = rows32(src3), rows32(tgt3)
    reset(engine, max_corr_distance=1.0, points_per_cell=6.0)
    engine.set_clouds(torch.from_numpy(tgt3).cuda(), torch.from_numpy(src3).cuda())
    ref = engine.align()
    qi, qd = engine.nn1(torch.from_numpy(src3).cuda())
    for mode in ("set_clouds", "prefetched", "separate"):
        if mode == "prefetched":
            engine.prefetch(0, tgt)
            engine.prefetch(1, src)
        if mode == "separate":
            engine.set_target(tgt)
            engine.set_source(src)
        else:
            engine.set_clouds(tgt, src)
        res = engine.align()
        assert np.array_equal(res["transform"], ref["transform"]), mode
        assert res["cost_evaluations"] == ref["cost_evaluations"]
    i2, d2 = engine.nn1(src)                      # staged query upload, stride 32 -> 12
    assert np.array_equal(i2, qi) and np.array_equal(d2, qd)
    m_dev, k_dev = engine.cloud_difference(torch.from_numpy(src3).cuda(), torch.from_numpy(tgt3).cuda(), 4e-4)
    m_host, k_host = engine.cloud_difference(src, tgt, 4e-4)
    assert k_host == k_dev and np.array_equal(m_host, m_dev.cpu().numpy())
    # whole rows through the same ring: transform (all 32 bytes travel) and the PointCloud2 gather
    moved = engine.transform_cloud(ref["transform"], src)
    moved_dev = engine.transform_cloud(ref["transform"], torch.from_numpy(src).cuda())
    assert np.array_equal(moved, moved_dev.cpu().numpy()) and np.all(moved[:, 4:] == 7.5)
    rows = engine.pointcloud2_to_xyzrgb(src, n, 1, 32, 32 * n, 0, 4, 8, 16)
    assert np.array_equal(rows[:, :3], src3) and np.all(rows[:, 3] == 1) and np.all(rows[:, 4] == 7.5)


def test_align_not_enough_correspondences(engine, cube_pair):
    src, tgt, _ = cube_pair
    reset(engine, max_corr_distance=1e-4)
    engine.set_target(tgt + np.float32(50.0))
    engine.set_source(src)
    res = engine.align(raise_on_failure=False)
    assert res["converged"] == 0 and res["rc"] == -4
    assert np.array_equal(res["transform"], np.eye(4, dtype=np.float32))


# ---- transform, difference ----------------------------------------------------------------------------------
@pytest.mark.parametrize("cols", [3, 4, 8])
def test_transform_cloud_bit_exact(engine, oracle, cube_pair, cols):
    src, _, _ = cube_pair
    T = oracle.apply_state([0.3, -0.2, 0.1, 0.2, -0.1, 0.4])
    cloud = np.zeros((len(src), cols), np.float32)
    cloud[:, :3] = src
    if cols > 3:
        cloud[:, 3:] = np.arange(cols - 3, dtype=np.float32) + 7.0
    out = engine.transform_cloud(T, cloud)
    assert np.array_equal(out[:, :3], oracle.transform(T, src))
    assert np.array_equal(out[:, 3:], cloud[:, 3:])
    assert np.array_equal(cloud[:, :3], src)  # input untouched


@pytest.mark.parametrize("thr", [4e-4, 4e-3 * 3, 0.0, 1.0])
def test_difference_mask_bit_exact(engine, oracle, cube_pair, thr):
    src, tgt, _ = cube_pair
    rng = np.random.default_rng(3)
    inp = np.concatenate([tgt + rng.normal(0, 0.01, tgt.shape).astype(np.float32),
                          (rng.random((500, 3)).astype(np.float32) - 0.5) * 6.0,
                          tgt[:50]])
    inp[11] = np.nan
    reset(engine)
    mask, kept = engine.cloud_difference(inp, tgt, thr)
    om, ok = oracle.difference(inp, tgt, thr)
    assert np.array_equal(mask, om)
    assert kept == ok


def test_difference_reference_fixture(engine, oracle):
    """reference test/test_filter.cpp:102-113: removeFromCloud(cube + 2, cube, resolution) keeps > 1 point."""
    from leica_point_cloud_processing_b200 import remove_from_cloud
    rng = np.random.default_rng(0)
    cube = rng.random((5000, 3)).astype(np.float32) * 1024.0 / 1024.0
    moved = cube + np.float32(2.0)
    res = oracle.resolution(cube)
    out, mask = remove_from_cloud(moved, cube, res, engine=engine)
    assert len(out) > 1
    om, _ = oracle.difference(moved, cube, res)
    assert np.array_equal(mask, om)


def test_difference_fod_blobs(engine, oracle):
    src, tgt, T_star = synth.make_pair(60_000, 60_000)
    aligned = synth.apply_rigid(T_star, src)
    with_fod, is_fod = synth.add_fod_blobs(aligned, n_blobs=6)
    reset(engine)
    for thr in (4e-3 * 0.1, 4e-3 * 3):
        mask, kept = engine.cloud_difference(with_fod, tgt, thr)
        om, ok = oracle.difference(with_fod, tgt, thr)
        assert np.array_equal(mask, om)
        assert kept == ok


# ---- the reference's own tests, re-expressed against the mirrored class --------------------------------------
def test_reference_testApplyTF(cube_pair):
    """reference test/test_gicp_alignment.cpp:50-75"""
    from leica_point_cloud_processing_b200 import GICPAlignment
    src, tgt, _ = cube_pair
    g = GICPAlignment(tgt, src, False)
    assert np.array_equal(g.getFineTransform(), np.eye(4, dtype=np.float32))
    g.run()
    g.applyTFtoCloud(src)
    aligned = g.getAlignedCloud()
    assert g.transform_exists_
    # what the reference test meant to check: after alignment the source lies on the target
    assert np.abs(aligned - tgt).max() <= 1e-2


def test_reference_testRun(cube_pair, oracle):
    """reference test/test_gicp_alignment.cpp:77-104"""
    from leica_point_cloud_processing_b200 import GICPAlignment
    src, tgt, T_true = cube_pair
    g = GICPAlignment(tgt, src, False)
    assert np.array_equal(g.getFineTransform(), np.eye(4, dtype=np.float32))
    g.setMaxIterations(100)
    g.setMaxCorrespondenceDistance(5)
    g.setRANSACOutlierTh(5e-2)
    g.setTfEpsilon(5e-4)
    assert g.ransac_outlier_th_ == 0.0  # int-typed setter truncates, as upstream
    g.run()
    aligned = g.getAlignedCloud()
    assert g.transform_exists_
    assert aligned.shape == src.shape
    assert synth.rotation_error_rad(g.getFineTransform(), T_true) < 1e-3
    assert np.abs(aligned - tgt).max() <= 1e-3


def test_reference_testRunWithCov(cube_pair):
    """reference test/test_gicp_alignment.cpp:106-131"""
    from leica_point_cloud_processing_b200 import GICPAlignment
    src, tgt, _ = cube_pair
    g = GICPAlignment(tgt, src, True)
    assert np.array_equal(g.getFineTransform(), np.eye(4, dtype=np.float32))
    g.run()
    g.getAlignedCloud()
    assert g.transform_exists_
    T1 = g.getFineTransform()
    g.iterate()
    assert g.transform_exists_
    # iterate() re-solves from the original source and left-multiplies the same transform (SURVEY App. A.6)
    assert np.allclose(g.getFineTransform(), T1 @ T1, atol=1e-6)
    # PCL's align() overwrote the cloud with T_new * source; undo() restores the pre-iterate copy (reference :139-142)
    g.aligned_cloud_ = g.aligned_cloud_ + np.float32(1.0)
    g.undo()
    assert np.array_equal(g.getAlignedCloud(), g.backup_cloud_)
    assert np.allclose(g.getFineTransform(), T1 @ T1, atol=1e-6)  # fine_tf_ is NOT rolled back, as upstream


@pytest.mark.parametrize("which", ["cube", "panel", "panel_far_from_origin"])
def test_normals_match_oracle(engine, oracle, cube_pair, which):
    """Utils::getNormals (reference src/Utils.cpp:27-44; SURVEY 8f row 2): the NaN pattern is bit-exact; the float moments
    are added in PCL's order with PCL's roundings, so the normal vectors and curvatures agree with the oracle to the few
    ulps by which CUDA's atan2f / cosf / sinf differ from glibc's inside pcl::eigen33, amplified by the eigen-gap."""
    if which == "cube":
        cloud, radius = cube_pair[0], 0.12
    else:
        cloud, radius = synth.panel_points(40000, 9, noise_sigma=5e-4), 0.035
        if which == "panel_far_from_origin":
            cloud = (cloud + np.array([30.0, -20.0, 10.0], np.float32)).astype(np.float32)
        cloud = np.concatenate([cloud, np.array([[50.0, 50.0, 50.0], [np.nan, 1.0, 1.0]], np.float32)])
    reset(engine)
    engine.set_target(cloud)
    nrm, kept = engine.normals(0, radius)
    ref, rk = oracle.normals(cloud, radius)
    mask, mk = engine.normal_validity(0, radius)
    assert kept == rk == mk
    assert np.array_equal(np.isnan(nrm), np.isnan(ref))
    assert np.array_equal(np.isfinite(nrm[:, 0]), mask.astype(bool))
    ok = np.isfinite(ref[:, 0])
    d = np.abs(nrm[ok, :3] - ref[ok, :3]).max(axis=1)
    # a flipped sign (n . p within an ulp of 0) or a different choice among equal cross products shows as a big jump: none
    assert d.max() < 1e-3, d.max()
    assert np.quantile(d, 0.999) <= 1e-6, np.quantile(d, [0.5, 0.99, 0.999, 1.0])
    assert (d == 0).mean() > 0.5          # most normals are bit-identical
    dc = np.abs(nrm[ok, 3] - ref[ok, 3])
    assert np.quantile(dc, 0.999) <= 1e-6 and dc.max() < 1e-4


def test_zero_gate_finds_no_pairs(engine, oracle, cube_pair):
    """setMaxCorrespondenceDistance(int) truncates (include/GICPAlignment.h:138): 0.5 becomes 0.  PCL then tests
    `nn_dists[0] < 0`, finds no pair, throws NotEnoughPointsException inside align() and hasConverged() stays false
    (reference :101,108 logs "GICP no converge").  A zero gate must therefore mean "no pair", not "no gate"."""
    from leica_point_cloud_processing_b200 import GICPAlignment
    from leica_point_cloud_processing_b200._capi import E_NOT_ENOUGH_CORRESPONDENCES
    from oracle.oracle import default_params
    src, tgt, _ = cube_pair
    ref = oracle.align(src, tgt, default_params(max_corr_distance=0.0))
    assert ref["converged"] == 0 and ref["n_pairs_last"] == 0
    reset(engine, max_corr_distance=0.0)
    engine.set_clouds(tgt, src)
    pairs, idx, d2, _ = engine.correspondences(np.eye(4, dtype=np.float32))
    assert pairs == 0 and np.all(idx == -1)
    res = engine.align(raise_on_failure=False)
    assert res["rc"] == E_NOT_ENOUGH_CORRESPONDENCES and res["converged"] == 0 and res["corr_pairs_last"] == 0
    assert np.array_equal(res["transform"], np.eye(4, dtype=np.float32))
    # the raw NN-1 hook keeps "max_dist <= 0 -> ungated"
    gi, gd = engine.nn1(src, max_dist=0.0)
    oi, od = oracle.nn1(tgt, src)
    assert np.array_equal(gi, oi) and np.array_equal(gd, od)
    g = GICPAlignment(tgt, src, False)
    g.setMaxCorrespondenceDistance(0.5)
    assert g.max_corresp_distance_ == 0.0
    g.run()
    assert not g.hasConverged() and not g.transform_exists_
    assert np.array_equal(g.getFineTransform(), np.eye(4, dtype=np.float32))
    reset(engine)


def test_iterate_keeps_the_clouds_of_the_last_run(cube_pair):
    """reference :111-127,166-174: setSourceCloud / setTargetCloud only swap the wrapper's pointers; gicp_ keeps the
    clouds of the last setInputSource / setInputTarget, so iterate() re-solves the OLD pair."""
    from leica_point_cloud_processing_b200 import GICPAlignment
    src, tgt, _ = cube_pair
    g = GICPAlignment(tgt, src, False)
    g.setMaxCorrespondenceDistance(5)
    g.setTfEpsilon(5e-4)
    g.run()
    T1 = g.getFineTransform()
    other = (src + np.float32(0.25)).astype(np.float32)
    g.setSourceCloud(other)
    g.iterate()
    assert g.hasConverged()
    assert np.allclose(g.getFineTransform(), T1 @ T1, atol=1e-6)   # the same solve as run(), not one on `other`
    fresh = GICPAlignment(tgt, src, False)
    fresh.iterate()                                                # align() before any input was set
    assert not fresh.hasConverged() and not fresh.transform_exists_


# ---- the use_covariances branch: resolution, radius-normal validity, in-place point removal --------------------
def test_cloud_resolution_matches_oracle(engine, oracle, cube_pair):
    """Utils::computeCloudResolution (reference src/Utils.cpp:145-174); the reference's test/test_utils.cpp:78-92 pins
    a 0.1 lattice to 0.1 +- 0.05."""
    src, tgt, _ = cube_pair
    reset(engine)
    engine.set_target(tgt)
    engine.set_source(src)
    for which, cloud in ((0, tgt), (1, src)):
        r = engine.cloud_resolution(which)
        assert abs(r - oracle.resolution(cloud)) <= 1e-12 * r
    assert abs(engine.cloud_resolution(1) - 0.03447) < 2e-5   # the fixture fact recorded in SURVEY section 4
    g = np.stack(np.meshgrid(*[np.arange(12) * 0.1] * 3, indexing="ij"), -1).reshape(-1, 3).astype(np.float32)
    engine.set_source(g)
    assert abs(engine.cloud_resolution(1) - 0.1) <= 1e-6
    with_nan = np.concatenate([g, np.full((3, 3), np.nan, np.float32)])
    engine.set_source(with_nan)
    assert abs(engine.cloud_resolution(1) - 0.1) <= 1e-6


@pytest.mark.parametrize("radius_factor", [0.6, 1.0, 2.0, 8.0])
def test_normal_validity_matches_oracle(engine, oracle, radius_factor):
    """Which points Utils::getNormals gives a finite normal (>= 3 points inside the radius), bit-exact mask."""
    rng = np.random.default_rng(11)
    src, tgt, _ = synth.make_pair(40_000, 40_000)
    # isolated points and pairs (no normal), a NaN point, duplicates
    extra = np.concatenate([rng.uniform(-3, 8, (40, 3)), [[50, 50, 50], [50, 50, 50.001]], [[np.nan, 0, 0]], src[:5]])
    cloud = np.concatenate([src, extra.astype(np.float32)])
    reset(engine)
    engine.set_source(cloud)
    radius = radius_factor * 2.0 * 2 * oracle.resolution(src)
    mask, kept = engine.normal_validity(1, radius)
    om, ok = oracle.normal_validity(cloud, radius)
    assert kept == ok == int(mask.sum())
    assert np.array_equal(mask, om)
    assert mask[len(src) + 42] == 0 and mask[len(src) + 40] == 0   # the NaN point and the isolated pair
    assert 0 < kept < len(cloud)


def test_use_covariances_filters_like_the_reference(oracle):
    """GICPAlignment(use_covariances=true).run(): the points without a finite radius normal are dropped (source first,
    then target, each with freshly computed resolutions, reference src/GICPAlignment.cpp:56-84), then GICP runs with
    its own kNN covariances on what is left."""
    from leica_point_cloud_processing_b200 import GICPAlignment
    from oracle.oracle import default_params
    rng = np.random.default_rng(5)
    src, tgt, _ = synth.make_pair(30_000, 30_000, angle_deg=1.0, offset_m=0.005)
    src = np.concatenate([src, rng.uniform(5, 9, (25, 3)).astype(np.float32)])      # stray points far from the part
    tgt = np.concatenate([tgt, rng.uniform(-9, -5, (30, 3)).astype(np.float32)])
    g = GICPAlignment(tgt, src, True)
    g.setMaxCorrespondenceDistance(1)
    g.run()
    # the same filtering, step by step, with the oracle
    r = 2.0 * (oracle.resolution(tgt) + oracle.resolution(src))
    ms, _ = oracle.normal_validity(src, r)
    src_f = src[ms.astype(bool)]
    r = 2.0 * (oracle.resolution(tgt) + oracle.resolution(src_f))
    mt, _ = oracle.normal_validity(tgt, r)
    tgt_f = tgt[mt.astype(bool)]
    assert len(src_f) < len(src) and len(tgt_f) < len(tgt)
    assert np.array_equal(g.source_cloud_, src_f) and np.array_equal(g.target_cloud_, tgt_f)
    assert g.transform_exists_
    ref = oracle.align(src_f, tgt_f, default_params(max_corr_distance=1.0))
    diag = float(np.linalg.norm(tgt_f.max(0) - tgt_f.min(0)))
    assert synth.rotation_error_rad(g.getFineTransform(), ref["T"]) <= ROT_TOL
    assert synth.translation_error(g.getFineTransform(), ref["T"]) <= 1e-5 * diag
    assert len(g.getAlignedCloud()) == len(src_f)
