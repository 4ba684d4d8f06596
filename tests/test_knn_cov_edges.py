"""kNN neighbourhoods (gicpb_knn) and GICP covariances (gicpb_get_covariances) at their edges, against the oracle.

knn_cov_kernel runs once per cloud in every job, and every Mahalanobis matrix and cost term is built from the covariance
normal it stores.  Each point's list is decided by the (d2, index) order alone, so it is compared bit for bit.

What a case asserts (check_knn_cov), on the target slot (0) and the source slot (1), whose far searches differ (the source
is searched without superbrick slabs):
  * gicpb_knn's idx and d2 equal Oracle.knn's bit for bit, the -1 / inf rows of non-finite points included;
  * gicpb_get_covariances lies within 2 x _cov_util.normal_error_bound of Oracle.covariances(k, eps) and of numpy's SVD
    of the raw matrix, and is NaN on the non-finite rows;
  * the number of points whose bound is below 1e-9 ("tight") is reported and has a floor, so that the bound cannot
    quietly become loose;
  * where the case is built for it, last_far_queries() is > 0 after the kNN call (the far instance ran) or 0 (it did not).

Cases: A every k from 2 to 32 on the cube and a panel at three cell sizes; B exact ties on lattices (the k-th neighbour
at the end of a distance shell and inside one, 0 / 1 km / 8 km out), 40 copies of points, and clusters of copies whose raw
covariance is exactly zero; C the cube and the panel 300 m to 10 km out, and points one float either side of the cell
faces; D the near / far split and neighbourhoods that must cross to another cluster; E non-finite rows and the k limit;
F k and gicp_epsilon changed on a context that already holds covariances, set_clouds against the separate calls; G a
1 M-point panel; H the cloud resolution (k = 2) of all three slots.

CPU part (-m "not gpu"): the fixtures are what they claim (complete shells, exact floats, ties kept after the offset,
exactly zero raw covariances, the finite-subset index map monotone).
"""
import contextlib
import time

import numpy as np
import pytest

from _cov_util import normal_error_bound, raw_covariances, regularised_from_svd
from leica_point_cloud_processing_b200 import synth

OFFSET_DIR = np.array([1.0, -0.5, 0.25])
SP = 2.0 ** -6                    # lattice spacing: every coordinate and every d2 of the lattices is an exact float
SHELLS = [1, 6, 12, 8, 6, 24]     # lattice points at d2 = 0, 1, 2, 3, 4, 5 spacings^2 around an interior point
LATTICE_K = [7, 19, 20, 26, 27, 32]
E_BADARG, E_TOO_FEW_POINTS = -1, -7
TIGHT = 1e-9


@contextlib.contextmanager
def timed(label):
    t0 = time.perf_counter()
    yield
    print(f"[time] {label}: {time.perf_counter() - t0:.2f} s")


# ---- fixtures ---------------------------------------------------------------------------------------------------------
def shifted(cloud, offset):
    return (cloud.astype(np.float64) + OFFSET_DIR * offset).astype(np.float32)


def panel(offset=0.0, n=30000, seed=3):
    return shifted(synth.panel_points(n, seed, noise_sigma=5e-4), offset)


def lattice(offset, side=12, seed=0):
    """side^3 lattice of spacing 2^-6 moved offset * (1, -0.5, 0.25) (multiples of 2^-6 for the offsets used), in a
    shuffled order so that the index decides the ties"""
    g = np.stack(np.meshgrid(*[np.arange(side)] * 3, indexing="ij"), -1).reshape(-1, 3) * SP
    return (g + OFFSET_DIR * offset)[np.random.default_rng(seed).permutation(len(g))].astype(np.float32)


def with_copies(base, n_pts, copies, seed):
    """base plus `copies` - 1 further copies of n_pts of its points, shuffled: more copies than k of one point"""
    rng = np.random.default_rng(seed)
    pick = rng.choice(len(base), n_pts, replace=False)
    c = np.concatenate([base] + [base[pick]] * (copies - 1))
    return c[rng.permutation(len(c))].astype(np.float32)


def zero_clusters(k, n_clusters=12, seed=1):
    """n_clusters clusters of k + 3 copies of one point whose coordinates are small multiples of 2^-6: x * x is exact in
    float, so sum(x * x) / k - mean^2 is exactly 0 for every neighbourhood inside a cluster; clusters 2 m apart"""
    rng = np.random.default_rng(seed)
    cen = (rng.integers(-64, 64, (n_clusters, 3)) * SP + 2.0 * np.arange(n_clusters)[:, None]).astype(np.float32)
    c = np.repeat(cen, k + 3, axis=0)
    return c[rng.permutation(len(c))]


def ordinary_clusters(k, n_clusters=12, seed=2):
    """the same with coordinates of full mantissas: the float squares round, and the raw covariance is rounding residue"""
    rng = np.random.default_rng(seed)
    cen = (rng.uniform(-1, 1, (n_clusters, 3)) + 2.0 * np.arange(n_clusters)[:, None]).astype(np.float32)
    c = np.repeat(cen, k + 3, axis=0)
    return c[rng.permutation(len(c))]


def face_ulps(offset, side=12):
    """the lattice with the cell forced to its spacing (C): after the offset every point moves one float up, one float
    down or stays, along one axis in turn, so points sit within rounding of the cell faces and of the ring bounds"""
    c = lattice(offset, side).astype(np.float32)
    i = np.arange(len(c))
    ax = (i // 3) % 3
    up, down = i % 3 == 1, i % 3 == 2
    c[up, ax[up]] = np.nextafter(c[up, ax[up]], np.float32(np.inf))
    c[down, ax[down]] = np.nextafter(c[down, ax[down]], np.float32(-np.inf))
    return c


def clump_and_outliers(seed=4, n=20000, n_out=300):
    """a dense clump and sparse outliers whose k-th neighbour lies far beyond kKnnMaxRing cells"""
    rng = np.random.default_rng(seed)
    clump = rng.random((n, 3)) * 0.1
    out = (rng.random((n_out, 3)) - 0.5) * 20.0
    return np.concatenate([clump, out]).astype(np.float32)


def two_clusters(k, seed=5):
    """a cluster of 4000 points and, 50 m away, one of k // 2 points whose lists must cross to the first"""
    rng = np.random.default_rng(seed)
    a = rng.normal(0, 0.05, (4000, 3))
    b = rng.normal(0, 0.05, (k // 2, 3)) + [50.0, -20.0, 10.0]
    return np.concatenate([a, b]).astype(np.float32)


def with_nonfinite(cloud, seed=6, every=17):
    c = np.array(cloud, np.float32)
    rng = np.random.default_rng(seed)
    c[::every, rng.integers(0, 3)] = np.nan
    c[5::every * 3, 1] = np.inf
    c[9::every * 5, 2] = -np.inf
    return c


# ---- the reference ----------------------------------------------------------------------------------------------------
_REF = {}


def reference(orc, cloud, k, eps=1e-3):
    """(idx, d2, cov, np_cov, bound) of the whole cloud: the oracle run on the finite rows only, indices mapped back
    through the (monotone) finite-subset map; -1 / inf / NaN on the non-finite rows.  Cached per cloud, k and eps."""
    key = (cloud.tobytes(), k, eps, id(orc))
    if key in _REF:
        return _REF[key]
    n = len(cloud)
    fin = np.isfinite(cloud[:, :3]).all(1)
    m = np.flatnonzero(fin)
    sub = np.ascontiguousarray(cloud[fin, :3])
    oi, od = orc.knn(sub, k)
    idx = np.full((n, k), -1, np.int32)
    d2 = np.full((n, k), np.inf, np.float32)
    idx[fin] = np.where(oi >= 0, m[np.maximum(oi, 0)], -1)
    d2[fin] = od
    cov = np.full((n, 3, 3), np.nan)
    cov[fin] = orc.covariances(sub, k, eps)
    npc = np.full((n, 3, 3), np.nan)
    bound = np.full(n, np.nan)
    for lo in range(0, len(sub), 100000):                   # raw_covariances takes ~ 12 * k bytes * 3 per point
        hi = min(len(sub), lo + 100000)
        r, sv = regularised_from_svd(raw_covariances(sub, oi[lo:hi]), eps)
        npc[m[lo:hi]] = r
        bound[m[lo:hi]] = normal_error_bound(sv)
    _REF[key] = (idx, d2, cov, npc, bound)
    if len(_REF) > 24:
        _REF.pop(next(iter(_REF)))
    return _REF[key]


def reset(engine, **kw):
    base = dict(max_iterations=100, transformation_epsilon=4e-3, rotation_epsilon=2e-3, max_corr_distance=4e-2,
                k_correspondences=20, gicp_epsilon=1e-3, max_inner_iterations=20, cell_size=0.0, points_per_cell=3.0,
                mahalanobis_fp32=0, use_previous_match=1, cost_moments=0, cost_persistent=1)
    base.update(kw)
    engine.set_params(**base)


def check_knn_cov(eng, orc, cloud, which, k, eps=1e-3, far=None, tight_min=0.0, label=""):
    """The contract of the module docstring for one slot.  far: True / False asserts that the kNN call did / did not run
    far queries, "all" that every query went far.  tight_min: floor on the fraction of finite points whose bound is
    < 1e-9 (the floors are the fixtures' fractions, measured with the oracle and numpy alone, rounded down)."""
    idx, d2 = eng.knn(which)
    far_q = eng.last_far_queries()
    cov = eng.covariances(which)
    ridx, rd2, rcov, npc, bound = reference(orc, cloud, k, eps)
    fin = np.isfinite(cloud[:, :3]).all(1)
    bad = np.flatnonzero((idx != ridx).any(1))
    assert bad.size == 0, f"{label}: {bad.size} kNN lists differ, first {bad[:5]}: {idx[bad[0]]} vs {ridx[bad[0]]}"
    assert np.array_equal(d2.view(np.uint32), rd2.view(np.uint32)), f"{label}: d2 differs"
    assert np.isnan(cov[~fin]).all(), f"{label}: a non-finite row has a covariance"
    assert not np.isnan(cov[fin]).any(), f"{label}: a finite row has NaN"
    err = np.abs(cov[fin] - rcov[fin]).max(axis=(1, 2))
    err_np = np.abs(cov[fin] - npc[fin]).max(axis=(1, 2))
    b = bound[fin]
    worst = int(np.argmax(err / b)) if len(b) else 0
    assert (err <= 2.0 * b).all(), f"{label}: covariance off by {err[worst]} (bound {b[worst]}) at finite row {worst}"
    assert (err_np <= 2.0 * b).all(), f"{label}: numpy SVD differs by {err_np.max()}"
    tight = b < TIGHT
    n_tight = int(tight.sum())
    if far == "all":
        assert far_q == int(fin.sum()), f"{label}: {far_q} of {int(fin.sum())} queries went far"
    elif far is True:
        assert far_q > 0, f"{label}: the far instance did not run"
    elif far is False:
        assert far_q == 0, f"{label}: far queries ran ({far_q})"
    print(f"{label} slot {which} k={k}: n={len(cloud)} finite={int(fin.sum())} far={far_q} tight={n_tight} "
          f"max_err_tight={err[tight].max() if n_tight else 0:.2e}")
    assert n_tight >= tight_min * int(fin.sum()), f"{label}: only {n_tight} of {int(fin.sum())} points checked tightly"
    return far_q


def both_slots(eng, orc, cloud, k, eps=1e-3, cell_size=0.0, **kw):
    reset(eng, k_correspondences=k, gicp_epsilon=eps, cell_size=cell_size)
    eng.set_target(cloud)
    eng.set_source(cloud)
    return [check_knn_cov(eng, orc, cloud, which, k, eps, **kw) for which in (0, 1)]


@pytest.fixture(scope="module")
def fast_oracle():
    from oracle.oracle import Oracle
    return Oracle(fast=True)


# ---- CPU: the fixtures are what they claim ----------------------------------------------------------------------------
def brute_d2(c):
    c = c.astype(np.float32)
    return ((c[:, None, :] - c[None, :, :]) ** 2).sum(-1)     # float32: exact for the lattices


@pytest.mark.parametrize("offset", [0.0, 1024.0, 8192.0])
def test_lattice_is_exact_and_its_shells_complete(offset):
    c = lattice(offset)
    ref = np.round((c.astype(np.float64) - OFFSET_DIR * offset) / SP)
    assert np.array_equal(ref * SP + OFFSET_DIR * offset, c.astype(np.float64)), "a coordinate is not an exact float"
    g = ref.astype(int)
    d2 = ((c[:, None, :].astype(np.float64) - c[None, :, :]) ** 2).sum(-1)
    assert np.array_equal(d2, np.float64(brute_d2(c))), "a float d2 rounds"
    units = np.rint(d2 / SP ** 2).astype(int)
    assert np.array_equal(units * SP ** 2, d2)
    inner = np.flatnonzero(((g >= 3) & (g <= 8)).all(1))   # 3 spacings from every face: shells up to d2 = 5 complete
    assert len(inner) == 216
    cum = np.cumsum(SHELLS)
    for i in inner:
        counts = np.bincount(units[i], minlength=6)[:6]
        assert counts.tolist() == SHELLS
    for k in LATTICE_K:
        s = np.searchsorted(cum, k)                        # the k-th neighbour lies in shell s
        assert (k == cum[s]) == (k in (7, 19, 27)), k      # 7, 19, 27 end a shell; 20, 26, 32 cut into one


def test_copies_push_the_point_out_of_its_own_list(oracle):
    base = panel(0.0, 2000)
    c = with_copies(base, 30, 40, 7)
    for k in (20, 32):
        idx, d2 = oracle.knn(c, k)
        u, inv, cnt = np.unique(c, axis=0, return_inverse=True, return_counts=True)
        many = np.flatnonzero(cnt[inv.ravel()] == 40)
        for i in many[:200]:
            same = np.flatnonzero((c == c[i]).all(1))
            assert np.array_equal(idx[i], same[:k]) and (d2[i] == 0).all()
        later = [i for i in many if i not in np.flatnonzero((c == c[i]).all(1))[:k]]
        assert later and all(i not in idx[i] for i in later[:200])


@pytest.mark.parametrize("k", [2, 20, 32])
def test_zero_clusters_have_exactly_zero_raw_covariance(oracle, k):
    c = zero_clusters(k)
    idx, _ = oracle.knn(c, k)
    raw = raw_covariances(c, idx)
    assert (raw == 0.0).all()
    _, sv = regularised_from_svd(raw)
    assert (normal_error_bound(sv) == 1e-13).all()
    # three equal singular values: the stable descending order leaves the last axis last, so the normal is e_z
    assert np.allclose(oracle.covariances(c, k), np.diag([1.0, 1.0, 1e-3]), rtol=0, atol=1e-13)
    o = ordinary_clusters(k)
    raw_o = raw_covariances(o, oracle.knn(o, k)[0])
    # residue of the float squares only: at most about an ulp of the largest x * x
    assert (raw_o != 0.0).any() and np.abs(raw_o).max() <= 2.0 ** -23 * float((o.astype(np.float64) ** 2).max())


@pytest.mark.parametrize("offset", [1000.0, 10000.0])
def test_face_ulp_lattice_sits_on_the_faces(offset):
    c = face_ulps(offset)
    e = lattice(offset)
    diff = (c != e).sum(1)
    assert (diff <= 1).all() and diff.sum() == 2 * len(c) // 3
    ulps = np.abs(c.view(np.int32).astype(np.int64) - e.view(np.int32).astype(np.int64)).sum(1)
    assert (ulps <= 1).all()


def test_finite_subset_map_is_monotone(oracle):
    c = with_nonfinite(panel(0.0, 3000))
    fin = np.isfinite(c).all(1)
    m = np.flatnonzero(fin)
    assert 0 < (~fin).sum() < len(c) and (np.diff(m) > 0).all()
    idx, d2, cov, npc, bound = reference(oracle, c, 20)
    assert (idx[~fin] == -1).all() and np.isinf(d2[~fin]).all() and np.isnan(cov[~fin]).all()
    assert fin[idx[fin]].all()
    # the brute-force lists of the finite rows, in the indices of the whole cloud: the map carries the tie rule over
    f = c[fin]
    d = brute_d2(f)
    for i in range(0, len(f), 97):
        order = np.lexsort((np.arange(len(f)), d[i]))[:20]
        assert np.array_equal(idx[m[i]], m[order])


# ---- A. every k ---------------------------------------------------------------------------------------------------------
CELLS = {"cube": [0.0, 0.03, 0.9], "panel": [0.0, 0.006, 0.15]}
# At k = 2 the raw matrix has rank 1: only where the 2nd neighbour's offset is far from the others is the smallest
# direction well separated (a noise-free cube face gives 28 %).
TIGHT_K2 = {"cube": 0.25, "panel": 0.9}


@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 3, 7, 16, 20, 31, 32])
@pytest.mark.parametrize("shape,cell", [(s, c) for s in ("cube", "panel") for c in CELLS[s]])
def test_every_k(engine, oracle, cube_pair, shape, cell, k):
    cloud = cube_pair[0] if shape == "cube" else panel()
    both_slots(engine, oracle, cloud, k, cell_size=cell, tight_min=TIGHT_K2[shape] if k == 2 else 0.98,
               label=f"A {shape} cell={cell}")


# ---- B. ties ------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("offset", [0.0, 1024.0, 8192.0])
@pytest.mark.parametrize("cell", [0.0, SP])
def test_lattice_ties(engine, oracle, offset, cell):
    cloud = lattice(offset)
    for k in LATTICE_K:   # at the origin the rounding-free symmetric neighbourhoods of the faces are degenerate
        both_slots(engine, oracle, cloud, k, cell_size=cell, tight_min=0.4 if offset == 0.0 else 0.0,
                   label=f"B lattice {offset} cell={cell}")


@pytest.mark.gpu
@pytest.mark.parametrize("k", [20, 32])
def test_copies(engine, oracle, k):
    cloud = with_copies(panel(0.0, 6000), 60, 40, 8)
    both_slots(engine, oracle, cloud, k, tight_min=0.98, label="B copies")


@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 3, 20, 32])
def test_copy_clusters(engine, oracle, k):
    """zero_clusters: raw covariance exactly 0, bound 1e-13 everywhere, so the "ties -> highest index" choice of the
    smallest eigenvalue is held to 1e-13 (the normal is e_z); ordinary_clusters: rounding residue"""
    both_slots(engine, oracle, zero_clusters(k), k, tight_min=1.0, label="B zero clusters")
    cov = engine.covariances(0)
    assert np.allclose(cov, np.diag([1.0, 1.0, 1e-3]), rtol=0, atol=1e-13)
    both_slots(engine, oracle, ordinary_clusters(k), k, tight_min=0.99, label="B ordinary clusters")


# ---- C. far from the origin ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 20, 32])
@pytest.mark.parametrize("offset", [300.0, 1000.0, 10000.0])
@pytest.mark.parametrize("shape", ["cube", "panel"])
def test_far_from_the_origin(engine, oracle, cube_pair, shape, offset, k):
    """From a few hundred metres out PCL's float products x * x make the raw covariance mostly rounding noise
    (computeCovariances sums float products in double).  That is PCL's behaviour, not a defect of the kernel: the kernel
    reproduces the same products and the same double operations in the same order, so its raw matrices equal the
    oracle's, and a noise matrix is well conditioned, so the bound stays sharp there.

    At the default cell size almost every query still ends near, even 10 km out.  So 10 km out the clouds run once more
    on 1 cm cells: there the grid margin (4e-6 |x| = 4 cm) cancels the four rings the near search reaches, a query can
    end near only if its k-th neighbour lies inside its own cell, and the far instance must run."""
    cloud = shifted(cube_pair[0], offset) if shape == "cube" else panel(offset)
    both_slots(engine, oracle, cloud, k, tight_min=0.98, label=f"C {shape} {offset}")
    if offset >= 10000.0:
        both_slots(engine, oracle, cloud, k, cell_size=0.01, far=True, tight_min=0.98, label=f"C {shape} {offset} 1 cm")


@pytest.mark.gpu
@pytest.mark.parametrize("offset", [1000.0, 8192.0])
def test_points_one_float_from_the_cell_faces(engine, oracle, offset):
    """face_ulps with the cell forced to the lattice spacing: the ring bounds of the near search sit within rounding of
    the points, on both sides"""
    cloud = face_ulps(offset)
    for k in (7, 20, 27, 32):
        both_slots(engine, oracle, cloud, k, cell_size=SP, label=f"C face ulps {offset}")


# ---- D. near / far split, sparse neighbourhoods ----------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 20, 32])
def test_clump_and_outliers_go_far(engine, oracle, k):
    both_slots(engine, oracle, clump_and_outliers(), k, far=True, tight_min=0.6 if k == 2 else 0.98,
               label="D clump+outliers")


@pytest.mark.gpu
@pytest.mark.parametrize("k", [3, 20, 32])
def test_lists_cross_to_the_other_cluster(engine, oracle, k):
    cloud = two_clusters(k)
    both_slots(engine, oracle, cloud, k, far=True, label="D two clusters")
    idx, _ = engine.knn(0)
    assert (idx[4000:] < 4000).any(1).all()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 3, 20, 32])
@pytest.mark.parametrize("extra", [0, 1])
def test_clouds_of_k_points(engine, oracle, k, extra):
    cloud = np.random.default_rng(k + extra).normal(0, 1, (k + extra, 3)).astype(np.float32)
    both_slots(engine, oracle, cloud, k, label=f"D {k + extra} points")


@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 20, 32])
def test_forced_all_near_and_all_far(engine, oracle, cube_pair, k):
    """the lattice (extent 0.17) in one cell of 0.5: the 3x3x3 box holds every point and the next ring bound is beyond
    all of them; in cells of 2^-9 the 4 rings reach 2^-7, less than the lattice spacing, so no query ends near.  The
    cube in cells of 0.9 (the box covers it) and of 0.01 (some queries go far)."""
    for off in (0.0, 1024.0):
        cloud = lattice(off)
        both_slots(engine, oracle, cloud, k, cell_size=0.5, far=False, label=f"D lattice {off} all near")
        both_slots(engine, oracle, cloud, k, cell_size=SP / 8, far="all", label=f"D lattice {off} all far")
    both_slots(engine, oracle, cube_pair[0], k, cell_size=0.9, far=False, label="D cube all near")
    both_slots(engine, oracle, cube_pair[0], k, cell_size=0.01, far=True, label="D cube far")


# ---- E. non-finite rows and the k limit --------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 20, 32])
def test_nonfinite_rows(engine, oracle, k):
    cloud = with_nonfinite(panel(0.0, 20000))
    both_slots(engine, oracle, cloud, k, tight_min=0.85 if k == 2 else 0.98, label="E NaN rows")
    both_slots(engine, oracle, with_nonfinite(clump_and_outliers()), k, far=True, tight_min=0.6 if k == 2 else 0.98,
               label="E NaN rows, outliers")


def _with_finite(n_finite, n_total, seed=9):
    rng = np.random.default_rng(seed)
    c = np.full((n_total, 3), np.nan, np.float32)
    rows = np.sort(rng.choice(n_total, n_finite, replace=False))
    c[rows] = rng.normal(0, 1, (n_finite, 3))
    return c


@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 20, 32])
def test_the_k_limit_counts_finite_points(engine, oracle, cube_pair, k):
    from leica_point_cloud_processing_b200 import GicpError
    ok = _with_finite(k, k + 7)
    both_slots(engine, oracle, ok, k, label="E n_finite = k")
    few = _with_finite(k - 1, k + 7)
    good = cube_pair[0]
    for tgt, src in ((few, good), (good, few)):
        reset(engine, k_correspondences=k)
        engine.set_target(tgt)
        engine.set_source(src)
        which = 0 if tgt is few else 1
        with pytest.raises(GicpError) as e:
            engine.knn(which)
        assert e.value.code == E_TOO_FEW_POINTS
        with pytest.raises(GicpError) as e:
            engine.compute_covariances()
        assert e.value.code == E_TOO_FEW_POINTS
        assert engine.align(raise_on_failure=False)["rc"] == E_TOO_FEW_POINTS
    # the context is still usable
    both_slots(engine, oracle, good, k, label="E after TOO_FEW_POINTS")


@pytest.mark.gpu
def test_k_outside_2_to_32_is_refused(engine, oracle, cube_pair):
    from leica_point_cloud_processing_b200 import GicpError
    cloud = cube_pair[0]
    reset(engine, k_correspondences=20)
    engine.set_target(cloud)
    engine.set_source(cloud)
    for bad in (1, 33, 0, -5):
        with pytest.raises(GicpError) as e:
            engine.set_params(k_correspondences=bad)
        assert e.value.code == E_BADARG
        assert engine.get_params().k_correspondences == 20
        check_knn_cov(engine, oracle, cloud, 0, 20, label=f"E after k={bad}")


# ---- F. state on one context ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_k_changes_without_new_clouds(engine, oracle, cube_pair):
    src, tgt, _ = cube_pair
    T = oracle.apply_state([0.01, 0.02, -0.01, 0.01, 0.02, 0.05])
    reset(engine, k_correspondences=20, max_corr_distance=5.0)
    engine.set_target(tgt)
    engine.set_source(src)
    for k in (20, 32, 2, 20):
        engine.set_params(k_correspondences=k)
        check_knn_cov(engine, oracle, tgt, 0, k, tight_min=0.25 if k == 2 else 0.98, label=f"F k -> {k}")
        check_knn_cov(engine, oracle, src, 1, k, tight_min=0.25 if k == 2 else 0.98, label=f"F k -> {k}")
        cov_s, cov_t = engine.covariances(1), engine.covariances(0)
        pairs, idx, d2, maha = engine.correspondences(T)
        cnt, oi, od, omaha = oracle.correspondences(src, tgt, cov_s, cov_t, T, 5.0)
        assert pairs == cnt == len(src)
        assert np.array_equal(idx, oi) and np.array_equal(d2, od)
        assert np.allclose(maha, omaha, rtol=1e-9, atol=1e-9)


@pytest.mark.gpu
def test_epsilon_changes_without_new_clouds(engine, oracle, cube_pair):
    src, tgt, _ = cube_pair
    reset(engine, k_correspondences=20)
    engine.set_target(tgt)
    engine.set_source(src)
    for eps in (1e-3, 1e-1, 1e-6):
        engine.set_params(gicp_epsilon=eps)
        for which, cloud in ((0, tgt), (1, src)):
            check_knn_cov(engine, oracle, cloud, which, 20, eps, tight_min=0.98, label=f"F eps -> {eps}")
        w = np.linalg.eigvalsh(engine.covariances(0))
        assert np.allclose(w[:, 0], eps, rtol=0, atol=1e-12) and np.allclose(w[:, 1:], 1.0, rtol=0, atol=1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 32])
def test_set_clouds_equals_the_separate_calls(engine, oracle, k):
    cloud_t = clump_and_outliers(10)
    cloud_s = clump_and_outliers(11, n=15000, n_out=200)
    reset(engine, k_correspondences=k)
    engine.set_target(cloud_t)
    engine.set_source(cloud_s)
    engine.compute_covariances()
    assert engine.last_far_queries() > 0
    sep = engine.covariances(0), engine.covariances(1)
    engine.set_clouds(cloud_t, cloud_s)
    assert engine.last_far_queries() > 0
    both = engine.covariances(0), engine.covariances(1)
    for a, b in zip(sep, both):
        assert np.array_equal(a.view(np.uint64), b.view(np.uint64))
    check_knn_cov(engine, oracle, cloud_t, 0, k, far=True, label="F set_clouds target")
    check_knn_cov(engine, oracle, cloud_s, 1, k, far=True, label="F set_clouds source")


# ---- G. scale -----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("k", [32, 2])
def test_one_million_points(engine, fast_oracle, k):
    cloud = panel(0.0, 1 << 20, seed=12)
    with timed(f"G 1 M panel k={k}"):
        both_slots(engine, fast_oracle, cloud, k, tight_min=0.85 if k == 2 else 0.98, label="G 1 M panel")
    _REF.clear()


# ---- H. resolution --------------------------------------------------------------------------------------------------------------
def resolution_reference(orc, cloud):
    """Utils::computeCloudResolution from Oracle.knn(., 2) on the finite rows: (mean of sqrt(d2[1]), count, sum of terms)"""
    fin = np.isfinite(cloud[:, :3]).all(1)
    if fin.sum() == 0:
        return 0.0, 0, 0.0
    idx, d2 = orc.knn(np.ascontiguousarray(cloud[fin, :3]), 2)
    has = idx[:, 1] >= 0
    terms = np.sqrt(d2[has, 1].astype(np.float64))
    cnt = int(has.sum())
    return (float(terms.sum()) / cnt if cnt else 0.0), cnt, float(terms.sum())


def resolution_fixtures(cube):
    rng = np.random.default_rng(13)
    base = panel(0.0, 8000)
    return {
        "copies": with_copies(base, 100, 40, 14),
        "nan_rows": with_nonfinite(base),
        "one_point": np.array([[0.5, -1.0, 2.0]], np.float32),
        "two_points": np.array([[0.5, -1.0, 2.0], [0.5, -1.0, 2.25]], np.float32),
        "two_points_one_nan": np.array([[0.5, -1.0, 2.0], [np.nan, 0, 0], [0.5, -1.0, 2.25]], np.float32),
        "cube_1km": shifted(cube, 1000.0),
        "panel_10km": panel(10000.0, 8000),
        "outliers": np.concatenate([base, (rng.random((200, 3)) - 0.5) * 40.0]).astype(np.float32),
    }


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["copies", "nan_rows", "one_point", "two_points", "two_points_one_nan", "cube_1km",
                                  "panel_10km", "outliers"])
def test_resolution(engine, oracle, cube_pair, name):
    cloud = resolution_fixtures(cube_pair[0])[name]
    ref, cnt, tsum = resolution_reference(oracle, cloud)
    # two sums of the same n double terms in different orders differ by at most 2 n 2^-53 sum(terms)
    tol = 2.0 * len(cloud) * 2.0 ** -53 * tsum / cnt if cnt else 0.0
    reset(engine, k_correspondences=20)
    engine.set_target(cloud)
    engine.set_source(cloud)
    engine.difference_set_subtract(cloud)
    for which in (0, 1, 2):
        r = engine.cloud_resolution(which)
        assert abs(r - ref) <= tol, (name, which, r, ref, tol)
    if cnt == 0:
        assert ref == 0.0 and engine.cloud_resolution(0) == 0.0
    print(f"H {name}: n={len(cloud)} count={cnt} res={ref:.9g} tol={tol:.2e}")

