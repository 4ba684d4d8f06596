"""Radius-search normals (gicpb_normals, gicpb_normal_validity) at their edges, against the oracle.

PCL adds a neighbourhood's nine moments in float, in (d2, index) order, and GICPAlignment(..., true) drops every point
whose normal is not finite.  From about 30 m out those float moments cancel so far that most neighbourhoods take
pcl::eigen33's roots2 path (curvature exactly 0), and up to 1 % of the points lose their normal.  On that path the kernel
and the oracle run the same single-rounding float operations, so every bit of a row depends on the neighbour set and on
the summation order: the sharpest check of the count, scan, fill and sort passes there is.

What a case asserts (check_normals):
  * the NaN pattern, n_valid and the normal_validity mask equal the oracle's, and the mask is "normal is finite";
  * rows where the oracle's roots are roots2's (branches 1, 2 and 4 of Oracle.normals_ex) are bit-identical as uint32,
    all four floats (any NaN equals any NaN: 0 / 0 gives a different NaN on the GPU and on the host);
  * rows of the trigonometric path (branch 3) lie within trig_bound of the oracle's;
  * a flipped sign only where the oracle's |cos_theta| is within |p| times that bound.
Branch 4 computes trigonometric roots and discards them for roots2's when the smallest is <= 0.  Only that decision
depends on atan2f / cosf / sinf, and it could legitimately differ from glibc's where the smallest trigonometric root is
within a few ulps of 0; on these seeded fixtures it never does, so branch 4 is held bit-exact like branch 2.

Cases: cancellation far from the origin on both search instances; the near/far switch of the query box; ties and the
strict radius on lattices; degenerate neighbourhoods and argument errors; list sizes at thread-block and scan-tile edges,
lists of 8192 entries and the 2^32 limit on all entries; the three cloud slots and the members of a group; the
use_covariances flow 300 m and 1 km out.

CPU part (-m "not gpu"): Oracle.normals_ex gives normals()' rows and brute-force neighbour counts; the fixtures are what
they claim (radii rounding to the intended float squares).
"""
import contextlib
import time

import numpy as np
import pytest

from leica_point_cloud_processing_b200 import synth

ROT_TOL = 1e-4          # rad, as tests/test_gpu_parity.py
TRANS_TOL_REL = 1e-5    # x bounding-box diagonal
OFFSET_DIR = np.array([1.0, -0.5, 0.25])
OFFSETS = [0.0, 30.0, 300.0, 1000.0, 10000.0]
U = 2.0 ** -24          # unit roundoff of float32


@contextlib.contextmanager
def timed(label):
    t0 = time.perf_counter()
    yield
    print(f"[time] {label}: {time.perf_counter() - t0:.2f} s")


@pytest.fixture(scope="module")
def fast_oracle():
    from oracle.oracle import Oracle
    return Oracle(fast=True)


# ---- fixtures ---------------------------------------------------------------------------------------------------------
def shifted(cloud, offset):
    return (cloud.astype(np.float64) + OFFSET_DIR * offset).astype(np.float32)


def panel(offset, n=40000):
    return shifted(synth.panel_points(n, 9, noise_sigma=5e-4), offset)


def cube(cube_pair, offset):
    return shifted(cube_pair[0], offset)


def tripled_lattice(offset, side=24, spacing=0.125):
    """a planar side x side lattice at z = 0.5 + offset, every point present three times, so that equal d2 sort by index;
    the offset is a multiple of the spacing, so every coordinate and every d2 stays exact in float.  At the origin the
    moments are exact too (zz covariance 0: roots2 everywhere); 1 km out x * x rounds and the summation order shows."""
    g = np.stack(np.meshgrid(np.arange(side) * spacing, np.arange(side) * spacing, indexing="ij"), -1).reshape(-1, 2)
    pts = np.concatenate([g, np.full((len(g), 1), 0.5)], axis=1) + offset
    return np.concatenate([pts, pts, pts])[np.random.default_rng(3).permutation(3 * len(pts))].astype(np.float32)


def radius_with_square(target_f32):
    """a double radius whose float(radius * radius) is exactly target_f32"""
    r = float(np.sqrt(np.float64(target_f32)))
    for _ in range(8):
        sq = np.float32(r * r)
        if sq == target_f32:
            return r
        r = float(np.nextafter(r, np.inf if sq < target_f32 else -np.inf))
    raise AssertionError(target_f32)


def lattice_radii():
    """(label, radius, float(r^2) vs the lattice d2): 0.125 and the next float radius around the axis neighbour at
    d2 = 2^-6; radii whose float squares are one float above and below the diagonal neighbour's d2 = 2^-5"""
    f = np.float32
    diag = f(0.03125)
    return [("axis_exact", 0.125, "equal"),
            ("axis_next", float(np.nextafter(f(0.125), f(1))), "above"),
            ("diag_above", radius_with_square(np.nextafter(diag, f(1))), "above"),
            ("diag_below", radius_with_square(np.nextafter(diag, f(0))), "below")]


def random_cloud(n, seed, nan_every=17):
    rng = np.random.default_rng(seed)
    c = rng.uniform(-0.2, 0.2, (n, 3)).astype(np.float32)
    c[:, 2] *= 0.05                                     # a slab: a clear smallest eigenvalue
    c[::nan_every, rng.integers(0, 3)] = np.nan
    c[5::nan_every * 3, 1] = np.inf
    return c


def ball(n, center, radius, seed):
    rng = np.random.default_rng(seed)
    v = rng.normal(size=(n, 3))
    v *= (rng.random((n, 1)) ** (1 / 3) * radius / np.linalg.norm(v, axis=1, keepdims=True))
    return (v + center).astype(np.float32)


# ---- the comparison ---------------------------------------------------------------------------------------------------
def trig_bound(gap, xyz):
    """Bound on |kernel - oracle| for a row of the trigonometric path, in the units of the unit normal.

    pcl::eigen33 scales the covariance by its largest |entry|, so its eigenvalues lie in [0, 3] and
    rho = sqrt(sum of squared eigenvalue gaps / 18) <= 1.25.  Each root is c2/3 + rho * (a cos(theta) + b sin(theta)) with
    |a| <= 2, |b| <= sqrt(3), theta = atan2(...) / 3.  CUDA documents atan2f within 3 ulp and cosf / sinf within 2 ulp;
    glibc is within 1 ulp; an ulp is at most 2 U of the value.  So cos and sin differ by <= 6 U, atan2 by <= 8 pi U and
    theta by <= 8.4 U, which moves a cos + b sin by <= (2 + sqrt 3) 8.4 U = 31 U.  Each root, and roots[1] - roots[0],
    therefore moves by <= rho (2 * 6 + sqrt(3) * 6 + 31) U = 53 rho U <= 67 U.  The normal is the normalised cross
    product of two rows of A - roots[0] I; a shift of roots[0] by e turns it by ~e / gap (first-order perturbation of the
    null vector of a matrix whose next singular value is the root gap), and the float rounding of the cross product adds
    ~4 U / gap.  With a factor of 2 for the second order:
        |dn| <= 2 (67 + 4) U / gap + 8 U = 142 U / gap + 8 U.
    The flip compares cos_theta = -p . n with 0, so a sign may differ where |cos_theta| <= |p| |dn| + 8 U.
    The curvature |roots[0] * scale / trace| moves by the root shift over c2 >= 1 (the largest entry of a PSD matrix is on
    its diagonal) plus its own rounding: |dc| <= 67 U + 4 ulp(c)."""
    with np.errstate(divide="ignore"):
        bn = np.where(gap > 0, 142.0 * U / gap, np.inf) + 8.0 * U
    return bn, bn * np.linalg.norm(xyz.astype(np.float64), axis=1) + 8.0 * U


def canon(a):
    b = np.ascontiguousarray(a, np.float32).view(np.uint32).copy()
    b[np.isnan(a)] = 0x7FC00000
    return b


def check_normals(eng, orc, cloud, radius, which=0, far=None, label=""):
    """The contract of the module docstring; far=True / False asserts that the fill pass did / did not run far queries.
    Returns (rows, info, stats)."""
    rows, kept = eng.normals(which, radius)
    far_q = eng.last_far_queries()
    mask, mk = eng.normal_validity(which, radius)
    ref, info, rk = orc.normals_ex(cloud, radius)
    assert kept == rk == mk == int(mask.sum()), (kept, rk, mk)
    assert np.array_equal(np.isnan(rows), np.isnan(ref))
    assert np.array_equal(mask.astype(bool), np.isfinite(rows[:, :3]).all(1))
    branch = info[:, 1].astype(int)
    same = (canon(rows) == canon(ref)).all(1)
    exact = (branch == 1) | (branch == 2) | (branch == 4)
    assert same[exact].all(), f"{label}: {int((~same[exact]).sum())} roots2 rows differ, first {np.flatnonzero(exact & ~same)[:5]}"
    bn, bflip = trig_bound(info[:, 2], cloud[:, :3])
    trig = (branch == 3) & ~same & np.isfinite(ref[:, 0])
    d = np.abs(rows[trig, :3].astype(np.float64) - ref[trig, :3])
    flip = np.abs(rows[trig, :3].astype(np.float64) + ref[trig, :3]).max(axis=1) < d.max(axis=1)
    dn = np.where(flip, np.abs(rows[trig, :3].astype(np.float64) + ref[trig, :3]).max(axis=1), d.max(axis=1))
    assert (dn <= bn[trig]).all(), f"{label}: normal off by {dn.max()} (bound {bn[trig][np.argmax(dn - bn[trig])]})"
    assert (np.abs(info[trig, 3][flip]) <= bflip[trig][flip]).all(), f"{label}: sign flipped with |cos_theta| large"
    dc = np.abs(rows[trig, 3].astype(np.float64) - ref[trig, 3])
    assert (dc <= 67 * U + 4 * np.spacing(np.abs(ref[trig, 3]))).all(), f"{label}: curvature off by {dc.max()}"
    if far is True:
        assert far_q > 0, f"{label}: the far instance did not run"
    elif far is False:
        assert far_q == 0, f"{label}: far queries ran ({far_q})"
    stats = dict(n=len(cloud), kept=kept, far=far_q, branches=np.bincount(branch, minlength=5).tolist(),
                 identical=int(same.sum()), max_count=int(info[:, 0].max()) if len(info) else 0)
    print(f"{label}: {stats}")
    return rows, info, stats


def reset(engine, **kw):
    base = dict(max_iterations=100, transformation_epsilon=4e-3, rotation_epsilon=2e-3, max_corr_distance=4e-2,
                k_correspondences=20, gicp_epsilon=1e-3, max_inner_iterations=20, cell_size=0.0, points_per_cell=3.0,
                mahalanobis_fp32=0, use_previous_match=1, cost_moments=0, cost_persistent=1)
    base.update(kw)
    engine.set_params(**base)


# ---- CPU: the oracle's extended call and the fixtures ----------------------------------------------------------------
@pytest.mark.parametrize("offset", [0.0, 300.0])
def test_oracle_normals_ex_gives_the_rows_of_normals(oracle, cube_pair, offset):
    for cloud, radius in ((panel(offset, 8000), 0.06), (cube(cube_pair, offset), 0.12), (tripled_lattice(0.0), 0.13)):
        cloud = np.concatenate([cloud, [[np.nan, 0, 0], [1e3, 1e3, 1e3]]]).astype(np.float32)
        rows, k = oracle.normals(cloud, radius)
        rows_ex, info, k_ex = oracle.normals_ex(cloud, radius)
        assert k == k_ex
        assert np.array_equal(canon(rows), canon(rows_ex))
        branch = info[:, 1]
        assert np.array_equal(branch == 0, info[:, 0] < 3)
        assert np.array_equal(np.isfinite(info[:, 3]), np.isfinite(rows[:, 0]))
        # roots2 gives a zero smallest root: curvature exactly 0 where the normal exists
        fin = np.isfinite(rows[:, 0])
        assert (rows[fin & ((branch == 2) | (branch == 4)), 3] == 0).all()
        assert (rows[fin & (branch == 3), 3] > 0).all()
        assert (np.isnan(rows[branch == 1, 0])).all()     # zero covariance: 0 / 0


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_oracle_neighbour_counts_brute_force(oracle, seed):
    """count = #{j : (dx*dx + dy*dy) + dz*dz < float32(r^2)} in float32, NaN rows count nothing and get 0"""
    rng = np.random.default_rng(seed)
    c = rng.uniform(0, 1, (600, 3)).astype(np.float32)
    c[::40] = np.floor(c[::40] * 8) / 8               # some lattice points: exact d2 ties at the radius
    c[7::50, 0] = np.nan
    for radius in (0.1, 0.125, 0.25, float(np.nextafter(0.125, np.inf))):
        _, info, _ = oracle.normals_ex(c, radius)
        r2 = np.float32(radius * radius)
        d = c[:, None, :] - c[None, :, :]
        d2 = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
        assert d2.dtype == np.float32
        with np.errstate(invalid="ignore"):
            cnt = (d2 < r2).sum(1)
        cnt[~np.isfinite(c).all(1)] = 0
        assert np.array_equal(info[:, 0].astype(np.int64), cnt)


def test_fixtures_are_what_they_claim(oracle):
    f = np.float32
    for label, r, rel in lattice_radii():
        sq = f(r * r)
        d2 = f(0.015625) if label.startswith("axis") else f(0.03125)
        assert {"equal": sq == d2, "above": sq > d2, "below": sq < d2}[rel], label
        if label.startswith("diag"):
            assert np.nextafter(d2, f(1) if rel == "above" else f(0)) == sq, label
    for off in (0.0, 1000.0):
        lat = tripled_lattice(off)
        _, info, _ = oracle.normals_ex(lat, 0.125)
        assert (info[:, 0] == 3).all()                                   # itself, three times
        # at the origin a zero covariance; 1 km out the float moments of three equal points do not cancel exactly
        assert (info[:, 1] == 1).all() if off == 0 else (info[:, 1] != 1).any()
        _, info, _ = oracle.normals_ex(lat, lattice_radii()[1][1])
        assert info[:, 0].max() == 15                                    # + the 4 axis neighbours, three times each
        assert (info[:, 1] == 2).all() if off == 0 else ((info[:, 1] == 2) | (info[:, 1] == 4)).all()
    assert f(1e-30 * 1e-30) == 0
    with np.errstate(over="ignore"):
        assert f(1e30 * 1e30) == np.inf


# ---- GPU --------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("radius", [0.035, 0.2])
@pytest.mark.parametrize("offset", OFFSETS)
@pytest.mark.parametrize("kind", ["panel", "cube"])
def test_cancellation_far_from_the_origin(engine, fast_oracle, cube_pair, kind, offset, radius):
    """A. The panel and the cube 0 m to 10 km out: 0.035 on the near instance, 0.2 on the far one (panel)."""
    cloud = panel(offset) if kind == "panel" else cube(cube_pair, offset)
    reset(engine)
    engine.set_target(cloud)
    far = (radius == 0.2) if kind == "panel" else None
    _, info, st = check_normals(engine, fast_oracle, cloud, radius, far=far, label=f"{kind} {offset} m r={radius}")
    b = np.array(st["branches"]) / len(cloud)
    if offset >= 300:
        assert b[2] + b[4] >= 0.8 * (1 - b[0]), b     # the roots2 path (bit-exact rows) for most points with neighbours
    if offset == 0 and kind == "panel":
        assert b[3] >= 0.999, b                       # near the origin next to nothing cancels
    if kind == "panel" and offset >= 300 and radius == 0.035:
        assert st["kept"] < len(cloud)                # some points lose their normal to the cancellation


@pytest.mark.gpu
@pytest.mark.parametrize("offset", [0.0, 300.0])
def test_near_far_switch(engine, fast_oracle, offset):
    """B. cell_size forced to h; radius 3.4 h ... 5 h takes the query box across kMaxBoxRows = 81 rows."""
    h = 0.01
    cloud = panel(offset)
    reset(engine, cell_size=h)
    engine.set_target(cloud)
    split = 0
    n = int(np.isfinite(cloud).all(1).sum())
    for f in np.linspace(3.4, 5.0, 9):
        _, _, st = check_normals(engine, fast_oracle, cloud, f * h, label=f"switch {offset} m r={f:.1f}h")
        split += 0 < st["far"] < n
    assert split >= 3          # e.g. 488, 21,971 and 33,710 of 40,000 queries far at 4.0 h, 4.2 h and 4.4 h
    reset(engine)


@pytest.mark.gpu
@pytest.mark.parametrize("offset", [0.0, 1000.0])
def test_ties_and_the_strict_radius(engine, fast_oracle, offset):
    """C. A tripled planar lattice: neighbours at d2 = r2 excluded, one float above included; equal d2 sorted by index."""
    lat = tripled_lattice(offset)
    reset(engine)
    engine.set_target(lat)
    for label, radius, rel in lattice_radii():
        _, info, st = check_normals(engine, fast_oracle, lat, radius, label=f"lattice {offset} {label}")
        if label == "axis_exact":
            assert (info[:, 0] == 3).all()
            assert st["kept"] == 0 if offset == 0 else 0 < st["kept"] < len(lat)
        if label == "axis_next":
            assert info[:, 0].max() == 15
            assert st["kept"] == len(lat) if offset == 0 else st["kept"] < len(lat)
        if label.startswith("diag"):
            assert info[:, 0].max() == (27 if rel == "above" else 15)
    # the same lattice on the far instance: with 1 cm cells a 0.45 m radius spans more than 81 rows along y
    reset(engine, cell_size=0.01)
    engine.set_target(lat)
    check_normals(engine, fast_oracle, lat, 0.45, far=True, label=f"lattice {offset} far")
    reset(engine)


def _degenerate_cases():
    f = np.float32
    far_pt = [[5.0, 5.0, 5.0]]
    return [
        ("one", np.array([[0.1, 0.2, 0.3]], f), 1.0),
        ("two", np.array([[0.1, 0.2, 0.3], [0.1, 0.2, 0.35]], f), 1.0),
        ("three", np.array([[0.1, 0.2, 0.3], [0.1, 0.25, 0.35], [0.15, 0.2, 0.3]], f), 1.0),
        ("three_identical", np.array([[0.1, 0.2, 0.3]] * 3, f), 1.0),
        ("three_collinear", np.array([[0.1, 0.2, 0.3], [0.2, 0.3, 0.4], [0.3, 0.4, 0.5]], f), 1.0),
        ("five_identical_and_far", np.array([[1.0, -2.0, 0.5]] * 5 + far_pt, f), 1.0),
        ("nonfinite_rows", np.array([[np.nan, 0, 0], [0.1, 0.2, 0.3], [np.inf, 1, 1], [0.1, 0.25, 0.35],
                                     [0, -np.inf, 0], [0.15, 0.2, 0.3], [np.nan] * 3], f), 1.0),
        ("square_underflows", np.array([[0.1, 0.2, 0.3]] * 4 + [[0.1, 0.2, 0.31]], f), 1e-30),
    ]


@pytest.mark.gpu
def test_degenerate_neighbourhoods_and_arguments(engine, oracle):
    """D. Tiny clouds, zero and rank-1 covariances, non-finite rows, every list the whole cloud, bad radii."""
    from leica_point_cloud_processing_b200._capi import E_BADARG, GicpError
    reset(engine)
    for label, cloud, radius in _degenerate_cases():
        engine.set_target(cloud)
        _, info, st = check_normals(engine, oracle, cloud, radius, label=label)
        if label in ("one", "two", "square_underflows"):
            assert st["kept"] == 0
        if label == "three_identical":
            assert st["kept"] == 0 and (info[:, 0] == 3).all() and (info[:, 1] == 1).all()
        if label == "five_identical_and_far":
            assert st["kept"] == 0 and (info[:5, 0] == 5).all() and info[5, 0] == 1
        if label == "square_underflows":
            assert (info[:, 0] == 0).all()
    rng = np.random.default_rng(4)
    c = rng.uniform(-1, 1, (3000, 3)).astype(np.float32)
    c[:, 2] *= 0.01
    engine.set_target(c)
    for radius in (np.inf, 1e30):
        _, info, _ = check_normals(engine, oracle, c, radius, label=f"whole cloud r={radius}")
        assert (info[:, 0] == len(c)).all()
    for radius in (0.0, -1.0, np.nan):
        for call in (engine.normals, engine.normal_validity):
            with pytest.raises(GicpError) as e:
                call(0, radius)
            assert e.value.code == E_BADARG


@pytest.mark.gpu
def test_long_lists_and_the_2_32_limit(engine, fast_oracle):
    """E. Lists of 8192 entries; 65,536^2 = 2^32 and 70,000^2 entries refused by both calls; the context stays usable."""
    from leica_point_cloud_processing_b200 import Engine
    from leica_point_cloud_processing_b200._capi import E_BADARG, GicpError
    ref_cloud = panel(300.0, 20000)
    reset(engine)
    engine.set_target(ref_cloud)
    before, _ = engine.normals(0, 0.035)
    for offset in (0.0, 300.0):
        b = ball(8192, OFFSET_DIR * offset, 0.05, 7)
        engine.set_target(b)
        with timed(f"8192 lists of 8192, {offset} m"):
            _, info, _ = check_normals(engine, fast_oracle, b, 1.0, label=f"ball 8192 {offset} m")
        assert (info[:, 0] == 8192).all()
    for n in (65536, 70000):
        engine.set_target(ball(n, np.zeros(3), 0.05, 8))
        for call in (engine.normals, engine.normal_validity):
            with pytest.raises(GicpError) as e:
                call(0, 1.0)
            assert e.value.code == E_BADARG and "more than 2^32 neighbour entries" in str(e.value)
        engine.set_target(ref_cloud)
        after, _ = engine.normals(0, 0.035)
        assert np.array_equal(canon(after), canon(before))
    fresh = Engine(0)
    try:
        reset(fresh)
        fresh.set_target(ref_cloud)
        assert np.array_equal(canon(fresh.normals(0, 0.035)[0]), canon(before))
    finally:
        fresh.close()


@pytest.mark.gpu
def test_block_and_tile_edges_and_scale(engine, oracle, fast_oracle):
    """E. n at the 128-thread block and 4096-entry scan tile edges with NaN rows; a 1 M-point panel; one context running
    big -> small -> big."""
    reset(engine)
    for n in (127, 128, 129, 4095, 4096, 4097):
        c = random_cloud(n, n)
        engine.set_target(c)
        check_normals(engine, oracle, c, 0.06, label=f"random {n}")
    big = shifted(synth.panel_points(1_000_000, 21, noise_sigma=5e-4), 300.0)
    engine.set_target(big)
    with timed("1 M panel"):
        first, _, st = check_normals(engine, fast_oracle, big, 0.01, label="1M panel 300 m")
    small = random_cloud(129, 5)
    engine.set_target(small)
    check_normals(engine, oracle, small, 0.06, label="small after big")
    engine.set_target(big)
    again, _ = engine.normals(0, 0.01)
    assert np.array_equal(canon(again), canon(first))


@pytest.mark.gpu
def test_which_cloud_and_group_members(engine, oracle):
    """F. Target, source and subtract slots give the same rows; group members on a windowed source and a windowed
    subtract equal a single context; a group align afterwards returns the same transform."""
    from leica_point_cloud_processing_b200 import EngineGroup
    src, tgt, _ = synth.make_pair(60_000, 60_000, angle_deg=1.0, offset_m=0.005)
    src, tgt = shifted(src, 300.0), shifted(tgt, 300.0)
    radius = 0.03
    reset(engine)
    engine.set_target(src)
    engine.set_source(src)
    engine.difference_set_subtract(src)
    rows = [engine.normals(w, radius)[0] for w in (0, 1, 2)]
    check_normals(engine, oracle, src, radius, which=1, label="which=1")
    assert np.array_equal(canon(rows[0]), canon(rows[1])) and np.array_equal(canon(rows[0]), canon(rows[2]))
    engine.difference_set_subtract(tgt)
    sub_rows = engine.normals(2, radius)[0]
    grp = EngineGroup([0, 0])
    try:
        grp.set_params(max_corr_distance=0.04)
        grp.set_clouds(tgt, src)
        first = grp.align()
        for r in range(grp.size):
            m = grp.member(r)
            assert m.grid_info(1)["n_points"] == len(src)
            assert np.array_equal(canon(m.normals(1, radius)[0]), canon(rows[1])), r
        grp.cloud_difference(src, tgt, 1e-4)
        for r in range(grp.size):
            assert np.array_equal(canon(grp.member(r).normals(2, radius)[0]), canon(sub_rows)), r
        again = grp.align()
        assert np.array_equal(again["transform"], first["transform"])
    finally:
        grp.close()


@pytest.mark.gpu
@pytest.mark.parametrize("offset", [300.0, 1000.0])
def test_use_covariances_far_from_the_origin(oracle, offset):
    """G. GICPAlignment(use_covariances=true).run() 300 m and 1 km out drops exactly the points the oracle's masks drop
    (source first, then target, each with freshly computed resolutions), then aligns like the oracle."""
    from leica_point_cloud_processing_b200 import GICPAlignment
    from oracle.oracle import default_params
    rng = np.random.default_rng(5)
    src, tgt, _ = synth.make_pair(30_000, 30_000, angle_deg=1.0, offset_m=0.005)
    src = np.concatenate([src, rng.uniform(5, 9, (25, 3)).astype(np.float32)])
    tgt = np.concatenate([tgt, rng.uniform(-9, -5, (30, 3)).astype(np.float32)])
    src, tgt = shifted(src, offset), shifted(tgt, offset)
    g = GICPAlignment(tgt, src, True)
    g.setMaxCorrespondenceDistance(1)
    g.run()
    r = 2.0 * (oracle.resolution(tgt) + oracle.resolution(src))
    ms, _ = oracle.normal_validity(src, r)
    src_f = src[ms.astype(bool)]
    r = 2.0 * (oracle.resolution(tgt) + oracle.resolution(src_f))
    mt, _ = oracle.normal_validity(tgt, r)
    tgt_f = tgt[mt.astype(bool)]
    print(f"{offset} m: kept {len(src_f)} / {len(src)} source, {len(tgt_f)} / {len(tgt)} target")
    assert len(src_f) < len(src) and len(tgt_f) < len(tgt)
    assert np.array_equal(g.source_cloud_, src_f) and np.array_equal(g.target_cloud_, tgt_f)
    assert g.transform_exists_
    ref = oracle.align(src_f, tgt_f, default_params(max_corr_distance=1.0))
    diag = float(np.linalg.norm(tgt_f.max(0) - tgt_f.min(0)))
    rot = synth.rotation_error_rad(g.getFineTransform(), ref["T"])
    tr = synth.translation_error(g.getFineTransform(), ref["T"])
    print(f"{offset} m: rotation {rot:.3e} rad, translation {tr:.3e} m (diag {diag:.2f})")
    assert rot <= ROT_TOL
    assert tr <= TRANS_TOL_REL * diag
