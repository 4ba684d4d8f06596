"""Euclidean clustering (gicpb_euclidean_clusters) and the voxel grid (gicpb_voxel_grid) at their edges and at scale,
against the oracle.

Voxel grid: PCL's leaf-size check on both sides of its boundary and in the window where div_b (up to dx + 1 per axis)
passes 2^31 or 2^32 while PCL's dx * dy * dz check passes; voxel totals at radix digit boundaries (1 to 4 sort passes);
valid point counts at sort-tile boundaries; faces, negative zero, large coordinates; strides 12 ... 32 from pageable,
pinned and device memory, written into a buffer of 0xFF bytes so that every byte the call leaves is seen.
Clustering: tolerances exactly at lattice pair distances, far from the origin (where the query box outgrows the near
search), a giant cluster, a deep chain, singletons, the size filter at cluster sizes.  One context is reused across
all of it, and the members of a group are used alone.

CPU part (-m "not gpu"): the fixtures are what they claim (brute-force components, PCL's index arithmetic in numpy).
GPU part (-m gpu): labels array-equal; voxel rows bit for bit as uint32 over every byte.  Large cases print their time.
"""
import contextlib
import ctypes
import time

import numpy as np
import pytest

from leica_point_cloud_processing_b200 import synth
from test_segment import components_brute_force, same_partition, xyzrgb

INT32_MAX = 2 ** 31 - 1
WARNING = "Leaf size is too small"


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
def pcl_dims(xyz, leaf):
    """PCL's check (dx, dy, dz) and its index extents div_b, in PCL's float arithmetic"""
    p = np.asarray(xyz, np.float32)
    p = p[np.isfinite(p).all(1)]
    inv = np.float32(1.0) / np.float32(leaf)
    lo, hi = p.min(0), p.max(0)
    d = ((hi - lo) * inv).astype(np.int64) + 1
    div = np.floor(hi * inv).astype(np.int64) - np.floor(lo * inv).astype(np.int64) + 1
    return [int(v) for v in d], [int(v) for v in div]


def overflow_cases():
    """(name, xyz, leaf, refused by PCL): a few points each, leaf 1"""
    f = np.float32
    cases = [
        # dx * dy = 46340 * 46341 = 2 147 441 940 < INT32_MAX, div_b the same
        ("below", [(0, 0, 0), (46339.5, 46340.5, 0), (7, 9, 0), (7.5, 9.5, 0)], False),
        # 46341^2 = 2 147 488 281 > INT32_MAX
        ("above", [(0, 0, 0), (46340.5, 46340.5, 0), (7, 9, 0)], True),
        # the window: dims 46340 x 46340 pass, div_b 46341 x 46341 would not
        ("window", [(0.5, 0.5, 0), (0.6, 0.6, 0), (46340.4, 46340.4, 0)], False),
        # dx * dy * dz = (2^30 + 1024) * 1 * 1 passes; div_b = (2^30 + 1025) * 2 * 2 > 2^32: PCL's index wraps, and the
        # last point (index 2^30 + 1024 + 3 div0 - 2^32 = 4099) is averaged with the point of voxel (4099, 0, 0)
        ("wrap", [(0.5, 0.9, 0.9), (2.0 ** 30 + 1024, 1.1, 1.1), (4099.5, 0.9, 0.9), (4100.5, 0.9, 0.9),
                  (77.25, 1.1, 0.9)], False),
    ]
    return [(n, np.array(p, f), 1.0, r) for n, p, r in cases]


def digit_cloud(dims, n, seed):
    """points in a box of dims[0] x dims[1] x dims[2] unit voxels (corners occupied), so div_b = dims"""
    rng = np.random.default_rng(seed)
    d = np.array(dims, np.float64)
    xyz = 0.5 + rng.random((n, 3)) * (d - 1.0)
    xyz[0] = 0.5
    xyz[-1] = d - 0.5
    return xyz.astype(np.float32)


def lattice(shape, s, origin=(0.0, 0.0, 0.0), jitter=0.0, seed=0):
    ijk = np.stack(np.meshgrid(*[np.arange(k) for k in shape], indexing="ij"), -1).reshape(-1, 3)
    xyz = np.asarray(origin, np.float64) + ijk * float(s)
    if jitter:
        xyz += np.random.default_rng(seed).uniform(-jitter, jitter, xyz.shape)
    return xyz.astype(np.float32)


def lattice_cases():
    """(name, xyz, tolerance): tolerances at the lattice's pair distances"""
    s = np.float32(0.25)
    up, down = np.nextafter(s, np.float32(1)), np.nextafter(s, np.float32(0))
    return [
        ("exact_s", lattice((9, 9, 9), s), float(s)),               # d2 == r2 everywhere: nothing joins
        ("s_plus_ulp", lattice((9, 9, 9), s), float(up)),           # every lattice edge joins
        ("s_minus_ulp", lattice((9, 9, 9), s), float(down)),
        ("tenth", lattice((10, 10, 10), 0.1), float(np.float32(0.1))),  # float differences straddle 0.1
        ("jittered", lattice((10, 10, 10), 0.05, jitter=2e-5, seed=3), 0.05),
        ("far_1e3", lattice((10, 10, 10), 0.05, origin=(1000.0, -2000.0, 500.0)), 0.05),
        ("far_1e4", lattice((10, 10, 10), 0.05, origin=(1e4, 1e4, -1e4)), 0.05),
        ("far_1e4_fine", lattice((10, 10, 10), 0.01, origin=(1e4, 3e3, -1e4)), 0.01),
    ]


def size_filter_cloud():
    """blobs of sizes 5, 3, 7, 5, 7, 1, 7 (3 cm spacing, 2 m apart), NaN at the first and the last index"""
    rng = np.random.default_rng(8)
    parts = [np.full((1, 3), np.nan, np.float32)]
    for b, k in enumerate([5, 3, 7, 5, 7, 1, 7]):
        c = np.array([2.0 * b, 0.5 * (b % 2), 0.0])
        parts.append((c + np.arange(k)[:, None] * [0.03, 0.0, 0.0] + rng.uniform(-1e-3, 1e-3, (k, 3))).astype(np.float32))
    parts.append(np.full((1, 3), np.nan, np.float32))
    xyz = np.concatenate(parts)
    xyz[-1, 1] = 0.0  # only y finite: still a non-finite point
    return xyz


def helix_chain(n, tol):
    """n points 0.9 tol apart along a helix whose turns are 5 tol apart: one component, as deep as it gets"""
    r, pitch = 1.0, 5.0 * tol
    dt = 0.9 * tol / np.hypot(r, pitch / (2 * np.pi))
    t = np.arange(n) * dt
    return np.stack([r * np.cos(t), r * np.sin(t), pitch * t / (2 * np.pi)], 1).astype(np.float32)


def rows(xyz, cols):
    """xyz as rows of `cols` float32 (4: w = 1, >= 5: PointXYZRGB-like with a colour word)"""
    if cols == 3:
        return np.ascontiguousarray(xyz, np.float32)
    return np.ascontiguousarray(xyzrgb(xyz, np.random.default_rng(len(xyz)))[:, :cols])


# ---- CPU: the fixtures are what they claim ----------------------------------------------------------------------------
@pytest.mark.parametrize("case", overflow_cases(), ids=lambda c: c[0])
def test_overflow_fixtures_straddle_pcl_check(oracle, case):
    name, xyz, leaf, refused = case
    d, div = pcl_dims(xyz, leaf)
    prod, divprod = d[0] * d[1] * d[2], div[0] * div[1] * div[2]
    assert (prod > INT32_MAX) == refused
    if name == "window":
        assert INT32_MAX < divprod < 2 ** 32
    if name == "wrap":
        assert divprod > 2 ** 32
    out = oracle.voxel_grid(xyz, leaf)
    assert (out is None) == refused
    if name == "window":
        assert len(out) == 2                                   # (0.5, 0.5) and (0.6, 0.6) share voxel 0
    if name == "wrap":
        # PCL's wrapped index merges the far point with the point of voxel (4099, 0, 0): 4 centroids of 5 points
        assert len(out) == 4
        merged = (np.float32(4099.5) + np.float32(2.0 ** 30 + 1024)) / np.float32(2)
        assert np.float32(merged) in out[:, 0]


@pytest.mark.parametrize("dims,passes", [((3, 5, 17), 1), ((4, 8, 8), 1), ((257, 1, 1), 2), ((15, 17, 257), 2),
                                         ((16, 64, 64), 2), ((195, 21, 4097), 3), ((97, 257, 673), 4)])
def test_digit_fixtures_have_the_voxel_totals(dims, passes):
    xyz = digit_cloud(dims, 1000, 1)
    d, div = pcl_dims(xyz, 1.0)
    assert d == list(dims) and div == list(dims)
    total = int(np.prod(dims))
    assert (max(1, int(total - 1).bit_length()) + 7) // 8 == passes   # keys below total


@pytest.mark.parametrize("case", lattice_cases(), ids=lambda c: c[0])
def test_lattice_fixtures_against_brute_force(oracle, case):
    name, xyz, tol = case
    labels, nc = oracle.euclidean_clusters(xyz, tol, min_size=1)
    n_ref, lab_ref = components_brute_force(xyz, tol)
    assert nc == n_ref and same_partition(labels, lab_ref)
    if name == "exact_s":
        assert nc == len(xyz)                                  # d2 == r2 must not join
    if name == "s_plus_ulp":
        assert nc == 1
    if name == "s_minus_ulp":
        assert nc == len(xyz)
    if name in ("tenth", "jittered", "far_1e4"):
        assert 1 < nc < len(xyz)                               # the pair distances straddle the tolerance


def test_size_filter_fixture_against_brute_force(oracle):
    xyz = size_filter_cloud()
    ok = np.isfinite(xyz).all(1)
    n_ref, lab_ref = components_brute_force(xyz[ok], 0.05)
    labels, nc = oracle.euclidean_clusters(xyz, 0.05, min_size=1)
    assert nc == n_ref == 7 and same_partition(labels[ok], lab_ref)
    assert labels[0] == -1 and labels[-1] == -1
    assert sorted(np.bincount(labels[ok]).tolist()) == [1, 3, 5, 5, 7, 7, 7]


def test_helix_chain_is_one_component():
    tol = 0.01
    xyz = helix_chain(4000, tol).astype(np.float64)
    step = np.linalg.norm(np.diff(xyz, axis=0), axis=1)
    assert (step < 0.91 * tol).all() and (step > 0.89 * tol).all()
    skip = np.linalg.norm(xyz[2:] - xyz[:-2], axis=1)
    assert (skip > 1.7 * tol).all()
    n_ref, _ = components_brute_force(xyz[:1500].astype(np.float32), tol)
    assert n_ref == 1
    # the nearest point of the next turn is 5 tol away
    from scipy.spatial import cKDTree
    pairs = cKDTree(xyz).query_pairs(1.2 * tol, output_type="ndarray")
    assert (np.abs(pairs[:, 0] - pairs[:, 1]) == 1).all()


# ---- GPU helpers ------------------------------------------------------------------------------------------------------
def _on(a, kind):
    import torch
    if kind == "pageable":
        return a
    t = torch.from_numpy(np.ascontiguousarray(a, np.float32))
    if kind == "pinned":
        p = torch.empty(t.shape, dtype=torch.float32, pin_memory=True)
        p.copy_(t)
        return p
    assert kind == "device"
    return t.cuda()


def voxel_direct(eng, cloud, leaf, kind="pageable"):
    """gicpb_voxel_grid through ctypes into an output buffer of 0xFF bytes: (rc, n_out, out as uint32 [n, cols], error)"""
    import torch
    a = np.ascontiguousarray(cloud, np.float32)
    n, cols = a.shape
    src = _on(a, kind)
    if kind == "pageable":
        out = np.full((n, cols), 0xFFFFFFFF, np.uint32)
        iptr, optr, dev = a.ctypes.data, out.ctypes.data, 0
    else:
        out = torch.empty((n, cols), dtype=torch.int32, pin_memory=(kind == "pinned"),
                          device="cuda" if kind == "device" else "cpu")
        out.fill_(-1)
        torch.cuda.synchronize()
        iptr, optr, dev = src.data_ptr(), out.data_ptr(), int(kind == "device")
    m = ctypes.c_int64(-1)
    rc = eng.lib.gicpb_voxel_grid(eng.h, iptr, n, cols * 4, dev, float(leaf), optr, ctypes.byref(m))
    err = (eng.lib.gicpb_last_error(eng.h) or b"").decode()
    host = out if kind == "pageable" else out.cpu().numpy().view(np.uint32)
    return rc, int(m.value), host, err


def check_voxel(eng, oracle, cloud, leaf, kind="pageable"):
    """the engine's rows equal the oracle's over every byte; nothing past them is written; the warning exactly when
    the oracle refuses the leaf"""
    a = np.ascontiguousarray(cloud, np.float32)
    n, cols = a.shape
    ref = oracle.voxel_grid(a, leaf)
    rc, m, out, err = voxel_direct(eng, a, leaf, kind)
    assert rc == 0, err
    if m > 0 and ref is not None and m == len(ref):
        last = out[m - 1].view(np.uint8)
        assert np.array_equal(last, ref[-1].view(np.uint8)), f"last row, bytes {np.nonzero(last != ref[-1].view(np.uint8))[0]}"
    if ref is None:
        assert m == n and WARNING in err
        nbytes = (n - 1) * cols * 4 + (20 if cols >= 5 else 12)
        assert np.array_equal(out.reshape(-1).view(np.uint8)[:nbytes], a.reshape(-1).view(np.uint8)[:nbytes])
        return None
    assert m == len(ref), (m, len(ref), err)
    assert np.array_equal(out[:m], ref.view(np.uint32))
    assert (out[m:] == 0xFFFFFFFF).all()
    assert err == ""                                           # no warning left from an earlier call
    return ref


def check_clusters(eng, orc, xyz, tol, min_size=1, max_size=0, kind="pageable", cols=3):
    olab, onc = orc.euclidean_clusters(xyz, tol, min_size, max_size)
    lab, nc = eng.euclidean_clusters(_on(rows(xyz, cols), kind), tol, min_size, max_size)
    assert nc == onc
    assert np.array_equal(lab, olab)
    return lab, nc


# ---- GPU: voxel grid --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", overflow_cases(), ids=lambda c: c[0])
@pytest.mark.parametrize("cols", [3, 8])
def test_voxel_overflow_check_matches_pcl(engine, oracle, case, cols):
    name, xyz, leaf, refused = case
    ref = check_voxel(engine, oracle, rows(xyz, cols), leaf)
    assert (ref is None) == refused


@pytest.mark.gpu
@pytest.mark.parametrize("dims", [(3, 5, 17), (4, 8, 8), (257, 1, 1), (15, 17, 257), (16, 64, 64), (195, 21, 4097),
                                  (97, 257, 673)])
def test_voxel_totals_at_digit_boundaries(engine, oracle, dims):
    xyz = digit_cloud(dims, 300_000, sum(dims))
    check_voxel(engine, oracle, rows(xyz, 8), 1.0)


@pytest.mark.gpu
def test_voxel_8m_points_28_bit_keys(engine, oracle):
    n = 2048 * 4096 + 1000                                      # 2049 sort tiles
    xyz = digit_cloud((1024, 1024, 256), n, 28)
    with timed("voxel grid, 8.4 M points, 28-bit keys"):
        ref = check_voxel(engine, oracle, rows(xyz, 4), 1.0, kind="device")
    assert len(ref) > 7_000_000


@pytest.mark.gpu
@pytest.mark.parametrize("n_valid", [1, 2, 4095, 4096, 4097, 8193])
def test_voxel_valid_counts_at_tile_boundaries(engine, oracle, n_valid):
    rng = np.random.default_rng(n_valid)
    n = n_valid + 4096 + 7                                      # n and n_valid in different sort tiles
    xyz = (rng.random((n, 3)) * 3.0 - 1.0).astype(np.float32)
    bad = np.ones(n, bool)
    bad[np.sort(rng.choice(np.arange(1, n - 1), n_valid, replace=False))] = False
    xyz[bad & (np.arange(n) % 3 == 0), 0] = np.nan
    xyz[bad & (np.arange(n) % 3 == 1), 1] = np.inf
    xyz[bad & (np.arange(n) % 3 == 2), 2] = -np.inf
    assert bad[0] and bad[-1] and np.isfinite(xyz).all(1).sum() == n_valid
    for cols in (3, 8):
        check_voxel(engine, oracle, rows(xyz, cols), 0.2)


@pytest.mark.gpu
def test_voxel_special_clouds(engine, oracle):
    # all non-finite: no rows, no error
    nan = np.full((5000, 3), np.nan, np.float32)
    assert len(check_voxel(engine, oracle, rows(nan, 8), 0.1)) == 0
    # 2 M points in one voxel: the float sums in input order
    rng = np.random.default_rng(2)
    one = (0.1 + 0.8 * rng.random((2_000_000, 3))).astype(np.float32)
    with timed("voxel grid, 2 M points in one voxel"):
        assert len(check_voxel(engine, oracle, rows(one, 8), 1.0)) == 1
    # every point in its own voxel, shuffled
    own = lattice((64, 64, 16), 1.0)[rng.permutation(64 * 64 * 16)] + np.float32(0.5)
    assert len(check_voxel(engine, oracle, rows(own, 5), 1.0)) == len(own)
    # 10 k copies of one point
    same = np.tile(np.array([[0.3, -7.1, 2.2]], np.float32), (10_000, 1))
    assert len(check_voxel(engine, oracle, rows(same, 8), 0.05)) == 1
    # points exactly on voxel faces (k * leaf), negative coordinates and -0.0
    faces = lattice((17, 17, 17), 0.25, origin=(-2.0, -2.0, -2.0))
    faces = np.concatenate([faces, np.array([[-0.0, -0.0, -0.0], [0.0, -0.0, 0.0], [-0.0, 0.25, -0.25]], np.float32)])
    check_voxel(engine, oracle, rows(faces, 6), 0.25)
    check_voxel(engine, oracle, rows(faces, 6), 0.5)


@pytest.mark.gpu
@pytest.mark.parametrize("center", [(5e4, 1e4, 1e4), (2e5, 5e4, 1e4)])
def test_voxel_large_coordinates(engine, oracle, center):
    """1 cm voxels 50 km and 200 km out: x / leaf passes 2^24 in the second, where the float product rounds"""
    rng = np.random.default_rng(4)
    xyz = (np.asarray(center) + rng.random((200_000, 3)) * [5.0, 3.0, 1.0]).astype(np.float32)
    check_voxel(engine, oracle, rows(xyz, 8), 0.01)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["pageable", "pinned", "device"])
@pytest.mark.parametrize("cols", [3, 4, 5, 6, 8])
def test_voxel_strides_and_memory(engine, oracle, kind, cols):
    rng = np.random.default_rng(cols)
    xyz = (rng.random((50_000, 3)) * [2.0, 1.0, 0.5] - 0.7).astype(np.float32)
    xyz[[0, 777, 49_999], [0, 1, 2]] = [np.nan, np.inf, np.nan]
    check_voxel(engine, oracle, rows(xyz, cols), 0.05, kind)
    # the overflow window and the wrap through the same layout
    for name, p, leaf, _ in overflow_cases()[2:]:
        check_voxel(engine, oracle, rows(p, cols), leaf, kind)


# ---- GPU: clustering --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", lattice_cases(), ids=lambda c: c[0])
def test_clusters_at_lattice_distances(engine, oracle, case):
    name, xyz, tol = case
    check_clusters(engine, oracle, xyz, tol)
    far = engine.last_far_queries()
    # the brick grid's cell is the tolerance; the search box is widened by 4e-6 |x|, so at 1e4 m and 1 cm the box
    # passes kMaxBoxRows and the queries run through the hierarchical (far) search
    if name == "far_1e4_fine":
        assert far > 0
    if name in ("exact_s", "tenth", "far_1e3"):
        assert far == 0


@pytest.mark.gpu
def test_clusters_size_filter_at_cluster_sizes(engine, oracle):
    xyz = size_filter_cloud()
    for lo, hi in [(1, 0), (5, 5), (4, 5), (6, 6), (5, 7), (7, 7), (8, 0), (3, 4), (1, 1), (6, 8)]:
        for kind, cols in [("pageable", 3), ("pinned", 4), ("device", 8)]:
            lab, nc = check_clusters(engine, oracle, xyz, 0.05, lo, hi, kind, cols)
            assert lab[0] == -1 and lab[-1] == -1
    one = np.array([[1.0, 2.0, 3.0]], np.float32)
    for kind in ("pageable", "pinned", "device"):
        lab, nc = check_clusters(engine, oracle, one, 0.1, 1, 0, kind, 4)
        assert nc == 1 and lab.tolist() == [0]
        lab, nc = check_clusters(engine, oracle, one, 0.1, 2, 0, kind, 4)
        assert nc == 0 and lab.tolist() == [-1]


@pytest.mark.gpu
def test_clusters_giant_cluster_deterministic(engine, fast_oracle):
    """a 2.25 M-point panel joined into one cluster; three runs on one context give identical labels"""
    rng = np.random.default_rng(6)
    g = lattice((1500, 1500, 1), 0.01)
    g[:, 2] = rng.normal(0, 5e-4, len(g)).astype(np.float32)
    xyz = g[rng.permutation(len(g))]
    with timed("clusters, 2.25 M points, one cluster (oracle)"):
        olab, onc = fast_oracle.euclidean_clusters(xyz, 0.015, 1, 0)
    assert onc == 1
    runs = []
    with timed("clusters, 2.25 M points, one cluster (3 GPU runs)"):
        for _ in range(3):
            runs.append(engine.euclidean_clusters(xyz, 0.015, 1, 0))
    for lab, nc in runs:
        assert nc == onc and np.array_equal(lab, olab)


@pytest.mark.gpu
def test_clusters_helix_chain(engine, fast_oracle):
    xyz = helix_chain(1_000_000, 0.01)
    with timed("clusters, 1 M-point helix chain"):
        lab, nc = check_clusters(engine, fast_oracle, xyz, 0.01, kind="device")
    assert nc == 1 and (lab == 0).all()


@pytest.mark.gpu
def test_clusters_mostly_singletons(engine, fast_oracle):
    rng = np.random.default_rng(9)
    xyz = (rng.random((1_000_000, 3)) * 10.0).astype(np.float32)
    with timed("clusters, 1 M points, mostly singletons"):
        lab, nc = check_clusters(engine, fast_oracle, xyz, 0.01, kind="pinned")
    assert nc > 900_000


@pytest.mark.gpu
def test_clusters_config4_difference_cloud(engine, fast_oracle):
    """10 M scan + 20 FOD blobs minus the 10 M CAD cloud, then the clusters of what is left (th * 100)"""
    n = 10_000_000
    with timed("config 4 clouds (host)"):
        src, tgt, T_star = synth.make_pair(n, n, length=12.0, width=4.0)
        inp, _ = synth.add_fod_blobs(synth.apply_rigid(T_star, src).astype(np.float32), n_blobs=20, length=12.0,
                                     width=4.0)
    th = 4e-3 * 0.1
    with timed("config 4 difference + clusters"):
        mask, kept = engine.cloud_difference(inp, tgt, th)
        diff = np.ascontiguousarray(inp[mask.astype(bool)])
        lab, nc = check_clusters(engine, fast_oracle, diff, th * 100, 3, 0)
    assert nc >= 20


# ---- GPU: one context in sequence, and group members ------------------------------------------------------------------
@pytest.mark.gpu
def test_one_context_in_sequence(oracle, cube_pair):
    """voxel grids whose point count and key width grow, shrink and grow again across tile counts, with clustering
    and an align in between, on one context: the sorter reuses its status words and epochs"""
    from leica_point_cloud_processing_b200 import Engine
    from oracle.oracle import default_params
    eng = Engine(0)
    try:
        rng = np.random.default_rng(12)
        src, tgt, _ = cube_pair
        for k, (dims, n) in enumerate([((64, 64, 64), 300_000), ((16, 16, 1), 5_000), ((1024, 512, 512), 2_000_000),
                                       ((8, 4, 2), 1_000), ((257, 255, 64), 600_000)]):
            xyz = digit_cloud(dims, n, 100 + k)
            xyz[rng.integers(0, n, n // 50)] = np.nan
            check_voxel(eng, oracle, rows(xyz, 8), 1.0, kind="pageable" if k % 2 else "device")
            blobs = (rng.random((20_000, 3)) * (1 + k)).astype(np.float32)
            check_clusters(eng, oracle, blobs, 0.02 * (1 + k), 3, 0)
            if k == 2:
                eng.set_params(max_corr_distance=5.0, transformation_epsilon=5e-4)
                eng.set_target(tgt)
                eng.set_source(src)
                res = eng.align()
                ref = oracle.align(src, tgt, default_params(max_corr_distance=5.0, transformation_epsilon=5e-4))
                assert synth.rotation_error_rad(res["transform"], ref["T"]) < 1e-4
                assert synth.translation_error(res["transform"], ref["T"]) < 6e-5
    finally:
        eng.close()


@pytest.mark.gpu
def test_group_members_cluster_and_downsample(oracle):
    from leica_point_cloud_processing_b200 import EngineGroup
    s, t, T_star = synth.make_pair(60_000, 60_000)
    inp, _ = synth.add_fod_blobs(synth.apply_rigid(T_star, s).astype(np.float32), n_blobs=8, seed=5)
    grp = EngineGroup([0, 0])
    try:
        grp.set_params(max_corr_distance=1.0)
        grp.set_clouds(t, s)
        grp.align()
        mask, kept = grp.cloud_difference(inp, t, 4e-4)
        diff = np.ascontiguousarray(inp[mask.astype(bool)])
        rgb = rows(s, 8)
        for r in range(2):
            m = grp.member(r)
            check_clusters(m, oracle, diff, 4e-2, 3, 0)
            check_voxel(m, oracle, rgb, 0.05)
            ref = oracle.voxel_grid(rgb, 0.05)
            assert np.array_equal(m.voxel_grid(rgb, 0.05).view(np.uint32), ref.view(np.uint32))
    finally:
        grp.close()
