"""SURVEY section 8f rows 1 and 3: Euclidean clustering (FODDetector::clusterPossibleFODs) and the voxel-grid
downsample (Filter::downsampleCloud).

CPU part (-m "not gpu"): the oracle restatements of pcl::EuclideanClusterExtraction / pcl::VoxelGrid against the
reference's own test fixtures (test/test_fod_detector.cpp, test/test_filter.cpp) and independent numpy / scipy checks.
GPU part (-m gpu): the CUDA path through the C ABI against the oracle: cluster label arrays identical, voxel
centroids bit-exact.
"""
import numpy as np
import pytest

from leica_point_cloud_processing_b200 import synth


# ---- fixtures of the reference's own tests ---------------------------------------------------------------------------
def cubes_point_cloud(pos, dim, step):
    """test/test_fod_detector.cpp:32-47 cubesPointCloud: float loop counters, i += step in float."""
    axis = []
    v = np.float32(pos)
    end = np.float32(np.float32(pos) + np.float32(dim))
    while v < end:
        axis.append(v)
        v = np.float32(v + np.float32(step))
    a = np.array(axis, np.float32)
    g = np.stack(np.meshgrid(a, a, a, indexing="ij"), axis=-1).reshape(-1, 3)
    return np.ascontiguousarray(g, dtype=np.float32)


def fod_fixture():
    """TEST_F(TestFODDetector, testFODClustering): three cubes at 0, 10, 20 (side 3, step 0.1)."""
    return np.concatenate([cubes_point_cloud(0, 3, 0.1), cubes_point_cloud(10, 3, 0.1), cubes_point_cloud(20, 3, 0.1)])


def plane_fixture(dim=3):
    """test/test_filter.cpp:48-66: white points on z = 0, 0.1 apart (float loop counters); PointXYZRGB rows."""
    axis = []
    v = np.float32(0)
    while v < np.float32(dim):
        axis.append(v)
        v = np.float32(v + np.float32(0.1))
    a = np.array(axis, np.float32)
    xy = np.stack(np.meshgrid(a, a, indexing="ij"), axis=-1).reshape(-1, 2)
    c = np.zeros((len(xy), 8), np.float32)
    c[:, :2] = xy
    c[:, 3] = 1.0
    c[:, 4] = np.array([0xFFFFFFFF], np.uint32).view(np.float32)[0]  # r = g = b = 255 (a defaults to 255)
    return c


def xyzrgb(xyz, rng):
    c = np.zeros((len(xyz), 8), np.float32)
    c[:, :3] = xyz
    c[:, 3] = 1.0
    c[:, 4] = rng.integers(0, 2 ** 32, len(xyz), dtype=np.uint64).astype(np.uint32).view(np.float32)
    return c


def components_brute_force(xyz, tol):
    """connected components of the d2 < float(tol^2) graph with float32 distances accumulated as FLANN does"""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components
    x = xyz.astype(np.float32)
    d = x[:, None, :] - x[None, :, :]
    d2 = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
    adj = d2 < np.float32(tol * tol)
    n, lab = connected_components(coo_matrix(adj), directed=False)
    return n, lab


def same_partition(a, b):
    """two label arrays describe the same set of clusters"""
    pairs = set(zip(a.tolist(), b.tolist()))
    return len(pairs) == len(set(a.tolist())) == len(set(b.tolist()))


# ---- CPU: the oracle --------------------------------------------------------------------------------------------------
def test_oracle_clusters_reference_fixture(oracle):
    cloud = fod_fixture()
    th = 4e-3 * 3
    labels, nc = oracle.euclidean_clusters(cloud, th * 10, min_size=3)
    assert nc == 3                                      # ASSERT_EQ(num_of_fods, 3)
    assert (labels >= 0).all()
    sizes = np.bincount(labels)
    assert sorted(sizes.tolist(), reverse=True) == sizes.tolist()   # extract(): largest cluster first
    assert same_partition(labels, (cloud[:, 0] // 5).astype(np.int32))
    l0, n0 = oracle.euclidean_clusters(np.zeros((0, 3), np.float32), th * 10, min_size=3)
    assert n0 == 0 and len(l0) == 0                     # TEST_F(TestFODDetector, testEmptyCloud)


@pytest.mark.parametrize("seed,tol", [(1, 0.05), (2, 0.11), (3, 0.3)])
def test_oracle_clusters_equal_connected_components(oracle, seed, tol):
    rng = np.random.default_rng(seed)
    xyz = rng.random((1500, 3)).astype(np.float32)
    labels, nc = oracle.euclidean_clusters(xyz, tol, min_size=1)
    n_ref, lab_ref = components_brute_force(xyz, tol)
    assert nc == n_ref and same_partition(labels, lab_ref)
    # the size filter drops whole clusters and keeps the order of the rest
    lab4, nc4 = oracle.euclidean_clusters(xyz, tol, min_size=4, max_size=50)
    sizes = np.bincount(labels)
    kept = [k for k in range(nc) if 4 <= sizes[k] <= 50]
    assert nc4 == len(kept)
    remap = {k: r for r, k in enumerate(kept)}
    assert np.array_equal(lab4, np.array([remap.get(l, -1) for l in labels], np.int32))


def test_oracle_voxel_grid_reference_fixture(oracle):
    cloud = plane_fixture()
    res = oracle.resolution(cloud[:, :3])
    out = oracle.voxel_grid(cloud, np.float32(2 * res))
    assert 0 < len(out) < len(cloud)
    assert oracle.resolution(out[:, :3]) > res          # EXPECT_GT(end_res, res)
    assert (out[:, 3] == 1.0).all() and (out[:, 4].view(np.uint32) == 0xFFFFFFFF).all() and (out[:, 5:] == 0).all()


def test_oracle_voxel_grid_against_numpy(oracle):
    rng = np.random.default_rng(5)
    cloud = xyzrgb((rng.random((4000, 3)) * [2.0, 1.0, 0.5] - 0.7).astype(np.float32), rng)
    cloud[17, 0] = np.nan
    leaf = np.float32(0.13)
    out = oracle.voxel_grid(cloud, leaf)
    ok = np.isfinite(cloud[:, :3]).all(1)
    p = cloud[ok]
    inv = np.float32(1.0) / leaf
    ijk = np.floor(p[:, :3] * inv).astype(np.int64)
    ijk -= np.floor(p[:, :3].min(0) * inv).astype(np.int64)
    div = ijk.max(0) + 1
    idx = ijk[:, 0] + ijk[:, 1] * div[0] + ijk[:, 2] * div[0] * div[1]
    order = np.argsort(idx, kind="stable")
    uniq, start, count = np.unique(idx[order], return_index=True, return_counts=True)
    assert len(out) == len(uniq)
    for v in (0, len(uniq) // 2, len(uniq) - 1):
        rows = p[order[start[v]:start[v] + count[v]]]
        s = np.zeros(3, np.float32)
        for r in rows:
            s = (s + r[:3]).astype(np.float32)
        assert np.array_equal(out[v, :3], (s / np.float32(count[v])).astype(np.float32))
        rgba = rows[:, 4].view(np.uint32)
        want = 0
        for shift in (24, 16, 8, 0):
            want |= int(np.float32(((rgba >> shift) & 255).astype(np.float32).sum()) / np.float32(count[v])) << shift
        assert int(out[v, 4].view(np.uint32)) == want
    # every centroid lies in its voxel; the point count is conserved
    assert np.allclose((out[:, :3].astype(np.float64) * count[:, None]).sum(0), p[:, :3].astype(np.float64).sum(0), rtol=1e-5)
    assert oracle.voxel_grid(cloud, 1e-4) is None       # "Leaf size is too small for the input dataset"


# ---- GPU: the CUDA path against the oracle ----------------------------------------------------------------------------
@pytest.mark.gpu
def test_reference_testFODClustering(engine, oracle):
    """test/test_fod_detector.cpp:52-72 and :75-90 through the Python mirror of FODDetector."""
    from leica_point_cloud_processing_b200 import FODDetector
    cloud = fod_fixture()
    th = 4e-3 * 3
    det = FODDetector(cloud, th * 10, 3, engine=engine)
    det.clusterPossibleFODs()
    fods = []
    assert det.fodIndicesToPointCloud(fods) == 3 and len(fods) == 3
    labels, nc = oracle.euclidean_clusters(cloud, th * 10, min_size=3)
    for k, idx in enumerate(det.getFODIndices()):
        assert np.array_equal(idx, np.nonzero(labels == k)[0])     # PointIndices of cluster k, ascending
        assert np.array_equal(fods[k], cloud[idx])
    empty = FODDetector(np.zeros((0, 3), np.float32), th * 10, 3, engine=engine)
    empty.clusterPossibleFODs()
    fods = []
    assert empty.fodIndicesToPointCloud(fods) == 0 and fods == []
    assert FODDetector(cloud, 0, 3, engine=engine).cluster_tolerance_ == 4e-3   # src/FODDetector.cpp:30-34


@pytest.mark.gpu
@pytest.mark.parametrize("seed,n,tol,min_size,max_size", [
    (1, 20000, 0.02, 1, 0),        # sparse: mostly singletons
    (2, 20000, 0.05, 3, 0),        # mixed
    (3, 20000, 0.05, 3, 40),       # upper size limit
    (4, 3000, 0.6, 1, 0),          # tolerance >> spacing: one cluster (the cell is never smaller than the tolerance,
                                   # so each ball spans a few cells: near search only; the far search runs where
                                   # the box margin grows with |x|, see test_segment_edges.py)
])
def test_clusters_match_oracle_random(engine, oracle, seed, n, tol, min_size, max_size):
    rng = np.random.default_rng(seed)
    xyz = rng.random((n, 3)).astype(np.float32)
    xyz[5] = np.nan                                      # a non-finite point is in no cluster
    xyz[9] = xyz[8]                                      # duplicates
    labels, nc = engine.euclidean_clusters(xyz, tol, min_size, max_size)
    olab, onc = oracle.euclidean_clusters(xyz, tol, min_size, max_size)
    assert nc == onc
    assert np.array_equal(labels, olab)
    assert labels[5] == -1


@pytest.mark.gpu
def test_clusters_on_the_fod_difference_cloud(engine, oracle):
    """The pipeline step of src/LeicaStateMachine.cpp:185-205: difference cloud -> clusters (tolerance th * 100)."""
    n = 200_000
    src, tgt, T_star = synth.make_pair(n, n)
    aligned = synth.apply_rigid(T_star, src)
    cloud, _ = synth.add_fod_blobs(aligned, n_blobs=8, seed=999)
    th = 4e-3 * 0.1
    mask, kept = engine.cloud_difference(cloud, tgt, th)
    diff = cloud[mask.astype(bool)]
    labels, nc = engine.euclidean_clusters(diff, th * 100, 3, 0)
    olab, onc = oracle.euclidean_clusters(diff, th * 100, 3, 0)
    assert nc == onc and nc >= 1
    assert np.array_equal(labels, olab)


@pytest.mark.gpu
def test_reference_testDownsample(engine, oracle):
    """test/test_filter.cpp:68-83 through downsample_cloud (Filter::downsampleCloud)."""
    from leica_point_cloud_processing_b200 import downsample_cloud
    cloud = plane_fixture()
    engine.set_target(cloud)
    res = engine.cloud_resolution(0)
    out = downsample_cloud(cloud, np.float32(2 * res), engine=engine)
    engine.set_target(out)
    assert engine.cloud_resolution(0) > res              # EXPECT_GT(end_res, res)
    ref = oracle.voxel_grid(cloud, np.float32(2 * res))
    assert out.shape == ref.shape and np.array_equal(out.view(np.uint32), ref.view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("cols", [3, 4, 8])
@pytest.mark.parametrize("leaf", [0.013, 0.13, 5.0])
def test_voxel_grid_bit_exact(engine, oracle, cols, leaf):
    rng = np.random.default_rng(11)
    xyz = (rng.random((50_000, 3)) * [2.0, 1.0, 0.5] - 0.7).astype(np.float32)
    cloud = xyzrgb(xyz, rng)[:, :cols].copy()
    if cols == 4:
        cloud[:, 3] = 1.0
    cloud[123, 1] = np.inf
    out = engine.voxel_grid(cloud, leaf)
    ref = oracle.voxel_grid(cloud, leaf)
    assert out.shape == ref.shape
    assert np.array_equal(out.view(np.uint32), ref.view(np.uint32))


@pytest.mark.gpu
def test_voxel_grid_panel_and_device_clouds(engine, oracle):
    import torch
    src, tgt, _ = synth.make_pair(300_000, 1000)
    engine.set_target(src)
    leaf = 10 * engine.cloud_resolution(0)               # src/LeicaStateMachine.cpp:61-65 leaf_size_factor = 10
    ref = oracle.voxel_grid(src, leaf)
    out = engine.voxel_grid(src, leaf)
    assert np.array_equal(out.view(np.uint32), ref.view(np.uint32))
    d_out = engine.voxel_grid(torch.from_numpy(src).cuda(), leaf)
    assert np.array_equal(d_out.cpu().numpy().view(np.uint32), ref.view(np.uint32))
    # leaf too small for 32-bit voxel indices: PCL warns and passes the input through
    same = engine.voxel_grid(src, 1e-4)
    assert oracle.voxel_grid(src, 1e-4) is None
    assert np.array_equal(same.view(np.uint32), src.view(np.uint32))
