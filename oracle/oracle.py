"""ctypes loader for the CPU oracle (oracle/gicp_oracle.cpp).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs.  The shipped package never imports this module.
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))

c_float_p = ctypes.POINTER(ctypes.c_float)
c_double_p = ctypes.POINTER(ctypes.c_double)
c_int_p = ctypes.POINTER(ctypes.c_int)
c_ubyte_p = ctypes.POINTER(ctypes.c_ubyte)


class OrcParams(ctypes.Structure):
    _fields_ = [
        ("max_iterations", ctypes.c_int),
        ("transformation_epsilon", ctypes.c_double),
        ("rotation_epsilon", ctypes.c_double),
        ("max_corr_distance", ctypes.c_double),
        ("k_correspondences", ctypes.c_int),
        ("gicp_epsilon", ctypes.c_double),
        ("max_inner_iterations", ctypes.c_int),
    ]


class OrcResult(ctypes.Structure):
    _fields_ = [
        ("T", ctypes.c_float * 16),
        ("converged", ctypes.c_int),
        ("outer_iterations", ctypes.c_int),
        ("n_f", ctypes.c_long),
        ("n_df", ctypes.c_long),
        ("n_fdf", ctypes.c_long),
        ("n_corr_queries", ctypes.c_long),
        ("n_pairs_last", ctypes.c_long),
        ("t_cov_s", ctypes.c_double),
        ("t_corr_s", ctypes.c_double),
        ("t_opt_s", ctypes.c_double),
        ("t_tree_s", ctypes.c_double),
    ]


def default_params(**kw):
    """Reference defaults: src/GICPAlignment.cpp:29-32 over PCL 1.8.1 gicp.h defaults."""
    p = OrcParams(100, 4e-3, 2e-3, 4e-2, 20, 1e-3, 20)
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def build(force=False):
    libs = [os.path.join(_HERE, n) for n in ("liboracle.so", "liboracle_fast.so")]
    src = os.path.join(_HERE, "gicp_oracle.cpp")
    stale = force or any((not os.path.exists(l)) or os.path.getmtime(l) < os.path.getmtime(src) for l in libs)
    if stale:
        subprocess.check_call(["make", "-C", _HERE, "-B"], stdout=subprocess.DEVNULL)
    return libs


def _f32(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    return a


def _xyz(a):
    a = _f32(a)
    assert a.ndim == 2 and a.shape[1] == 3, a.shape
    return a


def _p(a, t):
    return a.ctypes.data_as(t)


class Oracle:
    """fast=False: parity build (1 thread, -ffp-contract=off).  fast=True: -O3 + OpenMP timing build."""

    def __init__(self, fast=False):
        libs = build()
        self.lib = ctypes.CDLL(libs[1] if fast else libs[0])
        L = self.lib
        L.orc_num_threads.restype = ctypes.c_int
        L.orc_fitness.restype = ctypes.c_double
        L.orc_resolution.restype = ctypes.c_double
        L.orc_fitness.argtypes = [c_float_p, ctypes.c_int, c_float_p, ctypes.c_int, c_float_p, ctypes.c_double]
        L.orc_difference.argtypes = [c_float_p, ctypes.c_int, c_float_p, ctypes.c_int, ctypes.c_double, c_ubyte_p]
        L.orc_resolution.argtypes = [c_float_p, ctypes.c_int]
        L.orc_sample_mesh.argtypes = [c_float_p, ctypes.c_int, c_int_p, ctypes.c_int, ctypes.c_int, ctypes.c_long,
                                      c_float_p]
        L.orc_rotation_rpy.argtypes = [ctypes.c_double, ctypes.c_double, ctypes.c_double, c_float_p]
        L.orc_transform.argtypes = [c_float_p, c_float_p, ctypes.c_int, c_float_p]
        L.orc_apply_state.argtypes = [c_double_p, c_float_p]
        L.orc_nn1.argtypes = [c_float_p, ctypes.c_int, c_float_p, ctypes.c_int, ctypes.c_int, c_int_p, c_float_p]
        L.orc_knn.argtypes = [c_float_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_int_p, c_float_p]
        L.orc_covariances.argtypes = [c_float_p, ctypes.c_int, ctypes.c_int, ctypes.c_double, c_double_p]
        L.orc_cost.argtypes = [c_float_p, c_float_p, c_int_p, c_int_p, ctypes.c_int, c_double_p, ctypes.c_int,
                               c_double_p, c_double_p, c_double_p]
        L.orc_correspondences.argtypes = [c_float_p, ctypes.c_int, c_float_p, ctypes.c_int, c_double_p, c_double_p,
                                          c_float_p, ctypes.c_double, c_int_p, c_float_p, c_double_p]
        L.orc_correspondences.restype = ctypes.c_int
        L.orc_gicp_align.argtypes = [c_float_p, ctypes.c_int, c_float_p, ctypes.c_int, ctypes.POINTER(OrcParams),
                                     ctypes.c_int, ctypes.POINTER(OrcResult)]

    def num_threads(self):
        return int(self.lib.orc_num_threads())

    # ---- fixtures -------------------------------------------------------------------------------
    def sample_mesh(self, verts, faces, n, skip_draws=0):
        verts = _f32(verts)
        faces = np.ascontiguousarray(faces, dtype=np.int32)
        out = np.empty((n, 3), np.float32)
        self.lib.orc_sample_mesh(_p(verts, c_float_p), len(verts), _p(faces, c_int_p), len(faces), n, skip_draws,
                                 _p(out, c_float_p))
        return out

    def rotation_rpy(self, roll, pitch, yaw):
        T = np.empty((4, 4), np.float32)
        self.lib.orc_rotation_rpy(roll, pitch, yaw, _p(T, c_float_p))
        return T

    def transform(self, T, xyz):
        T = _f32(T).reshape(4, 4)
        xyz = _xyz(xyz)
        out = np.empty_like(xyz)
        self.lib.orc_transform(_p(T, c_float_p), _p(xyz, c_float_p), len(xyz), _p(out, c_float_p))
        return out

    def apply_state(self, x6):
        x = np.ascontiguousarray(x6, np.float64)
        T = np.empty((4, 4), np.float32)
        self.lib.orc_apply_state(_p(x, c_double_p), _p(T, c_float_p))
        return T

    # ---- searches -------------------------------------------------------------------------------
    def nn1(self, tgt, qry, use_tree=True):
        tgt, qry = _xyz(tgt), _xyz(qry)
        idx = np.empty(len(qry), np.int32)
        d2 = np.empty(len(qry), np.float32)
        self.lib.orc_nn1(_p(tgt, c_float_p), len(tgt), _p(qry, c_float_p), len(qry), int(use_tree), _p(idx, c_int_p),
                         _p(d2, c_float_p))
        return idx, d2

    def knn(self, xyz, k, use_tree=True):
        xyz = _xyz(xyz)
        idx = np.empty((len(xyz), k), np.int32)
        d2 = np.empty((len(xyz), k), np.float32)
        self.lib.orc_knn(_p(xyz, c_float_p), len(xyz), k, int(use_tree), _p(idx, c_int_p), _p(d2, c_float_p))
        return idx, d2

    def covariances(self, xyz, k=20, eps=1e-3):
        xyz = _xyz(xyz)
        cov = np.empty((len(xyz), 3, 3), np.float64)
        rc = self.lib.orc_covariances(_p(xyz, c_float_p), len(xyz), k, eps, _p(cov, c_double_p))
        if rc != 0:
            raise RuntimeError("orc_covariances: k > n")
        return cov

    # ---- GICP pieces ----------------------------------------------------------------------------
    def cost(self, src, tgt, isrc, itgt, maha, x6):
        src, tgt = _xyz(src), _xyz(tgt)
        isrc = np.ascontiguousarray(isrc, np.int32)
        itgt = np.ascontiguousarray(itgt, np.int32)
        maha = np.ascontiguousarray(maha, np.float64)
        x = np.ascontiguousarray(x6, np.float64)
        f = ctypes.c_double()
        g = np.empty(6, np.float64)
        self.lib.orc_cost(_p(src, c_float_p), _p(tgt, c_float_p), _p(isrc, c_int_p), _p(itgt, c_int_p), len(isrc),
                          _p(maha, c_double_p), len(src), _p(x, c_double_p), ctypes.byref(f), _p(g, c_double_p))
        return f.value, g

    def correspondences(self, src, tgt, cov_src, cov_tgt, T, max_corr_distance):
        src, tgt = _xyz(src), _xyz(tgt)
        cov_src = np.ascontiguousarray(cov_src, np.float64)
        cov_tgt = np.ascontiguousarray(cov_tgt, np.float64)
        T = _f32(T).reshape(4, 4)
        idx = np.empty(len(src), np.int32)
        d2 = np.empty(len(src), np.float32)
        maha = np.empty((len(src), 3, 3), np.float64)
        cnt = self.lib.orc_correspondences(_p(src, c_float_p), len(src), _p(tgt, c_float_p), len(tgt),
                                           _p(cov_src, c_double_p), _p(cov_tgt, c_double_p), _p(T, c_float_p),
                                           max_corr_distance, _p(idx, c_int_p), _p(d2, c_float_p),
                                           _p(maha, c_double_p))
        return cnt, idx, d2, maha

    def align(self, src, tgt, params=None, max_outer=0):
        src, tgt = _xyz(src), _xyz(tgt)
        params = params or default_params()
        res = OrcResult()
        rc = self.lib.orc_gicp_align(_p(src, c_float_p), len(src), _p(tgt, c_float_p), len(tgt),
                                     ctypes.byref(params), max_outer, ctypes.byref(res))
        out = {k: getattr(res, k) for k, _ in OrcResult._fields_ if k != "T"}
        out["T"] = np.array(res.T, np.float32).reshape(4, 4)
        out["rc"] = rc
        return out

    def fitness(self, src, tgt, T, max_range=float(np.finfo(np.float64).max)):
        src, tgt = _xyz(src), _xyz(tgt)
        T = _f32(T).reshape(4, 4)
        return float(self.lib.orc_fitness(_p(src, c_float_p), len(src), _p(tgt, c_float_p), len(tgt),
                                          _p(T, c_float_p), max_range))

    def difference(self, inp, sub, threshold):
        inp, sub = _xyz(inp), _xyz(sub)
        mask = np.empty(len(inp), np.uint8)
        kept = self.lib.orc_difference(_p(inp, c_float_p), len(inp), _p(sub, c_float_p), len(sub), threshold,
                                       _p(mask, c_ubyte_p))
        return mask, int(kept)

    def normal_validity(self, xyz, radius):
        """mask[i] = 1 iff Utils::getNormals gives point i a finite normal (>= 3 points inside the radius); (mask, count)"""
        a = _xyz(xyz)
        mask = np.zeros(len(a), np.uint8)
        self.lib.orc_normal_validity.restype = ctypes.c_int
        n = self.lib.orc_normal_validity(_p(a, c_float_p), ctypes.c_int(len(a)), ctypes.c_double(radius),
                                         _p(mask, c_ubyte_p))
        return mask, int(n)

    def normals(self, xyz, radius):
        """Utils::getNormals: float32 [n, 4] (nx, ny, nz, curvature; NaN where PCL gives no normal) and the finite count"""
        a = _xyz(xyz)
        out = np.empty((len(a), 4), np.float32)
        self.lib.orc_normals.restype = ctypes.c_int
        n = self.lib.orc_normals(_p(a, c_float_p), ctypes.c_int(len(a)), ctypes.c_double(radius), _p(out, c_float_p))
        return out, int(n)

    def normals_ex(self, xyz, radius):
        """normals() plus float64 [n, 4] info per point: neighbour count; branch (0 no normal: non-finite point or < 3
        neighbours, 1 zero covariance, 2 pcl::eigen33's c0 < eps -> roots2, 3 trigonometric roots, 4 trigonometric roots
        then the roots2 fallback); root gap roots[1] - roots[0] of the scaled matrix; cos_theta of the viewpoint flip.
        Returns (rows, info, finite count); the rows are the rows normals() gives."""
        a = _xyz(xyz)
        out = np.empty((len(a), 4), np.float32)
        info = np.empty((len(a), 4), np.float64)
        self.lib.orc_normals_ex.restype = ctypes.c_int
        n = self.lib.orc_normals_ex(_p(a, c_float_p), ctypes.c_int(len(a)), ctypes.c_double(radius), _p(out, c_float_p),
                                    _p(info, c_double_p))
        return out, info, int(n)

    def euclidean_clusters(self, xyz, tolerance, min_size=1, max_size=0):
        """pcl::EuclideanClusterExtraction::extract: (labels in PCL's cluster order, -1 = none; n_clusters)"""
        a = _xyz(xyz) if len(xyz) else np.zeros((0, 3), np.float32)
        labels = np.full(len(a), -1, np.int32)
        self.lib.orc_euclidean_clusters.restype = ctypes.c_int
        nc = self.lib.orc_euclidean_clusters(_p(a, c_float_p), ctypes.c_int(len(a)), ctypes.c_double(tolerance),
                                             ctypes.c_int(int(min_size)), ctypes.c_int(int(max_size)), _p(labels, c_int_p))
        return labels, int(nc)

    def voxel_grid(self, cloud, leaf_size):
        """pcl::VoxelGrid on a float32 [n, 3|4|8] array (8 = PointXYZRGB layout); None when PCL would refuse the leaf"""
        a = np.ascontiguousarray(cloud, dtype=np.float32)
        stride = a.shape[1] * 4
        out = np.zeros_like(a)
        self.lib.orc_voxel_grid.restype = ctypes.c_int64
        m = self.lib.orc_voxel_grid(ctypes.c_void_p(a.ctypes.data), ctypes.c_int64(len(a)), ctypes.c_int64(stride),
                                    ctypes.c_double(leaf_size), ctypes.c_void_p(out.ctypes.data))
        return None if m < 0 else out[: int(m)]

    def resolution(self, xyz):
        xyz = _xyz(xyz)
        return float(self.lib.orc_resolution(_p(xyz, c_float_p), len(xyz)))
