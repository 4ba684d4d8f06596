"""ctypes binding of libgicp_b200.so (C ABI declared in include/gicp_b200.h).

There is no CPU fallback: if the shared library is missing, or no sm_100 GPU is usable, loading / creating a
context raises.  PyTorch is not needed by this module; tensors can be passed by device pointer.
"""
import ctypes
import os

import numpy as np

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG_DIR, "libgicp_b200.so")

GICPB_OK = 0
E_BADARG, E_CUDA, E_NCCL, E_NOT_ENOUGH_CORRESPONDENCES, E_SOLVER, E_STATE, E_TOO_FEW_POINTS = -1, -2, -3, -4, -5, -6, -7

c_float_p = ctypes.POINTER(ctypes.c_float)
c_double_p = ctypes.POINTER(ctypes.c_double)
c_int32_p = ctypes.POINTER(ctypes.c_int32)
c_int64_p = ctypes.POINTER(ctypes.c_int64)
c_uint8_p = ctypes.POINTER(ctypes.c_uint8)


class Params(ctypes.Structure):
    """gicpb_params; defaults = reference src/GICPAlignment.cpp:29-32 over PCL 1.8.1 gicp.h defaults."""
    _fields_ = [
        ("max_iterations", ctypes.c_int),
        ("transformation_epsilon", ctypes.c_double),
        ("rotation_epsilon", ctypes.c_double),
        ("max_corr_distance", ctypes.c_double),
        ("k_correspondences", ctypes.c_int),
        ("gicp_epsilon", ctypes.c_double),
        ("max_inner_iterations", ctypes.c_int),
        ("cell_size", ctypes.c_float),
        ("points_per_cell", ctypes.c_float),
        ("mahalanobis_fp32", ctypes.c_int),
        ("use_previous_match", ctypes.c_int),
        ("l2_persist", ctypes.c_int),
        ("cost_moments", ctypes.c_int),
        ("cost_persistent", ctypes.c_int),
    ]


class AlignResult(ctypes.Structure):
    _fields_ = [
        ("transform", ctypes.c_float * 16),
        ("converged", ctypes.c_int),
        ("status", ctypes.c_int),
        ("outer_iterations", ctypes.c_int),
        ("inner_iterations", ctypes.c_int),
        ("cost_evaluations", ctypes.c_int64),
        ("corr_queries", ctypes.c_int64),
        ("corr_pairs_last", ctypes.c_int64),
        ("corr_far_queries", ctypes.c_int64),
        ("ms_total", ctypes.c_double),
        ("ms_corr", ctypes.c_double),
        ("ms_cost", ctypes.c_double),
    ]


class GridInfo(ctypes.Structure):
    _fields_ = [
        ("n_points", ctypes.c_int64),
        ("n_indexed", ctypes.c_int64),
        ("cell_size", ctypes.c_float),
        ("dims", ctypes.c_int * 3),
        ("n_bricks_occupied", ctypes.c_int64),
        ("n_cells_occupied", ctypes.c_int64),
        ("ms_build", ctypes.c_double),
    ]


class CostSessionInfo(ctypes.Structure):
    _fields_ = [
        ("persistent", ctypes.c_int),
        ("blocks", ctypes.c_int),
        ("threads", ctypes.c_int),
        ("stages", ctypes.c_int),
        ("pairs_per_block", ctypes.c_int),
        ("resident_cap", ctypes.c_int),
        ("resident", ctypes.c_int),
        ("epoch_first", ctypes.c_int),
        ("epoch_last", ctypes.c_int),
        ("launches", ctypes.c_int64),
        ("n_pairs", ctypes.c_int64),
    ]


class Pc2Layout(ctypes.Structure):
    """gicpb_pc2_layout: where a sensor_msgs/PointCloud2 payload keeps the fields a pcl::PointXYZRGB maps."""
    _fields_ = [
        ("width", ctypes.c_int64),
        ("height", ctypes.c_int64),
        ("point_step", ctypes.c_int64),
        ("row_step", ctypes.c_int64),
        ("off_x", ctypes.c_int32),
        ("off_y", ctypes.c_int32),
        ("off_z", ctypes.c_int32),
        ("off_rgb", ctypes.c_int32),
    ]


class PcdInfo(ctypes.Structure):
    _fields_ = [
        ("width", ctypes.c_int64),
        ("height", ctypes.c_int64),
        ("points", ctypes.c_int64),
        ("point_step", ctypes.c_int32),
        ("n_fields", ctypes.c_int32),
        ("data_kind", ctypes.c_int32),
        ("is_dense", ctypes.c_int32),
        ("off_x", ctypes.c_int32),
        ("off_y", ctypes.c_int32),
        ("off_z", ctypes.c_int32),
        ("off_rgb", ctypes.c_int32),
    ]


# every symbol include/gicp_b200.h declares: (name, restype, argtypes)
_VOID_P = ctypes.c_void_p
_SIGNATURES = [
    ("gicpb_default_params", None, [ctypes.POINTER(Params)]),
    ("gicpb_create", ctypes.c_int, [ctypes.c_int, ctypes.POINTER(_VOID_P)]),
    ("gicpb_destroy", None, [_VOID_P]),
    ("gicpb_last_error", ctypes.c_char_p, [_VOID_P]),
    ("gicpb_set_params", ctypes.c_int, [_VOID_P, ctypes.POINTER(Params)]),
    ("gicpb_get_params", ctypes.c_int, [_VOID_P, ctypes.POINTER(Params)]),
    ("gicpb_nccl_unique_id", ctypes.c_int, [ctypes.c_char_p, c_uint8_p]),
    ("gicpb_comm_init", ctypes.c_int, [_VOID_P, ctypes.c_char_p, ctypes.c_int, ctypes.c_int, c_uint8_p]),
    ("gicpb_comm_rank", ctypes.c_int, [_VOID_P, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]),
    ("gicpb_shard_info", ctypes.c_int, [_VOID_P, c_int64_p, c_int64_p, c_int64_p, c_int64_p]),
    ("gicpb_peer_export", ctypes.c_int, [_VOID_P, c_uint8_p]),
    ("gicpb_peer_import", ctypes.c_int, [_VOID_P, c_uint8_p, ctypes.c_int]),
    ("gicpb_peer_disable", ctypes.c_int, [_VOID_P]),
    ("gicpb_prefetch_cloud", ctypes.c_int, [_VOID_P, ctypes.c_int, _VOID_P, ctypes.c_int64, ctypes.c_int64]),
    ("gicpb_set_target", ctypes.c_int, [_VOID_P, _VOID_P, ctypes.c_int64, ctypes.c_int64, ctypes.c_int]),
    ("gicpb_set_source", ctypes.c_int, [_VOID_P, _VOID_P, ctypes.c_int64, ctypes.c_int64, ctypes.c_int]),
    ("gicpb_set_clouds", ctypes.c_int, [_VOID_P, _VOID_P, ctypes.c_int64, ctypes.c_int64, _VOID_P, ctypes.c_int64,
                                        ctypes.c_int64, ctypes.c_int]),
    ("gicpb_compute_covariances", ctypes.c_int, [_VOID_P]),
    ("gicpb_align", ctypes.c_int, [_VOID_P, ctypes.POINTER(AlignResult)]),
    ("gicpb_fitness", ctypes.c_int, [_VOID_P, c_float_p, ctypes.c_double, c_double_p]),
    ("gicpb_transform_cloud", ctypes.c_int, [_VOID_P, c_float_p, _VOID_P, _VOID_P, ctypes.c_int64, ctypes.c_int64,
                                             ctypes.c_int]),
    ("gicpb_cloud_difference", ctypes.c_int, [_VOID_P, _VOID_P, ctypes.c_int64, ctypes.c_int64, _VOID_P, ctypes.c_int64,
                                              ctypes.c_int64, ctypes.c_int, ctypes.c_double, _VOID_P, c_int64_p]),
    ("gicpb_difference_set_subtract", ctypes.c_int, [_VOID_P, _VOID_P, ctypes.c_int64, ctypes.c_int64, ctypes.c_int]),
    ("gicpb_difference_run", ctypes.c_int, [_VOID_P, _VOID_P, ctypes.c_int64, ctypes.c_int64, ctypes.c_int,
                                            ctypes.c_double, _VOID_P, ctypes.c_int, c_int64_p]),
    ("gicpb_nn1", ctypes.c_int, [_VOID_P, _VOID_P, ctypes.c_int64, ctypes.c_int64, ctypes.c_int, c_float_p,
                                 ctypes.c_double, c_int32_p, c_float_p]),
    ("gicpb_knn", ctypes.c_int, [_VOID_P, ctypes.c_int, c_int32_p, c_float_p]),
    ("gicpb_get_covariances", ctypes.c_int, [_VOID_P, ctypes.c_int, c_double_p]),
    ("gicpb_correspondences", ctypes.c_int, [_VOID_P, c_float_p, c_int32_p, c_float_p, c_double_p, c_int64_p]),
    ("gicpb_correspondences_pass", ctypes.c_int, [_VOID_P, c_float_p, ctypes.c_int, c_int32_p, c_float_p, c_double_p,
                                                  c_int64_p]),
    ("gicpb_cost", ctypes.c_int, [_VOID_P, c_double_p, c_double_p, c_double_p]),
    ("gicpb_cost_session", ctypes.c_int, [_VOID_P, ctypes.c_int, c_double_p, c_double_p, c_double_p,
                                          ctypes.POINTER(CostSessionInfo)]),
    ("gicpb_grid_info_get", ctypes.c_int, [_VOID_P, ctypes.c_int, ctypes.POINTER(GridInfo)]),
    ("gicpb_bench_kernel", ctypes.c_int, [_VOID_P, ctypes.c_int, c_float_p, ctypes.c_int, c_double_p, c_int64_p]),
    ("gicpb_cloud_resolution", ctypes.c_int, [_VOID_P, ctypes.c_int, c_double_p]),
    ("gicpb_normal_validity", ctypes.c_int, [_VOID_P, ctypes.c_int, ctypes.c_double, c_uint8_p, c_int64_p]),
    ("gicpb_normals", ctypes.c_int, [_VOID_P, ctypes.c_int, ctypes.c_double, c_float_p, c_int64_p]),
    ("gicpb_euclidean_clusters", ctypes.c_int, [_VOID_P, _VOID_P, ctypes.c_int64, ctypes.c_int64, ctypes.c_int,
                                                ctypes.c_double, ctypes.c_int64, ctypes.c_int64, c_int32_p, c_int64_p]),
    ("gicpb_voxel_grid", ctypes.c_int, [_VOID_P, _VOID_P, ctypes.c_int64, ctypes.c_int64, ctypes.c_int, ctypes.c_double,
                                        _VOID_P, c_int64_p]),
    ("gicpb_pointcloud2_to_xyzrgb", ctypes.c_int, [_VOID_P, _VOID_P, ctypes.c_int, ctypes.POINTER(Pc2Layout), _VOID_P,
                                                   ctypes.c_int]),
    ("gicpb_pcd_load_xyzrgb", ctypes.c_int, [_VOID_P, ctypes.c_char_p, _VOID_P, ctypes.c_int64, ctypes.c_int,
                                             ctypes.POINTER(PcdInfo)]),
    ("gicpb_group_create", ctypes.c_int, [ctypes.POINTER(ctypes.c_int), ctypes.c_int, ctypes.POINTER(_VOID_P)]),
    ("gicpb_group_destroy", None, [_VOID_P]),
    ("gicpb_group_last_error", ctypes.c_char_p, [_VOID_P]),
    ("gicpb_group_size", ctypes.c_int, [_VOID_P]),
    ("gicpb_group_fused", ctypes.c_int, [_VOID_P]),
    ("gicpb_group_ctx", ctypes.c_void_p, [_VOID_P, ctypes.c_int]),
    ("gicpb_group_set_params", ctypes.c_int, [_VOID_P, ctypes.POINTER(Params)]),
    ("gicpb_group_set_clouds", ctypes.c_int, [_VOID_P, _VOID_P, ctypes.c_int64, ctypes.c_int64, _VOID_P, ctypes.c_int64,
                                              ctypes.c_int64]),
    ("gicpb_group_align", ctypes.c_int, [_VOID_P, ctypes.POINTER(AlignResult)]),
    ("gicpb_group_fitness", ctypes.c_int, [_VOID_P, c_float_p, ctypes.c_double, c_double_p]),
    ("gicpb_group_cloud_difference", ctypes.c_int, [_VOID_P, _VOID_P, ctypes.c_int64, ctypes.c_int64, _VOID_P,
                                                    ctypes.c_int64, ctypes.c_int64, ctypes.c_double, _VOID_P, c_int64_p]),
    ("gicpb_launch_count", ctypes.c_int64, [_VOID_P]),
    ("gicpb_stream", ctypes.c_void_p, [_VOID_P]),
    ("gicpb_last_far_queries", ctypes.c_int64, [_VOID_P]),
]
EXPORTED_SYMBOLS = [s[0] for s in _SIGNATURES]

_lib = None


def load_library():
    """Load libgicp_b200.so (built in-tree by `make -C leica_point_cloud_processing_b200/csrc` or
    __graft_entry__.build()).  Raises if it is missing: there is no other implementation to fall back to."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `make -C {os.path.join(_PKG_DIR, 'csrc')}` "
            "(or __graft_entry__.build()); this package has no CPU fallback")
    lib = ctypes.CDLL(LIB_PATH)
    for name, restype, argtypes in _SIGNATURES:
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


class GicpError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libgicp_b200 error {code}: {msg}")
        self.code = code


def find_libnccl():
    """Path of the NCCL library torch ships (so the engine and torch.distributed share one libnccl)."""
    try:
        import nvidia.nccl  # noqa: F401
        for d in list(nvidia.nccl.__path__):
            cand = os.path.join(d, "lib", "libnccl.so.2")
            if os.path.exists(cand):
                return cand
    except Exception:
        pass
    return None


def _sync_producer(t):
    """The engine launches on its own non-blocking streams (include/gicp_b200.h, "Device pointers"): whatever torch has
    queued on its current stream for this tensor (a clone, an index_select, a kernel that writes it) must be complete
    before the engine reads or overwrites the memory.  Every engine call waits for its own work before it returns, so
    this one-sided wait orders both directions."""
    import torch
    torch.cuda.current_stream(t.device).synchronize()


def _as_cloud(a):
    """Return (keepalive, pointer, n, stride_bytes, on_device) for a numpy array [n, >=3] float32 (any row stride),
    a structured/byte numpy array of 32-byte points, or a CUDA torch tensor [n, 3|4|8] float32."""
    if hasattr(a, "is_cuda"):  # torch tensor
        if a.dtype.is_floating_point is False or a.element_size() != 4:
            raise TypeError("cloud tensor must be float32")
        if a.dim() != 2 or a.shape[1] < 3 or a.stride(1) != 1:
            raise TypeError("cloud tensor must be [n, >=3] with unit inner stride")
        if a.is_cuda:
            _sync_producer(a)
        return a, a.data_ptr(), int(a.shape[0]), int(a.stride(0)) * 4, 1 if a.is_cuda else 0
    a = np.asarray(a)
    if a.dtype != np.float32:
        a = a.astype(np.float32)
    if a.ndim != 2 or a.shape[1] < 3:
        raise TypeError("cloud array must be [n, >=3] float32")
    if a.strides[1] != 4 or a.strides[0] % 4 != 0 or a.strides[0] < 12:
        a = np.ascontiguousarray(a)
    return a, a.ctypes.data, int(a.shape[0]), int(a.strides[0]), 0


def _T(T):
    T = np.ascontiguousarray(np.asarray(T, dtype=np.float32).reshape(4, 4))
    return T, T.ctypes.data_as(c_float_p)


class Engine:
    """Thin object wrapper over one gicpb_ctx."""

    def __init__(self, device=0, _borrowed=None):
        self.lib = load_library()
        self._owned = _borrowed is None
        if _borrowed is not None:  # a member context of an EngineGroup: the group owns it
            self.h = _VOID_P(_borrowed)
            self.device = device
            return
        h = _VOID_P()
        rc = self.lib.gicpb_create(int(device), ctypes.byref(h))
        if rc != GICPB_OK:
            raise GicpError(rc, "gicpb_create failed (no usable sm_100 GPU?); there is no CPU fallback")
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            if self._owned:
                self.lib.gicpb_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != GICPB_OK:
            raise GicpError(rc, (self.lib.gicpb_last_error(self.h) or b"").decode())

    # ---- parameters ---------------------------------------------------------------------------------
    def get_params(self):
        p = Params()
        self._check(self.lib.gicpb_get_params(self.h, ctypes.byref(p)))
        return p

    def set_params(self, **kw):
        p = self.get_params()
        for k, v in kw.items():
            if not hasattr(p, k):
                raise AttributeError(k)
            setattr(p, k, v)
        self._check(self.lib.gicpb_set_params(self.h, ctypes.byref(p)))
        return p

    # ---- multi-GPU ----------------------------------------------------------------------------------
    def nccl_unique_id(self, libnccl=None):
        buf = (ctypes.c_uint8 * 128)()
        path = (libnccl or find_libnccl() or "").encode() or None
        rc = self.lib.gicpb_nccl_unique_id(path, buf)
        if rc != GICPB_OK:
            raise GicpError(rc, "gicpb_nccl_unique_id failed")
        return bytes(buf)

    def peer_export(self):
        buf = (ctypes.c_uint8 * 64)()
        self._check(self.lib.gicpb_peer_export(self.h, buf))
        return bytes(buf)

    def peer_import(self, handles):
        """handles: list of the 64-byte handles of all ranks, in rank order"""
        blob = b"".join(handles)
        buf = (ctypes.c_uint8 * len(blob)).from_buffer_copy(blob)
        self._check(self.lib.gicpb_peer_import(self.h, buf, len(handles)))

    def peer_disable(self):
        self._check(self.lib.gicpb_peer_disable(self.h))

    def comm_rank(self):
        r, w = ctypes.c_int(), ctypes.c_int()
        self._check(self.lib.gicpb_comm_rank(self.h, ctypes.byref(r), ctypes.byref(w)))
        return r.value, w.value

    def shard_info(self):
        """(lo, hi, source points indexed on this rank, times a window was widened): gicpb_shard_info"""
        v = [ctypes.c_int64() for _ in range(4)]
        self._check(self.lib.gicpb_shard_info(self.h, *[ctypes.byref(x) for x in v]))
        return tuple(int(x.value) for x in v)

    def shard(self):
        """[lo, hi) of this rank's sorted source points that it owns (csrc/engine.cu update_shard)"""
        return self.shard_info()[:2]

    def comm_init(self, rank, world, unique_id, libnccl=None):
        buf = (ctypes.c_uint8 * 128).from_buffer_copy(unique_id)
        path = (libnccl or find_libnccl() or "").encode() or None
        self._check(self.lib.gicpb_comm_init(self.h, path, rank, world, buf))

    # ---- clouds ---------------------------------------------------------------------------------------
    def prefetch(self, which, cloud):
        """Start uploading a HOST cloud (0 target, 1 source) beside whatever runs next; the following set_target /
        set_source of the same object uses that copy (gicpb_prefetch_cloud).  No-op for device clouds."""
        keep, ptr, n, stride, dev = _as_cloud(cloud)
        if dev:
            return
        self._check(self.lib.gicpb_prefetch_cloud(self.h, int(which), ptr, n, stride))
        if not hasattr(self, "_prefetched"):
            self._prefetched = {}
        self._prefetched[int(which)] = (cloud, keep, ptr, n, stride)  # same buffer (and pointer) for the set call

    def _cloud_args(self, which, cloud):
        pf = getattr(self, "_prefetched", {}).pop(which, None)
        if pf is not None and pf[0] is cloud:
            return pf[1], pf[2], pf[3], pf[4], 0
        return _as_cloud(cloud)

    def set_target(self, cloud):
        keep, ptr, n, stride, dev = self._cloud_args(0, cloud)
        self._check(self.lib.gicpb_set_target(self.h, ptr, n, stride, dev))

    def set_source(self, cloud):
        keep, ptr, n, stride, dev = self._cloud_args(1, cloud)
        self._check(self.lib.gicpb_set_source(self.h, ptr, n, stride, dev))

    def set_clouds(self, target, source):
        """set_target + set_source + compute_covariances in one call (the target's covariance pass overlaps the source's
        index build); both clouds on the host or both on the device."""
        kt, tptr, tn, tstride, tdev = self._cloud_args(0, target)
        ks, sptr, sn, sstride, sdev = self._cloud_args(1, source)
        if tdev != sdev:
            raise ValueError("set_clouds: both clouds must be host arrays or both device tensors")
        self._check(self.lib.gicpb_set_clouds(self.h, tptr, tn, tstride, sptr, sn, sstride, tdev))

    def compute_covariances(self):
        self._check(self.lib.gicpb_compute_covariances(self.h))

    def align(self, raise_on_failure=True):
        res = AlignResult()
        rc = self.lib.gicpb_align(self.h, ctypes.byref(res))
        if rc != GICPB_OK and (raise_on_failure or rc in (E_BADARG, E_CUDA, E_NCCL, E_STATE)):
            self._check(rc)
        out = {k: getattr(res, k) for k, _ in AlignResult._fields_ if k != "transform"}
        out["transform"] = np.array(res.transform, np.float32).reshape(4, 4)
        out["rc"] = rc
        return out

    def fitness(self, T, max_range=float(np.finfo(np.float64).max)):
        Tk, Tp = _T(T)
        s = ctypes.c_double()
        self._check(self.lib.gicpb_fitness(self.h, Tp, max_range, ctypes.byref(s)))
        return s.value

    def transform_cloud(self, T, cloud, out=None):
        Tk, Tp = _T(T)
        keep, ptr, n, stride, dev = _as_cloud(cloud)
        if out is None:
            if dev:
                import torch
                out = torch.empty_like(keep)  # the kernel writes every word of every point
            else:
                out = keep.copy()
        okeep, optr, on, ostride, odev = _as_cloud(out)
        if (on, ostride, odev) != (n, stride, dev):
            raise ValueError("out must match the input cloud's shape, stride and device")
        self._check(self.lib.gicpb_transform_cloud(self.h, Tp, ptr, optr, n, stride, dev))
        return okeep

    def cloud_difference(self, input_cloud, subtract_cloud, sqr_threshold):
        """mask (uint8 numpy, or uint8 CUDA tensor when the clouds are CUDA tensors) and kept count."""
        ik, iptr, n, istride, idev = _as_cloud(input_cloud)
        sk, sptr, ns, sstride, sdev = _as_cloud(subtract_cloud)
        if idev != sdev:
            raise ValueError("both clouds must live on the same side (host or device)")
        kept = ctypes.c_int64()
        if idev:
            import torch
            mask = torch.empty(n, dtype=torch.uint8, device=input_cloud.device)
            mptr = mask.data_ptr()
        else:
            mask = np.empty(n, np.uint8)
            mptr = mask.ctypes.data
        self._check(self.lib.gicpb_cloud_difference(self.h, iptr, n, istride, sptr, ns, sstride, idev,
                                                    float(sqr_threshold), mptr, ctypes.byref(kept)))
        return mask, int(kept.value)

    def difference_set_subtract(self, subtract_cloud):
        sk, sptr, ns, sstride, sdev = _as_cloud(subtract_cloud)
        self._check(self.lib.gicpb_difference_set_subtract(self.h, sptr, ns, sstride, sdev))

    def difference_run(self, input_cloud, sqr_threshold, mask=None):
        ik, iptr, n, istride, idev = _as_cloud(input_cloud)
        kept = ctypes.c_int64()
        if mask is None:
            if idev:
                import torch
                mask = torch.empty(n, dtype=torch.uint8, device=input_cloud.device)
            else:
                mask = np.empty(n, np.uint8)
        mdev = 1 if hasattr(mask, "is_cuda") and mask.is_cuda else 0
        mptr = mask.data_ptr() if hasattr(mask, "data_ptr") else mask.ctypes.data
        self._check(self.lib.gicpb_difference_run(self.h, iptr, n, istride, idev, float(sqr_threshold), mptr, mdev,
                                                  ctypes.byref(kept)))
        return mask, int(kept.value)

    # ---- the callers either side of the registration path ------------------------------------------------
    def euclidean_clusters(self, cloud, tolerance, min_size=1, max_size=0):
        """pcl::EuclideanClusterExtraction::extract: (labels int32 [n] in PCL's cluster order, -1 = none; n_clusters)."""
        n = int(cloud.shape[0])
        labels = np.full(n, -1, np.int32)
        nc = ctypes.c_int64()
        if n == 0:
            self._check(self.lib.gicpb_euclidean_clusters(self.h, None, 0, 32, 0, float(tolerance), int(min_size),
                                                          int(max_size), labels.ctypes.data_as(c_int32_p), ctypes.byref(nc)))
            return labels, 0
        keep, ptr, n, stride, dev = _as_cloud(cloud)
        self._check(self.lib.gicpb_euclidean_clusters(self.h, ptr, n, stride, dev, float(tolerance), int(min_size),
                                                      int(max_size), labels.ctypes.data_as(c_int32_p), ctypes.byref(nc)))
        return labels, int(nc.value)

    def voxel_grid(self, cloud, leaf_size):
        """pcl::VoxelGrid with leaf (l, l, l): the centroid points [m, same columns] in ascending voxel order."""
        n = int(cloud.shape[0])
        m = ctypes.c_int64()
        if n == 0:
            return cloud[:0]
        keep, ptr, n, stride, dev = _as_cloud(cloud)
        if dev:
            import torch
            out = torch.zeros((n, stride // 4), dtype=torch.float32, device=keep.device)
            optr = out.data_ptr()
        else:
            out = np.zeros((n, stride // 4), np.float32)
            optr = out.ctypes.data
        self._check(self.lib.gicpb_voxel_grid(self.h, ptr, n, stride, dev, float(leaf_size), optr, ctypes.byref(m)))
        return out[: int(m.value)]

    # ---- wire / on-disk formats (SURVEY 8f row 4) -------------------------------------------------------
    def pointcloud2_to_xyzrgb(self, data, width, height, point_step, row_step, off_x, off_y, off_z, off_rgb=-1,
                              device_out=False):
        """pcl::fromROSMsg into pcl::PointXYZRGB rows: float32 [width * height, 8] (x, y, z, 1, rgba bits, 0, 0, 0).
        `data`: the message payload (bytes / uint8 array, or a CUDA uint8 tensor)."""
        n = int(width) * int(height)
        lay = Pc2Layout(int(width), int(height), int(point_step), int(row_step), int(off_x), int(off_y), int(off_z),
                        int(off_rgb))
        if hasattr(data, "is_cuda"):
            dptr, ddev, keep = data.data_ptr(), 1 if data.is_cuda else 0, data
        else:
            keep = np.frombuffer(data, np.uint8) if isinstance(data, (bytes, bytearray, memoryview)) else np.ascontiguousarray(data).view(np.uint8)
            dptr, ddev = keep.ctypes.data, 0
        if device_out:
            import torch
            out = torch.empty((n, 8), dtype=torch.float32, device=f"cuda:{self.device}")
            optr, odev = out.data_ptr(), 1
        else:
            out = np.empty((n, 8), np.float32)
            optr, odev = out.ctypes.data, 0
        self._check(self.lib.gicpb_pointcloud2_to_xyzrgb(self.h, dptr if n else None, ddev, ctypes.byref(lay), optr if n else None, odev))
        return out

    def pcd_info(self, path):
        """Header of a PCD file (pcl::PCDReader::readHeader) as a dict."""
        info = PcdInfo()
        self._check(self.lib.gicpb_pcd_load_xyzrgb(self.h, os.fsencode(path), None, 0, 0, ctypes.byref(info)))
        return {k: int(getattr(info, k)) for k, _ in PcdInfo._fields_}

    def load_pcd(self, path, device_out=False):
        """pcl::io::loadPCDFile<pcl::PointXYZRGB>: (float32 [points, 8] rows as pointcloud2_to_xyzrgb, info dict)."""
        n = self.pcd_info(path)["points"]
        if device_out:
            import torch
            out = torch.empty((n, 8), dtype=torch.float32, device=f"cuda:{self.device}")
            optr, odev = out.data_ptr(), 1
        else:
            out = np.empty((n, 8), np.float32)
            optr, odev = out.ctypes.data, 0
        info = PcdInfo()
        # a dummy non-null pointer for an empty file: the call must still read the body section
        self._check(self.lib.gicpb_pcd_load_xyzrgb(self.h, os.fsencode(path), optr if n else ctypes.addressof(info), n, odev,
                                                   ctypes.byref(info)))
        return out, {k: int(getattr(info, k)) for k, _ in PcdInfo._fields_}

    # ---- hooks ----------------------------------------------------------------------------------------
    def nn1(self, queries, T=None, max_dist=0.0):
        keep, ptr, n, stride, dev = _as_cloud(queries)
        idx = np.empty(n, np.int32)
        d2 = np.empty(n, np.float32)
        Tp = None
        if T is not None:
            Tk, Tp = _T(T)
        self._check(self.lib.gicpb_nn1(self.h, ptr, n, stride, dev, Tp, float(max_dist),
                                       idx.ctypes.data_as(c_int32_p), d2.ctypes.data_as(c_float_p)))
        return idx, d2

    def knn(self, which):
        info = self.grid_info(which)
        k = self.get_params().k_correspondences
        idx = np.empty((info["n_points"], k), np.int32)
        d2 = np.empty((info["n_points"], k), np.float32)
        self._check(self.lib.gicpb_knn(self.h, which, idx.ctypes.data_as(c_int32_p), d2.ctypes.data_as(c_float_p)))
        return idx, d2

    def covariances(self, which):
        info = self.grid_info(which)
        cov = np.empty((info["n_points"], 3, 3), np.float64)
        self._check(self.lib.gicpb_get_covariances(self.h, which, cov.ctypes.data_as(c_double_p)))
        return cov

    def correspondences(self, T, seeded=False):
        """(pairs, idx, d2, maha) of one correspondence pass under T: the first pass of a job, or with seeded=True a later
        pass (more probe rings, seeded with the current pairs when use_previous_match is on)."""
        Tk, Tp = _T(T)
        n = self.grid_info(1)["n_points"]
        idx = np.empty(n, np.int32)
        d2 = np.full(n, np.inf, np.float32)
        maha = np.empty((n, 3, 3), np.float64)
        maha[:] = np.eye(3)
        pairs = ctypes.c_int64()
        self._check(self.lib.gicpb_correspondences_pass(self.h, Tp, 1 if seeded else 0, idx.ctypes.data_as(c_int32_p),
                                                        d2.ctypes.data_as(c_float_p), maha.ctypes.data_as(c_double_p),
                                                        ctypes.byref(pairs)))
        return int(pairs.value), idx, d2, maha

    def cost(self, x6):
        x = np.ascontiguousarray(x6, np.float64)
        f = ctypes.c_double()
        g = np.empty(6, np.float64)
        self._check(self.lib.gicpb_cost(self.h, x.ctypes.data_as(c_double_p), ctypes.byref(f),
                                        g.ctypes.data_as(c_double_p)))
        return f.value, g

    def cost_session(self, xs):
        """f [n], g [n, 6] of the states xs [n, 6] evaluated inside one evaluation session (gicpb_cost_session), and what
        ran as a dict (persistent, blocks, threads, stages, pairs_per_block, resident_cap, resident, epochs, launches)."""
        x = np.ascontiguousarray(np.asarray(xs, np.float64).reshape(-1, 6))
        n = len(x)
        f = np.empty(n, np.float64)
        g = np.empty((n, 6), np.float64)
        info = CostSessionInfo()
        self._check(self.lib.gicpb_cost_session(self.h, n, x.ctypes.data_as(c_double_p), f.ctypes.data_as(c_double_p),
                                                g.ctypes.data_as(c_double_p), ctypes.byref(info)))
        return f, g, {k: int(getattr(info, k)) for k, _ in CostSessionInfo._fields_}

    def grid_info(self, which):
        gi = GridInfo()
        self._check(self.lib.gicpb_grid_info_get(self.h, which, ctypes.byref(gi)))
        out = {k: getattr(gi, k) for k, _ in GridInfo._fields_ if k != "dims"}
        out["dims"] = tuple(gi.dims)
        return out

    def bench_kernel(self, which, T, iters=10):
        Tk, Tp = _T(T)
        ms = ctypes.c_double()
        launches = ctypes.c_int64()
        self._check(self.lib.gicpb_bench_kernel(self.h, which, Tp, iters, ctypes.byref(ms), ctypes.byref(launches)))
        return ms.value, int(launches.value)

    def cloud_resolution(self, which):
        """Utils::computeCloudResolution of an indexed cloud (0 target, 1 source, 2 subtract)."""
        r = ctypes.c_double()
        self._check(self.lib.gicpb_cloud_resolution(self.h, which, ctypes.byref(r)))
        return r.value

    def normal_validity(self, which, radius):
        """(mask, count): which points of an indexed cloud get a finite radius-search normal (>= 3 points in the radius)."""
        n = self.grid_info(which)["n_points"]
        mask = np.zeros(n, np.uint8)
        kept = ctypes.c_int64()
        self._check(self.lib.gicpb_normal_validity(self.h, which, float(radius), mask.ctypes.data_as(c_uint8_p),
                                                   ctypes.byref(kept)))
        return mask, int(kept.value)

    def normals(self, which, radius):
        """Utils::getNormals of an indexed cloud: (float32 [n, 4] = nx, ny, nz, curvature with NaN rows where PCL gives no
        normal, number of finite normals)."""
        n = self.grid_info(which)["n_points"]
        out = np.empty((n, 4), np.float32)
        kept = ctypes.c_int64()
        self._check(self.lib.gicpb_normals(self.h, which, float(radius), out.ctypes.data_as(c_float_p), ctypes.byref(kept)))
        return out, int(kept.value)

    def stream_handle(self):
        """cudaStream_t of the context as an integer (torch.cuda.ExternalStream(handle) wraps it)."""
        return int(self.lib.gicpb_stream(self.h) or 0)

    def last_far_queries(self):
        return int(self.lib.gicpb_last_far_queries(self.h))

    def launch_count(self):
        return int(self.lib.gicpb_launch_count(self.h))


class EngineGroup:
    """One process, several GPUs (gicpb_group): the source sharded over the devices, the target replicated, one host thread
    per GPU inside the library.  `devices` may name one GPU several times (host-mediated sums then; for tests on one GPU)."""

    def __init__(self, devices):
        self.lib = load_library()
        devs = (ctypes.c_int * len(devices))(*[int(d) for d in devices])
        h = _VOID_P()
        rc = self.lib.gicpb_group_create(devs, len(devices), ctypes.byref(h))
        if rc != GICPB_OK:
            raise GicpError(rc, "gicpb_group_create failed")
        self.h = h
        self.devices = list(devices)

    def close(self):
        if getattr(self, "h", None):
            self.lib.gicpb_group_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != GICPB_OK:
            raise GicpError(rc, (self.lib.gicpb_group_last_error(self.h) or b"").decode())

    @property
    def size(self):
        return int(self.lib.gicpb_group_size(self.h))

    @property
    def fused(self):
        return bool(self.lib.gicpb_group_fused(self.h))

    def member(self, rank):
        """Engine view of one member context (owned by the group)."""
        p = self.lib.gicpb_group_ctx(self.h, int(rank))
        if not p:
            raise IndexError(rank)
        return Engine(self.devices[rank], _borrowed=p)

    def set_params(self, **kw):
        p = self.member(0).get_params()
        for k, v in kw.items():
            if not hasattr(p, k):
                raise AttributeError(k)
            setattr(p, k, v)
        self._check(self.lib.gicpb_group_set_params(self.h, ctypes.byref(p)))
        return p

    def set_clouds(self, target, source):
        kt, tptr, tn, tstride, tdev = _as_cloud(target)
        ks, sptr, sn, sstride, sdev = _as_cloud(source)
        if tdev or sdev:
            raise ValueError("EngineGroup.set_clouds takes host clouds")
        self._check(self.lib.gicpb_group_set_clouds(self.h, tptr, tn, tstride, sptr, sn, sstride))

    def align(self, raise_on_failure=True):
        res = AlignResult()
        rc = self.lib.gicpb_group_align(self.h, ctypes.byref(res))
        if rc != GICPB_OK and (raise_on_failure or rc in (E_BADARG, E_CUDA, E_NCCL, E_STATE)):
            self._check(rc)
        out = {k: getattr(res, k) for k, _ in AlignResult._fields_ if k != "transform"}
        out["transform"] = np.array(res.transform, np.float32).reshape(4, 4)
        out["rc"] = rc
        return out

    def fitness(self, T, max_range=float(np.finfo(np.float64).max)):
        Tk, Tp = _T(T)
        s = ctypes.c_double()
        self._check(self.lib.gicpb_group_fitness(self.h, Tp, max_range, ctypes.byref(s)))
        return s.value

    def cloud_difference(self, input_cloud, subtract_cloud, sqr_threshold):
        """Engine.cloud_difference over the group's GPUs: (mask uint8 numpy, kept count).  Host clouds only."""
        ik, iptr, n, istride, idev = _as_cloud(input_cloud)
        sk, sptr, ns, sstride, sdev = _as_cloud(subtract_cloud)
        if idev or sdev:
            raise ValueError("EngineGroup.cloud_difference takes host clouds")
        kept = ctypes.c_int64()
        mask = np.empty(n, np.uint8)
        self._check(self.lib.gicpb_group_cloud_difference(self.h, iptr, n, istride, sptr, ns, sstride,
                                                          float(sqr_threshold), mask.ctypes.data, ctypes.byref(kept)))
        return mask, int(kept.value)
