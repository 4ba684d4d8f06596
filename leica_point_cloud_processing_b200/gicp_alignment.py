"""Host-side mirror of the reference's GICP stage classes, on top of the C ABI.

`GICPAlignment` keeps the public surface of the reference class (include/GICPAlignment.h:47-145, behaviour of
src/GICPAlignment.cpp:23-198): same method names, argument meaning, defaults and quirks, so the reference's own
tests (test/test_gicp_alignment.cpp) translate line by line.  `remove_from_cloud` mirrors
Filter::removeFromCloud (src/Filter.cpp:176-189).  The C++ drop-in with identical semantics is
include/GICPAlignment_b200.hpp.

Clouds are numpy float32 arrays [n, 3] (xyz), [n, 4] or [n, 8] (the 32-byte pcl::PointXYZRGB layout; columns past
xyz are carried through untouched), or CUDA torch tensors of the same shapes.
"""
import logging

import numpy as np

from ._capi import Engine, E_NOT_ENOUGH_CORRESPONDENCES, E_SOLVER, E_TOO_FEW_POINTS

log = logging.getLogger("leica_point_cloud_processing_b200")


def _copy(cloud):
    return cloud.clone() if hasattr(cloud, "clone") else np.array(cloud, copy=True)


def is_valid_transform(tf):
    """Utils::isValidTransform (reference src/Utils.cpp:71-82): no NaN entry."""
    return not bool(np.isnan(np.asarray(tf)).any())


class GICPAlignment:
    """Fine registration of `source_cloud` onto `target_cloud` with GICP (target first, as the reference ctor)."""

    def __init__(self, target_cloud, source_cloud, use_covariances, device=0, engine=None):
        # reference src/GICPAlignment.cpp:23-35
        self.target_cloud_ = target_cloud
        self.source_cloud_ = source_cloud
        self.covariances_ = bool(use_covariances)
        self.tf_epsilon_ = 4e-3
        self.max_iter_ = 100
        self.max_corresp_distance_ = 4e-2
        self.ransac_outlier_th_ = 1.0
        self.transform_exists_ = False
        self.fine_tf_ = np.eye(4, dtype=np.float32)
        self.aligned_cloud_ = None
        self.backup_cloud_ = None
        self._engine = engine if engine is not None else Engine(device)
        self._converged = False
        self._fitness = None
        self._inputs_set = False
        self._input_source_ = None
        self.last_result = None

    # ---- public surface (include/GICPAlignment.h:63-145) ---------------------------------------------
    def run(self):
        self._config_parameters()
        if self.covariances_:
            self._apply_covariances()
        self._fine_alignment()
        self.applyTFtoCloud(self.source_cloud_)

    def iterate(self):
        self._iterate_fine_alignment()

    def undo(self):
        if self.backup_cloud_ is not None:
            self.aligned_cloud_ = _copy(self.backup_cloud_)

    def getFineTransform(self):
        if not self.transform_exists_:
            log.error("No transform yet. Please run algorithm")
        return self.fine_tf_.copy()

    def getAlignedCloud(self, aligned_cloud=None):
        """Deep copy of the aligned cloud (reference :156-159).  If `aligned_cloud` is a list it is filled in
        place (the reference's out-parameter form); the copy is returned either way."""
        out = _copy(self.aligned_cloud_) if self.aligned_cloud_ is not None else np.zeros((0, 3), np.float32)
        if isinstance(aligned_cloud, list):
            aligned_cloud[:] = [out]
        return out

    def applyTFtoCloud(self, cloud):
        # reference :144-147: reads `cloud`, writes the INTERNAL aligned cloud; `cloud` itself is untouched
        self.aligned_cloud_ = self._engine.transform_cloud(self.fine_tf_, cloud)

    def setSourceCloud(self, source_cloud):
        # reference :166-169: only the wrapper's pointer changes.  gicp_ keeps the cloud it was given by
        # setInputSource in fineAlignment (:89), so a following iterate() still solves on the OLD pair; the new cloud
        # is used from the next run() on
        self.source_cloud_ = source_cloud

    def setTargetCloud(self, target_cloud):
        self.target_cloud_ = target_cloud  # reference :171-174, same remark

    def setMaxIterations(self, iterations):
        self.max_iter_ = int(iterations)
        self._config_parameters()

    def setTfEpsilon(self, tf_epsilon):
        self.tf_epsilon_ = float(tf_epsilon)
        self._config_parameters()

    def setMaxCorrespondenceDistance(self, max_corresp_distance):
        # the reference declares this parameter as `int` (include/GICPAlignment.h:138): fractions are truncated
        self.max_corresp_distance_ = float(int(max_corresp_distance))
        self._config_parameters()

    def setRANSACOutlierTh(self, ransac_threshold):
        # `int` in the reference as well (:145); GICP never uses the RANSAC threshold
        self.ransac_outlier_th_ = float(int(ransac_threshold))
        self._config_parameters()

    # ---- additions that do not break the reference surface ------------------------------------------
    def hasConverged(self):
        return self._converged

    def getFitnessScore(self):
        return self._fitness

    # ---- private, mirroring the reference's private methods -------------------------------------------
    def _config_parameters(self):
        # reference :48-54
        self._engine.set_params(max_iterations=self.max_iter_, max_corr_distance=self.max_corresp_distance_,
                                transformation_epsilon=self.tf_epsilon_)

    def _get_covariances(self, which):
        # reference :56-71 for one cloud (which: 1 source, 0 target).  Both resolutions are recomputed on every call,
        # as upstream does; the radius-search normals only decide WHICH points survive (those with a finite normal,
        # i.e. >= 3 points inside the radius); the covariances built from them are reset by setInputSource/Target.
        eng = self._engine
        eng.set_target(self.target_cloud_)
        eng.set_source(self.source_cloud_)
        target_res = eng.cloud_resolution(0)
        source_res = eng.cloud_resolution(1)
        normal_radius = (target_res + source_res) * 2.0
        log.info("Computing normals with radius: %f", normal_radius)
        mask, kept = eng.normal_validity(which, normal_radius)
        cloud = self.source_cloud_ if which == 1 else self.target_cloud_
        if kept != len(cloud):
            keep = mask.astype(bool)
            if hasattr(cloud, "is_cuda"):
                import torch
                keep = torch.from_numpy(keep).to(cloud.device)
            cloud = cloud[keep]
            if which == 1:
                self.source_cloud_ = cloud
            else:
                self.target_cloud_ = cloud
        self.covariance_radius_ = normal_radius
        return kept

    def _apply_covariances(self):
        # reference :73-84: source first, then target.  Upstream filters the caller's clouds IN PLACE through the shared
        # pointers; arrays cannot shrink in place, so the filtered clouds replace self.source_cloud_ / target_cloud_
        # (the C++ drop-in mutates the caller's clouds exactly like the reference).
        log.info("Extract covariances from clouds")
        self._get_covariances(1)
        self._get_covariances(0)
        self._inputs_set = False

    def _fine_alignment(self):
        # reference :86-109
        log.info("Perform GICP with %d iterations", self.max_iter_)
        self._engine.prefetch(0, self.target_cloud_)   # both uploads queue on the copy stream, target first:
        self._engine.prefetch(1, self.source_cloud_)   # the source uploads while the target is indexed
        self._engine.set_clouds(self.target_cloud_, self.source_cloud_)
        self._inputs_set = True
        self._input_source_ = self.source_cloud_   # what gicp_.setInputSource holds from here on (reference :89)
        res = self._engine.align(raise_on_failure=False)
        self.last_result = res
        log.info("GICP time: %f s", res["ms_total"] * 1e-3)
        self._converged = bool(res["converged"])
        if res["rc"] not in (0, E_NOT_ENOUGH_CORRESPONDENCES, E_SOLVER, E_TOO_FEW_POINTS):
            raise RuntimeError(f"gicpb_align failed with {res['rc']}")
        if self._converged:
            self._fitness = self._engine.fitness(res["transform"])
            log.info("Converged in %f FitnessScore", self._fitness)
            self.fine_tf_ = res["transform"].copy()
            self.transform_exists_ = is_valid_transform(self.fine_tf_)
        else:
            log.error("GICP no converge")

    def _iterate_fine_alignment(self):
        # reference :111-127.  PCL's align() re-solves from the ORIGINAL source at identity with the cached
        # covariances and overwrites the cloud it is given with final_transformation * source (SURVEY App. A.6).
        self.backup_cloud_ = _copy(self.aligned_cloud_) if self.aligned_cloud_ is not None else None
        log.info("Computing iteration...")
        if not self._inputs_set:
            # gicp_.align() without setInputSource / setInputTarget: PCL's initCompute fails, nothing converges
            log.error("GICP no converge")
            self._converged = False
            return
        res = self._engine.align(raise_on_failure=False)
        self.last_result = res
        self._converged = bool(res["converged"])
        if self._converged:
            temp_tf = res["transform"]
            self.fine_tf_ = (temp_tf @ self.fine_tf_).astype(np.float32)
            self._fitness = self._engine.fitness(temp_tf)
            log.info("Converged in %f FitnessScore", self._fitness)
        else:
            log.error("GICP no converge")
        # PCL's align() writes final_transformation * (the source given to setInputSource) into the cloud it is handed
        self.aligned_cloud_ = self._engine.transform_cloud(res["transform"], self._input_source_)


def remove_from_cloud(input_cloud, subtract_cloud, threshold, engine=None, device=0):
    """Filter::removeFromCloud (reference src/Filter.cpp:176-189): the points of `input_cloud` whose SQUARED
    distance to their nearest neighbour in `subtract_cloud` exceeds `threshold`, in input order.
    `engine` may be an EngineGroup (host clouds): the difference then runs on all of its GPUs.
    Returns (filtered_cloud, mask)."""
    eng = engine if engine is not None else Engine(device)
    log.info("Difference from segment with threshold: %f", threshold)
    mask, _ = eng.cloud_difference(input_cloud, subtract_cloud, threshold)
    keep = mask.bool() if hasattr(mask, "bool") else mask.astype(bool)
    return input_cloud[keep], mask
