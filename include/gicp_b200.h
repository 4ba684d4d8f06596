/* gicp_b200.h - C ABI of libgicp_b200.so, a B200 (sm_100a) GICP registration engine.
 *
 * This is the drop-in boundary for ONE path of catec/leica_point_cloud_processing: fine registration
 * behind `GICPAlignment` and the nearest-distance cloud difference behind `Filter::removeFromCloud`.
 * Each entry point names the reference interface it replaces (paths relative to the reference root).
 * The reference has no FFI layer (it is a plain C++ class linked against PCL), so the "binding" a
 * maintainer adds is the header-only C++ shim include/GICPAlignment_b200.hpp; see INTEGRATION.md.
 *
 * Conventions
 *   - plain pointers and sizes only; no C++ / torch / PCL types cross this boundary
 *   - every function returns GICPB_OK (0) or a negative GICPB_E_* code; gicpb_last_error(ctx) holds text
 *   - clouds are given as a base pointer to the first x, a point count and a byte stride between points
 *     (x, y, z are three consecutive float32).  stride 32 = pcl::PointXYZRGB as the reference holds it
 *     (include/GICPAlignment.h:35), stride 16 = float4, stride 12 = packed xyz
 *   - `on_device` != 0 means the pointer is a CUDA device pointer on the context's GPU; otherwise host
 *     (pinned host memory is copied as it is; pageable host clouds of 8 MB and more - a pcl::PointCloud - are gathered
 *     into packed xyz rows by a few host threads through a ring of pinned chunks, so 12 bytes per point cross PCIe)
 *   - Device pointers (stream contract): the library launches on its own non-blocking streams and every call waits
 *     for its work before it returns.  It does NOT order itself against the caller's streams: memory behind an
 *     `on_device` input must be completely written, and memory behind a device output no longer in use, before the
 *     call is made (synchronise the producing stream, or make gicpb_stream(ctx) wait on an event of it)
 *   - 4x4 transforms are float32, ROW-major (T[4*r + c]); Eigen::Matrix4f is column-major, the shim transposes
 *   - a context is bound to one GPU and is not thread-safe; distinct contexts are independent
 *   - there is no CPU fallback: without a usable GPU gicpb_create fails with GICPB_E_CUDA
 */
#ifndef GICP_B200_H_
#define GICP_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GICPB_OK 0
#define GICPB_E_BADARG (-1)
#define GICPB_E_CUDA (-2)
#define GICPB_E_NCCL (-3)
#define GICPB_E_NOT_ENOUGH_CORRESPONDENCES (-4) /* PCL NotEnoughPointsException: < 4 pairs            */
#define GICPB_E_SOLVER (-5)                     /* PCL SolverDidntConvergeException                     */
#define GICPB_E_STATE (-6)                      /* call order: clouds / covariances missing             */
#define GICPB_E_TOO_FEW_POINTS (-7)             /* k_correspondences > cloud size (gicp.hpp)            */

typedef struct gicpb_ctx gicpb_ctx;

/* Parameters of pcl::GeneralizedIterativeClosestPoint that the reference sets or inherits.
 * Defaults = reference src/GICPAlignment.cpp:29-32 over the PCL 1.8.1 gicp.h defaults. */
typedef struct gicpb_params {
  int max_iterations;             /* setMaximumIterations          src/GICPAlignment.cpp:50   (100)   */
  double transformation_epsilon;  /* setTransformationEpsilon      src/GICPAlignment.cpp:52   (4e-3)  */
  double rotation_epsilon;        /* PCL rotation_epsilon_                                    (2e-3)  */
  double max_corr_distance;       /* setMaxCorrespondenceDistance  src/GICPAlignment.cpp:51   (4e-2)  */
  int k_correspondences;          /* PCL k_correspondences_ (2..32)                           (20)    */
  double gicp_epsilon;            /* PCL gicp_epsilon_                                        (1e-3)  */
  int max_inner_iterations;       /* PCL max_inner_iterations_                                (20)    */
  /* engine knobs (no reference counterpart; results do not depend on them) */
  float cell_size;                /* uniform-grid cell edge in metres; <= 0 -> chosen from point density */
  float points_per_cell;          /* density target when cell_size <= 0                       (6.0)   */
  int mahalanobis_fp32;           /* 0: store M as 6 doubles (default); 1: 6 floats (56 B/pair cost pass) */
  int use_previous_match;         /* 1 (default): seed each NN search with last iteration's match     */
  int l2_persist;                 /* 1 (default): persisting-L2 window on the per-pair Mahalanobis array    */
  int cost_moments;               /* 0 (default): one cost-kernel pass over all pairs per evaluation, T*p rounded to
                                   * float exactly as PCL does: the BFGS path is PCL's step for step.
                                   * 1: one pass per OUTER iteration reduces the pairs to the 74 second-order moments
                                   * of the objective (a quadratic form in the 12 transform entries); every f / df
                                   * evaluation of the line search is then host arithmetic (and, sharded, there is
                                   * one all-reduce per outer iteration instead of one per evaluation).  Same
                                   * objective with exact T*p: values agree to ~1e-8 relative, which PCL's line
                                   * search amplifies to ~2e-4 in the final transform (see DESIGN.md section 4) */
  int cost_persistent;            /* 1 (default): the evaluations of one inner solve are commands to ONE resident kernel
                                   * (launched per outer iteration, a third of the pairs parked in shared memory) instead of
                                   * one launch each; the same terms, summed in another order (a block owns a
                                   * contiguous range of pairs): the sums agree with the per-launch kernel's to within
                                   * 2 n 2^-53 sum|terms|, and repeated evaluations of one state are bit-identical.
                                   * 0: one launch per evaluation */
} gicpb_params;

typedef struct gicpb_align_result {
  float transform[16];       /* getFinalTransformation()  src/GICPAlignment.cpp:104, row-major         */
  int converged;             /* hasConverged()            src/GICPAlignment.cpp:101                    */
  int status;                /* GICPB_OK or the GICPB_E_* that ended the outer loop                    */
  int outer_iterations;      /* nr_iterations_                                                         */
  int inner_iterations;      /* BFGS steps summed over the outer loop                                  */
  int64_t cost_evaluations;  /* cost/gradient kernel launches                                          */
  int64_t corr_queries;      /* source queries processed by the correspondence kernel (all outer its.) */
  int64_t corr_pairs_last;   /* correspondences of the last outer iteration (all ranks)                */
  int64_t corr_far_queries;  /* of corr_queries (this rank), those answered by the hierarchical far search */
  double ms_total;           /* wall ms of gicpb_align                                                 */
  double ms_corr;            /* device ms in the correspondence (NN + gate + Mahalanobis) kernel       */
  double ms_cost;            /* device ms in the cost/gradient kernel                                  */
} gicpb_align_result;

/* ---- lifetime -------------------------------------------------------------------------------------- */
void gicpb_default_params(gicpb_params* p);
int gicpb_create(int device, gicpb_ctx** out);                 /* ctor  src/GICPAlignment.cpp:23-35    */
void gicpb_destroy(gicpb_ctx* ctx);                            /* dtor  include/GICPAlignment.h:53     */
const char* gicpb_last_error(const gicpb_ctx* ctx);
int gicpb_set_params(gicpb_ctx* ctx, const gicpb_params* p);   /* configParameters :48-54              */
int gicpb_get_params(const gicpb_ctx* ctx, gicpb_params* p);

/* ---- multi-GPU: one process per GPU, source points sharded by rank, target replicated --------------
 * The per-evaluation partial sums are all-reduced with NCCL (ncclAllReduce, 14 doubles).  NCCL is
 * dlopen'ed from `libnccl_path` (NULL: "libnccl.so.2"), so the library has no link-time NCCL dependency. */
int gicpb_nccl_unique_id(const char* libnccl_path, unsigned char id_out[128]);
int gicpb_comm_init(gicpb_ctx* ctx, const char* libnccl_path, int rank, int world, const unsigned char id[128]);
int gicpb_comm_rank(const gicpb_ctx* ctx, int* rank, int* world);
/* This rank's shard [lo, hi) of its sorted source points, how many source points this rank has indexed (with more than one
 * rank: its window of brick planes, not the whole cloud) and how often a window had to be widened to the whole cloud. */
int gicpb_shard_info(gicpb_ctx* ctx, int64_t* lo, int64_t* hi, int64_t* n_indexed_here, int64_t* widened);
/* Optional, after gicpb_comm_init on every rank: fuse the cross-GPU sum of the 14 cost sums INTO the cost kernel over
 * NVLink peer memory (the kernel's last block sends its sums into every rank's slot block as self-validating 8-byte
 * words - half of a double and the evaluation counter - polls the words of the other ranks in its own block and adds
 * the sums in rank order), replacing the ncclAllReduce + copy per evaluation.
 * gicpb_peer_export returns this rank's cudaIpcMemHandle_t (64 bytes); the caller gathers the handles of all ranks
 * (rank order, 64 bytes each) and passes them to gicpb_peer_import.  All ranks must be processes on one node with
 * peer access between their GPUs; on failure the context keeps using NCCL. */
int gicpb_peer_export(gicpb_ctx* ctx, unsigned char handle_out[64]);
int gicpb_peer_import(gicpb_ctx* ctx, const unsigned char* handles, int world);
int gicpb_peer_disable(gicpb_ctx* ctx); /* back to ncclAllReduce (call on every rank) */

/* ---- one process, several GPUs ----------------------------------------------------------------------------------
 * The reference's consumer constructs GICPAlignment inside one process (src/LeicaStateMachine.cpp:138-171): a group makes
 * the sharded path reachable from there, without a launcher.  gicpb_group_create makes one context per entry of
 * `devices` (SURVEY 8b "create(cfg: device ids, n_gpus)"); every group call below runs the per-context call of the same
 * name on all of them, one host thread per GPU, the source sharded by rank and the target replicated exactly as with one
 * process per GPU.  The collectives stay inside the process: target covariances by peer copies, the per-evaluation sum
 * fused into the cost kernel over peer memory when every pair of devices can map each other (gicpb_group_fused), else
 * through the host.  No NCCL is needed.  All clouds are HOST clouds.  A group of one device is a plain context.
 * gicpb_group_ctx(g, r) is a full single-GPU context between group calls (transform, difference, clusters, resolution,
 * normals, ...): used on its own a member never waits for the others.  Clouds set through a member directly are that
 * member's alone; the next gicpb_group_set_clouds replaces them.  A member's source index is the group's (that rank's
 * window of the source): the first call on the member alone that needs the source (gicpb_align, gicpb_fitness,
 * gicpb_correspondences, gicpb_get_covariances, ...) indexes the whole source and works on all of it, with covariances
 * computed again for the whole cloud; the next group call goes back to the rank's shard and recomputes them on every member. */
typedef struct gicpb_group gicpb_group;
int gicpb_group_create(const int* devices, int n_devices, gicpb_group** out);
void gicpb_group_destroy(gicpb_group* group);
const char* gicpb_group_last_error(const gicpb_group* group);
int gicpb_group_size(const gicpb_group* group);
int gicpb_group_fused(const gicpb_group* group);
gicpb_ctx* gicpb_group_ctx(gicpb_group* group, int rank);
int gicpb_group_set_params(gicpb_group* group, const gicpb_params* p);                 /* configParameters :48-54 */
int gicpb_group_set_clouds(gicpb_group* group, const void* target, int64_t n_target, int64_t target_stride_bytes,
                           const void* source, int64_t n_source, int64_t source_stride_bytes); /* :89-90 */
int gicpb_group_align(gicpb_group* group, gicpb_align_result* out);                     /* gicp_.align :96,116 */
int gicpb_group_fitness(gicpb_group* group, const float transform[16], double max_range, double* score); /* :103,123 */
/* gicpb_cloud_difference over the group (Filter::removeFromCloud, src/Filter.cpp:176-189): host clouds and a host mask,
 * the same mask and n_kept as one context gives, the same argument errors.  Every member uploads its 1/N of the rows of
 * both clouds and gets the rest from the other members (GICPB_SHARD_UPLOAD=0: each uploads both clouds whole).  Member r
 * indexes only its own brick planes of the subtract cloud plus a halo of planes that covers sqrt(sqr_threshold) (the
 * whole cloud when that halo reaches both ends), answers the finite input points that fall into its own planes, and
 * writes the mask rows [n_input r / N, n_input (r + 1) / N) from the answers of every member.  A subtract cloud that
 * cannot be split by planes (too few of them, fewer than 1024 N finite points, a member without points) is indexed
 * whole by every member, each answering its row slice.  Afterwards a member's subtract index is that window
 * (gicpb_grid_info_get(ctx, 2) reports it); used on its own, the member indexes the whole subtract cloud again before
 * gicpb_difference_run, gicpb_cloud_resolution or gicpb_normals on it.  The target and source indexes, covariances and
 * correspondences of the group are not touched. */
int gicpb_group_cloud_difference(gicpb_group* group, const void* input, int64_t n_input, int64_t input_stride,
                                 const void* subtract, int64_t n_subtract, int64_t subtract_stride,
                                 double sqr_threshold, uint8_t* mask, int64_t* n_kept);

/* ---- clouds: upload once, index on the GPU (replaces setInputTarget / setInputSource and the two FLANN
 *      kd-tree builds, src/GICPAlignment.cpp:89-90; PCL Registration::initCompute[Reciprocal]) ------- */
/* Optional hint for HOST clouds: start uploading cloud `which` (0 target, 1 source) on a copy stream now and return
 * at once; a later gicpb_set_target / gicpb_set_source with the same (pointer, n, stride) uses that copy instead of
 * uploading again, so the upload of one cloud overlaps the indexing of the other (pinned host memory overlaps; pageable
 * memory is still correct).  The host buffer must stay valid and unchanged until that set call returns. */
int gicpb_prefetch_cloud(gicpb_ctx* ctx, int which, const void* xyz, int64_t n, int64_t stride_bytes);
int gicpb_set_target(gicpb_ctx* ctx, const void* xyz, int64_t n, int64_t stride_bytes, int on_device);
int gicpb_set_source(gicpb_ctx* ctx, const void* xyz, int64_t n, int64_t stride_bytes, int on_device);
/* gicpb_set_target + gicpb_set_source + gicpb_compute_covariances in one call, with the same results: the target's
 * covariance pass runs on a second stream while the source is being indexed (setInputTarget + setInputSource,
 * src/GICPAlignment.cpp:89-90, and the two computeCovariances passes of gicp_.align, :96).  Both clouds host or both
 * device; clouds announced with gicpb_prefetch_cloud are taken from there. */
int gicpb_set_clouds(gicpb_ctx* ctx, const void* target, int64_t n_target, int64_t target_stride_bytes,
                     const void* source, int64_t n_source, int64_t source_stride_bytes, int on_device);
/* kNN-k covariances of both clouds, regularised to (1, 1, gicp_epsilon) (PCL GICP::computeCovariances).
 * Called implicitly by gicpb_align when missing; cached until the cloud is set again (PCL A.1 semantics). */
int gicpb_compute_covariances(gicpb_ctx* ctx);

/* ---- the solve (replaces gicp_.align(), src/GICPAlignment.cpp:96,116; guess = identity as there) ---- */
int gicpb_align(gicpb_ctx* ctx, gicpb_align_result* out);
/* getFitnessScore(max_range) under `transform` (src/GICPAlignment.cpp:103,123); all ranks get the value */
int gicpb_fitness(gicpb_ctx* ctx, const float transform[16], double max_range, double* score);

/* ---- pcl::transformPointCloud (src/GICPAlignment.cpp:146, src/LeicaStateMachine.cpp:182): xyz of every
 *      point is replaced by T * xyz, all other bytes of the stride are copied.  in == out is allowed. -- */
int gicpb_transform_cloud(gicpb_ctx* ctx, const float transform[16], const void* in, void* out, int64_t n,
                          int64_t stride_bytes, int on_device);

/* ---- Filter::removeFromCloud (src/Filter.cpp:176-189 -> pcl::getPointCloudDifference): mask[i] = 1 iff
 *      input point i is finite and its squared NN distance in `subtract` is > sqr_threshold.
 *      n_kept may be NULL.  Does not touch the clouds set for alignment. ----------------------------- */
int gicpb_cloud_difference(gicpb_ctx* ctx, const void* input, int64_t n_input, int64_t input_stride,
                           const void* subtract, int64_t n_subtract, int64_t subtract_stride, int on_device,
                           double sqr_threshold, uint8_t* mask, int64_t* n_kept);
/* Two-step form for repeated differences against one cloud (index built once). */
int gicpb_difference_set_subtract(gicpb_ctx* ctx, const void* subtract, int64_t n, int64_t stride, int on_device);
int gicpb_difference_run(gicpb_ctx* ctx, const void* input, int64_t n, int64_t stride, int on_device,
                         double sqr_threshold, uint8_t* mask, int mask_on_device, int64_t* n_kept);

/* ---- the use_covariances branch (GICPAlignment::getCovariances, src/GICPAlignment.cpp:56-71) ---------------------
 * which = 0 target, 1 source (as set by gicpb_set_target / gicpb_set_source), 2 subtract.
 * Utils::computeCloudResolution (src/Utils.cpp:145-174): mean over the finite points of the distance to the 2nd
 * nearest neighbour (the 1st is the point itself). */
int gicpb_cloud_resolution(gicpb_ctx* ctx, int which, double* resolution);
/* valid[i] = 1 iff Utils::getNormals(cloud, radius) (src/Utils.cpp:27-44, pcl::NormalEstimation with a radius
 * search) gives point i a finite normal: the point is finite and has >= 3 points (itself included) closer than
 * `radius`.  getCovariances then drops the other points from the caller's cloud (src/GICPAlignment.cpp:63-67);
 * valid is a host array in ORIGINAL point order. */
int gicpb_normal_validity(gicpb_ctx* ctx, int which, double radius, uint8_t* valid, int64_t* n_valid);

/* Utils::getNormals (src/Utils.cpp:27-44): pcl::NormalEstimation<PointXYZRGB, Normal> with setRadiusSearch(radius) on an
 * indexed cloud (which: 0 target, 1 source, 2 subtract), viewpoint (0, 0, 0).  normals4[4 i .. 4 i + 3] = normal_x, normal_y,
 * normal_z, curvature of point i (original order): the eigenvector of the smallest eigenvalue of the neighbourhood's
 * covariance - accumulated in float over the neighbours sorted by (distance, index), as PCL 1.8.1 does - flipped towards
 * the viewpoint, and |lambda_0 / trace|.  NaN x 4 for a non-finite point and for fewer than 3 points inside the radius
 * (exactly the points gicpb_normal_validity marks 0).  *n_valid = number of finite normals.  Host output. */
int gicpb_normals(gicpb_ctx* ctx, int which, double radius, float* normals4, int64_t* n_valid);

/* ---- the callers either side of the registration path (SURVEY section 8f) ---------------------------------------
 * FODDetector::clusterPossibleFODs (src/FODDetector.cpp:45-58 -> pcl::EuclideanClusterExtraction::extract, called at
 * src/LeicaStateMachine.cpp:200-205 on the difference cloud): connected components of the graph joining two points
 * whose squared distance is < tolerance^2 (FLANN radius search, strict), kept when min_size <= size <= max_size
 * (max_size <= 0: no upper limit, the PCL default).  labels[i] = rank of point i's cluster in PCL's output order
 * (largest cluster first; equal sizes by lowest point index) or -1 (cluster dropped by the size filter, or a
 * non-finite point).  The indices of one cluster, ascending, are PCL's PointIndices::indices.  labels is a host
 * array of n; n = 0 is allowed (no clusters). */
int gicpb_euclidean_clusters(gicpb_ctx* ctx, const void* cloud, int64_t n, int64_t stride_bytes, int on_device,
                             double tolerance, int64_t min_size, int64_t max_size, int32_t* labels, int64_t* n_clusters);
/* Filter::downsampleCloud (src/Filter.cpp:91-105 -> pcl::VoxelGrid<PointXYZRGB>, leaf (l, l, l), all fields
 * downsampled): one point per occupied voxel, in ascending voxel index (PCL's output order): xyz = mean of the
 * voxel's points (float sums), stride >= 16: data[3] = 1, stride >= 20: the rgba word at byte 16 = per-channel
 * mean (truncated), all other bytes 0 (the last input point must extend through its rgba word).  `out` must have room for n points of the same stride (host or device like
 * `in`); every byte of the n_out rows is written.  When PCL's check refuses the leaf (dx * dy * dz > INT32_MAX with
 * d = int((max - min) / leaf) + 1) PCL warns and passes the input through: so does this call (n_out = n, the warning
 * is left in gicpb_last_error; a call that downsamples leaves gicpb_last_error empty).  Past that check PCL's 32-bit
 * voxel index may wrap; the output then matches PCL's, which averages the voxels that share a wrapped index. */
int gicpb_voxel_grid(gicpb_ctx* ctx, const void* in, int64_t n, int64_t stride_bytes, int on_device, double leaf_size,
                     void* out, int64_t* n_out);

/* ---- the wire and on-disk formats at the boundary (SURVEY section 8f row 4) ------------------------------------------
 * pcl::fromROSMsg(sensor_msgs::PointCloud2, pcl::PointCloud<pcl::PointXYZRGB>) (src/node.cpp:37,41, the two clouds the
 * node receives): the caller looks the fields up by name (pcl::FieldMatches: x, y, z FLOAT32 count 1; "rgb" FLOAT32 or
 * "rgba" UINT32) and passes their byte offsets; the GPU gathers them into 32-byte pcl::PointXYZRGB rows
 * (x, y, z, 1.0f, rgba word, 12 zero bytes) in `points32` (width * height rows, host or device).  off_rgb < 0: the
 * message has no colour field, every point keeps PointXYZRGB()'s default (r = g = b = 0, a = 255).  is_bigendian is
 * ignored, as PCL ignores it.  A message whose x, y, z are consecutive floats needs no unpacking at all:
 * gicpb_set_source(ctx, data + off_x, n, point_step, ...) reads it in place.
 * The reverse, pcl::toROSMsg (Utils::cloudToROSMsg, src/Utils.cpp:100-105), is a plain copy of the 32-byte rows: the
 * message is fields x@0 y@4 z@8 rgb@16 (FLOAT32, count 1), point_step 32, row_step 32 * width. */
typedef struct gicpb_pc2_layout {
  int64_t width, height;      /* points = width * height                                                   */
  int64_t point_step;         /* bytes between points of a row                                             */
  int64_t row_step;           /* bytes between rows (>= width * point_step)                                */
  int32_t off_x, off_y, off_z; /* byte offsets of the FLOAT32 fields inside a point                        */
  int32_t off_rgb;            /* byte offset of the 4-byte rgb / rgba field, < 0: none                     */
} gicpb_pc2_layout;
int gicpb_pointcloud2_to_xyzrgb(gicpb_ctx* ctx, const void* data, int data_on_device, const gicpb_pc2_layout* layout,
                                void* points32, int points_on_device);

/* pcl::io::loadPCDFile<pcl::PointXYZRGB> (src/load_and_publish_clouds.cpp:75): PCL 1.8.1's PCDReader (header v0.7,
 * DATA ascii / binary / binary_compressed) read on the host into the PointCloud2-style blob, fields mapped to
 * PointXYZRGB rows on the GPU as above.  points32 == NULL: only the header is read (info->points tells the caller how
 * many 32-byte rows to provide); otherwise `capacity` rows must be >= info->points. */
typedef struct gicpb_pcd_info {
  int64_t width, height, points;
  int32_t point_step;          /* bytes per point in the file's own layout                                  */
  int32_t n_fields;
  int32_t data_kind;           /* 0 ascii, 1 binary, 2 binary_compressed                                    */
  int32_t is_dense;            /* 0 if the body holds a NaN / Inf (only known after the body was read)      */
  int32_t off_x, off_y, off_z, off_rgb; /* where PointXYZRGB's fields sit in the file's layout, -1: absent  */
} gicpb_pcd_info;
int gicpb_pcd_load_xyzrgb(gicpb_ctx* ctx, const char* path, void* points32, int64_t capacity, int points_on_device,
                          gicpb_pcd_info* info);

/* ---- test / inspection hooks (parity checks against the oracle) ------------------------------------- */
/* exact NN-1 of `n` queries in the target: idx = ORIGINAL target index (-1: none), d2 = float32 squared
 * distance.  max_dist <= 0 -> ungated; else only neighbours with d2 < max_dist^2 (strict) are reported. */
int gicpb_nn1(gicpb_ctx* ctx, const void* queries, int64_t n, int64_t stride_bytes, int on_device,
              const float transform[16], double max_dist, int32_t* idx, float* d2);
/* self-kNN of the target (which = 0) or source (which = 1) cloud, k = params.k_correspondences, rows in
 * ORIGINAL point order, neighbours sorted by (d2, index); idx/d2 are host arrays of n*k. */
int gicpb_knn(gicpb_ctx* ctx, int which, int32_t* idx, float* d2);
/* regularised covariances (row-major 3x3 doubles, ORIGINAL point order, host array of 9*n). */
int gicpb_get_covariances(gicpb_ctx* ctx, int which, double* cov9);
/* correspondences + Mahalanobis matrices of one outer iteration under `transform`: host arrays in ORIGINAL
 * source order (this rank's shard only when sharded): nn_idx (-1 = gated out), d2, maha9 (9 doubles each). */
int gicpb_correspondences(gicpb_ctx* ctx, const float transform[16], int32_t* nn_idx, float* d2, double* maha9,
                          int64_t* n_pairs);
/* gicpb_correspondences with the pass chosen: mode 0 = the first pass of a job (unseeded, 1 near probe ring; what
 * gicpb_correspondences runs), mode 1 = every later pass of gicpb_align (kNearMaxRing rings, each query seeded with the
 * context's current pairs when use_previous_match is on and those pairs are valid for the same Mahalanobis width). */
int gicpb_correspondences_pass(gicpb_ctx* ctx, const float transform[16], int mode, int32_t* nn_idx, float* d2,
                               double* maha9, int64_t* n_pairs);
/* one evaluation of the objective for the correspondences of the last gicpb_correspondences / align
 * iteration at x = (tx,ty,tz,roll,pitch,yaw): f and g[6] as PCL's OptimizationFunctorWithIndices::fdf */
int gicpb_cost(gicpb_ctx* ctx, const double x[6], double* f, double g[6]);
/* n_x evaluations as one inner solve of gicpb_align makes them: x = xs[6 k .. 6 k + 5], f[k], g[6 k .. 6 k + 5], all inside
 * one evaluation session - one resident kernel when cost_persistent = 1 (and cost_moments = 0), one launch per evaluation
 * otherwise.  info reports what ran. */
typedef struct gicpb_cost_session_info {
  int persistent;              /* 1: the resident kernel evaluated them                                   */
  int blocks, threads, stages; /* its grid and ring shape (threads x stages)                              */
  int pairs_per_block;         /* pairs each block owns                                                   */
  int resident_cap;            /* pairs one block can park in shared memory                               */
  int resident;                /* pairs each block parks: min(pairs_per_block, resident_cap)              */
  int epoch_first, epoch_last; /* launch epochs of the session (they differ when the kernel was relaunched) */
  int64_t launches;            /* kernels launched by the call                                            */
  int64_t n_pairs;             /* pairs summed by the last evaluation                                     */
} gicpb_cost_session_info;
int gicpb_cost_session(gicpb_ctx* ctx, int n_x, const double* xs, double* f, double* g, gicpb_cost_session_info* info);
/* grid statistics of a cloud index: which = 0 target, 1 source, 2 subtract */
typedef struct gicpb_grid_info {
  int64_t n_points, n_indexed;
  float cell_size;
  int dims[3];
  int64_t n_bricks_occupied, n_cells_occupied;
  double ms_build;
} gicpb_grid_info;
int gicpb_grid_info_get(gicpb_ctx* ctx, int which, gicpb_grid_info* out);

/* ---- micro-benchmark hooks: run one kernel `iters` times on resident data, return mean device ms ----
 * which: 0 = correspondence pass (NN + gate + Mahalanobis) under `transform`
 *        1 = cost/gradient evaluation at x derived from `transform`
 *        2 = NN-1 only (no Mahalanobis build)
 *        3 = correspondence pass with the near-probe depth of the FIRST pass of a job (initial pose)       */
int gicpb_bench_kernel(gicpb_ctx* ctx, int which, const float transform[16], int iters, double* ms_mean,
                       int64_t* launches);
/* the CUDA stream (cudaStream_t) every kernel and copy of this context is issued on: record CUDA events on it to time
 * calls on the device */
void* gicpb_stream(const gicpb_ctx* ctx);
/* number of kernels this library launched since the context was created */
int64_t gicpb_launch_count(const gicpb_ctx* ctx);
/* how many queries of the most recent search (NN-1, kNN, correspondence, fitness or difference launch) were
 * answered by the hierarchical far instance instead of the near one; -1 on error */
int64_t gicpb_last_far_queries(gicpb_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* GICP_B200_H_ */
