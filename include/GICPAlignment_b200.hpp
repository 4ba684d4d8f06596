// GICPAlignment_b200.hpp - header-only C++ drop-in for the reference's GICPAlignment class
// (reference include/GICPAlignment.h:32-224, src/GICPAlignment.cpp:23-198) and for Filter::removeFromCloud
// (reference src/Filter.cpp:176-189), on top of the C ABI of libgicp_b200.so (include/gicp_b200.h).
//
// Same class name, constructor (TARGET first), public methods, argument types and public field
// `transform_exists_`, so that LeicaStateMachine.cpp:149-153 and test/test_gicp_alignment.cpp compile unchanged
// when this header replaces <GICPAlignment.h>.  Behaviour kept on purpose, quirks included:
//   - setMaxCorrespondenceDistance(int) / setRANSACOutlierTh(int) truncate to integers   (GICPAlignment.h:138,145)
//   - applyTFtoCloud(cloud) reads `cloud` and writes the INTERNAL aligned cloud          (GICPAlignment.cpp:144-147)
//   - iterate() re-solves from the original source at identity and LEFT-multiplies the result onto the stored
//     transform; undo() restores the aligned cloud only                                  (GICPAlignment.cpp:111-142)
//   - a solve that does not converge leaves fine_tf_ and transform_exists_ untouched and only logs (:101-108)
//   - use_covariances: the points without a finite radius-search normal are dropped from the CALLER's clouds
//     (:63-67); the covariances themselves are reset by setInputSource/Target in PCL 1.8.1 and never reach the
//     solver, see getCovariances() below.
//   - setSourceCloud / setTargetCloud do not reach gicp_: iterate() keeps solving the pair of the last run()  (:111-127,166-174)
//
// With -DGICPB_WITH_PCL the clouds are pcl::PointCloud<pcl::PointXYZRGB>::Ptr and the matrix Eigen::Matrix4f, as
// in the reference.  Without it (this repo's tests; PCL and Eigen are not in the image) the same code runs on the
// 32-byte POD stand-ins below, which have the memory layout of the PCL types.
// ROS is never needed: messages go through gicpb_shim::logger() (default: stderr).  getAlignedCloudROSMsg exists
// only under -DGICPB_WITH_ROS.
#pragma once
#ifndef GICP_ALIGNMENT_B200_HPP_
#define GICP_ALIGNMENT_B200_HPP_

#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "gicp_b200.h"

#ifdef GICPB_WITH_PCL
#include <pcl/point_cloud.h>
#include <pcl/point_types.h>
#include <Eigen/Core>
#endif
#ifdef GICPB_WITH_ROS
#include <pcl_conversions/pcl_conversions.h>
#include <sensor_msgs/PointCloud2.h>
#endif

class GICPAlignment;

namespace gicpb_shim {

// ---- logging (replaces ROS_INFO / ROS_ERROR) -----------------------------------------------------------------------
enum LogLevel { kInfo = 0, kWarn = 1, kError = 2 };
typedef void (*LogFn)(int level, const char* message);
inline void default_logger(int level, const char* message) {
  std::fprintf(stderr, "[%s] %s\n", level == kError ? "ERROR" : (level == kWarn ? " WARN" : " INFO"), message);
}
inline LogFn& logger() {
  static LogFn fn = &default_logger;
  return fn;
}
inline void log(int level, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  std::vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (logger()) logger()(level, buf);
}

#ifndef GICPB_WITH_PCL
// ---- stand-ins with the memory layout of pcl::PointXYZRGB / pcl::PointCloud / Eigen::Matrix4f -----------------------
struct alignas(16) PointXYZRGB {
  float x = 0.f, y = 0.f, z = 0.f, w = 1.f;  // PCL's padding float holds 1.0
  union {
    float rgb;
    struct { uint8_t b, g, r, a; };
  };
  float pad_[3] = {0.f, 0.f, 0.f};
  PointXYZRGB() : rgb(0.f) { a = 255; }  // pcl::PointXYZRGB(): r = g = b = 0, a = 255
};
static_assert(sizeof(PointXYZRGB) == 32, "pcl::PointXYZRGB is 32 bytes");

struct PointCloudRGB {
  typedef std::shared_ptr<PointCloudRGB> Ptr;
  std::vector<PointXYZRGB> points;
  uint32_t width = 0, height = 1;
  bool is_dense = true;
  size_t size() const { return points.size(); }
  bool empty() const { return points.empty(); }
  void resize(size_t n) {
    points.resize(n);
    width = (uint32_t)n;
    height = 1;
  }
};

struct Matrix4f {  // column-major like Eigen::Matrix4f
  float m[16];
  static Matrix4f Identity() {
    Matrix4f r;
    for (int i = 0; i < 16; ++i) r.m[i] = (i % 5 == 0) ? 1.f : 0.f;
    return r;
  }
  float& operator()(int row, int col) { return m[4 * col + row]; }
  float operator()(int row, int col) const { return m[4 * col + row]; }
  const float* data() const { return m; }
  float* data() { return m; }
  bool operator==(const Matrix4f& o) const { return std::memcmp(m, o.m, sizeof(m)) == 0; }
  bool operator!=(const Matrix4f& o) const { return !(*this == o); }
  Matrix4f operator*(const Matrix4f& o) const {  // float product, row by column in index order
    Matrix4f r;
    for (int i = 0; i < 4; ++i)
      for (int j = 0; j < 4; ++j) {
        float s = 0.f;
        for (int k = 0; k < 4; ++k) s += (*this)(i, k) * o(k, j);
        r(i, j) = s;
      }
    return r;
  }
};
typedef PointCloudRGB CloudT;
typedef Matrix4f Mat4T;
#else
typedef pcl::PointCloud<pcl::PointXYZRGB> CloudT;
typedef Eigen::Matrix4f Mat4T;
#endif

inline void to_row_major(const Mat4T& m, float out[16]) {
  for (int r = 0; r < 4; ++r)
    for (int c = 0; c < 4; ++c) out[4 * r + c] = m(r, c);
}
inline Mat4T from_row_major(const float in[16]) {
  Mat4T m = Mat4T::Identity();
  for (int r = 0; r < 4; ++r)
    for (int c = 0; c < 4; ++c) m(r, c) = in[4 * r + c];
  return m;
}
inline Mat4T identity4() { return Mat4T::Identity(); }

// Utils::isValidTransform (reference src/Utils.cpp:71-82): no NaN entry
inline bool isValidTransform(const Mat4T& tf) {
  for (int r = 0; r < 4; ++r)
    for (int c = 0; c < 4; ++c)
      if (std::isnan(tf(r, c))) return false;
  return true;
}

// One engine context (stream, pinned staging ring, device buffers) is shared by every shim object of the process by
// default - GICPAlignment, removeFromCloud, FODDetector, downsampleCloud, getNormals, the cloud I/O helpers - as one
// LeicaStateMachine run uses them one after the other (reference src/LeicaStateMachine.cpp:138-216): nothing is created
// and torn down per stage.  Device from GICPB_DEVICE (default 0).  A context is not thread-safe: objects used from
// several threads at once need their own (`Context::create()`).
class Context {
 public:
  // GICPB_DEVICES=0,1,2,3 (more than one GPU): the registration and removeFromCloud's difference run sharded over them
  // inside this process (gicpb_group); GICPB_DEVICE=n or nothing: one context on that GPU.  get() is always a full single-GPU context (the group's first).
  Context() {
    std::vector<int> devices;
    if (const char* e = std::getenv("GICPB_DEVICES")) {
      for (const char* p = e; *p;) {
        char* end = nullptr;
        const long d = std::strtol(p, &end, 10);
        if (end == p) break;
        devices.push_back((int)d);
        p = (*end == ',') ? end + 1 : end;
      }
    }
    if (devices.size() > 1) {
      const int rc = gicpb_group_create(devices.data(), (int)devices.size(), &group_);
      if (rc != GICPB_OK || !group_)
        throw std::runtime_error("gicpb_group_create failed (" + std::to_string(rc) + "): GICPB_DEVICES must name B200s");
      ctx_ = gicpb_group_ctx(group_, 0);
      return;
    }
    int device = devices.empty() ? 0 : devices[0];
    if (devices.empty())
      if (const char* e = std::getenv("GICPB_DEVICE")) device = std::atoi(e);
    const int rc = gicpb_create(device, &ctx_);
    if (rc != GICPB_OK || !ctx_)
      throw std::runtime_error("gicpb_create failed (" + std::to_string(rc) + "): libgicp_b200 needs a B200; there is no CPU path");
  }
  ~Context() {
    if (group_)
      gicpb_group_destroy(group_);
    else
      gicpb_destroy(ctx_);
  }
  Context(const Context&) = delete;
  Context& operator=(const Context&) = delete;
  gicpb_ctx* get() const { return ctx_; }
  bool grouped() const { return group_ != nullptr; }
  int gpus() const { return group_ ? gicpb_group_size(group_) : 1; }
  void check(int rc, const char* what) const {
    if (rc != GICPB_OK) throw std::runtime_error(std::string(what) + ": " + gicpb_last_error(ctx_));
  }
  void check_group(int rc, const char* what) const {
    if (rc != GICPB_OK) throw std::runtime_error(std::string(what) + ": " + gicpb_group_last_error(group_));
  }
  // the registration calls: on every GPU of the group, or on the one context
  void setParams(const gicpb_params& p) {
    if (group_)
      check_group(gicpb_group_set_params(group_, &p), "gicpb_group_set_params");
    else
      check(gicpb_set_params(ctx_, &p), "gicpb_set_params");
  }
  int align(gicpb_align_result* out) { return group_ ? gicpb_group_align(group_, out) : gicpb_align(ctx_, out); }
  void fitness(const float T[16], double max_range, double* score) {
    if (group_)
      check_group(gicpb_group_fitness(group_, T, max_range, score), "gicpb_group_fitness");
    else
      check(gicpb_fitness(ctx_, T, max_range, score), "gicpb_fitness");
  }
  // Filter::removeFromCloud's difference of two host clouds: on every GPU of the group, or on the one context
  void cloudDifference(const void* input, int64_t n_input, int64_t input_stride, const void* subtract, int64_t n_subtract,
                       int64_t subtract_stride, double sqr_threshold, uint8_t* mask, int64_t* n_kept) const {
    if (group_)
      check_group(gicpb_group_cloud_difference(group_, input, n_input, input_stride, subtract, n_subtract, subtract_stride,
                                               sqr_threshold, mask, n_kept),
                  "gicpb_group_cloud_difference");
    else
      check(gicpb_cloud_difference(ctx_, input, n_input, input_stride, subtract, n_subtract, subtract_stride, 0,
                                   sqr_threshold, mask, n_kept),
            "gicpb_cloud_difference");
  }
  const char* lastError() const { return group_ ? gicpb_group_last_error(group_) : gicpb_last_error(ctx_); }
  static std::shared_ptr<Context> create() { return std::make_shared<Context>(); }
  // the process-wide context (created on first use, destroyed at exit or by release_shared())
  static std::shared_ptr<Context>& shared_slot() {
    static std::shared_ptr<Context> slot;
    return slot;
  }
  static std::shared_ptr<Context> shared() {
    std::shared_ptr<Context>& slot = shared_slot();
    if (!slot) slot = create();
    return slot;
  }
  static void release_shared() { shared_slot().reset(); }
  // The registration inputs (target / source index, covariances) inside the context belong to the object that set them
  // last; an object that finds another owner sets its own inputs again before it solves.
  const void* inputs_owner = nullptr;

 private:
  gicpb_ctx* ctx_ = nullptr;
  gicpb_group* group_ = nullptr;
  friend class ::GICPAlignment;
};

inline Context* resolve(Context* given, std::shared_ptr<Context>& hold) {
  if (given) return given;
  hold = Context::shared();
  return hold.get();
}

// pcl::transformPointCloud(in, out, tf): every field copied, xyz <- tf * xyz (reference src/GICPAlignment.cpp:146)
inline void transformCloud(const Context& ctx, const CloudT& in, CloudT& out, const Mat4T& tf) {
  if (&in != &out) out = in;
  if (in.points.empty()) return;
  float T[16];
  to_row_major(tf, T);
  ctx.check(gicpb_transform_cloud(ctx.get(), T, &in.points[0].x, &out.points[0].x, (int64_t)in.points.size(),
                                  (int64_t)sizeof(in.points[0]), 0),
            "gicpb_transform_cloud");
}

// Filter::removeFromCloud (reference src/Filter.cpp:176-189): keep the points of `input_cloud` whose SQUARED distance
// to their nearest neighbour in `substract_cloud` exceeds `threshold`, in input order; height 1, is_dense true.
template <class CloudPtr>
inline void removeFromCloud(const CloudPtr& input_cloud, const CloudPtr& substract_cloud, double threshold,
                            const CloudPtr& cloud_filtered, Context* shared = nullptr) {
  log(kInfo, "Difference from segment with threshold: %f", threshold);
  std::shared_ptr<Context> hold;
  shared = resolve(shared, hold);
  const int64_t n = (int64_t)input_cloud->points.size();
  std::vector<uint8_t> mask((size_t)n);
  int64_t kept = 0;
  if (n > 0 && !substract_cloud->points.empty()) {
    shared->cloudDifference(&input_cloud->points[0].x, n, (int64_t)sizeof(input_cloud->points[0]), &substract_cloud->points[0].x,
                            (int64_t)substract_cloud->points.size(), (int64_t)sizeof(substract_cloud->points[0]), threshold,
                            mask.data(), &kept);
  }
  CloudT out;
  out.points.reserve((size_t)kept);
  for (int64_t i = 0; i < n; ++i)
    if (mask[(size_t)i]) out.points.push_back(input_cloud->points[(size_t)i]);
  out.width = (uint32_t)out.points.size();
  out.height = 1;
  out.is_dense = true;
  *cloud_filtered = out;  // safe when cloud_filtered aliases input_cloud
}

// Utils::computeCloudResolution (reference src/Utils.cpp:145-174): mean distance to the 2nd nearest neighbour (the 1st
// is the point itself) over the finite points
template <class CloudPtr>
inline double computeCloudResolution(const CloudPtr& cloud, Context* shared = nullptr) {
  if (cloud->points.empty()) return 0.0;
  std::shared_ptr<Context> hold;
  shared = resolve(shared, hold);
  double res = 0.0;
  shared->check(gicpb_difference_set_subtract(shared->get(), &cloud->points[0].x, (int64_t)cloud->points.size(),
                                              (int64_t)sizeof(cloud->points[0]), 0),
                "gicpb_difference_set_subtract");  // the context's third index slot
  shared->check(gicpb_cloud_resolution(shared->get(), 2, &res), "gicpb_cloud_resolution");
  return res;
}

#ifndef GICPB_WITH_PCL
struct alignas(16) Normal {  // memory layout of pcl::Normal
  float normal_x = 0.f, normal_y = 0.f, normal_z = 0.f, pad_n_ = 0.f;
  float curvature = 0.f, pad_c_[3] = {0.f, 0.f, 0.f};
};
static_assert(sizeof(Normal) == 32, "pcl::Normal is 32 bytes");
struct PointCloudNormal {
  typedef std::shared_ptr<PointCloudNormal> Ptr;
  std::vector<Normal> points;
  uint32_t width = 0, height = 1;
  bool is_dense = true;
  size_t size() const { return points.size(); }
};
typedef PointCloudNormal NormalCloudT;
#else
typedef pcl::PointCloud<pcl::Normal> NormalCloudT;
#endif

// Utils::getNormals (reference src/Utils.cpp:27-44): pcl::NormalEstimation with a radius search and the default viewpoint
// (0, 0, 0); one normal per point (NaN x 4 where PCL gives none, is_dense then false).  Returns what the reference
// returns: normals->size() == cloud->size().
template <class CloudPtr, class NormalsPtr>
inline bool getNormals(const CloudPtr& cloud, double normal_radius, const NormalsPtr& normals, Context* shared = nullptr) {
  log(kInfo, "Computing normals with radius: %f", normal_radius);
  std::shared_ptr<Context> hold;
  shared = resolve(shared, hold);
  const int64_t n = (int64_t)cloud->points.size();
  normals->points.resize((size_t)n);
  normals->width = (uint32_t)n;
  normals->height = 1;
  normals->is_dense = true;
  if (n == 0) return true;
  std::vector<float> out((size_t)n * 4);
  int64_t finite = 0;
  shared->check(gicpb_difference_set_subtract(shared->get(), &cloud->points[0].x, n, (int64_t)sizeof(cloud->points[0]), 0),
                "gicpb_difference_set_subtract");  // the context's third index slot
  shared->check(gicpb_normals(shared->get(), 2, normal_radius, out.data(), &finite), "gicpb_normals");
  for (int64_t i = 0; i < n; ++i) {
    normals->points[(size_t)i].normal_x = out[4 * (size_t)i];
    normals->points[(size_t)i].normal_y = out[4 * (size_t)i + 1];
    normals->points[(size_t)i].normal_z = out[4 * (size_t)i + 2];
    normals->points[(size_t)i].curvature = out[4 * (size_t)i + 3];
  }
  normals->is_dense = finite == n;
  return normals->points.size() == cloud->points.size();
}

}  // namespace gicpb_shim

class GICPAlignment {
 public:
  typedef gicpb_shim::CloudT PointCloudRGB;
  typedef std::shared_ptr<PointCloudRGB> PointCloudRGBPtr;
#ifdef GICPB_WITH_PCL
  typedef PointCloudRGB::Ptr CloudPtr;  // boost::shared_ptr in PCL 1.8
#else
  typedef PointCloudRGBPtr CloudPtr;
#endif
  typedef gicpb_shim::Mat4T Matrix4f;

  // reference src/GICPAlignment.cpp:23-35
  GICPAlignment(CloudPtr target_cloud, CloudPtr source_cloud, bool use_covariances)
      : transform_exists_(false), covariances_(use_covariances), fine_tf_(gicpb_shim::identity4()), max_iter_(100),
        tf_epsilon_(4e-3), max_corresp_distance_(4e-2), ransac_outlier_th_(1.0), target_cloud_(target_cloud),
        source_cloud_(source_cloud), aligned_cloud_(new PointCloudRGB), backup_cloud_(new PointCloudRGB),
        converged_(false), fitness_(-1.0), inputs_set_(false), tgt_indexed_(false), src_indexed_(false), last_(),
        ctx_holder_(gicpb_shim::Context::shared()), ctx_(*ctx_holder_) {}
  // the same, on a context of the caller's (one per thread when objects run concurrently)
  GICPAlignment(CloudPtr target_cloud, CloudPtr source_cloud, bool use_covariances, std::shared_ptr<gicpb_shim::Context> context)
      : transform_exists_(false), covariances_(use_covariances), fine_tf_(gicpb_shim::identity4()), max_iter_(100),
        tf_epsilon_(4e-3), max_corresp_distance_(4e-2), ransac_outlier_th_(1.0), target_cloud_(target_cloud),
        source_cloud_(source_cloud), aligned_cloud_(new PointCloudRGB), backup_cloud_(new PointCloudRGB),
        converged_(false), fitness_(-1.0), inputs_set_(false), tgt_indexed_(false), src_indexed_(false), last_(),
        ctx_holder_(context), ctx_(*ctx_holder_) {}

  ~GICPAlignment() {}

  bool transform_exists_;  // reference include/GICPAlignment.h:56

  void run() {  // :37-46
    tgt_indexed_ = src_indexed_ = false;  // the caller may have edited the clouds since the last call
    configParameters();
    if (covariances_) applyCovariances();
    fineAlignment();
    applyTFtoCloud(source_cloud_);
  }
  void iterate() { iterateFineAlignment(aligned_cloud_); }  // :129-132
  void undo() { *aligned_cloud_ = *backup_cloud_; }         // :139-142

  Matrix4f getFineTransform() {  // :149-154
    if (!transform_exists_) gicpb_shim::log(gicpb_shim::kError, "No transform yet. Please run algorithm");
    return fine_tf_;
  }
  void getAlignedCloud(CloudPtr aligned_cloud) { *aligned_cloud = *aligned_cloud_; }  // :156-159 (deep copy)
#ifdef GICPB_WITH_ROS
  void getAlignedCloudROSMsg(sensor_msgs::PointCloud2& aligned_cloud_msg) {  // :161-164
    pcl::toROSMsg(*aligned_cloud_, aligned_cloud_msg);
  }
#endif
  void applyTFtoCloud(CloudPtr cloud) {  // :144-147
    gicpb_shim::transformCloud(ctx_, *cloud, *aligned_cloud_, fine_tf_);
  }
  // :166-174: only the wrapper's pointers change.  gicp_ keeps the clouds given to setInputSource / setInputTarget by the
  // last fineAlignment (:89-90), so a following iterate() still solves the OLD pair; the new cloud counts from the next run()
  void setSourceCloud(CloudPtr source_cloud) { source_cloud_ = source_cloud; }
  void setTargetCloud(CloudPtr target_cloud) { target_cloud_ = target_cloud; }
  void setMaxIterations(int iterations) {  // :176-180
    max_iter_ = iterations;
    configParameters();
  }
  void setTfEpsilon(double tf_epsilon) {  // :182-186
    tf_epsilon_ = tf_epsilon;
    configParameters();
  }
  void setMaxCorrespondenceDistance(int max_corresp_distance) {  // :188-192, int on purpose
    max_corresp_distance_ = max_corresp_distance;
    configParameters();
  }
  void setRANSACOutlierTh(int ransac_threshold) {  // :194-198, int on purpose; GICP never uses it
    ransac_outlier_th_ = ransac_threshold;
    configParameters();
  }

  // ---- additions that do not break the reference surface (north_star: fitness score, convergence) ---------------
  bool hasConverged() const { return converged_; }
  double getFitnessScore() const { return fitness_; }
  const gicpb_align_result& lastResult() const { return last_; }

 private:
  bool covariances_;
  Matrix4f fine_tf_;
  int max_iter_;
  double tf_epsilon_;
  double max_corresp_distance_;
  double ransac_outlier_th_;
  CloudPtr target_cloud_, source_cloud_, aligned_cloud_, backup_cloud_;
  bool converged_;
  double fitness_;
  bool inputs_set_;                 // gicp_ holds input clouds (set by the last fineAlignment)
  bool tgt_indexed_, src_indexed_;  // within one run(): the context's index of that cloud is current
  CloudPtr input_target_, input_source_;  // what gicp_.setInputTarget / setInputSource were given (:89-90)
  gicpb_align_result last_;
  // replaces the pcl::GeneralizedIterativeClosestPoint member gicp_ (GICPAlignment.h:153)
  std::shared_ptr<gicpb_shim::Context> ctx_holder_;
  gicpb_shim::Context& ctx_;

  void configParameters() {  // :48-54
    gicpb_params p;
    ctx_.check(gicpb_get_params(ctx_.get(), &p), "gicpb_get_params");
    p.max_iterations = max_iter_;
    p.max_corr_distance = max_corresp_distance_;
    p.transformation_epsilon = tf_epsilon_;
    ctx_.setParams(p);
  }

  void indexCloud(int which, const CloudPtr& cloud) {
    if (cloud->points.empty()) throw std::runtime_error("empty cloud");
    const int rc = which == 0 ? gicpb_set_target(ctx_.get(), &cloud->points[0].x, (int64_t)cloud->points.size(),
                                                 (int64_t)sizeof(cloud->points[0]), 0)
                              : gicpb_set_source(ctx_.get(), &cloud->points[0].x, (int64_t)cloud->points.size(),
                                                 (int64_t)sizeof(cloud->points[0]), 0);
    ctx_.check(rc, which == 0 ? "gicpb_set_target" : "gicpb_set_source");
    ctx_.inputs_owner = this;
    (which == 0 ? tgt_indexed_ : src_indexed_) = true;
  }
  void ensureIndexed() {  // index only (no kNN-20 covariances): all the resolution and the normals need
    if (ctx_.inputs_owner != this) tgt_indexed_ = src_indexed_ = false;
    if (!tgt_indexed_) indexCloud(0, target_cloud_);
    if (!src_indexed_) indexCloud(1, source_cloud_);
  }

  // :56-71 for one cloud.  Both resolutions are recomputed on every call, as upstream does.  The radius-search normals
  // only decide WHICH points survive: pcl::NormalEstimation gives NaN to a point with fewer than 3 points inside the
  // radius, removeNaNNormalsFromPointCloud + Filter::extractIndices then drop it from the CALLER's cloud (:63-67).  The
  // covariances built from the normals (:70) are reset by setInputSource / setInputTarget in PCL 1.8.1 (:89-90,
  // SURVEY App. A.1) and never reach the solver, so they are not built.  A cloud is indexed again only after it lost
  // points: one run() with use_covariances builds 2 indices when nothing is dropped, at most 4.
  void getCovariances(CloudPtr cloud, bool is_source) {
    ensureIndexed();
    double target_res = 0, source_res = 0;
    ctx_.check(gicpb_cloud_resolution(ctx_.get(), 0, &target_res), "gicpb_cloud_resolution");
    ctx_.check(gicpb_cloud_resolution(ctx_.get(), 1, &source_res), "gicpb_cloud_resolution");
    const double normal_radius = (target_res + source_res) * 2.0;  // doubled
    gicpb_shim::log(gicpb_shim::kInfo, "Computing normals with radius: %f", normal_radius);
    std::vector<uint8_t> valid(cloud->points.size());
    int64_t kept = 0;
    ctx_.check(gicpb_normal_validity(ctx_.get(), is_source ? 1 : 0, normal_radius, valid.data(), &kept),
               "gicpb_normal_validity");
    if ((size_t)kept != cloud->points.size()) {
      size_t w = 0;
      for (size_t i = 0; i < cloud->points.size(); ++i)
        if (valid[i]) cloud->points[w++] = cloud->points[i];
      cloud->points.resize(w);
      cloud->width = (uint32_t)w;
      cloud->height = 1;
      (is_source ? src_indexed_ : tgt_indexed_) = false;
    }
  }

  void applyCovariances() {  // :73-84: source first, then target
    gicpb_shim::log(gicpb_shim::kInfo, "Extract covariances from clouds");
    getCovariances(source_cloud_, true);
    getCovariances(target_cloud_, false);
  }

  // gicp_.setInputSource / setInputTarget (:89-90) + the index builds and kNN-20 covariances PCL's align() starts with
  void setInputs(const CloudPtr& target, const CloudPtr& source, bool reuse_indices) {
    if (source->points.empty() || target->points.empty()) throw std::runtime_error("empty cloud");
    if (ctx_.inputs_owner != this) tgt_indexed_ = src_indexed_ = false;
    if (ctx_.grouped()) {
      // every GPU of the group uploads and indexes the target, and its shard's share of the work on the source
      ctx_.check_group(gicpb_group_set_clouds(ctx_.group_, &target->points[0].x, (int64_t)target->points.size(),
                                              (int64_t)sizeof(target->points[0]), &source->points[0].x,
                                              (int64_t)source->points.size(), (int64_t)sizeof(source->points[0])),
                       "gicpb_group_set_clouds");
    } else if (reuse_indices && (tgt_indexed_ || src_indexed_)) {
      // applyCovariances has just indexed these very clouds: index what changed since, then the covariances
      ensureIndexed();
      ctx_.check(gicpb_compute_covariances(ctx_.get()), "gicpb_compute_covariances");
    } else {
      // both uploads go to the copy stream, target first: the source uploads while the target is being indexed; then
      // one call indexes both clouds and computes their covariances (the target's beside the source's index build)
      ctx_.check(gicpb_prefetch_cloud(ctx_.get(), 0, &target->points[0].x, (int64_t)target->points.size(),
                                      (int64_t)sizeof(target->points[0])),
                 "gicpb_prefetch_cloud");
      ctx_.check(gicpb_prefetch_cloud(ctx_.get(), 1, &source->points[0].x, (int64_t)source->points.size(),
                                      (int64_t)sizeof(source->points[0])),
                 "gicpb_prefetch_cloud");
      ctx_.check(gicpb_set_clouds(ctx_.get(), &target->points[0].x, (int64_t)target->points.size(),
                                  (int64_t)sizeof(target->points[0]), &source->points[0].x, (int64_t)source->points.size(),
                                  (int64_t)sizeof(source->points[0]), 0),
                 "gicpb_set_clouds");
    }
    ctx_.inputs_owner = this;
    tgt_indexed_ = src_indexed_ = true;
    input_target_ = target;
    input_source_ = source;
    inputs_set_ = true;
  }

  // gicp_.align(): solver failures are not errors of the call (PCL swallows them: hasConverged() == false)
  int align() {
    const int rc = ctx_.align(&last_);
    if (rc == GICPB_E_BADARG || rc == GICPB_E_CUDA || rc == GICPB_E_NCCL || rc == GICPB_E_STATE)
      throw std::runtime_error(std::string("gicpb_align: ") + ctx_.lastError());
    converged_ = last_.converged != 0;
    return rc;
  }

  void fineAlignment() {  // :86-109
    gicpb_shim::log(gicpb_shim::kInfo, "Perform GICP with %d iterations", max_iter_);
    setInputs(target_cloud_, source_cloud_, true);
    const auto begin = std::chrono::steady_clock::now();
    gicpb_shim::log(gicpb_shim::kInfo, "This step may take a while ...");
    align();
    const double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - begin).count();
    gicpb_shim::log(gicpb_shim::kInfo, "GICP time: %lf s", secs);
    if (converged_) {
      ctx_.fitness(last_.transform, 1.7976931348623157e308, &fitness_);
      gicpb_shim::log(gicpb_shim::kInfo, "Converged in %f FitnessScore", fitness_);
      fine_tf_ = gicpb_shim::from_row_major(last_.transform);
      transform_exists_ = gicpb_shim::isValidTransform(fine_tf_);
    } else {
      gicpb_shim::log(gicpb_shim::kError, "GICP no converge");
    }
  }

  void iterateFineAlignment(CloudPtr cloud) {  // :111-127
    backUp(cloud);
    gicpb_shim::log(gicpb_shim::kInfo, "Computing iteration...");
    if (!inputs_set_) {  // gicp_.align() without input clouds: PCL's initCompute fails, nothing converges, `cloud` is untouched
      converged_ = false;
      gicpb_shim::log(gicpb_shim::kError, "GICP no converge");
      return;
    }
    // gicp_ still holds the clouds of the last fineAlignment, whatever setSourceCloud / setTargetCloud were given since;
    // if another object used the shared context in between, they are set again (the clouds are held by pointer, as in PCL)
    if (ctx_.inputs_owner != this) setInputs(input_target_, input_source_, false);
    align();  // PCL's align() restarts from the stored input source at identity (SURVEY App. A.6)
    const Matrix4f temp_tf = gicpb_shim::from_row_major(last_.transform);
    if (converged_) {
      fine_tf_ = temp_tf * fine_tf_;
      ctx_.fitness(last_.transform, 1.7976931348623157e308, &fitness_);
      gicpb_shim::log(gicpb_shim::kInfo, "Converged in %f FitnessScore", fitness_);
    } else {
      gicpb_shim::log(gicpb_shim::kError, "GICP no converge");
    }
    // align(*cloud) overwrites `cloud` with final_transformation * input source
    gicpb_shim::transformCloud(ctx_, *input_source_, *cloud, temp_tf);
  }

  void backUp(CloudPtr cloud) { *backup_cloud_ = *cloud; }  // :134-137
};

#endif  // GICP_ALIGNMENT_B200_HPP_
