// oracle/gicp_oracle.cpp
//
// TEST INFRASTRUCTURE ONLY.  CPU restatement of the reference's GICP hot path.  Nothing in the shipped
// library (leica_point_cloud_processing_b200/csrc) includes, links or calls this file; only tests/,
// __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs load it.
//
// PARITY UNPINNED: the arithmetic of this path lives in PCL 1.8.1 (+ FLANN 1.8, Eigen 3), which is a
// third-party dependency that is NOT vendored in /root/reference and is absent from this image
// (reference CMakeLists.txt:9, .travis.yml:11).  The reference's own tests hold no golden transform /
// fitness value for the path (test/test_gicp_alignment.cpp:50-131 only checks identity-at-construction
// and transform_exists_).  This file therefore restates the *published* PCL 1.8.1 / GSL algorithms and is
// anchored on the reference's call sites and on the fixture facts its tests imply (see tests/test_oracle.py).
//
// What is restated, and from where:
//   * cube fixture sampler ............ reference src/CADToPointCloud.cpp:101-190 (libc rand(), no srand)
//   * rotateCloud / transformPointCloud  reference src/Utils.cpp:215-232, PCL common/impl/transforms.hpp
//   * exact NN / kNN ................... PCL kdtree_flann (FLANN KDTreeSingleIndex, L2_Simple, exact search);
//                                        ties are broken towards the lowest index (BASELINE.json north_star)
//   * computeCovariances ............... PCL registration/impl/gicp.hpp (kNN-20, float products summed in
//                                        double, SVD, singular values -> (1, 1, gicp_epsilon))
//   * computeTransformation ............ PCL registration/impl/gicp.hpp (outer loop, Mahalanobis matrices,
//                                        delta test), call sites reference src/GICPAlignment.cpp:96,116
//   * estimateRigidTransformationBFGS .. PCL gicp.hpp + registration/bfgs.h (port of GSL vector_bfgs2 and
//                                        linear_minimize.c)
//   * getFitnessScore .................. PCL registration/impl/registration.hpp, reference
//                                        src/GICPAlignment.cpp:103,123
//   * getPointCloudDifference .......... PCL segmentation/impl/segment_differences.hpp, reference
//                                        src/Filter.cpp:176-189
//   * computeCloudResolution ........... reference src/Utils.cpp:145-174
//   * extractEuclideanClusters ......... PCL segmentation/impl/extract_clusters.hpp, reference
//                                        src/FODDetector.cpp:45-58
//   * VoxelGrid::applyFilter ........... PCL filters/impl/voxel_grid.hpp + common/impl/accumulators.hpp, reference
//                                        src/Filter.cpp:91-105
//
// Build (parity):  g++ -O2 -ffp-contract=off -fPIC -shared  (single thread, no FMA contraction)
// Build (timing):  g++ -O3 -march=native -fopenmp -fPIC -shared  (all host cores over points)

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <limits>
#include <numeric>
#include <vector>

#ifdef _OPENMP
#include <omp.h>
#endif

namespace {

// ----------------------------------------------------------------------------------------------------
// small linear algebra helpers (row-major 3x3 doubles, row-major 4x4 floats)
// ----------------------------------------------------------------------------------------------------
struct Mat3 {
  double m[9];
  double& operator()(int r, int c) { return m[3 * r + c]; }
  double operator()(int r, int c) const { return m[3 * r + c]; }
};

Mat3 mat3_zero() {
  Mat3 a;
  for (double& v : a.m) v = 0.0;
  return a;
}
Mat3 mat3_identity() {
  Mat3 a = mat3_zero();
  a(0, 0) = a(1, 1) = a(2, 2) = 1.0;
  return a;
}
Mat3 mat3_mul(const Mat3& a, const Mat3& b) {
  Mat3 c = mat3_zero();
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      double s = 0.0;
      for (int k = 0; k < 3; ++k) s += a(i, k) * b(k, j);
      c(i, j) = s;
    }
  return c;
}
Mat3 mat3_transpose(const Mat3& a) {
  Mat3 t;
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) t(i, j) = a(j, i);
  return t;
}
// 3x3 inverse through the adjugate, as Eigen does for fixed 3x3 matrices (Matrix3d::inverse()).
Mat3 mat3_inverse(const Mat3& a) {
  Mat3 c;
  c(0, 0) = a(1, 1) * a(2, 2) - a(1, 2) * a(2, 1);
  c(0, 1) = a(0, 2) * a(2, 1) - a(0, 1) * a(2, 2);
  c(0, 2) = a(0, 1) * a(1, 2) - a(0, 2) * a(1, 1);
  c(1, 0) = a(1, 2) * a(2, 0) - a(1, 0) * a(2, 2);
  c(1, 1) = a(0, 0) * a(2, 2) - a(0, 2) * a(2, 0);
  c(1, 2) = a(0, 2) * a(1, 0) - a(0, 0) * a(1, 2);
  c(2, 0) = a(1, 0) * a(2, 1) - a(1, 1) * a(2, 0);
  c(2, 1) = a(0, 1) * a(2, 0) - a(0, 0) * a(2, 1);
  c(2, 2) = a(0, 0) * a(1, 1) - a(0, 1) * a(1, 0);
  double det = a(0, 0) * c(0, 0) + a(0, 1) * c(1, 0) + a(0, 2) * c(2, 0);
  double inv = 1.0 / det;
  for (double& v : c.m) v *= inv;
  return c;
}

// Cyclic Jacobi eigen-decomposition of a symmetric 3x3 matrix (double).  For a symmetric positive
// semi-definite input this yields what Eigen::JacobiSVD(ComputeFullU) yields up to column signs:
// U = eigenvectors, singular values = |eigenvalues|.  Columns are returned sorted by descending |lambda|.
void sym3_eig_desc(const Mat3& in, double lam[3], Mat3& U) {
  Mat3 a = in;
  Mat3 v = mat3_identity();
  for (int sweep = 0; sweep < 64; ++sweep) {
    double off = std::fabs(a(0, 1)) + std::fabs(a(0, 2)) + std::fabs(a(1, 2));
    double diag = std::fabs(a(0, 0)) + std::fabs(a(1, 1)) + std::fabs(a(2, 2));
    if (off == 0.0 || off <= 1e-300 || off < 1e-22 * diag) break;
    for (int p = 0; p < 2; ++p)
      for (int q = p + 1; q < 3; ++q) {
        double apq = a(p, q);
        if (apq == 0.0) continue;
        double theta = (a(q, q) - a(p, p)) / (2.0 * apq);
        double t = (theta >= 0.0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
        double c = 1.0 / std::sqrt(t * t + 1.0);
        double s = t * c;
        // A <- J^T A J with J = rotation in the (p,q) plane
        for (int k = 0; k < 3; ++k) {
          double akp = a(k, p), akq = a(k, q);
          a(k, p) = c * akp - s * akq;
          a(k, q) = s * akp + c * akq;
        }
        for (int k = 0; k < 3; ++k) {
          double apk = a(p, k), aqk = a(q, k);
          a(p, k) = c * apk - s * aqk;
          a(q, k) = s * apk + c * aqk;
        }
        for (int k = 0; k < 3; ++k) {
          double vkp = v(k, p), vkq = v(k, q);
          v(k, p) = c * vkp - s * vkq;
          v(k, q) = s * vkp + c * vkq;
        }
      }
  }
  int order[3] = {0, 1, 2};
  double ev[3] = {a(0, 0), a(1, 1), a(2, 2)};
  std::stable_sort(order, order + 3, [&](int x, int y) { return std::fabs(ev[x]) > std::fabs(ev[y]); });
  for (int k = 0; k < 3; ++k) {
    lam[k] = ev[order[k]];
    for (int r = 0; r < 3; ++r) U(r, k) = v(r, order[k]);
  }
}

struct Mat4f {
  float m[16];  // row-major
  float& operator()(int r, int c) { return m[4 * r + c]; }
  float operator()(int r, int c) const { return m[4 * r + c]; }
};
Mat4f mat4f_identity() {
  Mat4f t;
  for (int i = 0; i < 16; ++i) t.m[i] = (i % 5 == 0) ? 1.0f : 0.0f;
  return t;
}
Mat4f mat4f_mul(const Mat4f& a, const Mat4f& b) {
  Mat4f c;
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 4; ++j) {
      float s = a(i, 0) * b(0, j);
      for (int k = 1; k < 4; ++k) s = s + a(i, k) * b(k, j);
      c(i, j) = s;
    }
  return c;
}

// Float point transform in the order Eigen's fixed-size 4x4 * 4x1 (w = 1) product evaluates it:
// ((c0*x + c1*y) + c2*z) + c3.  Used for `transformation_ * query` (gicp.hpp) and transformPointCloud.
inline void xform_point(const Mat4f& t, const float* p, float* q) {
  float x = p[0], y = p[1], z = p[2];
  q[0] = ((t(0, 0) * x + t(0, 1) * y) + t(0, 2) * z) + t(0, 3);
  q[1] = ((t(1, 0) * x + t(1, 1) * y) + t(1, 2) * z) + t(1, 3);
  q[2] = ((t(2, 0) * x + t(2, 1) * y) + t(2, 2) * z) + t(2, 3);
}

// squared distance the way FLANN's L2_Simple accumulates it in float: ((dx*dx) + dy*dy) + dz*dz
inline float sqdist(const float* a, const float* b) {
  float dx = a[0] - b[0], dy = a[1] - b[1], dz = a[2] - b[2];
  return (dx * dx + dy * dy) + dz * dz;
}

struct Quatf {
  float w, x, y, z;
};
Quatf quat_from_axis_angle(float angle, int axis) {  // Eigen: Quaternion = AngleAxis
  float ha = 0.5f * angle;
  Quatf q{std::cos(ha), 0.f, 0.f, 0.f};
  float s = std::sin(ha);
  if (axis == 0) q.x = s;
  if (axis == 1) q.y = s;
  if (axis == 2) q.z = s;
  return q;
}
Quatf quat_mul(const Quatf& a, const Quatf& b) {
  Quatf r;
  r.w = a.w * b.w - a.x * b.x - a.y * b.y - a.z * b.z;
  r.x = a.w * b.x + a.x * b.w + a.y * b.z - a.z * b.y;
  r.y = a.w * b.y + a.y * b.w + a.z * b.x - a.x * b.z;
  r.z = a.w * b.z + a.z * b.w + a.x * b.y - a.y * b.x;
  return r;
}
void quat_to_rot(const Quatf& q, float r[9]) {  // Eigen QuaternionBase::toRotationMatrix
  float tx = 2.f * q.x, ty = 2.f * q.y, tz = 2.f * q.z;
  float twx = tx * q.w, twy = ty * q.w, twz = tz * q.w;
  float txx = tx * q.x, txy = ty * q.x, txz = tz * q.x;
  float tyy = ty * q.y, tyz = tz * q.y, tzz = tz * q.z;
  r[0] = 1.f - (tyy + tzz);
  r[1] = txy - twz;
  r[2] = txz + twy;
  r[3] = txy + twz;
  r[4] = 1.f - (txx + tzz);
  r[5] = tyz - twx;
  r[6] = txz - twy;
  r[7] = tyz + twx;
  r[8] = 1.f - (txx + tyy);
}

// ----------------------------------------------------------------------------------------------------
// exact kd-tree (stand-in for FLANN KDTreeSingleIndex with exact search).  Ties -> lowest index.
// ----------------------------------------------------------------------------------------------------
class KdTree {
 public:
  KdTree(const float* xyz, int n) : pts_(xyz), n_(n) {
    idx_.reserve(n);
    for (int i = 0; i < n; ++i)
      if (std::isfinite(xyz[3 * i]) && std::isfinite(xyz[3 * i + 1]) && std::isfinite(xyz[3 * i + 2]))
        idx_.push_back(i);  // non-finite points are not indexed (kdtree_flann.hpp, !is_dense branch)
    nodes_.reserve(idx_.size() / 4 + 16);
    if (!idx_.empty()) build(0, (int)idx_.size());
  }
  int size() const { return (int)idx_.size(); }

  // nearest neighbour; returns false if the tree is empty
  bool nn1(const float* q, int& best_i, float& best_d) const {
    if (idx_.empty()) return false;
    best_i = -1;
    best_d = std::numeric_limits<float>::infinity();
    search1(0, q, best_i, best_d);
    return best_i >= 0;
  }
  // number of indexed points with d2 < r2 (strict, as FLANN's RadiusResultSet), counting stops at `cap`
  int count_within(const float* q, float r2, int cap) const {
    int found = 0;
    if (!nodes_.empty()) count(0, q, r2, cap, found);
    return found;
  }
  // all indexed points with d2 < r2 (strict, as FLANN's RadiusResultSet), appended to `out` in no particular order
  void radius(const float* q, float r2, std::vector<int>& out) const {
    if (!nodes_.empty()) collect(0, q, r2, out);
  }
  // k nearest, sorted ascending by (d2, index); returns number found
  int knn(const float* q, int k, int* out_i, float* out_d) const {
    int found = 0;
    searchk(0, q, k, out_i, out_d, found);
    return found;
  }

 private:
  struct Node {
    int lo, hi;       // range in idx_
    int left, right;  // children (-1 for a leaf)
    int axis;
    float split;
  };
  static constexpr int kLeaf = 12;

  int build(int lo, int hi) {
    int id = (int)nodes_.size();
    nodes_.push_back(Node{lo, hi, -1, -1, 0, 0.f});
    if (hi - lo <= kLeaf) return id;
    float mn[3] = {1e30f, 1e30f, 1e30f}, mx[3] = {-1e30f, -1e30f, -1e30f};
    for (int i = lo; i < hi; ++i)
      for (int a = 0; a < 3; ++a) {
        float v = pts_[3 * idx_[i] + a];
        mn[a] = std::min(mn[a], v);
        mx[a] = std::max(mx[a], v);
      }
    int axis = 0;
    if (mx[1] - mn[1] > mx[axis] - mn[axis]) axis = 1;
    if (mx[2] - mn[2] > mx[axis] - mn[axis]) axis = 2;
    if (mx[axis] == mn[axis]) return id;  // all points identical: keep as a (large) leaf
    int mid = (lo + hi) / 2;
    std::nth_element(idx_.begin() + lo, idx_.begin() + mid, idx_.begin() + hi,
                     [&](int a, int b) { return pts_[3 * a + axis] < pts_[3 * b + axis]; });
    float split = pts_[3 * idx_[mid] + axis];
    int l = build(lo, mid);
    int r = build(mid, hi);
    nodes_[id].left = l;
    nodes_[id].right = r;
    nodes_[id].axis = axis;
    nodes_[id].split = split;
    return id;
  }

  void count(int id, const float* q, float r2, int cap, int& found) const {
    const Node& nd = nodes_[id];
    if (nd.left < 0) {
      for (int i = nd.lo; i < nd.hi && found < cap; ++i)
        if (sqdist(q, pts_ + 3 * idx_[i]) < r2) ++found;
      return;
    }
    const float diff = q[nd.axis] - nd.split;
    const int near = diff < 0.f ? nd.left : nd.right, far = diff < 0.f ? nd.right : nd.left;
    count(near, q, r2, cap, found);
    if (found < cap && !(diff * diff >= r2)) count(far, q, r2, cap, found);
  }

  void collect(int id, const float* q, float r2, std::vector<int>& out) const {
    const Node& nd = nodes_[id];
    if (nd.left < 0) {
      for (int i = nd.lo; i < nd.hi; ++i)
        if (sqdist(q, pts_ + 3 * idx_[i]) < r2) out.push_back(idx_[i]);
      return;
    }
    const float diff = q[nd.axis] - nd.split;
    const int near = diff < 0.f ? nd.left : nd.right, far = diff < 0.f ? nd.right : nd.left;
    collect(near, q, r2, out);
    if (!(diff * diff >= r2)) collect(far, q, r2, out);
  }

  void search1(int id, const float* q, int& bi, float& bd) const {
    const Node& nd = nodes_[id];
    if (nd.left < 0) {
      for (int i = nd.lo; i < nd.hi; ++i) {
        int p = idx_[i];
        float d = sqdist(q, pts_ + 3 * p);
        if (d < bd || (d == bd && p < bi)) {
          bd = d;
          bi = p;
        }
      }
      return;
    }
    float diff = q[nd.axis] - nd.split;
    int near = diff < 0.f ? nd.left : nd.right;
    int far = diff < 0.f ? nd.right : nd.left;
    search1(near, q, bi, bd);
    // every point of the far side differs from q by at least |diff| along this axis; float rounding is
    // monotone, so diff*diff <= its d2.  Strict '>' keeps equal-distance candidates (tie -> lowest index).
    if (!(diff * diff > bd)) search1(far, q, bi, bd);
  }

  static bool less_pair(float d, int i, float d2, int i2) { return d < d2 || (d == d2 && i < i2); }

  void searchk(int id, const float* q, int k, int* oi, float* od, int& found) const {
    if (nodes_.empty()) return;
    const Node& nd = nodes_[id];
    if (nd.left < 0) {
      for (int i = nd.lo; i < nd.hi; ++i) {
        int p = idx_[i];
        float d = sqdist(q, pts_ + 3 * p);
        if (found == k && !less_pair(d, p, od[k - 1], oi[k - 1])) continue;
        int pos = (found < k) ? found : k - 1;
        while (pos > 0 && less_pair(d, p, od[pos - 1], oi[pos - 1])) {
          od[pos] = od[pos - 1];
          oi[pos] = oi[pos - 1];
          --pos;
        }
        od[pos] = d;
        oi[pos] = p;
        if (found < k) ++found;
      }
      return;
    }
    float diff = q[nd.axis] - nd.split;
    int near = diff < 0.f ? nd.left : nd.right;
    int far = diff < 0.f ? nd.right : nd.left;
    searchk(near, q, k, oi, od, found);
    if (found < k || !(diff * diff > od[k - 1])) searchk(far, q, k, oi, od, found);
  }

  const float* pts_;
  int n_;
  std::vector<int> idx_;
  std::vector<Node> nodes_;
};

// ----------------------------------------------------------------------------------------------------
// GICP state transform: applyState (gicp.hpp) - rotation built in FLOAT through quaternions,
// R = Rz(x5) * Ry(x4) * Rx(x3); t.topLeft3x3 = R * t.topLeft3x3; t.col(3) += (x0, x1, x2, 0).
// ----------------------------------------------------------------------------------------------------
void apply_state(Mat4f& t, const double x[6]) {
  Quatf qz = quat_from_axis_angle((float)x[5], 2);
  Quatf qy = quat_from_axis_angle((float)x[4], 1);
  Quatf qx = quat_from_axis_angle((float)x[3], 0);
  Quatf q = quat_mul(quat_mul(qz, qy), qx);
  float r[9];
  quat_to_rot(q, r);
  float nr[9];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      float s = r[3 * i] * t(0, j);
      s = s + r[3 * i + 1] * t(1, j);
      s = s + r[3 * i + 2] * t(2, j);
      nr[3 * i + j] = s;
    }
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) t(i, j) = nr[3 * i + j];
  t(0, 3) += (float)x[0];
  t(1, 3) += (float)x[1];
  t(2, 3) += (float)x[2];
}

// computeRDerivative (gicp.hpp): g[3..5] = tr(dR/dangle * Rsum)
void compute_r_derivative(const double x[6], const Mat3& R, double g[6]) {
  double phi = x[3], theta = x[4], psi = x[5];
  double cphi = std::cos(phi), sphi = std::sin(phi);
  double ctheta = std::cos(theta), stheta = std::sin(theta);
  double cpsi = std::cos(psi), spsi = std::sin(psi);
  Mat3 dphi = mat3_zero(), dth = mat3_zero(), dpsi = mat3_zero();
  dphi(0, 1) = sphi * spsi + cphi * cpsi * stheta;
  dphi(1, 1) = -cpsi * sphi + cphi * spsi * stheta;
  dphi(2, 1) = cphi * ctheta;
  dphi(0, 2) = cphi * spsi - cpsi * sphi * stheta;
  dphi(1, 2) = -cphi * cpsi - sphi * spsi * stheta;
  dphi(2, 2) = -ctheta * sphi;

  dth(0, 0) = -cpsi * stheta;
  dth(1, 0) = -spsi * stheta;
  dth(2, 0) = -ctheta;
  dth(0, 1) = cpsi * ctheta * sphi;
  dth(1, 1) = ctheta * sphi * spsi;
  dth(2, 1) = -sphi * stheta;
  dth(0, 2) = cphi * cpsi * ctheta;
  dth(1, 2) = cphi * ctheta * spsi;
  dth(2, 2) = -cphi * stheta;

  dpsi(0, 0) = -ctheta * spsi;
  dpsi(1, 0) = cpsi * ctheta;
  dpsi(0, 1) = -cphi * cpsi - sphi * spsi * stheta;
  dpsi(1, 1) = -cphi * spsi + cpsi * sphi * stheta;
  dpsi(0, 2) = cpsi * sphi - cphi * spsi * stheta;
  dpsi(1, 2) = sphi * spsi + cphi * cpsi * stheta;

  auto inner = [](const Mat3& a, const Mat3& b) {  // matricesInnerProd: sum_ij a(j,i) * b(i,j)
    double r = 0.0;
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) r += a(j, i) * b(i, j);
    return r;
  };
  g[3] = inner(dphi, R);
  g[4] = inner(dth, R);
  g[5] = inner(dpsi, R);
}

// ----------------------------------------------------------------------------------------------------
// The optimisation functor (gicp.hpp OptimizationFunctorWithIndices): base_transformation_ = identity.
// ----------------------------------------------------------------------------------------------------
struct Functor {
  const float* src;  // n_s x 3
  const float* tgt;  // n_t x 3
  const std::vector<int>* isrc;
  const std::vector<int>* itgt;
  const std::vector<Mat3>* maha;  // indexed by SOURCE index
  long n_f = 0, n_df = 0, n_fdf = 0;

  double f(const double x[6]) {
    ++n_f;
    Mat4f T = mat4f_identity();
    apply_state(T, x);
    const int m = (int)isrc->size();
    double acc = 0.0;
#ifdef _OPENMP
#pragma omp parallel for reduction(+ : acc) schedule(static)
#endif
    for (int i = 0; i < m; ++i) {
      const float* ps = src + 3 * (*isrc)[i];
      const float* pt = tgt + 3 * (*itgt)[i];
      float pp[3];
      xform_point(T, ps, pp);
      double res[3] = {(double)(pp[0] - pt[0]), (double)(pp[1] - pt[1]), (double)(pp[2] - pt[2])};
      const Mat3& M = (*maha)[(*isrc)[i]];
      double t0 = M(0, 0) * res[0] + M(0, 1) * res[1] + M(0, 2) * res[2];
      double t1 = M(1, 0) * res[0] + M(1, 1) * res[1] + M(1, 2) * res[2];
      double t2 = M(2, 0) * res[0] + M(2, 1) * res[1] + M(2, 2) * res[2];
      acc += res[0] * t0 + res[1] * t1 + res[2] * t2;
    }
    return acc / m;
  }

  void fdf_impl(const double x[6], double* fout, double g[6]) {
    Mat4f T = mat4f_identity();
    apply_state(T, x);
    const int m = (int)isrc->size();
    double acc = 0.0, g0 = 0.0, g1 = 0.0, g2 = 0.0;
    double r00 = 0, r01 = 0, r02 = 0, r10 = 0, r11 = 0, r12 = 0, r20 = 0, r21 = 0, r22 = 0;
#ifdef _OPENMP
#pragma omp parallel for reduction(+ : acc, g0, g1, g2, r00, r01, r02, r10, r11, r12, r20, r21, r22) schedule(static)
#endif
    for (int i = 0; i < m; ++i) {
      const float* ps = src + 3 * (*isrc)[i];
      const float* pt = tgt + 3 * (*itgt)[i];
      float pp[3];
      xform_point(T, ps, pp);
      double res[3] = {(double)(pp[0] - pt[0]), (double)(pp[1] - pt[1]), (double)(pp[2] - pt[2])};
      const Mat3& M = (*maha)[(*isrc)[i]];
      double t0 = M(0, 0) * res[0] + M(0, 1) * res[1] + M(0, 2) * res[2];
      double t1 = M(1, 0) * res[0] + M(1, 1) * res[1] + M(1, 2) * res[2];
      double t2 = M(2, 0) * res[0] + M(2, 1) * res[1] + M(2, 2) * res[2];
      acc += res[0] * t0 + res[1] * t1 + res[2] * t2;
      g0 += t0;
      g1 += t1;
      g2 += t2;
      double p0 = ps[0], p1 = ps[1], p2 = ps[2];  // base_transformation_ (identity) * p_src
      r00 += p0 * t0; r01 += p0 * t1; r02 += p0 * t2;
      r10 += p1 * t0; r11 += p1 * t1; r12 += p1 * t2;
      r20 += p2 * t0; r21 += p2 * t1; r22 += p2 * t2;
    }
    if (fout) *fout = acc / m;
    double sc = 2.0 / m;
    g[0] = g0 * sc;
    g[1] = g1 * sc;
    g[2] = g2 * sc;
    Mat3 R;
    R(0, 0) = r00 * sc; R(0, 1) = r01 * sc; R(0, 2) = r02 * sc;
    R(1, 0) = r10 * sc; R(1, 1) = r11 * sc; R(1, 2) = r12 * sc;
    R(2, 0) = r20 * sc; R(2, 1) = r21 * sc; R(2, 2) = r22 * sc;
    compute_r_derivative(x, R, g);
  }
  void df(const double x[6], double g[6]) {
    ++n_df;
    fdf_impl(x, nullptr, g);
  }
  void fdf(const double x[6], double& fo, double g[6]) {
    ++n_fdf;
    fdf_impl(x, &fo, g);
  }
};

// ----------------------------------------------------------------------------------------------------
// BFGS (PCL registration/bfgs.h == GSL multimin vector_bfgs2 + linear_minimize.c)
// ----------------------------------------------------------------------------------------------------
enum Status { NegativeGradientEpsilon = -3, NotStarted = -2, Running = -1, Success = 0, NoProgress = 1 };

struct Vec6 {
  double v[6];
  double& operator[](int i) { return v[i]; }
  double operator[](int i) const { return v[i]; }
};
double dot6(const Vec6& a, const Vec6& b) {
  double s = 0;
  for (int i = 0; i < 6; ++i) s += a[i] * b[i];
  return s;
}
double norm6(const Vec6& a) { return std::sqrt(dot6(a, a)); }

int solve_quadratic(double a, double b, double c, double* x0, double* x1) {  // gsl_poly_solve_quadratic
  if (a == 0) {
    if (b == 0) return 0;
    *x0 = -c / b;
    return 1;
  }
  double disc = b * b - 4 * a * c;
  if (disc > 0) {
    if (b == 0) {
      double r = std::sqrt(-c / a);
      *x0 = -r;
      *x1 = r;
    } else {
      double sgnb = (b > 0 ? 1 : -1);
      double temp = -0.5 * (b + sgnb * std::sqrt(disc));
      double r1 = temp / a;
      double r2 = c / temp;
      if (r1 < r2) {
        *x0 = r1;
        *x1 = r2;
      } else {
        *x0 = r2;
        *x1 = r1;
      }
    }
    return 2;
  } else if (disc == 0) {
    *x0 = -0.5 * b / a;
    *x1 = -0.5 * b / a;
    return 2;
  }
  return 0;
}

double interp_quad(double f0, double fp0, double f1, double zl, double zh) {
  double fl = f0 + zl * (fp0 + zl * (f1 - f0 - fp0));
  double fh = f0 + zh * (fp0 + zh * (f1 - f0 - fp0));
  double c = 2 * (f1 - f0 - fp0);
  double zmin = zl, fmin = fl;
  if (fh < fmin) {
    zmin = zh;
    fmin = fh;
  }
  if (c > 0) {
    double z = -fp0 / c;
    if (z > zl && z < zh) {
      double f = f0 + z * (fp0 + z * (f1 - f0 - fp0));
      if (f < fmin) {
        zmin = z;
        fmin = f;
      }
    }
  }
  return zmin;
}
double cubic(double c0, double c1, double c2, double c3, double z) { return c0 + z * (c1 + z * (c2 + z * c3)); }
void check_extremum(double c0, double c1, double c2, double c3, double z, double* zmin, double* fmin) {
  double y = cubic(c0, c1, c2, c3, z);
  if (y < *fmin) {
    *zmin = z;
    *fmin = y;
  }
}
double interp_cubic(double f0, double fp0, double f1, double fp1, double zl, double zh) {
  double eta = 3 * (f1 - f0) - 2 * fp0 - fp1;
  double xi = fp0 + fp1 - 2 * (f1 - f0);
  double c0 = f0, c1 = fp0, c2 = eta, c3 = xi;
  double zmin = zl, fmin = cubic(c0, c1, c2, c3, zl);
  check_extremum(c0, c1, c2, c3, zh, &zmin, &fmin);
  double z0, z1;
  int n = solve_quadratic(3 * c3, 2 * c2, c1, &z0, &z1);
  if (n == 2) {
    if (z0 > zl && z0 < zh) check_extremum(c0, c1, c2, c3, z0, &zmin, &fmin);
    if (z1 > zl && z1 < zh) check_extremum(c0, c1, c2, c3, z1, &zmin, &fmin);
  } else if (n == 1) {
    if (z0 > zl && z0 < zh) check_extremum(c0, c1, c2, c3, z0, &zmin, &fmin);
  }
  return zmin;
}
double interpolate(double a, double fa, double fpa, double b, double fb, double fpb, double xmin, double xmax,
                   int order) {
  double zmin = (xmin - a) / (b - a);
  double zmax = (xmax - a) / (b - a);
  if (zmin > zmax) std::swap(zmin, zmax);
  double z;
  if (order > 2 && !std::isnan(fpb))
    z = interp_cubic(fa, fpa * (b - a), fb, fpb * (b - a), zmin, zmax);
  else
    z = interp_quad(fa, fpa * (b - a), fb, zmin, zmax);
  return a + z * (b - a);
}

class Bfgs {
 public:
  struct Parameters {
    int max_iters = 400, bracket_iters = 100, section_iters = 100, order = 3;
    double rho = 0.01, sigma = 0.01, tau1 = 9, tau2 = 0.05, tau3 = 0.5, step_size = 1;
  } parameters;

  explicit Bfgs(Functor& fn) : functor(fn) {}

  Status minimizeInit(Vec6& x) {
    iter = 0;
    delta_f = 0;
    for (int i = 0; i < 6; ++i) dx0[i] = 0;
    functor.fdf(x.v, f, gradient.v);
    x0 = x;
    g0 = gradient;
    g0norm = norm6(g0);
    for (int i = 0; i < 6; ++i) p[i] = gradient[i] * -1 / g0norm;
    pnorm = norm6(p);
    fp0 = -g0norm;
    x_alpha = x0;
    x_cache_key = 0;
    f_alpha = f;
    f_cache_key = 0;
    g_alpha = g0;
    g_cache_key = 0;
    df_alpha = slope();
    df_cache_key = 0;
    return NotStarted;
  }

  Status minimizeOneStep(Vec6& x) {
    double alpha = 0.0, alpha1;
    double f0 = f;
    if (pnorm == 0.0 || g0norm == 0.0 || fp0 == 0) {
      for (int i = 0; i < 6; ++i) dx[i] = 0;
      return NoProgress;
    }
    if (delta_f < 0) {
      double del = std::max(-delta_f, 10 * std::numeric_limits<double>::epsilon() * std::fabs(f0));
      alpha1 = std::min(1.0, 2.0 * del / (-fp0));
    } else
      alpha1 = std::fabs(parameters.step_size);

    Status status = lineSearch(parameters.rho, parameters.sigma, parameters.tau1, parameters.tau2, parameters.tau3,
                               parameters.order, alpha1, alpha);
    if (status != Success) return status;

    updatePosition(alpha, x, f, gradient);
    delta_f = f - f0;

    // memoryless BFGS direction: p' = g1 - A dx - B dg
    {
      double dxg, dgg, dxdg, dgnorm, A, B;
      for (int i = 0; i < 6; ++i) dx0[i] = x[i] - x0[i];
      dx = dx0;
      for (int i = 0; i < 6; ++i) dg0[i] = gradient[i] - g0[i];
      dxg = dot6(dx0, gradient);
      dgg = dot6(dg0, gradient);
      dxdg = dot6(dx0, dg0);
      dgnorm = norm6(dg0);
      if (dxdg != 0) {
        B = dxg / dxdg;
        A = -(1.0 + dgnorm * dgnorm / dxdg) * B + dgg / dxdg;
      } else {
        B = 0;
        A = 0;
      }
      for (int i = 0; i < 6; ++i) p[i] = -A * dx0[i];
      for (int i = 0; i < 6; ++i) p[i] += gradient[i];
      for (int i = 0; i < 6; ++i) p[i] += -B * dg0[i];
    }
    g0 = gradient;
    x0 = x;
    g0norm = norm6(g0);
    pnorm = norm6(p);
    double dir = (dot6(p, gradient) > 0) ? -1.0 : 1.0;
    for (int i = 0; i < 6; ++i) p[i] *= dir / pnorm;
    pnorm = norm6(p);
    fp0 = dot6(p, g0);
    changeDirection();
    return Success;
  }

  Status testGradient(double epsilon) const {
    if (epsilon < 0) return NegativeGradientEpsilon;
    return (g0norm < epsilon) ? Success : Running;
  }

 private:
  void moveTo(double alpha) {
    if (alpha == x_cache_key) return;
    for (int i = 0; i < 6; ++i) x_alpha[i] = x0[i] + alpha * p[i];
    x_cache_key = alpha;
  }
  double slope() const { return dot6(g_alpha, p); }
  double getF(double alpha) {
    if (alpha == f_cache_key) return f_alpha;
    moveTo(alpha);
    f_alpha = functor.f(x_alpha.v);
    f_cache_key = alpha;
    return f_alpha;
  }
  double getDF(double alpha) {
    if (alpha == df_cache_key) return df_alpha;
    moveTo(alpha);
    if (alpha != g_cache_key) {
      functor.df(x_alpha.v, g_alpha.v);
      g_cache_key = alpha;
    }
    df_alpha = slope();
    df_cache_key = alpha;
    return df_alpha;
  }
  void getFDF(double alpha, double& fo, double& dfo) {
    if (alpha == f_cache_key && alpha == df_cache_key) {
      fo = f_alpha;
      dfo = df_alpha;
      return;
    }
    if (alpha == f_cache_key || alpha == df_cache_key) {
      fo = getF(alpha);
      dfo = getDF(alpha);
      return;
    }
    moveTo(alpha);
    functor.fdf(x_alpha.v, f_alpha, g_alpha.v);
    f_cache_key = alpha;
    g_cache_key = alpha;
    df_alpha = slope();
    df_cache_key = alpha;
    fo = f_alpha;
    dfo = df_alpha;
  }
  void updatePosition(double alpha, Vec6& x, double& fo, Vec6& g) {
    double fa, dfa;
    getFDF(alpha, fa, dfa);
    fo = f_alpha;
    x = x_alpha;
    g = g_alpha;
  }
  void changeDirection() {
    x_alpha = x0;
    x_cache_key = 0.0;
    f_cache_key = 0.0;
    g_alpha = g0;
    g_cache_key = 0.0;
    df_alpha = slope();
    df_cache_key = 0.0;
  }

  Status lineSearch(double rho, double sigma, double tau1, double tau2, double tau3, int order, double alpha1,
                    double& alpha_new) {
    double f0, fp0_, falpha, falpha_prev, fpalpha = 0, fpalpha_prev, delta, alpha_next;
    double alpha = alpha1, alpha_prev = 0.0;
    double a, b, fa, fb, fpa, fpb;
    int i = 0;
    getFDF(0.0, f0, fp0_);
    falpha_prev = f0;
    fpalpha_prev = fp0_;
    a = 0.0;
    b = alpha;
    fa = f0;
    fb = 0.0;
    fpa = fp0_;
    fpb = 0.0;
    // bracketing
    while (i++ < parameters.bracket_iters) {
      falpha = getF(alpha);
      if (falpha > f0 + alpha * rho * fp0_ || falpha >= falpha_prev) {
        a = alpha_prev;
        fa = falpha_prev;
        fpa = fpalpha_prev;
        b = alpha;
        fb = falpha;
        fpb = std::numeric_limits<double>::quiet_NaN();
        break;
      }
      fpalpha = getDF(alpha);
      if (std::fabs(fpalpha) <= -sigma * fp0_) {
        alpha_new = alpha;
        return Success;
      }
      if (fpalpha >= 0) {
        a = alpha;
        fa = falpha;
        fpa = fpalpha;
        b = alpha_prev;
        fb = falpha_prev;
        fpb = fpalpha_prev;
        break;
      }
      delta = alpha - alpha_prev;
      {
        double lower = alpha + delta;
        double upper = alpha + tau1 * delta;
        alpha_next = interpolate(alpha_prev, falpha_prev, fpalpha_prev, alpha, falpha, fpalpha, lower, upper, order);
      }
      alpha_prev = alpha;
      falpha_prev = falpha;
      fpalpha_prev = fpalpha;
      alpha = alpha_next;
    }
    // sectioning
    while (i++ < parameters.section_iters) {
      delta = b - a;
      {
        double lower = a + tau2 * delta;
        double upper = b - tau3 * delta;
        alpha = interpolate(a, fa, fpa, b, fb, fpb, lower, upper, order);
      }
      falpha = getF(alpha);
      if ((a - alpha) * fpa <= std::numeric_limits<double>::epsilon()) return NoProgress;
      if (falpha > f0 + rho * alpha * fp0_ || falpha >= fa) {
        b = alpha;
        fb = falpha;
        fpb = std::numeric_limits<double>::quiet_NaN();
      } else {
        fpalpha = getDF(alpha);
        if (std::fabs(fpalpha) <= -sigma * fp0_) {
          alpha_new = alpha;
          return Success;
        }
        if (((b - a) >= 0 && fpalpha >= 0) || ((b - a) <= 0 && fpalpha <= 0)) {
          b = a;
          fb = fa;
          fpb = fpa;
          a = alpha;
          fa = falpha;
          fpa = fpalpha;
        } else {
          a = alpha;
          fa = falpha;
          fpa = fpalpha;
        }
      }
    }
    return Success;
  }

  Functor& functor;
  int iter = 0;
  double step = 0, g0norm = 0, pnorm = 0, delta_f = 0, fp0 = 0, f = 0;
  Vec6 x0, dx, dx0, g0, dg0, p, gradient;
  Vec6 x_alpha, g_alpha;
  double f_alpha = 0, df_alpha = 0;
  double f_cache_key = 0, df_cache_key = 0, x_cache_key = 0, g_cache_key = 0;
};

// ----------------------------------------------------------------------------------------------------
// computeCovariances (gicp.hpp)
// ----------------------------------------------------------------------------------------------------
bool compute_covariances(const float* xyz, int n, const KdTree& tree, int k, double eps, std::vector<Mat3>& covs) {
  if (k > n) return false;
  covs.resize(n);
#ifdef _OPENMP
#pragma omp parallel
#endif
  {
    std::vector<int> nn(k);
    std::vector<float> nd(k);
#ifdef _OPENMP
#pragma omp for schedule(dynamic, 256)
#endif
    for (int i = 0; i < n; ++i) {
      Mat3 cov = mat3_zero();
      double mean[3] = {0, 0, 0};
      int found = tree.knn(xyz + 3 * i, k, nn.data(), nd.data());
      for (int j = 0; j < found; ++j) {
        const float* pt = xyz + 3 * nn[j];
        mean[0] += pt[0];
        mean[1] += pt[1];
        mean[2] += pt[2];
        // float * float products (rounded to float), accumulated in double, exactly as the PCL source does
        cov(0, 0) += pt[0] * pt[0];
        cov(1, 0) += pt[1] * pt[0];
        cov(1, 1) += pt[1] * pt[1];
        cov(2, 0) += pt[2] * pt[0];
        cov(2, 1) += pt[2] * pt[1];
        cov(2, 2) += pt[2] * pt[2];
      }
      for (double& m : mean) m /= (double)k;
      for (int a = 0; a < 3; ++a)
        for (int b = 0; b <= a; ++b) {
          cov(a, b) /= (double)k;
          cov(a, b) -= mean[a] * mean[b];
          cov(b, a) = cov(a, b);
        }
      double lam[3];
      Mat3 U;
      sym3_eig_desc(cov, lam, U);
      Mat3 out = mat3_zero();
      for (int c = 0; c < 3; ++c) {
        double v = (c == 2) ? eps : 1.0;
        for (int a = 0; a < 3; ++a)
          for (int b = 0; b < 3; ++b) out(a, b) += v * U(a, c) * U(b, c);
      }
      covs[i] = out;
    }
  }
  return true;
}

}  // namespace

// ====================================================================================================
// C interface (ctypes).  All clouds are contiguous float32 [n][3].  Matrices are row-major.
// ====================================================================================================
extern "C" {

struct OrcParams {
  int max_iterations;            // reference default 100 (src/GICPAlignment.cpp:30)
  double transformation_epsilon; // reference default 4e-3 (src/GICPAlignment.cpp:29)
  double rotation_epsilon;       // PCL default 2e-3
  double max_corr_distance;      // reference default 4e-2 (src/GICPAlignment.cpp:31)
  int k_correspondences;         // PCL default 20
  double gicp_epsilon;           // PCL default 1e-3
  int max_inner_iterations;      // PCL default 20
};

struct OrcResult {
  float T[16];           // final_transformation_, row-major
  int converged;
  int outer_iterations;
  long n_f, n_df, n_fdf; // functor evaluations over the whole align
  long n_corr_queries;   // sum over outer iterations of source queries
  long n_pairs_last;     // correspondences of the last outer iteration
  double t_cov_s, t_corr_s, t_opt_s, t_tree_s;
};

int orc_num_threads() {
#ifdef _OPENMP
  return omp_get_max_threads();
#else
  return 1;
#endif
}

// ---- fixture: area-weighted triangle sampling with libc rand() (reference src/CADToPointCloud.cpp:101-190)
void orc_sample_mesh(const float* verts, int nv, const int* faces, int nf, int n_samples, long skip_draws,
                     float* out_xyz) {
  (void)nv;
  std::vector<double> cum(nf, 0.0);
  double total = 0.0;
  for (int i = 0; i < nf; ++i) {
    double p1[3], p2[3], p3[3];
    for (int a = 0; a < 3; ++a) {
      p1[a] = verts[3 * faces[3 * i] + a];
      p2[a] = verts[3 * faces[3 * i + 1] + a];
      p3[a] = verts[3 * faces[3 * i + 2] + a];
    }
    auto d2 = [](const double* u, const double* v) {
      return (u[0] - v[0]) * (u[0] - v[0]) + (u[1] - v[1]) * (u[1] - v[1]) + (u[2] - v[2]) * (u[2] - v[2]);
    };
    double a = d2(p1, p2), b = d2(p2, p3), c = d2(p3, p1);  // vtkTriangle::TriangleArea
    total += 0.25 * std::sqrt(std::fabs(4.0 * a * c - (a - b + c) * (a - b + c)));
    cum[i] = total;
  }
  srand(1);  // the reference never calls srand(): glibc's initial state equals srand(1)
  for (long s = 0; s < skip_draws; ++s) (void)rand();
  auto uniform_deviate = [](int seed) { return seed * (1.0 / (RAND_MAX + 1.0)); };
  for (int i = 0; i < n_samples; ++i) {
    float r = static_cast<float>(uniform_deviate(rand()) * total);
    int el = (int)(std::lower_bound(cum.begin(), cum.end(), r) - cum.begin());
    float a1 = verts[3 * faces[3 * el]], a2 = verts[3 * faces[3 * el] + 1], a3 = verts[3 * faces[3 * el] + 2];
    float b1 = verts[3 * faces[3 * el + 1]], b2 = verts[3 * faces[3 * el + 1] + 1], b3 = verts[3 * faces[3 * el + 1] + 2];
    float c1 = verts[3 * faces[3 * el + 2]], c2 = verts[3 * faces[3 * el + 2] + 1], c3 = verts[3 * faces[3 * el + 2] + 2];
    float r1 = static_cast<float>(uniform_deviate(rand()));
    float r2 = static_cast<float>(uniform_deviate(rand()));
    float r1sqr = sqrtf(r1);
    float om1 = (1 - r1sqr);
    float om2 = (1 - r2);
    a1 *= om1; a2 *= om1; a3 *= om1;
    b1 *= om2; b2 *= om2; b3 *= om2;
    c1 = r1sqr * (r2 * c1 + b1) + a1;
    c2 = r1sqr * (r2 * c2 + b2) + a2;
    c3 = r1sqr * (r2 * c3 + b3) + a3;
    out_xyz[3 * i] = c1;
    out_xyz[3 * i + 1] = c2;
    out_xyz[3 * i + 2] = c3;
  }
}

// ---- Utils::rotateCloud matrix (reference src/Utils.cpp:215-229): q = Rx(roll) * Ry(pitch) * Rz(yaw)
void orc_rotation_rpy(double roll, double pitch, double yaw, float* T16) {
  Quatf q = quat_mul(quat_mul(quat_from_axis_angle((float)roll, 0), quat_from_axis_angle((float)pitch, 1)),
                     quat_from_axis_angle((float)yaw, 2));
  float r[9];
  quat_to_rot(q, r);
  Mat4f T = mat4f_identity();
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) T(i, j) = r[3 * i + j];
  std::memcpy(T16, T.m, sizeof(T.m));
}

// ---- pcl::transformPointCloud on xyz (reference src/GICPAlignment.cpp:146, src/LeicaStateMachine.cpp:182)
void orc_transform(const float* T16, const float* in, int n, float* out) {
  Mat4f T;
  std::memcpy(T.m, T16, sizeof(T.m));
#ifdef _OPENMP
#pragma omp parallel for schedule(static)
#endif
  for (int i = 0; i < n; ++i) {
    float q[3];
    xform_point(T, in + 3 * i, q);
    out[3 * i] = q[0];
    out[3 * i + 1] = q[1];
    out[3 * i + 2] = q[2];
  }
}

// ---- applyState exposed for tests (x = tx,ty,tz,roll,pitch,yaw)
void orc_apply_state(const double* x6, float* T16) {
  Mat4f T = mat4f_identity();
  apply_state(T, x6);
  std::memcpy(T16, T.m, sizeof(T.m));
}

// ---- exact NN-1 of every query in the target.  use_tree = 0 -> brute force.  Non-finite queries -> -1.
void orc_nn1(const float* tgt, int nt, const float* qry, int nq, int use_tree, int* idx, float* d2) {
  if (use_tree) {
    KdTree tree(tgt, nt);
#ifdef _OPENMP
#pragma omp parallel for schedule(dynamic, 1024)
#endif
    for (int i = 0; i < nq; ++i) {
      int bi = -1;
      float bd = std::numeric_limits<float>::infinity();
      const float* q = qry + 3 * i;
      if (std::isfinite(q[0]) && std::isfinite(q[1]) && std::isfinite(q[2])) tree.nn1(q, bi, bd);
      idx[i] = bi;
      d2[i] = bd;
    }
    return;
  }
  for (int i = 0; i < nq; ++i) {
    int bi = -1;
    float bd = std::numeric_limits<float>::infinity();
    const float* q = qry + 3 * i;
    if (std::isfinite(q[0]) && std::isfinite(q[1]) && std::isfinite(q[2]))
      for (int j = 0; j < nt; ++j) {
        const float* p = tgt + 3 * j;
        if (!(std::isfinite(p[0]) && std::isfinite(p[1]) && std::isfinite(p[2]))) continue;
        float d = sqdist(q, p);
        if (d < bd) {  // ascending j: strict '<' keeps the lowest index on ties
          bd = d;
          bi = j;
        }
      }
    idx[i] = bi;
    d2[i] = bd;
  }
}

// ---- exact self-kNN (the point itself is neighbour 0), sorted by (d2, index).  use_tree = 0 -> brute force.
void orc_knn(const float* xyz, int n, int k, int use_tree, int* idx, float* d2) {
  if (use_tree) {
    KdTree tree(xyz, n);
#ifdef _OPENMP
#pragma omp parallel for schedule(dynamic, 256)
#endif
    for (int i = 0; i < n; ++i) {
      int found = tree.knn(xyz + 3 * i, k, idx + (size_t)k * i, d2 + (size_t)k * i);
      for (int j = found; j < k; ++j) {
        idx[(size_t)k * i + j] = -1;
        d2[(size_t)k * i + j] = std::numeric_limits<float>::infinity();
      }
    }
    return;
  }
  std::vector<std::pair<float, int>> cand(n);
  for (int i = 0; i < n; ++i) {
    for (int j = 0; j < n; ++j) cand[j] = {sqdist(xyz + 3 * i, xyz + 3 * j), j};
    int kk = std::min(k, n);
    std::partial_sort(cand.begin(), cand.begin() + kk, cand.end());
    for (int j = 0; j < k; ++j) {
      idx[(size_t)k * i + j] = j < kk ? cand[j].second : -1;
      d2[(size_t)k * i + j] = j < kk ? cand[j].first : std::numeric_limits<float>::infinity();
    }
  }
}

// ---- GICP covariances (row-major 3x3 doubles per point).  Returns 0 on success.
int orc_covariances(const float* xyz, int n, int k, double eps, double* cov9) {
  KdTree tree(xyz, n);
  std::vector<Mat3> covs;
  if (!compute_covariances(xyz, n, tree, k, eps, covs)) return -1;
  for (int i = 0; i < n; ++i) std::memcpy(cov9 + 9 * (size_t)i, covs[i].m, sizeof(covs[i].m));
  return 0;
}

// ---- one evaluation of the GICP objective and gradient for a FIXED correspondence set, for tests:
//      pairs are (isrc[i], itgt[i]); maha9 is indexed by source index.  f and g[6] are returned.
void orc_cost(const float* src, const float* tgt, const int* isrc, const int* itgt, int m, const double* maha9,
              int n_src, const double* x6, double* f, double* g6) {
  std::vector<int> is(isrc, isrc + m), it(itgt, itgt + m);
  std::vector<Mat3> maha(n_src);
  for (int i = 0; i < n_src; ++i) std::memcpy(maha[i].m, maha9 + 9 * (size_t)i, sizeof(maha[i].m));
  Functor fn{src, tgt, &is, &it, &maha};
  fn.fdf(x6, *f, g6);
}

// ---- correspondences + Mahalanobis matrices of ONE outer iteration under transform T (float row-major),
//      as in gicp.hpp computeTransformation steps 1-2.  Outputs: nn index per source (-1 when gated out or
//      no NN), d2 per source, maha9 per source (identity when gated out).  Returns the pair count.
int orc_correspondences(const float* src, int ns, const float* tgt, int nt, const double* cov_src9,
                        const double* cov_tgt9, const float* T16, double max_corr_distance, int* nn_idx, float* nn_d2,
                        double* maha9) {
  KdTree tree(tgt, nt);
  Mat4f T;
  std::memcpy(T.m, T16, sizeof(T.m));
  Mat3 R;
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) R(i, j) = (double)T(i, j);
  double thr = max_corr_distance * max_corr_distance;
  int cnt = 0;
  for (int i = 0; i < ns; ++i) {
    float q[3];
    xform_point(T, src + 3 * i, q);
    int bi = -1;
    float bd = std::numeric_limits<float>::infinity();
    tree.nn1(q, bi, bd);
    nn_d2[i] = bd;
    Mat3 M = mat3_identity();
    if (bi >= 0 && bd < thr) {
      Mat3 C1, C2;
      std::memcpy(C1.m, cov_src9 + 9 * (size_t)i, sizeof(C1.m));
      std::memcpy(C2.m, cov_tgt9 + 9 * (size_t)bi, sizeof(C2.m));
      Mat3 tmp = mat3_mul(mat3_mul(R, C1), mat3_transpose(R));
      for (int e = 0; e < 9; ++e) tmp.m[e] += C2.m[e];
      M = mat3_inverse(tmp);
      nn_idx[i] = bi;
      ++cnt;
    } else
      nn_idx[i] = -1;
    std::memcpy(maha9 + 9 * (size_t)i, M.m, sizeof(M.m));
  }
  return cnt;
}

// ---- the whole align(): Registration::align + GICP::computeTransformation (guess = identity), as invoked by
//      reference src/GICPAlignment.cpp:96.  Returns 0; res->converged mirrors hasConverged().
int orc_gicp_align(const float* src, int ns, const float* tgt, int nt, const OrcParams* prm, int max_outer_override,
                   OrcResult* res) {
  auto now = []() {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec + 1e-9 * ts.tv_nsec;
  };
  std::memset(res, 0, sizeof(*res));
  Mat4f ident = mat4f_identity();
  std::memcpy(res->T, ident.m, sizeof(ident.m));
  if (ns <= 0 || nt <= 0) return -1;

  double t0 = now();
  KdTree tree_t(tgt, nt);  // Registration::initCompute
  KdTree tree_s(src, ns);  // initComputeReciprocal
  res->t_tree_s = now() - t0;

  t0 = now();
  std::vector<Mat3> cov_t, cov_s;
  std::vector<Mat3> maha(ns, mat3_identity());
  bool ok_t = compute_covariances(tgt, nt, tree_t, prm->k_correspondences, prm->gicp_epsilon, cov_t);
  bool ok_s = compute_covariances(src, ns, tree_s, prm->k_correspondences, prm->gicp_epsilon, cov_s);
  res->t_cov_s = now() - t0;
  if (!ok_t || !ok_s) return -2;

  Mat4f transformation = mat4f_identity(), previous = mat4f_identity();
  const double dist_threshold = prm->max_corr_distance * prm->max_corr_distance;
  int nr_iterations = 0;
  bool converged = false;
  const int max_iterations = max_outer_override > 0 ? max_outer_override : prm->max_iterations;
  std::vector<int> source_indices, target_indices;
  std::vector<int> nn_all(ns);
  std::vector<float> d2_all(ns);

  while (!converged) {
    t0 = now();
    Mat3 R;  // transform_R = double(transformation_) * double(guess = I)
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) R(i, j) = (double)transformation(i, j);
    const Mat3 Rt = mat3_transpose(R);
#ifdef _OPENMP
#pragma omp parallel for schedule(dynamic, 1024)
#endif
    for (int i = 0; i < ns; ++i) {
      float q[3];
      xform_point(transformation, src + 3 * i, q);
      int bi = -1;
      float bd = std::numeric_limits<float>::infinity();
      tree_t.nn1(q, bi, bd);
      if (bi >= 0 && bd < dist_threshold) {
        Mat3 tmp = mat3_mul(mat3_mul(R, cov_s[i]), Rt);
        for (int e = 0; e < 9; ++e) tmp.m[e] += cov_t[bi].m[e];
        maha[i] = mat3_inverse(tmp);
        nn_all[i] = bi;
      } else
        nn_all[i] = -1;
      d2_all[i] = bd;
    }
    source_indices.clear();
    target_indices.clear();
    for (int i = 0; i < ns; ++i)
      if (nn_all[i] >= 0) {
        source_indices.push_back(i);
        target_indices.push_back(nn_all[i]);
      }
    res->n_corr_queries += ns;
    res->n_pairs_last = (long)source_indices.size();
    res->t_corr_s += now() - t0;

    previous = transformation;
    t0 = now();
    // estimateRigidTransformationBFGS
    if (source_indices.size() < 4) break;  // NotEnoughPointsException -> converged_ stays false
    Vec6 x;
    x[0] = transformation(0, 3);
    x[1] = transformation(1, 3);
    x[2] = transformation(2, 3);
    x[3] = std::atan2((double)transformation(2, 1), (double)transformation(2, 2));
    x[4] = std::asin(-(double)transformation(2, 0));
    x[5] = std::atan2((double)transformation(1, 0), (double)transformation(0, 0));
    Functor fn{src, tgt, &source_indices, &target_indices, &maha};
    Bfgs bfgs(fn);
    bfgs.parameters.sigma = 0.01;
    bfgs.parameters.rho = 0.01;
    bfgs.parameters.tau1 = 9;
    bfgs.parameters.tau2 = 0.05;
    bfgs.parameters.tau3 = 0.5;
    bfgs.parameters.order = 3;
    int inner = 0;
    int result = bfgs.minimizeInit(x);
    result = Running;
    do {
      ++inner;
      result = bfgs.minimizeOneStep(x);
      if (result) break;
      result = bfgs.testGradient(1e-2);
    } while (result == Running && inner < prm->max_inner_iterations);
    res->n_f += fn.n_f;
    res->n_df += fn.n_df;
    res->n_fdf += fn.n_fdf;
    res->t_opt_s += now() - t0;
    if (result == NoProgress || result == Success || inner == prm->max_inner_iterations) {
      transformation = mat4f_identity();
      apply_state(transformation, x.v);
    } else
      break;  // SolverDidntConvergeException

    double delta = 0.0;
    for (int k = 0; k < 4; ++k)
      for (int l = 0; l < 4; ++l) {
        double ratio = (k < 3 && l < 3) ? 1.0 / prm->rotation_epsilon : 1.0 / prm->transformation_epsilon;
        double c_delta = ratio * std::fabs((double)(previous(k, l) - transformation(k, l)));
        if (c_delta > delta) delta = c_delta;
      }
    ++nr_iterations;
    if (nr_iterations >= max_iterations || delta < 1) {
      converged = true;
      previous = transformation;
    }
  }
  res->converged = converged ? 1 : 0;
  res->outer_iterations = nr_iterations;
  std::memcpy(res->T, previous.m, sizeof(previous.m));  // final_transformation_ = previous * guess
  return 0;
}

// ---- Registration::getFitnessScore(max_range): mean NN-1 d2 of T*source over points with d2 <= max_range
double orc_fitness(const float* src, int ns, const float* tgt, int nt, const float* T16, double max_range) {
  KdTree tree(tgt, nt);
  Mat4f T;
  std::memcpy(T.m, T16, sizeof(T.m));
  double sum = 0.0;
  long nr = 0;
#ifdef _OPENMP
#pragma omp parallel for reduction(+ : sum, nr) schedule(dynamic, 1024)
#endif
  for (int i = 0; i < ns; ++i) {
    float q[3];
    xform_point(T, src + 3 * i, q);
    int bi;
    float bd;
    if (!tree.nn1(q, bi, bd)) continue;
    if ((double)bd <= max_range) {
      sum += bd;
      ++nr;
    }
  }
  if (nr > 0) return sum / (double)nr;
  return std::numeric_limits<double>::max();
}

// ---- pcl::getPointCloudDifference (reference src/Filter.cpp:176-189): mask[i] = 1 iff input point i is finite
//      and its NN-1 squared distance in `subtract` is > threshold.  Returns the number kept.
int orc_difference(const float* input, int n_in, const float* subtract, int n_sub, double threshold,
                   unsigned char* mask) {
  KdTree tree(subtract, n_sub);
  int kept = 0;
#ifdef _OPENMP
#pragma omp parallel for reduction(+ : kept) schedule(dynamic, 1024)
#endif
  for (int i = 0; i < n_in; ++i) {
    const float* q = input + 3 * i;
    mask[i] = 0;
    if (!(std::isfinite(q[0]) && std::isfinite(q[1]) && std::isfinite(q[2]))) continue;
    int bi;
    float bd;
    if (!tree.nn1(q, bi, bd)) continue;
    if ((double)bd > threshold) {
      mask[i] = 1;
      ++kept;
    }
  }
  return kept;
}

// ---- Utils::computeCloudResolution (reference src/Utils.cpp:145-174): mean distance to the 2nd neighbour
double orc_resolution(const float* xyz, int n) {
  KdTree tree(xyz, n);
  double res = 0.0;
  long cnt = 0;
#ifdef _OPENMP
#pragma omp parallel for reduction(+ : res, cnt) schedule(dynamic, 1024)
#endif
  for (int i = 0; i < n; ++i) {
    if (!std::isfinite(xyz[3 * i])) continue;
    int nn[2];
    float nd[2];
    if (tree.knn(xyz + 3 * i, 2, nn, nd) == 2) {
      res += std::sqrt((double)nd[1]);  // the reference's unqualified sqrt() on a float: C's double sqrt(double)
      ++cnt;
    }
  }
  if (cnt) res /= (double)cnt;
  return res;
}

// Which points get a finite normal from Utils::getNormals (reference src/Utils.cpp:27-44): pcl::NormalEstimation with a
// radius search yields NaN for a non-finite point and for a point with fewer than 3 neighbours (itself included)
// inside the radius; GICPAlignment::getCovariances then drops exactly those points from the caller's cloud
// (reference src/GICPAlignment.cpp:63-67).  mask[i] = 1 iff the normal of point i is finite.  Returns the count.
int orc_normals(const float* xyz, int n, double radius, float* out4);
int orc_normal_validity(const float* xyz, int n, double radius, unsigned char* mask) {
  // pcl::removeNaNNormalsFromPointCloud: a point stays iff normal_x, normal_y and normal_z are finite - which is "at least 3
  // points inside the radius" except where the float moments cancel to a zero covariance (then pcl::eigen33 divides 0 by 0)
  std::vector<float> nrm((size_t)std::max(n, 1) * 4);
  orc_normals(xyz, n, radius, nrm.data());
  int kept = 0;
  for (int i = 0; i < n; ++i) {
    const float* o = &nrm[4 * (size_t)i];
    const bool ok = std::isfinite(o[0]) && std::isfinite(o[1]) && std::isfinite(o[2]);
    mask[i] = ok ? 1 : 0;
    kept += ok ? 1 : 0;
  }
  return kept;
}

// ---- Utils::getNormals (reference src/Utils.cpp:27-44) = pcl::NormalEstimation<PointXYZRGB, Normal> with a radius search,
//      restated from PCL 1.8.1 features/normal_3d.h(pp), common/impl/centroid.hpp and common/impl/eigen.hpp:
//        * neighbours = FLANN radiusSearch, d2 < float(radius^2), SORTED by (d2, index) (KdTreeFLANN sorted_ = true);
//        * computeMeanAndCovarianceMatrix with Scalar = float: nine FLOAT accumulators over the neighbours in that order
//          (xx xy xz yy yz zz x y z), divided by the count, cov = E[ab] - E[a]E[b];
//        * solvePlaneParameters: pcl::eigen33 (matrix scaled by its largest |entry|, closed-form roots of the
//          characteristic polynomial in float, eigenvector of the smallest root = the longest of the three row cross
//          products of A - lambda I), curvature = |lambda / trace|;
//        * flipNormalTowardsViewpoint with the default viewpoint (0, 0, 0).
//      A non-finite point, or one with fewer than 3 neighbours (itself included), gets NaN x 4.
//      out4: nx ny nz curvature per point.  Returns the number of finite normals.
namespace {
void roots2_f(float b, float c, float roots[3]) {
  roots[0] = 0.f;
  float d = (float)(b * b - 4.0 * c);
  if (d < 0.0) d = 0.0;
  const float sd = std::sqrt(d);
  roots[2] = 0.5f * (b + sd);
  roots[1] = 0.5f * (b - sd);
}
// *branch: 2 = c0 < epsilon -> roots2, 3 = trigonometric roots, 4 = trigonometric roots, then the roots2 fallback
void roots3_f(const float m[9], float roots[3], int* branch) {
  const float c0 = m[0] * m[4] * m[8] + 2.f * m[1] * m[2] * m[5] - m[0] * m[5] * m[5] - m[4] * m[2] * m[2] - m[8] * m[1] * m[1];
  const float c1 = m[0] * m[4] - m[1] * m[1] + m[0] * m[8] - m[2] * m[2] + m[4] * m[8] - m[5] * m[5];
  const float c2 = m[0] + m[4] + m[8];
  if (std::fabs(c0) < std::numeric_limits<float>::epsilon()) {
    *branch = 2;
    roots2_f(c2, c1, roots);
    return;
  }
  const float s_inv3 = (float)(1.0 / 3.0);
  const float s_sqrt3 = std::sqrt(3.0f);
  const float c2_over_3 = c2 * s_inv3;
  float a_over_3 = (c1 - c2 * c2_over_3) * s_inv3;
  if (a_over_3 > 0.f) a_over_3 = 0.f;
  const float half_b = 0.5f * (c0 + c2_over_3 * (2.f * c2_over_3 * c2_over_3 - c1));
  float q = half_b * half_b + a_over_3 * a_over_3 * a_over_3;
  if (q > 0.f) q = 0.f;
  const float rho = std::sqrt(-a_over_3);
  const float theta = std::atan2(std::sqrt(-q), half_b) * s_inv3;
  const float cos_theta = std::cos(theta), sin_theta = std::sin(theta);
  roots[0] = c2_over_3 + 2.f * rho * cos_theta;
  roots[1] = c2_over_3 - rho * (cos_theta + s_sqrt3 * sin_theta);
  roots[2] = c2_over_3 - rho * (cos_theta - s_sqrt3 * sin_theta);
  if (roots[0] >= roots[1]) std::swap(roots[0], roots[1]);
  if (roots[1] >= roots[2]) {
    std::swap(roots[1], roots[2]);
    if (roots[0] >= roots[1]) std::swap(roots[0], roots[1]);
  }
  *branch = 3;
  if (roots[0] <= 0.f) {
    *branch = 4;
    roots2_f(c2, c1, roots);
  }
}

// the normal of point i into o[0..3]; info (may be null): neighbour count, branch (0 no normal: non-finite point or < 3
// neighbours; 1 zero covariance: every |entry| <= FLT_MIN; 2..4 as roots3_f), root gap roots[1] - roots[0] of the scaled
// matrix, cos_theta of the viewpoint flip.  Returns whether the normal is finite.
bool normal_at(const KdTree& tree, const float* xyz, int i, float r2, float* o, double* info) {
  const float nan = std::numeric_limits<float>::quiet_NaN();
  o[0] = o[1] = o[2] = o[3] = nan;
  if (info) info[0] = info[1] = 0.0, info[2] = info[3] = nan;
  const float* p = xyz + 3 * i;
  if (!(std::isfinite(p[0]) && std::isfinite(p[1]) && std::isfinite(p[2]))) return false;
  std::vector<int> nn;
  tree.radius(p, r2, nn);
  if (info) info[0] = (double)nn.size();
  if (nn.size() < 3) return false;
  std::vector<std::pair<float, int>> order;
  order.reserve(nn.size());
  for (int j : nn) order.emplace_back(sqdist(p, xyz + 3 * j), j);
  std::sort(order.begin(), order.end());
  float accu[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  for (const auto& e : order) {
    const float* c = xyz + 3 * e.second;
    accu[0] += c[0] * c[0];
    accu[1] += c[0] * c[1];
    accu[2] += c[0] * c[2];
    accu[3] += c[1] * c[1];
    accu[4] += c[1] * c[2];
    accu[5] += c[2] * c[2];
    accu[6] += c[0];
    accu[7] += c[1];
    accu[8] += c[2];
  }
  const float cntf = (float)order.size();
  for (int k = 0; k < 9; ++k) accu[k] /= cntf;
  float m[9];
  m[0] = accu[0] - accu[6] * accu[6];
  m[1] = accu[1] - accu[6] * accu[7];
  m[2] = accu[2] - accu[6] * accu[8];
  m[4] = accu[3] - accu[7] * accu[7];
  m[5] = accu[4] - accu[7] * accu[8];
  m[8] = accu[5] - accu[8] * accu[8];
  m[3] = m[1];
  m[6] = m[2];
  m[7] = m[5];
  // pcl::eigen33(mat, eigenvalue, eigenvector)
  float scale = 0.f;
  for (int k = 0; k < 9; ++k) scale = std::max(scale, std::fabs(m[k]));
  const bool zero_cov = scale <= std::numeric_limits<float>::min();
  if (zero_cov) scale = 1.f;
  float sm[9];
  for (int k = 0; k < 9; ++k) sm[k] = m[k] / scale;
  float roots[3];
  int branch = 0;
  roots3_f(sm, roots, &branch);
  if (info) info[1] = zero_cov ? 1 : branch, info[2] = (double)roots[1] - (double)roots[0];
  const float eigenvalue = roots[0] * scale;
  sm[0] -= roots[0];
  sm[4] -= roots[0];
  sm[8] -= roots[0];
  auto cross = [](const float* a, const float* b, float* c) {
    c[0] = a[1] * b[2] - a[2] * b[1];
    c[1] = a[2] * b[0] - a[0] * b[2];
    c[2] = a[0] * b[1] - a[1] * b[0];
  };
  float v1[3], v2[3], v3[3];
  cross(sm, sm + 3, v1);
  cross(sm, sm + 6, v2);
  cross(sm + 3, sm + 6, v3);
  const float l1 = v1[0] * v1[0] + v1[1] * v1[1] + v1[2] * v1[2];
  const float l2 = v2[0] * v2[0] + v2[1] * v2[1] + v2[2] * v2[2];
  const float l3 = v3[0] * v3[0] + v3[1] * v3[1] + v3[2] * v3[2];
  const float* v = v3;
  float len = l3;
  if (l1 >= l2 && l1 >= l3) {
    v = v1;
    len = l1;
  } else if (l2 >= l1 && l2 >= l3) {
    v = v2;
    len = l2;
  }
  const float s = std::sqrt(len);
  float nx = v[0] / s, ny = v[1] / s, nz = v[2] / s;
  const float eig_sum = m[0] + m[4] + m[8];
  const float curvature = eig_sum != 0.f ? std::fabs(eigenvalue / eig_sum) : 0.f;
  // flipNormalTowardsViewpoint(point, 0, 0, 0, ...)
  const float vx = 0.f - p[0], vy = 0.f - p[1], vz = 0.f - p[2];
  const float cos_theta = vx * nx + vy * ny + vz * nz;
  if (info) info[3] = cos_theta;
  if (cos_theta < 0) {
    nx *= -1;
    ny *= -1;
    nz *= -1;
  }
  o[0] = nx;
  o[1] = ny;
  o[2] = nz;
  o[3] = curvature;
  // a covariance that cancelled to zero gives 0 / 0 above: the normal is NaN although the point has neighbours
  return std::isfinite(nx) && std::isfinite(ny) && std::isfinite(nz);
}

int normals_impl(const float* xyz, int n, double radius, float* out4, double* info4) {
  KdTree tree(xyz, n);
  const float r2 = (float)(radius * radius);
  int kept = 0;
#ifdef _OPENMP
#pragma omp parallel for reduction(+ : kept) schedule(dynamic, 256)
#endif
  for (int i = 0; i < n; ++i)
    kept += normal_at(tree, xyz, i, r2, out4 + 4 * (size_t)i, info4 ? info4 + 4 * (size_t)i : nullptr) ? 1 : 0;
  return kept;
}
}  // namespace

int orc_normals(const float* xyz, int n, double radius, float* out4) { return normals_impl(xyz, n, radius, out4, nullptr); }

// orc_normals plus, per point, info4 = (neighbour count, branch, root gap, cos_theta) - see normal_at.  The rows of out4 are
// the rows orc_normals gives.
int orc_normals_ex(const float* xyz, int n, double radius, float* out4, double* info4) {
  return normals_impl(xyz, n, radius, out4, info4);
}

// ---- pcl::EuclideanClusterExtraction::extract (reference src/FODDetector.cpp:45-58): extractEuclideanClusters
//      restated literally - for every unprocessed point a seed queue is grown with the radius neighbours
//      (d2 < float(tolerance^2), the query itself comes first in the sorted result and is skipped) of each queued
//      point; a queue of min_size..max_size points becomes a cluster (indices sorted); extract() then sorts the
//      clusters by size, largest first.  std::sort leaves the order of equal-sized clusters unspecified: here they keep
//      their discovery order (lowest seed index first).  labels[i] = rank of the cluster of point i, -1 = none.
//      Non-finite points are not in the tree and never seeded (the reference's difference cloud is dense).
int orc_euclidean_clusters(const float* xyz, int n, double tolerance, int min_size, int max_size, int* labels) {
  for (int i = 0; i < n; ++i) labels[i] = -1;
  if (n <= 0) return 0;
  if (max_size <= 0) max_size = std::numeric_limits<int>::max();
  KdTree tree(xyz, n);
  const float r2 = (float)(tolerance * tolerance);
  std::vector<char> processed((size_t)n, 0);
  std::vector<std::vector<int>> clusters;
  std::vector<int> nn;
  for (int i = 0; i < n; ++i) {
    if (processed[i]) continue;
    const float* p = xyz + 3 * i;
    if (!(std::isfinite(p[0]) && std::isfinite(p[1]) && std::isfinite(p[2]))) continue;
    std::vector<int> seed_queue;
    size_t sq_idx = 0;
    seed_queue.push_back(i);
    processed[i] = 1;
    while (sq_idx < seed_queue.size()) {
      nn.clear();
      tree.radius(xyz + 3 * seed_queue[sq_idx], r2, nn);
      for (size_t j = 0; j < nn.size(); ++j) {
        if (processed[nn[j]]) continue;  // includes the query itself (nn_start_idx = 1 in PCL)
        seed_queue.push_back(nn[j]);
        processed[nn[j]] = 1;
      }
      ++sq_idx;
    }
    if ((int64_t)seed_queue.size() >= min_size && (int64_t)seed_queue.size() <= max_size) {
      std::sort(seed_queue.begin(), seed_queue.end());
      clusters.push_back(std::move(seed_queue));
    }
  }
  std::stable_sort(clusters.begin(), clusters.end(),
                   [](const std::vector<int>& a, const std::vector<int>& b) { return a.size() > b.size(); });
  for (size_t k = 0; k < clusters.size(); ++k)
    for (int idx : clusters[k]) labels[idx] = (int)k;
  return (int)clusters.size();
}

// ---- pcl::VoxelGrid<PointXYZRGB>::applyFilter with leaf (l, l, l), downsample_all_data_ = true,
//      min_points_per_voxel_ = 0 (reference src/Filter.cpp:91-105).  `pts` holds n points of `stride` bytes (xyz
//      floats first; when stride >= 20 the packed rgba word sits at byte 16 as in PointXYZRGB).  One output point per
//      occupied voxel in ascending voxel index: xyz = float sum / count (AccumulatorXYZ), rgba channels =
//      uint32(float sum / count) (AccumulatorRGBA), data[3] = 1, remaining bytes 0.  PCL sorts the (voxel, point)
//      pairs with std::sort on the voxel index alone, which leaves the order inside a voxel unspecified; here it is
//      the original point order (a stable sort), which fixes the float summation order.
//      Returns the number of output points, or -1 when PCL would refuse the leaf size (index overflow) and copy
//      the input through.
int64_t orc_voxel_grid(const unsigned char* pts, int64_t n, int64_t stride, double leaf_size, unsigned char* out) {
  const float leaf = (float)leaf_size;
  const float inv = 1.0f / leaf;
  float min_p[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, max_p[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
  int64_t n_valid = 0;
  for (int64_t i = 0; i < n; ++i) {
    const float* p = reinterpret_cast<const float*>(pts + i * stride);
    if (!(std::isfinite(p[0]) && std::isfinite(p[1]) && std::isfinite(p[2]))) continue;
    ++n_valid;
    for (int a = 0; a < 3; ++a) {
      min_p[a] = std::min(min_p[a], p[a]);
      max_p[a] = std::max(max_p[a], p[a]);
    }
  }
  if (n_valid == 0) return 0;
  const int64_t dx = (int64_t)((max_p[0] - min_p[0]) * inv) + 1;
  const int64_t dy = (int64_t)((max_p[1] - min_p[1]) * inv) + 1;
  const int64_t dz = (int64_t)((max_p[2] - min_p[2]) * inv) + 1;
  // PCL tests dx*dy*dz (int64) against INT32_MAX; the running product is checked here so that it cannot wrap
  const int64_t lim = (int64_t)std::numeric_limits<int32_t>::max();
  if (dx > lim || dx * dy > lim || dx * dy * dz > lim) return -1;
  int min_b[3], div_b[3];
  for (int a = 0; a < 3; ++a) {
    min_b[a] = (int)std::floor(min_p[a] * inv);
    const int max_b = (int)std::floor(max_p[a] * inv);
    div_b[a] = max_b - min_b[a] + 1;
  }
  // PCL's int index arithmetic, in uint32_t so that it wraps with the same bits where div_b[0] * div_b[1] * div_b[2]
  // passes 2^31 (its dx * dy * dz check can pass while div_b, up to dx + 1 per axis, does not)
  const uint32_t mul[3] = {1u, (uint32_t)div_b[0], (uint32_t)div_b[0] * (uint32_t)div_b[1]};
  std::vector<std::pair<unsigned, int64_t>> index_vector;
  index_vector.reserve((size_t)n_valid);
  for (int64_t i = 0; i < n; ++i) {
    const float* p = reinterpret_cast<const float*>(pts + i * stride);
    if (!(std::isfinite(p[0]) && std::isfinite(p[1]) && std::isfinite(p[2]))) continue;
    const int ijk0 = (int)(std::floor(p[0] * inv) - (float)min_b[0]);
    const int ijk1 = (int)(std::floor(p[1] * inv) - (float)min_b[1]);
    const int ijk2 = (int)(std::floor(p[2] * inv) - (float)min_b[2]);
    index_vector.emplace_back((uint32_t)ijk0 * mul[0] + (uint32_t)ijk1 * mul[1] + (uint32_t)ijk2 * mul[2], i);
  }
  std::stable_sort(index_vector.begin(), index_vector.end(),
                   [](const std::pair<unsigned, int64_t>& a, const std::pair<unsigned, int64_t>& b) { return a.first < b.first; });
  int64_t n_out = 0;
  size_t first = 0;
  while (first < index_vector.size()) {
    size_t last = first + 1;
    while (last < index_vector.size() && index_vector[last].first == index_vector[first].first) ++last;
    float sx = 0.f, sy = 0.f, sz = 0.f, sr = 0.f, sg = 0.f, sb = 0.f, sa = 0.f;
    for (size_t k = first; k < last; ++k) {
      const unsigned char* pt = pts + index_vector[k].second * stride;
      const float* p = reinterpret_cast<const float*>(pt);
      sx += p[0];
      sy += p[1];
      sz += p[2];
      if (stride >= 20) {
        uint32_t c;
        std::memcpy(&c, pt + 16, 4);
        sb += (float)(c & 255u);
        sg += (float)((c >> 8) & 255u);
        sr += (float)((c >> 16) & 255u);
        sa += (float)(c >> 24);
      }
    }
    const float cnt = (float)(last - first);
    unsigned char* o = out + n_out * stride;
    std::memset(o, 0, (size_t)stride);
    const float c3[3] = {sx / cnt, sy / cnt, sz / cnt};
    std::memcpy(o, c3, 12);
    if (stride >= 16) {
      const float one = 1.0f;
      std::memcpy(o + 12, &one, 4);
    }
    if (stride >= 20) {
      const uint32_t c = ((uint32_t)(sa / cnt) << 24) | ((uint32_t)(sr / cnt) << 16) | ((uint32_t)(sg / cnt) << 8) |
                         (uint32_t)(sb / cnt);
      std::memcpy(o + 16, &c, 4);
    }
    ++n_out;
    first = last;
  }
  return n_out;
}

}  // extern "C"
