// knn_cov.cu - per-point k-nearest-neighbour search (k = 20 by default) on the brick grid and the GICP
// plane-to-plane covariance of each neighbourhood.
//
// Replaces pcl::GeneralizedIterativeClosestPoint::computeCovariances (PCL 1.8.1 gicp.hpp), run twice inside
// gicp_.align() at reference src/GICPAlignment.cpp:96: kNN-k of every point in its own cloud (the point itself
// is neighbour 0), mean / covariance accumulated in double from FLOAT products in neighbour order, SVD, and the
// singular values replaced by (1, 1, gicp_epsilon).  The rebuilt matrix equals I - (1 - eps) n n^T with n the
// singular vector of the smallest singular value, so only n (3 doubles) is stored per point.
//
// Mapping: one thread per query.  Consecutive threads hold consecutive points of the sorted cloud, i.e. spatial
// neighbours, so a warp walks the same few rows of cells and its loads hit L1.  Each thread keeps its k best
// candidates as a list sorted by (d2, original index) in shared memory (column layout: entry j of thread t at
// [j * blockDim + t], conflict-free), inserting only candidates that beat the current k-th.  The cells are visited
// in Chebyshev rings around the query's cell (the 3x3x3 box, then shells 2..kKnnMaxRing cut to the ball of the k-th
// distance); a query whose k-th neighbour is farther than that restarts on the hierarchical traversal (common.cuh).
#include <atomic>
#include <climits>
#include <cstdlib>

#include "kernels.hpp"
#include "knn_search.cuh"

namespace gicpb {

namespace {

constexpr int kKnnNearThreads = 256;  // consecutive (= neighbouring) queries of one block share its L1 lines
constexpr int kKnnFarThreads = 128;   // far_for_each needs 128

template <int P, int Q>
__device__ __forceinline__ void jacobi_rotate(double (&a)[9], double (&v)[9]) {
  const double apq = a[3 * P + Q];
  if (apq == 0.0) return;
  const double theta = (a[3 * Q + Q] - a[3 * P + P]) / (2.0 * apq);
  const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
  const double c = 1.0 / sqrt(t * t + 1.0);
  const double s = t * c;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const double akp = a[3 * k + P], akq = a[3 * k + Q];
    a[3 * k + P] = c * akp - s * akq;
    a[3 * k + Q] = s * akp + c * akq;
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const double apk = a[3 * P + k], aqk = a[3 * Q + k];
    a[3 * P + k] = c * apk - s * aqk;
    a[3 * Q + k] = s * apk + c * aqk;
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const double vkp = v[3 * k + P], vkq = v[3 * k + Q];
    v[3 * k + P] = c * vkp - s * vkq;
    v[3 * k + Q] = s * vkp + c * vkq;
  }
}

template <bool kFar, int kKnnThreads>
__global__ void __launch_bounds__(kKnnThreads) knn_cov_kernel(GridView g, int lo, int hi, int k,
                                                               double* __restrict__ normals,
                                                               int* __restrict__ knn_idx,
                                                               float* __restrict__ knn_d2, FarWork fw, int win_axis,
                                                               float win_lo, float win_hi,
                                                               unsigned* __restrict__ win_violations) {
  extern __shared__ __align__(8) int smem[];
  KnnVisitor<kKnnThreads> L;
  L.pts = g.pts;
  L.lkey = reinterpret_cast<unsigned long long*>(smem) + threadIdx.x;
  L.k = k;
  unsigned* qb = reinterpret_cast<unsigned*>(smem) + 2 * k * kKnnThreads + threadIdx.x;  // near instance only
  unsigned* qe = qb + kKnnQueueCap * kKnnThreads;
  auto body = [&](int item) {
  const int i = lo + item;
  const float4 qp = __ldg(&g.pts[i]);
  L.qx = qp.x;
  L.qy = qp.y;
  L.qz = qp.z;
  const Query q = make_query(g, qp.x, qp.y, qp.z);
  if (kFar) {
    knn_far(g, q, L);
  } else if (!knn_near<kKnnThreads, kKnnQueueCap>(g, q, L, qb, qe)) {
    fw.flags[item] = 1;
    return;
  }
  if (win_axis >= 0) {
    // A windowed index (sharded source) only holds the points between win_lo and win_hi along win_axis: the list is the
    // cloud's k nearest only if the k-th of them is no farther than the nearer end of the window.  Every point this
    // cannot be said of is counted; the caller then indexes the whole cloud instead.
    const float v = win_axis == 0 ? qp.x : (win_axis == 1 ? qp.y : qp.z);
    const float gap = fsub(fminf(fsub(v, win_lo), fsub(win_hi, v)), g.margin);
    const float kd = L.count == k ? L.d2_at(k - 1) : __int_as_float(0x7f800000);
    if (!(gap > 0.f && kd <= fmul(fmul(gap, gap), 0.999999f))) atomicAdd(win_violations, 1u);
  }
  if (knn_idx) {
    for (int j = 0; j < k; ++j) {
      const size_t row = (size_t)(i - lo) * k + j;
      knn_idx[row] = j < L.count ? L.oi_at(j) : -1;
      knn_d2[row] = j < L.count ? L.d2_at(j) : __int_as_float(0x7f800000);
    }
  }

  // ---- covariance in double from float products, in neighbour order (gicp.hpp) ---------------------------
  double mean0 = 0.0, mean1 = 0.0, mean2 = 0.0;
  double c00 = 0.0, c10 = 0.0, c11 = 0.0, c20 = 0.0, c21 = 0.0, c22 = 0.0;
  for (int j = 0; j < L.count; ++j) {
    const float4 p = __ldg(&g.pts[__ldg(&g.pos_of[L.oi_at(j)])]);
    mean0 += (double)p.x;
    mean1 += (double)p.y;
    mean2 += (double)p.z;
    c00 += (double)__fmul_rn(p.x, p.x);
    c10 += (double)__fmul_rn(p.y, p.x);
    c11 += (double)__fmul_rn(p.y, p.y);
    c20 += (double)__fmul_rn(p.z, p.x);
    c21 += (double)__fmul_rn(p.z, p.y);
    c22 += (double)__fmul_rn(p.z, p.z);
  }
  const double kd = (double)k;
  mean0 = __ddiv_rn(mean0, kd);
  mean1 = __ddiv_rn(mean1, kd);
  mean2 = __ddiv_rn(mean2, kd);
  double a[9], v[9] = {1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0};
  a[0] = __dsub_rn(__ddiv_rn(c00, kd), __dmul_rn(mean0, mean0));
  a[3] = __dsub_rn(__ddiv_rn(c10, kd), __dmul_rn(mean1, mean0));
  a[4] = __dsub_rn(__ddiv_rn(c11, kd), __dmul_rn(mean1, mean1));
  a[6] = __dsub_rn(__ddiv_rn(c20, kd), __dmul_rn(mean2, mean0));
  a[7] = __dsub_rn(__ddiv_rn(c21, kd), __dmul_rn(mean2, mean1));
  a[8] = __dsub_rn(__ddiv_rn(c22, kd), __dmul_rn(mean2, mean2));
  a[1] = a[3];
  a[2] = a[6];
  a[5] = a[7];
  for (int sweep = 0; sweep < 64; ++sweep) {
    const double off = fabs(a[1]) + fabs(a[2]) + fabs(a[5]);
    const double diag = fabs(a[0]) + fabs(a[4]) + fabs(a[8]);
    if (off == 0.0 || off <= 1e-300 || off < 1e-22 * diag) break;
    jacobi_rotate<0, 1>(a, v);
    jacobi_rotate<0, 2>(a, v);
    jacobi_rotate<1, 2>(a, v);
  }
  // singular vector of the smallest |eigenvalue| (ties -> highest index, as a stable descending sort leaves it last)
  const double e0 = fabs(a[0]), e1 = fabs(a[4]), e2 = fabs(a[8]);
  int best = 0;
  double eb = e0;
  if (e1 <= eb) { best = 1; eb = e1; }
  if (e2 <= eb) { best = 2; }
  const double nx = best == 0 ? v[0] : (best == 1 ? v[1] : v[2]);
  const double ny = best == 0 ? v[3] : (best == 1 ? v[4] : v[5]);
  const double nz = best == 0 ? v[6] : (best == 1 ? v[7] : v[8]);
  double* out = normals + 3 * (size_t)(i - lo);
  out[0] = nx;
  out[1] = ny;
  out[2] = nz;
  };
  if (kFar) {
    far_for_each(fw, hi - lo, body);
  } else {
    const int item = blockIdx.x * kKnnThreads + threadIdx.x;
    if (item < hi - lo) {
      fw.flags[item] = 0;
      body(item);
    }
  }
}

}  // namespace

void launch_knn_covariances(const GridView& g, int lo, int hi, int k, double* normals, int* knn_idx, float* knn_d2,
                            const FarWork& fw, cudaStream_t stream, const GridIndex::KnnWindow* win, unsigned* win_violations) {
  const int win_axis = (win && win_violations) ? win->axis : -1;
  const float win_lo = win ? win->lo : 0.f, win_hi = win ? win->hi : 0.f;
  const int n = hi - lo;
  if (n <= 0) return;
  reset_far(fw, n, stream);
  // threads per block of the near instance: 256 by default; GICPB_KNN_THREADS=128 for measurements
  static const int near_threads = [] {
    const char* e = std::getenv("GICPB_KNN_THREADS");
    return (e && std::atoi(e) == 128) ? 128 : kKnnNearThreads;
  }();
  const size_t heap_near = (size_t)2 * k * near_threads * sizeof(int);
  const size_t heap = (size_t)2 * k * kKnnFarThreads * sizeof(int);
  const size_t queue = (size_t)2 * kKnnQueueCap * near_threads * sizeof(unsigned);
  const unsigned nb = (unsigned)((n + near_threads - 1) / near_threads);
  static std::atomic<unsigned long long> attr_set{0ull};  // one bit per device: the attribute belongs to the device's context
  int dev = 0;
  GICPB_CUDA(cudaGetDevice(&dev));
  if (dev >= 64 || !((attr_set.load() >> dev) & 1ull)) {  // up to 88 KB of dynamic shared memory at k = 32
    GICPB_CUDA(cudaFuncSetAttribute(knn_cov_kernel<false, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    GICPB_CUDA(cudaFuncSetAttribute(knn_cov_kernel<false, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    GICPB_CUDA(cudaFuncSetAttribute(knn_cov_kernel<false, 256>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    if (dev < 64) attr_set.fetch_or(1ull << dev);
  }
  if (near_threads == 128)
    knn_cov_kernel<false, 128><<<nb, 128, heap_near + queue, stream>>>(g, lo, hi, k, normals, knn_idx, knn_d2, fw, win_axis, win_lo,
                                                                      win_hi, win_violations);
  else
    knn_cov_kernel<false, 256><<<nb, 256, heap_near + queue, stream>>>(g, lo, hi, k, normals, knn_idx, knn_d2, fw, win_axis, win_lo,
                                                                      win_hi, win_violations);
  GICPB_LAUNCHED();
  knn_cov_kernel<true, kKnnFarThreads><<<fw.far_blocks, kKnnFarThreads, heap, stream>>>(g, lo, hi, k, normals, knn_idx, knn_d2, fw,
                                                                                       win_axis, win_lo, win_hi, win_violations);
  GICPB_LAUNCHED();
}

}  // namespace gicpb
