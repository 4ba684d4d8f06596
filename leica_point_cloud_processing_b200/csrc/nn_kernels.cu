// nn_kernels.cu - nearest-neighbour kernels on the brick grid: the per-outer-iteration correspondence pass
// (transform, exact NN-1, distance gate, Mahalanobis matrix), the fitness score, the cloud difference, the raw
// NN-1 test hook and the cloud transform.
//
// Reference loops replaced (PCL 1.8.1 behind the reference's call sites):
//   correspondence_kernel  GICP::computeTransformation inner `for i < N` loop (gicp.hpp), reached from
//                          gicp_.align() at reference src/GICPAlignment.cpp:96,116
//   fitness_kernel         Registration::getFitnessScore, reference src/GICPAlignment.cpp:103,123
//   difference_kernel      pcl::getPointCloudDifference, reference src/Filter.cpp:176-189
//   transform_kernel       pcl::transformPointCloud, reference src/GICPAlignment.cpp:146
//
// Every search kernel exists in two instances.  The NEAR instance runs one thread per query: it answers the query
// from the cells around it (nn_near: queue the point ranges, then one flat scan) with a small register footprint,
// and appends the few queries that need more (nothing within a cell or two, or a seed that is far off) to a device
// work list.  The FAR instance walks that list with a persistent grid and runs the hierarchical traversal
// (nn_far) for each entry.  Both write the same outputs, so a query is answered by exactly one of them.
#include <climits>

#include "kernels.hpp"
#include "knn_search.cuh"

namespace gicpb {

namespace {

constexpr int kNnThreads = 128;

// gate2 >= 0: only candidates with d2 < gate2 count (gate2 == 0 admits none, as PCL's `nn_dists[0] < dist_threshold`
// with a zero threshold); gate2 < 0: ungated
__device__ __forceinline__ NNState nn_init(float gate2) {
  NNState s;
  if (gate2 >= 0.f) {
    s.best = gate2;  // strict '<' gate: nothing ties with the sentinel because its index is -1
    s.pos = -1;
    s.oi = -1;
  } else {
    s.best = __int_as_float(0x7f800000);
    s.pos = -1;
    s.oi = INT_MAX;
  }
  return s;
}

// Runs the search of one query in this instance.  false: the query was handed to the far instance (near only).
template <bool kFar, bool kEarlyExit>
__device__ __forceinline__ bool search_item(const GridView& g, float qx, float qy, float qz, NNState& s, int item,
                                            const FarWork& fw, unsigned* qb, unsigned* qe, bool& hit) {
  const Query q = make_query(g, qx, qy, qz);
  if (kFar) {
    hit = nn_far<kEarlyExit>(g, q, s);
    return true;
  }
  const int r = nn_near<kEarlyExit, kNnThreads, kNnQueueCap>(g, q, s, qb, qe, fw.near_rings);
  if (r == kNear_Far) {
    fw.flags[item] = 1;
    return false;
  }
  hit = (r == kNear_Stop);
  return true;
}

#define GICPB_NEAR_QUEUE()                                     \
  __shared__ unsigned s_qb[kFar ? 1 : kNnQueueCap * kNnThreads]; \
  __shared__ unsigned s_qe[kFar ? 1 : kNnQueueCap * kNnThreads]; \
  unsigned* qb = s_qb + (kFar ? 0 : threadIdx.x);              \
  unsigned* qe = s_qe + (kFar ? 0 : threadIdx.x)

// item loop shared by all search kernels: the near grid covers the items once (one per thread, and clears the item's
// far flag before the search may set it); the far grid works through the flagged items (kernels.hpp far_for_each)
#define GICPB_RUN_ITEMS(n_items, body)                            \
  if (kFar) {                                                     \
    far_for_each(fw, (int)(n_items), body);                       \
  } else {                                                        \
    const int k_ = blockIdx.x * kNnThreads + threadIdx.x;         \
    if (k_ < (int)(n_items)) {                                    \
      fw.flags[k_] = 0;                                           \
      body(k_);                                                   \
    }                                                             \
  }

template <bool kFar>
__global__ void __launch_bounds__(kNnThreads, kFar ? 6 : 8) nn1_kernel(GridView g, const float4* __restrict__ queries, int n, Rigid T,
                                                          float gate2, int* __restrict__ idx, float* __restrict__ d2,
                                                          int* __restrict__ pos_out, FarWork fw) {
  GICPB_NEAR_QUEUE();
  auto body = [&](int i) {
    const float4 p = __ldg(&queries[i]);
    NNState s = nn_init(gate2);
    if (finite3(p.x, p.y, p.z)) {
      const float3 q = xform(T, p.x, p.y, p.z);
      bool hit;
      if (finite3(q.x, q.y, q.z) && !search_item<kFar, false>(g, q.x, q.y, q.z, s, i, fw, qb, qe, hit)) return;
    }
    if (idx) idx[i] = s.pos >= 0 ? s.oi : -1;
    if (d2) d2[i] = s.pos >= 0 ? s.best : __int_as_float(0x7f800000);
    if (pos_out) pos_out[i] = s.pos;
  };
  GICPB_RUN_ITEMS(n, body)
}

// M = (R C1 R^T + C2)^-1 in double, C = I - (1 - eps) n n^T  (gicp.hpp: M = R*C1; temp = M*R^T; temp += C2)
template <typename MT>
__device__ __forceinline__ void write_mahalanobis(const RotD& R, const double* __restrict__ ns, const double* __restrict__ nt,
                                                  double eps, MT* __restrict__ m) {
  const double a = 1.0 - eps;
  const double sx = ns[0], sy = ns[1], sz = ns[2];
  const double tx = nt[0], ty = nt[1], tz = nt[2];
  double C1[9] = {1.0 - a * sx * sx, -a * sx * sy, -a * sx * sz, -a * sy * sx, 1.0 - a * sy * sy, -a * sy * sz,
                  -a * sz * sx, -a * sz * sy, 1.0 - a * sz * sz};
  double RC[9];
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int cc = 0; cc < 3; ++cc)
      RC[3 * r + cc] = R.m[3 * r] * C1[cc] + R.m[3 * r + 1] * C1[3 + cc] + R.m[3 * r + 2] * C1[6 + cc];
  double A[9];
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int cc = 0; cc < 3; ++cc)
      A[3 * r + cc] = RC[3 * r] * R.m[3 * cc] + RC[3 * r + 1] * R.m[3 * cc + 1] + RC[3 * r + 2] * R.m[3 * cc + 2];
  A[0] += 1.0 - a * tx * tx; A[1] += -a * tx * ty;      A[2] += -a * tx * tz;
  A[3] += -a * ty * tx;      A[4] += 1.0 - a * ty * ty; A[5] += -a * ty * tz;
  A[6] += -a * tz * tx;      A[7] += -a * tz * ty;      A[8] += 1.0 - a * tz * tz;
  // adjugate inverse (Eigen's fixed-size 3x3 path)
  const double c00 = A[4] * A[8] - A[5] * A[7];
  const double c01 = A[2] * A[7] - A[1] * A[8];
  const double c02 = A[1] * A[5] - A[2] * A[4];
  const double c10 = A[5] * A[6] - A[3] * A[8];
  const double c11 = A[0] * A[8] - A[2] * A[6];
  const double c12 = A[2] * A[3] - A[0] * A[5];
  const double c20 = A[3] * A[7] - A[4] * A[6];
  const double c22 = A[0] * A[4] - A[1] * A[3];
  const double inv = 1.0 / (A[0] * c00 + A[1] * c10 + A[2] * c20);
  m[0] = (MT)(c00 * inv);
  m[1] = (MT)(c01 * inv);
  m[2] = (MT)(c02 * inv);
  m[3] = (MT)(c11 * inv);
  m[4] = (MT)(c12 * inv);
  m[5] = (MT)(c22 * inv);
}

// One item per source point of this rank's shard [lo, hi) (sorted source order); item t <-> point lo + t.
template <typename MT, bool kUsePrev, bool kFar>
__global__ void __launch_bounds__(kNnThreads, kFar ? 6 : 8)
correspondence_kernel(GridView g, const float4* __restrict__ src, int lo, int hi, Rigid T, RotD R, float gate2,
                      const double* __restrict__ n_src, const double* __restrict__ n_tgt, double eps,
                      int* __restrict__ pair_pos, float* __restrict__ pair_d2, float4* __restrict__ pair_tgt,
                      MT* __restrict__ maha, FarWork fw) {
  GICPB_NEAR_QUEUE();
  auto body = [&](int t) {
    const float4 p = __ldg(&src[lo + t]);
    const float3 q = xform(T, p.x, p.y, p.z);
    NNState s = nn_init(gate2);
    if (kUsePrev) {
      const int prev = pair_pos[t];
      if (prev >= 0) {
        const float4 c = __ldg(&g.pts[prev]);
        const float d = dist2(q.x, q.y, q.z, c);
        const int oi = __float_as_int(c.w);
        if (cand_less(d, oi, s.best, s.oi)) {
          s.best = d;
          s.pos = prev;
          s.oi = oi;
        }
      }
    }
    bool hit;
    // a zero gate admits no candidate: nothing to search for
    if (gate2 != 0.f && finite3(q.x, q.y, q.z) && !search_item<kFar, false>(g, q.x, q.y, q.z, s, t, fw, qb, qe, hit)) return;
    pair_pos[t] = s.pos;
    pair_d2[t] = s.pos >= 0 ? s.best : __int_as_float(0x7f800000);
    if (s.pos < 0) {
      pair_tgt[t] = make_float4(0.f, 0.f, 0.f, 0.f);
      return;
    }
    const float4 c = __ldg(&g.pts[s.pos]);
    pair_tgt[t] = make_float4(c.x, c.y, c.z, 1.0f);
    write_mahalanobis<MT>(R, n_src + 3 * (size_t)t, n_tgt + 3 * (size_t)s.pos, eps, maha + 6 * (size_t)t);
  };
  GICPB_RUN_ITEMS(hi - lo, body)
}

// fitness: partial (sum d2, count) per block -> partials[(row0 + block)*2 + {0,1}]
// seed (nullable): pair_pos of the last correspondence pass - the match of each source point under a nearby pose is a
// first candidate that bounds the search ball (it is only a candidate: the result is the exact nearest neighbour)
template <bool kFar>
__global__ void __launch_bounds__(kNnThreads, kFar ? 6 : 8) fitness_kernel(GridView g, const float4* __restrict__ src, int lo, int hi,
                                                              Rigid T, double max_range, const int* __restrict__ seed,
                                                              double* __restrict__ partials, int row0, FarWork fw) {
  GICPB_NEAR_QUEUE();
  __shared__ double ssum[4], scnt[4];
  double sum = 0.0, cnt = 0.0;
  auto body = [&](int t) {
    const float4 p = __ldg(&src[lo + t]);
    const float3 q = xform(T, p.x, p.y, p.z);
    NNState s = nn_init(-1.f);
    if (seed) {
      const int prev = __ldg(&seed[t]);
      if (prev >= 0) {
        const float4 c = __ldg(&g.pts[prev]);
        s.best = dist2(q.x, q.y, q.z, c);
        s.pos = prev;
        s.oi = __float_as_int(c.w);
      }
    }
    bool hit;
    if (finite3(q.x, q.y, q.z) && !search_item<kFar, false>(g, q.x, q.y, q.z, s, t, fw, qb, qe, hit)) return;
    if (s.pos >= 0 && (double)s.best <= max_range) {
      sum += (double)s.best;
      cnt += 1.0;
    }
  };
  GICPB_RUN_ITEMS(hi - lo, body)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (!kFar) {
    // near instance: one row per WARP and no block-wide barrier - a warp whose queries are done leaves instead of holding
    // its place on the SM until the slowest warp of the block arrives (the barrier was 30 % of this kernel's stall samples)
    __syncwarp();
    sum = warp_sum(sum);
    cnt = warp_sum(cnt);
    if (lane == 0) {
      const size_t row = (size_t)row0 + (size_t)blockIdx.x * (kNnThreads / 32) + warp;
      partials[2 * row] = sum;
      partials[2 * row + 1] = cnt;
    }
    return;
  }
  __syncthreads();
  sum = warp_sum(sum);
  cnt = warp_sum(cnt);
  if (lane == 0) {
    ssum[warp] = sum;
    scnt[warp] = cnt;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    partials[2 * (size_t)(row0 + blockIdx.x)] = (ssum[0] + ssum[1]) + (ssum[2] + ssum[3]);
    partials[2 * (size_t)(row0 + blockIdx.x) + 1] = (scnt[0] + scnt[1]) + (scnt[2] + scnt[3]);
  }
}

// out[c] = sum over rows of partials[row*ncols + c], fixed order (deterministic): one block of 1024 threads, four
// independent partial sums per thread (rows t, t + 1024, ... taken four at a time) so that the loads are all in flight
constexpr int kReduceThreads = 1024;
__global__ void __launch_bounds__(kReduceThreads) reduce_partials_kernel(const double* __restrict__ partials, int nrows, int ncols,
                                                                          double* __restrict__ out) {
  __shared__ double sm[kReduceThreads / 32];
  for (int c = 0; c < ncols; ++c) {
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    int r = threadIdx.x;
    for (; r + 3 * kReduceThreads < nrows; r += 4 * kReduceThreads) {
      a0 += partials[(size_t)r * ncols + c];
      a1 += partials[(size_t)(r + kReduceThreads) * ncols + c];
      a2 += partials[(size_t)(r + 2 * kReduceThreads) * ncols + c];
      a3 += partials[(size_t)(r + 3 * kReduceThreads) * ncols + c];
    }
    for (; r < nrows; r += kReduceThreads) a0 += partials[(size_t)r * ncols + c];
    double v = (a0 + a1) + (a2 + a3);
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
      double t = 0.0;
      for (int w = 0; w < kReduceThreads / 32; ++w) t += sm[w];
      out[c] = t;
    }
    __syncthreads();
  }
}

// difference: mask[i] = 1 iff point i is finite and no subtract point lies within d2 <= thr (thr_next = the
// smallest float above thr, so "d2 < thr_next" == "!(d2 > thr)").  Kept count -> atomicAdd per warp.
template <bool kFar>
__global__ void __launch_bounds__(kNnThreads, kFar ? 6 : 8) difference_kernel(GridView g, const unsigned char* __restrict__ raw,
                                                                 int64_t n, int64_t stride, float thr_next,
                                                                 int mode, unsigned char* __restrict__ mask,
                                                                 unsigned long long* __restrict__ kept, FarWork fw) {
  GICPB_NEAR_QUEUE();
  unsigned mine = 0;
  auto body = [&](int i) {
    const float* p = reinterpret_cast<const float*>(raw + (int64_t)i * stride);
    const float x = p[0], y = p[1], z = p[2];
    bool keep = false;
    if (finite3(x, y, z) && mode != kDiffKeepNone) {
      if (mode == kDiffKeepAll) {
        keep = true;  // threshold < 0: every finite point with a neighbour is kept
      } else {
        NNState s;
        s.best = thr_next;
        s.pos = -1;
        s.oi = -1;
        bool hit = false;
        if (!search_item<kFar, true>(g, x, y, z, s, i, fw, qb, qe, hit)) return;
        keep = !hit;
      }
    }
    mask[i] = keep ? 1 : 0;
    mine += keep ? 1u : 0u;
  };
  GICPB_RUN_ITEMS(n, body)
  mine = __reduce_add_sync(kFullMask, mine);
  if ((threadIdx.x & 31) == 0 && mine) atomicAdd(kept, (unsigned long long)mine);
}

// ---- the use_covariances branch of the reference (src/GICPAlignment.cpp:56-71): the resolution here, the normals in normals.cu ----
// sum over the indexed points of sqrt(d2 to the 2nd nearest neighbour) (the point itself is the 1st) and their count:
// Utils::computeCloudResolution, reference src/Utils.cpp:145-174.  partials[(row0 + block)*2 + {0,1}]
template <bool kFar>
__global__ void __launch_bounds__(kNnThreads, kFar ? 4 : 6) resolution_kernel(GridView g, double* __restrict__ partials,
                                                                               int row0, FarWork fw) {
  GICPB_NEAR_QUEUE();
  __shared__ unsigned long long s_heap[2 * kNnThreads];
  __shared__ double ssum[4], scnt[4];
  double sum = 0.0, cnt = 0.0;
  auto body = [&](int i) {
    const float4 p = __ldg(&g.pts[i]);
    KnnVisitor<kNnThreads> L;
    L.pts = g.pts;
    L.lkey = s_heap + threadIdx.x;
    L.k = 2;
    L.qx = p.x;
    L.qy = p.y;
    L.qz = p.z;
    const Query q = make_query(g, p.x, p.y, p.z);
    if (kFar) {
      knn_far(g, q, L);
    } else if (!knn_near<kNnThreads, kNnQueueCap>(g, q, L, qb, qe)) {
      fw.flags[i] = 1;
      return;
    }
    if (L.count == 2) {
      sum += sqrt((double)L.d2_at(1));
      cnt += 1.0;
    }
  };
  GICPB_RUN_ITEMS(g.n, body)
  __syncthreads();
  sum = warp_sum(sum);
  cnt = warp_sum(cnt);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) {
    ssum[warp] = sum;
    scnt[warp] = cnt;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    partials[2 * (size_t)(row0 + blockIdx.x)] = (ssum[0] + ssum[1]) + (ssum[2] + ssum[3]);
    partials[2 * (size_t)(row0 + blockIdx.x) + 1] = (scnt[0] + scnt[1]) + (scnt[2] + scnt[3]);
  }
}

// xyz <- T * xyz for strided points; the other bytes of each point are copied (4-byte words).  in == out is allowed:
// every thread reads its own point completely before it writes it.
__global__ void __launch_bounds__(256) transform_kernel(const unsigned char* in, unsigned char* out, int64_t n,
                                                         int64_t stride, Rigid T) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t* p = reinterpret_cast<const uint32_t*>(in + i * stride);
  uint32_t* o = reinterpret_cast<uint32_t*>(out + i * stride);
  const float x = __uint_as_float(p[0]), y = __uint_as_float(p[1]), z = __uint_as_float(p[2]);
  const float3 q = xform(T, x, y, z);
  if (in != out) {
    const int words = (int)(stride >> 2);
    for (int k = 3; k < words; ++k) o[k] = p[k];
  }
  o[0] = __float_as_uint(q.x);
  o[1] = __float_as_uint(q.y);
  o[2] = __float_as_uint(q.z);
}

__global__ void __launch_bounds__(256) pack_queries_kernel(const unsigned char* __restrict__ raw, int64_t n,
                                                            int64_t stride, float4* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* p = reinterpret_cast<const float*>(raw + i * stride);
  out[i] = make_float4(p[0], p[1], p[2], 0.f);
}

inline unsigned nblocks(int64_t n, int threads) { return (unsigned)((n + threads - 1) / threads); }

}  // namespace

void reset_far(const FarWork& fw, int64_t n_items, cudaStream_t stream) {
  GICPB_CUDA(cudaMemsetAsync(fw.tile_counter, 0, 2 * sizeof(unsigned), stream));
  const int64_t padded = (n_items + kFarTile - 1) / kFarTile * kFarTile;  // flags past the last item must read 0
  if (padded > n_items) GICPB_CUDA(cudaMemsetAsync(fw.flags + n_items, 0, (size_t)(padded - n_items), stream));
}

namespace {

}  // namespace

void launch_nn1(const GridView& g, const float4* queries, int n, const Rigid& T, float gate2, int* idx, float* d2,
                int* pos, const FarWork& fw, cudaStream_t stream) {
  if (n <= 0) return;
  reset_far(fw, n, stream);
  nn1_kernel<false><<<nblocks(n, kNnThreads), kNnThreads, 0, stream>>>(g, queries, n, T, gate2, idx, d2, pos, fw);
  GICPB_LAUNCHED();
  nn1_kernel<true><<<fw.far_blocks, kNnThreads, 0, stream>>>(g, queries, n, T, gate2, idx, d2, pos, fw);
  GICPB_LAUNCHED();
}

template <typename MT, bool kUsePrev>
static void launch_corr_t(const GridView& g, const float4* src, int lo, int hi, const Rigid& T, const RotD& R, float gate2,
                          const double* n_src, const double* n_tgt, double eps, int* pair_pos, float* pair_d2,
                          float4* pair_tgt, void* maha, const FarWork& fw, cudaStream_t stream) {
  const unsigned nb = nblocks(hi - lo, kNnThreads);
  correspondence_kernel<MT, kUsePrev, false><<<nb, kNnThreads, 0, stream>>>(g, src, lo, hi, T, R, gate2, n_src, n_tgt, eps,
                                                                             pair_pos, pair_d2, pair_tgt, (MT*)maha, fw);
  GICPB_LAUNCHED();
  correspondence_kernel<MT, kUsePrev, true><<<fw.far_blocks, kNnThreads, 0, stream>>>(
      g, src, lo, hi, T, R, gate2, n_src, n_tgt, eps, pair_pos, pair_d2, pair_tgt, (MT*)maha, fw);
  GICPB_LAUNCHED();
}

void launch_correspondences(const GridView& g, const float4* src, int lo, int hi, const Rigid& T, const RotD& R,
                            float gate2, const double* n_src, const double* n_tgt, double eps, int* pair_pos,
                            float* pair_d2, float4* pair_tgt, void* maha, bool maha_fp32, bool use_prev,
                            const FarWork& fw, cudaStream_t stream) {
  if (hi - lo <= 0) return;
  reset_far(fw, hi - lo, stream);
  if (maha_fp32) {
    if (use_prev)
      launch_corr_t<float, true>(g, src, lo, hi, T, R, gate2, n_src, n_tgt, eps, pair_pos, pair_d2, pair_tgt, maha, fw, stream);
    else
      launch_corr_t<float, false>(g, src, lo, hi, T, R, gate2, n_src, n_tgt, eps, pair_pos, pair_d2, pair_tgt, maha, fw, stream);
  } else {
    if (use_prev)
      launch_corr_t<double, true>(g, src, lo, hi, T, R, gate2, n_src, n_tgt, eps, pair_pos, pair_d2, pair_tgt, maha, fw, stream);
    else
      launch_corr_t<double, false>(g, src, lo, hi, T, R, gate2, n_src, n_tgt, eps, pair_pos, pair_d2, pair_tgt, maha, fw, stream);
  }
}

// near instance: one row per warp; far instance: one row per block
int fitness_partial_rows(int n, int far_blocks) { return (int)nblocks(n, kNnThreads) * (kNnThreads / 32) + far_blocks; }

void launch_fitness(const GridView& g, const float4* src, int lo, int hi, const Rigid& T, double max_range,
                    const int* seed, double* partials, double* out2, const FarWork& fw, cudaStream_t stream) {
  const int n = hi - lo;
  if (n <= 0) {
    GICPB_CUDA(cudaMemsetAsync(out2, 0, 2 * sizeof(double), stream));
    return;
  }
  reset_far(fw, n, stream);
  const unsigned nb = nblocks(n, kNnThreads);
  fitness_kernel<false><<<nb, kNnThreads, 0, stream>>>(g, src, lo, hi, T, max_range, seed, partials, 0, fw);
  GICPB_LAUNCHED();
  const int near_rows = (int)nb * (kNnThreads / 32);
  fitness_kernel<true><<<fw.far_blocks, kNnThreads, 0, stream>>>(g, src, lo, hi, T, max_range, seed, partials, near_rows, fw);
  GICPB_LAUNCHED();
  reduce_partials_kernel<<<1, kReduceThreads, 0, stream>>>(partials, near_rows + fw.far_blocks, 2, out2);
  GICPB_LAUNCHED();
}

void launch_difference(const GridView& g, const unsigned char* raw, int64_t n, int64_t stride, float thr_next,
                       DiffMode mode, unsigned char* mask, unsigned long long* kept, const FarWork& fw,
                       cudaStream_t stream) {
  if (n <= 0) return;
  reset_far(fw, n, stream);
  difference_kernel<false><<<nblocks(n, kNnThreads), kNnThreads, 0, stream>>>(g, raw, n, stride, thr_next, mode, mask,
                                                                              kept, fw);
  GICPB_LAUNCHED();
  difference_kernel<true><<<fw.far_blocks, kNnThreads, 0, stream>>>(g, raw, n, stride, thr_next, mode, mask, kept, fw);
  GICPB_LAUNCHED();
}

void launch_resolution(const GridView& g, double* partials, double* out2, const FarWork& fw, cudaStream_t stream) {
  if (g.n <= 0) {
    GICPB_CUDA(cudaMemsetAsync(out2, 0, 2 * sizeof(double), stream));
    return;
  }
  reset_far(fw, g.n, stream);
  const unsigned nb = nblocks(g.n, kNnThreads);
  resolution_kernel<false><<<nb, kNnThreads, 0, stream>>>(g, partials, 0, fw);
  GICPB_LAUNCHED();
  resolution_kernel<true><<<fw.far_blocks, kNnThreads, 0, stream>>>(g, partials, (int)nb, fw);
  GICPB_LAUNCHED();
  reduce_partials_kernel<<<1, kReduceThreads, 0, stream>>>(partials, (int)nb + fw.far_blocks, 2, out2);
  GICPB_LAUNCHED();
}

void launch_transform(const unsigned char* in, unsigned char* out, int64_t n, int64_t stride, const Rigid& T,
                      cudaStream_t stream) {
  if (n <= 0) return;
  transform_kernel<<<nblocks(n, 256), 256, 0, stream>>>(in, out, n, stride, T);
  GICPB_LAUNCHED();
}

void launch_pack_queries(const unsigned char* raw, int64_t n, int64_t stride, float4* out, cudaStream_t stream) {
  if (n <= 0) return;
  pack_queries_kernel<<<nblocks(n, 256), 256, 0, stream>>>(raw, n, stride, out);
  GICPB_LAUNCHED();
}

}  // namespace gicpb
