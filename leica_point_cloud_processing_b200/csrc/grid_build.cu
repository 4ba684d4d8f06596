// grid_build.cu - builds the brick-grid spatial index of one cloud on the GPU (see common.cuh).
//
// Replaces the FLANN KDTreeSingleIndex builds of pcl::Registration::initCompute / initComputeReciprocal,
// triggered by gicp_.align() at reference src/GICPAlignment.cpp:96, and the pcl::search::KdTree of
// Filter::removeFromCloud (reference src/Filter.cpp:181-184).
//
// Pipeline (all kernels hand-written, no CUB/Thrust):
//   ingest   strided xyz -> float4 (x,y,z,id) + bounding box of the finite points (block reduce + atomics)
//   probe    multi-resolution occupancy bitmaps -> fractal-dimension estimate -> cell size for ~P points/cell
//   keys     key = brick_linear*512 + morton3(cell in brick); non-finite points get the sentinel key
//   sort     stable LSD radix sort of (key, id)            (sort_scan.cu)
//   reorder  gather float4 points into sorted order
//   tables   brick heads allocate pool slots; cell/brick (begin,end) ranges written by run heads / tails
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "engine.hpp"

namespace gicpb {

std::atomic<int64_t> g_launch_count{0};

namespace {

constexpr int kProbeLevels = 7;  // 4, 8, ..., 256 cells along the longest axis
constexpr int kMaxBricks = 1 << 22;

__device__ __forceinline__ unsigned f2ord(float f) {
  unsigned b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
inline float ord2f(unsigned u) {
  unsigned b = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
  float f;
  std::memcpy(&f, &b, 4);
  return f;
}

// scratch layout (uint32): [0..2] min xyz (ordered), [3..5] max xyz (ordered), [6] finite count, [7] slot counter,
// [8] occupied cell counter
__global__ void init_scratch_kernel(unsigned* s) {
  if (threadIdx.x < 3) s[threadIdx.x] = 0xffffffffu;
  else if (threadIdx.x < 6) s[threadIdx.x] = 0u;
  else if (threadIdx.x < 16) s[threadIdx.x] = 0u;
}

__global__ void __launch_bounds__(256) ingest_kernel(const unsigned char* __restrict__ raw, int64_t n, int64_t stride,
                                                      float4* __restrict__ pts, unsigned* __restrict__ scratch) {
  __shared__ unsigned smin[3][8], smax[3][8], scnt[8];
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float x = 0.f, y = 0.f, z = 0.f;
  bool ok = false;
  if (i < n) {
    const float* p = reinterpret_cast<const float*>(raw + i * stride);
    x = p[0];
    y = p[1];
    z = p[2];
    ok = finite3(x, y, z);
    pts[i] = make_float4(x, y, z, __int_as_float((int)i));
  }
  unsigned mn[3] = {ok ? f2ord(x) : 0xffffffffu, ok ? f2ord(y) : 0xffffffffu, ok ? f2ord(z) : 0xffffffffu};
  unsigned mx[3] = {ok ? f2ord(x) : 0u, ok ? f2ord(y) : 0u, ok ? f2ord(z) : 0u};
  unsigned c = ok ? 1u : 0u;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      mn[a] = min(mn[a], __shfl_xor_sync(kFullMask, mn[a], o));
      mx[a] = max(mx[a], __shfl_xor_sync(kFullMask, mx[a], o));
    }
    c += __shfl_xor_sync(kFullMask, c, o);
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) {
    for (int a = 0; a < 3; ++a) {
      smin[a][warp] = mn[a];
      smax[a][warp] = mx[a];
    }
    scnt[warp] = c;
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    unsigned lo = 0xffffffffu, hi = 0u;
    for (int w = 0; w < 8; ++w) {
      lo = min(lo, smin[threadIdx.x][w]);
      hi = max(hi, smax[threadIdx.x][w]);
    }
    atomicMin(&scratch[threadIdx.x], lo);
    atomicMax(&scratch[3 + threadIdx.x], hi);
  }
  if (threadIdx.x == 3) {
    unsigned t = 0;
    for (int w = 0; w < 8; ++w) t += scnt[w];
    if (t) atomicAdd(&scratch[6], t);
  }
}

struct ProbeParams {
  float ox, oy, oz;
  float inv_cell[kProbeLevels];
  int dim[kProbeLevels];            // cells per axis (cubic bitmaps of dim^3 bits)
  unsigned long long word_off[kProbeLevels];
};

// marks the occupied cells of every probe level for the points 0, sub, 2 sub, ... (a uniform subsample is enough
// for a density estimate; the search results do not depend on the cell size)
__global__ void __launch_bounds__(256) probe_kernel(const float4* __restrict__ pts, int64_t n, int sub, ProbeParams pp,
                                                     unsigned* __restrict__ bits) {
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * sub;
  if (i >= n) return;
  const float4 p = pts[i];
  if (!finite3(p.x, p.y, p.z)) return;
#pragma unroll
  for (int l = 0; l < kProbeLevels; ++l) {
    const int d = pp.dim[l];
    const int cx = clampi(__float2int_rd((p.x - pp.ox) * pp.inv_cell[l]), 0, d - 1);
    const int cy = clampi(__float2int_rd((p.y - pp.oy) * pp.inv_cell[l]), 0, d - 1);
    const int cz = clampi(__float2int_rd((p.z - pp.oz) * pp.inv_cell[l]), 0, d - 1);
    const unsigned long long bit = ((unsigned long long)cz * d + cy) * d + cx;
    const unsigned mask = 1u << (bit & 31);
    unsigned* w = bits + pp.word_off[l] + (bit >> 5);
    if (!(*w & mask)) atomicOr(w, mask);
  }
}

__global__ void __launch_bounds__(256) popcount_kernel(const unsigned* __restrict__ bits, ProbeParams pp,
                                                        unsigned long long total_words, unsigned* __restrict__ out) {
  // out[l] += popcount of level l's words
  const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total_words) return;
  int l = 0;
#pragma unroll
  for (int k = 1; k < kProbeLevels; ++k)
    if (i >= pp.word_off[k]) l = k;
  const unsigned c = __popc(bits[i]);
  if (c) atomicAdd(&out[l], c);
}

// key of every point, the occupancy mark of its brick and the digit histograms of all radix passes (RadixSorter::hist):
// one read of the points feeds the sort and the brick table
__global__ void __launch_bounds__(256) keys_kernel(const float4* __restrict__ pts, int64_t n, GridView g, uint32_t sentinel,
                                                    int passes, uint32_t* __restrict__ keys, uint32_t* __restrict__ vals,
                                                    uint32_t* __restrict__ occ, uint32_t* __restrict__ hist) {
  __shared__ uint32_t h[4][256];
  for (int i = threadIdx.x; i < 4 * 256; i += 256) (&h[0][0])[i] = 0u;
  __syncthreads();
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
    const float4 p = pts[i];
    uint32_t key = sentinel;
    if (finite3(p.x, p.y, p.z)) {
      const int cx = clampi(cell_of(p.x, g.ox, g.inv_h), 0, g.nx - 1);
      const int cy = clampi(cell_of(p.y, g.oy, g.inv_h), 0, g.ny - 1);
      const int cz = clampi(cell_of(p.z, g.oz, g.inv_h), 0, g.nz - 1);
      const uint32_t b = (uint32_t)brick_index(g, cx >> kBrickShift, cy >> kBrickShift, cz >> kBrickShift);
      key = b * kBrickCells + local_code(cx & 7, cy & 7, cz & 7);
      occ[b] = 1u;
    }
    keys[i] = key;
    vals[i] = (uint32_t)i;
    for (int p8 = 0; p8 < passes; ++p8) atomicAdd(&h[p8][(key >> (8 * p8)) & 255u], 1u);
  }
  __syncthreads();
  for (int p8 = 0; p8 < passes; ++p8)
    if (h[p8][threadIdx.x]) atomicAdd(&hist[p8 * 256 + threadIdx.x], h[p8][threadIdx.x]);
}

// gather the points into sorted order and record the inverse permutation (original index -> sorted position;
// the tail of vals, i >= n_valid, holds the non-finite points: position -1).  The original index is the point's w.
__global__ void __launch_bounds__(256) reorder_kernel(const float4* __restrict__ pts, const uint32_t* __restrict__ vals,
                                                       int64_t n_valid, int64_t n, float4* __restrict__ sorted,
                                                       int* __restrict__ pos_of) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 p = pts[vals[i]];
  const int oi = __float_as_int(p.w);
  if (i < n_valid) {
    sorted[i] = p;
    pos_of[oi] = (int)i;
  } else {
    pos_of[oi] = -1;
  }
}

// ---- sharded source: the window of brick planes one rank indexes (engine.hpp GridIndex::build, world > 1) ------------------
__device__ __forceinline__ int plane_of(const GridView& g, int axis, const float4& p) {
  const float v = axis == 0 ? p.x : (axis == 1 ? p.y : p.z);
  const float o = axis == 0 ? g.ox : (axis == 1 ? g.oy : g.oz);
  const int dim = axis == 0 ? g.nx : (axis == 1 ? g.ny : g.nz);
  return clampi(cell_of(v, o, g.inv_h), 0, dim - 1) >> kBrickShift;
}

// finite points per brick plane along `axis` (planes <= 8192: one shared-memory histogram per block)
__global__ void __launch_bounds__(256) plane_hist_kernel(const float4* __restrict__ pts, int64_t n, GridView g, int axis,
                                                          int planes, uint32_t* __restrict__ hist) {
  extern __shared__ uint32_t s_hist[];
  for (int i = threadIdx.x; i < planes; i += 256) s_hist[i] = 0u;
  __syncthreads();
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
    const float4 p = pts[i];
    if (finite3(p.x, p.y, p.z)) atomicAdd(&s_hist[plane_of(g, axis, p)], 1u);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < planes; i += 256)
    if (s_hist[i]) atomicAdd(&hist[i], s_hist[i]);
}

__global__ void __launch_bounds__(256) window_flags_kernel(const float4* __restrict__ pts, int64_t n, GridView g, int axis,
                                                            int w_lo, int w_hi, uint32_t* __restrict__ flags) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 p = pts[i];
  bool in = false;
  if (finite3(p.x, p.y, p.z)) {
    const int pl = plane_of(g, axis, p);
    in = pl >= w_lo && pl < w_hi;
  }
  flags[i] = in ? 1u : 0u;
}

// stable: pos = exclusive scan of the flags, so the window keeps the cloud's order (and the index its order inside a cell)
__global__ void __launch_bounds__(256) window_gather_kernel(const float4* __restrict__ pts, const uint32_t* __restrict__ flags,
                                                             const uint32_t* __restrict__ pos, int64_t n,
                                                             float4* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && flags[i]) out[pos[i]] = pts[i];
}

// ---- cloud difference over a group: the input rows whose brick plane (on the subtract's grid) a rank owns -----------------
__global__ void __launch_bounds__(256) route_flags_kernel(const unsigned char* __restrict__ raw, int64_t n, int64_t stride,
                                                           GridView g, int axis, int own_lo, int own_hi,
                                                           uint32_t* __restrict__ flags) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* p = reinterpret_cast<const float*>(raw + i * stride);
  const float4 q = make_float4(p[0], p[1], p[2], 0.f);
  bool in = false;
  if (finite3(q.x, q.y, q.z)) {
    const int pl = plane_of(g, axis, q);
    in = pl >= own_lo && pl < own_hi;
  }
  flags[i] = in ? 1u : 0u;
}

__global__ void __launch_bounds__(256) route_gather_kernel(const unsigned char* __restrict__ raw, int64_t n, int64_t stride,
                                                            const uint32_t* __restrict__ flags,
                                                            const uint32_t* __restrict__ pos, float4* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || !flags[i]) return;
  const float* p = reinterpret_cast<const float*>(raw + i * stride);
  out[pos[i]] = make_float4(p[0], p[1], p[2], __int_as_float((int)i));
}

__global__ void __launch_bounds__(256) scatter_keep_kernel(const float4* __restrict__ rows, const unsigned char* __restrict__ keep,
                                                            int64_t n_rows, unsigned char* __restrict__ full) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n_rows) full[__float_as_int(rows[j].w)] = keep[j];
}

__global__ void __launch_bounds__(256) or_parts_kernel(const unsigned char* __restrict__ parts, int n_parts, int64_t len,
                                                        unsigned char* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= len) return;
  unsigned char v = 0;
  for (int r = 0; r < n_parts; ++r) v |= parts[(int64_t)r * len + i];
  out[i] = v;
}

// brick table from the occupancy marks (rank = exclusive scan of occ): slot = rank of the brick among the occupied bricks
// (so slots ascend with the brick index), -1 for an empty brick; the brick's bit in its superbrick mask and the
// superbrick's bit in its hyperbrick mask; scratch[7] = number of occupied bricks
__global__ void __launch_bounds__(256) brick_table_kernel(const uint32_t* __restrict__ occ, const uint32_t* __restrict__ rank,
                                                           int n_bricks, GridView g, int* __restrict__ brick_slot,
                                                           unsigned long long* __restrict__ sb_mask,
                                                           unsigned long long* __restrict__ hb_mask,
                                                           unsigned* __restrict__ scratch) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n_bricks) return;
  const uint32_t o = occ[b], r = rank[b];
  if (b == n_bricks - 1) scratch[7] = r + o;
  if (!o) {
    brick_slot[b] = -1;
    return;
  }
  brick_slot[b] = (int)r;
  // b = bx * bsx + by * bsy + bz * bsz: peel the axes off from the slowest (g.bo2) to the fastest (g.bo0)
  int v[3];
  {
    const int s[3] = {g.bsx, g.bsy, g.bsz};
    int rest = b;
    v[g.bo2] = rest / s[g.bo2];
    rest -= v[g.bo2] * s[g.bo2];
    v[g.bo1] = rest / s[g.bo1];
    rest -= v[g.bo1] * s[g.bo1];
    v[g.bo0] = rest;
  }
  const int bx = v[0], by = v[1], bz = v[2];
  const int sx = bx >> 2, sy = by >> 2, sz = bz >> 2;
  atomicOr(&sb_mask[((size_t)sz * g.nsy + sy) * g.nsx + sx], 1ull << (((bz & 3) << 4) | ((by & 3) << 2) | (bx & 3)));
  atomicOr(&hb_mask[((size_t)(sz >> 2) * g.nhy + (sy >> 2)) * g.nhx + (sx >> 2)],
           1ull << (((sz & 3) << 4) | ((sy & 3) << 2) | (sx & 3)));
}

// cell_start in two steps.  Heads: the first sorted point of every occupied cell writes its index into the cell's entry
// (all other entries hold 0xffffffff) and the first point of every brick into brick_first[slot].  Fill: one warp per
// brick turns its 512 entries into "index of the first sorted point whose (slot, code) is >= this one" = the minimum of
// the head entries at or after it, or the first point of the next brick (a suffix minimum: head indices ascend with the
// code).  The last brick also writes the terminating entry.
__global__ void __launch_bounds__(256) cell_heads_kernel(const uint32_t* __restrict__ keys, int n_valid,
                                                          const int* __restrict__ brick_slot, uint32_t* __restrict__ cell_start,
                                                          uint32_t* __restrict__ brick_first, unsigned* __restrict__ scratch) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  bool head = false;
  if (i < n_valid) {
    const uint32_t k = keys[i];
    const uint32_t kp = i > 0 ? keys[i - 1] : ~k;
    head = kp != k;
    if (head) {
      const int slot = brick_slot[k >> 9];
      cell_start[(size_t)slot * kBrickCells + (k & 511u)] = (uint32_t)i;
      if (i == 0 || (kp >> 9) != (k >> 9)) brick_first[slot] = (uint32_t)i;
    }
  }
  const unsigned heads = __popc(__ballot_sync(kFullMask, head));
  if ((threadIdx.x & 31) == 0 && heads) atomicAdd(&scratch[8], heads);  // occupied cells (statistics only)
}

__global__ void __launch_bounds__(128) cell_fill_kernel(uint32_t* __restrict__ cell_start, const uint32_t* __restrict__ brick_first,
                                                         int n_slots, int n_valid) {
  const int slot = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (slot >= n_slots) return;
  const uint32_t carry = slot + 1 < n_slots ? brick_first[slot + 1] : (uint32_t)n_valid;
  uint4* cs = reinterpret_cast<uint4*>(cell_start + (size_t)slot * kBrickCells) + 4 * lane;  // entries [16 lane, 16 lane + 16)
  uint4 v[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) v[k] = cs[k];
  uint32_t lm = 0xffffffffu;
#pragma unroll
  for (int k = 0; k < 4; ++k) lm = min(lm, min(min(v[k].x, v[k].y), min(v[k].z, v[k].w)));
  uint32_t incl = lm;  // minimum over the lanes >= this one
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_down_sync(kFullMask, incl, o);
    if (lane + o < 32) incl = min(incl, t);
  }
  uint32_t run = __shfl_down_sync(kFullMask, incl, 1);
  run = lane == 31 ? carry : min(run, carry);
#pragma unroll
  for (int k = 3; k >= 0; --k) {
    run = min(run, v[k].w); v[k].w = run;
    run = min(run, v[k].z); v[k].z = run;
    run = min(run, v[k].y); v[k].y = run;
    run = min(run, v[k].x); v[k].x = run;
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) cs[k] = v[k];
  if (slot == n_slots - 1 && lane == 0) cell_start[(size_t)n_slots * kBrickCells] = (uint32_t)n_valid;
}

// GICPB_BUILD_TRACE=1: CUDA-event time of every phase of a build, printed to stderr (measurement aid, off by default)
struct BuildTrace {
  bool on;
  cudaStream_t stream;
  std::vector<std::pair<const char*, cudaEvent_t>> marks;
  explicit BuildTrace(cudaStream_t s) : stream(s) {
    static const bool enabled = [] {
      const char* e = std::getenv("GICPB_BUILD_TRACE");
      return e && *e && *e != '0';
    }();
    on = enabled;
  }
  void mark(const char* name) {
    if (!on) return;
    cudaEvent_t e;
    cudaEventCreate(&e);
    cudaEventRecord(e, stream);
    marks.emplace_back(name, e);
  }
  void report(int64_t n, double wall_ms) {
    if (!on) return;
    cudaStreamSynchronize(stream);
    std::string line = "[gicpb build trace] n " + std::to_string(n) + " wall " + std::to_string(wall_ms) + " ms:";
    for (size_t i = 1; i < marks.size(); ++i) {
      float ms = 0.f;
      cudaEventElapsedTime(&ms, marks[i - 1].second, marks[i].second);
      char buf[96];
      std::snprintf(buf, sizeof(buf), " %s %.3f", marks[i].first, ms);
      line += buf;
    }
    std::fprintf(stderr, "%s\n", line.c_str());
    for (auto& m : marks) cudaEventDestroy(m.second);
  }
};

inline unsigned blocks_for(int64_t n, int threads) { return (unsigned)((n + threads - 1) / threads); }

// GICPB_SB_PLANE=0 leaves the superbrick slabs out of the view (measurements)
inline bool use_sb_plane() {
  static const bool on = [] {
    const char* e = std::getenv("GICPB_SB_PLANE");
    return !(e && e[0] == '0');
  }();
  return on;
}

}  // namespace

// Oriented slab of every occupied brick (GridView::brick_plane, used by visit_brick): one warp per brick slot.  The
// direction is the eigenvector of the smallest eigenvalue of the covariance of the brick's points (any unit vector would
// be valid; this one makes the slab thin for a sheet); lo / hi are the extremes of plane_dot(n, p) over the brick's
// points, evaluated exactly as the search evaluates it for a query.
__device__ __forceinline__ void jacobi3(double (&a)[9], double (&v)[9], int p, int q) {
  const double apq = a[3 * p + q];
  if (apq == 0.0) return;
  const double theta = (a[3 * q + q] - a[3 * p + p]) / (2.0 * apq);
  const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
  const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
  for (int k = 0; k < 3; ++k) {
    const double akp = a[3 * k + p], akq = a[3 * k + q];
    a[3 * k + p] = c * akp - s * akq;
    a[3 * k + q] = s * akp + c * akq;
  }
  for (int k = 0; k < 3; ++k) {
    const double apk = a[3 * p + k], aqk = a[3 * q + k];
    a[3 * p + k] = c * apk - s * aqk;
    a[3 * q + k] = s * apk + c * aqk;
  }
  for (int k = 0; k < 3; ++k) {
    const double vkp = v[3 * k + p], vkq = v[3 * k + q];
    v[3 * k + p] = c * vkp - s * vkq;
    v[3 * k + q] = s * vkp + c * vkq;
  }
}

__global__ void __launch_bounds__(128) brick_plane_kernel(const float4* __restrict__ pts, const uint32_t* __restrict__ cell_start,
                                                           int n_slots, float* __restrict__ plane) {
  const int slot = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (slot >= n_slots) return;
  const unsigned b = cell_start[(size_t)slot * kBrickCells], e = cell_start[(size_t)(slot + 1) * kBrickCells];
  // moments about the brick's first point (keeps the sums small), in double, fixed order
  const float4 p0 = pts[b];
  double sm[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};  // x y z xx xy xz yy yz zz
  for (unsigned i = b + lane; i < e; i += 32) {
    const float4 p = pts[i];
    const double x = (double)p.x - (double)p0.x, y = (double)p.y - (double)p0.y, z = (double)p.z - (double)p0.z;
    sm[0] += x; sm[1] += y; sm[2] += z;
    sm[3] += x * x; sm[4] += x * y; sm[5] += x * z; sm[6] += y * y; sm[7] += y * z; sm[8] += z * z;
  }
#pragma unroll
  for (int k = 0; k < 9; ++k) sm[k] = warp_sum(sm[k]);
  const double m = (double)(e - b);
  const double mx = sm[0] / m, my = sm[1] / m, mz = sm[2] / m;
  double a[9], v[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
  a[0] = sm[3] / m - mx * mx; a[1] = sm[4] / m - mx * my; a[2] = sm[5] / m - mx * mz;
  a[4] = sm[6] / m - my * my; a[5] = sm[7] / m - my * mz; a[8] = sm[8] / m - mz * mz;
  a[3] = a[1]; a[6] = a[2]; a[7] = a[5];
  for (int sweep = 0; sweep < 24; ++sweep) {  // every lane runs the same arithmetic on the same sums
    const double off = fabs(a[1]) + fabs(a[2]) + fabs(a[5]);
    if (off == 0.0 || off < 1e-20 * (fabs(a[0]) + fabs(a[4]) + fabs(a[8]))) break;
    jacobi3(a, v, 0, 1);
    jacobi3(a, v, 0, 2);
    jacobi3(a, v, 1, 2);
  }
  int best = 0;
  if (fabs(a[4]) < fabs(a[0])) best = 1;
  if (fabs(a[8]) < fabs(a[4 * best])) best = 2;
  float nx = (float)v[best], ny = (float)v[3 + best], nz = (float)v[6 + best];
  if (!(fabsf(nx) + fabsf(ny) + fabsf(nz) > 0.5f)) { nx = 0.f; ny = 0.f; nz = 1.f; }  // degenerate input: any direction will do
  float lo = __int_as_float(0x7f800000), hi = __int_as_float(0xff800000);
  for (unsigned i = b + lane; i < e; i += 32) {
    const float4 p = pts[i];
    const float d = plane_dot(nx, ny, nz, p.x, p.y, p.z);
    lo = fminf(lo, d);
    hi = fmaxf(hi, d);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    lo = fminf(lo, __shfl_xor_sync(kFullMask, lo, o));
    hi = fmaxf(hi, __shfl_xor_sync(kFullMask, hi, o));
  }
  if (lane == 0) {
    float* out = plane + 5 * (size_t)slot;
    out[0] = nx; out[1] = ny; out[2] = nz; out[3] = lo; out[4] = hi;
  }
}

// The same slab for every occupied SUPERBRICK (GridView::sb_plane, used by visit_superbrick): one block per superbrick
// walks the points of its occupied bricks twice (moments, then the extremes of plane_dot along the PCA normal).  Empty
// superbricks get an empty slab; they are never looked at.
constexpr int kSbThreads = 512;
__global__ void __launch_bounds__(kSbThreads) sb_plane_kernel(GridView g, const float4* __restrict__ pts, const uint32_t* __restrict__ cell_start,
                                                               const int* __restrict__ brick_slot, const unsigned long long* __restrict__ sb_mask,
                                                               float* __restrict__ plane) {
  constexpr int kWarps = kSbThreads / 32;
  __shared__ unsigned s_b[64], s_pre[65];
  __shared__ double s_sum[kWarps][9];
  __shared__ float s_lo[kWarps], s_hi[kWarps];
  const int sb = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned long long occ = sb_mask[sb];
  float* out = plane + 5 * (size_t)sb;
  if (!occ) {
    if (threadIdx.x == 0) { out[0] = 0.f; out[1] = 0.f; out[2] = 1.f; out[3] = __int_as_float(0x7f800000); out[4] = __int_as_float(0xff800000); }
    return;
  }
  // the point ranges of the occupied bricks, all looked up at once, then ONE flat loop over the superbrick's points
  if (threadIdx.x < 64) {
    unsigned b = 0, e = 0;
    if ((occ >> threadIdx.x) & 1ull) {
      const int sx = sb % g.nsx, sy = (sb / g.nsx) % g.nsy, sz = sb / (g.nsx * g.nsy);
      const int bit = threadIdx.x;
      const int bx = (sx << 2) + (bit & 3), by = (sy << 2) + ((bit >> 2) & 3), bz = (sz << 2) + (bit >> 4);
      const int slot = brick_slot[brick_index(g, bx, by, bz)];
      b = cell_start[(size_t)slot * kBrickCells];
      e = cell_start[(size_t)(slot + 1) * kBrickCells];
    }
    s_b[threadIdx.x] = b;
    // inclusive scan of the 64 lengths over two warps
    unsigned incl = e - b;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned v = __shfl_up_sync(kFullMask, incl, o);
      if (lane >= o) incl += v;
    }
    s_pre[threadIdx.x + 1] = incl;
  }
  if (threadIdx.x == 0) s_pre[0] = 0u;
  __syncthreads();
  const unsigned first_half = s_pre[32];
  __syncthreads();
  if (threadIdx.x >= 32 && threadIdx.x < 64) s_pre[threadIdx.x + 1] += first_half;
  __syncthreads();
  const unsigned total = s_pre[64];
  auto point_at = [&](unsigned f) {  // f-th point of the superbrick: the last brick whose prefix is <= f
    int j = 0;
#pragma unroll
    for (int step = 32; step > 0; step >>= 1)
      if (s_pre[j + step] <= f) j += step;
    return s_b[j] + (f - s_pre[j]);
  };
  const float4 p0 = pts[point_at(0u)];  // moments about the first point (keeps the sums small), in double
  double sm[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};  // x y z xx xy xz yy yz zz
  for (unsigned f = threadIdx.x; f < total; f += kSbThreads) {
    const float4 p = pts[point_at(f)];
    const double x = (double)p.x - (double)p0.x, y = (double)p.y - (double)p0.y, z = (double)p.z - (double)p0.z;
    sm[0] += x; sm[1] += y; sm[2] += z;
    sm[3] += x * x; sm[4] += x * y; sm[5] += x * z; sm[6] += y * y; sm[7] += y * z; sm[8] += z * z;
  }
#pragma unroll
  for (int k = 0; k < 9; ++k) {
    sm[k] = warp_sum(sm[k]);
    if (lane == 0) s_sum[warp][k] = sm[k];
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 9; ++k) {  // the same value in every thread
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) t += s_sum[w][k];
    sm[k] = t;
  }
  const double m = (double)total;
  const double mx = sm[0] / m, my = sm[1] / m, mz = sm[2] / m;
  double a[9], v[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
  a[0] = sm[3] / m - mx * mx; a[1] = sm[4] / m - mx * my; a[2] = sm[5] / m - mx * mz;
  a[4] = sm[6] / m - my * my; a[5] = sm[7] / m - my * mz; a[8] = sm[8] / m - mz * mz;
  a[3] = a[1]; a[6] = a[2]; a[7] = a[5];
  for (int sweep = 0; sweep < 24; ++sweep) {
    const double off = fabs(a[1]) + fabs(a[2]) + fabs(a[5]);
    if (off == 0.0 || off < 1e-20 * (fabs(a[0]) + fabs(a[4]) + fabs(a[8]))) break;
    jacobi3(a, v, 0, 1);
    jacobi3(a, v, 0, 2);
    jacobi3(a, v, 1, 2);
  }
  int best = 0;
  if (fabs(a[4]) < fabs(a[0])) best = 1;
  if (fabs(a[8]) < fabs(a[4 * best])) best = 2;
  float nx = (float)v[best], ny = (float)v[3 + best], nz = (float)v[6 + best];
  if (!(fabsf(nx) + fabsf(ny) + fabsf(nz) > 0.5f)) { nx = 0.f; ny = 0.f; nz = 1.f; }
  float lo = __int_as_float(0x7f800000), hi = __int_as_float(0xff800000);
  for (unsigned f = threadIdx.x; f < total; f += kSbThreads) {
    const float4 p = pts[point_at(f)];
    const float d = plane_dot(nx, ny, nz, p.x, p.y, p.z);
    lo = fminf(lo, d);
    hi = fmaxf(hi, d);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    lo = fminf(lo, __shfl_xor_sync(kFullMask, lo, o));
    hi = fmaxf(hi, __shfl_xor_sync(kFullMask, hi, o));
  }
  if (lane == 0) { s_lo[warp] = lo; s_hi[warp] = hi; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < kWarps; ++w) { lo = fminf(lo, s_lo[w]); hi = fmaxf(hi, s_hi[w]); }
    out[0] = nx; out[1] = ny; out[2] = nz;
    out[3] = lo;
    out[4] = hi;
  }
}

// Ask for the largest shared-memory carve-out on every index-build kernel so that their blocks can share an SM with the
// kNN kernel (which needs it) when both run on different streams (gicpb_set_clouds).
void prefer_shared_carveout_grid() {
  const int pct = 100;
  cudaFuncSetAttribute(init_scratch_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
  cudaFuncSetAttribute(ingest_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
  cudaFuncSetAttribute(probe_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
  cudaFuncSetAttribute(popcount_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
  cudaFuncSetAttribute(keys_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
  cudaFuncSetAttribute(reorder_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
  cudaFuncSetAttribute(plane_hist_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
  cudaFuncSetAttribute(window_flags_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
  cudaFuncSetAttribute(window_gather_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
  cudaFuncSetAttribute(brick_table_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
  cudaFuncSetAttribute(cell_heads_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
  cudaFuncSetAttribute(cell_fill_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
  cudaFuncSetAttribute(brick_plane_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
  cudaFuncSetAttribute(sb_plane_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
  (void)cudaGetLastError();
}

// brick planes (8 cells each) indexed either side of a rank's own planes; GICPB_HALO_PLANES=0 makes the kNN check fail at
// every window edge (a test of the fall-back to the whole cloud)
static int halo_planes() {
  static const int v = [] {
    const char* e = std::getenv("GICPB_HALO_PLANES");
    return e && *e ? std::max(0, std::atoi(e)) : 1;
  }();
  return v;
}

// Halo of the subtract cloud's window (halo_m = the search radius sqrt(thr_next) of a difference).  A subtract point s that can
// hit a query q (float d2 < thr_next) has |s_a - q_a| <= halo_m along the split axis, up to the rounding of the float
// distance, which the grid's margin covers (it is the slack of every box bound of the searches).  cell_of is monotone in the
// coordinate, and floor() plus the rounding of (v - o) * inv_h move a cell index by less than one cell, so
// cell(s) < cell(q) + (halo_m + margin) / h + 1.  A query the rank owns has cell(q) < 8 own_hi, hence cell(s) < 8 (own_hi + H)
// - plane(s) < own_hi + H, inside the window - as soon as 8 h H >= halo_m + margin + h; the same holds below own_lo.  A query
// outside the grid is clamped to an end plane, and the points near it lie in the first (last) planes, in that window too.
static int difference_halo(double halo_m, double h, double margin, int planes) {
  const double H = std::ceil((halo_m + margin + h) / (8.0 * h));
  return H < (double)planes ? std::max(1, (int)H) : planes;  // INFINITY: the whole cloud
}

void GridIndex::build(const void* raw, int64_t n, int64_t stride_bytes, bool on_device, float cell_size,
                      float points_per_cell, cudaStream_t stream, HostStager* stager, int rank, int world, double halo_m) {
  const auto t_begin = std::chrono::steady_clock::now();
  BuildTrace trace(stream);
  trace.mark("begin");
  ready_ = false;
  if (n <= 0) throw ArgError("cloud is empty");
  if (n > 0x7fffff00LL) throw ArgError("cloud has more than 2^31 points");
  if (stride_bytes < 12 || (stride_bytes % 4) != 0) throw ArgError("stride must be a multiple of 4 and >= 12");
  if (raw == nullptr) throw ArgError("null cloud pointer");
  info_ = Info{};
  info_.n_points = n;

  // ---- ingest ---------------------------------------------------------------------------------------
  const unsigned char* d_raw = static_cast<const unsigned char*>(raw);
  if (!on_device) {
    raw_.reserve((size_t)n * stride_bytes);
    if (stager && HostStager::wants(raw, n, stride_bytes)) {  // pageable memory: packed xyz rows through pinned chunks
      stager->upload(raw_.get(), static_cast<const unsigned char*>(raw), n, stride_bytes, 12, stream);
      stride_bytes = 12;
    } else {
      GICPB_CUDA(cudaMemcpyAsync(raw_.get(), raw, (size_t)(n - 1) * stride_bytes + 12, cudaMemcpyHostToDevice, stream));
    }
    d_raw = raw_.get();
  }
  trace.mark("upload");
  pts_unsorted_.reserve(n);
  pts_sorted_.reserve(n);
  scratch_.reserve(64);
  init_scratch_kernel<<<1, 32, 0, stream>>>(scratch_.get());
  GICPB_LAUNCHED();
  ingest_kernel<<<blocks_for(n, 256), 256, 0, stream>>>(d_raw, n, stride_bytes, pts_unsorted_.get(), scratch_.get());
  GICPB_LAUNCHED();
  if (!h_pin_) GICPB_CUDA(cudaHostAlloc(&h_pin_, 32 * sizeof(unsigned), cudaHostAllocDefault));  // read-backs: no staging copy
  unsigned* hs = h_pin_;                  // 16 words of scratch
  unsigned* occ = h_pin_ + 16;            // kProbeLevels words of the density probe
  constexpr size_t kHsBytes = 16 * sizeof(unsigned);
  GICPB_CUDA(cudaMemcpyAsync(hs, scratch_.get(), kHsBytes, cudaMemcpyDeviceToHost, stream));
  trace.mark("ingest");
  GICPB_CUDA(cudaStreamSynchronize(stream));
  const int64_t n_valid = hs[6];
  info_.n_indexed = n_valid;
  if (n_valid == 0) throw ArgError("cloud has no finite point");
  float bmin[3], bmax[3], ext[3];
  for (int a = 0; a < 3; ++a) {
    bmin[a] = ord2f(hs[a]);
    bmax[a] = ord2f(hs[3 + a]);
    ext[a] = bmax[a] - bmin[a];
    info_.bbox_min[a] = bmin[a];
    info_.bbox_max[a] = bmax[a];
  }
  const float lmax = std::max(ext[0], std::max(ext[1], ext[2]));
  float max_abs = 0.f;
  for (int a = 0; a < 3; ++a) max_abs = std::max(max_abs, std::max(std::fabs(bmin[a]), std::fabs(bmax[a])));

  // ---- cell size ------------------------------------------------------------------------------------
  float h = cell_size;
  if (!(h > 0.f)) {
    if (!(lmax > 0.f)) {
      h = 1.0f;
    } else {
      ProbeParams pp{};
      pp.ox = bmin[0];
      pp.oy = bmin[1];
      pp.oz = bmin[2];
      unsigned long long words = 0;
      for (int l = 0; l < kProbeLevels; ++l) {
        const int d = 4 << l;
        pp.dim[l] = d;
        pp.inv_cell[l] = (float)d / (lmax * 1.0001f);
        pp.word_off[l] = words;
        words += ((unsigned long long)d * d * d + 31) / 32;
      }
      occ_bits_.reserve(words + 16);
      GICPB_CUDA(cudaMemsetAsync(occ_bits_.get(), 0, (words + 16) * sizeof(uint32_t), stream));
      // ~64 k samples are plenty for a density estimate (the finest well-populated level is found from them)
      const int sub = (int)std::max<int64_t>(1, std::min<int64_t>(64, n / 65536));
      probe_kernel<<<blocks_for((n + sub - 1) / sub, 256), 256, 0, stream>>>(pts_unsorted_.get(), n, sub, pp, occ_bits_.get());
      GICPB_LAUNCHED();
      popcount_kernel<<<blocks_for((int64_t)words, 256), 256, 0, stream>>>(occ_bits_.get(), pp, words,
                                                                           occ_bits_.get() + words);
      GICPB_LAUNCHED();
      static_assert(kProbeLevels <= 16, "probe read-back buffer");
      GICPB_CUDA(cudaMemcpyAsync(occ, occ_bits_.get() + words, kProbeLevels * sizeof(unsigned), cudaMemcpyDeviceToHost, stream));
      GICPB_CUDA(cudaStreamSynchronize(stream));
      const double N = (double)n_valid / sub;  // sampled points (the non-finite fraction is taken as uniform)
      const double tau = (points_per_cell > 0.f ? points_per_cell : 6.0) / sub;
      int ls = -1;  // finest level whose cells are still well populated
      for (int l = 0; l < kProbeLevels; ++l)
        if (occ[l] > 0 && N / occ[l] >= 8.0) ls = l;
      if (ls < 0) {
        h = (float)(lmax / std::max(1.0, std::cbrt(N / tau)));
      } else {
        double d = 2.0;
        if (ls >= 1 && occ[ls - 1] > 0) d = std::log2((double)occ[ls] / (double)occ[ls - 1]);
        d = std::min(3.0, std::max(1.0, d));
        const double H = lmax / (double)(4 << ls);
        const double ratio = std::min(1.0, tau * occ[ls] / N);
        h = (float)(H * std::pow(ratio, 1.0 / d));
      }
    }
  }
  if (!(h > 0.f) || !std::isfinite(h)) h = 1.0f;
  h = std::max(h, lmax / 60000.0f);
  int dims[3], bd[3];
  for (;;) {
    int64_t nb = 1;
    for (int a = 0; a < 3; ++a) {
      dims[a] = (int)std::floor(ext[a] / h) + 1;
      bd[a] = (dims[a] + 7) / 8;
      dims[a] = bd[a] * 8;
      nb *= bd[a];
    }
    if (nb <= kMaxBricks) break;
    h *= 1.2f;
  }
  const int64_t n_bricks = (int64_t)bd[0] * bd[1] * bd[2];
  const int maxdim = std::max(dims[0], std::max(dims[1], dims[2]));

  GridView g{};
  g.ox = bmin[0];
  g.oy = bmin[1];
  g.oz = bmin[2];
  g.h = h;
  g.inv_h = 1.0f / h;
  g.margin = h * (0.002f + 5e-7f * (float)maxdim) + 4e-6f * max_abs;
  g.nx = dims[0];
  g.ny = dims[1];
  g.nz = dims[2];
  g.nbx = bd[0];
  g.nby = bd[1];
  g.nbz = bd[2];
  g.n = (int)n_valid;

  g.nsx = (bd[0] + 3) / 4;
  g.nsy = (bd[1] + 3) / 4;
  g.nsz = (bd[2] + 3) / 4;
  g.nhx = (g.nsx + 3) / 4;
  g.nhy = (g.nsy + 3) / 4;
  g.nhz = (g.nsz + 3) / 4;
  g.bsx = 1;
  g.bsy = bd[0];
  g.bsz = bd[0] * bd[1];
  g.bo0 = 0;
  g.bo1 = 1;
  g.bo2 = 2;
  trace.mark("probe");

  // ---- sharded source: brick planes along the longest axis, numbered slowest, and this rank's window of them ---------
  win_ = Window{};
  win_.n_finite = n_valid;
  n_all_ = n;
  if (world > 1) {
    // The planes are cut across the SECOND longest axis when it has enough of them, so that every rank owns a strip that
    // runs the whole length of the cloud: the cost of a first correspondence pass grows with the distance from the centre
    // of the misalignment, and slabs across the longest axis would give the ranks at the two ends all the expensive
    // queries (measured on 8 GPUs, 8 M / 8 M: correspondence kernels of the slowest rank 4.5 ms against 2.9 ms).
    int order[3] = {0, 1, 2};
    std::sort(order, order + 3, [&](int a, int b) { return bd[a] != bd[b] ? bd[a] > bd[b] : a < b; });
    auto usable = [&](int a) { return bd[a] >= 4 * world && bd[a] <= 8192; };
    const int axis = usable(order[1]) ? order[1] : order[0];
    const int planes = bd[axis];
    if (usable(axis) && n_valid >= 1024 * (int64_t)world) {
      const int o0 = axis == 0 ? 1 : 0, o1 = axis == 2 ? 1 : 2;  // the other two axes, in x < y < z order
      int strides[3];
      strides[o0] = 1;
      strides[o1] = bd[o0];
      strides[axis] = bd[o0] * bd[o1];
      g.bsx = strides[0];
      g.bsy = strides[1];
      g.bsz = strides[2];
      g.bo0 = o0;
      g.bo1 = o1;
      g.bo2 = axis;
      plane_hist_.reserve((size_t)planes);
      GICPB_CUDA(cudaMemsetAsync(plane_hist_.get(), 0, (size_t)planes * sizeof(uint32_t), stream));
      plane_hist_kernel<<<std::min<unsigned>(blocks_for(n, 256 * 8), 148u * 4u), 256, (size_t)planes * sizeof(uint32_t), stream>>>(
          pts_unsorted_.get(), n, g, axis, planes, plane_hist_.get());
      GICPB_LAUNCHED();
      std::vector<uint32_t> hist((size_t)planes);
      GICPB_CUDA(cudaMemcpyAsync(hist.data(), plane_hist_.get(), (size_t)planes * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
      GICPB_CUDA(cudaStreamSynchronize(stream));
      win_.plane_prefix.assign((size_t)planes + 1, 0u);
      for (int p = 0; p < planes; ++p) win_.plane_prefix[(size_t)p + 1] = win_.plane_prefix[(size_t)p] + hist[(size_t)p];
      // rank r owns the planes [cut(r), cut(r + 1)): cut(r) = first plane with at least r / world of the points before it
      auto cut = [&](int r) {
        if (r <= 0) return 0;
        if (r >= world) return planes;
        const uint64_t want = (uint64_t)n_valid * (uint64_t)r / (uint64_t)world;
        int p = 0;
        while (p < planes && win_.plane_prefix[(size_t)p] < want) ++p;
        return p;
      };
      bool every_rank_owns_points = true;
      for (int r = 0; r < world; ++r)
        if (win_.plane_prefix[(size_t)cut(r + 1)] == win_.plane_prefix[(size_t)cut(r)]) every_rank_owns_points = false;
      if (every_rank_owns_points) {
        win_.active = true;
        win_.rank = rank;
        win_.world = world;
        win_.axis = axis;
        win_.planes = planes;
        win_.own_lo = cut(rank);
        win_.own_hi = cut(rank + 1);
        const int halo = halo_m >= 0 ? difference_halo(halo_m, g.h, g.margin, planes) : halo_planes();
        set_window(std::max(0, win_.own_lo - halo), std::min(planes, win_.own_hi + halo));
      } else {  // degenerate split: index everything, shards by index range (the default numbering again)
        g.bsx = 1; g.bsy = bd[0]; g.bsz = bd[0] * bd[1];
        g.bo0 = 0; g.bo1 = 1; g.bo2 = 2;
      }
    }
    trace.mark("window");
  }
  geom_ = g;
  int64_t n_local = 0;
  const float4* pts_in = pts_unsorted_.get();
  int64_t n_in = n, n_valid_in = n_valid;
  if (windowed()) {
    pts_in = window_points(stream, &n_local);
    n_in = n_valid_in = n_local;
  }
  index_points(pts_in, n_in, n_valid_in, geom_, stream, &trace);
  info_.ms_build =
      std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
  trace.report(n, info_.ms_build);
}

void GridIndex::set_window(int w_lo, int w_hi) {
  win_.w_lo = w_lo;
  win_.w_hi = w_hi;
  win_.shard_lo = (int)(win_.plane_prefix[(size_t)win_.own_lo] - win_.plane_prefix[(size_t)w_lo]);
  win_.shard_hi = (int)(win_.plane_prefix[(size_t)win_.own_hi] - win_.plane_prefix[(size_t)w_lo]);
}

GridIndex::KnnWindow GridIndex::knn_window() const {
  KnnWindow w;
  if (!windowed()) return w;
  const float o = win_.axis == 0 ? geom_.ox : (win_.axis == 1 ? geom_.oy : geom_.oz);
  const float hb = geom_.h * 8.0f;
  w.axis = win_.axis;
  w.lo = win_.w_lo > 0 ? o + (float)win_.w_lo * hb : -INFINITY;
  w.hi = win_.w_hi < win_.planes ? o + (float)win_.w_hi * hb : INFINITY;
  return w;
}

// the points of the window's planes, in the cloud's order
const float4* GridIndex::window_points(cudaStream_t stream, int64_t* n_local) {
  const int64_t n = n_all_;
  *n_local = (int64_t)(win_.plane_prefix[(size_t)win_.w_hi] - win_.plane_prefix[(size_t)win_.w_lo]);
  win_flags_.reserve((size_t)n);
  win_pos_.reserve((size_t)n);
  scan_tmp_.reserve(scan_tmp_entries(n));
  pts_local_.reserve((size_t)std::max<int64_t>(*n_local, 1));
  window_flags_kernel<<<blocks_for(n, 256), 256, 0, stream>>>(pts_unsorted_.get(), n, geom_, win_.axis, win_.w_lo, win_.w_hi,
                                                             win_flags_.get());
  GICPB_LAUNCHED();
  exclusive_scan_u32(win_flags_.get(), win_pos_.get(), n, scan_tmp_.get(), stream);
  window_gather_kernel<<<blocks_for(n, 256), 256, 0, stream>>>(pts_unsorted_.get(), win_flags_.get(), win_pos_.get(), n,
                                                              pts_local_.get());
  GICPB_LAUNCHED();
  return pts_local_.get();
}

int64_t GridIndex::owned_queries(const unsigned char* raw, int64_t n, int64_t stride, float4* out, uint32_t* flags,
                                 uint32_t* pos, uint32_t* tmp, cudaStream_t stream) const {
  // flags[n] = 0: the exclusive scan leaves the number of owned rows in pos[n]
  GICPB_CUDA(cudaMemsetAsync(flags + n, 0, sizeof(uint32_t), stream));
  route_flags_kernel<<<blocks_for(n, 256), 256, 0, stream>>>(raw, n, stride, geom_, win_.axis, win_.own_lo, win_.own_hi, flags);
  GICPB_LAUNCHED();
  exclusive_scan_u32(flags, pos, n + 1, tmp, stream);
  route_gather_kernel<<<blocks_for(n, 256), 256, 0, stream>>>(raw, n, stride, flags, pos, out);
  GICPB_LAUNCHED();
  uint32_t owned = 0;
  GICPB_CUDA(cudaMemcpyAsync(&owned, pos + n, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
  GICPB_CUDA(cudaStreamSynchronize(stream));
  return (int64_t)owned;
}

void scatter_keep(const float4* rows, const unsigned char* keep, int64_t n_rows, unsigned char* full, cudaStream_t stream) {
  if (n_rows <= 0) return;
  scatter_keep_kernel<<<blocks_for(n_rows, 256), 256, 0, stream>>>(rows, keep, n_rows, full);
  GICPB_LAUNCHED();
}

void or_parts(const unsigned char* parts, int n_parts, int64_t len, unsigned char* out, cudaStream_t stream) {
  if (len <= 0) return;
  or_parts_kernel<<<blocks_for(len, 256), 256, 0, stream>>>(parts, n_parts, len, out);
  GICPB_LAUNCHED();
}

void GridIndex::widen(cudaStream_t stream) {
  if (!windowed()) return;
  ready_ = false;
  set_window(0, win_.planes);
  index_points(pts_unsorted_.get(), n_all_, win_.n_finite, geom_, stream, nullptr);
}

// keys (+ brick occupancy + digit histograms) -> brick table -> sort -> reorder -> cell table -> brick slabs, for the points
// `pts` (w = original index; the first n_valid in the sort order are the finite ones) on the grid `geom`
void GridIndex::index_points(const float4* pts, int64_t n, int64_t n_valid, const GridView& geom, cudaStream_t stream,
                             void* trace_ptr) {
  BuildTrace none(stream);
  none.on = false;
  BuildTrace& trace = trace_ptr ? *static_cast<BuildTrace*>(trace_ptr) : none;
  GridView g = geom;
  g.n = (int)n_valid;
  const int64_t n_bricks = (int64_t)g.nbx * g.nby * g.nbz;
  const size_t n_sb = (size_t)g.nsx * g.nsy * g.nsz, n_hb = (size_t)g.nhx * g.nhy * g.nhz;
  unsigned* hs = h_pin_;
  constexpr size_t kHsBytes = 16 * sizeof(unsigned);
  pts_sorted_.reserve((size_t)std::max<int64_t>(n, 1));
  keys_a_.reserve(n);
  keys_b_.reserve(n);
  vals_a_.reserve(n);
  vals_b_.reserve(n);
  occ_.reserve(n_bricks);
  brick_rank_.reserve(n_bricks);
  scan_tmp_.reserve(scan_tmp_entries(std::max<int64_t>(n_bricks, n_all_)));
  brick_slot_.reserve(n_bricks);
  sb_mask_.reserve(n_sb);
  hb_mask_.reserve(n_hb);
  const uint32_t sentinel = (uint32_t)(n_bricks * kBrickCells);
  int key_bits = 1;
  while ((1ull << key_bits) <= (unsigned long long)sentinel) ++key_bits;
  sorter_.prepare(n, stream);
  GICPB_CUDA(cudaMemsetAsync(occ_.get(), 0, (size_t)n_bricks * sizeof(uint32_t), stream));
  GICPB_CUDA(cudaMemsetAsync(sb_mask_.get(), 0, n_sb * sizeof(unsigned long long), stream));
  GICPB_CUDA(cudaMemsetAsync(hb_mask_.get(), 0, n_hb * sizeof(unsigned long long), stream));
  GICPB_CUDA(cudaMemsetAsync(scratch_.get() + 7, 0, 2 * sizeof(unsigned), stream));  // slot and cell counters
  keys_kernel<<<std::min<unsigned>(blocks_for(n, 256 * 4), 148u * 4u), 256, 0, stream>>>(
      pts, n, g, sentinel, (key_bits + 7) / 8, keys_a_.get(), vals_a_.get(), occ_.get(), sorter_.hist());
  GICPB_LAUNCHED();
  trace.mark("keys");
  exclusive_scan_u32(occ_.get(), brick_rank_.get(), n_bricks, scan_tmp_.get(), stream);
  brick_table_kernel<<<blocks_for(n_bricks, 256), 256, 0, stream>>>(occ_.get(), brick_rank_.get(), (int)n_bricks, g,
                                                                    brick_slot_.get(), sb_mask_.get(), hb_mask_.get(),
                                                                    scratch_.get());
  GICPB_LAUNCHED();
  // the number of occupied bricks is read back while the sort runs
  if (!ev_slots_) GICPB_CUDA(cudaEventCreateWithFlags(&ev_slots_, cudaEventDisableTiming));
  GICPB_CUDA(cudaMemcpyAsync(hs, scratch_.get(), kHsBytes, cudaMemcpyDeviceToHost, stream));
  GICPB_CUDA(cudaEventRecord(ev_slots_, stream));
  trace.mark("bricks");
  const bool in_b = sorter_.sort(keys_a_.get(), vals_a_.get(), keys_b_.get(), vals_b_.get(), n, key_bits, true, stream);
  const uint32_t* skeys = in_b ? keys_b_.get() : keys_a_.get();
  const uint32_t* svals = in_b ? vals_b_.get() : vals_a_.get();
  trace.mark("sort");
  pos_of_.reserve((size_t)n_all_);
  if (n < n_all_)  // a window: the points outside it have no position
    GICPB_CUDA(cudaMemsetAsync(pos_of_.get(), 0xff, (size_t)n_all_ * sizeof(int), stream));
  reorder_kernel<<<blocks_for(n, 256), 256, 0, stream>>>(pts, svals, n_valid, n, pts_sorted_.get(), pos_of_.get());
  GICPB_LAUNCHED();

  trace.mark("reorder");
  // ---- cell table -----------------------------------------------------------------------------------------
  GICPB_CUDA(cudaEventSynchronize(ev_slots_));
  const int64_t n_slots = hs[7];
  cell_start_.reserve((size_t)n_slots * kBrickCells + 4);
  brick_first_.reserve((size_t)n_slots + 1);
  GICPB_CUDA(cudaMemsetAsync(cell_start_.get(), 0xff, ((size_t)n_slots * kBrickCells + 1) * sizeof(uint32_t), stream));
  cell_heads_kernel<<<blocks_for(n_valid, 256), 256, 0, stream>>>(skeys, (int)n_valid, brick_slot_.get(), cell_start_.get(),
                                                                   brick_first_.get(), scratch_.get());
  GICPB_LAUNCHED();
  cell_fill_kernel<<<blocks_for(n_slots * 32, 128), 128, 0, stream>>>(cell_start_.get(), brick_first_.get(), (int)n_slots,
                                                                      (int)n_valid);
  GICPB_LAUNCHED();
  trace.mark("cells");
  brick_plane_.reserve((size_t)n_slots * 5);
  brick_plane_kernel<<<blocks_for(n_slots * 32, 128), 128, 0, stream>>>(pts_sorted_.get(), cell_start_.get(), (int)n_slots,
                                                                        brick_plane_.get());
  GICPB_LAUNCHED();
  if (far_queries_ && use_sb_plane()) {
    sb_plane_.reserve(n_sb * 5);
    GridView gv = g;  // the kernel needs the geometry and the brick numbering only
    sb_plane_kernel<<<(unsigned)n_sb, kSbThreads, 0, stream>>>(gv, pts_sorted_.get(), cell_start_.get(), brick_slot_.get(), sb_mask_.get(),
                                                       sb_plane_.get());
    GICPB_LAUNCHED();
  }
  trace.mark("plane");
  GICPB_CUDA(cudaMemcpyAsync(hs, scratch_.get(), kHsBytes, cudaMemcpyDeviceToHost, stream));
  GICPB_CUDA(cudaStreamSynchronize(stream));

  g.pts = pts_sorted_.get();
  g.brick_plane = brick_plane_.get();
  g.sb_plane = (far_queries_ && use_sb_plane()) ? sb_plane_.get() : nullptr;
  g.brick_slot = brick_slot_.get();
  g.cell_start = cell_start_.get();
  g.pos_of = pos_of_.get();
  g.sb_mask = sb_mask_.get();
  g.hb_mask = hb_mask_.get();
  view_ = g;
  info_.n_indexed = n_valid;
  info_.cell_size = g.h;
  info_.dims[0] = g.nx;
  info_.dims[1] = g.ny;
  info_.dims[2] = g.nz;
  info_.n_bricks_occupied = n_slots;
  info_.n_cells_occupied = hs[8];
  ready_ = true;
}

}  // namespace gicpb
