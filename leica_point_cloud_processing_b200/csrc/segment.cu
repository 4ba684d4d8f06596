// segment.cu - the two callers either side of the registration path (SURVEY section 8f rows 1 and 3):
//
//   Euclidean clustering   FODDetector::clusterPossibleFODs (reference src/FODDetector.cpp:45-58) ->
//                          pcl::EuclideanClusterExtraction::extract: the clusters are the connected components of
//                          the graph that joins two points when their squared distance is < tolerance^2 (FLANN
//                          radius search, strict), of size in [min, max].  Here: the brick grid answers the radius
//                          queries and a lock-free union-find (atomicMin on the parent array) joins the points;
//                          which point reaches which first does not matter for a connected component.
//   voxel-grid downsample  Filter::downsampleCloud (reference src/Filter.cpp:91-105) -> pcl::VoxelGrid::applyFilter:
//                          voxel index per point exactly as PCL computes it in float, stable radix sort by voxel
//                          (sort_scan.cu), one centroid per occupied voxel (float sums in sorted order, rgb channel
//                          means), output in ascending voxel order.
#include <climits>
#include <cmath>
#include <cstring>

#include "kernels.hpp"

namespace gicpb {

namespace {

constexpr int kSegThreads = 128;
constexpr int kSegQueueCap = 16;

// ---- union-find on sorted positions: the root of a set is its smallest member ---------------------------------------
__device__ __forceinline__ int uf_find(volatile int* parent, int x) {
  for (;;) {
    const int p = parent[x];
    if (p == x) return x;
    const int gp = parent[p];
    if (gp != p) parent[x] = gp;  // path halving (a benign race: parents only ever move towards the root)
    x = p;
  }
}

__device__ __forceinline__ void uf_unite(int* parent, int a, int b) {
  for (;;) {
    a = uf_find(parent, a);
    b = uf_find(parent, b);
    if (a == b) return;
    if (a < b) { const int t = a; a = b; b = t; }  // a > b: hang the larger root under the smaller
    const int old = atomicMin(&parent[a], b);
    if (old == a) return;  // a was still a root: linked
    a = old;               // somebody re-parented a meanwhile: join that set with b instead
  }
}

struct UniteVisitor {
  const float4* pts;
  int* parent;
  float qx, qy, qz;
  float r2;
  unsigned self;  // sorted position of the query: every edge is handled once, from its larger end
  int root;       // last known root of the query's set: a neighbour already hanging under it needs no union
  __device__ __forceinline__ float bound() const { return r2; }
  __device__ __forceinline__ void apply(unsigned i, const float4& p) {
    if (i < self && dist2(qx, qy, qz, p) < r2) {
      if (*reinterpret_cast<volatile int*>(parent + i) == root) return;  // dense blobs: almost every pair ends here
      uf_unite(parent, (int)self, (int)i);
      root = uf_find(parent, (int)self);
    }
  }
  __device__ __forceinline__ bool point(unsigned i) {
    apply(i, __ldg(&pts[i]));
    return false;
  }
  __device__ __forceinline__ bool point2(unsigned i, bool two) {
    const float4 p0 = __ldg(&pts[i]);
    const float4 p1 = __ldg(&pts[two ? i + 1 : i]);
    apply(i, p0);
    if (two) apply(i + 1, p1);
    return false;
  }
  __device__ __forceinline__ bool range(unsigned b, unsigned e) {
    for (unsigned i = b; i < e && i < self; ++i) point(i);
    return false;
  }
};

__global__ void __launch_bounds__(256) iota_kernel(int* __restrict__ a, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) a[i] = i;
}

template <bool kFar>
__global__ void __launch_bounds__(kSegThreads, kFar ? 4 : 6) cluster_union_kernel(GridView g, float r2, int* __restrict__ parent,
                                                                                   FarWork fw) {
  __shared__ unsigned s_qb[kFar ? 1 : kSegQueueCap * kSegThreads];
  __shared__ unsigned s_qe[kFar ? 1 : kSegQueueCap * kSegThreads];
  unsigned* qb = s_qb + (kFar ? 0 : threadIdx.x);
  unsigned* qe = s_qe + (kFar ? 0 : threadIdx.x);
  auto body = [&](int i) {
    const float4 p = __ldg(&g.pts[i]);
    const Query q = make_query(g, p.x, p.y, p.z);
    UniteVisitor v{g.pts, parent, p.x, p.y, p.z, r2, (unsigned)i, i};
    if (kFar) {
      far_search(g, q, v);
      return;
    }
    const float rad = fadd(sqrt_up(r2), g.margin);
    const int x0 = max(cell_of(fsub(p.x, rad), g.ox, g.inv_h), 0), x1 = min(cell_of(fadd(p.x, rad), g.ox, g.inv_h), g.nx - 1);
    const int y0 = max(cell_of(fsub(p.y, rad), g.oy, g.inv_h), 0), y1 = min(cell_of(fadd(p.y, rad), g.oy, g.inv_h), g.ny - 1);
    const int z0 = max(cell_of(fsub(p.z, rad), g.oz, g.inv_h), 0), z1 = min(cell_of(fadd(p.z, rad), g.oz, g.inv_h), g.nz - 1);
    if ((long long)(y1 - y0 + 1) * (z1 - z0 + 1) > kMaxBoxRows) {
      fw.flags[i] = 1;
      return;
    }
    QueueVisitor<kSegThreads, kSegQueueCap, UniteVisitor> qv{qb, qe, 0, v};
    visit_box(g, q, x0, x1, y0, y1, z0, z1, qv);
    qv.drain();
  };
  if (kFar) {
    far_for_each(fw, g.n, body);
  } else {
    const int k = blockIdx.x * kSegThreads + threadIdx.x;
    if (k < g.n) {
      fw.flags[k] = 0;
      body(k);
    }
  }
}

// root_of[original index] = ORIGINAL index of the root point of its set (non-indexed points keep -1)
__global__ void __launch_bounds__(256) cluster_flatten_kernel(GridView g, int* __restrict__ parent, int* __restrict__ root_of) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= g.n) return;
  const int r = uf_find(parent, i);
  root_of[__float_as_int(__ldg(&g.pts[i]).w)] = __float_as_int(__ldg(&g.pts[r]).w);
}

// ---- voxel grid -----------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned vg_f2ord(float f) {
  const unsigned b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

// scratch: [0..2] min xyz (ordered bits), [3..5] max xyz, [6] finite count
__global__ void __launch_bounds__(256) voxel_minmax_kernel(const unsigned char* __restrict__ raw, int64_t n, int64_t stride,
                                                            unsigned* __restrict__ scratch) {
  __shared__ unsigned smin[3][8], smax[3][8], scnt[8];
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float x = 0.f, y = 0.f, z = 0.f;
  bool ok = false;
  if (i < n) {
    const float* p = reinterpret_cast<const float*>(raw + i * stride);
    x = p[0]; y = p[1]; z = p[2];
    ok = finite3(x, y, z);
  }
  unsigned mn[3] = {ok ? vg_f2ord(x) : 0xffffffffu, ok ? vg_f2ord(y) : 0xffffffffu, ok ? vg_f2ord(z) : 0xffffffffu};
  unsigned mx[3] = {ok ? vg_f2ord(x) : 0u, ok ? vg_f2ord(y) : 0u, ok ? vg_f2ord(z) : 0u};
  unsigned c = ok ? 1u : 0u;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    mn[a] = __reduce_min_sync(kFullMask, mn[a]);
    mx[a] = __reduce_max_sync(kFullMask, mx[a]);
  }
  c = __reduce_add_sync(kFullMask, c);
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

struct VoxelParams {
  float inv_leaf[3];
  int min_b[3];
  uint32_t mul[3];  // divb_mul_: 1, div0, div0 * div1 (wrapped to 32 bits, as PCL's int product)
};

__global__ void __launch_bounds__(256) voxel_finite_kernel(const unsigned char* __restrict__ raw, int64_t n, int64_t stride,
                                                            uint32_t* __restrict__ flags) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* p = reinterpret_cast<const float*>(raw + i * stride);
  flags[i] = finite3(p[0], p[1], p[2]) ? 1u : 0u;
}

// voxel_grid.hpp first pass: ijk = int(floor(x * inverse_leaf) - float(min_b)); idx = ijk . divb_mul in 32-bit
// arithmetic that wraps as PCL's int index does.  The finite points land at pos[i] (the exclusive scan of
// voxel_finite_kernel's flags), or at i when every point is finite (pos == nullptr).
__global__ void __launch_bounds__(256) voxel_keys_kernel(const unsigned char* __restrict__ raw, int64_t n, int64_t stride,
                                                          VoxelParams vp, const uint32_t* __restrict__ pos,
                                                          uint32_t* __restrict__ keys, uint32_t* __restrict__ vals) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* p = reinterpret_cast<const float*>(raw + i * stride);
  const float x = p[0], y = p[1], z = p[2];
  if (!finite3(x, y, z)) return;
  const int i0 = __float2int_rz(__fsub_rn(floorf(__fmul_rn(x, vp.inv_leaf[0])), (float)vp.min_b[0]));
  const int i1 = __float2int_rz(__fsub_rn(floorf(__fmul_rn(y, vp.inv_leaf[1])), (float)vp.min_b[1]));
  const int i2 = __float2int_rz(__fsub_rn(floorf(__fmul_rn(z, vp.inv_leaf[2])), (float)vp.min_b[2]));
  const uint32_t j = pos ? pos[i] : (uint32_t)i;
  keys[j] = (uint32_t)i0 * vp.mul[0] + (uint32_t)i1 * vp.mul[1] + (uint32_t)i2 * vp.mul[2];
  vals[j] = (uint32_t)i;
}

__global__ void __launch_bounds__(256) voxel_heads_kernel(const uint32_t* __restrict__ keys, int n_valid,
                                                           uint32_t* __restrict__ flags) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_valid) return;
  flags[i] = (i == 0 || keys[i - 1] != keys[i]) ? 1u : 0u;
}

// starts[rank of the voxel] = first sorted element of the voxel; starts[n_voxels] = n_valid
__global__ void __launch_bounds__(256) voxel_starts_kernel(const uint32_t* __restrict__ flags, const uint32_t* __restrict__ ranks,
                                                            int n_valid, uint32_t* __restrict__ starts,
                                                            unsigned* __restrict__ scratch) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_valid) return;
  if (flags[i]) starts[ranks[i]] = (uint32_t)i;
  if (i == n_valid - 1) {
    const uint32_t nv = ranks[i] + flags[i];
    starts[nv] = (uint32_t)n_valid;
    scratch[7] = nv;
  }
}

// One thread per voxel: pcl::CentroidPoint<PointXYZRGB> over the voxel's points in sorted (= original) order.
// AccumulatorXYZ: float sums, xyz / n; AccumulatorRGBA: float channel sums, uint32(channel / n).
__global__ void __launch_bounds__(128) voxel_centroid_kernel(const unsigned char* __restrict__ raw, int64_t stride,
                                                              const uint32_t* __restrict__ vals,
                                                              const uint32_t* __restrict__ starts, int n_voxels,
                                                              unsigned char* __restrict__ out) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n_voxels) return;
  const uint32_t b = starts[v], e = starts[v + 1];
  float sx = 0.f, sy = 0.f, sz = 0.f, sr = 0.f, sg = 0.f, sb = 0.f, sa = 0.f;
  const bool rgb = stride >= 20;
  for (uint32_t k = b; k < e; ++k) {
    const unsigned char* pt = raw + (int64_t)vals[k] * stride;
    const float* p = reinterpret_cast<const float*>(pt);
    sx = __fadd_rn(sx, p[0]);
    sy = __fadd_rn(sy, p[1]);
    sz = __fadd_rn(sz, p[2]);
    if (rgb) {
      const uint32_t c = *reinterpret_cast<const uint32_t*>(pt + 16);
      sb = __fadd_rn(sb, (float)(c & 255u));
      sg = __fadd_rn(sg, (float)((c >> 8) & 255u));
      sr = __fadd_rn(sr, (float)((c >> 16) & 255u));
      sa = __fadd_rn(sa, (float)(c >> 24));
    }
  }
  const float nf = (float)(e - b);
  unsigned char* o = out + (int64_t)v * stride;
  uint32_t* ow = reinterpret_cast<uint32_t*>(o);
  const int words = (int)(stride >> 2);
  for (int w = 3; w < words; ++w) ow[w] = 0u;
  ow[0] = __float_as_uint(__fdiv_rn(sx, nf));
  ow[1] = __float_as_uint(__fdiv_rn(sy, nf));
  ow[2] = __float_as_uint(__fdiv_rn(sz, nf));
  if (stride >= 16) ow[3] = __float_as_uint(1.0f);  // PointXYZRGB::data[3]
  if (rgb)
    ow[4] = ((uint32_t)__fdiv_rn(sa, nf) << 24) | ((uint32_t)__fdiv_rn(sr, nf) << 16) | ((uint32_t)__fdiv_rn(sg, nf) << 8) |
            (uint32_t)__fdiv_rn(sb, nf);
}

inline unsigned nblk(int64_t n, int t) { return (unsigned)((n + t - 1) / t); }

inline float ord2f(unsigned u) {
  unsigned b = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
  float f;
  std::memcpy(&f, &b, 4);
  return f;
}

}  // namespace

void launch_cluster_unions(const GridView& g, float r2, int* parent, int* root_of, const FarWork& fw, cudaStream_t stream) {
  if (g.n <= 0) return;
  iota_kernel<<<nblk(g.n, 256), 256, 0, stream>>>(parent, g.n);
  GICPB_LAUNCHED();
  reset_far(fw, g.n, stream);
  cluster_union_kernel<false><<<nblk(g.n, kSegThreads), kSegThreads, 0, stream>>>(g, r2, parent, fw);
  GICPB_LAUNCHED();
  cluster_union_kernel<true><<<fw.far_blocks, kSegThreads, 0, stream>>>(g, r2, parent, fw);
  GICPB_LAUNCHED();
  cluster_flatten_kernel<<<nblk(g.n, 256), 256, 0, stream>>>(g, parent, root_of);
  GICPB_LAUNCHED();
}

int64_t VoxelGrid::run(const unsigned char* d_in, int64_t n, int64_t stride, float leaf, unsigned char* d_out,
                       cudaStream_t stream, bool* overflow) {
  *overflow = false;
  scratch_.reserve(16);
  GICPB_CUDA(cudaMemsetAsync(scratch_.get(), 0xff, 3 * sizeof(unsigned), stream));
  GICPB_CUDA(cudaMemsetAsync(scratch_.get() + 3, 0, 13 * sizeof(unsigned), stream));
  voxel_minmax_kernel<<<nblk(n, 256), 256, 0, stream>>>(d_in, n, stride, scratch_.get());
  GICPB_LAUNCHED();
  unsigned hs[8];
  GICPB_CUDA(cudaMemcpyAsync(hs, scratch_.get(), sizeof(hs), cudaMemcpyDeviceToHost, stream));
  GICPB_CUDA(cudaStreamSynchronize(stream));
  const int64_t n_valid = hs[6];
  if (n_valid == 0) return 0;
  // voxel_grid.hpp: inverse_leaf_size_ = 1 / leaf (float); the index-overflow check; min_b / max_b / div_b / divb_mul
  const float inv = 1.0f / leaf;
  float min_p[3], max_p[3];
  int64_t cells = 1;
  VoxelParams vp{};
  int64_t div[3];
  for (int a = 0; a < 3; ++a) {
    min_p[a] = ord2f(hs[a]);
    max_p[a] = ord2f(hs[3 + a]);
    const int64_t d = (int64_t)((max_p[a] - min_p[a]) * inv) + 1;
    cells *= d;
    if (cells > (int64_t)INT32_MAX) {
      *overflow = true;  // "Leaf size is too small for the input dataset": PCL copies the input through
      return n;
    }
  }
  // div_b can exceed dx by one on every axis, so div0 * div1 * div2 may pass 2^31 and even 2^32 where PCL's check
  // passes; PCL's 32-bit index then wraps and voxels that share the wrapped index are averaged together.
  bool wide = false;  // an index may reach 2^24 voxels along an axis, where float(ijk) rounds: sort on all 32 bits
  double total = 1.0;
  for (int a = 0; a < 3; ++a) {
    vp.inv_leaf[a] = inv;
    vp.min_b[a] = (int)std::floor(min_p[a] * inv);
    const int64_t max_b = (int64_t)std::floor(max_p[a] * inv);
    div[a] = max_b - vp.min_b[a] + 1;
    wide = wide || div[a] > (1 << 24);
    total *= (double)div[a];
  }
  vp.mul[0] = 1u;
  vp.mul[1] = (uint32_t)div[0];
  vp.mul[2] = (uint32_t)div[0] * (uint32_t)div[1];
  int key_bits = 1;  // the keys are below total
  while (key_bits < 32 && (wide || (double)(1ull << key_bits) < total)) ++key_bits;
  keys_a_.reserve(n); keys_b_.reserve(n); vals_a_.reserve(n); vals_b_.reserve(n);
  scan_tmp_.reserve(scan_tmp_entries(n));
  sorter_.prepare(n_valid, stream);
  const uint32_t* pos = nullptr;
  if (n_valid < n) {  // compact the finite points, in input order, so that every 32-bit key is a voxel index
    voxel_finite_kernel<<<nblk(n, 256), 256, 0, stream>>>(d_in, n, stride, keys_b_.get());
    GICPB_LAUNCHED();
    exclusive_scan_u32(keys_b_.get(), vals_b_.get(), n, scan_tmp_.get(), stream);
    pos = vals_b_.get();
  }
  voxel_keys_kernel<<<nblk(n, 256), 256, 0, stream>>>(d_in, n, stride, vp, pos, keys_a_.get(), vals_a_.get());
  GICPB_LAUNCHED();
  const bool in_b = sorter_.sort(keys_a_.get(), vals_a_.get(), keys_b_.get(), vals_b_.get(), n_valid, key_bits, false,
                                 stream);
  const uint32_t* skeys = in_b ? keys_b_.get() : keys_a_.get();
  const uint32_t* svals = in_b ? vals_b_.get() : vals_a_.get();
  uint32_t* flags = in_b ? keys_a_.get() : keys_b_.get();
  uint32_t* ranks = in_b ? vals_a_.get() : vals_b_.get();
  voxel_heads_kernel<<<nblk(n_valid, 256), 256, 0, stream>>>(skeys, (int)n_valid, flags);
  GICPB_LAUNCHED();
  exclusive_scan_u32(flags, ranks, n_valid, scan_tmp_.get(), stream);
  starts_.reserve((size_t)n_valid + 1);
  voxel_starts_kernel<<<nblk(n_valid, 256), 256, 0, stream>>>(flags, ranks, (int)n_valid, starts_.get(), scratch_.get());
  GICPB_LAUNCHED();
  GICPB_CUDA(cudaMemcpyAsync(hs, scratch_.get(), sizeof(hs), cudaMemcpyDeviceToHost, stream));
  GICPB_CUDA(cudaStreamSynchronize(stream));
  const int64_t n_vox = hs[7];
  voxel_centroid_kernel<<<nblk(n_vox, 128), 128, 0, stream>>>(d_in, stride, svals, starts_.get(), (int)n_vox, d_out);
  GICPB_LAUNCHED();
  return n_vox;
}

}  // namespace gicpb
