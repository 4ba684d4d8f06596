// common.cuh - shared device-side definitions of libgicp_b200 (sm_100a).
//
// Spatial index ("brick grid"): a uniform grid of cubic cells of edge h over the cloud's bounding box, with three
// coarser occupancy levels above it so that empty space is skipped in O(log) steps however far a query is:
//
//   cell        edge h          points of one cell are contiguous in the sorted array
//   brick       8 x 8 x 8 cells only OCCUPIED bricks own a table: cell_start[slot*512 + code], code = (lz<<6)|(ly<<3)|lx,
//                               the exclusive prefix "first sorted point whose (brick, code) is >= this one".  Slots are
//                               numbered in brick order, so cell_start[slot*512 + code + 1] is always the END of a cell
//                               and every x-run of cells, every row (8 cells), slab (64) and brick (512) is ONE range.
//   superbrick  4 x 4 x 4 bricks        one 64-bit occupancy mask each, dense array
//   hyperbrick  4 x 4 x 4 superbricks   one 64-bit occupancy mask each, dense array
//
// Points are sorted by key = brick_linear * 512 + code with a stable radix sort, so inside one cell the sorted
// order is the original order.  This index replaces the two FLANN kd-trees the reference builds through
// pcl::Registration::initCompute / initComputeReciprocal (reference src/GICPAlignment.cpp:89-96) and the
// pcl::search::KdTree of Filter::removeFromCloud (reference src/Filter.cpp:181-184).
//
// Everything in this header is written so that it also compiles as plain host C++ (tests/host_emul builds the search
// on the CPU against brute force to check the traversal logic without a GPU).  The shipped library only ever calls
// these functions from kernels.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#include <cuda_runtime.h>
#define GICPB_HD __host__ __device__ __forceinline__
#else
#include <cmath>
#include <cstring>
#define GICPB_HD inline
struct float3 { float x, y, z; };
struct float4 { float x, y, z, w; };
struct uint2 { unsigned x, y; };
#endif

namespace gicpb {

constexpr int kBrickShift = 3;                  // 8 cells per brick edge
constexpr int kBrickCells = 512;                // 8*8*8
constexpr int kMaxBoxRows = 81;                 // NN-1: largest (y,z) row count searched as a plain cell box
constexpr int kSeedBoxRows = 4;                 // NN-1: a seed whose ball spans more rows is first improved by a probe
constexpr int kNearMaxRing = 3;                // NN-1: cell rings probed for a first candidate before the far search
constexpr int kKnnMaxRing = 4;                  // kNN: largest cell ring searched before the hierarchical fallback
// Point ranges a thread can queue before it scans them (QueueVisitor), as the kernels instantiate the near searches;
// tests/host_emul builds the same instances.  NN-1 (nn_kernels.cu): 3x3 rows, one of them split by a brick edge; 16
// entries took 16 KB of every block from L1: correspondence kernels of a job 1.616 -> 1.58 ms at 1 M, 27.5 -> 26.5 ms
// at 8 M.  kNN (knn_cov.cu): in dynamic shared memory beside the k-best lists.
constexpr int kNnQueueCap = 10;
constexpr int kKnnQueueCap = 8;
constexpr unsigned kFullMask = 0xffffffffu;

// ---- arithmetic with one rounding per operation on both sides (bit-exact against the oracle) -------------------------
#if defined(__CUDA_ARCH__)
GICPB_HD float fadd(float a, float b) { return __fadd_rn(a, b); }
GICPB_HD float fsub(float a, float b) { return __fsub_rn(a, b); }
GICPB_HD float fmul(float a, float b) { return __fmul_rn(a, b); }
GICPB_HD int floor_to_int(float v) { return __float2int_rd(v); }
// an upper bound of sqrt(v), only ever used to size a search box: the approximate square root (MUFU.SQRT, relative
// error <= 2^-23) times 1 + 2^-21 is never below the true root and costs two instructions instead of the
// range-checked Newton sequence of __fsqrt_ru
GICPB_HD float sqrt_up(float v) {
  float r;
  asm("sqrt.approx.f32 %0, %1;" : "=f"(r) : "f"(v));
  return __fmul_ru(r, 1.00000047683715820312f);
}
GICPB_HD int ffs64(unsigned long long m) { return __ffsll((long long)m); }
template <typename T>
GICPB_HD T ldg(const T* p) { return __ldg(p); }
GICPB_HD int f2i_bits(float f) { return __float_as_int(f); }
GICPB_HD float i2f_bits(int i) { return __int_as_float(i); }
#else
// host build (tests only): compile with -ffp-contract=off
GICPB_HD float fadd(float a, float b) { return a + b; }
GICPB_HD float fsub(float a, float b) { return a - b; }
GICPB_HD float fmul(float a, float b) { return a * b; }
GICPB_HD int floor_to_int(float v) {
  const float f = floorf(v);
  return f >= 2147483520.f ? 2147483647 : (f <= -2147483648.f ? -2147483647 - 1 : (int)f);
}
GICPB_HD float sqrt_up(float v) { return nextafterf(sqrtf(v), INFINITY); }
GICPB_HD int ffs64(unsigned long long m) { return __builtin_ffsll((long long)m); }
template <typename T>
GICPB_HD T ldg(const T* p) { return *p; }
GICPB_HD int f2i_bits(float f) { int i; memcpy(&i, &f, 4); return i; }
GICPB_HD float i2f_bits(int i) { float f; memcpy(&f, &i, 4); return f; }
#endif

GICPB_HD float fmin2(float a, float b) { return a < b ? a : b; }
GICPB_HD float fmax2(float a, float b) { return a > b ? a : b; }
GICPB_HD int imin2(int a, int b) { return a < b ? a : b; }
GICPB_HD int imax2(int a, int b) { return a > b ? a : b; }
GICPB_HD int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }
GICPB_HD float inf() { return i2f_bits(0x7f800000); }

struct GridView {
  const float4* pts;             // sorted points: x, y, z, w = original index (int bits)
  const int* brick_slot;         // [nbx*nby*nbz] -> table slot, -1 = empty brick; slots ascend with the brick index
  const uint32_t* cell_start;    // [n_slots*512 + 1] exclusive prefix (see the header comment); last entry = n
  const int* pos_of;             // [n_points] original index -> position in pts (-1 for a non-finite point)
  const unsigned long long* sb_mask;  // [nsx*nsy*nsz] occupancy of the 4x4x4 bricks of a superbrick, bit (lz<<4)|(ly<<2)|lx
  const unsigned long long* hb_mask;  // [nhx*nhy*nhz] occupancy of the 4x4x4 superbricks of a hyperbrick
  const float* brick_plane;      // [n_slots*5] or null: unit direction n of the brick's points (their PCA normal) and the
                                 // smallest / largest n.p over them: every point of the brick lies in that slab
  const float* sb_plane;         // [nsx*nsy*nsz*5] or null: the same slab for all points of a superbrick (indexed like sb_mask)
  float ox, oy, oz;              // origin (min corner of cell (0,0,0))
  float h, inv_h;                // cell edge and its reciprocal
  float margin;                  // conservative slack (metres) for all box-distance lower bounds
  int nx, ny, nz;                // grid size in cells (multiples of 8)
  int nbx, nby, nbz;             // grid size in bricks
  int bsx, bsy, bsz;             // linear brick index = bx * bsx + by * bsy + bz * bsz (default 1, nbx, nbx * nby)
  int bo0, bo1, bo2;             // the axes (0 x, 1 y, 2 z) from the fastest to the slowest in that index (default 0, 1, 2)
  int nsx, nsy, nsz;             // grid size in superbricks
  int nhx, nhy, nhz;             // grid size in hyperbricks
  int n;                         // number of indexed (finite) points
};

struct Rigid {                   // float 4x4 upper 3 rows, row-major: q = ((r0*x + r1*y) + r2*z) + t
  float m[12];
};

GICPB_HD float3 xform(const Rigid& T, float x, float y, float z) {
  // op order of Eigen's fixed-size Matrix4f * Vector4f (w = 1); no FMA contraction (bit-exact vs oracle)
  float3 q;
  q.x = fadd(fadd(fadd(fmul(T.m[0], x), fmul(T.m[1], y)), fmul(T.m[2], z)), T.m[3]);
  q.y = fadd(fadd(fadd(fmul(T.m[4], x), fmul(T.m[5], y)), fmul(T.m[6], z)), T.m[7]);
  q.z = fadd(fadd(fadd(fmul(T.m[8], x), fmul(T.m[9], y)), fmul(T.m[10], z)), T.m[11]);
  return q;
}

// squared distance exactly as FLANN L2_Simple accumulates it in float: (dx*dx + dy*dy) + dz*dz
GICPB_HD float dist2(float qx, float qy, float qz, const float4& p) {
  const float dx = fsub(qx, p.x), dy = fsub(qy, p.y), dz = fsub(qz, p.z);
  return fadd(fadd(fmul(dx, dx), fmul(dy, dy)), fmul(dz, dz));
}

GICPB_HD bool finite1(float v) { return (f2i_bits(v) & 0x7f800000) != 0x7f800000; }
GICPB_HD bool finite3(float x, float y, float z) { return finite1(x) && finite1(y) && finite1(z); }

// row-major cell code inside a brick: x fastest, then y, then z
GICPB_HD unsigned local_code(unsigned lx, unsigned ly, unsigned lz) { return (lz << 6) | (ly << 3) | lx; }

// cell coordinate of a coordinate value along one axis (NOT clamped); identical code for build and query
GICPB_HD int cell_of(float v, float origin, float inv_h) { return floor_to_int(fmul(fsub(v, origin), inv_h)); }

GICPB_HD int brick_index(const GridView& g, int bx, int by, int bz) { return bx * g.bsx + by * g.bsy + bz * g.bsz; }

// lower bound of |q - p| along one axis for any p stored in the box [lo, lo + size); never negative
GICPB_HD float axis_gap(float q, float lo, float size, float margin) {
  const float d = fmax2(fsub(lo, q), fsub(q, fadd(lo, size)));
  return fmax2(fsub(d, margin), 0.0f);
}
// the same for the node with integer coordinate c at a level whose nodes have edge `size`
GICPB_HD float node_gap(float q, float origin, int c, float size, float margin) {
  return axis_gap(q, fadd(origin, fmul((float)c, size)), size, margin);
}
GICPB_HD float sq3(float a, float b, float c) { return fadd(fadd(fmul(a, a), fmul(b, b)), fmul(c, c)); }

// candidate order: smaller d2 first, ties towards the lowest ORIGINAL index
GICPB_HD bool cand_less(float d, int oi, float d_ref, int oi_ref) {
  return d < d_ref || (d == d_ref && oi < oi_ref);
}

// occupancy-mask helpers for a 4x4x4 node: bit = (z<<4)|(y<<2)|x
GICPB_HD unsigned span4(int p, int r) {  // 4-bit mask of the coordinates in [p-r, p+r] cut to [0,3]
  const int lo = imax2(p - r, 0), hi = imin2(p + r, 3);
  return ((1u << (hi + 1)) - 1u) & ~((1u << lo) - 1u);
}
GICPB_HD unsigned long long spans_mask64(unsigned xm, unsigned ym, unsigned zm) {  // the box of three 4-bit coordinate sets
  const unsigned plane = xm * ((ym & 1u) | ((ym & 2u) << 3) | ((ym & 4u) << 6) | ((ym & 8u) << 9));
  const unsigned long long zs = (unsigned long long)(zm & 1u) | ((unsigned long long)(zm & 2u) << 15) |
                                ((unsigned long long)(zm & 4u) << 30) | ((unsigned long long)(zm & 8u) << 45);
  return (unsigned long long)plane * zs;
}
GICPB_HD unsigned long long box_mask64(int px, int py, int pz, int r) {
  return spans_mask64(span4(px, r), span4(py, r), span4(pz, r));
}
GICPB_HD unsigned range4(int lo, int hi) {  // 4-bit mask of the coordinates in [lo, hi] cut to [0,3]; 0 when empty
  lo = imax2(lo, 0);
  hi = imin2(hi, 3);
  return lo > hi ? 0u : (((1u << (hi + 1)) - 1u) & ~((1u << lo) - 1u));
}

// ---- query context: the query point and its (clamped) cell ---------------------------------------------------------------
struct Query {
  float x, y, z;
  int cx, cy, cz;
};
GICPB_HD Query make_query(const GridView& g, float qx, float qy, float qz) {
  Query q;
  q.x = qx; q.y = qy; q.z = qz;
  q.cx = clampi(cell_of(qx, g.ox, g.inv_h), 0, g.nx - 1);
  q.cy = clampi(cell_of(qy, g.oy, g.inv_h), 0, g.ny - 1);
  q.cz = clampi(cell_of(qz, g.oz, g.inv_h), 0, g.nz - 1);
  return q;
}

// The searches below are written against a visitor V:
//   float bound() const                 current squared search radius; a box whose lower bound is > bound() is skipped
//                                       (strictly: an equal-distance candidate can still win its tie)
//   bool range(unsigned b, unsigned e)  visit sorted points [b, e); return true to stop the whole search

// cells [x0, x1] of row (y, z); the run may cross brick boundaries
template <class V>
GICPB_HD bool visit_run(const GridView& g, int x0, int x1, int y, int z, V& v) {
  const int row = ((z & 7) << 6) | ((y & 7) << 3);
  const int by = y >> kBrickShift, bz = z >> kBrickShift;
  for (int bx = x0 >> kBrickShift; bx <= (x1 >> kBrickShift); ++bx) {
    const int slot = ldg(&g.brick_slot[brick_index(g, bx, by, bz)]);
    if (slot < 0) continue;
    const int lx0 = imax2(x0 - (bx << kBrickShift), 0), lx1 = imin2(x1 - (bx << kBrickShift), 7);
    const uint32_t* cs = g.cell_start + (size_t)slot * kBrickCells + row;
    const unsigned b = ldg(&cs[lx0]), e = ldg(&cs[lx1 + 1]);
    if (b < e && v.range(b, e)) return true;
  }
  return false;
}

// every cell of the box [x0,x1] x [y0,y1] x [z0,z1] (already cut to the grid) that can hold a point closer than bound()
template <class V>
GICPB_HD bool visit_box(const GridView& g, const Query& q, int x0, int x1, int y0, int y1, int z0, int z1, V& v) {
  const float h = g.h;
  for (int z = z0; z <= z1; ++z) {
    const float gz = node_gap(q.z, g.oz, z, h, g.margin);
    const float gz2 = fmul(gz, gz);
    if (gz2 > v.bound()) continue;
    for (int y = y0; y <= y1; ++y) {
      const float gy = node_gap(q.y, g.oy, y, h, g.margin);
      const float gyz2 = fadd(fmul(gy, gy), gz2);
      const float bnd = v.bound();
      if (gyz2 > bnd) continue;
      int xa = x0, xb = x1;
      if (bnd < 3.0e38f) {  // cut the run to the chord of the ball at this (y, z)
        const float rx = fadd(sqrt_up(fmax2(fsub(bnd, gyz2), 0.f)), g.margin);
        xa = imax2(xa, cell_of(fsub(q.x, rx), g.ox, g.inv_h));
        xb = imin2(xb, cell_of(fadd(q.x, rx), g.ox, g.inv_h));
        if (xa > xb) continue;
      }
      if (visit_run(g, xa, xb, y, z, v)) return true;
    }
  }
  return false;
}

// shell of Chebyshev radius R (>= 2) around the query's cell: the box of radius R minus the box of radius R - 1
template <class V>
GICPB_HD bool visit_shell(const GridView& g, const Query& q, int R, V& v) {
  const float h = g.h;
  const int z0 = imax2(q.cz - R, 0), z1 = imin2(q.cz + R, g.nz - 1);
  const int y0 = imax2(q.cy - R, 0), y1 = imin2(q.cy + R, g.ny - 1);
  for (int z = z0; z <= z1; ++z) {
    const float gz = node_gap(q.z, g.oz, z, h, g.margin);
    const float gz2 = fmul(gz, gz);
    if (gz2 > v.bound()) continue;
    const bool ez = (z - q.cz == R) || (q.cz - z == R);
    for (int y = y0; y <= y1; ++y) {
      const float gy = node_gap(q.y, g.oy, y, h, g.margin);
      const float gyz2 = fadd(fmul(gy, gy), gz2);
      const float bnd = v.bound();
      if (gyz2 > bnd) continue;
      int xa = 0, xb = g.nx - 1;
      if (bnd < 3.0e38f) {  // chord of the search ball at this (y, z)
        const float rx = fadd(sqrt_up(fmax2(fsub(bnd, gyz2), 0.f)), g.margin);
        xa = imax2(xa, cell_of(fsub(q.x, rx), g.ox, g.inv_h));
        xb = imin2(xb, cell_of(fadd(q.x, rx), g.ox, g.inv_h));
      }
      if (ez || (y - q.cy == R) || (q.cy - y == R)) {
        xa = imax2(xa, q.cx - R);
        xb = imin2(xb, q.cx + R);
        if (xa <= xb && visit_run(g, xa, xb, y, z, v)) return true;
      } else {
        const int xl = q.cx - R, xr = q.cx + R;
        if (xl >= xa && xl <= xb && visit_run(g, xl, xl, y, z, v)) return true;
        if (xr >= xa && xr <= xb && visit_run(g, xr, xr, y, z, v)) return true;
      }
    }
  }
  return false;
}

// n.p exactly as the index build evaluates it for the points of a brick (same operations, same order)
GICPB_HD float plane_dot(float nx, float ny, float nz, float x, float y, float z) {
  return fadd(fadd(fmul(nx, x), fmul(ny, y)), fmul(nz, z));
}
GICPB_HD float fabs1(float v) { return v < 0.f ? -v : v; }

// A visitor for which seeing a point twice is harmless (a running minimum) declares `static constexpr bool kRescanOk =
// true`; visit_brick then looks at the cell under the query's foot first.  Visitors that collect (kNN) or count do not.
template <class V>
GICPB_HD constexpr auto rescan_ok_impl(int) -> decltype(V::kRescanOk) { return V::kRescanOk; }
template <class V>
GICPB_HD constexpr bool rescan_ok_impl(long) { return false; }
template <class V>
GICPB_HD constexpr bool rescan_ok() { return rescan_ok_impl<V>(0); }

// lower bound of |f - p| along one axis for f anywhere in [flo, fhi] and p in the box [lo, lo + size); never negative
GICPB_HD float interval_gap(float flo, float fhi, float lo, float size, float margin) {
  const float d = fmax2(fsub(lo, fhi), fsub(flo, fadd(lo, size)));
  return fmax2(fsub(d, margin), 0.0f);
}

// one occupied brick: slabs (8x8x1 cells) and rows (8x1x1) nearest first, each pruned by its box distance.
//
// Oriented slab of the brick (g.brick_plane): its points satisfy lo <= n.p <= hi.  Split q - p = alpha n + w, w normal
// to n.  Then alpha = n.q - n.p lies in [n.q - hi, n.q - lo], |alpha| >= s (the distance from n.q to [lo, hi]), and per
// axis i   p_i = (q_i - alpha n_i) - w_i:   the point sits within |w_i| of the FOOT interval F_i = q_i - n_i [alpha range]
// (where the query lands on the slab along n).  A box whose interval on axis i is l_i away from F_i therefore holds no
// point closer than s^2 + sum_i l_i^2.  For a query far off a thin sheet F is as small as the sheet is thin, so only the
// boxes NEAR THE FOOT of the query are opened, where the plain box distance keeps every box within sqrt(2 R h) of the
// touch point (R = distance of the query, h = box edge).  Any direction n keeps the search exact.
template <class V>
GICPB_HD bool visit_brick(const GridView& g, const Query& q, int bx, int by, int bz, int slot, V& v) {
  const uint32_t* cs = g.cell_start + (size_t)slot * kBrickCells;
  const float h = g.h, hb = fmul(h, 8.0f);
  const float gx = node_gap(q.x, g.ox, bx, hb, g.margin);
  const float gyb = node_gap(q.y, g.oy, by, hb, g.margin);
  const float gx2 = fmul(gx, gx);
  const float gxy2 = fadd(gx2, fmul(gyb, gyb));
  const bool slab = g.brick_plane != nullptr;
  float slab2 = 0.f;                                                         // s^2
  float fxl = q.x, fxh = q.x, fyl = q.y, fyh = q.y, fzl = q.z, fzh = q.z;  // foot intervals
  float lxb2 = gx2, lyb = gyb;                                               // foot-to-brick gaps in x (squared) and y
  if (slab) {
    const float* pl = g.brick_plane + 5 * (size_t)slot;
    const float nx = ldg(&pl[0]), ny = ldg(&pl[1]), nz = ldg(&pl[2]), lo = ldg(&pl[3]), hi = ldg(&pl[4]);
    const float nq = plane_dot(nx, ny, nz, q.x, q.y, q.z);
    // the margin covers the rounding of both dot products and |n| = 1 +- 1e-7
    const float s = fmax2(fsub(fmax2(fsub(nq, hi), fsub(lo, nq)), g.margin), 0.f);
    slab2 = fmul(fmul(s, s), 0.999998f);
    const float al = fsub(fsub(nq, hi), g.margin), ah = fadd(fsub(nq, lo), g.margin);  // alpha range, widened
    const float x0 = fmul(nx, al), x1 = fmul(nx, ah), y0 = fmul(ny, al), y1 = fmul(ny, ah), z0 = fmul(nz, al), z1 = fmul(nz, ah);
    fxl = fsub(q.x, fmax2(x0, x1)); fxh = fsub(q.x, fmin2(x0, x1));
    fyl = fsub(q.y, fmax2(y0, y1)); fyh = fsub(q.y, fmin2(y0, y1));
    fzl = fsub(q.z, fmax2(z0, z1)); fzh = fsub(q.z, fmin2(z0, z1));
    const float lx = interval_gap(fxl, fxh, fadd(g.ox, fmul((float)bx, hb)), hb, g.margin);
    lyb = interval_gap(fyl, fyh, fadd(g.oy, fmul((float)by, hb)), hb, g.margin);
    const float lzb = interval_gap(fzl, fzh, fadd(g.oz, fmul((float)bz, hb)), hb, g.margin);
    lxb2 = fmul(lx, lx);
    if (fadd(slab2, fadd(lxb2, fadd(fmul(lyb, lyb), fmul(lzb, lzb)))) > v.bound()) return false;
  }
  if (slab && rescan_ok<V>()) {
    // The nearest point of a thin sheet lies next to the query's foot on it: the cell under the foot is scanned first, so
    // that the layers and rows below are already cut with a bound within a cell of the final one (counted on the host
    // build: point tests per far query 142 -> 105, row tests 25 -> 17).  Its points are seen again in their row.
    const int fx = clampi(cell_of(fmul(0.5f, fadd(fxl, fxh)), g.ox, g.inv_h) - (bx << 3), 0, 7);
    const int fy = clampi(cell_of(fmul(0.5f, fadd(fyl, fyh)), g.oy, g.inv_h) - (by << 3), 0, 7);
    const int fz = clampi(cell_of(fmul(0.5f, fadd(fzl, fzh)), g.oz, g.inv_h) - (bz << 3), 0, 7);
    const unsigned code = local_code((unsigned)fx, (unsigned)fy, (unsigned)fz);
    const unsigned b0 = ldg(&cs[code]), e0 = ldg(&cs[code + 1]);
    if (b0 < e0 && v.range(b0, e0)) return true;
  }
  const int zc = clampi(q.cz - (bz << 3), 0, 7), yc = clampi(q.cy - (by << 3), 0, 7);
  // layers of cells the foot interval can reach in z under the bound on entry (a later, smaller bound only narrows it)
  int za = 0, zb = 7;
  if (slab && v.bound() < 3.0e38f) {
    const float rz = fadd(sqrt_up(fmax2(fsub(fsub(v.bound(), slab2), fadd(lxb2, fmul(lyb, lyb))), 0.f)), g.margin);
    za = imax2(cell_of(fsub(fzl, rz), g.oz, g.inv_h) - (bz << 3), 0);
    zb = imin2(cell_of(fadd(fzh, rz), g.oz, g.inv_h) - (bz << 3), 7);
  }
  for (int kz = 0; kz < 8; ++kz) {
    const int lz = (zc + kz <= 7) ? zc + kz : 7 - kz;
    if (lz < za || lz > zb) continue;
    const unsigned sb = ldg(&cs[lz << 6]), se = ldg(&cs[(lz << 6) + 64]);
    if (sb == se) continue;
    const float gz = node_gap(q.z, g.oz, (bz << 3) + lz, h, g.margin);
    const float gz2 = fmul(gz, gz);
    if (fadd(gxy2, gz2) > v.bound()) continue;
    float slz2 = gz2;  // s^2 + the foot-to-cells gap in z, squared
    if (slab) {
      const float lzs = interval_gap(fzl, fzh, fadd(g.oz, fmul((float)((bz << 3) + lz), h)), h, g.margin);
      slz2 = fadd(slab2, fmul(lzs, lzs));
      if (fadd(slz2, fadd(lxb2, fmul(lyb, lyb))) > v.bound()) continue;
    }
    int ya = 0, yb = 7;  // rows of this layer the foot interval can reach in y
    if (slab && v.bound() < 3.0e38f) {
      const float ry = fadd(sqrt_up(fmax2(fsub(fsub(v.bound(), slz2), lxb2), 0.f)), g.margin);
      ya = imax2(cell_of(fsub(fyl, ry), g.oy, g.inv_h) - (by << 3), 0);
      yb = imin2(cell_of(fadd(fyh, ry), g.oy, g.inv_h) - (by << 3), 7);
    }
    for (int ky = 0; ky < 8; ++ky) {
      const int ly = (yc + ky <= 7) ? yc + ky : 7 - ky;
      if (ly < ya || ly > yb) continue;
      const unsigned rb = ldg(&cs[(lz << 6) + (ly << 3)]), re = ldg(&cs[(lz << 6) + (ly << 3) + 8]);
      if (rb == re) continue;
      const float gy = node_gap(q.y, g.oy, (by << 3) + ly, h, g.margin);
      const float gyz2 = fadd(fmul(gy, gy), gz2);
      const float bnd = v.bound();
      if (fadd(gx2, gyz2) > bnd) continue;
      float sl2 = 0.f;
      if (slab) {
        const float lyr = interval_gap(fyl, fyh, fadd(g.oy, fmul((float)((by << 3) + ly), h)), h, g.margin);
        sl2 = fadd(slz2, fmul(lyr, lyr));
        if (fadd(sl2, lxb2) > bnd) continue;
      }
      unsigned b = rb, e = re;
      if (bnd < 3.0e38f) {  // cut the row to the chord of the ball at this (y, z), and to the reach of the foot interval
        const float rx = fadd(sqrt_up(fmax2(fsub(bnd, gyz2), 0.f)), g.margin);
        float xlo = fsub(q.x, rx), xhi = fadd(q.x, rx);
        if (slab) {
          const float rw = fadd(sqrt_up(fmax2(fsub(bnd, sl2), 0.f)), g.margin);
          xlo = fmax2(xlo, fsub(fxl, rw));
          xhi = fmin2(xhi, fadd(fxh, rw));
        }
        const int xa = imax2(cell_of(xlo, g.ox, g.inv_h) - (bx << 3), 0);
        const int xb = imin2(cell_of(xhi, g.ox, g.inv_h) - (bx << 3), 7);
        if (xa > xb) continue;
        if (xa > 0) b = ldg(&cs[(lz << 6) + (ly << 3) + xa]);
        if (xb < 7) e = ldg(&cs[(lz << 6) + (ly << 3) + xb + 1]);
        if (b >= e) continue;
      }
      if (v.range(b, e)) return true;
    }
  }
  return false;
}

// the occupied children of one 4x4x4 mask, in Chebyshev rings around the child nearest to the query
template <class V>
GICPB_HD bool visit_superbrick(const GridView& g, const Query& q, int sx, int sy, int sz, V& v) {
  const size_t sbi = ((size_t)sz * g.nsy + sy) * g.nsx + sx;
  unsigned long long occ = ldg(&g.sb_mask[sbi]);
  if (!occ) return false;
  const float size = fmul(g.h, 8.0f);
  if (g.sb_plane != nullptr && v.bound() < 3.0e38f) {
    // Oriented slab of the whole superbrick (see visit_brick): a point p of it with |q - p|^2 <= bound lies, on every axis,
    // within sqrt(bound - s^2) of the foot interval F_i.  Only the bricks that box touches are looked at: for a query far
    // off a thin sheet that is the handful next to its foot instead of every brick the ball's own box covers.
    const float* pl = g.sb_plane + 5 * sbi;
    const float nx = ldg(&pl[0]), ny = ldg(&pl[1]), nz = ldg(&pl[2]), lo = ldg(&pl[3]), hi = ldg(&pl[4]);
    const float nq = plane_dot(nx, ny, nz, q.x, q.y, q.z);
    const float s = fmax2(fsub(fmax2(fsub(nq, hi), fsub(lo, nq)), g.margin), 0.f);
    const float slab2 = fmul(fmul(s, s), 0.999998f);
    const float bnd = v.bound();
    if (slab2 > bnd) return false;
    const float al = fsub(fsub(nq, hi), g.margin), ah = fadd(fsub(nq, lo), g.margin);  // alpha range, widened
    const float x0 = fmul(nx, al), x1 = fmul(nx, ah), y0 = fmul(ny, al), y1 = fmul(ny, ah), z0 = fmul(nz, al), z1 = fmul(nz, ah);
    const float rw = fadd(sqrt_up(fmax2(fsub(bnd, slab2), 0.f)), g.margin);
    const float xl = fsub(fsub(q.x, fmax2(x0, x1)), rw), xh = fadd(fsub(q.x, fmin2(x0, x1)), rw);
    const float yl = fsub(fsub(q.y, fmax2(y0, y1)), rw), yh = fadd(fsub(q.y, fmin2(y0, y1)), rw);
    const float zl = fsub(fsub(q.z, fmax2(z0, z1)), rw), zh = fadd(fsub(q.z, fmin2(z0, z1)), rw);
    // brick coordinates exactly as the build assigns them (clamped cells), relative to the superbrick
    const unsigned xm = range4((clampi(cell_of(xl, g.ox, g.inv_h), 0, g.nx - 1) >> 3) - (sx << 2),
                               (clampi(cell_of(xh, g.ox, g.inv_h), 0, g.nx - 1) >> 3) - (sx << 2));
    const unsigned ym = range4((clampi(cell_of(yl, g.oy, g.inv_h), 0, g.ny - 1) >> 3) - (sy << 2),
                               (clampi(cell_of(yh, g.oy, g.inv_h), 0, g.ny - 1) >> 3) - (sy << 2));
    const unsigned zm = range4((clampi(cell_of(zl, g.oz, g.inv_h), 0, g.nz - 1) >> 3) - (sz << 2),
                               (clampi(cell_of(zh, g.oz, g.inv_h), 0, g.nz - 1) >> 3) - (sz << 2));
    occ &= spans_mask64(xm, ym, zm);
    if (!occ) return false;
  }
  const int px = clampi((q.cx >> 3) - (sx << 2), 0, 3), py = clampi((q.cy >> 3) - (sy << 2), 0, 3),
            pz = clampi((q.cz >> 3) - (sz << 2), 0, 3);
  unsigned long long seen = 0ull;
  for (int r = 0; r < 4; ++r) {
    const unsigned long long box = box_mask64(px, py, pz, r);
    unsigned long long m = occ & box & ~seen;
    seen = box;
    while (m) {
      const int bit = ffs64(m) - 1;
      m &= m - 1ull;
      const int bx = (sx << 2) + (bit & 3), by = (sy << 2) + ((bit >> 2) & 3), bz = (sz << 2) + (bit >> 4);
      const float lb = sq3(node_gap(q.x, g.ox, bx, size, g.margin), node_gap(q.y, g.oy, by, size, g.margin),
                           node_gap(q.z, g.oz, bz, size, g.margin));
      if (lb > v.bound()) continue;
      const int slot = ldg(&g.brick_slot[brick_index(g, bx, by, bz)]);
      if (slot < 0) continue;  // cannot happen for a consistent index
      if (visit_brick(g, q, bx, by, bz, slot, v)) return true;
    }
    if ((occ & ~box) == 0ull) break;
  }
  return false;
}

template <class V>
GICPB_HD bool visit_hyperbrick(const GridView& g, const Query& q, int hx, int hy, int hz, V& v) {
  const unsigned long long occ = ldg(&g.hb_mask[((size_t)hz * g.nhy + hy) * g.nhx + hx]);
  if (!occ) return false;
  const float size = fmul(g.h, 32.0f);
  const int px = clampi((q.cx >> 5) - (hx << 2), 0, 3), py = clampi((q.cy >> 5) - (hy << 2), 0, 3),
            pz = clampi((q.cz >> 5) - (hz << 2), 0, 3);
  unsigned long long seen = 0ull;
  for (int r = 0; r < 4; ++r) {
    const unsigned long long box = box_mask64(px, py, pz, r);
    unsigned long long m = occ & box & ~seen;
    seen = box;
    while (m) {
      const int bit = ffs64(m) - 1;
      m &= m - 1ull;
      const int sx = (hx << 2) + (bit & 3), sy = (hy << 2) + ((bit >> 2) & 3), sz = (hz << 2) + (bit >> 4);
      const float lb = sq3(node_gap(q.x, g.ox, sx, size, g.margin), node_gap(q.y, g.oy, sy, size, g.margin),
                           node_gap(q.z, g.oz, sz, size, g.margin));
      if (lb > v.bound()) continue;
      if (visit_superbrick(g, q, sx, sy, sz, v)) return true;
    }
    if ((occ & ~box) == 0ull) break;
  }
  return false;
}

// Exhaustive, pruned, nearest-first traversal of the whole index: hyperbrick shells around the query, then the
// masks, bricks, slabs and rows.  Visits every point that can be closer than v.bound() (which the visitor tightens
// as it goes), so it is exact by itself whatever was searched before.
template <class V>
GICPB_HD bool far_search(const GridView& g, const Query& q, V& v) {
  const float hh = fmul(g.h, 128.0f);
  const int hx = q.cx >> 7, hy = q.cy >> 7, hz = q.cz >> 7;
  const float lox = fadd(g.ox, fmul((float)hx, hh)), loy = fadd(g.oy, fmul((float)hy, hh)),
              loz = fadd(g.oz, fmul((float)hz, hh));
  // distance from q to the nearest face of its own hyperbrick (0 when q lies outside the grid)
  float mh = fmin2(fmin2(fmin2(q.x - lox, lox + hh - q.x), fmin2(q.y - loy, loy + hh - q.y)),
                   fmin2(q.z - loz, loz + hh - q.z));
  mh = fmax2(mh, 0.0f);
  const int rmax = imax2(imax2(imax2(hx, g.nhx - 1 - hx), imax2(hy, g.nhy - 1 - hy)), imax2(hz, g.nhz - 1 - hz));
  for (int r = 0; r <= rmax; ++r) {
    if (r >= 1) {  // everything closer than (r-1)*hh + mh has been seen
      const float lb = fmax2(fsub(fadd(fmul((float)(r - 1), hh), mh), g.margin), 0.0f);
      if (fmul(lb, lb) > v.bound()) return false;
    }
    int x0 = hx - r, x1 = hx + r, y0 = hy - r, y1 = hy + r, z0 = hz - r, z1 = hz + r;
    const float bnd = v.bound();
    if (bnd < 3.0e38f) {  // cut the shell to the bounding box of the search ball
      const float rad = fadd(sqrt_up(bnd), g.margin);
      x0 = imax2(x0, cell_of(fsub(q.x, rad), g.ox, g.inv_h) >> 7);
      x1 = imin2(x1, cell_of(fadd(q.x, rad), g.ox, g.inv_h) >> 7);
      y0 = imax2(y0, cell_of(fsub(q.y, rad), g.oy, g.inv_h) >> 7);
      y1 = imin2(y1, cell_of(fadd(q.y, rad), g.oy, g.inv_h) >> 7);
      z0 = imax2(z0, cell_of(fsub(q.z, rad), g.oz, g.inv_h) >> 7);
      z1 = imin2(z1, cell_of(fadd(q.z, rad), g.oz, g.inv_h) >> 7);
    }
    x0 = imax2(x0, 0); y0 = imax2(y0, 0); z0 = imax2(z0, 0);
    x1 = imin2(x1, g.nhx - 1); y1 = imin2(y1, g.nhy - 1); z1 = imin2(z1, g.nhz - 1);
    for (int z = z0; z <= z1; ++z) {
      const bool ez = (z - hz == r) || (hz - z == r);
      const float gz = node_gap(q.z, g.oz, z, hh, g.margin);
      for (int y = y0; y <= y1; ++y) {
        const bool ezy = ez || (y - hy == r) || (hy - y == r);
        const float gy = node_gap(q.y, g.oy, y, hh, g.margin);
        const int step = (ezy || r == 0) ? 1 : 2 * r;  // interior rows: only the two x faces of the shell
        for (int x = ezy ? x0 : hx - r; x <= x1; x += step) {
          if (x < x0) continue;
          const float gx = node_gap(q.x, g.ox, x, hh, g.margin);
          if (sq3(gx, gy, gz) > v.bound()) continue;
          if (visit_hyperbrick(g, q, x, y, z, v)) return true;
        }
      }
    }
  }
  return false;
}

// ---- exact nearest neighbour -------------------------------------------------------------------------------------------------------
struct NNState {
  float best;  // best squared distance so far (or the gate^2 / +inf sentinel)
  int pos;     // position in the sorted target array, -1 = none
  int oi;      // original index of the best (sentinel: INT_MAX ungated, -1 gated)
};

template <bool kEarlyExit>
struct NNVisitor {
  static constexpr bool kRescanOk = true;  // a running minimum: a point seen twice changes nothing
  const float4* pts;
  float qx, qy, qz;
  NNState s;
  GICPB_HD float bound() const { return s.best; }
  GICPB_HD bool apply(unsigned i, const float4& p) {
    const float d = dist2(qx, qy, qz, p);
    const int oi = f2i_bits(p.w);
    if (cand_less(d, oi, s.best, s.oi)) {
      s.best = d;
      s.pos = (int)i;
      s.oi = oi;
      if (kEarlyExit) return true;
    }
    return false;
  }
  GICPB_HD bool point(unsigned i) { return apply(i, ldg(&pts[i])); }
  // points i and (if `two`) i + 1, both loads issued before either is used
  GICPB_HD bool point2(unsigned i, bool two) {
    const float4 p0 = ldg(&pts[i]);
    const float4 p1 = ldg(&pts[two ? i + 1 : i]);
    bool stop = apply(i, p0);
    if (two) stop = apply(i + 1, p1) || stop;
    return stop;
  }
  GICPB_HD bool range(unsigned b, unsigned e) {
    unsigned i = b;
    for (; i + 4 <= e; i += 4) {  // four independent loads in flight
      const float4 p0 = ldg(&pts[i]), p1 = ldg(&pts[i + 1]), p2 = ldg(&pts[i + 2]), p3 = ldg(&pts[i + 3]);
      bool stop = apply(i, p0);
      stop = apply(i + 1, p1) || stop;
      stop = apply(i + 2, p2) || stop;
      stop = apply(i + 3, p3) || stop;
      if (kEarlyExit && stop) return true;
    }
    for (; i < e; ++i)
      if (point(i)) return true;
    return false;
  }
};

// ---- range queue: enumerate first, scan later -------------------------------------------------------------------------------------
// A thread that walks cells and scans their points in nested loops keeps its warp waiting on every short loop.  The
// near searches therefore run in two flat phases: the cell walk only QUEUES the point ranges it finds (a handful),
// then one loop scans all queued points back to back.  Entry j of a thread lives at [j * kStride] (shared memory
// columns).  A full queue falls back to scanning the range at once, which is still exact.
template <int kStride, int kCap, class Scan>
struct QueueVisitor {
  unsigned* qb;
  unsigned* qe;
  int n;
  Scan& scan;
  GICPB_HD float bound() const { return scan.bound(); }
  GICPB_HD bool range(unsigned b, unsigned e) {
    if (n < kCap) {
      qb[n * kStride] = b;
      qe[n * kStride] = e;
      ++n;
      return false;
    }
    return scan.range(b, e);
  }
  GICPB_HD bool drain() {  // scan everything queued in one flat loop; true = the scan asked to stop
    int hd = 0;
    unsigned i = 0, e = 0;
    for (;;) {
      if (i >= e) {
        if (hd >= n) break;
        i = qb[hd * kStride];
        e = qe[hd * kStride];
        ++hd;
      }
      const bool two = i + 1 < e;
      if (scan.point2(i, two)) {
        n = 0;
        return true;
      }
      i += two ? 2u : 1u;
    }
    n = 0;
    return false;
  }
};

constexpr int kNear_Done = 0, kNear_Stop = 1, kNear_Far = 2;

// Near part of the exact nearest-neighbour search of (qx,qy,qz).  `s` must be initialised by the caller:
//   ungated: {+inf, -1, INT_MAX};  gated (d2 < gate2 strictly): {gate2, -1, -1};  or a known candidate (seed).
// kEarlyExit: stop as soon as ANY candidate beats the initial state (cloud difference) -> kNear_Stop.
// A candidate (seed) whose ball cuts few cells is refined by searching those cells as a plain box.  Otherwise the
// query's own cell, then the cell rings 1..rings around it, are probed for a (better) first candidate, whose ball is
// then searched -> kNear_Done.  When nothing turns up nearby, or the ball still spans too many rows, the answer is
// kNear_Far: the caller must run far_search (exact by itself) for this query.
template <bool kEarlyExit, int kStride, int kCap>
GICPB_HD int nn_near(const GridView& g, const Query& q, NNState& s, unsigned* qb, unsigned* qe, int rings = kNearMaxRing) {
  NNVisitor<kEarlyExit> v{g.pts, q.x, q.y, q.z, s};
  QueueVisitor<kStride, kCap, NNVisitor<kEarlyExit>> qv{qb, qe, 0, v};
  int result = kNear_Far;
  bool probed = false;
  for (;;) {
    if (v.s.pos >= 0) {  // a candidate bounds the ball: search the cells it cuts, if they are few
      const float rad = fadd(sqrt_up(v.s.best), g.margin);
      const int x0 = imax2(cell_of(fsub(q.x, rad), g.ox, g.inv_h), 0), x1 = imin2(cell_of(fadd(q.x, rad), g.ox, g.inv_h), g.nx - 1);
      const int y0 = imax2(cell_of(fsub(q.y, rad), g.oy, g.inv_h), 0), y1 = imin2(cell_of(fadd(q.y, rad), g.oy, g.inv_h), g.ny - 1);
      const int z0 = imax2(cell_of(fsub(q.z, rad), g.oz, g.inv_h), 0), z1 = imin2(cell_of(fadd(q.z, rad), g.oz, g.inv_h), g.nz - 1);
      if (x0 > x1 || y0 > y1 || z0 > z1) { result = kNear_Done; break; }  // the ball misses the grid: the candidate stands
      // A seed is searched directly only when its ball is small; a mediocre one (a match of a pose that has moved on)
      // is cheaper to improve first by probing the cells around the query than to scan its whole ball.
      if ((long long)(y1 - y0 + 1) * (z1 - z0 + 1) <= (probed ? kMaxBoxRows : kSeedBoxRows)) {
        bool stop = visit_box(g, q, x0, x1, y0, y1, z0, z1, qv);
        stop = stop || qv.drain();
        result = stop ? kNear_Stop : kNear_Done;
        break;
      }
    }
    if (probed) break;  // nothing (better) nearby: the far search takes over
    // No candidate yet, or only a poor one (a seed from a pose that has moved on): probe the query's own cell, then
    // the 3x3x3 block, then the cell shells 2..rings around it, until something closer turns up.
    probed = true;
    const int start_pos = v.s.pos;
    if (visit_run(g, q.cx, q.cx, q.cy, q.cz, v)) { result = kNear_Stop; break; }
    bool stop = false;
    for (int R = 1; R <= rings && v.s.pos == start_pos && !stop; ++R) {
      if (R == 1)
        stop = visit_box(g, q, imax2(q.cx - 1, 0), imin2(q.cx + 1, g.nx - 1), imax2(q.cy - 1, 0),
                         imin2(q.cy + 1, g.ny - 1), imax2(q.cz - 1, 0), imin2(q.cz + 1, g.nz - 1), qv);
      else
        stop = visit_shell(g, q, R, qv);
      stop = stop || qv.drain();
    }
    if (stop) { result = kNear_Stop; break; }
    if (v.s.pos < 0) break;  // nothing nearby at all: the far search takes over
  }
  s = v.s;
  return result;
}

// far part: the hierarchical traversal from the caller's initial state (it does not need what nn_near found)
template <bool kEarlyExit>
GICPB_HD bool nn_far(const GridView& g, const Query& q, NNState& s) {
  NNVisitor<kEarlyExit> v{g.pts, q.x, q.y, q.z, s};
  const bool stop = far_search(g, q, v);
  s = v.s;
  return stop;
}

#if defined(__CUDACC__)
// ---- block-level reduction of doubles (sum), result valid in thread 0 --------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFullMask, v, o);
  return v;
}
#endif

}  // namespace gicpb
