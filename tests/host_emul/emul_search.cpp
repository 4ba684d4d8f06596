// emul_search.cpp - host build of the index traversal code (csrc/common.cuh, csrc/knn_search.cuh) checked against
// brute force.  TEST INFRASTRUCTURE ONLY: it exists so the traversal logic (box search, hierarchical far search,
// kNN rings, tie rules, pruning margins) can be verified without a GPU; the shipped library has no host search.
// The index arrays are built here by a plain CPU restatement of grid_build.cu's layout.
//
// build: g++ -std=c++17 -O2 -ffp-contract=off -I../../leica_point_cloud_processing_b200/csrc emul_search.cpp
#include <algorithm>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <random>
#include <string>
#include <vector>

#include "knn_search.cuh"

using namespace gicpb;

struct HostIndex {
  std::vector<float4> pts;
  std::vector<int> brick_slot;
  std::vector<uint32_t> cell_start;
  std::vector<unsigned long long> sb, hb;
  std::vector<int> pos_of;
  std::vector<float> plane, sb_plane;
  GridView g{};
};

static void build_index(const std::vector<float3>& in, float h, HostIndex& ix) {
  float bmin[3] = {1e30f, 1e30f, 1e30f}, bmax[3] = {-1e30f, -1e30f, -1e30f};
  for (auto& p : in) {
    const float c[3] = {p.x, p.y, p.z};
    for (int a = 0; a < 3; ++a) { bmin[a] = std::min(bmin[a], c[a]); bmax[a] = std::max(bmax[a], c[a]); }
  }
  float max_abs = 0;
  int dims[3], bd[3];
  for (int a = 0; a < 3; ++a) {
    max_abs = std::max(max_abs, std::max(std::fabs(bmin[a]), std::fabs(bmax[a])));
    dims[a] = (int)std::floor((bmax[a] - bmin[a]) / h) + 1;
    bd[a] = (dims[a] + 7) / 8;
    dims[a] = bd[a] * 8;
  }
  GridView& g = ix.g;
  g.ox = bmin[0]; g.oy = bmin[1]; g.oz = bmin[2];
  g.h = h; g.inv_h = 1.0f / h;
  const int maxdim = std::max(dims[0], std::max(dims[1], dims[2]));
  g.margin = h * (0.002f + 5e-7f * (float)maxdim) + 4e-6f * max_abs;
  g.nx = dims[0]; g.ny = dims[1]; g.nz = dims[2];
  g.nbx = bd[0]; g.nby = bd[1]; g.nbz = bd[2];
  g.bsx = 1; g.bsy = bd[0]; g.bsz = bd[0] * bd[1];
  g.bo0 = 0; g.bo1 = 1; g.bo2 = 2;
  g.nsx = (bd[0] + 3) / 4; g.nsy = (bd[1] + 3) / 4; g.nsz = (bd[2] + 3) / 4;
  g.nhx = (g.nsx + 3) / 4; g.nhy = (g.nsy + 3) / 4; g.nhz = (g.nsz + 3) / 4;
  g.n = (int)in.size();
  const int n = g.n;
  std::vector<std::pair<uint32_t, int>> kv(n);
  for (int i = 0; i < n; ++i) {
    const int cx = clampi(cell_of(in[i].x, g.ox, g.inv_h), 0, g.nx - 1);
    const int cy = clampi(cell_of(in[i].y, g.oy, g.inv_h), 0, g.ny - 1);
    const int cz = clampi(cell_of(in[i].z, g.oz, g.inv_h), 0, g.nz - 1);
    const uint32_t b = (uint32_t)brick_index(g, cx >> 3, cy >> 3, cz >> 3);
    kv[i] = {b * 512u + local_code(cx & 7, cy & 7, cz & 7), i};
  }
  std::stable_sort(kv.begin(), kv.end(), [](auto& a, auto& b) { return a.first < b.first; });
  ix.pts.resize(n);
  ix.pos_of.assign(n, -1);
  for (int i = 0; i < n; ++i) {
    const float3& p = in[kv[i].second];
    ix.pts[i] = float4{p.x, p.y, p.z, i2f_bits(kv[i].second)};
    ix.pos_of[kv[i].second] = i;
  }
  ix.brick_slot.assign((size_t)bd[0] * bd[1] * bd[2], -1);
  ix.sb.assign((size_t)g.nsx * g.nsy * g.nsz, 0ull);
  ix.hb.assign((size_t)g.nhx * g.nhy * g.nhz, 0ull);
  int n_slots = 0;
  std::vector<int> slot_of(n);
  for (int i = 0; i < n; ++i) {
    const int b = (int)(kv[i].first >> 9);
    if (i == 0 || (int)(kv[i - 1].first >> 9) != b) {
      ix.brick_slot[b] = n_slots++;
      const int bx = b % g.nbx, by = (b / g.nbx) % g.nby, bz = b / (g.nbx * g.nby);
      const int sx = bx >> 2, sy = by >> 2, sz = bz >> 2;
      ix.sb[((size_t)sz * g.nsy + sy) * g.nsx + sx] |= 1ull << (((bz & 3) << 4) | ((by & 3) << 2) | (bx & 3));
      ix.hb[((size_t)(sz >> 2) * g.nhy + (sy >> 2)) * g.nhx + (sx >> 2)] |= 1ull << (((sz & 3) << 4) | ((sy & 3) << 2) | (sx & 3));
    }
    slot_of[i] = n_slots - 1;
  }
  ix.cell_start.assign((size_t)n_slots * 512 + 1, 0xdeadbeefu);
  // same fill rule as cell_start_kernel
  for (int i = 0; i < n; ++i) {
    const uint32_t c = kv[i].first & 511u;
    uint32_t* cs = ix.cell_start.data() + (size_t)slot_of[i] * 512;
    if (i == 0) {
      for (uint32_t code = 0; code <= c; ++code) cs[code] = 0;
    } else if (slot_of[i] == slot_of[i - 1]) {
      for (uint32_t code = (kv[i - 1].first & 511u) + 1; code <= c; ++code) cs[code] = i;
    } else {
      uint32_t* csp = cs - 512;
      for (uint32_t code = (kv[i - 1].first & 511u) + 1; code < 512; ++code) csp[code] = i;
      for (uint32_t code = 0; code <= c; ++code) cs[code] = i;
    }
    if (i == n - 1) for (uint32_t code = c + 1; code <= 512; ++code) cs[code] = n;
  }
  for (auto v : ix.cell_start) if (v == 0xdeadbeefu) { printf("cell_start entry not written\n"); exit(2); }
  g.pts = ix.pts.data();
  g.brick_slot = ix.brick_slot.data();
  g.cell_start = ix.cell_start.data();
  g.pos_of = ix.pos_of.data();
  g.sb_mask = ix.sb.data();
  g.hb_mask = ix.hb.data();
  // oriented slab per brick, as brick_plane_kernel builds it: PCA normal, extremes of plane_dot over the brick's points.
  // Every third brick gets an arbitrary (non-normal) direction instead: any direction must leave the search exact.
  ix.plane.assign((size_t)n_slots * 5, 0.f);
  std::vector<double> acc((size_t)n_slots * 10, 0.0);
  for (int i = 0; i < n; ++i) {
    double* a = &acc[(size_t)slot_of[i] * 10];
    const float4& p = ix.pts[i];
    a[0] += 1; a[1] += p.x; a[2] += p.y; a[3] += p.z;
    a[4] += (double)p.x * p.x; a[5] += (double)p.x * p.y; a[6] += (double)p.x * p.z;
    a[7] += (double)p.y * p.y; a[8] += (double)p.y * p.z; a[9] += (double)p.z * p.z;
  }
  for (int sl = 0; sl < n_slots; ++sl) {
    const double* a = &acc[(size_t)sl * 10];
    const double m = a[0], mx = a[1] / m, my = a[2] / m, mz = a[3] / m;
    double A[3][3] = {{a[4] / m - mx * mx, a[5] / m - mx * my, a[6] / m - mx * mz}, {0, a[7] / m - my * my, a[8] / m - my * mz}, {0, 0, a[9] / m - mz * mz}};
    A[1][0] = A[0][1]; A[2][0] = A[0][2]; A[2][1] = A[1][2];
    double V[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
    for (int sweep = 0; sweep < 30; ++sweep)
      for (int p = 0; p < 2; ++p)
        for (int q2 = p + 1; q2 < 3; ++q2) {
          if (std::fabs(A[p][q2]) < 1e-300) continue;
          const double th = (A[q2][q2] - A[p][p]) / (2 * A[p][q2]);
          const double tt = (th >= 0 ? 1 : -1) / (std::fabs(th) + std::sqrt(th * th + 1));
          const double c = 1 / std::sqrt(tt * tt + 1), s2 = tt * c;
          for (int k = 0; k < 3; ++k) { const double akp = A[k][p], akq = A[k][q2]; A[k][p] = c * akp - s2 * akq; A[k][q2] = s2 * akp + c * akq; }
          for (int k = 0; k < 3; ++k) { const double apk = A[p][k], aqk = A[q2][k]; A[p][k] = c * apk - s2 * aqk; A[q2][k] = s2 * apk + c * aqk; }
          for (int k = 0; k < 3; ++k) { const double vkp = V[k][p], vkq = V[k][q2]; V[k][p] = c * vkp - s2 * vkq; V[k][q2] = s2 * vkp + c * vkq; }
        }
    int best = 0;
    for (int k = 1; k < 3; ++k) if (std::fabs(A[k][k]) < std::fabs(A[best][best])) best = k;
    float* pl = &ix.plane[(size_t)sl * 5];
    pl[0] = (float)V[0][best]; pl[1] = (float)V[1][best]; pl[2] = (float)V[2][best];
    if (sl % 3 == 1) { pl[0] = 0.6f; pl[1] = -0.48f; pl[2] = 0.64f; }
    if (!(std::fabs(pl[0]) + std::fabs(pl[1]) + std::fabs(pl[2]) > 0.5f)) { pl[0] = 0; pl[1] = 0; pl[2] = 1; }
    pl[3] = inf(); pl[4] = -inf();
  }
  for (int i = 0; i < n; ++i) {
    float* pl = &ix.plane[(size_t)slot_of[i] * 5];
    const float4& p = ix.pts[i];
    const float d = plane_dot(pl[0], pl[1], pl[2], p.x, p.y, p.z);
    pl[3] = std::min(pl[3], d); pl[4] = std::max(pl[4], d);
  }
  g.brick_plane = ix.plane.data();
  // the same slab per SUPERBRICK (sb_plane_kernel): the direction of the superbrick's first occupied brick (for a sheet
  // that is close to the superbrick's own PCA normal; every third superbrick keeps an arbitrary direction: any unit
  // vector must leave the search exact), extremes of plane_dot over all points of the superbrick
  const size_t n_sb = (size_t)g.nsx * g.nsy * g.nsz;
  ix.sb_plane.assign(n_sb * 5, 0.f);
  for (size_t b = 0; b < n_sb; ++b) { float* pl = &ix.sb_plane[b * 5]; pl[2] = 1.f; pl[3] = inf(); pl[4] = -inf(); }
  std::vector<char> sb_has(n_sb, 0);
  auto sb_of = [&](int i) {
    const int b = (int)(kv[i].first >> 9);
    const int bx = b % g.nbx, by = (b / g.nbx) % g.nby, bz = b / (g.nbx * g.nby);
    return ((size_t)(bz >> 2) * g.nsy + (by >> 2)) * g.nsx + (bx >> 2);
  };
  for (int i = 0; i < n; ++i) {
    const size_t b = sb_of(i);
    if (sb_has[b]) continue;
    sb_has[b] = 1;
    float* pl = &ix.sb_plane[b * 5];
    const float* bp = &ix.plane[(size_t)slot_of[i] * 5];
    pl[0] = bp[0]; pl[1] = bp[1]; pl[2] = bp[2];
    if (b % 3 == 2) { pl[0] = -0.36f; pl[1] = 0.8f; pl[2] = 0.48f; }
  }
  for (int i = 0; i < n; ++i) {
    float* pl = &ix.sb_plane[sb_of(i) * 5];
    const float4& p = ix.pts[i];
    const float d = plane_dot(pl[0], pl[1], pl[2], p.x, p.y, p.z);
    pl[3] = std::min(pl[3], d); pl[4] = std::max(pl[4], d);
  }
  g.sb_plane = ix.sb_plane.data();
}

static long g_fail = 0, g_checks = 0, g_far = 0, g_knn_far = 0;
static bool mode_far_only = false;

static void brute_nn(const HostIndex& ix, float qx, float qy, float qz, NNState& s) {
  for (int i = 0; i < ix.g.n; ++i) {
    const float d = dist2(qx, qy, qz, ix.pts[i]);
    const int oi = f2i_bits(ix.pts[i].w);
    if (cand_less(d, oi, s.best, s.oi)) { s.best = d; s.pos = i; s.oi = oi; }
  }
}

// kCap: the queue length of the near searches (QueueVisitor).  The library's own caps (common.cuh), or 1, which sends every
// range through the overflow path (drain before the next range is queued).
template <int kCap>
static void check_nn(const HostIndex& ix, float qx, float qy, float qz, float gate2, int seed_pos, const char* what) {
  NNState a, b;
  if (gate2 > 0) { a.best = gate2; a.pos = -1; a.oi = -1; } else { a.best = inf(); a.pos = -1; a.oi = INT_MAX; }
  b = a;
  if (seed_pos >= 0) {
    const float d = dist2(qx, qy, qz, ix.pts[seed_pos]);
    const int oi = f2i_bits(ix.pts[seed_pos].w);
    if (cand_less(d, oi, a.best, a.oi)) { a.best = d; a.pos = seed_pos; a.oi = oi; }
  }
  const NNState a0 = a;
  unsigned qb[kCap], qe[kCap];
  const Query q = make_query(ix.g, qx, qy, qz);
  const int near = nn_near<false, 1, kCap>(ix.g, q, a, qb, qe);
  if (near == kNear_Far) { a = a0; nn_far<false>(ix.g, q, a); ++g_far; }
  if (mode_far_only) { a = a0; nn_far<false>(ix.g, q, a); }
  brute_nn(ix, qx, qy, qz, b);
  ++g_checks;
  if (a.pos != b.pos || a.oi != b.oi || f2i_bits(a.best) != f2i_bits(b.best)) {
    if (g_fail < 10) printf("NN mismatch (%s) q=(%g,%g,%g) got pos %d oi %d d %g, want pos %d oi %d d %g\n", what, qx, qy, qz,
                            a.pos, a.oi, a.best, b.pos, b.oi, b.best);
    ++g_fail;
  }
  // early-exit flavour (cloud difference): "is anything closer than thr" must agree with brute force
  if (gate2 > 0) {
    NNState e; e.best = gate2; e.pos = -1; e.oi = -1;
    const NNState e0 = e;
    const int r = nn_near<true, 1, kCap>(ix.g, q, e, qb, qe);
    bool hit = r == kNear_Stop;
    if (r == kNear_Far) { e = e0; hit = nn_far<true>(ix.g, q, e); }
    ++g_checks;
    if (hit != (b.pos >= 0)) { if (g_fail < 10) printf("early-exit mismatch (%s)\n", what); ++g_fail; }
  }
}

template <int kCap>
static void check_knn(const HostIndex& ix, int i, int k) {
  std::vector<unsigned long long> lk(k);
  KnnVisitor<1> v;
  v.pts = ix.pts.data(); v.lkey = lk.data(); v.k = k;
  const float4 q = ix.pts[i];
  v.qx = q.x; v.qy = q.y; v.qz = q.z;
  unsigned qb[kCap], qe[kCap];
  const Query qq = make_query(ix.g, q.x, q.y, q.z);
  if (mode_far_only || !knn_near<1, kCap>(ix.g, qq, v, qb, qe)) { knn_far(ix.g, qq, v); ++g_knn_far; }
  std::vector<std::pair<std::pair<float, int>, int>> all(ix.g.n);
  for (int j = 0; j < ix.g.n; ++j) all[j] = {{dist2(q.x, q.y, q.z, ix.pts[j]), f2i_bits(ix.pts[j].w)}, j};
  const int kk = std::min(k, ix.g.n);
  std::partial_sort(all.begin(), all.begin() + kk, all.end());
  ++g_checks;
  bool ok = v.count == kk;
  for (int j = 0; ok && j < kk; ++j) ok = ix.g.pos_of[v.oi_at(j)] == all[j].second && v.oi_at(j) == all[j].first.second && v.d2_at(j) == all[j].first.first;
  if (!ok) { if (g_fail < 10) printf("kNN mismatch at sorted point %d (count %d)\n", i, v.count); ++g_fail; }
}

// Every point set of run() is moved by offset * (1, -0.5, 0.25): far from the origin the grid margin (4e-6 |x|) widens and
// the near searches hand more queries to the far traversal.
template <int kNnCap, int kKnnCap>
static void run(float offset);

int main(int argc, char** argv) {
  // far: answer every query with the hierarchical traversal alone; cap1: queues of one entry; offset=X: see run()
  bool cap1 = false;
  float offset = 0.f;
  for (int a = 1; a < argc; ++a) {
    const std::string s = argv[a];
    if (s == "far") mode_far_only = true;
    else if (s == "cap1") cap1 = true;
    else if (s.rfind("offset=", 0) == 0) offset = std::strtof(s.c_str() + 7, nullptr);
    else { printf("unknown argument %s\n", s.c_str()); return 2; }
  }
  if (cap1) run<1, 1>(offset);
  else run<kNnQueueCap, kKnnQueueCap>(offset);
  printf("%ld checks, %ld failures (%ld NN and %ld kNN queries went through the far traversal)\n", g_checks, g_fail, g_far,
         g_knn_far);
  return g_fail ? 1 : 0;
}

template <int kNnCap, int kKnnCap>
static void run(float offset) {
  std::mt19937 rng(12345);
  std::uniform_real_distribution<float> U(0.f, 1.f);
  std::normal_distribution<float> N(0.f, 1.f);
  for (int scenario = 0; scenario < 10; ++scenario) {
    std::vector<float3> pts;
    float h = 0.05f;
    const char* name = "";
    if (scenario == 0) {  // curved sheet, like the bench panel
      name = "sheet";
      for (int i = 0; i < 20000; ++i) { float u = U(rng) * 4, s = U(rng) * 2; pts.push_back({u, s, 0.3f * std::sin(u) * std::cos(2 * s) + 0.001f * N(rng)}); }
      h = 0.035f;
    } else if (scenario == 1) {  // integer lattice: many exact distance ties
      name = "lattice";
      for (int x = 0; x < 14; ++x) for (int y = 0; y < 14; ++y) for (int z = 0; z < 14; ++z) pts.push_back({0.1f * x, 0.1f * y, 0.1f * z});
      h = 0.13f;
    } else if (scenario == 2) {  // volume + duplicates
      name = "volume+dups";
      for (int i = 0; i < 6000; ++i) pts.push_back({U(rng), U(rng), U(rng)});
      for (int i = 0; i < 500; ++i) pts.push_back(pts[i * 7]);
      h = 0.08f;
    } else if (scenario == 3) {  // two far-apart clusters and isolated outliers: hierarchy + sparse kNN fallback
      name = "clusters";
      for (int i = 0; i < 4000; ++i) pts.push_back({0.05f * N(rng), 0.05f * N(rng), 0.05f * N(rng)});
      for (int i = 0; i < 4000; ++i) pts.push_back({30.f + 0.05f * N(rng), 10.f + 0.05f * N(rng), -5.f + 0.05f * N(rng)});
      for (int i = 0; i < 30; ++i) pts.push_back({30.f * U(rng), 10.f * U(rng), -5.f * U(rng)});
      h = 0.02f;
    } else if (scenario == 4) {  // tiny cloud
      name = "tiny";
      for (int i = 0; i < 37; ++i) pts.push_back({U(rng), U(rng), U(rng)});
      h = 0.3f;
    } else if (scenario == 5) {  // all points identical except a few
      name = "degenerate";
      for (int i = 0; i < 300; ++i) pts.push_back({1.f, 2.f, 3.f});
      for (int i = 0; i < 40; ++i) pts.push_back({1.f + U(rng), 2.f, 3.f});
      h = 0.01f;
    } else if (scenario == 7) {  // thin sheet tilted against all three axes: the regime of the oriented brick slabs
      name = "tilted sheet";
      for (int i = 0; i < 30000; ++i) {
        const float a = U(rng) * 3 - 1.5f, b = U(rng) * 2 - 1.0f;
        pts.push_back({a + 0.31f * b, 0.93f * b - 0.2f * a, 0.37f * a + 0.29f * b + 0.0002f * N(rng)});
      }
      h = 0.02f;
    } else if (scenario == 8) {  // two parallel sheets 3 cells apart plus a step: slabs that are NOT thin
      name = "double sheet";
      for (int i = 0; i < 30000; ++i) {
        const float a = U(rng) * 2, b = U(rng) * 2;
        pts.push_back({a, b, (i & 1 ? 0.06f : 0.0f) + (a > 1.0f ? 0.15f : 0.0f) + 0.0005f * N(rng)});
      }
      h = 0.02f;
    } else if (scenario == 9) {  // lattice of spacing 2^-6 on cells of that edge, points one float either side of the faces
      name = "face ulps";
      for (int x = 0; x < 16; ++x) for (int y = 0; y < 16; ++y) for (int z = 0; z < 16; ++z)
        pts.push_back({0.015625f * x, 0.015625f * y, 0.015625f * z});
      h = 0.015625f;
    } else {  // cube faces (reference fixture shape), coarse cells
      name = "cube";
      for (int i = 0; i < 5000; ++i) {
        float a = 2 * U(rng) - 1, b = 2 * U(rng) - 1; int f = rng() % 6;
        float3 p = f == 0 ? float3{a, b, 1} : f == 1 ? float3{a, b, -1} : f == 2 ? float3{a, 1, b} : f == 3 ? float3{a, -1, b} : f == 4 ? float3{1, a, b} : float3{-1, a, b};
        pts.push_back(p);
      }
      h = 0.12f;
    }
    for (auto& p : pts) {
      p.x += offset;
      p.y -= 0.5f * offset;
      p.z += 0.25f * offset;
    }
    if (scenario == 9)  // after the offset: one float of the coordinate where it is, in turn up, down or not at all
      for (size_t i = 0; i < pts.size(); ++i) {
        float* c = (i / 3) % 3 == 0 ? &pts[i].x : ((i / 3) % 3 == 1 ? &pts[i].y : &pts[i].z);
        if (i % 3 == 1) *c = std::nextafter(*c, INFINITY);
        if (i % 3 == 2) *c = std::nextafter(*c, -INFINITY);
      }
    HostIndex ix;
    build_index(pts, h, ix);
    const GridView& g = ix.g;
    const long fail0 = g_fail;
    const float ext = std::max(g.nx, std::max(g.ny, g.nz)) * g.h;
    for (int t = 0; t < 3000; ++t) {
      float qx, qy, qz;
      const int mode = t % 6;
      const float3& p = pts[rng() % pts.size()];
      if (mode == 0) { qx = p.x + 0.2f * h * N(rng); qy = p.y + 0.2f * h * N(rng); qz = p.z + 0.2f * h * N(rng); }       // near
      else if (mode == 1) { qx = p.x + 3 * h * N(rng); qy = p.y + 3 * h * N(rng); qz = p.z + 3 * h * N(rng); }          // a few cells off
      else if (mode == 2) { qx = p.x + 40 * h * N(rng); qy = p.y + 40 * h * N(rng); qz = p.z + 40 * h * N(rng); }       // far
      else if (mode == 3) { qx = g.ox + ext * (3 * U(rng) - 1); qy = g.oy + ext * (3 * U(rng) - 1); qz = g.oz + ext * (3 * U(rng) - 1); }  // anywhere, also outside
      else if (mode == 4) { qx = p.x; qy = p.y; qz = p.z; }                                                               // exactly on a point
      else { qx = p.x + 0.5f * h; qy = p.y; qz = p.z; }
      check_nn<kNnCap>(ix, qx, qy, qz, 0.f, -1, name);
      check_nn<kNnCap>(ix, qx, qy, qz, (2.5f * h) * (2.5f * h), -1, name);
      check_nn<kNnCap>(ix, qx, qy, qz, (60.f * h) * (60.f * h), -1, name);
      check_nn<kNnCap>(ix, qx, qy, qz, 0.f, (int)(rng() % pts.size()), name);           // random (bad) seed
      check_nn<kNnCap>(ix, qx, qy, qz, (60.f * h) * (60.f * h), (int)(rng() % pts.size()), name);
    }
    const int n = (int)pts.size();
    for (int t = 0; t < 1500; ++t) check_knn<kKnnCap>(ix, (int)(rng() % pts.size()), std::min(20, n));
    for (const int k : {2, 3, 31, 32})
      for (int t = 0; t < 200; ++t) check_knn<kKnnCap>(ix, (int)(rng() % pts.size()), std::min(k, n));
    printf("scenario %-12s n=%6d grid %dx%dx%d bricks %dx%dx%d: %s\n", name, g.n, g.nx, g.ny, g.nz, g.nbx, g.nby, g.nbz,
           g_fail == fail0 ? "ok" : "FAILED");
  }
}
