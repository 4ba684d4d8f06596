// cost.cu - one evaluation of the GICP objective and its gradient sums over all correspondences.
//
// Replaces pcl::GeneralizedIterativeClosestPoint::OptimizationFunctorWithIndices::operator() / df / fdf
// (PCL 1.8.1 gicp.hpp), called by the BFGS line search inside gicp_.align() (reference
// src/GICPAlignment.cpp:96).  Per pair i:  pp = T * p_src (float);  res = double(pp - p_tgt) (float subtraction,
// as PCL);  t = M_i res;  f += res.t;  g_t += t;  Rsum += p_src t^T.  The 13 sums (+ the pair count) are reduced
// with warp shuffles, a shared-memory block tree and a last-block pass over the per-block partials, in a fixed
// order, so a given input always produces the same bits.  The host scales by 1/m, 2/m and applies
// computeRDerivative.  FP32 transform + FP64 accumulate: no dense contraction, tensor cores do not apply.
//
// Algorithmic bytes per pair: 16 (p_src float4) + 16 (p_tgt float4) + 48 (M, 6 doubles) or 24 (6 floats).
#include <algorithm>
#include <cstdlib>

#include "kernels.hpp"

namespace gicpb {

namespace {

constexpr int kCostThreads = 256;          // one pair per thread and tile
constexpr int kCostWarps = kCostThreads / 32;
constexpr int kCostStages = 2;             // shared-memory ring: 2 x 256 pairs x 80 B = 40 KB per CTA, 2 CTAs per SM

template <typename MT>
struct PairData {
  float4 q, p;
  MT m[6];
};

template <typename MT>
__device__ __forceinline__ void load_pair(const float4* __restrict__ src, const float4* __restrict__ pair_tgt,
                                          const MT* __restrict__ maha, int lo, int t, PairData<MT>& d) {
  d.q = __ldg(&pair_tgt[t]);
  d.p = __ldg(&src[lo + t]);
  const MT* m = maha + 6 * (size_t)t;
  if (sizeof(MT) == 8) {  // 48 B per pair, 16-byte aligned: three 128-bit loads
    const double2* m2 = reinterpret_cast<const double2*>(m);
    const double2 a = __ldg(m2), b = __ldg(m2 + 1), c = __ldg(m2 + 2);
    d.m[0] = (MT)a.x; d.m[1] = (MT)a.y; d.m[2] = (MT)b.x; d.m[3] = (MT)b.y; d.m[4] = (MT)c.x; d.m[5] = (MT)c.y;
  } else {                // 24 B per pair, 8-byte aligned: three 64-bit loads
    const float2* m2 = reinterpret_cast<const float2*>(m);
    const float2 a = __ldg(m2), b = __ldg(m2 + 1), c = __ldg(m2 + 2);
    d.m[0] = (MT)a.x; d.m[1] = (MT)a.y; d.m[2] = (MT)b.x; d.m[3] = (MT)b.y; d.m[4] = (MT)c.x; d.m[5] = (MT)c.y;
  }
}

// the same pair out of a shared-memory stage (rows of 16 / 16 / 6*sizeof(MT) bytes; 128-bit reads of the 48-byte M rows
// are conflict-free: the 8 lanes of a quarter warp start at banks 0 12 24 4 16 28 8 20)
template <typename MT>
__device__ __forceinline__ void load_pair_smem(const unsigned char* stage, int i, PairData<MT>& d) {
  d.q = *reinterpret_cast<const float4*>(stage + i * 16);
  d.p = *reinterpret_cast<const float4*>(stage + kCostThreads * 16 + i * 16);
  const unsigned char* m = stage + kCostThreads * 32 + i * (6 * (int)sizeof(MT));
  if (sizeof(MT) == 8) {
    const double2* m2 = reinterpret_cast<const double2*>(m);
    const double2 a = m2[0], b = m2[1], c = m2[2];
    d.m[0] = (MT)a.x; d.m[1] = (MT)a.y; d.m[2] = (MT)b.x; d.m[3] = (MT)b.y; d.m[4] = (MT)c.x; d.m[5] = (MT)c.y;
  } else {
    const float2* m2 = reinterpret_cast<const float2*>(m);
    const float2 a = m2[0], b = m2[1], c = m2[2];
    d.m[0] = (MT)a.x; d.m[1] = (MT)a.y; d.m[2] = (MT)b.x; d.m[3] = (MT)b.y; d.m[4] = (MT)c.x; d.m[5] = (MT)c.y;
  }
}

// the same with explicit row bases (q rows, p rows, M rows), for stages and resident blocks of any capacity
template <typename MT>
__device__ __forceinline__ void load_pair_smem_at(const unsigned char* qrows, const unsigned char* prows,
                                                  const unsigned char* mrows, int i, PairData<MT>& d) {
  d.q = *reinterpret_cast<const float4*>(qrows + i * 16);
  d.p = *reinterpret_cast<const float4*>(prows + i * 16);
  const unsigned char* m = mrows + i * (6 * (int)sizeof(MT));
  if (sizeof(MT) == 8) {
    const double2* m2 = reinterpret_cast<const double2*>(m);
    const double2 a = m2[0], b = m2[1], c = m2[2];
    d.m[0] = (MT)a.x; d.m[1] = (MT)a.y; d.m[2] = (MT)b.x; d.m[3] = (MT)b.y; d.m[4] = (MT)c.x; d.m[5] = (MT)c.y;
  } else {
    const float2* m2 = reinterpret_cast<const float2*>(m);
    const float2 a = m2[0], b = m2[1], c = m2[2];
    d.m[0] = (MT)a.x; d.m[1] = (MT)a.y; d.m[2] = (MT)b.x; d.m[3] = (MT)b.y; d.m[4] = (MT)c.x; d.m[5] = (MT)c.y;
  }
}

template <typename MT>
__device__ __forceinline__ void add_pair(const PairData<MT>& d, const Rigid& T, double (&acc)[kCostSums]) {
  if (d.q.w == 0.f) return;  // no correspondence inside the gate
  const double m00 = (double)d.m[0], m01 = (double)d.m[1], m02 = (double)d.m[2];
  const double m11 = (double)d.m[3], m12 = (double)d.m[4], m22 = (double)d.m[5];
  const float3 pp = xform(T, d.p.x, d.p.y, d.p.z);
  const double r0 = (double)__fsub_rn(pp.x, d.q.x);
  const double r1 = (double)__fsub_rn(pp.y, d.q.y);
  const double r2 = (double)__fsub_rn(pp.z, d.q.z);
  const double t0 = m00 * r0 + m01 * r1 + m02 * r2;
  const double t1 = m01 * r0 + m11 * r1 + m12 * r2;
  const double t2 = m02 * r0 + m12 * r1 + m22 * r2;
  acc[0] += r0 * t0 + r1 * t1 + r2 * t2;
  acc[1] += t0;
  acc[2] += t1;
  acc[3] += t2;
  const double p0 = (double)d.p.x, p1 = (double)d.p.y, p2 = (double)d.p.z;
  acc[4] += p0 * t0;  acc[5] += p0 * t1;  acc[6] += p0 * t2;
  acc[7] += p1 * t0;  acc[8] += p1 * t1;  acc[9] += p1 * t2;
  acc[10] += p2 * t0; acc[11] += p2 * t1; acc[12] += p2 * t2;
  acc[13] += 1.0;
}

// ---- bulk asynchronous copies (TMA, 1-D) into shared memory, completion counted in bytes on an mbarrier -------------------
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned arrivals) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(arrivals));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ uint4 ld_volatile_v4(const uint4* p) {
  uint4 v;
  asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_volatile_v4(uint4* p, const uint4& v) {
  asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  asm volatile(
      "{\n.reg .pred p;\nWAIT_%=:\nmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n@p bra DONE_%=;\nbra WAIT_%=;\nDONE_%=:\n}" ::"r"(
          smem_u32(bar)),
      "r"(parity)
      : "memory");
}

// ---- block / grid reduction of the 14 sums and their publication (shared by the per-launch and the persistent kernel) ----
// Warp shuffles -> shared-memory block tree -> per-block row of `partials` -> the last block to arrive (ticket) adds the
// rows in a fixed order (a given input always produces the same bits) and writes `out`.  stamp != 0: `out` is mapped host
// memory the host polls: the sums travel as stamped 8-byte words (kernels.hpp launch_cost).  kPeer: the sums are first
// exchanged with the other ranks through peer memory (kernels.hpp PeerReduce).  Must be called by every thread of the block.
// The arrivals are counted with atomicInc, which wraps to 0 in the very operation of the last block: no reset store that the
// blocks of the resident kernel's NEXT evaluation would have to see (with the result travelling to the host without a fence
// nothing would order such a store against it).
template <int kThreads, bool kPeer>
__device__ __forceinline__ void reduce_and_publish(const double (&acc)[kCostSums], double* __restrict__ partials,
                                                   unsigned* __restrict__ ticket, double* __restrict__ out,
                                                   const PeerReduce& pr, unsigned stamp) {
  constexpr int kWarps = kThreads / 32;
  __shared__ double sm[kWarps][kCostSums + 2];
  __shared__ double red[kThreads / 16][16];
  __shared__ bool is_last;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int c = 0; c < kCostSums; ++c) {
    const double v = warp_sum(acc[c]);
    if (lane == 0) sm[warp][c] = v;
  }
  __syncthreads();
  if (threadIdx.x < kCostSums) {
    double v = 0.0;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) v += sm[w][threadIdx.x];
    partials[(size_t)blockIdx.x * 16 + threadIdx.x] = v;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned done = atomicInc(ticket, gridDim.x - 1u);
    is_last = (done == gridDim.x - 1u);
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  // last block: column c = thread & 15, row group = thread >> 4; every thread sums its rows of the per-block partials
  // (rows are 16 doubles apart: one 128-byte line per row), then the groups are added in a fixed order
  const int c = threadIdx.x & 15, grp = threadIdx.x >> 4;
  double v = 0.0;
  if (c < kCostSums)
    for (int b = grp; b < (int)gridDim.x; b += kThreads / 16) v += __ldcg(&partials[(size_t)b * 16 + c]);
  red[grp][c] = v;
  __syncthreads();
  double s = 0.0;
  if (threadIdx.x < kCostSums) {
#pragma unroll
    for (int gi = 0; gi < kThreads / 16; ++gi) s += red[gi][threadIdx.x];
  }
  __shared__ double s_own[kCostSums];
  // stamp != 0: the result goes to the polling host as 28 self-validating 8-byte words (32 bits of a sum | stamp) behind the
  // 16 plain doubles of `out` (kCostOutWords): no fence and no separate flag between the sums and their "ready" mark
  auto publish = [&] {  // s_own holds the 14 results (written by the threads < kCostSums before a barrier)
    if (threadIdx.x < 2 * kCostSums) {
      const unsigned long long bits = (unsigned long long)__double_as_longlong(s_own[threadIdx.x >> 1]);
      const unsigned half = (threadIdx.x & 1) ? (unsigned)(bits >> 32) : (unsigned)bits;
      volatile unsigned long long* w = reinterpret_cast<volatile unsigned long long*>(out + kCostOutWords) + threadIdx.x;
      *w = ((unsigned long long)half << 32) | (unsigned long long)stamp;
    }
  };
  if (!kPeer) {
    if (!stamp) {
      if (threadIdx.x < kCostSums) out[threadIdx.x] = s;
      return;
    }
    if (threadIdx.x < kCostSums) s_own[threadIdx.x] = s;
    __syncthreads();
    publish();
    return;
  }
  // ---- sum over the ranks through peer memory (kernels.hpp PeerReduce) -------------------------------------------
  // Every sum travels as two self-validating 8-byte messages (32 bits of the double | the evaluation counter): an aligned
  // 8-byte store is single-copy atomic, so a word that shows `seq` shows this evaluation's payload - no fence between
  // payload and flag, no separate flag, one NVLink crossing per evaluation instead of two plus two system-wide fences.
  __shared__ unsigned s_rx[kMaxPeers][2 * kCostSums];
  __shared__ int timed_out;
  const int set = (int)(pr.seq & 1u);
  if (threadIdx.x < kCostSums) s_own[threadIdx.x] = s;
  if (threadIdx.x == 0) timed_out = 0;
  __syncthreads();
  if (threadIdx.x < 2 * kCostSums) {
    const unsigned long long bits = (unsigned long long)__double_as_longlong(s_own[threadIdx.x >> 1]);
    const unsigned half = (threadIdx.x & 1) ? (unsigned)(bits >> 32) : (unsigned)bits;
    const unsigned long long msg = ((unsigned long long)half << 32) | (unsigned long long)pr.seq;
    for (int p = 0; p < pr.world; ++p) {
      volatile unsigned long long* dst = &pr.peers[p]->msg[set][pr.rank][threadIdx.x];
      *dst = msg;
    }
  }
  for (int idx = threadIdx.x; idx < pr.world * 32; idx += kThreads) {
    const int r = idx >> 5, j = idx & 31;
    if (j >= 2 * kCostSums) continue;
    volatile unsigned long long* src_w = &pr.peers[pr.rank]->msg[set][r][j];
    unsigned long long t0 = 0, t1, w;
    unsigned spins = 0;
    while ((unsigned)((w = *src_w) & 0xffffffffull) != pr.seq) {
      if ((++spins & 0xffu) != 0u) continue;
      if (t0 == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
      if (t1 - t0 > pr.timeout_ns) {  // wall-clock nanoseconds (not SM cycles): a peer never launched this evaluation
        timed_out = 1;
        break;
      }
    }
    s_rx[r][j] = (unsigned)(w >> 32);
  }
  __syncthreads();
  if (threadIdx.x < kCostSums) {
    double t = 0.0;
    for (int r = 0; r < pr.world; ++r)  // rank order: the same sum, bit for bit, on every rank
      t += __longlong_as_double((long long)(((unsigned long long)s_rx[r][2 * threadIdx.x + 1] << 32) |
                                            (unsigned long long)s_rx[r][2 * threadIdx.x]));
    t = timed_out ? __longlong_as_double(0x7ff8000000000000LL) : t;
    if (stamp)
      s_own[threadIdx.x] = t;  // every thread has read s_own (its own sums) before the barrier above
    else
      out[threadIdx.x] = t;
  }
  if (stamp) {
    __syncthreads();
    publish();
  }
}


// Tiles of 256 consecutive pairs are three contiguous spans in global memory (pair_tgt, src, maha).  One elected thread
// streams them into a two-stage shared-memory ring with cp.async.bulk (TMA): the loads of the next tile are in flight
// while the block reduces the current one, no thread holds a second pair in registers (the former register
// double-buffer spilled at 64 registers and, at 10 M pairs, ran at half the bandwidth of this kernel:
// scripts/micro/cost_variants.cu).  A last partial tile is read with plain loads (its byte count need not be a
// multiple of 16).
template <typename MT, bool kPeer>
__global__ void __launch_bounds__(kCostThreads) cost_kernel(const float4* __restrict__ src, int lo, int n,
                                                             const float4* __restrict__ pair_tgt,
                                                             const MT* __restrict__ maha, Rigid T,
                                                             double* __restrict__ partials, unsigned* __restrict__ ticket,
                                                             double* __restrict__ out, PeerReduce pr, unsigned stamp) {
  constexpr int kRowM = 6 * (int)sizeof(MT);
  constexpr int kStageBytes = kCostThreads * (32 + kRowM);
  __shared__ __align__(128) unsigned char ring[kCostStages * kStageBytes];
  __shared__ __align__(8) unsigned long long full[kCostStages];
  double acc[kCostSums];
#pragma unroll
  for (int c = 0; c < kCostSums; ++c) acc[c] = 0.0;

  const int full_tiles = n / kCostThreads;
  auto issue = [&](int tile, int s) {
    const size_t t0 = (size_t)tile * kCostThreads;
    unsigned char* stage = ring + s * kStageBytes;
    mbar_expect_tx(&full[s], kStageBytes);
    bulk_g2s(stage, pair_tgt + t0, kCostThreads * 16, &full[s]);
    bulk_g2s(stage + kCostThreads * 16, src + lo + t0, kCostThreads * 16, &full[s]);
    bulk_g2s(stage + kCostThreads * 32, maha + 6 * t0, kCostThreads * kRowM, &full[s]);
  };
  if (threadIdx.x == 0) {
#pragma unroll
    for (int s = 0; s < kCostStages; ++s) mbar_init(&full[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) {
#pragma unroll
    for (int s = 0; s < kCostStages; ++s) {
      const int tile = blockIdx.x + s * gridDim.x;
      if (tile < full_tiles) issue(tile, s);
    }
  }
  int k = 0;
  for (int tile = blockIdx.x; tile < full_tiles; tile += gridDim.x, ++k) {
    const int s = k % kCostStages;
    mbar_wait(&full[s], (unsigned)(k / kCostStages) & 1u);
    PairData<MT> d;
    load_pair_smem<MT>(ring + s * kStageBytes, threadIdx.x, d);
    add_pair(d, T, acc);
    __syncthreads();  // every thread has read stage s: it may be refilled
    if (threadIdx.x == 0) {
      const int nt = tile + kCostStages * gridDim.x;
      if (nt < full_tiles) issue(nt, s);
    }
  }
  if ((int)blockIdx.x == full_tiles % (int)gridDim.x) {  // the partial tile, if any, goes to the next block in turn
    const int t = full_tiles * kCostThreads + threadIdx.x;
    if (t < n) {
      PairData<MT> d;
      load_pair(src, pair_tgt, maha, lo, t, d);
      add_pair(d, T, acc);
    }
  }

  reduce_and_publish<kCostThreads, kPeer>(acc, partials, ticket, out, pr, stamp);
}

// ---- persistent evaluation kernel: one launch per OUTER iteration, one command per evaluation ------------------------------
// The BFGS line search evaluates the same pairs 20-30 times per outer iteration with a different transform each time,
// and the host needs every result before it can choose the next transform: per evaluation the per-launch kernel pays a
// launch, the ramp of 296 blocks, 80 B per pair from L2 and a tail.  This kernel is launched once when the pairs of an
// outer iteration exist and stays resident, one block per SM:
//   * every block owns a fixed contiguous range of pairs; the first `resident` of them are copied into its shared
//     memory ONCE (one cp.async.bulk per span) and never leave it: at 1 M pairs that is 30 % of the pairs (all of them
//     up to 0.3 M pairs) that cost no L2 traffic in any evaluation; the rest streams through a ring of kStages tiles as
//     in cost_kernel, cyclically, so the first tiles of the NEXT evaluation are already in flight while the host thinks;
//   * a command (transform, stamp) arrives in mapped host memory; block 0 polls it and republishes it in device memory,
//     where the other blocks poll (one PCIe reader, not 148); the result goes back through the polled stamp as before;
//   * block 0 ends the kernel on an EXIT command, or by itself when no command arrived for idle_timeout_ns (a host that
//     threw an exception, was descheduled, or died): the host notices that the stream has drained and launches again.
// The per-pair arithmetic is cost_kernel's; the order of the sums is not (contiguous ranges per block instead of tiles dealt
// round-robin over twice as many blocks), so the two kernels agree to the rounding of a reordered sum, not bit for bit.  For
// one set of pairs and one block shape the order is fixed: the same state gives the same bits in every evaluation.
template <typename MT, bool kPeer, int kThreads, int kStages>
__global__ void __launch_bounds__(kThreads, 1)
cost_persistent_kernel(const float4* __restrict__ src, int lo, int n, const float4* __restrict__ pair_tgt,
                       const MT* __restrict__ maha, const CostCommand* hcmd, CostCommand* dcmd, unsigned epoch,
                       double* __restrict__ partials, unsigned* __restrict__ ticket, double* __restrict__ out, PeerReduce pr,
                       unsigned long long idle_timeout_ns, int resident_cap) {
  constexpr int kRowM = 6 * (int)sizeof(MT);
  constexpr int kRow = 32 + kRowM;
  constexpr int kStageBytes = kThreads * kRow;
  extern __shared__ __align__(128) unsigned char dyn[];
  __shared__ __align__(8) unsigned long long full[kStages];
  __shared__ __align__(8) unsigned long long res_bar;
  __shared__ struct { float T[12]; unsigned op, stamp, peer_seq; } s_cmd;
  unsigned char* ring = dyn;                                  // kStages stages of kThreads pairs
  unsigned char* res = dyn + (size_t)kStages * kStageBytes;   // resident pairs: q rows, p rows, M rows

  // pairs per block: a multiple of 16, so that every bulk copy starts on a 16-byte boundary whatever the row width
  const int per = ((n + (int)gridDim.x - 1) / (int)gridDim.x + 15) & ~15;
  const int b0 = min(n, (int)blockIdx.x * per);
  const int cnt = min(n - b0, per);
  const int r = min(cnt, resident_cap);
  const int streamed = cnt - r;
  const int ntiles = (streamed + kThreads - 1) / kThreads;
  auto tile_pairs = [&](int t) { return min(kThreads, streamed - t * kThreads); };
  auto issue = [&](unsigned k) {  // cyclic tile k into stage k % kStages (thread 0 only)
    const int t = (int)(k % (unsigned)ntiles), st = (int)(k % (unsigned)kStages);
    const int np = tile_pairs(t);
    const size_t t0 = (size_t)b0 + r + (size_t)t * kThreads;
    unsigned char* stage = ring + st * kStageBytes;
    // bulk copies move multiples of 16 bytes: an odd number of 24-byte float rows is rounded up (the 8 extra bytes are
    // the next pair's, or lie inside the allocation, which is sized for 48-byte rows)
    const int mbytes = (np * kRowM + 15) & ~15;
    mbar_expect_tx(&full[st], (unsigned)(np * 32 + mbytes));
    bulk_g2s(stage, pair_tgt + t0, np * 16, &full[st]);
    bulk_g2s(stage + kThreads * 16, src + lo + t0, np * 16, &full[st]);
    bulk_g2s(stage + kThreads * 32, maha + 6 * t0, mbytes, &full[st]);
  };
  if (threadIdx.x == 0) {
#pragma unroll
    for (int st = 0; st < kStages; ++st) mbar_init(&full[st], 1);
    mbar_init(&res_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (r > 0) {
      const int mbytes = (r * kRowM + 15) & ~15;
      mbar_expect_tx(&res_bar, (unsigned)(r * 32 + mbytes));
      bulk_g2s(res, pair_tgt + b0, r * 16, &res_bar);
      bulk_g2s(res + (size_t)resident_cap * 16, src + lo + b0, r * 16, &res_bar);
      bulk_g2s(res + (size_t)resident_cap * 32, maha + 6 * (size_t)b0, mbytes, &res_bar);
    }
    if (ntiles > 0)
      for (unsigned k = 0; k < (unsigned)kStages; ++k) issue(k);
  }
  if (r > 0) mbar_wait(&res_bar, 0u);

  unsigned consumed = 0;  // tiles consumed so far (all evaluations)
  unsigned count = 0;     // commands seen by this launch
  for (;;) {
    // ---- next command -------------------------------------------------------------------------------------------
    // lanes 0-4 of warp 0 each own one 16-byte chunk of the command (kernels.hpp CostCommand)
    if (threadIdx.x < 32) {
      const unsigned want = (epoch << 20) | ((count + 1u) & 0xfffffu);
      const int lane = threadIdx.x;
      uint4 v = make_uint4(0u, 0u, 0u, want);
      if (blockIdx.x == 0) {
        unsigned long long t0 = 0, t1;
        if (lane == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        bool dead = false;
        for (unsigned spins = 1;; ++spins) {
          if (lane < 5) v = ld_volatile_v4(reinterpret_cast<const uint4*>(&hcmd->chunk[lane]));
          if (__all_sync(kFullMask, lane >= 5 || v.w == want)) break;
          if ((spins & 0x1fu) == 0u) {
            int d = 0;
            if (lane == 0) {
              asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
              d = (t1 - t0 > idle_timeout_ns) ? 1 : 0;
            }
            if (__shfl_sync(kFullMask, d, 0)) { dead = true; break; }
          }
        }
        if (dead) v = make_uint4(kCostOpExit, 0u, 0u, want);  // only chunk 4's first word matters
        if (dead && lane != 4) v = make_uint4(0u, 0u, 0u, want);
        // republish for the other blocks: payload and sequence word of a chunk travel in one 16-byte store
        if (lane < 5) st_volatile_v4(reinterpret_cast<uint4*>(&dcmd->chunk[lane]), v);
      } else {
        for (;;) {
          if (lane < 5) v = ld_volatile_v4(reinterpret_cast<const uint4*>(&dcmd->chunk[lane]));
          if (__all_sync(kFullMask, lane >= 5 || v.w == want)) break;
        }
      }
      if (lane < 4) {
        s_cmd.T[3 * lane] = __uint_as_float(v.x);
        s_cmd.T[3 * lane + 1] = __uint_as_float(v.y);
        s_cmd.T[3 * lane + 2] = __uint_as_float(v.z);
      } else if (lane == 4) {
        s_cmd.op = v.x;
        s_cmd.stamp = v.y;
        s_cmd.peer_seq = v.z;
      }
    }
    __syncthreads();
    ++count;
    if (s_cmd.op != kCostOpEval) break;
    Rigid T;
#pragma unroll
    for (int i = 0; i < 12; ++i) T.m[i] = s_cmd.T[i];
    const unsigned stamp = s_cmd.stamp;
    PeerReduce prr = pr;
    prr.seq = s_cmd.peer_seq;

    double acc[kCostSums];
#pragma unroll
    for (int c = 0; c < kCostSums; ++c) acc[c] = 0.0;
    // resident pairs: no memory traffic beyond shared memory
    for (int i = threadIdx.x; i < r; i += kThreads) {
      PairData<MT> d;
      load_pair_smem_at<MT>(res, res + (size_t)resident_cap * 16, res + (size_t)resident_cap * 32, i, d);
      add_pair(d, T, acc);
    }
    // streamed pairs
    for (int t = 0; t < ntiles; ++t, ++consumed) {
      const int st = (int)(consumed % (unsigned)kStages);
      mbar_wait(&full[st], (consumed / (unsigned)kStages) & 1u);
      if ((int)threadIdx.x < tile_pairs((int)(consumed % (unsigned)ntiles))) {
        const unsigned char* stage = ring + st * kStageBytes;
        PairData<MT> d;
        load_pair_smem_at<MT>(stage, stage + kThreads * 16, stage + kThreads * 32, threadIdx.x, d);
        add_pair(d, T, acc);
      }
      __syncthreads();  // every thread has read stage st: it may be refilled (with a tile of this or the next evaluation)
      if (threadIdx.x == 0) issue(consumed + (unsigned)kStages);
    }
    reduce_and_publish<kThreads, kPeer>(acc, partials, ticket, out, prr, stamp);
    __syncthreads();
  }
  // leave no bulk copy in flight into this block's shared memory
  if (ntiles > 0)
    for (unsigned k = consumed; k < consumed + (unsigned)kStages; ++k)
      mbar_wait(&full[k % (unsigned)kStages], (k / (unsigned)kStages) & 1u);
}

// ---- second-order moments of the objective (one pass per OUTER iteration) ---------------------------------------------
// The objective is a quadratic form in the 12 entries of the rigid transform: with r0_i the residual at the transform
// T0 of this outer iteration (float, exactly as PCL evaluates it) and D = [R|t] - [R0|t0] (3x4),
//     r_i = r0_i + D p~_i,   p~ = (x, y, z, 1)
//     sum r^T M r   = c + sum_ak D[a][k] (B[a][k] + G[a][k])
//     sum (M r)_a p~_k = G[a][k] = B[a][k] + sum_bl H[kl][ab] D[b][l]
// with c = sum r0^T M r0, B[a][k] = sum p~_k (M r0)_a (12), H[kl][ab] = sum p~_k p~_l M_ab (10 x 6).  Once the 74
// sums are on the host every f / df / fdf evaluation of the BFGS line search (OptimizationFunctorWithIndices, PCL
// gicp.hpp) is O(1) host arithmetic: no kernel launch, no pass over the pairs, no collective.  At x = x0 the value
// is PCL's float-transform value bit for bit; away from it the products T p are exact instead of rounded to float.
//
// Layout of the 74 sums: [0] c, [1 + 4a + k] B[a][k], [13] pair count, [14 + 6*kl + ab] H, kl in the order
// 00 01 02 03 11 12 13 22 23 33, ab in the order 00 01 02 11 12 22.
constexpr int kMomThreads = 512;          // two roles of 256 threads: both walk the same pairs
constexpr int kMomRole = kMomThreads / 2;
constexpr int kMomAcc = 38;               // role 0: c, B, count, H kl 0..3 (38); role 1: H kl 4..9 (36)
constexpr int kMomRow = 80;               // doubles per partial row (74 used)

template <typename MT>
__global__ void __launch_bounds__(kMomThreads, 1) moments_kernel(const float4* __restrict__ src, int lo, int n,
                                                                  const float4* __restrict__ pair_tgt,
                                                                  const MT* __restrict__ maha, Rigid T0,
                                                                  double* __restrict__ partials,
                                                                  unsigned* __restrict__ ticket, double* __restrict__ out) {
  double acc[kMomAcc];
#pragma unroll
  for (int c = 0; c < kMomAcc; ++c) acc[c] = 0.0;
  const int role = threadIdx.x >= kMomRole ? 1 : 0;
  const int stride = gridDim.x * kMomRole;
  for (int t = blockIdx.x * kMomRole + (threadIdx.x & (kMomRole - 1)); t < n; t += stride) {
    PairData<MT> d;
    load_pair(src, pair_tgt, maha, lo, t, d);
    if (d.q.w == 0.f) continue;  // no correspondence inside the gate
    const double m[6] = {(double)d.m[0], (double)d.m[1], (double)d.m[2], (double)d.m[3], (double)d.m[4], (double)d.m[5]};
    const double px = (double)d.p.x, py = (double)d.p.y, pz = (double)d.p.z;
    if (role == 0) {
      const float3 pp = xform(T0, d.p.x, d.p.y, d.p.z);
      const double r0 = (double)__fsub_rn(pp.x, d.q.x);
      const double r1 = (double)__fsub_rn(pp.y, d.q.y);
      const double r2 = (double)__fsub_rn(pp.z, d.q.z);
      const double t0 = m[0] * r0 + m[1] * r1 + m[2] * r2;
      const double t1 = m[1] * r0 + m[3] * r1 + m[4] * r2;
      const double t2 = m[2] * r0 + m[4] * r1 + m[5] * r2;
      acc[0] += r0 * t0 + r1 * t1 + r2 * t2;
      acc[1] += px * t0; acc[2] += py * t0; acc[3] += pz * t0; acc[4] += t0;
      acc[5] += px * t1; acc[6] += py * t1; acc[7] += pz * t1; acc[8] += t1;
      acc[9] += px * t2; acc[10] += py * t2; acc[11] += pz * t2; acc[12] += t2;
      acc[13] += 1.0;
      const double w[4] = {px * px, px * py, px * pz, px};  // kl = 00 01 02 03
#pragma unroll
      for (int kl = 0; kl < 4; ++kl)
#pragma unroll
        for (int ab = 0; ab < 6; ++ab) acc[14 + 6 * kl + ab] += w[kl] * m[ab];
    } else {
      const double w[5] = {py * py, py * pz, py, pz * pz, pz};  // kl = 11 12 13 22 23
#pragma unroll
      for (int kl = 0; kl < 5; ++kl)
#pragma unroll
        for (int ab = 0; ab < 6; ++ab) acc[6 * kl + ab] += w[kl] * m[ab];
#pragma unroll
      for (int ab = 0; ab < 6; ++ab) acc[30 + ab] += m[ab];  // kl = 33
    }
  }

  __shared__ double sm[kMomThreads / 32][kMomAcc + 1];
  __shared__ double red[6][kMomRow];
  __shared__ bool is_last;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int c = 0; c < kMomAcc; ++c) {
    const double v = warp_sum(acc[c]);
    if (lane == 0) sm[warp][c] = v;
  }
  __syncthreads();
  if (threadIdx.x < 2 * kMomAcc) {  // column of role r, accumulator j: r * 38 + j  (role 1 uses 36 of its 38)
    const int r = threadIdx.x / kMomAcc, j = threadIdx.x % kMomAcc;
    double v = 0.0;
#pragma unroll
    for (int w = 0; w < kMomRole / 32; ++w) v += sm[r * (kMomRole / 32) + w][j];
    partials[(size_t)blockIdx.x * kMomRow + threadIdx.x] = v;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned done = atomicAdd(ticket, 1u);
    is_last = (done == gridDim.x - 1);
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  // last block: fixed-order sum of the per-block rows (deterministic)
  const int c = threadIdx.x % kMomRow, grp = threadIdx.x / kMomRow;
  if (grp < 6) {
    double v = 0.0;
    if (c < 2 * kMomAcc)
      for (int b = grp; b < (int)gridDim.x; b += 6) v += __ldcg(&partials[(size_t)b * kMomRow + c]);
    red[grp][c] = v;
  }
  __syncthreads();
  if (threadIdx.x < kMomentSums) out[threadIdx.x] = ((red[0][threadIdx.x] + red[1][threadIdx.x]) + (red[2][threadIdx.x] + red[3][threadIdx.x])) +
                                                     (red[4][threadIdx.x] + red[5][threadIdx.x]);
  if (threadIdx.x == 0) *ticket = 0u;
}

}  // namespace

int cost_grid_blocks(int n, int num_sms) {
  const int want = (n + kCostThreads - 1) / kCostThreads;
  const int cap = num_sms * 2;  // a multiple of the SM count; 2 resident CTAs (40 KB of staging each) per SM
  return std::max(1, std::min(want, cap));
}

void launch_cost(const float4* src, int lo, int n, const float4* pair_tgt, const void* maha, bool maha_fp32,
                 const Rigid& T, double* partials, unsigned* ticket, double* out14, int blocks, cudaStream_t stream,
                 const PeerReduce* peer, unsigned stamp) {
  PeerReduce pr{};
  if (peer) pr = *peer;
  if (maha_fp32) {
    if (peer)
      cost_kernel<float, true><<<blocks, kCostThreads, 0, stream>>>(src, lo, n, pair_tgt, (const float*)maha, T, partials,
                                                                    ticket, out14, pr, stamp);
    else
      cost_kernel<float, false><<<blocks, kCostThreads, 0, stream>>>(src, lo, n, pair_tgt, (const float*)maha, T, partials,
                                                                     ticket, out14, pr, stamp);
  } else {
    if (peer)
      cost_kernel<double, true><<<blocks, kCostThreads, 0, stream>>>(src, lo, n, pair_tgt, (const double*)maha, T, partials,
                                                                     ticket, out14, pr, stamp);
    else
      cost_kernel<double, false><<<blocks, kCostThreads, 0, stream>>>(src, lo, n, pair_tgt, (const double*)maha, T, partials,
                                                                      ticket, out14, pr, stamp);
  }
  GICPB_LAUNCHED();
}

// ---- persistent session ---------------------------------------------------------------------------------------------------
namespace {
template <typename MT, bool kPeer, int kThreads, int kStages>
void launch_persistent_v(const float4* src, int lo, int n, const float4* pair_tgt, const void* maha, const CostCommand* hcmd,
                         CostCommand* dcmd, unsigned epoch, double* partials, unsigned* ticket, double* out,
                         const PeerReduce& pr, unsigned long long idle_ns, int blocks, int smem_optin, cudaStream_t stream,
                         CostPersistentShape* shape) {
  constexpr int kRow = 32 + 6 * (int)sizeof(MT);
  auto kern = cost_persistent_kernel<MT, kPeer, kThreads, kStages>;
  static int static_smem = -1;  // of this instantiation
  if (static_smem < 0) {
    cudaFuncAttributes fa;
    GICPB_CUDA(cudaFuncGetAttributes(&fa, kern));
    static_smem = (int)fa.sharedSizeBytes;
  }
  const int ring = kStages * kThreads * kRow;
  const int budget = smem_optin - static_smem - ring - 1024;  // 1 KB of slack for alignment
  const int per = ((n + blocks - 1) / blocks + 15) & ~15;
  // a multiple of 16 pairs: the row bases of the resident block stay 128-byte aligned
  const int cap = std::max(0, (budget / kRow) & ~15);
  const int resident = std::min(per, cap);
  const size_t dyn = (size_t)ring + (size_t)resident * kRow;
  GICPB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
  kern<<<blocks, kThreads, dyn, stream>>>(src, lo, n, pair_tgt, (const MT*)maha, hcmd, dcmd, epoch, partials, ticket, out, pr,
                                          idle_ns, resident);
  GICPB_LAUNCHED();
  if (shape) *shape = CostPersistentShape{blocks, kThreads, kStages, per, cap, resident};
}

// block shape of the resident kernel: 512 threads x 2 stages keeps 80 KB in flight per SM and parks 26 % of 1 M pairs;
// from 2 M pairs on - where an evaluation is the stream from L2 / HBM and little else - a third stage (120 KB in flight) is
// worth the pairs it unparks (4 M pairs: 56 -> 51 us per evaluation; 1 M: 13.7 us either way).
template <typename MT, bool kPeer>
void launch_persistent_t(const float4* src, int lo, int n, const float4* pair_tgt, const void* maha, const CostCommand* hcmd,
                         CostCommand* dcmd, unsigned epoch, double* partials, unsigned* ticket, double* out,
                         const PeerReduce& pr, unsigned long long idle_ns, int blocks, int smem_optin, cudaStream_t stream,
                         CostPersistentShape* shape) {
  if (n >= 2000000)
    launch_persistent_v<MT, kPeer, 512, 3>(src, lo, n, pair_tgt, maha, hcmd, dcmd, epoch, partials, ticket, out, pr, idle_ns,
                                           blocks, smem_optin, stream, shape);
  else
    launch_persistent_v<MT, kPeer, 512, 2>(src, lo, n, pair_tgt, maha, hcmd, dcmd, epoch, partials, ticket, out, pr, idle_ns,
                                           blocks, smem_optin, stream, shape);
}
}  // namespace

int cost_persistent_blocks(int num_sms) { return num_sms; }

void launch_cost_persistent(const float4* src, int lo, int n, const float4* pair_tgt, const void* maha, bool maha_fp32,
                            const CostCommand* hcmd_dev, CostCommand* dcmd, unsigned epoch, double* partials, unsigned* ticket,
                            double* out16, const PeerReduce* peer, unsigned long long idle_timeout_ns, int blocks,
                            int smem_optin, cudaStream_t stream, CostPersistentShape* shape) {
  PeerReduce pr{};
  if (peer) pr = *peer;
  if (maha_fp32) {
    if (peer)
      launch_persistent_t<float, true>(src, lo, n, pair_tgt, maha, hcmd_dev, dcmd, epoch, partials, ticket, out16, pr,
                                       idle_timeout_ns, blocks, smem_optin, stream, shape);
    else
      launch_persistent_t<float, false>(src, lo, n, pair_tgt, maha, hcmd_dev, dcmd, epoch, partials, ticket, out16, pr,
                                        idle_timeout_ns, blocks, smem_optin, stream, shape);
  } else {
    if (peer)
      launch_persistent_t<double, true>(src, lo, n, pair_tgt, maha, hcmd_dev, dcmd, epoch, partials, ticket, out16, pr,
                                        idle_timeout_ns, blocks, smem_optin, stream, shape);
    else
      launch_persistent_t<double, false>(src, lo, n, pair_tgt, maha, hcmd_dev, dcmd, epoch, partials, ticket, out16, pr,
                                         idle_timeout_ns, blocks, smem_optin, stream, shape);
  }
}

int moments_grid_blocks(int n, int num_sms) {
  const int want = (n + kMomRole - 1) / kMomRole;
  return std::max(1, std::min(want, num_sms));  // one 512-thread CTA per SM
}

void launch_moments(const float4* src, int lo, int n, const float4* pair_tgt, const void* maha, bool maha_fp32,
                    const Rigid& T0, double* partials, unsigned* ticket, double* out74, int blocks, cudaStream_t stream) {
  if (maha_fp32)
    moments_kernel<float><<<blocks, kMomThreads, 0, stream>>>(src, lo, n, pair_tgt, (const float*)maha, T0, partials,
                                                              ticket, out74);
  else
    moments_kernel<double><<<blocks, kMomThreads, 0, stream>>>(src, lo, n, pair_tgt, (const double*)maha, T0, partials,
                                                               ticket, out74);
  GICPB_LAUNCHED();
}

}  // namespace gicpb
