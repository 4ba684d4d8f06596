// kernels.hpp - host-callable launchers of the CUDA kernels of libgicp_b200.
#pragma once
#include "engine.hpp"

namespace gicpb {

struct RotD {  // double 3x3, row-major: double(transformation_) top-left block (gicp.hpp transform_R)
  double m[9];
};

// Hand-over from a NEAR search kernel to its FAR instance (nn_kernels.cu, knn_cov.cu).  The near kernel writes one
// flag byte per query (1 = this query needs the hierarchical search).  The far kernel runs `far_blocks` persistent
// blocks; each block takes tiles of kFarTile consecutive queries from `tile_counter`, compacts the flagged ones IN
// ORDER into shared memory and works through them with full warps - so the lanes of a far warp still hold spatial
// neighbours (the queries are sorted by cell) and the warps of a block share cache lines.
// flags must have room for the item count rounded up to kFarTile; tile_counter[0..1] (tile cursor, number of far
// queries) are zeroed before each launch pair (reset_far).
constexpr int kFarTile = 256;   // 2 flags per thread of a 128-thread block: small tiles spread a clustered handful of
                                // far queries (FOD blobs, a seam) over many blocks instead of serialising them in one
constexpr int kFarFlagsPerThread = kFarTile / 128;
struct FarWork {
  unsigned char* flags;
  unsigned* tile_counter;
  int far_blocks;
  int near_rings;  // NN-1 near instance: cell rings probed for a first candidate (1..kNearMaxRing)
  // queries per tile: kFarTile, or half of it where there are few tiles per block to balance (far_tile_for: a first pass
  // over 1 M queries 1.06 -> 0.99 ms with 128; over 8 M queries 128 costs 3 % in cursor and barrier rounds)
  int tile = kFarTile;
};
inline int far_tile_for(int64_t n_items) { return n_items <= 2000000 ? kFarTile / 2 : kFarTile; }

#if defined(__CUDACC__)
// Far-instance driver: calls body(item) for every flagged item of [0, n_items); blockDim.x must be 128.
template <class F>
__device__ __forceinline__ void far_for_each(const FarWork& fw, int n_items, F body) {
  __shared__ int s_items[kFarTile];
  __shared__ int s_warp[4];
  __shared__ int s_tile, s_n, s_next;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (;;) {
    __syncthreads();
    if (threadIdx.x == 0) s_tile = (int)atomicAdd(fw.tile_counter, 1u);
    __syncthreads();
    const int fpt = fw.tile >> 7;  // flags per thread: 1 or 2 (kFarFlagsPerThread at most)
    const int base = s_tile * fw.tile;
    if (base >= n_items) break;
    // fpt consecutive flags per thread, in item order
    unsigned w = 0;
#pragma unroll
    for (int k = 0; k < kFarFlagsPerThread; ++k)
      if (k < fpt) w |= (unsigned)(fw.flags[base + threadIdx.x * fpt + k] & 1u) << k;
    const int cnt = __popc(w);
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(kFullMask, incl, o);
      if (lane >= o) incl += v;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    int off = incl - cnt;
    for (int k = 0; k < warp; ++k) off += s_warp[k];
    if (threadIdx.x == 127) {
      s_n = off + cnt;
      s_next = 0;
    }
#pragma unroll
    for (int k = 0; k < kFarFlagsPerThread; ++k)
      if ((w >> k) & 1u) s_items[off++] = base + threadIdx.x * fpt + k;
    __syncthreads();
    const int n = s_n;
    if (threadIdx.x == 0 && n) atomicAdd(fw.tile_counter + 1, (unsigned)n);  // statistics: queries answered here
    for (;;) {  // warps take 32 consecutive items at a time
      int k = 0;
      if (lane == 0) k = atomicAdd(&s_next, 32);
      k = __shfl_sync(kFullMask, k, 0);
      if (k >= n) break;
      if (k + lane < n) body(s_items[k + lane]);
      __syncwarp();
    }
  }
}
#endif

// ---- nn_kernels.cu ------------------------------------------------------------------------------------
void reset_far(const FarWork& fw, int64_t n_items, cudaStream_t stream);  // before every near / far launch pair
void launch_nn1(const GridView& g, const float4* queries, int n, const Rigid& T, float gate2, int* idx, float* d2,
                int* pos, const FarWork& fw, cudaStream_t stream);
void launch_correspondences(const GridView& g, const float4* src, int lo, int hi, const Rigid& T, const RotD& R,
                            float gate2, const double* n_src, const double* n_tgt, double eps, int* pair_pos,
                            float* pair_d2, float4* pair_tgt, void* maha, bool maha_fp32, bool use_prev,
                            const FarWork& fw, cudaStream_t stream);
int fitness_partial_rows(int n, int far_blocks);
// seed: nullptr, or one sorted-target position (-1 = none) per source point of [lo, hi) as a first candidate
void launch_fitness(const GridView& g, const float4* src, int lo, int hi, const Rigid& T, double max_range,
                    const int* seed, double* partials, double* out2, const FarWork& fw, cudaStream_t stream);
// what decides a difference's keep bytes: the search (d2 < thr_next hits), or the threshold alone (thr < 0 keeps every
// finite point, a NaN threshold none: PCL's `d2 > thr` is then always / never true)
enum DiffMode : int { kDiffSearch = 0, kDiffKeepAll = 1, kDiffKeepNone = 2 };
void launch_difference(const GridView& g, const unsigned char* raw, int64_t n, int64_t stride, float thr_next,
                       DiffMode mode, unsigned char* mask, unsigned long long* kept, const FarWork& fw,
                       cudaStream_t stream);
// use_covariances branch: the mean 2nd-neighbour distance sums (partials sized like the fitness ones); the normals: normals.cu
void launch_resolution(const GridView& g, double* partials, double* out2, const FarWork& fw, cudaStream_t stream);
void launch_transform(const unsigned char* in, unsigned char* out, int64_t n, int64_t stride, const Rigid& T,
                      cudaStream_t stream);
void launch_pack_queries(const unsigned char* raw, int64_t n, int64_t stride, float4* out, cudaStream_t stream);

// ---- normals.cu ---------------------------------------------------------------------------------------
// Utils::getNormals (pcl::NormalEstimation, radius search): counts[i] = neighbours (d2 < r2, the point included) of sorted
// point i; after an exclusive scan of the counts, fill writes every point's keys (d2 bits << 32 | original index) at
// keys[offsets[i] ...]; solve sorts each list and writes (nx, ny, nz, curvature) - NaN x 4 below 3 neighbours - to
// out4[ORIGINAL index] (entries of non-indexed points must be pre-set to NaN) and adds the finite count to *kept.
void launch_radius_counts(const GridView& g, float r2, unsigned* counts, const FarWork& fw, cudaStream_t stream);
void launch_sum_counts(const unsigned* counts, int n, unsigned long long* out, cudaStream_t stream);  // *out += sum, 64 bits
void launch_radius_fill(const GridView& g, float r2, const unsigned* offsets, unsigned long long* keys, const FarWork& fw,
                        cudaStream_t stream);
void launch_normals_solve(const GridView& g, const unsigned* counts, const unsigned* offsets, unsigned long long* keys,
                          float4* out4, unsigned long long* kept, cudaStream_t stream);

// ---- knn_cov.cu ---------------------------------------------------------------------------------------
// self-kNN (k <= 32) of sorted points [lo, hi) of grid g + regularised covariance normal per point.
// normals: 3 doubles per point, index (i - lo).  knn_idx / knn_d2 (nullable): k entries per point, row
// (i - lo), original indices.
// win (nullable, with win_violations): the index only holds the window's points (GridIndex::knn_window); *win_violations counts
// the points of [lo, hi) whose list cannot be vouched for (must be zeroed by the caller).
void launch_knn_covariances(const GridView& g, int lo, int hi, int k, double* normals, int* knn_idx, float* knn_d2,
                            const FarWork& fw, cudaStream_t stream, const GridIndex::KnnWindow* win = nullptr,
                            unsigned* win_violations = nullptr);

// ---- cost.cu ------------------------------------------------------------------------------------------
constexpr int kCostSums = 14;  // f, g_t[3], Rsum[9], pair count
int cost_grid_blocks(int n, int num_sms);

// Cross-GPU sum of the 14 cost sums INSIDE the cost kernel, over NVLink peer memory (no collective call, no extra
// launch): every rank owns one PeerSlots block in device memory that all ranks have mapped (cudaIpc).  The last block
// of a rank's cost kernel sends every sum to EVERY rank's block as two 8-byte words, each carrying 32 bits of the double
// and the evaluation counter `seq` (an aligned 8-byte store is single-copy atomic: a word that shows `seq` shows that
// evaluation's payload, so there is neither a fence between payload and flag nor a flag), polls the words of all
// `world` senders in its OWN block and adds the sums in rank order - the same order on every rank, so all ranks hold
// bit-identical sums and the host optimisers stay in lock step.  Two slot sets alternate (seq & 1): a rank can run at
// most one evaluation ahead of the slowest.  (Round 1 sent payload, fence, flag, fence: two NVLink crossings and two
// system-wide fences per evaluation: 27.7 us per evaluation on 2 GPUs against 22.1 us now.)
constexpr int kMaxPeers = 16;
struct PeerSlots {
  // msg[set][sender][2 c + half]: (32 bits of the sender's sum c) << 32 | evaluation counter - self-validating 8-byte words
  unsigned long long msg[2][kMaxPeers][32];
};
struct PeerReduce {
  PeerSlots* peers[kMaxPeers];  // peers[r] = rank r's block as mapped in this process (peers[rank] = own)
  int rank, world;
  unsigned seq;                 // evaluation counter, identical on all ranks, never 0
  unsigned long long timeout_ns;  // how long the last block waits for the other ranks' flags (GICPB_PEER_TIMEOUT_MS, default 30 s)
};
// sums over this rank's pairs; `partials` holds cost_grid_blocks * kCostSums doubles, `ticket` one zeroed uint.
// out14 may be device memory or mapped pinned host memory.
// peer != nullptr: out14 receives the sum over all ranks (see PeerReduce); a peer that does not show up within
// PeerReduce::timeout_ns makes every entry NaN.
void launch_cost(const float4* src, int lo, int n, const float4* pair_tgt, const void* maha, bool maha_fp32,
                 const Rigid& T, double* partials, unsigned* ticket, double* out14, int blocks, cudaStream_t stream,
                 const PeerReduce* peer = nullptr, unsigned stamp = 0);
// stamp != 0 (below 2^32, never 0): out14 must be mapped host memory of kCostOutDoubles doubles; the kernel then sends
// the 14 sums as 28 self-validating 8-byte words - (32 bits of sum j / 2, low half first) << 32 | stamp - at
// out14 + kCostOutWords, which the host polls instead of synchronising the stream: a word that shows the stamp shows its
// payload (aligned 8-byte stores are single-copy atomic), so the kernel needs no system-wide fence before a "ready" flag.
constexpr int kCostOutWords = 32;    // offset (in doubles) of the 32 result words behind the 16 plain doubles
constexpr int kCostOutDoubles = 64;

// Persistent evaluation kernel (cost.cu cost_persistent_kernel): launched once per outer iteration, one block per SM; every
// evaluation is a CostCommand the host writes into mapped pinned memory (seq LAST) and the kernel answers through the
// stamped result words behind out16 (launch_cost).  seq = (epoch << 20) | k for the k-th command (k = 1, 2, ...) of the launch with that epoch.
constexpr unsigned kCostOpEval = 1u, kCostOpExit = 2u;
// A command is five self-validating 16-byte chunks: each carries the sequence word in its last lane, and the host writes
// a chunk's payload before its sequence word.  A 16-byte read (one PCIe read inside one cache line, or one L2 access)
// that shows the expected sequence word therefore shows that command's payload: five lanes read the five chunks IN
// PARALLEL (one round trip) instead of seventeen dependent reads.
struct CostCommand {
  struct Chunk {
    unsigned w[3];  // chunks 0-3: the bits of T[3i .. 3i+2]; chunk 4: op, stamp, peer_seq
    unsigned seq;
  } chunk[5];
  unsigned pad[12];  // 128 bytes: two commands never share a line
};
static_assert(sizeof(CostCommand) == 128, "CostCommand layout");
int cost_persistent_blocks(int num_sms);
// hcmd_dev: device alias of the mapped host command slot of this launch (the host alternates between two slots by epoch,
// so the EXIT of one launch is never overwritten by the first command of the next); dcmd: one CostCommand in device memory; partials / ticket as
// launch_cost (blocks rows); out16: mapped host memory of kCostOutDoubles doubles; smem_optin: cudaDevAttrMaxSharedMemoryPerBlockOptin.
// shape (nullable) receives the block shape the launch took (gicpb_cost_session reports it).
struct CostPersistentShape {
  int blocks, threads, stages;
  int per_block;     // pairs each block owns (a multiple of 16; the last block may own fewer)
  int resident_cap;  // pairs one block can park in shared memory (a multiple of 16)
  int resident;      // pairs each full block parks: min(per_block, resident_cap)
};
void launch_cost_persistent(const float4* src, int lo, int n, const float4* pair_tgt, const void* maha, bool maha_fp32,
                            const CostCommand* hcmd_dev, CostCommand* dcmd, unsigned epoch, double* partials, unsigned* ticket,
                            double* out16, const PeerReduce* peer, unsigned long long idle_timeout_ns, int blocks,
                            int smem_optin, cudaStream_t stream, CostPersistentShape* shape = nullptr);

// ---- segment.cu -----------------------------------------------------------------------------------------
// Euclidean clustering: joins every pair of indexed points of `g` with d2 < r2 (strict) in a union-find over sorted
// positions (`parent`, g.n ints) and writes root_of[original index] = original index of the set's root point
// (entries of non-indexed points are left untouched: pre-set them to -1).
void launch_cluster_unions(const GridView& g, float r2, int* parent, int* root_of, const FarWork& fw, cudaStream_t stream);

// pcl::VoxelGrid::applyFilter on strided points (xyz first; rgba word at byte 16 when stride >= 20).  Writes one
// centroid point per occupied voxel to d_out (ascending voxel index, same stride) and returns their number.
// *overflow: PCL's check dx * dy * dz > INT32_MAX refuses the leaf ("leaf size too small"): nothing is written, n is
// returned.
class VoxelGrid {
 public:
  int64_t run(const unsigned char* d_in, int64_t n, int64_t stride, float leaf, unsigned char* d_out, cudaStream_t stream,
              bool* overflow);

 private:
  DevBuf<uint32_t> keys_a_, keys_b_, vals_a_, vals_b_, scan_tmp_, starts_;
  RadixSorter sorter_;
  DevBuf<unsigned> scratch_;
};

// second-order moments of the objective around T0 (cost.cu): 74 sums from which every later f / df evaluation of the
// outer iteration is host arithmetic.  `partials` holds moments_grid_blocks * 80 doubles, `ticket` one zeroed uint.
constexpr int kMomentSums = 74;
int moments_grid_blocks(int n, int num_sms);
void launch_moments(const float4* src, int lo, int n, const float4* pair_tgt, const void* maha, bool maha_fp32,
                    const Rigid& T0, double* partials, unsigned* ticket, double* out74, int blocks, cudaStream_t stream);

}  // namespace gicpb
