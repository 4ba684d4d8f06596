// engine.hpp - host-side declarations shared by the translation units of libgicp_b200.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <stdexcept>
#include <string>
#include <vector>

#include "common.cuh"
#include "upload.hpp"

namespace gicpb {

struct CudaError : std::runtime_error {
  explicit CudaError(const std::string& s) : std::runtime_error(s) {}
};
struct ArgError : std::runtime_error {
  explicit ArgError(const std::string& s) : std::runtime_error(s) {}
};
struct StateError : std::runtime_error {
  explicit StateError(const std::string& s) : std::runtime_error(s) {}
};

#define GICPB_CUDA(expr)                                                                              \
  do {                                                                                                \
    cudaError_t _e = (expr);                                                                          \
    if (_e != cudaSuccess)                                                                            \
      throw ::gicpb::CudaError(std::string(#expr) + ": " + cudaGetErrorString(_e) + " (" + __FILE__ + \
                               ":" + std::to_string(__LINE__) + ")");                                 \
  } while (0)

extern std::atomic<int64_t> g_launch_count;  // kernels launched by this library (all contexts, any host thread)
#define GICPB_LAUNCHED()                 \
  do {                                   \
    ++::gicpb::g_launch_count;           \
    GICPB_CUDA(cudaGetLastError());      \
  } while (0)

// RAII device buffer (cudaMalloc); never shrinks unless released
template <typename T>
class DevBuf {
 public:
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { release(); }
  void release() {
    if (p_) cudaFree(p_);
    p_ = nullptr;
    cap_ = 0;
  }
  void reserve(size_t n) {
    if (n <= cap_) return;
    release();
    GICPB_CUDA(cudaMalloc(&p_, std::max<size_t>(n, 1) * sizeof(T)));
    cap_ = n;
  }
  T* get() const { return p_; }
  size_t capacity() const { return cap_; }

 private:
  T* p_ = nullptr;
  size_t cap_ = 0;
};

// Stable LSD radix sort of (key, value) pairs, one kernel per 8-bit digit (sort_scan.cu "onesweep").  prepare() zeroes the
// digit histograms; the producer of the keys may count them itself into hist() ([pass][256], digit = (key >> 8 pass) & 255)
// and pass hist_ready = true.  sort() returns true if the result is in the *_b buffers.
class RadixSorter {
 public:
  void prepare(int64_t n, cudaStream_t stream);
  uint32_t* hist() const { return work_.get(); }
  bool sort(uint32_t* keys_a, uint32_t* vals_a, uint32_t* keys_b, uint32_t* vals_b, int64_t n, int key_bits, bool hist_ready,
            cudaStream_t stream);

 private:
  static constexpr size_t kWorkWords = 1024 + 8;  // 4 x 256 digit counts, 4 tile cursors
  DevBuf<uint32_t> work_;
  DevBuf<unsigned long long> status_;  // [tile][digit]: (epoch << 2 | kind) << 32 | count
  uint32_t epoch_ = 0;
};

// Per-cloud spatial index (see common.cuh).  build() runs the whole pipeline on `stream`:
// ingest (strided xyz -> float4 + bbox) -> density probe -> cell keys -> radix sort -> reorder -> brick/cell tables.
class GridIndex {
 public:
  GridIndex() = default;
  GridIndex(const GridIndex&) = delete;
  GridIndex& operator=(const GridIndex&) = delete;
  ~GridIndex() {
    if (h_pin_) cudaFreeHost(h_pin_);
    if (ev_slots_) cudaEventDestroy(ev_slots_);
  }
  struct Info {
    int64_t n_points = 0, n_indexed = 0;
    float cell_size = 0;
    int dims[3] = {0, 0, 0};
    int64_t n_bricks_occupied = 0, n_cells_occupied = 0;
    double ms_build = 0;
    float bbox_min[3] = {0, 0, 0}, bbox_max[3] = {0, 0, 0};
  };
  // `raw` points at the first x; device pointer iff on_device.  cell_size <= 0 -> from density.
  // stager (nullable): pageable host clouds are uploaded through it as packed xyz rows (upload.hpp)
  // world > 1 (the SOURCE of a sharded job): only the part of the cloud that rank `rank` needs is indexed - a window of
  // brick planes along the longest axis holding about 1 / world of the points (the rank's shard, [shard_lo, shard_hi) of
  // the sorted points) plus one halo plane either side, so that the k nearest neighbours of the shard's points are
  // in it (knn_window() tells the kNN kernel where the window ends; it reports every point it cannot vouch for, and the
  // caller then widens the window to the whole cloud with widen()).  Same grid geometry, keys and order as the whole
  // cloud's index: the window IS that index cut to its planes (bricks are numbered plane by plane for this).
  // halo_m >= 0 (the SUBTRACT cloud of a group's difference): the halo is as many planes as cover a search radius of halo_m
  // metres from any point of the rank's own planes (GICPB_HALO_PLANES does not apply); INFINITY: the whole cloud.
  void build(const void* raw, int64_t n, int64_t stride_bytes, bool on_device, float cell_size,
             float points_per_cell, cudaStream_t stream, HostStager* stager = nullptr, int rank = 0, int world = 1,
             double halo_m = -1.0);
  void widen(cudaStream_t stream);  // re-index with the window = the whole cloud (the shard stays the same set of points)
  bool windowed() const { return win_.active && !(win_.w_lo == 0 && win_.w_hi == win_.planes); }
  bool plane_sharded() const { return win_.active; }  // the shard is a range of brick planes (else: an index range)
  int shard_lo() const { return win_.shard_lo; }
  int shard_hi() const { return win_.shard_hi; }
  int64_t n_finite_total() const { return win_.n_finite; }  // finite points of the whole cloud
  struct KnnWindow {  // the window along `axis` in coordinates: neighbours beyond [lo, hi] are not indexed (axis -1: none)
    int axis = -1;
    float lo = 0.f, hi = 0.f;
  };
  KnnWindow knn_window() const;
  // plane_sharded(): the finite rows of a query cloud (raw, n, stride: xyz floats) whose brick plane on this grid - clamped to
  // the grid as the build clamps - is one of the rank's own planes, in row order, as float4 rows (x, y, z, w = row index as int
  // bits); returns how many.  Ownership partitions the finite rows over the ranks.  flags / pos hold n + 1 words, tmp
  // scan_tmp_entries(n + 1).  Synchronises `stream`.
  int64_t owned_queries(const unsigned char* raw, int64_t n, int64_t stride, float4* out, uint32_t* flags, uint32_t* pos,
                        uint32_t* tmp, cudaStream_t stream) const;
  bool ready() const { return ready_; }
  const GridView& view() const { return view_; }
  const Info& info() const { return info_; }
  int n_indexed() const { return view_.n; }
  int64_t n_points() const { return info_.n_points; }
  const float4* sorted_points() const { return pts_sorted_.get(); }
  void reset() { ready_ = false; }
  // false: a cloud that is only ever searched from its own points (the source of a registration job: kNN) - the superbrick
  // slabs, which pay off for queries far off the cloud, are then not built
  void expect_far_queries(bool yes) { far_queries_ = yes; }
  // device staging buffer for a host cloud that the caller uploads itself (prefetch on another stream)
  unsigned char* stage(size_t bytes) {
    raw_.reserve(bytes);
    return raw_.get();
  }

 private:
  bool ready_ = false;
  bool far_queries_ = true;
  GridView view_{};
  Info info_{};
  DevBuf<unsigned char> raw_;
  DevBuf<float4> pts_unsorted_, pts_sorted_;
  DevBuf<uint32_t> keys_a_, keys_b_, vals_a_, vals_b_, scan_tmp_;
  DevBuf<uint32_t> occ_, brick_rank_, brick_first_;  // brick occupancy marks, their ranks; first sorted point of every slot
  RadixSorter sorter_;
  cudaEvent_t ev_slots_ = nullptr;
  DevBuf<uint32_t> occ_bits_;
  DevBuf<int> brick_slot_;
  DevBuf<uint32_t> cell_start_;
  DevBuf<int> pos_of_;
  DevBuf<unsigned long long> sb_mask_, hb_mask_;
  DevBuf<float> brick_plane_;
  DevBuf<float> sb_plane_;
  DevBuf<uint32_t> scratch_;  // bbox (6) + counters
  unsigned* h_pin_ = nullptr; // pinned host words the build reads its counters back into
  // sharded source (world > 1)
  struct Window {
    bool active = false;
    int rank = 0, world = 1, axis = 0, planes = 0;
    int own_lo = 0, own_hi = 0, w_lo = 0, w_hi = 0;  // brick planes along `axis`: owned [own_lo, own_hi), indexed [w_lo, w_hi)
    int shard_lo = 0, shard_hi = 0;
    int64_t n_finite = 0;
    std::vector<uint32_t> plane_prefix;                // [planes + 1] finite points in the planes before each
  } win_;
  DevBuf<float4> pts_local_;
  DevBuf<uint32_t> plane_hist_, win_flags_, win_pos_;
  GridView geom_{};                                    // grid geometry of the whole cloud (pointers unset)
  int64_t n_all_ = 0;
  void index_points(const float4* pts, int64_t n_in, int64_t n_valid, const GridView& geom, cudaStream_t stream, void* trace);
  void set_window(int w_lo, int w_hi);
  const float4* window_points(cudaStream_t stream, int64_t* n_local);
};

// the index-build kernels ask for the largest shared-memory carve-out, like the kNN kernel they may share an SM with
// (gicpb_set_clouds); called once per context
void prefer_shared_carveout_grid();
void prefer_shared_carveout_sort();

// cloud difference over a group (grid_build.cu): keep[j] of the routed rows -> full[row index in rows[j].w]
void scatter_keep(const float4* rows, const unsigned char* keep, int64_t n_rows, unsigned char* full, cudaStream_t stream);
// out[i] = OR over r < n_parts of parts[r * len + i]
void or_parts(const unsigned char* parts, int n_parts, int64_t len, unsigned char* out, cudaStream_t stream);

// hand-written device-wide primitives (sort_scan.cu)
size_t scan_tmp_entries(int64_t n);
// exclusive prefix sum of n uint32 (in place allowed); tmp must hold scan_tmp_entries(n)
void exclusive_scan_u32(const uint32_t* in, uint32_t* out, int64_t n, uint32_t* tmp, cudaStream_t stream);

}  // namespace gicpb
