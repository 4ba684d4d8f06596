// engine.cu - context object, GICP outer loop and the C ABI of libgicp_b200 (include/gicp_b200.h).
//
// Host control flow restates pcl::GeneralizedIterativeClosestPoint::computeTransformation (PCL 1.8.1 gicp.hpp) as
// the reference drives it from GICPAlignment::fineAlignment / iterateFineAlignment (reference
// src/GICPAlignment.cpp:86-127): guess = identity, per outer iteration one correspondence pass (kernel) and one
// BFGS solve (host, optimizer.hpp) whose every evaluation is one cost-kernel launch (+ one NCCL all-reduce of 14
// doubles when the source is sharded over ranks).
#include <dlfcn.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <climits>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <memory>
#include <mutex>
#include <thread>

#include "../../include/gicp_b200.h"
#include "cloud_io.hpp"
#include "kernels.hpp"
#include "optimizer.hpp"

using namespace gicpb;

// ---- NCCL through dlopen -----------------------------------------------------------------------------------
namespace {

struct NcclApi {
  typedef struct ncclComm* comm_t;
  struct unique_id { char internal[128]; };
  int (*GetUniqueId)(unique_id*) = nullptr;
  int (*CommInitRank)(comm_t*, int, unique_id, int) = nullptr;
  int (*CommDestroy)(comm_t) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, comm_t, cudaStream_t) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, comm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  void* handle = nullptr;
};

NcclApi* load_nccl(const char* path, std::string& err) {
  static NcclApi api;
  if (api.handle) return &api;
  const char* name = (path && *path) ? path : "libnccl.so.2";
  void* h = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
  if (!h) {
    err = std::string("dlopen(") + name + ") failed: " + dlerror();
    return nullptr;
  }
  api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(dlsym(h, "ncclGetUniqueId"));
  api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(dlsym(h, "ncclCommInitRank"));
  api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(dlsym(h, "ncclCommDestroy"));
  api.AllReduce = reinterpret_cast<decltype(api.AllReduce)>(dlsym(h, "ncclAllReduce"));
  api.AllGather = reinterpret_cast<decltype(api.AllGather)>(dlsym(h, "ncclAllGather"));
  api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(dlsym(h, "ncclGetErrorString"));
  if (!api.GetUniqueId || !api.CommInitRank || !api.CommDestroy || !api.AllReduce || !api.AllGather || !api.GetErrorString) {
    err = "libnccl is missing a required symbol";
    return nullptr;
  }
  api.handle = h;
  return &api;
}
constexpr int kNcclFloat64 = 8, kNcclSum = 0;

struct NcclError : std::runtime_error {
  explicit NcclError(const std::string& s) : std::runtime_error(s) {}
};
struct AlignStop : std::runtime_error {
  int code;
  AlignStop(int c, const std::string& s) : std::runtime_error(s), code(c) {}
};

Rigid rigid_from_rowmajor(const float* T16) {
  Rigid r;
  for (int i = 0; i < 12; ++i) r.m[i] = T16[i];
  return r;
}
void identity16(float* T) {
  for (int i = 0; i < 16; ++i) T[i] = (i % 5 == 0) ? 1.f : 0.f;
}

// gicp.hpp applyState: R = Rz(x5) Ry(x4) Rx(x3) built in float through quaternions (Eigen AngleAxisf products),
// t.topLeft3x3 = R * t.topLeft3x3, t.col(3) += (x0,x1,x2).  Here t starts as the identity (base_transformation_).
struct Quat {
  float w, x, y, z;
};
Quat quat_axis(float angle, int axis) {
  const float ha = 0.5f * angle;
  Quat q{std::cos(ha), 0.f, 0.f, 0.f};
  const float s = std::sin(ha);
  (axis == 0 ? q.x : axis == 1 ? q.y : q.z) = s;
  return q;
}
Quat quat_mul(const Quat& a, const Quat& b) {
  return Quat{a.w * b.w - a.x * b.x - a.y * b.y - a.z * b.z, a.w * b.x + a.x * b.w + a.y * b.z - a.z * b.y,
              a.w * b.y + a.y * b.w + a.z * b.x - a.x * b.z, a.w * b.z + a.z * b.w + a.x * b.y - a.y * b.x};
}
void state_to_transform(const double* x, float* T16) {
  const Quat q = quat_mul(quat_mul(quat_axis((float)x[5], 2), quat_axis((float)x[4], 1)), quat_axis((float)x[3], 0));
  const float tx = 2.f * q.x, ty = 2.f * q.y, tz = 2.f * q.z;
  const float twx = tx * q.w, twy = ty * q.w, twz = tz * q.w;
  const float txx = tx * q.x, txy = ty * q.x, txz = tz * q.x;
  const float tyy = ty * q.y, tyz = tz * q.y, tzz = tz * q.z;
  const float R[9] = {1.f - (tyy + tzz), txy - twz, txz + twy, txy + twz, 1.f - (txx + tzz), tyz - twx,
                      txz - twy, tyz + twx, 1.f - (txx + tyy)};
  identity16(T16);
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      // R * I evaluated as Eigen's lazy product does: (r_i0*I_0j + r_i1*I_1j) + r_i2*I_2j
      float s = R[3 * i] * (j == 0 ? 1.f : 0.f);
      s = s + R[3 * i + 1] * (j == 1 ? 1.f : 0.f);
      s = s + R[3 * i + 2] * (j == 2 ? 1.f : 0.f);
      T16[4 * i + j] = s;
    }
  T16[3] += (float)x[0];
  T16[7] += (float)x[1];
  T16[11] += (float)x[2];
}
void transform_to_state(const float* T, double* x) {
  x[0] = T[3];
  x[1] = T[7];
  x[2] = T[11];
  x[3] = std::atan2((double)T[9], (double)T[10]);
  x[4] = std::asin(-(double)T[8]);
  x[5] = std::atan2((double)T[4], (double)T[0]);
}

// gicp.hpp computeRDerivative: g[3..5] = sum_ij dR(j,i) * Rsum(i,j)
void rotation_gradient(const double* x, const double* Rs, double* g) {
  const double cphi = std::cos(x[3]), sphi = std::sin(x[3]);
  const double cth = std::cos(x[4]), sth = std::sin(x[4]);
  const double cpsi = std::cos(x[5]), spsi = std::sin(x[5]);
  double dphi[9] = {0, sphi * spsi + cphi * cpsi * sth, cphi * spsi - cpsi * sphi * sth,
                    0, -cpsi * sphi + cphi * spsi * sth, -cphi * cpsi - sphi * spsi * sth,
                    0, cphi * cth, -cth * sphi};
  double dth[9] = {-cpsi * sth, cpsi * cth * sphi, cphi * cpsi * cth,
                   -spsi * sth, cth * sphi * spsi, cphi * cth * spsi,
                   -cth, -sphi * sth, -cphi * sth};
  double dpsi[9] = {-cth * spsi, -cphi * cpsi - sphi * spsi * sth, cpsi * sphi - cphi * spsi * sth,
                    cpsi * cth, -cphi * spsi + cpsi * sphi * sth, sphi * spsi + cphi * cpsi * sth,
                    0, 0, 0};
  auto inner = [&](const double* d) {
    double r = 0.0;
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) r += d[3 * j + i] * Rs[3 * i + j];
    return r;
  };
  g[3] = inner(dphi);
  g[4] = inner(dth);
  g[5] = inner(dpsi);
}

float round_up_to_float(double v) {  // smallest float >= v
  float f = (float)v;
  if ((double)f < v) f = std::nextafterf(f, INFINITY);
  return f;
}

// the correspondence gate of a max_corr_distance: PCL pairs iff (double)d2 < distance^2, i.e. d2 < the float rounded up;
// a NaN distance pairs nothing (d2 < NaN is false), as the zero gate does
float corr_gate2(double max_corr_distance) {
  const double thr = max_corr_distance * max_corr_distance;
  return std::isnan(thr) ? 0.f : round_up_to_float(thr);
}

double now_ms() {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

}  // namespace

// ---- the contexts of one gicpb_group (one process, several GPUs): what the ranks share ------------------------------------
struct gicpb_ctx;
struct GroupAbort : std::runtime_error {
  GroupAbort() : std::runtime_error("another GPU of the group failed") {}
};
struct LocalGroup {
  int world = 0;
  std::vector<gicpb_ctx*> members;
  std::vector<double> slots;  // [world][80]: small sums on their way through the host
  std::mutex mu;
  std::condition_variable cv;
  int waiting = 0;
  unsigned generation = 0;
  bool failed = false;
  // every rank's thread arrives; throws on all of them once one rank has failed (so nobody waits for ever)
  void barrier() {
    std::unique_lock<std::mutex> lk(mu);
    if (failed) throw GroupAbort();
    const unsigned gen = generation;
    if (++waiting == world) {
      waiting = 0;
      ++generation;
      cv.notify_all();
      return;
    }
    cv.wait(lk, [&] { return generation != gen || failed; });
    if (generation == gen) throw GroupAbort();
  }
  void fail() {
    std::lock_guard<std::mutex> lk(mu);
    failed = true;
    cv.notify_all();
  }
  void reset() {
    std::lock_guard<std::mutex> lk(mu);
    failed = false;
    waiting = 0;
  }
};

// ---- context ------------------------------------------------------------------------------------------------
struct gicpb_ctx {
  int device = 0;
  int num_sms = 148;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr;  // uploads started by gicpb_prefetch_cloud run here, beside the compute stream
  cudaStream_t aux_stream = nullptr;   // gicpb_set_clouds: target covariances beside the source index build
  cudaEvent_t ev_aux = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_order = nullptr;
  struct Prefetch {
    const void* host = nullptr;
    int64_t n = 0, stride = 0;
    unsigned char* dev = nullptr;
    int64_t dev_stride = 0;  // stride of the device copy (12 when the cloud went through the packed staged upload)
    cudaEvent_t done = nullptr;
    bool pending = false;
    bool sharded = false;    // only this rank's slice of the rows was uploaded: the other ranks' are gathered by do_prefetch
                             // on the copy stream (one process per GPU) or by take_prefetch (in-process group)
    int64_t chunk_rows = 0;  // rows per rank in the gathered buffer (the last rank's slice may be shorter, or empty)
  } prefetch[4];  // 0 target, 1 source, 2 subtract, 3 difference input (gicpb_group_cloud_difference)
  gicpb_params prm{};
  std::string err;

  GridIndex tgt, src, sub, clu;
  VoxelGrid voxel;
  DevBuf<int> uf_parent, uf_root;
  bool cov_ready = false;
  bool tgt_normals_gathered = false;  // start_target_cov has already exchanged the target's normal chunks (second stream)
  int shard_lo = 0, shard_hi = 0;
  DevBuf<double> n_tgt, n_src;
  DevBuf<int> pair_pos;
  DevBuf<float> pair_d2;
  DevBuf<float4> pair_tgt;
  DevBuf<double> maha;  // 6 doubles (or 6 floats) per shard point
  bool pairs_valid = false;
  bool pairs_fp32 = false;
  DevBuf<double> partials;
  DevBuf<unsigned> ticket;
  DevBuf<double> d_sums;          // 16 doubles on the device (NCCL path / fitness)
  DevBuf<double> mom_partials;    // moments pass: per-block rows
  DevBuf<double> d_mom;           // 80 doubles on the device
  double* h_mom = nullptr;        // pinned: the 74 moment sums of the current outer iteration (all ranks)
  float mom_T0[16];               // the transform the moments were taken around
  bool mom_valid = false;
  unsigned eval_stamp = 0;        // last stamp handed to a cost kernel (run_cost polls for it)
  double* h_sums = nullptr;       // pinned, mapped
  double* h_sums_dev = nullptr;   // device alias of h_sums
  unsigned* h_far = nullptr;      // pinned: far-query count of the last correspondence pass
  // persistent evaluation kernel (cost.cu cost_persistent_kernel): one launch per outer iteration, one command per evaluation
  CostCommand* h_cmd = nullptr;      // pinned, mapped: the host writes commands here
  CostCommand* h_cmd_dev = nullptr;  // device alias of h_cmd
  DevBuf<CostCommand> d_cmd;         // block 0 republishes every command here for the other blocks
  unsigned cost_epoch = 0, cost_count = 0;
  CostPersistentShape cost_shape{};  // block shape of the last resident launch
  bool cost_live = false;            // a persistent kernel is (believed to be) resident on the stream
  int smem_optin = 0;
  unsigned long long cost_idle_ns = 200000000ull;  // the kernel ends itself after this long without a command
  double cost_test_stall_ms = 0;     // test knob (GICPB_COST_TEST_STALL_MS): the host idles this long before every command
  DevBuf<float4> queries;
  DevBuf<unsigned char> io_a, io_b;
  HostStager stager;              // pageable host clouds reach the device through its pinned ring (upload.hpp)
  DevBuf<unsigned long long> counter;
  DevBuf<unsigned char> far_flags;  // near -> far hand-over (kernels.hpp FarWork)
  DevBuf<unsigned> far_counter;
  // gicpb_group_cloud_difference: routing of the input rows, this rank's keep bytes in row order, the pieces of its mask slice
  DevBuf<uint32_t> route_flags, route_pos, route_tmp;
  DevBuf<unsigned char> keep_full, keep_parts;

  NcclApi* nccl = nullptr;
  NcclApi::comm_t comm = nullptr;
  int rank = 0, world = 1;
  LocalGroup* local = nullptr;  // member of a gicpb_group: the collectives go over peer copies / the host, not NCCL
  bool peer_ipc = false;        // peer.peers[] are cudaIpc mappings (closed on destroy)
  // fused cost + cross-GPU sum over peer memory (kernels.hpp PeerReduce); falls back to ncclAllReduce when not set up
  PeerSlots* peer_own = nullptr;
  PeerReduce peer{};
  bool peer_ready = false;

  // accounting
  double ms_corr = 0, ms_cost = 0;
  int64_t far_queries = 0;
  int64_t cost_evals = 0;
  int64_t window_widened = 0;  // times a sharded source had to be indexed whole after all (GridIndex::widen)
};

namespace {

struct DeviceGuard {
  int prev = 0;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
  }
  ~DeviceGuard() { cudaSetDevice(prev); }
};

template <typename F>
int guarded(gicpb_ctx* ctx, F&& fn) {
  if (!ctx) return GICPB_E_BADARG;
  DeviceGuard guard(ctx->device);
  try {
    fn();
    return GICPB_OK;
  } catch (const ArgError& e) {
    ctx->err = e.what();
    return GICPB_E_BADARG;
  } catch (const StateError& e) {
    ctx->err = e.what();
    return GICPB_E_STATE;
  } catch (const CudaError& e) {
    ctx->err = e.what();
    return GICPB_E_CUDA;
  } catch (const NcclError& e) {
    ctx->err = e.what();
    return GICPB_E_NCCL;
  } catch (const AlignStop& e) {
    ctx->err = e.what();
    return e.code;
  } catch (const GroupAbort& e) {
    ctx->err = e.what();
    return GICPB_E_STATE;
  } catch (const std::exception& e) {
    ctx->err = e.what();
    return GICPB_E_CUDA;
  }
}

void check_nccl(gicpb_ctx* c, int rc, const char* what) {
  if (rc != 0) throw NcclError(std::string(what) + ": " + c->nccl->GetErrorString(rc));
}

// in-process group: `count` (<= 80) doubles of every rank through the host, added in rank order on every rank (identical sums)
void local_all_reduce(gicpb_ctx* c, double* dev, int count) {
  LocalGroup* lg = c->local;
  double* mine = lg->slots.data() + 80 * (size_t)c->rank;
  GICPB_CUDA(cudaMemcpyAsync(mine, dev, (size_t)count * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  GICPB_CUDA(cudaStreamSynchronize(c->stream));
  lg->barrier();
  double sum[80];
  for (int k = 0; k < count; ++k) {
    double v = 0.0;
    for (int r = 0; r < lg->world; ++r) v += lg->slots[80 * (size_t)r + k];
    sum[k] = v;
  }
  lg->barrier();  // everybody has read the slots: they may be written again
  GICPB_CUDA(cudaMemcpyAsync(dev, sum, (size_t)count * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  GICPB_CUDA(cudaStreamSynchronize(c->stream));
}

void all_reduce_sum(gicpb_ctx* c, double* dev, int count) {
  if (c->world <= 1) return;
  if (c->local) {
    local_all_reduce(c, dev, count);
    return;
  }
  check_nccl(c, c->nccl->AllReduce(dev, dev, (size_t)count, kNcclFloat64, kNcclSum, c->comm, c->stream), "ncclAllReduce");
}

constexpr int kFarBlocksPerSm = 6;

FarWork far_work(gicpb_ctx* c, int64_t n_items, int near_rings = kNearMaxRing) {
  c->far_flags.reserve((size_t)std::max<int64_t>(n_items, 1) + kFarTile);
  c->far_counter.reserve(4);
  return FarWork{c->far_flags.get(), c->far_counter.get(), c->num_sms * kFarBlocksPerSm, near_rings, far_tile_for(n_items)};
}

// The shard follows the context's current rank / world: a member of a gicpb_group is rank r of n during a group call and a
// single-GPU context (world 1) between them, while its source index stays the one the group built (a window of brick planes).
// With world 1 the window is widened to the whole source and the shard is all of it; the next group call takes the rank's
// planes again.  Covariances and pairs belong to one shard: they are dropped whenever the shard changes.
void update_shard(gicpb_ctx* c) {
  const int lo = c->shard_lo, hi = c->shard_hi;
  if (c->world == 1 && c->src.ready() && c->src.windowed()) c->src.widen(c->stream);
  if (c->world > 1 && c->src.ready() && c->src.plane_sharded()) {  // the rank's brick planes of the (windowed) source index
    c->shard_lo = c->src.shard_lo();
    c->shard_hi = c->src.shard_hi();
  } else {
    const int64_t n = c->src.ready() ? c->src.n_indexed() : 0;
    c->shard_lo = (int)(n * c->rank / c->world);
    c->shard_hi = (int)(n * (c->rank + 1) / c->world);
  }
  if (c->shard_lo != lo || c->shard_hi != hi) {
    c->cov_ready = false;
    c->pairs_valid = false;
  }
}

// Target covariances are needed in full on every rank, but each is a function of the target cloud alone: every rank
// computes one contiguous chunk of the (identically sorted) target (start_target_cov, on `knn_stream`) and the chunks
// are all-gathered in place (finish_covariances, on the context's stream).
int target_chunk(const gicpb_ctx* c) { return (c->tgt.n_indexed() + c->world - 1) / c->world; }

void check_k(const gicpb_ctx* c) {
  const int k = c->prm.k_correspondences;
  if (k < 2 || k > 32) throw ArgError("k_correspondences must be in [2, 32]");
}

void start_target_cov(gicpb_ctx* c, cudaStream_t knn_stream) {
  const int k = c->prm.k_correspondences;
  const int nt = c->tgt.n_indexed();
  const int chunk = target_chunk(c);
  const int t_lo = std::min(nt, c->rank * chunk), t_hi = std::min(nt, t_lo + chunk);
  c->n_tgt.reserve(3 * (size_t)chunk * c->world);
  const FarWork fw = far_work(c, chunk);
  launch_knn_covariances(c->tgt.view(), t_lo, t_hi, k, c->n_tgt.get() + 3 * (size_t)t_lo, nullptr, nullptr, fw, knn_stream);
  c->tgt_normals_gathered = false;
  if (c->world > 1 && !c->local && knn_stream != c->stream) {
    // gicpb_set_clouds: the chunks are exchanged on the second stream too, beside the source's index build (a chain of short
    // kernels that leaves the links and most of the SMs idle), not in front of the source's covariance pass
    check_nccl(c, c->nccl->AllGather(c->n_tgt.get() + 3 * (size_t)c->rank * chunk, c->n_tgt.get(), 3 * (size_t)chunk,
                                     kNcclFloat64, c->comm, knn_stream), "ncclAllGather");
    c->tgt_normals_gathered = true;
  }
}

// the rest, on the context's stream (which must already be ordered after start_target_cov's kernels)
void finish_covariances(gicpb_ctx* c) {
  const int k = c->prm.k_correspondences;
  update_shard(c);
  const int ns = c->shard_hi - c->shard_lo;
  const int chunk = target_chunk(c);
  c->n_src.reserve(3 * (size_t)std::max(ns, 1));
  const FarWork fw = far_work(c, std::max(chunk, ns));
  if (c->world > 1 && c->local) {
    // in-process group: every rank's chunk is complete and its buffer in place, then the other chunks come over NVLink
    GICPB_CUDA(cudaStreamSynchronize(c->stream));
    c->local->barrier();
    for (int r = 0; r < c->world; ++r) {
      if (r == c->rank) continue;
      const gicpb_ctx* o = c->local->members[(size_t)r];
      GICPB_CUDA(cudaMemcpyPeerAsync(c->n_tgt.get() + 3 * (size_t)r * chunk, c->device, o->n_tgt.get() + 3 * (size_t)r * chunk,
                                     o->device, 3 * (size_t)chunk * sizeof(double), c->stream));
    }
  } else if (c->world > 1 && !c->tgt_normals_gathered) {
    check_nccl(c, c->nccl->AllGather(c->n_tgt.get() + 3 * (size_t)c->rank * chunk, c->n_tgt.get(), 3 * (size_t)chunk,
                                     kNcclFloat64, c->comm, c->stream), "ncclAllGather");
  }
  c->tgt_normals_gathered = false;
  const GridIndex::KnnWindow win = c->src.knn_window();
  unsigned* violations = c->far_counter.get() + 2;  // far_work() reserved 4 words; [0..1] belong to the far hand-over
  if (win.axis >= 0) {
    GICPB_CUDA(cudaMemsetAsync(violations, 0, sizeof(unsigned), c->stream));
    launch_knn_covariances(c->src.view(), c->shard_lo, c->shard_hi, k, c->n_src.get(), nullptr, nullptr, fw, c->stream, &win,
                           violations);
    GICPB_CUDA(cudaMemcpyAsync(c->h_far + 2, violations, sizeof(unsigned), cudaMemcpyDeviceToHost, c->stream));
  } else {
    launch_knn_covariances(c->src.view(), c->shard_lo, c->shard_hi, k, c->n_src.get(), nullptr, nullptr, fw, c->stream);
  }
  GICPB_CUDA(cudaStreamSynchronize(c->stream));
  if (c->world > 1 && c->local) c->local->barrier();  // nobody touches its n_tgt again before every copy out of it is done
  if (win.axis >= 0 && c->h_far[2] != 0u) {
    // some neighbourhoods of this rank's shard reach beyond the halo of its window (a sparse region): index the whole source
    // after all - the shard stays the same set of points - and take the covariances from that
    c->src.widen(c->stream);
    update_shard(c);
    c->n_src.reserve(3 * (size_t)std::max(c->shard_hi - c->shard_lo, 1));
    launch_knn_covariances(c->src.view(), c->shard_lo, c->shard_hi, k, c->n_src.get(), nullptr, nullptr,
                           far_work(c, std::max(chunk, c->shard_hi - c->shard_lo)), c->stream);
    GICPB_CUDA(cudaStreamSynchronize(c->stream));
    ++c->window_widened;
  }
  c->cov_ready = true;
  c->pairs_valid = false;
}

void ensure_covariances(gicpb_ctx* c) {
  update_shard(c);
  if (c->cov_ready) return;
  if (!c->tgt.ready() || !c->src.ready()) throw StateError("set_target and set_source must be called first");
  check_k(c);
  const int k = c->prm.k_correspondences;
  if (k > c->tgt.n_indexed() || k > c->src.n_finite_total())
    throw AlignStop(GICPB_E_TOO_FEW_POINTS, "k_correspondences exceeds the number of points in a cloud");
  start_target_cov(c, c->stream);
  finish_covariances(c);
}

void ensure_pair_buffers(gicpb_ctx* c) {
  const size_t ns = (size_t)std::max(c->shard_hi - c->shard_lo, 1);
  c->pair_pos.reserve(ns);
  c->pair_d2.reserve(ns);
  c->pair_tgt.reserve(ns);
  c->maha.reserve(6 * ns);
  c->partials.reserve((size_t)c->num_sms * 4 * 16 + 2 * (size_t)fitness_partial_rows((int)ns, c->num_sms * kFarBlocksPerSm) + 64);
  c->ticket.reserve(4);
  c->d_sums.reserve(16);
  c->mom_partials.reserve((size_t)c->num_sms * 80);
  c->d_mom.reserve(80);
}

// one correspondence pass under transform T (row-major 4x4 float)
void run_correspondences(gicpb_ctx* c, const float* T16, bool first, int near_rings = 0) {
  if (near_rings <= 0) near_rings = first ? 1 : kNearMaxRing;
  ensure_pair_buffers(c);
  const Rigid T = rigid_from_rowmajor(T16);
  RotD R;
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) R.m[3 * i + j] = (double)T16[4 * i + j];
  const float gate2 = corr_gate2(c->prm.max_corr_distance);
  const bool fp32 = c->prm.mahalanobis_fp32 != 0;
  const bool use_prev = c->prm.use_previous_match != 0 && !first && c->pairs_valid && c->pairs_fp32 == fp32;
  GICPB_CUDA(cudaEventRecord(c->ev0, c->stream));
  launch_correspondences(c->tgt.view(), c->src.sorted_points(), c->shard_lo, c->shard_hi, T, R, gate2, c->n_src.get(),
                         c->n_tgt.get(), c->prm.gicp_epsilon, c->pair_pos.get(), c->pair_d2.get(), c->pair_tgt.get(),
                         c->maha.get(), fp32, use_prev, far_work(c, c->shard_hi - c->shard_lo, near_rings), c->stream);
  GICPB_CUDA(cudaEventRecord(c->ev1, c->stream));
  GICPB_CUDA(cudaMemcpyAsync(c->h_far, c->far_counter.get() + 1, sizeof(unsigned), cudaMemcpyDeviceToHost, c->stream));
  c->pairs_valid = true;
  c->pairs_fp32 = fp32;
  c->mom_valid = false;
  if (c->prm.cost_moments != 0) {
    // one pass over the pairs of this outer iteration: the 74 second-order moments around T (cost.cu); every cost /
    // gradient evaluation of the inner solve is then host arithmetic.  Sharded: ONE all-reduce per outer iteration.
    const int n = c->shard_hi - c->shard_lo;
    launch_moments(c->src.sorted_points(), c->shard_lo, n, c->pair_tgt.get(), c->maha.get(), fp32, T,
                   c->mom_partials.get(), c->ticket.get(), c->d_mom.get(), moments_grid_blocks(n, c->num_sms), c->stream);
    all_reduce_sum(c, c->d_mom.get(), kMomentSums);
    GICPB_CUDA(cudaMemcpyAsync(c->h_mom, c->d_mom.get(), kMomentSums * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    std::memcpy(c->mom_T0, T16, sizeof(c->mom_T0));
  }
}

// the 14 sums of run_cost from the moments (cost.cu header): D = [R|t](x) - [R0|t0], G = B + H D
void cost_from_moments(gicpb_ctx* c, const double* x, double* sums) {
  if (!c->mom_valid) {
    GICPB_CUDA(cudaStreamSynchronize(c->stream));
    c->mom_valid = true;
  }
  float T16[16];
  state_to_transform(x, T16);
  double D[3][4];
  for (int a = 0; a < 3; ++a)
    for (int k = 0; k < 4; ++k) D[a][k] = (double)T16[4 * a + k] - (double)c->mom_T0[4 * a + k];
  const double* mo = c->h_mom;
  static const int kl_of[4][4] = {{0, 1, 2, 3}, {1, 4, 5, 6}, {2, 5, 7, 8}, {3, 6, 8, 9}};
  static const int ab_of[3][3] = {{0, 1, 2}, {1, 3, 4}, {2, 4, 5}};
  double G[3][4];
  double f = mo[0];
  for (int a = 0; a < 3; ++a)
    for (int k = 0; k < 4; ++k) {
      double hd = 0.0;
      for (int b = 0; b < 3; ++b)
        for (int l = 0; l < 4; ++l) hd += mo[14 + 6 * kl_of[k][l] + ab_of[a][b]] * D[b][l];
      const double B = mo[1 + 4 * a + k];
      G[a][k] = B + hd;
      f += D[a][k] * (B + G[a][k]);
    }
  sums[0] = f;
  for (int a = 0; a < 3; ++a) sums[1 + a] = G[a][3];
  for (int k = 0; k < 3; ++k)
    for (int a = 0; a < 3; ++a) sums[4 + 3 * k + a] = G[a][k];
  sums[13] = mo[13];
  ++c->cost_evals;
}

// ---- persistent evaluation session (one per inner solve) --------------------------------------------------------------------
bool cost_session_wanted(const gicpb_ctx* c) {
  return c->prm.cost_persistent != 0 && c->prm.cost_moments == 0 && (c->world == 1 || c->peer_ready) && c->h_cmd != nullptr &&
         c->shard_hi > c->shard_lo;
}

void cost_session_begin(gicpb_ctx* c) {
  // 12 bits of the command sequence word, never 0, and consecutive launches alternate parity (so command slot) also where the
  // sequence wraps: 1 ... 4094, 1, ...
  c->cost_epoch = (c->cost_epoch % 4094u) + 1u;
  c->cost_count = 0;
  c->d_cmd.reserve(1);
  const bool fused = c->world > 1 && c->peer_ready;
  launch_cost_persistent(c->src.sorted_points(), c->shard_lo, c->shard_hi - c->shard_lo, c->pair_tgt.get(), c->maha.get(),
                         c->pairs_fp32, c->h_cmd_dev + (c->cost_epoch & 1u), c->d_cmd.get(), c->cost_epoch, c->partials.get(), c->ticket.get(),
                         c->h_sums_dev, fused ? &c->peer : nullptr, c->cost_idle_ns, cost_persistent_blocks(c->num_sms),
                         c->smem_optin, c->stream, &c->cost_shape);
  c->cost_live = true;
}

void cost_session_send(gicpb_ctx* c, unsigned op, const float* T16, unsigned stamp, unsigned peer_seq) {
  // two slots, alternating with the launch epoch: the EXIT of one launch and the first command of the next never share one
  CostCommand* h = c->h_cmd + (c->cost_epoch & 1u);
  ++c->cost_count;
  const unsigned seq = (c->cost_epoch << 20) | (c->cost_count & 0xfffffu);
  unsigned w[15] = {0};
  if (T16) std::memcpy(w, T16, 12 * sizeof(float));
  w[12] = op;
  w[13] = stamp;
  w[14] = peer_seq;
  for (int k = 0; k < 5; ++k) {
    volatile unsigned* ch = h->chunk[k].w;
    ch[0] = w[3 * k];
    ch[1] = w[3 * k + 1];
    ch[2] = w[3 * k + 2];
  }
  std::atomic_thread_fence(std::memory_order_release);  // payloads before sequence words (and x86 keeps store order)
  for (int k = 0; k < 5; ++k) *reinterpret_cast<volatile unsigned*>(&h->chunk[k].seq) = seq;
}

void cost_session_end(gicpb_ctx* c) {
  if (!c->cost_live) return;
  c->cost_live = false;
  cost_session_send(c, kCostOpExit, nullptr, 0u, 0u);  // nobody waits: the next kernel on the stream queues behind the exit
}

struct CostSession {  // ends the resident kernel however the inner solve is left
  gicpb_ctx* c;
  explicit CostSession(gicpb_ctx* ctx) : c(ctx) {
    if (cost_session_wanted(c)) cost_session_begin(c);
  }
  ~CostSession() { cost_session_end(c); }
};

// raw sums of one evaluation at x (all ranks): s[0] = sum r.Mr, s[1..3] = sum Mr, s[4..12] = sum p (Mr)^T, s[13] = m
void run_cost(gicpb_ctx* c, const double* x, double* sums) {
  if (c->prm.cost_moments != 0 && c->pairs_valid) {
    cost_from_moments(c, x, sums);
    return;
  }
  float T16[16];
  state_to_transform(x, T16);
  const Rigid T = rigid_from_rowmajor(T16);
  const int n = c->shard_hi - c->shard_lo;
  const int blocks = cost_grid_blocks(n, c->num_sms);
  const bool fused = c->world > 1 && c->peer_ready;
  double* out = (c->world > 1 && !fused) ? c->d_sums.get() : c->h_sums_dev;
  if (fused) {
    if (++c->peer.seq == 0u) c->peer.seq = 1u;
  }
  // the sums land in mapped host memory: the host polls the stamp the kernel stores after them (no driver call between
  // the kernel's last store and the optimiser's next step); the NCCL path still synchronises the stream
  const bool polled = out == c->h_sums_dev;
  unsigned stamp = 0;
  if (polled) {
    if (++c->eval_stamp == 0u || c->eval_stamp >= (1u << 30)) {
      c->eval_stamp = 1u;
      // no kernel is in flight here (every evaluation is waited for): forget the pre-wrap stamps
      std::memset(c->h_sums + kCostOutWords, 0, 32 * sizeof(unsigned long long));
    }
    stamp = c->eval_stamp;
  }
  const bool session = c->cost_live && polled;
  if (session && c->cost_test_stall_ms > 0) {
    const double t_end = now_ms() + c->cost_test_stall_ms;
    while (now_ms() < t_end) {
    }
  }
  if (session)
    cost_session_send(c, kCostOpEval, T16, stamp, c->peer.seq);
  else
    launch_cost(c->src.sorted_points(), c->shard_lo, n, c->pair_tgt.get(), c->maha.get(), c->pairs_fp32, T,
                c->partials.get(), c->ticket.get(), out, blocks, c->stream, fused ? &c->peer : nullptr, stamp);
  if (polled) {
    // 28 self-validating words (kernels.hpp launch_cost): every one must show this evaluation's stamp
    const volatile unsigned long long* words = reinterpret_cast<const volatile unsigned long long*>(c->h_sums + kCostOutWords);
    unsigned long long got[2 * kCostSums];
    int have = 0;  // words [0, have) have arrived
    auto arrived = [&] {
      while (have < 2 * kCostSums) {
        const unsigned long long w = words[have];
        if ((unsigned)(w & 0xffffffffull) != stamp) return false;
        got[have++] = w;
      }
      return true;
    };
    int relaunches = 0;
    for (unsigned spins = 1; !arrived(); ++spins) {
      if ((spins & 0x3fffu) == 0u) {  // every ~16 k polls: has the kernel died, or finished without publishing?
        const cudaError_t q = cudaStreamQuery(c->stream);
        if (q == cudaSuccess) {
          if (arrived()) break;
          if (session && relaunches < 3) {
            // the resident kernel ended itself (no command for cost_idle_ns: this thread was descheduled) before it saw
            // the command: launch it again and repeat the command
            ++relaunches;
            cost_session_begin(c);
            cost_session_send(c, kCostOpEval, T16, stamp, c->peer.seq);
            continue;
          }
          throw CudaError("cost kernel finished without publishing its sums");
        }
        if (q != cudaErrorNotReady) GICPB_CUDA(q);
        (void)cudaGetLastError();
      }
    }
    for (int i = 0; i < kCostSums; ++i) {
      const unsigned long long bits = (got[2 * i + 1] & 0xffffffff00000000ull) | (got[2 * i] >> 32);
      std::memcpy(&c->h_sums[i], &bits, sizeof(double));
    }
  } else {
    all_reduce_sum(c, c->d_sums.get(), kCostSums);
    GICPB_CUDA(cudaMemcpyAsync(c->h_sums, c->d_sums.get(), kCostSums * sizeof(double), cudaMemcpyDeviceToHost,
                               c->stream));
    GICPB_CUDA(cudaStreamSynchronize(c->stream));
  }
  for (int i = 0; i < kCostSums; ++i) sums[i] = c->h_sums[i];
  if (fused && std::isnan(sums[13])) {
    c->peer_ready = false;  // the slot flags are out of step from here on: this context goes back to ncclAllReduce
    throw NcclError("peer-memory reduction timed out: a rank did not launch this evaluation (GICPB_PEER_TIMEOUT_MS)");
  }
  ++c->cost_evals;
}

// f and g[6] exactly as OptimizationFunctorWithIndices::fdf scales them; returns the pair count
double cost_from_sums(const double* x, const double* s, double* f, double* g) {
  const double m = s[13];
  *f = s[0] / m;
  const double sc = 2.0 / m;
  g[0] = s[1] * sc;
  g[1] = s[2] * sc;
  g[2] = s[3] * sc;
  double Rs[9];
  for (int i = 0; i < 9; ++i) Rs[i] = s[4 + i] * sc;
  rotation_gradient(x, Rs, g);
  return m;
}

void do_align(gicpb_ctx* c, gicpb_align_result* out) {
  const double t_begin = now_ms();
  std::memset(out, 0, sizeof(*out));
  identity16(out->transform);
  if (!c->tgt.ready() || !c->src.ready()) throw StateError("set_target and set_source must be called first");
  ensure_covariances(c);
  ensure_pair_buffers(c);
  c->ms_corr = c->ms_cost = 0;
  c->cost_evals = 0;
  c->far_queries = 0;

  float T[16], prev[16];
  identity16(T);
  identity16(prev);
  int nr_iterations = 0, inner_total = 0;
  bool converged = false;
  int status = GICPB_OK;
  int64_t corr_queries = 0;
  double pairs_last = 0;
  const int max_iterations = c->prm.max_iterations;

  while (!converged) {
    run_correspondences(c, T, nr_iterations == 0);
    corr_queries += c->src.n_finite_total();
    std::memcpy(prev, T, sizeof(T));
    CostSession session(c);  // resident evaluation kernel for this inner solve (queued behind the correspondence kernels)

    double x[6];
    transform_to_state(T, x);
    double m_pairs = 0;
    bool first_eval = true;
    Bfgs6 bfgs([&](const double* xx, double* f, double* g) {
      double s[kCostSums];
      const double t0 = now_ms();
      run_cost(c, xx, s);
      c->ms_cost += now_ms() - t0;
      if (first_eval) {
        first_eval = false;
        float ms = 0.f;
        // run_cost may have polled instead of synchronising: the kernel it waited for ran after ev1 on this stream
        if (cudaEventSynchronize(c->ev1) == cudaSuccess && cudaEventElapsedTime(&ms, c->ev0, c->ev1) == cudaSuccess)
          c->ms_corr += ms;
        c->far_queries += c->h_far[0];
      }
      m_pairs = s[13];
      if (m_pairs < 4.0) return false;  // NotEnoughPointsException (< 4 correspondences)
      cost_from_sums(xx, s, f, g);
      return true;
    });
    if (!bfgs.init(x)) {
      pairs_last = m_pairs;
      status = GICPB_E_NOT_ENOUGH_CORRESPONDENCES;
      break;
    }
    pairs_last = m_pairs;
    int inner = 0;
    BfgsStatus result = BfgsStatus::kRunning;
    do {
      ++inner;
      result = bfgs.step(x);
      if (result != BfgsStatus::kSuccess) break;
      result = (bfgs.gradient_norm() < 1e-2) ? BfgsStatus::kSuccess : BfgsStatus::kRunning;
    } while (result == BfgsStatus::kRunning && inner < c->prm.max_inner_iterations);
    inner_total += inner;
    if (result == BfgsStatus::kNoProgress || result == BfgsStatus::kSuccess || inner == c->prm.max_inner_iterations) {
      state_to_transform(x, T);
    } else {
      status = GICPB_E_SOLVER;
      break;
    }
    double delta = 0.0;
    for (int k = 0; k < 4; ++k)
      for (int l = 0; l < 4; ++l) {
        const double ratio = (k < 3 && l < 3) ? 1.0 / c->prm.rotation_epsilon : 1.0 / c->prm.transformation_epsilon;
        const double cd = ratio * std::fabs((double)(prev[4 * k + l] - T[4 * k + l]));
        if (cd > delta) delta = cd;
      }
    ++nr_iterations;
    if (nr_iterations >= max_iterations || delta < 1) {
      converged = true;
      std::memcpy(prev, T, sizeof(T));
    }
  }
  std::memcpy(out->transform, prev, sizeof(prev));  // final_transformation_ = previous_transformation_ * guess
  out->converged = converged ? 1 : 0;
  out->status = status;
  out->outer_iterations = nr_iterations;
  out->inner_iterations = inner_total;
  out->cost_evaluations = c->cost_evals;
  out->corr_queries = corr_queries;
  out->corr_pairs_last = (int64_t)pairs_last;
  out->corr_far_queries = c->far_queries;
  out->ms_corr = c->ms_corr;
  out->ms_cost = c->ms_cost;
  out->ms_total = now_ms() - t_begin;
  if (status == GICPB_E_NOT_ENOUGH_CORRESPONDENCES) c->err = "fewer than 4 correspondences inside the distance gate";
  if (status == GICPB_E_SOLVER) c->err = "BFGS did not converge";
}

// `bytes` of host memory onto the device as they are: through the pinned ring when the memory is pageable and large
void upload_bytes(gicpb_ctx* c, unsigned char* dst, const void* src, size_t bytes) {
  if (HostStager::wants(src, (int64_t)bytes, 1))
    c->stager.upload(dst, static_cast<const unsigned char*>(src), (int64_t)bytes, 1, 1, c->stream);
  else
    GICPB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->stream));
}

// `bytes` of device memory into host memory; the stream is synchronised when this returns
void download_bytes(gicpb_ctx* c, void* dst, const unsigned char* src_dev, size_t bytes) {
  if (HostStager::wants(dst, (int64_t)bytes, 1)) {
    c->stager.download(static_cast<unsigned char*>(dst), src_dev, bytes, c->stream);
  } else {
    GICPB_CUDA(cudaMemcpyAsync(dst, src_dev, bytes, cudaMemcpyDeviceToHost, c->stream));
  }
  GICPB_CUDA(cudaStreamSynchronize(c->stream));
}

// xyz of a host cloud onto the device (only x, y, z are read from the staged copy); *stride becomes the stride of the copy
const unsigned char* stage_in(gicpb_ctx* c, DevBuf<unsigned char>& buf, const void* p, int64_t n, int64_t* stride,
                              bool on_device) {
  if (on_device) return static_cast<const unsigned char*>(p);
  buf.reserve((size_t)n * *stride);
  if (HostStager::wants(p, n, *stride)) {
    c->stager.upload(buf.get(), static_cast<const unsigned char*>(p), n, *stride, 12, c->stream);
    *stride = 12;
  } else {
    GICPB_CUDA(cudaMemcpyAsync(buf.get(), p, (size_t)(n - 1) * *stride + 12, cudaMemcpyHostToDevice, c->stream));
  }
  return buf.get();
}

void check_cloud_args(const void* p, int64_t n, int64_t stride) {
  if (!p) throw ArgError("null cloud pointer");
  if (n <= 0) throw ArgError("cloud is empty");
  if (stride < 12 || stride % 4) throw ArgError("stride must be a multiple of 4 and >= 12");
  if (reinterpret_cast<uintptr_t>(p) % 4) throw ArgError("cloud pointer must be 4-byte aligned");
}

// Sharded upload (world > 1, host clouds): every rank is given the same clouds, so each uploads only its 1 / world of the
// rows (packed xyz, 12 bytes per point) and the slices are exchanged between the GPUs - one in-place ncclAllGather, or peer
// copies inside a gicpb_group - instead of every rank pulling both whole clouds through its host.  GICPB_SHARD_UPLOAD=0: off.
bool shard_uploads(const gicpb_ctx* c) {
  static const bool enabled = [] {
    const char* e = std::getenv("GICPB_SHARD_UPLOAD");
    return !(e && *e == '0');
  }();
  return enabled && c->world > 1 && (c->local != nullptr || c->comm != nullptr);
}

// in-process group: the other members' slices are copied over from their staging buffers when the cloud is set
void gather_slices(gicpb_ctx* c, int which) {
  gicpb_ctx::Prefetch& p = c->prefetch[which];
  const size_t chunk_bytes = (size_t)p.chunk_rows * 12;
  GICPB_CUDA(cudaStreamSynchronize(c->stream));  // this rank's slice is in place (the stream waits for the copy stream)
  c->local->barrier();
  for (int r = 0; r < c->world; ++r) {
    if (r == c->rank) continue;
    const int64_t lo = std::min<int64_t>(p.n, (int64_t)r * p.chunk_rows), hi = std::min<int64_t>(p.n, lo + p.chunk_rows);
    if (hi <= lo) continue;
    const gicpb_ctx* o = c->local->members[(size_t)r];
    GICPB_CUDA(cudaMemcpyPeerAsync(p.dev + (size_t)r * chunk_bytes, c->device, o->prefetch[which].dev + (size_t)r * chunk_bytes,
                                   o->device, (size_t)(hi - lo) * 12, c->stream));
  }
  GICPB_CUDA(cudaStreamSynchronize(c->stream));
  c->local->barrier();  // every rank has what it needs from the others' staging buffers
}

// starts the upload of a host cloud on the copy stream (gicpb_prefetch_cloud)
void do_prefetch(gicpb_ctx* c, int which, const void* xyz, int64_t n, int64_t stride) {
  gicpb_ctx::Prefetch& p = c->prefetch[which];
  if (p.pending) GICPB_CUDA(cudaEventSynchronize(p.done));
  // the index of this cloud may still be in use on the compute stream (its staging buffer is about to be overwritten)
  GICPB_CUDA(cudaEventRecord(c->ev_order, c->stream));
  GICPB_CUDA(cudaStreamWaitEvent(c->copy_stream, c->ev_order, 0));
  auto stage = [&](size_t bytes) {  // the cloud's index keeps its staging buffer; the difference input goes to io_a
    if (which == 3) {
      c->io_a.reserve(bytes);
      return c->io_a.get();
    }
    return (which == 0 ? c->tgt : which == 1 ? c->src : c->sub).stage(bytes);
  };
  const unsigned char* src = static_cast<const unsigned char*>(xyz);
  p.sharded = shard_uploads(c);
  if (p.sharded) {
    p.chunk_rows = (n + c->world - 1) / c->world;
    const int64_t lo = std::min<int64_t>(n, (int64_t)c->rank * p.chunk_rows), hi = std::min<int64_t>(n, lo + p.chunk_rows);
    p.dev = stage((size_t)p.chunk_rows * c->world * 12);
    p.dev_stride = 12;
    if (hi > lo) {
      if (stride == 12 && !HostStager::wants(src + lo * stride, hi - lo, stride))
        GICPB_CUDA(cudaMemcpyAsync(p.dev + (size_t)lo * 12, src + lo * stride, (size_t)(hi - lo) * 12, cudaMemcpyHostToDevice,
                                   c->copy_stream));
      else  // wider rows, or pageable memory: packed by the host threads of the pinned ring
        c->stager.upload(p.dev + (size_t)lo * 12, src + lo * stride, hi - lo, stride, 12, c->copy_stream);
    }
  } else {
    p.dev = stage((size_t)n * stride);
    p.dev_stride = stride;
    if (HostStager::wants(xyz, n, stride)) {  // pageable: packed xyz rows (this call then lasts as long as the gather)
      c->stager.upload(p.dev, src, n, stride, 12, c->copy_stream);
      p.dev_stride = 12;
    } else {
      GICPB_CUDA(cudaMemcpyAsync(p.dev, xyz, (size_t)(n - 1) * stride + 12, cudaMemcpyHostToDevice, c->copy_stream));
    }
  }
  if (p.sharded && !c->local) {
    // one process per GPU: the slices are exchanged on the copy stream as soon as this rank's has arrived - for the source
    // that is WHILE the target is indexed on the compute stream, not in front of the source's own index build
    check_nccl(c, c->nccl->AllGather(p.dev + (size_t)c->rank * (size_t)p.chunk_rows * 12, p.dev, (size_t)p.chunk_rows * 12,
                                     /*ncclInt8*/ 0, c->comm, c->copy_stream), "ncclAllGather");
  }
  GICPB_CUDA(cudaEventRecord(p.done, c->copy_stream));
  p.host = xyz;
  p.n = n;
  p.stride = stride;
  p.pending = true;
}

// true: the host cloud (xyz, n, stride) was uploaded by gicpb_prefetch_cloud (or is uploaded here, in slices, when the job
// is sharded); the compute stream now waits for that copy
bool take_prefetch(gicpb_ctx* c, int which, const void* xyz, int64_t n, int64_t stride, int on_device) {
  gicpb_ctx::Prefetch& p = c->prefetch[which];
  if (p.pending && (on_device || p.host != xyz || p.n != n || p.stride != stride)) {
    p.pending = false;
    GICPB_CUDA(cudaEventSynchronize(p.done));  // a different cloud is being set: let the stale copy finish first
  }
  if (!p.pending && !on_device && shard_uploads(c)) do_prefetch(c, which, xyz, n, stride);
  if (!p.pending) return false;
  p.pending = false;
  GICPB_CUDA(cudaStreamWaitEvent(c->stream, p.done, 0));
  if (p.sharded && c->local) gather_slices(c, which);
  return true;
}

// keep iff (double)d2 > thr.  With thr_f = largest float <= thr this is d2 > thr_f, i.e. NOT (d2 < next(thr_f)).
// thr < 0 keeps every finite point and a NaN thr none, without a search (and without a NaN search radius).
float difference_thr_next(double thr, DiffMode* mode) {
  *mode = std::isnan(thr) ? kDiffKeepNone : thr < 0 ? kDiffKeepAll : kDiffSearch;
  if (*mode != kDiffSearch) return 0.f;
  float tf = (float)thr;
  if ((double)tf > thr) tf = std::nextafterf(tf, -INFINITY);
  return std::nextafterf(tf, INFINITY);
}

GridIndex& pick_grid(gicpb_ctx* c, int which) {
  if (which == 0) return c->tgt;
  if (which == 1) return c->src;
  if (which == 2) return c->sub;
  throw ArgError("which must be 0 (target), 1 (source) or 2 (subtract)");
}

// the calls that look at a WHOLE cloud (resolution, normals, the kNN hook): a source of which only this rank's window is
// indexed is indexed whole first
GridIndex& pick_whole_grid(gicpb_ctx* c, int which) {
  GridIndex& g = pick_grid(c, which);
  if (g.ready() && g.windowed()) {
    g.widen(c->stream);
    if (which == 1) {
      update_shard(c);
      c->cov_ready = false;
      c->pairs_valid = false;
    }
  }
  return g;
}

// Utils::getNormals on an indexed cloud: (nx, ny, nz, curvature) per point in ORIGINAL order into c->io_b (float4 rows, NaN x 4
// where PCL gives no normal); returns the number of finite normals, *total_points = rows written
int64_t compute_normals(gicpb_ctx* c, int which, double radius, int64_t* total_points) {
  if (!(radius > 0)) throw ArgError("radius must be > 0");
  GridIndex& g = pick_whole_grid(c, which);
  if (!g.ready()) throw StateError("cloud not set");
  const int64_t total = g.n_points();
  const int n = g.n_indexed();
  const float r2 = (float)(radius * radius);  // KdTreeFLANN::radiusSearch: float(radius * radius), d2 < r2
  DevBuf<unsigned> counts, offsets, scan_tmp;
  counts.reserve((size_t)n + 1);
  offsets.reserve((size_t)n + 1);
  scan_tmp.reserve(scan_tmp_entries(n + 1));
  // counts[n] = 0, so that the exclusive scan leaves the total in offsets[n]
  GICPB_CUDA(cudaMemsetAsync(counts.get() + n, 0, sizeof(unsigned), c->stream));
  launch_radius_counts(g.view(), r2, counts.get(), far_work(c, n), c->stream);
  exclusive_scan_u32(counts.get(), offsets.get(), (int64_t)n + 1, scan_tmp.get(), c->stream);
  GICPB_CUDA(cudaMemsetAsync(c->counter.get(), 0, sizeof(unsigned long long), c->stream));
  launch_sum_counts(counts.get(), n, c->counter.get(), c->stream);
  unsigned total_keys = 0;
  unsigned long long total_wide = 0;
  GICPB_CUDA(cudaMemcpyAsync(&total_keys, offsets.get() + n, sizeof(unsigned), cudaMemcpyDeviceToHost, c->stream));
  GICPB_CUDA(cudaMemcpyAsync(&total_wide, c->counter.get(), sizeof(total_wide), cudaMemcpyDeviceToHost, c->stream));
  GICPB_CUDA(cudaStreamSynchronize(c->stream));
  if (total_wide != (unsigned long long)total_keys)
    throw ArgError("normal radius too large: more than 2^32 neighbour entries (" + std::to_string(total_wide) + ")");
  DevBuf<unsigned long long> keys;
  keys.reserve((size_t)total_keys + 1);
  launch_radius_fill(g.view(), r2, offsets.get(), keys.get(), far_work(c, n), c->stream);
  c->io_b.reserve((size_t)total * 16);
  GICPB_CUDA(cudaMemsetAsync(c->io_b.get(), 0xff, (size_t)total * 16, c->stream));  // all-ones = a quiet NaN: no normal
  GICPB_CUDA(cudaMemsetAsync(c->counter.get(), 0, sizeof(unsigned long long), c->stream));
  launch_normals_solve(g.view(), counts.get(), offsets.get(), keys.get(), reinterpret_cast<float4*>(c->io_b.get()),
                       c->counter.get(), c->stream);
  unsigned long long kept = 0;
  GICPB_CUDA(cudaMemcpyAsync(&kept, c->counter.get(), sizeof(kept), cudaMemcpyDeviceToHost, c->stream));
  GICPB_CUDA(cudaStreamSynchronize(c->stream));
  *total_points = total;
  return (int64_t)kept;
}

}  // namespace

// ---- one process, several GPUs (include/gicp_b200.h "gicpb_group") ------------------------------------------------------
// The reference's consumer builds its GICPAlignment inside ONE process (reference src/LeicaStateMachine.cpp:138-171), so the
// multi-GPU path must be reachable without a launcher: a group owns one context per device, every group call runs the same
// per-rank call on all of them from one host thread per GPU (exactly what the ranks of a torchrun job do, optimisers in lock
// step), and the collectives stay inside the process: target covariances by peer copies, the 14 cost sums fused into the cost
// kernel over peer memory (kernels.hpp PeerReduce) when every pair of devices can map each other, else through the host.
struct gicpb_group {
  LocalGroup lg;
  std::vector<gicpb_ctx*> ctx;
  std::string err;
  bool fused = false;
};

namespace {

template <typename F>
int group_run(gicpb_group* g, F fn) {  // fn(rank, ctx) -> status, on one thread per GPU; the first failure is reported
  const int n = (int)g->ctx.size();
  std::vector<int> rc((size_t)n, GICPB_OK);
  g->lg.reset();
  // A member used on its own since the last group call worked on the whole source (update_shard) and has dropped the
  // covariances of its shard.  Computing them is a collective (the target's are gathered from every rank): when one member
  // needs them, all of them compute them again.
  bool all_ready = true;
  for (int r = 0; r < n; ++r) {
    gicpb_ctx* c = g->ctx[(size_t)r];
    c->rank = r;
    c->world = n;
    update_shard(c);
    all_ready = all_ready && c->cov_ready;
  }
  if (!all_ready)
    for (gicpb_ctx* c : g->ctx) {
      c->cov_ready = false;
      c->pairs_valid = false;
    }
  auto body = [&](int r) {
    // a member is rank r of n only while a group call runs on all members at once; used on its own (gicpb_group_ctx) it is
    // a plain single-GPU context, so that nothing it does waits for the other members
    gicpb_ctx* c = g->ctx[(size_t)r];
    c->rank = r;
    c->world = n;
    rc[(size_t)r] = fn(r, c);
    c->rank = 0;
    c->world = 1;
    if (rc[(size_t)r] != GICPB_OK) g->lg.fail();  // the others must not wait for this rank at a barrier
  };
  std::vector<std::thread> th;
  for (int r = 1; r < n; ++r) th.emplace_back(body, r);
  body(0);
  for (auto& t : th) t.join();
  int first = GICPB_OK;
  for (int r = 0; r < n; ++r) {
    // a rank that only gave up because another one failed is not the cause
    const bool abort_only = rc[(size_t)r] == GICPB_E_STATE && g->ctx[(size_t)r]->err == GroupAbort().what();
    if (rc[(size_t)r] != GICPB_OK && !abort_only && first == GICPB_OK) {
      first = rc[(size_t)r];
      g->err = "GPU " + std::to_string(g->ctx[(size_t)r]->device) + " (rank " + std::to_string(r) + "): " + g->ctx[(size_t)r]->err;
    }
  }
  if (first == GICPB_OK)
    for (int r = 0; r < n; ++r)
      if (rc[(size_t)r] != GICPB_OK) {
        first = rc[(size_t)r];
        g->err = g->ctx[(size_t)r]->err;
        break;
      }
  return first;
}

// the argument checks of gicpb_cloud_difference (set_subtract, then run), in its order and with its messages
void check_difference_args(const void* input, int64_t n_input, int64_t input_stride, const void* subtract,
                           int64_t n_subtract, int64_t subtract_stride, const uint8_t* mask) {
  check_cloud_args(subtract, n_subtract, subtract_stride);
  if (n_subtract > 0x7fffff00LL) throw ArgError("cloud has more than 2^31 points");
  if (!mask) throw ArgError("null mask");
  check_cloud_args(input, n_input, input_stride);
  if (n_input > 0x7fffff00LL) throw ArgError("cloud has more than 2^31 points");
}

// One rank of gicpb_group_cloud_difference (world > 1, host clouds and mask).  Every rank indexes the subtract planes it owns
// plus a halo that covers the search radius, answers the finite input rows of its own planes (the other points within the
// radius of those rows are all in its window) and then assembles the mask of its row slice [lo, hi) from every member's keep
// bytes.  When the subtract cannot be split by planes every rank indexes all of it and answers its row slice directly.
// Returns the number of points this rank kept.
unsigned long long group_difference_rank(gicpb_ctx* c, const void* input, int64_t n, int64_t input_stride,
                                         const void* subtract, int64_t n_sub, int64_t sub_stride, double thr,
                                         uint8_t* mask) {
  DiffMode mode = kDiffSearch;
  const float thr_next = difference_thr_next(thr, &mode);
  const double radius = std::sqrt((double)thr_next);
  // 1. both clouds: this rank's slice of the rows on the copy stream, the other slices from the other members
  const void* sub_p = subtract;
  bool sub_dev = false;
  const unsigned char* d_in = nullptr;
  try {
    if (shard_uploads(c)) {
      do_prefetch(c, 2, subtract, n_sub, sub_stride);
      do_prefetch(c, 3, input, n, input_stride);
    }
    if (take_prefetch(c, 2, subtract, n_sub, sub_stride, 0)) {
      sub_p = c->prefetch[2].dev;
      sub_stride = c->prefetch[2].dev_stride;
      sub_dev = true;
    }
    // 2. the window of the subtract's brick planes
    c->sub.build(sub_p, n_sub, sub_stride, sub_dev, c->prm.cell_size, c->prm.points_per_cell, c->stream, &c->stager, c->rank,
                 c->world, std::isfinite(radius) ? radius : INFINITY);
    if (take_prefetch(c, 3, input, n, input_stride, 0)) {
      d_in = c->prefetch[3].dev;
      input_stride = c->prefetch[3].dev_stride;
    } else {
      d_in = stage_in(c, c->io_a, input, n, &input_stride, false);
    }
  } catch (...) {
    for (int w : {2, 3})  // a copy started here must not be taken for a later call's clouds
      if (c->prefetch[w].pending) {
        c->prefetch[w].pending = false;
        cudaEventSynchronize(c->prefetch[w].done);
      }
    throw;
  }
  const int64_t lo = n * c->rank / c->world, hi = n * (c->rank + 1) / c->world, len = hi - lo;
  const bool routed = c->sub.plane_sharded();
  c->keep_full.reserve((size_t)n);
  GICPB_CUDA(cudaMemsetAsync(c->keep_full.get(), 0, (size_t)n, c->stream));
  GICPB_CUDA(cudaMemsetAsync(c->counter.get(), 0, sizeof(unsigned long long), c->stream));
  if (routed) {
    // 3. the rows of this rank's planes, compacted in row order, searched as float4 rows, their keep bytes put back in place
    c->route_flags.reserve((size_t)n + 1);
    c->route_pos.reserve((size_t)n + 1);
    c->route_tmp.reserve(scan_tmp_entries(n + 1));
    c->queries.reserve((size_t)n);
    const int64_t n_own = c->sub.owned_queries(d_in, n, input_stride, c->queries.get(), c->route_flags.get(),
                                                c->route_pos.get(), c->route_tmp.get(), c->stream);
    c->io_b.reserve((size_t)std::max<int64_t>(n_own, 1));
    launch_difference(c->sub.view(), reinterpret_cast<const unsigned char*>(c->queries.get()), n_own, 16, thr_next,
                      mode, c->io_b.get(), c->counter.get(), far_work(c, n_own), c->stream);
    scatter_keep(c->queries.get(), c->io_b.get(), n_own, c->keep_full.get(), c->stream);
  } else {
    launch_difference(c->sub.view(), d_in + lo * input_stride, len, input_stride, thr_next, mode,
                      c->keep_full.get() + lo, c->counter.get(), far_work(c, len), c->stream);
  }
  unsigned long long kept = 0;
  GICPB_CUDA(cudaMemcpyAsync(&kept, c->counter.get(), sizeof(kept), cudaMemcpyDeviceToHost, c->stream));
  GICPB_CUDA(cudaStreamSynchronize(c->stream));
  // 4. ownership partitions the finite rows: the mask of [lo, hi) is the OR of every member's keep bytes there
  c->local->barrier();  // every member's keep bytes are complete
  const unsigned char* slice = c->keep_full.get() + lo;
  if (routed && len > 0) {
    c->keep_parts.reserve((size_t)(c->world * len));
    for (int r = 0; r < c->world; ++r) {
      const gicpb_ctx* o = c->local->members[(size_t)r];
      GICPB_CUDA(cudaMemcpyPeerAsync(c->keep_parts.get() + r * len, c->device, o->keep_full.get() + lo, o->device, (size_t)len,
                                     c->stream));
    }
    c->io_b.reserve((size_t)len);
    or_parts(c->keep_parts.get(), c->world, len, c->io_b.get(), c->stream);
    slice = c->io_b.get();
  }
  GICPB_CUDA(cudaStreamSynchronize(c->stream));
  c->local->barrier();  // nobody reads another member's keep bytes any more
  if (len > 0) download_bytes(c, mask + lo, slice, (size_t)len);
  return kept;
}

}  // namespace

// ---- C ABI ---------------------------------------------------------------------------------------------------
extern "C" {

void gicpb_default_params(gicpb_params* p) {
  if (!p) return;
  p->max_iterations = 100;
  p->transformation_epsilon = 4e-3;
  p->rotation_epsilon = 2e-3;
  p->max_corr_distance = 4e-2;
  p->k_correspondences = 20;
  p->gicp_epsilon = 1e-3;
  p->max_inner_iterations = 20;
  p->cell_size = 0.f;
  p->points_per_cell = 6.0f;
  p->mahalanobis_fp32 = 0;
  p->use_previous_match = 1;
  p->cost_moments = 0;
  p->cost_persistent = 1;
  // GICPB_COST_PERSISTENT=0: one launch per evaluation (for runs under a profiler, which serialises launches and keeps the
  // host from talking to a resident kernel: every inner solve would first idle out, 200 ms, and then fall back)
  if (const char* e = std::getenv("GICPB_COST_PERSISTENT"))
    if (*e == '0') p->cost_persistent = 0;
}

int gicpb_create(int device, gicpb_ctx** out) {
  if (!out) return GICPB_E_BADARG;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) return GICPB_E_CUDA;
  std::unique_ptr<gicpb_ctx> c(new gicpb_ctx);
  c->device = device;
  gicpb_default_params(&c->prm);
  DeviceGuard guard(device);
  try {
    cudaDeviceProp prop;
    GICPB_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) throw CudaError("libgicp_b200 is built for sm_100a only; found sm_" +
                                         std::to_string(prop.major) + std::to_string(prop.minor));
    c->num_sms = prop.multiProcessorCount;
    GICPB_CUDA(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    {
      // gicpb_set_clouds runs the target's covariance pass on aux_stream beside the source's index build on the main
      // stream.  The build is a chain of short kernels and read-backs: its blocks must get onto the SMs as soon as
      // they are launched, so the main stream has the highest priority and aux_stream the lowest, and the build's
      // kernels ask for the same (largest) shared-memory carve-out as the kNN kernel so that both can share an SM
      // (measured at 1 M + 1 M points: 2.34 ms for the separate calls, 2.21 ms overlapped, 2.07 ms with both hints).
      int lo_p = 0, hi_p = 0;
      GICPB_CUDA(cudaDeviceGetStreamPriorityRange(&lo_p, &hi_p));
      GICPB_CUDA(cudaStreamCreateWithPriority(&c->stream, cudaStreamNonBlocking, hi_p));
      GICPB_CUDA(cudaStreamCreateWithPriority(&c->aux_stream, cudaStreamNonBlocking, lo_p));
      prefer_shared_carveout_grid();
      prefer_shared_carveout_sort();
    }
    c->src.expect_far_queries(false);  // the source is searched from its own points only (kNN, resolution, normals)
    GICPB_CUDA(cudaEventCreateWithFlags(&c->ev_aux, cudaEventDisableTiming));
    GICPB_CUDA(cudaEventCreate(&c->ev0));
    GICPB_CUDA(cudaEventCreate(&c->ev1));
    GICPB_CUDA(cudaEventCreateWithFlags(&c->ev_order, cudaEventDisableTiming));
    for (auto& p : c->prefetch) GICPB_CUDA(cudaEventCreateWithFlags(&p.done, cudaEventDisableTiming));
    GICPB_CUDA(cudaHostAlloc(&c->h_sums, kCostOutDoubles * sizeof(double), cudaHostAllocMapped));
    GICPB_CUDA(cudaHostGetDevicePointer(&c->h_sums_dev, c->h_sums, 0));
    std::memset(c->h_sums, 0, kCostOutDoubles * sizeof(double));  // the result words are polled for a stamp: recycled pinned pages may hold one
    GICPB_CUDA(cudaHostAlloc(&c->h_cmd, 2 * sizeof(CostCommand), cudaHostAllocMapped));
    GICPB_CUDA(cudaHostGetDevicePointer(&c->h_cmd_dev, c->h_cmd, 0));
    std::memset(c->h_cmd, 0, 2 * sizeof(CostCommand));
    c->d_cmd.reserve(1);
    GICPB_CUDA(cudaMemset(c->d_cmd.get(), 0, sizeof(CostCommand)));  // sequence words are never 0
    GICPB_CUDA(cudaDeviceGetAttribute(&c->smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
    if (const char* env = std::getenv("GICPB_COST_IDLE_MS"))
      if (*env) c->cost_idle_ns = (unsigned long long)(std::max(std::atof(env), 1.0) * 1e6);
    if (const char* env = std::getenv("GICPB_COST_TEST_STALL_MS"))
      if (*env) c->cost_test_stall_ms = std::atof(env);
    GICPB_CUDA(cudaHostAlloc(&c->h_mom, 80 * sizeof(double), cudaHostAllocDefault));
    GICPB_CUDA(cudaHostAlloc(&c->h_far, 4 * sizeof(unsigned), cudaHostAllocDefault));
    c->ticket.reserve(4);
    GICPB_CUDA(cudaMemset(c->ticket.get(), 0, 4 * sizeof(unsigned)));
    c->counter.reserve(2);
  } catch (const std::exception&) {
    return GICPB_E_CUDA;
  }
  *out = c.release();
  return GICPB_OK;
}

void gicpb_destroy(gicpb_ctx* c) {
  if (!c) return;
  DeviceGuard guard(c->device);
  if (c->comm && c->nccl) c->nccl->CommDestroy(c->comm);
  cost_session_end(c);
  if (c->stream) cudaStreamSynchronize(c->stream);
  if (c->h_sums) cudaFreeHost(c->h_sums);
  if (c->h_cmd) cudaFreeHost(c->h_cmd);
  if (c->h_mom) cudaFreeHost(c->h_mom);
  if (c->peer.world > 1 && c->peer_ipc)
    for (int r = 0; r < c->peer.world; ++r)
      if (r != c->rank && c->peer.peers[r]) cudaIpcCloseMemHandle(c->peer.peers[r]);
  if (c->peer_own) cudaFree(c->peer_own);
  if (c->h_far) cudaFreeHost(c->h_far);
  for (auto& p : c->prefetch) {
    if (p.pending) cudaEventSynchronize(p.done);
    if (p.done) cudaEventDestroy(p.done);
  }
  if (c->ev_order) cudaEventDestroy(c->ev_order);
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  if (c->aux_stream) cudaStreamDestroy(c->aux_stream);
  if (c->ev_aux) cudaEventDestroy(c->ev_aux);
  if (c->ev0) cudaEventDestroy(c->ev0);
  if (c->ev1) cudaEventDestroy(c->ev1);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;
}

const char* gicpb_last_error(const gicpb_ctx* c) { return c ? c->err.c_str() : "null context"; }

int gicpb_set_params(gicpb_ctx* c, const gicpb_params* p) {
  return guarded(c, [&] {
    if (!p) throw ArgError("null params");
    if (p->k_correspondences < 2 || p->k_correspondences > 32) throw ArgError("k_correspondences must be in [2, 32]");
    if (p->max_iterations < 1) throw ArgError("max_iterations must be >= 1");
    if (!(p->gicp_epsilon > 0)) throw ArgError("gicp_epsilon must be > 0");
    const bool cov_changed = p->k_correspondences != c->prm.k_correspondences;
    c->prm = *p;
    if (cov_changed) c->cov_ready = false;
  });
}

int gicpb_get_params(const gicpb_ctx* c, gicpb_params* p) {
  if (!c || !p) return GICPB_E_BADARG;
  *p = c->prm;
  return GICPB_OK;
}

int gicpb_nccl_unique_id(const char* libnccl_path, unsigned char id_out[128]) {
  std::string err;
  NcclApi* api = load_nccl(libnccl_path, err);
  if (!api || !id_out) return GICPB_E_NCCL;
  NcclApi::unique_id id;
  if (api->GetUniqueId(&id) != 0) return GICPB_E_NCCL;
  std::memcpy(id_out, id.internal, 128);
  return GICPB_OK;
}

int gicpb_comm_init(gicpb_ctx* c, const char* libnccl_path, int rank, int world, const unsigned char id[128]) {
  return guarded(c, [&] {
    if (world < 1 || rank < 0 || rank >= world) throw ArgError("bad rank / world");
    if (world == 1) {
      c->rank = 0;
      c->world = 1;
      return;
    }
    if (!id) throw ArgError("null NCCL unique id");
    std::string err;
    c->nccl = load_nccl(libnccl_path, err);
    if (!c->nccl) throw NcclError(err);
    NcclApi::unique_id uid;
    std::memcpy(uid.internal, id, 128);
    check_nccl(c, c->nccl->CommInitRank(&c->comm, world, uid, rank), "ncclCommInitRank");
    c->rank = rank;
    c->world = world;
    c->cov_ready = false;
    c->pairs_valid = false;
    update_shard(c);
  });
}

int gicpb_peer_export(gicpb_ctx* c, unsigned char handle_out[64]) {
  return guarded(c, [&] {
    if (!handle_out) throw ArgError("null handle");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    if (!c->peer_own) {
      GICPB_CUDA(cudaMalloc(&c->peer_own, sizeof(PeerSlots)));
      GICPB_CUDA(cudaMemset(c->peer_own, 0, sizeof(PeerSlots)));
    }
    cudaIpcMemHandle_t h;
    GICPB_CUDA(cudaIpcGetMemHandle(&h, c->peer_own));
    std::memcpy(handle_out, &h, 64);
  });
}

int gicpb_peer_import(gicpb_ctx* c, const unsigned char* handles, int world) {
  return guarded(c, [&] {
    if (!handles) throw ArgError("null handles");
    if (world != c->world || world < 2 || world > kMaxPeers) throw ArgError("world must match gicpb_comm_init (2..16)");
    if (!c->peer_own) throw StateError("gicpb_peer_export must be called first");
    c->peer_ready = false;
    // seq restarts at 0 below: the flag words of an earlier import must not look like evaluations already done
    GICPB_CUDA(cudaStreamSynchronize(c->stream));
    GICPB_CUDA(cudaMemset(c->peer_own, 0, sizeof(PeerSlots)));
    for (int r = 0; r < world; ++r) {
      if (r == c->rank) {
        c->peer.peers[r] = c->peer_own;
        continue;
      }
      cudaIpcMemHandle_t h;
      std::memcpy(&h, handles + 64 * (size_t)r, 64);
      void* p = nullptr;
      GICPB_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
      c->peer.peers[r] = static_cast<PeerSlots*>(p);
    }
    c->peer.rank = c->rank;
    c->peer.world = world;
    c->peer.seq = 0u;
    c->peer_ipc = true;
    {
      const char* env = std::getenv("GICPB_PEER_TIMEOUT_MS");
      const double ms = env && *env ? std::atof(env) : 30000.0;
      c->peer.timeout_ns = (unsigned long long)(std::max(ms, 1.0) * 1e6);
    }
    c->peer_ready = true;
  });
}

int gicpb_peer_disable(gicpb_ctx* c) {
  if (!c) return GICPB_E_BADARG;
  c->peer_ready = false;  // back to ncclAllReduce; mapped handles stay open until gicpb_destroy
  return GICPB_OK;
}

int gicpb_shard_info(gicpb_ctx* c, int64_t* lo, int64_t* hi, int64_t* n_indexed_here, int64_t* widened) {
  if (!c) return GICPB_E_BADARG;
  if (lo) *lo = c->shard_lo;
  if (hi) *hi = c->shard_hi;
  if (n_indexed_here) *n_indexed_here = c->src.ready() ? c->src.n_indexed() : 0;
  if (widened) *widened = c->window_widened;
  return GICPB_OK;
}

int gicpb_comm_rank(const gicpb_ctx* c, int* rank, int* world) {
  if (!c) return GICPB_E_BADARG;
  if (rank) *rank = c->rank;
  if (world) *world = c->world;
  return GICPB_OK;
}

int gicpb_prefetch_cloud(gicpb_ctx* c, int which, const void* xyz, int64_t n, int64_t stride) {
  return guarded(c, [&] {
    if (which != 0 && which != 1) throw ArgError("which must be 0 (target) or 1 (source)");
    check_cloud_args(xyz, n, stride);
    do_prefetch(c, which, xyz, n, stride);
  });
}

int gicpb_set_target(gicpb_ctx* c, const void* xyz, int64_t n, int64_t stride, int on_device) {
  return guarded(c, [&] {
    check_cloud_args(xyz, n, stride);
    c->cov_ready = false;
    c->pairs_valid = false;
    if (take_prefetch(c, 0, xyz, n, stride, on_device)) {
      xyz = c->prefetch[0].dev;
      stride = c->prefetch[0].dev_stride;
      on_device = 1;
    }
    c->tgt.build(xyz, n, stride, on_device != 0, c->prm.cell_size, c->prm.points_per_cell, c->stream, &c->stager);
  });
}

int gicpb_set_source(gicpb_ctx* c, const void* xyz, int64_t n, int64_t stride, int on_device) {
  return guarded(c, [&] {
    check_cloud_args(xyz, n, stride);
    c->cov_ready = false;
    c->pairs_valid = false;
    if (take_prefetch(c, 1, xyz, n, stride, on_device)) {
      xyz = c->prefetch[1].dev;
      stride = c->prefetch[1].dev_stride;
      on_device = 1;
    }
    c->src.build(xyz, n, stride, on_device != 0, c->prm.cell_size, c->prm.points_per_cell, c->stream, &c->stager, c->rank,
                 c->world);
    update_shard(c);
  });
}

// Both clouds in one call: the target is indexed, then its kNN covariances run on a second stream WHILE the source is
// indexed on the context's stream (the index build is a chain of small kernels and read-backs that leaves most of
// the GPU idle; the kNN kernel fills it), then the source covariances.  Same results as set_target + set_source +
// compute_covariances.  When k_correspondences does not fit the clouds the covariances are left to gicpb_align, which
// reports it as before.
int gicpb_set_clouds(gicpb_ctx* c, const void* target, int64_t n_target, int64_t target_stride, const void* source,
                     int64_t n_source, int64_t source_stride, int on_device) {
  return guarded(c, [&] {
    check_cloud_args(target, n_target, target_stride);
    check_cloud_args(source, n_source, source_stride);
    c->cov_ready = false;
    c->pairs_valid = false;
    int t_dev = on_device, s_dev = on_device;
    if (take_prefetch(c, 0, target, n_target, target_stride, on_device)) {
      target = c->prefetch[0].dev;
      target_stride = c->prefetch[0].dev_stride;
      t_dev = 1;
    }
    c->tgt.build(target, n_target, target_stride, t_dev != 0, c->prm.cell_size, c->prm.points_per_cell, c->stream, &c->stager);
    const int k = c->prm.k_correspondences;
    const bool overlap = k >= 2 && k <= 32 && k <= c->tgt.n_indexed();
    if (overlap) {  // the build has synchronised c->stream: the index is complete
      start_target_cov(c, c->aux_stream);
      GICPB_CUDA(cudaEventRecord(c->ev_aux, c->aux_stream));
    }
    try {
      if (take_prefetch(c, 1, source, n_source, source_stride, on_device)) {
        source = c->prefetch[1].dev;
        source_stride = c->prefetch[1].dev_stride;
        s_dev = 1;
      }
      c->src.build(source, n_source, source_stride, s_dev != 0, c->prm.cell_size, c->prm.points_per_cell, c->stream, &c->stager,
                   c->rank, c->world);
    } catch (...) {
      if (overlap) cudaStreamSynchronize(c->aux_stream);  // nothing may still be running on the target when we leave
      throw;
    }
    if (overlap) {
      GICPB_CUDA(cudaStreamWaitEvent(c->stream, c->ev_aux, 0));
      if (k <= c->src.n_finite_total()) {
        finish_covariances(c);
      } else {
        GICPB_CUDA(cudaStreamSynchronize(c->stream));
      }
    }
  });
}

int gicpb_compute_covariances(gicpb_ctx* c) {
  return guarded(c, [&] { ensure_covariances(c); });
}

int gicpb_align(gicpb_ctx* c, gicpb_align_result* out) {
  if (!out) return GICPB_E_BADARG;
  int rc = guarded(c, [&] { do_align(c, out); });
  if (rc == GICPB_OK && out->status != GICPB_OK) rc = out->status;
  return rc;
}

int gicpb_fitness(gicpb_ctx* c, const float transform[16], double max_range, double* score) {
  return guarded(c, [&] {
    if (!transform || !score) throw ArgError("null argument");
    if (!c->tgt.ready() || !c->src.ready()) throw StateError("set_target and set_source must be called first");
    update_shard(c);
    ensure_pair_buffers(c);
    const Rigid T = rigid_from_rowmajor(transform);
    double* partials = c->partials.get() + (size_t)c->num_sms * 4 * 16;
    // the matches of the last correspondence pass (same clouds, a nearby pose) seed the search
    const int* seed = (c->prm.use_previous_match != 0 && c->pairs_valid) ? c->pair_pos.get() : nullptr;
    launch_fitness(c->tgt.view(), c->src.sorted_points(), c->shard_lo, c->shard_hi, T, max_range, seed, partials,
                   c->d_sums.get(), far_work(c, c->shard_hi - c->shard_lo), c->stream);
    all_reduce_sum(c, c->d_sums.get(), 2);
    GICPB_CUDA(cudaMemcpyAsync(c->h_sums, c->d_sums.get(), 2 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    GICPB_CUDA(cudaStreamSynchronize(c->stream));
    *score = c->h_sums[1] > 0 ? c->h_sums[0] / c->h_sums[1] : std::numeric_limits<double>::max();
  });
}

int gicpb_transform_cloud(gicpb_ctx* c, const float transform[16], const void* in, void* out, int64_t n, int64_t stride,
                          int on_device) {
  return guarded(c, [&] {
    if (!transform || !out) throw ArgError("null argument");
    check_cloud_args(in, n, stride);
    const Rigid T = rigid_from_rowmajor(transform);
    if (on_device) {
      launch_transform(static_cast<const unsigned char*>(in), static_cast<unsigned char*>(out), n, stride, T, c->stream);
      GICPB_CUDA(cudaStreamSynchronize(c->stream));
      return;
    }
    // host clouds: `in` / `out` point at the first x; the last point may end right after its z
    const size_t bytes = (size_t)(n - 1) * stride + 12;
    const size_t full = (size_t)n * stride;
    c->io_a.reserve(full);
    upload_bytes(c, c->io_a.get(), in, bytes);
    launch_transform(c->io_a.get(), c->io_a.get(), n, stride, T, c->stream);
    download_bytes(c, out, c->io_a.get(), bytes);
  });
}

int gicpb_difference_set_subtract(gicpb_ctx* c, const void* subtract, int64_t n, int64_t stride, int on_device) {
  return guarded(c, [&] {
    check_cloud_args(subtract, n, stride);
    c->sub.build(subtract, n, stride, on_device != 0, c->prm.cell_size, c->prm.points_per_cell, c->stream, &c->stager);
  });
}

int gicpb_difference_run(gicpb_ctx* c, const void* input, int64_t n, int64_t stride, int on_device, double thr,
                         uint8_t* mask, int mask_on_device, int64_t* n_kept) {
  return guarded(c, [&] {
    if (!mask) throw ArgError("null mask");
    check_cloud_args(input, n, stride);
    if (!c->sub.ready()) throw StateError("difference_set_subtract must be called first");
    if (n > 0x7fffff00LL) throw ArgError("cloud has more than 2^31 points");
    if (c->sub.windowed()) c->sub.widen(c->stream);  // a group member's window of the subtract (gicpb_group_cloud_difference)
    const unsigned char* d_in = stage_in(c, c->io_a, input, n, &stride, on_device != 0);
    unsigned char* d_mask = mask;
    if (!mask_on_device) {
      c->io_b.reserve((size_t)n);
      d_mask = c->io_b.get();
    }
    GICPB_CUDA(cudaMemsetAsync(c->counter.get(), 0, sizeof(unsigned long long), c->stream));
    DiffMode mode = kDiffSearch;
    const float thr_next = difference_thr_next(thr, &mode);
    launch_difference(c->sub.view(), d_in, n, stride, thr_next, mode, d_mask, c->counter.get(), far_work(c, n), c->stream);
    unsigned long long kept = 0;
    GICPB_CUDA(cudaMemcpyAsync(&kept, c->counter.get(), sizeof(kept), cudaMemcpyDeviceToHost, c->stream));
    if (!mask_on_device) download_bytes(c, mask, d_mask, (size_t)n);
    GICPB_CUDA(cudaStreamSynchronize(c->stream));
    if (n_kept) *n_kept = (int64_t)kept;
  });
}

int gicpb_cloud_difference(gicpb_ctx* c, const void* input, int64_t n_input, int64_t input_stride, const void* subtract,
                           int64_t n_subtract, int64_t subtract_stride, int on_device, double thr, uint8_t* mask,
                           int64_t* n_kept) {
  int rc = gicpb_difference_set_subtract(c, subtract, n_subtract, subtract_stride, on_device);
  if (rc != GICPB_OK) return rc;
  return gicpb_difference_run(c, input, n_input, input_stride, on_device, thr, mask, on_device, n_kept);
}

int gicpb_nn1(gicpb_ctx* c, const void* queries, int64_t n, int64_t stride, int on_device, const float transform[16],
              double max_dist, int32_t* idx, float* d2) {
  return guarded(c, [&] {
    check_cloud_args(queries, n, stride);
    if (!c->tgt.ready()) throw StateError("set_target must be called first");
    if (n > INT_MAX) throw ArgError("too many queries");
    float ident[16];
    identity16(ident);
    const Rigid T = rigid_from_rowmajor(transform ? transform : ident);
    const unsigned char* d_in = stage_in(c, c->io_a, queries, n, &stride, on_device != 0);
    c->queries.reserve((size_t)n);
    launch_pack_queries(d_in, n, stride, c->queries.get(), c->stream);
    c->io_b.reserve((size_t)n * 8);
    int* d_idx = reinterpret_cast<int*>(c->io_b.get());
    float* d_d2 = reinterpret_cast<float*>(c->io_b.get() + (size_t)n * 4);
    const float gate2 = max_dist > 0 ? round_up_to_float(max_dist * max_dist) : -1.f;  // <= 0: ungated
    launch_nn1(c->tgt.view(), c->queries.get(), (int)n, T, gate2, d_idx, d_d2, nullptr, far_work(c, n), c->stream);
    if (idx) GICPB_CUDA(cudaMemcpyAsync(idx, d_idx, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
    if (d2) GICPB_CUDA(cudaMemcpyAsync(d2, d_d2, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
    GICPB_CUDA(cudaStreamSynchronize(c->stream));
  });
}

int gicpb_knn(gicpb_ctx* c, int which, int32_t* idx, float* d2) {
  return guarded(c, [&] {
    if (!idx || !d2) throw ArgError("null output");
    if (which != 0 && which != 1) throw ArgError("which must be 0 or 1");
    GridIndex& g = pick_whole_grid(c, which);
    if (!g.ready()) throw StateError("cloud not set");
    const int k = c->prm.k_correspondences;
    const int n = g.n_indexed();
    if (k > n) throw AlignStop(GICPB_E_TOO_FEW_POINTS, "k_correspondences exceeds the number of points");
    DevBuf<double> normals;
    DevBuf<int> d_idx;
    DevBuf<float> d_d2;
    normals.reserve(3 * (size_t)n);
    d_idx.reserve((size_t)n * k);
    d_d2.reserve((size_t)n * k);
    launch_knn_covariances(g.view(), 0, n, k, normals.get(), d_idx.get(), d_d2.get(), far_work(c, n), c->stream);
    std::vector<int> hi((size_t)n * k);
    std::vector<float> hd((size_t)n * k);
    std::vector<float4> hp((size_t)n);
    GICPB_CUDA(cudaMemcpyAsync(hi.data(), d_idx.get(), hi.size() * 4, cudaMemcpyDeviceToHost, c->stream));
    GICPB_CUDA(cudaMemcpyAsync(hd.data(), d_d2.get(), hd.size() * 4, cudaMemcpyDeviceToHost, c->stream));
    GICPB_CUDA(cudaMemcpyAsync(hp.data(), g.sorted_points(), hp.size() * sizeof(float4), cudaMemcpyDeviceToHost, c->stream));
    GICPB_CUDA(cudaStreamSynchronize(c->stream));
    const int64_t total = g.n_points();
    for (int64_t i = 0; i < total * k; ++i) {
      idx[i] = -1;
      d2[i] = INFINITY;
    }
    for (int s = 0; s < n; ++s) {
      int oi;
      std::memcpy(&oi, &hp[s].w, 4);
      std::memcpy(idx + (size_t)oi * k, hi.data() + (size_t)s * k, (size_t)k * 4);
      std::memcpy(d2 + (size_t)oi * k, hd.data() + (size_t)s * k, (size_t)k * 4);
    }
  });
}

int gicpb_get_covariances(gicpb_ctx* c, int which, double* cov9) {
  return guarded(c, [&] {
    if (!cov9) throw ArgError("null output");
    if (which != 0 && which != 1) throw ArgError("which must be 0 or 1");
    ensure_covariances(c);
    GridIndex& g = pick_grid(c, which);
    const int lo = which == 0 ? 0 : c->shard_lo;
    const int hi = which == 0 ? g.n_indexed() : c->shard_hi;
    const int n = hi - lo;
    std::vector<double> hn(3 * (size_t)std::max(n, 1));
    std::vector<float4> hp((size_t)g.n_indexed());
    GICPB_CUDA(cudaMemcpyAsync(hn.data(), (which == 0 ? c->n_tgt : c->n_src).get(), 3 * (size_t)n * sizeof(double),
                               cudaMemcpyDeviceToHost, c->stream));
    GICPB_CUDA(cudaMemcpyAsync(hp.data(), g.sorted_points(), hp.size() * sizeof(float4), cudaMemcpyDeviceToHost, c->stream));
    GICPB_CUDA(cudaStreamSynchronize(c->stream));
    const double a = 1.0 - c->prm.gicp_epsilon;
    const int64_t total = g.n_points();
    for (int64_t i = 0; i < 9 * total; ++i) cov9[i] = std::numeric_limits<double>::quiet_NaN();
    for (int s = 0; s < n; ++s) {
      int oi;
      std::memcpy(&oi, &hp[lo + s].w, 4);
      const double* nn = &hn[3 * (size_t)s];
      double* C = cov9 + 9 * (size_t)oi;
      for (int r = 0; r < 3; ++r)
        for (int q = 0; q < 3; ++q) C[3 * r + q] = (r == q ? 1.0 : 0.0) - a * nn[r] * nn[q];
    }
  });
}

int gicpb_correspondences(gicpb_ctx* c, const float transform[16], int32_t* nn_idx, float* d2, double* maha9,
                          int64_t* n_pairs) {
  return gicpb_correspondences_pass(c, transform, 0, nn_idx, d2, maha9, n_pairs);
}

int gicpb_correspondences_pass(gicpb_ctx* c, const float transform[16], int mode, int32_t* nn_idx, float* d2, double* maha9,
                               int64_t* n_pairs) {
  return guarded(c, [&] {
    if (!transform) throw ArgError("null transform");
    if (mode != 0 && mode != 1) throw ArgError("mode must be 0 (first pass) or 1 (a later pass)");
    ensure_covariances(c);
    run_correspondences(c, transform, mode == 0);
    const int lo = c->shard_lo, n = c->shard_hi - c->shard_lo;
    std::vector<int> hpos((size_t)std::max(n, 1));
    std::vector<float> hd2((size_t)std::max(n, 1));
    std::vector<float4> hs((size_t)c->src.n_indexed()), ht((size_t)c->tgt.n_indexed());
    std::vector<double> hm;
    std::vector<float> hmf;
    GICPB_CUDA(cudaMemcpyAsync(hpos.data(), c->pair_pos.get(), (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
    GICPB_CUDA(cudaMemcpyAsync(hd2.data(), c->pair_d2.get(), (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
    GICPB_CUDA(cudaMemcpyAsync(hs.data(), c->src.sorted_points(), hs.size() * sizeof(float4), cudaMemcpyDeviceToHost, c->stream));
    GICPB_CUDA(cudaMemcpyAsync(ht.data(), c->tgt.sorted_points(), ht.size() * sizeof(float4), cudaMemcpyDeviceToHost, c->stream));
    if (c->pairs_fp32) {
      hmf.resize(6 * (size_t)std::max(n, 1));
      GICPB_CUDA(cudaMemcpyAsync(hmf.data(), c->maha.get(), 6 * (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    } else {
      hm.resize(6 * (size_t)std::max(n, 1));
      GICPB_CUDA(cudaMemcpyAsync(hm.data(), c->maha.get(), 6 * (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    }
    GICPB_CUDA(cudaStreamSynchronize(c->stream));
    const int64_t total = c->src.n_points();
    if (nn_idx) for (int64_t i = 0; i < total; ++i) nn_idx[i] = -2;
    int64_t pairs = 0;
    for (int s = 0; s < n; ++s) {
      int oi;
      std::memcpy(&oi, &hs[lo + s].w, 4);
      int tj = -1;
      if (hpos[s] >= 0) {
        std::memcpy(&tj, &ht[hpos[s]].w, 4);
        ++pairs;
      }
      if (nn_idx) nn_idx[oi] = tj;
      if (d2) d2[oi] = hd2[s];
      if (maha9) {
        double* M = maha9 + 9 * (size_t)oi;
        if (tj < 0) {
          for (int e = 0; e < 9; ++e) M[e] = (e % 4 == 0) ? 1.0 : 0.0;
        } else {
          double v[6];
          for (int e = 0; e < 6; ++e) v[e] = c->pairs_fp32 ? (double)hmf[6 * (size_t)s + e] : hm[6 * (size_t)s + e];
          M[0] = v[0]; M[1] = v[1]; M[2] = v[2];
          M[3] = v[1]; M[4] = v[3]; M[5] = v[4];
          M[6] = v[2]; M[7] = v[4]; M[8] = v[5];
        }
      }
    }
    if (n_pairs) *n_pairs = pairs;
  });
}

int gicpb_cost(gicpb_ctx* c, const double x[6], double* f, double g[6]) {
  return guarded(c, [&] {
    if (!x || !f || !g) throw ArgError("null argument");
    update_shard(c);
    if (!c->pairs_valid) throw StateError("no correspondences: call gicpb_correspondences or gicpb_align first");
    double s[kCostSums];
    run_cost(c, x, s);
    if (s[13] < 1.0) throw AlignStop(GICPB_E_NOT_ENOUGH_CORRESPONDENCES, "no correspondences");
    cost_from_sums(x, s, f, g);
  });
}

int gicpb_cost_session(gicpb_ctx* c, int n_x, const double* xs, double* f, double* g, gicpb_cost_session_info* info) {
  return guarded(c, [&] {
    if (!xs || !f || !g || !info || n_x < 1) throw ArgError("bad argument");
    update_shard(c);
    if (!c->pairs_valid) throw StateError("no correspondences: call gicpb_correspondences or gicpb_align first");
    std::memset(info, 0, sizeof(*info));
    const int64_t before = g_launch_count.load();
    {
      CostSession session(c);
      info->persistent = c->cost_live ? 1 : 0;
      info->epoch_first = c->cost_live ? (int)c->cost_epoch : 0;
      for (int k = 0; k < n_x; ++k) {
        double s[kCostSums];
        run_cost(c, xs + 6 * (size_t)k, s);
        if (s[13] < 1.0) throw AlignStop(GICPB_E_NOT_ENOUGH_CORRESPONDENCES, "no correspondences");
        cost_from_sums(xs + 6 * (size_t)k, s, f + k, g + 6 * (size_t)k);
        info->n_pairs = (int64_t)s[13];
      }
      info->epoch_last = info->persistent ? (int)c->cost_epoch : 0;
    }
    GICPB_CUDA(cudaStreamSynchronize(c->stream));  // the resident kernel has taken its EXIT
    info->launches = g_launch_count.load() - before;
    if (info->persistent) {
      const CostPersistentShape& sh = c->cost_shape;
      info->blocks = sh.blocks;
      info->threads = sh.threads;
      info->stages = sh.stages;
      info->pairs_per_block = sh.per_block;
      info->resident_cap = sh.resident_cap;
      info->resident = sh.resident;
    }
  });
}

int gicpb_cloud_resolution(gicpb_ctx* c, int which, double* resolution) {
  return guarded(c, [&] {
    if (!resolution) throw ArgError("null output");
    GridIndex& g = pick_whole_grid(c, which);
    if (!g.ready()) throw StateError("cloud not set");
    const int n = g.n_indexed();
    const FarWork fw = far_work(c, n);
    c->partials.reserve((size_t)c->num_sms * 4 * 16 + 2 * (size_t)fitness_partial_rows(n, fw.far_blocks) + 64);
    c->d_sums.reserve(16);
    launch_resolution(g.view(), c->partials.get() + (size_t)c->num_sms * 4 * 16, c->d_sums.get(), fw, c->stream);
    GICPB_CUDA(cudaMemcpyAsync(c->h_sums, c->d_sums.get(), 2 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    GICPB_CUDA(cudaStreamSynchronize(c->stream));
    *resolution = c->h_sums[1] > 0 ? c->h_sums[0] / c->h_sums[1] : 0.0;
  });
}

// pcl::removeNaNNormalsFromPointCloud keeps a point iff all three components of its normal are finite.  That is "at least 3
// points inside the radius" almost always - but a neighbourhood whose float moments cancel to a zero covariance (a cloud far
// from the origin) gives 0 / 0 inside pcl::eigen33, and PCL drops that point too: the mask comes from the normals themselves.
int gicpb_normal_validity(gicpb_ctx* c, int which, double radius, uint8_t* valid, int64_t* n_valid) {
  return guarded(c, [&] {
    if (!valid) throw ArgError("null output");
    int64_t total = 0;
    const int64_t kept = compute_normals(c, which, radius, &total);
    std::vector<float> rows((size_t)total * 4);
    download_bytes(c, rows.data(), c->io_b.get(), (size_t)total * 16);
    for (int64_t i = 0; i < total; ++i)
      valid[i] = (std::isfinite(rows[4 * (size_t)i]) && std::isfinite(rows[4 * (size_t)i + 1]) &&
                  std::isfinite(rows[4 * (size_t)i + 2])) ? 1 : 0;
    if (n_valid) *n_valid = kept;
  });
}

int gicpb_normals(gicpb_ctx* c, int which, double radius, float* normals4, int64_t* n_valid) {
  return guarded(c, [&] {
    if (!normals4) throw ArgError("null output");
    int64_t total = 0;
    const int64_t kept = compute_normals(c, which, radius, &total);
    download_bytes(c, normals4, c->io_b.get(), (size_t)total * 16);
    if (n_valid) *n_valid = kept;
  });
}

int gicpb_euclidean_clusters(gicpb_ctx* c, const void* cloud, int64_t n, int64_t stride, int on_device, double tolerance,
                             int64_t min_size, int64_t max_size, int32_t* labels, int64_t* n_clusters) {
  return guarded(c, [&] {
    if (!labels && n > 0) throw ArgError("null labels");
    if (n_clusters) *n_clusters = 0;
    if (n == 0) return;  // pcl::EuclideanClusterExtraction on an empty cloud: no clusters
    check_cloud_args(cloud, n, stride);
    if (!(tolerance > 0)) throw ArgError("cluster tolerance must be > 0");
    if (max_size <= 0) max_size = INT_MAX;  // PCL default max_pts_per_cluster_
    // cells of the tolerance: the ball of a query cuts at most 3 x 3 x 3 of them
    bool any_finite = true;
    try {
      c->clu.build(cloud, n, stride, on_device != 0, (float)tolerance, c->prm.points_per_cell, c->stream, &c->stager);
    } catch (const ArgError& e) {
      if (std::string(e.what()) != "cloud has no finite point") throw;
      any_finite = false;
    }
    std::vector<int> root((size_t)n, -1);
    if (any_finite) {
      const GridView& g = c->clu.view();
      c->uf_parent.reserve((size_t)g.n);
      c->uf_root.reserve((size_t)n);
      GICPB_CUDA(cudaMemsetAsync(c->uf_root.get(), 0xff, (size_t)n * sizeof(int), c->stream));
      const float r2 = (float)(tolerance * tolerance);  // KdTreeFLANN::radiusSearch: float(radius * radius), d2 < r2
      launch_cluster_unions(g, r2, c->uf_parent.get(), c->uf_root.get(), far_work(c, g.n), c->stream);
      GICPB_CUDA(cudaMemcpyAsync(root.data(), c->uf_root.get(), (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
      GICPB_CUDA(cudaStreamSynchronize(c->stream));
    }
    // sizes, size filter, and PCL's output order: clusters by size, largest first (extract() sorts them; equal sizes
    // keep the order in which PCL's seed loop discovers them = by their lowest point index)
    std::vector<int> size((size_t)n, 0), first((size_t)n, -1);
    for (int64_t i = 0; i < n; ++i) {
      const int r = root[(size_t)i];
      if (r < 0) continue;
      if (size[(size_t)r]++ == 0) first[(size_t)r] = (int)i;
    }
    std::vector<int> keep;
    for (int64_t r = 0; r < n; ++r)
      if (size[(size_t)r] > 0 && size[(size_t)r] >= min_size && size[(size_t)r] <= max_size) keep.push_back((int)r);
    std::stable_sort(keep.begin(), keep.end(), [&](int a, int b) {
      if (size[(size_t)a] != size[(size_t)b]) return size[(size_t)a] > size[(size_t)b];
      return first[(size_t)a] < first[(size_t)b];
    });
    std::vector<int> rank((size_t)n, -1);
    for (size_t k = 0; k < keep.size(); ++k) rank[(size_t)keep[k]] = (int)k;
    for (int64_t i = 0; i < n; ++i) {
      const int r = root[(size_t)i];
      labels[i] = r >= 0 ? rank[(size_t)r] : -1;
    }
    if (n_clusters) *n_clusters = (int64_t)keep.size();
  });
}

int gicpb_voxel_grid(gicpb_ctx* c, const void* in, int64_t n, int64_t stride, int on_device, double leaf_size, void* out,
                     int64_t* n_out) {
  return guarded(c, [&] {
    if (!n_out) throw ArgError("null n_out");
    *n_out = 0;
    c->err.clear();  // the overflow warning below is the only text a successful call leaves
    if (n == 0) return;
    if (!out) throw ArgError("null output");
    check_cloud_args(in, n, stride);
    if (n > 0x7fffff00LL) throw ArgError("cloud has more than 2^31 points");
    if (!(leaf_size > 0)) throw ArgError("leaf size must be > 0");
    // the last point must reach through its z, and through its rgba word when the stride holds one
    const size_t full = (size_t)n * stride, bytes = (size_t)(n - 1) * stride + (stride >= 20 ? 20 : 12);
    const unsigned char* d_in = static_cast<const unsigned char*>(in);
    unsigned char* d_out = static_cast<unsigned char*>(out);
    if (!on_device) {
      c->io_a.reserve(full);
      c->io_b.reserve(full);
      GICPB_CUDA(cudaMemsetAsync(c->io_a.get() + bytes, 0, full - bytes, c->stream));
      upload_bytes(c, c->io_a.get(), in, bytes);
      d_in = c->io_a.get();
      d_out = c->io_b.get();
    }
    bool overflow = false;
    const int64_t m = c->voxel.run(d_in, n, stride, (float)leaf_size, d_out, c->stream, &overflow);
    if (overflow) {  // pcl::VoxelGrid: warns and passes the input through unchanged
      c->err = "Leaf size is too small for the input dataset. Integer indices would overflow.";
      if (on_device) {
        if (out != in) GICPB_CUDA(cudaMemcpyAsync(out, in, bytes, cudaMemcpyDeviceToDevice, c->stream));
      } else if (out != in) {
        std::memmove(out, in, bytes);
      }
      GICPB_CUDA(cudaStreamSynchronize(c->stream));
      *n_out = n;
      return;
    }
    if (!on_device && m > 0) download_bytes(c, out, d_out, (size_t)m * stride);  // whole rows: the zero bytes too
    GICPB_CUDA(cudaStreamSynchronize(c->stream));
    *n_out = m;
  });
}

// ---- SURVEY 8f row 4: PointCloud2 payloads and PCD files -> pcl::PointXYZRGB rows ------------------------------------------
namespace {
void unpack_pc2(gicpb_ctx* c, const void* data, bool data_on_device, const gicpb_pc2_layout& L, void* points32,
                bool points_on_device) {
  if (L.width < 0 || L.height < 0) throw ArgError("negative width / height");
  const int64_t n = L.width * L.height;
  if (n == 0) return;
  if (!data || !points32) throw ArgError("null pointer");
  if (n > 0x7fffff00LL) throw ArgError("cloud has more than 2^31 points");
  if (L.point_step < 12 || L.row_step < L.width * L.point_step) throw ArgError("point_step / row_step too small");
  const int32_t offs[3] = {L.off_x, L.off_y, L.off_z};
  for (int32_t o : offs)
    if (o < 0 || (int64_t)o + 4 > L.point_step) throw ArgError("x / y / z offset outside the point");
  if (L.off_rgb >= 0 && (int64_t)L.off_rgb + 4 > L.point_step) throw ArgError("rgb offset outside the point");
  const size_t in_bytes = (size_t)(L.height - 1) * L.row_step + (size_t)L.width * L.point_step;
  const unsigned char* d_in = static_cast<const unsigned char*>(data);
  if (!data_on_device) {
    c->io_a.reserve(in_bytes);
    upload_bytes(c, c->io_a.get(), data, in_bytes);
    d_in = c->io_a.get();
  }
  float4* d_out = static_cast<float4*>(points32);
  if (!points_on_device) {
    c->io_b.reserve((size_t)n * 32);
    d_out = reinterpret_cast<float4*>(c->io_b.get());
  } else if (reinterpret_cast<uintptr_t>(points32) % 16) {
    throw ArgError("device output must be 16-byte aligned");
  }
  launch_pc2_unpack(d_in, n, L.width, L.point_step, L.row_step, L.off_x, L.off_y, L.off_z, L.off_rgb, d_out, c->stream);
  if (!points_on_device) download_bytes(c, points32, reinterpret_cast<const unsigned char*>(d_out), (size_t)n * 32);
  GICPB_CUDA(cudaStreamSynchronize(c->stream));
}
}  // namespace

int gicpb_pointcloud2_to_xyzrgb(gicpb_ctx* c, const void* data, int data_on_device, const gicpb_pc2_layout* layout,
                                void* points32, int points_on_device) {
  return guarded(c, [&] {
    if (!layout) throw ArgError("null layout");
    unpack_pc2(c, data, data_on_device != 0, *layout, points32, points_on_device != 0);
  });
}

int gicpb_pcd_load_xyzrgb(gicpb_ctx* c, const char* path, void* points32, int64_t capacity, int points_on_device,
                          gicpb_pcd_info* info) {
  return guarded(c, [&] {
    if (!path || !info) throw ArgError("null path / info");
    PcdFile f;
    f.read_header(path);
    std::memset(info, 0, sizeof(*info));
    info->width = f.width;
    info->height = f.height;
    info->points = f.points;
    info->point_step = f.point_step;
    info->n_fields = (int32_t)f.fields.size();
    info->data_kind = f.data_kind;
    info->is_dense = 1;
    info->off_x = f.off_x;
    info->off_y = f.off_y;
    info->off_z = f.off_z;
    info->off_rgb = f.off_rgb;
    if (!points32) return;  // header only
    if (capacity < f.points) throw ArgError("output holds fewer rows than the file has points");
    if (f.off_x < 0 || f.off_y < 0 || f.off_z < 0) throw ArgError("PCD file has no FLOAT32 x / y / z fields");
    if (f.points == 0) return;
    // the body lands in pinned memory so that the upload is one asynchronous copy
    const size_t bytes = (size_t)f.points * f.point_step;
    unsigned char* blob = nullptr;
    GICPB_CUDA(cudaMallocHost(&blob, bytes));
    try {
      f.read_body(path, blob);
      info->is_dense = f.is_dense ? 1 : 0;
      gicpb_pc2_layout L{f.points, 1, f.point_step, f.points * (int64_t)f.point_step, f.off_x, f.off_y, f.off_z, f.off_rgb};
      unpack_pc2(c, blob, false, L, points32, points_on_device != 0);
    } catch (...) {
      cudaFreeHost(blob);
      throw;
    }
    cudaFreeHost(blob);
  });
}

int gicpb_grid_info_get(gicpb_ctx* c, int which, gicpb_grid_info* out) {
  return guarded(c, [&] {
    if (!out) throw ArgError("null output");
    GridIndex& g = pick_grid(c, which);
    if (!g.ready()) throw StateError("cloud not set");
    const GridIndex::Info& i = g.info();
    out->n_points = i.n_points;
    out->n_indexed = i.n_indexed;
    out->cell_size = i.cell_size;
    for (int a = 0; a < 3; ++a) out->dims[a] = i.dims[a];
    out->n_bricks_occupied = i.n_bricks_occupied;
    out->n_cells_occupied = i.n_cells_occupied;
    out->ms_build = i.ms_build;
  });
}

int gicpb_bench_kernel(gicpb_ctx* c, int which, const float transform[16], int iters, double* ms_mean, int64_t* launches) {
  return guarded(c, [&] {
    if (!transform || !ms_mean || iters < 1) throw ArgError("bad argument");
    ensure_covariances(c);
    ensure_pair_buffers(c);
    const Rigid T = rigid_from_rowmajor(transform);
    const int n = c->shard_hi - c->shard_lo;
    double x[6];
    transform_to_state(transform, x);
    if (which == 1 && !c->pairs_valid) run_correspondences(c, transform, true);
    if (which == 2) c->io_b.reserve((size_t)n * 8);
    const int64_t before = g_launch_count.load();
    if (which == 4 || which == 5) {
      // wall time of one evaluation as the optimiser sees it (command / launch -> sums on the host), mean over `iters`:
      // 4 = through the resident kernel of an inner solve, 5 = one launch per evaluation
      if (!c->pairs_valid) run_correspondences(c, transform, true);
      GICPB_CUDA(cudaStreamSynchronize(c->stream));
      const int keep = c->prm.cost_persistent;
      c->prm.cost_persistent = which == 4 ? 1 : 0;
      double s14[kCostSums];
      {
        CostSession session(c);
        for (int it = 0; it < 3; ++it) run_cost(c, x, s14);  // warm: the resident block is loaded, L2 holds the rest
        const double t0 = now_ms();
        for (int it = 0; it < iters; ++it) run_cost(c, x, s14);
        *ms_mean = (now_ms() - t0) / iters;
      }
      c->prm.cost_persistent = keep;
      GICPB_CUDA(cudaStreamSynchronize(c->stream));
      if (launches) *launches = g_launch_count.load() - before;
      return;
    }
    float total = 0.f;
    for (int it = 0; it < iters; ++it) {
      if (which == 0 || which == 3) {
        // records ev0 / ev1 around the kernel; 3 = as the first pass of a job runs it (1 probe ring: at the initial
        // pose most queries need the far search anyway), 0 = as every later pass does (3 rings), both unseeded
        run_correspondences(c, transform, true, which == 3 ? 1 : kNearMaxRing);
      } else if (which == 1) {
        float T16[16];
        state_to_transform(x, T16);
        GICPB_CUDA(cudaEventRecord(c->ev0, c->stream));
        launch_cost(c->src.sorted_points(), c->shard_lo, n, c->pair_tgt.get(), c->maha.get(), c->pairs_fp32,
                    rigid_from_rowmajor(T16), c->partials.get(), c->ticket.get(), c->d_sums.get(),
                    cost_grid_blocks(n, c->num_sms), c->stream);
        GICPB_CUDA(cudaEventRecord(c->ev1, c->stream));
      } else if (which == 2) {
        const float gate2 = corr_gate2(c->prm.max_corr_distance);
        GICPB_CUDA(cudaEventRecord(c->ev0, c->stream));
        launch_nn1(c->tgt.view(), c->src.sorted_points() + c->shard_lo, n, T, gate2,
                   reinterpret_cast<int*>(c->io_b.get()), reinterpret_cast<float*>(c->io_b.get() + (size_t)n * 4), nullptr,
                   far_work(c, n), c->stream);
        GICPB_CUDA(cudaEventRecord(c->ev1, c->stream));
      } else {
        throw ArgError("which must be 0 ... 5");
      }
      GICPB_CUDA(cudaEventSynchronize(c->ev1));
      float ms = 0.f;
      GICPB_CUDA(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
      total += ms;
    }
    *ms_mean = total / iters;
    if (launches) *launches = g_launch_count.load() - before;
  });
}

int64_t gicpb_launch_count(const gicpb_ctx*) { return g_launch_count.load(); }

void* gicpb_stream(const gicpb_ctx* c) { return c ? (void*)c->stream : nullptr; }

int64_t gicpb_last_far_queries(gicpb_ctx* c) {
  if (!c || !c->far_counter.get()) return -1;
  DeviceGuard guard(c->device);
  unsigned v[2] = {0, 0};
  if (cudaStreamSynchronize(c->stream) != cudaSuccess) return -1;
  if (cudaMemcpy(v, c->far_counter.get(), sizeof(v), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  return (int64_t)v[1];
}


int gicpb_group_create(const int* devices, int n_devices, gicpb_group** out) {
  if (!out) return GICPB_E_BADARG;
  *out = nullptr;
  if (!devices || n_devices < 1 || n_devices > kMaxPeers) return GICPB_E_BADARG;
  std::unique_ptr<gicpb_group> g(new gicpb_group);
  auto cleanup = [&] {
    for (gicpb_ctx* c : g->ctx) gicpb_destroy(c);
  };
  for (int r = 0; r < n_devices; ++r) {
    gicpb_ctx* c = nullptr;
    const int rc = gicpb_create(devices[r], &c);
    if (rc != GICPB_OK) {
      cleanup();
      return rc;
    }
    g->ctx.push_back(c);
  }
  if (n_devices == 1) {
    *out = g.release();
    return GICPB_OK;
  }
  g->lg.world = n_devices;
  g->lg.members = g->ctx;
  g->lg.slots.assign(80 * (size_t)n_devices, 0.0);
  // The fused sum makes each rank's cost kernel wait for the other ranks' kernels: only sound when every rank has a GPU of
  // its own (two such kernels on one GPU may never run at the same time) and every pair can map each other's memory.
  bool fused = true;
  for (int a = 0; a < n_devices && fused; ++a)
    for (int b = 0; b < n_devices && fused; ++b) {
      if (a == b) continue;
      int can = 0;
      if (devices[a] == devices[b] || cudaDeviceCanAccessPeer(&can, devices[a], devices[b]) != cudaSuccess || !can) fused = false;
    }
  if (const char* env = std::getenv("GICPB_NO_PEER"))
    if (*env == '1') fused = false;
  try {
    for (int r = 0; r < n_devices; ++r) {
      gicpb_ctx* c = g->ctx[(size_t)r];
      DeviceGuard guard(c->device);
      c->local = &g->lg;  // rank / world are set for the duration of each group call (group_run)
      if (!fused) continue;
      for (int b = 0; b < n_devices; ++b) {
        if (b == r) continue;
        const cudaError_t e = cudaDeviceEnablePeerAccess(devices[b], 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) GICPB_CUDA(e);
        (void)cudaGetLastError();
      }
      GICPB_CUDA(cudaMalloc(&c->peer_own, sizeof(PeerSlots)));
      GICPB_CUDA(cudaMemset(c->peer_own, 0, sizeof(PeerSlots)));
    }
    if (fused) {
      const char* env = std::getenv("GICPB_PEER_TIMEOUT_MS");
      const double ms = env && *env ? std::atof(env) : 30000.0;
      for (int r = 0; r < n_devices; ++r) {
        gicpb_ctx* c = g->ctx[(size_t)r];
        for (int b = 0; b < n_devices; ++b) c->peer.peers[b] = g->ctx[(size_t)b]->peer_own;  // plain device pointers (UVA)
        c->peer.rank = r;
        c->peer.world = n_devices;
        c->peer.seq = 0u;
        c->peer.timeout_ns = (unsigned long long)(std::max(ms, 1.0) * 1e6);
        c->peer_ipc = false;
        c->peer_ready = true;
      }
    }
  } catch (const std::exception&) {
    cleanup();
    return GICPB_E_CUDA;
  }
  g->fused = fused;
  *out = g.release();
  return GICPB_OK;
}

void gicpb_group_destroy(gicpb_group* g) {
  if (!g) return;
  for (gicpb_ctx* c : g->ctx) gicpb_destroy(c);
  delete g;
}

const char* gicpb_group_last_error(const gicpb_group* g) { return g ? g->err.c_str() : "null group"; }
int gicpb_group_size(const gicpb_group* g) { return g ? (int)g->ctx.size() : 0; }
int gicpb_group_fused(const gicpb_group* g) { return g && g->fused ? 1 : 0; }
gicpb_ctx* gicpb_group_ctx(gicpb_group* g, int rank) {
  return (g && rank >= 0 && rank < (int)g->ctx.size()) ? g->ctx[(size_t)rank] : nullptr;
}

int gicpb_group_set_params(gicpb_group* g, const gicpb_params* p) {
  if (!g) return GICPB_E_BADARG;
  for (gicpb_ctx* c : g->ctx) {
    const int rc = gicpb_set_params(c, p);
    if (rc != GICPB_OK) {
      g->err = c->err;
      return rc;
    }
  }
  return GICPB_OK;
}

int gicpb_group_set_clouds(gicpb_group* g, const void* target, int64_t n_target, int64_t target_stride, const void* source,
                           int64_t n_source, int64_t source_stride) {
  if (!g) return GICPB_E_BADARG;
  return group_run(g, [&](int, gicpb_ctx* c) {
    // host clouds: both uploads start on the copy stream (the source's runs beside the target's index build)
    int rc = gicpb_prefetch_cloud(c, 0, target, n_target, target_stride);
    if (rc == GICPB_OK) rc = gicpb_prefetch_cloud(c, 1, source, n_source, source_stride);
    if (rc == GICPB_OK) rc = gicpb_set_clouds(c, target, n_target, target_stride, source, n_source, source_stride, 0);
    return rc;
  });
}

int gicpb_group_align(gicpb_group* g, gicpb_align_result* out) {
  if (!g || !out) return GICPB_E_BADARG;
  std::vector<gicpb_align_result> res(g->ctx.size());
  const int rc = group_run(g, [&](int r, gicpb_ctx* c) { return gicpb_align(c, &res[(size_t)r]); });
  *out = res[0];
  // whole-job accounting: the ranks searched disjoint shards of the same passes
  for (size_t r = 1; r < res.size(); ++r) {
    out->corr_far_queries += res[r].corr_far_queries;
    out->ms_corr = std::max(out->ms_corr, res[r].ms_corr);
    if (rc == GICPB_OK && std::memcmp(res[r].transform, res[0].transform, sizeof(res[0].transform)) != 0) {
      g->err = "the GPUs of the group disagree on the transform";
      return GICPB_E_STATE;
    }
  }
  return rc;
}

int gicpb_group_fitness(gicpb_group* g, const float transform[16], double max_range, double* score) {
  if (!g || !score) return GICPB_E_BADARG;
  std::vector<double> sc(g->ctx.size(), 0.0);
  const int rc = group_run(g, [&](int r, gicpb_ctx* c) { return gicpb_fitness(c, transform, max_range, &sc[(size_t)r]); });
  *score = sc[0];
  return rc;
}

int gicpb_group_cloud_difference(gicpb_group* g, const void* input, int64_t n_input, int64_t input_stride,
                                 const void* subtract, int64_t n_subtract, int64_t subtract_stride, double sqr_threshold,
                                 uint8_t* mask, int64_t* n_kept) {
  if (!g) return GICPB_E_BADARG;
  try {
    check_difference_args(input, n_input, input_stride, subtract, n_subtract, subtract_stride, mask);
  } catch (const ArgError& e) {
    g->err = e.what();
    return GICPB_E_BADARG;
  }
  std::vector<int> rcs(g->ctx.size(), GICPB_OK);
  std::vector<unsigned long long> kept(g->ctx.size(), 0ull);
  const int rc = group_run(g, [&](int r, gicpb_ctx* c) {
    if (c->world == 1) {  // a group of one device is a plain context
      int64_t k = 0;
      rcs[(size_t)r] = gicpb_cloud_difference(c, input, n_input, input_stride, subtract, n_subtract, subtract_stride, 0,
                                              sqr_threshold, mask, &k);
      kept[(size_t)r] = (unsigned long long)k;
    } else {
      rcs[(size_t)r] = guarded(c, [&] {
        kept[(size_t)r] = group_difference_rank(c, input, n_input, input_stride, subtract, n_subtract, subtract_stride,
                                                sqr_threshold, mask);
      });
    }
    return rcs[(size_t)r];
  });
  if (rc == GICPB_E_BADARG)  // a bad cloud (no finite point) fails on every rank: report it as one context does
    for (size_t r = 0; r < rcs.size(); ++r)
      if (rcs[r] == GICPB_E_BADARG) {
        g->err = g->ctx[r]->err;
        break;
      }
  if (rc == GICPB_OK && n_kept) {
    unsigned long long total = 0;
    for (unsigned long long k : kept) total += k;
    *n_kept = (int64_t)total;
  }
  return rc;
}

}  // extern "C"
