// exchange.cu - the collectives of a sharded job (exchange.hpp): NCCL through dlopen, or peer copies and host sums inside a
// gicpb_group, and the set-up of the cost sum fused over peer memory.
#include <dlfcn.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "exchange.hpp"

namespace gicpb {

struct NcclApi {
  struct unique_id { char internal[128]; };
  int (*GetUniqueId)(unique_id*) = nullptr;
  int (*CommInitRank)(ncclComm**, int, unique_id, int) = nullptr;
  int (*CommDestroy)(ncclComm*) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, ncclComm*, cudaStream_t) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, ncclComm*, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  void* handle = nullptr;
};

namespace {

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
constexpr int kNcclInt8 = 0, kNcclFloat64 = 8, kNcclSum = 0;

void check_nccl(const NcclApi* nccl, int rc, const char* what) {
  if (rc != 0) throw NcclError(std::string(what) + ": " + nccl->GetErrorString(rc));
}

}  // namespace

bool nccl_unique_id(const char* libnccl_path, unsigned char id_out[128]) {
  std::string err;
  NcclApi* api = load_nccl(libnccl_path, err);
  if (!api || !id_out) return false;
  NcclApi::unique_id id;
  if (api->GetUniqueId(&id) != 0) return false;
  std::memcpy(id_out, id.internal, 128);
  return true;
}

Exchange::~Exchange() {
  if (comm && nccl) nccl->CommDestroy(comm);
  if (peer.world > 1 && peer_ipc)
    for (int r = 0; r < peer.world; ++r)
      if (r != peer.rank && peer.peers[r]) cudaIpcCloseMemHandle(peer.peers[r]);
  if (peer_own) cudaFree(peer_own);
}

void Exchange::init_nccl(const char* libnccl_path, int rank_, int world_, const unsigned char id[128]) {
  std::string err;
  nccl = load_nccl(libnccl_path, err);
  if (!nccl) throw NcclError(err);
  NcclApi::unique_id uid;
  std::memcpy(uid.internal, id, 128);
  check_nccl(nccl, nccl->CommInitRank(&comm, world_, uid, rank_), "ncclCommInitRank");
  rank = rank_;
  world = world_;
}

void Exchange::all_reduce_sum(double* dev, int count, cudaStream_t stream) {
  if (world <= 1) return;
  if (!local) {
    check_nccl(nccl, nccl->AllReduce(dev, dev, (size_t)count, kNcclFloat64, kNcclSum, comm, stream), "ncclAllReduce");
    return;
  }
  double* mine = local->slots.data() + 80 * (size_t)rank;
  GICPB_CUDA(cudaMemcpyAsync(mine, dev, (size_t)count * sizeof(double), cudaMemcpyDeviceToHost, stream));
  GICPB_CUDA(cudaStreamSynchronize(stream));
  local->barrier();
  double sum[80];
  for (int k = 0; k < count; ++k) {
    double v = 0.0;
    for (int r = 0; r < world; ++r) v += local->slots[80 * (size_t)r + k];
    sum[k] = v;
  }
  local->barrier();  // everybody has read the slots: they may be written again
  GICPB_CUDA(cudaMemcpyAsync(dev, sum, (size_t)count * sizeof(double), cudaMemcpyHostToDevice, stream));
  GICPB_CUDA(cudaStreamSynchronize(stream));
}

void Exchange::gather_send(void* buf, size_t chunk, cudaStream_t stream) {
  if (world <= 1 || local) return;
  check_nccl(nccl, nccl->AllGather(static_cast<unsigned char*>(buf) + (size_t)rank * chunk, buf, chunk, kNcclInt8, comm, stream),
             "ncclAllGather");
}

void Exchange::gather_recv(void* buf, size_t chunk, size_t total, cudaStream_t stream, const MemberBuf& member) {
  if (world <= 1 || !local) return;
  barrier(stream);  // every rank's chunk is complete and its buffer in place
  for (int r = 0; r < world; ++r) {
    const size_t lo = std::min(total, (size_t)r * chunk), hi = std::min(total, lo + chunk);
    if (r != rank && hi > lo)
      GICPB_CUDA(cudaMemcpyPeerAsync(static_cast<unsigned char*>(buf) + lo, local->devices[(size_t)rank],
                                     static_cast<const unsigned char*>(member(r)) + lo, local->devices[(size_t)r], hi - lo, stream));
  }
}

void Exchange::fetch_all(void* dst, size_t offset, size_t bytes, cudaStream_t stream, const MemberBuf& member) {
  barrier(stream);
  for (int r = 0; r < world && bytes > 0; ++r)
    GICPB_CUDA(cudaMemcpyPeerAsync(static_cast<unsigned char*>(dst) + (size_t)r * bytes, local->devices[(size_t)rank],
                                   static_cast<const unsigned char*>(member(r)) + offset, local->devices[(size_t)r], bytes,
                                   stream));
}

void Exchange::barrier(cudaStream_t stream) {
  if (world <= 1 || !local) return;
  GICPB_CUDA(cudaStreamSynchronize(stream));
  local->barrier();
}

void Exchange::alloc_peer_slots() {
  if (peer_own) return;
  GICPB_CUDA(cudaMalloc(&peer_own, sizeof(PeerSlots)));
  GICPB_CUDA(cudaMemset(peer_own, 0, sizeof(PeerSlots)));
}

void Exchange::arm_fused_sum(int rank_, int world_, PeerSlots* const* peers, bool ipc) {
  const char* env = std::getenv("GICPB_PEER_TIMEOUT_MS");
  const double ms = env && *env ? std::atof(env) : 30000.0;
  for (int r = 0; r < world_; ++r) peer.peers[r] = peers[r];
  peer.rank = rank_;
  peer.world = world_;
  peer.seq = 0u;
  peer.timeout_ns = (unsigned long long)(std::max(ms, 1.0) * 1e6);
  peer_ipc = ipc;
  peer_ready = true;
}

void Exchange::fused_sum_timed_out() {
  peer_ready = false;
  throw NcclError("peer-memory reduction timed out: a rank did not launch this evaluation (GICPB_PEER_TIMEOUT_MS)");
}

}  // namespace gicpb
