// exchange.hpp - how the ranks of a sharded job exchange data (exchange.cu): NCCL with one process per GPU (gicpb_comm_init),
// or peer copies and sums through the host between the members of a gicpb_group (one process, one host thread per GPU).
#pragma once
#include <condition_variable>
#include <functional>
#include <mutex>
#include <string>
#include <vector>

#include "kernels.hpp"

struct ncclComm;

namespace gicpb {

struct NcclError : std::runtime_error {
  using std::runtime_error::runtime_error;
};
struct GroupAbort : StateError {  // group_run matches the message: a rank that only gave up is not the cause
  GroupAbort() : StateError("another GPU of the group failed") {}
};

// libnccl through dlopen (path null or empty: libnccl.so.2); false if it cannot be loaded
bool nccl_unique_id(const char* libnccl_path, unsigned char id_out[128]);

// what the members of one gicpb_group share
struct LocalGroup {
  std::vector<int> devices;   // device of every rank
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
    if (++waiting == (int)devices.size()) {
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

struct NcclApi;

// who the ranks are and how they talk; a context holds one
struct Exchange {
  int rank = 0, world = 1;
  LocalGroup* local = nullptr;  // member of a gicpb_group: the collectives go over peer copies / the host, not NCCL
  NcclApi* nccl = nullptr;
  ncclComm* comm = nullptr;
  // fused cost + cross-GPU sum over peer memory (kernels.hpp PeerReduce); falls back to all_reduce_sum when not set up
  PeerSlots* peer_own = nullptr;
  PeerReduce peer{};
  bool peer_ready = false;
  bool peer_ipc = false;  // peer.peers[] are cudaIpc mappings (closed on destruction)

  Exchange() = default;
  Exchange(const Exchange&) = delete;
  Exchange& operator=(const Exchange&) = delete;
  ~Exchange();
  void init_nccl(const char* libnccl_path, int rank, int world, const unsigned char id[128]);

  // `count` (<= 80) device doubles summed over the ranks in place on `stream`; a group adds them in rank order on every
  // rank (identical sums) and synchronises `stream`
  void all_reduce_sum(double* dev, int count, cudaStream_t stream);

  // In-place all-gather of the chunks [r * chunk, (r + 1) * chunk) of rank r of a buffer held by every rank, clipped to
  // `total` bytes.  Every rank calls gather_send once its chunk is queued on `stream` (NCCL: ncclAllGather there), then
  // gather_recv before `stream` (ordered after that) reads the other chunks (a group: copies them out of member(r), rank
  // r's buffer), and barrier(stream) before it writes its buffer again.
  using MemberBuf = std::function<const void*(int rank)>;
  void gather_send(void* buf, size_t chunk, cudaStream_t stream);
  void gather_recv(void* buf, size_t chunk, size_t total, cudaStream_t stream, const MemberBuf& member);
  // group only: dst[r * bytes, (r + 1) * bytes) = member(r)[offset, offset + bytes) for every rank r, this one too
  void fetch_all(void* dst, size_t offset, size_t bytes, cudaStream_t stream, const MemberBuf& member);
  // a group waits for `stream`, then for every member (gather_recv and fetch_all begin with it); NCCL: nothing
  void barrier(cudaStream_t stream);

  bool may_shard_uploads() const { return world > 1 && (local != nullptr || comm != nullptr); }

  void alloc_peer_slots();  // this rank's zeroed slot block, once
  // peers[r]: rank r's slot block as mapped here (ipc: cudaIpc mappings, else plain device pointers)
  void arm_fused_sum(int rank, int world, PeerSlots* const* peers, bool ipc);
  // what the cost kernels take when they sum over the ranks themselves; null: all_reduce_sum
  const PeerReduce* fused_sum() const { return world > 1 && peer_ready ? &peer : nullptr; }
  // a fused sum came back NaN (a rank did not show up in time): back to all_reduce_sum, and throw NcclError
  [[noreturn]] void fused_sum_timed_out();
};

}  // namespace gicpb
