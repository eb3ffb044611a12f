// Communicator of the distributed loop-closure batch (dist.cu) as batch.cu sees it.
#pragma once
#include <functional>
#include <vector>

#include "common.cuh"

struct lgs_comm {
  void* comm = nullptr;  // ncclComm_t
  bool own = false;      // created by lgs_comm_init_rank (destroyed with the handle) or adopted from the caller
  int rank = 0, world = 1, device = 0;
  lgs::DevBuf send, recv;  // the per-rank capacity of records; W times that
  lgs::PinnedBuf host;     // gathered records on their way to the caller's array
};

namespace lgs {

void partition_pairs(const int64_t* sizes, int64_t n_total, int rank, int world, std::vector<int32_t>* mine);
// ncclAllGather of c->send (cap records of record_bytes per rank) on stream st; then place(record) for every gathered slot,
// which returns 1 when it stored the record, 0 for an unused slot, or an error code (having called set_error).
// *n_received = records placed.
int comm_all_gather(lgs_comm* c, cudaStream_t st, int64_t cap, size_t record_bytes, const std::function<int(const void*)>& place, int64_t* n_received);

}  // namespace lgs
