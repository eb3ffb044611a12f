// Multi-GPU plumbing of the loop-closure batch and of offline odometry (SURVEY section 8e): one process per GPU, work
// items (candidate pairs, sequences) dealt to the ranks by size with no data-path collective, and ONE ncclAllGather of
// fixed-size result records over NVLink / NVSwitch.  The batch's 96-byte records are written into the send buffer by the
// last kernel of each pair (nn.cu), so nothing is staged between the verification and the collective.
//
// NCCL is bound at run time (dlopen): a process that already holds a libnccl (PyTorch ships its own) keeps using that
// one, a plain C++ host gets the system library, and a single-GPU user of liblgs_b200.so needs no NCCL at all.
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <mutex>
#include <numeric>
#include <vector>

#include "dist.cuh"

namespace lgs {

namespace {

struct NcclApi {
  void* handle = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*CommCount)(const ncclComm_t, int*) = nullptr;
  ncclResult_t (*CommUserRank)(const ncclComm_t, int*) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GetVersion)(int*) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  std::string error;
};

NcclApi* nccl_api() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    const char* env = getenv("LGS_NCCL_LIB");
    void* h = nullptr;
    if (env && env[0]) h = dlopen(env, RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);  // the copy this process already uses, if any
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) {
      const char* e = dlerror();
      api.error = std::string("libnccl.so.2 not found (set LGS_NCCL_LIB): ") + (e ? e : "");
      return;
    }
    api.handle = h;
#define LGS_SYM(field, name)                                          \
  api.field = reinterpret_cast<decltype(api.field)>(dlsym(h, name)); \
  if (!api.field) api.error = std::string("symbol missing in libnccl: ") + name;
    LGS_SYM(GetUniqueId, "ncclGetUniqueId")
    LGS_SYM(CommInitRank, "ncclCommInitRank")
    LGS_SYM(CommDestroy, "ncclCommDestroy")
    LGS_SYM(CommCount, "ncclCommCount")
    LGS_SYM(CommUserRank, "ncclCommUserRank")
    LGS_SYM(AllGather, "ncclAllGather")
    LGS_SYM(GetVersion, "ncclGetVersion")
    LGS_SYM(GetErrorString, "ncclGetErrorString")
#undef LGS_SYM
  });
  return &api;
}

int require_nccl(NcclApi** out) {
  NcclApi* a = nccl_api();
  if (!a->handle || !a->error.empty()) {
    set_error("NCCL unavailable: %s", a->error.c_str());
    return LGS_ERR_STATE;
  }
  *out = a;
  return LGS_OK;
}

#define LGS_NCCL(api, call)                                                                              \
  do {                                                                                                   \
    ncclResult_t _r = (call);                                                                            \
    if (_r != ncclSuccess) {                                                                             \
      lgs::set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #call, (api)->GetErrorString(_r));      \
      return LGS_ERR_CUDA;                                                                               \
    }                                                                                                    \
  } while (0)

}  // namespace

// Deal the pairs to the ranks: descending size (index breaks ties), round-robin, so that every rank receives
// ceil(P/W) or floor(P/W) pairs of similar total size (SURVEY section 8e).  The local list is ascending in pair index.
void partition_pairs(const int64_t* sizes, int64_t n_total, int rank, int world, std::vector<int32_t>* mine) {
  std::vector<int32_t> order(static_cast<size_t>(n_total));
  std::iota(order.begin(), order.end(), 0);
  std::stable_sort(order.begin(), order.end(), [&](int32_t a, int32_t b) { return sizes[a] > sizes[b]; });
  mine->clear();
  for (int64_t p = rank; p < n_total; p += world) mine->push_back(order[static_cast<size_t>(p)]);
  std::sort(mine->begin(), mine->end());
}

int comm_all_gather(lgs_comm* c, cudaStream_t st, int64_t cap, size_t record_bytes, const std::function<int(const void*)>& place, int64_t* n_received) {
  NcclApi* api = nullptr;
  LGS_TRY(require_nccl(&api));
  const size_t bytes = static_cast<size_t>(cap) * record_bytes;
  LGS_TRY(c->recv.reserve(bytes * c->world));
  LGS_TRY(c->host.reserve(bytes * c->world));
  LGS_NCCL(api, api->AllGather(c->send.p, c->recv.p, bytes, ncclInt8, static_cast<ncclComm_t>(c->comm), st));
  LGS_CUDA(cudaMemcpyAsync(c->host.p, c->recv.p, bytes * c->world, cudaMemcpyDeviceToHost, st));
  LGS_CUDA(cudaStreamSynchronize(st));
  const unsigned char* h = c->host.as<unsigned char>();
  int64_t got = 0;
  for (int64_t i = 0; i < cap * c->world; i++) {
    const int r = place(h + static_cast<size_t>(i) * record_bytes);
    if (r < 0) return r;
    got += r;
  }
  if (n_received) *n_received = got;
  return LGS_OK;
}

}  // namespace lgs

using namespace lgs;

extern "C" {

int lgs_comm_get_unique_id(uint8_t* id128) {
  LGS_REQUIRE(id128, "null argument");
  NcclApi* api = nullptr;
  LGS_TRY(require_nccl(&api));
  static_assert(sizeof(ncclUniqueId) == LGS_COMM_ID_BYTES, "ncclUniqueId is 128 bytes");
  ncclUniqueId id;
  LGS_NCCL(api, api->GetUniqueId(&id));
  memcpy(id128, &id, sizeof(id));
  return LGS_OK;
}

int lgs_comm_init_rank(const uint8_t* id128, int32_t rank, int32_t world, int32_t device, lgs_comm** out) {
  LGS_REQUIRE(id128 && out, "null argument");
  LGS_REQUIRE(world >= 1 && rank >= 0 && rank < world, "rank / world out of range");
  NcclApi* api = nullptr;
  LGS_TRY(require_nccl(&api));
  LGS_CUDA(cudaSetDevice(device));
  ncclUniqueId id;
  memcpy(&id, id128, sizeof(id));
  ncclComm_t comm = nullptr;
  LGS_NCCL(api, api->CommInitRank(&comm, world, id, rank));
  lgs_comm* c = new lgs_comm;
  c->comm = comm;
  c->own = true;
  c->rank = rank;
  c->world = world;
  c->device = device;
  *out = c;
  return LGS_OK;
}

int lgs_comm_adopt(void* nccl_comm, int32_t device, lgs_comm** out) {
  LGS_REQUIRE(nccl_comm && out, "null argument");
  NcclApi* api = nullptr;
  LGS_TRY(require_nccl(&api));
  int rank = 0, world = 0;
  LGS_NCCL(api, api->CommUserRank(static_cast<ncclComm_t>(nccl_comm), &rank));
  LGS_NCCL(api, api->CommCount(static_cast<ncclComm_t>(nccl_comm), &world));
  lgs_comm* c = new lgs_comm;
  c->comm = nccl_comm;
  c->own = false;
  c->rank = rank;
  c->world = world;
  c->device = device;
  *out = c;
  return LGS_OK;
}

void lgs_comm_destroy(lgs_comm* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  c->send.release();
  c->recv.release();
  c->host.release();
  if (c->own && c->comm) {
    NcclApi* api = nccl_api();
    if (api->CommDestroy) api->CommDestroy(static_cast<ncclComm_t>(c->comm));
  }
  delete c;
}

int lgs_comm_info(lgs_comm* c, int32_t* rank, int32_t* world, int32_t* nccl_version) {
  LGS_REQUIRE(c, "null argument");
  if (rank) *rank = c->rank;
  if (world) *world = c->world;
  if (nccl_version) {
    NcclApi* api = nullptr;
    LGS_TRY(require_nccl(&api));
    int v = 0;
    LGS_NCCL(api, api->GetVersion(&v));
    *nccl_version = v;
  }
  return LGS_OK;
}

int lgs_batch_partition(const int64_t* sizes, int64_t n_total, int32_t rank, int32_t world, int32_t* out_ids, int64_t capacity, int64_t* n_mine) {
  LGS_REQUIRE(n_mine && (sizes || n_total == 0), "null argument");
  LGS_REQUIRE(n_total >= 0 && n_total < (int64_t(1) << 31), "pair count out of range");
  LGS_REQUIRE(world >= 1 && rank >= 0 && rank < world, "rank / world out of range");
  std::vector<int32_t> mine;
  partition_pairs(sizes, n_total, rank, world, &mine);
  *n_mine = static_cast<int64_t>(mine.size());
  if (out_ids) {
    LGS_REQUIRE(capacity >= *n_mine, "out_ids too small");
    std::copy(mine.begin(), mine.end(), out_ids);
  }
  return LGS_OK;
}

}  // extern "C"
