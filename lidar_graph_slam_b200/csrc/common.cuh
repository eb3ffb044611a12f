// Shared plumbing of liblgs_b200.so: error handling, the context (device + stream + arenas), growable
// device buffers and small device helpers.  sm_100a only.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include <nvtx3/nvToolsExt.h>

#include "../../include/lgs_c.h"

namespace lgs {

void set_error(const char* fmt, ...);

#define LGS_CUDA(call)                                                                                     \
  do {                                                                                                     \
    cudaError_t _e = (call);                                                                               \
    if (_e != cudaSuccess) {                                                                               \
      lgs::set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e));           \
      return LGS_ERR_CUDA;                                                                                 \
    }                                                                                                      \
  } while (0)

#define LGS_TRY(call)          \
  do {                         \
    int _r = (call);           \
    if (_r != LGS_OK) return _r; \
  } while (0)

#define LGS_REQUIRE(cond, msg)                 \
  do {                                         \
    if (!(cond)) {                             \
      lgs::set_error("%s: %s", __func__, msg); \
      return LGS_ERR_INVALID;                  \
    }                                          \
  } while (0)

// NVTX range over an API call (SURVEY section 5: the reference has no tracing; Nsight Systems / Compute timelines of a node
// that links this library show one range per registration call).  nvtx3 is header-only and a no-op without a tool attached.
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};
#define LGS_NVTX(name) lgs::NvtxRange lgs_nvtx_range_(name)

constexpr int kNumSMs = 148;  // B200

// Growable device allocation; never shrinks, so steady-state calls do not touch cudaMalloc.
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  int reserve(size_t bytes) {
    if (bytes <= cap) return LGS_OK;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 4 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) {
      set_error("cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
      p = nullptr;
      return LGS_ERR_CUDA;
    }
    cap = want;
    return LGS_OK;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <typename T>
  T* as() const {
    return static_cast<T*>(p);
  }
};

// Pinned host staging (results, small parameter blocks).
struct PinnedBuf {
  void* p = nullptr;
  size_t cap = 0;
  int reserve(size_t bytes) {
    if (bytes <= cap) return LGS_OK;
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
    cudaError_t e = cudaHostAlloc(&p, bytes + 256, cudaHostAllocDefault);
    if (e != cudaSuccess) {
      set_error("cudaHostAlloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
      p = nullptr;
      return LGS_ERR_CUDA;
    }
    cap = bytes + 256;
    return LGS_OK;
  }
  void release() {
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
  }
  template <typename T>
  T* as() const {
    return static_cast<T*>(p);
  }
};

// Result mailbox: a small block of host memory (pinned, mapped into the device address space) that the last CTA of
// a reduction kernel writes its result into.  Every value travels as one 16-byte record {value, token} written with
// a single 128-bit store, so each record validates itself (a 16-byte aligned record lies in one cache line and one
// PCIe write; the host reads the token first and the value after it): no fence, no flag, no D2H copy and no stream
// synchronisation - one posted PCIe write replaces ~15-25 us of copy + sync latency per Gauss-Newton / line-search
// evaluation.
constexpr int kMailboxRecords = 48;
struct MailboxRecord {
  double v;
  unsigned long long token;
};
struct MailboxHost {
  MailboxRecord r[kMailboxRecords];
};
struct Mailbox {  // kernel argument
  MailboxRecord* r;
  unsigned long long token;
};

}  // namespace lgs

struct lgs_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  int64_t launches = 0;
  lgs::DevBuf raw;       // AoS upload staging
  lgs::DevBuf tmp[8];    // general scratch arenas (per-call meaning)
  lgs::DevBuf sort_tmp;  // look-back scratch of the sort / scan primitives (sort.cuh)
  lgs::PinnedBuf pin;    // small D2H results
  lgs::PinnedBuf pin_up; // small H2D parameter blocks
  lgs::DevBuf vg_in, vg_out, vg_vidx, vg_rank;  // host-facing voxel-grid call: staged cloud + device-side outputs
  lgs::MailboxHost* mbox = nullptr;             // result mailbox (mapped pinned host memory)
  unsigned long long mbox_token = 0;
  bool polite_wait = false;  // batch workers: yield the core while waiting for a mailbox (several workers may share one)
  // One-shot record sink of the loop-closure batch (batch.cu, dist.cu): when set, the next getFitnessScore kernel on this
  // context - the last kernel of a candidate pair - completes rec_out_proto with the fitness it has just reduced and
  // stores the 96-byte record at rec_out_dev (a slot of the NCCL send buffer): no staging copy precedes the gather.
  lgs_align_result* rec_out_dev = nullptr;
  lgs_align_result rec_out_proto;
};

namespace lgs {

inline int use_device(const lgs_ctx* c) {
  LGS_CUDA(cudaSetDevice(c->device));
  return LGS_OK;
}

// Upload a host cloud with arbitrary record stride into packed float4 xyzi device storage.
int upload_cloud(lgs_ctx* ctx, const void* pts, int64_t n, int32_t stride_bytes, DevBuf* dst);
// The repack half of upload_cloud: n records of stride_bytes already in device memory -> packed float4 xyzi, on ctx's stream.
int repack_cloud(lgs_ctx* ctx, const void* raw_dev, int64_t n, int32_t stride_bytes, float4* dst);
// The input of every registration set_source / set_target entry point, validated on the host before anything is copied:
// host records of stride_bytes each (as upload_cloud) or, on_device, a packed float4 xyzi device array (copied device to
// device; stride_bytes unused).  pts may be null only when n == 0.
int load_cloud(lgs_ctx* ctx, const void* pts, int64_t n, int32_t stride_bytes, bool on_device, DevBuf* dst);

// dst = T * src as pcl::transformPointCloud (intensity kept); T column-major
int transform_cloud(lgs_ctx* ctx, const float4* src, int64_t n, const float* T, float4* dst);
// The aligned source cloud of align(output, guess): T * src through the device buffer scratch into out_host (n x 4 floats),
// waited for.  Nothing to do when n == 0.
int write_aligned_cloud(lgs_ctx* ctx, const float4* src, int64_t n, const float* T, DevBuf* scratch, float* out_host);

// Next mailbox token + kernel argument; mailbox_wait spins until the kernel has published k records with that token
// (checking the stream for errors now and then) and copies the values to out.
int mailbox_next(lgs_ctx* ctx, Mailbox* mb);
int mailbox_wait(lgs_ctx* ctx, const Mailbox& mb, int k, double* out);

inline int grid_for(int64_t n, int block) { return static_cast<int>((n + block - 1) / block); }

#ifdef __CUDACC__
// order-preserving float <-> uint encoding for atomic min/max
__device__ __forceinline__ unsigned enc_f(float f) {
  unsigned u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ __forceinline__ float dec_f_host(unsigned u) {
  unsigned v = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
  float f;
  memcpy(&f, &v, 4);
  return f;
}

// pcl::transformPointCloud order (PCL >= 1.10): c0*x + (c1*y + (c2*z + c3)), explicit rn ops so the
// compiler can neither contract nor reassociate.  T column-major.
// publish K doubles (threads 0..K-1 hold them) to the mailbox: one 128-bit store per value
template <int K>
__device__ __forceinline__ void mailbox_publish(const Mailbox& mb, double v) {
  static_assert(K <= kMailboxRecords, "mailbox too small");
  if (threadIdx.x < K) {
    const unsigned long long bits = static_cast<unsigned long long>(__double_as_longlong(v));
    asm volatile("st.global.v2.u64 [%0], {%1, %2};" ::"l"(mb.r + threadIdx.x), "l"(bits), "l"(mb.token) : "memory");
  }
}

// one value into record `slot` by the calling thread alone (single-thread finishers: look-back scans, atomic accumulators)
__device__ __forceinline__ void mailbox_publish_one(const Mailbox& mb, int slot, double v) {
  const unsigned long long bits = static_cast<unsigned long long>(__double_as_longlong(v));
  asm volatile("st.global.v2.u64 [%0], {%1, %2};" ::"l"(mb.r + slot), "l"(bits), "l"(mb.token) : "memory");
}

__device__ __forceinline__ float3 transform_pcl(const float* __restrict__ T, float x, float y, float z) {
  float3 r;
  r.x = __fadd_rn(__fmul_rn(T[0], x), __fadd_rn(__fmul_rn(T[4], y), __fadd_rn(__fmul_rn(T[8], z), T[12])));
  r.y = __fadd_rn(__fmul_rn(T[1], x), __fadd_rn(__fmul_rn(T[5], y), __fadd_rn(__fmul_rn(T[9], z), T[13])));
  r.z = __fadd_rn(__fmul_rn(T[2], x), __fadd_rn(__fmul_rn(T[6], y), __fadd_rn(__fmul_rn(T[10], z), T[14])));
  return r;
}
#endif

}  // namespace lgs
