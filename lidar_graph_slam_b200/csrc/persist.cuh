// Host -> resident-grid command channel shared by the persistent evaluators of ICP (icp.cu) and pclomp GICP (gicp_bfgs.cu).
//
// A command travels like a mailbox result in the other direction: 16-byte chunks {8 bytes of payload, sequence number}
// in mapped pinned host memory, each chunk validating itself (the host stores the payload word before the sequence
// word; a PCIe read returns a snapshot of the chunk), so warp 0 of CTA 0 fetches a whole command with ONE round of
// loads per poll.  It relays the payload into device memory (release); every CTA (CTA 0 included) acquires that copy
// from L2 and stages it in shared memory.  A command that does not arrive within ~0.5 s makes the grid give up: the
// host then finds a drained stream instead of a hang and goes on with plain launches (ResidentSession::recover).
//
// Two resident grids that each need every SM would wait for one another's SMs forever, so at most one session per
// device exists in the process (persist_try_acquire / persist_release, ctx.cu).
#pragma once
#include <atomic>

#include "common.cuh"

namespace lgs {

struct CmdChunk {
  unsigned long long data, seq;
};
template <int WORDS>
struct CmdHost {
  CmdChunk c[WORDS];
};
template <int WORDS>
struct CmdDev {
  unsigned long long data[WORDS];
  unsigned long long seq;
};

bool persist_try_acquire(int device);  // one resident evaluator per device and process
void persist_release(int device);
bool persist_env_enabled();            // LGS_NDT_PERSISTENT / injected CUDA tools (see ctx.cu)

// payload word first, sequence word second, chunk by chunk (x86 stores are not reordered with other stores)
template <int WORDS>
inline void persist_send(CmdHost<WORDS>* host, unsigned long long seq, const void* payload) {
  const unsigned long long* w = static_cast<const unsigned long long*>(payload);
  volatile CmdChunk* c = host->c;
  for (int i = 0; i < WORDS; i++) {
    c[i].data = w[i];
    std::atomic_thread_fence(std::memory_order_release);
    c[i].seq = seq;
  }
}

// Host side of one resident grid: the mapped command block, its device relay, the sequence counter and the device lock.
// While a session is open no other kernel may be put on its stream: one queued behind a grid that waits for commands
// would start only after the grid's time-out.  The owner closes the session first.
template <typename Cmd>
struct ResidentSession {
  static constexpr int kWords = static_cast<int>(sizeof(Cmd) / 8);
  static_assert(sizeof(Cmd) % 8 == 0, "commands are copied as 64-bit words");
  using Host = CmdHost<kWords>;
  using Dev = CmdDev<kWords>;

  Cmd quit;               // the command that makes the grid exit
  bool enabled = false;   // inside an align (SessionScope)
  bool active = false;    // a grid is resident and holds the lock of `device`
  bool broken = false;    // a grid timed out: plain launches from then on
  int device = -1;
  Host* host = nullptr;   // mapped pinned memory
  DevBuf dev;
  unsigned long long seq = 0;

  explicit ResidentSession(const Cmd& quit_cmd) : quit(quit_cmd) {}

  // whatever allocates or synchronises, before a grid becomes resident
  int prepare(lgs_ctx* ctx) {
    if (!host) {
      void* p = nullptr;
      LGS_CUDA(cudaHostAlloc(&p, sizeof(Host), cudaHostAllocMapped | cudaHostAllocPortable));
      memset(p, 0, sizeof(Host));
      host = static_cast<Host*>(p);
    }
    if (!dev.p) {
      LGS_TRY(dev.reserve(sizeof(Dev)));
      LGS_CUDA(cudaMemsetAsync(dev.p, 0, sizeof(Dev), ctx->stream));
    }
    return LGS_OK;
  }

  // Keeps or makes a grid resident when the session is enabled and not broken, LGS_NDT_PERSISTENT allows it, the grid
  // fits and the device lock is free; otherwise closes the session and the caller launches plainly.
  // launch(host block as the device sees it, device relay, first sequence number) puts the persistent kernel on the stream.
  template <typename Launch>
  int open(lgs_ctx* ctx, bool fits, Launch&& launch) {
    if (!enabled || broken || !fits || !persist_env_enabled()) {
      close();
      return LGS_OK;
    }
    if (active) return LGS_OK;
    LGS_TRY(prepare(ctx));
    void* dv = nullptr;
    LGS_CUDA(cudaHostGetDevicePointer(&dv, host, 0));
    if (!persist_try_acquire(ctx->device)) return LGS_OK;
    launch(static_cast<const Host*>(dv), dev.template as<Dev>(), seq + 1);
    ctx->launches++;
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
      persist_release(ctx->device);
      set_error("persistent kernel launch failed: %s", cudaGetErrorString(e));
      return LGS_ERR_CUDA;
    }
    active = true;
    device = ctx->device;
    return LGS_OK;
  }

  void send(const Cmd& c) { persist_send<kWords>(host, ++seq, &c); }

  void close() {
    if (!active) return;
    send(quit);
    active = false;
    persist_release(device);
  }

  // After a failed mailbox wait inside the session (the grid gave up, or the stream failed): closes the session, drains
  // the stream and re-arms the last-CTA counter the grid may have left mid-evaluation.  Returns whether plain launches can
  // go on; the session is then broken for good.
  bool recover(lgs_ctx* ctx, unsigned* counter) {
    close();
    if (cudaStreamSynchronize(ctx->stream) != cudaSuccess || cudaGetLastError() != cudaSuccess) return false;
    if (cudaMemsetAsync(counter, 0, sizeof(unsigned), ctx->stream) != cudaSuccess) return false;
    broken = true;
    return true;
  }

  // *_destroy: closes the session, drains the stream and frees the command buffers
  void release(lgs_ctx* ctx) {
    close();
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (host) cudaFreeHost(host);
    host = nullptr;
    dev.release();
  }
};

// Enables a session for one align; every exit path closes it.
template <typename Cmd>
struct SessionScope {
  ResidentSession<Cmd>& s;
  explicit SessionScope(ResidentSession<Cmd>& session) : s(session) { s.enabled = true; }
  ~SessionScope() {
    s.close();
    s.enabled = false;
  }
};

#ifdef __CUDACC__
__device__ __forceinline__ void ld_volatile_chunk(const CmdChunk* p, unsigned long long& data, unsigned long long& seq) {
  asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(data), "=l"(seq) : "l"(p) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_gpu_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

constexpr long long kCommandTimeoutCycles = 1000000000ll;  // ~0.5 s at 1.9 GHz

// Called by every thread of every CTA of the resident grid (NT threads per CTA, NT >= WORDS).  Returns false when the
// grid has to give up; otherwise command `seq` is in dst (shared memory, WORDS 64-bit words) and the CTA is synchronised.
template <int WORDS, int NT>
__device__ __forceinline__ bool persist_receive(const CmdHost<WORDS>* __restrict__ cmd_host, CmdDev<WORDS>* __restrict__ cmd_dev, unsigned long long seq,
                                                unsigned long long* dst, int* give_up) {
  static_assert(WORDS <= 128 && WORDS <= NT, "a command is at most four 16-byte chunks per lane of one warp");
  constexpr int kPerLane = (WORDS + 31) / 32;
  if (blockIdx.x == 0 && threadIdx.x < 32) {  // relay: host memory -> device memory
    const int lane = threadIdx.x;
    unsigned long long d[kPerLane], sq[kPerLane];
    const long long t0 = clock64();
    bool ok = true;
    while (true) {
      bool all = true;
#pragma unroll
      for (int c = 0; c < kPerLane; c++) {  // all loads of the round are in flight together: one PCIe latency per poll
        d[c] = 0;
        sq[c] = seq;
        if (lane + 32 * c < WORDS) ld_volatile_chunk(cmd_host->c + lane + 32 * c, d[c], sq[c]);
      }
#pragma unroll
      for (int c = 0; c < kPerLane; c++) all = all && sq[c] == seq;
      if (__all_sync(0xffffffffu, all)) break;
      if (clock64() - t0 > kCommandTimeoutCycles) ok = false;  // every lane reads the clock; any of them ends the wait for all
      ok = __all_sync(0xffffffffu, ok);
      if (!ok) break;
    }
    if (ok) {
#pragma unroll
      for (int c = 0; c < kPerLane; c++)
        if (lane + 32 * c < WORDS) cmd_dev->data[lane + 32 * c] = d[c];
      __threadfence();
      __syncwarp();
      if (lane == 0) st_release_gpu_u64(&cmd_dev->seq, seq);
    }
  }
  if (threadIdx.x == 0) {
    const long long t0 = clock64();
    while (ld_acquire_gpu_u64(&cmd_dev->seq) != seq)
      if (clock64() - t0 > kCommandTimeoutCycles + 100000000ll) {
        *give_up = 1;
        break;
      }
  }
  __syncthreads();
  if (*give_up) return false;
  if (threadIdx.x < WORDS) dst[threadIdx.x] = __ldcg(cmd_dev->data + threadIdx.x);
  __syncthreads();
  return true;
}
#endif

}  // namespace lgs
