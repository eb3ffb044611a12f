// Context, error reporting, cloud upload (host AoS records -> packed float4 xyzi in HBM) and the aligned output cloud.
#include <atomic>

#include <cstdlib>
#include <sched.h>

#include "persist.cuh"

namespace lgs {

static thread_local std::string g_last_error;

void set_error(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
}

// One thread per point: gather x,y,z (+ intensity) from the strided record.  Reads are 4-byte but
// consecutive lanes touch consecutive records, so every 32 B sector fetched is used for 32 B-stride
// PointXYZI up to its padding; the store is a coalesced float4.
__global__ void repack_kernel(const unsigned char* __restrict__ raw, int64_t n, int stride, int ioff, float4* __restrict__ out) {
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= n) return;
  const float* r = reinterpret_cast<const float*>(raw + i * stride);
  float4 v;
  v.x = r[0];
  v.y = r[1];
  v.z = r[2];
  v.w = ioff >= 0 ? *reinterpret_cast<const float*>(raw + i * stride + ioff) : 0.0f;
  out[i] = v;
}

int upload_cloud(lgs_ctx* ctx, const void* pts, int64_t n, int32_t stride, DevBuf* dst) {
  LGS_REQUIRE(n >= 0, "negative point count");
  LGS_REQUIRE(stride >= 12 && stride % 4 == 0, "stride_bytes must be a multiple of 4 and >= 12");
  LGS_REQUIRE(n == 0 || pts != nullptr, "null cloud");
  LGS_TRY(dst->reserve(static_cast<size_t>(n > 0 ? n : 1) * 16));
  if (n == 0) return LGS_OK;
  if (stride == 16) {
    LGS_CUDA(cudaMemcpyAsync(dst->p, pts, static_cast<size_t>(n) * 16, cudaMemcpyHostToDevice, ctx->stream));
    return LGS_OK;
  }
  LGS_TRY(ctx->raw.reserve(static_cast<size_t>(n) * stride));
  LGS_CUDA(cudaMemcpyAsync(ctx->raw.p, pts, static_cast<size_t>(n) * stride, cudaMemcpyHostToDevice, ctx->stream));
  return repack_cloud(ctx, ctx->raw.p, n, stride, dst->as<float4>());
}

int repack_cloud(lgs_ctx* ctx, const void* raw_dev, int64_t n, int32_t stride, float4* dst) {
  if (n == 0) return LGS_OK;
  int ioff = stride >= 20 ? 16 : -1;
  repack_kernel<<<grid_for(n, 256), 256, 0, ctx->stream>>>(static_cast<const unsigned char*>(raw_dev), n, stride, ioff, dst);
  ctx->launches++;
  LGS_CUDA(cudaGetLastError());
  return LGS_OK;
}

int load_cloud(lgs_ctx* ctx, const void* pts, int64_t n, int32_t stride_bytes, bool on_device, DevBuf* dst) {
  LGS_TRY(use_device(ctx));
  if (!on_device) return upload_cloud(ctx, pts, n, stride_bytes, dst);
  LGS_REQUIRE(n >= 0, "negative point count");
  LGS_REQUIRE(n == 0 || pts != nullptr, "null cloud");
  LGS_TRY(dst->reserve(static_cast<size_t>(n > 0 ? n : 1) * 16));
  if (n) LGS_CUDA(cudaMemcpyAsync(dst->p, pts, static_cast<size_t>(n) * 16, cudaMemcpyDeviceToDevice, ctx->stream));
  return LGS_OK;
}

struct Mat4f {  // a transform passed by value (64 bytes of kernel parameters), column-major
  float m[16];
};

__global__ void __launch_bounds__(256) transform_cloud_kernel(const float4* __restrict__ src, int64_t n, Mat4f T, float4* __restrict__ dst) {
  const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= n) return;
  const float4 p = src[i];
  const float3 t = transform_pcl(T.m, p.x, p.y, p.z);
  dst[i] = make_float4(t.x, t.y, t.z, p.w);
}

int transform_cloud(lgs_ctx* ctx, const float4* src, int64_t n, const float* T, float4* dst) {
  if (n == 0) return LGS_OK;
  Mat4f m;
  memcpy(m.m, T, sizeof(m.m));
  transform_cloud_kernel<<<grid_for(n, 256), 256, 0, ctx->stream>>>(src, n, m, dst);
  ctx->launches++;
  LGS_CUDA(cudaGetLastError());
  return LGS_OK;
}

int write_aligned_cloud(lgs_ctx* ctx, const float4* src, int64_t n, const float* T, DevBuf* scratch, float* out_host) {
  if (n == 0) return LGS_OK;
  LGS_TRY(scratch->reserve(static_cast<size_t>(n) * 16));
  LGS_TRY(transform_cloud(ctx, src, n, T, scratch->as<float4>()));
  LGS_CUDA(cudaMemcpyAsync(out_host, scratch->p, static_cast<size_t>(n) * 16, cudaMemcpyDeviceToHost, ctx->stream));
  LGS_CUDA(cudaStreamSynchronize(ctx->stream));
  return LGS_OK;
}

// ---- persistent evaluators (persist.cuh) ----------------------------------------------------------------------------
static std::atomic<int> g_persist_owner[64];

// The resident grids are sized for the B200's 148 SMs (kNumSMs) and need every CTA co-resident: on a device, MIG slice or MPS
// share with fewer SMs the CTAs that do not fit would never start while the resident ones spin.  Checked once per device.
static bool device_holds_resident_grids(int device) {
  static int sms[64] = {};
  if (sms[device] == 0) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) v = -1;
    sms[device] = v > 0 ? v : -1;
  }
  return sms[device] >= kNumSMs;
}

bool persist_try_acquire(int device) {
  if (device < 0 || device >= 64) return false;
  if (!device_holds_resident_grids(device)) return false;
  int expected = 0;
  return g_persist_owner[device].compare_exchange_strong(expected, 1, std::memory_order_acquire);
}
void persist_release(int device) {
  if (device >= 0 && device < 64) g_persist_owner[device].store(0, std::memory_order_release);
}

// LGS_NDT_PERSISTENT=0 turns the resident grids off, =1 forces them on.  By default they are off under an injected
// CUDA tool (Nsight Compute serialises kernels and blocks the host inside the launch call until the kernel has
// finished - a grid that waits for a host command would only end by its time-out).
bool persist_env_enabled() {
  static const bool on = [] {
    const char* e = getenv("LGS_NDT_PERSISTENT");
    if (e && e[0] == '0') return false;
    if (e && e[0] == '1') return true;
    for (const char* v : {"CUDA_INJECTION64_PATH", "NV_COMPUTE_PROFILER_PERFWORKS_DIR", "NV_NSIGHT_INJECTION_TRANSPORT_TYPE"})
      if (getenv(v)) return false;
    return true;
  }();
  return on;
}

int mailbox_next(lgs_ctx* ctx, Mailbox* mb) {
  if (!ctx->mbox) {
    void* p = nullptr;
    LGS_CUDA(cudaHostAlloc(&p, sizeof(MailboxHost), cudaHostAllocMapped | cudaHostAllocPortable));
    memset(p, 0, sizeof(MailboxHost));
    ctx->mbox = static_cast<MailboxHost*>(p);
  }
  void* dv = nullptr;
  LGS_CUDA(cudaHostGetDevicePointer(&dv, ctx->mbox, 0));
  mb->r = static_cast<MailboxHost*>(dv)->r;
  mb->token = ++ctx->mbox_token;
  return LGS_OK;
}

int mailbox_wait(lgs_ctx* ctx, const Mailbox& mb, int k, double* out) {
  const volatile MailboxRecord* r = ctx->mbox->r;
  unsigned spins = 0;
  for (int i = 0; i < k; i++) {
    while (r[i].token != mb.token) {
#if defined(__x86_64__) || defined(__i386__)
      __builtin_ia32_pause();
#endif
      if (ctx->polite_wait && (spins & 0x3fu) == 0x3fu) sched_yield();
      if ((++spins & 0x3fffu) == 0) {
        // a failed or finished-without-publishing launch must not hang the caller
        cudaError_t e = cudaStreamQuery(ctx->stream);
        if (e == cudaErrorNotReady) continue;
        if (e != cudaSuccess) {
          set_error("kernel failed while waiting for its result: %s", cudaGetErrorString(e));
          return LGS_ERR_CUDA;
        }
        if (r[i].token != mb.token) {
          set_error("stream drained but the result mailbox was not written (token %llu, record %d)", mb.token, i);
          return LGS_ERR_CUDA;
        }
      }
    }
    std::atomic_thread_fence(std::memory_order_acquire);  // token before value
    out[i] = r[i].v;
  }
  return LGS_OK;
}

}  // namespace lgs

extern "C" {

const char* lgs_last_error(void) { return lgs::g_last_error.c_str(); }
const char* lgs_version(void) { return "lgs_b200 0.1 (sm_100a)"; }

int lgs_ctx_create(int device, void* cuda_stream, lgs_ctx** out) {
  if (!out) {
    lgs::set_error("lgs_ctx_create: null out");
    return LGS_ERR_INVALID;
  }
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    lgs::set_error("no CUDA device available (%s); this library has no CPU fallback", cudaGetErrorString(e));
    return LGS_ERR_CUDA;
  }
  LGS_REQUIRE(device >= 0 && device < count, "device index out of range");
  LGS_CUDA(cudaSetDevice(device));
  lgs_ctx* c = new lgs_ctx;
  c->device = device;
  if (cuda_stream) {
    c->stream = static_cast<cudaStream_t>(cuda_stream);
    c->own_stream = false;
  } else {
    e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
      lgs::set_error("cudaStreamCreate failed: %s", cudaGetErrorString(e));
      delete c;
      return LGS_ERR_CUDA;
    }
    c->own_stream = true;
  }
  *out = c;
  return LGS_OK;
}

void lgs_ctx_destroy(lgs_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  c->raw.release();
  for (auto& b : c->tmp) b.release();
  c->sort_tmp.release();
  c->pin.release();
  c->pin_up.release();
  c->vg_in.release();
  c->vg_out.release();
  c->vg_vidx.release();
  c->vg_rank.release();
  c->ndt_many.release();
  if (c->mbox) cudaFreeHost(c->mbox);
  if (c->own_stream) cudaStreamDestroy(c->stream);
  delete c;
}

int lgs_ctx_synchronize(lgs_ctx* c) {
  LGS_REQUIRE(c, "null ctx");
  LGS_CUDA(cudaStreamSynchronize(c->stream));
  return LGS_OK;
}

int64_t lgs_ctx_launch_count(const lgs_ctx* c) { return c ? c->launches : 0; }

}  // extern "C"
