// lgs_linalg_batch: the small dense solvers of math.cuh / ndt_opt.cuh run one problem per GPU thread, so that their
// device results can be compared bit for bit with the oracle's Eigen restatement and with the host-compiled header.
// The kernels that use these routines inline them; this translation unit only adds its own kernel.
#include "common.cuh"
#include "math.cuh"
#include "ndt_opt.cuh"

namespace lgs {
namespace {

constexpr int kLinalgBlock = 128;

__host__ __device__ constexpr int linalg_in(int op) { return LGS_LINALG_IN(op); }
__host__ __device__ constexpr int linalg_out(int op) { return LGS_LINALG_OUT(op); }

__global__ void __launch_bounds__(kLinalgBlock) linalg_batch_kernel(int op, long long n, const double* __restrict__ in, double* __restrict__ out) {
  const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const double* a = in + t * linalg_in(op);
  double* o = out + t * linalg_out(op);
  double A[42];
  for (int i = 0; i < linalg_in(op); i++) A[i] = a[i];
  switch (op) {
    case LGS_LINALG_SVD3: {
      double U[9], S[3], V[9];
      m::svd_jacobi<3, double>(A, U, S, V);
      for (int i = 0; i < 9; i++) o[i] = U[i];
      for (int i = 0; i < 3; i++) o[9 + i] = S[i];
      for (int i = 0; i < 9; i++) o[12 + i] = V[i];
      break;
    }
    case LGS_LINALG_EIG3: {
      double w[3], Q[9];
      const bool ok = m::eig_sym3(A, w, Q);
      for (int i = 0; i < 3; i++) o[i] = w[i];
      for (int i = 0; i < 9; i++) o[3 + i] = Q[i];
      o[12] = ok ? 1.0 : 0.0;
      break;
    }
    case LGS_LINALG_INV3: {
      double R[9];
      m::inv3(A, R);
      for (int i = 0; i < 9; i++) o[i] = R[i];
      break;
    }
    case LGS_LINALG_SVD_SOLVE6: {
      double x[6];
      m::svd_solve<6>(A, A + 36, x);
      for (int i = 0; i < 6; i++) o[i] = x[i];
      break;
    }
    case LGS_LINALG_SCHUR6: {
      double x[6] = {0, 0, 0, 0, 0, 0};
      const bool ok = ndtopt::schur_solve6(A, A + 36, x);
      for (int i = 0; i < 6; i++) o[i] = x[i];
      o[6] = ok ? 1.0 : 0.0;
      break;
    }
    default: {  // LGS_LINALG_NEWTON6: Machine::solve on g = -b, with and without the exact Newton step
      ndtopt::Machine mc;
      for (int i = 0; i < 36; i++) mc.H[i] = A[i];
      for (int i = 0; i < 6; i++) mc.g[i] = -A[36 + i];
      for (int e = 0; e < 2; e++) {
        mc.exact_solve = e;
        mc.solve();
        for (int i = 0; i < 6; i++) o[6 * e + i] = mc.delta_p[i];
      }
      break;
    }
  }
}

}  // namespace
}  // namespace lgs

extern "C" int lgs_linalg_batch(lgs_ctx* ctx, int32_t op, int64_t n, const double* in, double* out) {
  using namespace lgs;
  LGS_REQUIRE(ctx, "null context");
  LGS_REQUIRE(op >= LGS_LINALG_SVD3 && op <= LGS_LINALG_NEWTON6, "unknown op");
  LGS_REQUIRE(n >= 0, "n must be >= 0");
  LGS_REQUIRE(n == 0 || (in && out), "null argument");
  if (n == 0) return LGS_OK;
  LGS_TRY(use_device(ctx));
  const size_t in_bytes = static_cast<size_t>(n) * linalg_in(op) * sizeof(double);
  const size_t out_bytes = static_cast<size_t>(n) * linalg_out(op) * sizeof(double);
  DevBuf din, dout;
  int rc = LGS_OK;
  do {
    if ((rc = din.reserve(in_bytes)) != LGS_OK) break;
    if ((rc = dout.reserve(out_bytes)) != LGS_OK) break;
    cudaMemcpyAsync(din.p, in, in_bytes, cudaMemcpyHostToDevice, ctx->stream);
    linalg_batch_kernel<<<grid_for(n, kLinalgBlock), kLinalgBlock, 0, ctx->stream>>>(op, n, din.as<double>(), dout.as<double>());
    ctx->launches++;
    if (cudaGetLastError() != cudaSuccess) {
      set_error("lgs_linalg_batch: launch failed");
      rc = LGS_ERR_CUDA;
      break;
    }
    cudaMemcpyAsync(out, dout.p, out_bytes, cudaMemcpyDeviceToHost, ctx->stream);
    if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) {
      set_error("lgs_linalg_batch: stream synchronize failed");
      rc = LGS_ERR_CUDA;
    }
  } while (false);
  din.release();
  dout.release();
  return rc;
}
