// PCL-style GICP: pclomp::GeneralizedIterativeClosestPoint behind pcl::Registration
// (GO = thirdparty/ndt_omp/include/pclomp/gicp_omp_impl.hpp, GO.h = .../gicp_omp.h; call sites LSM:73-96, GBS:120-141).
//
//   covariances     -> computeCovariances (GO:48-122): exact k-NN through the implicit BVH, f64 moments of the f32
//                      neighbours, 3x3 Jacobi SVD, singular values replaced by (1, 1, gicp_epsilon); one thread per point.
//   correspondences -> the body of the outer loop (GO:404-474): q = transformation_ * output[i] in f32, exact 1-NN in the
//                      target (one warp per point), distance gate, then M_i = (R C1 R^T + C2)^-1 in f64 stored as f32
//                      (one thread per point) and the number of correspondences.  The reference's sorted index lists
//                      (GO:458-474) are the ascending valid entries of corr[]: nothing is compacted, every functor
//                      kernel walks corr[] and skips the holes.
//   functor kernels -> OptimizationFunctorWithIndices::operator() / df / fdf (GO:245-367): streaming passes over
//                      (output[i], target[corr[i]], M_i) with 1 / 12 / 13 sums.  The sums are EXACT (128-bit fixed point,
//                      fixsum.cuh), hence independent of the reduction order: the line search compares costs that differ
//                      by less than the rounding noise of an f64 sum, and only exact sums make its path reproducible.
//                      Result published to the host mailbox (no D2H copy, no stream synchronisation).
//   BFGS + outer loop-> host (GO:180-242, 370-516; pcl/registration/bfgs.h restated: Fletcher line search of GSL's
//                      vector_bfgs2).  About 40 functor evaluations per outer iteration, each one kernel + one mailbox
//                      round trip.
#include <algorithm>
#include <cmath>
#include <limits>
#include <memory>

#include "fixsum.cuh"
#include "gicp.cuh"
#include "persist.cuh"

namespace lgs {

constexpr int kFunBlock = 128;
constexpr int kCovsPcl = 100;  // GicpCloud::covs_reg tag of the (1, 1, gicp_epsilon) covariances

__global__ void __launch_bounds__(128) pgicp_covariance_kernel(const float4* __restrict__ pts, int n, int k, double gicp_epsilon,
                                                              const int* __restrict__ knn_idx, double* __restrict__ covs) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int* nb = knn_idx + static_cast<size_t>(i) * k;
  double m0 = 0, m1 = 0, m2 = 0, c00 = 0, c10 = 0, c11 = 0, c20 = 0, c21 = 0, c22 = 0;
  for (int j = 0; j < k; j++) {
    const float4 p = __ldg(pts + nb[j]);
    m0 += static_cast<double>(p.x);
    m1 += static_cast<double>(p.y);
    m2 += static_cast<double>(p.z);
    c00 += static_cast<double>(__fmul_rn(p.x, p.x));  // f32 products widened at the += (GO:89-97)
    c10 += static_cast<double>(__fmul_rn(p.y, p.x));
    c11 += static_cast<double>(__fmul_rn(p.y, p.y));
    c20 += static_cast<double>(__fmul_rn(p.z, p.x));
    c21 += static_cast<double>(__fmul_rn(p.z, p.y));
    c22 += static_cast<double>(__fmul_rn(p.z, p.z));
  }
  const double kd = static_cast<double>(k);
  m0 /= kd;
  m1 /= kd;
  m2 /= kd;
  double cov[9];
  cov[0] = c00 / kd - m0 * m0;
  cov[3] = cov[1] = c10 / kd - m1 * m0;
  cov[4] = c11 / kd - m1 * m1;
  cov[6] = cov[2] = c20 / kd - m2 * m0;
  cov[7] = cov[5] = c21 / kd - m2 * m1;
  cov[8] = c22 / kd - m2 * m2;
  double U[9], S[3], V[9], out[9];
  m::svd_jacobi<3, double>(cov, U, S, V);
  for (int t = 0; t < 9; t++) out[t] = 0.0;
  for (int kk = 0; kk < 3; kk++) {
    const double v = kk == 2 ? gicp_epsilon : 1.0;
    for (int a = 0; a < 3; a++)
      for (int b = 0; b < 3; b++) out[a * 3 + b] += (v * U[a * 3 + kk]) * U[b * 3 + kk];
  }
  for (int t = 0; t < 9; t++) covs[static_cast<size_t>(i) * 9 + t] = out[t];
}

struct PgicpParams {
  float T[16];   // column-major: transformation_ (correspondences) or base_transformation_ with the state applied (functor)
  double R[9];   // rotation of transformation_ * guess, row-major (GO:411-417)
  double thr2;   // corr_dist_threshold_^2
};

// Matrix4f * (x, y, z, 1): ((c0 x + c1 y) + c2 z) + c3
__device__ __forceinline__ void mul4f_point(const float* __restrict__ T, const float4& p, float& x, float& y, float& z) {
  x = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(T[0], p.x), __fmul_rn(T[4], p.y)), __fmul_rn(T[8], p.z)), T[12]);
  y = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(T[1], p.x), __fmul_rn(T[5], p.y)), __fmul_rn(T[9], p.z)), T[13]);
  z = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(T[2], p.x), __fmul_rn(T[6], p.y)), __fmul_rn(T[10], p.z)), T[14]);
}

constexpr int kPCorrBlock = 256;
__global__ void __launch_bounds__(kPCorrBlock) pgicp_correspondence_kernel(NNView tv, const float4* __restrict__ out_cloud, int n, PgicpParams P,
                                                                          int* __restrict__ corr) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i = blockIdx.x * (kPCorrBlock / 32) + warp; i < n; i += gridDim.x * (kPCorrBlock / 32)) {
    const float4 a = __ldg(out_cloud + i);
    float qx, qy, qz;
    mul4f_point(P.T, a, qx, qy, qz);
    float d2;
    int id;
    nn_search1_warp(tv, qx, qy, qz, lane, d2, id);
    if (lane == 0) corr[i] = (static_cast<double>(d2) < P.thr2) ? id : -1;  // GO:436
  }
}

// Reduction of K per-thread exact sums (fixsum.cuh): warp shuffles, CTA, per-CTA partials, last CTA adds them and
// publishes the K doubles.  Integer addition: the result does not depend on the order of any of these steps.
template <int K>
__device__ __forceinline__ void fun_reduce_and_publish(Fix128 (&acc)[K], Fix128* __restrict__ partials, unsigned* __restrict__ counter,
                                                      const Mailbox& mb) {
  __shared__ Fix128 sm[kFunBlock / 32][K];
  __shared__ bool is_last;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < K; k++) {
    Fix128 v = acc[k];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      Fix128 o;
      o.lo = __shfl_xor_sync(0xffffffffu, v.lo, off);
      o.hi = __shfl_xor_sync(0xffffffffu, v.hi, off);
      fix_add(v, o);
    }
    if (lane == 0) sm[warp][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < K) {
    Fix128 v = sm[0][threadIdx.x];
#pragma unroll
    for (int w = 1; w < kFunBlock / 32; w++) fix_add(v, sm[w][threadIdx.x]);
    partials[static_cast<size_t>(blockIdx.x) * K + threadIdx.x] = v;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) is_last = atomicAdd(counter, 1u) == gridDim.x - 1;
  __syncthreads();
  if (is_last) {
    // integer sums: any order gives the same bits, so the per-CTA rows are added by eight groups of threads in parallel
    __threadfence();
    __shared__ Fix128 fin[kFunBlock / 16][16];
    static_assert(K <= 16, "one 16-thread group per slice of the rows");
    const int kk = threadIdx.x & 15, part = threadIdx.x >> 4;
    Fix128 v = fix_zero();
    if (kk < K) {
#pragma unroll 4
      for (unsigned b = part; b < gridDim.x; b += kFunBlock / 16) {
        const ulonglong2 t = __ldcg(reinterpret_cast<const ulonglong2*>(partials + static_cast<size_t>(b) * K + kk));
        Fix128 u;
        u.lo = t.x;
        u.hi = static_cast<long long>(t.y);
        fix_add(v, u);
      }
    }
    fin[part][kk] = v;
    __syncthreads();
    v = fix_zero();
    if (threadIdx.x < K) {
#pragma unroll
      for (int p = 0; p < kFunBlock / 16; p++) fix_add(v, fin[p][threadIdx.x]);
    }
    if (threadIdx.x == 0) *counter = 0;
    mailbox_publish<K>(mb, fix_value(v));
  }
}

// M_i = (R C1 R^T + C2)^-1, cast to f32 (GO:439-452); publishes the number of correspondences
__global__ void __launch_bounds__(kFunBlock) pgicp_mahalanobis_kernel(int n, PgicpParams P, const double* __restrict__ cov_src,
                                                                     const double* __restrict__ cov_tgt, const int* __restrict__ corr,
                                                                     float* __restrict__ mahal, Fix128* __restrict__ partials,
                                                                     unsigned* __restrict__ counter, const Mailbox mb) {
  Fix128 acc[1] = {fix_zero()};
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int c = corr[i];
    if (c < 0) continue;
    double C1[9], C2[9], M[9], Rt[9], temp[9], inv[9];
#pragma unroll
    for (int t = 0; t < 9; t++) {
      C1[t] = cov_src[static_cast<size_t>(i) * 9 + t];
      C2[t] = cov_tgt[static_cast<size_t>(c) * 9 + t];
    }
    m::mul3(P.R, C1, M);
#pragma unroll
    for (int a = 0; a < 3; a++)
#pragma unroll
      for (int b = 0; b < 3; b++) Rt[a * 3 + b] = P.R[b * 3 + a];
    m::mul3(M, Rt, temp);
#pragma unroll
    for (int t = 0; t < 9; t++) temp[t] += C2[t];
    m::inv3(temp, inv);
#pragma unroll
    for (int t = 0; t < 9; t++) mahal[static_cast<size_t>(i) * 9 + t] = static_cast<float>(inv[t]);
    fix_add(acc[0], 1.0);
  }
  fun_reduce_and_publish<1>(acc, partials, counter, mb);
}

// MODE 0: operator() (f32 arithmetic, GO:245-275)   sums: f
// MODE 1: df  (GO:278-330)                          sums: g_t[3], R[9]
// MODE 2: fdf (GO:333-367)                          sums: f, g_t[3], R[9]
// base_transformation_ is the identity (GO:394), so base_transformation_ * p_src is p_src itself.
template <int MODE>
__device__ __forceinline__ void pgicp_functor_body(const float4* __restrict__ out_cloud, const float4* __restrict__ tgt, int n, const float* __restrict__ T,
                                                   const int* __restrict__ corr, const float* __restrict__ mahal, Fix128* __restrict__ partials,
                                                   unsigned* __restrict__ counter, const Mailbox& mb) {
  constexpr int K = MODE == 0 ? 1 : (MODE == 1 ? 12 : 13);
  Fix128 acc[K];
#pragma unroll
  for (int k = 0; k < K; k++) acc[k] = fix_zero();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int c = corr[i];
    if (c < 0) continue;
    const float4 a = out_cloud[i];
    const float4 b = __ldg(tgt + c);
    float M[9];
#pragma unroll
    for (int t = 0; t < 9; t++) M[t] = mahal[static_cast<size_t>(i) * 9 + t];
    float px, py, pz;
    mul4f_point(T, a, px, py, pz);
    const float r0 = __fsub_rn(px, b.x), r1 = __fsub_rn(py, b.y), r2 = __fsub_rn(pz, b.z);
    if (MODE == 0) {
      const float t0 = __fadd_rn(__fadd_rn(__fmul_rn(M[0], r0), __fmul_rn(M[1], r1)), __fmul_rn(M[2], r2));
      const float t1 = __fadd_rn(__fadd_rn(__fmul_rn(M[3], r0), __fmul_rn(M[4], r1)), __fmul_rn(M[5], r2));
      const float t2 = __fadd_rn(__fadd_rn(__fmul_rn(M[6], r0), __fmul_rn(M[7], r1)), __fmul_rn(M[8], r2));
      // 4-lane SSE dot product, lane 3 is zero: (r0 t0 + r2 t2) + (r1 t1 + 0)
      fix_add(acc[0], static_cast<double>(__fadd_rn(__fadd_rn(__fmul_rn(r0, t0), __fmul_rn(r2, t2)), __fmul_rn(r1, t1))));
    } else {
      const double res[3] = {static_cast<double>(r0), static_cast<double>(r1), static_cast<double>(r2)};
      double temp[3];
#pragma unroll
      for (int r = 0; r < 3; r++)
        temp[r] = __dadd_rn(__dadd_rn(__dmul_rn(static_cast<double>(M[r * 3]), res[0]), __dmul_rn(static_cast<double>(M[r * 3 + 1]), res[1])),
                            __dmul_rn(static_cast<double>(M[r * 3 + 2]), res[2]));
      constexpr int o = MODE == 2 ? 1 : 0;
      if (MODE == 2) fix_add(acc[0], __dadd_rn(__dadd_rn(__dmul_rn(res[0], temp[0]), __dmul_rn(res[1], temp[1])), __dmul_rn(res[2], temp[2])));
      const double ps[3] = {static_cast<double>(a.x), static_cast<double>(a.y), static_cast<double>(a.z)};
#pragma unroll
      for (int r = 0; r < 3; r++) fix_add(acc[o + r], temp[r]);
#pragma unroll
      for (int r = 0; r < 3; r++)
#pragma unroll
        for (int cc = 0; cc < 3; cc++) fix_add(acc[o + 3 + r * 3 + cc], __dmul_rn(ps[r], temp[cc]));
    }
  }
  fun_reduce_and_publish<K>(acc, partials, counter, mb);
}

template <int MODE>
__global__ void __launch_bounds__(kFunBlock) pgicp_functor_kernel(const float4* __restrict__ out_cloud, const float4* __restrict__ tgt, int n,
                                                                 const __grid_constant__ PgicpParams P, const int* __restrict__ corr,
                                                                 const float* __restrict__ mahal, Fix128* __restrict__ partials,
                                                                 unsigned* __restrict__ counter, const __grid_constant__ Mailbox mb) {
  pgicp_functor_body<MODE>(out_cloud, tgt, n, P.T, corr, mahal, partials, counter, mb);
}

// Persistent functor evaluator: BFGS asks for ~50 cost / gradient evaluations per outer iteration and needs each answer
// before it can choose the next step, so the grid stays resident between update_correspondences calls and receives
// {T, mode, mailbox token} per evaluation through the command channel of persist.cuh (one launch + ~13 us of launch
// latency per evaluation otherwise, for ~10 us of work on a 30 000-point cloud).
struct PgicpPose {
  float T[16];
  int mode;  // 0: operator(), 1: df, 2: fdf, < 0: end of the run
  int pad;
  unsigned long long token;
};
using PgicpSession = ResidentSession<PgicpPose>;
constexpr int kPgWords = PgicpSession::kWords;
constexpr int kFunResident = 4;  // CTAs of the persistent grid per SM (all of them must be co-resident)

__global__ void __launch_bounds__(kFunBlock, kFunResident) pgicp_persistent_kernel(const float4* __restrict__ out_cloud, const float4* __restrict__ tgt, int n,
                                                                                  const int* __restrict__ corr, const float* __restrict__ mahal,
                                                                                  Fix128* __restrict__ partials, unsigned* __restrict__ counter,
                                                                                  MailboxRecord* mailbox, const PgicpSession::Host* __restrict__ cmd_host,
                                                                                  PgicpSession::Dev* __restrict__ cmd_dev, unsigned long long first_seq) {
  __shared__ __align__(16) PgicpPose pose;
  __shared__ int give_up;
  if (threadIdx.x == 0) give_up = 0;
  __syncthreads();
  for (unsigned long long seq = first_seq;; seq++) {
    if (!persist_receive<kPgWords, kFunBlock>(cmd_host, cmd_dev, seq, reinterpret_cast<unsigned long long*>(&pose), &give_up)) return;
    if (pose.mode < 0) return;
    Mailbox mb;
    mb.r = mailbox;
    mb.token = pose.token;
    if (pose.mode == 0)
      pgicp_functor_body<0>(out_cloud, tgt, n, pose.T, corr, mahal, partials, counter, mb);
    else if (pose.mode == 1)
      pgicp_functor_body<1>(out_cloud, tgt, n, pose.T, corr, mahal, partials, counter, mb);
    else
      pgicp_functor_body<2>(out_cloud, tgt, n, pose.T, corr, mahal, partials, counter, mb);
    __syncthreads();
  }
}

}  // namespace lgs

// =============================================================================================
using namespace lgs;

struct lgs_gicp_omp {
  lgs_ctx* ctx = nullptr;
  // GO.h:116-126
  int k = 20;
  double gicp_epsilon = 0.001;
  double rotation_eps = 2e-3, trans_eps = 5e-4;
  int max_inner_iterations = 20;
  int max_iterations = 200;
  double corr_dist_threshold = 5.0;
  std::shared_ptr<GicpCloud> source, target;
  DevBuf output, corr, mahal, partials, state, out_cloud;
  float base_T[16], T[16], prev_T[16], final_T[16], guess[16];
  int n_corr = 0;
  int f_calls = 0, df_calls = 0, fdf_calls = 0, inner_total = 0;
  PgicpSession session{PgicpPose{{}, -1, 0, 0}};  // persistent functor evaluator (between two update_correspondences calls of one align)
};

namespace {

// applyState (GO:518-529): t <- [Rz(x5) Ry(x4) Rx(x3) * t.linear | t.translation + x0..2], the rotation composed through
// f32 quaternions as Eigen's AngleAxisf products do
void apply_state(float* t, const double* x) {
  struct Quat {
    float w, x, y, z;
  };
  const float hz = 0.5f * static_cast<float>(x[5]), hy = 0.5f * static_cast<float>(x[4]), hx = 0.5f * static_cast<float>(x[3]);
  const Quat qz{std::cos(hz), 0.f, 0.f, std::sin(hz)}, qy{std::cos(hy), 0.f, std::sin(hy), 0.f}, qx{std::cos(hx), std::sin(hx), 0.f, 0.f};
  auto mul = [](const Quat& a, const Quat& b) {
    Quat r;
    r.w = a.w * b.w - a.x * b.x - a.y * b.y - a.z * b.z;
    r.x = a.w * b.x + a.x * b.w + a.y * b.z - a.z * b.y;
    r.y = a.w * b.y + a.y * b.w + a.z * b.x - a.x * b.z;
    r.z = a.w * b.z + a.z * b.w + a.x * b.y - a.y * b.x;
    return r;
  };
  const Quat q = mul(mul(qz, qy), qx);
  const float tx = 2 * q.x, ty = 2 * q.y, tz = 2 * q.z;
  const float twx = tx * q.w, twy = ty * q.w, twz = tz * q.w, txx = tx * q.x, txy = ty * q.x, txz = tz * q.x, tyy = ty * q.y, tyz = tz * q.y, tzz = tz * q.z;
  const float R[9] = {1 - (tyy + tzz), txy - twz, txz + twy, txy + twz, 1 - (txx + tzz), tyz - twx, txz - twy, tyz + twx, 1 - (txx + tyy)};
  float L[9];
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) L[r * 3 + c] = (R[r * 3] * t[c * 4] + R[r * 3 + 1] * t[c * 4 + 1]) + R[r * 3 + 2] * t[c * 4 + 2];
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) t[c * 4 + r] = L[r * 3 + c];
  t[12] += static_cast<float>(x[0]);
  t[13] += static_cast<float>(x[1]);
  t[14] += static_cast<float>(x[2]);
}

// computeRDerivative (GO:125-178): g[3..5] = <dR/dphi, R>, <dR/dtheta, R>, <dR/dpsi, R> (matricesInnerProd, GO.h:314-324)
void r_derivative(const double* x, const double* R, double* g) {
  const double cphi = std::cos(x[3]), sphi = std::sin(x[3]), cth = std::cos(x[4]), sth = std::sin(x[4]), cpsi = std::cos(x[5]), spsi = std::sin(x[5]);
  // row-major 3x3 each
  const double dPhi[9] = {0, sphi * spsi + cphi * cpsi * sth, cphi * spsi - cpsi * sphi * sth,
                          0, -cpsi * sphi + cphi * spsi * sth, -cphi * cpsi - sphi * spsi * sth,
                          0, cphi * cth, -cth * sphi};
  const double dTh[9] = {-cpsi * sth, cpsi * cth * sphi, cphi * cpsi * cth,
                         -spsi * sth, cth * sphi * spsi, cphi * cth * spsi,
                         -cth, -sphi * sth, -cphi * sth};
  const double dPsi[9] = {-cth * spsi, -cphi * cpsi - sphi * spsi * sth, cpsi * sphi - cphi * spsi * sth,
                          cpsi * cth, -cphi * spsi + cpsi * sphi * sth, sphi * spsi + cphi * cpsi * sth,
                          0, 0, 0};
  const double* D[3] = {dPhi, dTh, dPsi};
  for (int d = 0; d < 3; d++) {
    double r = 0;
    for (int i = 0; i < 3; i++)
      for (int j = 0; j < 3; j++) r += D[d][j * 3 + i] * R[i * 3 + j];
    g[3 + d] = r;
  }
}

// one row of partial sums per CTA goes through the last-CTA pass: no more CTAs than SMs (a 30 000-point cloud is 1.6 points per thread)
int fun_grid(int64_t n) { return std::max(1, std::min(grid_for(n, kFunBlock), kNumSMs)); }

// one functor evaluation on the device: mode 0 -> f; 1 -> g; 2 -> f and g
int functor_eval(lgs_gicp_omp* g, const double* x, int mode, double* f, double* grad) {
  lgs_ctx* ctx = g->ctx;
  (mode == 0 ? g->f_calls : mode == 1 ? g->df_calls : g->fdf_calls)++;
  PgicpParams P;
  memcpy(P.T, g->base_T, sizeof(P.T));
  apply_state(P.T, x);
  const int n = static_cast<int>(g->source->n);
  Fix128* partials = g->partials.as<Fix128>();
  unsigned* counter = g->state.as<unsigned>();
  Mailbox mb;
  LGS_TRY(mailbox_next(ctx, &mb));
  const float4* out = g->output.as<float4>();
  const float4* tgt = g->target->pts.as<float4>();
  const int grid = fun_grid(n);
  double h[kMailboxRecords];
  const int K = mode == 0 ? 1 : (mode == 1 ? 12 : 13);
  LGS_TRY(g->session.open(ctx, grid <= kNumSMs * kFunResident, [&](const PgicpSession::Host* host, PgicpSession::Dev* dev, unsigned long long first_seq) {
    pgicp_persistent_kernel<<<grid, kFunBlock, 0, ctx->stream>>>(out, tgt, n, g->corr.as<int>(), g->mahal.as<float>(), partials, counter, mb.r, host, dev,
                                                               first_seq);
  }));
  if (g->session.active) {
    PgicpPose pose;
    memcpy(pose.T, P.T, sizeof(pose.T));
    pose.mode = mode;
    pose.pad = 0;
    pose.token = mb.token;
    g->session.send(pose);
    const int rc = mailbox_wait(ctx, mb, K, h);
    if (rc != LGS_OK) {
      // the grid gave up (command time-out): the functor only reads, so if the stream is healthy this evaluation runs
      // again with a plain launch, and so do the ones after it
      if (!g->session.recover(ctx, counter)) return rc;
      (mode == 0 ? g->f_calls : mode == 1 ? g->df_calls : g->fdf_calls)--;
      return functor_eval(g, x, mode, f, grad);
    }
  } else {
    if (mode == 0)
      pgicp_functor_kernel<0><<<grid, kFunBlock, 0, ctx->stream>>>(out, tgt, n, P, g->corr.as<int>(), g->mahal.as<float>(), partials, counter, mb);
    else if (mode == 1)
      pgicp_functor_kernel<1><<<grid, kFunBlock, 0, ctx->stream>>>(out, tgt, n, P, g->corr.as<int>(), g->mahal.as<float>(), partials, counter, mb);
    else
      pgicp_functor_kernel<2><<<grid, kFunBlock, 0, ctx->stream>>>(out, tgt, n, P, g->corr.as<int>(), g->mahal.as<float>(), partials, counter, mb);
    ctx->launches++;
    LGS_CUDA(cudaGetLastError());
    LGS_TRY(mailbox_wait(ctx, mb, K, h));
  }
  const int m = g->n_corr;
  if (mode != 1) *f = h[0] / static_cast<double>(m);
  if (mode != 0) {
    const double* s = h + (mode == 2 ? 1 : 0);
    const double scale = 2.0 / m;
    double R[9];
    for (int a = 0; a < 6; a++) grad[a] = 0;
    for (int a = 0; a < 3; a++) grad[a] = s[a] * scale;
    for (int t = 0; t < 9; t++) R[t] = s[3 + t] * scale;
    r_derivative(x, R, grad);
  }
  return LGS_OK;
}

// ---- BFGS (pcl/registration/bfgs.h; Fletcher's line search as in GSL's vector_bfgs2) -------------------------
enum { kNegativeGradientEpsilon = -3, kNotStarted = -2, kRunning = -1, kSuccess = 0, kNoProgress = 1, kDeviceError = 100 };

struct Vec6 {
  double v[6];
  double& operator[](int i) { return v[i]; }
  double operator[](int i) const { return v[i]; }
};
double dot(const Vec6& a, const Vec6& b) {
  double s = 0;
  for (int i = 0; i < 6; i++) s += a[i] * b[i];
  return s;
}
double norm(const Vec6& a) { return std::sqrt(dot(a, a)); }

double cubic_at(const double* c, double z) { return c[0] + z * (c[1] + z * (c[2] + z * c[3])); }

int quadratic_roots(double a, double b, double c, double* lo, double* hi) {
  if (a == 0) {
    if (b == 0) return 0;
    *lo = -c / b;
    return 1;
  }
  const double disc = b * b - 4 * a * c;
  if (disc < 0) return 0;
  if (disc == 0) {
    *lo = *hi = -0.5 * b / a;
    return 2;
  }
  if (b == 0) {
    const double r = std::sqrt(-c / a);
    *lo = -r;
    *hi = r;
    return 2;
  }
  const double t = -0.5 * (b + (b > 0 ? 1 : -1) * std::sqrt(disc));
  const double r1 = t / a, r2 = c / t;
  *lo = std::min(r1, r2);
  *hi = std::max(r1, r2);
  return 2;
}

// minimiser of the cubic (order 3, both slopes known) or quadratic interpolant through (a, fa, fpa), (b, fb[, fpb]) over [xmin, xmax]
double interpolate(double a, double fa, double fpa, double b, double fb, double fpb, double xmin, double xmax, int order) {
  double lo = (xmin - a) / (b - a), hi = (xmax - a) / (b - a);
  if (lo > hi) std::swap(lo, hi);
  double y, fbest;
  auto consider = [&](const double* c, double z) {
    const double v = cubic_at(c, z);
    if (v < fbest) {
      y = z;
      fbest = v;
    }
  };
  if (order > 2 && !(fpb != fpb) && fpb != std::numeric_limits<double>::infinity()) {
    fpa *= (b - a);
    fpb *= (b - a);
    const double c[4] = {fa, fpa, 3 * (fb - fa) - 2 * fpa - fpb, fpa + fpb - 2 * (fb - fa)};
    y = lo;
    fbest = cubic_at(c, lo);
    consider(c, hi);
    double z0, z1;
    const int nr = quadratic_roots(3 * c[3], 2 * c[2], c[1], &z0, &z1);
    if (nr >= 1 && z0 > lo && z0 < hi) consider(c, z0);
    if (nr == 2 && z1 > lo && z1 < hi) consider(c, z1);
  } else {
    fpa *= (b - a);
    const double q = fb - fa - fpa;
    const double fl = fa + lo * (fpa + lo * q), fh = fa + hi * (fpa + hi * q);
    const double curv = 2 * q;
    y = lo;
    fbest = fl;
    if (fh < fbest) {
      y = hi;
      fbest = fh;
    }
    if (curv > a) {  // as published in PCL's port (GSL tests curv > 0)
      const double z = -fpa / curv;
      if (z > lo && z < hi) {
        const double v = fa + z * (fpa + z * q);
        if (v < fbest) {
          y = z;
          fbest = v;
        }
      }
    }
  }
  return a + y * (b - a);
}

struct Bfgs {
  lgs_gicp_omp* g;
  int err = LGS_OK;  // first device error seen by a functor call
  // parameters as set at GO:212-217 over the defaults of BFGS::Parameters
  int bracket_iters = 100, section_iters = 100, order = 3;
  double rho = 0.01, sigma = 0.01, tau1 = 9, tau2 = 0.05, tau3 = 0.5, step_size = 1;
  double f = 0, delta_f = 0, fp0 = 0, pnorm = 0, g0norm = 0;
  Vec6 gradient, x0, g0, p, x_alpha, g_alpha;
  double f_alpha = 0, df_alpha = 0;
  double f_key = 0, df_key = 0, x_key = 0, g_key = 0;  // the step the cached value / slope / point / gradient belong to

  void call(const Vec6& x, int mode, double* fo, Vec6* go) {
    if (err != LGS_OK) {
      if (fo) *fo = std::numeric_limits<double>::quiet_NaN();
      return;
    }
    err = functor_eval(g, x.v, mode, fo, go ? go->v : nullptr);
  }
  void move_to(double alpha) {
    if (alpha == x_key) return;
    for (int i = 0; i < 6; i++) x_alpha[i] = x0[i] + alpha * p[i];
    x_key = alpha;
  }
  double value_at(double alpha) {
    if (alpha == f_key) return f_alpha;
    move_to(alpha);
    call(x_alpha, 0, &f_alpha, nullptr);
    f_key = alpha;
    return f_alpha;
  }
  double slope_at(double alpha) {
    if (alpha == df_key) return df_alpha;
    move_to(alpha);
    if (alpha != g_key) {
      call(x_alpha, 1, nullptr, &g_alpha);
      g_key = alpha;
    }
    df_alpha = dot(g_alpha, p);
    df_key = alpha;
    return df_alpha;
  }
  void value_and_slope_at(double alpha, double& fo, double& dfo) {
    if (alpha == f_key && alpha == df_key) {
      fo = f_alpha;
      dfo = df_alpha;
      return;
    }
    if (alpha == f_key || alpha == df_key) {
      fo = value_at(alpha);
      dfo = slope_at(alpha);
      return;
    }
    move_to(alpha);
    call(x_alpha, 2, &f_alpha, &g_alpha);
    f_key = g_key = alpha;
    df_alpha = dot(g_alpha, p);
    df_key = alpha;
    fo = f_alpha;
    dfo = df_alpha;
  }
  void restart_line() {  // the caches describe step 0 of the new direction
    x_alpha = x0;
    x_key = 0;
    f_alpha = f;
    f_key = 0;
    g_alpha = g0;
    g_key = 0;
    df_alpha = dot(g_alpha, p);
    df_key = 0;
  }

  int init(Vec6& x) {
    delta_f = 0;
    call(x, 2, &f, &gradient);
    x0 = x;
    g0 = gradient;
    g0norm = norm(g0);
    for (int i = 0; i < 6; i++) p[i] = gradient[i] * (-1 / g0norm);
    pnorm = norm(p);
    fp0 = -g0norm;
    restart_line();
    return kNotStarted;
  }

  int line_search(double alpha1, double& alpha_new) {
    double f0, slope0, falpha, falpha_prev, fpalpha, fpalpha_prev;
    double alpha = alpha1, alpha_prev = 0.0;
    int i = 0;
    value_and_slope_at(0.0, f0, slope0);
    falpha_prev = f0;
    fpalpha_prev = slope0;
    double a = 0.0, b = alpha, fa = f0, fb = 0.0, fpa = slope0, fpb = 0.0;
    const double nan = std::numeric_limits<double>::quiet_NaN();
    while (i++ < bracket_iters) {  // bracketing
      falpha = value_at(alpha);
      if (falpha > f0 + alpha * rho * slope0 || falpha >= falpha_prev) {
        a = alpha_prev, fa = falpha_prev, fpa = fpalpha_prev;
        b = alpha, fb = falpha, fpb = nan;
        break;
      }
      fpalpha = slope_at(alpha);
      if (std::fabs(fpalpha) <= -sigma * slope0) {
        alpha_new = alpha;
        return kSuccess;
      }
      if (fpalpha >= 0) {
        a = alpha, fa = falpha, fpa = fpalpha;
        b = alpha_prev, fb = falpha_prev, fpb = fpalpha_prev;
        break;
      }
      const double delta = alpha - alpha_prev;
      const double next = interpolate(alpha_prev, falpha_prev, fpalpha_prev, alpha, falpha, fpalpha, alpha + delta, alpha + tau1 * delta, order);
      alpha_prev = alpha;
      falpha_prev = falpha;
      fpalpha_prev = fpalpha;
      alpha = next;
    }
    while (i++ < section_iters) {  // sectioning of [a, b]
      const double delta = b - a;
      alpha = interpolate(a, fa, fpa, b, fb, fpb, a + tau2 * delta, b - tau3 * delta, order);
      falpha = value_at(alpha);
      if ((a - alpha) * fpa <= std::numeric_limits<double>::epsilon()) return kNoProgress;
      if (falpha > f0 + rho * alpha * slope0 || falpha >= fa) {
        b = alpha, fb = falpha, fpb = nan;
      } else {
        fpalpha = slope_at(alpha);
        if (std::fabs(fpalpha) <= -sigma * slope0) {
          alpha_new = alpha;
          return kSuccess;
        }
        if (((b - a) >= 0 && fpalpha >= 0) || ((b - a) <= 0 && fpalpha <= 0)) {
          b = a, fb = fa, fpb = fpa;
        }
        a = alpha, fa = falpha, fpa = fpalpha;
      }
    }
    return kSuccess;
  }

  int step(Vec6& x) {
    double alpha = 0.0, alpha1;
    const double f0 = f;
    if (pnorm == 0.0 || g0norm == 0.0 || fp0 == 0) return kNoProgress;
    if (delta_f < 0) {
      const double del = std::max(-delta_f, 10 * std::numeric_limits<double>::epsilon() * std::fabs(f0));
      alpha1 = std::min(1.0, 2.0 * del / (-fp0));
    } else {
      alpha1 = std::fabs(step_size);
    }
    const int status = line_search(alpha1, alpha);
    if (status != kSuccess) return status;
    double fa, dfa;
    value_and_slope_at(alpha, fa, dfa);  // updatePosition
    f = f_alpha;
    x = x_alpha;
    gradient = g_alpha;
    delta_f = f - f0;
    Vec6 dx, dg;
    for (int i = 0; i < 6; i++) dx[i] = x[i] - x0[i];
    for (int i = 0; i < 6; i++) dg[i] = gradient[i] - g0[i];
    const double dxg = dot(dx, gradient), dgg = dot(dg, gradient), dxdg = dot(dx, dg), dgnorm = norm(dg);
    double A = 0, B = 0;
    if (dxdg != 0) {
      B = dxg / dxdg;
      A = -(1.0 + dgnorm * dgnorm / dxdg) * B + dgg / dxdg;
    }
    for (int i = 0; i < 6; i++) p[i] = (gradient[i] - A * dx[i]) - B * dg[i];
    g0 = gradient;
    x0 = x;
    g0norm = norm(g0);
    pnorm = norm(p);
    const double dir = dot(p, gradient) > 0 ? -1.0 : 1.0;
    for (int i = 0; i < 6; i++) p[i] *= dir / pnorm;
    pnorm = norm(p);
    fp0 = dot(p, g0);
    restart_line();
    return kSuccess;
  }

  int test_gradient(double epsilon) const {
    if (epsilon < 0) return kNegativeGradientEpsilon;
    return norm(gradient) < epsilon ? kSuccess : kRunning;
  }
};

// estimateRigidTransformationBFGS (GO:180-242).  *ok = false where the reference throws.
int estimate_bfgs(lgs_gicp_omp* g, float* tm, bool* ok) {
  *ok = false;
  if (g->n_corr < 4) return LGS_OK;  // NotEnoughPointsException
  Vec6 x;
  x[0] = tm[12];
  x[1] = tm[13];
  x[2] = tm[14];
  x[3] = std::atan2(tm[6], tm[10]);
  x[4] = std::asin(-tm[2]);
  x[5] = std::atan2(tm[1], tm[0]);
  Bfgs bfgs;
  bfgs.g = g;
  int inner = 0;
  int result = bfgs.init(x);
  result = kRunning;
  do {
    inner++;
    result = bfgs.step(x);
    if (result) break;
    result = bfgs.test_gradient(1e-2);
  } while (result == kRunning && inner < g->max_inner_iterations);
  g->inner_total += inner;
  if (bfgs.err != LGS_OK) return bfgs.err;
  if (result == kNoProgress || result == kSuccess || inner == g->max_inner_iterations) {
    identity16f(tm);
    apply_state(tm, x.v);
    *ok = true;
  }
  return LGS_OK;
}

int ensure_covs(lgs_gicp_omp* g, GicpCloud& c) {
  if (c.covs_ready && c.covs_k == g->k && c.covs_reg == kCovsPcl) return LGS_OK;
  lgs_ctx* ctx = g->ctx;
  if (g->k > c.n) {  // GO:54-58
    set_error("GeneralizedIterativeClosestPoint: number of points in cloud (%lld) is less than k_correspondences_ (%d)", static_cast<long long>(c.n), g->k);
    return LGS_ERR_STATE;
  }
  LGS_TRY(c.ensure_index(ctx));
  LGS_TRY(c.covs.reserve(static_cast<size_t>(c.n) * 72));
  LGS_TRY(ctx->tmp[1].reserve(static_cast<size_t>(c.n) * g->k * 4));
  int* knn_idx = ctx->tmp[1].as<int>();
  LGS_TRY(nn_self_knn(ctx, c.nn, g->k, knn_idx, nullptr));
  pgicp_covariance_kernel<<<grid_for(c.n, 128), 128, 0, ctx->stream>>>(c.pts.as<float4>(), static_cast<int>(c.n), g->k, g->gicp_epsilon, knn_idx,
                                                                      c.covs.as<double>());
  ctx->launches++;
  LGS_CUDA(cudaGetLastError());
  c.covs_ready = true;
  c.covs_k = g->k;
  c.covs_reg = kCovsPcl;
  return LGS_OK;
}

int ensure_ready(lgs_gicp_omp* g) {
  if (!g->source || !g->target || g->source->n == 0 || g->target->n == 0) {
    set_error("GeneralizedIterativeClosestPoint: setInputSource and setInputTarget must be called with non-empty clouds first");
    return LGS_ERR_STATE;
  }
  LGS_TRY(ensure_covs(g, *g->target));
  LGS_TRY(ensure_covs(g, *g->source));
  const size_t n = static_cast<size_t>(g->source->n);
  LGS_TRY(g->output.reserve(n * 16));
  LGS_TRY(g->corr.reserve(n * 4));
  LGS_TRY(g->mahal.reserve(n * 36));
  LGS_TRY(g->partials.reserve(static_cast<size_t>(fun_grid(g->source->n)) * 13 * sizeof(Fix128)));
  if (!g->state.p) {
    LGS_TRY(g->state.reserve(64));
    LGS_CUDA(cudaMemsetAsync(g->state.p, 0, 64, g->ctx->stream));
  }
  return LGS_OK;
}

// output = guess * source (GO:398)
int transform_source(lgs_gicp_omp* g) { return transform_cloud(g->ctx, g->source->pts.as<float4>(), g->source->n, g->guess, g->output.as<float4>()); }

// the correspondence / Mahalanobis half of one outer iteration (GO:404-474); sets g->n_corr
int update_correspondences(lgs_gicp_omp* g) {
  g->session.close();  // the correspondence / Mahalanobis kernels need the SMs; the next functor call opens a new run
  lgs_ctx* ctx = g->ctx;
  PgicpParams P;
  memcpy(P.T, g->T, sizeof(P.T));
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) {
      double s = 0;
      for (int k = 0; k < 4; k++) s += static_cast<double>(g->T[k * 4 + i]) * static_cast<double>(g->guess[j * 4 + k]);
      P.R[i * 3 + j] = s;
    }
  P.thr2 = g->corr_dist_threshold * g->corr_dist_threshold;
  const int n = static_cast<int>(g->source->n);
  const int cgrid = std::max(1, std::min(grid_for(n, kPCorrBlock / 32), kNumSMs * 8));
  pgicp_correspondence_kernel<<<cgrid, kPCorrBlock, 0, ctx->stream>>>(g->target->nn.view(), g->output.as<float4>(), n, P, g->corr.as<int>());
  Mailbox mb;
  LGS_TRY(mailbox_next(ctx, &mb));
  pgicp_mahalanobis_kernel<<<fun_grid(n), kFunBlock, 0, ctx->stream>>>(n, P, g->source->covs.as<double>(), g->target->covs.as<double>(), g->corr.as<int>(),
                                                                      g->mahal.as<float>(), g->partials.as<Fix128>(), g->state.as<unsigned>(), mb);
  ctx->launches += 2;
  LGS_CUDA(cudaGetLastError());
  double cnt = 0;
  LGS_TRY(mailbox_wait(ctx, mb, 1, &cnt));
  g->n_corr = static_cast<int>(cnt);
  return LGS_OK;
}

int set_cloud(lgs_gicp_omp* g, std::shared_ptr<GicpCloud>* slot, const void* pts, int64_t n, int32_t stride, bool on_device) {
  if (!*slot) *slot = std::make_shared<GicpCloud>();
  GicpCloud& c = **slot;
  c.nn_ready = false;
  c.covs_ready = false;  // GO.h:155,168: a new cloud drops its covariances
  LGS_TRY(load_cloud(g->ctx, pts, n, stride, on_device, &c.pts));
  c.n = n;
  return LGS_OK;
}

}  // namespace

extern "C" {

int lgs_gicp_omp_create(lgs_ctx* ctx, lgs_gicp_omp** out) {
  LGS_REQUIRE(ctx && out, "null argument");
  lgs_gicp_omp* g = new lgs_gicp_omp;
  g->ctx = ctx;
  for (float* T : {g->base_T, g->T, g->prev_T, g->final_T, g->guess}) identity16f(T);
  *out = g;
  return LGS_OK;
}

void lgs_gicp_omp_destroy(lgs_gicp_omp* g) {
  if (!g) return;
  g->session.release(g->ctx);
  g->source.reset();
  g->target.reset();
  for (DevBuf* b : {&g->output, &g->corr, &g->mahal, &g->partials, &g->state, &g->out_cloud}) b->release();
  delete g;
}

int lgs_gicp_omp_set_correspondence_randomness(lgs_gicp_omp* g, int32_t k) {
  LGS_REQUIRE(g, "null");
  LGS_REQUIRE(k >= 1 && k <= kMaxK, "k must be in [1, 32]");
  g->k = k;
  return LGS_OK;
}
int lgs_gicp_omp_set_max_correspondence_distance(lgs_gicp_omp* g, double d) { LGS_REQUIRE(g, "null"); g->corr_dist_threshold = d; return LGS_OK; }
int lgs_gicp_omp_set_transformation_epsilon(lgs_gicp_omp* g, double e) { LGS_REQUIRE(g, "null"); g->trans_eps = e; return LGS_OK; }
int lgs_gicp_omp_set_rotation_epsilon(lgs_gicp_omp* g, double e) { LGS_REQUIRE(g, "null"); g->rotation_eps = e; return LGS_OK; }
int lgs_gicp_omp_set_maximum_iterations(lgs_gicp_omp* g, int32_t n) { LGS_REQUIRE(g, "null"); g->max_iterations = n; return LGS_OK; }
int lgs_gicp_omp_set_maximum_optimizer_iterations(lgs_gicp_omp* g, int32_t n) { LGS_REQUIRE(g, "null"); g->max_inner_iterations = n; return LGS_OK; }

int lgs_gicp_omp_set_source(lgs_gicp_omp* g, const void* pts, int64_t n, int32_t stride) {
  LGS_REQUIRE(g, "null");
  return set_cloud(g, &g->source, pts, n, stride, false);
}
int lgs_gicp_omp_set_target(lgs_gicp_omp* g, const void* pts, int64_t n, int32_t stride) {
  LGS_REQUIRE(g, "null");
  return set_cloud(g, &g->target, pts, n, stride, false);
}
int lgs_gicp_omp_set_source_dev(lgs_gicp_omp* g, const float* pts_dev, int64_t n) {
  LGS_REQUIRE(g, "null");
  return set_cloud(g, &g->source, pts_dev, n, 16, true);
}
int lgs_gicp_omp_set_target_dev(lgs_gicp_omp* g, const float* pts_dev, int64_t n) {
  LGS_REQUIRE(g, "null");
  return set_cloud(g, &g->target, pts_dev, n, 16, true);
}

// pcl::Registration::align + computeTransformation (GO:370-516)
int lgs_gicp_omp_align(lgs_gicp_omp* g, const float* guess16, lgs_align_result* res, float* out_cloud) {
  LGS_NVTX("lgs_gicp_omp_align");
  LGS_REQUIRE(g && res, "null argument");
  SessionScope scope(g->session);
  memset(res, 0, sizeof(*res));
  LGS_TRY(use_device(g->ctx));
  LGS_TRY(ensure_ready(g));
  g->f_calls = g->df_calls = g->fdf_calls = g->inner_total = 0;
  identity16f(g->guess);
  if (guess16) memcpy(g->guess, guess16, sizeof(g->guess));
  for (float* T : {g->base_T, g->T, g->prev_T, g->final_T}) identity16f(T);
  LGS_TRY(transform_source(g));
  bool converged = false;
  int nr_iterations = 0;
  while (!converged) {
    LGS_TRY(update_correspondences(g));
    memcpy(g->prev_T, g->T, sizeof(g->T));
    bool ok = false;
    LGS_TRY(estimate_bfgs(g, g->T, &ok));
    if (!ok) break;  // GO:495-499: the exception ends the loop, converged_ stays false
    double delta = 0.;
    for (int k = 0; k < 4; k++)
      for (int l = 0; l < 4; l++) {
        const double ratio = (k < 3 && l < 3) ? 1. / g->rotation_eps : 1. / g->trans_eps;
        const double c_delta = ratio * std::abs(g->prev_T[l * 4 + k] - g->T[l * 4 + k]);
        if (c_delta > delta) delta = c_delta;
      }
    nr_iterations++;
    if (nr_iterations >= g->max_iterations || delta < 1) {
      converged = true;
      memcpy(g->prev_T, g->T, sizeof(g->T));
    }
  }
  g->session.close();  // before the output cloud's kernel
  mul4f(g->prev_T, g->guess, g->final_T);  // GO:512
  memcpy(res->T, g->final_T, sizeof(g->final_T));
  res->iterations = nr_iterations;
  res->converged = converged ? 1 : 0;
  res->evaluations = g->fdf_calls + g->df_calls;
  res->line_search_trials = g->f_calls;
  res->hessian_recomputes = g->inner_total;
  if (out_cloud) LGS_TRY(write_aligned_cloud(g->ctx, g->source->pts.as<float4>(), g->source->n, g->final_T, &g->out_cloud, out_cloud));  // GO:515
  return LGS_OK;
}

int lgs_gicp_omp_fitness(lgs_gicp_omp* g, double max_range, double* fitness) {
  LGS_REQUIRE(g && fitness, "null argument");
  if (!g->source || !g->target) {
    set_error("GeneralizedIterativeClosestPoint: target and source must be set");
    return LGS_ERR_STATE;
  }
  LGS_TRY(use_device(g->ctx));
  LGS_TRY(g->target->ensure_index(g->ctx));
  return nn_fitness(g->ctx, g->target->nn, g->source->pts.as<float4>(), g->source->n, g->final_T, max_range, fitness);
}

int lgs_gicp_omp_export_covariances(lgs_gicp_omp* g, int32_t which, double* covs) {
  LGS_REQUIRE(g && covs, "null argument");
  std::shared_ptr<GicpCloud> c = which == 0 ? g->source : g->target;
  if (!c || c->n == 0) {
    set_error("lgs_gicp_omp_export_covariances: cloud not set");
    return LGS_ERR_STATE;
  }
  LGS_TRY(use_device(g->ctx));
  LGS_TRY(ensure_covs(g, *c));
  LGS_CUDA(cudaMemcpyAsync(covs, c->covs.p, static_cast<size_t>(c->n) * 72, cudaMemcpyDeviceToHost, g->ctx->stream));
  LGS_CUDA(cudaStreamSynchronize(g->ctx->stream));
  return LGS_OK;
}

// parity hook: the set-up of one outer iteration at (transformation_, guess) and the three functor evaluations at x:
// out15 = f(x), df(x)[6], fdf(x) -> f, g[6], number of correspondences; corr / mahal (n_source ints / n_source x 9
// floats) are optional
int lgs_gicp_omp_functor(lgs_gicp_omp* g, const float* guess16, const float* transformation16, const double* x6, double* out15,
                         int32_t* corr, float* mahal) {
  LGS_REQUIRE(g && guess16 && transformation16 && x6 && out15, "null argument");
  LGS_TRY(use_device(g->ctx));
  LGS_TRY(ensure_ready(g));
  memcpy(g->guess, guess16, sizeof(g->guess));
  memcpy(g->T, transformation16, sizeof(g->T));
  identity16f(g->base_T);
  LGS_TRY(transform_source(g));
  LGS_TRY(update_correspondences(g));
  out15[14] = g->n_corr;
  double f_dummy = 0;
  LGS_TRY(functor_eval(g, x6, 0, out15, nullptr));
  LGS_TRY(functor_eval(g, x6, 1, &f_dummy, out15 + 1));
  LGS_TRY(functor_eval(g, x6, 2, out15 + 7, out15 + 8));
  cudaStream_t st = g->ctx->stream;
  if (corr) LGS_CUDA(cudaMemcpyAsync(corr, g->corr.p, static_cast<size_t>(g->source->n) * 4, cudaMemcpyDeviceToHost, st));
  if (mahal) LGS_CUDA(cudaMemcpyAsync(mahal, g->mahal.p, static_cast<size_t>(g->source->n) * 36, cudaMemcpyDeviceToHost, st));
  LGS_CUDA(cudaStreamSynchronize(st));
  return LGS_OK;
}

}  // extern "C"
