// GICP scan-to-map registration: fast_gicp::FastGICP over fast_gicp::LsqRegistration behind pcl::Registration.
//
//   covariances  -> calculate_covariances (FG:241-298): exact k-NN (k=20, self included) through the implicit BVH,
//                   f64 covariance of the neighbours in FLANN's ascending-distance order, 3x3 Jacobi SVD and the
//                   PLANE / MIN_EIG / NORMALIZED_MIN_EIG / FROBENIUS / NONE regularisations; one thread per point,
//                   threads walk the Morton-sorted cloud so that a warp's traversals stay coherent.
//   linearize    -> update_correspondences + linearize (FG:115-211) fused: f32 transform, exact 1-NN, fused
//                   Mahalanobis matrix (C_B + T C_A T^T)^-1 in f64, error, H (6x6) and b (6) accumulated in f64,
//                   block reduction + fixed-order last-block final reduction.
//   compute_error-> FG:214-237 with the stored correspondences / Mahalanobis matrices.
//   align        -> LsqRegistration::computeTransformation + step_lm (LSQ:53-79,125-172) on the host.
#include <algorithm>
#include <cmath>
#include <memory>

#include "gicp.cuh"
#include "reduce.cuh"

namespace lgs {

// ---------------------------------------------------------------------------------------------
// covariances

// list == nullptr: point i of n, neighbour row i.  Otherwise: point list[j] for j < *count, neighbour row j (lazy covariances).
__global__ void __launch_bounds__(128) gicp_covariance_kernel(NNView v, const float4* __restrict__ pts, int n, int k, int regularization,
                                                             const int* __restrict__ knn_idx, double* __restrict__ covs,
                                                             const int* __restrict__ list, const int* __restrict__ count) {
  const int j0 = blockIdx.x * blockDim.x + threadIdx.x;
  if (j0 >= (list ? *count : n)) return;
  const int i = list ? list[j0] : j0;  // original point index
  const int* nb = knn_idx + static_cast<size_t>(j0) * k;
  // neighbors.rowwise().mean(): sequential sum over the k columns, divided by k (missing columns are zero)
  double s0 = 0, s1 = 0, s2 = 0;
  for (int j = 0; j < k; j++) {
    const int id = nb[j];
    if (id >= 0) {
      const float4 p = __ldg(pts + id);
      s0 += static_cast<double>(p.x);
      s1 += static_cast<double>(p.y);
      s2 += static_cast<double>(p.z);
    }
  }
  const double m0 = s0 / k, m1 = s1 / k, m2 = s2 / k;
  double c00 = 0, c01 = 0, c02 = 0, c11 = 0, c12 = 0, c22 = 0;
  for (int j = 0; j < k; j++) {
    const int id = nb[j];
    double x = 0, y = 0, z = 0;
    if (id >= 0) {
      const float4 p = __ldg(pts + id);
      x = p.x; y = p.y; z = p.z;
    }
    x -= m0; y -= m1; z -= m2;
    c00 += x * x; c01 += x * y; c02 += x * z;
    c11 += y * y; c12 += y * z; c22 += z * z;
  }
  double cov[9] = {c00 / k, c01 / k, c02 / k, c01 / k, c11 / k, c12 / k, c02 / k, c12 / k, c22 / k};
  double out[9];
  if (regularization == LGS_REG_NONE) {
    for (int t = 0; t < 9; t++) out[t] = cov[t];
  } else if (regularization == LGS_REG_FROBENIUS) {
    const double lambda = 1e-3;
    double Cm[9], Ci[9];
    for (int t = 0; t < 9; t++) Cm[t] = cov[t] + ((t % 4 == 0) ? lambda : 0.0);
    m::inv3(Cm, Ci);
    double nrm = 0;
    for (int t = 0; t < 9; t++) nrm += Ci[t] * Ci[t];
    nrm = sqrt(nrm);
    for (int t = 0; t < 9; t++) Ci[t] /= nrm;
    m::inv3(Ci, out);
  } else {
    double U[9], S[3], V[9], val[3];
    m::svd_jacobi<3, double>(cov, U, S, V);
    if (regularization == LGS_REG_PLANE) {
      val[0] = 1; val[1] = 1; val[2] = 1e-3;
    } else if (regularization == LGS_REG_MIN_EIG) {
      for (int a = 0; a < 3; a++) val[a] = m::tmax(S[a], 1e-3);
    } else {  // std::max as the reference's Array max: 0 / 0 of an all-zero covariance stays NaN (fmax would give 1e-3)
      const double mx = m::tmax(S[0], m::tmax(S[1], S[2]));
      for (int a = 0; a < 3; a++) val[a] = m::tmax(S[a] / mx, 1e-3);
    }
    double UD[9];
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 3; c++) UD[r * 3 + c] = U[r * 3 + c] * val[c];
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 3; c++) out[r * 3 + c] = (UD[r * 3] * V[c * 3] + UD[r * 3 + 1] * V[c * 3 + 1]) + UD[r * 3 + 2] * V[c * 3 + 2];
  }
  for (int t = 0; t < 9; t++) covs[static_cast<size_t>(i) * 9 + t] = out[t];
}

int GicpCloud::ensure_index(lgs_ctx* ctx) {
  if (!nn_ready) {
    LGS_TRY(nn.build(ctx, pts.as<float4>(), n));
    nn_ready = true;
  }
  return LGS_OK;
}

int GicpCloud::ensure_covariances(lgs_ctx* ctx, int k, int regularization) {
  if (covs_ready && (covs_user || (covs_k == k && covs_reg == regularization))) return LGS_OK;
  LGS_REQUIRE(k >= 1 && k <= kMaxK, "k_correspondences must be in [1, 32]");
  LGS_TRY(ensure_index(ctx));
  LGS_TRY(covs.reserve(static_cast<size_t>(n > 0 ? n : 1) * 72));
  if (n > 0) {
    LGS_TRY(ctx->tmp[1].reserve(static_cast<size_t>(n) * k * 4));
    int* knn_idx = ctx->tmp[1].as<int>();
    LGS_TRY(nn_self_knn(ctx, nn, k, knn_idx, nullptr));
    gicp_covariance_kernel<<<grid_for(n, 128), 128, 0, ctx->stream>>>(nn.view(), pts.as<float4>(), static_cast<int>(n), k, regularization, knn_idx,
                                                                     covs.as<double>(), nullptr, nullptr);
    ctx->launches++;
    LGS_CUDA(cudaGetLastError());
  }
  covs_ready = true;
  covs_user = false;
  covs_lazy = false;
  covs_k = k;
  covs_reg = regularization;
  return LGS_OK;
}

// marks the target points that correspondences refer to and that have no covariance yet, and lists them
__global__ void __launch_bounds__(256) gicp_mark_needed_kernel(const int* __restrict__ corr, int n_corr, int* __restrict__ done, int* __restrict__ list,
                                                              int* __restrict__ count) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_corr) return;
  const int c = corr[i];
  if (c < 0) return;
  if (atomicExch(done + c, 1) == 0) list[atomicAdd(count, 1)] = c;
}

int GicpCloud::begin_lazy_covariances(lgs_ctx* ctx, int k, int regularization) {
  LGS_REQUIRE(k >= 1 && k <= kMaxK, "k_correspondences must be in [1, 32]");
  LGS_TRY(ensure_index(ctx));
  const size_t np = static_cast<size_t>(n > 0 ? n : 1);
  LGS_TRY(covs.reserve(np * 72));
  LGS_TRY(cov_done.reserve(np * 4));
  LGS_TRY(work_list.reserve(np * 4));
  LGS_TRY(work_count.reserve(64));
  LGS_CUDA(cudaMemsetAsync(cov_done.p, 0, np * 4, ctx->stream));
  covs_lazy = true;
  covs_ready = false;
  covs_user = false;
  covs_k = k;
  covs_reg = regularization;
  return LGS_OK;
}

int GicpCloud::cover_correspondences(lgs_ctx* ctx, const int* corr_dev, int64_t n_corr) {
  if (!covs_lazy || n == 0 || n_corr == 0) return LGS_OK;
  cudaStream_t st = ctx->stream;
  const int64_t cap = std::min<int64_t>(n_corr, n);  // at most one new point per correspondence
  LGS_TRY(ctx->tmp[1].reserve(static_cast<size_t>(cap) * covs_k * 4));
  int* count = work_count.as<int>();
  LGS_CUDA(cudaMemsetAsync(count, 0, 4, st));
  gicp_mark_needed_kernel<<<grid_for(n_corr, 256), 256, 0, st>>>(corr_dev, static_cast<int>(n_corr), cov_done.as<int>(), work_list.as<int>(), count);
  ctx->launches++;
  LGS_TRY(nn_knn_list(ctx, nn, pts.as<float4>(), work_list.as<int>(), count, cap, covs_k, ctx->tmp[1].as<int>()));
  gicp_covariance_kernel<<<grid_for(cap, 128), 128, 0, st>>>(nn.view(), pts.as<float4>(), static_cast<int>(n), covs_k, covs_reg, ctx->tmp[1].as<int>(),
                                                           covs.as<double>(), work_list.as<int>(), count);
  ctx->launches++;
  LGS_CUDA(cudaGetLastError());
  return LGS_OK;
}

// ---------------------------------------------------------------------------------------------
// linearize / compute_error

struct LinParams {
  double T[16];   // row-major Isometry3d
  float Tf[16];   // trans.cast<float>()
  double corr_thr2;  // corr_dist_threshold_^2 (f64 product of the f64 member, compared against the f32 distance)
};

constexpr int kLinBlock = 128;

// the per-CTA rows are folded in two groups, even rows and odd rows, each with sixteen loads in flight (reduce.cuh)
constexpr int kLinGroups = 2, kLinLoads = 16;

// error term of one correspondence: e = mean_B - T mean_A ; returns e^T M e and (optionally) accumulates H, b
template <bool WANT_HB>
__device__ __forceinline__ void gicp_point_terms(const LinParams& P, const float4& a, const float4& b, const double* __restrict__ M, double* acc) {
  const double mA[3] = {a.x, a.y, a.z};
  double tA[3], err[3];
#pragma unroll
  for (int r = 0; r < 3; r++) tA[r] = ((P.T[r * 4] * mA[0] + P.T[r * 4 + 1] * mA[1]) + P.T[r * 4 + 2] * mA[2]) + P.T[r * 4 + 3] * 1.0;
  err[0] = static_cast<double>(b.x) - tA[0];
  err[1] = static_cast<double>(b.y) - tA[1];
  err[2] = static_cast<double>(b.z) - tA[2];
  double eM[3];
#pragma unroll
  for (int c = 0; c < 3; c++) eM[c] = (err[0] * M[c] + err[1] * M[3 + c]) + err[2] * M[6 + c];
  acc[0] += (eM[0] * err[0] + eM[1] * err[1]) + eM[2] * err[2];
  if (WANT_HB) {
    // dtdx0 = [skewd(T mean_A), -I]
    const double J[3][6] = {{0, -tA[2], tA[1], -1, 0, 0}, {tA[2], 0, -tA[0], 0, -1, 0}, {-tA[1], tA[0], 0, 0, 0, -1}};
    double JtM[6][3];
#pragma unroll
    for (int r = 0; r < 6; r++)
#pragma unroll
      for (int c = 0; c < 3; c++) JtM[r][c] = (J[0][r] * M[c] + J[1][r] * M[3 + c]) + J[2][r] * M[6 + c];
#pragma unroll
    for (int r = 0; r < 6; r++) {
#pragma unroll
      for (int c = 0; c < 6; c++) acc[7 + r * 6 + c] += (JtM[r][0] * J[0][c] + JtM[r][1] * J[1][c]) + JtM[r][2] * J[2][c];
      acc[1 + r] += (JtM[r][0] * err[0] + JtM[r][1] * err[1]) + JtM[r][2] * err[2];
    }
  }
}

// update_correspondences, search half (FG:115-137): one warp per source point; pt = trans_f * input, exact 1-NN in
// the target, kept when its squared distance is below the threshold.  The Mahalanobis half (FG:139-150) is fused
// into gicp_linearize_kernel.
constexpr int kCorrBlock = 256;
__global__ void __launch_bounds__(kCorrBlock) gicp_correspondence_kernel(NNView tv, const float4* __restrict__ src, const float4* __restrict__ tgt, int n,
                                                                        LinParams P, int* __restrict__ corr, int* __restrict__ nn_prev, int use_seed) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i = blockIdx.x * (kCorrBlock / 32) + warp; i < n; i += gridDim.x * (kCorrBlock / 32)) {
    const float4 a = __ldg(src + i);
    // pt = trans_f * input (Isometry3f * Vector4f, column-by-column GEMV)
    const float qx = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(P.Tf[0], a.x), __fmul_rn(P.Tf[1], a.y)), __fmul_rn(P.Tf[2], a.z)), P.Tf[3]);
    const float qy = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(P.Tf[4], a.x), __fmul_rn(P.Tf[5], a.y)), __fmul_rn(P.Tf[6], a.z)), P.Tf[7]);
    const float qz = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(P.Tf[8], a.x), __fmul_rn(P.Tf[9], a.y)), __fmul_rn(P.Tf[10], a.z)), P.Tf[11]);
    float d2;
    int id;
    // seed: the neighbour found at the previous linearisation (the pose moved little since), see nn_search1_warp_seeded
    int seed = use_seed ? nn_prev[i] : -1;
    if (seed >= tv.n) seed = -1;  // the 'nothing found' sentinel of an empty index
    float seed_d = 0.f;
    if (seed >= 0) seed_d = nn_dist2(qx, qy, qz, __ldg(tgt + seed));
    nn_search1_warp_seeded(tv, qx, qy, qz, lane, seed_d, seed, d2, id);
    if (lane == 0) {
      corr[i] = (static_cast<double>(d2) < P.corr_thr2) ? id : -1;  // FG:136
      nn_prev[i] = id;
    }
  }
}

__global__ void __launch_bounds__(kLinBlock) gicp_linearize_kernel(const float4* __restrict__ src, const float4* __restrict__ tgt, int n,
                                                                  LinParams P, const double* __restrict__ cov_src,
                                                                  const double* __restrict__ cov_tgt, const int* __restrict__ corr,
                                                                  double* __restrict__ mahal, int want_hb, double* __restrict__ partials,
                                                                  unsigned* __restrict__ counter, const Mailbox mb) {
  double acc[43];
#pragma unroll
  for (int k = 0; k < 43; k++) acc[k] = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 a = src[i];
    const int c = corr[i];
    if (c < 0) continue;
    // RCR = cov_B + T cov_A T^T (3x3 block), mahalanobis = RCR^-1  (FG:146-150)
    const double* CA = cov_src + static_cast<size_t>(i) * 9;
    const double* CB = cov_tgt + static_cast<size_t>(c) * 9;
    double RC[9], RCR[9], M[9];
#pragma unroll
    for (int r = 0; r < 3; r++)
#pragma unroll
      for (int cc = 0; cc < 3; cc++) RC[r * 3 + cc] = (P.T[r * 4] * CA[cc] + P.T[r * 4 + 1] * CA[3 + cc]) + P.T[r * 4 + 2] * CA[6 + cc];
#pragma unroll
    for (int r = 0; r < 3; r++)
#pragma unroll
      for (int cc = 0; cc < 3; cc++)
        RCR[r * 3 + cc] = CB[r * 3 + cc] + ((RC[r * 3] * P.T[cc * 4] + RC[r * 3 + 1] * P.T[cc * 4 + 1]) + RC[r * 3 + 2] * P.T[cc * 4 + 2]);
    m::inv3(RCR, M);
    double* Mo = mahal + static_cast<size_t>(i) * 9;
#pragma unroll
    for (int t = 0; t < 9; t++) Mo[t] = M[t];
    const float4 b = __ldg(tgt + c);
    if (want_hb)
      gicp_point_terms<true>(P, a, b, M, acc);
    else
      gicp_point_terms<false>(P, a, b, M, acc);
  }
  grid_finish<43, kLinBlock, kLinGroups, kLinLoads>(cta_row<kLinBlock>(acc), partials, counter, mb);
}

__global__ void __launch_bounds__(kLinBlock) gicp_error_kernel(const float4* __restrict__ src, const float4* __restrict__ tgt, int n, LinParams P,
                                                              const int* __restrict__ corr, const double* __restrict__ mahal,
                                                              double* __restrict__ partials, unsigned* __restrict__ counter, const Mailbox mb) {
  double acc[1] = {0.0};
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int c = corr[i];
    if (c < 0) continue;
    const float4 a = src[i];
    const float4 b = __ldg(tgt + c);
    double M[9];
#pragma unroll
    for (int t = 0; t < 9; t++) M[t] = mahal[static_cast<size_t>(i) * 9 + t];
    gicp_point_terms<false>(P, a, b, M, acc);
  }
  grid_finish<1, kLinBlock, kLinGroups, kLinLoads>(cta_row<kLinBlock>(acc), partials, counter, mb);
}

}  // namespace lgs

// =============================================================================================
using namespace lgs;

namespace {

void identity_d(double* T) {
  for (int i = 0; i < 16; i++) T[i] = (i % 5 == 0) ? 1.0 : 0.0;
}

// Isometry3d * Isometry3d: linear = L L', translation = L t' + t
void iso_mul(const double* A, const double* B, double* C) {
  double R[16];
  identity_d(R);
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) R[i * 4 + j] = (A[i * 4] * B[j] + A[i * 4 + 1] * B[4 + j]) + A[i * 4 + 2] * B[8 + j];
  for (int i = 0; i < 3; i++) R[i * 4 + 3] = ((A[i * 4] * B[3] + A[i * 4 + 1] * B[7]) + A[i * 4 + 2] * B[11]) + A[i * 4 + 3];
  memcpy(C, R, sizeof(R));
}

// so3_exp (so3/so3.hpp:58-77) followed by Quaterniond::toRotationMatrix
void so3_exp_matrix(const double* w, double* R) {
  const double theta_sq = (w[0] * w[0] + w[1] * w[1]) + w[2] * w[2];
  double imag, real;
  if (theta_sq < 1e-10) {
    const double theta_quad = theta_sq * theta_sq;
    imag = 0.5 - 1.0 / 48.0 * theta_sq + 1.0 / 3840.0 * theta_quad;
    real = 1.0 - 1.0 / 8.0 * theta_sq + 1.0 / 384.0 * theta_quad;
  } else {
    const double theta = std::sqrt(theta_sq);
    const double half = 0.5 * theta;
    imag = std::sin(half) / theta;
    real = std::cos(half);
  }
  const double qw = real, qx = imag * w[0], qy = imag * w[1], qz = imag * w[2];
  const double tx = 2 * qx, ty = 2 * qy, tz = 2 * qz;
  const double twx = tx * qw, twy = ty * qw, twz = tz * qw;
  const double txx = tx * qx, txy = ty * qx, txz = tz * qx;
  const double tyy = ty * qy, tyz = tz * qy, tzz = tz * qz;
  R[0] = 1 - (tyy + tzz); R[1] = txy - twz;       R[2] = txz + twy;
  R[3] = txy + twz;       R[4] = 1 - (txx + tzz); R[5] = tyz - twx;
  R[6] = txz - twy;       R[7] = tyz + twx;       R[8] = 1 - (txx + tyy);
}

// every CTA contributes one row to the last-CTA pass: one CTA per SM at most (a 30 000-point cloud is 1.6 points per thread)
int lin_grid(int64_t n) { return std::max(1, std::min(grid_for(n, kLinBlock), kNumSMs)); }

int ensure_ready(lgs_gicp* g) {
  if (!g->source || !g->target) {
    set_error("FastGICP: setInputSource and setInputTarget must be called first");
    return LGS_ERR_STATE;
  }
  LGS_TRY(g->source->ensure_covariances(g->ctx, g->k, g->regularization));  // FG:104-109
  static const bool lazy_off = [] { const char* e = getenv("LGS_GICP_LAZY_TARGET"); return e && e[0] == '0'; }();
  GicpCloud& T = *g->target;
  const bool have = T.covs_ready && (T.covs_user || (T.covs_k == g->k && T.covs_reg == g->regularization));
  // worth it when the target is clearly larger than the source (scan against sub-map: a third of the target is ever matched);
  // between clouds of similar size nearly every target point is matched within a few iterations and the up-front pass is cheaper
  const bool small_target = 2 * T.n <= 3 * g->source->n;
  if (have || lazy_off || small_target || g->target == g->source) {
    LGS_TRY(T.ensure_covariances(g->ctx, g->k, g->regularization));
  } else if (!(T.covs_lazy && T.covs_k == g->k && T.covs_reg == g->regularization)) {
    LGS_TRY(T.begin_lazy_covariances(g->ctx, g->k, g->regularization));  // computed on first use (GicpCloud::cover_correspondences)
  }
  LGS_TRY(g->target->ensure_index(g->ctx));
  const size_t n = static_cast<size_t>(std::max<int64_t>(g->source->n, 1));
  LGS_TRY(g->corr.reserve(n * 4));
  LGS_TRY(g->nn_prev.reserve(n * 4));
  g->have_seed = false;  // a new align / hook call: the clouds may have changed since the seeds were written
  LGS_TRY(g->mahal.reserve(n * 72));
  const int grid = lin_grid(g->source->n);
  LGS_TRY(g->partials.reserve(static_cast<size_t>(grid) * 44 * 8));
  if (!g->counter.p) {
    LGS_TRY(g->counter.reserve(sizeof(unsigned)));
    LGS_CUDA(cudaMemsetAsync(g->counter.p, 0, sizeof(unsigned), g->ctx->stream));
  }
  return LGS_OK;
}

void fill_lin_params(const lgs_gicp* g, const double* T, LinParams* P) {
  for (int i = 0; i < 16; i++) {
    P->T[i] = T[i];
    P->Tf[i] = static_cast<float>(T[i]);
  }
  P->corr_thr2 = g->corr_dist_threshold * g->corr_dist_threshold;
}

// linearize (FG:155-211).  H/b may be null (cost only, but correspondences are still refreshed).
int linearize(lgs_gicp* g, const double* T, double* cost, double* H, double* b) {
  lgs_ctx* ctx = g->ctx;
  cudaStream_t st = ctx->stream;
  g->linearize_calls++;
  *cost = 0;
  if (H) std::fill(H, H + 36, 0.0);
  if (b) std::fill(b, b + 6, 0.0);
  const int n = static_cast<int>(g->source->n);
  if (n == 0) return LGS_OK;
  LinParams P;
  fill_lin_params(g, T, &P);
  unsigned* counter = g->counter.as<unsigned>();
  const int cgrid = std::max(1, std::min(grid_for(n, kCorrBlock / 32), kNumSMs * 8));
  Mailbox mb;
  LGS_TRY(mailbox_next(ctx, &mb));
  gicp_correspondence_kernel<<<cgrid, kCorrBlock, 0, st>>>(g->target->nn.view(), g->source->pts.as<float4>(), g->target->pts.as<float4>(), n, P, g->corr.as<int>(),
                                                          g->nn_prev.as<int>(), g->have_seed ? 1 : 0);
  g->have_seed = true;
  ctx->launches++;
  LGS_TRY(g->target->cover_correspondences(ctx, g->corr.as<int>(), n));
  gicp_linearize_kernel<<<lin_grid(n), kLinBlock, 0, st>>>(g->source->pts.as<float4>(), g->target->pts.as<float4>(), n, P,
                                                          g->source->covs.as<double>(), g->target->covs.as<double>(), g->corr.as<int>(),
                                                          g->mahal.as<double>(), (H && b) ? 1 : 0, g->partials.as<double>(), counter, mb);
  ctx->launches++;
  LGS_CUDA(cudaGetLastError());
  double h[kMailboxRecords];
  LGS_TRY(mailbox_wait(ctx, mb, 43, h));
  *cost = h[0];
  if (H && b) {
    memcpy(b, h + 1, 6 * 8);
    memcpy(H, h + 7, 36 * 8);
  }
  return LGS_OK;
}

// compute_error (FG:214-237)
int compute_error(lgs_gicp* g, const double* T, double* cost) {
  lgs_ctx* ctx = g->ctx;
  cudaStream_t st = ctx->stream;
  g->error_calls++;
  *cost = 0;
  const int n = static_cast<int>(g->source->n);
  if (n == 0) return LGS_OK;
  LinParams P;
  fill_lin_params(g, T, &P);
  unsigned* counter = g->counter.as<unsigned>();
  Mailbox mb;
  LGS_TRY(mailbox_next(ctx, &mb));
  gicp_error_kernel<<<lin_grid(n), kLinBlock, 0, st>>>(g->source->pts.as<float4>(), g->target->pts.as<float4>(), n, P, g->corr.as<int>(),
                                                      g->mahal.as<double>(), g->partials.as<double>(), counter, mb);
  ctx->launches++;
  LGS_CUDA(cudaGetLastError());
  LGS_TRY(mailbox_wait(ctx, mb, 1, cost));
  return LGS_OK;
}

// is_converged (LSQ:82-91)
bool is_converged(const lgs_gicp* g, const double* delta) {
  double r_max = 0, t_max = 0;
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) r_max = std::max(r_max, 1.0 / g->rotation_eps * std::fabs(delta[r * 4 + c] - (r == c ? 1.0 : 0.0)));
  for (int r = 0; r < 3; r++) t_max = std::max(t_max, 1.0 / g->trans_eps * std::fabs(delta[r * 4 + 3]));
  return std::max(r_max, t_max) < 1;
}

// step_lm (LSQ:125-172)
int step_lm(lgs_gicp* g, double* x0, double* delta, bool* ok) {
  double H[36], b[6], y0 = 0;
  LGS_TRY(linearize(g, x0, &y0, H, b));
  if (g->lm_lambda < 0.0) {
    double mx = 0;
    for (int i = 0; i < 6; i++) mx = std::max(mx, std::fabs(H[i * 7]));
    g->lm_lambda = g->lm_init_lambda_factor * mx;
  }
  double nu = 2.0;
  for (int i = 0; i < g->lm_max_iterations; i++) {
    double A[36], nb[6], d[6];
    for (int k = 0; k < 36; k++) A[k] = H[k] + ((k % 7 == 0) ? g->lm_lambda : 0.0);
    for (int k = 0; k < 6; k++) nb[k] = -b[k];
    m::ldlt_solve6(A, nb, d);
    identity_d(delta);
    double R[9];
    so3_exp_matrix(d, R);
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 3; c++) delta[r * 4 + c] = R[r * 3 + c];
    for (int r = 0; r < 3; r++) delta[r * 4 + 3] = d[3 + r];
    double xi[16], yi = 0;
    iso_mul(delta, x0, xi);
    LGS_TRY(compute_error(g, xi, &yi));
    double den = 0;
    for (int k = 0; k < 6; k++) den += d[k] * (g->lm_lambda * d[k] - b[k]);
    const double rho = (y0 - yi) / den;
    if (rho < 0) {
      if (is_converged(g, delta)) {
        *ok = true;
        return LGS_OK;
      }
      g->lm_lambda = nu * g->lm_lambda;
      nu = 2 * nu;
      continue;
    }
    memcpy(x0, xi, sizeof(xi));
    g->lm_lambda = g->lm_lambda * std::max(1.0 / 3.0, 1 - std::pow(2 * rho - 1, 3));
    memcpy(g->final_hessian, H, sizeof(H));
    *ok = true;
    return LGS_OK;
  }
  *ok = false;
  return LGS_OK;
}

int set_cloud(lgs_gicp* g, std::shared_ptr<GicpCloud>* slot, const void* pts, int64_t n, int32_t stride, bool on_device) {
  // a bundle nobody else holds (no swap partner, no exported alias) is recycled with its device buffers: steady-state
  // calls never reach cudaMalloc / cudaFree, which would serialise every stream of the device
  std::shared_ptr<GicpCloud> c;
  if (*slot && slot->use_count() == 1 && (g->source != g->target)) {
    c = *slot;
    c->nn_ready = false;
    c->covs_ready = false;
    c->covs_user = false;
    c->covs_lazy = false;
  } else {
    c = std::make_shared<GicpCloud>();
  }
  LGS_TRY(load_cloud(g->ctx, pts, n, stride, on_device, &c->pts));
  c->n = n;
  *slot = c;
  return LGS_OK;
}

}  // namespace

namespace lgs {
int gicp_align_impl(lgs_gicp* g, const float* guess16, lgs_align_result* res) {
  memset(res, 0, sizeof(*res));
  LGS_TRY(use_device(g->ctx));
  LGS_TRY(ensure_ready(g));
  g->linearize_calls = g->error_calls = 0;
  double x0[16];
  identity_d(x0);
  if (guess16)
    for (int r = 0; r < 4; r++)
      for (int c = 0; c < 4; c++) x0[r * 4 + c] = static_cast<double>(guess16[c * 4 + r]);
  g->lm_lambda = -1.0;
  bool converged = false;
  int nr_iterations = 0;
  for (int i = 0; i < g->max_iterations && !converged; i++) {  // LSQ:65-75
    nr_iterations = i;
    double delta[16];
    bool ok = false;
    LGS_TRY(step_lm(g, x0, delta, &ok));
    if (!ok) break;  // "lm not converged!!"
    converged = is_converged(g, delta);
  }
  for (int r = 0; r < 4; r++)
    for (int c = 0; c < 4; c++) g->final_T[c * 4 + r] = static_cast<float>(x0[r * 4 + c]);
  memcpy(res->T, g->final_T, sizeof(float) * 16);
  res->iterations = nr_iterations;
  res->converged = converged ? 1 : 0;
  res->evaluations = g->linearize_calls;
  res->line_search_trials = g->error_calls;
  return LGS_OK;
}

int gicp_fitness_impl(lgs_gicp* g, double max_range, double* fitness) {
  if (!g->source || !g->target) {
    set_error("FastGICP: target and source must be set");
    return LGS_ERR_STATE;
  }
  LGS_TRY(use_device(g->ctx));
  LGS_TRY(g->target->ensure_index(g->ctx));
  return nn_fitness(g->ctx, g->target->nn, g->source->pts.as<float4>(), g->source->n, g->final_T, max_range, fitness);
}
}  // namespace lgs

extern "C" {

int lgs_gicp_create(lgs_ctx* ctx, lgs_gicp** out) {
  LGS_REQUIRE(ctx && out, "null argument");
  lgs_gicp* g = new lgs_gicp;
  g->ctx = ctx;
  *out = g;
  return LGS_OK;
}

void lgs_gicp_destroy(lgs_gicp* g) {
  if (!g) return;
  cudaSetDevice(g->ctx->device);
  cudaStreamSynchronize(g->ctx->stream);
  g->source.reset();
  g->target.reset();
  for (DevBuf* b : {&g->corr, &g->nn_prev, &g->mahal, &g->partials, &g->counter, &g->out_cloud}) b->release();
  delete g;
}

int lgs_gicp_set_correspondence_randomness(lgs_gicp* g, int32_t k) {
  LGS_REQUIRE(g, "null");
  LGS_REQUIRE(k >= 1 && k <= kMaxK, "k must be in [1, 32]");
  g->k = k;
  return LGS_OK;
}
int lgs_gicp_set_max_correspondence_distance(lgs_gicp* g, double d) { LGS_REQUIRE(g, "null"); g->corr_dist_threshold = d; return LGS_OK; }
int lgs_gicp_set_transformation_epsilon(lgs_gicp* g, double e) { LGS_REQUIRE(g, "null"); g->trans_eps = e; return LGS_OK; }
int lgs_gicp_set_rotation_epsilon(lgs_gicp* g, double e) { LGS_REQUIRE(g, "null"); g->rotation_eps = e; return LGS_OK; }
int lgs_gicp_set_maximum_iterations(lgs_gicp* g, int32_t n) { LGS_REQUIRE(g, "null"); g->max_iterations = n; return LGS_OK; }
int lgs_gicp_set_regularization_method(lgs_gicp* g, int32_t m) {
  LGS_REQUIRE(g, "null");
  LGS_REQUIRE(m >= LGS_REG_NONE && m <= LGS_REG_FROBENIUS, "unknown regularization method");
  g->regularization = m;
  return LGS_OK;
}
int lgs_gicp_set_initial_lambda_factor(lgs_gicp* g, double f) { LGS_REQUIRE(g, "null"); g->lm_init_lambda_factor = f; return LGS_OK; }

int lgs_gicp_set_source(lgs_gicp* g, const void* pts, int64_t n, int32_t stride) {
  LGS_REQUIRE(g, "null");
  return set_cloud(g, &g->source, pts, n, stride, false);
}
int lgs_gicp_set_target(lgs_gicp* g, const void* pts, int64_t n, int32_t stride) {
  LGS_REQUIRE(g, "null");
  return set_cloud(g, &g->target, pts, n, stride, false);
}
int lgs_gicp_set_source_dev(lgs_gicp* g, const float* pts_dev, int64_t n) {
  LGS_REQUIRE(g, "null");
  return set_cloud(g, &g->source, pts_dev, n, 16, true);
}
int lgs_gicp_set_target_dev(lgs_gicp* g, const float* pts_dev, int64_t n) {
  LGS_REQUIRE(g, "null");
  return set_cloud(g, &g->target, pts_dev, n, 16, true);
}
int lgs_gicp_swap_source_and_target(lgs_gicp* g) {  // FG:50-57: clouds, trees and covariances travel together
  LGS_REQUIRE(g, "null");
  g->source.swap(g->target);
  return LGS_OK;
}
int lgs_gicp_clear_source(lgs_gicp* g) { LGS_REQUIRE(g, "null"); g->source.reset(); return LGS_OK; }
int lgs_gicp_clear_target(lgs_gicp* g) { LGS_REQUIRE(g, "null"); g->target.reset(); return LGS_OK; }

int lgs_gicp_align(lgs_gicp* g, const float* guess16, lgs_align_result* res, float* out_cloud) {
  LGS_NVTX("lgs_gicp_align");
  LGS_REQUIRE(g && res, "null argument");
  LGS_TRY(gicp_align_impl(g, guess16, res));
  if (out_cloud) LGS_TRY(write_aligned_cloud(g->ctx, g->source->pts.as<float4>(), g->source->n, g->final_T, &g->out_cloud, out_cloud));  // LSQ:77-78
  return LGS_OK;
}

int lgs_gicp_fitness(lgs_gicp* g, double max_range, double* fitness) {
  LGS_NVTX("lgs_gicp_fitness");
  LGS_REQUIRE(g && fitness, "null argument");
  return gicp_fitness_impl(g, max_range, fitness);
}

int lgs_gicp_final_hessian(lgs_gicp* g, double* H36) {
  LGS_REQUIRE(g && H36, "null argument");
  memcpy(H36, g->final_hessian, sizeof(g->final_hessian));
  return LGS_OK;
}

int lgs_gicp_export_covariances(lgs_gicp* g, int32_t which, double* covs) {
  LGS_REQUIRE(g && covs, "null argument");
  std::shared_ptr<GicpCloud> c = which == 0 ? g->source : g->target;
  if (!c) {
    set_error("lgs_gicp_export_covariances: cloud not set");
    return LGS_ERR_STATE;
  }
  LGS_TRY(use_device(g->ctx));
  LGS_TRY(c->ensure_covariances(g->ctx, g->k, g->regularization));
  if (c->n) {
    LGS_CUDA(cudaMemcpyAsync(covs, c->covs.p, static_cast<size_t>(c->n) * 72, cudaMemcpyDeviceToHost, g->ctx->stream));
    LGS_CUDA(cudaStreamSynchronize(g->ctx->stream));
  }
  return LGS_OK;
}

// evaluateCost (LSQ:48-50): compute_error at the given pose with the correspondences and Mahalanobis matrices of the
// last linearisation (FG:214-237 reads them as they are)
int lgs_gicp_evaluate_cost(lgs_gicp* g, const float* T16, double* cost) {
  LGS_REQUIRE(g && T16 && cost, "null argument");
  if (!g->source || !g->target || g->linearize_calls == 0) {
    set_error("lgs_gicp_evaluate_cost: no linearisation yet (call align or lgs_gicp_linearize first)");
    return LGS_ERR_STATE;
  }
  LGS_TRY(use_device(g->ctx));
  double T[16];
  for (int r = 0; r < 4; r++)
    for (int c = 0; c < 4; c++) T[r * 4 + c] = static_cast<double>(T16[c * 4 + r]);  // Isometry3d(relative_pose.cast<double>())
  const int keep = g->error_calls;
  const int rc = compute_error(g, T, cost);
  g->error_calls = keep;
  return rc;
}

// setSourceCovariances / setTargetCovariances (FG:93-101): the vector is taken as it is; as in computeTransformation
// (FG:104-109) it is used only when its size equals the cloud's, otherwise the covariances are computed at align time
int lgs_gicp_set_covariances(lgs_gicp* g, int32_t which, const double* covs, int64_t n) {
  LGS_REQUIRE(g && (covs || n == 0), "null argument");
  std::shared_ptr<GicpCloud> c = which == 0 ? g->source : g->target;
  if (!c || n != c->n || n == 0) {
    if (c) c->covs_ready = c->covs_user = false;
    return LGS_OK;
  }
  LGS_TRY(use_device(g->ctx));
  LGS_TRY(c->covs.reserve(static_cast<size_t>(n) * 72));
  LGS_CUDA(cudaMemcpyAsync(c->covs.p, covs, static_cast<size_t>(n) * 72, cudaMemcpyHostToDevice, g->ctx->stream));
  LGS_CUDA(cudaStreamSynchronize(g->ctx->stream));  // the caller's buffer is pageable and may go away
  c->covs_ready = true;
  c->covs_user = true;
  return LGS_OK;
}

int lgs_gicp_linearize(lgs_gicp* g, const double* T, double* cost, double* H36, double* b6, int32_t* correspondences) {
  LGS_REQUIRE(g && T && cost, "null argument");
  LGS_TRY(use_device(g->ctx));
  LGS_TRY(ensure_ready(g));
  LGS_TRY(linearize(g, T, cost, H36, b6));
  if (correspondences && g->source->n) {
    LGS_CUDA(cudaMemcpyAsync(correspondences, g->corr.p, static_cast<size_t>(g->source->n) * 4, cudaMemcpyDeviceToHost, g->ctx->stream));
    LGS_CUDA(cudaStreamSynchronize(g->ctx->stream));
  }
  return LGS_OK;
}

}  // extern "C"
