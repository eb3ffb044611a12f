// pcl::IterativeClosestPoint<PointXYZI, PointXYZI> behind pcl::Registration: the default loop-closure method of the graph
// SLAM node (graph_based_slam.param.yaml:9, constructed at GBS:142-151).  PCL is un-vendored; the algorithm is PCL
// 1.12's icp.hpp (computeTransformation), correspondence_estimation.hpp (determineCorrespondences),
// transformation_estimation_svd.hpp -> pcl::umeyama and default_convergence_criteria.hpp, restated.
//
// One kernel per iteration (icp_step_kernel, one warp per source point):
//   p <- transformation_ * p   the in-place transformCloud of the PREVIOUS iteration (icp.hpp), applied while the point
//                              is loaded and written back, so the cloud is read once and written once per iteration;
//   exact 1-NN of p in the target through the implicit BVH; kept unless d2 > max_dist^2;
//   17 f64 sums per kept pair {1, d2, p, q, q p^T} -> warp -> CTA -> fixed-order last-CTA pass -> host mailbox.
// The host turns the sums into Umeyama's R, t (f32 JacobiSVD as in Eigen) and runs the convergence criteria.
// Eigen's f32 column sums / GEMM inside umeyama have no specified order: means and cross-covariance are accumulated
// in f64 and rounded to f32 (same statement as the oracle's).
// Algorithmic bytes per iteration: 16 (read p) + 16 (write p) + 16 (matched q) per source point; the BVH walk is L2-latency bound.
#include <algorithm>
#include <cmath>
#include <limits>

#include "math.cuh"
#include "nn.cuh"
#include "persist.cuh"
#include "reduce.cuh"

namespace lgs {

constexpr int kIcpBlock = 256;
constexpr int kIcpSums = 17;

struct IcpParams {
  float T[16];       // column-major transform applied to every point before the search
  int apply;         // 0: T is the identity, the cloud is not rewritten
  int use_seed;      // nn_prev holds the neighbours of the previous iteration
  double max_dist2;
};

__device__ __forceinline__ void icp_step_body(const NNView& tv, const float4* __restrict__ tgt, float4* __restrict__ cloud, int* __restrict__ nn_prev, int n,
                                              const IcpParams& P, double* __restrict__ partials, unsigned* __restrict__ counter, const Mailbox& mb) {
  __shared__ double sm[kIcpBlock / 32][kIcpSums];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double acc = 0.0;  // lane k < 17 owns sum k of this warp
  for (int i = blockIdx.x * (kIcpBlock / 32) + warp; i < n; i += gridDim.x * (kIcpBlock / 32)) {
    float4 p = cloud[i];
    if (P.apply) {
      const float3 t = transform_pcl(P.T, p.x, p.y, p.z);
      p = make_float4(t.x, t.y, t.z, p.w);
      if (lane == 0) cloud[i] = p;
    }
    float d2;
    int id;
    // seeded with the previous iteration's neighbour (the cloud moved by one small transformation since)
    int seed = P.use_seed ? nn_prev[i] : -1;
    if (seed >= tv.n) seed = -1;  // the 'nothing found' sentinel of an empty index
    float seed_d = 0.f;
    if (seed >= 0) seed_d = nn_dist2(p.x, p.y, p.z, __ldg(tgt + seed));
    nn_search1_warp_seeded(tv, p.x, p.y, p.z, lane, seed_d, seed, d2, id);
    if (lane == 0) nn_prev[i] = id;
    if (id < 0 || static_cast<double>(d2) > P.max_dist2) continue;  // warp-uniform
    const float4 q = __ldg(tgt + id);  // id is the ORIGINAL index of the matched target point
    const double pv[3] = {static_cast<double>(p.x), static_cast<double>(p.y), static_cast<double>(p.z)};
    const double qv[3] = {static_cast<double>(q.x), static_cast<double>(q.y), static_cast<double>(q.z)};
    double term;
    if (lane == 0) term = 1.0;
    else if (lane == 1) term = static_cast<double>(d2);
    else if (lane < 5) term = pv[lane - 2];
    else if (lane < 8) term = qv[lane - 5];
    else if (lane < 17) term = __dmul_rn(qv[(lane - 8) / 3], pv[(lane - 8) % 3]);
    else term = 0.0;
    acc += term;
  }
  if (lane < kIcpSums) sm[warp][lane] = acc;
  __syncthreads();
  double v = 0;
  if (threadIdx.x < kIcpSums) {
#pragma unroll
    for (int w = 0; w < kIcpBlock / 32; w++) v += sm[w][threadIdx.x];
  }
  // eight groups of 32 threads fold the per-CTA rows, each with four loads in flight (reduce.cuh)
  grid_finish<kIcpSums, kIcpBlock, 8, 4>(v, partials, counter, mb);
}

__global__ void __launch_bounds__(kIcpBlock) icp_step_kernel(const __grid_constant__ NNView tv, const float4* __restrict__ tgt, float4* __restrict__ cloud,
                                                            int* __restrict__ nn_prev, int n, const __grid_constant__ IcpParams P,
                                                            double* __restrict__ partials, unsigned* __restrict__ counter,
                                                            const __grid_constant__ Mailbox mb) {
  icp_step_body(tv, tgt, cloud, nn_prev, n, P, partials, counter, mb);
}

// Persistent form: the grid stays resident for the iterations of one align and receives {transformation_, mailbox token}
// per iteration through the command channel of persist.cuh (the host needs the 17 sums of an iteration before it can
// estimate the next transformation).
struct IcpPose {
  float T[16];
  int apply;  // < 0: end of the run
  int use_seed;
  unsigned long long token;
};
using IcpSession = ResidentSession<IcpPose>;
constexpr int kIcpWords = IcpSession::kWords;
constexpr int kIcpResident = 4;  // CTAs per SM of the persistent grid (all co-resident)

__global__ void __launch_bounds__(kIcpBlock, kIcpResident) icp_persistent_kernel(const __grid_constant__ NNView tv, const float4* __restrict__ tgt,
                                                                                float4* __restrict__ cloud, int* __restrict__ nn_prev, int n, double max_dist2,
                                                                                double* __restrict__ partials, unsigned* __restrict__ counter,
                                                                                MailboxRecord* mailbox, const IcpSession::Host* __restrict__ cmd_host,
                                                                                IcpSession::Dev* __restrict__ cmd_dev, unsigned long long first_seq) {
  __shared__ __align__(16) IcpPose pose;
  __shared__ IcpParams P;
  __shared__ int give_up;
  if (threadIdx.x == 0) give_up = 0;
  __syncthreads();
  for (unsigned long long seq = first_seq;; seq++) {
    if (!persist_receive<kIcpWords, kIcpBlock>(cmd_host, cmd_dev, seq, reinterpret_cast<unsigned long long*>(&pose), &give_up)) return;
    if (pose.apply < 0) return;
    if (threadIdx.x < 16) P.T[threadIdx.x] = pose.T[threadIdx.x];
    if (threadIdx.x == 0) {
      P.apply = pose.apply;
      P.use_seed = pose.use_seed;
      P.max_dist2 = max_dist2;
    }
    __syncthreads();
    Mailbox mb;
    mb.r = mailbox;
    mb.token = pose.token;
    icp_step_body(tv, tgt, cloud, nn_prev, n, P, partials, counter, mb);
    __syncthreads();
  }
}

}  // namespace lgs

using namespace lgs;

struct lgs_icp {
  lgs_ctx* ctx = nullptr;
  // pcl::Registration / pcl::IterativeClosestPoint defaults
  int max_iterations = 10;
  double trans_eps = 0.0, rot_eps = 0.0;
  double fitness_eps = -std::numeric_limits<double>::max();
  double corr_dist_threshold = 1.3407807929942596e154;  // sqrt(DBL_MAX)
  int min_correspondences = 3;
  DevBuf source, target, target_copy, cloud, nn_prev, partials, state, out_cloud;
  bool have_seed = false;  // nn_prev belongs to the working cloud of the running align
  int64_t n_source = 0, n_target = 0;
  NNIndex nn;
  bool nn_ready = false;
  float final_T[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
  int convergence_state = 0;
  double last_mse = 0;
  int64_t last_correspondences = 0;
  // pcl::registration::DefaultConvergenceCriteria lives in the ICP object: correspondences_prev_mse_ and the
  // similar-transforms counter are set in its constructor only, so the first iteration of a second align on the same
  // object is compared with the last MSE of the align before (the reference re-uses one registration_ for every loop
  // closure, GBS:145-148).  lgs_icp_reset_convergence_criteria gives the state of a freshly constructed object.
  double crit_prev_mse = std::numeric_limits<double>::max();
  int crit_state = 0, crit_similar = 0;
  IcpSession session{IcpPose{{}, -1, 0, 0}};  // persistent evaluator (inside lgs_icp_align only)
};

namespace {

enum { kNotConverged = 0, kIterations = 1, kTransform = 2, kAbsMse = 3, kRelMse = 4, kNoCorrespondences = 5 };

float det3f(const float* m) {
  return m[0] * (m[4] * m[8] - m[5] * m[7]) - m[1] * (m[3] * m[8] - m[5] * m[6]) + m[2] * (m[3] * m[7] - m[4] * m[6]);
}

// pcl::umeyama(src, dst, false) from {n, -, sum p, sum q, sum q p^T}
void umeyama(const double* s, float* T) {
  const double n = s[0];
  float pm[3], qm[3], sigma[9], U[9], S[3], V[9], R[9];
  for (int a = 0; a < 3; a++) {
    pm[a] = static_cast<float>(s[2 + a] / n);
    qm[a] = static_cast<float>(s[5 + a] / n);
  }
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) sigma[r * 3 + c] = static_cast<float>(s[8 + r * 3 + c] / n - (s[5 + r] / n) * (s[2 + c] / n));
  m::svd_jacobi<3, float>(sigma, U, S, V);
  const float s2 = det3f(U) * det3f(V) < 0 ? -1.f : 1.f;
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) R[r * 3 + c] = ((U[r * 3] * 1.f) * V[c * 3] + (U[r * 3 + 1] * 1.f) * V[c * 3 + 1]) + (U[r * 3 + 2] * s2) * V[c * 3 + 2];
  identity16f(T);
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) T[c * 4 + r] = R[r * 3 + c];
  for (int r = 0; r < 3; r++) T[12 + r] = qm[r] - ((R[r * 3] * pm[0] + R[r * 3 + 1] * pm[1]) + R[r * 3 + 2] * pm[2]);
}

// pcl::registration::DefaultConvergenceCriteria::hasConverged
struct Criteria {
  int max_iterations, similar = 0, max_similar = 0, state = kNotConverged;
  double rot_thr, trans_thr, rel_thr, abs_thr = 1e-12;
  double prev_mse = std::numeric_limits<double>::max();
  bool check(int iterations, const float* T, double mse) {
    if (state != kNotConverged) {
      similar = 0;
      state = kNotConverged;
    }
    bool is_similar = false;
    if (iterations >= max_iterations) {
      state = kIterations;
      return true;
    }
    const double cos_angle = 0.5 * (T[0] + T[5] + T[10] - 1);
    const double translation_sqr = T[12] * T[12] + T[13] * T[13] + T[14] * T[14];
    auto hit = [&](int why) {
      if (similar >= max_similar) {
        state = why;
        return true;
      }
      is_similar = true;
      return false;
    };
    if (cos_angle >= rot_thr && translation_sqr <= trans_thr && hit(kTransform)) return true;
    if (std::fabs(mse - prev_mse) < abs_thr && hit(kAbsMse)) return true;
    if (std::fabs(mse - prev_mse) / prev_mse < rel_thr && hit(kRelMse)) return true;
    similar = is_similar ? similar + 1 : 0;
    prev_mse = mse;
    return false;
  }
};

int step_grid(int64_t n) { return std::max(1, std::min(grid_for(n, kIcpBlock / 32), kNumSMs * 4)); }

int ensure_ready(lgs_icp* g) {
  if (g->n_source == 0 || g->n_target == 0) {
    set_error("IterativeClosestPoint: setInputSource and setInputTarget must be called with non-empty clouds first");
    return LGS_ERR_STATE;
  }
  if (!g->nn_ready) {
    LGS_TRY(g->nn.build(g->ctx, g->target.as<float4>(), g->n_target));
    g->nn_ready = true;
  }
  LGS_TRY(g->cloud.reserve(static_cast<size_t>(g->n_source) * 16));
  LGS_TRY(g->nn_prev.reserve(static_cast<size_t>(g->n_source) * 4));
  LGS_TRY(g->partials.reserve(static_cast<size_t>(step_grid(g->n_source)) * kIcpSums * 8));
  if (!g->state.p) {
    LGS_TRY(g->state.reserve(64));
    LGS_CUDA(cudaMemsetAsync(g->state.p, 0, 64, g->ctx->stream));
  }
  return LGS_OK;
}

// transforms the working cloud by T (unless null) and returns the 17 sums of the correspondences found after it
int step(lgs_icp* g, const float* T, double* sums) {
  lgs_ctx* ctx = g->ctx;
  IcpParams P;
  P.apply = T ? 1 : 0;
  if (T) memcpy(P.T, T, sizeof(P.T)); else identity16f(P.T);
  P.max_dist2 = g->corr_dist_threshold * g->corr_dist_threshold;
  P.use_seed = g->have_seed ? 1 : 0;
  g->have_seed = true;
  Mailbox mb;
  LGS_TRY(mailbox_next(ctx, &mb));
  const int grid = step_grid(g->n_source);
  const int n = static_cast<int>(g->n_source);
  LGS_TRY(g->session.open(ctx, grid <= kNumSMs * kIcpResident, [&](const IcpSession::Host* host, IcpSession::Dev* dev, unsigned long long first_seq) {
    icp_persistent_kernel<<<grid, kIcpBlock, 0, ctx->stream>>>(g->nn.view(), g->target.as<float4>(), g->cloud.as<float4>(), g->nn_prev.as<int>(), n, P.max_dist2,
                                                             g->partials.as<double>(), g->state.as<unsigned>(), mb.r, host, dev, first_seq);
  }));
  if (g->session.active) {
    IcpPose pose;
    memcpy(pose.T, P.T, sizeof(pose.T));
    pose.apply = P.apply;
    pose.use_seed = P.use_seed;
    pose.token = mb.token;
    g->session.send(pose);
    const int rc = mailbox_wait(ctx, mb, kIcpSums, sums);
    if (rc == LGS_OK) return LGS_OK;
    // The grid gave up (command time-out).  It may have transformed part of the working cloud already, so this align
    // cannot be continued with plain launches: lgs_icp_align runs it again from the source cloud.
    if (g->session.recover(ctx, g->state.as<unsigned>()))
      set_error("IterativeClosestPoint: the resident evaluator timed out waiting for the host; call align again (plain launches from now on)");
    return rc;
  }
  icp_step_kernel<<<grid, kIcpBlock, 0, ctx->stream>>>(g->nn.view(), g->target.as<float4>(), g->cloud.as<float4>(), g->nn_prev.as<int>(), n, P, g->partials.as<double>(),
                                                      g->state.as<unsigned>(), mb);
  ctx->launches++;
  LGS_CUDA(cudaGetLastError());
  return mailbox_wait(ctx, mb, kIcpSums, sums);
}

int set_cloud(lgs_icp* g, DevBuf* dst, int64_t* cnt, const void* pts, int64_t n, int32_t stride, bool on_device) {
  LGS_TRY(load_cloud(g->ctx, pts, n, stride, on_device, dst));
  *cnt = n;
  return LGS_OK;
}

}  // namespace

extern "C" {

int lgs_icp_create(lgs_ctx* ctx, lgs_icp** out) {
  LGS_REQUIRE(ctx && out, "null argument");
  lgs_icp* g = new lgs_icp;
  g->ctx = ctx;
  *out = g;
  return LGS_OK;
}

void lgs_icp_destroy(lgs_icp* g) {
  if (!g) return;
  g->session.release(g->ctx);
  for (DevBuf* b : {&g->source, &g->target, &g->target_copy, &g->cloud, &g->nn_prev, &g->partials, &g->state, &g->out_cloud}) b->release();
  g->nn.release();
  delete g;
}

int lgs_icp_set_max_correspondence_distance(lgs_icp* g, double d) { LGS_REQUIRE(g, "null"); g->corr_dist_threshold = d; return LGS_OK; }
int lgs_icp_set_maximum_iterations(lgs_icp* g, int32_t n) { LGS_REQUIRE(g, "null"); g->max_iterations = n; return LGS_OK; }
int lgs_icp_set_transformation_epsilon(lgs_icp* g, double e) { LGS_REQUIRE(g, "null"); g->trans_eps = e; return LGS_OK; }
int lgs_icp_set_transformation_rotation_epsilon(lgs_icp* g, double e) { LGS_REQUIRE(g, "null"); g->rot_eps = e; return LGS_OK; }
int lgs_icp_set_euclidean_fitness_epsilon(lgs_icp* g, double e) { LGS_REQUIRE(g, "null"); g->fitness_eps = e; return LGS_OK; }
int lgs_icp_reset_convergence_criteria(lgs_icp* g) {
  LGS_REQUIRE(g, "null");
  g->crit_prev_mse = std::numeric_limits<double>::max();
  g->crit_state = 0;
  g->crit_similar = 0;
  return LGS_OK;
}

int lgs_icp_set_source(lgs_icp* g, const void* pts, int64_t n, int32_t stride) {
  LGS_REQUIRE(g, "null");
  return set_cloud(g, &g->source, &g->n_source, pts, n, stride, false);
}
int lgs_icp_set_source_dev(lgs_icp* g, const float* pts_dev, int64_t n) {
  LGS_REQUIRE(g, "null");
  return set_cloud(g, &g->source, &g->n_source, pts_dev, n, 16, true);
}
int lgs_icp_set_target(lgs_icp* g, const void* pts, int64_t n, int32_t stride) {
  LGS_REQUIRE(g, "null");
  g->nn_ready = false;
  return set_cloud(g, &g->target, &g->n_target, pts, n, stride, false);
}
int lgs_icp_set_target_dev(lgs_icp* g, const float* pts_dev, int64_t n) {
  LGS_REQUIRE(g, "null");
  g->nn_ready = false;
  return set_cloud(g, &g->target, &g->n_target, pts_dev, n, 16, true);
}

// pcl::Registration::align + IterativeClosestPoint::computeTransformation
static int icp_align(lgs_icp* g, const float* guess16, lgs_align_result* res, float* out_cloud);

int lgs_icp_align(lgs_icp* g, const float* guess16, lgs_align_result* res, float* out_cloud) {
  LGS_NVTX("lgs_icp_align");
  LGS_REQUIRE(g && res, "null argument");
  const bool was_broken = g->session.broken;
  const int rc = icp_align(g, guess16, res, out_cloud);
  // the resident grid timed out mid-align (see step()): run the whole align again, with plain launches now
  if (rc != LGS_OK && g->session.broken && !was_broken) return icp_align(g, guess16, res, out_cloud);
  return rc;
}

static int icp_align(lgs_icp* g, const float* guess16, lgs_align_result* res, float* out_cloud) {
  SessionScope scope(g->session);
  memset(res, 0, sizeof(*res));
  LGS_TRY(use_device(g->ctx));
  LGS_TRY(ensure_ready(g));
  cudaStream_t st = g->ctx->stream;
  float guess[16], T[16];
  identity16f(guess);
  if (guess16) memcpy(guess, guess16, sizeof(guess));
  memcpy(g->final_T, guess, sizeof(guess));
  bool is_identity = true;
  for (int i = 0; i < 16; i++)
    if (guess[i] != ((i % 5 == 0) ? 1.0f : 0.0f)) is_identity = false;
  g->have_seed = false;  // the seeds belong to one align (one working cloud, one target)
  // input_transformed = guess * input (or a copy)
  LGS_CUDA(cudaMemcpyAsync(g->cloud.p, g->source.p, static_cast<size_t>(g->n_source) * 16, cudaMemcpyDeviceToDevice, st));
  identity16f(T);
  Criteria crit;
  crit.prev_mse = g->crit_prev_mse;
  crit.state = g->crit_state;
  crit.similar = g->crit_similar;
  crit.max_iterations = g->max_iterations;
  crit.rel_thr = g->fitness_eps;
  crit.trans_thr = g->trans_eps;
  crit.rot_thr = g->rot_eps > 0 ? g->rot_eps : 1.0 - g->trans_eps;
  int nr_iterations = 0;
  bool converged = false;
  const float* pending = is_identity ? nullptr : guess;  // the transform the next step applies to the working cloud first
  double sums[kIcpSums];
  do {
    LGS_TRY(step(g, pending, sums));
    if (static_cast<int>(sums[0]) < g->min_correspondences) {  // "Not enough correspondences found"
      crit.state = kNoCorrespondences;
      converged = false;
      pending = nullptr;
      break;
    }
    umeyama(sums, T);
    pending = T;  // transformCloud(*input_transformed, *input_transformed, transformation_): fused into the next step
    mul4f(T, g->final_T, g->final_T);
    ++nr_iterations;
    g->last_correspondences = static_cast<int64_t>(sums[0]);
    g->last_mse = sums[1] / sums[0];
    converged = crit.check(nr_iterations, T, g->last_mse);
  } while (crit.state == kNotConverged);
  g->session.close();  // before the output cloud's kernel
  g->convergence_state = crit.state;
  g->crit_prev_mse = crit.prev_mse;
  g->crit_state = crit.state;
  g->crit_similar = crit.similar;
  memcpy(res->T, g->final_T, sizeof(g->final_T));
  res->iterations = nr_iterations;
  res->converged = converged ? 1 : 0;
  res->evaluations = nr_iterations;
  res->line_search_trials = crit.state;
  res->trans_probability = g->last_mse;
  if (out_cloud) LGS_TRY(write_aligned_cloud(g->ctx, g->source.as<float4>(), g->n_source, g->final_T, &g->out_cloud, out_cloud));
  return LGS_OK;
}

int lgs_icp_fitness(lgs_icp* g, double max_range, double* fitness) {
  LGS_REQUIRE(g && fitness, "null argument");
  LGS_TRY(use_device(g->ctx));
  LGS_TRY(ensure_ready(g));
  return nn_fitness(g->ctx, g->nn, g->source.as<float4>(), g->n_source, g->final_T, max_range, fitness);
}

// parity hook: one correspondence + Umeyama step on guess * source: the 17 sums {n, sum d2, sum p, sum q, sum q p^T} and the
// estimated transformation_; *ok = 0 when fewer than min_number_correspondences pairs were found
int lgs_icp_step(lgs_icp* g, const float* guess16, double* sums17, float* T16, int32_t* ok) {
  LGS_REQUIRE(g && guess16 && sums17 && T16 && ok, "null argument");
  LGS_TRY(use_device(g->ctx));
  LGS_TRY(ensure_ready(g));
  LGS_CUDA(cudaMemcpyAsync(g->cloud.p, g->source.p, static_cast<size_t>(g->n_source) * 16, cudaMemcpyDeviceToDevice, g->ctx->stream));
  g->have_seed = false;
  LGS_TRY(step(g, guess16, sums17));
  *ok = static_cast<int>(sums17[0]) >= g->min_correspondences ? 1 : 0;
  identity16f(T16);
  if (*ok) umeyama(sums17, T16);
  return LGS_OK;
}

}  // extern "C"
