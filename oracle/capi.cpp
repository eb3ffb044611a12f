// ORACLE (test infrastructure).  Flat C entry points for ctypes (tests/, smoke(), bench cpu_baseline only).
#include <chrono>
#include <cstring>
#ifdef _OPENMP
#include <omp.h>
#endif

#include "linalg.hpp"
#include "oracle.hpp"

using namespace lgs_oracle;

extern "C" {

int orc_max_threads() {
#ifdef _OPENMP
  return omp_get_max_threads();
#else
  return 1;
#endif
}

// ---- prefilter -------------------------------------------------------------------------------
struct OrcVG {
  VoxelGridResult r;
};
void* orc_vg_run(const float* pts, long n, const float* leaf3, int min_pts, double range_min, const double* box6) {
  OrcVG* h = new OrcVG;
  prefilter_voxel_grid(reinterpret_cast<const P4*>(pts), static_cast<size_t>(n), leaf3, min_pts, range_min, box6, &h->r);
  return h;
}
int orc_vg_status(void* h) { return static_cast<OrcVG*>(h)->r.status; }
long orc_vg_out_n(void* h) { return static_cast<long>(static_cast<OrcVG*>(h)->r.out.size()); }
long orc_vg_n_kept(void* h) { return static_cast<long>(static_cast<OrcVG*>(h)->r.n_kept); }
void orc_vg_get(void* h, float* out_pts, int* out_idx, int* out_count, int* voxel_idx, int* member_rank, int* grid9) {
  VoxelGridResult& r = static_cast<OrcVG*>(h)->r;
  if (out_pts) std::memcpy(out_pts, r.out.data(), r.out.size() * sizeof(P4));
  if (out_idx) std::memcpy(out_idx, r.out_idx.data(), r.out_idx.size() * sizeof(int));
  if (out_count) std::memcpy(out_count, r.out_count.data(), r.out_count.size() * sizeof(int));
  if (voxel_idx) std::memcpy(voxel_idx, r.voxel_idx.data(), r.voxel_idx.size() * sizeof(int));
  if (member_rank) std::memcpy(member_rank, r.member_rank.data(), r.member_rank.size() * sizeof(int));
  if (grid9)
    for (int a = 0; a < 3; a++) {
      grid9[a] = r.min_b[a];
      grid9[3 + a] = r.max_b[a];
      grid9[6 + a] = r.div_b[a];
    }
}
void orc_vg_free(void* h) { delete static_cast<OrcVG*>(h); }

// ---- NDT -------------------------------------------------------------------------------------
void* orc_ndt_create() { return new NDT; }
void orc_ndt_destroy(void* h) { delete static_cast<NDT*>(h); }
void orc_ndt_set_params(void* h, float resolution, double step_size, double trans_eps, int max_iter, double outlier_ratio, int search_method,
                        int num_threads) {
  NDT* n = static_cast<NDT*>(h);
  n->setResolution(resolution);
  n->step_size = step_size;
  n->transformation_epsilon = trans_eps;
  n->max_iterations = max_iter;
  n->outlier_ratio = outlier_ratio;
  n->search_method = search_method;
  if (num_threads > 0) n->num_threads = num_threads;
}
void orc_ndt_set_target(void* h, const float* pts, long n) { static_cast<NDT*>(h)->setInputTarget(reinterpret_cast<const P4*>(pts), n); }
void orc_ndt_set_source(void* h, const float* pts, long n) { static_cast<NDT*>(h)->setInputSource(reinterpret_cast<const P4*>(pts), n); }
void orc_ndt_align(void* h, const float* guess16, float* T16, int* iters, int* converged, double* trans_prob, float* out_cloud, int* stats3) {
  NDT* n = static_cast<NDT*>(h);
  std::vector<P4> out;
  n->align(guess16, &out);
  std::memcpy(T16, n->final_transformation, 16 * sizeof(float));
  *iters = n->nr_iterations;
  *converged = n->converged ? 1 : 0;
  *trans_prob = n->trans_probability;
  if (out_cloud) std::memcpy(out_cloud, out.data(), out.size() * sizeof(P4));
  if (stats3) {
    stats3[0] = n->stats.derivative_evals;
    stats3[1] = n->stats.line_search_trials;
    stats3[2] = n->stats.hessian_recomputes;
  }
}
double orc_ndt_fitness(void* h, double max_range) { return static_cast<NDT*>(h)->getFitnessScore(max_range); }
long orc_ndt_voxel_count(void* h) { return static_cast<long>(static_cast<NDT*>(h)->cells.leaves.size()); }
int orc_ndt_refused(void* h) { return static_cast<NDT*>(h)->cells.refused ? 1 : 0; }
// idx ascending; n = nr_points (-1 when invalidated); mean 3, cov 9, icov 9 (row-major); grid9 = min_b,max_b,div_b
void orc_ndt_export_voxels(void* h, int* idx, int* npts, double* mean, double* cov, double* icov, int* grid9) {
  NDT* n = static_cast<NDT*>(h);
  long k = 0;
  for (auto& kv : n->cells.leaves) {
    if (idx) idx[k] = static_cast<int>(kv.first);
    if (npts) npts[k] = kv.second.nr_points;
    if (mean) std::memcpy(mean + 3 * k, kv.second.mean, 3 * sizeof(double));
    if (cov) std::memcpy(cov + 9 * k, kv.second.cov, 9 * sizeof(double));
    if (icov) std::memcpy(icov + 9 * k, kv.second.icov, 9 * sizeof(double));
    k++;
  }
  if (grid9)
    for (int a = 0; a < 3; a++) {
      grid9[a] = n->cells.min_b[a];
      grid9[3 + a] = n->cells.max_b[a];
      grid9[6 + a] = n->cells.div_b[a];
    }
}
// One derivative evaluation at pose vector p with the source transformed by T (column-major f32).
// mode 0: computeDerivatives(compute_hessian=true); 1: gradient only; 2: computeHessian (f64 path; needs a prior mode-0/1 call for the angle tables)
double orc_ndt_derivatives(void* h, const float* T16, const double* p6, int mode, double* g6, double* H36) {
  NDT* n = static_cast<NDT*>(h);
  n->compute_gauss();
  std::vector<P4> tc(n->source.size());
  for (size_t i = 0; i < tc.size(); i++) tc[i] = transform_point(T16, n->source[i]);
  if (mode == 2) {
    n->computeAngleDerivatives(p6);
    n->computeHessian(H36, tc);
    return 0.0;
  }
  return n->computeDerivatives(g6, H36, tc, p6, mode == 0);
}
void orc_ndt_convert_transform(const double* p6, float* T16) { ndt_convert_transform(p6, T16); }
double orc_ndt_calculate_score(void* h, const float* T16) {
  NDT* n = static_cast<NDT*>(h);
  n->compute_gauss();
  std::vector<P4> tc(n->source.size());
  for (size_t i = 0; i < tc.size(); i++) tc[i] = transform_point(T16, n->source[i]);
  return n->calculateScore(tc);
}

// ---- GICP ------------------------------------------------------------------------------------
void* orc_gicp_create() { return new FastGICP; }
void orc_gicp_destroy(void* h) { delete static_cast<FastGICP*>(h); }
void orc_gicp_set_params(void* h, int k, double max_corr_dist, double trans_eps, double rot_eps, int max_iter, int regularization,
                         int num_threads) {
  FastGICP* g = static_cast<FastGICP*>(h);
  g->k_correspondences = k;
  if (max_corr_dist > 0) g->corr_dist_threshold = max_corr_dist;
  g->transformation_epsilon = trans_eps;
  g->rotation_epsilon = rot_eps;
  g->max_iterations = max_iter;
  g->regularization = regularization;
  if (num_threads > 0) g->num_threads = num_threads;
}
void orc_gicp_set_source(void* h, const float* pts, long n) { static_cast<FastGICP*>(h)->setInputSource(reinterpret_cast<const P4*>(pts), n); }
void orc_gicp_set_target(void* h, const float* pts, long n) { static_cast<FastGICP*>(h)->setInputTarget(reinterpret_cast<const P4*>(pts), n); }
void orc_gicp_swap(void* h) { static_cast<FastGICP*>(h)->swapSourceAndTarget(); }
void orc_gicp_align(void* h, const float* guess16, float* T16, int* iters, int* converged, float* out_cloud, int* stats2) {
  FastGICP* g = static_cast<FastGICP*>(h);
  std::vector<P4> out;
  g->align(guess16, out_cloud ? &out : nullptr);
  std::memcpy(T16, g->final_transformation, 16 * sizeof(float));
  *iters = g->nr_iterations;
  *converged = g->converged ? 1 : 0;
  if (out_cloud) std::memcpy(out_cloud, out.data(), out.size() * sizeof(P4));
  if (stats2) {
    stats2[0] = g->linearize_calls;
    stats2[1] = g->error_calls;
  }
}
double orc_gicp_fitness(void* h, double max_range) { return static_cast<FastGICP*>(h)->getFitnessScore(max_range); }
void orc_gicp_final_hessian(void* h, double* H36) { std::memcpy(H36, static_cast<FastGICP*>(h)->final_hessian, 36 * sizeof(double)); }
// which: 0 source, 1 target.  Computes them if missing.  9 doubles per point, row-major.
void orc_gicp_covariances(void* h, int which, double* covs) {
  FastGICP* g = static_cast<FastGICP*>(h);
  Cloud& c = which == 0 ? *g->source : *g->target;
  if (c.covs.size() != c.pts.size() * 9) g->calculate_covariances(c);
  std::memcpy(covs, c.covs.data(), c.covs.size() * sizeof(double));
}
// evaluateCost (LSQ:48-50): compute_error at Isometry3d(relative_pose.cast<double>()), column-major f32 in
double orc_gicp_evaluate_cost(void* h, const float* T16) {
  FastGICP* g = static_cast<FastGICP*>(h);
  double T[16];
  for (int r = 0; r < 4; r++)
    for (int c = 0; c < 4; c++) T[r * 4 + c] = static_cast<double>(T16[c * 4 + r]);
  const int keep = g->error_calls;
  const double v = g->compute_error(T);
  g->error_calls = keep;
  return v;
}
// setSourceCovariances / setTargetCovariances (FG:93-101): taken as they are; align recomputes them only when the
// size differs from the cloud's (FG:104-109)
void orc_gicp_set_covariances(void* h, int which, const double* covs, long n) {
  FastGICP* g = static_cast<FastGICP*>(h);
  Cloud& c = which == 0 ? *g->source : *g->target;
  c.covs.assign(covs, covs + static_cast<size_t>(n) * 9);
}
// linearize at a row-major f64 transform: returns cost, fills H/b and (optionally) correspondences
double orc_gicp_linearize(void* h, const double* T16_rowmajor, double* H36, double* b6, int* corr) {
  FastGICP* g = static_cast<FastGICP*>(h);
  if (g->source->covs.size() != g->source->pts.size() * 9) g->calculate_covariances(*g->source);
  if (g->target->covs.size() != g->target->pts.size() * 9) g->calculate_covariances(*g->target);
  double c = g->linearize(T16_rowmajor, H36, b6);
  if (corr) std::memcpy(corr, g->correspondences.data(), g->correspondences.size() * sizeof(int));
  return c;
}

// ---- pclomp::GeneralizedIterativeClosestPoint (BFGS) ---------------------------------------------
void* orc_pgicp_create() { return new PclGICP; }
void orc_pgicp_destroy(void* h) { delete static_cast<PclGICP*>(h); }
void orc_pgicp_set_params(void* h, int k, double max_corr_dist, double trans_eps, double rot_eps, int max_iter, int max_inner, double gicp_eps,
                          int num_threads) {
  PclGICP* g = static_cast<PclGICP*>(h);
  g->k_correspondences = k;
  g->corr_dist_threshold = max_corr_dist;
  g->transformation_epsilon = trans_eps;
  g->rotation_epsilon = rot_eps;
  g->max_iterations = max_iter;
  g->max_inner_iterations = max_inner;
  g->gicp_epsilon = gicp_eps;
  if (num_threads > 0) g->num_threads = num_threads;
}
void orc_pgicp_set_source(void* h, const float* pts, long n) { static_cast<PclGICP*>(h)->setInputSource(reinterpret_cast<const P4*>(pts), n); }
void orc_pgicp_set_target(void* h, const float* pts, long n) { static_cast<PclGICP*>(h)->setInputTarget(reinterpret_cast<const P4*>(pts), n); }
// stats5: f, df, fdf calls, total BFGS inner iterations, correspondences of the last outer iteration
void orc_pgicp_align(void* h, const float* guess16, float* T16, int* iters, int* converged, float* out_cloud, int* stats5) {
  PclGICP* g = static_cast<PclGICP*>(h);
  std::vector<P4> out;
  g->align(guess16, out_cloud ? &out : nullptr);
  std::memcpy(T16, g->final_transformation, 16 * sizeof(float));
  *iters = g->nr_iterations;
  *converged = g->converged ? 1 : 0;
  if (out_cloud) std::memcpy(out_cloud, out.data(), out.size() * sizeof(P4));
  if (stats5) {
    stats5[0] = g->f_calls;
    stats5[1] = g->df_calls;
    stats5[2] = g->fdf_calls;
    stats5[3] = g->inner_iterations_total;
    stats5[4] = static_cast<int>(g->corr_src.size());
  }
}
double orc_pgicp_fitness(void* h, double max_range) { return static_cast<PclGICP*>(h)->getFitnessScore(max_range); }
// which: 0 source, 1 target.  Computes them if missing.  9 doubles per point, row-major.
void orc_pgicp_covariances(void* h, int which, double* covs) {
  PclGICP* g = static_cast<PclGICP*>(h);
  if (which == 0) {
    if (g->source_covs.size() != g->source.size() * 9) g->computeCovariances(g->source, g->source_tree, g->source_covs);
    std::memcpy(covs, g->source_covs.data(), g->source_covs.size() * sizeof(double));
  } else {
    if (g->target_covs.size() != g->target.size() * 9) g->computeCovariances(g->target, g->target_tree, g->target_covs);
    std::memcpy(covs, g->target_covs.data(), g->target_covs.size() * sizeof(double));
  }
}
// One outer-iteration set-up at (transformation, guess) followed by the three functor evaluations at x:
// out15 = f(x), df(x)[6], fdf(x) -> f, g[6], number of correspondences.  corr (n_source ints, -1 = none) and
// mahal (n_source x 9 floats) are optional.
void orc_pgicp_functor(void* h, const float* guess16, const float* transformation16, const double* x6, double* out15, int* corr, float* mahal) {
  PclGICP* g = static_cast<PclGICP*>(h);
  if (g->target_covs.size() != g->target.size() * 9) g->computeCovariances(g->target, g->target_tree, g->target_covs);
  if (g->source_covs.size() != g->source.size() * 9) g->computeCovariances(g->source, g->source_tree, g->source_covs);
  g->output.resize(g->source.size());
  for (size_t i = 0; i < g->source.size(); i++) g->output[i] = transform_point(guess16, g->source[i]);
  std::memcpy(g->transformation, transformation16, 16 * sizeof(float));
  g->update_correspondences(guess16);
  out15[0] = g->functor_f(x6);
  g->functor_df(x6, out15 + 1);
  g->functor_fdf(x6, out15[7], out15 + 8);
  out15[14] = static_cast<double>(g->corr_src.size());
  if (corr) {
    for (size_t i = 0; i < g->source.size(); i++) corr[i] = -1;
    for (size_t i = 0; i < g->corr_src.size(); i++) corr[g->corr_src[i]] = g->corr_tgt[i];
  }
  if (mahal) std::memcpy(mahal, g->mahalanobis.data(), g->mahalanobis.size() * sizeof(float));
}

// pcl::transformPointCloud(Matrix4f) (transform_point_cloud of the nodes, LSM:206, GBS:305): out may alias pts
void orc_transform_cloud(const float* pts, long n, const float* T16, float* out) {
  const P4* p = reinterpret_cast<const P4*>(pts);
  P4* o = reinterpret_cast<P4*>(out);
  for (long i = 0; i < n; i++) o[i] = transform_point(T16, p[i]);
}

// ---- pcl::IterativeClosestPoint -------------------------------------------------------------------
void* orc_icp_create() { return new PclICP; }
void orc_icp_destroy(void* h) { delete static_cast<PclICP*>(h); }
void orc_icp_set_params(void* h, double max_corr_dist, int max_iter, double trans_eps, double rot_eps, double fitness_eps, int num_threads) {
  PclICP* g = static_cast<PclICP*>(h);
  g->corr_dist_threshold = max_corr_dist;
  g->max_iterations = max_iter;
  g->transformation_epsilon = trans_eps;
  g->transformation_rotation_epsilon = rot_eps;
  g->euclidean_fitness_epsilon = fitness_eps;
  if (num_threads > 0) g->num_threads = num_threads;
}
void orc_icp_set_source(void* h, const float* pts, long n) { static_cast<PclICP*>(h)->setInputSource(reinterpret_cast<const P4*>(pts), n); }
void orc_icp_set_target(void* h, const float* pts, long n) { static_cast<PclICP*>(h)->setInputTarget(reinterpret_cast<const P4*>(pts), n); }
// stats: {convergence state, correspondences of the last iteration}; mse: MSE of the last iteration
void orc_icp_align(void* h, const float* guess16, float* T16, int* iters, int* converged, float* out_cloud, long* stats2, double* mse) {
  PclICP* g = static_cast<PclICP*>(h);
  std::vector<P4> out;
  g->align(guess16, out_cloud ? &out : nullptr);
  std::memcpy(T16, g->final_transformation, 16 * sizeof(float));
  *iters = g->nr_iterations;
  *converged = g->converged ? 1 : 0;
  if (out_cloud) std::memcpy(out_cloud, out.data(), out.size() * sizeof(P4));
  if (stats2) {
    stats2[0] = g->convergence_state;
    stats2[1] = g->last_correspondences;
  }
  if (mse) *mse = g->last_mse;
}
double orc_icp_fitness(void* h, double max_range) { return static_cast<PclICP*>(h)->getFitnessScore(max_range); }
// one correspondence + umeyama step on guess * source: the 17 sums and the estimated transformation; returns 0 when
// there are fewer than min_number_correspondences
int orc_icp_step(void* h, const float* guess16, double* sums17, float* T16) {
  PclICP* g = static_cast<PclICP*>(h);
  std::vector<P4> cloud(g->source.size());
  for (size_t i = 0; i < cloud.size(); i++) cloud[i] = transform_point(guess16, g->source[i]);
  return g->estimate_step(cloud, sums17, T16) ? 1 : 0;
}

// ---- exact k-NN (tree built per call) -----------------------------------------------------------
void orc_knn(const float* pts, long n, const float* queries, long m, int k, int* idx, float* d2, int num_threads) {
  KdTree t;
  t.build(reinterpret_cast<const P4*>(pts), n);
  const P4* q = reinterpret_cast<const P4*>(queries);
  (void)num_threads;
#pragma omp parallel for num_threads(num_threads > 0 ? num_threads : 1) schedule(static)
  for (long i = 0; i < m; i++) {
    int f = t.knn(q[i], k, idx + i * k, d2 + i * k);
    for (int j = f; j < k; j++) {
      idx[i * k + j] = -1;
      d2[i * k + j] = 0;
    }
  }
}

// ---- the small dense solvers (linalg.hpp), n problems, f64 in and out, row-major ----------------
//   0 jacobi_svd<3>          A[9]        -> U[9], S[3], V[9]
//   1 self_adjoint_eigen3    A[9]        -> w[3], Q[9], ok
//   2 inverse3               A[9]        -> A^-1[9]
//   3 jacobi_svd_solve<6>    H[36], b[6] -> x[6]
//  16 jacobi_svd<3, float>   A[9]        -> U[9], S[3], V[9]   (inputs rounded to float, results widened exactly)
//  17 ldlt_solve6            H[36], b[6] -> x[6]
// Returns 0, or -1 for an unknown op.
int orc_linalg_batch(int op, long n, const double* in, double* out) {
  int nin, nout;
  switch (op) {
    case 0: case 16: nin = 9; nout = 21; break;
    case 1: nin = 9; nout = 13; break;
    case 2: nin = 9; nout = 9; break;
    case 3: case 17: nin = 42; nout = 6; break;
    default: return -1;
  }
  for (long t = 0; t < n; t++) {
    const double* a = in + t * nin;
    double* o = out + t * nout;
    if (op == 0) {
      jacobi_svd<3, double>(a, o, o + 9, o + 12);
    } else if (op == 1) {
      o[12] = self_adjoint_eigen3(a, o, o + 3) ? 1.0 : 0.0;
    } else if (op == 2) {
      inverse3(a, o);
    } else if (op == 3) {
      jacobi_svd_solve<6>(a, a + 36, o);
    } else if (op == 16) {
      float af[9], U[9], S[3], V[9];
      for (int i = 0; i < 9; i++) af[i] = static_cast<float>(a[i]);
      jacobi_svd<3, float>(af, U, S, V);
      for (int i = 0; i < 9; i++) o[i] = U[i];
      for (int i = 0; i < 3; i++) o[9 + i] = S[i];
      for (int i = 0; i < 9; i++) o[12 + i] = V[i];
    } else {
      ldlt_solve6(a, a + 36, o);
    }
  }
  return 0;
}

double orc_fitness(const float* tgt, long nt, const float* src, long ns, const float* T16, double max_range, int num_threads) {
  KdTree t;
  t.build(reinterpret_cast<const P4*>(tgt), nt);
  return fitness_score(t, reinterpret_cast<const P4*>(src), ns, T16, max_range, num_threads > 0 ? num_threads : 1);
}

}  // extern "C"
