// One registration handle of a given LGS_METHOD_* on a context, for the drivers that compose registrations (the
// loop-closure batch, the odometry loop).  Outside ndt.cu, gicp.cu, gicp_bfgs.cu and icp.cu this is the only code that
// knows which lgs_<method>_* call belongs to each step of a method's lifecycle.
#pragma once
#include <vector>

#include "keyframes.cuh"

namespace lgs {

// The settings the drivers apply, every default already resolved by the caller; each method reads its own subset.  The
// fields are in the order of lgs_batch_params and lgs_odometry_params.
struct MatcherSettings {
  int32_t max_iterations;
  double transformation_epsilon;
  double max_correspondence_distance;
  int32_t k_correspondences;
  float ndt_resolution;
  double ndt_step_size;
  int32_t max_optimizer_iterations;
  double euclidean_fitness_epsilon;
};

struct Matcher {
  int method = -1;  // -1: no handle
  union { lgs_ndt* ndt = nullptr; lgs_gicp* gicp; lgs_icp* icp; lgs_gicp_omp* gomp; };
  lgs_ctx* ctx = nullptr;
  DevBuf poses, target;  // set_target_keyframes of the methods without an incremental key-frame target

  Matcher() = default;
  Matcher(const Matcher&) = delete;
  Matcher& operator=(const Matcher&) = delete;
  ~Matcher() { destroy(); }

  int create(lgs_ctx* c, int m) {
    ctx = c;
    method = m;
    switch (m) {
      case LGS_METHOD_NDT: return lgs_ndt_create(c, &ndt);
      case LGS_METHOD_GICP: return lgs_gicp_create(c, &gicp);
      case LGS_METHOD_ICP: return lgs_icp_create(c, &icp);
      default: return lgs_gicp_omp_create(c, &gomp);
    }
  }
  void destroy() {
    switch (method) {
      case LGS_METHOD_NDT: lgs_ndt_destroy(ndt); break;
      case LGS_METHOD_GICP: lgs_gicp_destroy(gicp); break;
      case LGS_METHOD_ICP: lgs_icp_destroy(icp); break;
      case LGS_METHOD_GICP_OMP: lgs_gicp_omp_destroy(gomp); break;
    }
    method = -1;
    ndt = nullptr;
    poses.release();
    target.release();
  }
  int configure(const MatcherSettings& s) {
    switch (method) {
      case LGS_METHOD_NDT:
        LGS_TRY(lgs_ndt_set_resolution(ndt, s.ndt_resolution));
        LGS_TRY(lgs_ndt_set_step_size(ndt, s.ndt_step_size));
        LGS_TRY(lgs_ndt_set_transformation_epsilon(ndt, s.transformation_epsilon));
        return lgs_ndt_set_maximum_iterations(ndt, s.max_iterations);
      case LGS_METHOD_GICP:
        LGS_TRY(lgs_gicp_set_correspondence_randomness(gicp, s.k_correspondences));
        LGS_TRY(lgs_gicp_set_max_correspondence_distance(gicp, s.max_correspondence_distance));
        LGS_TRY(lgs_gicp_set_transformation_epsilon(gicp, s.transformation_epsilon));
        return lgs_gicp_set_maximum_iterations(gicp, s.max_iterations);
      case LGS_METHOD_ICP:
        LGS_TRY(lgs_icp_set_maximum_iterations(icp, s.max_iterations));
        LGS_TRY(lgs_icp_set_transformation_epsilon(icp, s.transformation_epsilon));
        LGS_TRY(lgs_icp_set_max_correspondence_distance(icp, s.max_correspondence_distance));
        LGS_TRY(lgs_icp_set_euclidean_fitness_epsilon(icp, s.euclidean_fitness_epsilon));
        return lgs_icp_set_transformation_rotation_epsilon(icp, 0.0);
      default:
        LGS_TRY(lgs_gicp_omp_set_correspondence_randomness(gomp, s.k_correspondences));
        LGS_TRY(lgs_gicp_omp_set_max_correspondence_distance(gomp, s.max_correspondence_distance));
        LGS_TRY(lgs_gicp_omp_set_transformation_epsilon(gomp, s.transformation_epsilon));
        LGS_TRY(lgs_gicp_omp_set_maximum_iterations(gomp, s.max_iterations));
        return lgs_gicp_omp_set_maximum_optimizer_iterations(gomp, s.max_optimizer_iterations);
    }
  }
  int set_target_dev(const float* pts, int64_t n) {
    switch (method) {
      case LGS_METHOD_NDT: return lgs_ndt_set_target_dev(ndt, pts, n);
      case LGS_METHOD_GICP: return lgs_gicp_set_target_dev(gicp, pts, n);
      case LGS_METHOD_ICP: return lgs_icp_set_target_dev(icp, pts, n);
      default: return lgs_gicp_omp_set_target_dev(gomp, pts, n);
    }
  }
  // the target is the key frames ids[], transformed by their poses and concatenated in that order
  int set_target_keyframes(lgs_keyframes* kf, const std::vector<int32_t>& ids) {
    const int32_t n_ids = static_cast<int32_t>(ids.size());
    if (method == LGS_METHOD_NDT) return lgs_ndt_set_target_keyframes(ndt, kf, ids.data(), n_ids, nullptr);
    int64_t n = 0;
    LGS_TRY(keyframes_assemble_into(kf, ctx, ids.data(), n_ids, &poses, &target, &n));
    return set_target_dev(target.as<float>(), n);
  }
  int set_source(const void* pts, int64_t n, int32_t stride) {
    switch (method) {
      case LGS_METHOD_NDT: return lgs_ndt_set_source(ndt, pts, n, stride);
      case LGS_METHOD_GICP: return lgs_gicp_set_source(gicp, pts, n, stride);
      case LGS_METHOD_ICP: return lgs_icp_set_source(icp, pts, n, stride);
      default: return lgs_gicp_omp_set_source(gomp, pts, n, stride);
    }
  }
  int set_source_dev(const float* pts, int64_t n) {
    switch (method) {
      case LGS_METHOD_NDT: return lgs_ndt_set_source_dev(ndt, pts, n);
      case LGS_METHOD_GICP: return lgs_gicp_set_source_dev(gicp, pts, n);
      case LGS_METHOD_ICP: return lgs_icp_set_source_dev(icp, pts, n);
      default: return lgs_gicp_omp_set_source_dev(gomp, pts, n);
    }
  }
  // ICP keeps its convergence criteria across aligns (PCL); a fresh criteria object makes a problem's result independent
  // of the problems before it
  int reset_between_problems() { return method == LGS_METHOD_ICP ? lgs_icp_reset_convergence_criteria(icp) : LGS_OK; }
  int align(const float* guess16, lgs_align_result* rec) {
    switch (method) {
      case LGS_METHOD_NDT: return lgs_ndt_align(ndt, guess16, rec, nullptr);
      case LGS_METHOD_GICP: return lgs_gicp_align(gicp, guess16, rec, nullptr);
      case LGS_METHOD_ICP: return lgs_icp_align(icp, guess16, rec, nullptr);
      default: return lgs_gicp_omp_align(gomp, guess16, rec, nullptr);
    }
  }
  int fitness(double max_range, double* f) {
    switch (method) {
      case LGS_METHOD_NDT: return lgs_ndt_fitness(ndt, max_range, f);
      case LGS_METHOD_GICP: return lgs_gicp_fitness(gicp, max_range, f);
      case LGS_METHOD_ICP: return lgs_icp_fitness(icp, max_range, f);
      default: return lgs_gicp_omp_fitness(gomp, max_range, f);
    }
  }
};

}  // namespace lgs
