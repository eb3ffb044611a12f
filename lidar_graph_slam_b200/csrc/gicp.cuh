// State of the GICP registration object (shared between gicp.cu and batch.cu).
#pragma once
#include <memory>

#include "math.cuh"
#include "nn.cuh"

namespace lgs {

// A cloud with everything fast_gicp keeps next to it: the search structure and the per-point covariances.
// swapSourceAndTarget (FG:50-57) swaps these bundles, which is what makes covariance reuse work.
struct GicpCloud {
  DevBuf pts;
  int64_t n = 0;
  NNIndex nn;
  bool nn_ready = false;
  DevBuf covs;  // n x 9 f64, row-major 3x3 block of the reference's Matrix4d
  bool covs_ready = false;
  int covs_k = 0, covs_reg = -1;
  bool covs_user = false;  // supplied through set*Covariances (FG:93-101): used as they are
  // Lazy covariances (a TARGET whose covariances nobody has asked for yet): fast_gicp computes the k-NN covariance of every
  // target point up front (FG:104-109, 241-298), but an align only ever reads those of the points some source point
  // corresponds to - a third of a 65 000-point sub-map for a 27 000-point scan.  A covariance depends on the cloud alone, so
  // computing it on first use gives the same bits; the k-NN search is the most expensive kernel of the loop-closure batch.
  bool covs_lazy = false;
  DevBuf cov_done, work_list, work_count;  // per point: covariance present; points to compute now; their number
  int ensure_index(lgs_ctx* ctx);
  int ensure_covariances(lgs_ctx* ctx, int k, int regularization);
  int begin_lazy_covariances(lgs_ctx* ctx, int k, int regularization);
  // computes the covariances of the not-yet-covered points among corr[0 .. n_corr) (device array, -1 = none)
  int cover_correspondences(lgs_ctx* ctx, const int* corr_dev, int64_t n_corr);
  ~GicpCloud() {
    pts.release();
    covs.release();
    nn.release();
    cov_done.release();
    work_list.release();
    work_count.release();
  }
};

}  // namespace lgs

struct lgs_gicp {
  lgs_ctx* ctx = nullptr;
  // defaults FG:16-20, LSQ:11-19
  int k = 20;
  double corr_dist_threshold = 3.4028234663852886e38;
  int regularization = LGS_REG_PLANE;
  int max_iterations = 64;
  double rotation_eps = 2e-3, trans_eps = 5e-4;
  int lm_max_iterations = 10;
  double lm_init_lambda_factor = 1e-9, lm_lambda = -1.0;
  std::shared_ptr<lgs::GicpCloud> source, target;
  lgs::DevBuf corr, mahal, partials, counter, out_cloud;  // partials, counter: the last-CTA reduction (reduce.cuh)
  lgs::DevBuf nn_prev;     // nearest target point of every source point at the previous linearisation (search seed)
  bool have_seed = false;  // nn_prev is valid for the current source / target pair
  double final_hessian[36] = {1, 0, 0, 0, 0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 1};
  float final_T[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
  int linearize_calls = 0, error_calls = 0;
};

namespace lgs {
int gicp_align_impl(lgs_gicp* g, const float* guess16, lgs_align_result* res);
int gicp_fitness_impl(lgs_gicp* g, double max_range, double* fitness);
}  // namespace lgs
