/*
 * lgs_c.h -- C ABI of the B200-native LiDAR front-end hot path (liblgs_b200.so).
 *
 * Drop-in boundary for RyuYamamoto/lidar_graph_slam: every entry point below replaces one call the
 * reference makes through pcl::VoxelGrid / pcl::Registration (SURVEY.md section 8b).  Citations are
 * file:line under the reference tree:
 *   PPF = points_prefiltering/src/points_prefiltering.cpp
 *   LSM = lidar_scan_matcher/src/lidar_scan_matcher.cpp
 *   GBS = graph_based_slam/src/graph_based_slam.cpp
 *   NDT.h / NDT = thirdparty/ndt_omp/include/pclomp/ndt_omp.h / ndt_omp_impl.hpp
 *   VGC = thirdparty/ndt_omp/include/pclomp/voxel_grid_covariance_omp_impl.hpp
 *   FG / FG.h = thirdparty/fast_gicp/include/fast_gicp/gicp/impl/fast_gicp_impl.hpp / fast_gicp.hpp
 *   LSQ / LSQ.h = .../gicp/impl/lsq_registration_impl.hpp / lsq_registration.hpp
 *
 * Conventions
 *   - plain C types only; every function returns LGS_OK (0) or a negative error code and never
 *     throws; lgs_last_error() returns the thread's last message.
 *   - all pointers are caller-owned HOST memory unless the parameter name ends in _dev.
 *   - point clouds: `pts` + `n` + `stride_bytes`.  x,y,z are floats at byte offsets 0,4,8 of each
 *     record; intensity is the float at offset 12 when stride_bytes == 16 (packed xyzi) and at offset
 *     16 when stride_bytes >= 20 (pcl::PointXYZI, 32-byte records); absent (0) when stride_bytes == 12.
 *   - 4x4 transforms are float[16] COLUMN-major (Eigen::Matrix4f memory order).
 *   - handles are not thread-safe; use one lgs_ctx per host thread (the reference's registration
 *     objects are stateful and non re-entrant as well, SURVEY.md section 8b "Threading").
 *   - there is no CPU fallback: without a CUDA device every call fails with LGS_ERR_CUDA.
 */
#ifndef LGS_C_H_
#define LGS_C_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LGS_OK 0
#define LGS_ERR_INVALID (-1)
#define LGS_ERR_CUDA (-2)
#define LGS_ERR_STATE (-3)

/* ------------------------------------------------------------------------------------------- */
/* context: one CUDA device + one stream + scratch arenas                                        */
typedef struct lgs_ctx lgs_ctx;

/* cuda_stream: a cudaStream_t to run on (e.g. torch.cuda.current_stream().cuda_stream), or NULL to
 * let the context create its own non-blocking stream. */
int lgs_ctx_create(int device, void* cuda_stream, lgs_ctx** out);
void lgs_ctx_destroy(lgs_ctx* ctx);
int lgs_ctx_synchronize(lgs_ctx* ctx);
const char* lgs_last_error(void);
const char* lgs_version(void);
/* number of kernel launches issued through this context since creation (bench.py "gpu_launches") */
int64_t lgs_ctx_launch_count(const lgs_ctx* ctx);

/* ------------------------------------------------------------------------------------------- */
/* prefilter: range crop + box crop + pcl::VoxelGrid                                             */
/*   replaces PPF:102-112 (distance_filter), PPF:89-100 (crop), PPF:114-121 (downsample ->        */
/*   VoxelGrid::setLeafSize/setInputCloud/filter) and the VoxelGrid calls at GBS:311-313,490-493 */
#define LGS_VG_OK 0
#define LGS_VG_REFUSED_OVERFLOW 1 /* dx*dy*dz > INT32_MAX: like pcl::VoxelGrid, output = cropped input */

typedef struct lgs_voxelgrid_info {
  int32_t status;    /* LGS_VG_OK or LGS_VG_REFUSED_OVERFLOW */
  int32_t reserved;
  int64_t n_kept;    /* points that survive the crop */
  int64_t n_out;     /* output points (occupied voxels with >= min_points_per_voxel) */
  int32_t min_b[3];  /* integer bounding box of the kept points, in leaf units */
  int32_t max_b[3];
  int32_t div_b[3];
} lgs_voxelgrid_info;

/* range_min < 0 disables the range test (keep iff range_min < |p|, strict, f32 norm as PPF:107-108);
 * box6 = {min_x,max_x,min_y,max_y,min_z,max_z} or NULL (strict inequalities as PPF:93-96).
 * out_pts: capacity n packed xyzi records (16 B each), centroids in ascending voxel-index order.
 * out_voxel_idx[n]: per input point its voxel index (-1 if cropped); out_member_rank[n]: row of out_pts
 * the point was averaged into (-1 if none).  Either may be NULL. */
int lgs_voxelgrid_filter(lgs_ctx* ctx, const void* pts, int64_t n, int32_t stride_bytes, const float leaf[3],
                         int32_t min_points_per_voxel, double range_min, const double* box6, float* out_pts,
                         int32_t* out_voxel_idx, int32_t* out_member_rank, lgs_voxelgrid_info* info);

/* Same, with the input cloud already resident in device memory as packed float4 xyzi and the three
 * outputs written to device memory (any of them may be NULL).  info is still returned on the host. */
int lgs_voxelgrid_filter_dev(lgs_ctx* ctx, const float* pts_dev, int64_t n, const float leaf[3],
                             int32_t min_points_per_voxel, double range_min, const double* box6, float* out_pts_dev,
                             int32_t* out_voxel_idx_dev, int32_t* out_member_rank_dev, lgs_voxelgrid_info* info);

/* ------------------------------------------------------------------------------------------- */
/* prefilter, second stage: pcl::StatisticalOutlierRemoval<PointXYZI>                            */
/*   replaces PPF:132-140 (outlier_filter: setInputCloud / setMeanK / setStddevMulThresh /        */
/*   filter), called on the voxel grid's output at PPF:79-80                                      */
typedef struct lgs_sor lgs_sor;

typedef struct lgs_sor_info {
  int64_t n_out;     /* points kept */
  double mean;       /* mean of the per-point mean neighbour distances */
  double stddev;     /* their sample standard deviation */
  double threshold;  /* mean + stddev_mul * stddev */
} lgs_sor_info;

int lgs_sor_create(lgs_ctx* ctx, lgs_sor** out);
void lgs_sor_destroy(lgs_sor* sor);
int lgs_sor_set_mean_k(lgs_sor* sor, int32_t mean_k);              /* setMeanK, PPF:137; 1..31 */
int lgs_sor_set_stddev_mul_thresh(lgs_sor* sor, double mul);       /* setStddevMulThresh, PPF:138 */
int lgs_sor_set_negative(lgs_sor* sor, int32_t negative);          /* pcl::FilterIndices::setNegative */
/* filter (PPF:139): out_pts (capacity n packed xyzi) receives the kept points in input order; out_keep[n] the per-point
 * decision; out_distances[n] the per-point mean distance to its mean_k nearest neighbours.  Any output may be NULL.
 * The cloud must be finite (the voxel grid's output always is). */
int lgs_sor_filter(lgs_sor* sor, const void* pts, int64_t n, int32_t stride_bytes, float* out_pts, uint8_t* out_keep,
                   float* out_distances, lgs_sor_info* info);
int lgs_sor_filter_dev(lgs_sor* sor, const float* pts_dev, int64_t n, float* out_pts_dev, uint8_t* out_keep_dev,
                       float* out_distances_dev, lgs_sor_info* info);

/* ------------------------------------------------------------------------------------------- */
/* ingest: sensor_msgs/PointCloud2 payload -> packed xyzi device cloud                            */
/*   replaces the host-side pcl::fromROSMsg of the nodes (PPF:65-70, LSM:122-130, GBS:287-295):   */
/*   the message bytes are uploaded as they are and repacked on the GPU; the result feeds every   */
/*   *_dev entry point (lgs_voxelgrid_filter_dev, lgs_*_set_source_dev / set_target_dev, ...)      */
#define LGS_PC2_INT8 1 /* sensor_msgs/PointField datatype constants */
#define LGS_PC2_UINT8 2
#define LGS_PC2_INT16 3
#define LGS_PC2_UINT16 4
#define LGS_PC2_INT32 5
#define LGS_PC2_UINT32 6
#define LGS_PC2_FLOAT32 7
#define LGS_PC2_FLOAT64 8

typedef struct lgs_pc2_layout {
  uint32_t width, height;      /* points = width * height */
  uint32_t point_step;         /* bytes per record, 12..256, any alignment (Velodyne: 22) */
  uint32_t row_step;           /* 0 or width * point_step */
  int32_t offset_x, offset_y, offset_z;
  int32_t datatype_xyz;        /* must be LGS_PC2_FLOAT32 */
  int32_t offset_intensity;    /* -1: the message has no intensity field */
  int32_t datatype_intensity;  /* anything but FLOAT32 is not mapped, like pcl::fromROSMsg: intensity = 0 */
  int32_t is_bigendian;        /* must be 0 */
  int32_t reserved;
} lgs_pc2_layout;

/* data: the message's `data` bytes (host).  out_dev: device buffer of width*height x 4 floats. */
int lgs_cloud_from_pointcloud2(lgs_ctx* ctx, const void* data, const lgs_pc2_layout* layout, float* out_dev, int64_t* n_points);

/* ------------------------------------------------------------------------------------------- */
/* shared result of one registration (both methods)                                              */
typedef struct lgs_align_result {
  float T[16];               /* getFinalTransformation(), column-major */
  double fitness;            /* filled by *_fitness / batch only; otherwise 0 */
  double trans_probability;  /* NDT getTransformationProbability() (NDT:170); 0 for GICP */
  int32_t iterations;        /* NDT getFinalNumIteration() / nr_iterations_ (LSQ:66 definition for GICP) */
  int32_t converged;         /* hasConverged() */
  int32_t evaluations;       /* derivative evaluations (NDT) / linearize calls (GICP) */
  int32_t line_search_trials;/* NDT More-Thuente inner iterations / GICP compute_error calls */
  int32_t hessian_recomputes;/* NDT computeHessian calls */
  int32_t pair_id;           /* batch API: index of the pair this record belongs to */
} lgs_align_result;

/* ------------------------------------------------------------------------------------------- */
/* NDT: pclomp::NormalDistributionsTransform behind pcl::Registration (NDT.h:71-502)             */
typedef struct lgs_ndt lgs_ndt;

#define LGS_NDT_KDTREE 0 /* enum order of ndt_omp.h:52-57; KDTREE is not supported (LGS_ERR_INVALID) */
#define LGS_NDT_DIRECT26 1
#define LGS_NDT_DIRECT7 2
#define LGS_NDT_DIRECT1 3

int lgs_ndt_create(lgs_ctx* ctx, lgs_ndt** out);
void lgs_ndt_destroy(lgs_ndt* ndt);
int lgs_ndt_set_resolution(lgs_ndt* ndt, float resolution);             /* NDT.h:132-142 setResolution */
int lgs_ndt_set_step_size(lgs_ndt* ndt, double step_size);              /* NDT.h:162-166 setStepSize */
/* Parity mode (no counterpart in the reference): solve every Newton step (NDT:127-129) with the restated JacobiSVD instead of
 * the block elimination.  The align then repeats the reference's arithmetic step by step (bit-identical transforms on every
 * fuzzed problem) at about twice the time per align; off by default.  LGS_NDT_EXACT_SOLVE=1 in the environment does the same. */
int lgs_ndt_set_exact_newton_step(lgs_ndt* ndt, int32_t on);
int lgs_ndt_set_transformation_epsilon(lgs_ndt* ndt, double eps);       /* pcl::Registration::setTransformationEpsilon, LSM:58 */
int lgs_ndt_set_maximum_iterations(lgs_ndt* ndt, int32_t n);            /* pcl::Registration::setMaximumIterations, LSM:66 */
int lgs_ndt_set_outlier_ratio(lgs_ndt* ndt, double ratio);              /* NDT.h:180-184 setOutlierRatio */
int lgs_ndt_set_search_method(lgs_ndt* ndt, int32_t method);            /* NDT.h:186-188 setNeighborhoodSearchMethod */
/* setInputTarget (NDT.h:122-127): uploads and re-voxelises on EVERY call -- the scan matcher mutates
 * the target cloud in place and passes the same pointer again (LSM:187-212). */
int lgs_ndt_set_target(lgs_ndt* ndt, const void* pts, int64_t n, int32_t stride_bytes);
int lgs_ndt_set_source(lgs_ndt* ndt, const void* pts, int64_t n, int32_t stride_bytes);   /* setInputSource, LSM:162 */
/* device-resident variants (packed float4 xyzi already in HBM).  Lifetime contract of every *_dev setter in this header:
 * the cloud is copied device-to-device on the CONTEXT's stream and the call may return before the copy has run, so
 * pts_dev must stay valid (and unmodified) until lgs_ctx_synchronize(ctx) or any later call on the same object that
 * returns a result to the host; a context created on the caller's own stream makes this ordinary stream ordering. */
int lgs_ndt_set_target_dev(lgs_ndt* ndt, const float* pts_dev, int64_t n);
int lgs_ndt_set_source_dev(lgs_ndt* ndt, const float* pts_dev, int64_t n);
/* The rolling local map of the scan matcher (LSM:187-212: on a key-frame change the node concatenates the last N key frames,
 * transformed by their poses, and calls setInputTarget, which re-voxelises all of them).  Here the target is given as a
 * list of key frames of a device-resident key-frame array and maintained INCREMENTALLY: the voxel partial sums of every
 * key frame are cached per (pose, resolution); a call voxelises only the key frames it has not seen (typically the one
 * that entered the window), drops those that left, and merges the cached sums in the order of ids[] - the order in which
 * the reference concatenates.  The voxel table equals setInputTarget(assembled cloud): occupancy, counts and validity
 * flags identical, means / covariances to the f64 rounding of adding per-frame sums (~1e-16 relative).  A moved key frame
 * (lgs_keyframes_set_pose) is re-voxelised.  *frames_voxelised (optional): key frames voxelised from their points by this
 * call.  getFitnessScore assembles the cloud on first use. */
typedef struct lgs_keyframes lgs_keyframes;
int lgs_ndt_set_target_keyframes(lgs_ndt* ndt, lgs_keyframes* kf, const int32_t* ids, int32_t n_ids, int32_t* frames_voxelised);
/* align (pcl::Registration::align + NDT:80-171, LSM:165, GBS:318).  guess may be NULL (identity).
 * out_cloud: NULL or capacity n_source packed xyzi records = source transformed by the final T. */
int lgs_ndt_align(lgs_ndt* ndt, const float* guess16, lgs_align_result* result, float* out_cloud);
/* No counterpart in the reference (ndt_omp runs one align per call): N aligns in one resident launch (per wave).  Record i is
 * bit-identical to lgs_ndt_align(ndts[i], guess i) run alone, and each handle ends in the state its last occurrence leaves;
 * handles may repeat; all on one context.  guesses16: N x 16 col-major floats or NULL (identity).  fitness_max_range:
 * NULL = no fitness, else records[i].fitness = getFitnessScore(*fitness_max_range) at record i's transform.
 * out_clouds: NULL or N pointers (each NULL or capacity n_source of ndts[i]).  records[i].pair_id = i.  n = 0 does nothing.
 * LGS_NDT_MANY_MAX_GROUPS (environment, read on every call): at most this many aligns per launch (default 1:
 * measured, grouped aligns were slower than consecutive ones; see DESIGN section 7). */
int lgs_ndt_align_many(lgs_ndt* const* ndts, int32_t n, const float* guesses16, const double* fitness_max_range,
                       lgs_align_result* records, float* const* out_clouds);
/* getFitnessScore(max_range) (PCL registration.hpp, GBS:321): exact 1-NN mean squared distance */
int lgs_ndt_fitness(lgs_ndt* ndt, double max_range, double* fitness);
/* calculateScore (NDT:934-982) of the source transformed by T */
int lgs_ndt_calculate_score(lgs_ndt* ndt, const float* T16, double* score);

/* parity hooks (SURVEY.md section 8b "export_voxels for parity tests") */
typedef struct lgs_ndt_grid_info {
  int32_t refused;   /* 1 when the target grid was refused (VGC:79-84) */
  int32_t dense;     /* 1 dense cell table, 0 hashed cell table */
  int64_t n_voxels;  /* occupied voxels (all leaves, including those with < 6 points) */
  int64_t n_valid;   /* voxels usable by the lookup (n >= 6 and covariance checks passed) */
  int32_t min_b[3];
  int32_t max_b[3];
  int32_t div_b[3];
  int32_t reserved;
} lgs_ndt_grid_info;
int lgs_ndt_grid_info_get(lgs_ndt* ndt, lgs_ndt_grid_info* info);
/* arrays of n_voxels entries, ascending idx: idx, nr_points (-1 when invalidated, VGC:339,363),
 * mean[3], cov[9], icov[9] (row-major f64).  Any pointer may be NULL. */
int lgs_ndt_export_voxels(lgs_ndt* ndt, int32_t* idx, int32_t* nr_points, double* mean, double* cov, double* icov);
/* one derivative evaluation with the source transformed by T16 and the angle tables of p6:
 * mode 0 = computeDerivatives(compute_hessian=true) (NDT:179-285), 1 = gradient only,
 * mode 2 = computeHessian (f64, NDT:539-644).  Outputs: score, g[6], H[36] row-major. */
int lgs_ndt_derivatives(lgs_ndt* ndt, const float* T16, const double* p6, int32_t mode, double* score, double* g6, double* H36);

/* measurement hook (bench.py roofline): returns and clears the CUDA-event timings gathered since the last
 * call, then enables (1) / disables (0) per-launch timing of the evaluation kernels.  out8 = {launches, ms} for
 * computeDerivatives with Hessian, gradient-only, and the f64 computeHessian kernel, then the number of accepted
 * (point, voxel) terms of the last evaluation and the source size.  out8 may be NULL. */
/* static convertTransform(x, trans) (NDT.h:214-238): (x, y, z, roll, pitch, yaw) -> column-major f32 4x4.  Host only. */
int lgs_ndt_convert_transform(const double* x6, float* T16);
int lgs_ndt_profile(lgs_ndt* ndt, int32_t enable, double* out8);
/* measurement hook: where the last device-resident align (one ndt_align_kernel launch) spent its time, as SM cycles of
 * CTA 0 summed over the align's evaluations: out16 = {evaluating, waiting for the other CTAs, adding the per-CTA rows,
 * optimiser step, publishing the next command, whole kernel, 0, 0; then the optimiser step in detail: More-Thuente /
 * exit rules (thread 0), 6x6 elimination (warp 0), Newton post-processing (thread 0), sines / cosines, transform +
 * angular tables, 0, 0, 0} */
int lgs_ndt_align_breakdown(lgs_ndt* ndt, double* out16);

/* ------------------------------------------------------------------------------------------- */
/* GICP: fast_gicp::FastGICP over LsqRegistration (FG.h:48-70, LSQ.h:48-60)                       */
typedef struct lgs_gicp lgs_gicp;

#define LGS_REG_NONE 0 /* enum order of gicp_settings.hpp:6 */
#define LGS_REG_MIN_EIG 1
#define LGS_REG_NORMALIZED_MIN_EIG 2
#define LGS_REG_PLANE 3
#define LGS_REG_FROBENIUS 4

int lgs_gicp_create(lgs_ctx* ctx, lgs_gicp** out);
void lgs_gicp_destroy(lgs_gicp* g);
int lgs_gicp_set_correspondence_randomness(lgs_gicp* g, int32_t k);     /* FG:40-42 */
int lgs_gicp_set_max_correspondence_distance(lgs_gicp* g, double d);    /* pcl::Registration, LSM:44 */
int lgs_gicp_set_transformation_epsilon(lgs_gicp* g, double eps);
int lgs_gicp_set_rotation_epsilon(lgs_gicp* g, double eps);             /* LSQ:28-30 */
int lgs_gicp_set_maximum_iterations(lgs_gicp* g, int32_t n);
int lgs_gicp_set_regularization_method(lgs_gicp* g, int32_t method);    /* FG:45-47 */
int lgs_gicp_set_initial_lambda_factor(lgs_gicp* g, double f);          /* LSQ:33-35 */
/* setInputSource / setInputTarget (FG:72-90).  Unlike the reference these never cache on pointer
 * identity: each call uploads and invalidates the cloud's covariances (SURVEY Appendix A #9). */
int lgs_gicp_set_source(lgs_gicp* g, const void* pts, int64_t n, int32_t stride_bytes);
int lgs_gicp_set_target(lgs_gicp* g, const void* pts, int64_t n, int32_t stride_bytes);
int lgs_gicp_set_source_dev(lgs_gicp* g, const float* pts_dev, int64_t n);
int lgs_gicp_set_target_dev(lgs_gicp* g, const float* pts_dev, int64_t n);
int lgs_gicp_swap_source_and_target(lgs_gicp* g);                       /* FG:50-57 */
int lgs_gicp_clear_source(lgs_gicp* g);                                 /* FG:60-63 */
int lgs_gicp_clear_target(lgs_gicp* g);                                 /* FG:66-69 */
int lgs_gicp_align(lgs_gicp* g, const float* guess16, lgs_align_result* result, float* out_cloud);
int lgs_gicp_fitness(lgs_gicp* g, double max_range, double* fitness);
int lgs_gicp_final_hessian(lgs_gicp* g, double* H36);                   /* LSQ:43-45 getFinalHessian */
/* parity hooks: which = 0 source, 1 target; covs = n x 9 f64 row-major (computed on demand, FG:241-298) */
int lgs_gicp_export_covariances(lgs_gicp* g, int32_t which, double* covs);
/* evaluateCost (LSQ.h:58, LSQ:48-50): the GICP cost at a pose (column-major f32 4x4) over the correspondences of the
 * last linearisation; LGS_ERR_STATE before the first align / linearize */
int lgs_gicp_evaluate_cost(lgs_gicp* g, const float* T16, double* cost);
/* setSourceCovariances / setTargetCovariances (FG.h:60-62, FG:93-101): n x 9 f64 row-major 3x3 blocks; used at align
 * time only if n equals the cloud's size (FG:104-109), and dropped by the next setInputSource / setInputTarget */
int lgs_gicp_set_covariances(lgs_gicp* g, int32_t which, const double* covs, int64_t n);
/* evaluateCost / linearize at a row-major f64 4x4 (LSQ:48-50, FG:155-211): cost, H[36], b[6], and
 * optionally the per-source-point correspondence index (-1 = none) */
int lgs_gicp_linearize(lgs_gicp* g, const double* T16_rowmajor, double* cost, double* H36, double* b6, int32_t* correspondences);

/* ------------------------------------------------------------------------------------------- */
/* PCL-style GICP: pclomp::GeneralizedIterativeClosestPoint (BFGS) behind pcl::Registration       */
/*   GO = thirdparty/ndt_omp/include/pclomp/gicp_omp_impl.hpp, GO.h = .../gicp_omp.h;             */
/*   constructed at LSM:73-96 and GBS:120-141 (registration_method "GICP")                        */
typedef struct lgs_gicp_omp lgs_gicp_omp;

int lgs_gicp_omp_create(lgs_ctx* ctx, lgs_gicp_omp** out);               /* defaults GO.h:116-126 */
void lgs_gicp_omp_destroy(lgs_gicp_omp* g);
int lgs_gicp_omp_set_correspondence_randomness(lgs_gicp_omp* g, int32_t k);      /* GO.h:248, LSM:94 */
int lgs_gicp_omp_set_max_correspondence_distance(lgs_gicp_omp* g, double d);     /* LSM:88 */
int lgs_gicp_omp_set_transformation_epsilon(lgs_gicp_omp* g, double eps);        /* LSM:92 */
int lgs_gicp_omp_set_rotation_epsilon(lgs_gicp_omp* g, double eps);              /* GO.h:234 */
int lgs_gicp_omp_set_maximum_iterations(lgs_gicp_omp* g, int32_t n);             /* LSM:89 */
int lgs_gicp_omp_set_maximum_optimizer_iterations(lgs_gicp_omp* g, int32_t n);   /* GO.h:262, LSM:91 */
/* setInputSource / setInputTarget (GO.h:139-169): upload, drop the cloud's covariances */
int lgs_gicp_omp_set_source(lgs_gicp_omp* g, const void* pts, int64_t n, int32_t stride_bytes);
int lgs_gicp_omp_set_target(lgs_gicp_omp* g, const void* pts, int64_t n, int32_t stride_bytes);
int lgs_gicp_omp_set_source_dev(lgs_gicp_omp* g, const float* pts_dev, int64_t n);
int lgs_gicp_omp_set_target_dev(lgs_gicp_omp* g, const float* pts_dev, int64_t n);
/* align (pcl::Registration::align + GO:370-516).  result: iterations = nr_iterations_ (outer iterations),
 * evaluations = df + fdf functor calls, line_search_trials = operator() calls, hessian_recomputes = BFGS
 * inner iterations summed over the outer iterations. */
int lgs_gicp_omp_align(lgs_gicp_omp* g, const float* guess16, lgs_align_result* result, float* out_cloud);
int lgs_gicp_omp_fitness(lgs_gicp_omp* g, double max_range, double* fitness);
/* parity hooks: covariances as lgs_gicp_export_covariances (GO:48-122); one outer-iteration set-up at
 * (transformation_, guess) followed by f(x), df(x), fdf(x) (GO:245-367): out15 = f, df[6], fdf f, fdf g[6],
 * number of correspondences; corr (n_source, -1 = none) and mahal (n_source x 9 f32) may be NULL */
int lgs_gicp_omp_export_covariances(lgs_gicp_omp* g, int32_t which, double* covs);
int lgs_gicp_omp_functor(lgs_gicp_omp* g, const float* guess16, const float* transformation16, const double* x6, double* out15,
                         int32_t* corr, float* mahal);

/* ------------------------------------------------------------------------------------------- */
/* ICP: pcl::IterativeClosestPoint<PointXYZI, PointXYZI> behind pcl::Registration                 */
/*   the graph SLAM node's default loop-closure method (graph_based_slam.param.yaml:9), built at  */
/*   GBS:142-151 with setMaxCorrespondenceDistance(30) / setMaximumIterations(100) /              */
/*   setTransformationEpsilon(1e-8) / setEuclideanFitnessEpsilon(1e-6) / setRANSACIterations(0)   */
typedef struct lgs_icp lgs_icp;

#define LGS_ICP_NOT_CONVERGED 0 /* pcl::registration::DefaultConvergenceCriteria::ConvergenceState */
#define LGS_ICP_ITERATIONS 1
#define LGS_ICP_TRANSFORM 2
#define LGS_ICP_ABS_MSE 3
#define LGS_ICP_REL_MSE 4
#define LGS_ICP_NO_CORRESPONDENCES 5

int lgs_icp_create(lgs_ctx* ctx, lgs_icp** out);   /* PCL defaults: 10 iterations, epsilons 0, distance sqrt(DBL_MAX) */
void lgs_icp_destroy(lgs_icp* icp);
int lgs_icp_set_max_correspondence_distance(lgs_icp* icp, double d);       /* GBS:145 */
int lgs_icp_set_maximum_iterations(lgs_icp* icp, int32_t n);               /* GBS:146 */
int lgs_icp_set_transformation_epsilon(lgs_icp* icp, double eps);          /* GBS:147 (compared with the SQUARED translation, as in PCL) */
int lgs_icp_set_transformation_rotation_epsilon(lgs_icp* icp, double eps); /* cos(angle) threshold; 0 = 1 - transformation_epsilon */
int lgs_icp_set_euclidean_fitness_epsilon(lgs_icp* icp, double eps);       /* GBS:148 (relative MSE threshold) */
/* The convergence criteria object lives in the ICP object, as in PCL: the previous-MSE it compares with survives from one
 * align to the next.  This gives it the state of a newly constructed pcl::IterativeClosestPoint (the loop-closure batch
 * calls it per pair so that a record does not depend on which pair its worker verified before). */
int lgs_icp_reset_convergence_criteria(lgs_icp* icp);
int lgs_icp_set_source(lgs_icp* icp, const void* pts, int64_t n, int32_t stride_bytes);
int lgs_icp_set_target(lgs_icp* icp, const void* pts, int64_t n, int32_t stride_bytes);
int lgs_icp_set_source_dev(lgs_icp* icp, const float* pts_dev, int64_t n);
int lgs_icp_set_target_dev(lgs_icp* icp, const float* pts_dev, int64_t n);
/* result: iterations = nr_iterations_, evaluations = correspondence/estimation steps, line_search_trials = the
 * LGS_ICP_* convergence state, trans_probability = MSE of the last correspondence set */
int lgs_icp_align(lgs_icp* icp, const float* guess16, lgs_align_result* result, float* out_cloud);
int lgs_icp_fitness(lgs_icp* icp, double max_range, double* fitness);
/* parity hook: one step on guess * source: sums17 = {n, sum d2, sum p[3], sum q[3], sum q p^T[9]}, T16 = the estimated
 * transformation_ (pcl::umeyama), *ok = 0 when fewer than 3 correspondences were found */
int lgs_icp_step(lgs_icp* icp, const float* guess16, double* sums17, float* T16, int32_t* ok);

/* exact k-NN of `queries` in `pts` (the search behind FG:133 and FG:254); idx/d2 are m x k, ascending */
int lgs_knn(lgs_ctx* ctx, const void* pts, int64_t n, int32_t stride_bytes, const void* queries, int64_t m, int32_t qstride_bytes,
            int32_t k, int32_t* idx, float* d2);
/* parity hook for the exact 1-NN of the correspondence searches (FG:133, ICP) and of getFitnessScore: idx/d2 are m
 * entries.  seeds (m entries, or NULL for the unseeded search) start query t from indexed point seeds[t], as the
 * correspondence searches start from the previous iteration's neighbour; a seed outside [0, n) means none.  The result
 * does not depend on the seed.  An empty cloud gives idx -1 and d2 +inf.  d2 may be NULL. */
int lgs_nn_search1(lgs_ctx* ctx, const void* pts, int64_t n, int32_t stride_bytes, const void* queries, int64_t m, int32_t qstride_bytes,
                   const int32_t* seeds, int32_t* idx, float* d2);

/* parity hook for the device radix sort that orders points by voxel (the std::sort of pcl::VoxelGrid::applyFilter
 * and the std::map iteration order of VGC:218-263): stable sort of n (key, value) pairs by the low `bits` key bits,
 * in place in the caller's host arrays */
int lgs_sort_pairs(lgs_ctx* ctx, uint32_t* keys, uint32_t* vals, int64_t n, int32_t bits);

/* parity hook for the small dense solvers the kernels run per voxel, per point and per Newton step (csrc/math.cuh,
 * csrc/ndt_opt.cuh): n independent problems, one GPU thread each, f64 in and f64 out, row-major, every output bit as the
 * device computes it.  in holds n records of LGS_LINALG_IN(op) doubles, out receives n records of LGS_LINALG_OUT(op).
 *   LGS_LINALG_SVD3        A[9]        -> U[9], S[3], V[9]        svd_jacobi<3, double> (FastGICP / pclomp GICP covariances)
 *   LGS_LINALG_EIG3        A[9]        -> w[3], Q[9], ok          eig_sym3, lower triangle read (NDT voxel covariances)
 *   LGS_LINALG_INV3        A[9]        -> A^-1[9]                 inv3
 *   LGS_LINALG_SVD_SOLVE6  H[36], b[6] -> x[6]                    svd_solve<6> (the JacobiSVD Newton step)
 *   LGS_LINALG_SCHUR6      H[36], b[6] -> x[6], accepted          schur_solve6 (x as left when declined)
 *   LGS_LINALG_NEWTON6     H[36], b[6] -> x[6], x_exact[6]        the NDT optimiser's step rule: Schur, else JacobiSVD;
 *                                                                 then with the exact Newton step on (JacobiSVD only)
 * Flags are 1.0 / 0.0.  An unknown op, n < 0 or a null pointer with n > 0 is LGS_ERR_INVALID and launches nothing. */
#define LGS_LINALG_SVD3 0
#define LGS_LINALG_EIG3 1
#define LGS_LINALG_INV3 2
#define LGS_LINALG_SVD_SOLVE6 3
#define LGS_LINALG_SCHUR6 4
#define LGS_LINALG_NEWTON6 5
#define LGS_LINALG_IN(op) ((op) <= LGS_LINALG_INV3 ? 9 : 42)
#define LGS_LINALG_OUT(op) ((op) == LGS_LINALG_SVD3 ? 21 : (op) == LGS_LINALG_EIG3 ? 13 : (op) == LGS_LINALG_INV3 ? 9 : (op) == LGS_LINALG_SVD_SOLVE6 ? 6 : (op) == LGS_LINALG_SCHUR6 ? 7 : 12)
int lgs_linalg_batch(lgs_ctx* ctx, int32_t op, int64_t n, const double* in, double* out);

/* ------------------------------------------------------------------------------------------- */
/* key-frame array + sub-map assembly, device resident                                            */
/*   replaces the per-key-frame fromROSMsg + transform_point_cloud + `*cloud += ...` loops and the */
/*   re-upload of the assembled map: LSM:196-212 (local map, newest first) and GBS:297-313         */
/*   (candidate neighbourhood, ascending index, then VoxelGrid).  A key frame is uploaded once.    */
/* (lgs_keyframes is declared with lgs_ndt_set_target_keyframes above) */

int lgs_keyframes_create(lgs_ctx* ctx, lgs_keyframes** out);
void lgs_keyframes_destroy(lgs_keyframes* kf);
/* key_frame_array_.keyframes.emplace_back (LSM:196-197): the cloud in its own frame + its pose (column-major
 * Matrix4f, what geometry_pose_to_matrix returns at LSM:205); id = index in the array */
int lgs_keyframes_push(lgs_keyframes* kf, const void* pts, int64_t n, int32_t stride_bytes, const float* pose16, int32_t* id);
int lgs_keyframes_push_dev(lgs_keyframes* kf, const float* pts_dev, int64_t n, const float* pose16, int32_t* id);
/* a pose-graph update moved the key frame (the optimised poses the back end publishes, GBS:343-352) */
int lgs_keyframes_set_pose(lgs_keyframes* kf, int32_t id, const float* pose16);
int lgs_keyframes_size(lgs_keyframes* kf, int64_t* count, int64_t* total_points);
/* key_frame.accum_distance (LSM:193) and detect_loop_with_accum_dist (GBS:157-187): all key frames at least
 * accumulate_distance_threshold of path behind `latest_id` and closer to it than search_for_candidate_threshold;
 * *nearest = the single candidate optimization_callback picks (GBS:263-280), -1 if none.  candidates may be NULL. */
int lgs_keyframes_set_accum_distance(lgs_keyframes* kf, int32_t id, double accum_distance);
/* key_frame.pose.position as the f64 geometry_msgs value (GBS:163-171 compares those); without it the loop detection falls
 * back to the f32 translation of the pose matrix, which can flip a candidate sitting on the 15 m / 100 m thresholds */
int lgs_keyframes_set_position(lgs_keyframes* kf, int32_t id, const double* xyz);
int lgs_keyframes_detect_loop(lgs_keyframes* kf, int32_t latest_id, double accumulate_distance_threshold, double search_for_candidate_threshold,
                              int32_t* candidates, int32_t capacity, int32_t* n_candidates, int32_t* nearest);
/* sub-map = concatenation, in the order of ids[], of pcl::transformPointCloud(key frame, pose); leaf > 0 applies
 * pcl::VoxelGrid(leaf) to the result (GBS:311-313).  *out_dev is a packed xyzi device cloud owned by kf, valid
 * until the next assemble call; feed it to lgs_*_set_target_dev / set_source_dev. */
int lgs_keyframes_assemble(lgs_keyframes* kf, const int32_t* ids, int32_t n_ids, float leaf, float** out_dev, int64_t* n_out);

/* ------------------------------------------------------------------------------------------- */
/* batched loop-closure verification: GBS:297-322 for a list of (scan, submap) pairs              */
#define LGS_METHOD_NDT 0      /* pclomp::NormalDistributionsTransform (GBS:101-119) */
#define LGS_METHOD_GICP 1     /* fast_gicp::FastGICP (GBS:82-100) */
#define LGS_METHOD_ICP 2      /* pcl::IterativeClosestPoint, the YAML default (GBS:142-151) */
#define LGS_METHOD_GICP_OMP 3 /* pclomp::GeneralizedIterativeClosestPoint (GBS:120-141) */

typedef struct lgs_batch_params {
  int32_t method;                 /* LGS_METHOD_* */
  int32_t max_iterations;         /* graph_based_slam.param.yaml */
  double transformation_epsilon;
  double max_correspondence_distance; /* GICP; <= 0 keeps FLT_MAX */
  int32_t k_correspondences;      /* GICP */
  float ndt_resolution;           /* NDT */
  double ndt_step_size;
  float submap_leaf;              /* VoxelGrid leaf applied to each submap before setInputTarget (GBS:61: 0.5); <= 0 disables */
  double fitness_max_range;       /* getFitnessScore(max_range); <= 0 means DBL_MAX (GBS:321) */
  int32_t n_workers;              /* concurrent pairs per GPU (each on its own stream); <= 0 picks a default */
  int32_t max_optimizer_iterations; /* GICP_OMP: BFGS inner iterations (GBS:136); <= 0 keeps 20 */
  double euclidean_fitness_epsilon; /* ICP (GBS:148); 0 keeps PCL's default (-DBL_MAX) */
} lgs_batch_params;

/* Each pair i: scan = scans[i] (n_scan[i] points), submap = submaps[i] (n_submap[i] points), all with the
 * same stride; guesses16 = n_pairs x 16 floats or NULL (identity, GBS:318).  records[n_pairs] receives
 * (T, fitness, iterations, converged, pair_id = pair_id0 + i).  records_dev, when not NULL, is a device
 * buffer of n_pairs records that receives the same data (the NCCL gather's send buffer). */
int lgs_batch_align(int device, void* cuda_stream, const lgs_batch_params* params, int64_t n_pairs, const void* const* scans,
                    const int64_t* n_scan, const void* const* submaps, const int64_t* n_submap, int32_t stride_bytes,
                    const float* guesses16, int32_t pair_id0, lgs_align_result* records, void* records_dev);

/* The same with both clouds of every pair taken from the device-resident key-frame array (optimization_callback,
 * GBS:247-251 + 297-322, for a list of candidates): pair i aligns key frame scan_ids[i], transformed by its pose, to the
 * submap_leaf-filtered concatenation of key frames center_ids[i] - K .. center_ids[i] + K (K = search_key_frame_num,
 * graph_based_slam.param.yaml:4), ascending, clipped to the array.  Only the records cross PCIe. */
int lgs_batch_align_keyframes(lgs_keyframes* kf, void* cuda_stream, const lgs_batch_params* params, int64_t n_pairs,
                              const int32_t* scan_ids, const int32_t* center_ids, int32_t search_key_frame_num,
                              const float* guesses16, int32_t pair_id0, lgs_align_result* records, void* records_dev);

/* ------------------------------------------------------------------------------------------- */
/* the same batch over the GPUs of a box: one process per GPU, one NCCL gather of the records    */
/*   SURVEY.md section 8b "batch_align_dist(ncclComm, rank, world, ...)" / section 8e.  The      */
/*   reference verifies one candidate per optimization_callback on one core (GBS:245-340); a     */
/*   pose graph with thousands of candidates (BASELINE configs[4]) is embarrassingly parallel:   */
/*   pairs are dealt to the ranks by size, every rank verifies its own, and the fixed-size        */
/*   records are exchanged with a single ncclAllGather over NVLink.                               */
typedef struct lgs_comm lgs_comm;
#define LGS_COMM_ID_BYTES 128 /* sizeof(ncclUniqueId) */

/* rank 0 calls lgs_comm_get_unique_id and hands the 128 bytes to the other ranks by any means it has (MPI, a file,
 * torch.distributed); every rank then calls lgs_comm_init_rank (ncclCommInitRank on `device`).  A host that already
 * owns an ncclComm_t passes it to lgs_comm_adopt instead (the handle is used, never destroyed). */
int lgs_comm_get_unique_id(uint8_t* id128);
int lgs_comm_init_rank(const uint8_t* id128, int32_t rank, int32_t world, int32_t device, lgs_comm** out);
int lgs_comm_adopt(void* nccl_comm, int32_t device, lgs_comm** out);
void lgs_comm_destroy(lgs_comm* comm);
int lgs_comm_info(lgs_comm* comm, int32_t* rank, int32_t* world, int32_t* nccl_version);

/* The partition rule, exported so that callers and tests can predict it: pairs sorted by descending size (index breaks
 * ties) and dealt round-robin; out_ids receives this rank's pair indices in ascending order.  Pure host arithmetic. */
int lgs_batch_partition(const int64_t* sizes, int64_t n_total, int32_t rank, int32_t world, int32_t* out_ids, int64_t capacity, int64_t* n_mine);

typedef struct lgs_batch_dist_info {
  int32_t rank, world;
  int64_t n_local;      /* pairs this rank verified */
  int64_t n_received;   /* records that came back from the gather (= n_pairs on success) */
  int64_t gather_bytes; /* bytes received by this rank in the ncclAllGather */
  double verify_ms;     /* host wall time of this rank's own pairs */
  double gather_ms;     /* ncclAllGather + D2H of the gathered records + placement */
} lgs_batch_dist_info;

/* Collective: every rank of `comm` calls it with the SAME list of n_pairs candidates (the pose graph is replicated, its
 * key-frame array resident on every GPU) and receives ALL n_pairs records in records_all[pair index], bit-identical on
 * every rank and for every world size.  Each pair's last kernel stores its record in the NCCL send buffer. */
int lgs_batch_align_keyframes_dist(lgs_keyframes* kf, lgs_comm* comm, const lgs_batch_params* params, int64_t n_pairs,
                                   const int32_t* scan_ids, const int32_t* center_ids, int32_t search_key_frame_num,
                                   const float* guesses16, lgs_align_result* records_all, lgs_batch_dist_info* info);
/* Host-array form: n_scan / n_submap are needed for all pairs on every rank (they drive the partition); scans[i] /
 * submaps[i] are read only on the rank that owns pair i and may be NULL elsewhere (each rank uploads only its own). */
int lgs_batch_align_dist(lgs_comm* comm, const lgs_batch_params* params, int64_t n_pairs, const void* const* scans,
                         const int64_t* n_scan, const void* const* submaps, const int64_t* n_submap, int32_t stride_bytes,
                         const float* guesses16, lgs_align_result* records_all, lgs_batch_dist_info* info);

/* ------------------------------------------------------------------------------------------- */
/* offline odometry: the scan matcher's key-frame loop (LSM:122-250) over whole recorded sequences */
/*   per frame: range crop + VoxelGrid + optional SOR in the sensor frame (the prefilter node),   */
/*   base_from_sensor (LSM:127-131), then frame 0 = key frame 0 and target; frame k > 0 =         */
/*   setInputSource + align(pose after frame k-1) (LSM:162-165), dropped when not converged       */
/*   (LSM:167-170); a key frame when |t(T) - t(T_kf)| >= keyframe_displacement (LSM:183), and    */
/*   then the target = the newest max_scan_accumulate_num key frames, newest first (LSM:187-212). */
/*   DESIGN.md section 8 records the contract.                                                   */
typedef struct lgs_odometry_params {
  int32_t method;                     /* LGS_METHOD_NDT / _GICP / _GICP_OMP (the scan matcher's three, LSM:37-97); ICP is refused */
  int32_t max_iterations;             /* fields up to max_optimizer_iterations mean what they mean in lgs_batch_params; a value */
  double transformation_epsilon;      /* <= 0 takes the scan-matcher YAML default (SURVEY Appendix C): NDT resolution 2.0,      */
  double max_correspondence_distance; /* step 0.1, eps 0.01, 64 iterations; GICP k 20, max correspondence distance 2.0, eps     */
  int32_t k_correspondences;          /* 0.01, 64 iterations; pclomp GICP 20 BFGS iterations                                  */
  float ndt_resolution;
  double ndt_step_size;
  int32_t max_optimizer_iterations;
  int32_t max_scan_accumulate_num;    /* key frames in the target window, >= 1 (lidar_scan_matcher.param.yaml: 20) */
  double keyframe_displacement;       /* metres (param.yaml: 1.0); <= 0 takes 1.0 */
  double range_min;                   /* keep iff range_min < |p| (PPF:102-112); < 0 disables; needs leaf > 0 (the crop is a VoxelGrid stage) */
  float leaf;                         /* VoxelGrid leaf (PPF:114-121); <= 0 disables */
  int32_t sor_mean_k;                 /* StatisticalOutlierRemoval mean_k (PPF:132-140), <= 31; <= 0 disables */
  double sor_stddev_mul;
  float base_from_sensor[16];         /* column-major extrinsic (LSM:127-131); all zeros = identity */
} lgs_odometry_params;

/* One per input frame, in (sequence, frame) order.  Fixed 112 bytes: the distributed run moves it as bytes. */
typedef struct lgs_odometry_frame {
  float T[16];               /* pose after the frame (map from base), column-major */
  double trans_probability;  /* the align's getTransformationProbability (NDT), else 0 */
  double accum_distance;     /* path length over the key frames so far (LSM:193) */
  int32_t sequence, frame;
  int32_t converged;         /* hasConverged(); frame 0 is 1 */
  int32_t iterations;        /* the align's iteration count; 0 for frame 0 */
  int32_t evaluations;       /* derivative evaluations (NDT) / linearize or functor calls (GICP) */
  int32_t keyframe_id;       /* id of the key frame this frame became, -1 if none */
  int64_t n_source;          /* points after the prefilter */
} lgs_odometry_frame;
#ifdef __cplusplus
static_assert(sizeof(lgs_odometry_frame) == 112, "lgs_odometry_frame is 112 bytes");
#else
_Static_assert(sizeof(lgs_odometry_frame) == 112, "lgs_odometry_frame is 112 bytes");
#endif

/* n_seq sequences; sequence s has n_frames[s] frames.  frames / n_points list the frames of all sequences flat, sequence
 * after sequence; records receives one record per frame in the same order.  Host form: records of stride_bytes as every host
 * cloud of this header; frame k+1 is uploaded through pinned staging on a copy stream while frame k aligns.  Device form:
 * packed xyzi device clouds on ctx's device, read on ctx's stream.  initial_poses: n_seq x 16 column-major or NULL (identity).
 * keyframes: NULL or n_seq entries, each NULL (the run uses scratch) or an EMPTY array on ctx's device that the run fills
 * with the sequence's key frames, their poses, accum_distance and f64 positions (ready for detect_loop /
 * lgs_batch_align_keyframes).  Every sequence starts from fresh registration objects; sequences run one after another.
 * Every argument is checked before anything runs: a rejected call launches nothing. */
int lgs_odometry_run(lgs_ctx* ctx, const lgs_odometry_params* params, int32_t n_seq, const int32_t* n_frames, const void* const* frames,
                     const int64_t* n_points, int32_t stride_bytes, const float* initial_poses, lgs_keyframes* const* keyframes,
                     lgs_odometry_frame* records);
int lgs_odometry_run_dev(lgs_ctx* ctx, const lgs_odometry_params* params, int32_t n_seq, const int32_t* n_frames, const float* const* frames_dev,
                         const int64_t* n_points, const float* initial_poses, lgs_keyframes* const* keyframes, lgs_odometry_frame* records);

/* measurement hook: with LGS_ODOMETRY_PROFILE=1 in the environment the runs of this thread time their stages with CUDA events;
 * out4 = {frames, prefilter ms (upload + range crop + VoxelGrid + SOR + extrinsic), align ms (setInputSource + align),
 * key-frame ms (push + target update)} summed since the last call, which clears them. */
int lgs_odometry_profile(double* out4);

typedef struct lgs_odometry_dist_info {
  int32_t rank, world;
  int64_t n_local_sequences;
  int64_t n_local_frames;
  int64_t n_received;   /* records that came back from the gather (= all frames on success) */
  int64_t gather_bytes; /* bytes received by this rank in the ncclAllGather */
  double run_ms;        /* host wall time of this rank's own sequences */
  double gather_ms;     /* ncclAllGather + D2H + placement */
} lgs_odometry_dist_info;

/* Collective over comm (on ctx's device): every rank passes the same n_seq, n_frames and n_points; the sequences are dealt by
 * lgs_batch_partition over each sequence's total point count; frames of sequences a rank does not own are not read and may
 * be NULL.  Each rank runs its share as lgs_odometry_run would (scratch key frames) and ONE ncclAllGather returns every
 * record to every rank in records_all, bit-identical to a one-rank run. */
int lgs_odometry_run_dist(lgs_ctx* ctx, lgs_comm* comm, const lgs_odometry_params* params, int32_t n_seq, const int32_t* n_frames,
                          const void* const* frames, const int64_t* n_points, int32_t stride_bytes, const float* initial_poses,
                          lgs_odometry_frame* records_all, lgs_odometry_dist_info* info);
int lgs_odometry_run_dist_dev(lgs_ctx* ctx, lgs_comm* comm, const lgs_odometry_params* params, int32_t n_seq, const int32_t* n_frames,
                              const float* const* frames_dev, const int64_t* n_points, const float* initial_poses,
                              lgs_odometry_frame* records_all, lgs_odometry_dist_info* info);

/* The per-worker device state of lgs_batch_align (stream, registration objects, staging buffers) is kept in a
 * process-wide pool between calls, the way the reference keeps one registration_ object per node for its lifetime
 * (graph_based_slam.hpp:108).  This frees it (call with no batch in flight, e.g. at node shutdown). */
void lgs_batch_release(void);

#ifdef __cplusplus
}
#endif
#endif /* LGS_C_H_ */
