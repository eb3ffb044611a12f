// lgs/registration.hpp -- header-only C++ shim that re-exposes the exact PCL method names the reference calls
// (SURVEY.md section 8b) on top of the C ABI in lgs_c.h.  PCL-free by default; define LGS_HAVE_PCL to also get
// adapters deriving from pcl::Registration / pcl::Filter whose virtual hooks forward to the GPU (see INTEGRATION.md).
//
//   lgs::VoxelGrid                      <- pcl::VoxelGrid<pcl::PointXYZI>            (PPF:118-120, GBS:61,311-313,490-493)
//   lgs::NormalDistributionsTransform   <- pclomp::NormalDistributionsTransform      (LSM:56-72, GBS:101-119)
//   lgs::FastGICP                       <- fast_gicp::FastGICP                       (LSM:38-54, GBS:82-100)
//   lgs::IterativeClosestPoint          <- pcl::IterativeClosestPoint                (GBS:142-151, the default method)
//   lgs::GeneralizedIterativeClosestPoint <- pclomp::GeneralizedIterativeClosestPoint (LSM:73-96, GBS:120-141)
//
// Clouds are std::vector<lgs::PointXYZI> with pcl::PointXYZI's 32-byte layout; transforms are float[16]
// column-major (Eigen::Matrix4f memory order), so `Eigen::Map<Eigen::Matrix4f>(m.data())` is a view, not a copy.
#pragma once
#include <array>
#include <cfloat>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../lgs_c.h"

namespace lgs {

struct alignas(16) PointXYZI {  // byte-compatible with pcl::PointXYZI
  float x, y, z, pad0;
  float intensity, pad1, pad2, pad3;
};
static_assert(sizeof(PointXYZI) == 32, "PointXYZI must match pcl::PointXYZI");

using PointCloud = std::vector<PointXYZI>;
using Matrix4f = std::array<float, 16>;  // column-major

inline Matrix4f Identity4f() { return Matrix4f{1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1}; }

// The reference never lets exceptions escape the registration call (SURVEY.md section 8b "Error convention"); the
// shim follows it: setters and align() record failures, hasConverged() turns false, lastError() has the message.
class Context {
 public:
  explicit Context(int device = 0, void* cuda_stream = nullptr) {
    if (lgs_ctx_create(device, cuda_stream, &ctx_) != LGS_OK) throw std::runtime_error(lgs_last_error());
  }
  ~Context() { lgs_ctx_destroy(ctx_); }
  Context(const Context&) = delete;
  Context& operator=(const Context&) = delete;
  lgs_ctx* get() const { return ctx_; }

 private:
  lgs_ctx* ctx_ = nullptr;
};

inline std::shared_ptr<Context> defaultContext() {
  static std::shared_ptr<Context> c = std::make_shared<Context>(0);
  return c;
}

class VoxelGrid {
 public:
  explicit VoxelGrid(std::shared_ptr<Context> ctx = defaultContext()) : ctx_(std::move(ctx)) {}
  void setLeafSize(float lx, float ly, float lz) { leaf_ = {lx, ly, lz}; }
  void setMinimumPointsNumberPerVoxel(unsigned n) { min_pts_ = static_cast<int>(n); }
  // the prefilter node's predicates (PPF:89-112), fused into the same pass
  void setRangeCrop(double min_distance) { range_min_ = min_distance; }
  void setBoxCrop(const std::array<double, 6>& box) { box_ = box; use_box_ = true; }
  void setInputCloud(const std::shared_ptr<const PointCloud>& cloud) { input_ = cloud; }
  void filter(PointCloud& output) {
    output.clear();
    if (!input_) return;
    const int64_t n = static_cast<int64_t>(input_->size());
    std::vector<float> packed(static_cast<size_t>(n > 0 ? n : 1) * 4);
    voxel_idx_.assign(static_cast<size_t>(n), -1);
    member_rank_.assign(static_cast<size_t>(n), -1);
    ok_ = lgs_voxelgrid_filter(ctx_->get(), input_->data(), n, sizeof(PointXYZI), leaf_.data(), min_pts_, range_min_,
                               use_box_ ? box_.data() : nullptr, packed.data(), voxel_idx_.data(), member_rank_.data(), &info_) == LGS_OK;
    if (!ok_) return;
    output.resize(static_cast<size_t>(info_.n_out));
    for (int64_t i = 0; i < info_.n_out; i++)
      output[i] = PointXYZI{packed[4 * i], packed[4 * i + 1], packed[4 * i + 2], 1.0f, packed[4 * i + 3], 0, 0, 0};
  }
  const std::vector<int32_t>& voxelIndices() const { return voxel_idx_; }
  const std::vector<int32_t>& memberRanks() const { return member_rank_; }
  const lgs_voxelgrid_info& info() const { return info_; }
  bool ok() const { return ok_; }

 private:
  std::shared_ptr<Context> ctx_;
  std::array<float, 3> leaf_{0.01f, 0.01f, 0.01f};
  int min_pts_ = 0;
  double range_min_ = -1.0;
  std::array<double, 6> box_{};
  bool use_box_ = false, ok_ = true;
  std::shared_ptr<const PointCloud> input_;
  std::vector<int32_t> voxel_idx_, member_rank_;
  lgs_voxelgrid_info info_{};
};

// pcl::StatisticalOutlierRemoval<PointXYZI> as the prefilter node drives it (PPF:132-140)
class StatisticalOutlierRemoval {
 public:
  explicit StatisticalOutlierRemoval(std::shared_ptr<Context> ctx = defaultContext()) : ctx_(std::move(ctx)) {
    ok_ = lgs_sor_create(ctx_->get(), &h_) == LGS_OK;
  }
  ~StatisticalOutlierRemoval() { lgs_sor_destroy(h_); }
  StatisticalOutlierRemoval(const StatisticalOutlierRemoval&) = delete;
  StatisticalOutlierRemoval& operator=(const StatisticalOutlierRemoval&) = delete;
  void setMeanK(int k) { ok_ = lgs_sor_set_mean_k(h_, k) == LGS_OK && ok_; }
  void setStddevMulThresh(double m) { ok_ = lgs_sor_set_stddev_mul_thresh(h_, m) == LGS_OK && ok_; }
  void setNegative(bool negative) { ok_ = lgs_sor_set_negative(h_, negative ? 1 : 0) == LGS_OK && ok_; }
  void setInputCloud(const std::shared_ptr<const PointCloud>& cloud) { input_ = cloud; }
  void filter(PointCloud& output) {
    output.clear();
    if (!input_ || !h_) return;
    const int64_t n = static_cast<int64_t>(input_->size());
    std::vector<float> packed(static_cast<size_t>(n > 0 ? n : 1) * 4);
    keep_.assign(static_cast<size_t>(n), 0);
    ok_ = lgs_sor_filter(h_, input_->data(), n, sizeof(PointXYZI), packed.data(), keep_.data(), nullptr, &info_) == LGS_OK;
    if (!ok_) return;
    output.resize(static_cast<size_t>(info_.n_out));
    for (int64_t i = 0; i < info_.n_out; i++)
      output[i] = PointXYZI{packed[4 * i], packed[4 * i + 1], packed[4 * i + 2], 1.0f, packed[4 * i + 3], 0, 0, 0};
  }
  const std::vector<uint8_t>& keptMask() const { return keep_; }
  const lgs_sor_info& info() const { return info_; }
  bool ok() const { return ok_; }

 private:
  std::shared_ptr<Context> ctx_;
  lgs_sor* h_ = nullptr;
  bool ok_ = true;
  std::shared_ptr<const PointCloud> input_;
  std::vector<uint8_t> keep_;
  lgs_sor_info info_{};
};

// pcl::Registration<PointXYZI, PointXYZI> surface shared by both methods
class Registration {
 public:
  virtual ~Registration() = default;
  virtual void setInputTarget(const std::shared_ptr<const PointCloud>& cloud) = 0;
  virtual void setInputSource(const std::shared_ptr<const PointCloud>& cloud) = 0;
  virtual void align(PointCloud& output, const Matrix4f& guess = Identity4f()) = 0;
  virtual double getFitnessScore(double max_range = DBL_MAX) = 0;
  bool hasConverged() const { return ok_ && result_.converged != 0; }
  Matrix4f getFinalTransformation() const {
    Matrix4f m;
    for (int i = 0; i < 16; i++) m[i] = result_.T[i];
    return m;
  }
  const lgs_align_result& result() const { return result_; }
  const std::string& lastError() const { return error_; }

 protected:
  void check(int rc) {
    if (rc != LGS_OK) {
      ok_ = false;
      error_ = lgs_last_error();
    }
  }
  void fill_output(PointCloud& output, const std::vector<float>& packed, size_t n) {
    output.resize(n);
    for (size_t i = 0; i < n; i++) output[i] = PointXYZI{packed[4 * i], packed[4 * i + 1], packed[4 * i + 2], 1.0f, packed[4 * i + 3], 0, 0, 0};
  }
  lgs_align_result result_{};
  bool ok_ = true;
  std::string error_;
  size_t n_source_ = 0;
};

enum NeighborSearchMethod { KDTREE = LGS_NDT_KDTREE, DIRECT26 = LGS_NDT_DIRECT26, DIRECT7 = LGS_NDT_DIRECT7, DIRECT1 = LGS_NDT_DIRECT1 };

class NormalDistributionsTransform : public Registration {
 public:
  explicit NormalDistributionsTransform(std::shared_ptr<Context> ctx = defaultContext()) : ctx_(std::move(ctx)) {
    if (lgs_ndt_create(ctx_->get(), &h_) != LGS_OK) throw std::runtime_error(lgs_last_error());
  }
  ~NormalDistributionsTransform() override { lgs_ndt_destroy(h_); }
  void setNumThreads(int) {}  // OpenMP knob of the reference (NDT.h:113-115)
  void setResolution(float r) { resolution_ = r; check(lgs_ndt_set_resolution(h_, r)); }
  float getResolution() const { return resolution_; }
  void setStepSize(double s) { step_ = s; check(lgs_ndt_set_step_size(h_, s)); }
  // no counterpart in the reference: every Newton step through the restated JacobiSVD (bit-identical transforms, ~2x the time)
  void setExactNewtonStep(bool on) { check(lgs_ndt_set_exact_newton_step(h_, on ? 1 : 0)); }
  double getStepSize() const { return step_; }
  void setOutlierRatio(double o) { outlier_ = o; check(lgs_ndt_set_outlier_ratio(h_, o)); }
  double getOutlierRatio() const { return outlier_; }
  void setTransformationEpsilon(double e) { check(lgs_ndt_set_transformation_epsilon(h_, e)); }
  void setMaximumIterations(int n) { check(lgs_ndt_set_maximum_iterations(h_, n)); }
  void setNeighborhoodSearchMethod(NeighborSearchMethod m) { check(lgs_ndt_set_search_method(h_, m)); }
  void setInputTarget(const std::shared_ptr<const PointCloud>& c) override {
    check(lgs_ndt_set_target(h_, c->data(), static_cast<int64_t>(c->size()), sizeof(PointXYZI)));
  }
  void setInputSource(const std::shared_ptr<const PointCloud>& c) override {
    n_source_ = c->size();
    check(lgs_ndt_set_source(h_, c->data(), static_cast<int64_t>(c->size()), sizeof(PointXYZI)));
  }
  void align(PointCloud& output, const Matrix4f& guess = Identity4f()) override {
    ok_ = true;
    std::vector<float> packed((n_source_ ? n_source_ : 1) * 4);
    check(lgs_ndt_align(h_, guess.data(), &result_, packed.data()));
    if (ok_) fill_output(output, packed, n_source_);
  }
  double getFitnessScore(double max_range = DBL_MAX) override {
    double f = DBL_MAX;
    check(lgs_ndt_fitness(h_, max_range, &f));
    return f;
  }
  static Matrix4f convertTransform(const std::array<double, 6>& x) {  // NDT.h:214-238
    Matrix4f T = Identity4f();
    lgs_ndt_convert_transform(x.data(), T.data());
    return T;
  }
  double getTransformationProbability() const { return result_.trans_probability; }
  int getFinalNumIteration() const { return result_.iterations; }
  double calculateScore(const Matrix4f& T) {
    double s = 0;
    check(lgs_ndt_calculate_score(h_, T.data(), &s));
    return s;
  }
  lgs_ndt* handle() const { return h_; }
  // No counterpart in the reference: align this source from every guess in one resident launch per wave
  // (lgs_ndt_align_many).  Record k is bit-identical to align(output, guesses[k]); afterwards result() is the last guess's.
  // fitness_max_range < 0: no fitness, else records[k].fitness = getFitnessScore(fitness_max_range) at record k's transform.
  std::vector<lgs_align_result> alignGuesses(const std::vector<Matrix4f>& guesses, double fitness_max_range = -1.0) {
    ok_ = true;
    std::vector<lgs_ndt*> hs(guesses.size(), h_);
    std::vector<float> packed(guesses.size() * 16);
    for (size_t k = 0; k < guesses.size(); k++) std::copy(guesses[k].begin(), guesses[k].end(), packed.begin() + 16 * k);
    std::vector<lgs_align_result> out(guesses.size());
    check(lgs_ndt_align_many(hs.data(), static_cast<int32_t>(hs.size()), packed.data(), fitness_max_range < 0 ? nullptr : &fitness_max_range,
                             out.data(), nullptr));
    if (ok_ && !out.empty()) result_ = out.back();
    return out;
  }
  friend std::vector<lgs_align_result> alignMany(const std::vector<NormalDistributionsTransform*>& ndts, const std::vector<Matrix4f>& guesses,
                                                 double fitness_max_range);

 private:
  std::shared_ptr<Context> ctx_;
  lgs_ndt* h_ = nullptr;
  float resolution_ = 1.0f;
  double step_ = 0.1, outlier_ = 0.55;
};

// No counterpart in the reference: ndts[i]->align(guesses[i]) for every i in one resident launch per wave (lgs_ndt_align_many);
// the objects may repeat and must share one Context.  guesses: empty (identity) or one per object.  Each object's result()
// becomes that of its last occurrence.  On failure every object records the error (hasConverged() false, lastError()).
inline std::vector<lgs_align_result> alignMany(const std::vector<NormalDistributionsTransform*>& ndts, const std::vector<Matrix4f>& guesses = {},
                                               double fitness_max_range = -1.0) {
  std::vector<lgs_ndt*> hs;
  for (auto* x : ndts) hs.push_back(x->h_);
  std::vector<float> packed(guesses.size() * 16);
  for (size_t k = 0; k < guesses.size(); k++) std::copy(guesses[k].begin(), guesses[k].end(), packed.begin() + 16 * k);
  std::vector<lgs_align_result> out(ndts.size());
  const int rc = (!guesses.empty() && guesses.size() != ndts.size())
                     ? LGS_ERR_INVALID
                     : lgs_ndt_align_many(hs.data(), static_cast<int32_t>(hs.size()), guesses.empty() ? nullptr : packed.data(),
                                          fitness_max_range < 0 ? nullptr : &fitness_max_range, out.data(), nullptr);
  for (size_t i = 0; i < ndts.size(); i++) {
    ndts[i]->ok_ = true;
    ndts[i]->check(rc);
    if (rc == LGS_OK) ndts[i]->result_ = out[i];
  }
  return out;
}

enum class RegularizationMethod { NONE = LGS_REG_NONE, MIN_EIG, NORMALIZED_MIN_EIG, PLANE, FROBENIUS };

class FastGICP : public Registration {
 public:
  explicit FastGICP(std::shared_ptr<Context> ctx = defaultContext()) : ctx_(std::move(ctx)) {
    if (lgs_gicp_create(ctx_->get(), &h_) != LGS_OK) throw std::runtime_error(lgs_last_error());
  }
  ~FastGICP() override { lgs_gicp_destroy(h_); }
  void setNumThreads(int) {}
  void setCorrespondenceRandomness(int k) { check(lgs_gicp_set_correspondence_randomness(h_, k)); }
  void setRegularizationMethod(RegularizationMethod m) { check(lgs_gicp_set_regularization_method(h_, static_cast<int>(m))); }
  void setMaxCorrespondenceDistance(double d) { check(lgs_gicp_set_max_correspondence_distance(h_, d)); }
  void setTransformationEpsilon(double e) { check(lgs_gicp_set_transformation_epsilon(h_, e)); }
  void setRotationEpsilon(double e) { check(lgs_gicp_set_rotation_epsilon(h_, e)); }
  void setMaximumIterations(int n) { check(lgs_gicp_set_maximum_iterations(h_, n)); }
  void setInitialLambdaFactor(double f) { check(lgs_gicp_set_initial_lambda_factor(h_, f)); }
  void swapSourceAndTarget() { check(lgs_gicp_swap_source_and_target(h_)); std::swap(n_source_, n_target_); }
  void clearSource() { check(lgs_gicp_clear_source(h_)); n_source_ = 0; }
  void clearTarget() { check(lgs_gicp_clear_target(h_)); n_target_ = 0; }
  void setInputTarget(const std::shared_ptr<const PointCloud>& c) override {
    n_target_ = c->size();
    check(lgs_gicp_set_target(h_, c->data(), static_cast<int64_t>(c->size()), sizeof(PointXYZI)));
  }
  void setInputSource(const std::shared_ptr<const PointCloud>& c) override {
    n_source_ = c->size();
    check(lgs_gicp_set_source(h_, c->data(), static_cast<int64_t>(c->size()), sizeof(PointXYZI)));
  }
  void align(PointCloud& output, const Matrix4f& guess = Identity4f()) override {
    ok_ = true;
    std::vector<float> packed((n_source_ ? n_source_ : 1) * 4);
    check(lgs_gicp_align(h_, guess.data(), &result_, packed.data()));
    if (ok_) fill_output(output, packed, n_source_);
  }
  double getFitnessScore(double max_range = DBL_MAX) override {
    double f = DBL_MAX;
    check(lgs_gicp_fitness(h_, max_range, &f));
    return f;
  }
  void setDebugPrint(bool) {}  // lsq_registration.hpp:36
  double evaluateCost(const Matrix4f& relative_pose) {  // LSQ:48-50
    double c = 0;
    check(lgs_gicp_evaluate_cost(h_, relative_pose.data(), &c));
    return c;
  }
  // FG.h:60-70: covariances as n x 9 doubles (row-major 3x3 blocks of the reference's Matrix4d)
  void setSourceCovariances(const std::vector<double>& covs) { check(lgs_gicp_set_covariances(h_, 0, covs.data(), static_cast<int64_t>(covs.size() / 9))); }
  void setTargetCovariances(const std::vector<double>& covs) { check(lgs_gicp_set_covariances(h_, 1, covs.data(), static_cast<int64_t>(covs.size() / 9))); }
  std::vector<double> getSourceCovariances() {
    std::vector<double> c(n_source_ * 9);
    if (n_source_) check(lgs_gicp_export_covariances(h_, 0, c.data()));
    return c;
  }
  std::vector<double> getTargetCovariances() {
    std::vector<double> c(n_target_ * 9);
    if (n_target_) check(lgs_gicp_export_covariances(h_, 1, c.data()));
    return c;
  }
  std::array<double, 36> getFinalHessian() {
    std::array<double, 36> H{};
    check(lgs_gicp_final_hessian(h_, H.data()));
    return H;
  }
  lgs_gicp* handle() const { return h_; }

 private:
  std::shared_ptr<Context> ctx_;
  lgs_gicp* h_ = nullptr;
  size_t n_target_ = 0;
};

// pclomp::GeneralizedIterativeClosestPoint (gicp_omp.h:116-270), the "GICP" registration_method of LSM:73-96 / GBS:120-141
class GeneralizedIterativeClosestPoint : public Registration {
 public:
  explicit GeneralizedIterativeClosestPoint(std::shared_ptr<Context> ctx = defaultContext()) : ctx_(std::move(ctx)) {
    if (lgs_gicp_omp_create(ctx_->get(), &h_) != LGS_OK) throw std::runtime_error(lgs_last_error());
  }
  ~GeneralizedIterativeClosestPoint() override { lgs_gicp_omp_destroy(h_); }
  void setCorrespondenceRandomness(int k) { k_ = k; check(lgs_gicp_omp_set_correspondence_randomness(h_, k)); }
  int getCorrespondenceRandomness() const { return k_; }
  void setMaxCorrespondenceDistance(double d) { check(lgs_gicp_omp_set_max_correspondence_distance(h_, d)); }
  void setTransformationEpsilon(double e) { check(lgs_gicp_omp_set_transformation_epsilon(h_, e)); }
  void setRotationEpsilon(double e) { rot_eps_ = e; check(lgs_gicp_omp_set_rotation_epsilon(h_, e)); }
  double getRotationEpsilon() const { return rot_eps_; }
  void setMaximumIterations(int n) { check(lgs_gicp_omp_set_maximum_iterations(h_, n)); }
  void setMaximumOptimizerIterations(int n) { max_inner_ = n; check(lgs_gicp_omp_set_maximum_optimizer_iterations(h_, n)); }
  int getMaximumOptimizerIterations() const { return max_inner_; }
  // set by the nodes (LSM:90,93, GBS:138-139) and never read by the reference's computeTransformation (GO:370-516)
  void setUseReciprocalCorrespondences(bool) {}
  void setEuclideanFitnessEpsilon(double) {}
  void setRANSACIterations(int) {}
  void setInputTarget(const std::shared_ptr<const PointCloud>& c) override {
    check(lgs_gicp_omp_set_target(h_, c->data(), static_cast<int64_t>(c->size()), sizeof(PointXYZI)));
  }
  void setInputSource(const std::shared_ptr<const PointCloud>& c) override {
    n_source_ = c->size();
    check(lgs_gicp_omp_set_source(h_, c->data(), static_cast<int64_t>(c->size()), sizeof(PointXYZI)));
  }
  void align(PointCloud& output, const Matrix4f& guess = Identity4f()) override {
    ok_ = true;
    std::vector<float> packed((n_source_ ? n_source_ : 1) * 4);
    check(lgs_gicp_omp_align(h_, guess.data(), &result_, packed.data()));
    if (ok_) fill_output(output, packed, n_source_);
  }
  double getFitnessScore(double max_range = DBL_MAX) override {
    double f = DBL_MAX;
    check(lgs_gicp_omp_fitness(h_, max_range, &f));
    return f;
  }
  lgs_gicp_omp* handle() const { return h_; }

 private:
  std::shared_ptr<Context> ctx_;
  lgs_gicp_omp* h_ = nullptr;
  int k_ = 20, max_inner_ = 20;
  double rot_eps_ = 2e-3;
};

// pcl::IterativeClosestPoint<PointXYZI, PointXYZI>: the default loop-closure method (GBS:142-151)
class IterativeClosestPoint : public Registration {
 public:
  explicit IterativeClosestPoint(std::shared_ptr<Context> ctx = defaultContext()) : ctx_(std::move(ctx)) {
    if (lgs_icp_create(ctx_->get(), &h_) != LGS_OK) throw std::runtime_error(lgs_last_error());
  }
  ~IterativeClosestPoint() override { lgs_icp_destroy(h_); }
  void setMaxCorrespondenceDistance(double d) { check(lgs_icp_set_max_correspondence_distance(h_, d)); }
  void setMaximumIterations(int n) { check(lgs_icp_set_maximum_iterations(h_, n)); }
  void setTransformationEpsilon(double e) { check(lgs_icp_set_transformation_epsilon(h_, e)); }
  void setTransformationRotationEpsilon(double e) { check(lgs_icp_set_transformation_rotation_epsilon(h_, e)); }
  void setEuclideanFitnessEpsilon(double e) { check(lgs_icp_set_euclidean_fitness_epsilon(h_, e)); }
  void setRANSACIterations(int) {}  // GBS:149: no rejector is installed, PCL never reads it
  void setInputTarget(const std::shared_ptr<const PointCloud>& c) override {
    check(lgs_icp_set_target(h_, c->data(), static_cast<int64_t>(c->size()), sizeof(PointXYZI)));
  }
  void setInputSource(const std::shared_ptr<const PointCloud>& c) override {
    n_source_ = c->size();
    check(lgs_icp_set_source(h_, c->data(), static_cast<int64_t>(c->size()), sizeof(PointXYZI)));
  }
  void align(PointCloud& output, const Matrix4f& guess = Identity4f()) override {
    ok_ = true;
    std::vector<float> packed((n_source_ ? n_source_ : 1) * 4);
    check(lgs_icp_align(h_, guess.data(), &result_, packed.data()));
    if (ok_) fill_output(output, packed, n_source_);
  }
  double getFitnessScore(double max_range = DBL_MAX) override {
    double f = DBL_MAX;
    check(lgs_icp_fitness(h_, max_range, &f));
    return f;
  }
  lgs_icp* handle() const { return h_; }

 private:
  std::shared_ptr<Context> ctx_;
  lgs_icp* h_ = nullptr;
};

// Device-resident key_frame_array_ (LSM:196-212, GBS:297-313): key frames are uploaded once; sub-maps are assembled on the
// GPU and handed to a registration as device clouds; loop candidates are verified without the clouds leaving the GPU.
class KeyFrameArray {
 public:
  explicit KeyFrameArray(std::shared_ptr<Context> ctx = defaultContext()) : ctx_(std::move(ctx)) {
    if (lgs_keyframes_create(ctx_->get(), &h_) != LGS_OK) throw std::runtime_error(lgs_last_error());
  }
  ~KeyFrameArray() { lgs_keyframes_destroy(h_); }
  KeyFrameArray(const KeyFrameArray&) = delete;
  KeyFrameArray& operator=(const KeyFrameArray&) = delete;
  // key_frame_array_.keyframes.emplace_back(key_frame): returns the key frame's id, -1 on failure
  int push(const PointCloud& cloud, const Matrix4f& pose, double accum_distance = 0.0) {
    int32_t id = -1;
    if (lgs_keyframes_push(h_, cloud.data(), static_cast<int64_t>(cloud.size()), sizeof(PointXYZI), pose.data(), &id) != LGS_OK) return -1;
    lgs_keyframes_set_accum_distance(h_, id, accum_distance);
    return id;
  }
  bool setPose(int id, const Matrix4f& pose) { return lgs_keyframes_set_pose(h_, id, pose.data()) == LGS_OK; }
  size_t size() const {
    int64_t n = 0;
    lgs_keyframes_size(h_, &n, nullptr);
    return static_cast<size_t>(n);
  }
  // detect_loop_with_accum_dist (GBS:157-187); returns the nearest candidate (the one GBS:263-280 picks) or -1
  int detectLoop(int latest_id, double accumulate_distance_threshold, double search_for_candidate_threshold, std::vector<int32_t>* candidates = nullptr) {
    std::vector<int32_t> c(size() ? size() : 1);
    int32_t n = 0, nearest = -1;
    if (lgs_keyframes_detect_loop(h_, latest_id, accumulate_distance_threshold, search_for_candidate_threshold, c.data(), static_cast<int32_t>(c.size()), &n,
                                  &nearest) != LGS_OK)
      return -1;
    if (candidates) candidates->assign(c.begin(), c.begin() + n);
    return nearest;
  }
  // the sub-map of `ids` (in that order), optionally VoxelGrid-filtered: a device cloud valid until the next call
  bool assemble(const std::vector<int32_t>& ids, float leaf, const float** cloud_dev, int64_t* n) {
    float* p = nullptr;
    const int rc = lgs_keyframes_assemble(h_, ids.data(), static_cast<int32_t>(ids.size()), leaf, &p, n);
    *cloud_dev = p;
    return rc == LGS_OK;
  }
  lgs_keyframes* handle() const { return h_; }

 private:
  std::shared_ptr<Context> ctx_;
  lgs_keyframes* h_ = nullptr;
};

// the flat frame list of lgs_odometry_run*
struct OdometryInput {
  std::vector<int32_t> n_frames;
  std::vector<const void*> frames;
  std::vector<int64_t> n_points;
  explicit OdometryInput(const std::vector<std::vector<PointCloud>>& sequences) {
    for (const auto& seq : sequences) {
      n_frames.push_back(static_cast<int32_t>(seq.size()));
      for (const auto& c : seq) {
        frames.push_back(c.data());
        n_points.push_back(static_cast<int64_t>(c.size()));
      }
    }
  }
};

// Offline odometry (lgs_odometry_run): the scan matcher's key-frame loop over each recorded sequence of sensor-frame sweeps.
// keyframes: empty, or one entry per sequence (nullptr or an empty array on ctx's device, which the run fills).  Returns the
// records in (sequence, frame) order; throws std::runtime_error with lgs_last_error() when the call is refused or fails.
inline std::vector<lgs_odometry_frame> odometry(const std::vector<std::vector<PointCloud>>& sequences, const lgs_odometry_params& params,
                                                const std::vector<Matrix4f>& initial_poses = {}, const std::vector<KeyFrameArray*>& keyframes = {},
                                                std::shared_ptr<Context> ctx = defaultContext()) {
  const OdometryInput in(sequences);
  std::vector<lgs_keyframes*> kf;
  for (KeyFrameArray* k : keyframes) kf.push_back(k ? k->handle() : nullptr);
  std::vector<lgs_odometry_frame> out(in.frames.size());
  const int rc = lgs_odometry_run(ctx->get(), &params, static_cast<int32_t>(sequences.size()), in.n_frames.data(), in.frames.data(), in.n_points.data(),
                                  sizeof(PointXYZI), initial_poses.empty() ? nullptr : initial_poses[0].data(), kf.empty() ? nullptr : kf.data(),
                                  out.data());
  if (rc != LGS_OK) throw std::runtime_error(lgs_last_error());
  return out;
}

// lgs_odometry_run_dist (collective over comm, on ctx's device): every rank passes the same sequence list; of the sequences this
// rank does not own only the cloud sizes are read.  Returns every record on every rank.
inline std::vector<lgs_odometry_frame> odometryDist(lgs_comm* comm, const std::vector<std::vector<PointCloud>>& sequences, const lgs_odometry_params& params,
                                                    const std::vector<Matrix4f>& initial_poses = {}, lgs_odometry_dist_info* info = nullptr,
                                                    std::shared_ptr<Context> ctx = defaultContext()) {
  const OdometryInput in(sequences);
  std::vector<lgs_odometry_frame> out(in.frames.size());
  const int rc = lgs_odometry_run_dist(ctx->get(), comm, &params, static_cast<int32_t>(sequences.size()), in.n_frames.data(), in.frames.data(),
                                       in.n_points.data(), sizeof(PointXYZI), initial_poses.empty() ? nullptr : initial_poses[0].data(), out.data(), info);
  if (rc != LGS_OK) throw std::runtime_error(lgs_last_error());
  return out;
}

}  // namespace lgs

#ifdef LGS_HAVE_PCL
// Adapters for a tree that has PCL: they derive from pcl::Registration so that the nodes' `registration_` pointer
// (lidar_scan_matcher.hpp:99, graph_based_slam.hpp:108) can hold them unchanged.  pcl::PointXYZI is a 32-byte record,
// so the cloud storage goes to the C ABI as is (stride 32), no host-side repacking.  Not compiled by this repo's
// tests (PCL is not installed in the build container); INTEGRATION.md shows the wiring.
#include <pcl/registration/registration.h>
namespace lgs {

// pcl::Registration::initCompute() (called by the non-virtual align shell) rebuilds PCL's FLANN kd-tree over the target after
// every setInputTarget unless the search method was installed with force_no_recompute: the adapters install an empty tree
// that way, so no host-side kd-tree over the 1 M-point map is ever built.  getFitnessScore is not virtual either: call it
// through the adapter type (INTEGRATION.md section 4).
template <typename Reg>
inline void lgs_skip_pcl_target_tree(Reg* reg) {
  typename Reg::KdTreePtr tree(new typename Reg::KdTree);
  reg->setSearchMethodTarget(tree, /*force_no_recompute=*/true);
}

class PclNdtAdapter : public pcl::Registration<pcl::PointXYZI, pcl::PointXYZI> {
 public:
  using Base = pcl::Registration<pcl::PointXYZI, pcl::PointXYZI>;
  NormalDistributionsTransform impl;
  PclNdtAdapter() {
    reg_name_ = "lgs::NormalDistributionsTransform";
    lgs_skip_pcl_target_tree(this);
  }
  void setInputTarget(const Base::PointCloudTargetConstPtr& cloud) override {
    Base::setInputTarget(cloud);
    lgs_ndt_set_target(impl.handle(), cloud->points.data(), static_cast<int64_t>(cloud->size()), sizeof(pcl::PointXYZI));
  }
  void setInputSource(const Base::PointCloudSourceConstPtr& cloud) override {
    Base::setInputSource(cloud);
    lgs_ndt_set_source(impl.handle(), cloud->points.data(), static_cast<int64_t>(cloud->size()), sizeof(pcl::PointXYZI));
  }
  double getFitnessScore(double max_range = std::numeric_limits<double>::max()) {
    double f = std::numeric_limits<double>::max();
    lgs_ndt_fitness(impl.handle(), max_range, &f);
    return f;
  }

 protected:
  void computeTransformation(Base::PointCloudSource& output, const Eigen::Matrix4f& guess) override {
    lgs_ndt_set_transformation_epsilon(impl.handle(), transformation_epsilon_);
    lgs_ndt_set_maximum_iterations(impl.handle(), max_iterations_);
    lgs_align_result r{};
    std::vector<float> packed(output.size() * 4 + 4);
    const int rc = lgs_ndt_align(impl.handle(), guess.data(), &r, packed.data());
    converged_ = rc == LGS_OK && r.converged != 0;
    nr_iterations_ = r.iterations;
    final_transformation_ = Eigen::Map<const Eigen::Matrix4f>(r.T);
    for (size_t i = 0; i < output.size(); i++) {
      output[i].x = packed[4 * i];
      output[i].y = packed[4 * i + 1];
      output[i].z = packed[4 * i + 2];
    }
  }
};

class PclGicpAdapter : public pcl::Registration<pcl::PointXYZI, pcl::PointXYZI> {
 public:
  using Base = pcl::Registration<pcl::PointXYZI, pcl::PointXYZI>;
  FastGICP impl;
  PclGicpAdapter() {
    reg_name_ = "lgs::FastGICP";
    lgs_skip_pcl_target_tree(this);
  }
  void setInputTarget(const Base::PointCloudTargetConstPtr& cloud) override {
    Base::setInputTarget(cloud);
    lgs_gicp_set_target(impl.handle(), cloud->points.data(), static_cast<int64_t>(cloud->size()), sizeof(pcl::PointXYZI));
  }
  void setInputSource(const Base::PointCloudSourceConstPtr& cloud) override {
    Base::setInputSource(cloud);
    lgs_gicp_set_source(impl.handle(), cloud->points.data(), static_cast<int64_t>(cloud->size()), sizeof(pcl::PointXYZI));
  }
  double getFitnessScore(double max_range = std::numeric_limits<double>::max()) {
    double f = std::numeric_limits<double>::max();
    lgs_gicp_fitness(impl.handle(), max_range, &f);
    return f;
  }

 protected:
  void computeTransformation(Base::PointCloudSource& output, const Eigen::Matrix4f& guess) override {
    lgs_gicp_set_transformation_epsilon(impl.handle(), transformation_epsilon_);
    lgs_gicp_set_maximum_iterations(impl.handle(), max_iterations_);
    lgs_gicp_set_max_correspondence_distance(impl.handle(), corr_dist_threshold_);
    lgs_align_result r{};
    std::vector<float> packed(output.size() * 4 + 4);
    const int rc = lgs_gicp_align(impl.handle(), guess.data(), &r, packed.data());
    converged_ = rc == LGS_OK && r.converged != 0;
    nr_iterations_ = r.iterations;
    final_transformation_ = Eigen::Map<const Eigen::Matrix4f>(r.T);
    for (size_t i = 0; i < output.size(); i++) {
      output[i].x = packed[4 * i];
      output[i].y = packed[4 * i + 1];
      output[i].z = packed[4 * i + 2];
    }
  }
};

// pclomp::GeneralizedIterativeClosestPoint ("GICP", LSM:73-96 / GBS:120-141) and pcl::IterativeClosestPoint ("ICP",
// GBS:142-151) behind the same pcl::Registration base.  The pcl::Registration members the nodes set
// (max_iterations_, transformation_epsilon_, corr_dist_threshold_, euclidean_fitness_epsilon_) are forwarded at align time.
class PclGicpOmpAdapter : public pcl::Registration<pcl::PointXYZI, pcl::PointXYZI> {
 public:
  using Base = pcl::Registration<pcl::PointXYZI, pcl::PointXYZI>;
  GeneralizedIterativeClosestPoint impl;
  PclGicpOmpAdapter() {
    reg_name_ = "lgs::GeneralizedIterativeClosestPoint";
    lgs_skip_pcl_target_tree(this);
    max_iterations_ = 200;            // gicp_omp.h:121-125
    transformation_epsilon_ = 5e-4;
    corr_dist_threshold_ = 5.;
  }
  void setInputTarget(const Base::PointCloudTargetConstPtr& cloud) override {
    Base::setInputTarget(cloud);
    lgs_gicp_omp_set_target(impl.handle(), cloud->points.data(), static_cast<int64_t>(cloud->size()), sizeof(pcl::PointXYZI));
  }
  void setInputSource(const Base::PointCloudSourceConstPtr& cloud) override {
    Base::setInputSource(cloud);
    lgs_gicp_omp_set_source(impl.handle(), cloud->points.data(), static_cast<int64_t>(cloud->size()), sizeof(pcl::PointXYZI));
  }
  double getFitnessScore(double max_range = std::numeric_limits<double>::max()) {
    double f = std::numeric_limits<double>::max();
    lgs_gicp_omp_fitness(impl.handle(), max_range, &f);
    return f;
  }

 protected:
  void computeTransformation(Base::PointCloudSource& output, const Eigen::Matrix4f& guess) override {
    lgs_gicp_omp_set_transformation_epsilon(impl.handle(), transformation_epsilon_);
    lgs_gicp_omp_set_maximum_iterations(impl.handle(), max_iterations_);
    lgs_gicp_omp_set_max_correspondence_distance(impl.handle(), corr_dist_threshold_);
    lgs_align_result r{};
    std::vector<float> packed(output.size() * 4 + 4);
    const int rc = lgs_gicp_omp_align(impl.handle(), guess.data(), &r, packed.data());
    converged_ = rc == LGS_OK && r.converged != 0;
    nr_iterations_ = r.iterations;
    final_transformation_ = Eigen::Map<const Eigen::Matrix4f>(r.T);
    for (size_t i = 0; i < output.size(); i++) {
      output[i].x = packed[4 * i];
      output[i].y = packed[4 * i + 1];
      output[i].z = packed[4 * i + 2];
    }
  }
};

class PclIcpAdapter : public pcl::Registration<pcl::PointXYZI, pcl::PointXYZI> {
 public:
  using Base = pcl::Registration<pcl::PointXYZI, pcl::PointXYZI>;
  IterativeClosestPoint impl;
  PclIcpAdapter() {
    reg_name_ = "lgs::IterativeClosestPoint";
    lgs_skip_pcl_target_tree(this);
  }
  void setInputTarget(const Base::PointCloudTargetConstPtr& cloud) override {
    Base::setInputTarget(cloud);
    lgs_icp_set_target(impl.handle(), cloud->points.data(), static_cast<int64_t>(cloud->size()), sizeof(pcl::PointXYZI));
  }
  void setInputSource(const Base::PointCloudSourceConstPtr& cloud) override {
    Base::setInputSource(cloud);
    lgs_icp_set_source(impl.handle(), cloud->points.data(), static_cast<int64_t>(cloud->size()), sizeof(pcl::PointXYZI));
  }
  double getFitnessScore(double max_range = std::numeric_limits<double>::max()) {
    double f = std::numeric_limits<double>::max();
    lgs_icp_fitness(impl.handle(), max_range, &f);
    return f;
  }

 protected:
  void computeTransformation(Base::PointCloudSource& output, const Eigen::Matrix4f& guess) override {
    lgs_icp_set_transformation_epsilon(impl.handle(), transformation_epsilon_);
    lgs_icp_set_transformation_rotation_epsilon(impl.handle(), transformation_rotation_epsilon_);
    lgs_icp_set_euclidean_fitness_epsilon(impl.handle(), euclidean_fitness_epsilon_);
    lgs_icp_set_maximum_iterations(impl.handle(), max_iterations_);
    lgs_icp_set_max_correspondence_distance(impl.handle(), corr_dist_threshold_);
    lgs_align_result r{};
    std::vector<float> packed(output.size() * 4 + 4);
    const int rc = lgs_icp_align(impl.handle(), guess.data(), &r, packed.data());
    converged_ = rc == LGS_OK && r.converged != 0;
    nr_iterations_ = r.iterations;
    final_transformation_ = Eigen::Map<const Eigen::Matrix4f>(r.T);
    for (size_t i = 0; i < output.size(); i++) {
      output[i].x = packed[4 * i];
      output[i].y = packed[4 * i + 1];
      output[i].z = packed[4 * i + 2];
    }
  }
};

}  // namespace lgs
#endif
