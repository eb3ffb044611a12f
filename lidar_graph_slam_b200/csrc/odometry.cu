// Offline multi-sequence odometry: the key-frame loop of the scan matcher's callback_cloud (LSM:122-250) run over whole
// recorded sequences, composed from the device paths the node's calls map to (DESIGN section 8):
//   prefilter (range crop + VoxelGrid, optional SOR; voxelgrid.cu, outlier.cu) in the sensor frame
//   -> base_from_sensor (transform_cloud, the transform_pcl arithmetic of the key-frame assembly)
//   -> setInputSource + align(pose after the previous frame) -> key-frame test on the host
//   -> on a key frame: push into the device key-frame array and rebuild the target from the newest window
//      (Matcher::set_target_keyframes: incremental for NDT, assemble + set_target_dev for GICP).
// The host reads only what the loop decides on: the align's record.  A sequence is one problem per GPU (the NDT align is
// a cooperative launch over every SM), so the sequences of one rank run one after another; lgs_odometry_run_dist deals
// whole sequences to the ranks and gathers the records once.
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <string>
#include <vector>

#include "dist.cuh"
#include "matcher.cuh"
#include "voxel_common.cuh"

using namespace lgs;

namespace {

struct Profile {
  double frames = 0, prefilter_ms = 0, align_ms = 0, keyframe_ms = 0;
};
thread_local Profile g_profile;

// The parameters with every default resolved (the scan-matcher column of SURVEY Appendix C).
struct Params {
  lgs_odometry_params p;
  float extrinsic[16];
};

int validate(lgs_ctx* ctx, const lgs_odometry_params* params, int32_t n_seq, const int32_t* n_frames, const void* const* frames,
             const int64_t* n_points, bool host, int32_t stride, const std::vector<char>& owned, lgs_keyframes* const* keyframes, Params* out) {
  LGS_REQUIRE(ctx && params, "null argument");
  LGS_REQUIRE(n_seq >= 0, "negative sequence count");
  LGS_REQUIRE(n_seq == 0 || (n_frames && n_points), "null frame counts");
  const lgs_odometry_params& q = *params;
  LGS_REQUIRE(q.method == LGS_METHOD_NDT || q.method == LGS_METHOD_GICP || q.method == LGS_METHOD_GICP_OMP,
              "method must be LGS_METHOD_NDT, _GICP or _GICP_OMP (the scan matcher offers no ICP)");
  LGS_REQUIRE(q.max_scan_accumulate_num >= 1, "max_scan_accumulate_num must be >= 1");
  LGS_REQUIRE(q.sor_mean_k <= 31, "sor_mean_k must be <= 31");
  LGS_REQUIRE(q.range_min < 0 || q.leaf > 0, "the range crop runs inside the VoxelGrid: range_min >= 0 needs leaf > 0");
  LGS_REQUIRE(!host || (stride >= 12 && stride % 4 == 0), "stride_bytes must be a multiple of 4 and >= 12");
  int64_t f = 0;
  for (int32_t s = 0; s < n_seq; s++) {
    LGS_REQUIRE(n_frames[s] >= 0, "negative frame count");
    f += n_frames[s];
    LGS_REQUIRE(f < (int64_t(1) << 31), "more than 2^31 frames");
  }
  int64_t i = 0;
  for (int32_t s = 0; s < n_seq; s++) {
    for (int32_t k = 0; k < n_frames[s]; k++, i++) {
      LGS_REQUIRE(n_points[i] >= 0 && n_points[i] < (int64_t(1) << 31), "point count out of range");
      if ((owned.empty() || owned[s]) && n_points[i] > 0) LGS_REQUIRE(frames && frames[i], "null cloud in a sequence this call runs");
    }
    if (keyframes && keyframes[s]) {
      LGS_REQUIRE(keyframes_count(keyframes[s]) == 0, "keyframes[s] must be empty");
      LGS_REQUIRE(keyframes_device(keyframes[s]) == ctx->device, "keyframes[s] lives on another device");
    }
  }
  Params& r = *out;
  r.p = q;
  lgs_odometry_params& p = r.p;
  if (p.method == LGS_METHOD_NDT) {
    if (p.ndt_resolution <= 0) p.ndt_resolution = 2.0f;
    if (p.ndt_step_size <= 0) p.ndt_step_size = 0.1;
    if (p.transformation_epsilon <= 0) p.transformation_epsilon = 0.01;
    if (p.max_iterations <= 0) p.max_iterations = 64;
  } else {
    if (p.k_correspondences <= 0) p.k_correspondences = 20;
    if (p.max_correspondence_distance <= 0) p.max_correspondence_distance = 2.0;
    if (p.transformation_epsilon <= 0) p.transformation_epsilon = 0.01;
    if (p.max_iterations <= 0) p.max_iterations = 64;
    if (p.max_optimizer_iterations <= 0) p.max_optimizer_iterations = 20;
  }
  if (p.keyframe_displacement <= 0) p.keyframe_displacement = 1.0;
  bool zero = true;
  for (int a = 0; a < 16; a++) zero = zero && p.base_from_sensor[a] == 0.0f;
  for (int a = 0; a < 16; a++) r.extrinsic[a] = zero ? ((a % 5) == 0 ? 1.0f : 0.0f) : p.base_from_sensor[a];
  return LGS_OK;
}

// Where the frames come from.  Device form: the caller's packed clouds.  Host form: two pinned staging buffers and two
// device buffers on a copy stream; frame k+1 is copied while frame k aligns, ordered by events in both directions.
struct FrameSource {
  lgs_ctx* ctx;
  const void* const* frames;
  const int64_t* n_points;
  bool host;
  int32_t stride;
  cudaStream_t copy = nullptr;
  PinnedBuf pin[2];
  DevBuf raw[2];
  DevBuf packed;
  cudaEvent_t uploaded[2] = {nullptr, nullptr}, consumed[2] = {nullptr, nullptr};
  int64_t staged[2] = {-1, -1};  // frame index held by each slot

  ~FrameSource() {
    if (copy) cudaStreamSynchronize(copy);
    for (int b = 0; b < 2; b++) {
      if (uploaded[b]) cudaEventDestroy(uploaded[b]);
      if (consumed[b]) cudaEventDestroy(consumed[b]);
      pin[b].release();
      raw[b].release();
    }
    packed.release();
    if (copy) cudaStreamDestroy(copy);
  }
  int init() {
    if (!host) return LGS_OK;
    LGS_CUDA(cudaStreamCreateWithFlags(&copy, cudaStreamNonBlocking));
    for (int b = 0; b < 2; b++) {
      LGS_CUDA(cudaEventCreateWithFlags(&uploaded[b], cudaEventDisableTiming));
      LGS_CUDA(cudaEventCreateWithFlags(&consumed[b], cudaEventDisableTiming));
    }
    return LGS_OK;
  }
  // host form: start the upload of frame i into slot i % 2
  int stage(int64_t i) {
    if (!host || i < 0) return LGS_OK;
    const int b = static_cast<int>(i & 1);
    const size_t bytes = static_cast<size_t>(n_points[i]) * stride;
    LGS_CUDA(cudaEventSynchronize(uploaded[b]));  // the slot's previous copy has left the pinned buffer
    staged[b] = i;
    if (bytes == 0) return LGS_OK;
    LGS_TRY(pin[b].reserve(bytes));
    memcpy(pin[b].p, frames[i], bytes);
    if (bytes > raw[b].cap) LGS_CUDA(cudaEventSynchronize(consumed[b]));  // reserve frees the old buffer
    LGS_TRY(raw[b].reserve(bytes));
    LGS_CUDA(cudaStreamWaitEvent(copy, consumed[b], 0));  // the previous frame of this slot has been read on ctx's stream
    LGS_CUDA(cudaMemcpyAsync(raw[b].p, pin[b].p, bytes, cudaMemcpyHostToDevice, copy));
    LGS_CUDA(cudaEventRecord(uploaded[b], copy));
    return LGS_OK;
  }
  // frame i as a packed xyzi device cloud, usable on ctx's stream
  int take(int64_t i, const float4** out) {
    const int64_t n = n_points[i];
    if (!host) {
      *out = static_cast<const float4*>(frames[i]);
      return LGS_OK;
    }
    const int b = static_cast<int>(i & 1);
    if (staged[b] != i) {
      set_error("odometry: frame %lld was not staged", static_cast<long long>(i));
      return LGS_ERR_STATE;
    }
    LGS_CUDA(cudaStreamWaitEvent(ctx->stream, uploaded[b], 0));
    if (stride == 16) {
      *out = raw[b].as<float4>();
      return LGS_OK;
    }
    LGS_TRY(packed.reserve(static_cast<size_t>(std::max<int64_t>(n, 1)) * 16));
    LGS_TRY(repack_cloud(ctx, raw[b].p, n, stride, packed.as<float4>()));
    *out = packed.as<float4>();
    return LGS_OK;
  }
  // ctx's stream has read everything it needs of frame i
  int release(int64_t i) {
    if (!host) return LGS_OK;
    LGS_CUDA(cudaEventRecord(consumed[i & 1], ctx->stream));
    return LGS_OK;
  }
};

struct StageTimer {
  bool on;
  cudaStream_t st;
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  explicit StageTimer(cudaStream_t s) : st(s) {
    const char* e = getenv("LGS_ODOMETRY_PROFILE");
    on = e && e[0] == '1';
    if (on)
      for (auto& x : ev) cudaEventCreate(&x);
  }
  ~StageTimer() {
    for (auto& x : ev)
      if (x) cudaEventDestroy(x);
  }
  void mark(int k) {
    if (on) cudaEventRecord(ev[k], st);
  }
  // ev[0..3] = frame start, prefilter done, align done, key-frame update done (the last one reused when nothing happens)
  int add(bool keyframe) {
    if (!on) return LGS_OK;
    LGS_CUDA(cudaEventSynchronize(ev[3]));
    float a = 0, b = 0, c = 0;
    LGS_CUDA(cudaEventElapsedTime(&a, ev[0], ev[1]));
    LGS_CUDA(cudaEventElapsedTime(&b, ev[1], ev[2]));
    LGS_CUDA(cudaEventElapsedTime(&c, ev[2], ev[3]));
    g_profile.frames += 1;
    g_profile.prefilter_ms += a;
    g_profile.align_ms += b;
    if (keyframe) g_profile.keyframe_ms += c;
    return LGS_OK;
  }
};

// Per-run buffers and objects shared by the sequences of one call.
struct Driver {
  lgs_ctx* ctx;
  const Params& P;
  FrameSource& src;
  lgs_sor* sor = nullptr;
  DevBuf vg_out, sor_out, base;
  Driver(lgs_ctx* c, const Params& p, FrameSource& s) : ctx(c), P(p), src(s) {}
  ~Driver() {
    if (sor) lgs_sor_destroy(sor);
    vg_out.release();
    sor_out.release();
    base.release();
  }
  int init() {
    if (P.p.sor_mean_k > 0) {  // PPF:136-138
      LGS_TRY(lgs_sor_create(ctx, &sor));
      LGS_TRY(lgs_sor_set_mean_k(sor, P.p.sor_mean_k));
      LGS_TRY(lgs_sor_set_stddev_mul_thresh(sor, P.p.sor_stddev_mul));
    }
    return src.init();
  }

  // frame i: prefilter in the sensor frame, then the base-frame cloud in `base`; returns its size
  int prefilter(int64_t i, int64_t* n_out) {
    const float4* cur = nullptr;
    LGS_TRY(src.take(i, &cur));
    int64_t n = src.n_points[i];
    if (P.p.leaf > 0 && n > 0) {  // PPF:102-121
      LGS_TRY(vg_out.reserve(static_cast<size_t>(n) * 16));
      const float leaf[3] = {P.p.leaf, P.p.leaf, P.p.leaf};
      lgs_voxelgrid_info info;
      LGS_TRY(voxelgrid_device(ctx, cur, n, leaf, 0, P.p.range_min, nullptr, vg_out.as<float4>(), nullptr, nullptr, &info));
      cur = vg_out.as<float4>();
      n = info.n_out;
    }
    if (sor && n > 0) {  // PPF:132-140
      LGS_TRY(sor_out.reserve(static_cast<size_t>(n) * 16));
      lgs_sor_info info;
      LGS_TRY(lgs_sor_filter_dev(sor, reinterpret_cast<const float*>(cur), n, sor_out.as<float>(), nullptr, nullptr, &info));
      cur = sor_out.as<float4>();
      n = info.n_out;
    }
    LGS_TRY(base.reserve(static_cast<size_t>(std::max<int64_t>(n, 1)) * 16));
    LGS_TRY(transform_cloud(ctx, cur, n, P.extrinsic, base.as<float4>()));  // LSM:127-131
    LGS_TRY(src.release(i));
    *n_out = n;
    return LGS_OK;
  }

  // a key frame (LSM:183-212): the base-frame cloud with pose T, its path length and f64 position, then the target window
  int add_keyframe(Matcher& reg, lgs_keyframes* kf, bool shared_stream, const float* T, double accum, int32_t* id) {
    if (!shared_stream) LGS_CUDA(cudaStreamSynchronize(ctx->stream));  // `base` is complete before the array's stream copies it
    LGS_TRY(lgs_keyframes_push_dev(kf, base.as<float>(), base_n, T, id));
    if (!shared_stream) LGS_TRY(keyframes_wait_resident(kf));  // and copied before ctx's stream reuses `base`
    LGS_TRY(lgs_keyframes_set_accum_distance(kf, *id, accum));
    const double pos[3] = {T[12], T[13], T[14]};
    LGS_TRY(lgs_keyframes_set_position(kf, *id, pos));
    std::vector<int32_t> ids;
    for (int32_t k = *id; k >= 0 && k > *id - P.p.max_scan_accumulate_num; k--) ids.push_back(k);  // newest first
    return reg.set_target_keyframes(kf, ids);  // LSM:199-212 without caching on identity (Appendix A #9)
  }

  int64_t base_n = 0;

  int run_sequence(int32_t seq, int64_t first, int32_t n_frames, const float* T0, lgs_keyframes* user_kf, int64_t next_first,
                   lgs_odometry_frame* out) {
    lgs_keyframes* kf = user_kf;
    lgs_keyframes* scratch = nullptr;
    if (!kf) {
      LGS_TRY(lgs_keyframes_create(ctx, &scratch));
      kf = scratch;
    }
    struct Free {
      lgs_keyframes* k;
      ~Free() {
        if (k) lgs_keyframes_destroy(k);
      }
    } free_scratch{scratch};
    Matcher reg;  // created fresh so that no state crosses from one sequence to the next, and destroyed before the scratch
                  // array its NDT target refers to
    LGS_TRY(reg.create(ctx, P.p.method));
    const lgs_odometry_params& p = P.p;  // NDT LSM:56-72, FastGICP LSM:38-54, pclomp GICP LSM:73-96
    LGS_TRY(reg.configure({p.max_iterations, p.transformation_epsilon, p.max_correspondence_distance, p.k_correspondences, p.ndt_resolution,
                           p.ndt_step_size, p.max_optimizer_iterations, 0.0}));
    // the array runs its copies on its own context's stream; with a context of its own it is synchronised around a push
    const bool shared_stream = keyframes_stream(kf) == ctx->stream;
    float T[16], T_kf[16];
    if (T0)
      memcpy(T, T0, sizeof(T));
    else
      for (int a = 0; a < 16; a++) T[a] = (a % 5) == 0 ? 1.0f : 0.0f;
    double accum = 0.0;
    StageTimer timer(ctx->stream);
    for (int32_t k = 0; k < n_frames; k++) {
      const int64_t i = first + k;
      timer.mark(0);
      LGS_TRY(prefilter(i, &base_n));
      LGS_TRY(src.stage(k + 1 < n_frames ? i + 1 : next_first));  // the next frame's copy runs under this frame's align
      timer.mark(1);
      lgs_odometry_frame& r = out[k];
      memset(&r, 0, sizeof(r));
      r.sequence = seq;
      r.frame = k;
      r.n_source = base_n;
      r.keyframe_id = -1;
      bool keyframe = false;
      if (k == 0) {  // LSM:133-160: the first cloud is key frame 0 and the target, at the initial pose
        timer.mark(2);
        LGS_TRY(add_keyframe(reg, kf, shared_stream, T, accum, &r.keyframe_id));
        memcpy(T_kf, T, sizeof(T));
        r.converged = 1;
        keyframe = true;
      } else {
        LGS_TRY(reg.set_source_dev(base.as<float>(), base_n));  // LSM:162
        lgs_align_result a;
        LGS_TRY(reg.align(T, &a));  // LSM:165, guess = the pose after the previous frame
        timer.mark(2);
        r.converged = a.converged;
        r.iterations = a.iterations;
        r.evaluations = a.evaluations;
        r.trans_probability = a.trans_probability;
        if (a.converged) {  // LSM:167-170: a frame that did not converge is dropped
          memcpy(T, a.T, sizeof(T));
          // LSM:183: f32 norm of the f32 translation difference, compared in f64
          const float dx = T[12] - T_kf[12], dy = T[13] - T_kf[13], dz = T[14] - T_kf[14];
          const float delta = std::sqrt((dx * dx + dy * dy) + dz * dz);
          if (static_cast<double>(delta) >= P.p.keyframe_displacement) {
            accum += static_cast<double>(delta);  // LSM:193
            LGS_TRY(add_keyframe(reg, kf, shared_stream, T, accum, &r.keyframe_id));
            memcpy(T_kf, T, sizeof(T));
            keyframe = true;
          }
        }
      }
      timer.mark(3);
      memcpy(r.T, T, sizeof(T));
      r.accum_distance = accum;
      LGS_TRY(timer.add(keyframe));
    }
    LGS_CUDA(cudaStreamSynchronize(ctx->stream));
    return LGS_OK;
  }
};

// Runs the sequences listed in `local` (ascending) one after another; records of sequence s go to out + offset[s].
int run_local(lgs_ctx* ctx, const Params& P, const int32_t* n_frames, const void* const* frames, const int64_t* n_points, bool host, int32_t stride,
              const float* initial_poses, lgs_keyframes* const* keyframes, const std::vector<int32_t>& local, const std::vector<int64_t>& offset,
              lgs_odometry_frame* out) {
  LGS_TRY(use_device(ctx));
  FrameSource src{ctx, frames, n_points, host, stride};
  Driver d(ctx, P, src);
  LGS_TRY(d.init());
  // the first non-empty local sequence's first frame is staged up front; each frame then stages the one after it
  std::vector<int64_t> first_of;
  for (int32_t s : local)
    if (n_frames[s] > 0) first_of.push_back(offset[s]);
  if (!first_of.empty()) LGS_TRY(src.stage(first_of[0]));
  size_t nxt = 0;
  for (int32_t s : local) {
    if (n_frames[s] == 0) continue;
    nxt++;
    const int64_t next_first = nxt < first_of.size() ? first_of[nxt] : -1;
    LGS_TRY(d.run_sequence(s, offset[s], n_frames[s], initial_poses ? initial_poses + 16 * static_cast<size_t>(s) : nullptr,
                           keyframes ? keyframes[s] : nullptr, next_first, out + offset[s]));
  }
  return LGS_OK;
}

std::vector<int64_t> frame_offsets(int32_t n_seq, const int32_t* n_frames) {
  std::vector<int64_t> off(static_cast<size_t>(n_seq) + 1, 0);
  for (int32_t s = 0; s < n_seq; s++) off[s + 1] = off[s] + n_frames[s];
  return off;
}

int run_all(lgs_ctx* ctx, const lgs_odometry_params* params, int32_t n_seq, const int32_t* n_frames, const void* const* frames, const int64_t* n_points,
            bool host, int32_t stride, const float* initial_poses, lgs_keyframes* const* keyframes, lgs_odometry_frame* records) {
  Params P;
  LGS_TRY(validate(ctx, params, n_seq, n_frames, frames, n_points, host, stride, {}, keyframes, &P));
  const std::vector<int64_t> off = frame_offsets(n_seq, n_frames);
  LGS_REQUIRE(records || off[n_seq] == 0, "null records");
  std::vector<int32_t> all(static_cast<size_t>(n_seq));
  for (int32_t s = 0; s < n_seq; s++) all[s] = s;
  return run_local(ctx, P, n_frames, frames, n_points, host, stride, initial_poses, keyframes, all, off, records);
}

int run_dist(lgs_ctx* ctx, lgs_comm* comm, const lgs_odometry_params* params, int32_t n_seq, const int32_t* n_frames, const void* const* frames,
             const int64_t* n_points, bool host, int32_t stride, const float* initial_poses, lgs_odometry_frame* records_all, lgs_odometry_dist_info* info) {
  LGS_REQUIRE(ctx && comm, "null argument");
  LGS_REQUIRE(n_seq >= 0 && (n_seq == 0 || (n_frames && n_points)), "null frame counts");
  for (int32_t s = 0; s < n_seq; s++) LGS_REQUIRE(n_frames[s] >= 0, "negative frame count");
  LGS_REQUIRE(comm->device == ctx->device, "the communicator and the context live on different devices");
  const std::vector<int64_t> off = frame_offsets(n_seq, n_frames);
  // the partition of every rank: sequences by total point count (lgs_batch_partition)
  std::vector<int64_t> sizes(static_cast<size_t>(n_seq), 0);
  for (int32_t s = 0; s < n_seq; s++)
    for (int64_t i = off[s]; i < off[s + 1]; i++) sizes[s] += std::max<int64_t>(n_points[i], 0);
  std::vector<int32_t> mine;
  int64_t cap = 1;  // records per rank in the gather: the largest frame total any rank owns
  for (int r = 0; r < comm->world; r++) {
    std::vector<int32_t> ids;
    partition_pairs(sizes.data(), n_seq, r, comm->world, &ids);
    int64_t f = 0;
    for (int32_t s : ids) f += n_frames[s];
    cap = std::max(cap, f);
    if (r == comm->rank) mine = ids;
  }
  std::vector<char> owned(static_cast<size_t>(std::max(n_seq, 1)), 0);
  for (int32_t s : mine) owned[s] = 1;
  Params P;
  LGS_TRY(validate(ctx, params, n_seq, n_frames, frames, n_points, host, stride, owned, nullptr, &P));
  LGS_REQUIRE(records_all || off[n_seq] == 0, "null records");
  LGS_TRY(use_device(ctx));
  // local records are packed rank-locally in the order of `mine`; the gather places them by (sequence, frame)
  std::vector<int64_t> local_off(static_cast<size_t>(n_seq) + 1, 0);
  int64_t n_local = 0;
  for (int32_t s : mine) {
    local_off[s] = n_local;
    n_local += n_frames[s];
  }
  std::vector<lgs_odometry_frame> local(static_cast<size_t>(cap));
  memset(local.data(), 0xFF, local.size() * sizeof(lgs_odometry_frame));  // sequence = -1: unused slot
  const auto t0 = std::chrono::steady_clock::now();
  // a rank whose own run fails still joins the gather (with no records), so that the other ranks return instead of waiting
  const int rc = run_local(ctx, P, n_frames, frames, n_points, host, stride, initial_poses, nullptr, mine, local_off, local.data());
  const std::string err = rc != LGS_OK ? lgs_last_error() : "";
  if (rc != LGS_OK) memset(local.data(), 0xFF, local.size() * sizeof(lgs_odometry_frame));
  const auto t1 = std::chrono::steady_clock::now();
  const size_t bytes = static_cast<size_t>(cap) * sizeof(lgs_odometry_frame);
  LGS_TRY(comm->send.reserve(bytes));
  LGS_CUDA(cudaMemcpyAsync(comm->send.p, local.data(), bytes, cudaMemcpyHostToDevice, ctx->stream));
  int64_t got = 0;
  LGS_TRY(comm_all_gather(comm, ctx->stream, cap, sizeof(lgs_odometry_frame), [&](const void* p) {
    const lgs_odometry_frame* r = static_cast<const lgs_odometry_frame*>(p);
    if (r->sequence < 0) return 0;
    if (r->sequence >= n_seq || r->frame < 0 || r->frame >= n_frames[r->sequence]) {
      set_error("gathered record carries (sequence %d, frame %d) outside the run", r->sequence, r->frame);
      return LGS_ERR_STATE;
    }
    records_all[off[r->sequence] + r->frame] = *r;
    return 1;
  }, &got));
  const auto t2 = std::chrono::steady_clock::now();
  if (info) {
    info->rank = comm->rank;
    info->world = comm->world;
    info->n_local_sequences = static_cast<int64_t>(mine.size());
    info->n_local_frames = n_local;
    info->n_received = got;
    info->gather_bytes = static_cast<int64_t>(bytes) * comm->world;
    info->run_ms = std::chrono::duration<double, std::milli>(t1 - t0).count();
    info->gather_ms = std::chrono::duration<double, std::milli>(t2 - t1).count();
  }
  if (rc != LGS_OK) {
    set_error("%s", err.c_str());
    return rc;
  }
  if (got != off[n_seq]) {
    set_error("the gather returned %lld of %lld records", static_cast<long long>(got), static_cast<long long>(off[n_seq]));
    return LGS_ERR_STATE;
  }
  return LGS_OK;
}

}  // namespace

extern "C" {

int lgs_odometry_run(lgs_ctx* ctx, const lgs_odometry_params* params, int32_t n_seq, const int32_t* n_frames, const void* const* frames,
                     const int64_t* n_points, int32_t stride_bytes, const float* initial_poses, lgs_keyframes* const* keyframes,
                     lgs_odometry_frame* records) {
  LGS_NVTX("lgs_odometry_run");
  return run_all(ctx, params, n_seq, n_frames, frames, n_points, true, stride_bytes, initial_poses, keyframes, records);
}

int lgs_odometry_run_dev(lgs_ctx* ctx, const lgs_odometry_params* params, int32_t n_seq, const int32_t* n_frames, const float* const* frames_dev,
                         const int64_t* n_points, const float* initial_poses, lgs_keyframes* const* keyframes, lgs_odometry_frame* records) {
  LGS_NVTX("lgs_odometry_run_dev");
  return run_all(ctx, params, n_seq, n_frames, reinterpret_cast<const void* const*>(frames_dev), n_points, false, 16, initial_poses, keyframes,
                 records);
}

int lgs_odometry_run_dist(lgs_ctx* ctx, lgs_comm* comm, const lgs_odometry_params* params, int32_t n_seq, const int32_t* n_frames,
                          const void* const* frames, const int64_t* n_points, int32_t stride_bytes, const float* initial_poses,
                          lgs_odometry_frame* records_all, lgs_odometry_dist_info* info) {
  LGS_NVTX("lgs_odometry_run_dist");
  return run_dist(ctx, comm, params, n_seq, n_frames, frames, n_points, true, stride_bytes, initial_poses, records_all, info);
}

int lgs_odometry_run_dist_dev(lgs_ctx* ctx, lgs_comm* comm, const lgs_odometry_params* params, int32_t n_seq, const int32_t* n_frames,
                              const float* const* frames_dev, const int64_t* n_points, const float* initial_poses,
                              lgs_odometry_frame* records_all, lgs_odometry_dist_info* info) {
  LGS_NVTX("lgs_odometry_run_dist_dev");
  return run_dist(ctx, comm, params, n_seq, n_frames, reinterpret_cast<const void* const*>(frames_dev), n_points, false, 16, initial_poses,
                  records_all, info);
}

int lgs_odometry_profile(double* out4) {
  if (out4) {
    out4[0] = g_profile.frames;
    out4[1] = g_profile.prefilter_ms;
    out4[2] = g_profile.align_ms;
    out4[3] = g_profile.keyframe_ms;
  }
  g_profile = Profile();
  return LGS_OK;
}

}  // extern "C"
