// Device-resident key-frame array and sub-map assembly (SURVEY section 8f item 2).
//
// The reference keeps every key frame as a serialised sensor_msgs/PointCloud2 inside key_frame_array_ and, on every
// key-frame change (LSM:187-212) and for every loop candidate (GBS:297-313), deserialises up to 20 / 41 of them
// (pcl::fromROSMsg), transforms each by its pose (pcl::transformPointCloud), concatenates them on the host and hands
// the result to setInputTarget, which copies ~1 M points to wherever the registration lives.  Here a key frame is
// uploaded ONCE, stays in HBM in its own frame, and a sub-map is one kernel: every output point finds its key frame
// (binary search over the segment offsets), applies that key frame's pose with pcl::transformPointCloud's operation
// order and stores one float4; optionally followed by the VoxelGrid of GBS:311-313.  The result is a device cloud for
// the *_set_target_dev / *_set_source_dev entry points, so no point of the map crosses PCIe again.
//
// Storage: chunked arena (a key frame never moves; 180 GB of HBM holds ~10^5 key frames of 10^5 points), poses on the
// host, refreshed by lgs_keyframes_set_pose after a pose-graph update (GBS:343-352 feeds corrected poses back).
// Algorithmic bytes of an assembly: 32 per output point (float4 in, float4 out); HBM-bound.
#include <algorithm>
#include <cmath>
#include <limits>
#include <vector>

#include "keyframes.cuh"
#include "voxel_common.cuh"

namespace lgs {

constexpr int kMaxSegments = 96;  // key frames per launch (LSM: 20, GBS: 41); longer lists are split

struct SubmapSegments {
  const float4* src[kMaxSegments];
  int begin[kMaxSegments + 1];  // first output row of each segment (relative to this launch); begin[count] = total
  int count;
};

// poses: count x 16 floats, column-major, in device memory
__global__ void __launch_bounds__(256) submap_assemble_kernel(SubmapSegments S, const float* __restrict__ poses, float4* __restrict__ out) {
  __shared__ float T[kMaxSegments][16];
  __shared__ int begin[kMaxSegments + 1];
  for (int t = threadIdx.x; t < S.count * 16; t += blockDim.x) T[t >> 4][t & 15] = poses[t];
  for (int t = threadIdx.x; t <= S.count; t += blockDim.x) begin[t] = S.begin[t];
  __syncthreads();
  const int total = begin[S.count];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    int lo = 0, hi = S.count - 1;  // last segment whose begin <= i
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (begin[mid] <= i) lo = mid; else hi = mid - 1;
    }
    const float4 p = __ldg(S.src[lo] + (i - begin[lo]));
    const float3 t = transform_pcl(T[lo], p.x, p.y, p.z);
    out[i] = make_float4(t.x, t.y, t.z, p.w);
  }
}

}  // namespace lgs

using namespace lgs;

struct lgs_keyframes {
  lgs_ctx* ctx = nullptr;
  struct Chunk {
    DevBuf buf;
    size_t used = 0;  // points
    size_t cap = 0;   // points
  };
  struct Frame {
    int chunk = -1;
    size_t offset = 0;  // points into the chunk
    int64_t n = 0;
    float pose[16];
    double accum_distance = 0;  // key_frame.accum_distance (LSM:193): path length at this key frame
    double position[3] = {0, 0, 0};  // key_frame.pose.position in f64 (geometry_msgs), what detect_loop compares (GBS:163-171)
    bool have_position = false;
  };
  std::vector<Chunk*> chunks;
  std::vector<Frame> frames;
  DevBuf assembled, filtered, poses_dev;
  size_t chunk_points = size_t(4) << 20;  // 4 Mi points = 64 MiB per chunk
};

namespace {

int frame_slot(lgs_keyframes* kf, int64_t n, lgs_keyframes::Frame* f) {
  size_t need = static_cast<size_t>(std::max<int64_t>(n, 1));
  if (kf->chunks.empty() || kf->chunks.back()->used + need > kf->chunks.back()->cap) {
    auto* c = new lgs_keyframes::Chunk;
    c->cap = std::max(kf->chunk_points, need);
    if (c->buf.reserve(c->cap * 16) != LGS_OK) {
      delete c;
      return LGS_ERR_CUDA;
    }
    kf->chunks.push_back(c);
  }
  lgs_keyframes::Chunk* c = kf->chunks.back();
  f->chunk = static_cast<int>(kf->chunks.size()) - 1;
  f->offset = c->used;
  f->n = n;
  c->used += need;
  return LGS_OK;
}

const float4* frame_ptr(const lgs_keyframes* kf, const lgs_keyframes::Frame& f) { return kf->chunks[f.chunk]->buf.as<float4>() + f.offset; }

int push(lgs_keyframes* kf, const void* pts, const float* pts_dev, int64_t n, int32_t stride, const float* pose16, int32_t* id) {
  LGS_REQUIRE(kf && pose16, "null argument");
  LGS_REQUIRE(n >= 0, "negative point count");
  LGS_TRY(use_device(kf->ctx));
  lgs_keyframes::Frame f;
  LGS_TRY(frame_slot(kf, n, &f));
  memcpy(f.pose, pose16, sizeof(f.pose));
  float4* dst = const_cast<float4*>(frame_ptr(kf, f));
  if (n) {
    if (pts_dev) {
      LGS_CUDA(cudaMemcpyAsync(dst, pts_dev, static_cast<size_t>(n) * 16, cudaMemcpyDeviceToDevice, kf->ctx->stream));
    } else {
      LGS_REQUIRE(pts != nullptr, "null cloud");
      // upload_cloud repacks into a DevBuf of its own: stage through tmp[0], then place the frame
      if (stride == 16) {
        LGS_CUDA(cudaMemcpyAsync(dst, pts, static_cast<size_t>(n) * 16, cudaMemcpyHostToDevice, kf->ctx->stream));
      } else {
        LGS_TRY(upload_cloud(kf->ctx, pts, n, stride, &kf->ctx->tmp[0]));
        LGS_CUDA(cudaMemcpyAsync(dst, kf->ctx->tmp[0].p, static_cast<size_t>(n) * 16, cudaMemcpyDeviceToDevice, kf->ctx->stream));
      }
    }
  }
  kf->frames.push_back(f);
  if (id) *id = static_cast<int32_t>(kf->frames.size()) - 1;
  return LGS_OK;
}

}  // namespace

namespace lgs {

int keyframes_wait_resident(const lgs_keyframes* kf) {
  LGS_CUDA(cudaSetDevice(kf->ctx->device));
  LGS_CUDA(cudaStreamSynchronize(kf->ctx->stream));
  return LGS_OK;
}
int64_t keyframes_count(const lgs_keyframes* kf) { return static_cast<int64_t>(kf->frames.size()); }
int keyframes_device(const lgs_keyframes* kf) { return kf->ctx->device; }
cudaStream_t keyframes_stream(const lgs_keyframes* kf) { return kf->ctx->stream; }
const float* keyframes_pose(const lgs_keyframes* kf, int64_t id) { return kf->frames[static_cast<size_t>(id)].pose; }
int64_t keyframes_points(const lgs_keyframes* kf, int64_t id) { return kf->frames[static_cast<size_t>(id)].n; }

int keyframes_assemble_into(const lgs_keyframes* kf, lgs_ctx* ctx, const int32_t* ids, int32_t n_ids, DevBuf* poses_dev, DevBuf* out, int64_t* n_out) {
  LGS_REQUIRE(n_ids >= 0, "negative id count");
  int64_t total = 0;
  for (int i = 0; i < n_ids; i++) {
    LGS_REQUIRE(ids[i] >= 0 && ids[i] < static_cast<int32_t>(kf->frames.size()), "key frame id out of range");
    total += kf->frames[ids[i]].n;
  }
  LGS_REQUIRE(total < (int64_t(1) << 31), "sub-map larger than 2^31 points");
  LGS_TRY(out->reserve(static_cast<size_t>(std::max<int64_t>(total, 1)) * 16));
  *n_out = total;
  if (total == 0) return LGS_OK;
  cudaStream_t st = ctx->stream;
  LGS_TRY(poses_dev->reserve(static_cast<size_t>(n_ids) * 64));
  LGS_TRY(ctx->pin_up.reserve(static_cast<size_t>(n_ids) * 64));
  float* hp = ctx->pin_up.as<float>();
  LGS_CUDA(cudaStreamSynchronize(st));  // the pinned staging block may still be in flight from an earlier call on this stream
  for (int i = 0; i < n_ids; i++) memcpy(hp + 16 * i, kf->frames[ids[i]].pose, 64);
  LGS_CUDA(cudaMemcpyAsync(poses_dev->p, hp, static_cast<size_t>(n_ids) * 64, cudaMemcpyHostToDevice, st));
  int64_t row = 0;
  for (int s0 = 0; s0 < n_ids; s0 += kMaxSegments) {
    SubmapSegments S;
    S.count = std::min(kMaxSegments, n_ids - s0);
    int acc = 0;
    for (int s = 0; s < S.count; s++) {
      const auto& f = kf->frames[ids[s0 + s]];
      S.src[s] = kf->chunks[f.chunk]->buf.as<float4>() + f.offset;
      S.begin[s] = acc;
      acc += static_cast<int>(f.n);
    }
    S.begin[S.count] = acc;
    if (acc > 0) {
      const int grid = std::max(1, std::min(grid_for(acc, 256), kNumSMs * 8));
      submap_assemble_kernel<<<grid, 256, 0, st>>>(S, poses_dev->as<float>() + 16 * s0, out->as<float4>() + row);
      ctx->launches++;
      LGS_CUDA(cudaGetLastError());
    }
    row += acc;
  }
  return LGS_OK;
}

}  // namespace lgs

extern "C" {

int lgs_keyframes_create(lgs_ctx* ctx, lgs_keyframes** out) {
  LGS_REQUIRE(ctx && out, "null argument");
  lgs_keyframes* kf = new lgs_keyframes;
  kf->ctx = ctx;
  *out = kf;
  return LGS_OK;
}

void lgs_keyframes_destroy(lgs_keyframes* kf) {
  if (!kf) return;
  cudaSetDevice(kf->ctx->device);
  cudaStreamSynchronize(kf->ctx->stream);
  for (auto* c : kf->chunks) {
    c->buf.release();
    delete c;
  }
  for (DevBuf* b : {&kf->assembled, &kf->filtered, &kf->poses_dev}) b->release();
  delete kf;
}

int lgs_keyframes_push(lgs_keyframes* kf, const void* pts, int64_t n, int32_t stride_bytes, const float* pose16, int32_t* id) {
  return push(kf, pts, nullptr, n, stride_bytes, pose16, id);
}
int lgs_keyframes_push_dev(lgs_keyframes* kf, const float* pts_dev, int64_t n, const float* pose16, int32_t* id) {
  LGS_REQUIRE(pts_dev || n == 0, "null cloud");
  return push(kf, nullptr, pts_dev, n, 16, pose16, id);
}

int lgs_keyframes_set_pose(lgs_keyframes* kf, int32_t id, const float* pose16) {
  LGS_REQUIRE(kf && pose16, "null argument");
  LGS_REQUIRE(id >= 0 && id < static_cast<int32_t>(kf->frames.size()), "key frame id out of range");
  memcpy(kf->frames[id].pose, pose16, sizeof(float) * 16);
  kf->frames[id].have_position = false;  // the f64 position, if any, belonged to the old pose
  return LGS_OK;
}

int lgs_keyframes_size(lgs_keyframes* kf, int64_t* count, int64_t* total_points) {
  LGS_REQUIRE(kf, "null argument");
  if (count) *count = static_cast<int64_t>(kf->frames.size());
  if (total_points) {
    int64_t t = 0;
    for (const auto& f : kf->frames) t += f.n;
    *total_points = t;
  }
  return LGS_OK;
}

int lgs_keyframes_assemble(lgs_keyframes* kf, const int32_t* ids, int32_t n_ids, float leaf, float** out_dev, int64_t* n_out) {
  LGS_NVTX("lgs_keyframes_assemble");
  LGS_REQUIRE(kf && out_dev && n_out && (ids || n_ids == 0), "null argument");
  lgs_ctx* ctx = kf->ctx;
  LGS_TRY(use_device(ctx));
  int64_t total = 0;
  LGS_TRY(keyframes_assemble_into(kf, ctx, ids, n_ids, &kf->poses_dev, &kf->assembled, &total));
  *out_dev = kf->assembled.as<float>();
  *n_out = total;
  if (leaf > 0.0f && total > 0) {  // GBS:311-313: voxel_grid_.setInputCloud(nearest_key_frame_cloud); filter
    LGS_TRY(kf->filtered.reserve(static_cast<size_t>(total) * 16));
    const float leaf3[3] = {leaf, leaf, leaf};
    lgs_voxelgrid_info info;
    LGS_TRY(voxelgrid_device(ctx, kf->assembled.as<float4>(), total, leaf3, 0, -1.0, nullptr, kf->filtered.as<float4>(), nullptr, nullptr, &info));
    *out_dev = kf->filtered.as<float>();
    *n_out = info.n_out;
  }
  return LGS_OK;
}

int lgs_keyframes_set_position(lgs_keyframes* kf, int32_t id, const double* xyz) {
  LGS_REQUIRE(kf && xyz, "null argument");
  LGS_REQUIRE(id >= 0 && id < static_cast<int32_t>(kf->frames.size()), "key frame id out of range");
  for (int a = 0; a < 3; a++) kf->frames[id].position[a] = xyz[a];
  kf->frames[id].have_position = true;
  return LGS_OK;
}

int lgs_keyframes_set_accum_distance(lgs_keyframes* kf, int32_t id, double accum_distance) {
  LGS_REQUIRE(kf, "null argument");
  LGS_REQUIRE(id >= 0 && id < static_cast<int32_t>(kf->frames.size()), "key frame id out of range");
  kf->frames[id].accum_distance = accum_distance;
  return LGS_OK;
}

// detect_loop_with_accum_dist (GBS:157-187): every key frame at least accumulate_distance_threshold of path behind the
// latest one and closer to it than search_for_candidate_threshold; *nearest = the one optimization_callback would
// pick (GBS:263-280: strictly smallest distance, first wins), -1 if none
int lgs_keyframes_detect_loop(lgs_keyframes* kf, int32_t latest_id, double accumulate_distance_threshold, double search_for_candidate_threshold,
                              int32_t* candidates, int32_t capacity, int32_t* n_candidates, int32_t* nearest) {
  LGS_REQUIRE(kf && n_candidates, "null argument");
  LGS_REQUIRE(latest_id >= 0 && latest_id < static_cast<int32_t>(kf->frames.size()), "key frame id out of range");
  const auto& L = kf->frames[latest_id];
  auto pos = [](const lgs_keyframes::Frame& f, int a) { return f.have_position ? f.position[a] : static_cast<double>(f.pose[12 + a]); };
  const double lp[3] = {pos(L, 0), pos(L, 1), pos(L, 2)};
  int32_t cnt = 0, best = -1;
  double min_dist = std::numeric_limits<double>::max();
  for (int32_t id = 0; id < static_cast<int32_t>(kf->frames.size()); id++) {
    const auto& f = kf->frames[id];
    if ((L.accum_distance - f.accum_distance) < accumulate_distance_threshold) continue;
    const double dx = lp[0] - pos(f, 0), dy = lp[1] - pos(f, 1), dz = lp[2] - pos(f, 2);
    const double dist = std::sqrt(dx * dx + dy * dy + dz * dz);
    if (dist < search_for_candidate_threshold) {
      if (candidates && cnt < capacity) candidates[cnt] = id;
      cnt++;
      if (dist < min_dist) {
        min_dist = dist;
        best = id;
      }
    }
  }
  *n_candidates = cnt;
  if (nearest) *nearest = best;
  return LGS_OK;
}

}  // extern "C"
