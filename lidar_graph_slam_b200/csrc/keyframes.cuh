// Internal view of the device-resident key-frame array (keyframes.cu) for the loop-closure batch (batch.cu).
#pragma once
#include "common.cuh"

struct lgs_keyframes;

namespace lgs {

// Sub-map of the key frames ids[0..n_ids) (transformed by their poses, concatenated in that order) written to `out`
// on ctx's stream; `poses_dev` is scratch for the poses.  ctx may be any context on the key-frame array's device:
// the arena is only read.  *n_out = number of points.
int keyframes_assemble_into(const lgs_keyframes* kf, lgs_ctx* ctx, const int32_t* ids, int32_t n_ids, DevBuf* poses_dev, DevBuf* out, int64_t* n_out);
// everything pushed so far is resident (the pushes are asynchronous on the array's own stream)
int keyframes_wait_resident(const lgs_keyframes* kf);
int64_t keyframes_count(const lgs_keyframes* kf);
int64_t keyframes_points(const lgs_keyframes* kf, int64_t id);  // points of key frame id
int keyframes_device(const lgs_keyframes* kf);
cudaStream_t keyframes_stream(const lgs_keyframes* kf);  // the stream pushes copy on (that of the array's context)
const float* keyframes_pose(const lgs_keyframes* kf, int64_t id);  // column-major 4x4 of key frame id

}  // namespace lgs
