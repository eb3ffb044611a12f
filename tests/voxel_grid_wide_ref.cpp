// Reference of the wide VoxelGrid (lgs_voxelgrid_filter_wide, DESIGN section 11) for the tests, built as a ctypes library
// by tests/voxel_grid_wide_ref.py.  It restates oracle/voxel.cpp's prefilter_voxel_grid (the same crop, bounding box,
// per-axis index and sequential f32 sums) with an int64 linear index, std::stable_sort over the 64-bit keys, and the wide
// grid's refusal: an axis of >= 2^31 cells, min_b / max_b outside int32, or more than 2^63 - 1 cells.
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstring>
#include <limits>
#include <utility>
#include <vector>

#include "oracle.hpp"

namespace {

using lgs_oracle::P4;
using lgs_oracle::sum3f;

struct VoxelGridWideResult {
  int status = 0;  // 0 ok, 1 refused (output = cropped input, original order)
  std::vector<P4> out;
  std::vector<int64_t> out_idx;
  std::vector<int32_t> out_count;
  std::vector<int64_t> voxel_idx;
  std::vector<int32_t> member_rank;
  int32_t min_b[3] = {0, 0, 0}, max_b[3] = {0, 0, 0}, div_b[3] = {0, 0, 0};
  size_t n_kept = 0;
};
constexpr int VG_OK = 0, VG_REFUSED_OVERFLOW = 1;

// The wide VoxelGrid: prefilter_voxel_grid with an int64 linear index.  The per-axis index keeps PCL's f32 expression
// floor(x * inv) - float(min_b) (cells beyond 2^24 leaf units merge as there), converted to int64; keys combine in
// 64-bit unsigned arithmetic and order as unsigned.
void prefilter_voxel_grid_wide(const P4* pts, size_t n, const float leaf[3], int min_points_per_voxel, double range_min, const double* box,
                               VoxelGridWideResult* res) {
  res->status = VG_OK;
  res->out.clear();
  res->out_idx.clear();
  res->out_count.clear();
  res->voxel_idx.assign(n, -1);
  res->member_rank.assign(n, -1);

  std::vector<uint32_t> kept;
  kept.reserve(n);
  for (size_t i = 0; i < n; i++) {
    const P4& p = pts[i];
    if (!std::isfinite(p.x) || !std::isfinite(p.y) || !std::isfinite(p.z)) continue;
    if (range_min >= 0.0) {
      const float norm = std::sqrt(sum3f(p.x * p.x, p.y * p.y, p.z * p.z));
      const double distance = norm;
      if (!(range_min < distance)) continue;
    }
    if (box) {
      if (!((box[0] < p.x && p.x < box[1]) && (box[2] < p.y && p.y < box[3]) && (box[4] < p.z && p.z < box[5]))) continue;
    }
    kept.push_back(uint32_t(i));
  }
  res->n_kept = kept.size();
  if (kept.empty()) return;

  float inv[3] = {1.0f / leaf[0], 1.0f / leaf[1], 1.0f / leaf[2]};
  float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
  for (uint32_t i : kept) {
    const float c[3] = {pts[i].x, pts[i].y, pts[i].z};
    for (int a = 0; a < 3; a++) {
      mn[a] = std::min(mn[a], c[a]);
      mx[a] = std::max(mx[a], c[a]);
    }
  }
  bool refuse = false;
  float fmin[3], fmax[3];
  int64_t div[3] = {0, 0, 0};
  for (int a = 0; a < 3; a++) {
    fmin[a] = std::floor(mn[a] * inv[a]);
    fmax[a] = std::floor(mx[a] * inv[a]);
    if (!(fmin[a] >= -2147483648.0f && fmax[a] < 2147483648.0f)) refuse = true;
    if (!((mx[a] - mn[a]) * inv[a] < 2147483648.0f)) refuse = true;
  }
  if (!refuse)
    for (int a = 0; a < 3; a++) {
      div[a] = static_cast<int64_t>(static_cast<int32_t>(fmax[a])) - static_cast<int32_t>(fmin[a]) + 1;
      if (div[a] > std::numeric_limits<int32_t>::max()) refuse = true;
    }
  if (!refuse) {
    const unsigned __int128 cells = static_cast<unsigned __int128>(div[0]) * static_cast<uint64_t>(div[1]) * static_cast<uint64_t>(div[2]);
    refuse = cells > static_cast<unsigned __int128>(std::numeric_limits<int64_t>::max());
  }
  if (refuse) {
    res->status = VG_REFUSED_OVERFLOW;
    for (uint32_t i : kept) res->out.push_back(pts[i]);
    return;
  }
  for (int a = 0; a < 3; a++) {
    res->min_b[a] = static_cast<int32_t>(fmin[a]);
    res->max_b[a] = static_cast<int32_t>(fmax[a]);
    res->div_b[a] = static_cast<int32_t>(div[a]);
  }
  const uint64_t mul[3] = {1, static_cast<uint64_t>(div[0]), static_cast<uint64_t>(div[0]) * static_cast<uint64_t>(div[1])};

  std::vector<std::pair<uint64_t, uint32_t>> iv;  // (idx, point index)
  iv.reserve(kept.size());
  for (uint32_t i : kept) {
    const float c[3] = {pts[i].x, pts[i].y, pts[i].z};
    uint64_t idx = 0;
    for (int a = 0; a < 3; a++) {
      const int64_t ijk = static_cast<int64_t>(std::floor(c[a] * inv[a]) - static_cast<float>(res->min_b[a]));
      idx += static_cast<uint64_t>(ijk) * mul[a];
    }
    res->voxel_idx[i] = static_cast<int64_t>(idx);
    iv.emplace_back(idx, i);
  }
  std::stable_sort(iv.begin(), iv.end(), [](const auto& a, const auto& b) { return a.first < b.first; });

  size_t index = 0;
  while (index < iv.size()) {
    size_t j = index + 1;
    while (j < iv.size() && iv[j].first == iv[index].first) ++j;
    if (j - index >= static_cast<size_t>(std::max(min_points_per_voxel, 0))) {
      float sx = 0, sy = 0, sz = 0, si = 0;
      for (size_t li = index; li < j; ++li) {
        const P4& p = pts[iv[li].second];
        sx += p.x;
        sy += p.y;
        sz += p.z;
        si += p.w;
        res->member_rank[iv[li].second] = static_cast<int32_t>(res->out.size());
      }
      const float cnt = static_cast<float>(j - index);
      res->out.push_back(P4{sx / cnt, sy / cnt, sz / cnt, si / cnt});
      res->out_idx.push_back(static_cast<int64_t>(iv[index].first));
      res->out_count.push_back(static_cast<int32_t>(j - index));
    }
    index = j;
  }
}

}  // namespace

extern "C" {

void* vgw_run(const float* pts, long n, const float* leaf3, int min_pts, double range_min, const double* box6) {
  auto* r = new VoxelGridWideResult;
  prefilter_voxel_grid_wide(reinterpret_cast<const P4*>(pts), static_cast<size_t>(n), leaf3, min_pts, range_min, box6, r);
  return r;
}
int vgw_status(void* h) { return static_cast<VoxelGridWideResult*>(h)->status; }
long vgw_out_n(void* h) { return static_cast<long>(static_cast<VoxelGridWideResult*>(h)->out.size()); }
long vgw_n_kept(void* h) { return static_cast<long>(static_cast<VoxelGridWideResult*>(h)->n_kept); }
void vgw_get(void* h, float* out_pts, long long* out_idx, int* out_count, long long* voxel_idx, int* member_rank, int* grid9) {
  const VoxelGridWideResult& r = *static_cast<VoxelGridWideResult*>(h);
  if (out_pts) std::memcpy(out_pts, r.out.data(), r.out.size() * sizeof(P4));
  if (out_idx) std::memcpy(out_idx, r.out_idx.data(), r.out_idx.size() * sizeof(int64_t));
  if (out_count) std::memcpy(out_count, r.out_count.data(), r.out_count.size() * sizeof(int));
  if (voxel_idx) std::memcpy(voxel_idx, r.voxel_idx.data(), r.voxel_idx.size() * sizeof(int64_t));
  if (member_rank) std::memcpy(member_rank, r.member_rank.data(), r.member_rank.size() * sizeof(int));
  if (grid9)
    for (int a = 0; a < 3; a++) {
      grid9[a] = r.min_b[a];
      grid9[3 + a] = r.max_b[a];
      grid9[6 + a] = r.div_b[a];
    }
}
void vgw_free(void* h) { delete static_cast<VoxelGridWideResult*>(h); }

}  // extern "C"
