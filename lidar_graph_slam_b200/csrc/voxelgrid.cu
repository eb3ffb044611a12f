// Prefilter: range/box crop + pcl::VoxelGrid downsampling on the GPU.
//
// Replaces PPF:102-112 (distance_filter), PPF:89-100 (crop) and pcl::VoxelGrid::filter as called at
// PPF:114-121 and GBS:311-313,490-493 (index arithmetic restated in-tree at VGC:67-103,218-223).
//
// Pipeline (all on ctx->stream):
//   K1 crop_bbox      16 B/pt read : crop predicate, bbox of the kept points (block reduce + 6 atomics)
//   -- 32-byte D2H of the bbox; the host derives min_b/div_b/divb_mul with the reference's f32 arithmetic
//   K2 voxel_key      16 B/pt read, 12 B/pt write: key = ijk . divb_mul (explicit IEEE f32 ops), value = point index
//   K3 radix sort     (key,value) pairs, only the bits the grid needs (stable => members stay in index order);
//                     own onesweep kernels, sort.cuh
//   K4 segment heads  single-pass look-back scan (sort.cuh) => start offset of every occupied voxel
//   K5 centroid       one thread per voxel: sequential f32 sums in ascending point index (the oracle's order),
//                     scatter of the per-point membership rank
// The wide grid (lgs_voxelgrid_filter_wide*, lgs_keyframes_export_map) runs the same stages.  Beyond INT32_MAX cells K2
// writes a 64-bit key, K3 orders it with two stable 32-bit sorts (radix_sort_indices64) and K4 compares whole keys.
// Integer outputs (voxel idx, occupancy, membership, order) are bit-exact by construction: no FMA
// contraction or reassociation can reach the key arithmetic because it is written with __f*_rn intrinsics.
#include <cfloat>
#include <cmath>
#include <limits>

#include "sort.cuh"
#include "voxel_common.cuh"

namespace lgs {

struct BBoxAcc {  // device-side accumulator
  unsigned mn[3];
  unsigned mx[3];
  unsigned long long kept;
  unsigned done;  // CTAs that have merged their part
  unsigned pad;
};
static_assert(sizeof(BBoxAcc) <= 48, "the segment count lives 48 bytes into the same scratch block");

__global__ void bbox_init_kernel(BBoxAcc* acc) {
  if (threadIdx.x == 0) {
    for (int a = 0; a < 3; a++) {
      acc->mn[a] = 0xFFFFFFFFu;
      acc->mx[a] = 0u;
    }
    acc->kept = 0ull;
    acc->done = 0u;
  }
}

__device__ __forceinline__ bool finite3(const float4& p) {
  return (__float_as_uint(p.x) & 0x7f800000u) != 0x7f800000u && (__float_as_uint(p.y) & 0x7f800000u) != 0x7f800000u &&
         (__float_as_uint(p.z) & 0x7f800000u) != 0x7f800000u;
}

// pcl::VoxelGrid / getMinMax3D / VGC:210-215 skip points with a non-finite coordinate (clouds that are not is_dense);
// here every cloud is treated that way: a NaN or Inf point never reaches the bounding box or a voxel.
__device__ __forceinline__ bool crop_keep(const float4& p, const CropParams& cp) {
  bool keep = finite3(p);
  if (cp.range_min >= 0.0) {
    // Eigen Vector3f::norm(): sqrt(x*x + (y*y + z*z)) in f32 (unrolled 3-element redux), compared in f64
    float n2 = __fadd_rn(__fmul_rn(p.x, p.x), __fadd_rn(__fmul_rn(p.y, p.y), __fmul_rn(p.z, p.z)));
    float nrm = __fsqrt_rn(n2);
    keep = keep && cp.range_min < static_cast<double>(nrm);
  }
  if (cp.use_box) {
    keep = keep && (cp.box[0] < p.x && p.x < cp.box[1]) && (cp.box[2] < p.y && p.y < cp.box[3]) && (cp.box[4] < p.z && p.z < cp.box[5]);
  }
  return keep;
}

// grid-stride, float4 loads; per-thread min/max -> warp shuffle -> one atomic set per block
__global__ void __launch_bounds__(256) crop_bbox_kernel(const float4* __restrict__ pts, int64_t n, CropParams cp, unsigned char* __restrict__ keep,
                                                       BBoxAcc* __restrict__ acc, const Mailbox mb) {
  float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
  unsigned cnt = 0;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    float4 p = pts[i];
    bool k = crop_keep(p, cp);
    if (keep) keep[i] = k ? 1 : 0;
    if (k) {
      cnt++;
      mn[0] = fminf(mn[0], p.x); mx[0] = fmaxf(mx[0], p.x);
      mn[1] = fminf(mn[1], p.y); mx[1] = fmaxf(mx[1], p.y);
      mn[2] = fminf(mn[2], p.z); mx[2] = fmaxf(mx[2], p.z);
    }
  }
  for (int off = 16; off > 0; off >>= 1) {
    for (int a = 0; a < 3; a++) {
      mn[a] = fminf(mn[a], __shfl_xor_sync(0xffffffffu, mn[a], off));
      mx[a] = fmaxf(mx[a], __shfl_xor_sync(0xffffffffu, mx[a], off));
    }
    cnt += __shfl_xor_sync(0xffffffffu, cnt, off);
  }
  __shared__ float smn[8][3], smx[8][3];
  __shared__ unsigned scnt[8];
  int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) {
    for (int a = 0; a < 3; a++) {
      smn[w][a] = mn[a];
      smx[w][a] = mx[a];
    }
    scnt[w] = cnt;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned total = 0;
    for (int ww = 0; ww < (blockDim.x >> 5); ww++) {
      total += scnt[ww];
      for (int a = 0; a < 3; a++) {
        mn[a] = fminf(mn[a], smn[ww][a]);
        mx[a] = fmaxf(mx[a], smx[ww][a]);
      }
    }
    if (total) {
      for (int a = 0; a < 3; a++) {
        atomicMin(&acc->mn[a], enc_f(mn[a]));
        atomicMax(&acc->mx[a], enc_f(mx[a]));
      }
      atomicAdd(&acc->kept, static_cast<unsigned long long>(total));
    }
    // the last CTA to arrive sends the finished box and count to the host mailbox (no D2H copy + stream synchronise)
    __threadfence();
    if (atomicAdd(&acc->done, 1u) == gridDim.x - 1) {
      __threadfence();
      volatile BBoxAcc* va = acc;
      for (int a = 0; a < 3; a++) {
        mailbox_publish_one(mb, a, static_cast<double>(va->mn[a]));
        mailbox_publish_one(mb, 3 + a, static_cast<double>(va->mx[a]));
      }
      mailbox_publish_one(mb, 6, static_cast<double>(va->kept));
    }
  }
}

// VGC:218-223 / pcl::VoxelGrid: ijk = int(floor(x * inv) - float(min_b)); idx = ijk . divb_mul
__device__ __forceinline__ int voxel_index(const float4& p, const GridParams& g) {
  int ijk0 = static_cast<int>(__fsub_rn(floorf(__fmul_rn(p.x, g.inv[0])), static_cast<float>(g.min_b[0])));
  int ijk1 = static_cast<int>(__fsub_rn(floorf(__fmul_rn(p.y, g.inv[1])), static_cast<float>(g.min_b[1])));
  int ijk2 = static_cast<int>(__fsub_rn(floorf(__fmul_rn(p.z, g.inv[2])), static_cast<float>(g.min_b[2])));
  return ijk0 * g.mul[0] + ijk1 * g.mul[1] + ijk2 * g.mul[2];
}

// IdxT: int for the narrow grid's index output, int64_t when the wide grid runs the narrow code (the index widened)
template <typename IdxT>
__global__ void __launch_bounds__(256) voxel_key_kernel(const float4* __restrict__ pts, const unsigned char* __restrict__ keep, int64_t n, GridParams g,
                                                       unsigned* __restrict__ keys, unsigned* __restrict__ vals, IdxT* __restrict__ voxel_idx,
                                                       int* __restrict__ member_rank) {
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= n) return;
  unsigned key = g.sentinel;
  int vi = -1;
  if (!keep || keep[i]) {
    vi = voxel_index(pts[i], g);
    key = static_cast<unsigned>(vi);
  }
  keys[i] = key;
  vals[i] = static_cast<unsigned>(i);
  if (voxel_idx) voxel_idx[i] = vi;
  if (member_rank) member_rank[i] = -1;
}

// The per-axis index exactly as voxel_index (so cells beyond 2^24 leaf units merge as they do there), converted to
// int64 and combined in 64-bit unsigned arithmetic
__device__ __forceinline__ unsigned long long voxel_index_wide(const float4& p, const GridParamsWide& g) {
  const long long ijk0 = static_cast<long long>(__fsub_rn(floorf(__fmul_rn(p.x, g.inv[0])), static_cast<float>(g.min_b[0])));
  const long long ijk1 = static_cast<long long>(__fsub_rn(floorf(__fmul_rn(p.y, g.inv[1])), static_cast<float>(g.min_b[1])));
  const long long ijk2 = static_cast<long long>(__fsub_rn(floorf(__fmul_rn(p.z, g.inv[2])), static_cast<float>(g.min_b[2])));
  return static_cast<unsigned long long>(ijk0) * g.mul[0] + static_cast<unsigned long long>(ijk1) * g.mul[1] +
         static_cast<unsigned long long>(ijk2) * g.mul[2];
}

// 64-bit keys: the whole key per point (read back by the high-word gather and the segment heads) and its low word as
// the first sort pass's key
__global__ void __launch_bounds__(256) voxel_key_wide_kernel(const float4* __restrict__ pts, const unsigned char* __restrict__ keep, int64_t n,
                                                            GridParamsWide g, unsigned* __restrict__ keys_lo, unsigned* __restrict__ vals,
                                                            unsigned long long* __restrict__ keys64, int64_t* __restrict__ voxel_idx,
                                                            int* __restrict__ member_rank) {
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= n) return;
  unsigned long long key = g.sentinel;
  int64_t vi = -1;
  if (!keep || keep[i]) {
    key = voxel_index_wide(pts[i], g);
    vi = static_cast<int64_t>(key);
  }
  keys_lo[i] = static_cast<unsigned>(key);
  vals[i] = static_cast<unsigned>(i);
  keys64[i] = key;
  if (voxel_idx) voxel_idx[i] = vi;
  if (member_rank) member_rank[i] = -1;
}

// scan_select functors (sort.cuh)
struct SegmentHeads {  // start offset of every run of equal keys
  const unsigned* keys;
  int* seg_start;
  __device__ bool flag(int64_t i) const { return i == 0 || keys[i] != keys[i - 1]; }
  __device__ void emit(int64_t i, int64_t pos, bool f) const {
    if (f) seg_start[pos] = static_cast<int>(i);
  }
};
struct SegmentHeadsWide {  // the same over 64-bit keys, read through the sorted point indices
  const unsigned* vals;
  const unsigned long long* keys64;
  int* seg_start;
  __device__ bool flag(int64_t i) const { return i == 0 || keys64[vals[i]] != keys64[vals[i - 1]]; }
  __device__ void emit(int64_t i, int64_t pos, bool f) const {
    if (f) seg_start[pos] = static_cast<int>(i);
  }
};
struct QualifiedVoxels {  // qual[v] = voxel holds >= min_pts points; out_rank[v] = its position among the qualified ones
  const int* seg_start;
  int n_seg;
  int n_kept;
  int min_pts;
  int* qual;
  int* out_rank;
  __device__ bool flag(int64_t v) const {
    const int b = seg_start[v];
    const int e = (v + 1 < n_seg) ? seg_start[v + 1] : n_kept;
    return e - b >= min_pts;
  }
  __device__ void emit(int64_t v, int64_t pos, bool f) const {
    qual[v] = f ? 1 : 0;
    out_rank[v] = static_cast<int>(pos);
  }
};
struct KeptPoints {  // compaction of the points that survive the crop, original order
  const float4* pts;
  const unsigned char* keep;
  float4* out;
  __device__ bool flag(int64_t i) const { return keep[i] != 0; }
  __device__ void emit(int64_t i, int64_t pos, bool f) const {
    if (f) out[pos] = pts[i];
  }
};

// One thread per occupied voxel.  CentroidPoint<PointXYZI> (PCL): f32 accumulators for xyz and
// intensity, divided by the point count; members are visited in ascending point index.
__global__ void __launch_bounds__(128) centroid_kernel(const float4* __restrict__ pts, const unsigned* __restrict__ vals, const int* __restrict__ seg_start,
                                                      const int* __restrict__ out_rank, const int* __restrict__ qual, int n_seg, int64_t n_kept,
                                                      float4* __restrict__ out_pts, int* __restrict__ member_rank) {
  int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n_seg) return;
  if (qual && !qual[v]) return;
  int b = seg_start[v];
  int e = (v + 1 < n_seg) ? seg_start[v + 1] : static_cast<int>(n_kept);
  int r = out_rank ? out_rank[v] : v;
  float sx = 0.f, sy = 0.f, sz = 0.f, si = 0.f;
  for (int j = b; j < e; j++) {
    unsigned pi = vals[j];
    float4 p = pts[pi];
    sx = __fadd_rn(sx, p.x);
    sy = __fadd_rn(sy, p.y);
    sz = __fadd_rn(sz, p.z);
    si = __fadd_rn(si, p.w);
    if (member_rank) member_rank[pi] = r;
  }
  float c = static_cast<float>(e - b);
  if (out_pts) out_pts[r] = make_float4(__fdiv_rn(sx, c), __fdiv_rn(sy, c), __fdiv_rn(sz, c), __fdiv_rn(si, c));
}

static int bits_for(uint64_t max_value, int cap = 32) {
  int b = 1;
  while (b < cap && (max_value >> b) != 0) b++;
  return b;
}

// start offset of every occupied voxel; n_kept > 0
template <class Heads>
static int segment_heads(lgs_ctx* ctx, Heads heads, int64_t n_kept, BBoxAcc* acc, SortedVoxels* out) {
  int* d_nseg = reinterpret_cast<int*>(reinterpret_cast<char*>(acc) + 48);
  Mailbox mb2;
  LGS_TRY(mailbox_next(ctx, &mb2));
  LGS_TRY(scan_select(ctx, heads, n_kept, d_nseg, &mb2));
  double nseg = 0;
  LGS_TRY(mailbox_wait(ctx, mb2, 1, &nseg));
  out->n_seg = static_cast<int>(nseg);
  return LGS_OK;
}

// The wide grid beyond INT32_MAX cells.  Refuses (returns with out->status set) when an axis spans >= 2^31 cells, when
// min_b or max_b does not fit int32, or when the cell product exceeds 2^63 - 1.
static int build_sorted_voxels_wide(lgs_ctx* ctx, const float4* pts, int64_t n, const unsigned char* keep, BBoxAcc* acc, const float mn[3],
                                    const float mx[3], const float inv[3], int64_t* voxel_idx_dev, int* member_rank_dev, SortedVoxels* out) {
  cudaStream_t st = ctx->stream;
  float fmin[3], fmax[3];
  bool refuse = false;
  for (int a = 0; a < 3; a++) {
    fmin[a] = std::floor(mn[a] * inv[a]);
    fmax[a] = std::floor(mx[a] * inv[a]);
    if (!(fmin[a] >= -2147483648.0f && fmax[a] < 2147483648.0f)) refuse = true;  // also NaN / inf: no float-to-int cast of it
    if (!((mx[a] - mn[a]) * inv[a] < 2147483648.0f)) refuse = true;              // PCL's per-axis extent
  }
  int64_t div[3] = {0, 0, 0};
  if (!refuse) {
    for (int a = 0; a < 3; a++) {
      div[a] = static_cast<int64_t>(static_cast<int>(fmax[a])) - static_cast<int>(fmin[a]) + 1;
      if (div[a] > std::numeric_limits<int32_t>::max()) refuse = true;
    }
  }
  if (!refuse) {
    const unsigned __int128 cells = static_cast<unsigned __int128>(div[0]) * static_cast<uint64_t>(div[1]) * static_cast<uint64_t>(div[2]);
    refuse = cells > static_cast<unsigned __int128>(std::numeric_limits<int64_t>::max());
  }
  if (refuse) {
    out->status = LGS_VG_REFUSED_OVERFLOW;
    if (voxel_idx_dev) LGS_CUDA(cudaMemsetAsync(voxel_idx_dev, 0xFF, n * sizeof(int64_t), st));
    if (member_rank_dev) LGS_CUDA(cudaMemsetAsync(member_rank_dev, 0xFF, n * sizeof(int), st));
    return LGS_OK;
  }
  GridParamsWide g;
  for (int a = 0; a < 3; a++) {
    out->min_b[a] = static_cast<int>(fmin[a]);
    out->max_b[a] = static_cast<int>(fmax[a]);
    out->div_b[a] = static_cast<int>(div[a]);
    g.inv[a] = inv[a];
    g.min_b[a] = out->min_b[a];
  }
  g.mul[0] = 1;
  g.mul[1] = static_cast<uint64_t>(div[0]);
  g.mul[2] = static_cast<uint64_t>(div[0]) * static_cast<uint64_t>(div[1]);
  const uint64_t total_cells = g.mul[2] * static_cast<uint64_t>(div[2]);
  out->total_cells = total_cells;
  // An axis index can exceed div_b - 1 where floor(x * inv) - float(min_b) rounds up (more than 2^24 cells on the axis);
  // the sentinel stays above the largest key the kernel can form, and the sort covers it.
  uint64_t max_key = 0;
  for (int a = 0; a < 3; a++) max_key += static_cast<uint64_t>(static_cast<int64_t>(fmax[a] - static_cast<float>(out->min_b[a]))) * g.mul[a];
  g.sentinel = std::max<uint64_t>(total_cells, max_key + 1);
  const int end_bit = bits_for(g.sentinel, 64);

  LGS_TRY(ctx->tmp[1].reserve(n * 4));
  LGS_TRY(ctx->tmp[2].reserve(n * 4));
  LGS_TRY(ctx->tmp[3].reserve(n * 4));
  LGS_TRY(ctx->tmp[4].reserve(n * 4));
  LGS_TRY(ctx->tmp[7].reserve(n * 8));
  unsigned *keys_lo = ctx->tmp[1].as<unsigned>(), *vals0 = ctx->tmp[2].as<unsigned>();
  unsigned long long* keys64 = ctx->tmp[7].as<unsigned long long>();
  voxel_key_wide_kernel<<<grid_for(n, 256), 256, 0, st>>>(pts, keep, n, g, keys_lo, vals0, keys64, voxel_idx_dev, member_rank_dev);
  ctx->launches++;
  unsigned* svals;
  LGS_TRY(radix_sort_indices64(ctx, keys64, keys_lo, vals0, ctx->tmp[3].as<unsigned>(), ctx->tmp[4].as<unsigned>(), n, end_bit, &svals));
  out->vals = svals;

  LGS_TRY(ctx->tmp[5].reserve(static_cast<size_t>(out->n_kept) * 4 + 64));
  int* seg_start = ctx->tmp[5].as<int>();
  LGS_TRY(segment_heads(ctx, SegmentHeadsWide{svals, keys64, seg_start}, out->n_kept, acc, out));
  out->seg_start = seg_start;
  return LGS_OK;
}

// Shared front half: crop, bbox, keys, sort, segment heads.
int build_sorted_voxels(lgs_ctx* ctx, const float4* pts, int64_t n, const float leaf[3], double range_min, const double* box6,
                        int* voxel_idx_dev, int* member_rank_dev, SortedVoxels* out, bool wide, int64_t* voxel_idx64_dev) {
  *out = SortedVoxels();
  LGS_REQUIRE(wide ? voxel_idx_dev == nullptr : voxel_idx64_dev == nullptr, "index output of the other width");
  LGS_REQUIRE(n >= 0 && n < (int64_t(1) << 31), "point count out of range");
  LGS_REQUIRE(leaf[0] > 0 && leaf[1] > 0 && leaf[2] > 0, "leaf size must be positive");
  if (n == 0) return LGS_OK;
  cudaStream_t st = ctx->stream;
  const bool cropping = true;  // the keep mask is always materialised: it also carries the finiteness test

  // arenas: tmp0 keep flags | tmp1 keys | tmp2 vals | tmp3 keys_alt | tmp4 vals_alt | tmp5 head flags, seg_start | tmp6 small
  if (cropping) LGS_TRY(ctx->tmp[0].reserve(n));
  LGS_TRY(ctx->tmp[6].reserve(sizeof(BBoxAcc) + 64));
  LGS_TRY(ctx->pin.reserve(256));
  unsigned char* keep = cropping ? ctx->tmp[0].as<unsigned char>() : nullptr;
  out->keep = keep;
  BBoxAcc* acc = ctx->tmp[6].as<BBoxAcc>();

  CropParams cp;
  cp.range_min = range_min;
  cp.use_box = box6 ? 1 : 0;
  for (int a = 0; a < 6; a++) cp.box[a] = box6 ? box6[a] : 0.0;

  bbox_init_kernel<<<1, 32, 0, st>>>(acc);
  int blocks = std::min(grid_for(n, 256), kNumSMs * 8);
  Mailbox mb;
  LGS_TRY(mailbox_next(ctx, &mb));
  crop_bbox_kernel<<<blocks, 256, 0, st>>>(pts, n, cp, keep, acc, mb);
  ctx->launches += 2;
  LGS_CUDA(cudaGetLastError());
  double hbox[kMailboxRecords];
  LGS_TRY(mailbox_wait(ctx, mb, 7, hbox));
  BBoxAcc hacc_v;
  BBoxAcc* hacc = &hacc_v;
  for (int a = 0; a < 3; a++) {
    hacc->mn[a] = static_cast<unsigned>(hbox[a]);
    hacc->mx[a] = static_cast<unsigned>(hbox[3 + a]);
  }
  hacc->kept = static_cast<unsigned long long>(hbox[6]);

  const int64_t n_kept = static_cast<int64_t>(hacc->kept);
  out->n_kept = n_kept;
  if (n_kept == 0) {
    if (voxel_idx_dev) LGS_CUDA(cudaMemsetAsync(voxel_idx_dev, 0xFF, n * sizeof(int), st));
    if (voxel_idx64_dev) LGS_CUDA(cudaMemsetAsync(voxel_idx64_dev, 0xFF, n * sizeof(int64_t), st));
    if (member_rank_dev) LGS_CUDA(cudaMemsetAsync(member_rank_dev, 0xFF, n * sizeof(int), st));
    return LGS_OK;
  }
  float mn[3], mx[3], inv[3];
  for (int a = 0; a < 3; a++) {
    mn[a] = dec_f_host(hacc->mn[a]);
    mx[a] = dec_f_host(hacc->mx[a]);
    inv[a] = 1.0f / leaf[a];  // VoxelGrid::setLeafSize: inverse_leaf_size_ = 1 / leaf_size_ (f32)
  }
  // overflow refusal (PCL voxel_grid.hpp; same test at VGC:75-84)
  int64_t d[3];
  bool too_large = false;
  for (int a = 0; a < 3; a++) {
    const float ext = (mx[a] - mn[a]) * inv[a];
    if (!(ext < 2147483648.0f)) too_large = true;  // also catches an extent that overflowed to inf: no float-to-int cast of it
    d[a] = too_large ? 0 : static_cast<int64_t>(ext) + 1;
  }
  if (wide) {
    // the narrow grid's decision with an exact product, and with min_b / max_b checked before they are cast
    bool narrow = !too_large;
    for (int a = 0; a < 3; a++) {
      const float lo = std::floor(mn[a] * inv[a]), hi = std::floor(mx[a] * inv[a]);
      narrow = narrow && lo >= -2147483648.0f && hi < 2147483648.0f;
    }
    narrow = narrow && static_cast<unsigned __int128>(d[0]) * static_cast<uint64_t>(d[1]) * static_cast<uint64_t>(d[2]) <=
                           static_cast<unsigned __int128>(std::numeric_limits<int32_t>::max());
    if (!narrow) return build_sorted_voxels_wide(ctx, pts, n, keep, acc, mn, mx, inv, voxel_idx64_dev, member_rank_dev, out);
  }
  if (too_large || d[0] * d[1] * d[2] > static_cast<int64_t>(std::numeric_limits<int32_t>::max())) {
    out->status = LGS_VG_REFUSED_OVERFLOW;
    if (voxel_idx_dev) LGS_CUDA(cudaMemsetAsync(voxel_idx_dev, 0xFF, n * sizeof(int), st));
    if (member_rank_dev) LGS_CUDA(cudaMemsetAsync(member_rank_dev, 0xFF, n * sizeof(int), st));
    return LGS_OK;
  }
  GridParams g;
  for (int a = 0; a < 3; a++) {
    out->min_b[a] = static_cast<int>(std::floor(mn[a] * inv[a]));
    out->max_b[a] = static_cast<int>(std::floor(mx[a] * inv[a]));
    out->div_b[a] = out->max_b[a] - out->min_b[a] + 1;
    g.inv[a] = inv[a];
    g.min_b[a] = out->min_b[a];
  }
  g.mul[0] = 1;
  g.mul[1] = out->div_b[0];
  g.mul[2] = out->div_b[0] * out->div_b[1];
  const uint64_t total_cells = static_cast<uint64_t>(out->div_b[0]) * out->div_b[1] * out->div_b[2];
  out->total_cells = total_cells;
  g.sentinel = static_cast<unsigned>(total_cells);  // <= 2^31 - 1, larger than any real index
  const int end_bit = bits_for(total_cells);

  LGS_TRY(ctx->tmp[1].reserve(n * 4));
  LGS_TRY(ctx->tmp[2].reserve(n * 4));
  LGS_TRY(ctx->tmp[3].reserve(n * 4));
  LGS_TRY(ctx->tmp[4].reserve(n * 4));
  unsigned *keys0 = ctx->tmp[1].as<unsigned>(), *vals0 = ctx->tmp[2].as<unsigned>();
  if (voxel_idx64_dev)
    voxel_key_kernel<int64_t><<<grid_for(n, 256), 256, 0, st>>>(pts, keep, n, g, keys0, vals0, voxel_idx64_dev, member_rank_dev);
  else
    voxel_key_kernel<int><<<grid_for(n, 256), 256, 0, st>>>(pts, keep, n, g, keys0, vals0, voxel_idx_dev, member_rank_dev);
  ctx->launches++;
  unsigned *skeys, *svals;
  LGS_TRY(radix_sort_pairs(ctx, keys0, vals0, ctx->tmp[3].as<unsigned>(), ctx->tmp[4].as<unsigned>(), n, end_bit, &skeys, &svals));
  out->keys = skeys;
  out->vals = svals;

  // segment heads -> start offsets
  LGS_TRY(ctx->tmp[5].reserve(static_cast<size_t>(n_kept) * 4 + 64));
  int* seg_start = ctx->tmp[5].as<int>();
  LGS_TRY(segment_heads(ctx, SegmentHeads{out->keys, seg_start}, n_kept, acc, out));  // n_kept > 0 here
  out->seg_start = seg_start;
  return LGS_OK;
}

// Prefilter core: everything device-side.  Outputs may be null.  out_pts in ascending voxel-index order.
int voxelgrid_device(lgs_ctx* ctx, const float4* pts, int64_t n, const float leaf[3], int min_pts, double range_min, const double* box6,
                     float4* out_pts_dev, int* voxel_idx_dev, int* member_rank_dev, lgs_voxelgrid_info* info, bool wide,
                     int64_t* voxel_idx64_dev) {
  memset(info, 0, sizeof(*info));
  SortedVoxels sv;
  LGS_TRY(build_sorted_voxels(ctx, pts, n, leaf, range_min, box6, voxel_idx_dev, member_rank_dev, &sv, wide, voxel_idx64_dev));
  cudaStream_t st = ctx->stream;
  info->status = sv.status;
  info->n_kept = sv.n_kept;
  for (int a = 0; a < 3; a++) {
    info->min_b[a] = sv.min_b[a];
    info->max_b[a] = sv.max_b[a];
    info->div_b[a] = sv.div_b[a];
  }
  if (sv.n_kept == 0) return LGS_OK;
  if (sv.status == LGS_VG_REFUSED_OVERFLOW) {
    info->n_out = sv.n_kept;
    if (out_pts_dev) {  // pcl::VoxelGrid: output = input (here: the cropped input, original order)
      if (!sv.keep) {
        LGS_CUDA(cudaMemcpyAsync(out_pts_dev, pts, static_cast<size_t>(n) * 16, cudaMemcpyDeviceToDevice, st));
      } else {
        LGS_TRY(ctx->tmp[5].reserve(64));
        LGS_TRY(scan_select(ctx, KeptPoints{pts, sv.keep, out_pts_dev}, n, ctx->tmp[5].as<int>()));
      }
      LGS_CUDA(cudaGetLastError());
    }
    return LGS_OK;
  }
  const int n_seg = sv.n_seg;
  const int64_t n_kept = sv.n_kept;
  int* h_small = ctx->pin.as<int>() + 32;
  int* qual = nullptr;
  int* out_rank = nullptr;
  int64_t n_out = n_seg;
  if (min_pts > 1) {
    LGS_TRY(ctx->tmp[7].reserve(static_cast<size_t>(n_seg) * 8 + 64));
    qual = ctx->tmp[7].as<int>();
    out_rank = qual + n_seg;
    LGS_TRY(scan_select(ctx, QualifiedVoxels{sv.seg_start, n_seg, static_cast<int>(n_kept), min_pts, qual, out_rank}, n_seg, nullptr));
    LGS_CUDA(cudaMemcpyAsync(h_small, qual + n_seg - 1, sizeof(int), cudaMemcpyDeviceToHost, st));
    LGS_CUDA(cudaMemcpyAsync(h_small + 1, out_rank + n_seg - 1, sizeof(int), cudaMemcpyDeviceToHost, st));
    LGS_CUDA(cudaStreamSynchronize(st));
    n_out = h_small[0] + h_small[1];
  }
  info->n_out = n_out;
  centroid_kernel<<<grid_for(n_seg, 128), 128, 0, st>>>(pts, sv.vals, sv.seg_start, out_rank, qual, n_seg, n_kept, out_pts_dev, member_rank_dev);
  ctx->launches++;
  LGS_CUDA(cudaGetLastError());
  return LGS_OK;
}

}  // namespace lgs

extern "C" {

int lgs_voxelgrid_filter_dev(lgs_ctx* ctx, const float* pts_dev, int64_t n, const float leaf[3], int32_t min_points_per_voxel, double range_min,
                             const double* box6, float* out_pts_dev, int32_t* out_voxel_idx_dev, int32_t* out_member_rank_dev,
                             lgs_voxelgrid_info* info) {
  LGS_NVTX("lgs_voxelgrid_filter_dev");
  LGS_REQUIRE(ctx && info && leaf, "null argument");
  LGS_TRY(lgs::use_device(ctx));
  return lgs::voxelgrid_device(ctx, reinterpret_cast<const float4*>(pts_dev), n, leaf, min_points_per_voxel, range_min, box6,
                               reinterpret_cast<float4*>(out_pts_dev), out_voxel_idx_dev, out_member_rank_dev, info);
}

int lgs_voxelgrid_filter(lgs_ctx* ctx, const void* pts, int64_t n, int32_t stride_bytes, const float leaf[3], int32_t min_points_per_voxel,
                         double range_min, const double* box6, float* out_pts, int32_t* out_voxel_idx, int32_t* out_member_rank,
                         lgs_voxelgrid_info* info) {
  LGS_NVTX("lgs_voxelgrid_filter");
  LGS_REQUIRE(ctx && info && leaf, "null argument");
  LGS_TRY(lgs::use_device(ctx));
  struct Arena {
    lgs::DevBuf &in, &out, &vidx, &rank;
  } arena{ctx->vg_in, ctx->vg_out, ctx->vg_vidx, ctx->vg_rank};
  Arena* A = &arena;
  LGS_TRY(lgs::upload_cloud(ctx, pts, n, stride_bytes, &A->in));
  const size_t nn = static_cast<size_t>(n > 0 ? n : 1);
  LGS_TRY(A->out.reserve(nn * 16));
  if (out_voxel_idx) LGS_TRY(A->vidx.reserve(nn * 4));
  if (out_member_rank) LGS_TRY(A->rank.reserve(nn * 4));
  LGS_TRY(lgs::voxelgrid_device(ctx, A->in.as<float4>(), n, leaf, min_points_per_voxel, range_min, box6, A->out.as<float4>(),
                                out_voxel_idx ? A->vidx.as<int>() : nullptr, out_member_rank ? A->rank.as<int>() : nullptr, info));
  cudaStream_t st = ctx->stream;
  if (out_pts && info->n_out) LGS_CUDA(cudaMemcpyAsync(out_pts, A->out.p, static_cast<size_t>(info->n_out) * 16, cudaMemcpyDeviceToHost, st));
  if (out_voxel_idx && n) LGS_CUDA(cudaMemcpyAsync(out_voxel_idx, A->vidx.p, static_cast<size_t>(n) * 4, cudaMemcpyDeviceToHost, st));
  if (out_member_rank && n) LGS_CUDA(cudaMemcpyAsync(out_member_rank, A->rank.p, static_cast<size_t>(n) * 4, cudaMemcpyDeviceToHost, st));
  LGS_CUDA(cudaStreamSynchronize(st));
  return LGS_OK;
}

// The wide entry points check every argument before anything is queued (the narrow ones above keep their behaviour).
static int check_wide_args(lgs_ctx* ctx, const void* pts, int64_t n, const float* leaf, lgs_voxelgrid_info* info) {
  LGS_REQUIRE(ctx && info && leaf, "null argument");
  LGS_REQUIRE(n >= 0 && n < (int64_t(1) << 31), "point count out of range");
  LGS_REQUIRE(n == 0 || pts != nullptr, "null cloud");
  LGS_REQUIRE(leaf[0] > 0 && leaf[1] > 0 && leaf[2] > 0, "leaf size must be positive");
  return LGS_OK;
}

int lgs_voxelgrid_filter_wide_dev(lgs_ctx* ctx, const float* pts_dev, int64_t n, const float leaf[3], int32_t min_points_per_voxel, double range_min,
                                  const double* box6, float* out_pts_dev, int64_t* out_voxel_idx_dev, int32_t* out_member_rank_dev,
                                  lgs_voxelgrid_info* info) {
  LGS_NVTX("lgs_voxelgrid_filter_wide_dev");
  LGS_TRY(check_wide_args(ctx, pts_dev, n, leaf, info));
  LGS_TRY(lgs::use_device(ctx));
  return lgs::voxelgrid_device(ctx, reinterpret_cast<const float4*>(pts_dev), n, leaf, min_points_per_voxel, range_min, box6,
                               reinterpret_cast<float4*>(out_pts_dev), nullptr, out_member_rank_dev, info, true, out_voxel_idx_dev);
}

int lgs_voxelgrid_filter_wide(lgs_ctx* ctx, const void* pts, int64_t n, int32_t stride_bytes, const float leaf[3], int32_t min_points_per_voxel,
                              double range_min, const double* box6, float* out_pts, int64_t* out_voxel_idx, int32_t* out_member_rank,
                              lgs_voxelgrid_info* info) {
  LGS_NVTX("lgs_voxelgrid_filter_wide");
  LGS_TRY(check_wide_args(ctx, pts, n, leaf, info));
  LGS_REQUIRE(stride_bytes >= 12 && stride_bytes % 4 == 0, "stride_bytes must be a multiple of 4 and >= 12");
  LGS_TRY(lgs::use_device(ctx));
  LGS_TRY(lgs::upload_cloud(ctx, pts, n, stride_bytes, &ctx->vg_in));
  const size_t nn = static_cast<size_t>(n > 0 ? n : 1);
  LGS_TRY(ctx->vg_out.reserve(nn * 16));
  if (out_voxel_idx) LGS_TRY(ctx->vg_vidx.reserve(nn * 8));
  if (out_member_rank) LGS_TRY(ctx->vg_rank.reserve(nn * 4));
  LGS_TRY(lgs::voxelgrid_device(ctx, ctx->vg_in.as<float4>(), n, leaf, min_points_per_voxel, range_min, box6, ctx->vg_out.as<float4>(), nullptr,
                                out_member_rank ? ctx->vg_rank.as<int>() : nullptr, info, true, out_voxel_idx ? ctx->vg_vidx.as<int64_t>() : nullptr));
  cudaStream_t st = ctx->stream;
  if (out_pts && info->n_out) LGS_CUDA(cudaMemcpyAsync(out_pts, ctx->vg_out.p, static_cast<size_t>(info->n_out) * 16, cudaMemcpyDeviceToHost, st));
  if (out_voxel_idx && n) LGS_CUDA(cudaMemcpyAsync(out_voxel_idx, ctx->vg_vidx.p, static_cast<size_t>(n) * 8, cudaMemcpyDeviceToHost, st));
  if (out_member_rank && n) LGS_CUDA(cudaMemcpyAsync(out_member_rank, ctx->vg_rank.p, static_cast<size_t>(n) * 4, cudaMemcpyDeviceToHost, st));
  LGS_CUDA(cudaStreamSynchronize(st));
  return LGS_OK;
}

}  // extern "C"
