// Build and query kernels of the exact nearest-neighbour index (see nn.cuh).

#include <cfloat>

#include "nn.cuh"
#include "sort.cuh"

namespace lgs {

struct BoxAcc {
  unsigned mn[3];
  unsigned mx[3];
};

__global__ void nn_box_init_kernel(BoxAcc* acc) {
  if (threadIdx.x < 3) {
    acc->mn[threadIdx.x] = 0xFFFFFFFFu;
    acc->mx[threadIdx.x] = 0u;
  }
}

__global__ void __launch_bounds__(256) nn_bbox_kernel(const float4* __restrict__ pts, int64_t n, BoxAcc* __restrict__ acc) {
  float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    float4 p = pts[i];
    mn[0] = fminf(mn[0], p.x); mx[0] = fmaxf(mx[0], p.x);
    mn[1] = fminf(mn[1], p.y); mx[1] = fmaxf(mx[1], p.y);
    mn[2] = fminf(mn[2], p.z); mx[2] = fmaxf(mx[2], p.z);
  }
  for (int off = 16; off > 0; off >>= 1)
    for (int a = 0; a < 3; a++) {
      mn[a] = fminf(mn[a], __shfl_xor_sync(0xffffffffu, mn[a], off));
      mx[a] = fmaxf(mx[a], __shfl_xor_sync(0xffffffffu, mx[a], off));
    }
  if ((threadIdx.x & 31) == 0)
    for (int a = 0; a < 3; a++) {
      atomicMin(&acc->mn[a], enc_f(mn[a]));
      atomicMax(&acc->mx[a], enc_f(mx[a]));
    }
}

__device__ __forceinline__ unsigned expand10(unsigned v) {
  v = (v * 0x00010001u) & 0xFF0000FFu;
  v = (v * 0x00000101u) & 0x0F00F00Fu;
  v = (v * 0x00000011u) & 0xC30C30C3u;
  v = (v * 0x00000005u) & 0x49249249u;
  return v;
}

__global__ void __launch_bounds__(256) nn_morton_kernel(const float4* __restrict__ pts, int64_t n, const BoxAcc* __restrict__ acc,
                                                       unsigned* __restrict__ codes, unsigned* __restrict__ perm) {
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= n) return;
  float4 p = pts[i];
  float lo[3], hi[3];
  for (int a = 0; a < 3; a++) {
    lo[a] = dec_f_host(acc->mn[a]);
    hi[a] = dec_f_host(acc->mx[a]);
  }
  const float c[3] = {p.x, p.y, p.z};
  unsigned q[3];
  for (int a = 0; a < 3; a++) {
    float ext = hi[a] - lo[a];
    float t = ext > 0.f ? (c[a] - lo[a]) / ext : 0.f;
    t = fminf(fmaxf(t * 1024.0f, 0.0f), 1023.0f);
    q[a] = static_cast<unsigned>(t);
  }
  codes[i] = (expand10(q[0]) << 2) | (expand10(q[1]) << 1) | expand10(q[2]);
  perm[i] = static_cast<unsigned>(i);
}

__global__ void __launch_bounds__(256) nn_gather_kernel(const float4* __restrict__ pts, const unsigned* __restrict__ perm, int64_t n,
                                                       float4* __restrict__ spts) {
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= n) return;
  unsigned src = perm[i];
  float4 p = pts[src];
  p.w = __int_as_float(static_cast<int>(src));
  spts[i] = p;
}

// level 0: one warp per leaf of 32 consecutive sorted points (coalesced 512-byte load, butterfly min / max)
__global__ void __launch_bounds__(256) nn_leaf_box_kernel(const float4* __restrict__ spts, int n, int n_leaves, float4* __restrict__ bmin,
                                                         float4* __restrict__ bmax) {
  const int leaf = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (leaf >= n_leaves) return;
  const float inf = __int_as_float(0x7f800000);
  float mn[3] = {inf, inf, inf}, mx[3] = {-inf, -inf, -inf};
  const int j = leaf * kLeaf + lane;
  if (j < n) {
    const float4 p = spts[j];
    mn[0] = mx[0] = p.x;
    mn[1] = mx[1] = p.y;
    mn[2] = mx[2] = p.z;
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1)
#pragma unroll
    for (int a = 0; a < 3; a++) {
      mn[a] = fminf(mn[a], __shfl_xor_sync(kFullMask, mn[a], off));
      mx[a] = fmaxf(mx[a], __shfl_xor_sync(kFullMask, mx[a], off));
    }
  if (lane == 0) {
    bmin[leaf] = make_float4(mn[0], mn[1], mn[2], 0.f);
    bmax[leaf] = make_float4(mx[0], mx[1], mx[2], 0.f);
  }
}

// level l + 1 from level l: one thread per node, union of its (up to) 32 child boxes
__global__ void __launch_bounds__(128) nn_node_box_kernel(int child_off, int child_cnt, int node_off, int node_cnt, float4* __restrict__ bmin,
                                                         float4* __restrict__ bmax) {
  const int node = blockIdx.x * blockDim.x + threadIdx.x;
  if (node >= node_cnt) return;
  const int b = node * kLeaf, e = min(b + kLeaf, child_cnt);
  float4 lo = bmin[child_off + b], hi = bmax[child_off + b];
  for (int c = b + 1; c < e; c++) {
    const float4 a = bmin[child_off + c], z = bmax[child_off + c];
    lo.x = fminf(lo.x, a.x); lo.y = fminf(lo.y, a.y); lo.z = fminf(lo.z, a.z);
    hi.x = fmaxf(hi.x, z.x); hi.y = fmaxf(hi.y, z.y); hi.z = fmaxf(hi.z, z.z);
  }
  bmin[node_off + node] = lo;
  bmax[node_off + node] = hi;
}

int NNIndex::build(lgs_ctx* ctx, const float4* pts, int64_t n_in) {
  LGS_REQUIRE(n_in >= 0 && n_in < (int64_t(1) << 31), "point count out of range");
  n = n_in;
  n_levels = 0;
  if (n == 0) return LGS_OK;
  cudaStream_t st = ctx->stream;
  // level sizes: cnt[0] leaves, then ceil(/32) per level; padded to 3 or 6 levels (see nn.cuh)
  int64_t c = (n + kLeaf - 1) / kLeaf, total = 0;
  for (int l = 0; l < kMaxLevels; l++) {
    cnt[l] = static_cast<int>(c);
    off[l] = static_cast<int>(total);
    total += c;
    c = (c + kLeaf - 1) / kLeaf;
  }
  n_levels = cnt[2] <= kLeaf ? 3 : 6;
  LGS_TRY(spts.reserve(static_cast<size_t>(n) * 16));
  LGS_TRY(bmin.reserve(static_cast<size_t>(total) * 16));
  LGS_TRY(bmax.reserve(static_cast<size_t>(total) * 16));
  LGS_TRY(codes.reserve(static_cast<size_t>(n) * 4));
  LGS_TRY(codes_alt.reserve(static_cast<size_t>(n) * 4));
  LGS_TRY(perm.reserve(static_cast<size_t>(n) * 4));
  LGS_TRY(perm_alt.reserve(static_cast<size_t>(n) * 4));
  LGS_TRY(small.reserve(64));
  BoxAcc* acc = small.as<BoxAcc>();
  nn_box_init_kernel<<<1, 32, 0, st>>>(acc);
  nn_bbox_kernel<<<std::min(grid_for(n, 256), kNumSMs * 8), 256, 0, st>>>(pts, n, acc);
  nn_morton_kernel<<<grid_for(n, 256), 256, 0, st>>>(pts, n, acc, codes.as<unsigned>(), perm.as<unsigned>());
  unsigned *sorted_codes, *sorted_perm;
  LGS_TRY(radix_sort_pairs(ctx, codes.as<unsigned>(), perm.as<unsigned>(), codes_alt.as<unsigned>(), perm_alt.as<unsigned>(), n, 30, &sorted_codes,
                           &sorted_perm));
  nn_gather_kernel<<<grid_for(n, 256), 256, 0, st>>>(pts, sorted_perm, n, spts.as<float4>());
  nn_leaf_box_kernel<<<grid_for(static_cast<int64_t>(cnt[0]) * 32, 256), 256, 0, st>>>(spts.as<float4>(), static_cast<int>(n), cnt[0],
                                                                                     bmin.as<float4>(), bmax.as<float4>());
  ctx->launches += 5;
  for (int l = 1; l < n_levels; l++) {
    nn_node_box_kernel<<<grid_for(cnt[l], 128), 128, 0, st>>>(off[l - 1], cnt[l - 1], off[l], cnt[l], bmin.as<float4>(), bmax.as<float4>());
    ctx->launches++;
  }
  LGS_CUDA(cudaGetLastError());
  return LGS_OK;
}

// ---------------------------------------------------------------------------------------------
// fitness: pcl::Registration::getFitnessScore

constexpr int kFitBlock = 256;
constexpr int kFitWarps = kFitBlock / 32;

// one warp per source point; lane 0 of every warp accumulates its points in index order, warps and blocks are
// combined in a fixed order: reproducible sums
struct FitTransform {
  float m[16];  // column-major
};
struct FitRecord {  // loop-closure batch: the pair's record, completed with the fitness and stored by the last block
  lgs_align_result* dst;
  lgs_align_result proto;
};

__global__ void record_write_kernel(const FitRecord rec) {
  if (threadIdx.x == 0) *rec.dst = rec.proto;
}

__global__ void __launch_bounds__(kFitBlock) nn_fitness_kernel(NNView v, const float4* __restrict__ src, int n, const FitTransform Tp,
                                                              double max_range, double* __restrict__ partials, double* __restrict__ result,
                                                              unsigned* __restrict__ counter, const Mailbox mb, const FitRecord rec) {
  __shared__ float T[16];
  if (threadIdx.x < 16) T[threadIdx.x] = Tp.m[threadIdx.x];
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double sum = 0.0, cnt = 0.0;
  for (int i = blockIdx.x * kFitWarps + warp; i < n; i += gridDim.x * kFitWarps) {
    const float4 p = __ldg(src + i);
    const float3 q = transform_pcl(T, p.x, p.y, p.z);
    float d;
    int id;
    nn_search1_warp(v, q.x, q.y, q.z, lane, d, id);
    if (static_cast<double>(d) <= max_range) {
      sum += static_cast<double>(d);
      cnt += 1.0;
    }
  }
  __shared__ double ssum[kFitWarps], scnt[kFitWarps];
  __shared__ bool is_last;
  if (lane == 0) {
    ssum[warp] = sum;
    scnt[warp] = cnt;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0, c = 0;
    for (int w = 0; w < kFitWarps; w++) {
      s += ssum[w];
      c += scnt[w];
    }
    partials[2 * blockIdx.x] = s;
    partials[2 * blockIdx.x + 1] = c;
    __threadfence();
    is_last = atomicAdd(counter, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (is_last && threadIdx.x < 32) {
    __threadfence();
    double s = 0, c = 0;
    for (unsigned b = lane; b < gridDim.x; b += 32) {
      s += __ldcg(partials + 2 * b);
      c += __ldcg(partials + 2 * b + 1);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      s += __shfl_xor_sync(kFullMask, s, off);
      c += __shfl_xor_sync(kFullMask, c, off);
    }
    if (lane == 0) {
      result[0] = s;
      result[1] = c;
      *counter = 0;
      mailbox_publish_one(mb, 0, s);  // the host reads sum and count from mapped pinned memory: no D2H copy, no synchronise
      mailbox_publish_one(mb, 1, c);
      if (rec.dst) {  // same f64 division as the host's (nn_fitness below): the two copies of the record are bit-identical
        lgs_align_result r = rec.proto;
        r.fitness = c > 0 ? s / c : 1.7976931348623157e308;
        *rec.dst = r;
      }
    }
  }
}

int nn_fitness(lgs_ctx* ctx, const NNIndex& index, const float4* src, int64_t n_src, const float* T16, double max_range, double* fitness) {
  *fitness = std::numeric_limits<double>::max();
  cudaStream_t st = ctx->stream;
  FitRecord rec;
  rec.dst = ctx->rec_out_dev;
  rec.proto = ctx->rec_out_proto;
  ctx->rec_out_dev = nullptr;  // one-shot
  if (n_src == 0 || index.n == 0) {
    if (rec.dst) {
      rec.proto.fitness = *fitness;
      record_write_kernel<<<1, 32, 0, st>>>(rec);
      ctx->launches++;
      LGS_CUDA(cudaGetLastError());
    }
    return LGS_OK;
  }
  const int grid = std::max(1, std::min(grid_for(n_src, kFitWarps), kNumSMs * 8));
  LGS_TRY(ctx->tmp[0].reserve(static_cast<size_t>(grid) * 16 + 256));
  double* partials = ctx->tmp[0].as<double>();
  double* result = partials + 2 * grid;
  unsigned* counter = reinterpret_cast<unsigned*>(result + 2);
  FitTransform Tp;
  memcpy(Tp.m, T16, sizeof(Tp.m));
  Mailbox mb;
  LGS_TRY(mailbox_next(ctx, &mb));
  LGS_CUDA(cudaMemsetAsync(counter, 0, 4, st));
  nn_fitness_kernel<<<grid, kFitBlock, 0, st>>>(index.view(), src, static_cast<int>(n_src), Tp, max_range, partials, result, counter, mb, rec);
  ctx->launches++;
  LGS_CUDA(cudaGetLastError());
  double h[2];
  LGS_TRY(mailbox_wait(ctx, mb, 2, h));
  if (h[1] > 0) *fitness = h[0] / h[1];
  return LGS_OK;
}

// ---------------------------------------------------------------------------------------------
// k-NN

constexpr int kKnnBlock = 256;
constexpr int kKnnWarps = kKnnBlock / 32;

// one warp per query.  SELF: query t is sorted point t (consecutive warps search neighbouring regions, so the boxes
// and leaves they touch are shared through L1) and the row written is the point's original index.
template <bool SELF>
__global__ void __launch_bounds__(kKnnBlock) nn_knn_kernel(NNView v, const float4* __restrict__ queries, int m, int k, int* __restrict__ out_idx,
                                                          float* __restrict__ out_d2) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int t = blockIdx.x * kKnnWarps + warp; t < m; t += gridDim.x * kKnnWarps) {
    const float4 qp = SELF ? __ldg(v.spts + t) : __ldg(queries + t);
    const int row = SELF ? __float_as_int(qp.w) : t;
    NNKBest B;
    nn_searchk_warp(v, qp.x, qp.y, qp.z, lane, k, B);
    if (lane < k) {
      const bool have = B.bi() != 0x7fffffff;
      out_idx[static_cast<size_t>(row) * k + lane] = have ? B.bi() : -1;
      if (out_d2) out_d2[static_cast<size_t>(row) * k + lane] = have ? B.bd() : 0.f;
    }
  }
}

// the same search for a device-side list of indexed points (lazy covariances, gicp.cu)
__global__ void __launch_bounds__(kKnnBlock) nn_knn_list_kernel(NNView v, const float4* __restrict__ pts, const int* __restrict__ list,
                                                               const int* __restrict__ count, int k, int* __restrict__ out_idx) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int m = *count;
  for (int t = blockIdx.x * kKnnWarps + warp; t < m; t += gridDim.x * kKnnWarps) {
    const float4 qp = __ldg(pts + list[t]);
    NNKBest B;
    nn_searchk_warp(v, qp.x, qp.y, qp.z, lane, k, B);
    if (lane < k) out_idx[static_cast<size_t>(t) * k + lane] = B.bi() != 0x7fffffff ? B.bi() : -1;
  }
}

// the 1-NN of the correspondence searches (gicp_correspondence_kernel, icp_step_body) with their seed handling: seeds[t]
// outside [0, n) means no seed, otherwise the search starts from that point of the original (unsorted) cloud `pts`.
// seeds == nullptr: the unseeded search of getFitnessScore and pclomp GICP.
__global__ void __launch_bounds__(kKnnBlock) nn_search1_kernel(NNView v, const float4* __restrict__ pts, const float4* __restrict__ queries, int m,
                                                              const int* __restrict__ seeds, int* __restrict__ out_idx, float* __restrict__ out_d2) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int t = blockIdx.x * kKnnWarps + warp; t < m; t += gridDim.x * kKnnWarps) {
    const float4 q = __ldg(queries + t);
    float d2;
    int id;
    if (seeds) {
      int seed = seeds[t];
      if (seed >= v.n) seed = -1;
      float seed_d = 0.f;
      if (seed >= 0) seed_d = nn_dist2(q.x, q.y, q.z, __ldg(pts + seed));
      nn_search1_warp_seeded(v, q.x, q.y, q.z, lane, seed_d, seed, d2, id);
    } else {
      nn_search1_warp(v, q.x, q.y, q.z, lane, d2, id);
    }
    if (lane == 0) {
      out_idx[t] = id;
      if (out_d2) out_d2[t] = d2;
    }
  }
}

static int knn_grid(int64_t m) { return static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((m + kKnnWarps - 1) / kKnnWarps, kNumSMs * 64))); }

int nn_self_knn(lgs_ctx* ctx, const NNIndex& index, int k, int* out_idx_dev, float* out_d2_dev) {
  LGS_REQUIRE(k >= 1 && k <= kMaxK, "k must be in [1, 32]");
  if (index.n == 0) return LGS_OK;
  nn_knn_kernel<true><<<knn_grid(index.n), kKnnBlock, 0, ctx->stream>>>(index.view(), nullptr, static_cast<int>(index.n), k, out_idx_dev, out_d2_dev);
  ctx->launches++;
  LGS_CUDA(cudaGetLastError());
  return LGS_OK;
}

int nn_knn_list(lgs_ctx* ctx, const NNIndex& index, const float4* pts, const int* list_dev, const int* count_dev, int64_t capacity, int k,
                int* out_idx_dev) {
  LGS_REQUIRE(k >= 1 && k <= kMaxK, "k must be in [1, 32]");
  if (capacity == 0 || index.n == 0) return LGS_OK;
  // a quarter of the capacity's grid: the list is usually much shorter than its bound and the kernel strides
  nn_knn_list_kernel<<<std::max(1, knn_grid(capacity) / 4), kKnnBlock, 0, ctx->stream>>>(index.view(), pts, list_dev, count_dev, k, out_idx_dev);
  ctx->launches++;
  LGS_CUDA(cudaGetLastError());
  return LGS_OK;
}

int nn_knn(lgs_ctx* ctx, const NNIndex& index, const float4* queries, int64_t m, int k, int* out_idx_dev, float* out_d2_dev) {
  LGS_REQUIRE(k >= 1 && k <= kMaxK, "k must be in [1, 32]");
  if (m == 0) return LGS_OK;
  if (index.n == 0) {
    LGS_CUDA(cudaMemsetAsync(out_idx_dev, 0xFF, static_cast<size_t>(m) * k * 4, ctx->stream));
    if (out_d2_dev) LGS_CUDA(cudaMemsetAsync(out_d2_dev, 0, static_cast<size_t>(m) * k * 4, ctx->stream));
    return LGS_OK;
  }
  nn_knn_kernel<false><<<knn_grid(m), kKnnBlock, 0, ctx->stream>>>(index.view(), queries, static_cast<int>(m), k, out_idx_dev, out_d2_dev);
  ctx->launches++;
  LGS_CUDA(cudaGetLastError());
  return LGS_OK;
}

}  // namespace lgs

extern "C" int lgs_knn(lgs_ctx* ctx, const void* pts, int64_t n, int32_t stride_bytes, const void* queries, int64_t m, int32_t qstride_bytes, int32_t k,
                       int32_t* idx, float* d2) {
  using namespace lgs;
  LGS_REQUIRE(ctx && idx, "null argument");
  LGS_REQUIRE(k >= 1 && k <= kMaxK, "k must be in [1, 32]");
  LGS_TRY(use_device(ctx));
  DevBuf cloud, q, oi, od;
  NNIndex index;
  int rc = LGS_OK;
  do {
    if ((rc = upload_cloud(ctx, pts, n, stride_bytes, &cloud)) != LGS_OK) break;
    if ((rc = upload_cloud(ctx, queries, m, qstride_bytes, &q)) != LGS_OK) break;
    if ((rc = index.build(ctx, cloud.as<float4>(), n)) != LGS_OK) break;
    if ((rc = oi.reserve(static_cast<size_t>(m > 0 ? m : 1) * k * 4)) != LGS_OK) break;
    if ((rc = od.reserve(static_cast<size_t>(m > 0 ? m : 1) * k * 4)) != LGS_OK) break;
    if ((rc = nn_knn(ctx, index, q.as<float4>(), m, k, oi.as<int>(), od.as<float>())) != LGS_OK) break;
    if (m) {
      cudaMemcpyAsync(idx, oi.p, static_cast<size_t>(m) * k * 4, cudaMemcpyDeviceToHost, ctx->stream);
      if (d2) cudaMemcpyAsync(d2, od.p, static_cast<size_t>(m) * k * 4, cudaMemcpyDeviceToHost, ctx->stream);
    }
    if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) {
      set_error("lgs_knn: stream synchronize failed");
      rc = LGS_ERR_CUDA;
    }
  } while (false);
  cloud.release();
  q.release();
  oi.release();
  od.release();
  index.release();
  return rc;
}

extern "C" int lgs_nn_search1(lgs_ctx* ctx, const void* pts, int64_t n, int32_t stride_bytes, const void* queries, int64_t m, int32_t qstride_bytes,
                              const int32_t* seeds, int32_t* idx, float* d2) {
  using namespace lgs;
  LGS_REQUIRE(ctx && idx, "null argument");
  LGS_TRY(use_device(ctx));
  DevBuf cloud, q, s, oi, od;
  NNIndex index;
  int rc = LGS_OK;
  do {
    if ((rc = upload_cloud(ctx, pts, n, stride_bytes, &cloud)) != LGS_OK) break;
    if ((rc = upload_cloud(ctx, queries, m, qstride_bytes, &q)) != LGS_OK) break;
    if (m == 0) break;
    if (n == 0) {  // nothing indexed: no neighbour, at infinite distance
      for (int64_t t = 0; t < m; t++) {
        idx[t] = -1;
        if (d2) d2[t] = std::numeric_limits<float>::infinity();
      }
      break;
    }
    if ((rc = index.build(ctx, cloud.as<float4>(), n)) != LGS_OK) break;
    if ((rc = oi.reserve(static_cast<size_t>(m) * 4)) != LGS_OK) break;
    if ((rc = od.reserve(static_cast<size_t>(m) * 4)) != LGS_OK) break;
    if (seeds) {
      if ((rc = s.reserve(static_cast<size_t>(m) * 4)) != LGS_OK) break;
      cudaMemcpyAsync(s.p, seeds, static_cast<size_t>(m) * 4, cudaMemcpyHostToDevice, ctx->stream);
    }
    nn_search1_kernel<<<knn_grid(m), kKnnBlock, 0, ctx->stream>>>(index.view(), cloud.as<float4>(), q.as<float4>(), static_cast<int>(m),
                                                                  seeds ? s.as<int>() : nullptr, oi.as<int>(), od.as<float>());
    ctx->launches++;
    if (cudaGetLastError() != cudaSuccess) {
      set_error("lgs_nn_search1: launch failed");
      rc = LGS_ERR_CUDA;
      break;
    }
    cudaMemcpyAsync(idx, oi.p, static_cast<size_t>(m) * 4, cudaMemcpyDeviceToHost, ctx->stream);
    if (d2) cudaMemcpyAsync(d2, od.p, static_cast<size_t>(m) * 4, cudaMemcpyDeviceToHost, ctx->stream);
    if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) {
      set_error("lgs_nn_search1: stream synchronize failed");
      rc = LGS_ERR_CUDA;
    }
  } while (false);
  cloud.release();
  q.release();
  s.release();
  oi.release();
  od.release();
  index.release();
  return rc;
}
