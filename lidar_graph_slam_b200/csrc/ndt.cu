// NDT scan-to-map registration: pclomp::NormalDistributionsTransform behind the pcl::Registration surface.
//
//   set_target   -> VoxelGridCovariance::applyFilter (VGC:48-370): bbox, keys, stable radix sort, then one thread
//                   per occupied voxel accumulates sum(x), sum(x x^T) in f64 in ascending point index (the
//                   reference's serial order => bit-identical sums), finishes mean / covariance / eigen
//                   regularisation / inverse, and publishes a 64-byte lookup record + a cell-table entry.
//   derivatives  -> computeDerivatives (NDT:179-285) fused with transformPointCloud and getNeighborhoodAtPoint7
//                   (VGC:373-433): float4 point load, on-the-fly f32 transform, <=27 cell-table probes,
//                   f32 point terms (NDT:397-439,483-536), f64 accumulation, block reduction of 43 doubles,
//                   last-block fixed-order final reduction (deterministic).
//   hessian_f64  -> computeHessian / updateHessian (NDT:539-644) in f64.
//   align        -> computeTransformation (NDT:80-171) + computeStepLengthMT (NDT:771-931) driven from the host;
//                   each evaluation is one kernel launch + one 352-byte D2H.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <limits>
#include <utility>
#include <vector>

#include "keyframes.cuh"
#include "math.cuh"
#include "nn.cuh"
#include "sort.cuh"
#include "voxel_common.cuh"

namespace lgs {

// 64-byte voxel record read by the derivative kernels (4 x 16-byte loads)
struct __align__(16) VoxelRec {
  double mean[3];
  float icov[9];
  int n;
};
static_assert(sizeof(VoxelRec) == 64, "VoxelRec must be 64 bytes");

struct CellTable {
  int dense;            // 1: table[lin] = record index or -1 ; 0: open-addressing hash
  const int* table;     // dense table, or hash values
  const int* hkeys;     // hash keys (-1 = empty)
  unsigned hmask;
  float leaf[3];
  float inv_leaf[3];    // exact reciprocals when every leaf is a power of two (leaf_pow2): x / leaf == x * inv_leaf bit for bit
  int leaf_pow2;
  int min_b[3], max_b[3], mul[3];
};

__device__ __forceinline__ unsigned hash_u32(unsigned x) {
  x ^= x >> 16;
  x *= 0x7feb352du;
  x ^= x >> 15;
  x *= 0x846ca68bu;
  x ^= x >> 16;
  return x;
}

__device__ __forceinline__ int cell_lookup(const CellTable& ct, int lin) {
  if (ct.dense) return __ldg(ct.table + lin);
  unsigned h = hash_u32(static_cast<unsigned>(lin)) & ct.hmask;
  while (true) {
    int k = __ldg(ct.hkeys + h);
    if (k == lin) return __ldg(ct.table + h);
    if (k == -1) return -1;
    h = (h + 1) & ct.hmask;
  }
}

// ---------------------------------------------------------------------------------------------
// target voxelisation

struct VoxelExport {  // f64 per-voxel data, ascending idx (parity hook + operands of the f64 Hessian path)
  int* idx;
  int* nr_points;
  double* mean;  // 3
  double* cov;   // 9
  double* icov;  // 9
};

// pass 1 (VGC:233-237): mean_ += p ; cov_ += p p^T in f64, members in ascending point index - the reference's serial
// order, which is what makes the sums (and with them the validity flags) bit-identical to the oracle's.  One WARP per
// voxel.  The lanes fetch 32 members at a time (index, then point: two dependent gathers, pipelined two chunks deep; a
// single thread would pay their latency once per member, and the largest voxel of a map - hundreds of points - used to set
// the kernel's duration).  Every lane widens ITS member and forms the nine addends x, y, z, xx, xy, xz, yy, yz, zz once
// (exactly the products the serial loop forms) and parks them in shared memory; then lane a (0..8) adds addend a of member
// 0, 1, 2, ... in order.  Per member that is one shared-memory read off the critical path and one DADD on it: ~8 cycles,
// the latency of the addition chain that the order fixes (tools/microbench/chain.cu; selecting operands per member after
// three shuffles costs 47, a per-lane `?:` that compiles to divergent branches 260).
constexpr int kSumsPerVoxel = 9;
constexpr int kSumsWarps = 8;
__global__ void __launch_bounds__(kSumsWarps * 32) voxel_sums_kernel(const float4* __restrict__ pts, const unsigned* __restrict__ vals,
                                                                    const int* __restrict__ seg_start, int n_seg, int64_t n_pts, double* __restrict__ sums) {
  __shared__ double addend[kSumsWarps][2][32][kSumsPerVoxel];  // [warp][buffer][member][addend], 36 KB
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int v = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (v >= n_seg) return;
  const int b = seg_start[v];
  const int e = (v + 1 < n_seg) ? seg_start[v + 1] : static_cast<int>(n_pts);
  auto park = [&](int buf, const float4& p) {
    const double x = static_cast<double>(p.x), y = static_cast<double>(p.y), z = static_cast<double>(p.z);
    double* a = addend[warp][buf][lane];
    a[0] = x;
    a[1] = y;
    a[2] = z;
    a[3] = __dmul_rn(x, x);
    a[4] = __dmul_rn(x, y);
    a[5] = __dmul_rn(x, z);
    a[6] = __dmul_rn(y, y);
    a[7] = __dmul_rn(y, z);
    a[8] = __dmul_rn(z, z);
  };
  double acc = 0.0;
  const int col = lane < kSumsPerVoxel ? lane : 0;
  float4 cur = make_float4(0.f, 0.f, 0.f, 0.f);
  if (b + lane < e) cur = __ldg(pts + __ldg(vals + b + lane));
  int idx_next = b + 32 + lane < e ? static_cast<int>(__ldg(vals + b + 32 + lane)) : -1;
  int buf = 0;
  for (int c0 = b; c0 < e; c0 += 32, buf ^= 1) {
    float4 nxt = make_float4(0.f, 0.f, 0.f, 0.f);
    if (idx_next >= 0) nxt = __ldg(pts + idx_next);  // points of the next chunk and indices of the one after: in flight
    idx_next = c0 + 64 + lane < e ? static_cast<int>(__ldg(vals + c0 + 64 + lane)) : -1;
    park(buf, cur);
    __syncwarp();
    const int cnt = min(32, e - c0);
    const double* mine = &addend[warp][buf][0][col];
#pragma unroll 8
    for (int t = 0; t < cnt; t++) acc = __dadd_rn(acc, mine[t * kSumsPerVoxel]);
    cur = nxt;  // (the other buffer is parked next: a lane still reading this one is never overtaken by more than one chunk,
  }             //  and the __syncwarp above separates its reads from the writes two chunks later)
  if (lane < kSumsPerVoxel) sums[static_cast<size_t>(v) * kSumsPerVoxel + lane] = acc;
}

// pass 2 (VGC:282-367): one thread per voxel finishes mean / covariance / eigen regularisation / inverse and publishes the
// lookup record and the cell-table entry.
// counts: members per voxel when a voxel's entries are partial sums of several key frames (rolling map); otherwise the
// segment length is the member count.
__global__ void __launch_bounds__(128) voxel_stats_kernel(const double* __restrict__ sums, const unsigned* __restrict__ keys,
                                                         const int* __restrict__ seg_start, const int* __restrict__ counts, int n_seg,
                                                         int64_t n_pts, int min_pts, double eig_mult, VoxelExport ex, VoxelRec* __restrict__ recs,
                                                         int* __restrict__ dense_table, int* __restrict__ hkeys, int* __restrict__ hvals,
                                                         unsigned hmask, int* __restrict__ n_valid) {
  int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n_seg) return;
  const int b = seg_start[v];
  const int e = (v + 1 < n_seg) ? seg_start[v + 1] : static_cast<int>(n_pts);
  const int key = static_cast<int>(keys[b]);
  const double* sv = sums + static_cast<size_t>(v) * kSumsPerVoxel;
  const double s0 = sv[0], s1 = sv[1], s2 = sv[2], c00 = sv[3], c01 = sv[4], c02 = sv[5], c11 = sv[6], c12 = sv[7], c22 = sv[8];
  int n = counts ? counts[v] : e - b;
  double cov[9] = {c00, c01, c02, c01, c11, c12, c02, c12, c22};
  double sum[3] = {s0, s1, s2};
  double mean[3] = {s0 / n, s1 / n, s2 / n};  // VGC:293
  double icov[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  int nr_points = n;
  if (n >= min_pts) {
    // VGC:329-330
    const double dn = n;
    for (int a = 0; a < 3; a++)
      for (int c = 0; c < 3; c++) cov[a * 3 + c] = (cov[a * 3 + c] - 2 * (sum[a] * mean[c])) / dn + mean[a] * mean[c];
    const double f = (n - 1.0) / n;
    for (int k = 0; k < 9; k++) cov[k] *= f;
    double ev[3], V[9];
    m::eig_sym3(cov, ev, V);  // VGC:333-335
    if (ev[0] < 0 || ev[1] < 0 || ev[2] <= 0) {
      nr_points = -1;  // VGC:337-341
    } else {
      const double min_ev = eig_mult * ev[2];  // VGC:345-356
      if (ev[0] < min_ev) {
        ev[0] = min_ev;
        if (ev[1] < min_ev) ev[1] = min_ev;
        double D[9] = {ev[0], 0, 0, 0, ev[1], 0, 0, 0, ev[2]};
        double Vi[9], VD[9];
        m::inv3(V, Vi);
        m::mul3(V, D, VD);
        m::mul3(VD, Vi, cov);
      }
      m::inv3(cov, icov);  // VGC:359-364
      double mxc = icov[0], mnc = icov[0];
      for (int k = 1; k < 9; k++) {
        mxc = fmax(mxc, icov[k]);
        mnc = fmin(mnc, icov[k]);
      }
      const double finf = static_cast<double>(__int_as_float(0x7f800000));
      if (mxc == finf || mnc == -finf) nr_points = -1;
    }
  }
  ex.idx[v] = key;
  ex.nr_points[v] = nr_points;
  for (int a = 0; a < 3; a++) ex.mean[v * 3 + a] = mean[a];
  for (int k = 0; k < 9; k++) {
    ex.cov[v * 9 + k] = cov[k];
    ex.icov[v * 9 + k] = icov[k];
  }
  if (nr_points >= min_pts) {  // visible to the lookup (VGC:395)
    VoxelRec r;
    for (int a = 0; a < 3; a++) r.mean[a] = mean[a];
    for (int k = 0; k < 9; k++) r.icov[k] = static_cast<float>(icov[k]);  // c_inv.cast<float>() (NDT:493)
    r.n = nr_points;
    recs[v] = r;
    if (dense_table) {
      dense_table[key] = v;
    } else {
      unsigned h = hash_u32(static_cast<unsigned>(key)) & hmask;
      while (true) {
        int prev = atomicCAS(hkeys + h, -1, key);
        if (prev == -1 || prev == key) {
          hvals[h] = v;
          break;
        }
        h = (h + 1) & hmask;
      }
    }
    atomicAdd(n_valid, 1);
  }
}

// ---------------------------------------------------------------------------------------------
// rolling map: merging cached per-key-frame voxel partial sums (lgs_ndt_set_target_keyframes)

// per key frame, after its own voxelisation: local voxel index and member count of every occupied voxel
__global__ void __launch_bounds__(256) frame_pack_kernel(const unsigned* __restrict__ keys, const int* __restrict__ seg_start, int n_seg, int64_t n_kept,
                                                        unsigned* __restrict__ out_keys, int* __restrict__ out_cnt) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n_seg) return;
  const int b = seg_start[v];
  const int e = (v + 1 < n_seg) ? seg_start[v + 1] : static_cast<int>(n_kept);
  out_keys[v] = keys[b];
  out_cnt[v] = e - b;
}

constexpr int kMergeFrames = 40;  // key frames per gather launch (kernel parameter space); longer lists are split
struct MergeSegments {
  const unsigned* keys[kMergeFrames];
  const int* cnt[kMergeFrames];
  const double* sums[kMergeFrames];
  int begin[kMergeFrames + 1];  // first entry of each frame (relative to this launch)
  int fmin[kMergeFrames][3];    // the frame grid's min_b minus the map's min_b
  int fdx[kMergeFrames], fdxy[kMergeFrames];
  int gmul[3];
  int count;
};

// every cached entry (frame-major, i.e. in the order the reference concatenates the key frames) gets its voxel index in the
// MAP's grid; counts and sums are copied next to it
__global__ void __launch_bounds__(256) frame_gather_kernel(const MergeSegments S, int out0, unsigned* __restrict__ gkeys, unsigned* __restrict__ gvals,
                                                          int* __restrict__ ccnt, double* __restrict__ csum) {
  __shared__ int begin[kMergeFrames + 1];
  for (int t = threadIdx.x; t <= S.count; t += blockDim.x) begin[t] = S.begin[t];
  __syncthreads();
  const int total = begin[S.count];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    int lo = 0, hi = S.count - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (begin[mid] <= i) lo = mid; else hi = mid - 1;
    }
    const int l = i - begin[lo];
    const unsigned key = S.keys[lo][l];
    const int iz = static_cast<int>(key / static_cast<unsigned>(S.fdxy[lo]));
    const int rem = static_cast<int>(key % static_cast<unsigned>(S.fdxy[lo]));
    const int iy = rem / S.fdx[lo], ix = rem % S.fdx[lo];
    const int g = (ix + S.fmin[lo][0]) * S.gmul[0] + (iy + S.fmin[lo][1]) * S.gmul[1] + (iz + S.fmin[lo][2]) * S.gmul[2];
    const int o = out0 + i;
    gkeys[o] = static_cast<unsigned>(g);
    gvals[o] = static_cast<unsigned>(o);
    ccnt[o] = S.cnt[lo][l];
#pragma unroll
    for (int c = 0; c < kSumsPerVoxel; c++) csum[static_cast<size_t>(o) * kSumsPerVoxel + c] = S.sums[lo][static_cast<size_t>(l) * kSumsPerVoxel + c];
  }
}

struct MergeHeads {  // start offset of every run of equal map voxel indices (sort.cuh scan_select functor)
  const unsigned* keys;
  int* seg_start;
  __device__ bool flag(int64_t i) const { return i == 0 || keys[i] != keys[i - 1]; }
  __device__ void emit(int64_t i, int64_t pos, bool f) const {
    if (f) seg_start[pos] = static_cast<int>(i);
  }
};

// one thread per (map voxel, sum): the key frames' partial sums are added in key-frame order (the stable sort kept it)
__global__ void __launch_bounds__(256) frame_merge_kernel(const unsigned* __restrict__ svals, const int* __restrict__ seg_start, int n_seg, int n_entries,
                                                         const int* __restrict__ ccnt, const double* __restrict__ csum, double* __restrict__ msum,
                                                         int* __restrict__ mcnt) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int v = t / (kSumsPerVoxel + 1), c = t % (kSumsPerVoxel + 1);
  if (v >= n_seg) return;
  const int b = seg_start[v];
  const int e = (v + 1 < n_seg) ? seg_start[v + 1] : n_entries;
  if (c == kSumsPerVoxel) {
    int n = 0;
    for (int j = b; j < e; j++) n += ccnt[svals[j]];
    mcnt[v] = n;
  } else {
    double a = 0.0;
    for (int j = b; j < e; j++) a = __dadd_rn(a, csum[static_cast<size_t>(svals[j]) * kSumsPerVoxel + c]);
    msum[static_cast<size_t>(v) * kSumsPerVoxel + c] = a;
  }
}

// ---------------------------------------------------------------------------------------------
// derivative evaluation

struct EvalParams {
  float T[16];          // column-major transform applied to the source points
  float j_ang[8][3];    // NDT:339-346 (rows a..h), f32
  float h_ang[15][3];   // NDT:373-392 (rows a2..f3), f32
  double j_ang_d[8][3]; // f64 copies for computeHessian (NDT:329-336, 351-370)
  double h_ang_d[15][3];
  double gauss_d1, gauss_d2;
  float gauss_d2f;
  int n_offsets;
  signed char off[27][3];
};

constexpr int kEvalBlock = 128;
constexpr int kNumAcc = 44;  // score, g[6], H[36], term count

// block-wide sum of K doubles held per thread -> partials[blockIdx][k]; the last block to finish adds the
// per-block partials in block order (fixed tree => run-to-run reproducible) and writes result[k].
template <int K>
__device__ __forceinline__ void block_reduce_and_finish(double (&acc)[K], double* __restrict__ partials, double* __restrict__ result,
                                                       unsigned* __restrict__ counter, const Mailbox& mb) {
  __shared__ double sm[kEvalBlock / 32][K];
  __shared__ bool is_last;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < K; k++) {
    double v = acc[k];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    if (lane == 0) sm[warp][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < K) {
    double v = 0;
#pragma unroll
    for (int w = 0; w < kEvalBlock / 32; w++) v += sm[w][threadIdx.x];
    partials[static_cast<size_t>(blockIdx.x) * K + threadIdx.x] = v;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned done = atomicAdd(counter, 1u);
    is_last = (done == gridDim.x - 1);
  }
  __syncthreads();
  if (is_last) {
    __threadfence();
    double v = 0;
    if (threadIdx.x < K) {
      for (unsigned b0 = 0; b0 < gridDim.x; b0 += 8) {  // eight independent loads in flight, added in block order
        double t[8];
#pragma unroll
        for (int u = 0; u < 8; u++) t[u] = b0 + u < gridDim.x ? __ldcg(partials + static_cast<size_t>(b0 + u) * K + threadIdx.x) : 0.0;
#pragma unroll
        for (int u = 0; u < 8; u++) v += t[u];
      }
      result[threadIdx.x] = v;
    }
    if (threadIdx.x == 0) *counter = 0;  // re-arm for the next launch on this stream
    mailbox_publish<K>(mb, v);
  }
}

}  // namespace lgs

#include "ndt_opt.cuh"
#include "ndt_deriv.cuh"

namespace lgs {

// calculateScore (NDT:934-982)
__global__ void __launch_bounds__(kEvalBlock) ndt_score_kernel(const float4* __restrict__ src, int n, EvalParams P, CellTable ct,
                                                             const double* __restrict__ vmean, const double* __restrict__ vicov, double gauss_d3,
                                                             double* __restrict__ partials, double* __restrict__ result, unsigned* __restrict__ counter, const Mailbox mb) {
  double acc[1] = {0.0};
  auto s3 = [](double a, double b, double c) { return a + (b + c); };
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 p = src[i];
    const float3 xt = transform_pcl(P.T, p.x, p.y, p.z);
    const int ix = static_cast<int>(floorf(__fdiv_rn(xt.x, ct.leaf[0])));
    const int iy = static_cast<int>(floorf(__fdiv_rn(xt.y, ct.leaf[1])));
    const int iz = static_cast<int>(floorf(__fdiv_rn(xt.z, ct.leaf[2])));
    int slots[27];
    int cnt = 0;
    for (int o = 0; o < P.n_offsets; o++) {
      const int cx = ix + P.off[o][0], cy = iy + P.off[o][1], cz = iz + P.off[o][2];
      if (cx < ct.min_b[0] || cx > ct.max_b[0] || cy < ct.min_b[1] || cy > ct.max_b[1] || cz < ct.min_b[2] || cz > ct.max_b[2]) continue;
      const int lin = (cx - ct.min_b[0]) * ct.mul[0] + (cy - ct.min_b[1]) * ct.mul[1] + (cz - ct.min_b[2]) * ct.mul[2];
      const int slot = cell_lookup(ct, lin);
      if (slot >= 0) slots[cnt++] = slot;
    }
    for (int k = 0; k < cnt; k++) {
      const double* mean = vmean + static_cast<size_t>(slots[k]) * 3;
      const double* C = vicov + static_cast<size_t>(slots[k]) * 9;
      const double xx[3] = {static_cast<double>(xt.x) - mean[0], static_cast<double>(xt.y) - mean[1], static_cast<double>(xt.z) - mean[2]};
      double Cx[3];
      for (int r = 0; r < 3; r++) Cx[r] = s3(C[r * 3] * xx[0], C[r * 3 + 1] * xx[1], C[r * 3 + 2] * xx[2]);
      double e = exp(-P.gauss_d2 * s3(xx[0] * Cx[0], xx[1] * Cx[1], xx[2] * Cx[2]) / 2);
      double score_inc = -P.gauss_d1 * e - gauss_d3;
      acc[0] += score_inc / cnt;
    }
  }
  block_reduce_and_finish<1>(acc, partials, result, counter, mb);
}

}  // namespace lgs

// =============================================================================================
// host side

using namespace lgs;

struct lgs_ndt {
  lgs_ctx* ctx = nullptr;
  // parameters, defaults NDT:49-51,71-75
  float resolution = 1.0f;
  double step_size = 0.1, outlier_ratio = 0.55, trans_eps = 0.1;
  int max_iter = 35;
  bool exact_newton_step = false;  // lgs_ndt_set_exact_newton_step
  int search = LGS_NDT_DIRECT7;
  // clouds
  DevBuf target, source, out_cloud;
  int64_t n_target = 0, n_source = 0;
  bool have_target = false, have_source = false;
  // voxel structure
  bool grid_ready = false, refused = false;
  int dense = 1;
  int64_t n_voxels = 0, n_valid = 0;
  int min_b[3] = {0, 0, 0}, max_b[3] = {0, 0, 0}, div_b[3] = {0, 0, 0};
  DevBuf table, hkeys, recs, ex_idx, ex_n, ex_mean, ex_cov, ex_icov, small, vsums;
  unsigned hmask = 0;
  // reduction scratch
  DevBuf partials, result;
  // nearest-neighbour structure over the target for getFitnessScore (lazy)
  NNIndex nn;
  bool nn_ready = false;
  // state of the last align
  float final_T[16];
  double gauss_d1 = 0, gauss_d2 = 0, gauss_d3 = 0;
  EvalParams P;
  int evals = 0, trials = 0, hess_recomputes = 0;
  double last_terms = 0;
  // rolling map (lgs_ndt_set_target_keyframes): the target is a list of key frames of a device-resident key-frame array; every
  // key frame's voxel partial sums are cached (per pose and resolution), a key-frame change voxelises only the new frame
  struct FrameVox {
    int32_t id = -1;
    float pose[16];
    float res = 0;
    int64_t n_points = 0;
    int n_vox = 0;
    int min_b[3] = {0, 0, 0}, div_b[3] = {1, 1, 1}, max_b[3] = {0, 0, 0};
    DevBuf keys, cnt, sums;  // n_vox: local linear voxel index (u32), members (int), 9 f64 sums
    int64_t last_used = 0;
  };
  std::vector<FrameVox*> frame_cache;
  const lgs_keyframes* roll_kf = nullptr;
  std::vector<int32_t> roll_ids;
  bool target_from_frames = false, target_cloud_stale = false;
  int64_t roll_epoch = 0;
  int roll_frames_voxelised = 0;  // key frames voxelised from their points by the last set_target_keyframes
  DevBuf roll_frame, roll_gkeys, roll_gvals, roll_gkeys_alt, roll_gvals_alt, roll_ccnt, roll_csum, roll_msum, roll_mcnt, roll_seg, roll_small, roll_poses;
  // device-resident align (ndt_align_kernel): the hand-over block of the resident grid, and how the last align ran
  lgs::DevBuf align_dev;
  int align_launches = 0;      // ndt_align_kernel launches of the last align (1, or 0 when the host stepped the optimiser)
  double align_trace[16] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};  // CTA 0's cycle breakdown of the last device-resident align
  double terms_total = 0;      // accepted (point, voxel) terms over all evaluations of the last device-resident align
  // optional per-kernel timing (bench.py roofline): CUDA event pairs around each evaluation launch
  int profiling = 0;  // 1: per-evaluation launches timed (host-stepped optimiser), 2: ndt_align_kernel launches timed
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> prof_events[4];  // modes 0, 1, 2 and whole aligns
  double prof_align_evals = 0, prof_align_terms = 0;
};

namespace {

constexpr uint64_t kDenseCellLimit = uint64_t(1) << 26;  // 64 Mi cells (256 MiB of int32) before switching to the hash

// NDT.h:214-231 (ndt_opt.cuh holds the arithmetic, shared with the device-resident optimiser)
void pose_to_matrix(const double x[6], float* T) {
  ndtopt::Trig t;
  ndtopt::trig_of_pose(x, &t);
  ndtopt::pose_to_matrix(x, t, T);
}

using ndtopt::matrix_to_pose;  // NDT:103-111 (ndt_opt.cuh)

void compute_gauss(lgs_ndt* n) {  // NDT:86-93
  double c1 = 10 * (1 - n->outlier_ratio);
  double c2 = n->outlier_ratio / std::pow(static_cast<double>(n->resolution), 3);
  n->gauss_d3 = -std::log(c2);
  n->gauss_d1 = -std::log(c1 + c2) - n->gauss_d3;
  n->gauss_d2 = -2 * std::log((-std::log(c1 * std::exp(-0.5) + c2) - n->gauss_d3) / n->gauss_d1);
}

// computeAngleDerivatives (NDT:288-394; arithmetic in ndt_opt.cuh)
void angle_derivatives(const double p[6], EvalParams* P) {
  ndtopt::Trig t;
  ndtopt::trig_of_pose(p, &t);
  ndtopt::angle_tables(t, P->j_ang_d, P->h_ang_d, P->j_ang, P->h_ang);
}

void fill_offsets(int method, EvalParams* P) {
  static const signed char off7[7][3] = {{0, 0, 0}, {1, 0, 0}, {-1, 0, 0}, {0, 1, 0}, {0, -1, 0}, {0, 0, 1}, {0, 0, -1}};  // VGC:423-430
  if (method == LGS_NDT_DIRECT1) {
    P->n_offsets = 1;
    P->off[0][0] = P->off[0][1] = P->off[0][2] = 0;
  } else if (method == LGS_NDT_DIRECT26) {
    // pcl::getAllNeighborCellIndices: 13 half offsets then their negations (no centre cell)
    int c = 0;
    signed char half[13][3];
    for (int i = -1; i < 2; i++)
      for (int j = -1; j < 2; j++) {
        half[c][0] = i; half[c][1] = j; half[c][2] = -1; c++;
      }
    for (int i = -1; i < 2; i++) {
      half[c][0] = i; half[c][1] = -1; half[c][2] = 0; c++;
    }
    half[c][0] = -1; half[c][1] = 0; half[c][2] = 0;
    for (int t = 0; t < 13; t++)
      for (int a = 0; a < 3; a++) {
        P->off[t][a] = half[t][a];
        P->off[13 + t][a] = -half[t][a];
      }
    P->n_offsets = 26;
  } else {
    P->n_offsets = 7;
    for (int t = 0; t < 7; t++)
      for (int a = 0; a < 3; a++) P->off[t][a] = off7[t][a];
  }
}

CellTable make_cell_table(const lgs_ndt* n) {
  CellTable ct;
  ct.dense = n->dense;
  ct.table = n->table.as<int>();
  ct.hkeys = n->hkeys.as<int>();
  ct.hmask = n->hmask;
  int mant_exp = 0;
  ct.leaf_pow2 = std::frexp(n->resolution, &mant_exp) == 0.5f && mant_exp > -100 && mant_exp < 100 ? 1 : 0;
  for (int a = 0; a < 3; a++) {
    ct.inv_leaf[a] = 1.0f / n->resolution;
    ct.leaf[a] = n->resolution;
    ct.min_b[a] = n->min_b[a];
    ct.max_b[a] = n->max_b[a];
  }
  ct.mul[0] = 1;
  ct.mul[1] = n->div_b[0];
  ct.mul[2] = n->div_b[0] * n->div_b[1];
  return ct;
}

int eval_grid(int64_t n) { return std::max(1, std::min(grid_for(n, kEvalBlock), kNumSMs * 4)); }

// second half of the target build: from per-voxel sums (ascending voxel index) to records, export arrays and cell table
int finish_grid(lgs_ndt* n, int V, uint64_t total_cells, const unsigned* keys, const int* seg_start, int64_t n_entries, const double* sums,
                const int* counts) {
  lgs_ctx* ctx = n->ctx;
  cudaStream_t st = ctx->stream;
  n->n_voxels = V;
  n->dense = total_cells <= kDenseCellLimit ? 1 : 0;
  LGS_TRY(n->recs.reserve(static_cast<size_t>(V) * sizeof(VoxelRec)));
  LGS_TRY(n->ex_idx.reserve(static_cast<size_t>(V) * 4));
  LGS_TRY(n->ex_n.reserve(static_cast<size_t>(V) * 4));
  LGS_TRY(n->ex_mean.reserve(static_cast<size_t>(V) * 24));
  LGS_TRY(n->ex_cov.reserve(static_cast<size_t>(V) * 72));
  LGS_TRY(n->ex_icov.reserve(static_cast<size_t>(V) * 72));
  LGS_TRY(n->small.reserve(64));
  LGS_CUDA(cudaMemsetAsync(n->small.p, 0, 64, st));
  if (n->dense) {
    LGS_TRY(n->table.reserve(total_cells * 4));
    LGS_CUDA(cudaMemsetAsync(n->table.p, 0xFF, total_cells * 4, st));
    n->hmask = 0;
  } else {
    uint64_t cap = 1024;
    while (cap < static_cast<uint64_t>(V) * 2) cap <<= 1;
    n->hmask = static_cast<unsigned>(cap - 1);
    LGS_TRY(n->table.reserve(cap * 4));
    LGS_TRY(n->hkeys.reserve(cap * 4));
    LGS_CUDA(cudaMemsetAsync(n->hkeys.p, 0xFF, cap * 4, st));
  }
  VoxelExport ex{n->ex_idx.as<int>(), n->ex_n.as<int>(), n->ex_mean.as<double>(), n->ex_cov.as<double>(), n->ex_icov.as<double>()};
  voxel_stats_kernel<<<grid_for(V, 128), 128, 0, st>>>(sums, keys, seg_start, counts, V, n_entries, 6, 0.01, ex, n->recs.as<VoxelRec>(),
                                                      n->dense ? n->table.as<int>() : nullptr, n->hkeys.as<int>(), n->table.as<int>(), n->hmask,
                                                      n->small.as<int>());
  ctx->launches++;
  LGS_CUDA(cudaGetLastError());
  LGS_TRY(ctx->pin.reserve(256));
  int* h = ctx->pin.as<int>();
  LGS_CUDA(cudaMemcpyAsync(h, n->small.p, 4, cudaMemcpyDeviceToHost, st));
  LGS_CUDA(cudaStreamSynchronize(st));
  n->n_valid = h[0];
  n->grid_ready = true;
  return LGS_OK;
}

// init() (NDT.h:276-283): (re)voxelise the target at the current resolution
int build_grid_from_frames(lgs_ndt* n);
int build_grid(lgs_ndt* n) {
  if (n->target_from_frames) return build_grid_from_frames(n);
  lgs_ctx* ctx = n->ctx;
  cudaStream_t st = ctx->stream;
  n->grid_ready = false;
  n->refused = false;
  n->n_voxels = n->n_valid = 0;
  if (!n->have_target) return LGS_OK;
  const float leaf[3] = {n->resolution, n->resolution, n->resolution};
  SortedVoxels sv;
  LGS_TRY(build_sorted_voxels(ctx, n->target.as<float4>(), n->n_target, leaf, -1.0, nullptr, nullptr, nullptr, &sv));
  if (n->n_target == 0 || sv.n_kept == 0 || sv.status == LGS_VG_REFUSED_OVERFLOW) {  // VGC:79-84: grid cleared, every lookup misses (also: no finite point)
    n->refused = true;
    n->grid_ready = true;
    return LGS_OK;
  }
  for (int a = 0; a < 3; a++) {
    n->min_b[a] = sv.min_b[a];
    n->max_b[a] = sv.max_b[a];
    n->div_b[a] = sv.div_b[a];
  }
  const int V = sv.n_seg;
  LGS_TRY(n->vsums.reserve(static_cast<size_t>(V) * kSumsPerVoxel * sizeof(double)));
  voxel_sums_kernel<<<grid_for(static_cast<int64_t>(V) * 32, 256), 256, 0, st>>>(n->target.as<float4>(), sv.vals, sv.seg_start, V, sv.n_kept, n->vsums.as<double>());
  ctx->launches++;
  return finish_grid(n, V, sv.total_cells, sv.keys, sv.seg_start, sv.n_kept, n->vsums.as<double>(), nullptr);
}

// ---- rolling map ---------------------------------------------------------------------------------------------------
static int bits_for_cells(uint64_t max_value) {
  int b = 1;
  while (b < 32 && (max_value >> b) != 0) b++;
  return b;
}

// voxel partial sums of ONE key frame (transformed by its pose) in the frame's own grid
int voxelise_frame(lgs_ndt* n, const lgs_keyframes* kf, int32_t id, lgs_ndt::FrameVox* f) {
  lgs_ctx* ctx = n->ctx;
  cudaStream_t st = ctx->stream;
  f->id = id;
  memcpy(f->pose, keyframes_pose(kf, id), sizeof(f->pose));
  f->res = n->resolution;
  f->n_points = keyframes_points(kf, id);
  f->n_vox = 0;
  int64_t n_out = 0;
  LGS_TRY(keyframes_assemble_into(kf, ctx, &id, 1, &n->roll_poses, &n->roll_frame, &n_out));
  if (n_out == 0) return LGS_OK;
  const float leaf[3] = {n->resolution, n->resolution, n->resolution};
  SortedVoxels sv;
  LGS_TRY(build_sorted_voxels(ctx, n->roll_frame.as<float4>(), n_out, leaf, -1.0, nullptr, nullptr, nullptr, &sv));
  if (sv.status == LGS_VG_REFUSED_OVERFLOW) {
    set_error("key frame %d alone exceeds the voxel index range at resolution %g", id, n->resolution);
    return LGS_ERR_INVALID;
  }
  if (sv.n_kept == 0) return LGS_OK;
  const int V = sv.n_seg;
  for (int a = 0; a < 3; a++) {
    f->min_b[a] = sv.min_b[a];
    f->max_b[a] = sv.max_b[a];
    f->div_b[a] = sv.div_b[a];
  }
  LGS_TRY(f->keys.reserve(static_cast<size_t>(V) * 4));
  LGS_TRY(f->cnt.reserve(static_cast<size_t>(V) * 4));
  LGS_TRY(f->sums.reserve(static_cast<size_t>(V) * kSumsPerVoxel * sizeof(double)));
  voxel_sums_kernel<<<grid_for(static_cast<int64_t>(V) * 32, 256), 256, 0, st>>>(n->roll_frame.as<float4>(), sv.vals, sv.seg_start, V, sv.n_kept, f->sums.as<double>());
  frame_pack_kernel<<<grid_for(V, 256), 256, 0, st>>>(sv.keys, sv.seg_start, V, sv.n_kept, f->keys.as<unsigned>(), f->cnt.as<int>());
  ctx->launches += 2;
  LGS_CUDA(cudaGetLastError());
  f->n_vox = V;
  return LGS_OK;
}

// (Re)builds the voxel structure from the key frames of n->roll_ids: cached partial sums for the frames seen before (same
// pose, same resolution), a fresh voxelisation for the others, then one merge.  Equals the full build on the concatenated
// cloud up to the f64 rounding of adding per-frame partial sums instead of one running sum (~1e-16 relative).
int build_grid_from_frames(lgs_ndt* n) {
  lgs_ctx* ctx = n->ctx;
  cudaStream_t st = ctx->stream;
  const lgs_keyframes* kf = n->roll_kf;
  n->grid_ready = false;
  n->refused = false;
  n->n_voxels = n->n_valid = 0;
  n->roll_epoch++;
  n->roll_frames_voxelised = 0;
  std::vector<lgs_ndt::FrameVox*> use;
  for (int32_t id : n->roll_ids) {
    lgs_ndt::FrameVox* f = nullptr;
    for (auto* c : n->frame_cache)
      if (c->id == id) f = c;
    const bool valid = f && f->res == n->resolution && f->n_points == keyframes_points(kf, id) && memcmp(f->pose, keyframes_pose(kf, id), sizeof(f->pose)) == 0;
    if (!valid) {
      if (!f) {
        f = new lgs_ndt::FrameVox;
        n->frame_cache.push_back(f);
      }
      LGS_TRY(voxelise_frame(n, kf, id, f));
      n->roll_frames_voxelised++;
    }
    f->last_used = n->roll_epoch;
    use.push_back(f);
  }
  // evict the frames that left the window
  for (size_t i = 0; i < n->frame_cache.size();) {
    if (n->frame_cache[i]->last_used != n->roll_epoch) {
      lgs_ndt::FrameVox* f = n->frame_cache[i];
      LGS_CUDA(cudaStreamSynchronize(st));
      f->keys.release();
      f->cnt.release();
      f->sums.release();
      delete f;
      n->frame_cache.erase(n->frame_cache.begin() + i);
    } else {
      i++;
    }
  }
  int64_t M = 0;
  bool any = false;
  int gmin[3] = {0, 0, 0}, gmax[3] = {0, 0, 0};
  for (auto* f : use) {
    if (f->n_vox == 0) continue;
    M += f->n_vox;
    for (int a = 0; a < 3; a++) {
      gmin[a] = any ? std::min(gmin[a], f->min_b[a]) : f->min_b[a];
      gmax[a] = any ? std::max(gmax[a], f->max_b[a]) : f->max_b[a];
    }
    any = true;
  }
  int64_t d[3];
  for (int a = 0; a < 3; a++) d[a] = static_cast<int64_t>(gmax[a]) - gmin[a] + 1;
  if (!any || d[0] * d[1] * d[2] > static_cast<int64_t>(std::numeric_limits<int32_t>::max()) || M >= (int64_t(1) << 31)) {  // VGC:79-84
    n->refused = true;
    n->grid_ready = true;
    return LGS_OK;
  }
  for (int a = 0; a < 3; a++) {
    n->min_b[a] = gmin[a];
    n->max_b[a] = gmax[a];
    n->div_b[a] = static_cast<int>(d[a]);
  }
  const uint64_t total_cells = static_cast<uint64_t>(d[0]) * d[1] * d[2];
  LGS_TRY(n->roll_gkeys.reserve(static_cast<size_t>(M) * 4));
  LGS_TRY(n->roll_gvals.reserve(static_cast<size_t>(M) * 4));
  LGS_TRY(n->roll_gkeys_alt.reserve(static_cast<size_t>(M) * 4));
  LGS_TRY(n->roll_gvals_alt.reserve(static_cast<size_t>(M) * 4));
  LGS_TRY(n->roll_ccnt.reserve(static_cast<size_t>(M) * 4));
  LGS_TRY(n->roll_csum.reserve(static_cast<size_t>(M) * kSumsPerVoxel * sizeof(double)));
  int64_t out0 = 0;
  for (size_t s0 = 0; s0 < use.size(); s0 += kMergeFrames) {
    MergeSegments S;
    S.count = 0;
    int acc = 0;
    for (size_t s = s0; s < std::min(use.size(), s0 + kMergeFrames); s++) {
      const lgs_ndt::FrameVox* f = use[s];
      if (f->n_vox == 0) continue;
      const int k = S.count++;
      S.keys[k] = f->keys.as<unsigned>();
      S.cnt[k] = f->cnt.as<int>();
      S.sums[k] = f->sums.as<double>();
      S.begin[k] = acc;
      acc += f->n_vox;
      for (int a = 0; a < 3; a++) S.fmin[k][a] = f->min_b[a] - gmin[a];
      S.fdx[k] = f->div_b[0];
      S.fdxy[k] = f->div_b[0] * f->div_b[1];
    }
    S.begin[S.count] = acc;
    S.gmul[0] = 1;
    S.gmul[1] = static_cast<int>(d[0]);
    S.gmul[2] = static_cast<int>(d[0] * d[1]);
    if (acc > 0) {
      frame_gather_kernel<<<std::max(1, std::min(grid_for(acc, 256), kNumSMs * 8)), 256, 0, st>>>(S, static_cast<int>(out0), n->roll_gkeys.as<unsigned>(),
                                                                                              n->roll_gvals.as<unsigned>(), n->roll_ccnt.as<int>(),
                                                                                              n->roll_csum.as<double>());
      ctx->launches++;
    }
    out0 += acc;
  }
  LGS_CUDA(cudaGetLastError());
  unsigned *skeys, *svals;
  LGS_TRY(radix_sort_pairs(ctx, n->roll_gkeys.as<unsigned>(), n->roll_gvals.as<unsigned>(), n->roll_gkeys_alt.as<unsigned>(), n->roll_gvals_alt.as<unsigned>(), M,
                           bits_for_cells(total_cells), &skeys, &svals));
  LGS_TRY(n->roll_seg.reserve(static_cast<size_t>(M) * 4 + 64));
  LGS_TRY(n->roll_small.reserve(64));
  Mailbox mb;
  LGS_TRY(mailbox_next(ctx, &mb));
  LGS_TRY(scan_select(ctx, MergeHeads{skeys, n->roll_seg.as<int>()}, M, n->roll_small.as<int>(), &mb));
  double nseg = 0;
  LGS_TRY(mailbox_wait(ctx, mb, 1, &nseg));
  const int V = static_cast<int>(nseg);
  LGS_TRY(n->roll_msum.reserve(static_cast<size_t>(V) * kSumsPerVoxel * sizeof(double)));
  LGS_TRY(n->roll_mcnt.reserve(static_cast<size_t>(V) * 4));
  frame_merge_kernel<<<grid_for(static_cast<int64_t>(V) * (kSumsPerVoxel + 1), 256), 256, 0, st>>>(svals, n->roll_seg.as<int>(), V, static_cast<int>(M), n->roll_ccnt.as<int>(),
                                                                                                 n->roll_csum.as<double>(), n->roll_msum.as<double>(),
                                                                                                 n->roll_mcnt.as<int>());
  ctx->launches++;
  return finish_grid(n, V, total_cells, skeys, n->roll_seg.as<int>(), M, n->roll_msum.as<double>(), n->roll_mcnt.as<int>());
}

// getFitnessScore needs the target as a cloud: assembled from the key frames on first use
int ensure_target_cloud(lgs_ndt* n) {
  if (!n->target_from_frames || !n->target_cloud_stale) return LGS_OK;
  int64_t total = 0;
  LGS_TRY(keyframes_assemble_into(n->roll_kf, n->ctx, n->roll_ids.data(), static_cast<int32_t>(n->roll_ids.size()), &n->roll_poses, &n->target, &total));
  n->n_target = total;
  n->target_cloud_stale = false;
  n->nn_ready = false;
  return LGS_OK;
}

// one-time (per device) opt-in for > 48 KB of dynamic shared memory + the co-residency check of the align grid
struct DeviceCaps {
  bool ready = false;
  int num_sms = 0;
  int align_ctas_per_sm[2] = {0, 0};  // ndt_align_kernel<D7 = false / true>
  int group_ctas_per_sm[2] = {0, 0};  // ndt_align_group_kernel<D7 = false / true>
};
int device_caps(lgs_ctx* ctx, const DeviceCaps** out) {
  static DeviceCaps caps[64];
  DeviceCaps& c = caps[ctx->device & 63];
  if (!c.ready) {
    const int smem = static_cast<int>(sizeof(DerivSmem));
    LGS_CUDA(cudaFuncSetAttribute(ndt_derivatives_kernel<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    LGS_CUDA(cudaFuncSetAttribute(ndt_derivatives_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    LGS_CUDA(cudaFuncSetAttribute(ndt_derivatives_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    LGS_CUDA(cudaFuncSetAttribute(ndt_derivatives_kernel<0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    LGS_CUDA(cudaFuncSetAttribute(ndt_derivatives_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    LGS_CUDA(cudaFuncSetAttribute(ndt_derivatives_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    LGS_CUDA(cudaFuncSetAttribute(ndt_align_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    LGS_CUDA(cudaFuncSetAttribute(ndt_align_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    LGS_CUDA(cudaFuncSetAttribute(ndt_align_group_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    LGS_CUDA(cudaFuncSetAttribute(ndt_align_group_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    LGS_CUDA(cudaDeviceGetAttribute(&c.num_sms, cudaDevAttrMultiProcessorCount, ctx->device));
    int coop = 0;
    LGS_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, ctx->device));
    if (coop) {
      LGS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&c.align_ctas_per_sm[0], ndt_align_kernel<false>, kDerivThreads, sizeof(DerivSmem)));
      LGS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&c.align_ctas_per_sm[1], ndt_align_kernel<true>, kDerivThreads, sizeof(DerivSmem)));
      LGS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&c.group_ctas_per_sm[0], ndt_align_group_kernel<false>, kDerivThreads, sizeof(DerivSmem)));
      LGS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&c.group_ctas_per_sm[1], ndt_align_group_kernel<true>, kDerivThreads, sizeof(DerivSmem)));
    }
    c.ready = true;
  }
  *out = &c;
  return LGS_OK;
}

bool device_align_env_enabled() {  // LGS_NDT_DEVICE_ALIGN=0: the host steps the optimiser, one launch per evaluation
  static const bool on = [] {
    const char* e = getenv("LGS_NDT_DEVICE_ALIGN");
    return !(e && e[0] == '0');
  }();
  return on;
}

void fill_eval_constants(lgs_ndt* n) {
  EvalParams& P = n->P;
  P.gauss_d1 = n->gauss_d1;
  P.gauss_d2 = n->gauss_d2;
  P.gauss_d2f = static_cast<float>(n->gauss_d2);
  fill_offsets(n->search, &P);
}

int ensure_reduction_buffers(lgs_ndt* n, int grid) {
  cudaStream_t st = n->ctx->stream;
  LGS_TRY(n->partials.reserve(static_cast<size_t>(std::max(grid, kNumSMs)) * (kRow + 8) * sizeof(double)));  // rows + LGS_DERIV_TRACE words
  if (!n->result.p) {
    LGS_TRY(n->result.reserve(kNumAcc * sizeof(double) + 64));
    LGS_CUDA(cudaMemsetAsync(n->result.p, 0, kNumAcc * sizeof(double) + 64, st));
  }
  return LGS_OK;
}

// one computeDerivatives / computeHessian evaluation as one kernel launch, with the transform and the angular tables
// already in n->P.  mode 0: score+g+H (f32 terms), 1: score+g, 2: f64 Hessian.  sums[kRow]: the kernel's packed result (44 / 8 /
// 22 doubles, zeros when there is nothing to evaluate).
int evaluate_launch(lgs_ndt* n, int mode, double* sums) {
  lgs_ctx* ctx = n->ctx;
  cudaStream_t st = ctx->stream;
  fill_eval_constants(n);
  const int K = mode == 0 ? kSumsHess : (mode == 1 ? kSumsGrad : kSumsF64);
  std::fill(sums, sums + kRow, 0.0);
  if (mode == 2) n->hess_recomputes++; else n->evals++;
  if (n->n_source == 0 || n->refused || n->n_valid == 0) return LGS_OK;
  const DeviceCaps* caps = nullptr;
  LGS_TRY(device_caps(ctx, &caps));
  const int ns = static_cast<int>(n->n_source);
  // one CTA per SM (fewer when the cloud has fewer rounds of 32 points than SMs)
  const int dgrid = std::max(1, std::min(kNumSMs, (ns + 31) / 32));
  LGS_TRY(ensure_reduction_buffers(n, dgrid));
  double* result = n->result.as<double>();
  unsigned* counter = reinterpret_cast<unsigned*>(result + kNumAcc);
  const CellTable ct = make_cell_table(n);
  const float4* src = n->source.as<float4>();
  const EvalParams& P = n->P;
  Mailbox mb;
  LGS_TRY(mailbox_next(ctx, &mb));
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  if (n->profiling == 1) {
    LGS_CUDA(cudaEventCreate(&ev0));
    LGS_CUDA(cudaEventCreate(&ev1));
    LGS_CUDA(cudaEventRecord(ev0, st));
  }
  {
    const u64 one2 = 0x3f8000003f800000ull;  // (1.0f, 1.0f): see ndt_deriv.cuh
    const bool d7 = n->search == LGS_NDT_DIRECT7;
    VoxelRec* rc = n->recs.as<VoxelRec>();
    const double *vm = n->ex_mean.as<double>(), *vc = n->ex_icov.as<double>();
    double* pt = n->partials.as<double>();
#define LGS_LAUNCH(M, D) ndt_derivatives_kernel<M, D><<<dgrid, kDerivThreads, sizeof(DerivSmem), st>>>(src, ns, P, ct, rc, vm, vc, pt, result, counter, one2, mb)
    if (mode == 0 && d7) LGS_LAUNCH(0, true);
    else if (mode == 0) LGS_LAUNCH(0, false);
    else if (mode == 1 && d7) LGS_LAUNCH(1, true);
    else if (mode == 1) LGS_LAUNCH(1, false);
    else if (d7) LGS_LAUNCH(2, true);
    else LGS_LAUNCH(2, false);
#undef LGS_LAUNCH
  }
  if (n->profiling == 1) {
    LGS_CUDA(cudaEventRecord(ev1, st));
    n->prof_events[mode].emplace_back(ev0, ev1);
  }
  ctx->launches++;
  LGS_CUDA(cudaGetLastError());
  // the last CTA publishes the K sums to the host mailbox; no D2H copy, no stream synchronisation
  LGS_TRY(mailbox_wait(ctx, mb, K, sums));
  n->last_terms = sums[K - 1];
  return LGS_OK;
}

// the parity-hook form: transform T, tables of pose p
int evaluate(lgs_ndt* n, const float* T, const double p[6], int mode, double* score, double* g, double* H) {
  memcpy(n->P.T, T, sizeof(float) * 16);
  if (p) angle_derivatives(p, &n->P);
  double sums[kRow];
  LGS_TRY(evaluate_launch(n, mode, sums));
  if (mode == 2) {
    for (int i = 0; i < 6; i++)
      for (int j = i; j < 6; j++) H[i * 6 + j] = H[j * 6 + i] = sums[tri(i, j)];
    return LGS_OK;
  }
  if (score) *score = sums[0];
  if (g) memcpy(g, sums + 1, 6 * sizeof(double));
  if (H) {
    std::fill(H, H + 36, 0.0);
    if (mode == 0)  // all 36 entries, as the reference forms them (its two triangles differ in f32 rounding)
      for (int i = 0; i < 6; i++)
        for (int j = 0; j < 6; j++) H[i * 6 + j] = sums[hidx(i, j)];
  }
  return LGS_OK;
}

void command_to_params(const ndtopt::Command& c, EvalParams* P) {
  memcpy(P->T, c.T, sizeof(P->T));
  memcpy(P->j_ang, c.j_ang, sizeof(P->j_ang));
  memcpy(P->h_ang, c.h_ang, sizeof(P->h_ang));
  memcpy(P->j_ang_d, c.j_ang_d, sizeof(P->j_ang_d));
  memcpy(P->h_ang_d, c.h_ang_d, sizeof(P->h_ang_d));
}

struct AlignOutcome {
  float T[16];
  int iterations, converged, evals, trials, hess;
  double trans_probability;
};

// the optimiser stepped by the host: one kernel launch per evaluation (small or empty inputs, profiling of the
// per-evaluation kernels, LGS_NDT_DEVICE_ALIGN=0)
// parity mode: the reference's JacobiSVD for every Newton step (setter, or LGS_NDT_EXACT_SOLVE=1 read at every align)
bool exact_solve_requested(const lgs_ndt* n) {
  const char* e = getenv("LGS_NDT_EXACT_SOLVE");
  return n->exact_newton_step || (e && e[0] && e[0] != '0');
}

int align_host_stepped(lgs_ndt* n, const double p0[6], const float T0[16], AlignOutcome* out) {
  ndtopt::Machine m;
  ndtopt::Command c;
  m.begin(p0, T0, n->step_size, n->trans_eps, n->max_iter, static_cast<double>(n->n_source), &c, exact_solve_requested(n) ? 1 : 0);
  n->evals = n->hess_recomputes = 0;
  while (true) {
    command_to_params(c, &n->P);
    double sums[kRow];
    LGS_TRY(evaluate_launch(n, c.mode, sums));
    static const bool eval_trace = getenv("LGS_NDT_EVAL_TRACE") != nullptr;  // tests/diag_ndt_eval_diff.py
    if (eval_trace) {
      fprintf(stderr, "EV mode %d P", c.mode);
      for (int i = 0; i < 6; i++) fprintf(stderr, " %a", m.pending == 0 ? m.p[i] : m.x_t[i]);
      fprintf(stderr, " T");
      for (int i = 0; i < 12; i++) fprintf(stderr, " %a", static_cast<double>(n->P.T[i]));
      fprintf(stderr, " | S");
      for (int i = 0; i < (c.mode == 0 ? 43 : 28); i++) fprintf(stderr, " %a", sums[i]);  // score, g, upper triangle, strict lower triangle
      fprintf(stderr, "\n");
    }
    if (!m.advance(sums, &c)) break;
  }
  memcpy(out->T, m.final_T, sizeof(out->T));
  out->iterations = m.nr_iterations;
  out->converged = m.converged;
  out->evals = m.evals;
  out->trials = m.trials;
  out->hess = m.hess_recomputes;
  out->trans_probability = m.trans_probability;
  return LGS_OK;
}

// Evaluating CTAs of a device-resident align of n (one per round of 32 points at most, one CTA per SM, the optimiser's SM
// excluded).  G also fixes which points each CTA adds and in what order the rows are summed: every launch form of the align
// must use this G to produce the same bits.
int align_eval_ctas(const lgs_ndt* n, const DeviceCaps* caps) {
  return std::max(1, std::min(std::min(kNumSMs, caps->num_sms) - 1, static_cast<int>((n->n_source + 31) / 32)));
}

// The inputs of a device-resident align of n from guess T0 (pose p0): the first command in n->P (NDT:119: the guess and the
// tables of its pose; the machine on the device builds the same one) and the machine's arguments.
void align_launch_inputs(lgs_ndt* n, const double p0[6], const float T0[16], NdtAlignArgs* args) {
  fill_eval_constants(n);
  memcpy(n->P.T, T0, sizeof(float) * 16);
  angle_derivatives(p0, &n->P);
  memcpy(args->p0, p0, sizeof(args->p0));
  memcpy(args->T0, T0, sizeof(args->T0));
  args->step_size = n->step_size;
  args->trans_eps = n->trans_eps;
  args->n_in = static_cast<double>(n->n_source);
  args->max_iter = n->max_iter;
  args->exact_solve = exact_solve_requested(n) ? 1 : 0;
}

// the whole align as one cooperative launch of ndt_align_kernel; *used = false when the device cannot hold the grid
int align_on_device(lgs_ndt* n, const double p0[6], const float T0[16], AlignOutcome* out, bool* used) {
  *used = false;
  lgs_ctx* ctx = n->ctx;
  cudaStream_t st = ctx->stream;
  const DeviceCaps* caps = nullptr;
  LGS_TRY(device_caps(ctx, &caps));
  const bool d7 = n->search == LGS_NDT_DIRECT7;
  const int ns = static_cast<int>(n->n_source);
  const int grid = align_eval_ctas(n, caps) + 1;  // + the optimiser CTA
  if (caps->num_sms < 2 || caps->align_ctas_per_sm[d7 ? 1 : 0] * caps->num_sms < grid) return LGS_OK;  // the grid must be co-resident
  LGS_TRY(ensure_reduction_buffers(n, grid));
  if (!n->align_dev.p) LGS_TRY(n->align_dev.reserve(sizeof(NdtAlignDev)));
  NdtAlignArgs args;
  align_launch_inputs(n, p0, T0, &args);
  Mailbox mb;
  LGS_TRY(mailbox_next(ctx, &mb));
  LGS_CUDA(cudaMemsetAsync(n->align_dev.p, 0, 48, st));  // seq, the arrival counter, the trace words
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  if (n->profiling == 2) {
    LGS_CUDA(cudaEventCreate(&ev0));
    LGS_CUDA(cudaEventCreate(&ev1));
    LGS_CUDA(cudaEventRecord(ev0, st));
  }
  const float4* src = n->source.as<float4>();
  CellTable ct = make_cell_table(n);
  const VoxelRec* rc = n->recs.as<VoxelRec>();
  const double *vm = n->ex_mean.as<double>(), *vc = n->ex_icov.as<double>();
  double* pt = n->partials.as<double>();
  NdtAlignDev* dev = n->align_dev.as<NdtAlignDev>();
  u64 one2 = 0x3f8000003f800000ull;
  int ns_arg = ns;
  void* kargs[] = {&src, &ns_arg, &n->P, &ct, &rc, &vm, &vc, &pt, &dev, &args, &one2, &mb};
  const void* fn = d7 ? reinterpret_cast<const void*>(ndt_align_kernel<true>) : reinterpret_cast<const void*>(ndt_align_kernel<false>);
  cudaError_t le = cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(kDerivThreads), kargs, sizeof(DerivSmem), st);
  if (le != cudaSuccess) {
    set_error("ndt_align_kernel cooperative launch failed: %s", cudaGetErrorString(le));
    return LGS_ERR_CUDA;
  }
  if (n->profiling == 2) {
    LGS_CUDA(cudaEventRecord(ev1, st));
    n->prof_events[3].emplace_back(ev0, ev1);
  }
  ctx->launches++;
  n->align_launches = 1;
  double h[kMailboxRecords];
  LGS_TRY(mailbox_wait(ctx, mb, kAlignResultRecords, h));
  for (int i = 0; i < 16; i++) out->T[i] = static_cast<float>(h[i]);
  out->trans_probability = h[23];
  out->iterations = static_cast<int>(h[24]);
  out->converged = static_cast<int>(h[25]);
  out->evals = static_cast<int>(h[26]);
  out->trials = static_cast<int>(h[27]);
  out->hess = static_cast<int>(h[28]);
  n->last_terms = h[29];
  n->terms_total = h[30];
  for (int i = 0; i < 16; i++) n->align_trace[i] = h[32 + i];
  if (n->profiling == 2) {
    n->prof_align_evals += h[26] + h[28];
    n->prof_align_terms += h[30];
  }
  *used = true;
  return LGS_OK;
}

// getFitnessScore(max_range) of n's source under T (the 1-NN structure over the target is built on first use)
int fitness_at(lgs_ndt* n, const float* T, double max_range, double* fitness) {
  LGS_TRY(ensure_target_cloud(n));
  if (!n->nn_ready) {
    LGS_TRY(n->nn.build(n->ctx, n->target.as<float4>(), n->n_target));
    n->nn_ready = true;
  }
  return nn_fitness(n->ctx, n->nn, n->source.as<float4>(), n->n_source, T, max_range, fitness);
}

// ---- several aligns in one launch (lgs_ndt_align_many) --------------------------------------------------------------
// Groups per ndt_align_group_kernel launch (a wave), unless LGS_NDT_MANY_MAX_GROUPS says otherwise (read on every call).
// 1: measured on a B200 (DESIGN section 7), every grouping of 2 to 16 problems was slower than the same aligns one after
// another - a group's aligns end at different evaluation counts, and the SMs of the groups that finish first idle.
constexpr int kManyDefaultGroups = 1;
int many_max_groups() {
  const char* e = getenv("LGS_NDT_MANY_MAX_GROUPS");
  const int v = e && e[0] ? atoi(e) : 0;
  return v > 0 ? v : kManyDefaultGroups;
}

struct ManyProblem {
  int i;  // index in the caller's list
  lgs_ndt* n;
  double p0[6];
  float T0[16];
  int G;  // evaluating CTAs of the same align alone (align_eval_ctas)
};

constexpr size_t kManyRowsPerGroup = static_cast<size_t>(kNumSMs) * (kRow + 8);  // doubles: G <= kNumSMs - 1 rows (+ trace words)
inline size_t round_up_256(size_t b) { return (b + 255) & ~size_t(255); }

// One cooperative launch of ndt_align_group_kernel<d7> for probs[0..k): group sizes roughly proportional to G with
// 1 <= g <= G and sum(g + 1) <= capacity; record r of problem j lands in out[j * kAlignResultRecords + r].
int run_many_wave(lgs_ctx* ctx, bool d7, int capacity, const ManyProblem* probs, int k, double* out) {
  cudaStream_t st = ctx->stream;
  if (k == 1) {  // a lone problem: lgs_ndt_align's own launch, without the descriptor and record copies
    lgs_ndt* n = probs[0].n;
    AlignOutcome o;
    bool used = false;
    LGS_TRY(align_on_device(n, probs[0].p0, probs[0].T0, &o, &used));
    LGS_REQUIRE(used, "the align grid does not fit the device");
    std::fill(out, out + kAlignResultRecords, 0.0);
    for (int r = 0; r < 16; r++) out[r] = static_cast<double>(o.T[r]);
    out[23] = o.trans_probability;
    out[24] = o.iterations;
    out[25] = o.converged;
    out[26] = o.evals;
    out[27] = o.trials;
    out[28] = o.hess;
    out[29] = n->last_terms;
    out[30] = n->terms_total;
    for (int r = 0; r < 16; r++) out[32 + r] = n->align_trace[r];
    return LGS_OK;
  }
  const size_t desc_b = round_up_256(sizeof(NdtGroupDesc) * k), dev_b = round_up_256(sizeof(NdtAlignDev) * k);
  const size_t rec_b = round_up_256(sizeof(double) * kAlignResultRecords * k), rows_b = sizeof(double) * kManyRowsPerGroup * k;
  // an earlier call may still have a copy out of the pinned staging blocks in flight on this stream (keyframes.cu does the same)
  LGS_CUDA(cudaStreamSynchronize(st));
  LGS_TRY(ctx->ndt_many.reserve(desc_b + dev_b + rec_b + rows_b));
  LGS_TRY(ctx->pin_up.reserve(sizeof(NdtGroupDesc) * k));
  LGS_TRY(ctx->pin.reserve(sizeof(double) * kAlignResultRecords * k));
  char* base = ctx->ndt_many.as<char>();
  NdtGroupDesc* descs = reinterpret_cast<NdtGroupDesc*>(base);
  NdtAlignDev* devs = reinterpret_cast<NdtAlignDev*>(base + desc_b);
  double* recs = reinterpret_cast<double*>(base + desc_b + dev_b);
  double* rows = reinterpret_cast<double*>(base + desc_b + dev_b + rec_b);
  int64_t sum_G = 0;
  for (int j = 0; j < k; j++) sum_G += probs[j].G;
  const int64_t spare = capacity - 2 * k;  // evaluating CTAs beyond the one every group has
  NdtGroupDesc* h = ctx->pin_up.as<NdtGroupDesc>();
  int cta = 0;
  for (int j = 0; j < k; j++) {
    lgs_ndt* n = probs[j].n;
    NdtGroupDesc& d = h[j];
    align_launch_inputs(n, probs[j].p0, probs[j].T0, &d.args);
    d.P0 = n->P;
    d.ct = make_cell_table(n);
    d.src = n->source.as<float4>();
    d.recs = n->recs.as<VoxelRec>();
    d.vmean = n->ex_mean.as<double>();
    d.vicov = n->ex_icov.as<double>();
    d.partials = rows + kManyRowsPerGroup * j;
    d.dev = devs + j;
    d.record = recs + static_cast<size_t>(kAlignResultRecords) * j;
    d.n = static_cast<int>(n->n_source);
    d.G = probs[j].G;
    d.g = static_cast<int>(std::min<int64_t>(probs[j].G, 1 + spare * probs[j].G / sum_G));
    d.cta0 = cta;
    cta += d.g + 1;
  }
  LGS_CUDA(cudaMemcpyAsync(descs, h, sizeof(NdtGroupDesc) * k, cudaMemcpyHostToDevice, st));
  LGS_CUDA(cudaMemsetAsync(devs, 0, sizeof(NdtAlignDev) * k, st));
  const NdtGroupDesc* descs_arg = descs;
  int k_arg = k;
  u64 one2 = 0x3f8000003f800000ull;  // (1.0f, 1.0f): see ndt_deriv.cuh
  void* kargs[] = {&descs_arg, &k_arg, &one2};
  const void* fn = d7 ? reinterpret_cast<const void*>(ndt_align_group_kernel<true>) : reinterpret_cast<const void*>(ndt_align_group_kernel<false>);
  cudaError_t le = cudaLaunchCooperativeKernel(fn, dim3(cta), dim3(kDerivThreads), kargs, sizeof(DerivSmem), st);
  if (le != cudaSuccess) {
    set_error("ndt_align_group_kernel cooperative launch failed: %s", cudaGetErrorString(le));
    return LGS_ERR_CUDA;
  }
  ctx->launches++;
  LGS_CUDA(cudaMemcpyAsync(ctx->pin.p, recs, sizeof(double) * kAlignResultRecords * k, cudaMemcpyDeviceToHost, st));
  LGS_CUDA(cudaStreamSynchronize(st));
  memcpy(out, ctx->pin.p, sizeof(double) * kAlignResultRecords * k);
  return LGS_OK;
}

}  // namespace

extern "C" {

int lgs_ndt_create(lgs_ctx* ctx, lgs_ndt** out) {
  LGS_REQUIRE(ctx && out, "null argument");
  lgs_ndt* n = new lgs_ndt;
  n->ctx = ctx;
  identity16f(n->final_T);
  memset(&n->P, 0, sizeof(n->P));
  compute_gauss(n);
  *out = n;
  return LGS_OK;
}

void lgs_ndt_destroy(lgs_ndt* n) {
  if (!n) return;
  cudaSetDevice(n->ctx->device);
  cudaStreamSynchronize(n->ctx->stream);
  n->align_dev.release();
  for (auto* f : n->frame_cache) {
    f->keys.release();
    f->cnt.release();
    f->sums.release();
    delete f;
  }
  for (DevBuf* b : {&n->roll_frame, &n->roll_gkeys, &n->roll_gvals, &n->roll_gkeys_alt, &n->roll_gvals_alt, &n->roll_ccnt, &n->roll_csum, &n->roll_msum,
                    &n->roll_mcnt, &n->roll_seg, &n->roll_small, &n->roll_poses})
    b->release();
  for (DevBuf* b : {&n->target, &n->source, &n->out_cloud, &n->table, &n->hkeys, &n->recs, &n->ex_idx, &n->ex_n, &n->ex_mean, &n->ex_cov, &n->ex_icov,
                    &n->small, &n->partials, &n->result, &n->vsums})
    b->release();
  n->nn.release();
  delete n;
}

int lgs_ndt_set_resolution(lgs_ndt* n, float r) {  // NDT.h:132-142: re-init only when the value changes and a source is set
  LGS_REQUIRE(n && r > 0, "bad argument");
  if (n->resolution != r) {
    n->resolution = r;
    n->grid_ready = false;
    if (n->have_source && n->have_target) {
      LGS_TRY(use_device(n->ctx));
      LGS_TRY(build_grid(n));
    }
  }
  return LGS_OK;
}
int lgs_ndt_set_step_size(lgs_ndt* n, double s) { LGS_REQUIRE(n, "null"); n->step_size = s; return LGS_OK; }
int lgs_ndt_set_exact_newton_step(lgs_ndt* n, int32_t on) { LGS_REQUIRE(n, "null"); n->exact_newton_step = on != 0; return LGS_OK; }
int lgs_ndt_set_transformation_epsilon(lgs_ndt* n, double e) { LGS_REQUIRE(n, "null"); n->trans_eps = e; return LGS_OK; }
int lgs_ndt_set_maximum_iterations(lgs_ndt* n, int32_t it) { LGS_REQUIRE(n, "null"); n->max_iter = it; return LGS_OK; }
int lgs_ndt_set_outlier_ratio(lgs_ndt* n, double o) { LGS_REQUIRE(n, "null"); n->outlier_ratio = o; return LGS_OK; }
int lgs_ndt_set_search_method(lgs_ndt* n, int32_t m) {
  LGS_REQUIRE(n, "null");
  LGS_REQUIRE(m == LGS_NDT_DIRECT1 || m == LGS_NDT_DIRECT7 || m == LGS_NDT_DIRECT26, "only DIRECT1/7/26 are supported (KDTREE radius search is not)");
  n->search = m;
  return LGS_OK;
}

static int after_target(lgs_ndt* n) {
  n->have_target = true;
  n->nn_ready = false;
  n->target_from_frames = false;
  return build_grid(n);
}

int lgs_ndt_set_target(lgs_ndt* n, const void* pts, int64_t cnt, int32_t stride) {
  LGS_NVTX("lgs_ndt_set_target");
  LGS_REQUIRE(n, "null");
  LGS_TRY(load_cloud(n->ctx, pts, cnt, stride, false, &n->target));
  n->n_target = cnt;
  return after_target(n);
}
int lgs_ndt_set_target_dev(lgs_ndt* n, const float* pts_dev, int64_t cnt) {
  LGS_NVTX("lgs_ndt_set_target_dev");
  LGS_REQUIRE(n, "null");
  LGS_TRY(load_cloud(n->ctx, pts_dev, cnt, 16, true, &n->target));
  n->n_target = cnt;
  return after_target(n);
}
int lgs_ndt_set_target_keyframes(lgs_ndt* n, lgs_keyframes* kf, const int32_t* ids, int32_t n_ids, int32_t* frames_voxelised) {
  LGS_NVTX("lgs_ndt_set_target_keyframes");
  LGS_REQUIRE(n && kf && (ids || n_ids == 0) && n_ids >= 0, "bad argument");
  LGS_REQUIRE(keyframes_device(kf) == n->ctx->device, "the key-frame array lives on another device");
  const int64_t count = keyframes_count(kf);
  for (int32_t i = 0; i < n_ids; i++) LGS_REQUIRE(ids[i] >= 0 && ids[i] < count, "key frame id out of range");
  LGS_TRY(use_device(n->ctx));
  LGS_TRY(keyframes_wait_resident(kf));
  if (n->roll_kf != kf) {  // another array: nothing cached applies
    for (auto* f : n->frame_cache) f->id = -1;
  }
  n->roll_kf = kf;
  n->roll_ids.assign(ids, ids + n_ids);
  n->target_from_frames = true;
  n->target_cloud_stale = true;
  n->have_target = true;
  n->nn_ready = false;
  const int rc = build_grid_from_frames(n);
  if (frames_voxelised) *frames_voxelised = n->roll_frames_voxelised;
  return rc;
}

int lgs_ndt_set_source(lgs_ndt* n, const void* pts, int64_t cnt, int32_t stride) {
  LGS_REQUIRE(n, "null");
  LGS_TRY(load_cloud(n->ctx, pts, cnt, stride, false, &n->source));
  n->n_source = cnt;
  n->have_source = true;
  return LGS_OK;
}
int lgs_ndt_set_source_dev(lgs_ndt* n, const float* pts_dev, int64_t cnt) {
  LGS_REQUIRE(n, "null");
  LGS_TRY(load_cloud(n->ctx, pts_dev, cnt, 16, true, &n->source));
  n->n_source = cnt;
  n->have_source = true;
  return LGS_OK;
}

// pcl::Registration::align shell + computeTransformation (NDT:80-171)
int lgs_ndt_align(lgs_ndt* n, const float* guess16, lgs_align_result* res, float* out_cloud) {
  LGS_NVTX("lgs_ndt_align");
  LGS_REQUIRE(n && res, "null argument");
  memset(res, 0, sizeof(*res));
  if (!n->have_target || !n->have_source) {
    set_error("lgs_ndt_align: setInputTarget and setInputSource must be called first");
    return LGS_ERR_STATE;
  }
  LGS_TRY(use_device(n->ctx));
  if (!n->grid_ready) LGS_TRY(build_grid(n));
  const auto t0 = std::chrono::steady_clock::now();
  n->evals = n->trials = n->hess_recomputes = 0;
  n->align_launches = 0;
  compute_gauss(n);
  float guess[16];
  identity16f(guess);
  if (guess16) memcpy(guess, guess16, sizeof(guess));  // NDT:95-101; the evaluation transforms by the guess on the fly
  double p0[6];
  matrix_to_pose(guess, p0);  // NDT:103-111
  AlignOutcome out;
  bool on_device = false;
  const bool nothing_to_evaluate = n->n_source == 0 || n->refused || n->n_valid == 0;
  if (!nothing_to_evaluate && n->profiling != 1 && device_align_env_enabled()) LGS_TRY(align_on_device(n, p0, guess, &out, &on_device));
  if (!on_device) LGS_TRY(align_host_stepped(n, p0, guess, &out));
  memcpy(n->final_T, out.T, sizeof(float) * 16);
  memcpy(res->T, out.T, sizeof(float) * 16);
  res->trans_probability = out.trans_probability;
  res->iterations = out.iterations;
  res->converged = out.converged;
  res->evaluations = out.evals;
  res->line_search_trials = out.trials;
  res->hessian_recomputes = out.hess;
  n->evals = out.evals;
  n->trials = out.trials;
  n->hess_recomputes = out.hess;
  if (getenv("LGS_NDT_TRACE"))
    fprintf(stderr, "[lgs ndt] align %.1f us (%s): %d evaluations (%d trials, %d f64 Hessians), %d iterations\n",
            std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t0).count(), on_device ? "one resident launch" : "host-stepped",
            res->evaluations, res->line_search_trials, res->hessian_recomputes, res->iterations);
  if (out_cloud) LGS_TRY(write_aligned_cloud(n->ctx, n->source.as<float4>(), n->n_source, n->final_T, &n->out_cloud, out_cloud));
  return LGS_OK;
}

int lgs_ndt_fitness(lgs_ndt* n, double max_range, double* fitness) {
  LGS_NVTX("lgs_ndt_fitness");
  LGS_REQUIRE(n && fitness, "null argument");
  if (!n->have_target || !n->have_source) {
    set_error("lgs_ndt_fitness: target and source must be set");
    return LGS_ERR_STATE;
  }
  LGS_TRY(use_device(n->ctx));
  return fitness_at(n, n->final_T, max_range, fitness);
}

// N aligns as if lgs_ndt_align(ndts[i], guess i, &records[i], out_clouds[i]) ran for i = 0 .. n - 1 in turn.  The problems a
// lone align would run in one ndt_align_kernel launch go to ndt_align_group_kernel launches (one per wave of at most
// many_max_groups() problems of one search-method class); every other problem runs through lgs_ndt_align itself.
int lgs_ndt_align_many(lgs_ndt* const* ndts, int32_t count, const float* guesses16, const double* fitness_max_range, lgs_align_result* records,
                       float* const* out_clouds) {
  LGS_NVTX("lgs_ndt_align_many");
  LGS_REQUIRE(count >= 0, "negative count");
  if (count == 0) return LGS_OK;
  LGS_REQUIRE(ndts && records, "null argument");
  for (int32_t i = 0; i < count; i++) LGS_REQUIRE(ndts[i], "null handle");
  lgs_ctx* ctx = ndts[0]->ctx;
  for (int32_t i = 0; i < count; i++) LGS_REQUIRE(ndts[i]->ctx == ctx, "all handles must belong to one context");
  for (int32_t i = 0; i < count; i++) {
    if (!ndts[i]->have_target || !ndts[i]->have_source) {
      set_error("lgs_ndt_align_many: handle %d: setInputTarget and setInputSource must be called first", i);
      return LGS_ERR_STATE;
    }
  }
  LGS_TRY(use_device(ctx));
  const DeviceCaps* caps = nullptr;
  LGS_TRY(device_caps(ctx, &caps));
  std::vector<lgs_ndt*> prepared;
  for (int32_t i = 0; i < count; i++) {
    lgs_ndt* n = ndts[i];
    if (std::find(prepared.begin(), prepared.end(), n) != prepared.end()) continue;
    prepared.push_back(n);
    if (!n->grid_ready) LGS_TRY(build_grid(n));
    compute_gauss(n);
  }
  // route: a problem joins a group launch exactly when lgs_ndt_align would run it as one ndt_align_kernel launch
  std::vector<ManyProblem> cls[2];  // DIRECT1 / DIRECT26, DIRECT7: D7 is a template parameter of the kernel
  std::vector<int> slot(count, -1);  // problem i's place in its class, -1: runs through lgs_ndt_align
  for (int32_t i = 0; i < count; i++) {
    lgs_ndt* n = ndts[i];
    const int c = n->search == LGS_NDT_DIRECT7 ? 1 : 0;
    const int G = align_eval_ctas(n, caps);
    const bool nothing_to_evaluate = n->n_source == 0 || n->refused || n->n_valid == 0;
    const bool fits = caps->num_sms >= 2 && caps->align_ctas_per_sm[c] * caps->num_sms >= G + 1 && caps->group_ctas_per_sm[c] * caps->num_sms >= 2;
    if (nothing_to_evaluate || n->profiling != 0 || !device_align_env_enabled() || !fits) continue;
    ManyProblem p;
    p.i = i;
    p.n = n;
    identity16f(p.T0);
    if (guesses16) memcpy(p.T0, guesses16 + 16 * static_cast<size_t>(i), sizeof(p.T0));
    matrix_to_pose(p.T0, p.p0);
    p.G = G;
    slot[i] = static_cast<int>(cls[c].size());
    cls[c].push_back(p);
  }
  std::vector<double> rec[2];
  for (int c = 0; c < 2; c++) {
    rec[c].resize(cls[c].size() * kAlignResultRecords);
    const int capacity = caps->group_ctas_per_sm[c] * caps->num_sms;
    const int M = std::max(1, std::min(many_max_groups(), capacity / 2));
    for (size_t w0 = 0; w0 < cls[c].size(); w0 += M) {
      const int k = static_cast<int>(std::min(cls[c].size() - w0, static_cast<size_t>(M)));
      LGS_TRY(run_many_wave(ctx, c == 1, capacity, cls[c].data() + w0, k, rec[c].data() + w0 * kAlignResultRecords));
    }
  }
  // publish in the caller's order: each handle ends in the state of its last occurrence
  for (int32_t i = 0; i < count; i++) {
    lgs_ndt* n = ndts[i];
    lgs_align_result* res = records + i;
    float* out_cloud = out_clouds ? out_clouds[i] : nullptr;
    if (slot[i] < 0) {
      float guess[16];
      identity16f(guess);
      if (guesses16) memcpy(guess, guesses16 + 16 * static_cast<size_t>(i), sizeof(guess));
      LGS_TRY(lgs_ndt_align(n, guess, res, out_cloud));
    } else {
      const double* h = rec[n->search == LGS_NDT_DIRECT7 ? 1 : 0].data() + static_cast<size_t>(slot[i]) * kAlignResultRecords;
      memset(res, 0, sizeof(*res));
      for (int k = 0; k < 16; k++) res->T[k] = n->final_T[k] = static_cast<float>(h[k]);
      res->trans_probability = h[23];
      res->iterations = static_cast<int>(h[24]);
      res->converged = static_cast<int>(h[25]);
      res->evaluations = n->evals = static_cast<int>(h[26]);
      res->line_search_trials = n->trials = static_cast<int>(h[27]);
      res->hessian_recomputes = n->hess_recomputes = static_cast<int>(h[28]);
      n->last_terms = h[29];
      n->terms_total = h[30];
      for (int k = 0; k < 16; k++) n->align_trace[k] = h[32 + k];
      n->align_launches = 1;
      if (out_cloud) LGS_TRY(write_aligned_cloud(ctx, n->source.as<float4>(), n->n_source, n->final_T, &n->out_cloud, out_cloud));
    }
    if (fitness_max_range) LGS_TRY(fitness_at(n, res->T, *fitness_max_range, &res->fitness));
    res->pair_id = i;
  }
  return LGS_OK;
}

int lgs_ndt_calculate_score(lgs_ndt* n, const float* T16, double* score) {
  LGS_REQUIRE(n && T16 && score, "null argument");
  LGS_TRY(use_device(n->ctx));
  if (!n->grid_ready) LGS_TRY(build_grid(n));
  compute_gauss(n);
  *score = 0;
  if (n->n_source == 0) return LGS_OK;
  lgs_ctx* ctx = n->ctx;
  cudaStream_t st = ctx->stream;
  EvalParams& P = n->P;
  memcpy(P.T, T16, sizeof(float) * 16);
  P.gauss_d1 = n->gauss_d1;
  P.gauss_d2 = n->gauss_d2;
  fill_offsets(n->search, &P);
  if (!(n->refused || n->n_valid == 0)) {
    const int grid = eval_grid(n->n_source);
    LGS_TRY(n->partials.reserve(static_cast<size_t>(grid) * kNumAcc * sizeof(double)));
    if (!n->result.p) {
      LGS_TRY(n->result.reserve(kNumAcc * sizeof(double) + 64));
      LGS_CUDA(cudaMemsetAsync(n->result.p, 0, kNumAcc * sizeof(double) + 64, st));
    }
    double* result = n->result.as<double>();
    unsigned* counter = reinterpret_cast<unsigned*>(result + kNumAcc);
    Mailbox mb;
    LGS_TRY(mailbox_next(ctx, &mb));
    ndt_score_kernel<<<grid, kEvalBlock, 0, st>>>(n->source.as<float4>(), static_cast<int>(n->n_source), P, make_cell_table(n),
                                                 n->ex_mean.as<double>(), n->ex_icov.as<double>(), n->gauss_d3, n->partials.as<double>(), result, counter, mb);
    ctx->launches++;
    LGS_CUDA(cudaGetLastError());
    LGS_TRY(mailbox_wait(ctx, mb, 1, score));
  }
  *score /= static_cast<double>(n->n_source);
  return LGS_OK;
}

int lgs_ndt_grid_info_get(lgs_ndt* n, lgs_ndt_grid_info* info) {
  LGS_REQUIRE(n && info, "null argument");
  memset(info, 0, sizeof(*info));
  if (n->have_target && !n->grid_ready) {
    LGS_TRY(use_device(n->ctx));
    LGS_TRY(build_grid(n));
  }
  info->refused = n->refused ? 1 : 0;
  info->dense = n->dense;
  info->n_voxels = n->n_voxels;
  info->n_valid = n->n_valid;
  for (int a = 0; a < 3; a++) {
    info->min_b[a] = n->min_b[a];
    info->max_b[a] = n->max_b[a];
    info->div_b[a] = n->div_b[a];
  }
  return LGS_OK;
}

int lgs_ndt_export_voxels(lgs_ndt* n, int32_t* idx, int32_t* nr_points, double* mean, double* cov, double* icov) {
  LGS_REQUIRE(n, "null argument");
  LGS_TRY(use_device(n->ctx));
  if (n->have_target && !n->grid_ready) LGS_TRY(build_grid(n));
  const size_t V = static_cast<size_t>(n->n_voxels);
  if (V == 0) return LGS_OK;
  cudaStream_t st = n->ctx->stream;
  if (idx) LGS_CUDA(cudaMemcpyAsync(idx, n->ex_idx.p, V * 4, cudaMemcpyDeviceToHost, st));
  if (nr_points) LGS_CUDA(cudaMemcpyAsync(nr_points, n->ex_n.p, V * 4, cudaMemcpyDeviceToHost, st));
  if (mean) LGS_CUDA(cudaMemcpyAsync(mean, n->ex_mean.p, V * 24, cudaMemcpyDeviceToHost, st));
  if (cov) LGS_CUDA(cudaMemcpyAsync(cov, n->ex_cov.p, V * 72, cudaMemcpyDeviceToHost, st));
  if (icov) LGS_CUDA(cudaMemcpyAsync(icov, n->ex_icov.p, V * 72, cudaMemcpyDeviceToHost, st));
  LGS_CUDA(cudaStreamSynchronize(st));
  return LGS_OK;
}

int lgs_ndt_profile(lgs_ndt* n, int32_t enable, double* out8) {
  LGS_REQUIRE(n, "null argument");
  LGS_REQUIRE(enable >= 0 && enable <= 2, "enable must be 0, 1 or 2");
  LGS_TRY(use_device(n->ctx));
  LGS_CUDA(cudaStreamSynchronize(n->ctx->stream));
  auto total_ms = [](std::vector<std::pair<cudaEvent_t, cudaEvent_t>>& v) {
    double ms = 0;
    for (auto& pr : v) {
      float t = 0;
      cudaEventElapsedTime(&t, pr.first, pr.second);
      ms += t;
    }
    return ms;
  };
  if (out8) {
    if (n->profiling == 2) {  // whole aligns: launches, ms, evaluations and accepted terms summed over them
      out8[0] = static_cast<double>(n->prof_events[3].size());
      out8[1] = total_ms(n->prof_events[3]);
      out8[2] = n->prof_align_evals;
      out8[3] = n->prof_align_terms;
      out8[4] = out8[5] = 0;
    } else {
      for (int m = 0; m < 3; m++) {
        out8[2 * m] = static_cast<double>(n->prof_events[m].size());
        out8[2 * m + 1] = total_ms(n->prof_events[m]);
      }
    }
    out8[6] = n->last_terms;
    out8[7] = static_cast<double>(n->n_source);
  }
  for (int m = 0; m < 4; m++) {
    for (auto& pr : n->prof_events[m]) {
      cudaEventDestroy(pr.first);
      cudaEventDestroy(pr.second);
    }
    n->prof_events[m].clear();
  }
  n->prof_align_evals = n->prof_align_terms = 0;
  n->profiling = enable;
  return LGS_OK;
}

int lgs_ndt_align_breakdown(lgs_ndt* n, double* out16) {
  LGS_REQUIRE(n && out16, "null argument");
  memcpy(out16, n->align_trace, sizeof(n->align_trace));
  return LGS_OK;
}

#ifdef LGS_DERIV_TRACE
// development aid: per-CTA phase stamps of the last derivative launch (see ndt_deriv.cuh), 8 doubles per CTA
int lgs_ndt_debug_trace(lgs_ndt* n, double* out, int32_t n_cta) {
  LGS_TRY(use_device(n->ctx));
  LGS_CUDA(cudaMemcpy(out, n->partials.as<double>() + static_cast<size_t>(n_cta) * kRow, sizeof(double) * 8 * n_cta, cudaMemcpyDeviceToHost));
  return LGS_OK;
}
#endif

// static convertTransform (NDT.h:214-238): Translation(x, y, z) * AngleAxis(roll, X) * AngleAxis(pitch, Y) * AngleAxis(yaw, Z)
// in f32, as the optimiser builds its poses.  Pure host arithmetic: needs no device.
int lgs_ndt_convert_transform(const double* x6, float* T16) {
  LGS_REQUIRE(x6 && T16, "null argument");
  pose_to_matrix(x6, T16);
  return LGS_OK;
}

int lgs_ndt_derivatives(lgs_ndt* n, const float* T16, const double* p6, int32_t mode, double* score, double* g6, double* H36) {
  LGS_REQUIRE(n && T16 && p6 && H36, "null argument");
  LGS_REQUIRE(mode >= 0 && mode <= 2, "mode must be 0, 1 or 2");
  if (!n->have_target || !n->have_source) {
    set_error("lgs_ndt_derivatives: target and source must be set");
    return LGS_ERR_STATE;
  }
  LGS_TRY(use_device(n->ctx));
  if (!n->grid_ready) LGS_TRY(build_grid(n));
  compute_gauss(n);
  double s = 0, g[6];
  LGS_TRY(evaluate(n, T16, p6, mode, &s, g, H36));
  if (score) *score = s;
  if (g6) memcpy(g6, g, sizeof(g));
  return LGS_OK;
}

}  // extern "C"
