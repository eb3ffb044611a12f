// Device-wide primitives of the voxelisation front half, written for this library (no CUB / Thrust); the radix
// kernels live in sort.cu, the templated scan in this header:
//
//   radix_sort_pairs   stable LSD radix sort of (u32 key, u32 value) pairs, 8-bit digits, one pass per digit over only
//                      the key bits the caller needs.  One histogram kernel reads the keys once for all passes; each
//                      pass is a single "onesweep" kernel: a tile of keys is ranked in shared memory, the tile's
//                      per-digit counts are chained to the previous tiles by decoupled look-back (one self-validating
//                      64-bit status word per (tile, digit): flag and count travel in the same store, so no fence),
//                      and the tile is scattered as runs of equal digits.  Traffic per pass: 8 B read + 8 B written
//                      per pair, the minimum for an out-of-place pass.
//   scan_select        single-pass flagged selection / exclusive scan over an index range with the same look-back
//                      chaining: a functor supplies flag(i) and receives emit(i, position, flagged).
//
// Stability matters beyond sorting: members of a voxel must stay in ascending point index because the reference
// accumulates them serially in that order (VGC:218-263) and the sums have to round identically.
// Tiles take their index from an atomic ticket, so a tile only ever waits on tiles that are already running.
#pragma once
#include "common.cuh"

namespace lgs {

typedef unsigned long long u64_t;

constexpr int kSortThreads = 256;
constexpr int kSortWarps = kSortThreads / 32;
constexpr int kRadix = 256;
constexpr u64_t kStatusValueMask = (u64_t(1) << 48) - 1;

// scratch layout of ctx->sort_tmp: [0, 64) tickets (u32 per pass / call) | [64, 64 + 4 * 256 * 8) digit histograms |
// status words after that
constexpr size_t kSortTicketBytes = 64;
constexpr size_t kSortHistBytes = 4 * kRadix * sizeof(u64_t);

__device__ __forceinline__ u64_t ld_status(const u64_t* p) {
  u64_t v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_status(u64_t* p, u64_t v) { asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory"); }

// exclusive scan of one value per thread over a 256-thread block; returns the exclusive prefix, *total gets the sum
template <typename T>
__device__ __forceinline__ T block_excl_scan(T v, T* warp_sums /* [kSortWarps + 1] shared */, T* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  T inc = v;
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    T o = __shfl_up_sync(0xffffffffu, inc, off);
    if (lane >= off) inc += o;
  }
  if (lane == 31) warp_sums[warp] = inc;
  __syncthreads();
  if (threadIdx.x == 0) {
    T s = 0;
#pragma unroll
    for (int w = 0; w < kSortWarps; w++) {
      T t = warp_sums[w];
      warp_sums[w] = s;
      s += t;
    }
    warp_sums[kSortWarps] = s;
  }
  __syncthreads();
  const T r = warp_sums[warp] + inc - v;
  if (total) *total = warp_sums[kSortWarps];
  __syncthreads();  // warp_sums may be reused by the caller
  return r;
}

// Single-pass scan + select over [0, n): pos(i) = number of flagged j < i.  F: bool flag(int64_t i) const;
// void emit(int64_t i, int64_t pos, bool flagged) const.  *total_out receives the number of flagged elements.
constexpr int kScanItems = 8;
constexpr int kScanTile = kSortThreads * kScanItems;

template <class F>
__global__ void __launch_bounds__(kSortThreads) scan_select_kernel(F f, int64_t n, u64_t* __restrict__ status, unsigned* __restrict__ ticket,
                                                                  int* __restrict__ total_out, const Mailbox mb) {
  __shared__ unsigned scan32[kSortWarps + 1];
  __shared__ unsigned tile_s;
  __shared__ u64_t excl_s;
  if (threadIdx.x == 0) tile_s = atomicAdd(ticket, 1u);
  __syncthreads();
  const unsigned tile = tile_s;
  const int64_t base = static_cast<int64_t>(tile) * kScanTile + static_cast<int64_t>(threadIdx.x) * kScanItems;  // blocked: thread owns a run
  bool fl[kScanItems];
  unsigned c = 0;
#pragma unroll
  for (int j = 0; j < kScanItems; j++) {
    fl[j] = base + j < n && f.flag(base + j);
    c += fl[j] ? 1u : 0u;
  }
  unsigned tile_n;
  const unsigned local = block_excl_scan<unsigned>(c, scan32, &tile_n);
  constexpr u64_t flag_agg = u64_t(1) << 56, flag_pre = u64_t(2) << 56;
  if (threadIdx.x == 0) {
    st_status(status + tile, (tile == 0 ? flag_pre : flag_agg) | tile_n);
    u64_t excl = 0;
    if (tile > 0) {
      long long t = static_cast<long long>(tile) - 1;
      while (true) {
        const u64_t s = ld_status(status + t);
        const u64_t fg = s & ~kStatusValueMask;
        if (fg == flag_pre) {
          excl += s & kStatusValueMask;
          break;
        }
        if (fg == flag_agg) {
          excl += s & kStatusValueMask;
          t--;
        }
      }
      st_status(status + tile, flag_pre | (excl + tile_n));
    }
    excl_s = excl;
    if (static_cast<int64_t>(tile + 1) * kScanTile >= n) {  // the last tile knows the total
      if (total_out) *total_out = static_cast<int>(excl + tile_n);
      if (mb.r) mailbox_publish_one(mb, 0, static_cast<double>(excl + tile_n));  // the host gets it without a copy + synchronise
    }
  }
  __syncthreads();
  int64_t pos = static_cast<int64_t>(excl_s) + local;
#pragma unroll
  for (int j = 0; j < kScanItems; j++) {
    if (base + j < n) {
      f.emit(base + j, pos, fl[j]);
      pos += fl[j] ? 1 : 0;
    }
  }
}

// host side (sort.cu) ------------------------------------------------------------------------------------------

// Sorts n pairs by the low `bits` bits of the key.  (keys, vals) hold the input; the sorted pairs end up in
// (*keys_out, *vals_out), which point at either the input or the alt buffers.  Stable.
int radix_sort_pairs(lgs_ctx* ctx, unsigned* keys, unsigned* vals, unsigned* keys_alt, unsigned* vals_alt, int64_t n, int bits,
                     unsigned** keys_out, unsigned** vals_out);

// Stable sort of n indices by a 64-bit key, over the low `bits` (<= 64) key bits: vals holds indices into keys64 and
// keys_lo[i] the low word of keys64[vals[i]].  Two radix_sort_pairs composed least-significant word first: (low word,
// index) over min(bits, 32) bits, then the high words gathered through that permutation and (high word, permutation)
// sorted over bits - 32 bits.  Stability of both keeps equal keys in their input order.  The sorted indices end up in
// *vals_out (vals or vals_alt); keys_lo and keys_alt are overwritten.
int radix_sort_indices64(lgs_ctx* ctx, const u64_t* keys64, unsigned* keys_lo, unsigned* vals, unsigned* keys_alt, unsigned* vals_alt, int64_t n,
                         int bits, unsigned** vals_out);

// reserves and zeroes the look-back scratch for one scan_select launch over n elements
int scan_select_prepare(lgs_ctx* ctx, int64_t n, u64_t** status, unsigned** ticket);

// mb (optional): a mailbox the total is published to as well; ask for it only with n > 0
template <class F>
int scan_select(lgs_ctx* ctx, const F& f, int64_t n, int* total_out_dev, const Mailbox* mb = nullptr) {
  if (n <= 0) {
    if (total_out_dev) LGS_CUDA(cudaMemsetAsync(total_out_dev, 0, sizeof(int), ctx->stream));
    return LGS_OK;
  }
  Mailbox none;
  none.r = nullptr;
  none.token = 0;
  u64_t* status;
  unsigned* ticket;
  LGS_TRY(scan_select_prepare(ctx, n, &status, &ticket));
  scan_select_kernel<F><<<grid_for(n, kScanTile), kSortThreads, 0, ctx->stream>>>(f, n, status, ticket, total_out_dev, mb ? *mb : none);
  ctx->launches++;
  LGS_CUDA(cudaGetLastError());
  return LGS_OK;
}

}  // namespace lgs
