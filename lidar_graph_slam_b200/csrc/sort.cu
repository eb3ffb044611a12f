// Radix-sort kernels and the host side of the sort / scan primitives (see sort.cuh).
#include "sort.cuh"

#include <algorithm>
#include <utility>

namespace lgs {

// digit histograms of every pass in one read of the keys: ghist[pass][digit]
__global__ void __launch_bounds__(kSortThreads) radix_hist_kernel(const unsigned* __restrict__ keys, int64_t n, int npass, u64_t* __restrict__ ghist) {
  __shared__ unsigned h[4 * kRadix];
  for (int i = threadIdx.x; i < 4 * kRadix; i += kSortThreads) h[i] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * kSortThreads;
  const int64_t n_up = (n + 31) & ~int64_t(31);  // whole warps iterate together (match_any needs every lane)
  for (int64_t i = blockIdx.x * static_cast<int64_t>(kSortThreads) + threadIdx.x; i < n_up; i += stride) {
    const bool valid = i < n;
    const unsigned key = valid ? __ldg(keys + i) : 0u;
    for (int p = 0; p < npass; p++) {
      // neighbouring points of a sweep fall into the same voxel: aggregate equal digits inside the warp first
      const unsigned d = valid ? ((key >> (8 * p)) & 255u) : (256u + lane);
      const unsigned peers = __match_any_sync(0xffffffffu, d);
      if (valid && lane == __ffs(peers) - 1) atomicAdd(&h[p * kRadix + d], static_cast<unsigned>(__popc(peers)));
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < npass * kRadix; i += kSortThreads)
    if (h[i]) atomicAdd(ghist + i, static_cast<u64_t>(h[i]));
}

// one radix pass.  ITEMS keys per thread, warp-striped inside the tile: element (warp, round j, lane) has tile offset
// warp * 32 * ITEMS + j * 32 + lane, so "warp order, then round order, then lane order" is ascending input order.
template <int ITEMS>
__global__ void __launch_bounds__(kSortThreads) radix_onesweep_kernel(const unsigned* __restrict__ kin, const unsigned* __restrict__ vin,
                                                                     unsigned* __restrict__ kout, unsigned* __restrict__ vout, int64_t n, int pass,
                                                                     const u64_t* __restrict__ ghist, u64_t* __restrict__ status,
                                                                     unsigned* __restrict__ tickets) {
  constexpr int TILE = kSortThreads * ITEMS;
  __shared__ unsigned warp_hist[kSortWarps][kRadix];
  __shared__ unsigned skeys[TILE], svals[TILE];
  __shared__ unsigned dstart[kRadix];       // first tile-local position of each digit
  __shared__ long long goff[kRadix];        // global position of tile-local position 0 of each digit, minus dstart
  __shared__ u64_t scan64[kSortWarps + 1];
  __shared__ unsigned scan32[kSortWarps + 1];
  __shared__ unsigned tile_s;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) tile_s = atomicAdd(tickets + pass, 1u);
  for (int i = threadIdx.x; i < kSortWarps * kRadix; i += kSortThreads) (&warp_hist[0][0])[i] = 0;
  __syncthreads();
  const unsigned tile = tile_s;
  const int64_t tile_base = static_cast<int64_t>(tile) * TILE;
  const int shift = 8 * pass;
  const u64_t flag_agg = static_cast<u64_t>(2 * pass + 1) << 56, flag_pre = static_cast<u64_t>(2 * pass + 2) << 56;

  unsigned key[ITEMS], val[ITEMS], rank[ITEMS];
  bool valid[ITEMS];
#pragma unroll
  for (int j = 0; j < ITEMS; j++) {
    const int64_t i = tile_base + warp * (32 * ITEMS) + j * 32 + lane;
    valid[j] = i < n;
    key[j] = valid[j] ? __ldg(kin + i) : 0xffffffffu;
    val[j] = valid[j] ? __ldg(vin + i) : 0u;
  }
  // stable rank of every key among the keys of its warp with the same digit
#pragma unroll
  for (int j = 0; j < ITEMS; j++) {
    const unsigned d = valid[j] ? ((key[j] >> shift) & 255u) : 256u;
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    const int leader = __ffs(peers) - 1;
    unsigned old = 0;
    if (lane == leader && valid[j]) {
      old = warp_hist[warp][d];
      warp_hist[warp][d] = old + __popc(peers);
    }
    old = __shfl_sync(0xffffffffu, old, leader);
    rank[j] = old + __popc(peers & ((1u << lane) - 1u));
    __syncwarp();
  }
  __syncthreads();
  // thread d owns digit d: exclusive offsets of the warps, the tile's count, and the look-back over earlier tiles
  const int d = threadIdx.x;
  unsigned cnt = 0;
#pragma unroll
  for (int w = 0; w < kSortWarps; w++) {
    const unsigned t = warp_hist[w][d];
    warp_hist[w][d] = cnt;
    cnt += t;
  }
  u64_t* my_status = status + static_cast<size_t>(tile) * kRadix + d;
  st_status(my_status, (tile == 0 ? flag_pre : flag_agg) | cnt);
  u64_t excl = 0;
  if (tile > 0) {
    long long t = static_cast<long long>(tile) - 1;
    while (true) {
      const u64_t s = ld_status(status + static_cast<size_t>(t) * kRadix + d);
      const u64_t f = s & ~kStatusValueMask;
      if (f == flag_pre) {
        excl += s & kStatusValueMask;
        break;
      }
      if (f == flag_agg) {
        excl += s & kStatusValueMask;
        t--;
      }
    }
    st_status(my_status, flag_pre | (excl + cnt));
  }
  const u64_t gbase = block_excl_scan<u64_t>(ghist[pass * kRadix + d], scan64, nullptr);
  unsigned tile_n;
  const unsigned ds = block_excl_scan<unsigned>(cnt, scan32, &tile_n);
  dstart[d] = ds;
  goff[d] = static_cast<long long>(gbase + excl) - static_cast<long long>(ds);
  __syncthreads();
  // reorder inside the tile, then write runs of equal digits
#pragma unroll
  for (int j = 0; j < ITEMS; j++) {
    if (valid[j]) {
      const unsigned dd = (key[j] >> shift) & 255u;
      const unsigned lp = dstart[dd] + warp_hist[warp][dd] + rank[j];
      skeys[lp] = key[j];
      svals[lp] = val[j];
    }
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < ITEMS; j++) {
    const unsigned i = j * kSortThreads + threadIdx.x;
    if (i < tile_n) {
      const unsigned k = skeys[i];
      const long long o = goff[(k >> shift) & 255u] + i;
      kout[o] = k;
      vout[o] = svals[i];
    }
  }
}

// look-back scratch: tickets | digit histograms | status words; zeroed once per sort / scan call
static int reserve_sort_tmp(lgs_ctx* ctx, size_t status_words, unsigned** tickets, u64_t** ghist, u64_t** status) {
  const size_t bytes = kSortTicketBytes + kSortHistBytes + status_words * sizeof(u64_t);
  LGS_TRY(ctx->sort_tmp.reserve(bytes));
  LGS_CUDA(cudaMemsetAsync(ctx->sort_tmp.p, 0, bytes, ctx->stream));
  char* base = ctx->sort_tmp.as<char>();
  *tickets = reinterpret_cast<unsigned*>(base);
  *ghist = reinterpret_cast<u64_t*>(base + kSortTicketBytes);
  *status = reinterpret_cast<u64_t*>(base + kSortTicketBytes + kSortHistBytes);
  return LGS_OK;
}

int radix_sort_pairs(lgs_ctx* ctx, unsigned* keys, unsigned* vals, unsigned* keys_alt, unsigned* vals_alt, int64_t n, int bits,
                     unsigned** keys_out, unsigned** vals_out) {
  *keys_out = keys;
  *vals_out = vals;
  if (n <= 1 || bits <= 0) return LGS_OK;
  LGS_REQUIRE(bits <= 32, "key bits out of range");
  cudaStream_t st = ctx->stream;
  const int npass = (bits + 7) / 8;
  // small inputs: smaller tiles so that the pass still spreads over the SMs
  const bool big = n >= (int64_t(1) << 20);
  const int tile = kSortThreads * (big ? 16 : 4);
  const int64_t ntiles = (n + tile - 1) / tile;
  unsigned* tickets;
  u64_t *ghist, *status;
  LGS_TRY(reserve_sort_tmp(ctx, static_cast<size_t>(ntiles) * kRadix, &tickets, &ghist, &status));
  radix_hist_kernel<<<std::min<int64_t>(grid_for(n, kSortThreads * 8), kNumSMs * 4), kSortThreads, 0, st>>>(keys, n, npass, ghist);
  ctx->launches++;
  unsigned *kin = keys, *vin = vals, *kout = keys_alt, *vout = vals_alt;
  for (int p = 0; p < npass; p++) {
    if (big)
      radix_onesweep_kernel<16><<<static_cast<unsigned>(ntiles), kSortThreads, 0, st>>>(kin, vin, kout, vout, n, p, ghist, status, tickets);
    else
      radix_onesweep_kernel<4><<<static_cast<unsigned>(ntiles), kSortThreads, 0, st>>>(kin, vin, kout, vout, n, p, ghist, status, tickets);
    ctx->launches++;
    std::swap(kin, kout);
    std::swap(vin, vout);
  }
  LGS_CUDA(cudaGetLastError());
  *keys_out = kin;
  *vals_out = vin;
  return LGS_OK;
}

// hi[j] = high word of the key of the index at position j (the second pass's keys)
__global__ void __launch_bounds__(256) key_high_gather_kernel(const unsigned* __restrict__ perm, const u64_t* __restrict__ keys64, int64_t n,
                                                             unsigned* __restrict__ hi) {
  const int64_t j = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (j < n) hi[j] = static_cast<unsigned>(keys64[perm[j]] >> 32);
}

int radix_sort_indices64(lgs_ctx* ctx, const u64_t* keys64, unsigned* keys_lo, unsigned* vals, unsigned* keys_alt, unsigned* vals_alt, int64_t n,
                         int bits, unsigned** vals_out) {
  LGS_REQUIRE(bits >= 0 && bits <= 64, "key bits out of range");
  unsigned *k1, *v1;
  LGS_TRY(radix_sort_pairs(ctx, keys_lo, vals, keys_alt, vals_alt, n, std::min(bits, 32), &k1, &v1));
  *vals_out = v1;
  if (bits <= 32 || n <= 1) return LGS_OK;
  // the low words are no longer needed: their buffer takes the gathered high words, the other pair is the alt side
  unsigned* k_other = k1 == keys_lo ? keys_alt : keys_lo;
  unsigned* v_other = v1 == vals ? vals_alt : vals;
  key_high_gather_kernel<<<grid_for(n, 256), 256, 0, ctx->stream>>>(v1, keys64, n, k1);
  ctx->launches++;
  LGS_CUDA(cudaGetLastError());
  unsigned* k2;
  return radix_sort_pairs(ctx, k1, v1, k_other, v_other, n, bits - 32, &k2, vals_out);
}

int scan_select_prepare(lgs_ctx* ctx, int64_t n, u64_t** status, unsigned** ticket) {
  u64_t* ghist;
  return reserve_sort_tmp(ctx, static_cast<size_t>((n + kScanTile - 1) / kScanTile), ticket, &ghist, status);
}

}  // namespace lgs

extern "C" int lgs_sort_pairs(lgs_ctx* ctx, uint32_t* keys, uint32_t* vals, int64_t n, int32_t bits) {
  LGS_REQUIRE(ctx && (n == 0 || (keys && vals)), "null argument");
  LGS_REQUIRE(n >= 0 && n < (int64_t(1) << 31) && bits >= 0 && bits <= 32, "argument out of range");
  LGS_TRY(lgs::use_device(ctx));
  if (n == 0) return LGS_OK;
  cudaStream_t st = ctx->stream;
  const size_t bytes = static_cast<size_t>(n) * 4;
  for (int i = 1; i <= 4; i++) LGS_TRY(ctx->tmp[i].reserve(bytes));
  LGS_CUDA(cudaMemcpyAsync(ctx->tmp[1].p, keys, bytes, cudaMemcpyHostToDevice, st));
  LGS_CUDA(cudaMemcpyAsync(ctx->tmp[2].p, vals, bytes, cudaMemcpyHostToDevice, st));
  unsigned *ko, *vo;
  LGS_TRY(lgs::radix_sort_pairs(ctx, ctx->tmp[1].as<unsigned>(), ctx->tmp[2].as<unsigned>(), ctx->tmp[3].as<unsigned>(), ctx->tmp[4].as<unsigned>(), n,
                                bits, &ko, &vo));
  LGS_CUDA(cudaMemcpyAsync(keys, ko, bytes, cudaMemcpyDeviceToHost, st));
  LGS_CUDA(cudaMemcpyAsync(vals, vo, bytes, cudaMemcpyDeviceToHost, st));
  LGS_CUDA(cudaStreamSynchronize(st));
  return LGS_OK;
}
