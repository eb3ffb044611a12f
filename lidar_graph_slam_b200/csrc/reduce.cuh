// The last-CTA reduction behind every value an evaluation returns to the host (DESIGN section 2, "Reductions").
//
// Each CTA reduces its threads to one row of K sums and stores the row in `partials`; it fences and arrives on a counter.
// The last CTA to arrive folds the G rows, re-arms the counter and publishes the K sums to the mailbox (common.cuh).
// The fold has NG groups: group g adds rows g, g + NG, g + 2 NG, ... in that order, starting from zero; the NG group sums
// are then added in group order, starting from zero.  The order is a fixed function of G and NG, so the sums are the same
// bits run after run; NG is part of each call site's result.  lgs_grid_fold_check (linalg_check.cu) runs this code on
// given rows, so that tests can compare it with the same fold written out in Python.
//
// T is double (rounded sums: the order above is what makes them reproducible) or Fix128 (fixsum.cuh: exact sums, which
// any order gives).
#pragma once
#include "common.cuh"
#include "fixsum.cuh"

namespace lgs {

__device__ __forceinline__ void sum_add(double& a, double b) { a += b; }
__device__ __forceinline__ void sum_add(Fix128& a, const Fix128& b) { fix_add(a, b); }
__device__ __forceinline__ double sum_value(double a) { return a; }
__device__ __forceinline__ double sum_value(const Fix128& a) { return fix_value(a); }
__device__ __forceinline__ double shfl_xor(double v, int off) { return __shfl_xor_sync(0xffffffffu, v, off); }
__device__ __forceinline__ Fix128 shfl_xor(const Fix128& v, int off) {
  Fix128 o;
  o.lo = __shfl_xor_sync(0xffffffffu, v.lo, off);
  o.hi = __shfl_xor_sync(0xffffffffu, v.hi, off);
  return o;
}
__device__ __forceinline__ double load_row(const double* p) { return __ldcg(p); }
__device__ __forceinline__ Fix128 load_row(const Fix128* p) {
  const ulonglong2 t = __ldcg(reinterpret_cast<const ulonglong2*>(p));
  Fix128 v;
  v.lo = t.x;
  v.hi = static_cast<long long>(t.y);
  return v;
}

// The CTA row of K per-thread sums (NT threads): each sum is reduced across its warp by shuffle-xor (16, 8, 4, 2, 1),
// then the warps are added in order.  Thread k < K gets sum k.
template <int NT, int K, typename T>
__device__ __forceinline__ T cta_row(const T (&acc)[K]) {
  __shared__ T warp_sums[NT / 32][K];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < K; k++) {
    T v = acc[k];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) sum_add(v, shfl_xor(v, off));
    if (lane == 0) warp_sums[warp][k] = v;
  }
  __syncthreads();
  T r{};
  if (threadIdx.x < K) {
#pragma unroll
    for (int w = 0; w < NT / 32; w++) sum_add(r, warp_sums[w][threadIdx.x]);
  }
  return r;
}

// The fold of columns 0 .. K-1 of the G rows rows[b * S + k] in the order stated at the top, by all NT threads of one
// CTA: group g is threads g * NT / NG ... (g + 1) * NT / NG - 1, whose thread c adds columns c, c + NT / NG, ...; each
// keeps the loads of U rows in flight (rows past G load as zero: adding zero to a sum that started from +0 changes no
// bit).  Thread k < K gets the sum of column k.  K <= KMAX <= S: the last pass over the columns may also add columns
// K .. KMAX-1, whose sums are dropped.
template <int NT, int NG, int U, int KMAX, typename T>
__device__ __forceinline__ T grid_fold(const T* __restrict__ rows, unsigned G, int S, int K) {
  static_assert(NT % NG == 0, "equal groups");
  constexpr int CW = NT / NG;
  __shared__ T group_sums[NG][KMAX];
  const int g = threadIdx.x / CW;
  for (int h = 0; h * CW < K; h++) {
    const int c = h * CW + threadIdx.x % CW;
    T v{};
    for (unsigned b0 = g; b0 < G; b0 += U * NG) {
      T t[U];
#pragma unroll
      for (int u = 0; u < U; u++) {
        const unsigned b = b0 + u * NG;
        t[u] = (b < G && c < KMAX) ? load_row(rows + static_cast<size_t>(b) * S + c) : T{};
      }
#pragma unroll
      for (int u = 0; u < U; u++) sum_add(v, t[u]);
    }
    if (c < KMAX) group_sums[g][c] = v;
  }
  __syncthreads();
  T r{};
  if (static_cast<int>(threadIdx.x) < K) {
#pragma unroll
    for (int h = 0; h < NG; h++) sum_add(r, group_sums[h][threadIdx.x]);
  }
  return r;
}

// The grid half, once this CTA's row is in partials[blockIdx.x * S + k] (k < K), stored by any of its threads: fence and
// arrive; the last CTA folds the rows, re-arms the counter and publishes the K sums.  Callable any number of times in
// one launch (the persistent grids call it once per evaluation).
template <int K, int S, int NT, int NG, int U, typename T>
__device__ __forceinline__ void grid_finish_rows(const T* __restrict__ partials, unsigned* __restrict__ counter, const Mailbox& mb) {
  __shared__ bool is_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) is_last = atomicAdd(counter, 1u) == gridDim.x - 1;
  __syncthreads();
  if (is_last) {
    __threadfence();
    const T r = grid_fold<NT, NG, U, K>(partials, gridDim.x, S, K);
    if (threadIdx.x == 0) *counter = 0;
    mailbox_publish<K>(mb, sum_value(r));
  }
}

// The same with thread k < K holding this CTA's sum k.
template <int K, int NT, int NG, int U, typename T>
__device__ __forceinline__ void grid_finish(T v, T* __restrict__ partials, unsigned* __restrict__ counter, const Mailbox& mb) {
  if (threadIdx.x < K) partials[static_cast<size_t>(blockIdx.x) * K + threadIdx.x] = v;
  grid_finish_rows<K, K, NT, NG, U>(partials, counter, mb);
}

}  // namespace lgs
