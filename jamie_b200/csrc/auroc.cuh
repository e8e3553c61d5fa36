// Per-feature AUROC of an imputation against the measured modality read as present / absent (jb_metric_feature_auroc,
// jamie_b200/evaluation.py imputation_auroc; the reference's AUROC panel, jamie/evaluation.py:468-490, sklearn
// roc_auc_score on measured > threshold). Exact integer Mann-Whitney statistic per column:
//   2U = sum over (positive p, negative q) of 2 [s_q < s_p] + [s_q == s_p]
//      = sum over negatives q of 2P - lt(s_q) - le(s_q),   lt / le = #positives with a score < / <= s_q,
// computed as (the same sum over all rows) - (the sum over the positive rows), modulo 2^64 (the true value is < 2^62).
// Per column batch: k_auroc_keys turns the [n, w] fp32 slab into order-preserving uint32 keys, transposed to [w, n] so
// that a column is contiguous; k_auroc_col (one CTA per column) gathers the positives' keys, sorts them with a stable
// LSD radix sort (4 x 8-bit digits, ranks within a warp from __match_any_sync), and binary-searches every row's key in
// the sorted positives. Only integer arithmetic: results do not depend on the batch split or the schedule.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

namespace jb {

constexpr int AU_THREADS = 256;          // one thread per radix digit in the scan
constexpr int AU_WARPS = AU_THREADS / 32;
constexpr int AU_SMEM_ROWS = 26 * 1024;  // n up to this: the sort's two key buffers (8 B per positive) in shared memory

// order-preserving key of a finite fp32 score; -0.0 and +0.0 are one key
__device__ __forceinline__ uint32_t au_key(float f) {
  uint32_t u = __float_as_uint(f);
  if (u == 0x80000000u) u = 0u;
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// keys[c, r] = au_key(slab[r, c]) for a [n, w] row-major slab, through a 32 x 32 shared tile (both sides coalesced)
__global__ void __launch_bounds__(256) k_auroc_keys(const float* __restrict__ slab, long long n, int w, uint32_t* __restrict__ keys) {
  __shared__ uint32_t t[32][33];
  const long long r0 = static_cast<long long>(blockIdx.x) * 32;
  const int c0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += 8) {
    const long long r = r0 + i;
    const int c = c0 + threadIdx.x;
    if (r < n && c < w) t[i][threadIdx.x] = au_key(slab[r * w + c]);
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int c = c0 + i;
    const long long r = r0 + threadIdx.x;
    if (r < n && c < w) keys[c * n + r] = t[threadIdx.x][i];
  }
}

// #{i < P: a[i] < k} (UPPER: a[i] <= k) in the sorted a
template <bool UPPER>
__device__ __forceinline__ uint32_t au_bound(const uint32_t* a, uint32_t P, uint32_t k) {
  uint32_t lo = 0, hi = P;
  while (lo < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (UPPER ? a[mid] <= k : a[mid] < k) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

// One CTA per column of the batch. keys [w, n]; the positives of column c are rows[ptr[c] - ptr[0], ptr[c + 1] - ptr[0]).
// SH: the sort's buffers (2 x pcap keys, pcap >= every P of the batch) in dynamic shared memory; else 2 n keys of
// `scratch` per column. u2[c] = 2U of the column.
template <bool SH>
__global__ void __launch_bounds__(AU_THREADS) k_auroc_col(const uint32_t* __restrict__ keys, long long n, const long long* __restrict__ ptr,
                                                         const int* __restrict__ rows, int pcap, uint32_t* __restrict__ scratch,
                                                         unsigned long long* __restrict__ u2) {
  extern __shared__ uint32_t au_sm[];
  __shared__ uint32_t run[256];              // per digit: the next output position
  __shared__ uint32_t wcnt[AU_WARPS][256];   // per warp and digit: elements of the current tile
  __shared__ uint32_t wsum[AU_WARPS];
  __shared__ unsigned long long red[AU_WARPS];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned lt_mask = (1u << lane) - 1u;
  const long long c = blockIdx.x;
  const uint32_t* kc = keys + c * n;
  const int* pr = rows + (ptr[c] - ptr[0]);
  const uint32_t P = static_cast<uint32_t>(ptr[c + 1] - ptr[c]);
  uint32_t *A, *B;
  if (SH) {
    A = au_sm;
    B = au_sm + pcap;
  } else {
    A = scratch + c * 2 * n;
    B = A + n;
  }
  for (int q = 0; q < AU_WARPS; ++q) wcnt[q][tid] = 0u;
  for (uint32_t i = tid; i < P; i += AU_THREADS) A[i] = kc[pr[i]];
  __syncthreads();

  for (int shift = 0; shift < 32; shift += 8) {
    // digit histogram (one atomic per group of equal digits in a warp), then its exclusive scan: thread = digit
    run[tid] = 0u;
    __syncthreads();
    for (uint32_t t0 = 0; t0 < P; t0 += AU_THREADS) {
      const uint32_t i = t0 + tid;
      const uint32_t dig = i < P ? (A[i] >> shift) & 255u : 256u;
      const unsigned peers = __match_any_sync(0xffffffffu, dig);
      if (i < P && (peers & lt_mask) == 0u) atomicAdd(&run[dig], static_cast<uint32_t>(__popc(peers)));
    }
    __syncthreads();
    const uint32_t h = run[tid];
    uint32_t x = h;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) wsum[warp] = x;
    __syncthreads();
    uint32_t off = 0;
    for (int q = 0; q < warp; ++q) off += wsum[q];
    run[tid] = off + x - h;
    __syncthreads();
    // stable scatter, one tile of AU_THREADS elements at a time in order: position = run[digit] + the tile's equal
    // digits in lower warps + the equal digits in lower lanes of this warp
    for (uint32_t t0 = 0; t0 < P; t0 += AU_THREADS) {
      const uint32_t i = t0 + tid;
      const uint32_t k = i < P ? A[i] : 0u;
      const uint32_t dig = i < P ? (k >> shift) & 255u : 256u;
      const unsigned peers = __match_any_sync(0xffffffffu, dig);
      if (i < P && (peers & lt_mask) == 0u) wcnt[warp][dig] = static_cast<uint32_t>(__popc(peers));
      __syncthreads();
      if (i < P) {
        uint32_t pos = run[dig] + static_cast<uint32_t>(__popc(peers & lt_mask));
        for (int q = 0; q < warp; ++q) pos += wcnt[q][dig];
        B[pos] = k;
      }
      __syncthreads();
      uint32_t s = 0;
#pragma unroll
      for (int q = 0; q < AU_WARPS; ++q) {
        s += wcnt[q][tid];
        wcnt[q][tid] = 0u;
      }
      run[tid] += s;
      __syncthreads();
    }
    uint32_t* tmp = A;
    A = B;
    B = tmp;
  }

  // sum of 2P - lt - le over all rows, minus the same over the positives (A, sorted)
  unsigned long long acc = 0;
  for (long long r = tid; r < n; r += AU_THREADS) {
    const uint32_t k = kc[r];
    acc += 2ull * P - au_bound<false>(A, P, k) - au_bound<true>(A, P, k);
  }
  for (uint32_t i = tid; i < P; i += AU_THREADS) {
    const uint32_t k = A[i];
    acc -= 2ull * P - au_bound<false>(A, P, k) - au_bound<true>(A, P, k);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) red[warp] = acc;
  __syncthreads();
  if (tid == 0) {
    unsigned long long s = 0;
    for (int q = 0; q < AU_WARPS; ++q) s += red[q];
    u2[c] = s;
  }
}

}  // namespace jb
