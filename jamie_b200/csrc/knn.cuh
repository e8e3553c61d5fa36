// Exact euclidean k-nearest-neighbour search and the kNN average of a reference matrix (jb_knn, jb_knn_average).
// The search is FOSCTTM's tile arithmetic (mt_tile: float64 squared distances of fp32 rows) with a selecting consumer:
// each query keeps its k best (distance, reference index) pairs, ordered by the float64 squared sum and then by the
// index (a stable argsort's order), without storing a distance matrix. Integer atomics in shared memory only: the pairs
// form a total order, so the lists do not depend on the order in which candidates arrive, the schedule or the split of
// the queries and references into batches and ranges.
#pragma once
#include <cuda_runtime.h>
#include <climits>
#include <cstdint>

#include "metrics.cuh"

namespace jb {

constexpr int KN_MAXK = 1024;   // largest k
constexpr int KN_BUF = 112;     // candidates per query buffered in shared memory before they are merged into its list
constexpr size_t KN_SMEM = static_cast<size_t>(MT_TILE) * KN_BUF * (sizeof(double) + sizeof(int));

__device__ __forceinline__ bool kn_less(double da, int ja, double db, int jb) { return da < db || (da == db && ja < jb); }

// Merges the buffered candidates of query row li into its sorted list, by one warp. Each element's place in the merged
// list is its rank: its position in its own sequence plus the number of elements of the other sequence that precede it
// (the buffer is unsorted, so its own rank is counted too). The lists of a query alternate between two arrays of k.
__device__ __forceinline__ void kn_flush(int li, int k, const double* bd, const int* bj, int* cnt, int* len, int* which,
                                         double* thr_d, int* thr_j, double* ld, int* lj) {
  const int lane = threadIdx.x & 31;
  const int nb = cnt[li], m = len[li], src = which[li];
  const double* Bd = bd + li * KN_BUF;
  const int* Bj = bj + li * KN_BUF;
  const double* Sd = ld + static_cast<long long>(src) * k;
  const int* Sj = lj + static_cast<long long>(src) * k;
  double* Dd = ld + static_cast<long long>(1 - src) * k;
  int* Dj = lj + static_cast<long long>(1 - src) * k;
  for (int e = lane; e < nb; e += 32) {
    const double d = Bd[e];
    const int j = Bj[e];
    int r = 0;
    for (int f = 0; f < nb; ++f) r += kn_less(Bd[f], Bj[f], d, j);
    int lo = 0, hi = m;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (kn_less(Sd[mid], Sj[mid], d, j)) lo = mid + 1; else hi = mid;
    }
    r += lo;
    if (r < k) { Dd[r] = d; Dj[r] = j; }
    if (r == k - 1) { thr_d[li] = d; thr_j[li] = j; }
  }
  for (int p = lane; p < m; p += 32) {
    const double d = Sd[p];
    const int j = Sj[p];
    int r = p;
    for (int f = 0; f < nb; ++f) r += kn_less(Bd[f], Bj[f], d, j);
    if (r < k) { Dd[r] = d; Dj[r] = j; }
    if (r == k - 1) { thr_d[li] = d; thr_j[li] = j; }
  }
  __syncwarp();
  if (lane == 0) {
    len[li] = m + nb < k ? m + nb : k;
    which[li] = 1 - src;
    cnt[li] = 0;
  }
  __syncwarp();
}

// Block (query tile x, reference range y): the sorted k best of the range for each of 64 query rows. A candidate enters
// the shared buffer of its query when it precedes the query's current k-th best; a buffer that may not take another
// tile's 64 candidates is merged after the tile, and every buffer at the end. Lists: ld / lj [ranges, nq, 2, k], meta
// [ranges, nq] = (length, which of the two arrays holds the list).
__global__ void __launch_bounds__(MT_THREADS) k_knn_search(const float* __restrict__ q, long long nq, const float* __restrict__ r,
                                                           long long nr, int L, int k, long long tiles_per_range,
                                                           double* __restrict__ ld, int* __restrict__ lj, int2* __restrict__ meta) {
  __shared__ float As[MT_TILE][MT_LC + 1], Bs[MT_TILE][MT_LC + 1];
  __shared__ double thr_d[MT_TILE];
  __shared__ int thr_j[MT_TILE], cnt[MT_TILE], len[MT_TILE], which[MT_TILE];
  extern __shared__ double knn_smem[];
  double* bd = knn_smem;                                   // [64][KN_BUF]
  int* bj = reinterpret_cast<int*>(knn_smem + MT_TILE * KN_BUF);
  const long long i0 = static_cast<long long>(blockIdx.x) * MT_TILE;
  const long long tiles = (nr + MT_TILE - 1) / MT_TILE;
  const long long t0 = blockIdx.y * tiles_per_range, t1 = t0 + tiles_per_range < tiles ? t0 + tiles_per_range : tiles;
  const long long row0 = static_cast<long long>(blockIdx.y) * nq + i0;   // list of query i0 of this range
  double* bld = ld + row0 * 2 * k;
  int* blj = lj + row0 * 2 * k;
  const int warp = threadIdx.x >> 5;
  if (threadIdx.x < MT_TILE) {
    thr_d[threadIdx.x] = __longlong_as_double(0x7ff0000000000000LL);   // +inf: every candidate enters until k are held
    thr_j[threadIdx.x] = INT_MAX;
    cnt[threadIdx.x] = len[threadIdx.x] = which[threadIdx.x] = 0;
  }
  for (long long t = t0; t < t1; ++t) {
    int full = 0;
    mt_tile(q, nq, r, nr, L, i0, t * MT_TILE, As, Bs, [&](long long i, long long j, double d) {
      const int li = static_cast<int>(i - i0), jj = static_cast<int>(j);
      if (kn_less(d, jj, thr_d[li], thr_j[li])) {
        const int s = atomicAdd(&cnt[li], 1);
        bd[li * KN_BUF + s] = d;
        bj[li * KN_BUF + s] = jj;
        full |= s >= KN_BUF - MT_TILE;
      }
    });
    const bool last = t + 1 == t1;
    if (__syncthreads_or(full) || last) {
      for (int li = warp; li < MT_TILE; li += MT_THREADS / 32)
        if (cnt[li] > (last ? 0 : KN_BUF - MT_TILE))
          kn_flush(li, k, bd, bj, cnt, len, which, thr_d, thr_j, bld + static_cast<long long>(li) * 2 * k, blj + static_cast<long long>(li) * 2 * k);
    }
    // the next tile's first barrier (inside mt_tile) orders these merges before its candidates are tested
  }
  __syncthreads();
  if (threadIdx.x < MT_TILE && i0 + threadIdx.x < nq) meta[row0 + threadIdx.x] = make_int2(len[threadIdx.x], which[threadIdx.x]);
}

// One block per query row: merges the sorted lists of the reference ranges (each element placed at its rank among all
// of them) into the first k, and writes the indices and sqrt of the squared sums.
constexpr int KM_THREADS = 128;
__global__ void __launch_bounds__(KM_THREADS) k_knn_merge(const double* __restrict__ ld, const int* __restrict__ lj,
                                                          const int2* __restrict__ meta, int ranges, long long nq, int k,
                                                          long long* __restrict__ idx, double* __restrict__ dist) {
  const long long qi = blockIdx.x;
  for (long long e = threadIdx.x; e < static_cast<long long>(ranges) * k; e += KM_THREADS) {
    const int s = static_cast<int>(e / k), p = static_cast<int>(e % k);
    const int2 ms = meta[s * nq + qi];
    if (p >= ms.x) continue;
    const long long base = (s * nq + qi) * 2 * k + static_cast<long long>(ms.y) * k;
    const double d = ld[base + p];
    const int j = lj[base + p];
    int rank = p;
    for (int t = 0; t < ranges && rank < k; ++t) {
      if (t == s) continue;
      const int2 mt = meta[t * nq + qi];
      const double* Td = ld + (t * nq + qi) * 2 * k + static_cast<long long>(mt.y) * k;
      const int* Tj = lj + (t * nq + qi) * 2 * k + static_cast<long long>(mt.y) * k;
      int lo = 0, hi = mt.x;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (kn_less(Td[mid], Tj[mid], d, j)) lo = mid + 1; else hi = mid;
      }
      rank += lo;
    }
    if (rank < k) {
      idx[qi * k + rank] = j;
      if (dist) dist[qi * k + rank] = sqrt(d);
    }
  }
}

// out[q, c] = sum_t w[q, t] v[idx[q, t], c] / sum_t w[q, t] over a column slab v [nr, ws], float64, summed in list order
// (w = 1 when null). Products and sums are rounded separately, as numpy's sum of the products does.
constexpr int KA_THREADS = 128;
__global__ void __launch_bounds__(KA_THREADS) k_knn_average(const long long* __restrict__ idx, const double* __restrict__ w,
                                                            int k, const double* __restrict__ v, int ws, double* __restrict__ out) {
  const long long qi = blockIdx.x;
  const int c = blockIdx.y * KA_THREADS + threadIdx.x;
  if (c >= ws) return;
  double s = 0.0, sw = 0.0;
  for (int t = 0; t < k; ++t) {
    const double wt = w ? w[qi * k + t] : 1.0;
    s = __dadd_rn(s, __dmul_rn(wt, v[idx[qi * k + t] * ws + c]));
    sw = __dadd_rn(sw, wt);
  }
  out[qi * ws + c] = s / sw;
}

}  // namespace jb
