// Silhouette sums of the euclidean distances of rows sorted by label (jb_silhouette): for each query row i and label c,
// S[i, c] = sum over the rows j of label c of sqrt(|x_i - x_j|^2), the squared distances from FOSCTTM's tile arithmetic
// (mt_tile: float64 sums of squared fp32 differences), then intra[i] = S[i, l_i] and inter[i] = min over c != l_i of
// S[i, c] / n_c (sklearn's _silhouette_reduce before its intra division). The reference rows are cut into chunks of
// SL_CHUNK_TILES tiles that depend on n only; a chunk's sum for each (row, label) it holds goes to its own workspace slot
// and the slots of a label are folded in chunk order. No floating-point atomics: every sum's order depends only on the
// row, the tile and the chunk, so results are bit-identical for any query batch and device.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

#include "metrics.cuh"

namespace jb {

constexpr int SL_CHUNK_TILES = 64;                    // reference tiles (of MT_TILE rows) per chunk
constexpr int SL_CHUNK = SL_CHUNK_TILES * MT_TILE;    // 4096 reference rows per chunk
constexpr int SL_LD = 4 * 17;                         // staged tile row: four 16-column quarters, each padded by one
constexpr size_t SL_SMEM = static_cast<size_t>(MT_TILE) * SL_LD * sizeof(double);

// Block (chunk x, query tile y): the 64 query rows [64 y, 64 y + 64) of the batch (sorted rows q0 + ...) against the
// reference rows of chunk x. Each tile's 64 x 64 distances are staged in shared memory; the 4 threads
// of a query row (quarter q = threadIdx & 3) then add the tile into the row's running sum of the current label segment.
// A tile inside one segment is summed as four 16-column quarters in column order, combined as (q0 + q1) + (q2 + q3); a
// tile that crosses a segment end is walked column by column. A finished segment is written once, to
// ws[slot * nb + row] with slot = slot_base[chunk] + label - first_label[chunk].
__global__ void __launch_bounds__(MT_THREADS) k_sil_partial(const float* __restrict__ x, long long n, int L, long long q0, long long nb,
                                                            const long long* __restrict__ label_off,
                                                            const long long* __restrict__ slot_base, const int* __restrict__ first_label,
                                                            double* __restrict__ ws) {
  __shared__ float As[MT_TILE][MT_LC + 1], Bs[MT_TILE][MT_LC + 1];
  extern __shared__ double sil_smem[];   // [MT_TILE][SL_LD]
  const long long ch = blockIdx.x;
  const long long i0 = static_cast<long long>(blockIdx.y) * MT_TILE;   // first query row of the block, in the batch
  const long long c0 = ch * SL_CHUNK, c1 = c0 + SL_CHUNK < n ? c0 + SL_CHUNK : n;
  const int li = threadIdx.x >> 2, q = threadIdx.x & 3;
  const bool own = q == 0 && i0 + li < nb;   // this thread writes the row's slots
  double* row_ws = ws + (i0 + li);
  const long long base = slot_base[ch];
  const int lab0 = first_label[ch];
  int c = lab0;
  long long e = label_off[c + 1] < c1 ? label_off[c + 1] : c1;   // end of the current segment (every thread tracks it)
  double acc = 0.0;
  for (long long j0 = c0; j0 < c1; j0 += MT_TILE) {
    const long long j1 = j0 + MT_TILE < c1 ? j0 + MT_TILE : c1;
    mt_tile(x + q0 * L, nb, x, n, L, i0, j0, As, Bs, [&](long long i, long long j, double d) {
      const int r = static_cast<int>(i - i0), k = static_cast<int>(j - j0);
      sil_smem[r * SL_LD + (k >> 4) * 17 + (k & 15)] = sqrt(d);
    });
    __syncthreads();
    const double* D = sil_smem + li * SL_LD;
    if (e >= j1) {   // the whole tile lies in segment c
      const int k0 = 16 * q, k1 = static_cast<int>(j1 - j0) < k0 + 16 ? static_cast<int>(j1 - j0) : k0 + 16;
      double s = 0.0;
      for (int k = k0; k < k1; ++k) s += D[q * 17 + (k & 15)];
      s += __shfl_xor_sync(0xffffffffu, s, 1);   // q0 + q1 and q2 + q3, the same bits in both lanes of a pair
      s += __shfl_xor_sync(0xffffffffu, s, 2);
      acc += s;
    } else {
      for (long long j = j0; j < j1; ++j) {
        if (j == e) {
          if (own) row_ws[(base + c - lab0) * nb] = acc;
          acc = 0.0;
          ++c;
          e = label_off[c + 1] < c1 ? label_off[c + 1] : c1;
        }
        const int k = static_cast<int>(j - j0);
        acc += D[(k >> 4) * 17 + (k & 15)];
      }
    }
    if (e == j1) {   // the segment ends with the tile
      if (own) row_ws[(base + c - lab0) * nb] = acc;
      acc = 0.0;
      if (j1 < c1) {
        ++c;
        e = label_off[c + 1] < c1 ? label_off[c + 1] : c1;
      }
    }
    // the next tile's first barrier (inside mt_tile) orders these reads before the staged tile is overwritten
  }
}

// One thread per query row of the batch: S[c] = the row's chunk slots of label c folded in chunk order; intra = S[l_i],
// inter = min over c != l_i of S[c] / n_c (one correctly rounded division, as numpy's).
constexpr int SF_THREADS = 128;
__global__ void __launch_bounds__(SF_THREADS) k_sil_finish(const double* __restrict__ ws, long long q0, long long nb,
                                                           const long long* __restrict__ label_off, int n_labels,
                                                           const long long* __restrict__ slot_base, const int* __restrict__ first_label,
                                                           double* __restrict__ intra, double* __restrict__ inter) {
  const long long r = static_cast<long long>(blockIdx.x) * SF_THREADS + threadIdx.x;
  if (r >= nb) return;
  const long long i = q0 + r;   // sorted row index
  int lo = 0, hi = n_labels - 1;   // the row's label: the last c with label_off[c] <= i
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (label_off[mid] <= i) lo = mid; else hi = mid - 1;
  }
  const int li = lo;
  double a = 0.0, b = __longlong_as_double(0x7ff0000000000000LL);   // +inf
  for (int c = 0; c < n_labels; ++c) {
    const long long s0 = label_off[c], s1 = label_off[c + 1];
    double S = 0.0;
    for (long long ch = s0 / SL_CHUNK; ch <= (s1 - 1) / SL_CHUNK; ++ch) S += ws[(slot_base[ch] + c - first_label[ch]) * nb + r];
    if (c == li) a = S;
    else b = fmin(b, __ddiv_rn(S, static_cast<double>(s1 - s0)));
  }
  intra[r] = a;
  inter[r] = b;
}

}  // namespace jb
