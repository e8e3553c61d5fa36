// Distances of the F estimation on the GPU (SURVEY.md 8f row N2): compute_distances (jamie/jamie.py:839-890) and the
// geodesic distance of unioncom's geodesic_distances (kNN graph, all-pairs shortest paths, unreachable pairs at twice the
// largest finite distance). One n x n float64 matrix D per handle, built in four steps:
//   k_dist_accum  D[i, j] += sum_c f(x_ic, x_jc) over a [n, w] float64 column slab, f = (a - b)^2, |a - b| or a b.
//                 64 x 64 register tiles of CUDA-core fp64 fma (B200's fp64 tensor rate is no higher than its vector
//                 rate), upper-triangle tiles only, each sum written to D[i, j] and D[j, i]: D is bitwise symmetric and
//                 its diagonal is exactly 0 for the difference forms. Columns are summed in index order whatever the
//                 slab width, so the result is deterministic.
//   k_dist_finish sqrt (euclidean), 1 - g clipped to [0, 2] with a zero diagonal (sklearn cosine, scipy correlation),
//                 (1 - clip(g, -1, 1)) / 2 (np.corrcoef for pearson / spearman). NaN stays NaN.
//   k_knn_rows    per row the k smallest entries in ascending order, equal values by the lowest column (a stable
//                 argsort): radix select on the bit patterns of the non-negative doubles, then a rank by counting.
//   k_fw_*        blocked Floyd-Warshall (min-plus, float64, in place) on the kNN graph written into D.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

namespace jb {

enum DistKind { DIST_SQDIFF = 0, DIST_ABSDIFF = 1, DIST_PRODUCT = 2 };
enum DistTransform { DIST_NONE = 0, DIST_SQRT = 1, DIST_ONE_MINUS = 2, DIST_HALF_ONE_MINUS = 3 };

constexpr int DA_TILE = 64;     // rows x rows per block
constexpr int DA_LC = 16;       // slab columns per shared-memory chunk
constexpr int DA_THREADS = 256; // 16 x 16 threads, 4 x 4 pairs each

// Tile t of the upper triangle (ti <= tj) in row-major order of the triangle.
__device__ __forceinline__ void tri_tile(long long t, long long tiles, long long& ti, long long& tj) {
  // row ti holds tiles - ti tiles; find ti by a float guess corrected in integers
  const double T = static_cast<double>(tiles);
  long long r = static_cast<long long>(T + 0.5 - sqrt((T + 0.5) * (T + 0.5) - 2.0 * static_cast<double>(t)));
  if (r < 0) r = 0;
  if (r > tiles - 1) r = tiles - 1;
  auto start = [&](long long q) { return q * tiles - q * (q - 1) / 2; };
  while (r > 0 && start(r) > t) --r;
  while (r + 1 < tiles && start(r + 1) <= t) ++r;
  ti = r;
  tj = r + (t - start(r));
}

template <int KIND>
__global__ void __launch_bounds__(DA_THREADS) k_dist_accum(const double* __restrict__ slab, long long n, int w, long long ld,
                                                           double* __restrict__ D) {
  __shared__ double As[DA_TILE][DA_LC + 1], Bs[DA_TILE][DA_LC + 1];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const long long tiles = (n + DA_TILE - 1) / DA_TILE, ntri = tiles * (tiles + 1) / 2;
  for (long long t = blockIdx.x; t < ntri; t += gridDim.x) {
    long long ti, tj;
    tri_tile(t, tiles, ti, tj);
    const long long i0 = ti * DA_TILE, j0 = tj * DA_TILE;
    double acc[4][4];
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        const long long i = i0 + ty + 16 * u, j = j0 + tx + 16 * v;
        acc[u][v] = (i < n && j < n && i <= j) ? D[i * n + j] : 0.0;
      }
    for (int c0 = 0; c0 < w; c0 += DA_LC) {
      __syncthreads();
      for (int e = threadIdx.x; e < DA_TILE * DA_LC; e += DA_THREADS) {
        const int r = e / DA_LC, c = e % DA_LC;
        As[r][c] = (i0 + r < n && c0 + c < w) ? slab[(i0 + r) * ld + c0 + c] : 0.0;
        Bs[r][c] = (j0 + r < n && c0 + c < w) ? slab[(j0 + r) * ld + c0 + c] : 0.0;
      }
      __syncthreads();
      // zero-padded columns add f(0, 0) = 0 exactly: the sum is the same as without padding
#pragma unroll 4
      for (int c = 0; c < DA_LC; ++c) {
        double av[4], bv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) { av[u] = As[ty + 16 * u][c]; bv[u] = Bs[tx + 16 * u][c]; }
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
          for (int v = 0; v < 4; ++v) {
            if (KIND == DIST_SQDIFF) {
              const double d = av[u] - bv[v];
              acc[u][v] = fma(d, d, acc[u][v]);
            } else if (KIND == DIST_ABSDIFF) {
              acc[u][v] += fabs(av[u] - bv[v]);
            } else {
              acc[u][v] = fma(av[u], bv[v], acc[u][v]);
            }
          }
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        const long long i = i0 + ty + 16 * u, j = j0 + tx + 16 * v;
        if (i < n && j < n && i <= j) {
          D[i * n + j] = acc[u][v];
          D[j * n + i] = acc[u][v];
        }
      }
  }
}

__global__ void k_dist_finish(double* __restrict__ D, long long n, int transform) {
  const long long nn = n * n;
  for (long long q = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; q < nn; q += static_cast<long long>(gridDim.x) * blockDim.x) {
    double g = D[q];
    if (transform == DIST_SQRT) {
      g = sqrt(g);
    } else if (transform == DIST_ONE_MINUS) {
      g = 1.0 - g;
      g = g < 0.0 ? 0.0 : (g > 2.0 ? 2.0 : g);   // comparisons, not fmin / fmax: NaN propagates
      if (q / n == q % n) g = 0.0;
    } else if (transform == DIST_HALF_ONE_MINUS) {
      g = g < -1.0 ? -1.0 : (g > 1.0 ? 1.0 : g);
      g = (1.0 - g) / 2.0;
    }
    D[q] = g;
  }
}

// One block per row of D (non-negative doubles: their bit patterns order as the values). T = the k-th smallest pattern
// (8 radix passes of 8 bits); the entries below T and the first `need` entries equal to T (in column order) are
// gathered, then each one's rank among them by (value, column) places it in the output.
constexpr int KN_THREADS = 256;
__global__ void __launch_bounds__(KN_THREADS) k_knn_rows(const double* __restrict__ D, long long n, int k, int* __restrict__ idx,
                                                         double* __restrict__ dist) {
  extern __shared__ __align__(16) unsigned char kn_smem[];
  unsigned long long* cv = reinterpret_cast<unsigned long long*>(kn_smem);   // [k] candidate values
  int* ci = reinterpret_cast<int*>(cv + k);                                  // [k] candidate columns
  __shared__ unsigned int hist[256];
  __shared__ unsigned long long s_prefix;
  __shared__ unsigned int s_need, s_run, s_cnt;
  __shared__ unsigned int wcnt[KN_THREADS / 32];
  const long long row = blockIdx.x;
  const unsigned long long* r = reinterpret_cast<const unsigned long long*>(D + row * n);
  const int tid = threadIdx.x;
  if (tid == 0) { s_prefix = 0ull; s_need = static_cast<unsigned int>(k); }
  for (int shift = 56; shift >= 0; shift -= 8) {
    hist[tid] = 0u;
    __syncthreads();
    const unsigned long long prefix = s_prefix, mask = shift == 56 ? 0ull : (~0ull << (shift + 8));
    for (long long j = tid; j < n; j += KN_THREADS) {
      const unsigned long long v = r[j];
      if ((v & mask) == prefix) atomicAdd(&hist[(v >> shift) & 255u], 1u);
    }
    __syncthreads();
    if (tid == 0) {
      unsigned int need = s_need, b = 0;
      for (; b < 256u; ++b) {
        if (hist[b] >= need) break;
        need -= hist[b];
      }
      s_prefix = prefix | (static_cast<unsigned long long>(b) << shift);
      s_need = need;
    }
    __syncthreads();
  }
  const unsigned long long T = s_prefix;
  if (tid == 0) { s_run = 0u; s_cnt = 0u; }
  __syncthreads();
  // gather: the slot order is arbitrary, the ranking below makes the output order exact
  for (long long j0 = 0; j0 < n; j0 += KN_THREADS) {
    const long long j = j0 + tid;
    const unsigned long long v = j < n ? r[j] : ~0ull;
    if (j < n && v < T) {
      const unsigned int s = atomicAdd(&s_cnt, 1u);
      cv[s] = v; ci[s] = static_cast<int>(j);
    }
    const bool tie = j < n && v == T;
    const unsigned int bal = __ballot_sync(0xffffffffu, tie);
    if ((tid & 31) == 0) wcnt[tid >> 5] = __popc(bal);
    __syncthreads();
    if (tie) {   // ties in column order: the first s_need of them are among the k nearest
      unsigned int before = s_run;
      for (int w = 0; w < (tid >> 5); ++w) before += wcnt[w];
      before += __popc(bal & ((1u << (tid & 31)) - 1u));
      if (before < s_need) {
        const unsigned int s = atomicAdd(&s_cnt, 1u);
        cv[s] = v; ci[s] = static_cast<int>(j);
      }
    }
    __syncthreads();
    if (tid == 0) {
      unsigned int s = 0;
      for (int w = 0; w < KN_THREADS / 32; ++w) s += wcnt[w];
      s_run += s;
    }
    __syncthreads();
  }
  for (int a = tid; a < k; a += KN_THREADS) {
    const unsigned long long va = cv[a];
    const int ia = ci[a];
    int rank = 0;
    for (int b = 0; b < k; ++b) rank += (cv[b] < va || (cv[b] == va && ci[b] < ia)) ? 1 : 0;
    idx[row * k + rank] = ia;
    dist[row * k + rank] = __longlong_as_double(static_cast<long long>(va));
  }
}

// kNN graph of the first k of the K neighbours of every row, undirected (an edge if either end lists the other, as
// scipy's directed=False reads it): D = inf except the diagonal (0) and the edges. Both directions of an edge carry
// the same weight (D was bitwise symmetric), so the unordered stores race only between equal values.
__global__ void k_graph_fill(double* __restrict__ D, long long n) {
  const long long nn = n * n;
  for (long long q = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; q < nn; q += static_cast<long long>(gridDim.x) * blockDim.x)
    D[q] = (q / n == q % n) ? 0.0 : __longlong_as_double(0x7ff0000000000000LL);
}
__global__ void k_graph_edges(double* __restrict__ D, long long n, const int* __restrict__ idx, const double* __restrict__ dist, int K, int k) {
  const long long q = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (q >= n * k) return;
  const long long i = q / k, t = q % k, j = idx[i * K + t];
  if (i == j) return;
  const double w = dist[i * K + t];
  D[i * n + j] = w;
  D[j * n + i] = w;
}

// Blocked Floyd-Warshall, FW_B x FW_B blocks, round kb: phase 1 closes the diagonal block (kb, kb), phase 2 the blocks
// of row kb and column kb through it, phase 3 every other block (i, j) with min(D_ij, D_i,kb + D_kb,j). Within a block the
// in-place updates of phases 1 and 2 are safe: row / column kk of the pivot block does not change in step kk (D_kk,kk = 0).
// Out-of-range entries read as +inf and are never written.
constexpr int FW_B = 64;
constexpr int FW_THREADS = 256;   // 16 x 16 threads, 4 x 4 entries each
constexpr int FW_KC = 32;         // pivot columns per shared chunk of phase 3

__device__ __forceinline__ double fw_load(const double* D, long long n, long long i, long long j) {
  return (i < n && j < n) ? D[i * n + j] : __longlong_as_double(0x7ff0000000000000LL);
}

__global__ void __launch_bounds__(FW_THREADS) k_fw_diag(double* __restrict__ D, long long n, int kb) {
  __shared__ double P[FW_B][FW_B + 1];
  const long long o = static_cast<long long>(kb) * FW_B;
  for (int e = threadIdx.x; e < FW_B * FW_B; e += FW_THREADS) P[e / FW_B][e % FW_B] = fw_load(D, n, o + e / FW_B, o + e % FW_B);
  __syncthreads();
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  for (int kk = 0; kk < FW_B; ++kk) {
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        const int i = ty + 16 * u, j = tx + 16 * v;
        const double s = P[i][kk] + P[kk][j];
        if (s < P[i][j]) P[i][j] = s;
      }
    __syncthreads();
  }
  for (int e = threadIdx.x; e < FW_B * FW_B; e += FW_THREADS) {
    const long long i = o + e / FW_B, j = o + e % FW_B;
    if (i < n && j < n) D[i * n + j] = P[e / FW_B][e % FW_B];
  }
}

// blockIdx.y = 0: block (kb, other) of the pivot row; 1: block (other, kb) of the pivot column
constexpr int FW_CROSS_SMEM = 2 * FW_B * (FW_B + 1) * static_cast<int>(sizeof(double));   // dynamic: above the 48 KB static limit
__global__ void __launch_bounds__(FW_THREADS) k_fw_cross(double* __restrict__ D, long long n, int kb) {
  extern __shared__ __align__(16) double fw_smem[];
  double (*P)[FW_B + 1] = reinterpret_cast<double (*)[FW_B + 1]>(fw_smem);
  double (*C)[FW_B + 1] = P + FW_B;
  const int other = blockIdx.x < static_cast<unsigned>(kb) ? blockIdx.x : blockIdx.x + 1;
  const bool row = blockIdx.y == 0;
  const long long o = static_cast<long long>(kb) * FW_B;
  const long long ci = row ? o : static_cast<long long>(other) * FW_B, cj = row ? static_cast<long long>(other) * FW_B : o;
  for (int e = threadIdx.x; e < FW_B * FW_B; e += FW_THREADS) {
    P[e / FW_B][e % FW_B] = fw_load(D, n, o + e / FW_B, o + e % FW_B);
    C[e / FW_B][e % FW_B] = fw_load(D, n, ci + e / FW_B, cj + e % FW_B);
  }
  __syncthreads();
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  for (int kk = 0; kk < FW_B; ++kk) {
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        const int i = ty + 16 * u, j = tx + 16 * v;
        const double s = row ? P[i][kk] + C[kk][j] : C[i][kk] + P[kk][j];
        if (s < C[i][j]) C[i][j] = s;
      }
    __syncthreads();
  }
  for (int e = threadIdx.x; e < FW_B * FW_B; e += FW_THREADS) {
    const long long i = ci + e / FW_B, j = cj + e % FW_B;
    if (i < n && j < n) D[i * n + j] = C[e / FW_B][e % FW_B];
  }
}

__global__ void __launch_bounds__(FW_THREADS) k_fw_rest(double* __restrict__ D, long long n, int kb) {
  if (blockIdx.x == static_cast<unsigned>(kb) || blockIdx.y == static_cast<unsigned>(kb)) return;
  __shared__ double A[FW_B][FW_KC + 1], B[FW_KC][FW_B];
  const long long o = static_cast<long long>(kb) * FW_B, i0 = static_cast<long long>(blockIdx.y) * FW_B, j0 = static_cast<long long>(blockIdx.x) * FW_B;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  double acc[4][4];
#pragma unroll
  for (int u = 0; u < 4; ++u)
#pragma unroll
    for (int v = 0; v < 4; ++v) acc[u][v] = fw_load(D, n, i0 + ty + 16 * u, j0 + tx + 16 * v);
  for (int k0 = 0; k0 < FW_B; k0 += FW_KC) {
    __syncthreads();
    for (int e = threadIdx.x; e < FW_B * FW_KC; e += FW_THREADS) {
      A[e / FW_KC][e % FW_KC] = fw_load(D, n, i0 + e / FW_KC, o + k0 + e % FW_KC);
      B[e / FW_B][e % FW_B] = fw_load(D, n, o + k0 + e / FW_B, j0 + e % FW_B);
    }
    __syncthreads();
#pragma unroll 4
    for (int kk = 0; kk < FW_KC; ++kk) {
      double av[4], bv[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) { av[u] = A[ty + 16 * u][kk]; bv[u] = B[kk][tx + 16 * u]; }
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) acc[u][v] = fmin(acc[u][v], av[u] + bv[v]);
    }
  }
#pragma unroll
  for (int u = 0; u < 4; ++u)
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      const long long i = i0 + ty + 16 * u, j = j0 + tx + 16 * v;
      if (i < n && j < n) D[i * n + j] = acc[u][v];
    }
}

// largest finite entry (non-negative doubles order as their bit patterns: an integer max, order-independent)
__global__ void k_finite_max(const double* __restrict__ D, long long nn, unsigned long long* __restrict__ out) {
  unsigned long long m = 0ull;
  const unsigned long long inf = 0x7ff0000000000000ull;
  const unsigned long long* p = reinterpret_cast<const unsigned long long*>(D);
  for (long long q = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; q < nn; q += static_cast<long long>(gridDim.x) * blockDim.x) {
    const unsigned long long v = p[q];
    if (v < inf && v > m) m = v;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long x = __shfl_xor_sync(0xffffffffu, m, o);
    m = x > m ? x : m;
  }
  if ((threadIdx.x & 31) == 0) atomicMax(out, m);
}

// the unreachable rule of geodesic_distances: every entry above the largest finite one becomes twice that
__global__ void k_fill_unreachable(double* __restrict__ D, long long nn, const unsigned long long* __restrict__ fmax_bits) {
  const double fmax = __longlong_as_double(static_cast<long long>(*fmax_bits));
  for (long long q = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; q < nn; q += static_cast<long long>(gridDim.x) * blockDim.x)
    if (D[q] > fmax) D[q] = 2.0 * fmax;
}

}  // namespace jb
