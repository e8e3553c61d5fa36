// Kernels of the jb_pcaop handle (randomized PCA fit, jamie_b200/pca_fit.py randomized_fit_transform): the implicitly
// centred operand Xc = X - 1 mu^T applied to thin dense matrices, and the per-column statistics that give mu.
//
// Sparse X is held as CSR of X and CSR of X^T (= CSC of X), so ONE kernel, k_csr_dense, serves Xc B and Xc^T B:
//   Y[r, j] = sum_p val[p] * B[idx[p], j]  -  a[r] * v[j]
// The sum runs over the nonzeros of row r in index order, each fp32 x fp32 product exact in float64 and added in
// float64; the centring is the rank-1 term a[r] v[j] (a = 1, v = mu^T B for Xc B; a = mu, v = 1^T B for Xc^T B), also in
// float64, and the result is rounded to fp32 once. A row longer than PO_SEG nonzeros is cut into segments whose float64
// partials k_seg_finish adds in segment order. No floating-point atomics anywhere: the results are bit-reproducible.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

namespace jb {

constexpr int PO_SEG = 4096;          // nonzeros per work item: longer rows are split into segments
constexpr int PO_WARPS = 8;           // work items (one per warp) per 256-thread block of k_csr_dense
constexpr int PO_SLAB = 64;           // columns of B per warp pass (two per lane); gridDim.y = column slabs
constexpr int PO_STAT_SLABS = 64;     // row slabs of the dense column statistics / column reductions

// One unit of sparse work: nonzeros [begin, end) of row `row`. slot < 0: the whole row, finished in place; else the
// float64 partial of one segment, stored in part[slot].
struct PoItem {
  long long begin, end;
  int row, slot;
};
// A row that was split: its partials are part[first .. first + count), added in that order.
struct PoLong {
  int row, first, count;
};

__global__ void __launch_bounds__(PO_WARPS * 32)
k_csr_dense(const PoItem* __restrict__ items, long long n_items, const int* __restrict__ idx, const float* __restrict__ val,
            const float* __restrict__ B, int l, const double* __restrict__ a, const double* __restrict__ v,
            float* __restrict__ Y, double* __restrict__ part) {
  const int lane = threadIdx.x & 31;
  const long long w = static_cast<long long>(blockIdx.x) * PO_WARPS + (threadIdx.x >> 5);
  if (w >= n_items) return;
  const PoItem it = items[w];
  const int j0 = blockIdx.y * PO_SLAB + lane, j1 = j0 + 32;
  const bool ok0 = j0 < l, ok1 = j1 < l;
  double s0 = 0.0, s1 = 0.0;
  for (long long p0 = it.begin; p0 < it.end; p0 += 32) {
    // 32 nonzeros per round: lane q loads nonzero p0 + q (coalesced), then every lane walks them in order
    const int cnt = it.end - p0 < 32 ? static_cast<int>(it.end - p0) : 32;
    int my_c = 0;
    float my_x = 0.f;
    if (lane < cnt) { my_c = __ldg(idx + p0 + lane); my_x = __ldg(val + p0 + lane); }
    int q = 0;
    for (; q + 4 <= cnt; q += 4) {   // four independent row gathers in flight, added in index order
      float b0[4], b1[4], x[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int c = __shfl_sync(0xffffffffu, my_c, q + u);
        x[u] = __shfl_sync(0xffffffffu, my_x, q + u);
        const float* row = B + static_cast<size_t>(c) * l;
        b0[u] = ok0 ? __ldg(row + j0) : 0.f;
        b1[u] = ok1 ? __ldg(row + j1) : 0.f;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        s0 += static_cast<double>(x[u]) * static_cast<double>(b0[u]);
        s1 += static_cast<double>(x[u]) * static_cast<double>(b1[u]);
      }
    }
    for (; q < cnt; ++q) {
      const int c = __shfl_sync(0xffffffffu, my_c, q);
      const float x = __shfl_sync(0xffffffffu, my_x, q);
      const float* row = B + static_cast<size_t>(c) * l;
      if (ok0) s0 += static_cast<double>(x) * static_cast<double>(__ldg(row + j0));
      if (ok1) s1 += static_cast<double>(x) * static_cast<double>(__ldg(row + j1));
    }
  }
  if (it.slot >= 0) {
    double* o = part + static_cast<size_t>(it.slot) * l;
    if (ok0) o[j0] = s0;
    if (ok1) o[j1] = s1;
    return;
  }
  const double ar = a ? a[it.row] : 1.0;
  float* o = Y + static_cast<size_t>(it.row) * l;
  if (ok0) o[j0] = static_cast<float>(v ? s0 - ar * v[j0] : s0);
  if (ok1) o[j1] = static_cast<float>(v ? s1 - ar * v[j1] : s1);
}

// rows split into segments: Y[row, j] = sum of the segment partials in order - a[row] v[j]
__global__ void k_seg_finish(const PoLong* __restrict__ longs, int n_long, const double* __restrict__ part, int l,
                             const double* __restrict__ a, const double* __restrict__ v, float* __restrict__ Y) {
  const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= static_cast<long long>(n_long) * l) return;
  const PoLong L = longs[t / l];
  const int j = static_cast<int>(t % l);
  double s = 0.0;
  for (int q = 0; q < L.count; ++q) s += part[static_cast<size_t>(L.first + q) * l + j];
  if (v) s -= (a ? a[L.row] : 1.0) * v[j];
  Y[static_cast<size_t>(L.row) * l + j] = static_cast<float>(s);
}

// partial column sums over row slabs: part[slab][j] = sum_{k in slab} w[k] B[k, j] (w = NULL: weights 1), float64
__global__ void k_wcolsum(const float* __restrict__ B, long long K, int l, long long rows_per_slab, const double* __restrict__ w,
                          double* __restrict__ part) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= l) return;
  const long long k0 = blockIdx.y * rows_per_slab, k1 = k0 + rows_per_slab < K ? k0 + rows_per_slab : K;
  double s = 0.0;
  for (long long k = k0; k < k1; ++k) {
    const double b = static_cast<double>(B[k * l + j]);
    s += w ? w[k] * b : b;
  }
  part[static_cast<size_t>(blockIdx.y) * l + j] = s;
}

// partial centred sums of squares of a dense [n, d] matrix over row slabs: part[slab][c] = sum (x - mean[c])^2
__global__ void k_col_sqdev(const float* __restrict__ x, long long n, long long d, long long rows_per_slab,
                            const double* __restrict__ mean, double* __restrict__ part) {
  const long long c = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (c >= d) return;
  const long long r0 = blockIdx.y * rows_per_slab, r1 = r0 + rows_per_slab < n ? r0 + rows_per_slab : n;
  const double m = mean[c];
  double s = 0.0;
  for (long long r = r0; r < r1; ++r) {
    const double e = static_cast<double>(x[r * d + c]) - m;
    s += e * e;
  }
  part[static_cast<long long>(blockIdx.y) * d + c] = s;
}

// out[c] = (sum over the slabs in order of part[slab][c]) / div
__global__ void k_sum_parts(const double* __restrict__ part, int slabs, long long cols, double div, double* __restrict__ out) {
  const long long c = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  double s = 0.0;
  for (int q = 0; q < slabs; ++q) s += part[static_cast<size_t>(q) * cols + c];
  out[c] = s / div;
}

// per-column mean and variance (ddof 0) of a sparse matrix from its CSC rows: one warp per column, two passes over the
// nonzeros (lane-strided, then a fixed butterfly), the n - nnz_c zeros contributing mu^2 each to the second
__global__ void k_csc_stats(const long long* __restrict__ ptr, const float* __restrict__ val, long long d, long long n,
                            double* __restrict__ mean, double* __restrict__ var) {
  const int lane = threadIdx.x & 31;
  const long long c = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  if (c >= d) return;
  const long long b = ptr[c], e = ptr[c + 1];
  double s = 0.0;
  for (long long p = b + lane; p < e; p += 32) s += static_cast<double>(val[p]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const double mu = s / static_cast<double>(n);
  double q = 0.0;
  for (long long p = b + lane; p < e; p += 32) {
    const double t = static_cast<double>(val[p]) - mu;
    q += t * t;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  if (lane == 0) {
    mean[c] = mu;
    var[c] = (q + static_cast<double>(n - (e - b)) * mu * mu) / static_cast<double>(n);
  }
}

__global__ void k_f64_to_f32(const double* __restrict__ a, long long count, float* __restrict__ y) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < count) y[i] = static_cast<float>(a[i]);
}

}  // namespace jb
