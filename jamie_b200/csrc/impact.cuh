// Batched feature ablation (jb_feature_impact, SURVEY.md 3.2): the reference's notebooks replace one raw input feature,
// rerun the imputation and score it, once per feature. With a linear input map an ablation of raw column j changes the
// network's input by a rank-1 term, Z(j) = Z + dz[:, j] w_j^T, so a batch of ablated inputs is built on the device from
// Z, w and dz alone, and only per-feature sums leave it.
#pragma once
#include <cuda_runtime.h>

namespace jb {

// Rows per partial sum of k_impact_moments. Row ranges start at multiples of it, so the slabs sit at fixed absolute rows.
constexpr int IMP_SLAB = 32;

// out[s * R + i, :] = Z[r0 + i, :] for slot s = 0 (the unablated rows), and for slot s >= 1 (feature j = j0 + s - 1)
//   dense w : Z[r, c] + dz[s - 1][r] * w[j, c]
//   w_col   : Z[r, c] + (c == w_col[j] ? dz[s - 1][r] * w[j] : 0)
// in float64, rounded once to fp32. dz holds the batch's columns, [a][n].
__global__ void k_ablate_rows(const double* __restrict__ Z, int D, long long n, long long r0, int R, int j0,
                              const double* __restrict__ dz, const double* __restrict__ w, const int* __restrict__ w_col,
                              float* __restrict__ out, long long ldo) {
  const long long b = blockIdx.x;
  const int s = static_cast<int>(b / R), i = static_cast<int>(b % R);
  const long long r = r0 + i;
  const double* z = Z + r * D;
  float* o = out + b * ldo;
  if (s == 0) {
    for (int c = threadIdx.x; c < D; c += blockDim.x) o[c] = static_cast<float>(z[c]);
    return;
  }
  const int j = j0 + s - 1;
  const double dv = dz[static_cast<long long>(s - 1) * n + r];
  if (w_col) {
    const int cj = w_col[j];
    const double add = dv * w[j];
    for (int c = threadIdx.x; c < D; c += blockDim.x) o[c] = static_cast<float>(c == cj ? z[c] + add : z[c]);
  } else {
    const double* wj = w + static_cast<long long>(j) * D;
    for (int c = threadIdx.x; c < D; c += blockDim.x) o[c] = static_cast<float>(z[c] + dv * wj[c]);
  }
}

// Per (slot, output column): acc[s][c] += {sum y, sum y^2, sum y t, sum |y - y0|} over the rows [r0, r0 + R) of the
// batch's predictions P ([(a + 1) R, ldp], slot 0 = the unablated y0), one partial per IMP_SLAB rows added in row order.
// Feature batches and row ranges thus give the same left fold over the slabs whatever their sizes: no atomics.
// aff_scale / aff_shift (or NULL): the output map y = fp32(v * scale[c] + shift[c]) of a side standardised per column.
// T: the target [n, d] (or NULL: t = 0). tacc (or NULL): {sum t, sum t^2} per column, accumulated by slot 0.
__global__ void k_impact_moments(const float* __restrict__ P, long long ldp, int R, long long r0, int d,
                                 const float* __restrict__ T, const double* __restrict__ aff_scale,
                                 const double* __restrict__ aff_shift, double* __restrict__ acc, double* __restrict__ tacc) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= d) return;
  const int s = blockIdx.y;
  const float* p = P + static_cast<long long>(s) * R * ldp + c;
  const float* p0 = P + c;
  const double sc = aff_scale ? aff_scale[c] : 1.0, sh = aff_shift ? aff_shift[c] : 0.0;
  auto val = [&](float v) {
    return aff_scale ? static_cast<double>(static_cast<float>(static_cast<double>(v) * sc + sh)) : static_cast<double>(v);
  };
  double* a = acc + (static_cast<long long>(s) * d + c) * 4;
  double a0 = a[0], a1 = a[1], a2 = a[2], a3 = a[3];
  const bool do_t = tacc && s == 0 && T;
  double t0 = do_t ? tacc[2 * c] : 0.0, t1 = do_t ? tacc[2 * c + 1] : 0.0;
  for (int i0 = 0; i0 < R; i0 += IMP_SLAB) {
    const int i1 = i0 + IMP_SLAB < R ? i0 + IMP_SLAB : R;
    double q0 = 0, q1 = 0, q2 = 0, q3 = 0, u0 = 0, u1 = 0;
    for (int i = i0; i < i1; ++i) {
      const double y = val(p[static_cast<long long>(i) * ldp]);
      const double y0 = val(p0[static_cast<long long>(i) * ldp]);
      const double t = T ? static_cast<double>(T[(r0 + i) * d + c]) : 0.0;
      q0 += y; q1 += y * y; q2 += y * t; q3 += fabs(y - y0);
      u0 += t; u1 += t * t;
    }
    a0 += q0; a1 += q1; a2 += q2; a3 += q3;
    t0 += u0; t1 += u1;
  }
  a[0] = a0; a[1] = a1; a[2] = a2; a[3] = a3;
  if (do_t) { tacc[2 * c] = t0; tacc[2 * c + 1] = t1; }
}

}  // namespace jb
