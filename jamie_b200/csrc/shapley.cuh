// Shapley values by permutation walks (jb_shapley, jamie_b200/shapley.py). A walk goes from a background row b to the
// explained row x, adding the raw features in the order of a permutation pi. With a linear input map the network input
// changes by one rank-1 term per step, z_t = z_{t-1} + (x_j - b_j) w_j with j = pi_t, so the walk is a prefix sum built
// on the device from z_b, w and the raw rows. A step with x_j == b_j changes nothing and gets no chain row.
//
// A segment is one (explained row, background row) pair of a batch, g = x * nb + b. All segments of a batch follow the
// same permutation, so one block reads a w_j tile once for SHP_SG segments, and the blocks of one step chunk are adjacent
// in launch order so that they find the tile in L2.
#pragma once
#include <cuda_runtime.h>

namespace jb {

constexpr int SHP_TC = 128;   // steps per walk chunk; the chunking depends on d only, never on the batch
constexpr int SHP_SG = 16;    // segments per block of k_shap_walk
constexpr int SHP_CT = 128;   // network-input columns per block of k_shap_walk, one per thread

// cnt[g] = number of raw features where x and b differ (the segment's chain rows, for every permutation)
__global__ void k_shap_count(const double* __restrict__ X, const double* __restrict__ B, int d, int nb,
                             long long* __restrict__ cnt) {
  const long long g = blockIdx.x;
  const double* x = X + (g / nb) * d;
  const double* b = B + (g % nb) * d;
  long long c = 0;
  for (int j = threadIdx.x; j < d; j += blockDim.x) c += x[j] != b[j];
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  __shared__ long long part[32];
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    long long s = 0;
    for (int i = 0; i < static_cast<int>(blockDim.x >> 5); ++i) s += part[i];
    cnt[g] = s;
  }
}

// One step chunk q (blockIdx.y) of SHP_SG segments (blockIdx.x) on SHP_CT input columns (blockIdx.z), segments
// s0 + [0, S) of the call, permutation perm. w: dense [d, D] (w_col == NULL), else w_j = w[j] at column w_col[j].
//   EMIT = false: part[s][q][c] = the sum over the chunk's active steps of d_t w_{pi_t}[c] (float64, in step order) and,
//                 from column tile 0, ccnt[s][q] = the chunk's active steps.
//   EMIT = true : part[s][q][c] holds the chunk's start value (k_shap_chunk_start); the running sum in float64 is
//                 rounded once to fp32 per active step and written to out[coff[s][q] + rank, c], rank = the step's index
//                 among the chunk's active steps of the segment (the same in every column tile). Column tile 0 writes
//                 rowof[s][t] = that row, or -1 for an inactive step.
template <bool EMIT>
__global__ void __launch_bounds__(SHP_CT) k_shap_walk(const double* __restrict__ X, const double* __restrict__ B, int d,
                                                      int nb, long long s0, int S, const int* __restrict__ perm,
                                                      const double* __restrict__ w, const int* __restrict__ w_col, int D,
                                                      double* __restrict__ part, int* __restrict__ ccnt,
                                                      const int* __restrict__ coff, float* __restrict__ out, long long ldo,
                                                      int* __restrict__ rowof) {
  __shared__ double sd[SHP_SG][SHP_TC];   // d_t = x_j - b_j per segment and step
  __shared__ short srank[SHP_SG][SHP_TC];  // rank among the chunk's active steps, -1 inactive
  __shared__ int sj[SHP_TC];
  __shared__ unsigned smask[SHP_TC];       // bit s: the step is active in segment s
  const int Q = (d + SHP_TC - 1) / SHP_TC;
  const int sg = blockIdx.x * SHP_SG, q = blockIdx.y;
  const int t0 = q * SHP_TC;
  const int nt = d - t0 < SHP_TC ? d - t0 : SHP_TC;
  const int ns = S - sg < SHP_SG ? S - sg : SHP_SG;
  for (int t = threadIdx.x; t < SHP_TC; t += blockDim.x) sj[t] = t < nt ? perm[t0 + t] : 0;
  __syncthreads();
  for (int i = threadIdx.x; i < SHP_SG * SHP_TC; i += blockDim.x) {
    const int s = i / SHP_TC, t = i % SHP_TC;
    double v = 0.0;
    if (s < ns && t < nt) {
      const long long g = s0 + sg + s;
      const int j = sj[t];
      v = X[(g / nb) * d + j] - B[(g % nb) * d + j];
    }
    sd[s][t] = v;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int s = warp; s < SHP_SG; s += SHP_CT / 32) {
    int base = 0;
    for (int tb = 0; tb < SHP_TC; tb += 32) {
      const bool a = sd[s][tb + lane] != 0.0;
      const unsigned bal = __ballot_sync(0xffffffffu, a);
      srank[s][tb + lane] = static_cast<short>(a ? base + __popc(bal & ((1u << lane) - 1u)) : -1);
      base += __popc(bal);
    }
    if (!EMIT && blockIdx.z == 0 && lane == 0 && s < ns) ccnt[static_cast<long long>(sg + s) * Q + q] = base;
  }
  __syncthreads();
  for (int t = threadIdx.x; t < SHP_TC; t += blockDim.x) {
    unsigned m = 0;
    for (int s = 0; s < SHP_SG; ++s) m |= (srank[s][t] >= 0 ? 1u : 0u) << s;
    smask[t] = m;
  }
  __syncthreads();
  if (EMIT && blockIdx.z == 0) {
    for (int i = threadIdx.x; i < ns * SHP_TC; i += blockDim.x) {
      const int s = i / SHP_TC, t = i % SHP_TC;
      if (t >= nt) continue;
      const int rk = srank[s][t];
      rowof[static_cast<long long>(sg + s) * d + t0 + t] = rk < 0 ? -1 : coff[static_cast<long long>(sg + s) * Q + q] + rk;
    }
  }
  const int c = blockIdx.z * SHP_CT + threadIdx.x;
  if (c >= D) return;
  double acc[SHP_SG];
  int orow[SHP_SG];
#pragma unroll
  for (int s = 0; s < SHP_SG; ++s) {
    const long long sq = static_cast<long long>(sg + s) * Q + q;
    acc[s] = EMIT && s < ns ? part[sq * D + c] : 0.0;
    orow[s] = EMIT && s < ns ? coff[sq] : 0;
  }
  for (int t = 0; t < nt; ++t) {
    const unsigned m = smask[t];
    if (!m) continue;
    const int j = sj[t];
    const double wv = w_col ? (w_col[j] == c ? w[j] : 0.0) : w[static_cast<long long>(j) * D + c];
#pragma unroll
    for (int s = 0; s < SHP_SG; ++s) {
      if (m >> s & 1u) {
        acc[s] += sd[s][t] * wv;
        if (EMIT) out[static_cast<long long>(orow[s] + srank[s][t]) * ldo + c] = static_cast<float>(acc[s]);
      }
    }
  }
  if (!EMIT) {
#pragma unroll
    for (int s = 0; s < SHP_SG; ++s)
      if (s < ns) part[(static_cast<long long>(sg + s) * Q + q) * D + c] = acc[s];
  }
}

// Chunk start values and row offsets of segment s (one block per segment): part[s][q][:] becomes
// z_b + part[s][0] + ... + part[s][q - 1] (a left fold in chunk order), coff[s][q] = first[s] + ccnt[s][0 .. q - 1].
// Zb [nb, D] float64: the preprocessed background rows. first[s]: the segment's first row in the batch.
__global__ void k_shap_chunk_start(const double* __restrict__ Zb, int D, int nb, long long s0, int Q,
                                   double* __restrict__ part, const int* __restrict__ ccnt, const int* __restrict__ first,
                                   int* __restrict__ coff) {
  const long long s = blockIdx.x;
  const double* zb = Zb + ((s0 + s) % nb) * D;
  double* p = part + s * Q * D;
  for (int c = threadIdx.x; c < D; c += blockDim.x) {
    double run = zb[c];
    for (int q = 0; q < Q; ++q) {
      const double v = p[static_cast<long long>(q) * D + c];
      p[static_cast<long long>(q) * D + c] = run;
      run += v;
    }
  }
  if (threadIdx.x == 0) {
    int r = first[s];
    for (int q = 0; q < Q; ++q) {
      coff[s * Q + q] = r;
      r += ccnt[s * Q + q];
    }
  }
}

// The value of output o of chain / inverse row y: map_kind 1 (PCA inverse, restricted to the selected columns) reads
// column o; kinds 0 / 2 read column ocol[o] of the chain's output, kind 2 as fp32(y * aff_scale + aff_shift).
struct ShapOut {
  const float* Y;
  long long ldy;
  int map_kind;
  const int* ocol;
  const double* sc;
  const double* sh;
  __device__ float at(long long r, int o) const {
    if (map_kind == 1) return Y[r * ldy + o];
    const int c = ocol[o];
    const float v = Y[r * ldy + c];
    return map_kind == 2 ? static_cast<float>(static_cast<double>(v) * sc[c] + sh[c]) : v;
  }
};

// f(b) of background rows b0 + [0, rows): fB[b][o] (fp32, the mapped output) and base[o] += f(b)[o] in row order.
__global__ void k_shap_base(ShapOut Y, int rows, long long b0, int n_out, float* __restrict__ fB, double* __restrict__ base) {
  const int o = blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= n_out) return;
  double acc = base[o];
  for (int i = 0; i < rows; ++i) {
    const float v = Y.at(i, o);
    fB[(b0 + i) * n_out + o] = v;
    acc += static_cast<double>(v);
  }
  base[o] = acc;
}

// Difference fold of one batch (segments s0 + [0, S) of the call): for explained row x = s0 / nb + blockIdx.x, step t
// and output o, phi[x, perm[t], o] += y(row of step t) - y(the segment's previous row, or f(b) at its first row), one
// term at a time over the batch's segments of x in background-row order, in float64. Each accumulator thus receives its
// terms in (permutation, background row) order whatever the batches: no atomics.
__global__ void k_shap_fold(ShapOut Y, const float* __restrict__ fB, const int* __restrict__ rowof,
                            const int* __restrict__ first, const int* __restrict__ perm, int d, int nb, long long s0, int S,
                            int n_out, double* __restrict__ phi) {
  const int o = blockIdx.z * 32 + threadIdx.x, t = blockIdx.y * 8 + threadIdx.y;
  if (o >= n_out || t >= d) return;
  const long long x = s0 / nb + blockIdx.x;
  const long long g_lo = x * nb > s0 ? x * nb : s0;
  const long long g_hi = (x + 1) * nb < s0 + S ? (x + 1) * nb : s0 + S;
  double* acc = phi + (x * d + perm[t]) * n_out + o;
  double a = *acc;
  for (long long g = g_lo; g < g_hi; ++g) {
    const long long s = g - s0;
    const int r = rowof[s * d + t];
    if (r < 0) continue;
    const double y = static_cast<double>(Y.at(r, o));
    const double prev = static_cast<double>(r == first[s] ? fB[(g % nb) * n_out + o] : Y.at(r - 1, o));
    a += y - prev;
  }
  *acc = a;
}

// rows [rows, ld] fp32 = Z[r0 + i, :D] (float64 rows, one rounding)
__global__ void k_shap_rows_f32(const double* __restrict__ Z, int D, long long r0, float* __restrict__ out, long long ld) {
  const long long i = blockIdx.x;
  for (int c = threadIdx.x; c < D; c += blockDim.x) out[i * ld + c] = static_cast<float>(Z[(r0 + i) * D + c]);
}

}  // namespace jb
