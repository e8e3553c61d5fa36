// The whole JAMIE training step as ONE persistent cooperative kernel (round 2).
//
// Round 1 ran the step as a CUDA graph of 31 kernels, 29 of them on the critical path; its own trace showed that ~8 of
// every 12-14 us GEMM link were launch latency, prologue (barrier init, TMEM allocation, tensor-map fetch), pipeline fill
// and epilogue, and that the BatchNorm / latent / optimizer kernels were latency chains of a few microseconds each
// (profiles/README.md, round 1). Here one CTA per SM (148 x 512 threads) stays resident for any number of optimizer
// steps and walks the phases of the step, separated by grid barriers (ptx.cuh: grid_barrier, ~1.2 us): the operand ring,
// the mbarriers, the TMEM allocation and the tensor maps live for the whole kernel, the GEMM phases run the fp16-split
// tcgen05 pipeline of hgemm.cuh (4 B per operand element instead of round 1's 8), and the element-wise phases use all
// 16 warps of all SMs.
//
// Phases of one step (StepPhase). "slab" = a CTA owns 16 feature columns and all B rows, so BatchNorm statistics are
// CTA-local; "row" = one warp per (modality, batch row). Split-K partial sums of a GEMM are reduced by the phase that
// consumes them (fixed order: deterministic, no atomics anywhere).
//   GATHER   rows: x = data[idx] + fp16 operand planes; CTA strips: P / F blocks (row sums + normalise + transposes)
//   ENC1     GEMM  y1 = x W1^T + b1                        BN1  slab: batch stats, LeakyReLU, dropout -> h1 planes
//   ENC2     GEMM  y2 = h1 W2^T + b2 (split-K)             BN2  slab -> h2 planes
//   HEADS    GEMM  [mu | logvar] = h2 Wmv^T + bmv (split-K)
//   REPARAM  elements: eps (Philox or injected), z         COMBINE rows: sigma-weighted combine over the nonzeros of
//            the correspondence rows (+ latent loss partials when F is absent)     LATLOSS rows: planes of c with their
//            dynamic scale (+ the F loss partials when F is present)
//   DEC1..3  GEMMs + BN3, BN4 slabs                         REC  slab: reconstruction loss, d xhat planes, bias grad
//   DG5, DG4, DG3 dgrad GEMMs + BNB4, BNB3 backward slabs   LATBC, LATBZ rows: latent backward (KL with the reference's
//            logvar quirk, "CosSim", F loss, combine, reparameterisation) -> d[mu | logvar] planes
//   LATFIN   d[mu | logvar] planes with their dynamic scale; loss scalars, d sigma, head bias gradients
//   DGH      dgrad GEMM of the heads
//   BNB2, DG2, BNB1                                         WGRAD all 12 weight gradients (3-pass, 128 x 256 tiles)
//   NORM     sum g^2 partials                               ADAM  clip + Adam over the flat buffer + fp16 weight planes
// The backward pass carries the loss scale `gs` (a power of two): d xhat and the latent loss gradients are multiplied by
// it, every write into the gradient buffer divides it out (exactly), so small gradients stay in fp16's normal range.
#pragma once
#include "hgemm.cuh"
#include "kernels.cuh"

namespace jb {

// Loads of data written by OTHER CTAs earlier in the same launch. The grid barrier's gpu-scope acquire fence invalidates
// the SM's L1 (CCTL.IVALL), so after the barrier plain loads are coherent. The first version used __ldcg here, which
// compiles to LDG.E.STRONG.GPU: measured 1.65 us for eight independent L2 hits per thread (~234 cycles each: issued one
// after the other) instead of one latency for all eight.
template <class T> __device__ __forceinline__ T sk_ld(const T* p) { return *p; }
constexpr int SK_THREADS = 512;
constexpr int SK_WARPS = SK_THREADS / 32;
constexpr int SK_MAX_CTAS = 160;

enum StepPhase : int {
  PH_GATHER = 0, PH_ENC1, PH_BN1, PH_ENC2, PH_BN2, PH_HEADS, PH_REPARAM, PH_COMBINE, PH_LATLOSS, PH_DEC1, PH_BN3, PH_DEC2,
  PH_BN4, PH_DEC3, PH_REC, PH_DG5, PH_BNB4, PH_DG4, PH_BNB3, PH_DG3, PH_LATBC, PH_LATBZ, PH_LATFIN, PH_DGH, PH_BNB2, PH_DG2, PH_BNB1,
  PH_WGRAD, PH_NORM, PH_ADAM, PH_COUNT
};
// index of a GEMM phase in StepCtx::gph, or -1
__host__ __device__ inline int gemm_index(int ph) {
  switch (ph) {
    case PH_ENC1: return 0; case PH_ENC2: return 1; case PH_HEADS: return 2; case PH_DEC1: return 3; case PH_DEC2: return 4;
    case PH_DEC3: return 5; case PH_DG5: return 6; case PH_DG4: return 7; case PH_DG3: return 8; case PH_DGH: return 9;
    case PH_DG2: return 10; case PH_WGRAD: return 11; default: return -1;
  }
}
constexpr int SK_NUM_GEMM = 12;

struct Parts {       // a GEMM output as split-K partial sums: element e of partial p at ptr[p * stride + e]
  float* ptr; long long stride; int n;
};
__device__ __forceinline__ float ld_parts(const Parts& q, long long e) {
  float s = sk_ld(q.ptr + e);
  for (int p = 1; p < q.n; ++p) s += sk_ld(q.ptr + p * q.stride + e);
  return s;
}

struct BnLayer {     // one BatchNorm(+LeakyReLU+Dropout) layer of one modality, forward and backward views; one pitch
  Parts Y;                         // pre-BN Linear output (reduced in place into partial 0 by the forward slab)
  __half *Hh, *Hl;                 // post-dropout activation, operand planes
  const float *gamma, *beta;
  float *mean, *invstd, *var, *run_mean, *run_var;   // var: biased batch variance (fused path)
  const unsigned char* mask;       // injected keep mask [B, N] or null
  Parts dH;                        // gradient wrt the layer output (dgrad result)
  __half *dYh, *dYl;               // gradient wrt the pre-BN output, operand planes
  float *dgamma, *dbeta, *dbias;
  const float* gdyn;               // extra dynamic factor of the parameter-gradient writes (encoder layers: dyn[1]) or null
  int N, ld;
  int lcw;                         // log2 of the columns per slab item
  unsigned layer_id;
};

struct ModCtx {      // per modality
  const float* data; long long ld_data;
  const float* stage[2];           // host-batch steps: the two H2D landing buffers
  const int* idx;                  // plan [nsteps][B]
  float* x; __half *xh, *xl;       // gathered rows [B, ldD] + planes
  Parts mulv;                      // heads output [B, ldmv]: mu | logvar
  float *eps, *z, *c, *S, *g, *den, *rs;   // latent [B, LP] / [B]
  const float* inj_eps;
  __half *ch, *cl;                 // planes of c
  Parts dc;                        // decoder dgrad wrt c [B, LP]
  float* dmulv; __half *dmh, *dml; // gradient wrt the heads output + planes
  Parts xhat;                      // reconstruction [B, ldD]
  __half *dxh, *dxl;               // d loss / d xhat planes
  float* db5;                      // bias gradient of the last decoder Linear
  float* rec_part;                 // [rec_items] partial sums of squares (one per slab item of the REC phase)
  int rec_items, rec_lcw;
  float* dbias_heads;              // [2L]
  int D, ldD;
};

struct StepCtx {
  int B, L, LP, ldmv;
  ModCtx m[2];
  BnLayer bn[4][2];                // enc1, enc2, dec1, dec2
  // correspondence blocks
  const float *p_diag, *p_dense, *f_dense; long long pn1;
  float *corr, *corr_t, *fblk, *fblk_t;
  int2* corr_hint;                 // diagonal priors: per row of corr (then corr^T) {number of nonzeros, column of the first}; else null
  float pf_ratio;
  int f_present;
  // latent scratch
  float* lat_r; float* rowpart;
  int cosine;                      // dist_method == 'cosine' (jamie/jamie.py:485-494); 0: euclidean
  float* lat_coef;                 // cosine: per row [i][row] {a_zz, a_x, a_cc, -}: d loss / dz = a_zz z + a_x c, d loss / dc = a_x z + a_cc c
  // dynamic power-of-two operand scales (fp16 range): per-CTA maxima of |c| and |d mulv|, and the published inverse
  // scales dyn[0] = 1 / s_c (c planes hold s_c c), dyn[1] = 1 / s_b (d mulv planes and everything downstream of them in
  // the encoder backward hold s_b times the loss-scaled gradient). Both are exactly 1 unless a value leaves fp16's range.
  float *cmax_part, *dmax_part, *dyn;
  // parameters / optimizer
  float *theta, *grad, *adam_m, *adam_v; __half *theta_hi, *theta_lo;
  long long n_flat;
  const float* sigma; float* dsigma;
  double* norm_part;               // [SK_MAX_CTAS]
  // clip norm without the NORM sweep (launches that contain every weight-gradient GEMM and ADAM): the weight-gradient
  // epilogues leave per-warp sums of squares in norm_tile [n_norm_tile]; the gradients of the small tensors (biases,
  // BatchNorm affine, sigma: norm_rng (offset, length) pairs) are summed by warps without a GEMM role during WGRAD into
  // norm_small [4 ncta]
  float *norm_tile, *norm_small;
  int n_norm_tile, n_norm_rng;
  int norm_rng[32][2];
  // plan / control / outputs
  const float* plan_kl; float* out_loss; Ctl* ctl;
  StepConsts sc;
  float gs, inv_gs;                // loss scale of the backward pass and its inverse
  int merge_latent;                // no F: LATLOSS / LATFIN folded into COMBINE / LATBZ / the DEC1 and DGH phases (optimistic operand scales)
  int eps_early;                   // the reparameterisation noise is drawn during ENC1 (heads tail fused)
  // in-kernel data-parallel exchange (sk_exchange); xworld <= 1: off
  float* xg[8]; unsigned int* xf[8]; int xrank, xworld, xdbg;   // xdbg: timing experiments (JB_XCHG_DBG bit 0: no sweep, bit 1: no cross-GPU barriers)
  int xfence;                      // 1: every exchange fence at system scope (JB_XCHG_FENCE=sys); 0: see fence_light
  long long x_adam0;               // optimizer step count when the exchange was configured (epoch 0 of the flags)
  float* xmc;                      // NVSwitch multicast address of the gradient buffers (NULL: peer loads / stores)
  unsigned long long phase_mask;   // bit ph set: the phase runs (fused layers drop the BatchNorm / REC / REPARAM phases)
  // GEMM tables
  HgPhase gph[SK_NUM_GEMM];
};
// The whole description of a step travels as ONE kernel parameter (constant bank: every phase begins by reading its
// pointers and sizes, and loads from global memory would each cost an L2 round trip after every grid barrier, because
// the barrier's acquire invalidates L1). The tensor maps inside are used by TMA straight from parameter space.
constexpr int SK_MAX_PROBS = 36;
struct StepParams {
  StepCtx cx;
  HgProblem probs[SK_MAX_PROBS];
};
static_assert(sizeof(StepParams) <= 32000, "kernel parameter space");

struct StepVars {    // per-step scalars (one copy per CTA in shared memory)
  long long row;
  float kl_base, kl_coef, step_size, inv_bc2_sqrt;
  uint2 key;
  int inject, accum, host_slot;
};

// ------------------------------------------------------------------------------------------------ helpers
__device__ __forceinline__ void st_h4(__half* p, float a, float b, float c, float d, bool lo_of = false) { (void)lo_of;
  const __half2 u = h2_sat(a, b), v = h2_sat(c, d);
  uint2 w;
  w.x = *reinterpret_cast<const uint32_t*>(&u); w.y = *reinterpret_cast<const uint32_t*>(&v);
  *reinterpret_cast<uint2*>(p) = w;
}
// split four values into the hi / lo planes with two 8-byte stores
__device__ __forceinline__ void split4_store(__half* hi, __half* lo, float a, float b, float c, float d) {
  const __half ha = h_sat(a), hb = h_sat(b), hc = h_sat(c), hd = h_sat(d);
  const __half2 h01 = __halves2half2(ha, hb), h23 = __halves2half2(hc, hd);
  const __half2 l01 = h2_sat((a - __half2float(ha)) * HG_LO_SCALE, (b - __half2float(hb)) * HG_LO_SCALE);
  const __half2 l23 = h2_sat((c - __half2float(hc)) * HG_LO_SCALE, (d - __half2float(hd)) * HG_LO_SCALE);
  uint2 wh, wl;
  wh.x = *reinterpret_cast<const uint32_t*>(&h01); wh.y = *reinterpret_cast<const uint32_t*>(&h23);
  wl.x = *reinterpret_cast<const uint32_t*>(&l01); wl.y = *reinterpret_cast<const uint32_t*>(&l23);
  *reinterpret_cast<uint2*>(hi) = wh;
  *reinterpret_cast<uint2*>(lo) = wl;
}

// ------------------------------------------------------------------------------------------------ GATHER
__device__ __forceinline__ float sk_p_entry(const StepCtx& cx, int i0, int i1) {
  if (cx.p_dense) return __ldg(cx.p_dense + static_cast<long long>(i0) * cx.pn1 + i1);
  if (cx.p_diag) return i0 == i1 ? __ldg(cx.p_diag + i0) : 0.f;
  return 0.f;
}
// P / F blocks of the step (jamie/jamie.py:586-604): one warp per block row: row sums, then the normalised row of corr
// (coalesced) and the same values into column `a` of the transposed blocks (the entries are recomputed in the second
// pass instead of being held in registers: rolled loops, small code). fblk / fblk_t only exist with a dense F.
__device__ __forceinline__ void sk_corr_row(const StepCtx& cx, long long base, int a, int lane) {
  const int B = cx.B;
  const int i0 = cx.m[0].idx[base + a];
  const int* __restrict__ idx1 = cx.m[1].idx + base;
  const float* __restrict__ pd = cx.p_dense != nullptr ? cx.p_dense + static_cast<long long>(i0) * cx.pn1 : nullptr;
  const float* __restrict__ fd = cx.f_dense != nullptr ? cx.f_dense + static_cast<long long>(i0) * cx.pn1 : nullptr;
  const float diag = (pd == nullptr && cx.p_diag != nullptr) ? __ldg(cx.p_diag + i0) : 0.f;   // P = diag(m): entry m[i0] where i1 == i0
  float p = 0.f, f = 0.f;
#pragma unroll 1
  for (int b0 = lane; b0 < B; b0 += 128) {     // four entries in flight per lane
    int i1[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) i1[u] = b0 + 32 * u < B ? idx1[b0 + 32 * u] : -1;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (i1[u] < 0) continue;
      p += pd != nullptr ? __ldg(pd + i1[u]) : (i1[u] == i0 ? diag : 0.f);
      if (fd != nullptr) f += __ldg(fd + i1[u]);
    }
  }
  p = warp_sum(p); f = warp_sum(f);
  const float rp = p == 0.f ? 1.f : p, rf = f == 0.f ? 1.f : f;
  const float pfr = cx.pf_ratio;
  float* crow = cx.corr + static_cast<long long>(a) * B;
  float* frow = cx.fblk + static_cast<long long>(a) * B;
#pragma unroll 1
  for (int b0 = lane; b0 < B; b0 += 128) {
    int i1[4];
    float pv[4], fv[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) i1[u] = b0 + 32 * u < B ? idx1[b0 + 32 * u] : -1;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      pv[u] = 0.f; fv[u] = 0.f;
      if (i1[u] < 0) continue;
      pv[u] = pd != nullptr ? __ldg(pd + i1[u]) : (i1[u] == i0 ? diag : 0.f);
      if (fd != nullptr) fv[u] = __ldg(fd + i1[u]);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (i1[u] < 0) continue;
      const int b = b0 + 32 * u;
      const float fvn = fv[u] / rf;
      const float c = pfr * (pv[u] / rp) + (1.f - pfr) * fvn;
      crow[b] = c;
      cx.corr_t[static_cast<long long>(b) * B + a] = c;
      if (fd != nullptr) { frow[b] = fvn; cx.fblk_t[static_cast<long long>(b) * B + a] = fvn; }
    }
  }
}
// P = diag(m), no F (the identity / partially matched priors of every large run): corr[a][b] = pf m[i0[a]] [i1[b] == i0[a]] /
// rowsum_a with rowsum_a = m[i0[a]] * #{b': i1[b'] == i0[a]} (1 if that is 0). A matching pair (a, b) shares the cell id,
// so the row sum of a is also known from b's side: one warp writes row a of corr (it = a) or row b of corr^T (it = B + b),
// both coalesced; the general path above scatters the transposed entries 4 bytes at a time (measured: GATHER 20 us).
__device__ __forceinline__ void sk_corr_row_diag(const StepCtx& cx, long long base, int it, int lane) {
  const int B = cx.B;
  const bool tr = it >= B;
  const int a = tr ? it - B : it;
  const int* __restrict__ idx_self = cx.m[tr ? 1 : 0].idx + base;    // the cell of this row
  const int* __restrict__ idx_other = cx.m[tr ? 0 : 1].idx + base;   // the cells along the row
  const int* __restrict__ idx1 = cx.m[1].idx + base;
  const int cell = idx_self[a];
  const float diag = __ldg(cx.p_diag + cell);
  int cnt = 0;
#pragma unroll 1
  for (int b0 = lane; b0 < B; b0 += 128) {
    int v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = b0 + 32 * u < B ? idx1[b0 + 32 * u] : -1;
#pragma unroll
    for (int u = 0; u < 4; ++u) cnt += v[u] == cell ? 1 : 0;
  }
  cnt = __reduce_add_sync(0xffffffffu, cnt);
  float p = 0.f;
  for (int k = 0; k < cnt; ++k) p += diag;   // the same additions as the general path's row sum (cnt is 0 or 1 in practice)
  const float rp = p == 0.f ? 1.f : p;
  const float val = cx.pf_ratio * (diag / rp) + (1.f - cx.pf_ratio) * 0.f;
  float* row = (tr ? cx.corr_t : cx.corr) + static_cast<long long>(a) * B;
  int nn = 0, first = B;   // nonzeros along the row and the column of the first one (the consumers' shortcut, sk_row_times)
#pragma unroll 1
  for (int b0 = lane; b0 < B; b0 += 128) {
    int v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = b0 + 32 * u < B ? idx_other[b0 + 32 * u] : -1;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const bool hit = v[u] == cell;
      if (b0 + 32 * u < B) row[b0 + 32 * u] = hit ? val : 0.f;
      if (hit) { ++nn; first = min(first, b0 + 32 * u); }
    }
  }
  nn = __reduce_add_sync(0xffffffffu, nn);
  first = __reduce_min_sync(0xffffffffu, first);
  if (lane == 0 && cx.corr_hint != nullptr) cx.corr_hint[it] = val != 0.f ? make_int2(nn, first) : make_int2(0, 0);
}
// x_i[b, :] = data_i[idx_i[row][b], :] (jamie/jamie.py:583) + operand planes; one warp per (modality, row)
__device__ __forceinline__ void sk_gather_row(const StepCtx& cx, const StepVars& sv, int use_stage, int it, int lane) {
  const int B = cx.B;
  const int i = it / B, b = it - i * B;
  const ModCtx& M = cx.m[i];
  const float* s;
  if (use_stage) s = M.stage[sv.host_slot != 0 ? 1 : 0] + static_cast<long long>(b) * M.ldD;
  else s = M.data + static_cast<long long>(M.idx[sv.row * B + b]) * M.ld_data;
  const long long o = static_cast<long long>(b) * M.ldD;
  float* d = M.x + o;
  __half* dh = M.xh + o;
  __half* dl = M.xl + o;
  const int D = M.D;
  int j0 = 0;
  if ((reinterpret_cast<uintptr_t>(s) & 15) == 0) {
    const int nv = D >> 2;
    for (int j = lane; j < nv; j += 128) {      // four 16-byte loads in flight per lane
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (j + 32 * u < nv) v[u] = __ldg(reinterpret_cast<const float4*>(s) + j + 32 * u);
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (j + 32 * u < nv) {
          reinterpret_cast<float4*>(d)[j + 32 * u] = v[u];
          split4_store(dh + 4 * (j + 32 * u), dl + 4 * (j + 32 * u), v[u].x, v[u].y, v[u].z, v[u].w);
        }
    }
    j0 = nv << 2;
  }
  for (int j = j0 + lane; j < D; j += 32) {
    const float v = __ldg(s + j);
    d[j] = v;
    h_split(v, dh[j], dl[j]);
  }
}

// ------------------------------------------------------------------------------------------------ column slabs
// A CTA item owns cw = 2^lcw feature columns (16 at the headline widths, 8 where that would leave half the grid idle)
// and all B rows, so BatchNorm statistics are CTA-local. Thread t has column t & (cw - 1) and row slot t >> lcw.
// The slab is staged in shared memory (the GEMM operand ring is idle in these phases) and walked with ROLLED loops:
// the first version kept the column in registers with everything unrolled, and ncu showed the phases bound by
// instruction fetch (stall_no_instruction the top reason: a 400 KB kernel whose phase bodies run once per step).
// Only the global loads are unrolled (8 rows in flight per thread).
constexpr int SK_UNR = 8;

// sums a, b over all threads of the CTA that share a column (fixed order), broadcast. All 512 threads must call.
__device__ __noinline__ void sk_colsum2(float& a, float& b, float* sh, int lcw, int warp, int lane) {
  const int cw = 1 << lcw;
  for (int o = 16; o >= cw; o >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, o);
    b += __shfl_xor_sync(0xffffffffu, b, o);
  }
  if (lane < cw) { sh[warp * 32 + lane] = a; sh[512 + warp * 32 + lane] = b; }
  __syncthreads();
  if (warp == 0 && lane < cw) {
    float x = 0.f, y = 0.f;
#pragma unroll
    for (int w = 0; w < SK_WARPS; ++w) { x += sh[w * 32 + lane]; y += sh[512 + w * 32 + lane]; }
    sh[1024 + lane] = x; sh[1056 + lane] = y;
  }
  __syncthreads();
  a = sh[1024 + (lane & (cw - 1))]; b = sh[1056 + (lane & (cw - 1))];
  __syncthreads();
}
__device__ __noinline__ uint4 sk_rand4(uint2 key, unsigned layer_id, int col, int rgroup) { return rand4(key, layer_id, col, rgroup); }

// Linear output Y [B, N] -> BatchNorm1d (batch statistics, two-pass variance) -> LeakyReLU(0.01) -> Dropout(p)
// (jamie/model.py:151-154 and siblings) -> fp16 operand planes of the next GEMM. Also reduces the split-K partials of Y
// into partial 0 (the backward slab reads one array) and updates the running statistics.
// Code-size rules of the slab phases (the step kernel is bound by INSTRUCTION FETCH: a phase body runs once per step, its
// code comes from L2 at ~234 cycles per 128-byte line): 32-bit element offsets, clamped indices instead of per-load
// branches, rolled loops everywhere except the 8 independent loads of a round.
__device__ __forceinline__ void sk_bn_fwd_item(const BnLayer& Lr, const StepCtx& cx, const StepVars& sv, int cb, float* slab, float* sh,
                                            int tid, int warp, int lane, long long* stamp = nullptr) {
  if (stamp != nullptr && tid == 0) stamp[0] = clock64();
  const int B = cx.B;
  const int lcw = Lr.lcw, cw = 1 << lcw, slots = SK_THREADS >> lcw;
  const int cl = tid & (cw - 1), slot = tid >> lcw;
  const int N = Lr.N, ld = Lr.ld;
  const int c = (cb << lcw) + cl;
  const bool cok = c < N;
  const int cc = cok ? c : N - 1;
  float* const Y = Lr.Y.ptr + cc;
  const int nparts = Lr.Y.n;
  const long long pstride = Lr.Y.stride;
  float* const sl = slab + cl;
  float s = 0.f, dummy = 0.f;
#pragma unroll 1
  for (int r0 = slot; r0 < B; r0 += SK_UNR * slots) {
    float v[SK_UNR];
#pragma unroll
    for (int k = 0; k < SK_UNR; ++k) v[k] = sk_ld(Y + min(r0 + k * slots, B - 1) * ld);
#pragma unroll 1
    for (int p = 1; p < nparts; ++p) {
      const float* Yp = Y + p * pstride;
#pragma unroll
      for (int k = 0; k < SK_UNR; ++k) v[k] += sk_ld(Yp + min(r0 + k * slots, B - 1) * ld);
    }
#pragma unroll
    for (int k = 0; k < SK_UNR; ++k) {
      const int r = r0 + k * slots;
      if (r < B) {
        s += v[k];
        sl[r << lcw] = v[k];
        if (nparts > 1 && cok) Y[r * ld] = v[k];
      }
    }
  }
  if (stamp != nullptr && tid == 0) stamp[1] = clock64();
  sk_colsum2(s, dummy, sh, lcw, warp, lane);
  if (stamp != nullptr && tid == 0) stamp[2] = clock64();
  const float mean = s / static_cast<float>(B);
  float q = 0.f;
#pragma unroll 4
  for (int r = slot; r < B; r += slots) {
    const float d = sl[r << lcw] - mean;
    q += d * d;
  }
  dummy = 0.f;
  sk_colsum2(q, dummy, sh, lcw, warp, lane);
  const float var = q / static_cast<float>(B);
  const float invx = 1.0f / sqrtf(var + BN_EPS);
  if (slot == 0 && cok) {
    Lr.mean[c] = mean;
    Lr.invstd[c] = invx;
    const float unb = B > 1 ? var * (static_cast<float>(B) / static_cast<float>(B - 1)) : var;
    Lr.run_mean[c] = (1.f - BN_MOM) * Lr.run_mean[c] + BN_MOM * mean;
    Lr.run_var[c] = (1.f - BN_MOM) * Lr.run_var[c] + BN_MOM * unb;
  }
  if (stamp != nullptr && tid == 0) stamp[3] = clock64();
  if (!cok) return;   // no block-wide synchronisation below
  const float p = cx.sc.dropout;
  const float g = __ldg(Lr.gamma + c), be = __ldg(Lr.beta + c);
  if (stamp != nullptr && tid == 0) stamp[4] = clock64() + (g == 12345.f ? 1 : 0);
  const float scale = p > 0.f ? 1.f / (1.f - p) : 1.f;
  const bool inject = sv.inject != 0 && Lr.mask != nullptr;
  const bool draw = p > 0.f && !inject;
  const uint32_t thresh = p > 0.f ? static_cast<uint32_t>(fminf(p * 4294967296.0f, 4294967040.0f)) : 0u;
  const unsigned char* const mask = Lr.mask + c;
  __half* const Hh = Lr.Hh + c;
  __half* const Hl = Lr.Hl + c;
  const uint2 key = sv.key;
  const unsigned lid = Lr.layer_id;
  const int ngroups = (B + 3) >> 2;
#pragma unroll 1
  for (int gq = slot; gq < ngroups; gq += slots) {
    uint4 rnd = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
    if (draw) rnd = sk_rand4(key, lid, c, gq);
    const uint32_t rr[4] = {rnd.x, rnd.y, rnd.z, rnd.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int r = gq * 4 + k;
      if (r < B) {
        const float a = g * ((sl[r << lcw] - mean) * invx) + be;
        float out = a > 0.f ? a : LRELU * a;
        if (p > 0.f) {
          const bool keep = inject ? (mask[r * N] != 0) : (rr[k] >= thresh);
          out = keep ? out * scale : 0.f;
        }
        h_split(out, Hh[r * ld], Hl[r * ld]);
      }
    }
  }
  if (stamp != nullptr && tid == 0) stamp[5] = clock64();
}

// Backward of the slab: dH -> dY (through dropout, LeakyReLU, BatchNorm), dgamma, dbeta; the pre-BN bias gradient is
// identically zero (BN subtracts the batch mean) and is written as 0. slab holds [B][cw] of d a and [B][cw] of x_hat.
__device__ __forceinline__ void sk_bn_bwd_item(const BnLayer& Lr, const StepCtx& cx, const StepVars& sv, int cb, float* slab, float* sh,
                                            int tid, int warp, int lane) {
  const int B = cx.B;
  const int lcw = Lr.lcw, cw = 1 << lcw, slots = SK_THREADS >> lcw;
  const int cl = tid & (cw - 1), slot = tid >> lcw;
  const int N = Lr.N, ld = Lr.ld;
  const int c = (cb << lcw) + cl;
  const bool cok = c < N;
  const int cc = cok ? c : N - 1;
  float* const sl = slab + cl;
  float* const xl = sl + (B << lcw);
  const float p = cx.sc.dropout;
  const float mean = sk_ld(Lr.mean + cc), inv = sk_ld(Lr.invstd + cc);
  const float g = __ldg(Lr.gamma + cc), be = __ldg(Lr.beta + cc);
  const float scale = p > 0.f ? 1.f / (1.f - p) : 1.f;
  const bool inject = sv.inject != 0 && Lr.mask != nullptr;
  const bool draw = p > 0.f && !inject;
  const uint32_t thresh = p > 0.f ? static_cast<uint32_t>(fminf(p * 4294967296.0f, 4294967040.0f)) : 0u;
  const unsigned char* const mask = Lr.mask + cc;
  const float* const Y = Lr.Y.ptr + cc;
  const float* const dH = Lr.dH.ptr + cc;
  const int nparts = Lr.dH.n;
  const long long pstride = Lr.dH.stride;
  const uint2 key = sv.key;
  const unsigned lid = Lr.layer_id;
  const int ngroups = (B + 3) >> 2;
  float s1 = 0.f, s2 = 0.f;
  // two row groups (8 rows) per iteration: all loads first
#pragma unroll 1
  for (int g0 = slot; g0 < ngroups; g0 += 2 * slots) {
    float y[8], d[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int o = min((g0 + (k >> 2) * slots) * 4 + (k & 3), B - 1) * ld;
      y[k] = sk_ld(Y + o);
      d[k] = sk_ld(dH + o);
    }
#pragma unroll 1
    for (int q = 1; q < nparts; ++q) {
      const float* dHq = dH + q * pstride;
#pragma unroll
      for (int k = 0; k < 8; ++k) d[k] += sk_ld(dHq + min((g0 + (k >> 2) * slots) * 4 + (k & 3), B - 1) * ld);
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int gq = g0 + h * slots;
      uint4 rnd = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
      if (draw && gq < ngroups) rnd = sk_rand4(key, lid, c, gq);
      const uint32_t rr[4] = {rnd.x, rnd.y, rnd.z, rnd.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int r = gq * 4 + k;
        if (r < B) {
          const float xhat = (y[4 * h + k] - mean) * inv;
          const float a = g * xhat + be;
          float dd = cok ? d[4 * h + k] : 0.f;
          if (p > 0.f) {
            const bool keep = inject ? (mask[r * N] != 0) : (rr[k] >= thresh);
            dd = keep ? dd * scale : 0.f;
          }
          dd = a > 0.f ? dd : LRELU * dd;
          s1 += dd;
          s2 += dd * xhat;
          sl[r << lcw] = dd;
          xl[r << lcw] = xhat;
        }
      }
    }
  }
  sk_colsum2(s1, s2, sh, lcw, warp, lane);
  if (!cok) return;
  if (slot == 0) {
    const float ig = Lr.gdyn != nullptr ? cx.inv_gs * sk_ld(Lr.gdyn) : cx.inv_gs;
    if (sv.accum) { Lr.dbeta[c] += s1 * ig; Lr.dgamma[c] += s2 * ig; }
    else { Lr.dbeta[c] = s1 * ig; Lr.dgamma[c] = s2 * ig; Lr.dbias[c] = 0.f; }
  }
  const float fb = static_cast<float>(B);
  const float k0 = inv * g / fb;
  __half* const dYh = Lr.dYh + c;
  __half* const dYl = Lr.dYl + c;
#pragma unroll 4
  for (int r = slot; r < B; r += slots)
    h_split(k0 * (fb * sl[r << lcw] - s1 - xl[r << lcw] * s2), dYh[r * ld], dYl[r * ld]);
}

// ------------------------------------------------------------------------------------------------ cluster-fused tails
// With B <= 4 x 128 rows the step kernel runs as clusters of HG_CLUSTER = 4 CTAs: the four CTAs of a cluster compute the
// four M tiles of one column block of a layer (hgemm.cuh: HgProblem::fuse), so the whole batch of every feature column
// sits in one cluster and the BatchNorm batch statistics are a cluster-local reduction through distributed shared memory.
// The element-wise work that used to be separate slab phases (each a grid barrier plus an L2 round trip of the layer
// output) becomes the tail of the GEMM work item: all 16 warps read the tile from the staging blocks.
//
// Code-size rule (measured, round 2): a phase body runs once per step, so its instructions come from L2 at ~20 cycles
// per instruction (no overlap: ~10 ns per STATIC instruction); the first version of these tails (8 columns per thread,
// everything unrolled: ~1300 instructions each) cost 25 us per work item cold and 10 us warm. Hence ROLLED loops over
// the rows, tile values re-read from shared memory instead of living in registers, and the dropout keep bits are
// produced by the six warps without a GEMM role while the main loop runs (sk_side_mask).
//   thread mapping: warp = octet of rows (16 octets = 128 rows); lane = pair of adjacent columns (bn = 64), or
//   lane & 15 = pair and lane >> 4 = half of the octet (bn = 32). Pairs: 8-byte shared loads, float2 / half2 stores.
// Scratch (operand ring, idle while the tail runs; float offsets): red [16 warps][32 pairs] float4, xbuf [32] float4
// (read by the peers), then a [128][64] tile buffer (y / x prefetch, x_hat).
enum StepFuse : int { FUSE_NONE = 0, FUSE_BN_FWD = 1, FUSE_BN_BWD = 2, FUSE_REC = 3, FUSE_HEADS = 4, FUSE_LATBC = 5 };
constexpr int SKT_RED = 0, SKT_XBUF = 16 * 32 * 4, SKT_TILE = SKT_XBUF + 32 * 4;

struct TailArgs {
  uint8_t* stage; float* scr; const uint8_t* keep; int m0, n0, bn, tid, warp, lane; uint32_t rank;
  long long* stamp;   // profiling: SM clock stamps of thread 0 (8 slots) or null
};
__device__ __forceinline__ void tail_stamp(const TailArgs& ta, int k) { if (ta.stamp != nullptr && ta.tid == 0) ta.stamp[k] = clock64(); }
struct TailGeo {
  int pr, cl, r0, nk, fold;
  uint32_t sbase;   // byte offset of (row 0, column cl) in the staging blocks, without the row swizzle
  int u;            // 16-byte unit of the column pair inside its 128-byte row
};
__device__ __forceinline__ TailGeo tail_geo(int bn, int warp, int lane) {
  TailGeo g;
  g.fold = bn > 32 ? 0 : 1;
  g.pr = g.fold ? (lane & 15) : lane;
  g.cl = 2 * g.pr;
  g.nk = g.fold ? 4 : 8;
  g.r0 = warp * 8 + (g.fold ? (lane >> 4) * 4 : 0);
  g.sbase = static_cast<uint32_t>((g.cl >> 5) * 16384 + (g.cl & 3) * 4);
  g.u = (g.cl & 31) >> 2;
  return g;
}
// elements (r, cl), (r, cl + 1) of the staged tile (hgemm.cuh: hg_stage_ptr)
__device__ __forceinline__ float2* tail_stg(const TailArgs& ta, const TailGeo& g, int r) {
  return reinterpret_cast<float2*>(ta.stage + g.sbase + r * 128 + ((g.u ^ (r & 7)) << 4));
}
__device__ __forceinline__ int tile_rows(int B, int rank) { const int n = B - rank * HG_BM; return n < 0 ? 0 : (n > HG_BM ? HG_BM : n); }
// v = per-thread partial sums {a of column 0, a of column 1, b of column 0, b of column 1}: summed over all rows of the
// tile (the two halves of an octet, then the 16 warps in a fixed order) and broadcast. All 512 threads must call.
__device__ __noinline__ float4 tail_sum4(float4 v, float* scr, int pr, int warp, int fold) {
  if (fold) {
    v.x += __shfl_xor_sync(0xffffffffu, v.x, 16); v.y += __shfl_xor_sync(0xffffffffu, v.y, 16);
    v.z += __shfl_xor_sync(0xffffffffu, v.z, 16); v.w += __shfl_xor_sync(0xffffffffu, v.w, 16);
  }
  float4* red = reinterpret_cast<float4*>(scr + SKT_RED);
  red[warp * 32 + pr] = v;
  __syncthreads();
  float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
  for (int w = 0; w < SK_WARPS; ++w) { const float4 x = red[w * 32 + pr]; t.x += x.x; t.y += x.y; t.z += x.z; t.w += x.w; }
  __syncthreads();
  return t;
}
// 8 x 16 random bits for rows 8 oc8 .. 8 oc8 + 7 of column c (dropout of the fused layers; oc8 counts octets of the batch)
__device__ __forceinline__ uint4 sk_rand8(uint2 key, unsigned layer_id, int col, int oc8) {
  return philox4x32(make_uint4(static_cast<uint32_t>(oc8), static_cast<uint32_t>(col), layer_id + 64u, 0x4A4Du), key);
}
// Dropout keep bits of a fused BatchNorm tile: keep[oc * 64 + col] bit k = row 8 oc + k of the tile is kept. Written by
// the warps without a GEMM role (side = 0 .. HG_NSIDE - 1) while the roles run; forward and backward regenerate the
// same bits (Philox keyed by step, layer, column, octet) or pack the injected mask.
__device__ __forceinline__ void sk_side_mask(const StepCtx& cx, const StepVars& sv, const BnLayer& Lr, const HgTile& T, uint8_t* keep, int side, int lane) {
  const float pdrop = cx.sc.dropout;
  const bool inject = sv.inject != 0 && Lr.mask != nullptr;
  const uint32_t thresh = pdrop > 0.f ? static_cast<uint32_t>(fminf(pdrop * 65536.0f + 0.5f, 65535.0f)) : 0u;
  const int lbn = T.bn > 32 ? 6 : 5;
  const int N = Lr.N;
#pragma unroll 1
  for (int it = side * 32 + lane; it < (16 << lbn); it += HG_NSIDE * 32) {
    const int oc = it >> lbn, cl = it & (T.bn - 1);
    const int c = T.n0 + cl;
    uint32_t bits = 0xffu;
    if (pdrop > 0.f && c < N) {
      bits = 0u;
      if (inject) {
#pragma unroll 1
        for (int k = 0; k < 8; ++k) {
          const int row = T.m0 + oc * 8 + k;
          if (row < cx.B && Lr.mask[static_cast<long long>(row) * N + c] != 0) bits |= 1u << k;
        }
      } else {
        const uint4 r = sk_rand8(sv.key, Lr.layer_id, c, (T.m0 >> 3) + oc);
        bits |= ((r.x & 0xffffu) >= thresh ? 1u : 0u) | ((r.x >> 16) >= thresh ? 2u : 0u);
        bits |= ((r.y & 0xffffu) >= thresh ? 4u : 0u) | ((r.y >> 16) >= thresh ? 8u : 0u);
        bits |= ((r.z & 0xffffu) >= thresh ? 16u : 0u) | ((r.z >> 16) >= thresh ? 32u : 0u);
        bits |= ((r.w & 0xffffu) >= thresh ? 64u : 0u) | ((r.w >> 16) >= thresh ? 128u : 0u);
      }
    }
    keep[oc * 64 + cl] = static_cast<uint8_t>(bits);
  }
}
__device__ __forceinline__ float4 ld_dsmem_f4(uint32_t addr) { return ld_shared_cluster_f4(addr); }
__device__ __forceinline__ void split2(float a, float b, __half2& hi, __half2& lo) {
  hi = h2_sat(a, b);
  const float2 f = __half22float2(hi);
  lo = h2_sat((a - f.x) * HG_LO_SCALE, (b - f.y) * HG_LO_SCALE);
}

// Linear output tile -> BatchNorm1d (batch statistics over the cluster: per-CTA mean / M2, merged with Chan's formula in
// rank order) -> LeakyReLU(0.01) -> Dropout(p) -> fp16 operand planes of the next GEMM; stores the pre-BN output y for
// the backward pass; rank 0 updates the running statistics   (jamie/model.py:151-154 and siblings)
__device__ __forceinline__ void sk_tail_bn_fwd(const StepCtx& cx, const StepVars& sv, const BnLayer& Lr, const float* __restrict__ biasp, const TailArgs& ta) {
  const int B = cx.B, N = Lr.N, ld = Lr.ld;
  const TailGeo g = tail_geo(ta.bn, ta.warp, ta.lane);
  const int c = ta.n0 + g.cl;
  const bool cok = c < N, cok1 = c + 1 < N;
  const int c0 = cok ? c : N - 1, c1 = cok1 ? c + 1 : N - 1;
  const float bias0 = __ldg(biasp + c0), bias1 = __ldg(biasp + c1);
  const float ga0 = __ldg(Lr.gamma + c0), ga1 = __ldg(Lr.gamma + c1), be0 = __ldg(Lr.beta + c0), be1 = __ldg(Lr.beta + c1);
  const int nc = tile_rows(B, static_cast<int>(ta.rank));
  int nv = nc - g.r0; nv = nv < 0 ? 0 : (nv > g.nk ? g.nk : nv);   // valid rows of this thread
  tail_stamp(ta, 0);
  // one pass: sums of (x - p) and (x - p)^2 with the pivot p = row 0 of the tile (shifted-data variance: the cancellation
  // in S2 - S1^2 / n is governed by (mean - p)^2 / var = O(1), not by mean^2 / var)
  const float2 pv0 = *tail_stg(ta, g, 0);
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 2
  for (int k = 0; k < nv; ++k) {
    const float2 f = *tail_stg(ta, g, g.r0 + k);
    const float d0 = f.x - pv0.x, d1 = f.y - pv0.y;
    s.x += d0; s.y += d1; s.z += d0 * d0; s.w += d1 * d1;
  }
  s = tail_sum4(s, ta.scr, g.pr, ta.warp, g.fold);
  tail_stamp(ta, 1);
  const float rnc = nc > 0 ? 1.f / static_cast<float>(nc) : 0.f;
  const float mc0 = nc > 0 ? pv0.x + bias0 + s.x * rnc : 0.f, mc1 = nc > 0 ? pv0.y + bias1 + s.y * rnc : 0.f;
  s.x = fmaxf(s.z - s.x * s.x * rnc, 0.f);   // M2 about the CTA mean
  s.y = fmaxf(s.w - s.y * s.y * rnc, 0.f);
  float4* xb = reinterpret_cast<float4*>(ta.scr + SKT_XBUF);
  tail_stamp(ta, 2);
  if (ta.warp == 0) xb[g.pr] = make_float4(mc0, mc1, s.x, s.y);
  cluster_sync_all();
  tail_stamp(ta, 3);
  // batch mean = sum n_r mean_r / B; M2 = sum [M2_r + n_r (mean_r - mean)^2]   (the ranks in a fixed order)
  const float rB = 1.f / static_cast<float>(B);
  float mean0 = 0.f, mean1 = 0.f, m20 = 0.f, m21 = 0.f;
  {
    const uint32_t xa = smem_u32(xb + g.pr);
    float4 pv[HG_CLUSTER];
#pragma unroll
    for (int r = 0; r < HG_CLUSTER; ++r) pv[r] = ld_dsmem_f4(mapa_shared(xa, static_cast<uint32_t>(r)));
#pragma unroll
    for (int r = 0; r < HG_CLUSTER; ++r) {
      const float nr = static_cast<float>(tile_rows(B, r));
      mean0 += nr * pv[r].x; mean1 += nr * pv[r].y;
    }
    mean0 *= rB; mean1 *= rB;
#pragma unroll
    for (int r = 0; r < HG_CLUSTER; ++r) {
      const float nr = static_cast<float>(tile_rows(B, r));
      const float d0 = pv[r].x - mean0, d1 = pv[r].y - mean1;
      if (nr > 0.f) { m20 += pv[r].z + nr * d0 * d0; m21 += pv[r].w + nr * d1 * d1; }
    }
  }
  const float var0 = m20 * rB, var1 = m21 * rB;
  const float inv0 = rsqrtf(var0 + BN_EPS), inv1 = rsqrtf(var1 + BN_EPS);
  if (ta.rank == 0 && ta.warp == 0 && ta.lane == g.pr) {   // the running statistics follow in the WGRAD phase (sk_running_stats)
    if (cok) { Lr.mean[c] = mean0; Lr.invstd[c] = inv0; Lr.var[c] = var0; }
    if (cok1) { Lr.mean[c + 1] = mean1; Lr.invstd[c + 1] = inv1; Lr.var[c + 1] = var1; }
  }
  tail_stamp(ta, 4);
  if (!cok) return;   // no block-wide synchronisation below
  const float pdrop = cx.sc.dropout;
  const float scale = pdrop > 0.f ? 1.f / (1.f - pdrop) : 1.f;
  const uint32_t kb = *reinterpret_cast<const uint16_t*>(ta.keep + ta.warp * 64 + g.cl) >> (g.r0 & 7);   // bits k (column 0), 8 + k (column 1)
  // a = gamma (v - mean) inv + beta as one FMA per element; a column beyond N gets a = 0
  const float sc0 = ga0 * inv0, sc1 = cok1 ? ga1 * inv1 : 0.f;
  const float sh0 = be0 - mean0 * sc0, sh1 = cok1 ? be1 - mean1 * sc1 : 0.f;
  int o = (ta.m0 + g.r0) * ld + c;
#pragma unroll 2
  for (int k = 0; k < nv; ++k, o += ld) {
    const float2 f = *tail_stg(ta, g, g.r0 + k);
    const float v0 = f.x + bias0, v1 = f.y + bias1;
    const float a0 = v0 * sc0 + sh0, a1 = v1 * sc1 + sh1;
    const float o0 = fmaxf(a0, LRELU * a0) * (((kb >> k) & 1u) ? scale : 0.f);          // LeakyReLU: max(a, 0.01 a)
    const float o1 = fmaxf(a1, LRELU * a1) * (((kb >> (8 + k)) & 1u) ? scale : 0.f);
    __half2 hi, lo;
    split2(o0, o1, hi, lo);
    *reinterpret_cast<float2*>(Lr.Y.ptr + o) = make_float2(v0, v1);
    *reinterpret_cast<__half2*>(Lr.Hh + o) = hi;
    *reinterpret_cast<__half2*>(Lr.Hl + o) = lo;
  }
  tail_stamp(ta, 5);
}

// dgrad tile dH -> through Dropout, LeakyReLU and BatchNorm (batch sums over the cluster) -> dY planes; rank 0 writes
// d gamma, d beta (the pre-BN bias gradient is identically zero)
__device__ __forceinline__ void sk_tail_bn_bwd(const StepCtx& cx, const StepVars& sv, const BnLayer& Lr, const TailArgs& ta) {
  const int B = cx.B, N = Lr.N, ld = Lr.ld;
  const TailGeo g = tail_geo(ta.bn, ta.warp, ta.lane);
  const int c = ta.n0 + g.cl;
  const bool cok = c < N, cok1 = c + 1 < N;
  const int c0 = cok ? c : N - 1, c1 = cok1 ? c + 1 : N - 1;
  const int nc = tile_rows(B, static_cast<int>(ta.rank));
  int nv = nc - g.r0; nv = nv < 0 ? 0 : (nv > g.nk ? g.nk : nv);
  float2* const xt = reinterpret_cast<float2*>(ta.scr + SKT_TILE + g.cl);   // [r * 32]: y, then x_hat
  // prefetch this thread's y values (all loads in flight together; row indices clamped instead of branches)
  {
    const float* const Y = Lr.Y.ptr + (cok ? c : 0);
    const int rl = nc > 0 ? ta.m0 + nc - 1 : B - 1;   // last valid row (a CTA without rows reads row B - 1 and ignores it)
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int row = ta.m0 + g.r0 + k;
      const float2 y = sk_ld(reinterpret_cast<const float2*>(Y + (row < rl ? row : rl) * ld));
      if (k < g.nk) xt[(g.r0 + k) * 32] = y;
    }
  }
  const float mean0 = sk_ld(Lr.mean + c0), mean1 = sk_ld(Lr.mean + c1), inv0 = sk_ld(Lr.invstd + c0), inv1 = sk_ld(Lr.invstd + c1);
  const float ga0 = __ldg(Lr.gamma + c0), ga1 = __ldg(Lr.gamma + c1), be0 = __ldg(Lr.beta + c0), be1 = __ldg(Lr.beta + c1);
  const float pdrop = cx.sc.dropout;
  const float scale = pdrop > 0.f ? 1.f / (1.f - pdrop) : 1.f;
  uint32_t kb = *reinterpret_cast<const uint16_t*>(ta.keep + ta.warp * 64 + g.cl) >> (g.r0 & 7);
  if (!cok) kb = 0u;
  if (!cok1) kb &= 0xffu;   // a column beyond N: d = 0 (its y is finite: the forward tail wrote the padding)
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 2
  for (int k = 0; k < nv; ++k) {
    float2* const sp = tail_stg(ta, g, g.r0 + k);
    const float2 y = xt[(g.r0 + k) * 32];
    float2 d = *sp;
    const float x0 = (y.x - mean0) * inv0, x1 = (y.y - mean1) * inv1;
    const float a0 = ga0 * x0 + be0, a1 = ga1 * x1 + be1;
    d.x *= (((kb >> k) & 1u) ? scale : 0.f) * (a0 > 0.f ? 1.f : LRELU);
    d.y *= (((kb >> (8 + k)) & 1u) ? scale : 0.f) * (a1 > 0.f ? 1.f : LRELU);
    s.x += d.x; s.y += d.y; s.z += d.x * x0; s.w += d.y * x1;
    *sp = d;
    xt[(g.r0 + k) * 32] = make_float2(x0, x1);
  }
  s = tail_sum4(s, ta.scr, g.pr, ta.warp, g.fold);
  float4* xb = reinterpret_cast<float4*>(ta.scr + SKT_XBUF);
  if (ta.warp == 0) xb[g.pr] = s;
  cluster_sync_all();
  {
    const uint32_t xa = smem_u32(xb + g.pr);
    float4 pv[HG_CLUSTER];
#pragma unroll
    for (int r = 0; r < HG_CLUSTER; ++r) pv[r] = ld_dsmem_f4(mapa_shared(xa, static_cast<uint32_t>(r)));
    s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int r = 0; r < HG_CLUSTER; ++r)
      if (tile_rows(B, r) > 0) { s.x += pv[r].x; s.y += pv[r].y; s.z += pv[r].z; s.w += pv[r].w; }
  }
  if (!cok) return;
  if (ta.rank == 0 && ta.warp == 0 && ta.lane == g.pr) {
    const float ig = Lr.gdyn != nullptr ? cx.inv_gs * sk_ld(Lr.gdyn) : cx.inv_gs;
    if (sv.accum) {
      Lr.dbeta[c] += s.x * ig; Lr.dgamma[c] += s.z * ig;
      if (cok1) { Lr.dbeta[c + 1] += s.y * ig; Lr.dgamma[c + 1] += s.w * ig; }
    } else {
      Lr.dbeta[c] = s.x * ig; Lr.dgamma[c] = s.z * ig; Lr.dbias[c] = 0.f;
      if (cok1) { Lr.dbeta[c + 1] = s.y * ig; Lr.dgamma[c + 1] = s.w * ig; Lr.dbias[c + 1] = 0.f; }
    }
  }
  // dy = (gamma inv / B) (B d - s1 - x_hat s2) = A d - (K s1) - x_hat (K s2),  K = gamma inv / B
  const float rB = 1.f / static_cast<float>(B);
  const float A0 = inv0 * ga0, A1 = cok1 ? inv1 * ga1 : 0.f;
  const float K0 = A0 * rB, K1 = A1 * rB;
  const float b0 = K0 * s.x, b1 = K1 * s.y, e0 = K0 * s.z, e1 = K1 * s.w;
  int o = (ta.m0 + g.r0) * ld + c;
#pragma unroll 2
  for (int k = 0; k < nv; ++k, o += ld) {
    const float2 d = *tail_stg(ta, g, g.r0 + k);
    const float2 x = xt[(g.r0 + k) * 32];
    __half2 hi, lo;
    split2(A0 * d.x - b0 - x.x * e0, A1 * d.y - b1 - x.y * e1, hi, lo);
    *reinterpret_cast<__half2*>(Lr.dYh + o) = hi;
    *reinterpret_cast<__half2*>(Lr.dYl + o) = lo;
  }
}

// last decoder Linear: xhat tile -> reconstruction loss partial, d xhat planes, bias gradient (column sums over the
// cluster)   (jamie/jamie.py:637-643)
__device__ __forceinline__ void sk_tail_rec(const StepCtx& cx, const StepVars& sv, const ModCtx& M, const float* __restrict__ biasp, const TailArgs& ta) {
  const int B = cx.B, N = M.D, ld = M.ldD;
  const TailGeo g = tail_geo(ta.bn, ta.warp, ta.lane);
  const int c = ta.n0 + g.cl;
  const bool cok = c < N, cok1 = c + 1 < N;
  const int c0 = cok ? c : N - 1, c1 = cok1 ? c + 1 : N - 1;
  const int nc = tile_rows(B, static_cast<int>(ta.rank));
  int nv = nc - g.r0; nv = nv < 0 ? 0 : (nv > g.nk ? g.nk : nv);
  if (!cok) nv = 0;
  float2 xv[8];
  {
    const float* const X = M.x + (cok ? c : 0);
    const int rl = nc > 0 ? ta.m0 + nc - 1 : B - 1;   // last valid row (a CTA without rows reads row B - 1 and ignores it)
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int row = ta.m0 + g.r0 + k;
      xv[k] = sk_ld(reinterpret_cast<const float2*>(X + (row < rl ? row : rl) * ld));
    }
  }
  float2* const xt = reinterpret_cast<float2*>(ta.scr + SKT_TILE + g.cl);
#pragma unroll
  for (int k = 0; k < 8; ++k)
    if (k < g.nk) xt[(g.r0 + k) * 32] = xv[k];
  const float kk = cx.gs * cx.sc.w[1] * 2.f / (static_cast<float>(B) * static_cast<float>(N));
  const float bias0 = __ldg(biasp + c0), bias1 = __ldg(biasp + c1);
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);   // column sums of d xhat (x, y), squared error (z)
  int o = (ta.m0 + g.r0) * ld + c;
#pragma unroll 2
  for (int k = 0; k < nv; ++k, o += ld) {
    const float2 f = *tail_stg(ta, g, g.r0 + k);
    const float2 x = xt[(g.r0 + k) * 32];
    const float h0 = f.x + bias0, h1 = f.y + bias1;
    const float d0 = h0 - x.x, d1 = cok1 ? h1 - x.y : 0.f;
    s.z += d0 * d0 + d1 * d1;
    const float g0 = kk * d0, g1 = kk * d1;
    s.x += g0; s.y += g1;
    __half2 hi, lo;
    split2(g0, g1, hi, lo);
    *reinterpret_cast<float2*>(M.xhat.ptr + o) = make_float2(h0, h1);
    *reinterpret_cast<__half2*>(M.dxh + o) = hi;
    *reinterpret_cast<__half2*>(M.dxl + o) = lo;
  }
  s = tail_sum4(s, ta.scr, g.pr, ta.warp, g.fold);
  float4* xb = reinterpret_cast<float4*>(ta.scr + SKT_XBUF);
  if (ta.warp == 0) xb[g.pr] = s;
  cluster_sync_all();   // (also a CTA barrier)
  if (ta.warp == 1) {   // CTA partial of the squared error: the column pairs of the tile in a fixed order
    float t = (ta.bn > 32 || ta.lane < 16) ? xb[ta.lane].z : 0.f;
    t = warp_sum(t);
    if (ta.lane == 0) M.rec_part[(ta.n0 / ta.bn) * HG_CLUSTER + static_cast<int>(ta.rank)] = t;
  }
  if (ta.rank == 0 && ta.warp == 0 && ta.lane == g.pr && cok) {
    const uint32_t xa = smem_u32(xb + g.pr);
    float s0 = 0.f, s1 = 0.f;
#pragma unroll
    for (int r = 0; r < HG_CLUSTER; ++r) {
      const float4 pv = ld_dsmem_f4(mapa_shared(xa, static_cast<uint32_t>(r)));
      if (tile_rows(B, r) > 0) { s0 += pv.x; s1 += pv.y; }
    }
    const float v0 = s0 * cx.inv_gs, v1 = s1 * cx.inv_gs;
    M.db5[c] = sv.accum ? M.db5[c] + v0 : v0;
    if (cok1) M.db5[c + 1] = sv.accum ? M.db5[c + 1] + v1 : v1;
  }
}

// eps of both modalities for this step (injected or Philox Box-Muller, jamie/model.py:230-240): drawn by the warps without
// a GEMM role at the start of ENC1, off the critical path (the heads tail of 8 CTAs used to spend 7 us on it)
__device__ __forceinline__ void sk_draw_eps(const StepCtx& cx, const StepVars& sv, int gt, int nt) {
  const int B = cx.B, L = cx.L;
#pragma unroll 1
  for (int t = gt; t < 2 * B * L; t += nt) {
    const int i = t / (B * L), rem = t - i * B * L, b = rem / L, l = rem - b * L;
    const ModCtx& M = cx.m[i];
    float e;
    if (sv.inject) {
      e = M.inj_eps[static_cast<long long>(b) * cx.LP + l];
    } else {
      const uint4 r = philox4x32(make_uint4(static_cast<uint32_t>(b), static_cast<uint32_t>(l), 0xE950u + i, 0x4A4Du), sv.key);
      const float u1 = (static_cast<float>(r.x >> 8) + 0.5f) * (1.0f / 16777216.0f);
      const float u2 = (static_cast<float>(r.y >> 8) + 0.5f) * (1.0f / 16777216.0f);
      e = sqrtf(-2.f * logf(u1)) * cospif(2.f * u2);
    }
    M.eps[static_cast<long long>(b) * cx.LP + l] = e;
  }
}
// heads tile [mu | logvar] (2 L <= 64 columns) -> z = mu + (exp(logvar/2) + 1e-7) eps   (jamie/model.py:230-240)
// element (r, c) of the staged tile of cluster rank rk (distributed shared memory)
__device__ __forceinline__ float tail_stage_remote(const TailArgs& ta, int r, int c, uint32_t rk) {
  float v;
  asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(mapa_shared(smem_u32(reinterpret_cast<const float*>(hg_stage_ptr(ta.stage, r, c & ~3)) + (c & 3)), rk)) : "memory");
  return v;
}
__device__ __forceinline__ void sk_tail_heads(const StepCtx& cx, const StepVars& sv, const ModCtx& M, int mod, const float* __restrict__ bias, const TailArgs& ta, int ks) {
  const int B = cx.B, L = cx.L;
  if (ks) cluster_sync_all();   // K split over the cluster: the four partial tiles are staged; this CTA finishes rows [32 rank, +32)
  const int r_lo = ks ? 32 * static_cast<int>(ta.rank) : 0, n_r = ks ? 32 : HG_BM;
#pragma unroll 1
  for (int idx = ta.tid; idx < n_r * L; idx += SK_THREADS) {
    const int r = r_lo + idx / L, l = idx % L;
    const int b = ta.m0 + r;
    if (b >= B) break;
    const float e = sk_ld(M.eps + static_cast<long long>(b) * cx.LP + l);
    float mu = __ldg(bias + l), lv = __ldg(bias + L + l);
    if (ks) {
#pragma unroll
      for (uint32_t rk = 0; rk < HG_CLUSTER; ++rk) { mu += tail_stage_remote(ta, r, l, rk); lv += tail_stage_remote(ta, r, L + l, rk); }
    } else {
      mu += reinterpret_cast<const float*>(hg_stage_ptr(ta.stage, r, l & ~3))[l & 3];
      lv += reinterpret_cast<const float*>(hg_stage_ptr(ta.stage, r, (L + l) & ~3))[(L + l) & 3];
    }
    const long long om = static_cast<long long>(b) * cx.ldmv;
    M.mulv.ptr[om + l] = mu;
    M.mulv.ptr[om + L + l] = lv;
    M.z[static_cast<long long>(b) * cx.LP + l] = mu + (expf(lv * 0.5f) + 1e-7f) * e;
  }
}

// ------------------------------------------------------------------------------------------------ reconstruction loss
// d xhat = gs * w_rec * 2 (xhat - x) / (B D); per-item partial of sum (xhat - x)^2; bias gradient of the last decoder
// Linear = column sums of d xhat / gs   (jamie/jamie.py:637-643). One pass, no staging.
__device__ __forceinline__ void sk_rec_item(const ModCtx& M, const StepCtx& cx, const StepVars& sv, int cb, int item, float* sh, int tid,
                                         int warp, int lane) {
  const int B = cx.B;
  const int lcw = M.rec_lcw, cw = 1 << lcw, slots = SK_THREADS >> lcw;
  const int cl = tid & (cw - 1), slot = tid >> lcw;
  const int c = (cb << lcw) + cl;
  const bool cok = c < M.D;
  const int cc = cok ? c : M.D - 1;
  const int ld = M.ldD;
  const float kk = cx.gs * cx.sc.w[1] * 2.f / (static_cast<float>(B) * static_cast<float>(M.D));
  const int nparts = M.xhat.n;
  const long long pstride = M.xhat.stride;
  float* const XH = M.xhat.ptr + cc;
  const float* const X = M.x + cc;
  __half* const dxh = M.dxh + cc;
  __half* const dxl = M.dxl + cc;
  float sq = 0.f, cs = 0.f;
#pragma unroll 1
  for (int r0 = slot; r0 < B; r0 += SK_UNR * slots) {
    float xh[SK_UNR], xx[SK_UNR];
#pragma unroll
    for (int k = 0; k < SK_UNR; ++k) {
      const int o = min(r0 + k * slots, B - 1) * ld;
      xh[k] = sk_ld(XH + o);
      xx[k] = sk_ld(X + o);
    }
#pragma unroll 1
    for (int q = 1; q < nparts; ++q) {
      const float* XHq = XH + q * pstride;
#pragma unroll
      for (int k = 0; k < SK_UNR; ++k) xh[k] += sk_ld(XHq + min(r0 + k * slots, B - 1) * ld);
    }
#pragma unroll
    for (int k = 0; k < SK_UNR; ++k) {
      const int r = r0 + k * slots;
      if (cok && r < B) {
        const float d = xh[k] - xx[k];
        sq += d * d;
        const float gx = kk * d;
        cs += gx;
        if (nparts > 1) XH[r * ld] = xh[k];
        h_split(gx, dxh[r * ld], dxl[r * ld]);
      }
    }
  }
  sk_colsum2(sq, cs, sh, lcw, warp, lane);
  if (warp == 0) {
    if (lane < cw && cok) {
      const float v = cs * cx.inv_gs;
      M.db5[c] = sv.accum ? M.db5[c] + v : v;
    }
    float t = (lane < cw && cok) ? sq : 0.f;
    t = warp_sum(t);
    if (lane == 0) M.rec_part[item] = t;
  }
}

// ------------------------------------------------------------------------------------------------ dynamic operand scales
// fp16 operand planes overflow above 65504. Post-BatchNorm activations and weights are bounded by construction, the
// backward pass carries the static loss scale, but two tensors are unbounded: the latent c (z = mu + exp(logvar / 2) eps
// with a large logvar: observed 1e5 within 60 steps of the 1M-cell benchmark) and d[mu | logvar] (the same exp factor).
// Their producers record the per-CTA maximum magnitude; the phase that writes the planes (after a grid barrier) derives
// an exact power-of-two scale from the global maximum, identical in every CTA. s = 1 whenever max <= 2^15.
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// every thread passes its running maximum; writes the CTA maximum to part[cta]. All threads of the CTA must call.
__device__ __forceinline__ void sk_cta_max_store(float v, float* part, int cta, float* sh, int tid, int warp, int lane) {
  v = warp_max(v);
  __syncthreads();
  if (lane == 0) sh[warp] = v;
  __syncthreads();
  if (tid == 0) {
    float m = 0.f;
#pragma unroll
    for (int w = 0; w < SK_WARPS; ++w) m = fmaxf(m, sh[w]);
    part[cta] = m;
  }
  __syncthreads();
}
// (scale, inverse scale) from the per-CTA maxima; warp-cooperative, same result in every warp of every CTA
__device__ __forceinline__ float2 sk_dyn_scale(const float* part, int ncta, int lane) {
  float v[SK_MAX_CTAS / 32];
#pragma unroll
  for (int u = 0; u < SK_MAX_CTAS / 32; ++u) v[u] = sk_ld(part + min(lane + 32 * u, ncta - 1));   // all loads in flight together
  float m = 0.f;
#pragma unroll
  for (int u = 0; u < SK_MAX_CTAS / 32; ++u) m = fmaxf(m, v[u]);
  m = warp_max(m);
  if (!(m > 32768.f)) return make_float2(1.f, 1.f);
  int e = 128;
  if (m < 3.0e38f) frexpf(m, &e);          // m <= 2^e
  return make_float2(ldexpf(1.f, 15 - e), ldexpf(1.f, e - 15));
}

// ------------------------------------------------------------------------------------------------ latent stage
// eps (injected or Philox Box-Muller) and z = mu + (exp(logvar/2) + 1e-7) eps   (jamie/model.py:230-240); also reduces
// the split-K partials of the heads GEMM into partial 0.
__device__ __forceinline__ void sk_reparam(const StepCtx& cx, const StepVars& sv, int gt, int nt) {
  const int B = cx.B, L = cx.L;
  for (int t = gt; t < 2 * B * L; t += nt) {
    const int i = t / (B * L), rem = t - i * B * L, b = rem / L, l = rem - b * L;
    const ModCtx& M = cx.m[i];
    float e;
    if (sv.inject) {
      e = M.inj_eps[static_cast<long long>(b) * cx.LP + l];
    } else {
      const uint4 r = philox4x32(make_uint4(static_cast<uint32_t>(b), static_cast<uint32_t>(l), 0xE950u + i, 0x4A4Du), sv.key);
      const float u1 = (static_cast<float>(r.x >> 8) + 0.5f) * (1.0f / 16777216.0f);
      const float u2 = (static_cast<float>(r.y >> 8) + 0.5f) * (1.0f / 16777216.0f);
      e = sqrtf(-2.f * logf(u1)) * cospif(2.f * u2);
    }
    const long long om = static_cast<long long>(b) * cx.ldmv;
    const float mu = ld_parts(M.mulv, om + l);
    const float lv = ld_parts(M.mulv, om + L + l);
    if (M.mulv.n > 1) { M.mulv.ptr[om + l] = mu; M.mulv.ptr[om + L + l] = lv; }
    M.eps[static_cast<long long>(b) * cx.LP + l] = e;
    M.z[static_cast<long long>(b) * cx.LP + l] = mu + (expf(lv * 0.5f) + 1e-7f) * e;
  }
}

// out[l] (per lane, LAT_MAXT strided) = sum_b M[row, b] * V[b, l], skipping zero entries; also returns the row sum.
// 128 entries of the row per iteration (four loads in flight per lane), then a ballot loop over the nonzeros.
// hint (diagonal priors, written by sk_corr_row_diag): {nonzeros of the row, column of the first}: rows without a nonzero
// (unmatched cells) and rows with exactly one (every matched cell unless the batch repeats it) skip the scan of the dense
// row -- four dependent L2 round trips on the critical path of COMBINE and LATBZ. Same arithmetic: 0 + x = x.
__device__ __forceinline__ float sk_row_times(const float* __restrict__ Mrow, const float* __restrict__ V, int B, int LP, int L, int lane,
                                              float (&acc)[LAT_MAXT], const int2* __restrict__ hint = nullptr) {
#pragma unroll
  for (int t = 0; t < LAT_MAXT; ++t) acc[t] = 0.f;
  float rs = 0.f;
  if (hint != nullptr) {
    const int2 h = sk_ld(hint);
    if (h.x == 0) return 0.f;
    if (h.x == 1) {
      const float mv = sk_ld(Mrow + h.y);
      const float* v = V + static_cast<long long>(h.y) * LP;
#pragma unroll
      for (int t = 0; t < LAT_MAXT; ++t) {
        const int l = lane + 32 * t;
        if (l < L) acc[t] += mv * sk_ld(v + l);
      }
      return rs + mv;
    }
  }
#pragma unroll 1
  for (int sup = 0; sup < B; sup += 128) {
    float m[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int b = sup + 32 * i + lane;
      m[i] = b < B ? sk_ld(Mrow + b) : 0.f;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      unsigned nz = __ballot_sync(0xffffffffu, m[i] != 0.f);
      while (nz) {
        const int src = __ffs(nz) - 1;
        nz &= nz - 1;
        const float mv = __shfl_sync(0xffffffffu, m[i], src);
        rs += mv;
        const float* v = V + static_cast<long long>(sup + 32 * i + src) * LP;
#pragma unroll
        for (int t = 0; t < LAT_MAXT; ++t) {
          const int l = lane + 32 * t;
          if (l < L) acc[t] += mv * sk_ld(v + l);
        }
      }
    }
  }
  return rs;
}

// dist_method == 'cosine' (jamie/jamie.py:485-494, 655-657): the row's loss term is (1 - cos(z, c))^2 instead of |z - c|^2.
// From the row sums z.c, z.z, c.c: returns the loss term; lane 0 leaves the coefficients of its gradient,
//   d/dz = k d (cos z / |z|^2 - c / (|z| |c|)),  d/dc = k d (cos c / |c|^2 - z / (|z| |c|)),  d = 1 - cos, k = the weight k_cos
__device__ __forceinline__ float sk_cos_row(const StepCtx& cx, int i, int row, float szc, float szz, float scc, int lane) {
  const float nz = sqrtf(szz), nc = sqrtf(scc);
  const float cosv = szc / (nz * nc), d = 1.f - cosv;
  if (lane == 0) {
    const float k = cx.gs * cx.sc.w[2] * 32.f * 2.f / (static_cast<float>(cx.B) * static_cast<float>(cx.L));
    const float kd = k * d;
    reinterpret_cast<float4*>(cx.lat_coef)[static_cast<long long>(i) * cx.B + row] = make_float4(kd * cosv / szz, -kd / (nz * nc), kd * cosv / scc, 0.f);
  }
  return d * d;
}
// combine (jamie/model.py:245-259): c_i = (s_i z_i + s_j C_i z_j) / (s_i + s_j rowsum(C_i)), C_0 = corr, C_1 = corr^T.
// Without F the latent loss partials need nothing of another row and are emitted here (fuse_loss).
__device__ __forceinline__ void sk_combine(const StepCtx& cx, int gw, int nw, int lane, int cta, float* sh, int tid, int warp) {
  const int B = cx.B, L = cx.L, LP = cx.LP;
  const int fuse_loss = cx.f_present ? 0 : 1;
  float cmax = 0.f;
  for (int w = gw; w < 2 * B; w += nw) {
    const int i = w / B, row = w - i * B, j = 1 - i;
    const ModCtx& M = cx.m[i];
    const float si = sk_ld(cx.sigma + i), sj = sk_ld(cx.sigma + j);
    const float* Ci = (i == 0 ? cx.corr : cx.corr_t) + static_cast<long long>(row) * B;
    float acc[LAT_MAXT];
    const float rs = sk_row_times(Ci, cx.m[j].z, B, LP, L, lane, acc, cx.corr_hint != nullptr ? cx.corr_hint + w : nullptr);
    const float den = si + sj * rs;
    if (lane == 0) { M.den[row] = den; M.rs[row] = rs; }
    float smu = 0.f, scs = 0.f, sr = 0.f, szc = 0.f, szz = 0.f, scc = 0.f;
#pragma unroll
    for (int t = 0; t < LAT_MAXT; ++t) {
      const int l = lane + 32 * t;
      if (l < L) {
        const long long o = static_cast<long long>(row) * LP + l;
        M.S[o] = acc[t];
        const float zv = sk_ld(M.z + o);
        const float cv = (si * zv + sj * acc[t]) / den;
        M.c[o] = cv;
        cmax = fmaxf(cmax, fabsf(cv));
        if (cx.merge_latent) h_split(cv, M.ch[o], M.cl[o]);   // scale 1; DEC1 re-scales if the global maximum leaves fp16's range
        if (fuse_loss) {
          const float mu = sk_ld(M.mulv.ptr + static_cast<long long>(row) * cx.ldmv + l);
          smu += mu * mu;
          const float d = zv - cv;
          scs += d * d;
          if (cx.cosine) { szc += zv * cv; szz += zv * zv; scc += cv * cv; }
          if (i == 0) { cx.lat_r[o] = cv; sr += cv * cv; }
        }
      }
    }
    if (fuse_loss) {
      smu = warp_sum(smu); scs = warp_sum(scs); sr = warp_sum(sr);
      if (cx.cosine) scs = sk_cos_row(cx, i, row, warp_sum(szc), warp_sum(szz), warp_sum(scc), lane);
      if (lane == 0) {
        float* rp = cx.rowpart + (static_cast<long long>(i) * B + row) * 8;
        rp[0] = smu; rp[1] = scs; rp[2] = sr;
      }
    }
  }
  sk_cta_max_store(cmax, cx.cmax_part, cta, sh, tid, warp, lane);
}
// Row partial sums (rowpart[i][row][k]): 0: sum mu^2  1: sum (z - c)^2  2: sum r^2 (i = 0)  3: sum g z  4: sum g c  5: sum g S
// F residual r = c0 - F c1 (jamie/jamie.py:663-665).
// Also writes the operand planes of c with the dynamic scale s_c (always; the loss part only when F is present).
__device__ __forceinline__ void sk_latloss(const StepCtx& cx, int gw, int nw, int lane, int ncta) {
  const int B = cx.B, L = cx.L, LP = cx.LP;
  const float2 sc = sk_dyn_scale(cx.cmax_part, ncta, lane);
  if (gw == 0 && lane == 0) cx.dyn[0] = sc.y;
  for (int w = gw; w < 2 * B; w += nw) {
    const int i = w / B, row = w - i * B;
    const ModCtx& M = cx.m[i];
#pragma unroll
    for (int t = 0; t < LAT_MAXT; ++t) {
      const int l = lane + 32 * t;
      if (l < L) {
        const long long o = static_cast<long long>(row) * LP + l;
        h_split(sk_ld(M.c + o) * sc.x, M.ch[o], M.cl[o]);
      }
    }
    if (!cx.f_present) continue;
    float acc[LAT_MAXT];
    if (i == 0) sk_row_times(cx.fblk + static_cast<long long>(row) * B, cx.m[1].c, B, LP, L, lane, acc);
    else {
#pragma unroll
      for (int t = 0; t < LAT_MAXT; ++t) acc[t] = 0.f;
    }
    float smu = 0.f, scs = 0.f, sr = 0.f, szc = 0.f, szz = 0.f, scc = 0.f;
#pragma unroll
    for (int t = 0; t < LAT_MAXT; ++t) {
      const int l = lane + 32 * t;
      if (l < L) {
        const long long o = static_cast<long long>(row) * LP + l;
        const float mu = sk_ld(M.mulv.ptr + static_cast<long long>(row) * cx.ldmv + l);
        smu += mu * mu;
        const float zv = sk_ld(M.z + o), cv = sk_ld(M.c + o);
        const float d = zv - cv;
        scs += d * d;
        if (cx.cosine) { szc += zv * cv; szz += zv * zv; scc += cv * cv; }
        if (i == 0) {
          const float r = cv - acc[t];
          cx.lat_r[o] = r;
          sr += r * r;
        }
      }
    }
    smu = warp_sum(smu); scs = warp_sum(scs); sr = warp_sum(sr);
    if (cx.cosine) scs = sk_cos_row(cx, i, row, warp_sum(szc), warp_sum(szz), warp_sum(scc), lane);
    if (lane == 0) {
      float* rp = cx.rowpart + (static_cast<long long>(i) * B + row) * 8;
      rp[0] = smu; rp[1] = scs; rp[2] = sr;
    }
  }
}
// slow path of the optimistic operand scales: re-write the planes of c (d[mu|logvar]) with the scale derived from the
// per-CTA maxima; every CTA takes the same decision (same data). Returns true if the planes were rewritten.
__device__ __forceinline__ bool sk_rescale_c(const StepCtx& cx, int gt, int nt, int lane, int ncta, int* flag, int tid) {
  if (tid < 32) {
    const float2 sc = sk_dyn_scale(cx.cmax_part, ncta, lane);
    if (lane == 0) { flag[0] = sc.x != 1.f ? 1 : 0; reinterpret_cast<float*>(flag)[1] = sc.x; reinterpret_cast<float*>(flag)[2] = sc.y; }
  }
  __syncthreads();
  const bool need = flag[0] != 0;
  const float sx = reinterpret_cast<const float*>(flag)[1], sy = reinterpret_cast<const float*>(flag)[2];
  __syncthreads();
  // every CTA publishes the (identical) inverse scale before its own epilogues read it: no barrier separates this from the
  // GEMM below in the fast path, so a single writer would race with the other CTAs' readers
  if (tid == 0) cx.dyn[0] = need ? sy : 1.f;
  if (!need) return false;
  const int B = cx.B, L = cx.L;
#pragma unroll 1
  for (int t = gt; t < 2 * B * L; t += nt) {
    const int i = t / (B * L), rem = t - i * B * L, b = rem / L, l = rem - b * L;
    const long long o = static_cast<long long>(b) * cx.LP + l;
    h_split(sk_ld(cx.m[i].c + o) * sx, cx.m[i].ch[o], cx.m[i].cl[o]);
  }
  return true;
}
__device__ __forceinline__ bool sk_rescale_dmulv(const StepCtx& cx, int gt, int nt, int lane, int ncta, int* flag, int tid) {
  if (tid < 32) {
    const float2 sc = sk_dyn_scale(cx.dmax_part, ncta, lane);
    if (lane == 0) { flag[0] = sc.x != 1.f ? 1 : 0; reinterpret_cast<float*>(flag)[1] = sc.x; reinterpret_cast<float*>(flag)[2] = sc.y; }
  }
  __syncthreads();
  const bool need = flag[0] != 0;
  const float sx = reinterpret_cast<const float*>(flag)[1], sy = reinterpret_cast<const float*>(flag)[2];
  __syncthreads();
  if (tid == 0) cx.dyn[1] = need ? sy : 1.f;
  if (!need) return false;
  const int B = cx.B, L2 = 2 * cx.L;
#pragma unroll 1
  for (int t = gt; t < 2 * B * L2; t += nt) {
    const int i = t / (B * L2), rem = t - i * B * L2, b = rem / L2, l = rem - b * L2;
    const long long o = static_cast<long long>(b) * cx.ldmv + l;
    h_split(sk_ld(cx.m[i].dmulv + o) * sx, cx.m[i].dmh[o], cx.m[i].dml[o]);
  }
  return true;
}
// g_i = d(loss)/dc_i / den_i with d/dc_i = decoder dgrad - k_cos (z_i - c_i) + F term (everything times the loss scale).
__device__ __forceinline__ void sk_latbc(const StepCtx& cx, int gw, int nw, int lane) {
  const int B = cx.B, L = cx.L, LP = cx.LP;
  const float k_cos = cx.gs * cx.sc.w[2] * 32.f * 2.f / (static_cast<float>(B) * static_cast<float>(L));
  const float k_f = cx.gs * cx.sc.w[3] * 2.f / (static_cast<float>(B) * static_cast<float>(L));
  for (int w = gw; w < 2 * B; w += nw) {
    const int i = w / B, row = w - i * B;
    const ModCtx& M = cx.m[i];
    float acc[LAT_MAXT];
    if (i == 1 && cx.f_present) sk_row_times(cx.fblk_t + static_cast<long long>(row) * B, cx.lat_r, B, LP, L, lane, acc);
    else {
#pragma unroll
      for (int t = 0; t < LAT_MAXT; ++t) acc[t] = 0.f;
    }
    const float den = sk_ld(M.den + row);
    float4 cf = make_float4(0.f, 0.f, 0.f, 0.f);
    if (cx.cosine) cf = sk_ld(reinterpret_cast<const float4*>(cx.lat_coef) + static_cast<long long>(i) * B + row);
    float p3 = 0.f, p4 = 0.f, p5 = 0.f;
#pragma unroll
    for (int t = 0; t < LAT_MAXT; ++t) {
      const int l = lane + 32 * t;
      if (l < L) {
        const long long o = static_cast<long long>(row) * LP + l;
        const float z = sk_ld(M.z + o), c = sk_ld(M.c + o);
        const float dcd = ld_parts(M.dc, o);
        if (M.dc.n > 1) M.dc.ptr[o] = dcd;
        float dc = cx.cosine ? dcd + (cf.y * z + cf.z * c) : dcd - k_cos * (z - c);
        dc += i == 0 ? k_f * sk_ld(cx.lat_r + o) : -k_f * acc[t];
        const float g = dc / den;
        M.g[o] = g;
        p3 += g * z; p4 += g * c; p5 += g * sk_ld(M.S + o);
      }
    }
    p3 = warp_sum(p3); p4 = warp_sum(p4); p5 = warp_sum(p5);
    if (lane == 0) {
      float* rp = cx.rowpart + (static_cast<long long>(i) * B + row) * 8;
      rp[3] = p3; rp[4] = p4; rp[5] = p5;
    }
  }
}
// dz_i = k_cos (z_i - c_i) + s_i g_i + s_i C_i g_j ; then through the reparameterisation and the KL term
// (jamie/jamie.py:619-632 with the reference's logvar quirk: only rows 0 and 1 of modality 1's logvar get KL
// gradient, each scaled by the broadcast over the batch).
__device__ __forceinline__ void sk_latbz(const StepCtx& cx, const StepVars& sv, int gw, int nw, int lane, int cta, float* sh, int tid, int warp) {
  const int B = cx.B, L = cx.L, LP = cx.LP;
  float dmax = 0.f;
  const float k_cos = cx.gs * cx.sc.w[2] * 32.f * 2.f / (static_cast<float>(B) * static_cast<float>(L));
  const float kkl = cx.gs * sv.kl_coef;
  const float fbl = static_cast<float>(B) * static_cast<float>(L);
  for (int w = gw; w < 2 * B; w += nw) {
    const int i = w / B, row = w - i * B, j = 1 - i;
    const ModCtx& M = cx.m[i];
    const float si = sk_ld(cx.sigma + i);
    const float* Ci = (i == 0 ? cx.corr : cx.corr_t) + static_cast<long long>(row) * B;
    float acc[LAT_MAXT];
    sk_row_times(Ci, cx.m[j].g, B, LP, L, lane, acc, cx.corr_hint != nullptr ? cx.corr_hint + w : nullptr);
    float4 cf = make_float4(0.f, 0.f, 0.f, 0.f);
    if (cx.cosine) cf = sk_ld(reinterpret_cast<const float4*>(cx.lat_coef) + static_cast<long long>(i) * B + row);
#pragma unroll
    for (int t = 0; t < LAT_MAXT; ++t) {
      const int l = lane + 32 * t;
      if (l < L) {
        const long long o = static_cast<long long>(row) * LP + l;
        const long long om = static_cast<long long>(row) * cx.ldmv;
        const float mu = sk_ld(M.mulv.ptr + om + l), lv = sk_ld(M.mulv.ptr + om + L + l);
        const float zv = sk_ld(M.z + o), cv = sk_ld(M.c + o);
        const float dz = (cx.cosine ? cf.x * zv + cf.y * cv : k_cos * (zv - cv)) + si * sk_ld(M.g + o) + si * acc[t];
        const float dmu = dz + kkl * mu / fbl;
        float dlv = dz * sk_ld(M.eps + o) * 0.5f * expf(lv * 0.5f);
        if (i == 1 && row < 2) dlv += kkl * -0.5f * (1.f - expf(lv)) / static_cast<float>(L);
        M.dmulv[om + l] = dmu;
        M.dmulv[om + L + l] = dlv;
        if (cx.merge_latent) { h_split(dmu, M.dmh[om + l], M.dml[om + l]); h_split(dlv, M.dmh[om + L + l], M.dml[om + L + l]); }
        dmax = fmaxf(dmax, fmaxf(fabsf(dmu), fabsf(dlv)));
      }
    }
  }
  sk_cta_max_store(dmax, cx.dmax_part, cta, sh, tid, warp, lane);
}
// operand planes of d[mu | logvar] with the dynamic scale s_b (the encoder backward carries it from here on)
__device__ __forceinline__ void sk_dmulv_planes(const StepCtx& cx, int gt, int nt, int lane, int ncta) {
  const int B = cx.B, L2 = 2 * cx.L;
  const float2 sb = sk_dyn_scale(cx.dmax_part, ncta, lane);
  if (gt == 0) cx.dyn[1] = sb.y;
  for (int t = gt; t < 2 * B * L2; t += nt) {
    const int i = t / (B * L2), rem = t - i * B * L2, b = rem / L2, l = rem - b * L2;
    const ModCtx& M = cx.m[i];
    const long long o = static_cast<long long>(b) * cx.ldmv + l;
    h_split(sk_ld(M.dmulv + o) * sb.x, M.dmh[o], M.dml[o]);
  }
}
// FINAL, CTA item 0: loss scalars and d sigma (fixed-order sums); items 1 ..: head bias gradients (16 of the 4L columns).
__device__ __forceinline__ void sk_final_item(const StepCtx& cx, const StepVars& sv, int item, float* sh, int tid, int warp, int lane) {
  const int B = cx.B, L = cx.L;
  if (item > 0) {   // head bias gradients: column sums of d[mu | logvar] (16 columns per item)
    const int col = (item - 1) * 16 + (tid & 15);
    const int slot = tid >> 4;
    const bool cok = col < 4 * L;
    const int i = cok ? col / (2 * L) : 0, cidx = cok ? col - i * 2 * L : 0;
    const float* src = cx.m[i].dmulv + cidx;
    float s = 0.f, dummy = 0.f;
    for (int r0 = slot; r0 < B; r0 += SK_UNR * 32) {
      float v[SK_UNR];
#pragma unroll
      for (int k = 0; k < SK_UNR; ++k) {
        const int r = r0 + k * 32;
        v[k] = (cok && r < B) ? sk_ld(src + static_cast<long long>(r) * cx.ldmv) : 0.f;
      }
#pragma unroll
      for (int k = 0; k < SK_UNR; ++k) s += v[k];
    }
    sk_colsum2(s, dummy, sh, 4, warp, lane);
    if (slot == 0 && cok) {
      float* dst = cx.m[i].dbias_heads + cidx;
      const float v = s * cx.inv_gs;
      *dst = sv.accum ? *dst + v : v;
    }
    return;
  }
  float* tot = sh + 64;    // [14]: [i * 7 + k], k = 0..5 the rowpart sums, k = 6: sum_r (g.c)[r] * rowsum_i[r]
  float* aux = sh + 80;    // [0,1]: sum_l (1 + lv - exp lv) of logvar rows 0 / 1 (modality 1); [2,3]: sum (xhat - x)^2
  float* wpart = sh + 96;  // [SK_WARPS][16] per-warp partial sums
  {
    // every thread takes rows tid, tid + 512, ... of both modalities: the 8 row partials are two 16-byte loads
    float acc[14];
#pragma unroll
    for (int k = 0; k < 14; ++k) acc[k] = 0.f;
    for (int r = tid; r < B; r += SK_THREADS) {
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const float4* rp = reinterpret_cast<const float4*>(cx.rowpart + (static_cast<long long>(i) * B + r) * 8);
        const float4 u = sk_ld(rp), v = sk_ld(rp + 1);
        const float rs = sk_ld(cx.m[i].rs + r);
        acc[i * 7 + 0] += u.x; acc[i * 7 + 1] += u.y; acc[i * 7 + 2] += u.z; acc[i * 7 + 3] += u.w;
        acc[i * 7 + 4] += v.x; acc[i * 7 + 5] += v.y; acc[i * 7 + 6] += v.x * rs;
      }
    }
#pragma unroll
    for (int k = 0; k < 14; ++k) {
      const float t = warp_sum(acc[k]);
      if (lane == 0) wpart[warp * 16 + k] = t;
    }
  }
  if (warp == 14) {
    for (int i = 0; i < 2; ++i) {
      float t1 = 0.f;
      for (int l = lane; l < L; l += 32) {
        const float lv = sk_ld(cx.m[1].mulv.ptr + static_cast<long long>(i) * cx.ldmv + L + l);
        t1 += 1.f + lv - expf(lv);
      }
      t1 = warp_sum(t1);
      if (lane == 0) aux[i] = t1;
    }
  } else if (warp == 15) {
    for (int i = 0; i < 2; ++i) {
      float sacc = 0.f;
      const int nb = cx.m[i].rec_items;
      for (int b = lane; b < nb; b += 32) sacc += sk_ld(cx.m[i].rec_part + b);
      sacc = warp_sum(sacc);
      if (lane == 0) aux[2 + i] = sacc;
    }
  }
  __syncthreads();
  if (tid < 14) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < SK_WARPS; ++w) t += wpart[w * 16 + tid];
    tot[tid] = t;
  }
  __syncthreads();
  if (tid == 0) {
    const float fB = static_cast<float>(B), fL = static_cast<float>(L);
    // KL value (jamie/jamie.py:619-628) with logvars = rows 0/1 of modality 1's logvar
    float kl = 0.f;
    for (int i = 0; i < 2; ++i) kl += -0.5f * (aux[i] / fL - tot[i * 7 + 0] / (fB * fL));
    const float l_kl = sv.kl_base * kl;
    float rec = 0.f;
    for (int i = 0; i < 2; ++i) rec += aux[2 + i] / (fB * static_cast<float>(cx.m[i].D));
    const float l_cos = 32.f * (tot[1] + tot[7 + 1]) / (fB * fL);
    const float l_f = tot[2] / (fB * fL);
    // d sigma (combine backward): i = 0: d s0 += sum g0.z0 - sum g0.c0 ; d s1 += sum g0.S0 - sum (g0.c0) rs0 (and symmetrically)
    const float ds0 = ((tot[3] - tot[4]) + (tot[7 + 5] - tot[7 + 6])) * cx.inv_gs;
    const float ds1 = ((tot[7 + 3] - tot[7 + 4]) + (tot[5] - tot[6])) * cx.inv_gs;
    cx.dsigma[0] = sv.accum ? cx.dsigma[0] + ds0 : ds0;
    cx.dsigma[1] = sv.accum ? cx.dsigma[1] + ds1 : ds1;
    const StepConsts& sc = cx.sc;
    const float total = sc.w[0] * l_kl + sc.w[1] * rec + sc.w[2] * l_cos + sc.w[3] * l_f;
    float* o = cx.out_loss + sv.row * 8;
    o[0] = l_kl; o[1] = rec; o[2] = l_cos; o[3] = l_f; o[4] = total; o[6] = 0.f; o[7] = 0.f;
    float* gt = cx.grad + cx.n_flat;   // 8 floats behind the flat gradients: the data-parallel all-reduce carries them
    gt[0] = l_kl; gt[1] = rec; gt[2] = l_cos; gt[3] = l_f; gt[4] = total;
  }
  __syncthreads();
}

__device__ __forceinline__ void ld8(const float* p, float (&x)[8]) {
  const float4 a = sk_ld(reinterpret_cast<const float4*>(p)), b = sk_ld(reinterpret_cast<const float4*>(p + 4));
  x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = b.x; x[5] = b.y; x[6] = b.z; x[7] = b.w;
}
__device__ __forceinline__ void st8(float* p, const float (&x)[8]) {
  *reinterpret_cast<float4*>(p) = make_float4(x[0], x[1], x[2], x[3]);
  *reinterpret_cast<float4*>(p + 4) = make_float4(x[4], x[5], x[6], x[7]);
}
// decoder dgrad tile d c (L <= 64 columns, no F) -> g = d(loss)/dc / den and the row partials of d sigma: the LATBC phase as
// the tail of the DG3 work item. Thread = (row, group of 8 latent columns): every load of a thread is independent (the
// first version walked 8 rows per warp one after the other: 8 L2 round trips, 19 us for the phase).
__device__ __forceinline__ void sk_tail_latbc(const StepCtx& cx, const ModCtx& M, int mod, const TailArgs& ta, int ks) {
  if (ks) cluster_sync_all();   // K split over the cluster: sum the four staged partial tiles; this CTA finishes rows [32 rank, +32)
  const int B = cx.B, L = cx.L, LP = cx.LP;
  const float k_cos = cx.gs * cx.sc.w[2] * 32.f * 2.f / (static_cast<float>(B) * static_cast<float>(L));
  const float k_f = mod == 0 ? cx.gs * cx.sc.w[3] * 2.f / (static_cast<float>(B) * static_cast<float>(L)) : 0.f;
  const int r = (ks ? 32 * static_cast<int>(ta.rank) : 0) + (ta.tid >> 2), q = ta.tid & 3, row = ta.m0 + r;
  const bool rok = row < B && (!ks || ta.tid < 128);
  const int rr = rok ? row : B - 1;
  const float rden = 1.f / sk_ld(M.den + rr);
  float4 cf = make_float4(0.f, 0.f, 0.f, 0.f);
  if (cx.cosine) cf = sk_ld(reinterpret_cast<const float4*>(cx.lat_coef) + static_cast<long long>(mod) * B + rr);
  float p3 = 0.f, p4 = 0.f, p5 = 0.f;
#pragma unroll 1
  for (int l0 = q * 8; l0 < LP; l0 += 32) {
    const long long o = static_cast<long long>(rr) * LP + l0;
    float z[8], c[8], S[8], lr[8], g[8];
    ld8(M.z + o, z); ld8(M.c + o, c); ld8(M.S + o, S); ld8(cx.lat_r + o, lr);
    float4 d0, d1;
    if (ks) {
      d0 = make_float4(0.f, 0.f, 0.f, 0.f); d1 = d0;
      const int rs = ta.tid < 128 ? r : 0;
#pragma unroll
      for (uint32_t rk = 0; rk < HG_CLUSTER; ++rk) {
        const float4 a = ld_shared_cluster_f4(mapa_shared(smem_u32(hg_stage_ptr(ta.stage, rs, l0)), rk));
        const float4 b = ld_shared_cluster_f4(mapa_shared(smem_u32(hg_stage_ptr(ta.stage, rs, l0 + 4)), rk));
        d0.x += a.x; d0.y += a.y; d0.z += a.z; d0.w += a.w; d1.x += b.x; d1.y += b.y; d1.z += b.z; d1.w += b.w;
      }
    } else {
      d0 = *hg_stage_ptr(ta.stage, r, l0); d1 = *hg_stage_ptr(ta.stage, r, l0 + 4);
    }
    const float dcd[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const bool ok = l0 + j < L;
      const float dd = cx.cosine ? cf.y * z[j] + cf.z * c[j] : -k_cos * (z[j] - c[j]);
      g[j] = ok ? (dcd[j] + dd + k_f * lr[j]) * rden : 0.f;
      p3 += g[j] * z[j]; p4 += g[j] * c[j]; p5 += g[j] * S[j];
    }
    if (rok) { st8(M.g + o, g); st8(M.dc.ptr + o, dcd); }
  }
  p3 += __shfl_xor_sync(0xffffffffu, p3, 1); p4 += __shfl_xor_sync(0xffffffffu, p4, 1); p5 += __shfl_xor_sync(0xffffffffu, p5, 1);
  p3 += __shfl_xor_sync(0xffffffffu, p3, 2); p4 += __shfl_xor_sync(0xffffffffu, p4, 2); p5 += __shfl_xor_sync(0xffffffffu, p5, 2);
  if (q == 0 && rok) {
    float* rp = cx.rowpart + (static_cast<long long>(mod) * B + row) * 8;
    rp[3] = p3; rp[4] = p4; rp[5] = p5;
  }
}

// ------------------------------------------------------------------------------------------------ in-kernel gradient exchange
// Data-parallel training without leaving the step kernel (SURVEY.md 8e: one all-reduce of the flat gradient buffer per
// step). Every rank's gradient buffer lives in NVLink symmetric memory and is mapped into every peer (xg[q]); xf[q] is
// rank q's flag / partial block: [0, R) = "gradients ready" epochs (slot = source rank), [16] = "delivered" arrival counter,
// doubles from byte 256: [src rank][SK_MAX_CTAS] partial sums of squares of the reduced slices.
//   1. (after the WGRAD grid barrier) tell every peer "my gradients of this step are complete"; wait for all peers
//   2. reduce-scatter + all-gather in one sweep: this rank owns 1/R of the buffer; each CTA sums its part of the slice over
//      the ranks in rank order (peer loads over NVLink), writes the sum into EVERY rank's buffer (peer stores), and
//      leaves the sum of squares of what it reduced in every rank's partial block: the clip norm of the summed gradient
//      needs no sweep and no further collective
//   3. grid barrier (all of this rank's remote writes are issued and fenced), tell every peer "my slice is delivered";
//      wait for all peers. ADAM then reads the local buffer.
// Spins are bounded (a protocol error traps instead of hanging the box).
// One system-scope fence per side of a flag: release = fence + relaxed store / red, acquire = relaxed polls + fence (a
// .release store / .acquire load per poll would each carry a fence of their own: measured 16 us of fences per exchange).
__device__ __forceinline__ void fence_sys() { asm volatile("fence.acq_rel.sys;" ::: "memory"); }
__device__ __forceinline__ void fence_gpu() { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }
// A system-scope fence costs ~3.5 us on B200 (measured: JB_XCHG_DBG=31 vs 15) and the exchange has four on its critical
// path. Only ONE of them orders accesses that a GPU-scope fence does not already order on this hardware: the one
// between this CTA's peer STORES (slice sums, norm partial) and its "delivered" arrival at the peer, which must wait for
// the NVLink write acknowledgements. The other three sit between accesses to LOCAL memory and a flag: local stores are
// visible to the peers' NVLink loads once they are performed at GPU scope (the L2 is the point of coherence for peer
// accesses too), the sweep's peer loads are .relaxed.sys (never served from L1) and are issued after the flag was
// observed (no load speculation across the bar.sync), and the consumers of what the peers wrote here read L2 (TMA) or
// L1 lines that the GPU-scope acquire invalidates. xfence != 0 (JB_XCHG_FENCE=sys) makes all four system-scope, as the
// PTX memory model formally asks.
__device__ __forceinline__ void fence_light(const StepCtx& cx) { if (cx.xfence) fence_sys(); else fence_gpu(); }
__device__ __forceinline__ unsigned int ld_relaxed_sys_u32(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void xchg_signal(const StepCtx& cx, int slot0, unsigned int epoch, int tid) {
  if (tid < cx.xworld) {
    fence_light(cx);
    asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(cx.xf[tid] + slot0 + cx.xrank), "r"(epoch) : "memory");
  }
}
__device__ __forceinline__ void xchg_wait(const StepCtx& cx, int slot0, unsigned int epoch, int tid) {
  if (tid < cx.xworld) {
    const unsigned int* f = cx.xf[cx.xrank] + slot0 + tid;
    unsigned int spins = 0;
    while (static_cast<int>(ld_relaxed_sys_u32(f) - epoch) < 0)
      if (++spins > (1u << 26)) __trap();
    fence_light(cx);
  }
  __syncthreads();
}
__device__ __forceinline__ float4 ld_sys_f4(const float4* p) {
  float4 v;
  asm volatile("ld.relaxed.sys.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
  return v;
}
// sum of [a, b) (float4 units) over the ranks, in rank order, written to every rank; returns this thread's sum of squares.
// MAXR loads per element are always issued (ranks beyond the world re-read the local buffer and are not added): no
// predicated loads into the register array.
template <int MAXR>
__device__ __forceinline__ double xchg_sweep(const StepCtx& cx, long long a, long long b, int tid) {
  constexpr int U = 8 / MAXR;   // elements per thread per round: U x MAXR = 8 loads of 16 bytes in flight (an NVLink round
                                // trip is 3 - 5 us: with one element per round the sweep was 60 us at two ranks)
  const int R = cx.xworld;
  float sq = 0.f;   // at most a few dozen squares per thread: fp32 here, double from the CTA reduction on (FP64 is slow on B200)
#pragma unroll 1
  for (long long i0 = a + tid; i0 < b; i0 += U * SK_THREADS) {
    float4 v[U][MAXR];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long i = i0 + u * SK_THREADS < b ? i0 + u * SK_THREADS : b - 1;   // clamped, not predicated
#pragma unroll
      for (int q = 0; q < MAXR; ++q) v[u][q] = ld_sys_f4(reinterpret_cast<const float4*>(cx.xg[q < R ? q : cx.xrank]) + i);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long i = i0 + u * SK_THREADS;
      if (i < b) {
        float4 s = v[u][0];
#pragma unroll
        for (int q = 1; q < MAXR; ++q)
          if (q < R) { s.x += v[u][q].x; s.y += v[u][q].y; s.z += v[u][q].z; s.w += v[u][q].w; }
        if (i * 4 < cx.n_flat) sq += s.x * s.x + s.y * s.y + s.z * s.z + s.w * s.w;
#pragma unroll
        for (int q = 0; q < MAXR; ++q)
          if (q < R) reinterpret_cast<float4*>(cx.xg[q])[i] = s;
      }
    }
  }
  return static_cast<double>(sq);
}
// the same sweep through the switch (NVLS): multimem.ld_reduce returns the sum over all ranks' copies of the address in ONE
// load (reduced inside the NVSwitch), multimem.st writes every rank's copy in ONE store: 1/R of the instructions and of
// the bytes through this GPU's links. Every rank receives the same bits; the order of the in-switch sum is the switch's.
__device__ __forceinline__ double xchg_sweep_mc(const StepCtx& cx, long long a, long long b, int tid) {
  constexpr int U = 8;
  float sq = 0.f;
  float4* const mc = reinterpret_cast<float4*>(cx.xmc);
#pragma unroll 1
  for (long long i0 = a + tid; i0 < b; i0 += U * SK_THREADS) {
    float4 v[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long i = i0 + u * SK_THREADS < b ? i0 + u * SK_THREADS : b - 1;   // clamped, not predicated
      asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];"
                   : "=f"(v[u].x), "=f"(v[u].y), "=f"(v[u].z), "=f"(v[u].w) : "l"(mc + i) : "memory");
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long i = i0 + u * SK_THREADS;
      if (i < b) {
        const float4 s = v[u];
        if (i * 4 < cx.n_flat) sq += s.x * s.x + s.y * s.y + s.z * s.z + s.w * s.w;
        asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc + i), "f"(s.x), "f"(s.y), "f"(s.z), "f"(s.w) : "memory");
      }
    }
  }
  return static_cast<double>(sq);
}
// (Measured and removed: the same sweep as TMA bulk copies through the idle operand ring -- R bulk loads per sub-chunk into
// shared memory, sum, R bulk stores. 39.8 vs 40.5 us per exchange at two ranks, i.e. the sweep is bound by the NVLink
// stream, not by load issue; and the bulk loads of peer memory returned stale lines in ~1e-3 of the elements, which the
// .relaxed.sys register loads below cannot.)
__device__ __forceinline__ void sk_exchange(const StepCtx& cx, unsigned int epoch, int cta, int ncta, int tid, double* shd) {
  const int R = cx.xworld, me = cx.xrank;
  if (!(cx.xdbg & 2)) {
    if (cta == 0) xchg_signal(cx, 0, epoch, tid);
    xchg_wait(cx, 0, epoch, tid);
  }
  const long long n4 = (cx.n_flat + 8) / 4;                       // gradients + the 8 loss scalars behind them
  const long long lo = n4 * me / R, hi = n4 * (me + 1) / R;       // this rank's slice
  const long long per = (hi - lo + ncta - 1) / ncta;
  const long long a = lo + per * cta, b = a + per < hi ? a + per : hi;
  double sq = 0.0;
  if (cx.xdbg & 1) sq = 1.0;
  else if (cx.xmc != nullptr) sq = xchg_sweep_mc(cx, a, b, tid);
  else if (R <= 2) sq = xchg_sweep<2>(cx, a, b, tid);
  else if (R <= 4) sq = xchg_sweep<4>(cx, a, b, tid);
  else sq = xchg_sweep<8>(cx, a, b, tid);
  shd[tid] = sq;
  __syncthreads();   // (also: every thread's peer stores of the sweep are ordered before the fence below)
  if (!(cx.xdbg & 4)) {
    for (int o = SK_THREADS / 2; o > 0; o >>= 1) {
      if (tid < o) shd[tid] += shd[tid + o];
      __syncthreads();
    }
  }
  // "delivered": every CTA of every rank counts itself in at every rank (one remote atomic per destination) once its part
  // of the slice and its norm partial are written and fenced; a CTA goes on to ADAM when its own rank's counter shows all
  // R x ncta arrivals of this epoch. No grid barrier and no single signalling CTA on the way (the phase's own grid barrier
  // is skipped as well): the counter orders the local CTAs among themselves too.
  if (tid < R) {
    if (!(cx.xdbg & 8)) reinterpret_cast<double*>(reinterpret_cast<char*>(cx.xf[tid]) + 256)[me * SK_MAX_CTAS + cta] = shd[0];
    if (!(cx.xdbg & 16)) fence_sys();
    if (!(cx.xdbg & 2) || tid == me)
      asm volatile("red.relaxed.sys.global.add.u32 [%0], 1;" ::"l"(cx.xf[tid] + 16) : "memory");
  }
  if (tid == 0) {
    const unsigned int want = epoch * static_cast<unsigned int>(((cx.xdbg & 2) ? 1 : R) * ncta);
    const unsigned int* f = cx.xf[me] + 16;
    unsigned int spins = 0;
    while (static_cast<int>(ld_relaxed_sys_u32(f) - want) < 0)
      if (++spins > (1u << 26)) __trap();
    if (!(cx.xdbg & 16)) fence_light(cx);
  }
  __syncthreads();
  fence_proxy_async_global();   // the reduced gradients (peer stores) -> the Adam stream's bulk loads
}

// ------------------------------------------------------------------------------------------------ clip + Adam
__device__ __forceinline__ void sk_norm(const StepCtx& cx, int cta, int ncta, double* shd, int tid) {
  const long long n4 = cx.n_flat / 4;
  double s = 0.0;
  const float4* g4 = reinterpret_cast<const float4*>(cx.grad);
  const long long stride = static_cast<long long>(ncta) * SK_THREADS;
  for (long long i0 = static_cast<long long>(cta) * SK_THREADS + tid; i0 < n4; i0 += 4 * stride) {   // 4 loads in flight
    float4 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = i0 + u * stride < n4 ? sk_ld(g4 + i0 + u * stride) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int u = 0; u < 4; ++u)
      s += static_cast<double>(v[u].x) * v[u].x + static_cast<double>(v[u].y) * v[u].y + static_cast<double>(v[u].z) * v[u].z +
           static_cast<double>(v[u].w) * v[u].w;
  }
  shd[tid] = s;
  __syncthreads();
  for (int o = SK_THREADS / 2; o > 0; o >>= 1) {
    if (tid < o) shd[tid] += shd[tid + o];
    __syncthreads();
  }
  if (tid == 0) cx.norm_part[cta] = shd[0];
  __syncthreads();
}
// The Adam sweep as a TMA-staged stream (round 2): with plain loads the phase holds 8 x 16 bytes per thread in flight (64 KB
// per SM; 16 loads per thread spill inside the 128-register budget) and ran at 3.9 TB/s. Here one thread moves 8 KB
// chunks of g, m, v, theta into the (idle) operand ring with 1-D bulk copies, ADAM_STAGES - 2 chunks ahead; all threads
// update one float4 of each array in shared memory; m, v, theta and the fp16 planes go back with bulk stores.
constexpr int ADAM_CHUNK = 2048;                 // floats per array per stage
constexpr int ADAM_STAGE_BYTES = 4 * ADAM_CHUNK * 4;
constexpr int ADAM_STAGES = HG_RING_BYTES / ADAM_STAGE_BYTES;   // 6
__device__ __forceinline__ void sk_adam_stream(const StepCtx& cx, uint8_t* ring, uint64_t* bars, int cta, int ncta, int tid,
                                               float coef, float b1, float b2, float eps, float step, float ibc2) {
  const long long nchunk = (cx.n_flat + ADAM_CHUNK - 1) / ADAM_CHUNK;
  const int mine = cta < nchunk ? static_cast<int>((nchunk - cta + ncta - 1) / ncta) : 0;   // chunks cta, cta + ncta, ...
  // bars[0 .. STAGES) are initialised once per launch (k_step prologue); bars[STAGES] holds their parity bits between
  // uses (an initialised mbarrier must not be initialised again)
  uint32_t par = *reinterpret_cast<volatile uint32_t*>(&bars[ADAM_STAGES]);
  __syncthreads();
  auto issue = [&](int k) {   // thread 0: loads of this CTA's k-th chunk
    const long long c = cta + static_cast<long long>(k) * ncta;
    const long long e0 = c * ADAM_CHUNK;
    const long long left = cx.n_flat - e0;
    const uint32_t bytes = static_cast<uint32_t>((left < ADAM_CHUNK ? left : ADAM_CHUNK) * 4);
    uint8_t* st = ring + (k % ADAM_STAGES) * ADAM_STAGE_BYTES;
    uint64_t* bar = &bars[k % ADAM_STAGES];
    mbar_arrive_expect_tx(bar, 4 * bytes);
    bulk_load(st, cx.grad + e0, bytes, bar);
    bulk_load(st + ADAM_CHUNK * 4, cx.adam_m + e0, bytes, bar);
    bulk_load(st + 2 * ADAM_CHUNK * 4, cx.adam_v + e0, bytes, bar);
    bulk_load(st + 3 * ADAM_CHUNK * 4, cx.theta + e0, bytes, bar);
  };
  if (tid == 0)
    for (int k = 0; k < ADAM_STAGES - 2 && k < mine; ++k) issue(k);
#pragma unroll 1
  for (int k = 0; k < mine; ++k) {
    if (tid == 0) {
      bulk_wait_read_1();   // the stores of chunk k - 2 have read their stage: it is the one chunk k + STAGES - 2 lands in
      if (k + ADAM_STAGES - 2 < mine) issue(k + ADAM_STAGES - 2);
    }
    uint8_t* st = ring + (k % ADAM_STAGES) * ADAM_STAGE_BYTES;
    mbar_wait(&bars[k % ADAM_STAGES], (par >> (k % ADAM_STAGES)) & 1u);
    par ^= 1u << (k % ADAM_STAGES);
    const long long c = cta + static_cast<long long>(k) * ncta;
    const long long e0 = c * ADAM_CHUNK;
    const long long left = cx.n_flat - e0;
    const int n = static_cast<int>(left < ADAM_CHUNK ? left : ADAM_CHUNK);
    float4* sg = reinterpret_cast<float4*>(st);
    float4* sm = sg + ADAM_CHUNK / 4;
    float4* sv4 = sm + ADAM_CHUNK / 4;
    float4* stt = sv4 + ADAM_CHUNK / 4;
    const bool act = tid * 4 < n;
    float4 g4 = make_float4(0.f, 0.f, 0.f, 0.f), m4 = g4, v4 = g4, t4 = g4;
    if (act) { g4 = sg[tid]; m4 = sm[tid]; v4 = sv4[tid]; t4 = stt[tid]; }
    __syncthreads();   // the planes below overwrite the g part of the stage, which other threads read above
    if (act) {
      const float gx[4] = {g4.x * coef, g4.y * coef, g4.z * coef, g4.w * coef};
      float* mp = reinterpret_cast<float*>(&m4);
      float* vp = reinterpret_cast<float*>(&v4);
      float* tp = reinterpret_cast<float*>(&t4);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        mp[j] = mp[j] + (gx[j] - mp[j]) * (1.f - b1);
        vp[j] = vp[j] * b2 + gx[j] * gx[j] * (1.f - b2);
        const float denom = sqrtf(vp[j]) * ibc2 + eps;
        tp[j] = tp[j] - step * (mp[j] / denom);
      }
      sm[tid] = m4; sv4[tid] = v4; stt[tid] = t4;
      // the planes of theta replace g in the stage: hi in its first half, lo in the second
      split4_store(reinterpret_cast<__half*>(st) + 4 * tid, reinterpret_cast<__half*>(st + ADAM_CHUNK * 2) + 4 * tid, t4.x, t4.y, t4.z, t4.w);
    }
    fence_proxy_async_smem();
    __syncthreads();
    if (tid == 0) {
      const uint32_t bytes = static_cast<uint32_t>(n) * 4;
      bulk_store(cx.adam_m + e0, st + ADAM_CHUNK * 4, bytes);
      bulk_store(cx.adam_v + e0, st + 2 * ADAM_CHUNK * 4, bytes);
      bulk_store(cx.theta + e0, st + 3 * ADAM_CHUNK * 4, bytes);
      bulk_store(cx.theta_hi + e0, st, bytes / 2);
      bulk_store(cx.theta_lo + e0, st + ADAM_CHUNK * 2, bytes / 2);
      tma_store_commit();
    }
  }
  if (tid == 0) {
    tma_store_wait_all();       // every bulk store complete
    fence_proxy_async_all();    // async-proxy writes -> generic / async reads after the next grid barrier
    *reinterpret_cast<volatile uint32_t*>(&bars[ADAM_STAGES]) = par;
  }
  __syncthreads();
}
// every CTA re-reduces the partials in the same order (identical clip coefficient everywhere), then
// g *= grad_scale * clip;  m, v, theta updated with torch.optim.Adam's formulas (jamie/jamie.py:739-741).
// theta, m, v are not prefetched into L2 during WGRAD: measured on B200, a bulk L2 prefetch by the warps without a GEMM
// role took 3.5 us off ADAM but added 9.4 us to WGRAD (it competes with the operand loads).
__device__ __forceinline__ void sk_adam(const StepCtx& cx, const StepVars& sv, int cta, int ncta, double* shd, int tid, bool fused_norm, uint8_t* ring, uint64_t* abars) {
  double s = 0.0;
  if (cx.xworld > 1) {   // partial sums of squares of the reduced slices, delivered by every rank (sk_exchange)
    const double* xp = reinterpret_cast<const double*>(reinterpret_cast<const char*>(cx.xf[cx.xrank]) + 256);
    for (int i = tid; i < cx.xworld * SK_MAX_CTAS; i += SK_THREADS)
      if (i % SK_MAX_CTAS < ncta) s += sk_ld(xp + i);
  } else if (fused_norm) {
    for (int i = tid; i < cx.n_norm_tile; i += SK_THREADS) s += static_cast<double>(sk_ld(cx.norm_tile + i));
    for (int i = tid; i < 4 * ncta; i += SK_THREADS) s += static_cast<double>(sk_ld(cx.norm_small + i));
  } else {
    for (int i = tid; i < ncta; i += SK_THREADS) s += sk_ld(cx.norm_part + i);
  }
  shd[tid] = s;
  __syncthreads();
  for (int o = SK_THREADS / 2; o > 0; o >>= 1) {
    if (tid < o) shd[tid] += shd[tid + o];
    __syncthreads();
  }
  const StepConsts& sc = cx.sc;
  const double norm = sqrt(shd[0]) * static_cast<double>(sc.grad_scale);
  const float coef = static_cast<float>(fmin(1.0, static_cast<double>(sc.max_norm) / (norm + 1e-6))) * sc.grad_scale;
  if (cta == 0 && tid == 0) cx.out_loss[sv.row * 8 + 5] = static_cast<float>(norm);
  __syncthreads();
  const float b1 = sc.beta1, b2 = sc.beta2, eps = sc.adam_eps;
  const float step = sv.step_size, ibc2 = sv.inv_bc2_sqrt;
  sk_adam_stream(cx, ring, abars, cta, ncta, tid, coef, b1, b2, eps, step, ibc2);
}

// sum of squares of the gradients of the small tensors (everything that is not a weight matrix): 128 threads per CTA
// (the four warps without a role during WGRAD), one partial per warp
__device__ __forceinline__ void sk_norm_small(const StepCtx& cx, int cta, int ncta, int w4, int lane) {
  const int gt = (cta * 4 + w4) * 32 + lane, nt = ncta * 128;
  float s = 0.f;
  int base = 0;
#pragma unroll 1
  for (int r = 0; r < cx.n_norm_rng; ++r) {
    const int len = cx.norm_rng[r][1];
    const float* g = cx.grad + cx.norm_rng[r][0];
    // element e of the concatenated ranges belongs to thread e mod nt
    int first = gt - (base % nt);
    if (first < 0) first += nt;
#pragma unroll 1
    for (int i = first; i < len; i += nt) { const float v = sk_ld(g + i); s += v * v; }
    base += len;
  }
  s = warp_sum(s);
  if (lane == 0) cx.norm_small[cta * 4 + w4] = s;
}

// running_mean / running_var of the eight BatchNorm layers from the batch statistics the fused forward tails stored
// (jamie/model.py BatchNorm1d, momentum 0.1, unbiased variance). Runs on warps without a GEMM role at the start of WGRAD,
// i.e. once per forward pass and off the critical path (in the tail it was four serialised L2 round trips: 2.4 us).
__device__ __forceinline__ void sk_running_stats(const StepCtx& cx, int gt, int nt) {
  const float fB = static_cast<float>(cx.B);
  const float ub = cx.B > 1 ? fB / static_cast<float>(cx.B - 1) : 1.f;
#pragma unroll 1
  for (int ki = 0; ki < 8; ++ki) {
    const BnLayer& Lr = cx.bn[ki >> 1][ki & 1];
#pragma unroll 1
    for (int c = gt; c < Lr.N; c += nt) {
      const float m = sk_ld(Lr.mean + c), v = sk_ld(Lr.var + c);
      Lr.run_mean[c] = (1.f - BN_MOM) * Lr.run_mean[c] + BN_MOM * m;
      Lr.run_var[c] = (1.f - BN_MOM) * Lr.run_var[c] + BN_MOM * v * ub;
    }
  }
}

// theta -> fp16 planes over the whole flat buffer (after jb_set_params)
__global__ void k_hsplit_flat(const float* __restrict__ src, __half* __restrict__ hi, __half* __restrict__ lo, long long n) {
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<long long>(gridDim.x) * blockDim.x)
    h_split(src[i], hi[i], lo[i]);
}
// fp32 -> fp16 over a flat buffer (the folded inference weights)
__global__ void k_to_half(const float* __restrict__ src, __half* __restrict__ dst, long long n) {
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<long long>(gridDim.x) * blockDim.x)
    dst[i] = __float2half_rn(src[i]);
}
__global__ void k_set_accum(Ctl* ctl, int v) { ctl->accum = v; }
// after a launch of k_step: advance the plan cursor / optimizer step count / Philox stream, clear the injection flag
__global__ void k_ctl_advance(Ctl* ctl, int d_cursor, int d_adam, int clear_inject) {
  ctl->cursor += d_cursor;
  ctl->stream_id += static_cast<unsigned long long>(d_cursor);
  ctl->adam_t += d_adam;
  if (clear_inject) ctl->inject = 0;
}

// ------------------------------------------------------------------------------------------------ the kernel
// Runs phases [ph_lo, ph_hi) of `nsteps` consecutive steps (plan rows ctl->cursor ...). A launch that contains PH_ADAM
// uses optimizer step counts ctl->adam_t + 1 ...; the host advances ctl with k_ctl_advance after the launch.
// use_stage: the batch rows were copied into ModCtx::stage[ctl->host_slot] (host-batch step). row_bias: -1 for an
// update-only launch (the cursor was already advanced by the backward launch). ts (optional): CTA 0 records the global
// timer at kernel start (ts[0]) and at the end of every phase (ts[1 + step * PH_COUNT + phase]); behind those, every CTA
// records {SM clock at phase begin, SM clock at the end of its work, global time at the end of its work} per phase.
// The launch is self-contained (no memset / control kernels around it, which cost a stream operation each in the split
// data-parallel and host-batch paths): `bar` points at the barrier counter of this launch, bar_next at the one of the
// next launch, which is zeroed here; when the last phase is done CTA 0 advances the control block by adv = {plan rows, optimizer
// steps, clear the injection flag} (every CTA read it before its first grid barrier).
__global__ void __launch_bounds__(SK_THREADS, 1) k_step(const __grid_constant__ StepParams prm, int ph_lo, int ph_hi, int nsteps,
                                                         unsigned int* bar, int use_stage, int row_bias,
                                                         unsigned long long* ts, int3 adv, unsigned int* bar_next) {
  extern __shared__ uint8_t sk_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(sk_smem_raw) + 1023) & ~uintptr_t(1023));
  HgCtrl* ctrl = reinterpret_cast<HgCtrl*>(smem);
  StepVars* svp = reinterpret_cast<StepVars*>(smem + 896);
  HgTile* first_tiles = reinterpret_cast<HgTile*>(smem + 256);   // [SK_NUM_GEMM] this CTA's first work item of every GEMM phase
  uint8_t* ring = smem + HG_CTRL_BYTES;
  uint8_t* stage = ring + HG_RING_BYTES;
  float* sh = reinterpret_cast<float*>(stage);            // reduction scratch of the element-wise phases (GEMM idle)
  double* shd = reinterpret_cast<double*>(stage + 4096);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int cta = blockIdx.x, ncta = gridDim.x;
  const int gw = cta * SK_WARPS + warp, nw = ncta * SK_WARPS;
  const StepCtx& cx = prm.cx;
  static_assert(sizeof(HgCtrl) <= 192 && (ADAM_STAGES + 1) * 8 <= 64 && sizeof(HgTile) * SK_NUM_GEMM <= 640 && sizeof(StepVars) <= 128, "control block layout");
  if (warp == 2 && lane < SK_NUM_GEMM && cta < cx.gph[lane].total_tiles) first_tiles[lane] = hg_decode(prm.probs, cx.gph[lane], cta);
  if (tid == 0) {   // barriers of the Adam stream (sk_adam_stream) + their parity word
    uint64_t* abars = reinterpret_cast<uint64_t*>(smem + 192);
    for (int s = 0; s < ADAM_STAGES; ++s) mbar_init(&abars[s], 1);
    abars[ADAM_STAGES] = 0;
  }
  const uint32_t tmem_d = hg_setup(ctrl, warp, lane);   // (fences the barrier initialisation, __syncthreads)
  HgPipe pp;
  unsigned int target = 0;
  if (cta == 0 && tid == 0) *bar_next = 0u;
  const int B = cx.B;
  // the counters CTA 0 advances at the end are read once, before this CTA's first grid barrier (used by thread 0 only)
  long long ctl_cursor0 = 0, ctl_adam0 = 0;
  unsigned long long ctl_stream0 = 0;
  if (tid == 0) { ctl_cursor0 = cx.ctl->cursor; ctl_adam0 = cx.ctl->adam_t; ctl_stream0 = cx.ctl->stream_id; }
  const long long ctl_xepoch = cx.xworld > 1 ? cx.ctl->adam_t - cx.x_adam0 : 0;   // exchange epochs = optimizer steps: the same on every rank

  const bool norm_fused = ph_lo <= PH_DG3 && ph_hi > PH_ADAM && cx.xworld <= 1;   // every weight-gradient epilogue of the step is in this launch
  if (ts != nullptr && cta == 0 && tid == 0) ts[0] = globaltimer_ns();
  long long clk_begin = clock64();
  for (int s = 0; s < nsteps; ++s) {
    if (tid == 0) {
      StepVars v;
      const long long cursor0 = ctl_cursor0, adam0 = ctl_adam0;
      const unsigned long long stream0 = ctl_stream0, seed = cx.ctl->seed;
      const int inject = cx.ctl->inject, accum = cx.ctl->accum, host_slot = cx.ctl->host_slot;
      v.row = cursor0 + s + row_bias;
      const long long t = adam0 + s + 1;
      v.kl_base = cx.plan_kl[v.row];
      v.kl_coef = cx.sc.w[0] * v.kl_base;
      const double bc1 = 1.0 - pow(static_cast<double>(cx.sc.beta1), static_cast<double>(t));
      const double bc2 = 1.0 - pow(static_cast<double>(cx.sc.beta2), static_cast<double>(t));
      v.step_size = static_cast<float>(static_cast<double>(cx.sc.lr) / bc1);
      v.inv_bc2_sqrt = static_cast<float>(1.0 / sqrt(bc2));
      const unsigned long long sid = stream0 + static_cast<unsigned long long>(s) + 1ull;
      const unsigned long long k = seed ^ (sid * 0x9E3779B97F4A7C15ull);
      v.key = make_uint2(static_cast<uint32_t>(k), static_cast<uint32_t>(k >> 32));
      v.inject = inject; v.accum = accum; v.host_slot = host_slot;
      *svp = v;
    }
    __syncthreads();
    const StepVars& sv = *svp;

    for (int ph = ph_lo; ph < ph_hi; ++ph) {
      if (!((cx.phase_mask >> ph) & 1ull) || (ph == PH_NORM && norm_fused)) {   // phase folded away: no work, no barrier
        if (ts != nullptr && tid == 0) {
          unsigned long long* d = ts + 1 + static_cast<long long>(nsteps) * PH_COUNT + ((static_cast<long long>(s) * PH_COUNT + ph) * ncta + cta) * 3;
          d[0] = d[1] = static_cast<unsigned long long>(clk_begin);
          d[2] = globaltimer_ns();
          if (cta == 0) ts[1 + s * PH_COUNT + ph] = d[2];
        }
        continue;
      }
      const int gi = gemm_index(ph);
      if (gi >= 0) {
        if (ts != nullptr && cta == 0) {   // role stamps of CTA 0's first tile (profiling)
          pp.dbg = reinterpret_cast<long long*>(ts + 1 + static_cast<long long>(nsteps) * PH_COUNT * (1 + 3 * ncta)) +
                   (static_cast<long long>(s) * SK_NUM_GEMM + gi) * 8;
          if (tid == 0) pp.dbg[7] = clk_begin;
        }
        const HgPhase& gphase = cx.gph[gi];
        if (ph == PH_WGRAD && warp >= HG_WARP_EPI0 + HG_NEPI) {
          if (!((cx.phase_mask >> PH_BN1) & 1ull)) sk_running_stats(cx, cta * 128 + (tid - 32 * (HG_WARP_EPI0 + HG_NEPI)), ncta * 128);
          if (norm_fused) sk_norm_small(cx, cta, ncta, warp - (HG_WARP_EPI0 + HG_NEPI), lane);
        }
        if (ph == PH_ENC1 && cx.eps_early && warp >= HG_WARP_EPI0 + HG_NEPI)
          sk_draw_eps(cx, sv, cta * 128 + (tid - 32 * (HG_WARP_EPI0 + HG_NEPI)), ncta * 128);
        if (cx.merge_latent && (ph == PH_DEC1 || ph == PH_DGH)) {
          // optimistic operand scales: COMBINE / LATBZ wrote the planes of c / d[mu|logvar] with scale 1; if a value left
          // fp16's range every CTA sees the same maxima, rewrites the planes with the exact power-of-two scale and meets
          // at an extra grid barrier
          const bool redo = ph == PH_DEC1 ? sk_rescale_c(cx, cta * SK_THREADS + tid, ncta * SK_THREADS, lane, ncta, reinterpret_cast<int*>(sh), tid)
                                          : sk_rescale_dmulv(cx, cta * SK_THREADS + tid, ncta * SK_THREADS, lane, ncta, reinterpret_cast<int*>(sh), tid);
          if (redo) {
            target += static_cast<unsigned int>(ncta);
            grid_barrier(bar, target);
          }
        }
        hg_run_phase(prm.probs, gphase, cta, ncta, ctrl, ring, stage, tmem_d, pp, warp, lane, first_tiles + gi,
                     [&](const HgTile& T, const HgProblem& P, bool more) {
          TailArgs ta;
          ta.stage = stage; ta.scr = reinterpret_cast<float*>(ring); ta.keep = smem + 1024; ta.m0 = T.m0; ta.n0 = T.n0; ta.bn = T.bn;
          ta.tid = tid; ta.warp = warp; ta.lane = lane; ta.rank = static_cast<uint32_t>(cta & (HG_CLUSTER - 1));
          ta.stamp = nullptr;
          if (ts != nullptr && cta == 0) {
            ta.stamp = reinterpret_cast<long long*>(ts + 1 + static_cast<long long>(nsteps) * PH_COUNT * (1 + 3 * ncta) + static_cast<long long>(nsteps) * SK_NUM_GEMM * 8) +
                       (static_cast<long long>(s) * PH_COUNT + ph) * 8;
            if (tid == 0) ta.stamp[7] = clk_begin;
          }
          const int arg = P.fuse_arg;
          switch (P.fuse) {
            case FUSE_BN_FWD: sk_tail_bn_fwd(cx, sv, cx.bn[arg >> 1][arg & 1], P.bias, ta); break;
            case FUSE_BN_BWD: sk_tail_bn_bwd(cx, sv, cx.bn[arg >> 1][arg & 1], ta); break;
            case FUSE_REC: sk_tail_rec(cx, sv, cx.m[arg], P.bias, ta); break;
            case FUSE_HEADS: sk_tail_heads(cx, sv, cx.m[arg], arg, P.bias, ta, P.fuse_ks); break;
            case FUSE_LATBC: sk_tail_latbc(cx, cx.m[arg], arg, ta, P.fuse_ks); break;
            default: break;
          }
          fence_proxy_async_smem();   // the scratch is operand-ring memory: generic accesses before the next TMA writes
          if (more) cluster_sync_all();   // the peers have read this CTA's exchange buffer; staging blocks reusable
        },
                     [&](const HgTile& T, const HgProblem& P, int side) {
          if (P.fuse == FUSE_BN_FWD || P.fuse == FUSE_BN_BWD)
            sk_side_mask(cx, sv, cx.bn[P.fuse_arg >> 1][P.fuse_arg & 1], T, smem + 1024, side, lane);
        });
        if (warp == HG_WARP_TMA && lane == 0) {
          // the tensor maps of this CTA's first work item of the NEXT GEMM phase (a TMA issue stalls on a cold descriptor:
          // four of them cost ~1.6 us at the head of every GEMM phase)
          const int gn = gi + 1 == SK_NUM_GEMM ? 0 : gi + 1;
          if (cta < cx.gph[gn].total_tiles && !first_tiles[gn].null) {
            const HgProblem& Pn = prm.probs[first_tiles[gn].p];
            tma_prefetch_desc(&Pn.tmA_hi); tma_prefetch_desc(&Pn.tmB_hi);
            if (Pn.mode != HG_SINGLE) { tma_prefetch_desc(&Pn.tmA_lo); tma_prefetch_desc(&Pn.tmB_lo); }
          }
        }
        if (cx.merge_latent && (ph == PH_DGH || ph == PH_DG2)) {
          // head bias gradients (DGH) and loss scalars + d sigma (DG2): CTAs from the top down, which have no GEMM work in
          // these phases at the headline shape (80 resp. 128 work items on 132 CTAs)
          const int nitems = 1 + (4 * cx.L + 15) / 16;
          for (int it = ph == PH_DG2 ? 0 : 1; it < (ph == PH_DG2 ? 1 : nitems); ++it)
            if ((ncta - 1 - (it % ncta)) == cta) { __syncthreads(); sk_final_item(cx, sv, it, sh, tid, warp, lane); }
        }
      } else {
        switch (ph) {
          case PH_GATHER: {
            // warp items: B rows of the P / F blocks (from the top of the grid down), then 2 B batch rows
            const long long base = sv.row * B;
            if (cx.p_diag != nullptr && cx.p_dense == nullptr && cx.f_dense == nullptr) {   // 2 B rows of corr / corr^T, then 2 B batch rows
              for (int it = nw - 1 - gw; it < 4 * B; it += nw) {
                if (it < 2 * B) sk_corr_row_diag(cx, base, it, lane);
                else sk_gather_row(cx, sv, use_stage, it - 2 * B, lane);
              }
            } else {
              for (int it = nw - 1 - gw; it < 3 * B; it += nw) {
                if (it < B) sk_corr_row(cx, base, it, lane);
                else sk_gather_row(cx, sv, use_stage, it - B, lane);
              }
            }
            break;
          }
          case PH_BN1: case PH_BN2: case PH_BN3: case PH_BN4: {
            const int which = ph == PH_BN1 ? 0 : (ph == PH_BN2 ? 1 : (ph == PH_BN3 ? 2 : 3));
            const int lcw = cx.bn[which][0].lcw;
            const int nb0 = (cx.bn[which][0].N + (1 << lcw) - 1) >> lcw, nb1 = (cx.bn[which][1].N + (1 << lcw) - 1) >> lcw;
            for (int it = cta; it < nb0 + nb1; it += ncta) {
              const int i = it >= nb0 ? 1 : 0;
              long long* est = nullptr;
              if (ts != nullptr && cta == 0 && it == cta) {
                est = reinterpret_cast<long long*>(ts + 1 + static_cast<long long>(nsteps) * PH_COUNT * (1 + 3 * ncta) + static_cast<long long>(nsteps) * SK_NUM_GEMM * 8) +
                      (static_cast<long long>(s) * PH_COUNT + ph) * 8;
                if (tid == 0) est[7] = clk_begin;
              }
              sk_bn_fwd_item(cx.bn[which][i], cx, sv, it - (i ? nb0 : 0), reinterpret_cast<float*>(ring), sh, tid, warp, lane, est);
              __syncthreads();
              if (est != nullptr && tid == 0) est[6] = clock64();
            }
            fence_proxy_async_smem();   // the slab is operand-ring memory: generic writes before the next TMA writes
            break;
          }
          case PH_BNB1: case PH_BNB2: case PH_BNB3: case PH_BNB4: {
            const int which = ph == PH_BNB1 ? 0 : (ph == PH_BNB2 ? 1 : (ph == PH_BNB3 ? 2 : 3));
            const int lcw = cx.bn[which][0].lcw;
            const int nb0 = (cx.bn[which][0].N + (1 << lcw) - 1) >> lcw, nb1 = (cx.bn[which][1].N + (1 << lcw) - 1) >> lcw;
            for (int it = cta; it < nb0 + nb1; it += ncta) {
              const int i = it >= nb0 ? 1 : 0;
              sk_bn_bwd_item(cx.bn[which][i], cx, sv, it - (i ? nb0 : 0), reinterpret_cast<float*>(ring), sh, tid, warp, lane);
              __syncthreads();
            }
            fence_proxy_async_smem();
            break;
          }
          case PH_REC: {
            const int lcw = cx.m[0].rec_lcw;
            const int nb0 = (cx.m[0].D + (1 << lcw) - 1) >> lcw, nb1 = (cx.m[1].D + (1 << lcw) - 1) >> lcw;
            for (int it = cta; it < nb0 + nb1; it += ncta) {
              const int i = it >= nb0 ? 1 : 0;
              sk_rec_item(cx.m[i], cx, sv, it - (i ? nb0 : 0), it - (i ? nb0 : 0), sh, tid, warp, lane);
            }
            break;
          }
          case PH_REPARAM: sk_reparam(cx, sv, cta * SK_THREADS + tid, ncta * SK_THREADS); break;
          case PH_COMBINE: sk_combine(cx, gw, nw, lane, cta, sh, tid, warp); break;
          case PH_LATLOSS: sk_latloss(cx, gw, nw, lane, ncta); break;
          case PH_LATBC: sk_latbc(cx, gw, nw, lane); break;
          case PH_LATBZ: sk_latbz(cx, sv, gw, nw, lane, cta, sh, tid, warp); break;
          case PH_LATFIN: {
            // operand planes of d[mu | logvar]; then FINAL (loss scalars, d sigma, head bias gradients) on the CTAs from
            // the top down
            sk_dmulv_planes(cx, cta * SK_THREADS + tid, ncta * SK_THREADS, lane, ncta);
            const int nitems = 1 + (4 * cx.L + 15) / 16;
            for (int it = 0; it < nitems; ++it)
              if ((ncta - 1 - (it % ncta)) == cta) sk_final_item(cx, sv, it, sh, tid, warp, lane);
            break;
          }
          case PH_NORM:
            if (cx.xworld > 1) sk_exchange(cx, static_cast<unsigned int>(ctl_xepoch + s + 1), cta, ncta, tid, shd);
            else sk_norm(cx, cta, ncta, shd, tid);
            break;
          case PH_ADAM: sk_adam(cx, sv, cta, ncta, shd, tid, norm_fused, ring, reinterpret_cast<uint64_t*>(smem + 192)); break;
          default: break;
        }
      }
      const bool last = (ph == ph_hi - 1) && (s == nsteps - 1);
      if (ts != nullptr) {   // per-CTA detail: SM clock at the end of this CTA's work, global time at that moment
        __syncthreads();
        if (tid == 0) {
          unsigned long long* d = ts + 1 + static_cast<long long>(nsteps) * PH_COUNT + ((static_cast<long long>(s) * PH_COUNT + ph) * ncta + cta) * 3;
          d[0] = static_cast<unsigned long long>(clk_begin);
          d[1] = static_cast<unsigned long long>(clock64());
          d[2] = globaltimer_ns();
        }
      }
      // no barrier between ADAM and the next step's GATHER: the gather / correspondence-block build reads nothing that
      // the optimizer writes and writes nothing that the optimizer reads, so it overlaps Adam's tail; the barrier after
      // GATHER orders both before ENC1
      const bool fused_next = ph == PH_ADAM && ph_lo == PH_GATHER && s + 1 < nsteps;
      const bool xchg_done = ph == PH_NORM && cx.xworld > 1;   // sk_exchange ends with its own (cross-GPU) barrier
      if (!last && !fused_next && !xchg_done) {
        target += static_cast<unsigned int>(ncta);
        grid_barrier(bar, target);
      } else if (fused_next) {
        __syncthreads();   // the next step's StepVars overwrite this step's
      }
      if (ts != nullptr) {
        if (cta == 0 && tid == 0) ts[1 + s * PH_COUNT + ph] = globaltimer_ns();
        clk_begin = clock64();
      }
    }
  }
  if (cta == 0 && tid == 0 && (adv.x | adv.y | adv.z) != 0) {
    Ctl* c = cx.ctl;
    c->cursor = ctl_cursor0 + adv.x;
    c->stream_id = ctl_stream0 + static_cast<unsigned long long>(adv.x);
    c->adam_t = ctl_adam0 + adv.y;
    if (adv.z) c->inject = 0;
  }
  hg_teardown(tmem_d, warp);
}

}  // namespace jb
