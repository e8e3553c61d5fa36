// jamie_b200 engine: device state of one JAMIE model (both modalities' encoder/decoder MLPs, Adam moments, BatchNorm
// statistics, resident datasets) and the C ABI declared in include/jamie_b200.h.
//
// Memory layout:
//   theta / grad / adam_m / adam_v (fp32) : one flat buffer each with the SAME padded layout. Every tensor starts on a
//       128-byte boundary and 2-D weights use a row pitch rounded up to 8 elements so that TMA can address them directly
//       in fp32 and in fp16 (tensor maps need 16-byte aligned bases and pitches). Padding stays zero forever (zero
//       gradient -> zero Adam update), so clip-norm and Adam run over the whole buffer with 128-bit accesses.
//       fc_mus.i / fc_vars.i are stored as ONE [2L, D] matrix per modality (mu rows, then logvar rows): one heads GEMM.
//   theta_hi / theta_lo (fp16)            : the GEMM operand planes of theta (hgemm.cuh), same element offsets,
//       rewritten by every Adam step.
//   activations: [B, pitch] row-major per layer and modality, pitch = width rounded up to 8 elements; GEMM outputs are
//       fp32 (with room for split-K partial sums), GEMM inputs are fp16 hi / lo planes.
// One training step = the phases of ONE persistent cooperative kernel (stepk.cuh); every step-varying scalar (plan row,
// KL anneal, Adam bias corrections, Philox stream) derives from a device-side control block, so jb_train_steps(n) is a
// single launch for n optimizer steps.
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/jamie_b200.h"
#include "gemm_tf32.cuh"
#include "gemm_persistent.cuh"
#include "kernels.cuh"
#include "hgemm.cuh"
#include "stepk.cuh"
#include "metrics.cuh"
#include "distances.cuh"
#include "pcaop.cuh"
#include "impact.cuh"
#include "shapley.cuh"
#include "auroc.cuh"
#include "knn.cuh"
#include "silhouette.cuh"

namespace {

thread_local std::string g_err;
int fail(const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return 1;
}
#define CU(x)                                                                                      \
  do {                                                                                             \
    cudaError_t e_ = (x);                                                                          \
    if (e_ != cudaSuccess) return fail("%s failed: %s (%s:%d)", #x, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

inline int r4(int x) { return (x + 3) & ~3; }
inline int r8(int x) { return (x + 7) & ~7; }
inline long long r32(long long x) { return (x + 31) & ~31LL; }

struct Seg {  // one tensor of the padded flat layout
  long long off = 0;
  int rows = 0, cols = 0, ld = 0;
  long long span() const { return static_cast<long long>(rows) * ld; }
};
struct PackMap {  // packed (reference order) tensor -> location in the padded flat buffer
  long long dst_off;
  int rows, cols, ld;
};

struct ModSegs {
  Seg W1, b1, g1, be1, W2, b2, g2, be2;  // encoder: Linear(D,2D) BN(2D) | Linear(2D,D) BN(D)
  Seg Wmv, bmv;                          // heads: [2L, D] (fc_mus rows, fc_vars rows), [2L]
  Seg W3, b3, g3, be3, W4, b4, g4, be4, W5, b5;  // decoder: Linear(L,D) BN(D) | Linear(D,2D) BN(2D) | Linear(2D,D)
};

using jb::HPlanes;
struct ModActs {  // activations and gradients of one modality (device pointers; pitches in elements)
  float* x; HPlanes xp;
  float* x_stage[2];                                     // host-batch steps: two H2D landing buffers for x
  HPlanes h1, h2, cp, g1, g2;                            // forward GEMM operands
  HPlanes dxhat, dy4, dy3, dmp, dy2, dy1;                // backward GEMM operands
  float* dmulv;
  float *z, *c, *S, *g, *eps, *inj_eps, *den, *rs;
  float *bn_mean[4], *bn_inv[4], *bn_var[4];  // enc1, enc2, dec1, dec2
  unsigned char* inj_mask[4];
  float* rec_part;
  // GEMM outputs (fp32, split-K partial sums; carved per table build)
  jb::Parts y1, y2, mulv, y3, y4, xhat, dg2, dg1, dc, dh2, dh1;
  int ldD, ld2D;
};

}  // namespace

struct HostPin {
  long long cursor_val[2];   // {0, 1}: plan row of a slot, copied into the control block before the step
  int slot_val[2];           // {0, 1}
  float kl[2];
  float losses[2][8];
  int idx[1];                // [slot][modality][Bmax]
};

struct jb_engine {
  jb_config cfg{};
  int D[2]{}, L = 0, LP = 0, ldmv = 0, Bmax = 0;
  // flat parameter layout
  ModSegs ms[2];
  Seg sigma;
  long long n_flat = 0;  // padded float count (multiple of 32)
  std::vector<PackMap> packmap;
  long long n_packed = 0;
  float *theta = nullptr, *grad = nullptr, *adam_m = nullptr, *adam_v = nullptr, *theta_eval = nullptr;
  float* xg[8]{}; unsigned int* xf[8]{}; float* xmc = nullptr; int xrank = 0, xworld = 0; long long x_adam0 = 0;   // in-kernel exchange (jb_set_exchange)
  float* grad_own = nullptr;        // the engine's own gradient buffer while a caller-owned one is in use (jb_set_grad_buffer)
  __half* theta_eval_h = nullptr;   // fp16 copy of the folded inference weights (operands of the fp16 layers of the chain)
  __half *theta_hi = nullptr, *theta_lo = nullptr;   // fp16 operand planes of theta (same element offsets)
  float* state_slab = nullptr;   // one allocation: theta | adam_m | adam_v | theta_hi, theta_lo
  size_t slab_bytes = 0;
  // BatchNorm running statistics: 8 layers in packed order (enc0.1, enc0.5, enc1.1, enc1.5, dec0.1, dec0.5, dec1.1, dec1.5)
  float* bn_run = nullptr;
  long long bn_off[8]{};
  int bn_w[8]{};
  long long n_bn = 0;
  long long nbt[8]{};  // num_batches_tracked (host side; every training step increments all 8)
  // datasets and priors
  float* data[2]{};
  long long data_n[2]{}, data_ld[2]{};
  float *p_diag = nullptr, *p_dense = nullptr, *f_dense = nullptr;
  long long pn0 = 0, pn1 = 0, p_diag_n = 0;
  // plan
  int* plan_idx[2]{};
  float* plan_kl = nullptr;
  float* out_loss = nullptr;
  int plan_cap = 0, plan_steps = 0, plan_B = 0;
  jb::Ctl* ctl = nullptr;
  double* norm_part = nullptr;
  float *norm_tile = nullptr, *norm_small = nullptr;   // fused clip norm (stepk.cuh)
  int norm_tile_cap = 0;
  unsigned int* bar = nullptr;          // grid barrier counters of k_step: [0] and [32], used by alternate launches
  int bar_parity = 0;
  unsigned long long* d_ts = nullptr;   // phase timestamps (profiling)
  // workspaces
  char* arena = nullptr;
  size_t arena_bytes = 0;
  char* parts_arena = nullptr;          // GEMM outputs with their split-K partials (depends on the batch size)
  ModActs act[2]{};
  float *corr = nullptr, *corr_t = nullptr, *fblk = nullptr, *fblk_t = nullptr;
  float *lat_r = nullptr, *rowpart = nullptr, *lat_coef = nullptr;
  int2* corr_hint = nullptr;
  int cosine = 0;                   // jb_set_dist_method
  float *cmax_part = nullptr, *dmax_part = nullptr, *dyn = nullptr;   // dynamic operand scales (stepk.cuh)
  // step tables at batch size step_B
  std::vector<jb::HgProblem> h_probs;
  jb::StepParams* h_prm = nullptr;   // the step kernel's parameter block (host copy; passed by value at every launch)
  jb::StepCtx& h_ctx_ref() { return h_prm->cx; }
  int step_B = 0;
  int grid = 132;            // CTAs of k_step: HG_CLUSTER x the co-resident clusters (33 x 4 on B200; set in jb_create)
  int fused = 0;             // the current step tables use the cluster-fused tails
  int accumulate = 0, accumulate_dev = 0;
  float gs = 1.f;
  // Host-batch steps (data resident on the host): two slots so that the copies of batch k + 1 run while step k computes.
  struct HostPin* h_pin = nullptr;   // pinned: constants, per-slot kl / losses / indices
  cudaStream_t h2d_stream = nullptr;
  cudaEvent_t ev_h2d[2]{}, ev_slot_free[2]{}, ev_loss[2]{};
  bool slot_used[2]{};
  int hb_slot = 0, hb_oldest = 0, hb_outstanding = 0;
  int num_sms = 148;
  // eval
  bool eval_dirty = true;
  int eval_chunk = 8192;     // rows per pass of the folded chain (set in jb_create); activations of a chunk stay in L2
  float *ev_a = nullptr, *ev_b = nullptr, *ev_in = nullptr, *ev_out = nullptr;
  jb::GemmProblem* d_ev_probs = nullptr;
  int ev_probs_cap = 0;
  cudaStream_t ev_stream[2]{};
  cudaEvent_t ev_done[2]{}, ev_free[2]{};
  std::vector<float> prof_gemm;     // last jb_profile_step: per GEMM phase 6 role stamps of CTA 0 (us after the phase began)
  std::vector<float> prof_detail;   // last jb_profile_step: per phase {total, longest CTA work, mean CTA work, barrier tail} us
  long long launches = 0;
};

namespace {

using jb::GemmProblem;

// ------------------------------------------------------------------------------------------- layout
void add_seg(jb_engine* e, Seg& s, int rows, int cols) {
  s.rows = rows; s.cols = cols; s.ld = rows > 1 ? r8(cols) : cols;
  s.off = e->n_flat;
  e->n_flat = r32(e->n_flat + (rows > 1 ? s.span() : cols));
}
void build_layout(jb_engine* e) {
  const int L = e->L;
  e->n_flat = 0;
  add_seg(e, e->sigma, 1, 2);
  for (int i = 0; i < 2; ++i) {
    const int D = e->D[i];
    ModSegs& m = e->ms[i];
    add_seg(e, m.W1, 2 * D, D); add_seg(e, m.b1, 1, 2 * D); add_seg(e, m.g1, 1, 2 * D); add_seg(e, m.be1, 1, 2 * D);
    add_seg(e, m.W2, D, 2 * D); add_seg(e, m.b2, 1, D); add_seg(e, m.g2, 1, D); add_seg(e, m.be2, 1, D);
  }
  for (int i = 0; i < 2; ++i) {
    const int D = e->D[i];
    ModSegs& m = e->ms[i];
    add_seg(e, m.Wmv, 2 * L, D); add_seg(e, m.bmv, 1, 2 * L);
    add_seg(e, m.W3, D, L); add_seg(e, m.b3, 1, D); add_seg(e, m.g3, 1, D); add_seg(e, m.be3, 1, D);
    add_seg(e, m.W4, 2 * D, D); add_seg(e, m.b4, 1, 2 * D); add_seg(e, m.g4, 1, 2 * D); add_seg(e, m.be4, 1, 2 * D);
    add_seg(e, m.W5, D, 2 * D); add_seg(e, m.b5, 1, D);
  }
  // packed (reference named_parameters) order -> flat locations
  auto pm = [&](const Seg& s, int row0, int rows, int cols) {
    PackMap p;
    p.dst_off = s.off + static_cast<long long>(row0) * (s.rows > 1 ? s.ld : 1);
    p.rows = rows; p.cols = cols; p.ld = s.rows > 1 ? s.ld : cols;
    e->packmap.push_back(p);
    e->n_packed += static_cast<long long>(rows) * cols;
  };
  auto whole = [&](const Seg& s) { pm(s, 0, s.rows, s.cols); };
  e->packmap.clear(); e->n_packed = 0;
  whole(e->sigma);
  for (int i = 0; i < 2; ++i) {
    ModSegs& m = e->ms[i];
    whole(m.W1); whole(m.b1); whole(m.g1); whole(m.be1); whole(m.W2); whole(m.b2); whole(m.g2); whole(m.be2);
  }
  for (int i = 0; i < 2; ++i) { pm(e->ms[i].Wmv, 0, L, e->D[i]); pm(e->ms[i].bmv, 0, 1, L); }           // fc_mus
  for (int i = 0; i < 2; ++i) { pm(e->ms[i].Wmv, L, L, e->D[i]); PackMap p; p.dst_off = e->ms[i].bmv.off + L; p.rows = 1; p.cols = L; p.ld = L; e->packmap.push_back(p); e->n_packed += L; }  // fc_vars
  for (int i = 0; i < 2; ++i) {
    ModSegs& m = e->ms[i];
    whole(m.W3); whole(m.b3); whole(m.g3); whole(m.be3); whole(m.W4); whole(m.b4); whole(m.g4); whole(m.be4);
    whole(m.W5); whole(m.b5);
  }
  // BatchNorm running stats
  const int widths[8] = {2 * e->D[0], e->D[0], 2 * e->D[1], e->D[1], e->D[0], 2 * e->D[0], e->D[1], 2 * e->D[1]};
  long long off = 0;
  for (int k = 0; k < 8; ++k) { e->bn_w[k] = widths[k]; e->bn_off[k] = off; off += 2LL * widths[k]; }
  e->n_bn = off;
}

int copy_packed(jb_engine* e, float* flat, float* packed_host, bool to_device) {
  // packed host <-> padded device, tensor by tensor (2-D copies honour the padded pitch)
  long long src = 0;
  for (const PackMap& p : e->packmap) {
    if (to_device)
      CU(cudaMemcpy2D(flat + p.dst_off, static_cast<size_t>(p.ld) * 4, packed_host + src, static_cast<size_t>(p.cols) * 4,
                      static_cast<size_t>(p.cols) * 4, p.rows, cudaMemcpyHostToDevice));
    else
      CU(cudaMemcpy2D(packed_host + src, static_cast<size_t>(p.cols) * 4, flat + p.dst_off, static_cast<size_t>(p.ld) * 4,
                      static_cast<size_t>(p.cols) * 4, p.rows, cudaMemcpyDeviceToHost));
    src += static_cast<long long>(p.rows) * p.cols;
  }
  return 0;
}

// ------------------------------------------------------------------------------------------- arena
struct Carver {
  char* base; size_t off = 0; bool dry;
  explicit Carver(char* b) : base(b), dry(b == nullptr) {}
  template <class T> T* take(size_t n) {
    off = (off + 255) & ~size_t(255);
    T* p = dry ? nullptr : reinterpret_cast<T*>(base + off);
    off += n * sizeof(T);
    return p;
  }
};
void carve(jb_engine* e, Carver& c) {
  const size_t B = e->Bmax;
  for (int i = 0; i < 2; ++i) {
    ModActs& a = e->act[i];
    const int D = e->D[i];
    a.ldD = r8(D); a.ld2D = r8(2 * D);
    auto planes = [&](HPlanes& p, size_t n) { p.hi = c.take<__half>(n); p.lo = c.take<__half>(n); };
    a.x = c.take<float>(B * a.ldD); planes(a.xp, B * a.ldD);
    a.x_stage[0] = c.take<float>(B * a.ldD); a.x_stage[1] = c.take<float>(B * a.ldD);
    planes(a.h1, B * a.ld2D); planes(a.h2, B * a.ldD); planes(a.g1, B * a.ldD); planes(a.g2, B * a.ld2D);
    planes(a.dxhat, B * a.ldD); planes(a.dy4, B * a.ld2D); planes(a.dy3, B * a.ldD);
    a.dmulv = c.take<float>(B * e->ldmv); planes(a.dmp, B * e->ldmv); planes(a.dy2, B * a.ldD); planes(a.dy1, B * a.ld2D);
    a.z = c.take<float>(B * e->LP); a.c = c.take<float>(B * e->LP); planes(a.cp, B * e->LP); a.S = c.take<float>(B * e->LP);
    a.g = c.take<float>(B * e->LP); a.eps = c.take<float>(B * e->LP); a.inj_eps = c.take<float>(B * e->LP);
    a.den = c.take<float>(B); a.rs = c.take<float>(B);
    const int w[4] = {2 * D, D, D, 2 * D};
    for (int k = 0; k < 4; ++k) {
      a.bn_mean[k] = c.take<float>(w[k]); a.bn_inv[k] = c.take<float>(w[k]); a.bn_var[k] = c.take<float>(w[k]);
      a.inj_mask[k] = c.take<unsigned char>(B * w[k]);
    }
    a.rec_part = c.take<float>(D);   // one partial per slab item of the reconstruction phase (at most D items)
  }
  e->corr = c.take<float>(B * B); e->corr_t = c.take<float>(B * B);
  e->fblk = c.take<float>(B * B); e->fblk_t = c.take<float>(B * B);
  e->lat_r = c.take<float>(B * e->LP); e->rowpart = c.take<float>(2 * B * 8); e->lat_coef = c.take<float>(2 * B * 4); e->corr_hint = c.take<int2>(2 * B);
  e->cmax_part = c.take<float>(jb::SK_MAX_CTAS); e->dmax_part = c.take<float>(jb::SK_MAX_CTAS); e->dyn = c.take<float>(8);
}

// ------------------------------------------------------------------------------------------- step tables
// Forward GEMMs and dgrads run the fp32-class 3-pass mode on the fp16 hi / lo planes (HG_PRECISE): pre-activation errors
// flip LeakyReLU' decisions and dX errors propagate down the chain. Weight gradients run three passes without the
// accumulator drains (HG_MEDIUM, ~1e-6): their rounding stays local to the gradient tensor, but a single pass (3e-4 at
// the headline shape, up to 1.2e-3 at small ones, measured in round 1) would eat the whole 1e-3 parity budget.
struct StageSpec {   // one problem of a GEMM phase before its split-K factor is known
  HPlanes A; int lda, a_mn; HPlanes Bm; int ldb, b_mn;
  jb::Parts* out;    // activation output (partials carved later) or null ...
  float* C;          // ... for weight gradients, which go straight into the gradient buffer
  int ldc, M, N, K, bn, mode, epi;
  const float* bias;
  float out_scale;
  int acc_dynamic;
  int dyn;           // index into StepCtx::dyn of an extra dynamic output factor, or -1
  int fuse = 0, fuse_arg = 0, fuse_ks = 0;
};

int build_step(jb_engine* e, int B) {
  const int L = e->L;
  float* T = e->theta;
  float* G = e->grad;
  auto W = [&](const Seg& s) { return HPlanes{e->theta_hi + s.off, e->theta_lo + s.off}; };
  auto bias = [&](const Seg& s) { return T + s.off; };
  // loss scale of the backward pass: d xhat = gs * 2 w (xhat - x) / (B D) is O(xhat - x)
  {
    const int Dm = e->D[0] > e->D[1] ? e->D[0] : e->D[1];
    float wmax = 1.f;
    for (int k = 0; k < 4; ++k) wmax = fmaxf(wmax, fabsf(e->cfg.loss_w[k]));
    const int ex = static_cast<int>(ceil(log2(static_cast<double>(B) * Dm))) - static_cast<int>(ceil(log2(static_cast<double>(wmax))));
    e->gs = ldexpf(1.f, ex < 0 ? 0 : (ex > 30 ? 30 : ex));
  }
  const float inv_gs = 1.f / e->gs;
  // Forward / dgrad mode by reduction length: the tensor core adds products into its fp32 accumulator with truncation, a
  // bias that grows with the number of accumulation steps. Up to K = 1024 (64 steps) three undrained passes (HG_MEDIUM)
  // stay at 7e-6 of the fp32 oracle at the headline shape and save 9 us per step; longer reductions (2000-wide inputs
  // without PCA: measured 6e-4 undrained) keep the drained HG_PRECISE mode.
  auto fmode_for = [](int K) { return static_cast<int>(K <= 1024 ? jb::HG_MEDIUM : jb::HG_PRECISE); };
  std::vector<std::vector<StageSpec>> st(jb::SK_NUM_GEMM);
  // Cluster-fused tails need all rows of a column block in one cluster: B <= HG_CLUSTER M tiles. Larger batches run
  // BatchNorm / reconstruction / reparameterisation as separate slab phases.
  const bool fused = B <= jb::HG_CLUSTER * jb::HG_BM;
  e->fused = fused ? 1 : 0;
  const int nclusters = e->grid / jb::HG_CLUSTER;
  // N tile of the forward / dgrad stages: 64 columns, or 32 when the 64-wide column blocks of both modalities would leave
  // half of the clusters idle (fused) / for narrow outputs
  auto fbn = [&](int N) { return N <= 32 ? 32 : 64; };
  auto fbn2 = [&](int N0, int N1) {
    if (!fused) return 64;
    const int blocks64 = (N0 + 63) / 64 + (N1 + 63) / 64;
    return 2 * blocks64 <= nclusters ? 32 : 64;
  };
  for (int i = 0; i < 2; ++i) {
    ModActs& a = e->act[i]; ModSegs& m = e->ms[i]; const int D = e->D[i];
    auto fwd = [&](int stage, HPlanes X, int ldx, const Seg& w, const Seg& b, jb::Parts* out, int ldy, int n_out, int n_in) {
      StageSpec sp{X, ldx, 0, W(w), w.ld, 0, out, nullptr, ldy, B, n_out, n_in, fbn(n_out), fmode_for(n_in), jb::EPI_BIAS, bias(b), 1.f, 0,
                   stage == 3 ? 0 : -1};   // the c planes carry the dynamic scale s_c
      if (fused) {
        static const int bn_layer[6] = {0, 1, -1, 2, 3, -1};
        if (bn_layer[stage] >= 0) { sp.fuse = jb::FUSE_BN_FWD; sp.fuse_arg = bn_layer[stage] * 2 + i; }
        else if (stage == 5) { sp.fuse = jb::FUSE_REC; sp.fuse_arg = i; }
        else if (stage == 2 && 2 * L <= 64) { sp.fuse = jb::FUSE_HEADS; sp.fuse_arg = i; sp.fuse_ks = n_in >= 8 * jb::HG_BK; }
        // narrow column blocks only pay where the main loop is long (K >= 256); short-K stages keep 64
        if (stage != 2 && n_out > 32 && n_in >= 256) sp.bn = stage == 0 || stage == 4 ? fbn2(2 * e->D[0], 2 * e->D[1]) : fbn2(e->D[0], e->D[1]);
      }
      st[stage].push_back(sp);
    };
    fwd(0, a.xp, a.ldD, m.W1, m.b1, &a.y1, a.ld2D, 2 * D, D);
    fwd(1, a.h1, a.ld2D, m.W2, m.b2, &a.y2, a.ldD, D, 2 * D);
    fwd(2, a.h2, a.ldD, m.Wmv, m.bmv, &a.mulv, e->ldmv, 2 * L, D);
    fwd(3, a.cp, e->LP, m.W3, m.b3, &a.y3, a.ldD, D, L);
    fwd(4, a.g1, a.ldD, m.W4, m.b4, &a.y4, a.ld2D, 2 * D, D);
    fwd(5, a.g2, a.ld2D, m.W5, m.b5, &a.xhat, a.ldD, D, 2 * D);
    // dgrad dX[B, N_in] = dY W   (A = dY planes K-major, B = W planes MN-major, K = N_out)
    auto dgrad = [&](int stage, HPlanes dY, int lddy, const Seg& s, jb::Parts* out, int lddx, int n_out, int n_in) {
      StageSpec sp{dY, lddy, 0, W(s), s.ld, 1, out, nullptr, lddx, B, n_in, n_out, fbn(n_in), fmode_for(n_out), jb::EPI_STORE, nullptr, 1.f, 0, -1};
      if (fused && stage == 8) {   // d c: the LATBC phase becomes the tail (no F, one column block)
        if (e->f_dense == nullptr && L <= 64) { sp.fuse = jb::FUSE_LATBC; sp.fuse_arg = i; sp.fuse_ks = n_out >= 8 * jb::HG_BK; }
      } else if (fused) {   // the dgrad result feeds a BatchNorm backward: stage 6 -> dec2, 7 -> dec1, 9 -> enc2, 10 -> enc1
        const int k = stage == 6 ? 3 : (stage == 7 ? 2 : (stage == 9 ? 1 : 0));
        sp.fuse = jb::FUSE_BN_BWD; sp.fuse_arg = k * 2 + i;
        if (n_in > 32 && n_out >= 256) sp.bn = (k == 0 || k == 3) ? fbn2(2 * e->D[0], 2 * e->D[1]) : fbn2(e->D[0], e->D[1]);
      }
      st[stage].push_back(sp);
    };
    dgrad(6, a.dxhat, a.ldD, m.W5, &a.dg2, a.ld2D, D, 2 * D);
    dgrad(7, a.dy4, a.ld2D, m.W4, &a.dg1, a.ldD, 2 * D, D);
    dgrad(8, a.dy3, a.ldD, m.W3, &a.dc, e->LP, D, L);
    dgrad(9, a.dmp, e->ldmv, m.Wmv, &a.dh2, a.ldD, 2 * L, D);
    dgrad(10, a.dy2, a.ldD, m.W2, &a.dh1, a.ld2D, D, 2 * D);
  }
  // wgrad dW[N_out, N_in] = dY^T X / gs  (A = dY planes MN-major, B = X planes MN-major, K = batch); largest first
  // The two small weight gradients do not wait for the WGRAD phase: d W3 = d y3^T c runs beside the DG3 GEMM (8 + 8 work
  // items at the headline shape) and d Wmv = d[mu|logvar]^T h2 beside DGH, on CTAs those phases leave idle; WGRAD is then
  // exactly one work item per CTA (128 items of 128 x 256 on 132 CTAs).
  auto wgrad = [&](HPlanes dY, int lddy, HPlanes X, int ldx, const Seg& s, int n_out, int n_in, int dyn, int stage = 11) {
    int bn = n_in <= 32 ? 32 : (n_in <= 64 || stage != 11 ? 64 : (n_in >= 256 ? 256 : 128));
    st[stage].push_back(StageSpec{dY, lddy, 1, X, ldx, 1, nullptr, G + s.off, s.ld, n_out, n_in, B, bn, jb::HG_MEDIUM, jb::EPI_STORE, nullptr, inv_gs, 1, dyn});
  };
  for (int i = 0; i < 2; ++i) { ModActs& a = e->act[i]; ModSegs& m = e->ms[i]; const int D = e->D[i];
    // encoder-side gradients carry the dynamic scale s_b of d[mu | logvar] (dyn 1); dW3's B operand is the c planes (dyn 0)
    wgrad(a.dxhat, a.ldD, a.g2, a.ld2D, m.W5, D, 2 * D, -1); wgrad(a.dy4, a.ld2D, a.g1, a.ldD, m.W4, 2 * D, D, -1);
    wgrad(a.dy2, a.ldD, a.h1, a.ld2D, m.W2, D, 2 * D, 1); wgrad(a.dy1, a.ld2D, a.xp, a.ldD, m.W1, 2 * D, D, 1); }
  for (int i = 0; i < 2; ++i) { ModActs& a = e->act[i]; ModSegs& m = e->ms[i]; const int D = e->D[i];
    wgrad(a.dmp, e->ldmv, a.h2, a.ldD, m.Wmv, 2 * L, D, 1, 9); wgrad(a.dy3, a.ldD, a.cp, e->LP, m.W3, D, L, 0, 8); }
  // split-K factor per problem: fill the grid, at least two k-blocks per partial, at most kMaxKsplit partials
  constexpr int kMaxKsplit = 8;
  size_t parts_bytes = 0;
  std::vector<std::vector<int>> ks(jb::SK_NUM_GEMM);
  for (int g = 0; g < jb::SK_NUM_GEMM; ++g) {
    int tiles = 0;
    for (const StageSpec& s : st[g]) tiles += ((s.M + jb::HG_BM - 1) / jb::HG_BM) * ((s.N + s.bn - 1) / s.bn);
    for (const StageSpec& s : st[g]) {
      int k = 1;
      if (s.out != nullptr) {
        const int kb = (s.K + jb::HG_BK - 1) / jb::HG_BK;
        k = s.fuse ? (s.fuse_ks ? jb::HG_CLUSTER : 1) : e->grid / (tiles > 0 ? tiles : 1);
        if (k > kb / 2) k = kb / 2;
        if (k > kMaxKsplit) k = kMaxKsplit;
        if (k < 1) k = 1;
        parts_bytes = ((parts_bytes + 255) & ~size_t(255)) + static_cast<size_t>(k) * s.M * s.ldc * 4;
      }
      ks[g].push_back(k);
    }
  }
  if (e->parts_arena) { cudaFree(e->parts_arena); e->parts_arena = nullptr; }
  CU(cudaMalloc(&e->parts_arena, parts_bytes + 256));
  CU(cudaMemset(e->parts_arena, 0, parts_bytes + 256));
  Carver pc(e->parts_arena);
  e->h_probs.clear();
  if (!e->h_prm) e->h_prm = new jb::StepParams();
  jb::StepCtx& cx = e->h_prm->cx;
  cx = jb::StepCtx{};
  int n_norm_tile = 0;
  for (int g = 0; g < jb::SK_NUM_GEMM; ++g) {
    const int first = static_cast<int>(e->h_probs.size());
    if (st[g].size() > static_cast<size_t>(jb::HG_MAX_PROBS) || e->h_probs.size() + st[g].size() > static_cast<size_t>(jb::SK_MAX_PROBS))
      return fail("too many problems in a GEMM phase");
    for (size_t q = 0; q < st[g].size(); ++q) {
      const StageSpec& s = st[g][q];
      const int k = ks[g][q];
      float* C = s.C;
      long long pstride = 0;
      if (s.out != nullptr) {
        pstride = static_cast<long long>(s.M) * s.ldc;
        C = pc.take<float>(static_cast<size_t>(k) * pstride);
        *s.out = jb::Parts{C, pstride, k};
      }
      jb::HgProblem hp;
      int rc = jb::hg_problem_fill(&hp, s.A, s.lda, s.a_mn, s.Bm, s.ldb, s.b_mn, C, s.ldc, s.M, s.N, s.K, s.bn, s.mode, s.epi, s.bias, k,
                                   pstride, 0, s.out_scale, jb::LRELU);
      if (rc) return fail("hgemm problem fill failed (%d) for M%d N%d K%d lda%d ldb%d bn%d mode%d", rc, s.M, s.N, s.K, s.lda, s.ldb, s.bn, s.mode);
      if (hp.ksplit != k && s.out != nullptr) s.out->n = hp.ksplit;
      if (s.fuse && s.out != nullptr) s.out->n = 1;   // fused tails store the finished tensor (K parts are summed over DSMEM)
      if (s.fuse_ks && hp.ksplit != jb::HG_CLUSTER) return fail("cluster K split needs %d parts, got %d", jb::HG_CLUSTER, hp.ksplit);
      if (s.acc_dynamic) hp.acc_flag = &e->ctl->accum;
      if (s.dyn >= 0) hp.dyn_scale = e->dyn + s.dyn;
      hp.fuse = s.fuse; hp.fuse_arg = s.fuse_arg; hp.fuse_ks = s.fuse_ks;
      if (s.out == nullptr) {   // weight gradient: per-warp sums of squares of what the epilogue stored (offset now, base below)
        hp.norm_out = reinterpret_cast<float*>(static_cast<uintptr_t>(n_norm_tile) * 4 + 4);   // +4: distinguishes offset 0 from "none"
        n_norm_tile += hp.tiles_m * hp.tiles_n * jb::HG_NEPI;
      }
      if (s.fuse && hp.tiles_m > jb::HG_CLUSTER) return fail("fused stage with %d M tiles", hp.tiles_m);
      e->h_probs.push_back(hp);
    }
    cx.gph[g] = jb::hg_phase_finalize(e->h_probs.data(), first, static_cast<int>(st[g].size()));
  }
  if (n_norm_tile > e->norm_tile_cap) {
    if (e->norm_tile) cudaFree(e->norm_tile);
    e->norm_tile = nullptr; e->norm_tile_cap = 0;
    CU(cudaMalloc(&e->norm_tile, static_cast<size_t>(n_norm_tile) * 4));
    e->norm_tile_cap = n_norm_tile;
  }
  if (n_norm_tile > 0) CU(cudaMemset(e->norm_tile, 0, static_cast<size_t>(n_norm_tile) * 4));
  for (jb::HgProblem& hp : e->h_probs)
    if (hp.norm_out != nullptr) hp.norm_out = e->norm_tile + (reinterpret_cast<uintptr_t>(hp.norm_out) - 4) / 4;
  for (size_t q = 0; q < e->h_probs.size(); ++q) e->h_prm->probs[q] = e->h_probs[q];
  // ---- the rest of the step context
  cx.B = B; cx.L = L; cx.LP = e->LP; cx.ldmv = e->ldmv;
  for (int i = 0; i < 2; ++i) {
    ModActs& a = e->act[i]; ModSegs& m = e->ms[i];
    jb::ModCtx& M = cx.m[i];
    M.data = e->data[i]; M.ld_data = e->data_ld[i]; M.stage[0] = a.x_stage[0]; M.stage[1] = a.x_stage[1];
    M.idx = e->plan_idx[i]; M.x = a.x; M.xh = a.xp.hi; M.xl = a.xp.lo;
    M.mulv = a.mulv; M.eps = a.eps; M.z = a.z; M.c = a.c; M.S = a.S; M.g = a.g; M.den = a.den; M.rs = a.rs;
    M.inj_eps = a.inj_eps; M.ch = a.cp.hi; M.cl = a.cp.lo; M.dc = a.dc; M.dmulv = a.dmulv; M.dmh = a.dmp.hi; M.dml = a.dmp.lo;
    M.xhat = a.xhat; M.dxh = a.dxhat.hi; M.dxl = a.dxhat.lo; M.db5 = G + m.b5.off; M.rec_part = a.rec_part;
    M.dbias_heads = G + m.bmv.off; M.D = e->D[i]; M.ldD = a.ldD;
    const int D = e->D[i];
    const struct { jb::Parts Y; HPlanes H; const Seg *g, *be, *b; jb::Parts dH; HPlanes dY; int N, ld; } bl[4] = {
        {a.y1, a.h1, &m.g1, &m.be1, &m.b1, a.dh1, a.dy1, 2 * D, a.ld2D},
        {a.y2, a.h2, &m.g2, &m.be2, &m.b2, a.dh2, a.dy2, D, a.ldD},
        {a.y3, a.g1, &m.g3, &m.be3, &m.b3, a.dg1, a.dy3, D, a.ldD},
        {a.y4, a.g2, &m.g4, &m.be4, &m.b4, a.dg2, a.dy4, 2 * D, a.ld2D}};
    for (int k = 0; k < 4; ++k) {
      jb::BnLayer& l = cx.bn[k][i];
      const int bnidx = k < 2 ? (2 * i + k) : (4 + 2 * i + (k - 2));
      l.Y = bl[k].Y; l.Hh = bl[k].H.hi; l.Hl = bl[k].H.lo;
      l.gamma = T + bl[k].g->off; l.beta = T + bl[k].be->off;
      l.mean = a.bn_mean[k]; l.invstd = a.bn_inv[k]; l.var = a.bn_var[k];
      l.run_mean = e->bn_run + e->bn_off[bnidx]; l.run_var = l.run_mean + e->bn_w[bnidx];
      l.mask = a.inj_mask[k];
      l.dH = bl[k].dH; l.dYh = bl[k].dY.hi; l.dYl = bl[k].dY.lo;
      l.dgamma = G + bl[k].g->off; l.dbeta = G + bl[k].be->off; l.dbias = G + bl[k].b->off;
      l.gdyn = k < 2 ? e->dyn + 1 : nullptr;   // encoder layers sit downstream of d[mu | logvar]
      l.N = bl[k].N; l.ld = bl[k].ld; l.layer_id = static_cast<unsigned>(bnidx);
    }
    M.rec_lcw = 0; M.rec_items = 0;   // set below (both modalities share the slab width of a phase)
  }
  // slab width per element-wise phase: 16 columns per CTA item unless that leaves most of the grid idle (then 8); halved
  // further until the backward slab (2 x B x cw floats) fits the operand ring
  auto slab_lcw = [&](int n0, int n1) {
    int lcw = 4;
    if (((n0 + 15) / 16 + (n1 + 15) / 16) * 10 < e->grid * 6) lcw = 3;
    while (lcw > 0 && static_cast<size_t>(B) * (1u << lcw) * 8 > static_cast<size_t>(jb::HG_RING_BYTES)) --lcw;
    return lcw;
  };
  if (static_cast<size_t>(B) * 8 > static_cast<size_t>(jb::HG_RING_BYTES)) return fail("batch size %d too large for the slab phases", B);
  for (int k = 0; k < 4; ++k) {
    const int lcw = slab_lcw(cx.bn[k][0].N, cx.bn[k][1].N);
    cx.bn[k][0].lcw = cx.bn[k][1].lcw = lcw;
  }
  {
    const int lcw = slab_lcw(e->D[0], e->D[1]);
    for (int i = 0; i < 2; ++i) { cx.m[i].rec_lcw = lcw; cx.m[i].rec_items = (e->D[i] + (1 << lcw) - 1) >> lcw; }
  }
  cx.phase_mask = ~0ull;
  if (fused) {
    for (int ph : {jb::PH_BN1, jb::PH_BN2, jb::PH_BN3, jb::PH_BN4, jb::PH_BNB1, jb::PH_BNB2, jb::PH_BNB3, jb::PH_BNB4, jb::PH_REC})
      cx.phase_mask &= ~(1ull << ph);
    if (2 * L <= 64) { cx.phase_mask &= ~(1ull << jb::PH_REPARAM); cx.eps_early = 1; }
    for (int i = 0; i < 2; ++i) {   // one squared-error partial per (column block, cluster rank) of the last decoder GEMM
      const jb::HgProblem& hp = e->h_probs[cx.gph[5].first + i];
      cx.m[i].rec_items = hp.tiles_n * jb::HG_CLUSTER;
    }
  }
  cx.norm_tile = e->norm_tile; cx.norm_small = e->norm_small; cx.n_norm_tile = n_norm_tile;
  {
    int nr = 0;
    auto rng = [&](const Seg& sg) { cx.norm_rng[nr][0] = static_cast<int>(sg.off); cx.norm_rng[nr][1] = sg.cols; ++nr; };
    rng(e->sigma);
    for (int i = 0; i < 2; ++i) {
      const ModSegs& m = e->ms[i];
      for (const Seg* sg : {&m.b1, &m.g1, &m.be1, &m.b2, &m.g2, &m.be2, &m.bmv, &m.b3, &m.g3, &m.be3, &m.b4, &m.g4, &m.be4, &m.b5}) rng(*sg);
    }
    cx.n_norm_rng = nr;
  }
  cx.merge_latent = e->f_dense == nullptr ? 1 : 0;
  if (cx.merge_latent) cx.phase_mask &= ~((1ull << jb::PH_LATLOSS) | (1ull << jb::PH_LATFIN));
  if (e->h_probs[cx.gph[8].first].fuse == jb::FUSE_LATBC) cx.phase_mask &= ~(1ull << jb::PH_LATBC);
  cx.p_diag = e->p_diag; cx.p_dense = e->p_dense; cx.f_dense = e->f_dense; cx.pn1 = e->pn1;
  cx.corr = e->corr; cx.corr_t = e->corr_t; cx.fblk = e->fblk; cx.fblk_t = e->fblk_t;
  cx.pf_ratio = e->cfg.pf_ratio; cx.f_present = e->f_dense != nullptr;
  // the row shortcut of COMBINE / LATBZ exists where GATHER builds the blocks with sk_corr_row_diag (same condition as there)
  cx.corr_hint = (e->p_diag != nullptr && e->p_dense == nullptr && e->f_dense == nullptr) ? e->corr_hint : nullptr;
  cx.lat_r = e->lat_r; cx.rowpart = e->rowpart; cx.lat_coef = e->lat_coef; cx.cosine = e->cosine;
  cx.cmax_part = e->cmax_part; cx.dmax_part = e->dmax_part; cx.dyn = e->dyn;
  {
    const float ones[8] = {1.f, 1.f, 1.f, 1.f, 1.f, 1.f, 1.f, 1.f};
    CU(cudaMemcpy(e->dyn, ones, sizeof ones, cudaMemcpyHostToDevice));
  }
  cx.theta = e->theta; cx.grad = e->grad; cx.adam_m = e->adam_m; cx.adam_v = e->adam_v;
  cx.theta_hi = e->theta_hi; cx.theta_lo = e->theta_lo; cx.n_flat = e->n_flat;
  cx.sigma = T + e->sigma.off; cx.dsigma = G + e->sigma.off; cx.norm_part = e->norm_part;
  cx.plan_kl = e->plan_kl; cx.out_loss = e->out_loss; cx.ctl = e->ctl;
  jb::StepConsts& sc = cx.sc;
  sc.lr = e->cfg.lr; sc.beta1 = e->cfg.beta1; sc.beta2 = e->cfg.beta2; sc.adam_eps = e->cfg.adam_eps;
  sc.max_norm = e->cfg.max_grad_norm;
  for (int k = 0; k < 4; ++k) sc.w[k] = e->cfg.loss_w[k];
  sc.pf_ratio = e->cfg.pf_ratio; sc.dropout = e->cfg.dropout;
  sc.grad_scale = 1.0f / static_cast<float>(e->cfg.world_size > 0 ? e->cfg.world_size : 1);
  sc.B = B; sc.L = L; sc.D[0] = e->D[0]; sc.D[1] = e->D[1];
  cx.gs = e->gs; cx.inv_gs = inv_gs;
  for (int q = 0; q < 8; ++q) { cx.xg[q] = e->xg[q]; cx.xf[q] = e->xf[q]; }
  cx.xrank = e->xrank; cx.xworld = e->xworld; cx.xmc = e->xworld > 1 ? e->xmc : nullptr; cx.x_adam0 = e->x_adam0;
  cx.xdbg = getenv("JB_XCHG_DBG") ? atoi(getenv("JB_XCHG_DBG")) : 0;
  cx.xfence = (getenv("JB_XCHG_FENCE") && strcmp(getenv("JB_XCHG_FENCE"), "sys") == 0) ? 1 : 0;
  e->step_B = B;
  return 0;
}

int ensure_step(jb_engine* e, int B) {
  if (e->step_B == B) return 0;
  CU(cudaDeviceSynchronize());
  return build_step(e, B);
}

// k_step always runs as thread-block clusters of HG_CLUSTER CTAs (cooperative: all CTAs co-resident; the grid barrier spins).
int launch_kstep_raw(jb_engine* e, void** args, cudaStream_t s) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(e->grid); cfg.blockDim = dim3(jb::SK_THREADS); cfg.dynamicSmemBytes = jb::HG_SMEM_BYTES; cfg.stream = s;
  cudaLaunchAttribute at[2];
  at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = jb::HG_CLUSTER; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  at[1].id = cudaLaunchAttributeCooperative; at[1].val.cooperative = 1;
  // JB_COOP=0 (profilers that cannot replay a cooperative cluster launch): a plain cluster launch; the grid still fits the
  // device in one wave, which is all the software grid barrier needs when nothing else runs on the GPU
  static const bool coop = !(getenv("JB_COOP") && atoi(getenv("JB_COOP")) == 0);
  cfg.attrs = at; cfg.numAttrs = coop ? 2 : 1;
  CU(cudaLaunchKernelExC(&cfg, reinterpret_cast<const void*>(jb::k_step), args));
  return 0;
}

// One launch of the step kernel: phases [lo, hi) of nsteps consecutive steps, then the control-block update.
int launch_step(jb_engine* e, int lo, int hi, int nsteps, int use_stage, cudaStream_t s, unsigned long long* ts = nullptr) {
  if (e->accumulate != e->accumulate_dev) {
    jb::k_set_accum<<<1, 1, 0, s>>>(e->ctl, e->accumulate);
    e->accumulate_dev = e->accumulate;
    ++e->launches;
  }
  int row_bias = lo > jb::PH_GATHER ? -1 : 0;
  const int fwd = lo == jb::PH_GATHER ? nsteps : 0, upd = hi == jb::PH_COUNT ? nsteps : 0;
  int3 adv = make_int3(fwd, upd, fwd > 0 ? 1 : 0);
  unsigned int* bar = e->bar + (e->bar_parity ? 32 : 0);   // this launch's counter; the kernel zeroes the other one
  unsigned int* bar_next = e->bar + (e->bar_parity ? 0 : 32);
  e->bar_parity ^= 1;
  void* args[] = {e->h_prm, &lo, &hi, &nsteps, &bar, &use_stage, &row_bias, &ts, &adv, &bar_next};
  if (launch_kstep_raw(e, args, s)) return 1;
  CU(cudaGetLastError());
  e->launches += 1;
  return 0;
}

// ------------------------------------------------------------------------------------------- eval path
int prepare_eval(jb_engine* e, cudaStream_t s) {
  if (!e->eval_dirty) return 0;
  CU(cudaMemcpyAsync(e->theta_eval, e->theta, e->n_flat * 4, cudaMemcpyDeviceToDevice, s));
  for (int i = 0; i < 2; ++i) {
    ModSegs& m = e->ms[i];
    const Seg* Ws[4] = {&m.W1, &m.W2, &m.W3, &m.W4};
    const Seg* bs[4] = {&m.b1, &m.b2, &m.b3, &m.b4};
    const Seg* gs[4] = {&m.g1, &m.g2, &m.g3, &m.g4};
    const Seg* es[4] = {&m.be1, &m.be2, &m.be3, &m.be4};
    const int bnidx[4] = {2 * i, 2 * i + 1, 4 + 2 * i, 4 + 2 * i + 1};
    for (int k = 0; k < 4; ++k) {
      jb::FoldArgs fa{};
      fa.W = e->theta + Ws[k]->off; fa.b = e->theta + bs[k]->off; fa.gamma = e->theta + gs[k]->off; fa.beta = e->theta + es[k]->off;
      fa.rm = e->bn_run + e->bn_off[bnidx[k]]; fa.rv = fa.rm + e->bn_w[bnidx[k]];
      fa.Wf = e->theta_eval + Ws[k]->off; fa.bf = e->theta_eval + bs[k]->off;
      fa.rows = Ws[k]->rows; fa.cols = Ws[k]->cols; fa.ld = Ws[k]->ld;
      jb::k_fold<<<fa.rows, 128, 0, s>>>(fa);
      ++e->launches;
    }
  }
  jb::k_to_half<<<296, 256, 0, s>>>(e->theta_eval, e->theta_eval_h, e->n_flat);
  ++e->launches;
  CU(cudaGetLastError());
  e->eval_dirty = false;
  return 0;
}

// Runs the folded chain on `rows` rows: in [rows, ld_in] (device, TMA-addressable) -> out [rows, ld_out].
// to < 0: encoder + mu head only.
int run_chain(jb_engine* e, int from, int to, const float* in, int ld_in, int rows, float* out, int ld_out, cudaStream_t s,
              float* bufA, float* bufB, GemmProblem* d_tab) {
  const float* T = e->theta_eval;
  const int L = e->L;
  ModSegs& mf = e->ms[from];
  const int Df = e->D[from];
  std::vector<GemmProblem> tab;
  // fp16 chain: the wide layers exchange fp16 activations and read fp16 weights (half the operand bytes); the first
  // layer of each half reads fp32 (the caller's rows, the fp32 embedding) as TF32; embeddings and outputs stay fp32
  const __half* Th = e->theta_eval_h;
  __half* hA = reinterpret_cast<__half*>(bufA);
  __half* hB = reinterpret_cast<__half*>(bufB);
  auto addc = [&](const void* A, int lda, const Seg& Wt, const Seg& bt, void* C, int ldc, int N, int K, int epi, int f16_ops, int out_f16) {
    GemmProblem g;
    int bn = N <= 32 ? 32 : (N <= 64 ? 64 : (N >= 256 ? 256 : 128));
    if (out_f16 && bn < 64) bn = 64;
    const void* Bw = f16_ops ? static_cast<const void*>(Th + Wt.off) : static_cast<const void*>(T + Wt.off);
    int rc = jb::gemm_chain_problem_fill(&g, A, lda, Bw, Wt.ld, C, ldc, rows, N, K, bn, epi, T + bt.off, jb::LRELU, f16_ops, out_f16);
    if (rc) return fail("eval tensor map encode failed (%d)", rc);
    jb::gemm_table_finalize(&g, 1);
    tab.push_back(g);
    return 0;
  };
  const int h2f = r8(2 * Df), hf = r8(Df);
  if (addc(in, ld_in, mf.W1, mf.b1, hA, h2f, 2 * Df, Df, jb::EPI_BIAS_LRELU, 0, 1)) return 1;
  if (addc(hA, h2f, mf.W2, mf.b2, hB, hf, Df, 2 * Df, jb::EPI_BIAS_LRELU, 1, 1)) return 1;
  if (to < 0) {
    if (addc(hB, hf, mf.Wmv, mf.bmv, out, ld_out, L, Df, jb::EPI_BIAS, 1, 0)) return 1;   // first L rows of Wmv = fc_mus
  } else {
    ModSegs& mt = e->ms[to];
    const int Dt = e->D[to];
    const int h2t = r8(2 * Dt), ht = r8(Dt);
    if (addc(hB, hf, mf.Wmv, mf.bmv, bufA, e->LP, L, Df, jb::EPI_BIAS, 1, 0)) return 1;
    if (addc(bufA, e->LP, mt.W3, mt.b3, hB, ht, Dt, L, jb::EPI_BIAS_LRELU, 0, 1)) return 1;
    if (addc(hB, ht, mt.W4, mt.b4, hA, h2t, 2 * Dt, Dt, jb::EPI_BIAS_LRELU, 1, 1)) return 1;
    if (addc(hA, h2t, mt.W5, mt.b5, out, ld_out, Dt, 2 * Dt, jb::EPI_BIAS, 1, 0)) return 1;
  }
  CU(cudaMemcpyAsync(d_tab, tab.data(), tab.size() * sizeof(GemmProblem), cudaMemcpyHostToDevice, s));
  for (size_t k = 0; k < tab.size(); ++k) {
    // programmatic dependent launch inside the chain: GEMM k + 1 sets up while GEMM k drains (the kernel waits for its
    // predecessor before touching memory)
    CU(jb::gemm_launch_persistent(d_tab + k, tab[k], e->num_sms, s, k > 0));
    ++e->launches;
  }
  return 0;
}

int eval_common(jb_engine* e, int from, int to, const float* X, long long n, long long ldx, float* out, long long ldo,
                int on_device, cudaStream_t s) {
  if (from < 0 || from > 1 || to > 1) return fail("modality index out of range");
  if (n <= 0) return 0;
  const int Din = e->D[from];
  const int Dout = to < 0 ? e->L : e->D[to];
  if (ldx < Din || ldo < Dout) return fail("row pitch smaller than the row width");
  if (prepare_eval(e, s)) return 1;
  const int CH = e->eval_chunk;
  const int ldin_p = r4(Din), ldout_p = r4(Dout);
  if (on_device) {
    const bool in_ok = (ldx % 4 == 0) && ((reinterpret_cast<uintptr_t>(X) & 15) == 0);
    const bool out_ok = (ldo % 4 == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
    // device-resident rows need no copy / compute double-buffering: both workspace slots form one chunk of 2 CH rows
    // (measured: 111.6 vs 105.3 M rows/s)
    const long long CHd = 2LL * CH;
    int slot = 0;
    for (long long r0 = 0; r0 < n; r0 += CHd, slot ^= 1) {
      const int rows = static_cast<int>(n - r0 < CHd ? n - r0 : CHd);
      const float* in = X + r0 * ldx;
      int ld_in = static_cast<int>(ldx);
      if (!in_ok) {
        jb::k_copy2d<<<rows, 128, 0, s>>>(in, ldx, e->ev_in, ldin_p, rows, Din); ++e->launches;
        in = e->ev_in; ld_in = ldin_p;
      }
      float* o = out + r0 * ldo;
      int ld_o = static_cast<int>(ldo);
      if (!out_ok) { o = e->ev_out; ld_o = ldout_p; }
      // the per-chunk tables alternate between two device slots; a slot is reused only after the stream has
      // consumed it (same-stream ordering of the H2D table copy after the previous chunk's kernels)
      if (run_chain(e, from, to, in, ld_in, rows, o, ld_o, s, e->ev_a, e->ev_b, e->d_ev_probs + slot * 8)) return 1;
      if (!out_ok) { jb::k_copy2d<<<rows, 128, 0, s>>>(e->ev_out, ldout_p, out + r0 * ldo, ldo, rows, Dout); ++e->launches; }
      // the host-side table vector of run_chain is pageable: the async copy has been staged by the driver on return
    }
    CU(cudaGetLastError());
    return 0;
  }
  // host pointers: stream chunks through two device staging slots so that H2D, compute and D2H overlap
  CU(cudaStreamSynchronize(s));
  const size_t in_slot = static_cast<size_t>(CH) * ldin_p, out_slot = static_cast<size_t>(CH) * ldout_p;
  const size_t a_slot = static_cast<size_t>(CH) * r4(2 * (e->D[0] > e->D[1] ? e->D[0] : e->D[1]));
  int slot = 0;
  for (long long r0 = 0; r0 < n; r0 += CH, slot ^= 1) {
    cudaStream_t cs = e->ev_stream[slot];
    const int rows = static_cast<int>(n - r0 < CH ? n - r0 : CH);
    float* din = e->ev_in + slot * in_slot;
    float* dout = e->ev_out + slot * out_slot;
    CU(cudaMemcpy2DAsync(din, static_cast<size_t>(ldin_p) * 4, X + r0 * ldx, static_cast<size_t>(ldx) * 4,
                         static_cast<size_t>(Din) * 4, rows, cudaMemcpyHostToDevice, cs));
    if (run_chain(e, from, to, din, ldin_p, rows, dout, ldout_p, cs, e->ev_a + slot * a_slot, e->ev_b + slot * a_slot,
                  e->d_ev_probs + slot * 8)) return 1;
    CU(cudaMemcpy2DAsync(out + r0 * ldo, static_cast<size_t>(ldo) * 4, dout, static_cast<size_t>(ldout_p) * 4,
                         static_cast<size_t>(Dout) * 4, rows, cudaMemcpyDeviceToHost, cs));
  }
  CU(cudaStreamSynchronize(e->ev_stream[0]));
  CU(cudaStreamSynchronize(e->ev_stream[1]));
  return 0;
}


}  // namespace

// =============================================================================================== C ABI
namespace {
template <class T> struct DevArr {   // scoped device allocation of any type
  T* p = nullptr;
  ~DevArr() { if (p) cudaFree(p); }
  int alloc(size_t n) { CU(cudaMalloc(&p, (n ? n : 1) * sizeof(T))); return 0; }
  int upload(const T* h, size_t n) { if (alloc(n)) return 1; CU(cudaMemcpy(p, h, n * sizeof(T), cudaMemcpyHostToDevice)); return 0; }
};
int metric_grid(long long tiles) {
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const long long g = static_cast<long long>(sms) * 4;
  return static_cast<int>(tiles < g ? (tiles > 0 ? tiles : 1) : g);
}
}  // namespace

struct jb_pcaop {   // one centred PCA operand Xc = X - 1 mu^T on one device (jb_pcaop_*)
  long long n = 0, d = 0, nnz = 0;
  int device = 0;
  int sparse = 0;
  cudaStream_t s = nullptr;
  cudaEvent_t ev_in = nullptr, ev_out = nullptr;   // order jb_pcaop_apply after / before the caller's stream
  double* mu = nullptr;          // [d] column means (0 until jb_pcaop_stats)
  double* var = nullptr;         // [d]
  // dense operand
  float* X = nullptr;            // [n, d] as given
  float* mu32 = nullptr;         // [d]
  float* x_hi = nullptr;         // [n, ldd] 3xTF32 planes of X - mu
  float* x_lo = nullptr;
  long long ldd = 0;
  double* stat_part = nullptr;   // [PO_STAT_SLABS, d] partial column sums
  jb::GemmProblem* probs = nullptr;   // one table entry per reduction chunk of a product
  int n_probs = 0;
  std::vector<jb::GemmProblem> host_probs;
  // sparse operand: CSR of X (rp, ci, rv) and CSR of X^T (cp, ri, cv); work items of both directions
  long long* rp = nullptr; int* ci = nullptr; float* rv = nullptr;
  long long* cp = nullptr; int* ri = nullptr; float* cv = nullptr;
  jb::PoItem* items[2] = {nullptr, nullptr};
  long long n_items[2] = {0, 0};
  jb::PoLong* longs[2] = {nullptr, nullptr};
  int n_long[2] = {0, 0};
  int n_part[2] = {0, 0};
  // workspaces of width ws_l (grown on demand by jb_pcaop_apply)
  int ws_l = 0;
  float* b_hi = nullptr; float* b_lo = nullptr; float* t32 = nullptr;   // dense: planes of B, one chunk's fp32 product
  double* acc = nullptr;                                                // dense: float64 sum over the chunks
  double* part = nullptr;                                               // sparse: segment partials
  double* vpart = nullptr; double* vvec = nullptr;                      // sparse: the l-vector of the rank-1 correction
};

struct jb_dist {   // one n x n float64 distance matrix on one device (jb_dist_*)
  long long n = 0;
  int device = 0;
  cudaStream_t s = nullptr;
  double* D = nullptr;
  double* slab = nullptr;   // device copy of the current column slab
  size_t slab_cap = 0;      // doubles
  int* knn_idx = nullptr;   // [n, knn_k] neighbour lists of the last jb_dist_knn
  double* knn_dist = nullptr;
  int knn_k = 0;
  unsigned long long* scratch = nullptr;
};

extern "C" {

const char* jb_last_error(void) { return g_err.c_str(); }
int jb_version(void) { return 200; }

int jb_create(const jb_config* cfg, jb_engine** out) {
  if (!cfg || !out) return fail("null argument");
  if (cfg->dims[0] <= 0 || cfg->dims[1] <= 0 || cfg->latent <= 0 || cfg->max_batch < 2)
    return fail("invalid dims/latent/batch (%d, %d, %d, %d)", cfg->dims[0], cfg->dims[1], cfg->latent, cfg->max_batch);
  if (cfg->latent > 32 * jb::LAT_MAXT) return fail("output_dim %d exceeds the supported maximum %d", cfg->latent, 32 * jb::LAT_MAXT);
  if (!(cfg->dropout >= 0.f && cfg->dropout < 1.f)) return fail("dropout must be in [0, 1)");
  CU(cudaSetDevice(cfg->device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, cfg->device));
  if (prop.major != 10) return fail("jamie_b200 needs an sm_100 (B200) device, found sm_%d%d", prop.major, prop.minor);
  if (!prop.cooperativeLaunch) return fail("the device does not support cooperative launches");
  jb_engine* e = new jb_engine();
  e->cfg = *cfg;
  e->D[0] = cfg->dims[0]; e->D[1] = cfg->dims[1]; e->L = cfg->latent; e->LP = r8(cfg->latent); e->ldmv = r8(2 * cfg->latent);
  e->Bmax = cfg->max_batch;
  build_layout(e);
  const size_t fb = static_cast<size_t>(e->n_flat + 32) * 4;
  auto alloc0 = [&](float** p, size_t bytes) -> int {
    CU(cudaMalloc(p, bytes));
    CU(cudaMemset(*p, 0, bytes));
    return 0;
  };
  // theta, the Adam moments (fp32) and the fp16 operand planes live in ONE slab (fb is a multiple of 128 B)
  e->slab_bytes = 4 * fb;
  if (alloc0(&e->state_slab, e->slab_bytes) || alloc0(&e->grad, fb) || alloc0(&e->theta_eval, fb) ||
      alloc0(&e->bn_run, e->n_bn * 4)) { jb_destroy(e); return 1; }
  e->theta = e->state_slab; e->adam_m = e->theta + fb / 4; e->adam_v = e->adam_m + fb / 4;
  e->theta_hi = reinterpret_cast<__half*>(e->adam_v + fb / 4); e->theta_lo = e->theta_hi + fb / 4;
  {  // BatchNorm defaults: running_mean 0, running_var 1; gamma = 1 is set through jb_set_params
    std::vector<float> h(e->n_bn, 0.f);
    for (int k = 0; k < 8; ++k)
      for (int j = 0; j < e->bn_w[k]; ++j) h[e->bn_off[k] + e->bn_w[k] + j] = 1.f;
    CU(cudaMemcpy(e->bn_run, h.data(), e->n_bn * 4, cudaMemcpyHostToDevice));
  }
  Carver dry(nullptr);
  carve(e, dry);
  e->arena_bytes = dry.off + 256;
  CU(cudaMalloc(&e->arena, e->arena_bytes));
  CU(cudaMemset(e->arena, 0, e->arena_bytes));
  Carver real(e->arena);
  carve(e, real);
  CU(cudaMalloc(&e->ctl, sizeof(jb::Ctl)));
  jb::Ctl c0{};
  c0.seed = cfg->seed;
  CU(cudaMemcpy(e->ctl, &c0, sizeof c0, cudaMemcpyHostToDevice));
  CU(cudaMalloc(&e->norm_part, jb::SK_MAX_CTAS * sizeof(double)));
  e->norm_tile = nullptr; e->norm_tile_cap = 0;   // sized by build_step (one partial per epilogue warp and weight-gradient work item)
  CU(cudaMalloc(&e->norm_small, jb::SK_MAX_CTAS * 4 * sizeof(float)));
  CU(cudaMemset(e->norm_small, 0, jb::SK_MAX_CTAS * 4 * sizeof(float)));
  CU(cudaMalloc(&e->bar, 512));
  CU(cudaMemset(e->bar, 0, 512));
  CU(cudaFuncSetAttribute(jb::gemm_tf32_grouped_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, jb::GEMM_SMEM_BYTES));
  CU(cudaFuncSetAttribute(jb::k_step, cudaFuncAttributeMaxDynamicSharedMemorySize, jb::HG_SMEM_BYTES));
  e->num_sms = prop.multiProcessorCount;
  {  // the step kernel is cooperative and runs as clusters of HG_CLUSTER CTAs, one CTA per SM: every cluster must be
     // co-resident (33 clusters = 132 CTAs on a 148-SM B200: GPCs with 18 SMs seat four clusters of four)
    CU(cudaFuncSetAttribute(jb::k_step, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cudaLaunchConfig_t lc = {};
    lc.gridDim = dim3(jb::HG_CLUSTER * 64); lc.blockDim = dim3(jb::SK_THREADS); lc.dynamicSmemBytes = jb::HG_SMEM_BYTES;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = jb::HG_CLUSTER; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    lc.attrs = at; lc.numAttrs = 1;
    int nclusters = 0;
    CU(cudaOccupancyMaxActiveClusters(&nclusters, jb::k_step, &lc));
    if (nclusters < 1) { jb_destroy(e); return fail("the step kernel does not fit on the device (shared memory / registers / clusters)"); }
    e->grid = nclusters * jb::HG_CLUSTER;
    if (e->grid > jb::SK_MAX_CTAS) e->grid = (jb::SK_MAX_CTAS / jb::HG_CLUSTER) * jb::HG_CLUSTER;
  }
  // rows per pass of the folded chain: one 128-row M tile per SM, so every GEMM of the chain is a whole number of waves
  // (measured on B200, 1M rows 512 -> 512: 8192 rows 59.1, 9472 rows 66.7, 18944 rows 69.0 M rows/s)
  e->eval_chunk = 128 * e->num_sms;
  CU(cudaMalloc(&e->theta_eval_h, static_cast<size_t>(e->n_flat + 32) * 2));
  // eval workspaces: two slots of chunk activations
  {
    const int Dm = e->D[0] > e->D[1] ? e->D[0] : e->D[1];
    const size_t a = static_cast<size_t>(e->eval_chunk) * r4(2 * Dm);
    const size_t io = static_cast<size_t>(e->eval_chunk) * r4(Dm > e->L ? Dm : e->L);
    CU(cudaMalloc(&e->ev_a, 2 * a * 4)); CU(cudaMalloc(&e->ev_b, 2 * a * 4));
    CU(cudaMalloc(&e->ev_in, 2 * io * 4)); CU(cudaMalloc(&e->ev_out, 2 * io * 4));
    CU(cudaMalloc(&e->d_ev_probs, 16 * sizeof(GemmProblem)));
    for (int k = 0; k < 2; ++k) CU(cudaStreamCreateWithFlags(&e->ev_stream[k], cudaStreamNonBlocking));
  }
  *out = e;
  return 0;
}

void jb_destroy(jb_engine* e) {
  if (!e) return;
  cudaDeviceSynchronize();
  if (e->h_pin) cudaFreeHost(e->h_pin);
  if (e->h2d_stream) cudaStreamDestroy(e->h2d_stream);
  for (int k = 0; k < 2; ++k) {
    if (e->ev_h2d[k]) cudaEventDestroy(e->ev_h2d[k]);
    if (e->ev_slot_free[k]) cudaEventDestroy(e->ev_slot_free[k]);
    if (e->ev_loss[k]) cudaEventDestroy(e->ev_loss[k]);
  }
  void* ptrs[] = {e->state_slab, e->grad_own ? e->grad_own : e->grad, e->theta_eval, e->bn_run, e->data[0], e->data[1], e->p_diag,
                  e->p_dense, e->f_dense, e->plan_idx[0], e->plan_idx[1], e->plan_kl, e->out_loss, e->ctl, e->norm_part,
                  e->arena, e->parts_arena, e->bar, e->d_ts, e->ev_a, e->ev_b, e->ev_in, e->ev_out,
                  e->d_ev_probs, e->theta_eval_h, e->norm_tile, e->norm_small};
  for (void* p : ptrs) if (p) cudaFree(p);
  for (int k = 0; k < 2; ++k) if (e->ev_stream[k]) cudaStreamDestroy(e->ev_stream[k]);
  delete e->h_prm;
  delete e;
}

long long jb_num_params(const jb_engine* e) { return e ? e->n_packed : 0; }
long long jb_num_bn_floats(const jb_engine* e) { return e ? e->n_bn : 0; }

int jb_set_params(jb_engine* e, const float* packed, long long n) {
  if (!e || !packed) return fail("null argument");
  if (n != e->n_packed) return fail("expected %lld parameters, got %lld", e->n_packed, n);
  CU(cudaDeviceSynchronize());
  e->eval_dirty = true;
  if (copy_packed(e, e->theta, const_cast<float*>(packed), true)) return 1;
  jb::k_hsplit_flat<<<296, 256>>>(e->theta, e->theta_hi, e->theta_lo, e->n_flat);   // operand planes of the training GEMMs
  ++e->launches;
  CU(cudaGetLastError());
  CU(cudaDeviceSynchronize());
  return 0;
}
int jb_get_params(jb_engine* e, float* packed, long long n) {
  if (!e || !packed) return fail("null argument");
  if (n != e->n_packed) return fail("expected %lld parameters, got %lld", e->n_packed, n);
  CU(cudaDeviceSynchronize());
  return copy_packed(e, e->theta, packed, false);
}
int jb_get_grads(jb_engine* e, float* packed, long long n) {
  if (!e || !packed) return fail("null argument");
  if (n != e->n_packed) return fail("expected %lld parameters, got %lld", e->n_packed, n);
  CU(cudaDeviceSynchronize());
  return copy_packed(e, e->grad, packed, false);
}
int jb_get_adam_state(jb_engine* e, float* m, float* v, long long n, long long* t) {
  if (!e || !m || !v || !t) return fail("null argument");
  if (n != e->n_packed) return fail("expected %lld parameters, got %lld", e->n_packed, n);
  CU(cudaDeviceSynchronize());
  if (copy_packed(e, e->adam_m, m, false) || copy_packed(e, e->adam_v, v, false)) return 1;
  jb::Ctl c;
  CU(cudaMemcpy(&c, e->ctl, sizeof c, cudaMemcpyDeviceToHost));
  *t = c.adam_t;
  return 0;
}
int jb_set_adam_state(jb_engine* e, const float* m, const float* v, long long n, long long t) {
  if (!e || !m || !v) return fail("null argument");
  if (n != e->n_packed) return fail("expected %lld parameters, got %lld", e->n_packed, n);
  CU(cudaDeviceSynchronize());
  if (copy_packed(e, e->adam_m, const_cast<float*>(m), true) || copy_packed(e, e->adam_v, const_cast<float*>(v), true)) return 1;
  jb::Ctl c;
  CU(cudaMemcpy(&c, e->ctl, sizeof c, cudaMemcpyDeviceToHost));
  if (e->xworld > 1) { e->x_adam0 += t - c.adam_t; e->step_B = 0; }   // exchange epochs keep counting from where they were
  c.adam_t = t;
  CU(cudaMemcpy(e->ctl, &c, sizeof c, cudaMemcpyHostToDevice));
  return 0;
}
int jb_set_bn_stats(jb_engine* e, const float* packed, long long n, const long long nbt[8]) {
  if (!e || !packed) return fail("null argument");
  if (n != e->n_bn) return fail("expected %lld BatchNorm floats, got %lld", e->n_bn, n);
  CU(cudaDeviceSynchronize());
  CU(cudaMemcpy(e->bn_run, packed, n * 4, cudaMemcpyHostToDevice));
  if (nbt) for (int k = 0; k < 8; ++k) e->nbt[k] = nbt[k];
  e->eval_dirty = true;
  return 0;
}
int jb_get_bn_stats(jb_engine* e, float* packed, long long n, long long nbt[8]) {
  if (!e || !packed) return fail("null argument");
  if (n != e->n_bn) return fail("expected %lld BatchNorm floats, got %lld", e->n_bn, n);
  CU(cudaDeviceSynchronize());
  CU(cudaMemcpy(packed, e->bn_run, n * 4, cudaMemcpyDeviceToHost));
  if (nbt) for (int k = 0; k < 8; ++k) nbt[k] = e->nbt[k];
  return 0;
}

int jb_set_dataset(jb_engine* e, int mod, const float* X, long long n, long long ld, int on_device, void* stream) {
  if (!e || !X) return fail("null argument");
  if (mod < 0 || mod > 1) return fail("modality index out of range");
  if (ld < e->D[mod] || n <= 0) return fail("bad dataset shape");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  CU(cudaDeviceSynchronize());
  if (e->data[mod]) { cudaFree(e->data[mod]); e->data[mod] = nullptr; }
  const long long ldd = r4(e->D[mod]);
  CU(cudaMalloc(&e->data[mod], static_cast<size_t>(n) * ldd * 4));
  CU(cudaMemcpy2DAsync(e->data[mod], static_cast<size_t>(ldd) * 4, X, static_cast<size_t>(ld) * 4,
                       static_cast<size_t>(e->D[mod]) * 4, n, on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, s));
  CU(cudaStreamSynchronize(s));
  e->data_n[mod] = n; e->data_ld[mod] = ldd;
  e->step_B = 0;   // pointers are baked into the step context
  return 0;
}

int jb_set_prior_diag(jb_engine* e, const float* m, long long n) {
  if (!e) return fail("null argument");
  CU(cudaDeviceSynchronize());
  if (e->p_diag) { cudaFree(e->p_diag); e->p_diag = nullptr; }
  if (e->p_dense) { cudaFree(e->p_dense); e->p_dense = nullptr; }
  if (m) {
    CU(cudaMalloc(&e->p_diag, static_cast<size_t>(n) * 4));
    CU(cudaMemcpy(e->p_diag, m, static_cast<size_t>(n) * 4, cudaMemcpyHostToDevice));
  }
  e->p_diag_n = m ? n : 0;
  e->step_B = 0;
  return 0;
}
int jb_set_prior_dense(jb_engine* e, const float* P, long long n0, long long n1) {
  if (!e || !P) return fail("null argument");
  CU(cudaDeviceSynchronize());
  if (e->p_diag) { cudaFree(e->p_diag); e->p_diag = nullptr; }
  if (e->p_dense) { cudaFree(e->p_dense); e->p_dense = nullptr; }
  if (e->f_dense && (e->pn0 != n0 || e->pn1 != n1)) return fail("P and F shapes differ");
  CU(cudaMalloc(&e->p_dense, static_cast<size_t>(n0) * n1 * 4));
  CU(cudaMemcpy(e->p_dense, P, static_cast<size_t>(n0) * n1 * 4, cudaMemcpyHostToDevice));
  e->pn0 = n0; e->pn1 = n1;
  e->step_B = 0;
  return 0;
}
int jb_set_f_dense(jb_engine* e, const float* F, long long n0, long long n1) {
  if (!e) return fail("null argument");
  CU(cudaDeviceSynchronize());
  if (e->f_dense) { cudaFree(e->f_dense); e->f_dense = nullptr; }
  if (F) {
    if (e->p_dense && (e->pn0 != n0 || e->pn1 != n1)) return fail("P and F shapes differ");
    CU(cudaMalloc(&e->f_dense, static_cast<size_t>(n0) * n1 * 4));
    CU(cudaMemcpy(e->f_dense, F, static_cast<size_t>(n0) * n1 * 4, cudaMemcpyHostToDevice));
    e->pn0 = n0; e->pn1 = n1;
  }
  e->step_B = 0;
  return 0;
}

int jb_upload_plan(jb_engine* e, const long long* idx0, const long long* idx1, const double* kl_anneal, int nsteps, int batch,
                   void* stream) {
  if (!e || !idx0 || !idx1 || !kl_anneal) return fail("null argument");
  if (batch < 2 || batch > e->Bmax) return fail("batch %d outside [2, %d]", batch, e->Bmax);
  if (nsteps <= 0) return fail("nsteps must be positive");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  CU(cudaStreamSynchronize(s));
  if (nsteps > e->plan_cap || batch != e->plan_B) {
    CU(cudaDeviceSynchronize());
    for (int i = 0; i < 2; ++i) if (e->plan_idx[i]) { cudaFree(e->plan_idx[i]); e->plan_idx[i] = nullptr; }
    if (e->plan_kl) { cudaFree(e->plan_kl); e->plan_kl = nullptr; }
    if (e->out_loss) { cudaFree(e->out_loss); e->out_loss = nullptr; }
    const int cap = nsteps > e->plan_cap ? nsteps : e->plan_cap;
    for (int i = 0; i < 2; ++i) CU(cudaMalloc(&e->plan_idx[i], static_cast<size_t>(cap) * batch * 4));
    CU(cudaMalloc(&e->plan_kl, static_cast<size_t>(cap) * 4));
    CU(cudaMalloc(&e->out_loss, static_cast<size_t>(cap) * 8 * 4));
    e->plan_cap = cap; e->plan_B = batch;
    e->step_B = 0;  // plan pointers are baked into the step context
  }
  std::vector<int> h(static_cast<size_t>(nsteps) * batch);
  const long long* src[2] = {idx0, idx1};
  for (int i = 0; i < 2; ++i) {
    for (size_t k = 0; k < h.size(); ++k) {
      const long long v = src[i][k];
      if (v < 0 || (e->data[i] && v >= e->data_n[i])) return fail("batch index %lld out of range for modality %d (n = %lld)", v, i, e->data_n[i]);
      h[k] = static_cast<int>(v);
    }
    CU(cudaMemcpy(e->plan_idx[i], h.data(), h.size() * 4, cudaMemcpyHostToDevice));
  }
  std::vector<float> kl(nsteps);
  for (int k = 0; k < nsteps; ++k) kl[k] = static_cast<float>(32 * 1e-3 * kl_anneal[k]);
  CU(cudaMemcpy(e->plan_kl, kl.data(), static_cast<size_t>(nsteps) * 4, cudaMemcpyHostToDevice));
  CU(cudaMemset(e->out_loss, 0, static_cast<size_t>(nsteps) * 8 * 4));
  long long zero = 0;
  CU(cudaMemcpy(&e->ctl->cursor, &zero, sizeof zero, cudaMemcpyHostToDevice));
  e->plan_steps = nsteps;
  return 0;
}

int jb_inject_randomness(jb_engine* e, const float* eps0, const float* eps1, const unsigned char* const masks[8], void* stream) {
  if (!e || !eps0 || !eps1 || !masks) return fail("null argument");
  if (!e->plan_B) return fail("jb_upload_plan must be called first");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int B = e->plan_B;
  const float* eps[2] = {eps0, eps1};
  for (int i = 0; i < 2; ++i) {
    CU(cudaMemcpy2DAsync(e->act[i].inj_eps, static_cast<size_t>(e->LP) * 4, eps[i], static_cast<size_t>(e->L) * 4,
                         static_cast<size_t>(e->L) * 4, B, cudaMemcpyHostToDevice, s));
    const int D = e->D[i];
    const int w[4] = {2 * D, D, D, 2 * D};
    // draw order: enc_i d1, d2 are masks[2i], masks[2i+1]; dec_i d1, d2 are masks[4+2i], masks[4+2i+1]
    const unsigned char* src[4] = {masks[2 * i], masks[2 * i + 1], masks[4 + 2 * i], masks[4 + 2 * i + 1]};
    for (int k = 0; k < 4; ++k) {
      if (!src[k]) return fail("null mask pointer");
      CU(cudaMemcpyAsync(e->act[i].inj_mask[k], src[k], static_cast<size_t>(B) * w[k], cudaMemcpyHostToDevice, s));
    }
  }
  int one = 1;
  CU(cudaMemcpyAsync(&e->ctl->inject, &one, sizeof one, cudaMemcpyHostToDevice, s));
  CU(cudaStreamSynchronize(s));
  return 0;
}

int jb_train_steps(jb_engine* e, int nsteps, void* stream) {
  if (!e) return fail("null argument");
  if (nsteps <= 0) return 0;
  if (!e->plan_B) return fail("jb_upload_plan must be called first");
  if (!e->data[0] || !e->data[1]) return fail("jb_set_dataset must be called for both modalities before jb_train_steps");
  if (ensure_step(e, e->plan_B)) return 1;
  if (launch_step(e, jb::PH_GATHER, jb::PH_COUNT, nsteps, 0, static_cast<cudaStream_t>(stream))) return 1;
  for (int k = 0; k < 8; ++k) e->nbt[k] += nsteps;
  e->eval_dirty = true;
  return 0;
}
int jb_step_backward(jb_engine* e, void* stream) {
  if (!e) return fail("null argument");
  if (!e->plan_B) return fail("jb_upload_plan must be called first");
  if (!e->data[0] || !e->data[1]) return fail("jb_set_dataset must be called for both modalities before jb_step_backward");
  if (ensure_step(e, e->plan_B)) return 1;
  if (launch_step(e, jb::PH_GATHER, jb::PH_NORM, 1, 0, static_cast<cudaStream_t>(stream))) return 1;
  for (int k = 0; k < 8; ++k) e->nbt[k] += 1;
  e->eval_dirty = true;
  return 0;
}
int jb_step_update(jb_engine* e, void* stream) {
  if (!e) return fail("null argument");
  if (!e->step_B) return fail("jb_step_backward must run before jb_step_update");
  if (launch_step(e, jb::PH_NORM, jb::PH_COUNT, 1, 0, static_cast<cudaStream_t>(stream))) return 1;
  e->eval_dirty = true;
  return 0;
}
int jb_grad_buffer(jb_engine* e, float** dev_ptr, long long* n_floats) {
  if (!e || !dev_ptr || !n_floats) return fail("null argument");
  *dev_ptr = e->grad;
  *n_floats = e->n_flat + 8;  // flat gradients + the loss scalars appended by the loss phase
  return 0;
}
int jb_set_grad_buffer(jb_engine* e, float* dev_ptr, long long n_floats) {
  if (!e) return fail("null argument");
  CU(cudaDeviceSynchronize());
  if (dev_ptr == nullptr) {
    if (e->grad_own) e->grad = e->grad_own;
  } else {
    if (n_floats < e->n_flat + 8) return fail("gradient buffer too small (%lld floats, need %lld)", n_floats, e->n_flat + 8);
    if (reinterpret_cast<uintptr_t>(dev_ptr) & 15) return fail("gradient buffer must be 16-byte aligned");
    if (!e->grad_own) e->grad_own = e->grad;
    CU(cudaMemset(dev_ptr, 0, static_cast<size_t>(e->n_flat + 8) * 4));   // the padding stays zero forever
    e->grad = dev_ptr;
  }
  e->step_B = 0;   // the step tables hold the address
  return 0;
}
long long jb_exchange_scratch_bytes(void) { return 256 + 8LL * jb::SK_MAX_CTAS * 8; }
int jb_set_exchange(jb_engine* e, int rank, int world, float* const* grad_ptrs, unsigned int* const* flag_ptrs, float* grad_multicast) {
  if (!e) return fail("null argument");
  CU(cudaDeviceSynchronize());
  e->xworld = 0; e->xmc = nullptr;
  if (world > 1 && grad_ptrs && flag_ptrs) {
    if (world > 8 || rank < 0 || rank >= world) return fail("exchange over %d ranks (rank %d): at most 8 ranks of one box", world, rank);
    if (world != e->cfg.world_size) return fail("exchange world %d != jb_config.world_size %d", world, e->cfg.world_size);
    if (grad_ptrs[rank] != e->grad) return fail("grad_ptrs[rank] must be the buffer given to jb_set_grad_buffer");
    for (int q = 0; q < world; ++q) {
      if (!grad_ptrs[q] || !flag_ptrs[q]) return fail("null peer pointer for rank %d", q);
      e->xg[q] = grad_ptrs[q]; e->xf[q] = flag_ptrs[q];
    }
    e->xrank = rank; e->xworld = world; e->xmc = grad_multicast;
    jb::Ctl c;   // exchange epochs count from the optimizer step at which the (zeroed) scratch blocks were handed over
    CU(cudaMemcpy(&c, e->ctl, sizeof c, cudaMemcpyDeviceToHost));
    e->x_adam0 = c.adam_t;
  }
  e->step_B = 0;
  return 0;
}
int jb_set_dist_method(jb_engine* e, int method) {
  if (!e) return fail("null argument");
  if (method != 0 && method != 1) return fail("dist_method %d: 0 = euclidean, 1 = cosine", method);
  CU(cudaDeviceSynchronize());
  e->cosine = method;
  e->step_B = 0;   // the step context holds the flag
  return 0;
}
int jb_set_grad_accumulate(jb_engine* e, int accumulate) {
  if (!e) return fail("null argument");
  e->accumulate = accumulate ? 1 : 0;   // reaches the device control block with the next launch (no re-build, no sync)
  return 0;
}

// Enqueues one host-batch step in slot e->hb_slot: index / kl / row copies on the copy stream, then (after an event) the
// control-block pokes, the step kernel and the loss read-back on the caller's stream. Nothing here blocks the host.
static int hostbatch_submit(jb_engine* e, const float* x0, const float* x1, const long long* idx0, const long long* idx1,
                            int batch, double kl_anneal, bool with_update, void* stream) {
  if (!e || !x0 || !x1 || !idx0 || !idx1) return fail("null argument");
  if (with_update && e->hb_outstanding >= 2) return fail("two host-batch steps are in flight: call jb_hostbatch_wait first");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (e->plan_B != batch || e->plan_cap < 2) {   // first call: allocate a two-row plan (one row per slot) through the normal path
    std::vector<long long> z(2 * static_cast<size_t>(batch), 0);
    double k0[2] = {0, 0};
    if (jb_upload_plan(e, z.data(), z.data(), k0, 2, batch, stream)) return 1;
  }
  if (ensure_step(e, batch)) return 1;
  if (!e->h_pin) {
    CU(cudaMallocHost(reinterpret_cast<void**>(&e->h_pin), sizeof(HostPin) + 4 * static_cast<size_t>(e->Bmax) * sizeof(int)));
    e->h_pin->cursor_val[0] = 0; e->h_pin->cursor_val[1] = 1;
    e->h_pin->slot_val[0] = 0; e->h_pin->slot_val[1] = 1;
    CU(cudaStreamCreateWithFlags(&e->h2d_stream, cudaStreamNonBlocking));
    for (int k = 0; k < 2; ++k) {
      CU(cudaEventCreateWithFlags(&e->ev_h2d[k], cudaEventDisableTiming));
      CU(cudaEventCreateWithFlags(&e->ev_slot_free[k], cudaEventDisableTiming));
      CU(cudaEventCreateWithFlags(&e->ev_loss[k], cudaEventDisableTiming));
    }
  }
  const int slot = e->hb_slot;
  HostPin* hp = e->h_pin;
  // the slot's pinned index / kl area is reused: its previous copies (two submits ago) must have been consumed
  if (e->slot_used[slot]) CU(cudaEventSynchronize(e->ev_h2d[slot]));
  int* hi = hp->idx + static_cast<size_t>(slot) * 2 * e->Bmax;
  const long long* src[2] = {idx0, idx1};
  for (int i = 0; i < 2; ++i)
    for (int k = 0; k < batch; ++k) {
      const long long v = src[i][k];
      long long lim = 1LL << 31;
      if (e->p_diag) lim = e->p_diag_n;
      else if (e->p_dense || e->f_dense) lim = i == 0 ? e->pn0 : e->pn1;
      if (v < 0 || v >= lim) return fail("cell id %lld out of range for the prior (limit %lld)", v, lim);
      hi[i * e->Bmax + k] = static_cast<int>(v);
    }
  hp->kl[slot] = static_cast<float>(32 * 1e-3 * kl_anneal);
  // copy stream: wait until the step that last used this slot's device buffers has run, then bring the batch in
  cudaStream_t cs = e->h2d_stream;
  if (e->slot_used[slot]) CU(cudaStreamWaitEvent(cs, e->ev_slot_free[slot], 0));
  const float* xs[2] = {x0, x1};
  for (int i = 0; i < 2; ++i) {
    CU(cudaMemcpyAsync(e->plan_idx[i] + static_cast<size_t>(slot) * batch, hi + i * e->Bmax, static_cast<size_t>(batch) * 4,
                       cudaMemcpyHostToDevice, cs));
    CU(cudaMemcpy2DAsync(e->act[i].x_stage[slot], static_cast<size_t>(e->act[i].ldD) * 4, xs[i], static_cast<size_t>(e->D[i]) * 4,
                         static_cast<size_t>(e->D[i]) * 4, batch, cudaMemcpyHostToDevice, cs));
  }
  CU(cudaMemcpyAsync(e->plan_kl + slot, &hp->kl[slot], 4, cudaMemcpyHostToDevice, cs));
  CU(cudaEventRecord(e->ev_h2d[slot], cs));
  // compute stream
  CU(cudaStreamWaitEvent(s, e->ev_h2d[slot], 0));
  CU(cudaMemcpyAsync(&e->ctl->cursor, &hp->cursor_val[slot], sizeof(long long), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(&e->ctl->host_slot, &hp->slot_val[slot], sizeof(int), cudaMemcpyHostToDevice, s));
  for (int k = 0; k < 8; ++k) e->nbt[k] += 1;
  if (e->plan_steps < 2) e->plan_steps = 2;
  e->eval_dirty = true;
  if (!with_update) {   // data-parallel form: forward + backward only
    if (launch_step(e, jb::PH_GATHER, jb::PH_NORM, 1, 1, s)) return 1;
  } else {
    if (launch_step(e, jb::PH_GATHER, jb::PH_COUNT, 1, 1, s)) return 1;
    CU(cudaMemcpyAsync(hp->losses[slot], e->out_loss + static_cast<size_t>(slot) * 8, 8 * 4, cudaMemcpyDeviceToHost, s));
    CU(cudaEventRecord(e->ev_loss[slot], s));
    ++e->hb_outstanding;
  }
  CU(cudaEventRecord(e->ev_slot_free[slot], s));
  e->slot_used[slot] = true;
  e->hb_slot ^= 1;
  return 0;
}
int jb_hostbatch_submit(jb_engine* e, const float* x0, const float* x1, const long long* idx0, const long long* idx1, int batch,
                        double kl_anneal, void* stream) {
  return hostbatch_submit(e, x0, x1, idx0, idx1, batch, kl_anneal, true, stream);
}
int jb_hostbatch_wait(jb_engine* e, float out_losses[8]) {
  if (!e || !out_losses) return fail("null argument");
  if (e->hb_outstanding <= 0) return fail("no host-batch step in flight");
  const int slot = e->hb_oldest;
  CU(cudaEventSynchronize(e->ev_loss[slot]));
  memcpy(out_losses, e->h_pin->losses[slot], 8 * 4);
  e->hb_oldest ^= 1;
  --e->hb_outstanding;
  return 0;
}
int jb_train_step_hostbatch(jb_engine* e, const float* x0, const float* x1, const long long* idx0, const long long* idx1,
                            int batch, double kl_anneal, float out_losses[8], void* stream) {
  if (!out_losses) return fail("null argument");
  if (e && e->hb_outstanding > 0) return fail("asynchronous host-batch steps are in flight: call jb_hostbatch_wait first");
  if (hostbatch_submit(e, x0, x1, idx0, idx1, batch, kl_anneal, true, stream)) return 1;
  return jb_hostbatch_wait(e, out_losses);
}
int jb_step_backward_hostbatch(jb_engine* e, const float* x0, const float* x1, const long long* idx0, const long long* idx1,
                               int batch, double kl_anneal, void* stream) {
  return hostbatch_submit(e, x0, x1, idx0, idx1, batch, kl_anneal, false, stream);
}

int jb_num_phases(void) { return jb::PH_COUNT; }
const char* jb_phase_name(int ph) {
  static const char* names[jb::PH_COUNT] = {
      "gather+corr", "gemm enc1", "bn1", "gemm enc2", "bn2", "gemm heads", "reparam", "combine", "latloss", "gemm dec1", "bn3",
      "gemm dec2", "bn4", "gemm dec3", "rec", "dgrad W5", "bnb4", "dgrad W4", "bnb3", "dgrad W3", "latbc", "latbz",
      "dmulv planes+final", "dgrad heads", "bnb2", "dgrad W2", "bnb1", "wgrad x12", "gradnorm", "adam"};
  return ph >= 0 && ph < jb::PH_COUNT ? names[ph] : "";
}

// Times ONE phase alone: `iters` launches of k_step over [phase, phase + 1) on `stream` (CUDA events on that stream; each
// launch includes the kernel's setup, so this is an upper bound of the phase's share of a step). flops: GEMM phases only.
int jb_bench_stage(jb_engine* e, int phase, int iters, float* avg_us, double* flops, void* stream) {
  if (!e || !avg_us || !flops) return fail("null argument");
  if (phase < -1 || phase >= jb::PH_COUNT || iters <= 0) return fail("bad phase / iters");   // -1: an empty launch (setup + teardown only)
  if (!e->plan_B) return fail("jb_upload_plan must be called first");
  if (ensure_step(e, e->plan_B)) return 1;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  double fl = 0;
  const int gi = jb::gemm_index(phase);
  if (gi >= 0) {
    const jb::HgPhase& ph = e->h_prm->cx.gph[gi];
    for (int i = ph.first; i < ph.first + ph.count; ++i)
      fl += 2.0 * e->h_probs[i].M * e->h_probs[i].N * e->h_probs[i].K;
  }
  int lo = phase < 0 ? 0 : phase, hi = phase + 1, one = 1, zero = 0;
  unsigned int* bar = e->bar + 64;     // (a single phase: no grid barrier)
  unsigned long long* ts = nullptr;
  int3 adv0 = make_int3(0, 0, 0);
  unsigned int* bar_next = e->bar + 96;
  void* args[] = {e->h_prm, &lo, &hi, &one, &bar, &zero, &zero, &ts, &adv0, &bar_next};
  cudaEvent_t a, b;
  CU(cudaEventCreate(&a)); CU(cudaEventCreate(&b));
  int nwarm = 3;
  if (const char* pv = getenv("JB_STAGE_WARM")) nwarm = atoi(pv);   // 0 under ncu: one profiled launch per phase
  for (int i = 0; i < nwarm; ++i)
    if (launch_kstep_raw(e, args, s)) return 1;
  CU(cudaEventRecord(a, s));
  for (int i = 0; i < iters; ++i)
    if (launch_kstep_raw(e, args, s)) return 1;
  CU(cudaEventRecord(b, s));
  CU(cudaEventSynchronize(b));
  float ms = 0;
  CU(cudaEventElapsedTime(&ms, a, b));
  cudaEventDestroy(a); cudaEventDestroy(b);
  e->launches += iters + 3;
  *avg_us = ms * 1000.f / static_cast<float>(iters);
  *flops = fl;
  return 0;
}

// In-kernel phase timeline: runs `iters` (+1 warm-up) training steps in ONE launch with CTA 0 recording the global timer at
// every phase boundary; out_us[p] = average microseconds of phase p INSIDE the persistent kernel (barrier included).
// Consumes plan row 0 for every step (the cursor is rewound) and takes optimizer steps like jb_train_steps.
int jb_profile_step(jb_engine* e, int iters, float* out_us, int cap, int* n_launches, void* stream) {
  if (!e || !out_us || !n_launches || iters <= 0) return fail("bad argument");
  if (!e->plan_B) return fail("jb_upload_plan must be called first");
  if (!e->data[0] || !e->data[1]) return fail("jb_set_dataset must be called for both modalities first");
  if (iters + 1 > e->plan_steps) iters = e->plan_steps - 1;
  if (iters < 1) return fail("the plan needs at least two rows for a profile");
  if (ensure_step(e, e->plan_B)) return 1;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const size_t nhead = 1 + static_cast<size_t>(iters + 1) * jb::PH_COUNT;
  const size_t ndet = static_cast<size_t>(iters + 1) * jb::PH_COUNT * e->grid * 3;
  const size_t ngem = static_cast<size_t>(iters + 1) * jb::SK_NUM_GEMM * 8;
  const size_t nts = nhead + ndet + ngem + static_cast<size_t>(iters + 1) * jb::PH_COUNT * 8;
  if (e->d_ts) { cudaFree(e->d_ts); e->d_ts = nullptr; }
  CU(cudaMalloc(&e->d_ts, nts * 8));
  CU(cudaMemsetAsync(e->d_ts, 0, nts * 8, s));
  CU(cudaMemsetAsync(&e->ctl->cursor, 0, sizeof(long long), s));
  if (launch_step(e, jb::PH_GATHER, jb::PH_COUNT, iters + 1, 0, s, e->d_ts)) return 1;
  std::vector<unsigned long long> ts(nts);
  CU(cudaMemcpyAsync(ts.data(), e->d_ts, nts * 8, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  std::vector<double> acc(jb::PH_COUNT, 0.0);
  for (int it = 1; it <= iters; ++it)
    for (int p = 0; p < jb::PH_COUNT; ++p) {
      const size_t k = 1 + static_cast<size_t>(it) * jb::PH_COUNT + p;
      acc[p] += static_cast<double>(ts[k] - ts[k - 1]) * 1e-3;
    }
  {  // per-CTA detail
    const int nc = e->grid;
    auto det = [&](int it, int p, int cta, int k) { return ts[nhead + ((static_cast<size_t>(it) * jb::PH_COUNT + p) * nc + cta) * 3 + k]; };
    // SM clock rate from CTA 0: cycles per ns over steps 1 .. iters
    const double cyc = static_cast<double>(det(iters, jb::PH_COUNT - 1, 0, 1) - det(1, 0, 0, 0));
    const double ns = static_cast<double>(det(iters, jb::PH_COUNT - 1, 0, 2) - ts[1 + jb::PH_COUNT - 1]);
    const double ghz = ns > 0 ? cyc / ns : 1.9;
    // GEMM role stamps of CTA 0 (cycles after the phase began): first TMA issued, last TMA issued, first stage landed,
    // last stage landed, accumulator final, tile stored
    e->prof_gemm.assign(jb::SK_NUM_GEMM * 7, 0.f);
    for (int gi = 0; gi < jb::SK_NUM_GEMM; ++gi)
      for (int it = 1; it <= iters; ++it) {
        const unsigned long long* d = &ts[nhead + ndet + (static_cast<size_t>(it) * jb::SK_NUM_GEMM + gi) * 8];
        for (int k = 0; k < 7; ++k)
          e->prof_gemm[gi * 7 + k] += static_cast<float>(static_cast<double>(static_cast<long long>(d[k] - d[7])) / ghz * 1e-3 / iters);
      }
    if (getenv("JB_PROF_ELEM")) {   // element-wise phase stamps of CTA 0 (BatchNorm forward): cycles after the phase began
      for (int p : {static_cast<int>(jb::PH_ENC1), static_cast<int>(jb::PH_ENC2), static_cast<int>(jb::PH_DEC1), static_cast<int>(jb::PH_DEC2), static_cast<int>(jb::PH_BN1), static_cast<int>(jb::PH_BN2)}) {
        double a[7] = {0, 0, 0, 0, 0, 0, 0};
        for (int it = 1; it <= iters; ++it) {
          const unsigned long long* d = &ts[nhead + ndet + ngem + (static_cast<size_t>(it) * jb::PH_COUNT + p) * 8];
          for (int k = 0; k < 7; ++k) a[k] += static_cast<double>(static_cast<long long>(d[k] - d[7])) / ghz * 1e-3 / iters;
        }
        fprintf(stderr, "bn fwd (tail / slab) phase %d CTA0, us after the phase began: enter %.2f | pass 1 + sum %.2f | pass 2 + sum %.2f | cluster sync %.2f | merge + stats %.2f | apply %.2f | %.2f\n",
                p, a[0], a[1], a[2], a[3], a[4], a[5], a[6]);
      }
    }
    if (const char* pv = getenv("JB_PROF_CTA_PHASE")) {   // per-CTA work of one phase (us, averaged over the steps)
      const int p = atoi(pv);
      if (p >= 0 && p < jb::PH_COUNT) {
        fprintf(stderr, "phase %d work per CTA (us):", p);
        for (int c = 0; c < nc; ++c) {
          double w = 0;
          for (int it = 1; it <= iters; ++it) w += static_cast<double>(det(it, p, c, 1) - det(it, p, c, 0)) / ghz * 1e-3;
          fprintf(stderr, "%s%.1f", c % 16 == 0 ? "\n  " : " ", w / iters);
        }
        fprintf(stderr, "\n");
      }
    }
    e->prof_detail.assign(jb::PH_COUNT * 4, 0.f);
    for (int p = 0; p < jb::PH_COUNT; ++p) {
      double wmax = 0, wavg = 0, tail = 0;
      for (int it = 1; it <= iters; ++it) {
        double m = 0, a = 0;
        unsigned long long latest = 0;
        for (int c = 0; c < nc; ++c) {
          const double w = static_cast<double>(det(it, p, c, 1) - det(it, p, c, 0)) / ghz * 1e-3;
          m = w > m ? w : m; a += w;
          latest = det(it, p, c, 2) > latest ? det(it, p, c, 2) : latest;
        }
        wmax += m; wavg += a / nc;
        const unsigned long long end = ts[1 + static_cast<size_t>(it) * jb::PH_COUNT + p];
        tail += end > latest ? static_cast<double>(end - latest) * 1e-3 : 0.0;
      }
      e->prof_detail[p * 4 + 0] = static_cast<float>(acc[p] / iters);
      e->prof_detail[p * 4 + 1] = static_cast<float>(wmax / iters);
      e->prof_detail[p * 4 + 2] = static_cast<float>(wavg / iters);
      e->prof_detail[p * 4 + 3] = static_cast<float>(tail / iters);
    }
  }
  for (int k = 0; k < 8; ++k) e->nbt[k] += iters + 1;
  e->eval_dirty = true;
  *n_launches = jb::PH_COUNT;
  for (int p = 0; p < jb::PH_COUNT && p < cap; ++p) out_us[p] = static_cast<float>(acc[p] / iters);
  return 0;
}

int jb_profile_detail(jb_engine* e, float* out, int cap) {
  if (!e || !out) return fail("null argument");
  if (e->prof_detail.empty()) return fail("jb_profile_step has not run");
  for (size_t k = 0; k < e->prof_detail.size() && k < static_cast<size_t>(cap); ++k) out[k] = e->prof_detail[k];
  for (size_t k = 0; k < e->prof_gemm.size() && e->prof_detail.size() + k < static_cast<size_t>(cap); ++k) out[e->prof_detail.size() + k] = e->prof_gemm[k];
  return 0;
}

int jb_read_losses(jb_engine* e, float* out, int nsteps, void* stream) {
  if (!e || !out) return fail("null argument");
  if (nsteps > e->plan_steps) return fail("only %d steps in the plan", e->plan_steps);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  CU(cudaMemcpyAsync(out, e->out_loss, static_cast<size_t>(nsteps) * 8 * 4, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  return 0;
}

int jb_encode(jb_engine* e, int mod, const float* X, long long n, long long ldx, float* out, long long ldo, int on_device,
              void* stream) {
  if (!e || !X || !out) return fail("null argument");
  return eval_common(e, mod, -1, X, n, ldx, out, ldo, on_device, static_cast<cudaStream_t>(stream));
}
int jb_predict(jb_engine* e, int from, int to, const float* X, long long n, long long ldx, float* out, long long ldo,
               int on_device, void* stream) {
  if (!e || !X || !out) return fail("null argument");
  if (to < 0) return fail("modality index out of range");
  return eval_common(e, from, to, X, n, ldx, out, ldo, on_device, static_cast<cudaStream_t>(stream));
}

// ---------------------------------------------------------------------------------------------- PCA projection
namespace {
struct DevBuf {  // scoped device allocation
  float* p = nullptr;
  ~DevBuf() { if (p) cudaFree(p); }
  int alloc(size_t floats) {
    CU(cudaMalloc(&p, floats * 4));
    return 0;
  }
};
int launch_one(jb_engine* e, GemmProblem& g, GemmProblem* d_slot, cudaStream_t s) {
  jb::gemm_table_finalize(&g, 1);
  CU(cudaMemcpyAsync(d_slot, &g, sizeof g, cudaMemcpyHostToDevice, s));
  CU(jb::gemm_launch(d_slot, 1, g.tiles_m * g.tiles_n, s));
  ++e->launches;
  return 0;
}
// rows per chunk so that one [rows, ld] fp32 temporary stays around 256 MB
long long pca_chunk_rows(long long ld) {
  long long r = (64LL << 20) / (ld > 0 ? ld : 1);
  if (r < 128) r = 128;
  if (r > 16384) r = 16384;
  return r;
}
}  // namespace

int jb_pca_project(jb_engine* e, const float* X, long long n, long long d, const float* comp, const float* mean, int k,
                   float m, float sdev, float* out, int on_device, void* stream) {
  if (!e || !X || !comp || !mean || !out) return fail("null argument");
  if (n <= 0 || d <= 0 || k <= 0) return fail("bad PCA shape");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const long long ldd = r4(static_cast<int>(d));
  const int ldk = r4(k);
  const long long R = pca_chunk_rows(ldd);
  DevBuf c_raw, c_hi, c_lo, d_mean, x_raw, x_hi, x_lo, z;
  if (c_raw.alloc(static_cast<size_t>(k) * d) || c_hi.alloc(static_cast<size_t>(k) * ldd) || c_lo.alloc(static_cast<size_t>(k) * ldd) ||
      d_mean.alloc(d) || x_hi.alloc(static_cast<size_t>(R) * ldd) || x_lo.alloc(static_cast<size_t>(R) * ldd) ||
      z.alloc(static_cast<size_t>(R) * ldk)) return 1;
  if (!on_device && x_raw.alloc(static_cast<size_t>(R) * d)) return 1;
  CU(cudaMemcpyAsync(c_raw.p, comp, static_cast<size_t>(k) * d * 4, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(d_mean.p, mean, static_cast<size_t>(d) * 4, cudaMemcpyHostToDevice, s));
  jb::k_split_tf32<<<k, 256, 0, s>>>(c_raw.p, d, k, static_cast<int>(d), 2, nullptr, 1.f, 0.f, c_hi.p, c_lo.p, ldd); ++e->launches;
  DevBuf out_dev;
  if (!on_device && out_dev.alloc(static_cast<size_t>(R) * k)) return 1;
  for (long long r0 = 0; r0 < n; r0 += R) {
    const long long rows = n - r0 < R ? n - r0 : R;
    const float* src = X + r0 * d;
    if (!on_device) {
      CU(cudaMemcpyAsync(x_raw.p, src, static_cast<size_t>(rows) * d * 4, cudaMemcpyHostToDevice, s));
      src = x_raw.p;
    }
    jb::k_split_tf32<<<static_cast<unsigned>(rows), 256, 0, s>>>(src, d, rows, static_cast<int>(d), 0, d_mean.p, 1.f, 0.f, x_hi.p, x_lo.p, ldd); ++e->launches;
    {
      GemmProblem g;   // one 3xTF32 launch on the hi/lo planes
      const int bn = k <= 32 ? 32 : 64;
      int rc = jb::gemm_problem_fill(&g, x_hi.p, static_cast<int>(ldd), 0, c_hi.p, static_cast<int>(ldd), 0, z.p, ldk,
                                     static_cast<int>(rows), k, static_cast<int>(d), bn, jb::EPI_STORE, nullptr, 0.f, 0, 0,
                                     x_lo.p, c_lo.p);
      if (rc) return fail("PCA tensor map encode failed (%d)", rc);
      if (launch_one(e, g, e->d_ev_probs, s)) return 1;
    }
    float* dst = on_device ? out + r0 * k : out_dev.p;
    jb::k_standardise<<<static_cast<unsigned>(rows), 128, 0, s>>>(z.p, ldk, rows, k, m, sdev, dst, k); ++e->launches;
    if (!on_device) CU(cudaMemcpyAsync(out + r0 * k, out_dev.p, static_cast<size_t>(rows) * k * 4, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));  // temporaries and table slots are reused by the next chunk
  }
  CU(cudaGetLastError());
  return 0;
}

// PCA fit, GPU part (jamie/jamie.py:436-452: sklearn PCA(n_components).fit): column sums and the centred Gram matrix; the
// d x d symmetric eigenproblem stays with the caller (host LAPACK, independent of n), as does the all-reduce of both
// results when the rows are sharded over ranks.
int jb_pca_colsum(jb_engine* e, const float* X, long long n, long long d, double* colsum, int on_device, void* stream) {
  if (!e || !X || !colsum) return fail("null argument");
  if (n <= 0 || d <= 0) return fail("bad PCA shape");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const long long R = pca_chunk_rows(d);
  const int slabs = 64;
  DevBuf x_raw;
  DevArr<double> part;
  if (part.alloc(static_cast<size_t>(slabs) * d)) return 1;
  if (!on_device && x_raw.alloc(static_cast<size_t>(R) * d)) return 1;
  std::vector<double> h(static_cast<size_t>(slabs) * d);
  for (long long c = 0; c < d; ++c) colsum[c] = 0.0;
  for (long long r0 = 0; r0 < n; r0 += R) {
    const long long rows = n - r0 < R ? n - r0 : R;
    const float* src = X + r0 * d;
    if (!on_device) {
      CU(cudaMemcpyAsync(x_raw.p, src, static_cast<size_t>(rows) * d * 4, cudaMemcpyHostToDevice, s));
      src = x_raw.p;
    }
    const long long per = (rows + slabs - 1) / slabs;
    jb::k_col_sums<<<dim3(static_cast<unsigned>((d + 127) / 128), slabs), 128, 0, s>>>(src, rows, d, per, part.p); ++e->launches;
    CU(cudaMemcpyAsync(h.data(), part.p, h.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    for (int sl = 0; sl < slabs; ++sl)   // fixed order: deterministic
      if (sl * per < rows)
        for (long long c = 0; c < d; ++c) colsum[c] += h[static_cast<size_t>(sl) * d + c];
  }
  CU(cudaGetLastError());
  return 0;
}

int jb_pca_gram(jb_engine* e, const float* X, long long n, long long d, const double* mean, double* gram, int on_device, void* stream) {
  if (!e || !X || !mean || !gram) return fail("null argument");
  if (n <= 0 || d <= 0) return fail("bad PCA shape");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const long long ldd = r4(static_cast<int>(d));
  const long long R = pca_chunk_rows(ldd);
  DevBuf d_mean, x_raw, x_hi, x_lo, g32;
  DevArr<double> g64;
  if (d_mean.alloc(d) || x_hi.alloc(static_cast<size_t>(R) * ldd) || x_lo.alloc(static_cast<size_t>(R) * ldd) ||
      g32.alloc(static_cast<size_t>(d) * ldd) || g64.alloc(static_cast<size_t>(d) * d)) return 1;
  if (!on_device && x_raw.alloc(static_cast<size_t>(R) * d)) return 1;
  {
    std::vector<float> mf(d);
    for (long long c = 0; c < d; ++c) mf[c] = static_cast<float>(mean[c]);
    CU(cudaMemcpyAsync(d_mean.p, mf.data(), static_cast<size_t>(d) * 4, cudaMemcpyHostToDevice, s));
    CU(cudaStreamSynchronize(s));
  }
  CU(cudaMemsetAsync(g64.p, 0, static_cast<size_t>(d) * d * sizeof(double), s));
  for (long long r0 = 0; r0 < n; r0 += R) {
    const long long rows = n - r0 < R ? n - r0 : R;
    const float* src = X + r0 * d;
    if (!on_device) {
      CU(cudaMemcpyAsync(x_raw.p, src, static_cast<size_t>(rows) * d * 4, cudaMemcpyHostToDevice, s));
      src = x_raw.p;
    }
    jb::k_split_tf32<<<static_cast<unsigned>(rows), 256, 0, s>>>(src, d, rows, static_cast<int>(d), 0, d_mean.p, 1.f, 0.f, x_hi.p, x_lo.p, ldd); ++e->launches;
    {
      GemmProblem g;   // G[d, d] = Xc^T Xc over this chunk: both operands are the same [rows][ldd] planes, MN-major (K = rows)
      int rc = jb::gemm_problem_fill(&g, x_hi.p, static_cast<int>(ldd), 1, x_hi.p, static_cast<int>(ldd), 1, g32.p, static_cast<int>(ldd),
                                     static_cast<int>(d), static_cast<int>(d), static_cast<int>(rows), 64, jb::EPI_STORE, nullptr, 0.f, 0, 0,
                                     x_lo.p, x_lo.p);
      if (rc) return fail("PCA Gram tensor map encode failed (%d)", rc);
      if (launch_one(e, g, e->d_ev_probs, s)) return 1;
    }
    jb::k_acc_f64<<<static_cast<unsigned>(d), 256, 0, s>>>(g32.p, ldd, g64.p, d); ++e->launches;
    CU(cudaStreamSynchronize(s));  // temporaries and the table slot are reused by the next chunk
  }
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(gram, g64.p, static_cast<size_t>(d) * d * sizeof(double), cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  return 0;
}

namespace {
// preclass.inverse_transform with PCA on device rows: out = (Z * s + m) @ comp + mean. The component hi/lo planes are split
// once (prepare); apply then maps any number of row blocks (jb_pca_inverse's chunks, jb_feature_impact's batches).
struct PcaInverse {
  DevBuf c_raw, c_hi, c_lo, d_mean;
  int k = 0, ldk = 0;
  long long d = 0, ldd = 0;
  float m = 0.f, s = 1.f;
  int prepare(jb_engine* e, const float* comp, const float* mean, int k_, long long d_, float m_, float s_, cudaStream_t st) {
    k = k_; d = d_; m = m_; s = s_;
    ldd = r4(static_cast<int>(d));
    ldk = r4(k);
    if (c_raw.alloc(static_cast<size_t>(k) * d) || c_hi.alloc(static_cast<size_t>(k) * ldd) ||
        c_lo.alloc(static_cast<size_t>(k) * ldd) || d_mean.alloc(d)) return 1;
    CU(cudaMemcpyAsync(c_raw.p, comp, static_cast<size_t>(k) * d * 4, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_mean.p, mean, static_cast<size_t>(d) * 4, cudaMemcpyHostToDevice, st));
    jb::k_split_tf32<<<k, 256, 0, st>>>(c_raw.p, d, k, static_cast<int>(d), 2, nullptr, 1.f, 0.f, c_hi.p, c_lo.p, ldd); ++e->launches;
    return 0;
  }
  // Z: [rows, ldz] device; z_hi / z_lo: [rows, ldk] scratch; out: [rows, ldd] device
  int apply(jb_engine* e, const float* Z, long long ldz, long long rows, float* z_hi, float* z_lo, float* out, cudaStream_t st) {
    jb::k_split_tf32<<<static_cast<unsigned>(rows), 128, 0, st>>>(Z, ldz, rows, k, 1, nullptr, s, m, z_hi, z_lo, ldk); ++e->launches;
    GemmProblem g;   // out[rows, d] = A[rows, k] * comp[k, d]: B is logically [N = d, K = k] stored [k][d] -> MN-major
    int rc = jb::gemm_problem_fill(&g, z_hi, ldk, 0, c_hi.p, static_cast<int>(ldd), 1, out, static_cast<int>(ldd),
                                   static_cast<int>(rows), static_cast<int>(d), k, 64, jb::EPI_BIAS, d_mean.p, 0.f, 0, 0,
                                   z_lo, c_lo.p);
    if (rc) return fail("PCA tensor map encode failed (%d)", rc);
    return launch_one(e, g, e->d_ev_probs, st);
  }
};
}  // namespace

int jb_pca_inverse(jb_engine* e, const float* Z, long long n, int k, const float* comp, const float* mean, long long d,
                   float m, float sdev, float* out, int on_device, void* stream) {
  if (!e || !Z || !comp || !mean || !out) return fail("null argument");
  if (n <= 0 || d <= 0 || k <= 0) return fail("bad PCA shape");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PcaInverse inv;
  if (inv.prepare(e, comp, mean, k, d, m, sdev, s)) return 1;
  const long long ldd = inv.ldd;
  const long long R = pca_chunk_rows(ldd);
  DevBuf z_raw, z_hi, z_lo, o;
  if (z_hi.alloc(static_cast<size_t>(R) * inv.ldk) || z_lo.alloc(static_cast<size_t>(R) * inv.ldk) ||
      o.alloc(static_cast<size_t>(R) * ldd)) return 1;
  if (!on_device && z_raw.alloc(static_cast<size_t>(R) * k)) return 1;
  for (long long r0 = 0; r0 < n; r0 += R) {
    const long long rows = n - r0 < R ? n - r0 : R;
    const float* src = Z + r0 * k;
    if (!on_device) {
      CU(cudaMemcpyAsync(z_raw.p, src, static_cast<size_t>(rows) * k * 4, cudaMemcpyHostToDevice, s));
      src = z_raw.p;
    }
    if (inv.apply(e, src, k, rows, z_hi.p, z_lo.p, o.p, s)) return 1;
    CU(cudaMemcpy2DAsync(out + r0 * d, static_cast<size_t>(d) * 4, o.p, static_cast<size_t>(ldd) * 4, static_cast<size_t>(d) * 4,
                         rows, on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
  }
  CU(cudaGetLastError());
  return 0;
}

// ---------------------------------------------------------------------------------------------- feature ablation (SURVEY 3.2)

int jb_feature_impact(jb_engine* e, int from, int to, const double* Z, long long n, long long n_feat, const double* dz,
                      const double* w, const int* w_col, int map_kind, const float* comp, const float* mean, float m, float sdev,
                      const double* aff_scale, const double* aff_shift, long long d_out, const float* target, double* base_r,
                      double* r, double* shift, long long batch_bytes, void* stream) {
  if (!e || !Z || (n_feat > 0 && (!dz || !w || !shift))) return fail("null argument");
  if (from < 0 || from > 1 || to < -1 || to > 1) return fail("modality index out of range");
  if (n <= 0 || n_feat < 0 || d_out <= 0) return fail("bad feature-impact shape");
  const int D_in = e->D[from];
  const int D_to = to < 0 ? e->L : e->D[to];
  if (map_kind == 1) {
    if (!comp || !mean || to < 0) return fail("the PCA output map needs comp, mean and an output modality");
  } else if (map_kind == 2) {
    if (!aff_scale || !aff_shift || d_out != D_to) return fail("the per-column output map needs %d scales and shifts", D_to);
  } else if (map_kind != 0 || d_out != D_to) {
    return fail("output map %d with %lld output columns (the network gives %d)", map_kind, d_out, D_to);
  }
  if (target && (!base_r || !r)) return fail("a target needs base_r and r");
  if (d_out > (1LL << 30) || n > (1LL << 40)) return fail("bad feature-impact shape");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const long long SL = jb::IMP_SLAB;
  const long long ldin = r4(D_in), ldto = r4(D_to), ldo = map_kind == 1 ? r4(static_cast<int>(d_out)) : ldto;
  // bytes per row of one slot (ablated input, chain output, and for PCA the split planes and the inverse's output), per slot
  // (its moment sums) and per feature (its dz column over all rows)
  const double row_b = 4.0 * (ldin + ldto + (map_kind == 1 ? 2.0 * ldto + ldo : 0.0));
  const double slot_b = 32.0 * d_out, feat_b = 8.0 * n;
  const double fixed = 8.0 * n * D_in + (w_col ? 12.0 * n_feat : 8.0 * n_feat * D_in) + (target ? 4.0 * n * d_out : 0.0) +
                       (map_kind == 1 ? 12.0 * D_to * ldo + 4.0 * d_out : 0.0) + (map_kind == 2 ? 16.0 * d_out : 0.0) + 16.0 * d_out;
  auto batch = [&](long long a, long long R) { return (a + 1) * (R * row_b + slot_b) + a * feat_b; };
  const long long n_pad = (n + SL - 1) / SL * SL;
  const long long a_min = n_feat > 0 ? 1 : 0;
  size_t free_b = 0, total_b = 0;
  CU(cudaMemGetInfo(&free_b, &total_b));
  const double avail = static_cast<double>(free_b) - (256.0 * (1 << 20));   // GEMM tables, tensor maps, allocator slack
  const double need_min = fixed + batch(a_min, n_pad < SL ? n_pad : SL);
  if (need_min > avail)
    return fail("feature impact needs %.2f GB of device memory for its smallest batch (one feature, %lld rows); %.2f GB free",
                need_min / 1e9, SL < n_pad ? SL : n_pad, static_cast<double>(free_b) / 1e9);
  // row range: up to 1024 rows, halved while two slots of it exceed the budget; then as many features as fit
  const double budget = static_cast<double>(batch_bytes) < avail - fixed ? static_cast<double>(batch_bytes) : avail - fixed;
  long long R = n_pad < 1024 ? n_pad : 1024;
  while (R > SL && batch(a_min, R) > budget) R = (R / 2 + SL - 1) / SL * SL;
  long long a = a_min;
  if (n_feat > 0) {
    a = static_cast<long long>((budget - (R * row_b + slot_b)) / (R * row_b + slot_b + feat_b));
    if (a < 1) a = 1;
    if (a > n_feat) a = n_feat;
    if (a > 65534) a = 65534;
    while (a > 1 && fixed + batch(a, R) > avail) a /= 2;
  }
  const long long S = a + 1;
  if ((S * R) > (1LL << 31) - 1) return fail("feature-impact batch of %lld rows", S * R);
  if (prepare_eval(e, s)) return 1;

  DevArr<double> dZ, dW, dDz, dAcc, dTacc, dSc, dSh;
  DevArr<int> dWc;
  DevArr<float> dT;
  DevBuf xin, cout, zhi, zlo, o;
  PcaInverse inv;
  if (dZ.upload(Z, static_cast<size_t>(n) * D_in) || dAcc.alloc(static_cast<size_t>(S) * d_out * 4) ||
      dTacc.alloc(static_cast<size_t>(2) * d_out) || xin.alloc(static_cast<size_t>(S * R) * ldin) ||
      cout.alloc(static_cast<size_t>(S * R) * ldto)) return 1;
  if (n_feat > 0) {
    if (w_col ? (dW.upload(w, n_feat) || dWc.upload(w_col, n_feat)) : dW.upload(w, static_cast<size_t>(n_feat) * D_in)) return 1;
    if (dDz.alloc(static_cast<size_t>(a) * n)) return 1;
  }
  if (target && dT.upload(target, static_cast<size_t>(n) * d_out)) return 1;
  if (map_kind == 2 && (dSc.upload(aff_scale, d_out) || dSh.upload(aff_shift, d_out))) return 1;
  if (map_kind == 1) {
    if (inv.prepare(e, comp, mean, D_to, d_out, m, sdev, s) || zhi.alloc(static_cast<size_t>(S * R) * inv.ldk) ||
        zlo.alloc(static_cast<size_t>(S * R) * inv.ldk) || o.alloc(static_cast<size_t>(S * R) * ldo)) return 1;
  }
  CU(cudaMemsetAsync(dTacc.p, 0, static_cast<size_t>(2) * d_out * sizeof(double), s));
  std::vector<double> acc(static_cast<size_t>(S) * d_out * 4), tacc(static_cast<size_t>(2) * d_out);
  const double N = static_cast<double>(n);
  const unsigned mgrid = static_cast<unsigned>((d_out + 127) / 128);
  for (long long j0 = 0; j0 < (n_feat > 0 ? n_feat : 1); j0 += (a > 0 ? a : 1)) {
    const long long na = n_feat - j0 < a ? n_feat - j0 : a;   // features of this batch (slots 1 .. na)
    if (na > 0) CU(cudaMemcpyAsync(dDz.p, dz + j0 * n, static_cast<size_t>(na) * n * 8, cudaMemcpyHostToDevice, s));
    CU(cudaMemsetAsync(dAcc.p, 0, static_cast<size_t>(na + 1) * d_out * 4 * sizeof(double), s));
    for (long long r0 = 0; r0 < n; r0 += R) {
      const int rows = static_cast<int>(n - r0 < R ? n - r0 : R);
      const long long brows = (na + 1) * rows;
      jb::k_ablate_rows<<<static_cast<unsigned>(brows), 128, 0, s>>>(dZ.p, D_in, n, r0, rows, static_cast<int>(j0), dDz.p,
                                                                     dW.p, dWc.p, xin.p, ldin); ++e->launches;
      if (eval_common(e, from, to, xin.p, brows, ldin, cout.p, ldto, 1, s)) return 1;
      const float* P = cout.p;
      if (map_kind == 1) {
        if (inv.apply(e, cout.p, ldto, brows, zhi.p, zlo.p, o.p, s)) return 1;
        P = o.p;
      }
      jb::k_impact_moments<<<dim3(mgrid, static_cast<unsigned>(na + 1)), 128, 0, s>>>(
          P, ldo, rows, r0, static_cast<int>(d_out), dT.p, dSc.p, dSh.p, dAcc.p, j0 == 0 ? dTacc.p : nullptr); ++e->launches;
    }
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(acc.data(), dAcc.p, static_cast<size_t>(na + 1) * d_out * 4 * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (j0 == 0) CU(cudaMemcpyAsync(tacc.data(), dTacc.p, tacc.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    // r as jb_metric_feature_pearson finishes it (x = the prediction, y = the target); a constant column gives nan
    auto pearson = [&](const double* q, long long c) {
      const double st = tacc[2 * c], stt = tacc[2 * c + 1];
      const double cxy = q[2] - q[0] * st / N, cxx = q[1] - q[0] * q[0] / N, cyy = stt - st * st / N;
      return cxy / std::sqrt(cxx * cyy);
    };
    if (j0 == 0 && target)
      for (long long c = 0; c < d_out; ++c) base_r[c] = pearson(&acc[static_cast<size_t>(c) * 4], c);
    for (long long q = 0; q < na; ++q)
      for (long long c = 0; c < d_out; ++c) {
        const double* v = &acc[(static_cast<size_t>(q + 1) * d_out + c) * 4];
        shift[(j0 + q) * d_out + c] = v[3] / N;
        if (target) r[(j0 + q) * d_out + c] = pearson(v, c);
      }
  }
  return 0;
}

// ---------------------------------------------------------------------------------------------- Shapley values (SURVEY 3.2)

int jb_shapley(jb_engine* e, int from, int to, const double* X, long long nx, const double* B, long long nb, long long d,
               const double* Zb, const int* perms, long long n_perm, const double* w, const int* w_col, int map_kind,
               const float* comp, const float* mean, float m, float sdev, const double* aff_scale, const double* aff_shift,
               const int* out_cols, long long n_out, double* phi, double* base, long long* stats, long long batch_bytes,
               void* stream) {
  if (!e || !X || !B || !Zb || !perms || !w || !phi || !base) return fail("null argument");
  if (from < 0 || from > 1 || to < -1 || to > 1) return fail("modality index out of range");
  if (nx <= 0 || nb <= 0 || d <= 0 || n_perm <= 0 || n_out <= 0) return fail("bad Shapley shape");
  if (d > 8LL * 65535 || n_out > 32LL * 65535 || nx * nb > (1LL << 31) - 1) return fail("Shapley problem too large to index");
  const int D_in = e->D[from];
  const int D_to = to < 0 ? e->L : e->D[to];
  if (map_kind == 1) {
    if (!comp || !mean || to < 0) return fail("the PCA output map needs comp, mean and an output modality");
  } else if (map_kind == 0 || map_kind == 2) {
    if (!out_cols) return fail("output map %d needs the selected output columns", map_kind);
    if (map_kind == 2 && (!aff_scale || !aff_shift)) return fail("the per-column output map needs %d scales and shifts", D_to);
    if (n_out > D_to) return fail("%lld output columns selected, the network gives %d", n_out, D_to);
    for (long long o = 0; o < n_out; ++o)
      if (out_cols[o] < 0 || out_cols[o] >= D_to) return fail("output column %d out of range [0, %d)", out_cols[o], D_to);
  } else {
    return fail("unknown output map %d", map_kind);
  }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const long long S_all = nx * nb;
  const int di = static_cast<int>(d);
  const long long Q = (d + jb::SHP_TC - 1) / jb::SHP_TC;
  const long long ldin = r4(D_in), ldto = r4(D_to), ldo = r4(static_cast<int>(n_out)), ldk = r4(D_to);
  // bytes per chain row (walk row, chain output, and for PCA the split planes and the inverse's output), per segment of a
  // batch (chunk sums, chunk counts and offsets, step -> row map), and fixed (raw rows, z_b, w, permutations, phi, f(b))
  const double row_b = 4.0 * (ldin + ldto + (map_kind == 1 ? 2.0 * ldk + ldo : 0.0));
  const double seg_b = 8.0 * Q * D_in + 8.0 * Q + 4.0 * d + 4.0;
  const double fixed = 8.0 * (nx + nb) * d + 8.0 * nb * D_in + 4.0 * n_perm * d + (w_col ? 12.0 * d : 8.0 * d * D_in) +
                       8.0 * nx * d * n_out + 4.0 * nb * n_out + 16.0 * S_all + 12.0 * n_out +
                       (map_kind == 1 ? 12.0 * D_to * ldo + 4.0 * n_out : 0.0) + (map_kind == 2 ? 16.0 * D_to : 0.0);
  size_t free_b = 0, total_b = 0;
  CU(cudaMemGetInfo(&free_b, &total_b));
  const double avail = static_cast<double>(free_b) - (256.0 * (1 << 20));   // GEMM tables, tensor maps, allocator slack
  const double need_min = fixed + d * row_b + seg_b;                         // one segment, every step active
  if (need_min > avail)
    return fail("Shapley values need %.2f GB of device memory for their smallest batch (one segment of %lld steps); "
                "%.2f GB free", need_min / 1e9, d, static_cast<double>(free_b) / 1e9);
  const double budget = static_cast<double>(batch_bytes) < avail - fixed ? static_cast<double>(batch_bytes) : avail - fixed;
  if (prepare_eval(e, s)) return 1;

  DevArr<double> dX, dB, dZb, dW, dPhi, dBase, dSc, dSh, dPart;
  DevArr<int> dPerm, dWc, dOc, dCcnt, dCoff, dFirst, dRowof;
  DevArr<long long> dCnt;
  DevArr<float> dFB;
  DevBuf xin, cout, zhi, zlo, o;
  PcaInverse inv;
  if (dX.upload(X, static_cast<size_t>(nx) * d) || dB.upload(B, static_cast<size_t>(nb) * d) ||
      dZb.upload(Zb, static_cast<size_t>(nb) * D_in) || dPerm.upload(perms, static_cast<size_t>(n_perm) * d) ||
      (w_col ? (dW.upload(w, d) || dWc.upload(w_col, d)) : dW.upload(w, static_cast<size_t>(d) * D_in)) ||
      dPhi.upload(phi, static_cast<size_t>(nx) * d * n_out) || dBase.upload(base, n_out) ||
      dFB.alloc(static_cast<size_t>(nb) * n_out) || dCnt.alloc(S_all)) return 1;
  if (map_kind != 1 && dOc.upload(out_cols, n_out)) return 1;
  if (map_kind == 2 && (dSc.upload(aff_scale, D_to) || dSh.upload(aff_shift, D_to))) return 1;
  if (map_kind == 1 && inv.prepare(e, comp, mean, D_to, n_out, m, sdev, s)) return 1;

  // chain rows per segment (the same for every permutation), then batches: runs of segments in order whose rows and
  // per-segment buffers fit the budget; a segment is never split
  jb::k_shap_count<<<static_cast<unsigned>(S_all), 256, 0, s>>>(dX.p, dB.p, di, static_cast<int>(nb), dCnt.p); ++e->launches;
  CU(cudaGetLastError());
  std::vector<long long> cnt(S_all);
  CU(cudaMemcpyAsync(cnt.data(), dCnt.p, S_all * sizeof(long long), cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  struct Batch { long long s0, S, rows; };
  std::vector<Batch> batches;
  long long Smax = 1, Rmax = 0, total_rows = 0;
  for (long long g = 0; g < S_all;) {
    Batch bt{g, 0, 0};
    while (g < S_all && (bt.S == 0 || ((bt.rows + cnt[g]) * row_b + (bt.S + 1) * seg_b <= budget &&
                                       bt.rows + cnt[g] <= (1LL << 30) && bt.S < (1LL << 24)))) {
      bt.rows += cnt[g++];
      ++bt.S;
    }
    batches.push_back(bt);
    Smax = bt.S > Smax ? bt.S : Smax;
    Rmax = bt.rows > Rmax ? bt.rows : Rmax;
    total_rows += bt.rows;
  }
  const long long Rb = nb < d ? nb : d;   // rows per chunk of the f(b) pass
  const long long R = Rmax > Rb ? Rmax : Rb;
  if (xin.alloc(static_cast<size_t>(R) * ldin) || cout.alloc(static_cast<size_t>(R) * ldto) ||
      dPart.alloc(static_cast<size_t>(Smax) * Q * D_in) || dCcnt.alloc(static_cast<size_t>(Smax) * Q) ||
      dCoff.alloc(static_cast<size_t>(Smax) * Q) || dFirst.alloc(Smax) || dRowof.alloc(static_cast<size_t>(Smax) * d)) return 1;
  if (map_kind == 1 && (zhi.alloc(static_cast<size_t>(R) * inv.ldk) || zlo.alloc(static_cast<size_t>(R) * inv.ldk) ||
                        o.alloc(static_cast<size_t>(R) * ldo))) return 1;
  // the chain (and for PCA the inverse) of `rows` walk rows in xin; the mapped outputs are then read through ShapOut
  auto chain = [&](long long rows, jb::ShapOut* out) -> int {
    if (eval_common(e, from, to, xin.p, rows, ldin, cout.p, ldto, 1, s)) return 1;
    *out = jb::ShapOut{cout.p, ldto, map_kind, dOc.p, dSc.p, dSh.p};
    if (map_kind == 1) {
      if (inv.apply(e, cout.p, ldto, rows, zhi.p, zlo.p, o.p, s)) return 1;
      out->Y = o.p;
      out->ldy = ldo;
    }
    return 0;
  };
  const unsigned ogrid = static_cast<unsigned>((n_out + 127) / 128);
  for (long long b0 = 0; b0 < nb; b0 += Rb) {   // f(b) and base += sum_b f(b)
    const long long rows = nb - b0 < Rb ? nb - b0 : Rb;
    jb::k_shap_rows_f32<<<static_cast<unsigned>(rows), 128, 0, s>>>(dZb.p, D_in, b0, xin.p, ldin); ++e->launches;
    jb::ShapOut Y{};
    if (chain(rows, &Y)) return 1;
    jb::k_shap_base<<<ogrid, 128, 0, s>>>(Y, static_cast<int>(rows), b0, static_cast<int>(n_out), dFB.p, dBase.p); ++e->launches;
  }
  std::vector<int> first(Smax);
  for (long long p = 0; p < n_perm; ++p) {
    const int* perm = dPerm.p + p * d;
    for (const Batch& bt : batches) {
      if (bt.rows == 0) continue;
      const int S = static_cast<int>(bt.S);
      long long r = 0;
      for (long long i = 0; i < bt.S; ++i) { first[i] = static_cast<int>(r); r += cnt[bt.s0 + i]; }
      CU(cudaMemcpyAsync(dFirst.p, first.data(), bt.S * sizeof(int), cudaMemcpyHostToDevice, s));
      const dim3 wgrid(static_cast<unsigned>((S + jb::SHP_SG - 1) / jb::SHP_SG), static_cast<unsigned>(Q),
                       static_cast<unsigned>((D_in + jb::SHP_CT - 1) / jb::SHP_CT));
      jb::k_shap_walk<false><<<wgrid, jb::SHP_CT, 0, s>>>(dX.p, dB.p, di, static_cast<int>(nb), bt.s0, S, perm, dW.p, dWc.p,
                                                          D_in, dPart.p, dCcnt.p, nullptr, nullptr, 0, nullptr); ++e->launches;
      jb::k_shap_chunk_start<<<static_cast<unsigned>(S), 128, 0, s>>>(dZb.p, D_in, static_cast<int>(nb), bt.s0,
                                                                      static_cast<int>(Q), dPart.p, dCcnt.p, dFirst.p,
                                                                      dCoff.p); ++e->launches;
      jb::k_shap_walk<true><<<wgrid, jb::SHP_CT, 0, s>>>(dX.p, dB.p, di, static_cast<int>(nb), bt.s0, S, perm, dW.p, dWc.p,
                                                         D_in, dPart.p, nullptr, dCoff.p, xin.p, ldin, dRowof.p); ++e->launches;
      jb::ShapOut Y{};
      if (chain(bt.rows, &Y)) return 1;
      const long long xa = bt.s0 / nb, xb = (bt.s0 + bt.S - 1) / nb;
      const dim3 fgrid(static_cast<unsigned>(xb - xa + 1), static_cast<unsigned>((d + 7) / 8),
                       static_cast<unsigned>((n_out + 31) / 32));
      jb::k_shap_fold<<<fgrid, dim3(32, 8), 0, s>>>(Y, dFB.p, dRowof.p, dFirst.p, perm, di, static_cast<int>(nb), bt.s0, S,
                                                    static_cast<int>(n_out), dPhi.p); ++e->launches;
      // `first` is reused by the next batch: its pageable copy has been staged by the driver on return, as in eval_common
    }
  }
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(phi, dPhi.p, static_cast<size_t>(nx) * d * n_out * sizeof(double), cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(base, dBase.p, static_cast<size_t>(n_out) * sizeof(double), cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  if (stats) {
    stats[0] += n_perm * total_rows;
    stats[1] += n_perm * (S_all * d - total_rows);
  }
  return 0;
}

// ---------------------------------------------------------------------------------------------- evaluation metrics (N4)

int jb_metric_foscttm(const float* emb0, const float* emb1, long long n, int L, int device, unsigned long long* raw_count_closer) {
  if (!emb0 || !emb1 || !raw_count_closer) return fail("null argument");
  if (n <= 0 || L <= 0) return fail("bad embedding shape");
  CU(cudaSetDevice(device));
  DevArr<float> a, b; DevArr<double> diag; DevArr<unsigned long long> cnt;
  if (a.upload(emb0, static_cast<size_t>(n) * L) || b.upload(emb1, static_cast<size_t>(n) * L) || diag.alloc(n) || cnt.alloc(1)) return 1;
  CU(cudaMemset(cnt.p, 0, sizeof(unsigned long long)));
  jb::k_pair_diag<<<static_cast<unsigned>((n + 255) / 256), 256>>>(a.p, b.p, n, L, diag.p);
  const long long tiles = (n + jb::MT_TILE - 1) / jb::MT_TILE;
  jb::k_foscttm<<<metric_grid(tiles * tiles), jb::MT_THREADS>>>(a.p, b.p, n, L, diag.p, cnt.p);
  CU(cudaGetLastError());
  CU(cudaMemcpy(raw_count_closer, cnt.p, sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  return 0;
}

int jb_metric_knn_vote(const float* query, long long nq, const float* ref, const int* ref_class, long long nr, int L, int k,
                       int n_classes, int device, int* pred_class) {
  if (!query || !ref || !ref_class || !pred_class) return fail("null argument");
  if (nq <= 0 || nr <= 0 || L <= 0) return fail("bad embedding shape");
  if (k < 1 || k > nr) return fail("k = %d neighbours of %lld reference rows", k, nr);
  if (n_classes < 1 || n_classes > 8192) return fail("%d classes (1 .. 8192)", n_classes);
  for (long long j = 0; j < nr; ++j)
    if (ref_class[j] < 0 || ref_class[j] >= n_classes) return fail("class index %d of row %lld out of range", ref_class[j], j);
  CU(cudaSetDevice(device));
  long long Q = (512LL << 20) / (4 * nr);   // query rows per chunk: a 512 MB distance slab
  if (Q < 1) Q = 1;
  if (Q > nq) Q = nq;
  DevArr<float> q, r, D; DevArr<int> cls, pred;
  if (q.upload(query, static_cast<size_t>(nq) * L) || r.upload(ref, static_cast<size_t>(nr) * L) || cls.upload(ref_class, nr) ||
      D.alloc(static_cast<size_t>(Q) * nr) || pred.alloc(nq)) return 1;
  for (long long q0 = 0; q0 < nq; q0 += Q) {
    const long long rows = nq - q0 < Q ? nq - q0 : Q;
    const long long tiles = ((rows + jb::MT_TILE - 1) / jb::MT_TILE) * ((nr + jb::MT_TILE - 1) / jb::MT_TILE);
    jb::k_dist_rows<<<metric_grid(tiles), jb::MT_THREADS>>>(q.p + q0 * L, rows, r.p, nr, L, D.p);
    jb::k_knn_vote<<<static_cast<unsigned>(rows), jb::KV_THREADS, static_cast<size_t>(n_classes) * sizeof(int)>>>(D.p, nr, k, cls.p, n_classes, pred.p + q0);
  }
  CU(cudaGetLastError());
  CU(cudaMemcpy(pred_class, pred.p, static_cast<size_t>(nq) * sizeof(int), cudaMemcpyDeviceToHost));
  return 0;
}

int jb_metric_feature_pearson(const float* x, const float* y, long long n, long long d, int device, double* r) {
  if (!x || !y || !r) return fail("null argument");
  if (n <= 0 || d <= 0) return fail("bad matrix shape");
  CU(cudaSetDevice(device));
  const int slabs = static_cast<int>(n < 64 ? 1 : (n / 64 < 256 ? n / 64 : 256));
  const long long per = (n + slabs - 1) / slabs;
  DevArr<float> dx, dy; DevArr<double> part;
  if (dx.upload(x, static_cast<size_t>(n) * d) || dy.upload(y, static_cast<size_t>(n) * d) || part.alloc(static_cast<size_t>(slabs) * d * 5)) return 1;
  jb::k_col_moments<<<dim3(static_cast<unsigned>((d + 127) / 128), slabs), 128>>>(dx.p, dy.p, n, d, per, part.p);
  CU(cudaGetLastError());
  std::vector<double> h(static_cast<size_t>(slabs) * d * 5);
  CU(cudaMemcpy(h.data(), part.p, h.size() * sizeof(double), cudaMemcpyDeviceToHost));
  const double N = static_cast<double>(n);
  for (long long c = 0; c < d; ++c) {
    double m[5] = {0, 0, 0, 0, 0};
    for (int sl = 0; sl < slabs; ++sl)   // fixed order: deterministic
      for (int q = 0; q < 5; ++q) m[q] += h[(static_cast<size_t>(sl) * d + c) * 5 + q];
    const double cxy = m[4] - m[0] * m[1] / N, cxx = m[2] - m[0] * m[0] / N, cyy = m[3] - m[1] * m[1] / N;
    r[c] = cxy / std::sqrt(cxx * cyy);   // constant feature: 0 / 0 = nan, as the host definition gives
  }
  return 0;
}

namespace {
struct AurocStreams {   // compute and copy streams of jb_metric_feature_auroc; synchronised before the buffers are freed
  cudaStream_t s = nullptr, sc = nullptr;
  cudaEvent_t copied = nullptr, keyed = nullptr, done[2] = {nullptr, nullptr};
  int create() {
    CU(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&sc, cudaStreamNonBlocking));
    for (cudaEvent_t* ev : {&copied, &keyed, &done[0], &done[1]}) CU(cudaEventCreateWithFlags(ev, cudaEventDisableTiming));
    return 0;
  }
  ~AurocStreams() {
    if (s) cudaStreamSynchronize(s);
    if (sc) cudaStreamSynchronize(sc);
    for (cudaEvent_t ev : {copied, keyed, done[0], done[1]})
      if (ev) cudaEventDestroy(ev);
    if (s) cudaStreamDestroy(s);
    if (sc) cudaStreamDestroy(sc);
  }
};
}  // namespace

int jb_metric_feature_auroc(const float* scores, long long n, long long d, const long long* pos_ptr, const int* pos_row,
                            long long batch_bytes, int device, unsigned long long* u2, long long* n_pos) {
  if (!scores || !pos_ptr || !u2 || !n_pos) return fail("null argument");
  if (n <= 0 || d <= 0 || n > (1LL << 31) - 1) return fail("bad matrix shape: %lld rows, %lld columns", n, d);
  CU(cudaSetDevice(device));
  const bool shared = n <= jb::AU_SMEM_ROWS;
  // bytes per column of a batch: the fp32 slab, its keys, two buffers of positive lists (n rows each at most) and, above
  // the shared-memory regime, the sort's two key buffers
  const double col_b = (shared ? 16.0 : 24.0) * static_cast<double>(n);
  const double fixed = 16.0 * static_cast<double>(d) + 8.0;
  size_t free_b = 0, total_b = 0;
  CU(cudaMemGetInfo(&free_b, &total_b));
  const double avail = static_cast<double>(free_b) - (64.0 * (1 << 20));
  if (fixed + col_b > avail)
    return fail("AUROC needs %.2f GB of device memory for one column of %lld rows; %.2f GB free", (fixed + col_b) / 1e9, n,
                static_cast<double>(free_b) / 1e9);
  if (pos_ptr[0] != 0 || (pos_ptr[d] > 0 && !pos_row)) return fail("bad positive lists");
  for (long long c = 0; c < d; ++c) {
    const long long a = pos_ptr[c], b = pos_ptr[c + 1];
    if (b < a || b - a > n) return fail("column %lld has %lld positives in %lld rows", c, b - a, n);
    for (long long i = a; i < b; ++i)
      if (pos_row[i] < 0 || pos_row[i] >= n || (i > a && pos_row[i] <= pos_row[i - 1]))
        return fail("the positive rows of column %lld must increase and lie in [0, %lld)", c, n);
    n_pos[c] = b - a;
  }
  const double budget = static_cast<double>(batch_bytes) < avail - fixed ? static_cast<double>(batch_bytes) : avail - fixed;
  long long w = static_cast<long long>(budget / col_b);
  if (w < 1) w = 1;
  if (w > d) w = d;
  if (w > 65535LL * 32) w = 65535LL * 32;   // column tiles of k_auroc_keys in grid.y
  long long lmax = 0;                        // the largest batch's positive lists
  for (long long j0 = 0; j0 < d; j0 += w) {
    const long long j1 = j0 + w < d ? j0 + w : d;
    lmax = pos_ptr[j1] - pos_ptr[j0] > lmax ? pos_ptr[j1] - pos_ptr[j0] : lmax;
  }
  if (shared) CU(cudaFuncSetAttribute(jb::k_auroc_col<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * jb::AU_SMEM_ROWS));

  DevArr<long long> dPtr;
  DevArr<unsigned long long> dU2;
  DevArr<float> slab;
  DevArr<uint32_t> keys, scratch;
  DevArr<int> rows[2];
  if (dPtr.upload(pos_ptr, static_cast<size_t>(d) + 1) || dU2.alloc(d) || slab.alloc(static_cast<size_t>(n) * w) ||
      keys.alloc(static_cast<size_t>(n) * w) || rows[0].alloc(lmax) || rows[1].alloc(lmax) ||
      (!shared && scratch.alloc(static_cast<size_t>(2 * n) * w))) return 1;
  AurocStreams st;   // declared after the buffers: its destructor synchronises before they are freed
  if (st.create()) return 1;
  // batch b: the copy stream uploads the slab once batch b - 1 has been keyed and the lists once batch b - 2 is done, so
  // that the host-to-device copy of one batch overlaps the sort of the previous one
  int b = 0;
  for (long long j0 = 0; j0 < d; j0 += w, ++b) {
    const long long wb = d - j0 < w ? d - j0 : w;
    const long long l0 = pos_ptr[j0], nl = pos_ptr[j0 + wb] - l0;
    long long pcap = 0;
    for (long long c = j0; c < j0 + wb; ++c) pcap = n_pos[c] > pcap ? n_pos[c] : pcap;
    CU(cudaStreamWaitEvent(st.sc, st.keyed, 0));
    CU(cudaMemcpy2DAsync(slab.p, static_cast<size_t>(wb) * 4, scores + j0, static_cast<size_t>(d) * 4, static_cast<size_t>(wb) * 4,
                         static_cast<size_t>(n), cudaMemcpyHostToDevice, st.sc));
    CU(cudaStreamWaitEvent(st.sc, st.done[b & 1], 0));
    if (nl > 0) CU(cudaMemcpyAsync(rows[b & 1].p, pos_row + l0, static_cast<size_t>(nl) * 4, cudaMemcpyHostToDevice, st.sc));
    CU(cudaEventRecord(st.copied, st.sc));
    CU(cudaStreamWaitEvent(st.s, st.copied, 0));
    jb::k_auroc_keys<<<dim3(static_cast<unsigned>((n + 31) / 32), static_cast<unsigned>((wb + 31) / 32)), dim3(32, 8), 0, st.s>>>(
        slab.p, n, static_cast<int>(wb), keys.p);
    CU(cudaEventRecord(st.keyed, st.s));
    if (shared)
      jb::k_auroc_col<true><<<static_cast<unsigned>(wb), jb::AU_THREADS, static_cast<size_t>(pcap) * 8, st.s>>>(
          keys.p, n, dPtr.p + j0, rows[b & 1].p, static_cast<int>(pcap), nullptr, dU2.p + j0);
    else
      jb::k_auroc_col<false><<<static_cast<unsigned>(wb), jb::AU_THREADS, 0, st.s>>>(keys.p, n, dPtr.p + j0, rows[b & 1].p, 0,
                                                                                   scratch.p, dU2.p + j0);
    CU(cudaEventRecord(st.done[b & 1], st.s));
  }
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(u2, dU2.p, static_cast<size_t>(d) * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st.s));
  CU(cudaStreamSynchronize(st.s));
  return 0;
}

// ---------------------------------------------------------------------------------------------- kNN search and average

namespace {
struct KnnStream {   // the stream of jb_knn / jb_knn_average; synchronised before the buffers are freed
  cudaStream_t s = nullptr;
  int create() { CU(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking)); return 0; }
  ~KnnStream() {
    if (s) { cudaStreamSynchronize(s); cudaStreamDestroy(s); }
  }
};
double knn_avail() {   // free device memory less a margin for the context's own allocations
  size_t free_b = 0, total_b = 0;
  if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) return 0.0;
  return static_cast<double>(free_b) - (64.0 * (1 << 20));
}
}  // namespace

int jb_knn(const float* query, long long nq, const float* ref, long long nr, int L, int k, long long batch_bytes, int device,
           long long* idx, double* dist) {
  if (!query || !ref || !idx) return fail("null argument");
  if (nq <= 0 || nr <= 0 || L <= 0) return fail("bad embedding shape: %lld query rows, %lld reference rows, %d columns", nq, nr, L);
  if (nq > INT_MAX || nr > INT_MAX) return fail("%lld query rows, %lld reference rows: jb_knn takes fewer than 2^31 of each", nq, nr);
  if (k < 1 || k > jb::KN_MAXK || k > nr) return fail("k = %d neighbours: 1 <= k <= %d and k <= %lld reference rows", k, jb::KN_MAXK, nr);
  CU(cudaSetDevice(device));
  // device bytes: the reference rows (resident), and for each query row of a batch its fp32 row and output lists, and
  // per reference range its two list arrays and their length
  const double ref_b = 4.0 * static_cast<double>(nr) * L;
  const double row_b = 4.0 * L + 16.0 * k, range_b = 24.0 * k + 8.0;
  const double avail = knn_avail();
  if (ref_b + row_b + range_b > avail)
    return fail("kNN search needs %.2f GB of device memory for %lld reference rows and one query row; %.2f GB free",
                (ref_b + row_b + range_b) / 1e9, nr, (avail > 0 ? avail : 0) / 1e9);
  const double budget = static_cast<double>(batch_bytes) < avail - ref_b ? static_cast<double>(batch_bytes) : avail - ref_b;
  long long nqb = static_cast<long long>(budget / (row_b + range_b));
  if (nqb > nq) nqb = nq;
  if (nqb >= jb::MT_TILE) nqb -= nqb % jb::MT_TILE;
  if (nqb < 1) nqb = 1;
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  const long long target = 4LL * sms;   // blocks per batch: split the reference rows into ranges until a small batch has them
  const long long tiles_r = (nr + jb::MT_TILE - 1) / jb::MT_TILE;
  const long long min_tiles = 2 * ((k + jb::MT_TILE - 1) / jb::MT_TILE);   // per range: k rows and as many again to select from
  auto ranges_for = [&](long long rows, long long cap_lists) {
    const long long tq = (rows + jb::MT_TILE - 1) / jb::MT_TILE;
    long long S = (target + tq - 1) / tq;
    if (S > tiles_r / min_tiles) S = tiles_r / min_tiles;
    if (S > cap_lists / rows) S = cap_lists / rows;
    if (S < 1) S = 1;
    return S;
  };
  long long fit = static_cast<long long>((budget - static_cast<double>(nqb) * row_b) / (static_cast<double>(nqb) * range_b));
  const long long cap_lists = ranges_for(nqb, (fit > 1 ? fit : 1) * nqb) * nqb;   // (range, query) lists allocated
  CU(cudaFuncSetAttribute(jb::k_knn_search, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(jb::KN_SMEM)));

  DevArr<float> dr, dq;
  DevArr<double> ld, odist;
  DevArr<int> lj;
  DevArr<int2> meta;
  DevArr<long long> oidx;
  if (dr.alloc(static_cast<size_t>(nr) * L) || dq.alloc(static_cast<size_t>(nqb) * L) || ld.alloc(static_cast<size_t>(cap_lists) * 2 * k) ||
      lj.alloc(static_cast<size_t>(cap_lists) * 2 * k) || meta.alloc(cap_lists) || oidx.alloc(static_cast<size_t>(nqb) * k) ||
      (dist && odist.alloc(static_cast<size_t>(nqb) * k))) return 1;
  KnnStream st;   // declared after the buffers: its destructor synchronises before they are freed
  if (st.create()) return 1;
  CU(cudaMemcpyAsync(dr.p, ref, static_cast<size_t>(nr) * L * 4, cudaMemcpyHostToDevice, st.s));
  for (long long q0 = 0; q0 < nq; q0 += nqb) {
    const long long nb = nq - q0 < nqb ? nq - q0 : nqb;
    long long S = ranges_for(nb, cap_lists);
    const long long per = (tiles_r + S - 1) / S;
    S = (tiles_r + per - 1) / per;   // no empty range
    CU(cudaMemcpyAsync(dq.p, query + q0 * L, static_cast<size_t>(nb) * L * 4, cudaMemcpyHostToDevice, st.s));
    jb::k_knn_search<<<dim3(static_cast<unsigned>((nb + jb::MT_TILE - 1) / jb::MT_TILE), static_cast<unsigned>(S)), jb::MT_THREADS,
                       jb::KN_SMEM, st.s>>>(dq.p, nb, dr.p, nr, L, k, per, ld.p, lj.p, meta.p);
    jb::k_knn_merge<<<static_cast<unsigned>(nb), jb::KM_THREADS, 0, st.s>>>(ld.p, lj.p, meta.p, static_cast<int>(S), nb, k, oidx.p,
                                                                           dist ? odist.p : nullptr);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(idx + q0 * k, oidx.p, static_cast<size_t>(nb) * k * 8, cudaMemcpyDeviceToHost, st.s));
    if (dist) CU(cudaMemcpyAsync(dist + q0 * k, odist.p, static_cast<size_t>(nb) * k * 8, cudaMemcpyDeviceToHost, st.s));
  }
  CU(cudaStreamSynchronize(st.s));
  return 0;
}

int jb_knn_average(const long long* idx, const double* weights, long long nq, int k, const double* values, long long nr, long long w,
                   long long ldv, long long batch_bytes, int device, double* out) {
  if (!idx || !values || !out) return fail("null argument");
  if (nq <= 0 || nr <= 0 || w <= 0 || ldv < w) return fail("bad shape: %lld query rows, %lld reference rows, %lld columns, pitch %lld", nq, nr, w, ldv);
  if (nq > INT_MAX) return fail("%lld query rows: jb_knn_average takes fewer than 2^31", nq);
  if (k < 1 || k > jb::KN_MAXK) return fail("k = %d neighbours: 1 <= k <= %d", k, jb::KN_MAXK);
  for (long long e = 0; e < nq * k; ++e)
    if (idx[e] < 0 || idx[e] >= nr) return fail("neighbour index %lld of query row %lld out of range [0, %lld)", idx[e], e / k, nr);
  CU(cudaSetDevice(device));
  // device bytes: the lists and weights (resident), and per column of a slab the reference values and the output
  const double fixed = (weights ? 16.0 : 8.0) * static_cast<double>(nq) * k;
  const double col_b = 8.0 * static_cast<double>(nr + nq);
  const double avail = knn_avail();
  if (fixed + col_b > avail)
    return fail("kNN average needs %.2f GB of device memory for one column of %lld reference and %lld query rows; %.2f GB free",
                (fixed + col_b) / 1e9, nr, nq, (avail > 0 ? avail : 0) / 1e9);
  const double budget = static_cast<double>(batch_bytes) < avail - fixed ? static_cast<double>(batch_bytes) : avail - fixed;
  long long ws = static_cast<long long>(budget / col_b);
  if (ws < 1) ws = 1;
  if (ws > w) ws = w;
  if (ws > 65535LL * jb::KA_THREADS) ws = 65535LL * jb::KA_THREADS;   // column blocks in grid.y

  DevArr<long long> didx;
  DevArr<double> dw, vs, os;
  if (didx.alloc(static_cast<size_t>(nq) * k) || (weights && dw.alloc(static_cast<size_t>(nq) * k)) || vs.alloc(static_cast<size_t>(nr) * ws) ||
      os.alloc(static_cast<size_t>(nq) * ws)) return 1;
  KnnStream st;   // declared after the buffers: its destructor synchronises before they are freed
  if (st.create()) return 1;
  CU(cudaMemcpyAsync(didx.p, idx, static_cast<size_t>(nq) * k * 8, cudaMemcpyHostToDevice, st.s));
  if (weights) CU(cudaMemcpyAsync(dw.p, weights, static_cast<size_t>(nq) * k * 8, cudaMemcpyHostToDevice, st.s));
  for (long long c0 = 0; c0 < w; c0 += ws) {
    const long long wb = w - c0 < ws ? w - c0 : ws;
    CU(cudaMemcpy2DAsync(vs.p, static_cast<size_t>(wb) * 8, values + c0, static_cast<size_t>(ldv) * 8, static_cast<size_t>(wb) * 8,
                         static_cast<size_t>(nr), cudaMemcpyHostToDevice, st.s));
    jb::k_knn_average<<<dim3(static_cast<unsigned>(nq), static_cast<unsigned>((wb + jb::KA_THREADS - 1) / jb::KA_THREADS)), jb::KA_THREADS, 0,
                        st.s>>>(didx.p, weights ? dw.p : nullptr, k, vs.p, static_cast<int>(wb), os.p);
    CU(cudaGetLastError());
    CU(cudaMemcpy2DAsync(out + c0, static_cast<size_t>(w) * 8, os.p, static_cast<size_t>(wb) * 8, static_cast<size_t>(wb) * 8,
                         static_cast<size_t>(nq), cudaMemcpyDeviceToHost, st.s));
  }
  CU(cudaStreamSynchronize(st.s));
  return 0;
}

// ---------------------------------------------------------------------------------------------- silhouette sums

int jb_silhouette(const float* x, long long n, int L, const long long* label_off, int n_labels, long long batch_bytes,
                  int device, double* intra, double* inter) {
  if (!x || !label_off || !intra || !inter) return fail("null argument");
  if (n <= 0 || L <= 0) return fail("bad embedding shape: %lld rows, %d columns", n, L);
  if (n > INT_MAX) return fail("%lld rows: jb_silhouette takes fewer than 2^31", n);
  if (n_labels < 2 || n_labels > n) return fail("%d labels of %lld rows: 2 <= labels <= rows", n_labels, n);
  if (label_off[0] != 0 || label_off[n_labels] != n)
    return fail("label offsets must run from 0 to %lld rows, got %lld to %lld", n, label_off[0], label_off[n_labels]);
  for (int c = 0; c < n_labels; ++c)
    if (label_off[c + 1] <= label_off[c]) return fail("label %d is empty or its offsets decrease (%lld, %lld)", c, label_off[c], label_off[c + 1]);
  // per chunk of reference rows: its first label and the offset of its slots (one per label it holds)
  const long long nch = (n + jb::SL_CHUNK - 1) / jb::SL_CHUNK;
  std::vector<long long> slot_base(nch + 1, 0);
  std::vector<int> first_label(nch);
  for (long long ch = 0, c = 0; ch < nch; ++ch) {
    const long long r0 = ch * jb::SL_CHUNK, r1 = (r0 + jb::SL_CHUNK < n ? r0 + jb::SL_CHUNK : n) - 1;
    while (label_off[c + 1] <= r0) ++c;
    long long c2 = c;
    while (label_off[c2 + 1] <= r1) ++c2;
    first_label[ch] = static_cast<int>(c);
    slot_base[ch + 1] = slot_base[ch] + (c2 - c + 1);
  }
  const long long P = slot_base[nch];
  CU(cudaSetDevice(device));
  // device bytes: the rows and the label / slot tables (resident), and per query row of a batch its P slots and outputs
  const double res_b = 4.0 * static_cast<double>(n) * L + 8.0 * (n_labels + 1) + 12.0 * static_cast<double>(nch) + 8.0;
  const double row_b = 8.0 * static_cast<double>(P) + 16.0;
  const double avail = knn_avail();
  if (res_b + row_b > avail)
    return fail("silhouette needs %.2f GB of device memory for %lld rows and one query row's workspace; %.2f GB free",
                (res_b + row_b) / 1e9, n, (avail > 0 ? avail : 0) / 1e9);
  const double budget = static_cast<double>(batch_bytes) < avail - res_b ? static_cast<double>(batch_bytes) : avail - res_b;
  long long nqb = static_cast<long long>(budget / row_b);
  if (nqb > n) nqb = n;
  if (nqb > 65535LL * jb::MT_TILE) nqb = 65535LL * jb::MT_TILE;   // query tiles in grid.y
  if (nqb >= jb::MT_TILE) nqb -= nqb % jb::MT_TILE;
  if (nqb < 1) nqb = 1;
  CU(cudaFuncSetAttribute(jb::k_sil_partial, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(jb::SL_SMEM)));

  DevArr<float> dx;
  DevArr<long long> doff, dbase;
  DevArr<int> dfirst;
  DevArr<double> ws, da, db;
  if (dx.alloc(static_cast<size_t>(n) * L) || doff.alloc(n_labels + 1) || dbase.alloc(nch + 1) || dfirst.alloc(nch) ||
      ws.alloc(static_cast<size_t>(nqb) * P) || da.alloc(nqb) || db.alloc(nqb)) return 1;
  KnnStream st;   // declared after the buffers: its destructor synchronises before they are freed
  if (st.create()) return 1;
  CU(cudaMemcpyAsync(dx.p, x, static_cast<size_t>(n) * L * 4, cudaMemcpyHostToDevice, st.s));
  CU(cudaMemcpyAsync(doff.p, label_off, static_cast<size_t>(n_labels + 1) * 8, cudaMemcpyHostToDevice, st.s));
  CU(cudaMemcpyAsync(dbase.p, slot_base.data(), static_cast<size_t>(nch + 1) * 8, cudaMemcpyHostToDevice, st.s));
  CU(cudaMemcpyAsync(dfirst.p, first_label.data(), static_cast<size_t>(nch) * 4, cudaMemcpyHostToDevice, st.s));
  for (long long q0 = 0; q0 < n; q0 += nqb) {
    const long long nb = n - q0 < nqb ? n - q0 : nqb;
    jb::k_sil_partial<<<dim3(static_cast<unsigned>(nch), static_cast<unsigned>((nb + jb::MT_TILE - 1) / jb::MT_TILE)), jb::MT_THREADS,
                        jb::SL_SMEM, st.s>>>(dx.p, n, L, q0, nb, doff.p, dbase.p, dfirst.p, ws.p);
    jb::k_sil_finish<<<static_cast<unsigned>((nb + jb::SF_THREADS - 1) / jb::SF_THREADS), jb::SF_THREADS, 0, st.s>>>(
        ws.p, q0, nb, doff.p, n_labels, dbase.p, dfirst.p, da.p, db.p);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(intra + q0, da.p, static_cast<size_t>(nb) * 8, cudaMemcpyDeviceToHost, st.s));
    CU(cudaMemcpyAsync(inter + q0, db.p, static_cast<size_t>(nb) * 8, cudaMemcpyDeviceToHost, st.s));
  }
  CU(cudaStreamSynchronize(st.s));
  return 0;
}

// ---------------------------------------------------------------------------------------------- F-estimation distances (N2)

int jb_dist_create(long long n, int device, jb_dist** out) {
  if (!out) return fail("null argument");
  *out = nullptr;
  if (n < 1 || n > (1LL << 31) - 1) return fail("bad number of rows %lld", n);
  CU(cudaSetDevice(device));
  size_t free_b = 0, total_b = 0;
  CU(cudaMemGetInfo(&free_b, &total_b));
  const double need = 8.0 * static_cast<double>(n) * static_cast<double>(n);
  if (need > static_cast<double>(free_b))
    return fail("n = %lld rows need %.2f GB for the n x n float64 distance matrix; %.2f GB of device %d are free", n, need / 1e9,
                free_b / 1e9, device);
  jb_dist* h = new jb_dist();
  h->n = n;
  h->device = device;
  cudaError_t ce = cudaStreamCreateWithFlags(&h->s, cudaStreamNonBlocking);
  if (ce == cudaSuccess) ce = cudaMalloc(&h->D, static_cast<size_t>(n) * n * sizeof(double));
  if (ce == cudaSuccess) ce = cudaMalloc(&h->scratch, sizeof(unsigned long long));
  if (ce == cudaSuccess) ce = cudaMemsetAsync(h->D, 0, static_cast<size_t>(n) * n * sizeof(double), h->s);
  if (ce != cudaSuccess) {
    jb_dist_destroy(h);
    return fail("distance handle of %lld rows: %s", n, cudaGetErrorString(ce));
  }
  *out = h;
  return 0;
}

void jb_dist_destroy(jb_dist* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  if (h->s) cudaStreamSynchronize(h->s);
  cudaFree(h->D); cudaFree(h->slab); cudaFree(h->knn_idx); cudaFree(h->knn_dist); cudaFree(h->scratch);
  if (h->s) cudaStreamDestroy(h->s);
  delete h;
}

int jb_dist_accumulate(jb_dist* h, int kind, const double* slab, long long w, long long ld) {
  if (!h || !slab) return fail("null argument");
  if (kind < jb::DIST_SQDIFF || kind > jb::DIST_PRODUCT) return fail("unknown distance kind %d", kind);
  if (w < 1 || w > (1LL << 30) || ld < w) return fail("bad slab shape: %lld columns, row pitch %lld", w, ld);
  CU(cudaSetDevice(h->device));
  const size_t span = static_cast<size_t>(h->n - 1) * ld + w;
  if (span > h->slab_cap) {
    CU(cudaStreamSynchronize(h->s));
    cudaFree(h->slab);
    h->slab = nullptr; h->slab_cap = 0;
    CU(cudaMalloc(&h->slab, span * sizeof(double)));
    h->slab_cap = span;
  }
  // stream-ordered after the previous slab's kernel; from pageable memory it returns once `slab` has been staged
  CU(cudaMemcpyAsync(h->slab, slab, span * sizeof(double), cudaMemcpyHostToDevice, h->s));
  const long long tiles = (h->n + jb::DA_TILE - 1) / jb::DA_TILE;
  const int grid = metric_grid(tiles * (tiles + 1) / 2);
  const int wi = static_cast<int>(w);
  if (kind == jb::DIST_SQDIFF) jb::k_dist_accum<jb::DIST_SQDIFF><<<grid, jb::DA_THREADS, 0, h->s>>>(h->slab, h->n, wi, ld, h->D);
  else if (kind == jb::DIST_ABSDIFF) jb::k_dist_accum<jb::DIST_ABSDIFF><<<grid, jb::DA_THREADS, 0, h->s>>>(h->slab, h->n, wi, ld, h->D);
  else jb::k_dist_accum<jb::DIST_PRODUCT><<<grid, jb::DA_THREADS, 0, h->s>>>(h->slab, h->n, wi, ld, h->D);
  CU(cudaGetLastError());
  return 0;
}

int jb_dist_finish(jb_dist* h, int transform, double* out) {
  if (!h) return fail("null argument");
  if (transform < jb::DIST_NONE || transform > jb::DIST_HALF_ONE_MINUS) return fail("unknown distance transform %d", transform);
  CU(cudaSetDevice(h->device));
  const size_t nn = static_cast<size_t>(h->n) * h->n;
  if (transform != jb::DIST_NONE) {
    jb::k_dist_finish<<<metric_grid(static_cast<long long>((nn + 255) / 256)), 256, 0, h->s>>>(h->D, h->n, transform);
    CU(cudaGetLastError());
  }
  if (out) CU(cudaMemcpyAsync(out, h->D, nn * sizeof(double), cudaMemcpyDeviceToHost, h->s));
  CU(cudaStreamSynchronize(h->s));
  return 0;
}

int jb_dist_knn(jb_dist* h, int k, int* idx, double* dist) {
  if (!h || !idx) return fail("null argument");
  if (k < 1 || k > h->n || k > 16384) return fail("k = %d neighbours of %lld rows (1 .. min(n, 16384))", k, h->n);
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->s));
  cudaFree(h->knn_idx); cudaFree(h->knn_dist);
  h->knn_idx = nullptr; h->knn_dist = nullptr; h->knn_k = 0;
  const size_t nk = static_cast<size_t>(h->n) * k;
  CU(cudaMalloc(&h->knn_idx, nk * sizeof(int)));
  CU(cudaMalloc(&h->knn_dist, nk * sizeof(double)));
  const size_t smem = static_cast<size_t>(k) * (sizeof(unsigned long long) + sizeof(int));
  CU(cudaFuncSetAttribute(jb::k_knn_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  jb::k_knn_rows<<<static_cast<unsigned>(h->n), jb::KN_THREADS, smem, h->s>>>(h->D, h->n, k, h->knn_idx, h->knn_dist);
  CU(cudaGetLastError());
  h->knn_k = k;
  CU(cudaMemcpyAsync(idx, h->knn_idx, nk * sizeof(int), cudaMemcpyDeviceToHost, h->s));
  if (dist) CU(cudaMemcpyAsync(dist, h->knn_dist, nk * sizeof(double), cudaMemcpyDeviceToHost, h->s));
  CU(cudaStreamSynchronize(h->s));
  return 0;
}

int jb_dist_geodesic(jb_dist* h, int k, double* out) {
  if (!h) return fail("null argument");
  if (h->knn_k < 1) return fail("jb_dist_geodesic needs the neighbour lists of jb_dist_knn first");
  if (k < 1 || k > h->knn_k) return fail("k = %d, but the neighbour lists hold %d per row", k, h->knn_k);
  CU(cudaSetDevice(h->device));
  const long long n = h->n;
  const size_t nn = static_cast<size_t>(n) * n;
  const int eg = metric_grid(static_cast<long long>((nn + 255) / 256));
  jb::k_graph_fill<<<eg, 256, 0, h->s>>>(h->D, n);
  jb::k_graph_edges<<<static_cast<unsigned>((n * k + 255) / 256), 256, 0, h->s>>>(h->D, n, h->knn_idx, h->knn_dist, h->knn_k, k);
  const int nb = static_cast<int>((n + jb::FW_B - 1) / jb::FW_B);
  CU(cudaFuncSetAttribute(jb::k_fw_cross, cudaFuncAttributeMaxDynamicSharedMemorySize, jb::FW_CROSS_SMEM));
  for (int kb = 0; kb < nb; ++kb) {
    jb::k_fw_diag<<<1, jb::FW_THREADS, 0, h->s>>>(h->D, n, kb);
    if (nb > 1) {
      jb::k_fw_cross<<<dim3(nb - 1, 2), jb::FW_THREADS, jb::FW_CROSS_SMEM, h->s>>>(h->D, n, kb);
      jb::k_fw_rest<<<dim3(nb, nb), jb::FW_THREADS, 0, h->s>>>(h->D, n, kb);
    }
  }
  CU(cudaMemsetAsync(h->scratch, 0, sizeof(unsigned long long), h->s));
  jb::k_finite_max<<<eg, 256, 0, h->s>>>(h->D, static_cast<long long>(nn), h->scratch);
  jb::k_fill_unreachable<<<eg, 256, 0, h->s>>>(h->D, static_cast<long long>(nn), h->scratch);
  CU(cudaGetLastError());
  if (out) CU(cudaMemcpyAsync(out, h->D, nn * sizeof(double), cudaMemcpyDeviceToHost, h->s));
  CU(cudaStreamSynchronize(h->s));
  return 0;
}

// ---------------------------------------------------------------------------------------------- randomized PCA operand (N3)

namespace {
constexpr long long PO_KCHUNK = 8192;   // dense products: reduction length of one GEMM, accumulated over chunks in float64

int po_check_fits(double need, int device, const char* what) {
  size_t free_b = 0, total_b = 0;
  CU(cudaMemGetInfo(&free_b, &total_b));
  if (need > static_cast<double>(free_b))
    return fail("%s needs %.2f GB of device memory; %.2f GB of device %d are free", what, need / 1e9, free_b / 1e9, device);
  return 0;
}

// CSR consistency: ptr[0] = 0, non-decreasing, ptr[rows] = nnz, every index in [0, cols)
int po_check_csr(const char* name, long long rows, long long cols, long long nnz, const long long* ptr, const int* idx) {
  if (ptr[0] != 0) return fail("%s: indptr[0] = %lld, expected 0", name, ptr[0]);
  if (ptr[rows] != nnz) return fail("%s: indptr[%lld] = %lld, expected nnz = %lld", name, rows, ptr[rows], nnz);
  for (long long r = 0; r < rows; ++r)
    if (ptr[r + 1] < ptr[r]) return fail("%s: indptr decreases at row %lld", name, r);
  for (long long p = 0; p < nnz; ++p)
    if (idx[p] < 0 || idx[p] >= cols) return fail("%s: index %d at position %lld out of range [0, %lld)", name, idx[p], p, cols);
  return 0;
}

// one work item per row, or one per PO_SEG-long segment of a longer row
void po_items(const long long* ptr, long long rows, std::vector<jb::PoItem>& items, std::vector<jb::PoLong>& longs, int& n_part) {
  n_part = 0;
  for (long long r = 0; r < rows; ++r) {
    const long long b = ptr[r], e = ptr[r + 1];
    if (e - b <= jb::PO_SEG) { items.push_back({b, e, static_cast<int>(r), -1}); continue; }
    const int first = n_part;
    for (long long p = b; p < e; p += jb::PO_SEG) items.push_back({p, p + jb::PO_SEG < e ? p + jb::PO_SEG : e, static_cast<int>(r), n_part++});
    longs.push_back({static_cast<int>(r), first, n_part - first});
  }
}

double po_ws_bytes(const jb_pcaop* h, int l) {
  const double M = static_cast<double>(h->n > h->d ? h->n : h->d);
  if (!h->sparse) return M * r4(l) * 4.0 * 3 + M * l * 8.0;
  const int np = h->n_part[0] > h->n_part[1] ? h->n_part[0] : h->n_part[1];
  return static_cast<double>(np) * l * 8.0 + (jb::PO_STAT_SLABS + 1.0) * l * 8.0;
}

void po_free_ws(jb_pcaop* h) {
  cudaFree(h->b_hi); cudaFree(h->b_lo); cudaFree(h->t32); cudaFree(h->acc); cudaFree(h->part); cudaFree(h->vpart); cudaFree(h->vvec);
  h->b_hi = h->b_lo = h->t32 = nullptr; h->acc = h->part = h->vpart = h->vvec = nullptr;
  h->ws_l = 0;
}

int po_ensure_ws(jb_pcaop* h, int l) {
  if (l <= h->ws_l) return 0;
  CU(cudaStreamSynchronize(h->s));   // the old workspaces may still be in use
  po_free_ws(h);
  char what[96];
  snprintf(what, sizeof what, "the workspaces of a width-%d product", l);
  if (po_check_fits(po_ws_bytes(h, l), h->device, what)) return 1;
  const size_t M = static_cast<size_t>(h->n > h->d ? h->n : h->d);
  cudaError_t ce = cudaSuccess;
  if (!h->sparse) {
    const size_t pl = M * r4(l);
    ce = cudaMalloc(&h->b_hi, pl * 4);
    if (ce == cudaSuccess) ce = cudaMalloc(&h->b_lo, pl * 4);
    if (ce == cudaSuccess) ce = cudaMalloc(&h->t32, pl * 4);
    if (ce == cudaSuccess) ce = cudaMalloc(&h->acc, M * l * 8);
  } else {
    const int np = h->n_part[0] > h->n_part[1] ? h->n_part[0] : h->n_part[1];
    ce = cudaMalloc(&h->part, static_cast<size_t>(np > 0 ? np : 1) * l * 8);
    if (ce == cudaSuccess) ce = cudaMalloc(&h->vpart, static_cast<size_t>(jb::PO_STAT_SLABS) * l * 8);
    if (ce == cudaSuccess) ce = cudaMalloc(&h->vvec, static_cast<size_t>(l) * 8);
  }
  if (ce != cudaSuccess) {
    po_free_ws(h);
    return fail("workspaces of a width-%d product: %s", l, cudaGetErrorString(ce));
  }
  h->ws_l = l;
  return 0;
}

// hi/lo planes of X - mu (fp32 mean subtracted during the split), on the handle's stream
int po_split_dense(jb_pcaop* h) {
  jb::k_f64_to_f32<<<static_cast<unsigned>((h->d + 255) / 256), 256, 0, h->s>>>(h->mu, h->d, h->mu32);
  jb::k_split_tf32<<<static_cast<unsigned>(h->n), 256, 0, h->s>>>(h->X, h->d, h->n, static_cast<int>(h->d), 0, h->mu32, 1.f, 0.f,
                                                                  h->x_hi, h->x_lo, h->ldd);
  CU(cudaGetLastError());
  return 0;
}

jb_pcaop* po_new(long long n, long long d, int device, int sparse) {
  jb_pcaop* h = new jb_pcaop();
  h->n = n; h->d = d; h->device = device; h->sparse = sparse;
  return h;
}

// stream, events, mu / var: common to both operand kinds
cudaError_t po_common_alloc(jb_pcaop* h) {
  cudaError_t ce = cudaStreamCreateWithFlags(&h->s, cudaStreamNonBlocking);
  if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&h->ev_in, cudaEventDisableTiming);
  if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&h->ev_out, cudaEventDisableTiming);
  if (ce == cudaSuccess) ce = cudaMalloc(&h->mu, static_cast<size_t>(h->d) * 8);
  if (ce == cudaSuccess) ce = cudaMalloc(&h->var, static_cast<size_t>(h->d) * 8);
  if (ce == cudaSuccess) ce = cudaMemsetAsync(h->mu, 0, static_cast<size_t>(h->d) * 8, h->s);
  return ce;
}
}  // namespace

int jb_pcaop_create_dense(const float* X, long long n, long long d, int device, jb_pcaop** out) {
  if (!X || !out) return fail("null argument");
  *out = nullptr;
  if (n < 1 || d < 1 || n > (1LL << 31) - 1 || d > (1LL << 31) - 32) return fail("bad operand shape %lld x %lld", n, d);
  CU(cudaSetDevice(device));
  const long long ldd = r4(static_cast<int>(d));
  const long long chunks = ((n > d ? n : d) + PO_KCHUNK - 1) / PO_KCHUNK;
  const double need = 4.0 * n * d + 8.0 * n * ldd + 20.0 * d + 8.0 * jb::PO_STAT_SLABS * d +
                      static_cast<double>(chunks) * sizeof(jb::GemmProblem);
  char what[96];
  snprintf(what, sizeof what, "a dense %lld x %lld PCA operand", n, d);
  if (po_check_fits(need, device, what)) return 1;
  jb_pcaop* h = po_new(n, d, device, 0);
  h->ldd = ldd;
  h->n_probs = static_cast<int>(chunks);
  cudaError_t ce = po_common_alloc(h);
  if (ce == cudaSuccess) ce = cudaMalloc(&h->X, static_cast<size_t>(n) * d * 4);
  if (ce == cudaSuccess) ce = cudaMalloc(&h->x_hi, static_cast<size_t>(n) * ldd * 4);
  if (ce == cudaSuccess) ce = cudaMalloc(&h->x_lo, static_cast<size_t>(n) * ldd * 4);
  if (ce == cudaSuccess) ce = cudaMalloc(&h->mu32, static_cast<size_t>(d) * 4);
  if (ce == cudaSuccess) ce = cudaMalloc(&h->stat_part, static_cast<size_t>(jb::PO_STAT_SLABS) * d * 8);
  if (ce == cudaSuccess) ce = cudaMalloc(&h->probs, static_cast<size_t>(chunks) * sizeof(jb::GemmProblem));
  if (ce == cudaSuccess) ce = cudaMemcpyAsync(h->X, X, static_cast<size_t>(n) * d * 4, cudaMemcpyHostToDevice, h->s);
  if (ce != cudaSuccess) {
    jb_pcaop_destroy(h);
    return fail("dense PCA operand of %lld x %lld: %s", n, d, cudaGetErrorString(ce));
  }
  if (po_split_dense(h)) { jb_pcaop_destroy(h); return 1; }
  ce = cudaStreamSynchronize(h->s);
  if (ce != cudaSuccess) {
    jb_pcaop_destroy(h);
    return fail("dense PCA operand of %lld x %lld: %s", n, d, cudaGetErrorString(ce));
  }
  *out = h;
  return 0;
}

int jb_pcaop_create_sparse(long long n, long long d, long long nnz, const long long* row_ptr, const int* col_idx,
                           const float* row_val, const long long* col_ptr, const int* row_idx, const float* col_val,
                           int device, jb_pcaop** out) {
  if (!out || !row_ptr || !col_ptr || (nnz > 0 && (!col_idx || !row_val || !row_idx || !col_val))) return fail("null argument");
  *out = nullptr;
  if (n < 1 || d < 1 || n > (1LL << 31) - 1 || d > (1LL << 31) - 1 || nnz < 0) return fail("bad operand shape %lld x %lld, %lld nonzeros", n, d, nnz);
  if (po_check_csr("CSR of X", n, d, nnz, row_ptr, col_idx) || po_check_csr("CSR of X^T", d, n, nnz, col_ptr, row_idx)) return 1;
  std::vector<jb::PoItem> items[2];
  std::vector<jb::PoLong> longs[2];
  int n_part[2];
  po_items(row_ptr, n, items[0], longs[0], n_part[0]);
  po_items(col_ptr, d, items[1], longs[1], n_part[1]);
  CU(cudaSetDevice(device));
  const double need = 8.0 * (n + 1) + 8.0 * (d + 1) + 16.0 * nnz + 16.0 * d +
                      sizeof(jb::PoItem) * static_cast<double>(items[0].size() + items[1].size()) +
                      sizeof(jb::PoLong) * static_cast<double>(longs[0].size() + longs[1].size());
  char what[128];
  snprintf(what, sizeof what, "a sparse %lld x %lld PCA operand with %lld nonzeros", n, d, nnz);
  if (po_check_fits(need, device, what)) return 1;
  jb_pcaop* h = po_new(n, d, device, 1);
  h->nnz = nnz;
  cudaError_t ce = po_common_alloc(h);
  auto up = [&](auto** dst, const auto* src, size_t count) {
    if (ce != cudaSuccess) return;
    ce = cudaMalloc(dst, (count ? count : 1) * sizeof(**dst));
    if (ce == cudaSuccess && count) ce = cudaMemcpyAsync(*dst, src, count * sizeof(**dst), cudaMemcpyHostToDevice, h->s);
  };
  up(&h->rp, row_ptr, static_cast<size_t>(n) + 1);
  up(&h->ci, col_idx, static_cast<size_t>(nnz));
  up(&h->rv, row_val, static_cast<size_t>(nnz));
  up(&h->cp, col_ptr, static_cast<size_t>(d) + 1);
  up(&h->ri, row_idx, static_cast<size_t>(nnz));
  up(&h->cv, col_val, static_cast<size_t>(nnz));
  for (int t = 0; t < 2; ++t) {
    h->n_items[t] = static_cast<long long>(items[t].size());
    h->n_long[t] = static_cast<int>(longs[t].size());
    h->n_part[t] = n_part[t];
    up(&h->items[t], items[t].data(), items[t].size());
    up(&h->longs[t], longs[t].data(), longs[t].size());
  }
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(h->s);   // the host vectors above go out of scope
  if (ce != cudaSuccess) {
    jb_pcaop_destroy(h);
    return fail("sparse PCA operand of %lld x %lld: %s", n, d, cudaGetErrorString(ce));
  }
  *out = h;
  return 0;
}

int jb_pcaop_stats(jb_pcaop* h, double* mean, double* var) {
  if (!h) return fail("null argument");
  CU(cudaSetDevice(h->device));
  const long long n = h->n, d = h->d;
  if (h->sparse) {
    jb::k_csc_stats<<<static_cast<unsigned>((d * 32 + 255) / 256), 256, 0, h->s>>>(h->cp, h->cv, d, n, h->mu, h->var);
  } else {
    const long long per = (n + jb::PO_STAT_SLABS - 1) / jb::PO_STAT_SLABS;
    const dim3 g(static_cast<unsigned>((d + 127) / 128), jb::PO_STAT_SLABS);
    const unsigned gs = static_cast<unsigned>((d + 255) / 256);
    jb::k_col_sums<<<g, 128, 0, h->s>>>(h->X, n, d, per, h->stat_part);
    jb::k_sum_parts<<<gs, 256, 0, h->s>>>(h->stat_part, jb::PO_STAT_SLABS, d, static_cast<double>(n), h->mu);
    jb::k_col_sqdev<<<g, 128, 0, h->s>>>(h->X, n, d, per, h->mu, h->stat_part);
    jb::k_sum_parts<<<gs, 256, 0, h->s>>>(h->stat_part, jb::PO_STAT_SLABS, d, static_cast<double>(n), h->var);
    if (po_split_dense(h)) return 1;
  }
  CU(cudaGetLastError());
  if (mean) CU(cudaMemcpyAsync(mean, h->mu, static_cast<size_t>(d) * 8, cudaMemcpyDeviceToHost, h->s));
  if (var) CU(cudaMemcpyAsync(var, h->var, static_cast<size_t>(d) * 8, cudaMemcpyDeviceToHost, h->s));
  CU(cudaStreamSynchronize(h->s));
  return 0;
}

int jb_pcaop_apply(jb_pcaop* h, int trans, const float* B, int l, float* Y, void* stream) {
  if (!h || !B || !Y) return fail("null argument");
  if (trans != 0 && trans != 1) return fail("trans must be 0 or 1, not %d", trans);
  if (l < 1 || l > 65536) return fail("bad product width %d (1 .. 65536)", l);
  CU(cudaSetDevice(h->device));
  if (po_ensure_ws(h, l)) return 1;
  cudaStream_t cs = static_cast<cudaStream_t>(stream);
  CU(cudaEventRecord(h->ev_in, cs));
  CU(cudaStreamWaitEvent(h->s, h->ev_in, 0));
  const long long K = trans ? h->n : h->d, M = trans ? h->d : h->n;   // B [K, l], Y [M, l]
  if (h->sparse) {
    // the l-vector of the rank-1 correction: mu^T B (trans 0, a = 1) or 1^T B (trans 1, a = mu), in a fixed order
    const long long per = (K + jb::PO_STAT_SLABS - 1) / jb::PO_STAT_SLABS;
    jb::k_wcolsum<<<dim3(static_cast<unsigned>((l + 127) / 128), jb::PO_STAT_SLABS), 128, 0, h->s>>>(B, K, l, per, trans ? nullptr : h->mu, h->vpart);
    jb::k_sum_parts<<<static_cast<unsigned>((l + 255) / 256), 256, 0, h->s>>>(h->vpart, jb::PO_STAT_SLABS, l, 1.0, h->vvec);
    const double* a = trans ? h->mu : nullptr;
    const int* idx = trans ? h->ri : h->ci;
    const float* val = trans ? h->cv : h->rv;
    const dim3 g(static_cast<unsigned>((h->n_items[trans] + jb::PO_WARPS - 1) / jb::PO_WARPS), static_cast<unsigned>((l + jb::PO_SLAB - 1) / jb::PO_SLAB));
    jb::k_csr_dense<<<g, jb::PO_WARPS * 32, 0, h->s>>>(h->items[trans], h->n_items[trans], idx, val, B, l, a, h->vvec, Y, h->part);
    if (h->n_long[trans]) {
      const long long t = static_cast<long long>(h->n_long[trans]) * l;
      jb::k_seg_finish<<<static_cast<unsigned>((t + 255) / 256), 256, 0, h->s>>>(h->longs[trans], h->n_long[trans], h->part, l, a, h->vvec, Y);
    }
  } else {
    // Y = Xc B (trans 0: A = the [n, d] planes, K-major) or Xc^T B (trans 1: the same planes read MN-major); B [K, l] is
    // MN-major. One 3xTF32 GEMM per PO_KCHUNK slice of K, each added to a float64 accumulator, then one rounding to fp32.
    const int ldl = r4(l);
    jb::k_split_tf32<<<static_cast<unsigned>(K), 256, 0, h->s>>>(B, l, K, l, 2, nullptr, 1.f, 0.f, h->b_hi, h->b_lo, ldl);
    CU(cudaMemsetAsync(h->acc, 0, static_cast<size_t>(M) * l * 8, h->s));
    const int chunks = static_cast<int>((K + PO_KCHUNK - 1) / PO_KCHUNK);
    const int bn = l <= 32 ? 32 : 64;
    h->host_probs.assign(static_cast<size_t>(chunks), jb::GemmProblem{});
    for (int c = 0; c < chunks; ++c) {
      const long long k0 = c * PO_KCHUNK, kc = K - k0 < PO_KCHUNK ? K - k0 : PO_KCHUNK;
      const long long a_off = trans ? k0 * h->ldd : k0;
      jb::GemmProblem& g = h->host_probs[static_cast<size_t>(c)];
      int rc = jb::gemm_problem_fill(&g, h->x_hi + a_off, static_cast<int>(h->ldd), trans, h->b_hi + k0 * ldl, ldl, 1, h->t32, ldl,
                                     static_cast<int>(M), l, static_cast<int>(kc), bn, jb::EPI_STORE, nullptr, 0.f, 0, 0,
                                     h->x_lo + a_off, h->b_lo + k0 * ldl);
      if (rc) return fail("PCA operand tensor map encode failed (%d)", rc);
      jb::gemm_table_finalize(&g, 1);
    }
    CU(cudaMemcpyAsync(h->probs, h->host_probs.data(), static_cast<size_t>(chunks) * sizeof(jb::GemmProblem), cudaMemcpyHostToDevice, h->s));
    for (int c = 0; c < chunks; ++c) {
      const jb::GemmProblem& g = h->host_probs[static_cast<size_t>(c)];
      CU(jb::gemm_launch(h->probs + c, 1, g.tiles_m * g.tiles_n, h->s));
      jb::k_acc_f64<<<static_cast<unsigned>(M), 256, 0, h->s>>>(h->t32, ldl, h->acc, l);
    }
    jb::k_f64_to_f32<<<static_cast<unsigned>((M * l + 255) / 256), 256, 0, h->s>>>(h->acc, M * l, Y);
  }
  CU(cudaGetLastError());
  CU(cudaEventRecord(h->ev_out, h->s));
  CU(cudaStreamWaitEvent(cs, h->ev_out, 0));
  return 0;
}

void jb_pcaop_destroy(jb_pcaop* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  if (h->s) cudaStreamSynchronize(h->s);
  po_free_ws(h);
  cudaFree(h->mu); cudaFree(h->var); cudaFree(h->X); cudaFree(h->mu32); cudaFree(h->x_hi); cudaFree(h->x_lo);
  cudaFree(h->stat_part); cudaFree(h->probs);
  cudaFree(h->rp); cudaFree(h->ci); cudaFree(h->rv); cudaFree(h->cp); cudaFree(h->ri); cudaFree(h->cv);
  for (int t = 0; t < 2; ++t) { cudaFree(h->items[t]); cudaFree(h->longs[t]); }
  if (h->ev_in) cudaEventDestroy(h->ev_in);
  if (h->ev_out) cudaEventDestroy(h->ev_out);
  if (h->s) cudaStreamDestroy(h->s);
  delete h;
}

long long jb_debug_read(jb_engine* e, const char* name, float* out, long long cap) {
  if (!e || !name || !out) { fail("null argument"); return -1; }
  cudaDeviceSynchronize();
  const int B = e->step_B ? e->step_B : e->plan_B;
  // a tap is an fp32 array (optionally the sum of split-K partials) or a pair of fp16 operand planes (hi + lo / 2^11);
  // backward taps carry the loss scale, which is divided out here
  // (parts that the consuming phase reduces in place hold the sum in partial 0: read with parts = 1)
  struct Tap { const char* n; const float* p; const __half* hi; const __half* lo; long long rows, cols, ld; int parts; long long pstride; float scale; };
  std::vector<Tap> taps;
  char nm[2][24][16];
  const float ig = 1.f / e->gs;
  for (int i = 0; i < 2; ++i) {
    ModActs& a = e->act[i];
    const int D = e->D[i], L = e->L;
    int k = 0;
    auto f32 = [&](const char* base, const float* p, int cols, int ld, float scale = 1.f) {
      snprintf(nm[i][k], sizeof nm[i][k], "%s%d", base, i);
      taps.push_back({nm[i][k], p, nullptr, nullptr, B, cols, ld, 1, 0, scale}); ++k;
    };
    auto prt = [&](const char* base, const jb::Parts& q, int cols, int ld, float scale = 1.f, bool reduced = true) {
      snprintf(nm[i][k], sizeof nm[i][k], "%s%d", base, i);
      taps.push_back({nm[i][k], q.ptr, nullptr, nullptr, B, cols, ld, reduced ? 1 : q.n, q.stride, scale}); ++k;
    };
    auto pl = [&](const char* base, const HPlanes& h, int cols, int ld, float scale = 1.f) {
      snprintf(nm[i][k], sizeof nm[i][k], "%s%d", base, i);
      taps.push_back({nm[i][k], nullptr, h.hi, h.lo, B, cols, ld, 1, 0, scale}); ++k;
    };
    f32("x", a.x, D, a.ldD); prt("y1_", a.y1, 2 * D, a.ld2D); pl("h1_", a.h1, 2 * D, a.ld2D); prt("y2_", a.y2, D, a.ldD);
    pl("h2_", a.h2, D, a.ldD); prt("mulv", a.mulv, 2 * L, e->ldmv); f32("z", a.z, L, e->LP); f32("c", a.c, L, e->LP);
    f32("eps", a.eps, L, e->LP); pl("g1_", a.g1, D, a.ldD); pl("g2_", a.g2, 2 * D, a.ld2D); prt("xhat", a.xhat, D, a.ldD);
    pl("dxhat", a.dxhat, D, a.ldD, ig); prt("dg2_", a.dg2, 2 * D, a.ld2D, ig, false); pl("dy4_", a.dy4, 2 * D, a.ld2D, ig);
    prt("dg1_", a.dg1, D, a.ldD, ig, false); pl("dy3_", a.dy3, D, a.ldD, ig); prt("dc", a.dc, L, e->LP, ig);
    f32("dmulv", a.dmulv, 2 * L, e->ldmv, ig); prt("dh2_", a.dh2, D, a.ldD, ig, false); pl("dy2_", a.dy2, D, a.ldD, ig);
    prt("dh1_", a.dh1, 2 * D, a.ld2D, ig, false); pl("dy1_", a.dy1, 2 * D, a.ld2D, ig); f32("S", a.S, L, e->LP);
  }
  taps.push_back({"corr", e->corr, nullptr, nullptr, B, B, B, 1, 0, 1.f});
  taps.push_back({"fblk", e->fblk, nullptr, nullptr, B, B, B, 1, 0, 1.f});
  taps.push_back({"grad", e->grad, nullptr, nullptr, 1, e->n_flat, e->n_flat, 1, 0, 1.f});
  taps.push_back({"theta", e->theta, nullptr, nullptr, 1, e->n_flat, e->n_flat, 1, 0, 1.f});
  for (const Tap& t : taps) {
    if (strcmp(t.n, name) != 0) continue;
    const long long need = t.rows * t.cols;
    if (need > cap) { fail("buffer too small: need %lld floats", need); return -1; }
    if (t.p) {
      if (!e->step_B && t.parts > 0 && t.p == nullptr) { fail("no step has run yet"); return -1; }
      std::vector<float> tmp(static_cast<size_t>(need));
      for (long long q = 0; q < need; ++q) out[q] = 0.f;
      for (int p = 0; p < t.parts; ++p) {
        cudaError_t ce = cudaMemcpy2D(tmp.data(), static_cast<size_t>(t.cols) * 4, t.p + p * t.pstride, static_cast<size_t>(t.ld) * 4,
                                      static_cast<size_t>(t.cols) * 4, t.rows, cudaMemcpyDeviceToHost);
        if (ce != cudaSuccess) { fail("debug read failed: %s", cudaGetErrorString(ce)); return -1; }
        for (long long q = 0; q < need; ++q) out[q] += tmp[static_cast<size_t>(q)];
      }
    } else {
      std::vector<__half> hi(static_cast<size_t>(need)), lo(static_cast<size_t>(need));
      cudaError_t ce = cudaMemcpy2D(hi.data(), static_cast<size_t>(t.cols) * 2, t.hi, static_cast<size_t>(t.ld) * 2,
                                    static_cast<size_t>(t.cols) * 2, t.rows, cudaMemcpyDeviceToHost);
      if (ce == cudaSuccess)
        ce = cudaMemcpy2D(lo.data(), static_cast<size_t>(t.cols) * 2, t.lo, static_cast<size_t>(t.ld) * 2,
                          static_cast<size_t>(t.cols) * 2, t.rows, cudaMemcpyDeviceToHost);
      if (ce != cudaSuccess) { fail("debug read failed: %s", cudaGetErrorString(ce)); return -1; }
      for (long long q = 0; q < need; ++q) out[q] = __half2float(hi[static_cast<size_t>(q)]) + __half2float(lo[static_cast<size_t>(q)]) * jb::HG_LO_INV;
    }
    if (t.scale != 1.f) for (long long q = 0; q < need; ++q) out[q] *= t.scale;
    return need;
  }
  fail("unknown tap '%s'", name);
  return -1;
}

long long jb_launch_count(const jb_engine* e) { return e ? e->launches : 0; }

}  // extern "C"
