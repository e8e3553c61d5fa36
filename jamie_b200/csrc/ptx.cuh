// Thin inline-PTX wrappers for the sm_100a features the kernels use:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld), tf32 rounding.
// Everything here is device-only and header-only.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace jb {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }
__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// One lane of a converged warp. Keeping the surrounding control flow warp-uniform (whole warp runs the loop, only the
// issuing instruction is predicated) lets the compiler keep descriptors in uniform registers.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---------------------------------------------------------------- programmatic dependent launch
// wait: blocks until every prerequisite grid has completed and its memory is visible (a no-op when the kernel was
// launched without the programmatic-serialization attribute). launch: lets the dependent grid start its prologue.
__device__ __forceinline__ void grid_dep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void grid_dep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---------------------------------------------------------------- thread-block clusters
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_nctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
  return r;
}
// All threads of all CTAs of the cluster (release / acquire: also orders mbarrier initialisation before remote use).
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// Address of the same shared-memory location in CTA `rank` of the cluster (distributed shared memory window).
__device__ __forceinline__ uint32_t mapa_shared(uint32_t local_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ float4 ld_shared_cluster_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void st_shared_cluster_f4(uint32_t addr, float a, float b, float c, float d) {
  asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded spin: a protocol bug traps (launch error) instead of hanging the GPU box.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 26)) __trap();
  }
}

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
// 2-D tiled load global -> shared, completion signalled on an mbarrier (complete_tx::bytes).
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const void* tmap, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// 2-D tiled store shared -> global (bulk_group completion).
__device__ __forceinline__ void tma_store_2d(const void* tmap, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(tmap)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// the issued bulk stores have finished READING their shared-memory source (it may be overwritten)
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// generic-proxy writes (st.global / st.shared of any thread, once visible to this thread) -> visible to the async proxy
// (TMA loads issued afterwards by this thread), all state spaces
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }

// ---------------------------------------------------------------- 1-D bulk copies (TMA without a tensor map)
// global -> shared, completion on an mbarrier (complete_tx::bytes); 16-byte aligned addresses, size a multiple of 16
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
               "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// shared -> global, bulk-group completion
__device__ __forceinline__ void bulk_store(void* gdst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(reinterpret_cast<uint64_t>(gdst)), "r"(smem_u32(smem_src)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_wait_read_1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }

// ---------------------------------------------------------------- L2 prefetch
// TMA prefetch of one tensor-map box into L2 (no shared-memory destination, no barrier)
__device__ __forceinline__ void tma_prefetch_2d(const void* tmap, int c0, int c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];" ::"l"(reinterpret_cast<uint64_t>(tmap)), "r"(c0), "r"(c1) : "memory");
}

// ---------------------------------------------------------------- grid-wide barrier (persistent kernels, all CTAs co-resident)
// One monotonically increasing counter in global memory (never reset inside a launch; the host zeroes it before the
// launch): every CTA adds 1 per barrier and waits until the count reaches `target` = barriers so far * CTAs.
// Release / acquire at gpu scope; the bracketing __syncthreads make the whole CTA's writes part of the release and the
// whole CTA a reader of the acquire. The proxy fences order generic global writes before later TMA (async proxy) reads.
// A protocol bug traps (launch error) instead of hanging the box.
__device__ __forceinline__ void fence_proxy_async_global() { asm volatile("fence.proxy.async.global;" ::: "memory"); }
__device__ __forceinline__ void grid_barrier(unsigned int* counter, unsigned int target) {
  fence_proxy_async_global();   // this thread's generic global writes -> async proxy (a later TMA load of any CTA)
  __syncthreads();
  if (threadIdx.x == 0) {
    // release: cumulative over the CTA's writes ordered before it by the bar.sync above
    asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(counter) : "memory");
    unsigned int v, spins = 0;
    do {
      asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
      if (++spins > (1u << 24)) __trap();
    } while (static_cast<int>(v - target) < 0);
    asm volatile("fence.acq_rel.gpu;" ::: "memory");   // acquire (also invalidates this SM's L1)
  }
  __syncthreads();
}
// the first version measured on B200: 1.66 us per barrier (tools/hgemm_lab bar); kept for A/B
__device__ __forceinline__ void grid_barrier_v0(unsigned int* counter, unsigned int target) {
  fence_proxy_async_all();
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(counter) : "memory");
    unsigned int v, spins = 0;
    do {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
      if (++spins > (1u << 24)) __trap();
    } while (static_cast<int>(v - target) < 0);
    __threadfence();
  }
  __syncthreads();
  fence_proxy_async_all();
}

// ---------------------------------------------------------------- tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {  // whole warp
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc], kind::tf32, issued by ONE thread.
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier when all previously issued MMAs of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// TMEM -> registers: thread t of warp w reads lane (32*(w%4)+t), 32 consecutive fp32 columns.
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, float (&v)[32]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------- numerics
// Round-to-nearest (ties away) to TF32, result kept in an fp32 container: the tensor core only
// reads the top 19 bits, so un-rounded operands would be truncated (biased).
__device__ __forceinline__ float tf32_rna(float x) {
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
  return __uint_as_float(u);
}
// x = hi + lo + r with hi, lo TF32-representable and |r| <= 2^-23 |x|: the operand planes of the 3xTF32 GEMMs.
__device__ __forceinline__ void tf32_split(float x, float& hi, float& lo) {
  hi = tf32_rna(x);
  lo = tf32_rna(x - hi);
}

// ---------------------------------------------------------------- UMMA descriptors
// Shared-memory matrix descriptor (sm_100 "version 1").
//   bits [0,14)  start address >> 4       bits [16,30) leading byte offset >> 4
//   bits [32,46) stride byte offset >> 4  bits [46,48) version = 1   bits [61,64) layout type
//   K-major operands use SWIZZLE_128B (layout 2); MN-major tf32 operands must use SWIZZLE_128B_BASE32B
//   (layout 1: 32-byte swizzle atoms, 4 K-rows of 128 B per atom) -- the only MN-major layout the tensor core
//   accepts for 32-bit elements.
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                                   uint32_t layout_type) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr >> 4) & 0x3FFFu);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(layout_type & 7u) << 61;
  return d;
}
// Instruction descriptor, kind::tf32, fp32 accumulate, M = 128.
//   c_format [4,6)=1 (F32); a_format [7,10)=2, b_format [10,13)=2 (TF32); a_major bit 15, b_major bit 16
//   (0 = K-major, 1 = MN-major); n_dim [17,23) = N>>3; m_dim [24,29) = M>>4.
__host__ __device__ __forceinline__ uint32_t umma_idesc_tf32(int m, int n, int a_mn, int b_mn) {
  uint32_t d = 0;
  d |= 1u << 4;
  d |= 2u << 7;
  d |= 2u << 10;
  d |= static_cast<uint32_t>(a_mn & 1) << 15;
  d |= static_cast<uint32_t>(b_mn & 1) << 16;
  d |= static_cast<uint32_t>(n >> 3) << 17;
  d |= static_cast<uint32_t>(m >> 4) << 24;
  return d;
}

}  // namespace jb
