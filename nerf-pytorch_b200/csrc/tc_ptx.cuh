// tc_ptx.cuh -- thin inline-PTX wrappers for sm_100a: mbarrier, bulk async copy (TMA engine,
// SASS UBLKCP), tcgen05 (alloc / mma / commit / ld / fences) and UMMA descriptors.
#pragma once
#include <stdint.h>
#include <cuda_runtime.h>

namespace nb {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier --------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
               : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) { }
}

// ---- proxy fences ----------------------------------------------------------------------------
// generic-proxy st.shared  ->  async-proxy (tcgen05.mma / bulk copy) readers
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- bulk async copy global -> shared (TMA engine, completes on an mbarrier) -------------------
__device__ __forceinline__ void bulk_g2s(uint32_t dst_smem, const void* src_gmem, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst_smem), "l"(src_gmem), "r"(bytes), "r"(bar) : "memory");
}

// ---- bulk async copy shared -> global (TMA engine, bulk-group completion; per-thread groups) ------
__device__ __forceinline__ void bulk_s2g(void* dst_gmem, uint32_t src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(src_smem), "r"(bytes) : "memory");
}
// the same with an L2 eviction-priority hint (createpolicy): streaming records are written / read once
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void bulk_s2g_hint(void* dst_gmem, uint32_t src_smem, uint32_t bytes, uint64_t policy) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(dst_gmem), "r"(src_smem), "r"(bytes), "l"(policy) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all of this thread's committed groups have finished READING shared memory (the source may be overwritten)
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ---- tcgen05: TMEM allocation ------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem_addr, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem_addr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() { asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---- tcgen05.mma (kind::f16, A and B from shared memory descriptors, D in TMEM) -----------------
__device__ __forceinline__ void mma_f16_ss(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// completion of all previously issued tcgen05 ops of this thread -> one arrive on an mbarrier
__device__ __forceinline__ void mma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// ---- tcgen05.ld: 32 lanes x 32 columns of 32-bit (thread t of warp w reads TMEM lane 32*(w%4)+t) -
__device__ __forceinline__ void tmem_ld_x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- UMMA descriptors (cute/arch/mma_sm100_desc.hpp bit layout) ---------------------------------
// shared-memory matrix descriptor, K-major canonical layouts:
//   SWIZZLE_128B: rows of 128 B (64 fp16), 8-row atoms of 1024 B, SBO = 1024, layout_type = 2
//   SWIZZLE_64B : rows of  64 B (32 fp16), 8-row atoms of  512 B, SBO =  512, layout_type = 4
constexpr uint64_t UMMA_SW128 = 2, UMMA_SW64 = 4, UMMA_SW32 = 6;
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr, uint32_t sbo_bytes, uint64_t layout_type) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);        // start address  [0,14)
  d |= (uint64_t)1 << 16;                              // LBO (unused for swizzled K-major) [16,30)
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;    // SBO            [32,46)
  d |= (uint64_t)1 << 46;                              // descriptor version = 1 (Blackwell) [46,48)
  d |= layout_type << 61;                              // layout type    [61,64)
  return d;
}
// full form: explicit leading-dimension byte offset (MN-major operands use both strides)
__device__ __forceinline__ uint64_t umma_desc_full(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint64_t layout_type) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= layout_type << 61;
  return d;
}
// instruction descriptor: D=f32, A=B=f16, both K-major, M x N
__host__ __device__ constexpr uint32_t umma_idesc_f16(int M, int N) {
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// same with MN-major A and/or B (bits 15 / 16): the operand's contiguous dimension is M (N), not K
__host__ __device__ constexpr uint32_t umma_idesc_f16_major(int M, int N, int a_mn, int b_mn) {
  return umma_idesc_f16(M, N) | ((uint32_t)(a_mn & 1) << 15) | ((uint32_t)(b_mn & 1) << 16);
}

// one elected lane of a fully converged warp (the surrounding control flow stays warp-uniform, so the
// compiler keeps descriptors / addresses in uniform registers instead of a per-lane waterfall loop)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.b32 %0, 1, 0, P;\n\t}" : "=r"(pred));
  return pred != 0;
}

// ---- thread-block clusters / CTA pairs (cta_group::2) ---------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cta address of this CTA -> shared::cluster address of the same offset in CTA `rank`
__device__ __forceinline__ uint32_t mapa(uint32_t addr, uint32_t rank) {
  uint32_t r; asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank)); return r;
}
// remote arrive with the default semantics (.release at .cta scope), as CUTLASS' ClusterBarrier::arrive(cta_id) does.
// The .release.cluster form below costs ~1.5 k cycles per arrive on B200 (measured in the pair kernel: the peer's
// epilogue warps reached the arrive together with the leader's, their arrivals landed 1.3-1.8 k cycles later).
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// 2D tensor-map TMA load into this CTA's shared memory whose completion bytes are counted on the LEADER CTA's
// mbarrier (cta_group::2: the peer bit of the mbarrier address is cleared, as in CUTLASS' SM100_TMA_2SM_LOAD)
__device__ __forceinline__ void tma2_load_2d(uint32_t dst_smem, const void* tmap, int c0, int c1, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
               ::"r"(dst_smem), "l"(tmap), "r"(c0), "r"(c1), "r"(bar & 0xFEFFFFFFu) : "memory");
}
// relaxed remote arrive: pure signal (the waiter's data dependency is carried by the control dependency on the
// local wait that precedes it; no data written by this thread is published)
__device__ __forceinline__ void mbar_arrive_cluster_relaxed(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait_cluster(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
               : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) { while (!mbar_try_wait_cluster(bar, parity)) { } }
__device__ __forceinline__ void tmem_alloc2(uint32_t dst_smem_addr, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem_addr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish2() { asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// pair MMA: M = 256 rows (128 per CTA, each CTA's own A tile and accumulator), B split across the pair (N/2 rows each)
__device__ __forceinline__ void mma2_f16_ss(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// completion of prior pair MMAs -> one arrive on the barrier at this offset in every CTA of `mask`
__device__ __forceinline__ void mma2_commit_mc(uint32_t bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"(mask) : "memory");
}

// ---- packing helpers ----------------------------------------------------------------------------
// {lo = a, hi = b} as fp16 pair with ReLU fused into the conversion
__device__ __forceinline__ uint32_t cvt_relu_f16x2(float a, float b) {
  uint32_t r;
  asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
__device__ __forceinline__ uint32_t cvt_f16x2(float a, float b) {
  uint32_t r;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
// saturating variant (+-65504 instead of inf): loss-scaled gradients of the fp16 backward
__device__ __forceinline__ uint32_t cvt_sat_f16x2(float a, float b) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

}  // namespace ptx
}  // namespace nb
