// tc_ptx.cuh -- raw-PTX device helpers shared by the tcgen05 kernels (mbarrier, TMA, UMMA
// descriptors, tcgen05.mma / commit / ld / alloc) and the split-FP16 operand encoding.  sm_100a only.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include "kernels.h"

namespace kkx {

// fp16 hi = rn(v), lo = rn(v - hi) of an already scaled v, as raw 16-bit patterns.  Every split-FP16 plane (activation
// operands, weights, attention Q / K / V^T) is encoded here, so a value gives the same planes whichever kernel wrote them.
__host__ __device__ __forceinline__ void split_f16(float v, uint32_t& hi, uint32_t& lo) {
  const __half h = __float2half_rn(v);
  hi = __half_as_ushort(h);
  lo = __half_as_ushort(__float2half_rn(v - __half2float(h)));
}
// GEMM activation operand: kSplitF16Scale * v, saturated at the fp16 range, then split (the GEMM epilogue divides by
// kSplitF16Scale again through its wscale)
__device__ __forceinline__ void split_f16_operand(float v, uint32_t& hi, uint32_t& lo) {
  split_f16(fminf(fmaxf(v * kSplitF16Scale, -65504.f), 65504.f), hi, lo);
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void prefetch_tmap(const void* p) { asm volatile("prefetch.tensormap [%0];" ::"l"(p) : "memory"); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
// after the barrier inits of a CTA: make them visible to the async proxy (TMA, tcgen05.commit) and to the cluster
__device__ __forceinline__ void mbar_init_fence() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"   // suspend-time hint: the warp sleeps in
      "@p bra DONE_%=;\n\t"                                            // hardware instead of spinning on issue slots
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(bar), "r"(parity), "r"(0x989680u) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const void* tmap, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(tmap), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// TMEM of a CTA (CG = 1) or of a CTA pair (CG = 2, the same warp of both CTAs): one whole warp allocates `cols`
// columns, writes the base address to the shared-memory word `slot` and gives up the right to allocate more; the
// other warps read the base after the CTA (cluster) barrier that follows.
template <int CG>
__device__ __forceinline__ void tmem_alloc(uint32_t slot, uint32_t cols) {
  static_assert(CG == 1 || CG == 2, "cta_group is 1 or 2");
  if constexpr (CG == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  } else {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
}
__device__ __forceinline__ uint32_t tmem_base_of(uint32_t slot) {
  uint32_t base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(base) : "r"(slot) : "memory");
  return base;
}
template <int CG>
__device__ __forceinline__ void tmem_dealloc(uint32_t base, uint32_t cols) {
  static_assert(CG == 1 || CG == 2, "cta_group is 1 or 2");
  if constexpr (CG == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(cols) : "memory");
  else asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(cols) : "memory");
}

// SM100 shared-memory matrix descriptor, K-major, SWIZZLE_128B: start>>4 | LBO(1)<<16 | SBO(1024B>>4)<<32 |
// version 1 <<46 | layout SWIZZLE_128B (2) << 61
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// instruction descriptor kind::f16: D=f32 (1<<4), A=bf16 (1<<7), B=bf16 (1<<10), K-major both,
// N>>3 at bit 17, M>>4 at bit 24
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
// kind::tf32: A/B format 2 (TF32), fp32 accumulate; K = 8 per instruction
__host__ __device__ constexpr uint32_t umma_idesc_tf32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
// kind::f16 with fp16 operands (A/B format 0), fp32 accumulate; K = 16 per instruction
__host__ __device__ constexpr uint32_t umma_idesc_f16(int M, int N) {
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// split-precision product: tf32 planes (f16 = false) or fp16 planes (f16 = true); both step 32 bytes of K per
// instruction, so the smem descriptors advance identically
__device__ __forceinline__ void umma_split(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc, bool f16) {
  if (f16) umma_bf16(tmem_d, adesc, bdesc, idesc, acc);     // kind::f16; the instruction descriptor selects fp16
  else umma_tf32(tmem_d, adesc, bdesc, idesc, acc);
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// ---- CTA pairs (cta_group::2): two CTAs of a cluster run ONE tcgen05.mma of M = 256; each supplies its own 128 rows
// of A and its own half (N/2 rows) of B from shared memory at the same offsets, and owns the accumulator rows of its A.
// address of the same shared-memory offset in CTA `rank` of the cluster (shared::cluster window)
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
// TMA load into this CTA's shared memory whose completion bytes are counted on an mbarrier of the pair's leader CTA
// (`bar_cluster` is a shared::cluster address, see mapa_u32)
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const void* tmap, int c0, int c1, uint32_t bar_cluster) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(tmap), "r"(bar_cluster), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void umma_f16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
// arrive on the mbarrier at this offset in both CTAs of the pair once the pair-MMAs issued so far have completed
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"((uint16_t)3) : "memory");
}
// arrive on an mbarrier of another CTA of the cluster (shared::cluster address).  Default semantics (.release.cta) on
// purpose: a cluster-scope release makes every arrive wait for the thread's outstanding global stores -- measured, it
// turned the 3.5 Mcycle accumulator drain of the pair GEMM into 24 Mcycles.  What is handed over here is TMEM, and
// that is ordered by tcgen05.wait::ld + tcgen05.fence::before_thread_sync ahead of the arrive.
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar_cluster) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(bar_cluster) : "memory");
}
// wait on a local mbarrier whose arrivals may come from the other CTA of the cluster
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAITC_%=:\n\t"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1, %2;\n\t"
      "@p bra DONEC_%=;\n\t"
      "bra WAITC_%=;\n\t"
      "DONEC_%=:\n\t}" ::"r"(bar), "r"(parity), "r"(0x989680u) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// 64 columns in one instruction: one TMEM round trip instead of two (the split-precision GEMMs drain an accumulator
// chain per 64 K-elements, so the latency of these loads is on the critical path of the epilogue warps)
__device__ __forceinline__ void tmem_ld64(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x64.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32, %33, %34, %35, %36, %37, %38, %39, %40, %41, %42, %43, %44, %45, %46, %47, %48, %49, %50, %51, %52, %53, %54, %55, %56, %57, %58, %59, %60, %61, %62, %63}, [%64];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31]), "=r"(v[32]), "=r"(v[33]), "=r"(v[34]), "=r"(v[35]), "=r"(v[36]), "=r"(v[37]), "=r"(v[38]), "=r"(v[39]), "=r"(v[40]), "=r"(v[41]), "=r"(v[42]), "=r"(v[43]), "=r"(v[44]), "=r"(v[45]), "=r"(v[46]), "=r"(v[47]), "=r"(v[48]), "=r"(v[49]), "=r"(v[50]), "=r"(v[51]), "=r"(v[52]), "=r"(v[53]), "=r"(v[54]), "=r"(v[55]), "=r"(v[56]), "=r"(v[57]), "=r"(v[58]), "=r"(v[59]), "=r"(v[60]), "=r"(v[61]), "=r"(v[62]), "=r"(v[63])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

}  // namespace kkx
