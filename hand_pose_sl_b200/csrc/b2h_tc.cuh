// Thin inline-PTX layer for sm_100a: tcgen05 (UMMA) + TMEM + mbarrier + bulk async copies.
// Field layouts follow the PTX ISA "tcgen05 matrix/instruction descriptor" tables.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace b2h {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// one lane of a fully-active warp (warp-uniform predicate the compiler can keep on the uniform datapath)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\t"
      "elect.sync rx|px, 0xFFFFFFFF;\n\t"
      "@px mov.s32 %0, 1;\n\t}"
      : "+r"(pred));
  return pred != 0;
}

// ---- mbarrier -------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ uint32_t mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok;
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}

#ifndef B2H_TC_NO_STATUS
// Device-side status word: a wait that exceeds its budget records the site and returns so a
// descriptor / protocol bug ends as a wrong answer + error code, never as a hung GPU.
__device__ int g_tc_status = 0;
// Data-parallel exchange: set (with status 51) when a wait for a peer's gradient words gave up; while it is set the
// fused train kernel writes no parameter / moment (sticky until the host reads the status) -- see b2h_tc_status.
__device__ int g_dp_abort = 0;

__device__ __forceinline__ bool mbar_wait(uint64_t* bar, uint32_t parity, int site) {
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) {  // ~2 s at 2 GHz
      atomicExch(&g_tc_status, site);
      return false;
    }
  }
  return true;
}
// Whole-warp wait with ONE polling lane: 256 threads spinning on try_wait keep the SM's barrier unit busy enough to
// delay the MMA-issuing thread's own barrier traffic (measured: 538 -> ~260 cycles per weight stage of the wide kernel).
__device__ __forceinline__ bool mbar_wait_warp(uint64_t* bar, uint32_t parity, int site) {
  int ok = 1;
  if ((threadIdx.x & 31) == 0) ok = mbar_wait(bar, parity, site) ? 1 : 0;
  ok = __shfl_sync(0xffffffffu, ok, 0);     // also orders lane 0's acquire before the other lanes' later accesses
  return ok != 0;
}
#endif  // B2H_TC_NO_STATUS

// named barrier `id` (1..15; 0 is __syncthreads) over `nthreads` (whole warps)
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---- proxies / fences -------------------------------------------------------------------------
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// Programmatic dependent launch (sm_90+).  `launch_dependents`: the next kernel on the stream, if it was launched with the
// programmatic-serialization attribute, may start its CTAs once every CTA of this grid has passed this point (or exited).
// `wait`: blocks until the preceding grid has completed and its memory is visible; a no-op for a normal launch.
__device__ __forceinline__ void griddep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---- TMEM -------------------------------------------------------------------------------------
// warp-collective; ncols power of two in [32, 512]
__device__ __forceinline__ void tmem_alloc(uint32_t* slot_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot_smem)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

#define B2H_TMEM_LD_REGS16(v, o) \
  "=r"(v[o + 0]), "=r"(v[o + 1]), "=r"(v[o + 2]), "=r"(v[o + 3]), "=r"(v[o + 4]), "=r"(v[o + 5]), "=r"(v[o + 6]), \
      "=r"(v[o + 7]), "=r"(v[o + 8]), "=r"(v[o + 9]), "=r"(v[o + 10]), "=r"(v[o + 11]), "=r"(v[o + 12]),           \
      "=r"(v[o + 13]), "=r"(v[o + 14]), "=r"(v[o + 15])

// 32 lanes x 32-bit, 16 consecutive columns: thread i of the warp receives row (lane_base+i)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : B2H_TMEM_LD_REGS16(v, 0)
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : B2H_TMEM_LD_REGS16(v, 0), B2H_TMEM_LD_REGS16(v, 16)
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- UMMA descriptors ---------------------------------------------------------------------------
// Shared-memory matrix descriptor, SWIZZLE_NONE ("interleave"): core matrix = 8 rows x 16 bytes,
// stored as 128 contiguous bytes.
//   K-major  operand: LBO = byte distance between the two 16-B K-chunks of one MMA (K=16 bf16),
//                     SBO = byte distance between consecutive 8-row (M/N) groups.
//   MN-major operand: LBO = byte distance between consecutive 8-element K groups,
//                     SBO = byte distance between consecutive 8-element (16-B) M/N groups.
// bits [0,14) start>>4 | [16,30) LBO>>4 | [32,46) SBO>>4 | [46,48) version=1 | [61,64) layout=0
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t version = 1) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)(version & 3) << 46;
  return d;
}

// Instruction descriptor, kind::f16: D=f32 (bits 4-5 = 1), A=B=bf16 (bits 7-9, 10-12 = 1),
// a_major bit 15, b_major bit 16 (0 = K-major, 1 = MN-major), N>>3 at bits 17-22, M>>4 at bits 24-28.
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread on behalf of the CTA.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// all previously issued MMAs of this thread arrive on `bar` when complete (implies fence::before_thread_sync)
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ---- bulk async copy (TMA engine, 1-D): global -> shared, completion on an mbarrier ---------------
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// shared -> global bulk store (TMA engine), bulk-group completion
__device__ __forceinline__ void bulk_s2g(void* gdst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(smem_src)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

}  // namespace tc
}  // namespace b2h
