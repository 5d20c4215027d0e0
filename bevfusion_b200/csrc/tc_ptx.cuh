// tcgen05 / TMA / mbarrier PTX wrappers shared by the sparse-conv kernels (sm_100a).  Internal header.
#pragma once
#include "common.cuh"

namespace bevb200 {

// ---- PTX wrappers ----------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, 0x989680;\n\t"   // suspend, do not spin
      "@p bra WAIT_DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t}"
      ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_copy_g2s(uint32_t dst_smem, const void *src, uint32_t bytes,
                                              uint32_t bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
      ::"r"(dst_smem), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// one elected lane of a fully converged warp (elect.sync): the compiler keeps the tcgen05 issue
// sequence on the uniform datapath; an `if (lane == 0)` branch instead makes it wrap every
// UTCHMMA in an ELECT / BRA.U.ANY waterfall loop (measured: ~100 clk per MMA issue)
__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];"
               ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                            uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, float v[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// UMMA shared-memory descriptor, K-major, SWIZZLE_128B (cute/arch/mma_sm100_desc.hpp layout):
//   [0,14) start address >> 4, [16,30) leading byte offset >> 4 (unused for swizzled K-major),
//   [32,46) stride byte offset >> 4 (= 1024 B between 8-row groups), [46,48) version = 1,
//   [61,64) layout type = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  uint64_t d = (uint64_t)((smem_addr & 0x3ffff) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// instruction descriptor for kind::tf32: c=F32 (bit 4), a=b=TF32 (2 at bits 7, 10), both K-major,
// N >> 3 at bit 17, M >> 4 at bit 24
__host__ __device__ inline uint32_t umma_idesc_tf32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// instruction descriptor for kind::f16 with bf16 operands: c=F32 (bit 4), a=b=BF16 (1 at bits 7, 10)
__host__ __device__ inline uint32_t umma_idesc_bf16(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// two fp32 -> packed bf16x2 (round to nearest even): `lo` lands in bits 0..15, `hi` in bits 16..31
__device__ __forceinline__ uint32_t cvt_bf16x2(float hi, float lo) {
  uint32_t d;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}

// 16-byte cp.async; `row` < 0 = the ignore-src form: nothing is read, the 16 bytes are zero-filled
__device__ __forceinline__ void cp_async16_row(uint32_t dst_smem, unsigned long long src, int row) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.lt.s32 p, %2, 0;\n\t"
      "cp.async.cg.shared.global [%0], [%1], 16, p;\n\t}"
      ::"r"(dst_smem), "l"(src), "r"(row) : "memory");
}

__device__ __forceinline__ void cp_async_mbar_arrive_noinc(uint32_t bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}

}  // namespace bevb200
