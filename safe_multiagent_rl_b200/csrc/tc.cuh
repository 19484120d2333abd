// tcgen05 / TMEM / mbarrier wrappers (sm_100a inline PTX) for the one GEMM-shaped piece of the path: fc1 of the
// fused per-agent policies (policy_tc.cu).  Single-CTA MMAs (cta_group::1), operands in shared memory in the canonical
// K-major no-swizzle layout, accumulators in tensor memory.
//
// Shared-memory matrix descriptor (64 bit), no swizzle, K-major ("core matrix" = 8 rows x 16 bytes, stored as 128
// contiguous bytes):
//   bits  0..13  start address >> 4
//   bits 16..29  leading-dimension byte offset >> 4 : distance between the two core matrices one MMA reads along K
//   bits 32..45  stride-dimension byte offset >> 4  : distance between 8-row groups along M / N
//   bits 46..47  descriptor version (1 on sm_100)
//   bits 61..63  swizzle mode (0 = none)
// Instruction descriptor (32 bit) for kind::f16 with bf16 inputs and f32 accumulation:
//   bits 4..5 D format (1 = f32), 7..9 A format (1 = bf16), 10..12 B format (1 = bf16), 15 / 16 A / B major (0 = K),
//   17..22 N >> 3, 24..28 M >> 4.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "mbarrier.cuh"

namespace smarl {
namespace tc {

using ::smarl::mbar_init;
using ::smarl::mbar_try_wait;
using ::smarl::mbar_wait;
using ::smarl::smem_u32;

__host__ __device__ constexpr uint64_t smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | ((uint64_t)1 << 46);
}

__host__ __device__ constexpr uint32_t idesc_bf16_f32(int m, int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// ---- tensor memory -------------------------------------------------------------------------------------------
// One full warp allocates `cols` (power of two >= 32) columns; the base address lands in *slot (shared memory).
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// generic-proxy shared-memory writes -> visible to the async proxy (the MMA reads its operands through it)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// 32 lanes x 16 consecutive 32-bit columns: thread i of the warp gets lane (taddr.lane + i), columns taddr.col .. +15.
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
// The same load into raw registers, and a wait that names them: the loaded registers are only defined after
// tcgen05.wait::ld, so the wait takes them as read-write operands and every use is ordered behind it (lets the
// caller keep the next load in flight while it computes on the previous one).
__device__ __forceinline__ void tmem_ld16_raw(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait_regs(uint32_t (&r)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
               :
               : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- MMA ------------------------------------------------------------------------------------------------------
// D[tmem] (+)= A[smem] * B[smem]^T, one thread issues for the CTA.
__device__ __forceinline__ void mma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, bool accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"((uint32_t)accumulate)
      : "memory");
}
// All MMAs issued so far by this thread -> one arrival on the mbarrier when they have completed.
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ---- packed fp32 pairs (FFMA2 on sm_100: two fused multiply-adds per issue slot) -----------------------------
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;"
      : "=l"(d)
      : "l"(*reinterpret_cast<const uint64_t*>(&a)), "l"(*reinterpret_cast<const uint64_t*>(&b)),
        "l"(*reinterpret_cast<const uint64_t*>(&c)));
  return *reinterpret_cast<float2*>(&d);
}

}  // namespace tc
}  // namespace smarl
