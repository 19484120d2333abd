// Shared device/host helpers for libsmarl (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <type_traits>
#include <utility>

#include "../../include/smarl.h"

namespace smarl {

// ---------------------------------------------------------------------------------------
// Error plumbing (thread-local message behind smarl_last_error()).
// ---------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);

#define SMARL_REQUIRE(cond, ...)                \
  do {                                          \
    if (!(cond)) {                              \
      ::smarl::set_error(__VA_ARGS__);          \
      return SMARL_EINVAL;                      \
    }                                           \
  } while (0)

#define SMARL_CUDA(call)                                                                  \
  do {                                                                                    \
    cudaError_t err__ = (call);                                                           \
    if (err__ != cudaSuccess) {                                                           \
      ::smarl::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(err__),       \
                         __FILE__, __LINE__);                                             \
      return SMARL_ECUDA;                                                                 \
    }                                                                                     \
  } while (0)

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// smarl_set_kernel_variant's current setting for an env kind (-1 = automatic).
int kernel_variant(int env_kind);

// Programmatic dependent launch of the per-step kernels (on unless SMARL_PDL=0 in the environment).
bool pdl_enabled();

// Checks the shared layout contract of smarl.h for one call.
int check_layout(int64_t n_envs, int64_t ld);

// Checks the accounting arguments every fused rollout and returns entry point takes: acc present,
// 1 <= n_steps <= max_steps, 0 <= g_mode <= max_g_mode, G present unless g_mode is 0, stats and stats_scratch together.
int check_accounting(const SmarlAccounting* acc, int max_steps, int max_g_mode, const float* G, const double* stats,
                     const double* stats_scratch);

// Selects a compile-time value: calls f(std::integral_constant<int, N>{}) for the N in Lo..Hi that equals n and returns
// its result.  Outside Lo..Hi it sets the error from fmt (one %d, given n) and returns SMARL_EUNSUPPORTED.
template <int Lo, typename F, int... I>
int dispatch_seq(int n, F& f, const char* fmt, std::integer_sequence<int, I...>) {
  int rc = SMARL_EUNSUPPORTED;
  if (!((n == Lo + I && (rc = f(std::integral_constant<int, Lo + I>{}), true)) || ...)) set_error(fmt, n);
  return rc;
}
template <int Lo, int Hi, typename F>
int dispatch(int n, F&& f, const char* fmt = "n_agents=%d outside 1..32") {
  return dispatch_seq<Lo>(n, f, fmt, std::make_integer_sequence<int, Hi - Lo + 1>{});
}

// Which translation unit of a split source this compile is (build.py builds a source once per -DSMARL_TU=k, k from 0
// to the largest k the source names in SMARL_TU_IS(k); -1, the default, builds everything).
#ifndef SMARL_TU
#define SMARL_TU -1
#endif
#define SMARL_TU_IS(k) (SMARL_TU == -1 || SMARL_TU == (k))

#ifdef __CUDACC__
// ---------------------------------------------------------------------------------------
// Programmatic dependent launch (PDL) for the per-step kernels.  A closed loop is T x (policy, step) launches on one
// stream; with small batches (BASELINE configs[0] / [1], or 2^19 envs per GPU of the sharded configs[3]) the ~2-3 us
// between two kernels is a large share of the step.  launch_pdl() lets the NEXT kernel's CTAs be scheduled while this
// one still runs; pdl_prologue() -- the first statement of every such kernel -- then blocks until the previous grid
// has COMPLETED and its memory is visible (griddepcontrol.wait), and only after that allows the kernel behind it to be
// scheduled, so at most two grids overlap and nothing is read before the wait.  Without the launch attribute (or
// behind a kernel that is not PDL-aware) both instructions are no-ops.  Stream capture records the edge as a
// programmatic dependency, so CUDA-graph replays keep the overlap.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_prologue() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
template <typename Arg>
inline cudaError_t launch_pdl(void (*kern)(Arg), dim3 grid, dim3 block, size_t smem, cudaStream_t st, const Arg& a) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = pdl_enabled() ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, a);
}

// ---------------------------------------------------------------------------------------
// Streaming global access.  Every byte of the batched state is touched once per launch,
// so loads bypass L1 allocation and stores are marked evict-first ("streaming").
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t ld_stream_u32(const void* p) {
  uint32_t v;
  asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ float4 ld_stream_f4(const void* p) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p));
  return v;
}
// State that is re-read by the NEXT launch (positions between env steps): ask L2 to keep it
// (evict_last) so that, when a batch's positions fit in the 126 MB L2, they never round-trip HBM.
__device__ __forceinline__ uint64_t l2_keep_policy() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ uint32_t ld_keep_u32(const void* p, uint64_t pol) {
  uint32_t v;
  asm volatile("ld.global.L1::no_allocate.L2::cache_hint.u32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
  return v;
}
__device__ __forceinline__ void st_keep_u32(void* p, uint32_t v, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.u32 [%0], %1, %2;" ::"l"(p), "r"(v), "l"(pol) : "memory");
}
// Coherent load for data this kernel wrote itself earlier (scratch re-reads): never .nc.
__device__ __forceinline__ float4 ld_f4(const void* p) {
  float4 v;
  asm volatile("ld.global.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p)
               : "memory");
  return v;
}
__device__ __forceinline__ void st_stream_u32(void* p, uint32_t v) {
  asm volatile("st.global.cs.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void st_stream_f4(void* p, float4 v) {
  asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
               "f"(v.w)
               : "memory");
}
__device__ __forceinline__ void st_stream_i4(void* p, int4 v) {
  asm volatile("st.global.cs.v4.s32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z),
               "r"(v.w)
               : "memory");
}

// Byte k (0..3) of a packed word as float, exact: PRMT builds 0x4B0000bb (= 2^23 + b), one FADD.
__device__ __forceinline__ float byte_to_float(uint32_t w, int k) {
  uint32_t bits = __byte_perm(w, 0x4B000000u, 0x7440u | (uint32_t)k);
  return __uint_as_float(bits) - 8388608.0f;
}
__device__ __forceinline__ float4 bytes_to_float4(uint32_t w) {
  return make_float4(byte_to_float(w, 0), byte_to_float(w, 1), byte_to_float(w, 2),
                     byte_to_float(w, 3));
}

// ---------------------------------------------------------------------------------------
// Grid moves on four envs at once (one byte per env).  Direction table shared by
// envs/coverage.py:176 and envs/congestion.py:55:  0:(+1,0) 1:(-1,0) 2:(0,-1) 3:(0,+1) 4:stay,
// then clamp to [0,size] (coverage.py:185-186, congestion.py:70-71).  Valid bytes are <= 254,
// so +1 never carries into the neighbouring env; padding lanes may hold garbage, which the
// clamp pulls into range (and a carry out of a padding byte only reaches higher padding bytes).
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void grid_move4(uint32_t& xw, uint32_t& yw, uint32_t aw, uint32_t size4) {
  const uint32_t k1 = 0x01010101u;
  const uint32_t b0 = aw & k1, b1 = (aw >> 1) & k1, b2 = (aw >> 2) & k1;
  const uint32_t inc_x = (b0 | b1 | b2) ^ k1;   // a == 0
  const uint32_t dec_x = b0 & ~b1;              // a == 1  (a <= 4, so b0 => !b2)
  const uint32_t dec_y = b1 & ~b0;              // a == 2
  const uint32_t inc_y = b0 & b1;               // a == 3
  xw = __vsubus4(__vminu4(xw + inc_x, size4), dec_x);
  yw = __vsubus4(__vminu4(yw + inc_y, size4), dec_y);
}
// Same move for grids with size <= 127 (Coverage): with the top bit of every byte free, per-byte
// comparisons are carry-free adds -- bit 7 of (x + 128 - S) is [x >= S], bit 7 of (x + 127) is
// [x >= 1] -- so the clamp costs 7 plain integer ops per coordinate word instead of the emulated
// SIMD min / saturating-subtract intrinsics.  ge_bias = (128 - S) * 0x01010101.
__device__ __forceinline__ void grid_move4_s127(uint32_t& xw, uint32_t& yw, uint32_t aw, uint32_t ge_bias) {
  const uint32_t k1 = 0x01010101u, k7f = 0x7F7F7F7Fu;
  const uint32_t b0 = aw & k1, b1 = (aw >> 1) & k1, b2 = (aw >> 2) & k1;
  const uint32_t inc_x = (b0 | b1 | b2) ^ k1;   // a == 0
  const uint32_t dec_x = b0 & ~b1;              // a == 1
  const uint32_t dec_y = b1 & ~b0;              // a == 2
  const uint32_t inc_y = b0 & b1;               // a == 3
  xw = xw + (inc_x & ~((xw + ge_bias) >> 7)) - (dec_x & ((xw + k7f) >> 7));
  yw = yw + (inc_y & ~((yw + ge_bias) >> 7)) - (dec_y & ((yw + k7f) >> 7));
}
// p += lam where bit (mask) of w is set: one predicate-producing LOP3 + one predicated DADD.
__device__ __forceinline__ void add_if_bit(double& p, double lam, uint32_t w, uint32_t mask) {
  asm("{\n\t.reg .pred q;\n\t.reg .b32 t;\n\tand.b32 t, %2, %3;\n\tsetp.ne.u32 q, t, 0;\n\t@q add.rn.f64 %0, %0, %1;\n\t}"
      : "+d"(p)
      : "d"(lam), "r"(w), "r"(mask));
}
// cost byte = 1 for a non-stay action (coverage.py:191-196: [1,1,1,1,0][a]).
__device__ __forceinline__ uint32_t move_cost4(uint32_t aw) { return ((aw >> 2) & 0x01010101u) ^ 0x01010101u; }

// ---------------------------------------------------------------------------------------
// Philox4x32-10 (oracle/philox.py restates it; Random123 known answers are tested there).
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    // one 32 x 32 -> 64 multiply per product (IMAD.WIDE.U32) instead of a high and a low one
    const uint64_t p0 = (uint64_t)0xD2511F53u * c.x, p1 = (uint64_t)0xCD9E8D57u * c.z;
    const uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0;
    const uint32_t hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}

// ---------------------------------------------------------------------------------------
// Deterministic block reduction of NV doubles per thread -> partial[blockIdx.x][NV] written
// by thread 0.  Fixed shuffle tree + fixed warp order: bit-reproducible for a given launch
// shape.  `smem` needs NV * (blockDim.x/32) doubles.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
#endif  // __CUDACC__

}  // namespace smarl
