// CoverageDiscrete device code shared by the step kernel and the fused rollout kernel.
#pragma once
#include "common.cuh"

namespace smarl {

// Coverage grids are limited to size <= 127 so that doubled coordinates fit a byte (see
// coverage_pack2).  Largest penalty table kept in shared memory (entries): fv^2 <= this.
// (the fused rollout kernel keeps a 32-byte static reduction buffer beside the table: (12279 + 1) * 4 + 32 = 48 KB)
constexpr int kCoverageMaxLut = 12279;

// ---------------------------------------------------------------------------------------
// Fused open-loop episode: positions, cost counters and discounted sums never leave
// registers for the whole horizon; per step a thread reads A action words (1 B / agent-step).
// Replaces main.py:28-57 (minus the policy nets) + buffer.py:30-39 + meta_agent.py:18-30 +
// agent.py:129-132 / :200-206 for four envs per thread.
// ---------------------------------------------------------------------------------------
struct CoverageRolloutArgs {
  const uint8_t* start_x;
  const uint8_t* start_y;
  const uint8_t* actions;   // [T][A][ld]
  const double* lambdas;
  uint8_t* final_x;
  uint8_t* final_y;
  float* R;
  float* modR;
  int32_t* C;
  float* G;                 // [T][A][ld]
  float* g_scratch;         // [2][T][ld]
  double* partials;         // [gridDim.x][stats_len]
  const double* thresholds;
  const float* lut;
  const float* weights;
  double gamma;
  int64_t n_groups;
  int64_t n_envs;
  int64_t ld;
  int32_t size;
  int32_t lut_len;
  int32_t n_steps;
  int32_t g_mode;
};

constexpr int kRolloutThreads = 128;

inline int check_coverage(const SmarlCoverageParams* p) {
  SMARL_REQUIRE(p != nullptr, "params is NULL");
  SMARL_REQUIRE(p->size >= 1 && p->size <= 127, "size=%d outside 1..127", p->size);
  SMARL_REQUIRE(p->lut_len >= 0 && (p->lut_len == 0 || p->lut != nullptr), "bad penalty table");
  if (p->lut_len > kCoverageMaxLut) {
    set_error("lut_len=%d exceeds the shared-memory table limit %d", p->lut_len, kCoverageMaxLut);
    return SMARL_EUNSUPPORTED;
  }
  return SMARL_OK;
}

// Agents of env lane k packed for the pair loop: p[a] = (2x | 2y << 8), upper bytes zero.
// One PRMT gathers (x_k, y_k) and zero-fills bytes 2,3 by replicating the (clear) sign bit of
// x_k -- coordinates are <= 127 -- and one add doubles both bytes without carry.
__device__ __forceinline__ uint32_t coverage_pack2(uint32_t xw, uint32_t yw, uint32_t sel) {
  uint32_t p;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(p) : "r"(xw), "r"(yw), "r"(sel));
  return p + p;
}
// selector for env lane k: byte0 = x.b[k], byte1 = y.b[k], byte2 = byte3 = sign(x.b[k]) = 0
__device__ __forceinline__ uint32_t coverage_pack_sel(int k) {
  return (uint32_t)k | ((uint32_t)(k + 4) << 4) | ((uint32_t)(8 + k) << 8) | ((uint32_t)(8 + k) << 12);
}

// Sum of pair penalties of ONE env whose agents are packed by coverage_pack2.
//
// Replaces the i<j double loop over scipy's distance_matrix in CoverageContinuous.reward
// (envs/coverage.py:76-83).  For integer coordinates the distance is sqrt(q) with
// q = dx^2 + dy^2 an integer, so the penalty is a table lookup: 2|dx|, 2|dy| for the pair come
// from one SIMD byte abs-diff (VABSDIFF4), 4q -- already the byte offset into the f32 table --
// from one dp4a (IDP.4A), clamped (VIMNMX) to the table's trailing zero entry, then LDS + FADD.
// The clamp is not only a bounds guard: most pairs are farther apart than the field of view, so their lookups all
// hit the ONE trailing zero entry (a broadcast) and the rest a table of a few hundred bytes.  A table covering every
// q (no VIMNMX, measured in round 2) scatters the 32 lanes over ~2000 entries: shared-memory bank conflicts took the
// step kernel from 205 to 302 us and the fused rollout from 6.0 to 12.1 ms.  Rejected.
// Canonical summation order (every kernel that produces rewards uses this function, so
// step-mode and fused-mode rewards are bit-identical): pair n in the reference's i-major
// order goes to accumulator n % 4, result = (acc0 + acc1) + (acc2 + acc3), all f32.
template <int A>
__device__ __forceinline__ float coverage_pair_penalty(const uint32_t (&p)[A],
                                                       const float* __restrict__ s_lut,
                                                       uint32_t lut_bytes) {
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  int n = 0;
  const char* base = reinterpret_cast<const char*>(s_lut);
#pragma unroll
  for (int i = 0; i < A; ++i) {
#pragma unroll
    for (int j = i + 1; j < A; ++j) {
      const uint32_t v = __vabsdiffu4(p[i], p[j]);
      const uint32_t off = min(__dp4a(v, v, 0u), lut_bytes);
      acc[n & 3] += *reinterpret_cast<const float*>(base + off);
      ++n;
    }
  }
  return (acc[0] + acc[1]) + (acc[2] + acc[3]);
}

// Stage the penalty table: s_lut[0..lut_len) = lut, s_lut[lut_len] = 0.
__device__ __forceinline__ void coverage_load_lut(float* s_lut, const float* __restrict__ lut,
                                                  int lut_len) {
  for (int i = threadIdx.x; i <= lut_len; i += blockDim.x) s_lut[i] = i < lut_len ? __ldg(lut + i) : 0.f;
  __syncthreads();
}

}  // namespace smarl
