// CoverageDiscrete, lane-cooperative step kernel for large agent counts (sm_100a).
//
// coverage.cu keeps all A agents of four envs in one thread (3A state words + the packed pair operands): from
// A ~ 20 that is 255 registers, two CTAs per SM, and the kernel falls from 0.83-0.89 of the HBM roofline (A <= 16)
// to 0.59 (A = 32).  Here a group of S = 2 or 4 lanes shares one quad of four envs; lane s owns agents
// i = j*S + s (j = 0..B-1, B = ceil(A/S)), still as SIMD-in-word bytes (one byte per env).  A warp covers 32/S
// quads; lane = s*(32/S) + q, so each load / store instruction touches S rows x (32/S) consecutive 4-byte words
// (u8 rows) or 16-byte vectors (f32 rows) of the agent-major SoA arrays: whole 32-byte sectors.
//
//   moves, costs, obs, done       own agents only, the byte-SIMD code of coverage.cu (common.cuh)
//   reward (coverage.py:76-89)    every lane publishes its agents' packed positions (2x | 2y << 8, one word per
//                                 env) to shared memory; agent i then sums the table penalties of the partners
//                                 (i + k) mod A, k = 1..A/2 -- each unordered pair exactly once, balanced over the
//                                 lanes -- and the S partial sums meet in an xor-shuffle tree (identical on every
//                                 lane of the group because a + b == b + a).
//   penalty <lambda, c>           per-lane partial sums over own agents in f64, same shuffle tree
//
// Parity: moves / costs are the same integer code; the reward is an f32 sum of the same table entries in another
// association than coverage.cu (<= 1e-6 relative apart, tests hold 1e-5 against the f64 oracle).
#include "coverage.cuh"

namespace smarl {

constexpr int kCovCoopThreads = 128;

template <int A, int S>
struct CovCoop {
  static constexpr int B = (A + S - 1) / S;          // agents per lane
  static constexpr int EPW = 32 / S;                 // env quads per warp
  static constexpr int EPC = kCovCoopThreads / S;    // env quads per CTA
  static constexpr int H = A / 2;                    // circular partner window (last offset halved for even A)
  static constexpr bool kGhost = (A % S) != 0;
  static constexpr int PA = (((A + S - 1) / S) | 1) * S;   // words per (env lane, quad): S * odd => conflict-free LDS.32
  static constexpr size_t kPosWords = (size_t)4 * EPC * PA;
};

// CoverageStepArgs is declared in coverage.cu; the launcher below takes the same fields.
struct CoverageCoopArgs {
  uint8_t* pos_x;
  uint8_t* pos_y;
  const uint8_t* actions;
  float* obs;
  float* reward;
  uint8_t* cost;
  uint8_t* done;
  const double* lambdas;
  float* penalty;
  const float* lut;
  const float* weights;
  int64_t n_groups;
  int64_t ld;
  int32_t size;
  int32_t lut_len;
  int32_t reward_rows;
};

template <int A, int S>
__global__ void __launch_bounds__(kCovCoopThreads, 4) coverage_coop_step_kernel(const CoverageCoopArgs a) {
  pdl_prologue();   // programmatic dependent launch: the previous grid has completed past this point (common.cuh)
  using C = CovCoop<A, S>;
  constexpr int B = C::B, EPW = C::EPW, EPC = C::EPC, H = C::H, PA = C::PA;
  extern __shared__ float s_lut[];                                        // [lut_len + 1] then the packed positions
  uint32_t* s_p = reinterpret_cast<uint32_t*>(s_lut + ((a.lut_len + 1 + 3) & ~3));   // [4][EPC][PA]
  coverage_load_lut(s_lut, a.lut, a.lut_len);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int q = lane % EPW, s = lane / EPW;
  const int ql = warp * EPW + q;                                          // quad within the CTA
  const int64_t gq = (int64_t)blockIdx.x * EPC + ql;
  const bool live = gq < a.n_groups;
  const uint32_t ld = (uint32_t)a.ld;
  const uint32_t e0 = (uint32_t)(live ? gq : 0) * 4u;
  const uint32_t row0 = (uint32_t)s * ld + e0;                            // agent s, this quad (32-bit offsets, host-checked)

  uint32_t xw[B], yw[B], aw[B];
#pragma unroll
  for (int j = 0; j < B; ++j) {
    const uint32_t off = row0 + (uint32_t)(j * S) * ld;
    if (!C::kGhost || j < B - 1 || j * S + s < A) {
      xw[j] = ld_stream_u32(a.pos_x + off);
      yw[j] = ld_stream_u32(a.pos_y + off);
      aw[j] = ld_stream_u32(a.actions + off);
    } else {
      xw[j] = yw[j] = 0u;
      aw[j] = 0x04040404u;                                                // padding agent: stays, costs nothing
    }
  }
  const uint32_t ge_bias = (uint32_t)(128 - a.size) * 0x01010101u;
  double pen[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
  for (int j = 0; j < B; ++j) {
    const bool own = !C::kGhost || j < B - 1 || j * S + s < A;
    grid_move4_s127(xw[j], yw[j], aw[j], ge_bias);                        // coverage.py:174-189
    const uint32_t cw = move_cost4(aw[j]);                                // coverage.py:191-196
    if (own && live) {
      const uint32_t off = row0 + (uint32_t)(j * S) * ld;
      st_stream_u32(a.pos_x + off, xw[j]);
      st_stream_u32(a.pos_y + off, yw[j]);
      st_stream_u32(a.cost + off, cw);
      if (a.done) st_stream_u32(a.done + off, 0u);                        // coverage.py:97-98
      if (a.obs) {
        const uint32_t o2 = 2u * off - e0;                                // row 2i
        st_stream_f4(a.obs + o2, bytes_to_float4(xw[j]));
        st_stream_f4(a.obs + (o2 + ld), bytes_to_float4(yw[j]));
      }
    }
    if (a.penalty && own) {                                               // meta_agent.py:21-22
      const double lam = __ldg(a.lambdas + (j * S + s));
#pragma unroll
      for (int k = 0; k < 4; ++k) add_if_bit(pen[k], lam, cw, 1u << (8 * k));
    }
    // publish the packed position of every env lane: s_p[k][quad][agent]
    if (own) {
#pragma unroll
      for (int k = 0; k < 4; ++k)
        s_p[(k * EPC + ql) * PA + j * S + s] = coverage_pack2(xw[j], yw[j], coverage_pack_sel(k));
    }
  }
  if (a.penalty) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
#pragma unroll
      for (int off = 1; off < S; off <<= 1) pen[k] += __shfl_xor_sync(0xffffffffu, pen[k], off * EPW);
    }
    if (s == 0 && live)
      st_stream_f4(a.penalty + e0, make_float4((float)pen[0], (float)pen[1], (float)pen[2], (float)pen[3]));
  }
  __syncwarp();

  // pair penalties: agent i against partners (i + k) mod A, k = 1..H (for even A the offset H pairs each couple
  // twice: only i < H counts it)
  const uint32_t lut_bytes = (uint32_t)a.lut_len * 4u;
  const char* lut_base = reinterpret_cast<const char*>(s_lut);
  float r[4];
#pragma unroll 1
  for (int k = 0; k < 4; ++k) {
    const uint32_t sel = coverage_pack_sel(k);
    uint32_t p[B];
#pragma unroll
    for (int j = 0; j < B; ++j) {
      p[j] = coverage_pack2(xw[j], yw[j], sel);
      // a padding agent differs from every real one by 255 in byte 2: all its pairs land on the table's zero entry
      if (C::kGhost && j == B - 1 && j * S + s >= A) p[j] = 0x00FF0000u;
    }
    const uint32_t* sp = s_p + (k * EPC + ql) * PA + s;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    int n = 0;
#pragma unroll
    for (int c = 1; c <= (B - 1) * S + H; ++c) {
      // partner index (s + c) mod A: compile-time except for the S-1 offsets around the wrap
      uint32_t pp;
      if (c + S - 1 < A) pp = sp[c];
      else if (c >= A) pp = sp[c - A];
      else pp = sp[(s + c >= A) ? c - A : c];
#pragma unroll
      for (int j = 0; j < B; ++j) {
        const int kk = c - j * S;
        if (kk >= 1 && kk <= H) {
          const uint32_t v = __vabsdiffu4(p[j], pp);
          uint32_t off = min(__dp4a(v, v, 0u), lut_bytes);
          if (A % 2 == 0 && kk == H) off = (j * S + s < H) ? off : lut_bytes;
          acc[n & 3] += *reinterpret_cast<const float*>(lut_base + off);
          ++n;
        }
      }
    }
    float t = (acc[0] + acc[1]) + (acc[2] + acc[3]);
#pragma unroll
    for (int off = 1; off < S; off <<= 1) t += __shfl_xor_sync(0xffffffffu, t, off * EPW);
    r[k] = -t;                                                            // coverage.py:79-83
  }
  if (!live) return;
  if (a.reward_rows == 1) {                      // one unweighted row; the accounting applies w_a
    if (s == 0) st_stream_f4(a.reward + e0, make_float4(r[0], r[1], r[2], r[3]));
    return;
  }
#pragma unroll
  for (int j = 0; j < B; ++j) {
    if (C::kGhost && j == B - 1 && j * S + s >= A) continue;
    const float w = a.weights ? __ldg(a.weights + (j * S + s)) : 1.0f;    // coverage.py:86-87
    st_stream_f4(a.reward + (row0 + (uint32_t)(j * S) * ld), make_float4(r[0] * w, r[1] * w, r[2] * w, r[3] * w));
  }
}

template <int S>
static int launch_s(int A, const CoverageCoopArgs& a, cudaStream_t st) {
  return dispatch<9, 32>(A, [&](auto kA) {
    using C = CovCoop<kA, S>;
    auto kern = coverage_coop_step_kernel<kA, S>;
    const size_t smem = (size_t)((a.lut_len + 1 + 3) & ~3) * sizeof(float) + C::kPosWords * sizeof(uint32_t);
    if (smem > 48 * 1024)
      SMARL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const unsigned grid = (unsigned)((a.n_groups + C::EPC - 1) / C::EPC);
    SMARL_CUDA(launch_pdl(kern, grid, kCovCoopThreads, smem, st, a));
    SMARL_CUDA(cudaGetLastError());
    return SMARL_OK;
  }, "cooperative Coverage kernels cover n_agents 9..32 (got %d)");
}

// Entry used by smarl_coverage_step (coverage.cu).
int launch_coverage_coop_step(int A, int S, uint8_t* pos_x, uint8_t* pos_y, const uint8_t* actions, float* obs,
                              float* reward, uint8_t* cost, uint8_t* done, const double* lambdas, float* penalty,
                              const float* lut, const float* weights, int64_t n_groups, int64_t ld, int size,
                              int lut_len, int reward_rows, cudaStream_t st) {
  CoverageCoopArgs a;
  a.pos_x = pos_x; a.pos_y = pos_y; a.actions = actions; a.obs = obs; a.reward = reward; a.cost = cost; a.done = done;
  a.lambdas = lambdas; a.penalty = penalty; a.lut = lut; a.weights = weights; a.n_groups = n_groups; a.ld = ld;
  a.size = size; a.lut_len = lut_len; a.reward_rows = reward_rows;
  return S == 2 ? launch_s<2>(A, a, st) : launch_s<4>(A, a, st);
}

}  // namespace smarl
