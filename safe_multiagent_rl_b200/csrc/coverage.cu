// CoverageDiscrete ("Explore") on sm_100a: step kernel, shared grid reset, fused rollout.
//
// Thread mapping: one thread owns FOUR consecutive envs.  All arrays are agent-major SoA
// ([row][ld], env fastest), so for every row a warp moves 32 x 4 B = 128 contiguous bytes of
// u8 state per load and 32 x 16 B = 512 contiguous bytes of f32 output per store.  The four
// envs share the SIMD-in-word move / cost logic (one byte per env); the pair loop runs per env
// on agents packed (x | y << 8).  No shared-memory staging of state: every byte is touched
// once, already coalesced.  Shared memory only holds the penalty table.
#include <stdlib.h>

#include "coverage.cuh"
#include "stats.cuh"

// Built as three translation units (build.py compiles this file once per SMARL_TU value):
//   0 step kernel   1 fused rollout kernel   2 reset kernel + C entry points

namespace smarl {

struct CoverageStepArgs {
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
  int64_t n_groups;   // ceil(n_envs / 4)
  int64_t ld;
  int32_t size;
  int32_t lut_len;
  int32_t reward_rows;
  int32_t keep_pos;   // positions fit in L2: load/store them with an evict_last policy
};

constexpr int kStepThreads = 128;

int launch_coverage_step(int A, const CoverageStepArgs& a, unsigned grid, cudaStream_t s);
int launch_coverage_coop_step(int A, int S, uint8_t* pos_x, uint8_t* pos_y, const uint8_t* actions, float* obs,
                              float* reward, uint8_t* cost, uint8_t* done, const double* lambdas, float* penalty,
                              const float* lut, const float* weights, int64_t n_groups, int64_t ld, int size,
                              int lut_len, int reward_rows, cudaStream_t st);
int launch_coverage_rollout(int A, const CoverageRolloutArgs& a, unsigned grid, cudaStream_t s);

#if SMARL_TU_IS(0)
// KEEP: positions fit in L2 and are loaded / stored with an evict_last policy (a compile-time switch: as a
// run-time branch inside the load loop it cost the reward_rows = 1 path 13 % of its bandwidth).
template <int A, bool KEEP>
__global__ void __launch_bounds__(kStepThreads) coverage_step_kernel(const CoverageStepArgs a) {
  pdl_prologue();   // programmatic dependent launch: the previous grid has completed past this point (common.cuh)
  extern __shared__ float s_lut[];
  coverage_load_lut(s_lut, a.lut, a.lut_len);
  const int64_t g = (int64_t)blockIdx.x * kStepThreads + threadIdx.x;
  if (g >= a.n_groups) return;
  // 32-bit element offsets (host checks (2A+1) * ld < 2^32): one add per row, one wide add per access
  const uint32_t ld = (uint32_t)a.ld;
  const uint32_t e0 = (uint32_t)g * 4u;

  uint32_t xw[A], yw[A], aw[A];
  const uint64_t keep = KEEP ? l2_keep_policy() : 0ull;
  {
    uint32_t off = e0;
#pragma unroll
    for (int i = 0; i < A; ++i, off += ld) {
      if (KEEP) {
        xw[i] = ld_keep_u32(a.pos_x + off, keep);
        yw[i] = ld_keep_u32(a.pos_y + off, keep);
      } else {
        xw[i] = ld_stream_u32(a.pos_x + off);
        yw[i] = ld_stream_u32(a.pos_y + off);
      }
      aw[i] = ld_stream_u32(a.actions + off);
    }
  }
  const uint32_t ge_bias = (uint32_t)(128 - a.size) * 0x01010101u;
  double pen[4] = {0.0, 0.0, 0.0, 0.0};
  {
    uint32_t off = e0, obs_off = e0;
#pragma unroll
    for (int i = 0; i < A; ++i, off += ld, obs_off += 2u * ld) {
      grid_move4_s127(xw[i], yw[i], aw[i], ge_bias);       // coverage.py:174-189
      const uint32_t cw = move_cost4(aw[i]);               // coverage.py:191-196
      if (KEEP) {
        st_keep_u32(a.pos_x + off, xw[i], keep);
        st_keep_u32(a.pos_y + off, yw[i], keep);
      } else {
        st_stream_u32(a.pos_x + off, xw[i]);
        st_stream_u32(a.pos_y + off, yw[i]);
      }
      st_stream_u32(a.cost + off, cw);
      if (a.done) st_stream_u32(a.done + off, 0u);         // coverage.py:97-98
      if (a.obs) {
        st_stream_f4(a.obs + obs_off, bytes_to_float4(xw[i]));
        st_stream_f4(a.obs + (obs_off + ld), bytes_to_float4(yw[i]));
      }
      if (a.penalty) {                                      // meta_agent.py:21-22
        const double lam = __ldg(a.lambdas + i);
#pragma unroll
        for (int k = 0; k < 4; ++k) add_if_bit(pen[k], lam, cw, 1u << (8 * k));
      }
    }
  }
  if (a.penalty)
    st_stream_f4(a.penalty + e0, make_float4((float)pen[0], (float)pen[1], (float)pen[2], (float)pen[3]));

  float r0 = 0.f, r1 = 0.f, r2 = 0.f, r3 = 0.f;
  const uint32_t lut_bytes = (uint32_t)a.lut_len * 4u;
#pragma unroll 1
  for (int k = 0; k < 4; ++k) {
    const uint32_t sel = coverage_pack_sel(k);
    uint32_t p[A];
#pragma unroll
    for (int i = 0; i < A; ++i) p[i] = coverage_pack2(xw[i], yw[i], sel);
    const float r = -coverage_pair_penalty<A>(p, s_lut, lut_bytes);              // coverage.py:79-83
    r0 = k == 0 ? r : r0;
    r1 = k == 1 ? r : r1;
    r2 = k == 2 ? r : r2;
    r3 = k == 3 ? r : r3;
  }
  if (a.reward_rows == 1) {                      // one unweighted row; the accounting applies w_a
    st_stream_f4(a.reward + e0, make_float4(r0, r1, r2, r3));
    return;
  }
  {
    uint32_t off = e0;
#pragma unroll
    for (int i = 0; i < A; ++i, off += ld) {
      const float w = a.weights ? __ldg(a.weights + i) : 1.0f;                   // coverage.py:86-87
      st_stream_f4(a.reward + off, make_float4(r0 * w, r1 * w, r2 * w, r3 * w));
    }
  }
}

int launch_coverage_step(int A, const CoverageStepArgs& a, unsigned grid, cudaStream_t s) {
  const size_t smem = (size_t)(a.lut_len + 1) * sizeof(float);
  if (a.keep_pos)
    return dispatch<1, 32>(A, [&](auto kA) {
      SMARL_CUDA(launch_pdl(coverage_step_kernel<kA, true>, grid, kStepThreads, smem, s, a));
      SMARL_CUDA(cudaGetLastError());
      return SMARL_OK;
    });
  return dispatch<1, 32>(A, [&](auto kA) {
    SMARL_CUDA(launch_pdl(coverage_step_kernel<kA, false>, grid, kStepThreads, smem, s, a));
    SMARL_CUDA(cudaGetLastError());
    return SMARL_OK;
  });
}
#endif

#if SMARL_TU_IS(1)
// Up to 4 agents the kernel is capped at 64 registers (8 CTAs per SM; A = 3 / 4 on 2^22 envs +4 % / +1.5 %); from A = 8 on a cap
// was measured slower (A = 8 at 96 registers -3 %, A = 16 at 128 registers -13 %).
template <int A>
__global__ void __launch_bounds__(kRolloutThreads, (A <= 4 ? 8 : 0)) coverage_rollout_kernel(const CoverageRolloutArgs a) {
  extern __shared__ float s_lut[];
  coverage_load_lut(s_lut, a.lut, a.lut_len);
  const int64_t g = (int64_t)blockIdx.x * kRolloutThreads + threadIdx.x;
  const bool live = g < a.n_groups;
  const int64_t e0 = (live ? g : 0) * 4;
  const int64_t ld = a.ld;
  const int T = a.n_steps;

  uint32_t xw[A], yw[A], cnt[A];
  double lam[A];
#pragma unroll
  for (int i = 0; i < A; ++i) {
    xw[i] = ld_stream_u32(a.start_x + i * ld + e0);
    yw[i] = ld_stream_u32(a.start_y + i * ld + e0);
    cnt[i] = 0u;
    lam[i] = a.lambdas ? __ldg(a.lambdas + i) : 0.0;
  }
  const uint32_t ge_bias = (uint32_t)(128 - a.size) * 0x01010101u;
  double s_rew[4] = {0, 0, 0, 0}, s_pen[4] = {0, 0, 0, 0};
  double disc = 1.0;

  for (int t = 0; t < T; ++t) {
    const uint8_t* act_t = a.actions + (int64_t)t * A * ld;          // uniform; per-thread offsets stay 32-bit
    uint32_t aw[A];
    {
      uint32_t off = (uint32_t)e0;
#pragma unroll
      for (int i = 0; i < A; ++i, off += (uint32_t)ld) aw[i] = ld_stream_u32(act_t + off);
    }
    double pen[4] = {0, 0, 0, 0};
#pragma unroll
    for (int i = 0; i < A; ++i) {
      grid_move4_s127(xw[i], yw[i], aw[i], ge_bias);
      const uint32_t cw = move_cost4(aw[i]);
      cnt[i] += cw;                                   // four byte counters, T <= 255
#pragma unroll
      for (int k = 0; k < 4; ++k) add_if_bit(pen[k], lam[i], cw, 1u << (8 * k));
    }
    float r0 = 0.f, r1 = 0.f, r2 = 0.f, r3 = 0.f;
#pragma unroll 1
    for (int k = 0; k < 4; ++k) {
      const uint32_t sel = coverage_pack_sel(k);
      uint32_t p[A];
#pragma unroll
      for (int i = 0; i < A; ++i) p[i] = coverage_pack2(xw[i], yw[i], sel);
      const float r = -coverage_pair_penalty<A>(p, s_lut, (uint32_t)a.lut_len * 4u);
      r0 = k == 0 ? r : r0;
      r1 = k == 1 ? r : r1;
      r2 = k == 2 ? r : r2;
      r3 = k == 3 ? r : r3;
    }
    const float rr[4] = {r0, r1, r2, r3};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      pen[k] = (double)(float)pen[k];                 // the step kernel publishes the penalty as f32
      s_rew[k] += disc * (double)rr[k];
      s_pen[k] += disc * pen[k];
    }
    if (a.g_mode == 1 && live) {
      st_stream_f4(a.g_scratch + (int64_t)t * ld + e0, make_float4(r0, r1, r2, r3));
      st_stream_f4(a.g_scratch + ((int64_t)T + t) * ld + e0,
                   make_float4((float)pen[0], (float)pen[1], (float)pen[2], (float)pen[3]));
    } else if (a.g_mode == 2 && live) {               // agent.py:129-132: gamma^t * m_t
#pragma unroll
      for (int i = 0; i < A; ++i) {
        const double w = a.weights ? (double)__ldg(a.weights + i) : 1.0;
        float4 o;
        o.x = (float)(disc * ((double)(r0 * (float)w) - pen[0]));
        o.y = (float)(disc * ((double)(r1 * (float)w) - pen[1]));
        o.z = (float)(disc * ((double)(r2 * (float)w) - pen[2]));
        o.w = (float)(disc * ((double)(r3 * (float)w) - pen[3]));
        st_stream_f4(a.G + ((int64_t)t * A + i) * ld + e0, o);
      }
    }
    disc *= a.gamma;
  }

  // Episode products.  reward_a = w_a * rew is linear in rew, so one discounted sum per env
  // serves every agent:  R_a = w_a * S_rew,  modR_a = w_a * S_rew - S_pen.
  if (live) {
#pragma unroll
    for (int i = 0; i < A; ++i) {
      const double w = a.weights ? (double)__ldg(a.weights + i) : 1.0;
      if (a.final_x) st_stream_u32(a.final_x + i * ld + e0, xw[i]);
      if (a.final_y) st_stream_u32(a.final_y + i * ld + e0, yw[i]);
      st_stream_f4(a.R + i * ld + e0, make_float4((float)(w * s_rew[0]), (float)(w * s_rew[1]),
                                                  (float)(w * s_rew[2]), (float)(w * s_rew[3])));
      st_stream_f4(a.modR + i * ld + e0,
                   make_float4((float)(w * s_rew[0] - s_pen[0]), (float)(w * s_rew[1] - s_pen[1]),
                               (float)(w * s_rew[2] - s_pen[2]), (float)(w * s_rew[3] - s_pen[3])));
      st_stream_i4(a.C + i * ld + e0, make_int4(cnt[i] & 0xFF, (cnt[i] >> 8) & 0xFF,
                                                (cnt[i] >> 16) & 0xFF, cnt[i] >> 24));
    }
    if (a.g_mode == 1) {                               // agent.py:200-206, backward Horner
      double g_rew[4] = {0, 0, 0, 0}, g_pen[4] = {0, 0, 0, 0};
      for (int t = T - 1; t >= 0; --t) {
        const float4 r = ld_f4(a.g_scratch + (int64_t)t * ld + e0);
        const float4 q = ld_f4(a.g_scratch + ((int64_t)T + t) * ld + e0);
        const float rr[4] = {r.x, r.y, r.z, r.w}, qq[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          g_rew[k] = (double)rr[k] + a.gamma * g_rew[k];
          g_pen[k] = (double)qq[k] + a.gamma * g_pen[k];
        }
#pragma unroll
        for (int i = 0; i < A; ++i) {
          const double w = a.weights ? (double)__ldg(a.weights + i) : 1.0;
          st_stream_f4(a.G + ((int64_t)t * A + i) * ld + e0,
                       make_float4((float)(w * g_rew[0] - g_pen[0]), (float)(w * g_rew[1] - g_pen[1]),
                                   (float)(w * g_rew[2] - g_pen[2]), (float)(w * g_rew[3] - g_pen[3])));
        }
      }
    }
  }

  // Block partials of the statistics the meta-agent's lambda update consumes (meta_agent.py:32-36)
  // -- the only quantities that ever cross GPUs.  Padding lanes are masked out here.
  if (a.partials) {
    __shared__ double s_red[kRolloutThreads / 32];
    double* out = a.partials + (int64_t)blockIdx.x * stats_len(A, A);
    double v_rew = 0.0, v_pen = 0.0;
    bool valid[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      valid[k] = live && (e0 + k < a.n_envs);
      v_rew += valid[k] ? s_rew[k] : 0.0;
      v_pen += valid[k] ? s_pen[k] : 0.0;
    }
    const double b_rew = block_sum<kRolloutThreads>(v_rew, s_red);
    const double b_pen = block_sum<kRolloutThreads>(v_pen, s_red);
#pragma unroll      // keep cnt[] statically indexed: a rolled loop would push the counters into local memory
    for (int i = 0; i < A; ++i) {
      double c = 0.0, viol = 0.0;
      const double thr = a.thresholds ? __ldg(a.thresholds + i) : 0.0;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const double ck = (double)((cnt[i] >> (8 * k)) & 0xFFu);
        c += valid[k] ? ck : 0.0;
        viol += (valid[k] && a.thresholds && ck > thr) ? 1.0 : 0.0;
      }
      const double bc = block_sum<kRolloutThreads>(c, s_red);
      const double bv = block_sum<kRolloutThreads>(viol, s_red);
      if (threadIdx.x == 0) {
        const double w = a.weights ? (double)__ldg(a.weights + i) : 1.0;
        out[i] = bc;
        out[A + i] = bv;
        out[2 * A + i] = w * b_rew;
        out[3 * A + i] = w * b_rew - b_pen;
      }
    }
    if (threadIdx.x == 0) out[4 * A] = 0.0;           // count is filled by the finalize kernel
  }
}

int launch_coverage_rollout(int A, const CoverageRolloutArgs& a, unsigned grid, cudaStream_t s) {
  const size_t smem = (size_t)(a.lut_len + 1) * sizeof(float);
  return dispatch<1, 32>(A, [&](auto kA) {
    coverage_rollout_kernel<kA><<<grid, kRolloutThreads, smem, s>>>(a);
    SMARL_CUDA(cudaGetLastError());
    return SMARL_OK;
  });
}
#endif

#if SMARL_TU_IS(2)
// state <- start and rebuild the float observation (coverage.py:45-52, congestion.py:39-47).
__global__ void grid_reset_kernel(const uint8_t* __restrict__ start_x, const uint8_t* __restrict__ start_y,
                                  uint8_t* __restrict__ pos_x, uint8_t* __restrict__ pos_y,
                                  float* __restrict__ obs, int64_t n_groups, int64_t ld) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_groups) return;
  const int64_t off = (int64_t)blockIdx.y * ld + g * 4;
  const uint32_t xw = ld_stream_u32(start_x + off), yw = ld_stream_u32(start_y + off);
  st_stream_u32(pos_x + off, xw);
  st_stream_u32(pos_y + off, yw);
  if (obs) {
    st_stream_f4(obs + (2 * (int64_t)blockIdx.y) * ld + g * 4, bytes_to_float4(xw));
    st_stream_f4(obs + (2 * (int64_t)blockIdx.y + 1) * ld + g * 4, bytes_to_float4(yw));
  }
}

// ---------------------------------------------------------------------------------------
// Host side
// ---------------------------------------------------------------------------------------
// Lanes per env quad of the step kernel: 0 = one thread per four envs (this file), 2 / 4 = lane-cooperative
// kernel (coverage_coop.cu).  Crossover measured on B200 (profiles/r02); smarl_set_kernel_variant overrides it.
static int coverage_coop_lanes(int A) {
  if (A < 9) return 0;
  const int forced = kernel_variant(SMARL_ENV_COVERAGE);
  if (forced >= 0) return forced;
  return A >= 22 ? 2 : 0;       // A = 20: 0.76 vs 0.75 (tie), A = 24: 0.66 -> 0.71, A = 32: 0.58 -> 0.65 of the HBM peak, closed loop
}

#endif

}  // namespace smarl

using namespace smarl;

#if SMARL_TU_IS(2)
extern "C" int smarl_grid_reset(const uint8_t* start_x, const uint8_t* start_y, uint8_t* pos_x,
                                uint8_t* pos_y, float* obs, int32_t n_agents, int64_t n_envs,
                                int64_t ld, smarl_stream_t stream) {
  if (int rc = check_layout(n_envs, ld)) return rc;
  SMARL_REQUIRE(start_x && start_y && pos_x && pos_y, "null state pointer");
  SMARL_REQUIRE(n_agents >= 1 && n_agents <= SMARL_MAX_AGENTS, "n_agents=%d outside 1..32", n_agents);
  SMARL_REQUIRE(aligned16(start_x) && aligned16(start_y) && aligned16(pos_x) && aligned16(pos_y) &&
                    aligned16(obs), "pointers must be 16-byte aligned");
  const int64_t n_groups = (n_envs + 3) / 4;
  dim3 grid((unsigned)((n_groups + 255) / 256), (unsigned)n_agents);
  grid_reset_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(start_x, start_y, pos_x, pos_y, obs,
                                                            n_groups, ld);
  SMARL_CUDA(cudaGetLastError());
  return SMARL_OK;
}

extern "C" int smarl_coverage_step(const SmarlCoverageParams* p, uint8_t* pos_x, uint8_t* pos_y,
                                   const uint8_t* actions, float* obs, float* reward, uint8_t* cost,
                                   uint8_t* done, const double* lambdas, float* penalty,
                                   int64_t n_envs, int64_t ld, smarl_stream_t stream) {
  if (int rc = check_coverage(p)) return rc;
  if (int rc = check_layout(n_envs, ld)) return rc;
  SMARL_REQUIRE(pos_x && pos_y && actions && reward && cost, "null required pointer");
  SMARL_REQUIRE((lambdas == nullptr) == (penalty == nullptr), "lambdas and penalty go together");
  SMARL_REQUIRE(aligned16(pos_x) && aligned16(pos_y) && aligned16(actions) && aligned16(obs) &&
                    aligned16(reward) && aligned16(cost) && aligned16(done) && aligned16(penalty),
                "pointers must be 16-byte aligned");
  CoverageStepArgs a;
  a.pos_x = pos_x; a.pos_y = pos_y; a.actions = actions; a.obs = obs; a.reward = reward;
  a.cost = cost; a.done = done; a.lambdas = lambdas; a.penalty = penalty;
  a.lut = p->lut; a.weights = p->weights;
  a.n_groups = (n_envs + 3) / 4; a.ld = ld; a.size = p->size; a.lut_len = p->lut_len;
  a.reward_rows = p->reward_rows == 1 ? 1 : 0;
  {
    // positions (2 B per agent and env) are re-read by the next step: keep them in L2 when they fit comfortably
    static const char* env_keep = getenv("SMARL_KEEP_POS");
    const int64_t pos_bytes = 2 * (int64_t)p->n_agents * n_envs;
    a.keep_pos = env_keep ? atoi(env_keep) : (pos_bytes <= (48ll << 20) ? 1 : 0);
  }
  if ((int64_t)(2 * p->n_agents + 1) * ld >= (1ll << 32)) {
    set_error("(2A+1)*ld = %lld exceeds 32-bit element offsets; split the env batch", (long long)((2 * p->n_agents + 1) * ld));
    return SMARL_EUNSUPPORTED;
  }
  if (const int lanes = coverage_coop_lanes(p->n_agents))
    return launch_coverage_coop_step(p->n_agents, lanes, pos_x, pos_y, actions, obs, reward, cost, done, lambdas, penalty,
                                     p->lut, p->weights, a.n_groups, ld, p->size, p->lut_len, a.reward_rows,
                                     (cudaStream_t)stream);
  const unsigned grid = (unsigned)((a.n_groups + kStepThreads - 1) / kStepThreads);
  if (int rc = launch_coverage_step(p->n_agents, a, grid, (cudaStream_t)stream)) return rc;
  return SMARL_OK;
}

extern "C" int smarl_coverage_rollout(const SmarlCoverageParams* p, const SmarlAccounting* acc,
                                      const uint8_t* start_x, const uint8_t* start_y,
                                      const uint8_t* actions, const double* lambdas,
                                      uint8_t* final_x, uint8_t* final_y, float* R, float* modR,
                                      int32_t* C, float* G, float* g_scratch, double* stats,
                                      double* stats_scratch, int64_t n_envs, int64_t ld,
                                      smarl_stream_t stream) {
  if (int rc = check_coverage(p)) return rc;
  if (int rc = check_layout(n_envs, ld)) return rc;
  if (int rc = check_accounting(acc, 255, 2, G, stats, stats_scratch)) return rc;
  SMARL_REQUIRE(start_x && start_y && actions && R && modR && C, "null required pointer");
  SMARL_REQUIRE(acc->g_mode != 1 || g_scratch, "g_mode 1 needs g_scratch [2][T][ld]");
  SMARL_REQUIRE(aligned16(start_x) && aligned16(start_y) && aligned16(actions) && aligned16(final_x) &&
                    aligned16(final_y) && aligned16(R) && aligned16(modR) && aligned16(C) &&
                    aligned16(G) && aligned16(g_scratch), "pointers must be 16-byte aligned");
  CoverageRolloutArgs a;
  a.start_x = start_x; a.start_y = start_y; a.actions = actions; a.lambdas = lambdas;
  a.final_x = final_x; a.final_y = final_y; a.R = R; a.modR = modR; a.C = C; a.G = G;
  a.g_scratch = g_scratch; a.partials = stats_scratch; a.thresholds = acc->thresholds;
  a.lut = p->lut; a.weights = p->weights; a.gamma = acc->gamma;
  a.n_groups = (n_envs + 3) / 4; a.n_envs = n_envs; a.ld = ld; a.size = p->size;
  a.lut_len = p->lut_len; a.n_steps = acc->n_steps; a.g_mode = acc->g_mode;
  const unsigned grid = (unsigned)((a.n_groups + kRolloutThreads - 1) / kRolloutThreads);
  if (int rc = launch_coverage_rollout(p->n_agents, a, grid, (cudaStream_t)stream)) return rc;
  if (stats)
    return launch_stats_finalize(stats_scratch, grid, p->n_agents, p->n_agents, n_envs, stats,
                                 (cudaStream_t)stream);
  return SMARL_OK;
}
#endif
