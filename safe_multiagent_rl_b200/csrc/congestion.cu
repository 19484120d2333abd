// Congestion on sm_100a: step kernel (+ fused rollout).  Same thread mapping and SoA layout as
// coverage.cu: one thread owns four consecutive envs, one byte per env in every state word.
#include "congestion.cuh"
#include "stats.cuh"

// Built as several translation units (build.py compiles this file once per SMARL_TU value) so the
// 32 agent-count instantiations of each kernel compile in parallel:
//   0,1,2 step kernel noise mode 0/1/2   3,4,5 rollout kernel mode 0/1/2   6 C entry points

namespace smarl {

constexpr int kCongThreads = 128;
// Both Congestion kernels are issue / latency-bound, so up to 8 agents the register budget is capped for more
// resident CTAs: 80 per thread in the step kernel (6 CTAs of 128; with the byte-SIMD class counting a tighter cap
// spills more than the occupancy returns: config 2 closed loop 5.38 ms at 64 registers, 5.29 at 72, 5.18 at 80) and
// 128 in the rollout kernel (8 CTAs of 64: rollout 5.28 -> 4.39 ms when introduced).  Larger agent counts would
// spill hundreds of bytes and get slower, so they keep the compiler's choice.
constexpr int cong_step_min_blocks(int A) { return A <= 8 ? 6 : 0; }   // 0 = unspecified (1 would lift the register heuristic to 255)
constexpr int cong_min_blocks(int A) { return A <= 8 ? 8 : (A <= 12 ? 5 : 0); }   // A = 9..12: 168 registers (A = 12 fused +9 %)

// ---------------------------------------------------------------------------------------
// Fused open-loop episode (main.py:28-57 minus the policy nets, buffer.py:30-39,
// meta_agent.py:18-30, agent.py:129-132 / :200-206).  Positions stay in registers; the
// per-agent discounted sums (A x 4 envs, f64) live in shared memory, indexed
// [agent][env lane][thread] so that every access is conflict-free.
// ---------------------------------------------------------------------------------------
// (CongestionRolloutArgs lives in congestion.cuh: the cooperative rollout kernel of congestion_coop.cu shares it)

#if SMARL_TU_IS(0) || SMARL_TU_IS(1) || SMARL_TU_IS(2)
template <int A, int MODE>
__global__ void __launch_bounds__(kCongThreads, cong_step_min_blocks(A)) congestion_step_kernel(const CongestionStepArgs a) {
  pdl_prologue();   // programmatic dependent launch: the previous grid has completed past this point (common.cuh)
  const int64_t g = (int64_t)blockIdx.x * kCongThreads + threadIdx.x;
  if (g >= a.n_groups) return;
  // 32-bit element offsets (the host checks (2A+1) * ld < 2^32): one add per row and one wide add per
  // access instead of a 64-bit multiply-add chain (a sixth of the kernel's instructions before).
  const uint32_t ld = (uint32_t)a.ld;
  const uint32_t e0 = (uint32_t)g * 4u;

  uint32_t xw[A], yw[A], aw[A], mw[A];
  {
    uint32_t off = e0;
#pragma unroll
    for (int i = 0; i < A; ++i, off += ld) {
      xw[i] = ld_stream_u32(a.pos_x + off);
      yw[i] = ld_stream_u32(a.pos_y + off);
      aw[i] = ld_stream_u32(a.actions + off);
      if (MODE == 1) mw[i] = ld_stream_u32(a.moves + off);
      if (MODE == 0) mw[i] = aw[i];
    }
  }
  if (MODE == 2)
    congestion_noise_moves<A>(aw, mw, a.seed, a.keep_threshold, a.env_offset + (int64_t)g * 4, (uint32_t)a.t,
                              a.episode + (a.episode_dev ? __ldg(a.episode_dev) : 0u));

  uint32_t dcw[A];
  congestion_transition<A>(xw, yw, mw, dcw, (uint32_t)a.size * 0x01010101u);
  {
    uint32_t off = e0, obs_off = e0;
#pragma unroll
    for (int i = 0; i < A; ++i, off += ld, obs_off += 2u * ld) {
      st_stream_u32(a.pos_x + off, xw[i]);
      st_stream_u32(a.pos_y + off, yw[i]);
      if (MODE != 1 && a.moves) st_stream_u32(a.moves + off, mw[i]);
      if (a.done) st_stream_u32(a.done + off, 0u);                       // congestion.py:103-104
      if (a.obs) {
        st_stream_f4(a.obs + obs_off, bytes_to_float4(xw[i]));
        st_stream_f4(a.obs + (obs_off + ld), bytes_to_float4(yw[i]));
      }
    }
  }

  uint32_t conw[A];
  const uint32_t org = congestion_classes<A, kSimdClassAgentsStep>(xw, yw, dcw, aw, conw);
  // congestion.py:93-100: cost = max(0, A // 3 - #agents on node (0,0)) per env lane
  const int c0 = max(0, A / 3 - (int)(org & 0xFFu)), c1 = max(0, A / 3 - (int)((org >> 8) & 0xFFu)),
            c2 = max(0, A / 3 - (int)((org >> 16) & 0xFFu)), c3 = max(0, A / 3 - (int)(org >> 24));
  st_stream_i4(a.cost + e0, make_int4(c0, c1, c2, c3));
  if (a.penalty) {                                                       // meta_agent.py:21-22
    const double lam = __ldg(a.lambdas);
    st_stream_f4(a.penalty + e0, make_float4((float)(lam * c0), (float)(lam * c1), (float)(lam * c2),
                                             (float)(lam * c3)));
  }
  const int W = a.size + 1;
  if (a.wait_reward) {
    uint32_t off = e0;
#pragma unroll
    for (int i = 0; i < A; ++i, off += ld)
      st_stream_f4(a.reward + off, congestion_reward4<true>(aw[i], conw[i], xw[i], yw[i], a.demand, W, a.wait_reward));
  } else {
    uint32_t off = e0;
#pragma unroll 1
    for (int i = 0; i < A; ++i, off += ld)
      st_stream_f4(a.reward + off, congestion_reward4<false>(aw[i], conw[i], xw[i], yw[i], a.demand, W, nullptr));
  }
}

template <int M>
int launch_congestion_step(int A, const CongestionStepArgs& a, unsigned grid, cudaStream_t s) {
  return dispatch<1, 32>(A, [&](auto kA) {
    SMARL_CUDA(launch_pdl(congestion_step_kernel<kA, M>, grid, kCongThreads, 0, s, a));
    SMARL_CUDA(cudaGetLastError());
    return SMARL_OK;
  });
}
#endif
#if SMARL_TU_IS(0)
template int launch_congestion_step<0>(int, const CongestionStepArgs&, unsigned, cudaStream_t);
#endif
#if SMARL_TU_IS(1)
template int launch_congestion_step<1>(int, const CongestionStepArgs&, unsigned, cudaStream_t);
#endif
#if SMARL_TU_IS(2)
template int launch_congestion_step<2>(int, const CongestionStepArgs&, unsigned, cudaStream_t);
#endif

#if SMARL_TU_IS(3) || SMARL_TU_IS(4) || SMARL_TU_IS(5)

template <int A, int MODE>
__global__ void __launch_bounds__(kCongRollThreads, cong_min_blocks(A)) congestion_rollout_kernel(const CongestionRolloutArgs a) {
  extern __shared__ double s_acc[];                      // [A][4][kCongRollThreads]
  __shared__ double s_red[kCongRollThreads / 32];
  const int tid = threadIdx.x;
  const int64_t g = (int64_t)blockIdx.x * kCongRollThreads + tid;
  const bool live = g < a.n_groups;
  const int64_t e0 = (live ? g : 0) * 4;
  const int64_t ld = a.ld;
  const int T = a.n_steps;
  const int W = a.size + 1;
  const uint32_t size4 = (uint32_t)a.size * 0x01010101u;
  const double lam = a.lambdas ? __ldg(a.lambdas) : 0.0;
  const uint32_t episode = a.episode + ((MODE == 2 && a.episode_dev) ? __ldg(a.episode_dev) : 0u);

  uint32_t xw[A], yw[A];
#pragma unroll
  for (int i = 0; i < A; ++i) {
    xw[i] = ld_stream_u32(a.start_x + i * ld + e0);
    yw[i] = ld_stream_u32(a.start_y + i * ld + e0);
#pragma unroll
    for (int k = 0; k < 4; ++k) s_acc[(i * 4 + k) * kCongRollThreads + tid] = 0.0;
  }
  double s_pen[4] = {0, 0, 0, 0};
  int csum[4] = {0, 0, 0, 0};
  double disc = 1.0;

  for (int t = 0; t < T; ++t) {
    uint32_t aw[A], mw[A];
    {
      const uint8_t* act_t = a.actions + (int64_t)t * A * ld;            // uniform; per-thread offsets stay 32-bit
      const uint8_t* mov_t = MODE == 1 ? a.moves + (int64_t)t * A * ld : nullptr;
      uint32_t off = (uint32_t)e0;
#pragma unroll
      for (int i = 0; i < A; ++i, off += (uint32_t)ld) {
        aw[i] = ld_stream_u32(act_t + off);
        if (MODE == 1) mw[i] = ld_stream_u32(mov_t + off);
        if (MODE == 0) mw[i] = aw[i];
      }
    }
    if (MODE == 2) congestion_noise_moves<A>(aw, mw, a.seed, a.keep_threshold, a.env_offset + e0, (uint32_t)t, episode);
    uint32_t dcw[A], conw[A];
    congestion_transition<A>(xw, yw, mw, dcw, size4);
    const uint32_t org = congestion_classes<A, kSimdClassAgentsRollout>(xw, yw, dcw, aw, conw);
    const int cost[4] = {max(0, A / 3 - (int)(org & 0xFFu)), max(0, A / 3 - (int)((org >> 8) & 0xFFu)),
                         max(0, A / 3 - (int)((org >> 16) & 0xFFu)), max(0, A / 3 - (int)(org >> 24))};
    float pen[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      pen[k] = (float)(lam * cost[k]);                  // the step kernel publishes the penalty as f32
      s_pen[k] += disc * (double)pen[k];
      csum[k] += cost[k];
    }
    if (a.g_mode == 1 && live) st_stream_f4(a.g_scratch + (int64_t)t * ld + e0, make_float4(pen[0], pen[1], pen[2], pen[3]));
#pragma unroll
    for (int i = 0; i < A; ++i) {
      const float4 r4 = a.wait_reward ? congestion_reward4<true>(aw[i], conw[i], xw[i], yw[i], a.demand, W, a.wait_reward)
                                      : congestion_reward4<false>(aw[i], conw[i], xw[i], yw[i], a.demand, W, nullptr);
      const float r[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) s_acc[(i * 4 + k) * kCongRollThreads + tid] += disc * (double)r[k];
      if (a.g_mode == 1 && live) {
        st_stream_f4(a.G + ((int64_t)t * A + i) * ld + e0, make_float4(r[0], r[1], r[2], r[3]));
      } else if (a.g_mode == 2 && live) {               // agent.py:129-132
        st_stream_f4(a.G + ((int64_t)t * A + i) * ld + e0,
                     make_float4((float)(disc * ((double)r[0] - (double)pen[0])), (float)(disc * ((double)r[1] - (double)pen[1])),
                                 (float)(disc * ((double)r[2] - (double)pen[2])), (float)(disc * ((double)r[3] - (double)pen[3]))));
      }
    }
    disc *= a.gamma;
  }

  bool valid[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) valid[k] = live && (e0 + k < a.n_envs);
  double* out = a.partials ? a.partials + (int64_t)blockIdx.x * stats_len(A, 1) : nullptr;
  if (live) {
    st_stream_i4(a.C + e0, make_int4(csum[0], csum[1], csum[2], csum[3]));
  }
  if (live) {   // unrolled: dynamic indices would push the position words into local memory for the whole episode
#pragma unroll
    for (int i = 0; i < A; ++i) {
      if (a.final_x) st_stream_u32(a.final_x + i * ld + e0, xw[i]);
      if (a.final_y) st_stream_u32(a.final_y + i * ld + e0, yw[i]);
    }
  }
#pragma unroll 1
  for (int i = 0; i < A; ++i) {
    double raw[4], mod[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      raw[k] = s_acc[(i * 4 + k) * kCongRollThreads + tid];
      mod[k] = raw[k] - s_pen[k];
    }
    if (live) {
      st_stream_f4(a.R + i * ld + e0, make_float4((float)raw[0], (float)raw[1], (float)raw[2], (float)raw[3]));
      st_stream_f4(a.modR + i * ld + e0, make_float4((float)mod[0], (float)mod[1], (float)mod[2], (float)mod[3]));
    }
    if (out) {
      double v_raw = 0.0, v_mod = 0.0;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        v_raw += valid[k] ? raw[k] : 0.0;
        v_mod += valid[k] ? mod[k] : 0.0;
      }
      const double b_raw = block_sum<kCongRollThreads>(v_raw, s_red);
      const double b_mod = block_sum<kCongRollThreads>(v_mod, s_red);
      if (tid == 0) {
        out[2 + i] = b_raw;
        out[2 + A + i] = b_mod;
      }
    }
  }
  if (out) {
    const double thr = a.thresholds ? __ldg(a.thresholds) : 0.0;
    double c = 0.0, viol = 0.0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      c += valid[k] ? (double)csum[k] : 0.0;
      viol += (valid[k] && a.thresholds && (double)csum[k] > thr) ? 1.0 : 0.0;
    }
    const double bc = block_sum<kCongRollThreads>(c, s_red);
    const double bv = block_sum<kCongRollThreads>(viol, s_red);
    if (tid == 0) {
      out[0] = bc;
      out[1] = bv;
      out[2 + 2 * A] = 0.0;
    }
  }

  if (a.g_mode == 1 && live) {                          // agent.py:200-206, in place over the stored rewards
#pragma unroll
    for (int i = 0; i < A; ++i)
#pragma unroll
      for (int k = 0; k < 4; ++k) s_acc[(i * 4 + k) * kCongRollThreads + tid] = 0.0;
    for (int t = T - 1; t >= 0; --t) {
      const float4 q = ld_f4(a.g_scratch + (int64_t)t * ld + e0);
      const float qq[4] = {q.x, q.y, q.z, q.w};
#pragma unroll 4
      for (int i = 0; i < A; ++i) {
        float* gp = a.G + ((int64_t)t * A + i) * ld + e0;
        const float4 r = ld_f4(gp);
        const float rr[4] = {r.x, r.y, r.z, r.w};
        float o[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          double& run = s_acc[(i * 4 + k) * kCongRollThreads + tid];
          run = ((double)rr[k] - (double)qq[k]) + a.gamma * run;
          o[k] = (float)run;
        }
        st_stream_f4(gp, make_float4(o[0], o[1], o[2], o[3]));
      }
    }
  }
}

template <int M>
int launch_congestion_rollout(int A, const CongestionRolloutArgs& a, unsigned grid, cudaStream_t s) {
  const size_t smem = sizeof(double) * 4 * kCongRollThreads * (size_t)A;
  return dispatch<1, 32>(A, [&](auto kA) {
    auto kern = congestion_rollout_kernel<kA, M>;
    if (smem + 64 > 48 * 1024)   // + the static reduction buffer
      SMARL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, kCongRollThreads, smem, s>>>(a);
    SMARL_CUDA(cudaGetLastError());
    return SMARL_OK;
  });
}
#endif
#if SMARL_TU_IS(3)
template int launch_congestion_rollout<0>(int, const CongestionRolloutArgs&, unsigned, cudaStream_t);
#endif
#if SMARL_TU_IS(4)
template int launch_congestion_rollout<1>(int, const CongestionRolloutArgs&, unsigned, cudaStream_t);
#endif
#if SMARL_TU_IS(5)
template int launch_congestion_rollout<2>(int, const CongestionRolloutArgs&, unsigned, cudaStream_t);
#endif

#if SMARL_TU_IS(6)
// Lanes per env quad of the step kernel: 0 = one thread per four envs (this file), 2 / 4 = lane-cooperative
// scan kernel (congestion_coop.cu).  Crossover measured on B200 (profiles/r02); smarl_set_kernel_variant overrides.
static int congestion_coop_lanes(int A) {
  if (A < 9) return 0;
  const int forced = kernel_variant(SMARL_ENV_CONGESTION);
  if (forced >= 0) return forced;
  return A >= 12 ? 4 : 0;       // closed loop, of the HBM peak: A = 12 0.63 -> 0.68, 16 0.56 -> 0.65, 20 0.38 -> 0.60, 32 0.30 -> 0.48
}

// The fused rollout: 0 = one thread per four envs (this file), 4 = lane-cooperative rollout (congestion_coop.cu; a
// forced 2 also takes it, the rollout is built for four lanes only).  B200, 2^20 envs, T = 20 (profiles/r02).
static int congestion_coop_rollout_lanes(int A) {
  if (A < 9) return 0;
  const int forced = kernel_variant(SMARL_ENV_CONGESTION);
  if (forced >= 0) return forced ? 4 : 0;
  return A >= 12 ? 4 : 0;       // fused ms per 2^20 envs x T = 20: A = 12 1.12 -> 1.09, 16 1.75 -> 1.55, 24 3.90 -> 3.01, 32 9.33 -> 4.80
}

#endif

}  // namespace smarl

using namespace smarl;

#if SMARL_TU_IS(6)
extern "C" int smarl_congestion_step(const SmarlCongestionParams* p, uint8_t* pos_x, uint8_t* pos_y,
                                     const uint8_t* actions, uint8_t* moves, float* obs, float* reward,
                                     int32_t* cost, uint8_t* done, const double* lambdas, float* penalty,
                                     int32_t t, int64_t n_envs, int64_t ld, smarl_stream_t stream) {
  if (int rc = check_congestion(p)) return rc;
  if (int rc = check_layout(n_envs, ld)) return rc;
  SMARL_REQUIRE(pos_x && pos_y && actions && reward && cost, "null required pointer");
  SMARL_REQUIRE(p->noise_mode != 1 || moves, "noise_mode 1 needs the recorded moves");
  SMARL_REQUIRE((lambdas == nullptr) == (penalty == nullptr), "lambdas and penalty go together");
  SMARL_REQUIRE((2 * (int64_t)p->n_agents + 1) * ld < (1ll << 32),
                "(2A+1)*ld = %lld exceeds 32-bit element offsets; split the env batch",
                (long long)((2 * (int64_t)p->n_agents + 1) * ld));
  SMARL_REQUIRE(aligned16(pos_x) && aligned16(pos_y) && aligned16(actions) && aligned16(moves) &&
                    aligned16(obs) && aligned16(reward) && aligned16(cost) && aligned16(done) &&
                    aligned16(penalty), "pointers must be 16-byte aligned");
  CongestionStepArgs a;
  a.pos_x = pos_x; a.pos_y = pos_y; a.actions = actions; a.moves = moves; a.obs = obs;
  a.reward = reward; a.cost = cost; a.done = done; a.lambdas = lambdas; a.penalty = penalty;
  a.demand = p->demand; a.wait_reward = p->wait_reward; a.keep_threshold = p->keep_threshold; a.seed = p->seed;
  a.env_offset = p->env_offset; a.n_groups = (n_envs + 3) / 4; a.ld = ld; a.size = p->size; a.t = t;
  a.episode = p->episode; a.episode_dev = p->episode_dev;
  const unsigned grid = (unsigned)((a.n_groups + kCongThreads - 1) / kCongThreads);
  cudaStream_t s = (cudaStream_t)stream;
  const int lanes = congestion_coop_lanes(p->n_agents);
  return dispatch<0, 2>(p->noise_mode, [&](auto m) {
    return lanes ? launch_congestion_coop_step<m>(p->n_agents, lanes, a, s) : launch_congestion_step<m>(p->n_agents, a, grid, s);
  }, "bad noise_mode %d");
}

extern "C" int smarl_congestion_rollout(const SmarlCongestionParams* p, const SmarlAccounting* acc,
                                        const uint8_t* start_x, const uint8_t* start_y,
                                        const uint8_t* actions, const uint8_t* moves,
                                        const double* lambdas, uint8_t* final_x, uint8_t* final_y,
                                        float* R, float* modR, int32_t* C, float* G, float* g_scratch,
                                        double* stats, double* stats_scratch, int64_t n_envs,
                                        int64_t ld, smarl_stream_t stream) {
  if (int rc = check_congestion(p)) return rc;
  if (int rc = check_layout(n_envs, ld)) return rc;
  if (int rc = check_accounting(acc, INT32_MAX, 2, G, stats, stats_scratch)) return rc;
  SMARL_REQUIRE(start_x && start_y && actions && R && modR && C, "null required pointer");
  SMARL_REQUIRE(p->noise_mode != 1 || moves, "noise_mode 1 needs the recorded moves [T][A][ld]");
  SMARL_REQUIRE(acc->g_mode != 1 || g_scratch, "g_mode 1 needs g_scratch");
  SMARL_REQUIRE((int64_t)p->n_agents * ld < (1ll << 32), "A*ld = %lld exceeds 32-bit element offsets; split the env batch",
                (long long)((int64_t)p->n_agents * ld));
  SMARL_REQUIRE(aligned16(start_x) && aligned16(start_y) && aligned16(actions) && aligned16(moves) &&
                    aligned16(final_x) && aligned16(final_y) && aligned16(R) && aligned16(modR) &&
                    aligned16(C) && aligned16(G) && aligned16(g_scratch), "pointers must be 16-byte aligned");
  CongestionRolloutArgs a;
  a.start_x = start_x; a.start_y = start_y; a.actions = actions; a.moves = moves; a.lambdas = lambdas;
  a.final_x = final_x; a.final_y = final_y; a.R = R; a.modR = modR; a.C = C; a.G = G;
  a.g_scratch = g_scratch; a.partials = stats_scratch; a.thresholds = acc->thresholds;
  a.demand = p->demand; a.wait_reward = p->wait_reward; a.gamma = acc->gamma; a.keep_threshold = p->keep_threshold;
  a.seed = p->seed;
  a.env_offset = p->env_offset; a.n_groups = (n_envs + 3) / 4; a.n_envs = n_envs; a.ld = ld;
  a.size = p->size; a.n_steps = acc->n_steps; a.g_mode = acc->g_mode;
  a.episode = p->episode; a.episode_dev = p->episode_dev;
  const unsigned grid = (unsigned)((a.n_groups + kCongRollThreads - 1) / kCongRollThreads);
  cudaStream_t s = (cudaStream_t)stream;
  const bool coop = congestion_coop_rollout_lanes(p->n_agents) != 0;
  unsigned rows = grid;                                 // CTAs launched = rows of stats partials
  if (int rc = dispatch<0, 2>(p->noise_mode, [&](auto m) {
        return coop ? launch_congestion_coop_rollout<m>(p->n_agents, a, &rows, s)
                    : launch_congestion_rollout<m>(p->n_agents, a, grid, s);
      }, "bad noise_mode %d"))
    return rc;
  if (stats)
    return launch_stats_finalize(stats_scratch, rows, p->n_agents, 1, n_envs, stats, s);
  return SMARL_OK;
}
#endif
