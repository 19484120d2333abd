// CoverageContinuous / CoverageDiscretized on sm_100a (float64 positions).  One thread owns one
// env; all arrays agent-major SoA.  Compiled with -fmad=false: positions follow the reference's
// float64 operations one by one (bit-exact); the pair penalty uses a multiply where the reference's
// numpy scalar power calls libm pow (<= 1 ulp per term, invisible after the f32 rounding of rewards).
#include "coverage_float.cuh"
#include "stats.cuh"

namespace smarl {

#if SMARL_TU_IS(0) || SMARL_TU_IS(1)
template <int A, int MODE>
__global__ void __launch_bounds__(kCovFThreads) coverage_float_step_kernel(const CoverageFloatArgs a) {
  pdl_prologue();   // programmatic dependent launch: the previous grid has completed past this point (common.cuh)
  const int64_t e = (int64_t)blockIdx.x * kCovFThreads + threadIdx.x;
  if (e >= a.n_envs) return;
  const int64_t ld = a.ld;
  double px[A], py[A], cost[A];
  double pen = 0.0, rew;
#pragma unroll
  for (int i = 0; i < A; ++i) {
    px[i] = a.pos_x[i * ld + e];
    py[i] = a.pos_y[i * ld + e];
  }
  const void* act = MODE == 0 ? static_cast<const void*>(static_cast<const float*>(a.actions) + e)
                              : static_cast<const void*>(static_cast<const uint8_t*>(a.actions) + e);
  coverage_float_env_step<A, MODE>(px, py, act, ld, a, cost, rew);
#pragma unroll
  for (int i = 0; i < A; ++i) {
    a.pos_x[i * ld + e] = px[i];
    a.pos_y[i * ld + e] = py[i];
    a.cost[i * ld + e] = (float)cost[i];
    if (a.done) a.done[i * ld + e] = 0;                                 // :97-98
    if (a.obs) {
      a.obs[(2 * i) * ld + e] = (float)px[i];
      a.obs[(2 * i + 1) * ld + e] = (float)py[i];
    }
    if (a.penalty) pen += __ldg(a.lambdas + i) * cost[i];               // meta_agent.py:21-22
    const double w = a.weights ? (double)__ldg(a.weights + i) : 1.0;
    a.reward[i * ld + e] = (float)__dmul_rn(rew, w);
  }
  if (a.penalty) a.penalty[e] = (float)pen;
}

template <int M>
int launch_coverage_float_step(int A, const CoverageFloatArgs& a, unsigned grid, cudaStream_t s) {
  return dispatch<1, 32>(A, [&](auto kA) {
    SMARL_CUDA(launch_pdl(coverage_float_step_kernel<kA, M>, grid, kCovFThreads, 0, s, a));
    SMARL_CUDA(cudaGetLastError());
    return SMARL_OK;
  });
}
#endif
#if SMARL_TU_IS(0)
template int launch_coverage_float_step<0>(int, const CoverageFloatArgs&, unsigned, cudaStream_t);
#endif
#if SMARL_TU_IS(1)
template int launch_coverage_float_step<1>(int, const CoverageFloatArgs&, unsigned, cudaStream_t);
#endif

#if SMARL_TU_IS(3) || SMARL_TU_IS(4)
// Fused open-loop episode of the float-position Coverage envs: positions, per-agent cost sums and the
// (S_rew, S_pen) discounted sums stay in registers; reward_a = w_a * rew, so one pair serves every agent.
// CAP: 64 registers (8 CTAs per SM) for A <= 4 on batches >= 2^18 envs (2^20 envs: Continuous 1.69 -> 1.26 ms, Discretized
// 2.34 -> 2.00 ms per batch); a one-wave batch of 65 536 envs is latency-bound per thread and loses 8 % to the spills.
template <int A, int MODE, bool CAP>
__global__ void __launch_bounds__(kCovFThreads, (CAP ? 8 : 0)) coverage_float_rollout_kernel(const CoverageFloatRolloutArgs r) {
  __shared__ double s_red[kCovFThreads / 32];
  const CoverageFloatArgs& a = r.env;
  const int64_t eg = (int64_t)blockIdx.x * kCovFThreads + threadIdx.x;
  const bool live = eg < a.n_envs;
  const int64_t e = live ? eg : 0;
  const int64_t ld = a.ld;
  const int T = r.n_steps;
  constexpr int kRows = MODE == 0 ? 2 * A : A;
  double px[A], py[A], csum[A], lam[A];
#pragma unroll
  for (int i = 0; i < A; ++i) {
    px[i] = a.pos_x[i * ld + e];
    py[i] = a.pos_y[i * ld + e];
    csum[i] = 0.0;
    lam[i] = a.lambdas ? __ldg(a.lambdas + i) : 0.0;
  }
  double s_rew = 0.0, s_pen = 0.0, disc = 1.0;
  for (int t = 0; t < T; ++t) {
    const void* act = MODE == 0
        ? static_cast<const void*>(static_cast<const float*>(a.actions) + (int64_t)t * kRows * ld + e)
        : static_cast<const void*>(static_cast<const uint8_t*>(a.actions) + (int64_t)t * kRows * ld + e);
    double cost[A], rew, pen = 0.0;
    coverage_float_env_step<A, MODE>(px, py, act, ld, a, cost, rew);
#pragma unroll
    for (int i = 0; i < A; ++i) {
      csum[i] += (double)(float)cost[i];             // the step kernel publishes costs as f32
      pen += lam[i] * cost[i];
    }
    const float pf = (float)pen;
    s_rew += disc * rew;
    s_pen += disc * (double)pf;
    if (r.g_mode == 1 && live) {
      r.g_scratch[(int64_t)t * ld + e] = (float)rew;
      r.g_scratch[((int64_t)T + t) * ld + e] = pf;
    } else if (r.g_mode == 2 && live) {
#pragma unroll
      for (int i = 0; i < A; ++i) {
        const double w = a.weights ? (double)__ldg(a.weights + i) : 1.0;
        r.G[((int64_t)t * A + i) * ld + e] = (float)(disc * ((double)(float)__dmul_rn(rew, w) - (double)pf));
      }
    }
    disc *= r.gamma;
  }
  if (live) {
#pragma unroll
    for (int i = 0; i < A; ++i) {
      const double w = a.weights ? (double)__ldg(a.weights + i) : 1.0;
      if (r.final_x) r.final_x[i * ld + e] = px[i];
      if (r.final_y) r.final_y[i * ld + e] = py[i];
      r.R[i * ld + e] = (float)(w * s_rew);
      r.modR[i * ld + e] = (float)(w * s_rew - s_pen);
      r.C[i * ld + e] = (float)csum[i];
    }
  }
  if (r.partials) {
    double* out = r.partials + (int64_t)blockIdx.x * stats_len(A, A);
    const double b_rew = block_sum<kCovFThreads>(live ? s_rew : 0.0, s_red);
    const double b_pen = block_sum<kCovFThreads>(live ? s_pen : 0.0, s_red);
#pragma unroll
    for (int i = 0; i < A; ++i) {
      const double thr = r.thresholds ? __ldg(r.thresholds + i) : 0.0;
      const double c = (double)(float)csum[i];
      const double bc = block_sum<kCovFThreads>(live ? c : 0.0, s_red);
      const double bv = block_sum<kCovFThreads>((live && r.thresholds && c > thr) ? 1.0 : 0.0, s_red);
      if (threadIdx.x == 0) {
        const double w = a.weights ? (double)__ldg(a.weights + i) : 1.0;
        out[i] = bc;
        out[A + i] = bv;
        out[2 * A + i] = w * b_rew;
        out[3 * A + i] = w * b_rew - b_pen;
      }
    }
    if (threadIdx.x == 0) out[4 * A] = 0.0;
  }
  if (r.g_mode == 1 && live) {                          // agent.py:200-206
    double g_rew = 0.0, g_pen = 0.0;
    for (int t = T - 1; t >= 0; --t) {
      g_rew = (double)r.g_scratch[(int64_t)t * ld + e] + r.gamma * g_rew;
      g_pen = (double)r.g_scratch[((int64_t)T + t) * ld + e] + r.gamma * g_pen;
#pragma unroll
      for (int i = 0; i < A; ++i) {
        const double w = a.weights ? (double)__ldg(a.weights + i) : 1.0;
        r.G[((int64_t)t * A + i) * ld + e] = (float)(w * g_rew - g_pen);
      }
    }
  }
}
template <int M>
int launch_coverage_float_rollout(int A, const CoverageFloatRolloutArgs& a, unsigned grid, cudaStream_t s) {
  if (A <= 4 && a.env.n_envs >= (1 << 18))
    return dispatch<1, 4>(A, [&](auto kA) {
      coverage_float_rollout_kernel<kA, M, true><<<grid, kCovFThreads, 0, s>>>(a);
      SMARL_CUDA(cudaGetLastError());
      return SMARL_OK;
    });
  return dispatch<1, 32>(A, [&](auto kA) {
    coverage_float_rollout_kernel<kA, M, false><<<grid, kCovFThreads, 0, s>>>(a);
    SMARL_CUDA(cudaGetLastError());
    return SMARL_OK;
  });
}
#endif
#if SMARL_TU_IS(3)
template int launch_coverage_float_rollout<0>(int, const CoverageFloatRolloutArgs&, unsigned, cudaStream_t);
#endif
#if SMARL_TU_IS(4)
template int launch_coverage_float_rollout<1>(int, const CoverageFloatRolloutArgs&, unsigned, cudaStream_t);
#endif

#if SMARL_TU_IS(2)
__global__ void coverage_float_reset_kernel(const double* __restrict__ start_x, const double* __restrict__ start_y,
                                            double* __restrict__ pos_x, double* __restrict__ pos_y,
                                            float* __restrict__ obs, int A, int64_t n_envs, int64_t ld) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_envs) return;
  for (int i = 0; i < A; ++i) {
    const double x = start_x[i * ld + e], y = start_y[i * ld + e];
    pos_x[i * ld + e] = x;
    pos_y[i * ld + e] = y;
    if (obs) {
      obs[(2 * i) * ld + e] = (float)x;
      obs[(2 * i + 1) * ld + e] = (float)y;
    }
  }
}
#endif

}  // namespace smarl

using namespace smarl;

#if SMARL_TU_IS(2)
extern "C" int smarl_coverage_float_reset(const double* start_x, const double* start_y, double* pos_x,
                                          double* pos_y, float* obs, int32_t n_agents, int64_t n_envs,
                                          int64_t ld, smarl_stream_t stream) {
  if (int rc = check_layout(n_envs, ld)) return rc;
  SMARL_REQUIRE(start_x && start_y && pos_x && pos_y, "null state pointer");
  SMARL_REQUIRE(n_agents >= 1 && n_agents <= SMARL_MAX_AGENTS, "n_agents=%d outside 1..32", n_agents);
  coverage_float_reset_kernel<<<(unsigned)((n_envs + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      start_x, start_y, pos_x, pos_y, obs, n_agents, n_envs, ld);
  SMARL_CUDA(cudaGetLastError());
  return SMARL_OK;
}

extern "C" int smarl_coverage_float_step(const SmarlCoverageFloatParams* p, double* pos_x, double* pos_y,
                                         const void* actions, float* obs, float* reward, float* cost,
                                         uint8_t* done, const double* lambdas, float* penalty,
                                         int64_t n_envs, int64_t ld, smarl_stream_t stream) {
  SMARL_REQUIRE(p != nullptr, "params is NULL");
  if (int rc = check_layout(n_envs, ld)) return rc;
  SMARL_REQUIRE(p->size >= 1, "size=%d must be >= 1", p->size);
  SMARL_REQUIRE(p->mode == 0 || p->mode == 1, "bad mode %d", p->mode);
  SMARL_REQUIRE(p->mode == 0 || p->zoom > 0.0, "mode 1 needs zoom > 0");
  SMARL_REQUIRE(pos_x && pos_y && actions && reward && cost, "null required pointer");
  SMARL_REQUIRE((lambdas == nullptr) == (penalty == nullptr), "lambdas and penalty go together");
  CoverageFloatArgs a;
  coverage_float_args(p, a);
  a.pos_x = pos_x; a.pos_y = pos_y; a.actions = actions; a.obs = obs; a.reward = reward; a.cost = cost;
  a.done = done; a.lambdas = lambdas; a.penalty = penalty; a.n_envs = n_envs; a.ld = ld;
  const unsigned grid = (unsigned)((n_envs + kCovFThreads - 1) / kCovFThreads);
  return dispatch<0, 1>(p->mode, [&](auto m) { return launch_coverage_float_step<m>(p->n_agents, a, grid, (cudaStream_t)stream); },
                        "bad mode %d");
}

extern "C" int smarl_coverage_float_rollout(const SmarlCoverageFloatParams* p, const SmarlAccounting* acc,
                                            const double* start_x, const double* start_y, const void* actions,
                                            const double* lambdas, double* final_x, double* final_y, float* R,
                                            float* modR, float* C, float* G, float* g_scratch, double* stats,
                                            double* stats_scratch, int64_t n_envs, int64_t ld,
                                            smarl_stream_t stream) {
  SMARL_REQUIRE(p != nullptr, "params is NULL");
  if (int rc = check_layout(n_envs, ld)) return rc;
  SMARL_REQUIRE(p->size >= 1 && (p->mode == 0 || p->mode == 1), "bad size / mode");
  SMARL_REQUIRE(p->mode == 0 || p->zoom > 0.0, "mode 1 needs zoom > 0");
  if (int rc = check_accounting(acc, INT32_MAX, 2, G, stats, stats_scratch)) return rc;
  SMARL_REQUIRE(start_x && start_y && actions && R && modR && C, "null required pointer");
  SMARL_REQUIRE(acc->g_mode != 1 || g_scratch, "g_mode 1 needs g_scratch [2][T][ld]");
  CoverageFloatRolloutArgs r;
  CoverageFloatArgs& a = r.env;
  coverage_float_args(p, a);
  a.pos_x = const_cast<double*>(start_x); a.pos_y = const_cast<double*>(start_y); a.actions = actions;
  a.lambdas = lambdas; a.n_envs = n_envs; a.ld = ld;
  r.final_x = final_x; r.final_y = final_y; r.R = R; r.modR = modR; r.C = C; r.G = G; r.g_scratch = g_scratch;
  r.partials = stats_scratch; r.thresholds = acc->thresholds; r.gamma = acc->gamma; r.n_steps = acc->n_steps;
  r.g_mode = acc->g_mode;
  const unsigned grid = (unsigned)((n_envs + kCovFThreads - 1) / kCovFThreads);
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = dispatch<0, 1>(p->mode, [&](auto m) { return launch_coverage_float_rollout<m>(p->n_agents, r, grid, st); },
                              "bad mode %d"))
    return rc;
  if (stats) return launch_stats_finalize(stats_scratch, grid, p->n_agents, p->n_agents, n_envs, stats, st);
  return SMARL_OK;
}
#endif
