// Whole on-policy CoverageContinuous episodes in one launch (sm_100a): reset + T x (every agent's ContinuousPolicy on
// the current observation, sample, env step, MetaAgent.act) + Buffer.step + compute_returns, i.e. main.py:28-57 with
// the policies (agent.py:48-76) inside.  The closed loop runs the same episode as 2T + 1 dependent launches
// (smarl_policy_act_gaussian + smarl_coverage_float_step per step, then smarl_rollout_returns).
//
// One thread owns one env, as in coverage_float_rollout_kernel: the f64 positions, cost sums and discounted sums stay in
// registers for all T steps, every agent's weights sit in shared memory and are read as warp-wide broadcasts.  Per step
// the thread builds the f32 observation (x_i, y_i: what the reset / step kernels write to env.obs), evaluates the A
// networks and samples them with gauss_policy.cuh (policy_gauss.cu's arithmetic and Philox counter), steps the env with
// coverage_float_env_step_regs from coverage_float.cuh and accumulates R / modR / C / G / stats exactly as
// coverage_float_rollout_kernel does.  Compiled with -fmad=false like coverage_float.cu.
//
// The weight staging and the accounting are copies of collision_policy.cu's and coverage_float_rollout_kernel's:
// moving either into a shared function changed the SASS of the kernel it came from (DESIGN.md section 3.12).
#include "coverage_float.cuh"
#include "gauss_policy.cuh"
#include "stats.cuh"

namespace smarl {

constexpr int kCovPolMaxA = 8;      // one thread per env: the A networks' registers

struct CoverageFloatPolicyArgs {
  CoverageFloatRolloutArgs r;       // r.env.pos_x / pos_y = start positions, r.env.actions unused
  float* obs_rec;                   // [T][2A][ld] or NULL
  float* act_rec;                   // [T][2A][ld] or NULL
  float* logp_rec;                  // [T][A][ld]  or NULL
  GaussPolicyArgs pol;              // S = 2A
};

// kCovFThreads threads per CTA keep coverage_float_rollout_kernel's summation tree of the stats partials (one row per
// 128 envs), so the stats are bit-identical to the open-loop rollout of the recorded actions.  Shared memory is static:
// the observation has no landmark rows, S = 2A, and the weights take A (16 S + 84) floats (10.9 KB at A = 8).
template <int A>
__global__ void __launch_bounds__(kCovFThreads) coverage_float_policy_rollout_kernel(const CoverageFloatPolicyArgs p) {
  constexpr int S = 2 * A, H = kPolHidden, W1S = S * H + H;
  __shared__ __align__(16) float s_w1[A * W1S];        // [A][W1S]: w1[a][k][u], then b1[a][u]
  __shared__ __align__(16) float s_hd[A * kHeadFloats];
  __shared__ double s_red[kCovFThreads / 32];
  const CoverageFloatRolloutArgs& r = p.r;
  const CoverageFloatArgs& a = r.env;
  const int tid = threadIdx.x;
  for (int i = tid; i < A * S * H; i += kCovFThreads) s_w1[(i / (S * H)) * W1S + i % (S * H)] = __ldg(p.pol.w1 + i);
  for (int i = tid; i < A * H; i += kCovFThreads) s_w1[(i / H) * W1S + S * H + i % H] = __ldg(p.pol.b1 + i);
  for (int i = tid; i < A * kHeadFloats; i += kCovFThreads) {
    const int ag = i / kHeadFloats, j = i % kHeadFloats;
    float v;
    if (j < H * 4) {
      const int u = j / 4, c = j % 4;
      v = c < 2 ? __ldg(p.pol.w_mu + (ag * H + u) * 2 + c) : __ldg(p.pol.w_var + (ag * H + u) * 2 + (c - 2));
    } else {
      const int c = j - H * 4;
      v = c < 2 ? __ldg(p.pol.b_mu + ag * 2 + c) : __ldg(p.pol.b_var + ag * 2 + (c - 2));
    }
    s_hd[i] = v;
  }

  const int64_t eg = (int64_t)blockIdx.x * kCovFThreads + tid;
  const bool live = eg < a.n_envs;                     // lanes past n_envs replay env 0 and store nothing
  const int64_t e = live ? eg : 0;
  const int64_t ld = a.ld;
  const int T = r.n_steps;
  double px[A], py[A], csum[A], lam[A];
#pragma unroll
  for (int i = 0; i < A; ++i) {
    px[i] = a.pos_x[i * ld + e];
    py[i] = a.pos_y[i * ld + e];
    csum[i] = 0.0;
    lam[i] = a.lambdas ? __ldg(a.lambdas + i) : 0.0;
  }
  const uint2 key = make_uint2((uint32_t)p.pol.seed, (uint32_t)(p.pol.seed >> 32) ^ 0x47415553u);   // "GAUS"
  const uint32_t episode = p.pol.episode + (p.pol.episode_dev ? __ldg(p.pol.episode_dev) : 0u);
  const uint32_t t_base = episode << 16, ep_hi = gauss_episode_hi(episode);
  const uint64_t id = (uint64_t)(p.pol.env_offset + e);
  __syncthreads();

  double s_rew = 0.0, s_pen = 0.0, disc = 1.0;
  for (int t = 0; t < T; ++t) {
    float x[S];
#pragma unroll
    for (int i = 0; i < A; ++i) {
      x[2 * i] = (float)px[i];
      x[2 * i + 1] = (float)py[i];
    }
    if (p.obs_rec && live) {
      float* o = p.obs_rec + (int64_t)t * S * ld + e;
#pragma unroll
      for (int k = 0; k < S; ++k) o[k * ld] = x[k];
    }
    // every agent's policy (agent.py:60-74): one Philox block serves agents 2j and 2j + 1
    float fa[2 * A];                                   // the sampled rows dx0, dy0, dx1, ... the env step takes
    const uint32_t ma[1] = {0u};
    const uint32_t t_word = t_base + (uint32_t)t;
#pragma unroll
    for (int j = 0; j < (A + 1) / 2; ++j) {
      const uint4 w = philox4x32_10(make_uint4((uint32_t)id, (uint32_t)(id >> 32), t_word, ep_hi | (uint32_t)j), key);
#pragma unroll
      for (int h = 0; h < 2 && 2 * j + h < A; ++h) {
        const int ag = 2 * j + h;
        float2 mu;
        float v0, v1, lp;
        agent_heads<A, 1>(x, nullptr, 0, s_w1 + ag * W1S, s_hd + ag * kHeadFloats, mu, v0, v1);
        gauss_sample(h ? w.z : w.x, h ? w.w : w.y, mu, v0, v1, fa[2 * ag], fa[2 * ag + 1], lp);
        if (live) {
          if (p.act_rec) {
            p.act_rec[((int64_t)t * S + 2 * ag) * ld + e] = fa[2 * ag];
            p.act_rec[((int64_t)t * S + 2 * ag + 1) * ld + e] = fa[2 * ag + 1];
          }
          if (p.logp_rec) p.logp_rec[((int64_t)t * A + ag) * ld + e] = lp;
        }
      }
    }
    // the env step and the accounting, exactly as coverage_float_rollout_kernel
    double cost[A], rew, pen = 0.0;
    coverage_float_env_step_regs<A, 0>(px, py, fa, ma, a, cost, rew);
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
      if (tid == 0) {
        const double w = a.weights ? (double)__ldg(a.weights + i) : 1.0;
        out[i] = bc;
        out[A + i] = bv;
        out[2 * A + i] = w * b_rew;
        out[3 * A + i] = w * b_rew - b_pen;
      }
    }
    if (tid == 0) out[4 * A] = 0.0;
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

}  // namespace smarl

using namespace smarl;

extern "C" int smarl_coverage_float_policy_rollout(const SmarlCoverageFloatParams* p, const SmarlGaussianPolicy* pol,
                                                   const SmarlAccounting* acc, const double* start_x,
                                                   const double* start_y, const double* lambdas, float* obs_rec,
                                                   float* actions, float* logp, double* final_x, double* final_y,
                                                   float* R, float* modR, float* C, float* G, float* g_scratch,
                                                   double* stats, double* stats_scratch, int64_t n_envs, int64_t ld,
                                                   smarl_stream_t stream) {
  SMARL_REQUIRE(p != nullptr && pol != nullptr && acc != nullptr, "params is NULL");
  SMARL_REQUIRE(p->n_agents >= 1 && p->n_agents <= SMARL_MAX_AGENTS, "n_agents=%d outside 1..32", p->n_agents);
  if (p->n_agents > kCovPolMaxA) {
    set_error("the on-policy rollout runs one thread per env: n_agents=%d above %d", p->n_agents, kCovPolMaxA);
    return SMARL_EUNSUPPORTED;
  }
  SMARL_REQUIRE(p->mode == 0 || p->mode == 1, "bad mode %d", p->mode);
  if (p->mode != 0) {
    set_error("the on-policy rollout runs the continuous-action env (mode 0), not mode %d", p->mode);
    return SMARL_EUNSUPPORTED;
  }
  SMARL_REQUIRE(p->size >= 1, "size=%d must be >= 1", p->size);
  if (int rc = check_layout(n_envs, ld)) return rc;
  if (int rc = check_accounting(acc, 65536, 2, G, stats, stats_scratch)) return rc;   // 16 bits of the Philox counter
  const int A = p->n_agents;
  if (int rc = check_gaussian_policy(pol, A, 2 * A)) return rc;
  SMARL_REQUIRE(start_x && start_y && R && modR && C, "null required pointer");
  SMARL_REQUIRE(acc->g_mode != 1 || g_scratch, "g_mode 1 needs g_scratch [2][T][ld]");
  CoverageFloatPolicyArgs k;
  CoverageFloatRolloutArgs& r = k.r;
  coverage_float_args(p, r.env);
  r.env.pos_x = const_cast<double*>(start_x); r.env.pos_y = const_cast<double*>(start_y); r.env.lambdas = lambdas;
  r.env.n_envs = n_envs; r.env.ld = ld;
  r.final_x = final_x; r.final_y = final_y; r.R = R; r.modR = modR; r.C = C; r.G = G; r.g_scratch = g_scratch;
  r.partials = stats_scratch; r.thresholds = acc->thresholds; r.gamma = acc->gamma; r.n_steps = acc->n_steps;
  r.g_mode = acc->g_mode;
  k.obs_rec = obs_rec; k.act_rec = actions; k.logp_rec = logp; k.pol = gauss_policy_args(pol);
  const unsigned grid = (unsigned)((n_envs + kCovFThreads - 1) / kCovFThreads);
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = dispatch<1, 8>(A, [&](auto kA) {
        coverage_float_policy_rollout_kernel<kA><<<grid, kCovFThreads, 0, st>>>(k);
        SMARL_CUDA(cudaGetLastError());
        return SMARL_OK;
      }))
    return rc;
  if (stats) return launch_stats_finalize(stats_scratch, grid, A, A, n_envs, stats, st);
  return SMARL_OK;
}
