// Whole on-policy CoverageDiscretized episodes in one launch (sm_100a): reset + T x (every agent's DiscretePolicy on the
// current observation, sample, env step, MetaAgent.act) + Buffer.step + compute_returns, i.e. main.py:28-57 with the
// policies (agent.py:23-47, 9 actions from coverage.py:210-241) inside.  The closed loop runs the same episode as
// 2T + 1 dependent launches (smarl_policy_act_discretized + smarl_coverage_float_step per step, then
// smarl_rollout_returns).
//
// One thread owns one env, as in coverage_float_rollout_kernel: the f64 positions, cost sums and discounted sums stay in
// registers for all T steps, every agent's weights sit in static shared memory and are read as warp-wide broadcasts.
// Per step the thread builds the f32 observation (x_i, y_i: what the reset / step kernels write to env.obs), evaluates
// the A networks in the operation order of policy.cuh's policy_act_discrete_kernel<A, 9> (fc1 as packed FFMA2 from b1
// over k = 0..2A-1, relu, fc2 as an fmaf chain over u = 0..15 from log2(e) b2), samples each with policy_head<9> on the
// shared Philox word, steps the env with coverage_float_env_step_regs<A, 1> and accumulates R / modR / C / G / stats
// exactly as coverage_float_rollout_kernel does.  Compiled with -fmad=false like coverage_float.cu: every multiply-add
// the contraction-on policy kernel fuses is an explicit fmaf / ffma2 here.
//
// Only the policy arguments (DiscretePolicyArgs) are shared with the other on-policy rollouts; the one-env network is
// this kernel's own, and the accounting is a copy of coverage_float_rollout_kernel's (as in coverage_float_policy.cu):
// moving it into a shared function changed the SASS of the kernel it came from (DESIGN.md section 3.12).
#include "coverage_float.cuh"
#include "policy.cuh"
#include "stats.cuh"
#include "tc.cuh"

namespace smarl {

constexpr int kCovDzPolMaxA = 8;    // one thread per env: the A networks' registers

struct CoverageDiscretizedPolicyArgs {
  CoverageFloatRolloutArgs r;       // r.env.pos_x / pos_y = start positions, r.env.actions unused
  float* obs_rec;                   // [T][2A][ld] or NULL
  uint8_t* act_rec;                 // [T][A][ld]  or NULL
  float* logp_rec;                  // [T][A][ld]  or NULL
  DiscretePolicyArgs pol;
};

// kCovFThreads threads per CTA keep coverage_float_rollout_kernel's summation tree of the stats partials (one row per
// 128 envs), so the stats are bit-identical to the open-loop rollout of the recorded actions.  Shared memory is static:
// A (32 A + 16 + 144 + 9) floats, 13.6 KB at A = 8.
template <int A>
__global__ void __launch_bounds__(kCovFThreads) coverage_discretized_policy_rollout_kernel(
    const CoverageDiscretizedPolicyArgs p) {
  constexpr int S = 2 * A, H = kPolHidden, NA = kDiscretizedActions, W1S = S * H + H, W2S = H * NA + NA;
  __shared__ __align__(16) float s_w1[A * W1S];        // [A][W1S]: w1[a][k][u], then b1[a][u]
  __shared__ float s_w2[A * W2S];                      // [A][W2S]: log2(e) w2[a][u][c], then log2(e) b2[a][c]
  __shared__ double s_red[kCovFThreads / 32];
  const CoverageFloatRolloutArgs& r = p.r;
  const CoverageFloatArgs& a = r.env;
  const int tid = threadIdx.x;
  for (int i = tid; i < A * S * H; i += kCovFThreads) s_w1[(i / (S * H)) * W1S + i % (S * H)] = __ldg(p.pol.w1 + i);
  for (int i = tid; i < A * H; i += kCovFThreads) s_w1[(i / H) * W1S + S * H + i % H] = __ldg(p.pol.b1 + i);
  for (int i = tid; i < A * H * NA; i += kCovFThreads) s_w2[(i / (H * NA)) * W2S + i % (H * NA)] = __ldg(p.pol.w2 + i) * kLog2e;
  for (int i = tid; i < A * NA; i += kCovFThreads) s_w2[(i / NA) * W2S + H * NA + i % NA] = __ldg(p.pol.b2 + i) * kLog2e;

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
  const uint2 key = policy_key(p.pol.seed);
  const uint32_t episode = p.pol.episode + (p.pol.episode_dev ? __ldg(p.pol.episode_dev) : 0u);
  const uint32_t t_base = episode << 16, ep_hi = policy_episode_hi(episode);
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
    // every agent's policy (agent.py:33-46); one Philox block serves four consecutive agents
    const float fa[1] = {0.f};
    uint32_t ma[A];
    const uint32_t t_word = t_base + (uint32_t)t;
    uint4 words;
#pragma unroll
    for (int ag = 0; ag < A; ++ag) {
      if ((ag & 3) == 0) words = policy_words(id, t_word, ep_hi, ag >> 2, key);
      const float* w1 = s_w1 + ag * W1S;
      const float* w2 = s_w2 + ag * W2S;
      float2 h2[H / 2];
#pragma unroll
      for (int q = 0; q < H / 2; ++q) h2[q] = *reinterpret_cast<const float2*>(w1 + S * H + 2 * q);
#pragma unroll
      for (int k = 0; k < S; ++k) {
        const float2 xx = make_float2(x[k], x[k]);
        const float4* wr = reinterpret_cast<const float4*>(w1 + k * H);
#pragma unroll
        for (int v = 0; v < H / 4; ++v) {
          const float4 w = wr[v];
          h2[2 * v] = tc::ffma2(xx, make_float2(w.x, w.y), h2[2 * v]);
          h2[2 * v + 1] = tc::ffma2(xx, make_float2(w.z, w.w), h2[2 * v + 1]);
        }
      }
      float l[NA];
#pragma unroll
      for (int c = 0; c < NA; ++c) l[c] = w2[H * NA + c];
#pragma unroll
      for (int u = 0; u < H; ++u) {
        const float rl = fmaxf((u & 1) ? h2[u >> 1].y : h2[u >> 1].x, 0.f);
#pragma unroll
        for (int c = 0; c < NA; ++c) l[c] = fmaf(rl, w2[u * NA + c], l[c]);
      }
      int pick;
      float lp;
      policy_head(l, word_of(words, ag & 3), pick, lp);
      ma[ag] = (uint32_t)pick;
      if (live) {
        if (p.act_rec) p.act_rec[((int64_t)t * A + ag) * ld + e] = (uint8_t)pick;
        if (p.logp_rec) p.logp_rec[((int64_t)t * A + ag) * ld + e] = lp;
      }
    }
    // the env step and the accounting, exactly as coverage_float_rollout_kernel
    double cost[A], rew, pen = 0.0;
    coverage_float_env_step_regs<A, 1>(px, py, fa, ma, a, cost, rew);
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

extern "C" int smarl_coverage_discretized_policy_rollout(const SmarlCoverageFloatParams* p,
                                                         const SmarlDiscretePolicy* pol, const SmarlAccounting* acc,
                                                         const double* start_x, const double* start_y,
                                                         const double* lambdas, float* obs_rec, uint8_t* actions,
                                                         float* logp, double* final_x, double* final_y, float* R,
                                                         float* modR, float* C, float* G, float* g_scratch,
                                                         double* stats, double* stats_scratch, int64_t n_envs,
                                                         int64_t ld, smarl_stream_t stream) {
  SMARL_REQUIRE(p != nullptr && pol != nullptr && acc != nullptr, "params is NULL");
  SMARL_REQUIRE(p->n_agents >= 1 && p->n_agents <= SMARL_MAX_AGENTS, "n_agents=%d outside 1..32", p->n_agents);
  if (p->n_agents > kCovDzPolMaxA) {
    set_error("the on-policy rollout runs one thread per env: n_agents=%d above %d", p->n_agents, kCovDzPolMaxA);
    return SMARL_EUNSUPPORTED;
  }
  SMARL_REQUIRE(p->mode == 0 || p->mode == 1, "bad mode %d", p->mode);
  if (p->mode != 1) {
    set_error("the on-policy rollout with the DiscretePolicy runs the discretized env (mode 1), not mode %d; "
              "smarl_coverage_float_policy_rollout runs mode 0", p->mode);
    return SMARL_EUNSUPPORTED;
  }
  SMARL_REQUIRE(p->size >= 1, "size=%d must be >= 1", p->size);
  SMARL_REQUIRE(p->zoom > 0.0, "mode 1 needs zoom > 0");
  if (int rc = check_layout(n_envs, ld)) return rc;
  if (int rc = check_accounting(acc, 65536, 2, G, stats, stats_scratch)) return rc;   // 16 bits of the Philox counter
  const int A = p->n_agents;
  if (int rc = check_discrete_policy(pol, A, kDiscretizedActions)) return rc;
  SMARL_REQUIRE(start_x && start_y && R && modR && C, "null required pointer");
  SMARL_REQUIRE(acc->g_mode != 1 || g_scratch, "g_mode 1 needs g_scratch [2][T][ld]");
  CoverageDiscretizedPolicyArgs k;
  CoverageFloatRolloutArgs& r = k.r;
  coverage_float_args(p, r.env);
  r.env.pos_x = const_cast<double*>(start_x); r.env.pos_y = const_cast<double*>(start_y); r.env.lambdas = lambdas;
  r.env.n_envs = n_envs; r.env.ld = ld;
  r.final_x = final_x; r.final_y = final_y; r.R = R; r.modR = modR; r.C = C; r.G = G; r.g_scratch = g_scratch;
  r.partials = stats_scratch; r.thresholds = acc->thresholds; r.gamma = acc->gamma; r.n_steps = acc->n_steps;
  r.g_mode = acc->g_mode;
  k.obs_rec = obs_rec; k.act_rec = actions; k.logp_rec = logp;
  k.pol = discrete_policy_args(pol);
  const unsigned grid = (unsigned)((n_envs + kCovFThreads - 1) / kCovFThreads);
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = dispatch<1, kCovDzPolMaxA>(A, [&](auto kA) {
        coverage_discretized_policy_rollout_kernel<kA><<<grid, kCovFThreads, 0, st>>>(k);
        SMARL_CUDA(cudaGetLastError());
        return SMARL_OK;
      }))
    return rc;
  if (stats) return launch_stats_finalize(stats_scratch, grid, A, A, n_envs, stats, st);
  return SMARL_OK;
}
