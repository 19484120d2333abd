// Whole on-policy CoverageDiscrete episodes in one launch (sm_100a): reset + T x (every agent's DiscretePolicy on the
// joint state, sample, env step, MetaAgent.act) + Buffer.step + compute_returns, i.e. main.py:28-57 with the policies
// (agent.py:23-47) inside.  The closed loop runs the same episode as 2T + 1 dependent launches
// (smarl_policy_act_discrete + smarl_coverage_step per step, then smarl_rollout_returns).
//
// One thread owns four consecutive envs, as in coverage_rollout_kernel: the packed u8 positions, the byte cost counters
// and the discounted sums stay in registers for all T steps.  Every agent's weights sit in shared memory beside the
// penalty table and are read as warp-wide broadcasts; they are staged by policy.cuh's stage_discrete_policy.  Per step the
// thread evaluates the A networks on the joint observation (x0, y0, x1, ...: what the reset / step kernels write to
// env.obs) in exactly policy_act_discrete_kernel's operation order: fc1 as packed FFMA2 from b1 over the inputs
// k = 0..2A-1, relu, fc2 from log2(e) b2 over the 16 hidden units (packed FFMA2 over env pairs: per env policy.cu's fmaf
// chain), then policy_head with the same Philox word.  So the actions and log-probabilities are the bits of the
// FP32-pipe build of smarl_policy_act_discrete.  That per-step loop is a copy of policy.cuh's discrete_policy_step4,
// which congestion_policy.cu calls: calling it here made the one launch without records 4.7 % slower on a B200 at
// 50 envs x 3 agents (DESIGN.md section 3.13).  The env step and the accounting are copies of coverage_rollout_kernel's,
// compiled with the same flags (contraction on), so the products are the bits of smarl_coverage_rollout fed the recorded
// actions.
#include "coverage.cuh"
#include "policy.cuh"
#include "stats.cuh"
#include "tc.cuh"

namespace smarl {

constexpr int kCovDiscPolMaxA = 8;      // one thread per four envs: the 64 hidden accumulators and A agents' state

struct CoveragePolicyArgs {
  CoverageRolloutArgs r;                // r.actions unused
  float* obs_rec;                       // [T][2A][ld] or NULL
  uint8_t* act_rec;                     // [T][A][ld]  or NULL
  float* logp_rec;                      // [T][A][ld]  or NULL
  DiscretePolicyArgs pol;
};

template <int A>
__global__ void __launch_bounds__(kRolloutThreads) coverage_policy_rollout_kernel(const CoveragePolicyArgs p) {
  using Cfg = PolCfg<A, kPolActions>;
  constexpr int IN = Cfg::IN, H = kPolHidden, NA = kPolActions;
  extern __shared__ __align__(16) float s_mem[];
  const float* s_w1 = s_mem;                         // [A][W1S]  w1[a][k][u]
  const float* s_w2 = s_w1 + A * Cfg::W1S;           // [A][W2S]  log2(e) w2[a][u][c]
  const float* s_b1 = s_w2 + A * Cfg::W2S;           // [A][16]
  const float* s_b2 = s_b1 + A * H;                  // [A][8]    log2(e) b2[a][c]
  float* s_lut = s_mem + Cfg::kWeightFloats;
  const CoverageRolloutArgs& a = p.r;
  const int tid = threadIdx.x;
  stage_discrete_policy<A, kPolActions, kRolloutThreads>(s_mem, p.pol, tid);
  coverage_load_lut(s_lut, a.lut, a.lut_len);       // its barrier also covers the weights
  const int64_t g = (int64_t)blockIdx.x * kRolloutThreads + tid;
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
  const uint2 key = policy_key(p.pol.seed);
  const uint32_t episode = p.pol.episode + (p.pol.episode_dev ? __ldg(p.pol.episode_dev) : 0u);
  const uint32_t t_base = episode << 16, ep_hi = policy_episode_hi(episode);
  const uint64_t id0 = (uint64_t)(p.pol.env_offset + e0);
  double s_rew[4] = {0, 0, 0, 0}, s_pen[4] = {0, 0, 0, 0};
  double disc = 1.0;

  for (int t = 0; t < T; ++t) {
    if (p.obs_rec && live) {                           // main.py:33: np.array(state).flatten()
      float* o = p.obs_rec + (int64_t)t * IN * ld + e0;
#pragma unroll
      for (int i = 0; i < A; ++i) {
        st_stream_f4(o + (2 * i) * ld, bytes_to_float4(xw[i]));
        st_stream_f4(o + (2 * i + 1) * ld, bytes_to_float4(yw[i]));
      }
    }
    // every agent's policy (agent.py:33-46); one Philox block serves four consecutive agents of an env
    const uint32_t t_word = t_base + (uint32_t)t;
    uint32_t aw[A];
    uint4 words[4];
#pragma unroll
    for (int ag = 0; ag < A; ++ag) {
      if ((ag & 3) == 0) {
#pragma unroll
        for (int k = 0; k < 4; ++k) words[k] = policy_words(id0 + k, t_word, ep_hi, ag >> 2, key);
      }
      const float* w1 = s_w1 + ag * Cfg::W1S;
      const float* w2 = s_w2 + ag * Cfg::W2S;
      float2 h2[4][H / 2];
#pragma unroll
      for (int q = 0; q < H / 2; ++q) {
        const float2 b = *reinterpret_cast<const float2*>(s_b1 + ag * H + 2 * q);
        h2[0][q] = h2[1][q] = h2[2][q] = h2[3][q] = b;
      }
#pragma unroll
      for (int k = 0; k < IN; ++k) {
        const float4 x = bytes_to_float4((k & 1) ? yw[k >> 1] : xw[k >> 1]);
        const float2 xx[4] = {make_float2(x.x, x.x), make_float2(x.y, x.y), make_float2(x.z, x.z), make_float2(x.w, x.w)};
        const float4* wr = reinterpret_cast<const float4*>(w1 + k * H);
#pragma unroll
        for (int v = 0; v < H / 4; ++v) {
          const float4 w = wr[v];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            h2[e][2 * v] = tc::ffma2(xx[e], make_float2(w.x, w.y), h2[e][2 * v]);
            h2[e][2 * v + 1] = tc::ffma2(xx[e], make_float2(w.z, w.w), h2[e][2 * v + 1]);
          }
        }
      }
      // fc2 as packed FFMA2 over the env pairs (0, 1) and (2, 3): per env the fmaf chain over u = 0..15 of policy.cu
      float2 l2[2][NA];
#pragma unroll
      for (int c = 0; c < NA; ++c) l2[0][c] = l2[1][c] = make_float2(s_b2[ag * 8 + c], s_b2[ag * 8 + c]);
#pragma unroll
      for (int u = 0; u < H; ++u) {
        float r[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) r[e] = fmaxf((u & 1) ? h2[e][u >> 1].y : h2[e][u >> 1].x, 0.f);
        const float2 r01 = make_float2(r[0], r[1]), r23 = make_float2(r[2], r[3]);
#pragma unroll
        for (int c = 0; c < NA; ++c) {
          const float w = w2[u * NA + c];
          l2[0][c] = tc::ffma2(r01, make_float2(w, w), l2[0][c]);
          l2[1][c] = tc::ffma2(r23, make_float2(w, w), l2[1][c]);
        }
      }
      uint32_t act4 = 0u;
      float lp[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        float l[NA];
#pragma unroll
        for (int c = 0; c < NA; ++c) l[c] = (k & 1) ? l2[k >> 1][c].y : l2[k >> 1][c].x;
        int pick;
        policy_head(l, word_of(words[k], ag & 3), pick, lp[k]);
        act4 |= (uint32_t)pick << (8 * k);
      }
      aw[ag] = act4;
      if (live) {
        if (p.act_rec) st_stream_u32(p.act_rec + ((int64_t)t * A + ag) * ld + e0, act4);
        if (p.logp_rec) st_stream_f4(p.logp_rec + ((int64_t)t * A + ag) * ld + e0, make_float4(lp[0], lp[1], lp[2], lp[3]));
      }
    }
    // the env step and the accounting, exactly as coverage_rollout_kernel
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
      uint32_t pk[A];
#pragma unroll
      for (int i = 0; i < A; ++i) pk[i] = coverage_pack2(xw[i], yw[i], sel);
      const float r = -coverage_pair_penalty<A>(pk, s_lut, (uint32_t)a.lut_len * 4u);
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

  // Episode products: R_a = w_a * S_rew,  modR_a = w_a * S_rew - S_pen (coverage_rollout_kernel)
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

  // Block partials of the statistics (meta_agent.py:32-36), in coverage_rollout_kernel's summation tree
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
#pragma unroll
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

}  // namespace smarl

using namespace smarl;

extern "C" int smarl_coverage_policy_rollout(const SmarlCoverageParams* p, const SmarlDiscretePolicy* pol,
                                             const SmarlAccounting* acc, const uint8_t* start_x, const uint8_t* start_y,
                                             const double* lambdas, float* obs_rec, uint8_t* actions, float* logp,
                                             uint8_t* final_x, uint8_t* final_y, float* R, float* modR, int32_t* C,
                                             float* G, float* g_scratch, double* stats, double* stats_scratch,
                                             int64_t n_envs, int64_t ld, smarl_stream_t stream) {
  SMARL_REQUIRE(p != nullptr && pol != nullptr && acc != nullptr, "params is NULL");
  SMARL_REQUIRE(p->n_agents >= 1 && p->n_agents <= SMARL_MAX_AGENTS, "n_agents=%d outside 1..32", p->n_agents);
  if (p->n_agents > kCovDiscPolMaxA) {
    set_error("the on-policy rollout runs one thread per four envs: n_agents=%d above %d", p->n_agents,
              kCovDiscPolMaxA);
    return SMARL_EUNSUPPORTED;
  }
  if (int rc = check_coverage(p)) return rc;
  if (int rc = check_layout(n_envs, ld)) return rc;
  if (int rc = check_accounting(acc, 255, 2, G, stats, stats_scratch)) return rc;   // byte cost counters
  const int A = p->n_agents;
  if (int rc = check_discrete_policy(pol, A)) return rc;
  SMARL_REQUIRE(start_x && start_y && R && modR && C, "null required pointer");
  SMARL_REQUIRE(acc->g_mode != 1 || g_scratch, "g_mode 1 needs g_scratch [2][T][ld]");
  SMARL_REQUIRE(aligned16(start_x) && aligned16(start_y) && aligned16(obs_rec) && aligned16(actions) &&
                    aligned16(logp) && aligned16(final_x) && aligned16(final_y) && aligned16(R) && aligned16(modR) &&
                    aligned16(C) && aligned16(G) && aligned16(g_scratch), "pointers must be 16-byte aligned");
  CoveragePolicyArgs k;
  CoverageRolloutArgs& r = k.r;
  r.start_x = start_x; r.start_y = start_y; r.actions = nullptr; r.lambdas = lambdas;
  r.final_x = final_x; r.final_y = final_y; r.R = R; r.modR = modR; r.C = C; r.G = G;
  r.g_scratch = g_scratch; r.partials = stats_scratch; r.thresholds = acc->thresholds;
  r.lut = p->lut; r.weights = p->weights; r.gamma = acc->gamma;
  r.n_groups = (n_envs + 3) / 4; r.n_envs = n_envs; r.ld = ld; r.size = p->size;
  r.lut_len = p->lut_len; r.n_steps = acc->n_steps; r.g_mode = acc->g_mode;
  k.obs_rec = obs_rec; k.act_rec = actions; k.logp_rec = logp;
  k.pol = discrete_policy_args(pol);
  const unsigned grid = (unsigned)((r.n_groups + kRolloutThreads - 1) / kRolloutThreads);
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = dispatch<1, kCovDiscPolMaxA>(A, [&](auto kA) {
        auto kern = coverage_policy_rollout_kernel<kA>;
        const size_t smem = (size_t)(PolCfg<kA, kPolActions>::kWeightFloats + p->lut_len + 1) * sizeof(float);
        if (smem > 48 * 1024) SMARL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<grid, kRolloutThreads, smem, st>>>(k);
        SMARL_CUDA(cudaGetLastError());
        return SMARL_OK;
      }))
    return rc;
  if (stats) return launch_stats_finalize(stats_scratch, grid, A, A, n_envs, stats, st);
  return SMARL_OK;
}
