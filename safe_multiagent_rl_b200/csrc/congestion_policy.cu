// Whole on-policy Congestion episodes in one launch (sm_100a): reset + T x (every agent's DiscretePolicy on the joint
// state, sample, Congestion.step, MetaAgent.act) + Buffer.step + compute_returns, i.e. main.py:28-57 with the policies
// (agent.py:23-47) inside.  The closed loop runs the same episode as 2T + 1 dependent launches
// (smarl_policy_act_discrete + smarl_congestion_step per step, then smarl_rollout_returns).
//
// One thread owns four consecutive envs, as in congestion_rollout_kernel: the packed u8 positions stay in registers for
// all T steps, the per-agent f64 discounted sums in the [A][4][threads] shared-memory array, and the CTA has
// kCongRollThreads threads, so the stats partials come out of the same block summation tree.  Every agent's weights sit
// in dynamic shared memory after the sums and are read as warp-wide broadcasts.  The policy part is policy.cuh's:
// stage_discrete_policy, then per step discrete_policy_step4 on the joint observation
// (x0, y0, x1, ...: what the reset / step kernels write to env.obs), so the actions and log-probabilities are the bits
// of the FP32-pipe build of smarl_policy_act_discrete.  The env step (noise modes 0 and 2) and the accounting are copies
// of congestion_rollout_kernel's (DESIGN.md section 3.14), compiled with the same flags (contraction on), so the
// products are the bits of smarl_congestion_rollout fed the recorded actions.
#include "congestion.cuh"
#include "policy.cuh"
#include "stats.cuh"

namespace smarl {

constexpr int kCongPolMaxA = 8;         // one thread per four envs: the 64 hidden accumulators and A agents' state

struct CongestionPolicyArgs {
  CongestionRolloutArgs r;              // r.actions, r.moves unused
  float* obs_rec;                       // [T][2A][ld] or NULL
  uint8_t* act_rec;                     // [T][A][ld]  or NULL
  float* logp_rec;                      // [T][A][ld]  or NULL
  DiscretePolicyArgs pol;
};

// Dynamic shared memory: the reward sums [A][4][kCongRollThreads] and penalty sums [4][kCongRollThreads] in f64, then
// the weights (stage_discrete_policy).  The penalty sums live in shared memory too: kept in registers across the policy
// part they made A = 7 spill.
template <int A>
struct CongPolCfg {
  static constexpr size_t kSmem =
      sizeof(double) * 4 * kCongRollThreads * (A + 1) + sizeof(float) * PolCfg<A, kPolActions>::kWeightFloats;
};

// Launcher of noise mode M (0 or 2), each mode instantiated in its own translation unit
template <int M> int launch_congestion_policy_rollout(int A, const CongestionPolicyArgs& k, unsigned grid, cudaStream_t st);

#if SMARL_TU_IS(0) || SMARL_TU_IS(1)
template <int A, int MODE>
__global__ void __launch_bounds__(kCongRollThreads) congestion_policy_rollout_kernel(const CongestionPolicyArgs p) {
  constexpr int IN = 2 * A;
  extern __shared__ __align__(16) double s_acc[];             // [A][4][kCongRollThreads]
  __shared__ double s_red[kCongRollThreads / 32];
  double* s_pen = s_acc + 4 * kCongRollThreads * A;           // [4][kCongRollThreads]
  float* s_w = reinterpret_cast<float*>(s_pen + 4 * kCongRollThreads);
  const CongestionRolloutArgs& a = p.r;
  const int tid = threadIdx.x;
  stage_discrete_policy<A, kPolActions, kCongRollThreads>(s_w, p.pol, tid);
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
#pragma unroll
  for (int k = 0; k < 4; ++k) s_pen[k * kCongRollThreads + tid] = 0.0;
  __syncthreads();                                            // the weights
  const uint2 key = policy_key(p.pol.seed);
  const uint32_t policy_episode = p.pol.episode + (p.pol.episode_dev ? __ldg(p.pol.episode_dev) : 0u);
  const uint32_t t_base = policy_episode << 16, ep_hi = policy_episode_hi(policy_episode);
  const uint64_t id0 = (uint64_t)(p.pol.env_offset + e0);
  int csum[4] = {0, 0, 0, 0};
  double disc = 1.0;

  for (int t = 0; t < T; ++t) {
    if (p.obs_rec && live) {                                  // main.py:33: np.array(state).flatten()
      float* o = p.obs_rec + (int64_t)t * IN * ld + e0;
#pragma unroll
      for (int i = 0; i < A; ++i) {
        st_stream_f4(o + (2 * i) * ld, bytes_to_float4(xw[i]));
        st_stream_f4(o + (2 * i + 1) * ld, bytes_to_float4(yw[i]));
      }
    }
    // every agent's policy (agent.py:33-46)
    uint32_t aw[A];
    discrete_policy_step4<A>(xw, yw, s_w, key, id0, t_base + (uint32_t)t, ep_hi, aw, p.act_rec, p.logp_rec, live, t, ld,
                             e0);
    // the env step and the accounting, exactly as congestion_rollout_kernel
    uint32_t mw[A];
    if (MODE == 0) {
#pragma unroll
      for (int i = 0; i < A; ++i) mw[i] = aw[i];
    } else {
      congestion_noise_moves<A>(aw, mw, a.seed, a.keep_threshold, a.env_offset + e0, (uint32_t)t, episode);
    }
    uint32_t dcw[A], conw[A];
    congestion_transition<A>(xw, yw, mw, dcw, size4);
    const uint32_t org = congestion_classes<A, kSimdClassAgentsRollout>(xw, yw, dcw, aw, conw);
    const int cost[4] = {max(0, A / 3 - (int)(org & 0xFFu)), max(0, A / 3 - (int)((org >> 8) & 0xFFu)),
                         max(0, A / 3 - (int)((org >> 16) & 0xFFu)), max(0, A / 3 - (int)(org >> 24))};
    float pen[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      pen[k] = (float)(lam * cost[k]);                        // the step kernel publishes the penalty as f32
      s_pen[k * kCongRollThreads + tid] += disc * (double)pen[k];
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
      } else if (a.g_mode == 2 && live) {                     // agent.py:129-132
        st_stream_f4(a.G + ((int64_t)t * A + i) * ld + e0,
                     make_float4((float)(disc * ((double)r[0] - (double)pen[0])), (float)(disc * ((double)r[1] - (double)pen[1])),
                                 (float)(disc * ((double)r[2] - (double)pen[2])), (float)(disc * ((double)r[3] - (double)pen[3]))));
      }
    }
    disc *= a.gamma;
  }

  // Episode products and block partials of the statistics (meta_agent.py:32-36), as congestion_rollout_kernel
  bool valid[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) valid[k] = live && (e0 + k < a.n_envs);
  double* out = a.partials ? a.partials + (int64_t)blockIdx.x * stats_len(A, 1) : nullptr;
  if (live) {
    st_stream_i4(a.C + e0, make_int4(csum[0], csum[1], csum[2], csum[3]));
  }
  if (live) {
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
      mod[k] = raw[k] - s_pen[k * kCongRollThreads + tid];
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

  if (a.g_mode == 1 && live) {                                // agent.py:200-206, in place over the stored rewards
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
int launch_congestion_policy_rollout(int A, const CongestionPolicyArgs& k, unsigned grid, cudaStream_t st) {
  return dispatch<1, kCongPolMaxA>(A, [&](auto kA) {
    auto kern = congestion_policy_rollout_kernel<kA, M>;
    const size_t smem = CongPolCfg<kA>::kSmem;
    if (smem + 64 > 48 * 1024)   // + the static reduction buffer
      SMARL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, kCongRollThreads, smem, st>>>(k);
    SMARL_CUDA(cudaGetLastError());
    return SMARL_OK;
  });
}
#endif
#if SMARL_TU_IS(0)
template int launch_congestion_policy_rollout<0>(int, const CongestionPolicyArgs&, unsigned, cudaStream_t);
#endif
#if SMARL_TU_IS(1)
template int launch_congestion_policy_rollout<2>(int, const CongestionPolicyArgs&, unsigned, cudaStream_t);
#endif

}  // namespace smarl

using namespace smarl;

#if SMARL_TU_IS(2)

extern "C" int smarl_congestion_policy_rollout(const SmarlCongestionParams* p, const SmarlDiscretePolicy* pol,
                                               const SmarlAccounting* acc, const uint8_t* start_x,
                                               const uint8_t* start_y, const double* lambdas, float* obs_rec,
                                               uint8_t* actions, float* logp, uint8_t* final_x, uint8_t* final_y,
                                               float* R, float* modR, int32_t* C, float* G, float* g_scratch,
                                               double* stats, double* stats_scratch, int64_t n_envs, int64_t ld,
                                               smarl_stream_t stream) {
  if (int rc = check_congestion(p)) return rc;
  SMARL_REQUIRE(pol != nullptr && acc != nullptr, "params is NULL");
  SMARL_REQUIRE(p->n_agents >= 1 && p->n_agents <= SMARL_MAX_AGENTS, "n_agents=%d outside 1..32", p->n_agents);
  if (p->n_agents > kCongPolMaxA) {
    set_error("the on-policy rollout runs one thread per four envs: n_agents=%d above %d", p->n_agents, kCongPolMaxA);
    return SMARL_EUNSUPPORTED;
  }
  if (p->noise_mode == 1) {
    set_error("noise_mode 1 replays recorded moves, which cannot follow the sampled actions of an on-policy rollout");
    return SMARL_EUNSUPPORTED;
  }
  if (int rc = check_layout(n_envs, ld)) return rc;
  if (int rc = check_accounting(acc, 65536, 2, G, stats, stats_scratch)) return rc;   // 16 bits of the Philox counter
  const int A = p->n_agents;
  if (int rc = check_discrete_policy(pol, A)) return rc;
  SMARL_REQUIRE(start_x && start_y && R && modR && C, "null required pointer");
  SMARL_REQUIRE(acc->g_mode != 1 || g_scratch, "g_mode 1 needs g_scratch [T][ld]");
  SMARL_REQUIRE((int64_t)A * ld < (1ll << 32), "A*ld = %lld exceeds 32-bit element offsets; split the env batch",
                (long long)((int64_t)A * ld));
  SMARL_REQUIRE(aligned16(start_x) && aligned16(start_y) && aligned16(obs_rec) && aligned16(actions) &&
                    aligned16(logp) && aligned16(final_x) && aligned16(final_y) && aligned16(R) && aligned16(modR) &&
                    aligned16(C) && aligned16(G) && aligned16(g_scratch), "pointers must be 16-byte aligned");
  CongestionPolicyArgs k;
  CongestionRolloutArgs& r = k.r;
  r.start_x = start_x; r.start_y = start_y; r.actions = nullptr; r.moves = nullptr; r.lambdas = lambdas;
  r.final_x = final_x; r.final_y = final_y; r.R = R; r.modR = modR; r.C = C; r.G = G;
  r.g_scratch = g_scratch; r.partials = stats_scratch; r.thresholds = acc->thresholds;
  r.demand = p->demand; r.wait_reward = p->wait_reward; r.gamma = acc->gamma; r.keep_threshold = p->keep_threshold;
  r.seed = p->seed; r.env_offset = p->env_offset; r.n_groups = (n_envs + 3) / 4; r.n_envs = n_envs; r.ld = ld;
  r.size = p->size; r.n_steps = acc->n_steps; r.g_mode = acc->g_mode;
  r.episode = p->episode; r.episode_dev = p->episode_dev;
  k.obs_rec = obs_rec; k.act_rec = actions; k.logp_rec = logp;
  k.pol = discrete_policy_args(pol);
  const unsigned grid = (unsigned)((r.n_groups + kCongRollThreads - 1) / kCongRollThreads);
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = p->noise_mode == 2 ? launch_congestion_policy_rollout<2>(A, k, grid, st)
                                  : launch_congestion_policy_rollout<0>(A, k, grid, st))
    return rc;
  if (stats) return launch_stats_finalize(stats_scratch, grid, A, 1, n_envs, stats, st);
  return SMARL_OK;
}
#endif
