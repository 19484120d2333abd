// Whole on-policy CollisionAvoidance episodes in one launch (sm_100a): reset + T x (every agent's ContinuousPolicy on
// the current observation, sample, env step, MetaAgent.act) + Buffer.step + compute_returns, i.e. main.py:28-57 with
// the policies (agent.py:48-76) inside.  The closed loop runs the same episode as 2T + 1 dependent launches
// (smarl_policy_act_gaussian + smarl_collision_step per step, then smarl_rollout_returns).
//
// One thread owns one env, as in collision_rollout_kernel (collision.cu): the f64 positions and the done mask stay in
// registers for all T steps, every agent's weights sit in shared memory and are read as warp-wide broadcasts.  Per
// step the thread builds the f32 observation, evaluates the A networks, samples by Philox Box-Muller, steps the env
// with the collision.cuh code the fused rollout uses (collision_transition_compact, collision_env_step) and accumulates
// R / modR / C / G the way that kernel does.
//
// Bit-identity with the closed loop is the contract: the policy code (gauss_policy.cuh, shared with
// coverage_float_policy.cu) keeps policy_gauss.cu's evaluation order and its Philox counter.  This file is compiled with
// -fmad=false like collision.cu (the accounting relies on uncontracted f64 sums), which gauss_policy.cuh's explicit
// fmaf form expects.  Actions and log-probabilities are sampled for every (t, agent, env), including done agents and
// envs past their episode end, as the policy kernel of the closed loop does.
//
// The weight staging and the accounting are copies of coverage_float_policy.cu's and collision_rollout_kernel's (DESIGN.md
// section 3.12 says why they are not shared).
#include "collision.cuh"
#include "gauss_policy.cuh"

namespace smarl {

// CTA size.  128 keeps smarl_collision_rollout's summation tree of the stats partials (one row per 128 envs), so the
// stats are bit-identical to the open-loop rollout of the recorded actions; other multiples of 32 (a build-time
// experiment, see DESIGN.md section 3.11) change only the order of the stats sums.
#ifndef SMARL_POLICY_ROLLOUT_THREADS
#define SMARL_POLICY_ROLLOUT_THREADS 128
#endif
constexpr int kPolRollThreads = SMARL_POLICY_ROLLOUT_THREADS;
constexpr int kPolRollMaxA = 8;                  // one thread per env: collision_coop_lanes returns 0 below A = 9

struct CollisionPolicyArgs {
  CollisionRolloutArgs r;    // r.actions unused
  float* obs_rec;            // [T][S][ld]  or NULL
  float* act_rec;            // [T][2A][ld] or NULL
  float* logp_rec;           // [T][A][ld]  or NULL
  GaussPolicyArgs pol;
  int32_t S;
  int32_t obs_landmarks;
  int32_t normalize;
};

// Static shared memory of the kernel: the block-sum slots and the warps' action-clip slots.  A launch without the opt-in
// may ask for 48 KB minus this much dynamic shared memory.
constexpr size_t kPolRollStaticSmem = sizeof(double) * (kPolRollThreads / 32) +
                                      sizeof(double2) * (kPolRollThreads / 32) * kClipSlots;

// Dynamic shared memory (floats): per agent w1 [S][16] and b1 [16] (W1S = 16 S + 16), heads [kHeadFloats]; then the
// landmark part of the observation, constant over the episode, one column per thread: [2L][kPolRollThreads].
inline size_t policy_rollout_smem(int A, int S, int L, int obs_landmarks) {
  return sizeof(float) * ((size_t)A * (S * kPolHidden + kPolHidden + kHeadFloats) +
                          (obs_landmarks ? (size_t)2 * L * kPolRollThreads : 0));
}

template <int A>
__global__ void __launch_bounds__(kPolRollThreads) collision_policy_rollout_kernel(const CollisionPolicyArgs p) {
  constexpr int H = kPolHidden;
  const CollisionRolloutArgs& a = p.r;
  extern __shared__ float s_pol[];
  __shared__ double s_red[kPolRollThreads / 32];
  __shared__ double2 s_clip[kPolRollThreads / 32][kClipSlots];
  const int S = p.S, W1S = S * H + H, n_lobs = S - 2 * A;
  float* s_w1 = s_pol;                                 // [A][W1S]: w1[a][k][u], then b1[a][u]
  float* s_hd = s_w1 + A * W1S;                        // [A][kHeadFloats]
  float* s_lobs = s_hd + A * kHeadFloats;              // [n_lobs][kPolRollThreads]
  const int tid = threadIdx.x;
  for (int i = tid; i < A * S * H; i += kPolRollThreads) s_w1[(i / (S * H)) * W1S + i % (S * H)] = __ldg(p.pol.w1 + i);
  for (int i = tid; i < A * H; i += kPolRollThreads) s_w1[(i / H) * W1S + S * H + i % H] = __ldg(p.pol.b1 + i);
  for (int i = tid; i < A * kHeadFloats; i += kPolRollThreads) {
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

  const int64_t eg = (int64_t)blockIdx.x * kPolRollThreads + tid;
  const bool live = eg < a.n_envs;
  const int64_t e = live ? eg : 0;
  const int64_t ld = a.ld;
  const int T = a.n_steps;
  const double size = a.size;
  float* lobs = s_lobs + tid;
  for (int k = 0; k < n_lobs; ++k) lobs[k * kPolRollThreads] = obs_value(a.landmarks[k * ld + e], size, p.normalize);
  double px[A], py[A];
#pragma unroll
  for (int i = 0; i < A; ++i) {
    px[i] = a.start_x[i * ld + e];
    py[i] = a.start_y[i * ld + e];
  }
  const uint2 key = make_uint2((uint32_t)p.pol.seed, (uint32_t)(p.pol.seed >> 32) ^ 0x47415553u);   // "GAUS"
  const uint32_t episode = p.pol.episode + (p.pol.episode_dev ? __ldg(p.pol.episode_dev) : 0u);
  const uint32_t t_base = episode << 16, ep_hi = gauss_episode_hi(episode);
  const uint64_t id = (uint64_t)(p.pol.env_offset + e);
  __syncthreads();

  const uint32_t all = (1u << A) - 1u;
  const double lam = a.lambdas ? __ldg(a.lambdas) : 0.0;
  uint32_t done_mask = 0u;
  double s_rew = 0.0, s_pen = 0.0, disc = 1.0;
  int csum = 0, steps = 0;
  for (int t = 0; t < T; ++t) {
    // the observation (collision_avoidance.py:141-147): what the reset / step kernels write to env.obs
    float x[2 * A];
#pragma unroll
    for (int i = 0; i < A; ++i) {
      x[2 * i] = p.normalize ? obs_normalized(px[i], size) : (float)px[i];
      x[2 * i + 1] = p.normalize ? obs_normalized(py[i], size) : (float)py[i];
    }
    if (p.obs_rec && live) {
      float* o = p.obs_rec + (int64_t)t * S * ld + e;
#pragma unroll
      for (int k = 0; k < 2 * A; ++k) o[k * ld] = x[k];
      for (int k = 0; k < n_lobs; ++k) o[(2 * A + k) * ld] = lobs[k * kPolRollThreads];
    }
    // every agent's policy (agent.py:60-74): one Philox block serves agents 2j and 2j + 1
    float adx[A], ady[A];
    const uint32_t t_word = t_base + (uint32_t)t;
#pragma unroll
    for (int j = 0; j < (A + 1) / 2; ++j) {
      const uint4 w = philox4x32_10(make_uint4((uint32_t)id, (uint32_t)(id >> 32), t_word, ep_hi | (uint32_t)j), key);
#pragma unroll
      for (int h = 0; h < 2 && 2 * j + h < A; ++h) {
        const int ag = 2 * j + h;
        float2 mu;
        float v0, v1, lp;
        agent_heads<A, kPolRollThreads>(x, lobs, n_lobs, s_w1 + ag * W1S, s_hd + ag * kHeadFloats, mu, v0, v1);
        gauss_sample(h ? w.z : w.x, h ? w.w : w.y, mu, v0, v1, adx[ag], ady[ag], lp);
        if (live) {
          if (p.act_rec) {
            p.act_rec[((int64_t)t * 2 * A + 2 * ag) * ld + e] = adx[ag];
            p.act_rec[((int64_t)t * 2 * A + 2 * ag + 1) * ld + e] = ady[ag];
          }
          if (p.logp_rec) p.logp_rec[((int64_t)t * A + ag) * ld + e] = lp;
        }
      }
    }
    // the env step and the accounting, exactly as collision_rollout_kernel
    double reward = 0.0;
    int collisions = 0;
    const bool active = done_mask != all;               // main.py:51 (lanes past n_envs replay env 0 and store nothing)
    collision_transition_compact<A>(px, py, done_mask, active, adx, ady, size, s_clip[tid >> 5]);
    if (active) {
      collision_env_step<A, false>(px, py, done_mask, a.landmarks + e, ld, a.L, 0.0, 0.0, size, a.agents_size, reward,
                                   collisions);
      ++steps;
    }
    const float rf = (float)reward;
    const float pf = (float)(lam * (double)collisions);
    s_rew += disc * (double)rf;
    s_pen += disc * (double)pf;
    csum += collisions;
    if (a.g_mode == 1 && live) {
      a.g_scratch[(int64_t)t * ld + e] = rf;
      a.g_scratch[((int64_t)T + t) * ld + e] = pf;
    } else if (a.g_mode == 2 && live) {
      const float o = (float)(disc * ((double)rf - (double)pf));
#pragma unroll
      for (int i = 0; i < A; ++i) a.G[((int64_t)t * A + i) * ld + e] = o;
    }
    disc *= a.gamma;
  }
  if (live) {
    const float r = (float)s_rew, m = (float)(s_rew - s_pen);
#pragma unroll
    for (int i = 0; i < A; ++i) {
      if (a.final_x) a.final_x[i * ld + e] = px[i];
      if (a.final_y) a.final_y[i * ld + e] = py[i];
      if (a.final_done) a.final_done[i * ld + e] = (uint8_t)((done_mask >> i) & 1u);
      a.R[i * ld + e] = r;
      a.modR[i * ld + e] = m;
    }
    a.C[e] = csum;
    if (a.n_active) a.n_active[e] = steps;
  }
  if (a.partials) {
    double* out = a.partials + (int64_t)blockIdx.x * stats_len(A, 1);
    const double thr = a.thresholds ? __ldg(a.thresholds) : 0.0;
    const double bc = block_sum<kPolRollThreads>(live ? (double)csum : 0.0, s_red);
    const double bv = block_sum<kPolRollThreads>((live && a.thresholds && (double)csum > thr) ? 1.0 : 0.0, s_red);
    const double br = block_sum<kPolRollThreads>(live ? s_rew : 0.0, s_red);
    const double bm = block_sum<kPolRollThreads>(live ? s_rew - s_pen : 0.0, s_red);
    if (tid == 0) {
      out[0] = bc;
      out[1] = bv;
      for (int i = 0; i < A; ++i) {
        out[2 + i] = br;
        out[2 + A + i] = bm;
      }
      out[2 + 2 * A] = 0.0;
    }
  }
  if (a.g_mode == 1 && live) {                            // agent.py:200-206
    double g_rew = 0.0, g_pen = 0.0;
    for (int t = T - 1; t >= 0; --t) {
      g_rew = (double)a.g_scratch[(int64_t)t * ld + e] + a.gamma * g_rew;
      g_pen = (double)a.g_scratch[((int64_t)T + t) * ld + e] + a.gamma * g_pen;
      const float o = (float)(g_rew - g_pen);
#pragma unroll
      for (int i = 0; i < A; ++i) a.G[((int64_t)t * A + i) * ld + e] = o;
    }
  }
}

}  // namespace smarl

using namespace smarl;

extern "C" int smarl_collision_policy_rollout(const SmarlCollisionParams* p, const SmarlGaussianPolicy* pol,
                                              const SmarlAccounting* acc, const double* start_x, const double* start_y,
                                              const double* landmarks, const double* lambdas, float* obs_rec,
                                              float* actions, float* logp, double* final_x, double* final_y,
                                              uint8_t* final_done, int32_t* n_active, float* R, float* modR, int32_t* C,
                                              float* G, float* g_scratch, double* stats, double* stats_scratch,
                                              int64_t n_envs, int64_t ld, smarl_stream_t stream) {
  SMARL_REQUIRE(p != nullptr && pol != nullptr && acc != nullptr, "params is NULL");
  SMARL_REQUIRE(p->n_agents >= 1 && p->n_agents <= SMARL_MAX_AGENTS, "n_agents=%d outside 1..32", p->n_agents);
  if (p->n_agents > kPolRollMaxA) {
    set_error("the on-policy rollout runs one thread per env: n_agents=%d above %d", p->n_agents, kPolRollMaxA);
    return SMARL_EUNSUPPORTED;
  }
  if (int rc = check_collision(p)) return rc;
  if (int rc = check_layout(n_envs, ld)) return rc;
  if (int rc = check_accounting(acc, 65536, 2, G, stats, stats_scratch)) return rc;   // 16 bits of the Philox counter
  const int A = p->n_agents, S = 2 * A + (p->obs_landmarks ? 2 * p->n_landmarks : 0);
  if (int rc = check_gaussian_policy(pol, A, S)) return rc;
  SMARL_REQUIRE(start_x && start_y && landmarks && R && modR && C, "null required pointer");
  SMARL_REQUIRE(acc->g_mode != 1 || g_scratch, "g_mode 1 needs g_scratch [2][T][ld]");
  CollisionPolicyArgs k;
  CollisionRolloutArgs& a = k.r;
  a.start_x = start_x; a.start_y = start_y; a.landmarks = landmarks; a.actions = nullptr;
  a.lambdas = lambdas; a.final_x = final_x; a.final_y = final_y; a.final_done = final_done;
  a.n_active = n_active; a.R = R; a.modR = modR; a.C = C; a.G = G; a.g_scratch = g_scratch;
  a.partials = stats_scratch; a.thresholds = acc->thresholds; a.gamma = acc->gamma; a.n_envs = n_envs;
  a.ld = ld; a.size = (double)p->size; a.agents_size = p->agents_size; a.L = p->n_landmarks;
  a.n_steps = acc->n_steps; a.g_mode = acc->g_mode;
  k.obs_rec = obs_rec; k.act_rec = actions; k.logp_rec = logp; k.pol = gauss_policy_args(pol);
  k.S = S; k.obs_landmarks = p->obs_landmarks; k.normalize = p->normalize_state;
  const size_t smem = policy_rollout_smem(A, S, p->n_landmarks, p->obs_landmarks);
  const unsigned grid = (unsigned)((n_envs + kPolRollThreads - 1) / kPolRollThreads);
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = dispatch<1, 8>(A, [&](auto kA) {
        auto kern = collision_policy_rollout_kernel<kA>;
        if (smem + kPolRollStaticSmem > 48 * 1024)
          SMARL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<grid, kPolRollThreads, smem, st>>>(k);
        SMARL_CUDA(cudaGetLastError());
        return SMARL_OK;
      }))
    return rc;
  if (stats) return launch_stats_finalize(stats_scratch, grid, A, 1, n_envs, stats, st);
  return SMARL_OK;
}
