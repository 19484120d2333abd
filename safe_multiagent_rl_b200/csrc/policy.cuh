// The reference's DiscretePolicy (agent.py:23-47) as every fused kernel evaluates it: arguments, the Philox stream and
// the softmax / inverse-CDF sampling head of both closed-loop builds (policy.cu / policy_discretized.cu: FP32 pipes,
// policy_tc.cu: fc1 on the tensor cores); the FP32-pipe closed-loop kernel and its launcher; the weight staging of the
// grid envs' on-policy rollouts (coverage_policy.cu, congestion_policy.cu) and the four-env evaluation of Congestion's
// (coverage_policy.cu keeps a copy of it, which is faster there).
#pragma once

#include "common.cuh"
#include "tc.cuh"

namespace smarl {

constexpr int kPolHidden = 16;
constexpr int kPolActions = 5;             // the grid envs
constexpr int kDiscretizedActions = 9;     // CoverageDiscretized (coverage.py:210-241)
constexpr float kLog2e = 1.4426950408889634f;

struct PolicyArgs {
  const uint8_t* pos_x;
  const uint8_t* pos_y;
  uint8_t* actions;
  float* logp;
  const float* w1;     // [A][2A][16]
  const float* b1;     // [A][16]
  const float* w2;     // [A][16][NA]
  const float* b2;     // [A][NA]
  uint64_t seed;
  int64_t env_offset;
  int64_t n_envs;
  int64_t ld;
  int64_t n_tiles;
  uint32_t t;
  uint32_t episode;    // *episode_dev is added on the device
  const uint32_t* episode_dev;
  const float* obs;    // [2A][ld] f32 observation rows, the 9-action input (pos_x / pos_y unused); last, so that the
                       // tensor-core kernel's parameter offsets stay put
};

// The policy part of the on-policy rollout kernels' arguments: every agent's weights and the sampling stream.
struct DiscretePolicyArgs {
  const float* w1;     // [A][2A][16]
  const float* b1;     // [A][16]
  const float* w2;     // [A][16][NA]
  const float* b2;     // [A][NA]
  uint64_t seed;
  int64_t env_offset;
  uint32_t episode;    // *episode_dev is added on the device
  const uint32_t* episode_dev;
};

inline DiscretePolicyArgs discrete_policy_args(const SmarlDiscretePolicy* pol) {
  DiscretePolicyArgs d;
  d.w1 = pol->w1; d.b1 = pol->b1; d.w2 = pol->w2; d.b2 = pol->b2;
  d.seed = pol->seed; d.env_offset = pol->env_offset; d.episode = pol->episode; d.episode_dev = pol->episode_dev;
  return d;
}

// tensor-core build (policy_tc.cu); SMARL_EUNSUPPORTED when the shape does not fit it
int launch_policy_tc(const PolicyArgs& a, int n_agents, int group_max, int sms, cudaStream_t st);

// The policy checks of the entry points that run the DiscretePolicy (p not NULL) for an env of A agents and n_actions
// actions: 5 on the grid envs, 9 on CoverageDiscretized (policy_discretized.cu).
inline int check_discrete_policy(const SmarlDiscretePolicy* p, int A, int n_actions = kPolActions) {
  SMARL_REQUIRE(p->n_agents == A, "policy has %d agents, the env %d", p->n_agents, A);
  if (n_actions == kPolActions)
    SMARL_REQUIRE(p->hidden == kPolHidden && p->n_actions == kPolActions,
                  "only the reference's DiscretePolicy shape (hidden 16, 5 actions) is built (got %d, %d)", p->hidden,
                  p->n_actions);
  else
    SMARL_REQUIRE(p->hidden == kPolHidden && p->n_actions == n_actions,
                  "CoverageDiscretized runs the reference's DiscretePolicy of hidden 16 and %d actions (got %d, %d)",
                  n_actions, p->hidden, p->n_actions);
  SMARL_REQUIRE(p->w1 && p->b1 && p->w2 && p->b2, "null pointer");
  return SMARL_OK;
}

#ifdef __CUDACC__
__device__ __forceinline__ uint2 policy_key(uint64_t seed) {
  return make_uint2((uint32_t)seed, (uint32_t)(seed >> 32) ^ 0x504C4359u);   // "PLCY"
}
// One Philox block serves four consecutive agents of one env and step: counter (env id lo, hi, t | episode << 16,
// agent >> 2 | (episode >> 16) << 3), agent a uses word a & 3 (oracle/philox.policy_words restates it).  The episode's
// bits above the 16 of the step word sit above the agent quad (8 quads for 32 agents), so the streams of episodes
// 65 536 apart differ; ep_hi is policy_episode_hi(episode).
__device__ __forceinline__ uint32_t policy_episode_hi(uint32_t episode) { return (episode >> 16) << 3; }
__device__ __forceinline__ uint4 policy_words(uint64_t env_id, uint32_t t_word, uint32_t ep_hi, int agent_quad,
                                              uint2 key) {
  return philox4x32_10(make_uint4((uint32_t)env_id, (uint32_t)(env_id >> 32), t_word, ep_hi | (uint32_t)agent_quad),
                       key);
}
// The Gaussian stream's counter (policy_gauss.cu) carries the same episode bits above its agent pair (16 pairs).
__device__ __forceinline__ uint32_t gauss_episode_hi(uint32_t episode) { return (episode >> 16) << 4; }
__device__ __forceinline__ uint32_t word_of(const uint4& o, int i) {
  return i == 0 ? o.x : (i == 1 ? o.y : (i == 2 ? o.z : o.w));
}

__device__ __forceinline__ float ex2_ftz(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float lg2_ftz(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// softmax (agent.py:35), Categorical sample by inverse CDF and log_prob (:44-46) of one agent and env over NA actions
// (5 on the grid envs, 9 on CoverageDiscretized; deduced from the logits array).  The logits
// arrive in log2 units, l2_c = log2(e) * logit_c (both builds scale their shared-memory copies of fc2 by log2(e)), so
// e_c = exp(logit_c - max) is one subtraction and one MUFU.EX2:
// u = min(((word >> 8) + 0.5) * 2^-24, 1 - 2^-24); action = #{c < NA - 1 : sum_{c' <= c} e_c' <= u * sum e}.
// In float32, (word >> 8) + 0.5 rounds to 2^24 for the top word, so u would be 1 and u * sum == sum would pick the last
// action whatever its probability; below 1, fl(u * sum) < sum for every sum >= 1, and an action of probability 0
// (its e_c flushed to 0) is never drawn.
template <int NA>
__device__ __forceinline__ void policy_head(const float (&l2)[NA], uint32_t word, int& pick, float& logp) {
  float m = l2[0];
#pragma unroll
  for (int c = 1; c < NA; ++c) m = fmaxf(m, l2[c]);
  float ex[NA], sum = 0.f;
#pragma unroll
  for (int c = 0; c < NA; ++c) {
    ex[c] = ex2_ftz(l2[c] - m);
    sum += ex[c];
  }
  const float target = fminf(((float)(word >> 8) + 0.5f) * (1.0f / 16777216.0f), 0x1.fffffep-1f) * sum;
  float cum = 0.f, l_pick = l2[0];
  pick = 0;
#pragma unroll
  for (int c = 0; c < NA - 1; ++c) {
    cum += ex[c];
    if (cum <= target) {
      pick = c + 1;
      l_pick = l2[c + 1];
    }
  }
  logp = ((l_pick - m) - lg2_ftz(sum)) * 0.693147180559945309f;     // log_softmax at the sampled action (sum >= 1)
}

// Layout of the FP32-pipe evaluations: every agent's weights in shared memory, per-agent strides padded by 4 floats so
// that agents land on different banks; then, in the closed-loop kernel, the tile's joint observation [IN][TE].
template <int A, int NA>
struct PolCfg {
  static constexpr int IN = 2 * A;
  // closed loop: env quads per tile, all A agents x QPT quads = one CTA of 96..256 threads
  static constexpr int QPT = A >= 16 ? 8 : (A >= 8 ? 16 : (A >= 4 ? 32 : 64));
  static constexpr int THREADS = A * QPT;
  static constexpr int TE = 4 * QPT;                          // envs per tile
  static constexpr int W1S = IN * kPolHidden + 4;
  static constexpr int W2S = kPolHidden * NA + 4;
  static constexpr int B2S = (NA + 3) / 4 * 4;                // NA biases, padded so that s_in stays 16-byte aligned
  static constexpr int kWeightFloats = A * W1S + A * W2S + A * kPolHidden + A * B2S;
  static constexpr size_t kSmemFloats = (size_t)kWeightFloats + (size_t)IN * TE;
  static_assert(kSmemFloats * sizeof(float) <= 227 * 1024, "weights exceed the shared memory of one SM");
};

// Stage the weights w1, b1, w2, b2 of every agent (a PolicyArgs or DiscretePolicyArgs p) at s_w, the THREADS threads
// of the CTA cooperating (tid: the kernel's threadIdx.x, whose range ptxas knows from the kernel's launch bounds):
// w1 [A][W1S], log2(e) w2 [A][W2S], b1 [A][16], log2(e) b2 [A][B2S] (fc2 scaled so that the logits arrive in
// policy_head's log2 units).  The caller's barrier follows.
template <int A, int NA, int THREADS, class P>
__device__ __forceinline__ void stage_discrete_policy(float* s_w, const P& p, int tid) {
  using C = PolCfg<A, NA>;
  constexpr int IN = C::IN, H = kPolHidden;
  float* s_w1 = s_w;
  float* s_w2 = s_w1 + A * C::W1S;
  float* s_b1 = s_w2 + A * C::W2S;
  float* s_b2 = s_b1 + A * H;
  for (int i = tid; i < A * IN * H; i += THREADS) s_w1[(i / (IN * H)) * C::W1S + i % (IN * H)] = __ldg(p.w1 + i);
  for (int i = tid; i < A * H * NA; i += THREADS) s_w2[(i / (H * NA)) * C::W2S + i % (H * NA)] = __ldg(p.w2 + i) * kLog2e;
  for (int i = tid; i < A * H; i += THREADS) s_b1[i] = __ldg(p.b1 + i);
  for (int i = tid; i < A * NA; i += THREADS) s_b2[(i / NA) * C::B2S + i % NA] = __ldg(p.b2 + i) * kLog2e;
}

// The closed-loop policy on the FP32 pipes (all multiply-adds as packed FFMA2 or fmaf).  Thread mapping: one thread =
// one agent x four consecutive envs (64 hidden accumulators in registers); a CTA = all A agents x QPT env quads, looping
// over tiles of 4*QPT envs (persistent grid), so the weights are staged once per CTA.  Per input k a thread issues one
// LDS.128 for the four envs' value and four LDS.128 for the 16 weights (both conflict-free broadcasts) against 64 FFMA.
template <int A, int NA>
__global__ void __launch_bounds__(PolCfg<A, NA>::THREADS) policy_act_discrete_kernel(const PolicyArgs a) {
  pdl_prologue();   // programmatic dependent launch: the previous grid has completed past this point (common.cuh)
  using C = PolCfg<A, NA>;
  constexpr int IN = C::IN, QPT = C::QPT, TE = C::TE, H = kPolHidden;
  extern __shared__ float s_mem[];
  float* s_w1 = s_mem;                               // [A][W1S]  w1[a][k][u]
  float* s_w2 = s_w1 + A * C::W1S;                   // [A][W2S]  log2(e) w2[a][u][c]
  float* s_b1 = s_w2 + A * C::W2S;                   // [A][16]
  float* s_b2 = s_b1 + A * H;                        // [A][B2S]  log2(e) b2[a][c]
  float* s_in = s_b2 + A * C::B2S;                   // [IN][TE] the joint observation of the tile, as floats
  const int tid = threadIdx.x;
  stage_discrete_policy<A, NA, C::THREADS>(s_mem, a, tid);
  const int ag = tid / QPT, quad = tid % QPT;
  const uint2 key = policy_key(a.seed);
  const uint32_t episode = a.episode + (a.episode_dev ? __ldg(a.episode_dev) : 0u);
  const uint32_t t_word = a.t | episode << 16, ep_hi = policy_episode_hi(episode);
  const float* w1 = s_w1 + ag * C::W1S;
  const float* w2 = s_w2 + ag * C::W2S;

  for (int64_t tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int64_t e_tile = tile * TE;
    if (tile != (int64_t)blockIdx.x) __syncthreads();   // previous tile fully consumed; the first tile's input loads
                                                        // go out right behind the weight loads (one barrier covers both)
    // stage the tile's joint observation (main.py:33: np.array(state).flatten()): row 2i = x_i, row 2i+1 = y_i.  The
    // grid envs (5 actions) keep u8 cells, read from their position rows; CoverageDiscretized (9 actions) has f64
    // positions, read from the f32 observation rows its step kernel publishes.
    for (int i = tid; i < IN * QPT; i += C::THREADS) {
      const int row = i / QPT, qd = i % QPT;
      const int64_t e = e_tile + 4 * qd;
      float4 v;
      if constexpr (NA == kPolActions) {
        const uint8_t* src = (row & 1) ? a.pos_y : a.pos_x;
        v = bytes_to_float4(e < a.ld ? ld_stream_u32(src + (int64_t)(row >> 1) * a.ld + e) : 0u);
      } else {
        v = e < a.ld ? ld_stream_f4(a.obs + (int64_t)row * a.ld + e) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      *reinterpret_cast<float4*>(s_in + row * TE + 4 * qd) = v;
    }
    __syncthreads();
    const int64_t e0 = e_tile + 4 * quad;
    // fc1 (agent.py:33) as packed FFMA2: h2[k][p] = (h[k][2p], h[k][2p+1]) for the four envs k of this thread
    float2 h2[4][H / 2];
#pragma unroll
    for (int p = 0; p < H / 2; ++p) {
      const float2 b = *reinterpret_cast<const float2*>(s_b1 + ag * H + 2 * p);
      h2[0][p] = h2[1][p] = h2[2][p] = h2[3][p] = b;
    }
#pragma unroll 4
    for (int k = 0; k < IN; ++k) {
      const float4 x = *reinterpret_cast<const float4*>(s_in + k * TE + 4 * quad);
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
    // relu, fc2 (agent.py:34) as one fmaf chain per action, softmax (:35), Categorical sample + log_prob (:44-46)
    uint32_t act4 = 0u;
    float lp[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float l[NA];
#pragma unroll
      for (int c = 0; c < NA; ++c) l[c] = s_b2[ag * C::B2S + c];
#pragma unroll
      for (int u = 0; u < H; ++u) {
        const float r = fmaxf((u & 1) ? h2[k][u >> 1].y : h2[k][u >> 1].x, 0.f);
#pragma unroll
        for (int c = 0; c < NA; ++c) l[c] = fmaf(r, w2[u * NA + c], l[c]);
      }
      const uint64_t id = (uint64_t)(a.env_offset + e0 + k);
      const uint4 o = policy_words(id, t_word, ep_hi, ag >> 2, key);
      int pick;
      policy_head(l, word_of(o, ag & 3), pick, lp[k]);
      act4 |= (uint32_t)pick << (8 * k);
    }
    if (e0 < a.ld) {
      st_stream_u32(a.actions + (int64_t)ag * a.ld + e0, act4);
      if (a.logp) st_stream_f4(a.logp + (int64_t)ag * a.ld + e0, make_float4(lp[0], lp[1], lp[2], lp[3]));
    }
  }
}

// Launch policy_act_discrete_kernel<A, NA> for a.ld envs (a.n_tiles is set here) on a persistent grid of at most the
// resident CTAs of sms SMs.
template <int NA>
int launch_policy_fp32(PolicyArgs a, int n_agents, int sms, cudaStream_t st) {
  return dispatch<1, 32>(n_agents, [&](auto kA) {
    using C = PolCfg<kA, NA>;
    auto kern = policy_act_discrete_kernel<kA, NA>;
    const size_t smem = C::kSmemFloats * sizeof(float);
    if (smem > 48 * 1024) SMARL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 1;
    SMARL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, C::THREADS, smem));
    if (per_sm < 1) per_sm = 1;
    a.n_tiles = (a.ld + C::TE - 1) / C::TE;
    const int64_t grid = a.n_tiles < (int64_t)sms * per_sm ? a.n_tiles : (int64_t)sms * per_sm;
    SMARL_CUDA(launch_pdl(kern, (unsigned)grid, C::THREADS, smem, st, a));
    SMARL_CUDA(cudaGetLastError());
    return SMARL_OK;
  });
}

// Every agent's policy for the four consecutive envs of one on-policy rollout thread at one step, on the joint
// observation held as packed u8 position words (x_i of env k in byte k of xw[i]), in policy_act_discrete_kernel<A, 5>'s
// operation order, so the actions and log-probabilities are its bits: fc1 as packed FFMA2 from b1 over k = 0..2A-1,
// relu, fc2 from log2(e) b2 over u = 0..15 (packed FFMA2 over the env pairs (0, 1) and (2, 3): per env the closed loop's
// fmaf chain, with half the issue slots), then policy_head.  One Philox block serves four consecutive agents of an env.
// s_w holds the weights as stage_discrete_policy<A, kPolActions, .> put them.  aw[i] receives agent i's four action
// bytes.  A live thread (one whose envs exist) stores them and the log-probabilities at step t, env e0 of the [T][A][ld]
// records act_rec / logp_rec that are not NULL.
template <int A>
__device__ __forceinline__ void discrete_policy_step4(const uint32_t (&xw)[A], const uint32_t (&yw)[A], const float* s_w,
                                                      uint2 key, uint64_t id0, uint32_t t_word, uint32_t ep_hi,
                                                      uint32_t (&aw)[A], uint8_t* act_rec, float* logp_rec, bool live,
                                                      int t, int64_t ld, int64_t e0) {
  using C = PolCfg<A, kPolActions>;
  constexpr int IN = C::IN, H = kPolHidden, NA = kPolActions;
  const float* s_w1 = s_w;
  const float* s_w2 = s_w1 + A * C::W1S;
  const float* s_b1 = s_w2 + A * C::W2S;
  const float* s_b2 = s_b1 + A * H;
  uint4 words[4];
#pragma unroll
  for (int ag = 0; ag < A; ++ag) {
    if ((ag & 3) == 0) {
#pragma unroll
      for (int k = 0; k < 4; ++k) words[k] = policy_words(id0 + k, t_word, ep_hi, ag >> 2, key);
    }
    const float* w1 = s_w1 + ag * C::W1S;
    const float* w2 = s_w2 + ag * C::W2S;
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
    float2 l2[2][NA];
#pragma unroll
    for (int c = 0; c < NA; ++c) l2[0][c] = l2[1][c] = make_float2(s_b2[ag * C::B2S + c], s_b2[ag * C::B2S + c]);
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
      if (act_rec) st_stream_u32(act_rec + ((int64_t)t * A + ag) * ld + e0, act4);
      if (logp_rec) st_stream_f4(logp_rec + ((int64_t)t * A + ag) * ld + e0, make_float4(lp[0], lp[1], lp[2], lp[3]));
    }
  }
}
#endif

}  // namespace smarl
