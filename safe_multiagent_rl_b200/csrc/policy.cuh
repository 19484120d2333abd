// Shared by the two builds of the fused per-agent discrete policy (policy.cu: FP32 pipes, policy_tc.cu: fc1 on the
// tensor cores): arguments, the Philox stream, and the softmax / inverse-CDF sampling head.
#pragma once

#include "common.cuh"

namespace smarl {

constexpr int kPolHidden = 16;
constexpr int kPolActions = 5;
constexpr float kLog2e = 1.4426950408889634f;

struct PolicyArgs {
  const uint8_t* pos_x;
  const uint8_t* pos_y;
  uint8_t* actions;
  float* logp;
  const float* w1;     // [A][2A][16]
  const float* b1;     // [A][16]
  const float* w2;     // [A][16][5]
  const float* b2;     // [A][5]
  uint64_t seed;
  int64_t env_offset;
  int64_t n_envs;
  int64_t ld;
  int64_t n_tiles;
  uint32_t t;
  uint32_t episode;    // *episode_dev is added on the device
  const uint32_t* episode_dev;
};

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
#endif

}  // namespace smarl
