// The reference's ContinuousPolicy (agent.py:48-76) evaluated by one thread for one env, with every agent's weights
// in shared memory: the network, the Gaussian head and the Philox Box-Muller sample of the on-policy rollouts
// (collision_policy.cu, coverage_float_policy.cu), and the host side of their policy arguments.
//
// Bit-identity with smarl_policy_act_gaussian is the contract: the arithmetic keeps policy_gauss.cu's evaluation order
// (h[u] = b1[u], then fma(x_k, w1[k][u], .) for k = 0..S-1; the heads from their bias over u = 0..15).  policy_gauss.cu
// is compiled with contraction on, the files including this header with -fmad=false (their f64 accounting relies on
// uncontracted sums): every multiply-add ptxas fuses there is written as an explicit fmaf / ffma2 here.
#pragma once

#include <math.h>

#include "policy.cuh"
#include "tc.cuh"

namespace smarl {

constexpr int kHeadFloats = kPolHidden * 4 + 4;  // per agent: heads [u][mu0 mu1 v0 v1], then b_mu0 b_mu1 b_var0 b_var1

// The policy part of the on-policy rollout kernels' arguments: every agent's weights and the sampling stream.
struct GaussPolicyArgs {
  const float* w1;           // [A][S][16]
  const float* b1;           // [A][16]
  const float* w_mu;         // [A][16][2]
  const float* b_mu;         // [A][2]
  const float* w_var;        // [A][16][2]
  const float* b_var;        // [A][2]
  uint64_t seed;
  int64_t env_offset;
  uint32_t episode;
  const uint32_t* episode_dev;
};

inline GaussPolicyArgs gauss_policy_args(const SmarlGaussianPolicy* pol) {
  GaussPolicyArgs g;
  g.w1 = pol->w1; g.b1 = pol->b1; g.w_mu = pol->w_mu; g.b_mu = pol->b_mu; g.w_var = pol->w_var; g.b_var = pol->b_var;
  g.seed = pol->seed; g.env_offset = pol->env_offset; g.episode = pol->episode; g.episode_dev = pol->episode_dev;
  return g;
}

// A policy for an env of A agents whose observation has S rows, in the one shape the on-policy rollouts build.
inline int check_gaussian_policy(const SmarlGaussianPolicy* pol, int A, int S) {
  SMARL_REQUIRE(pol->n_agents == A, "policy has %d agents, the env %d", pol->n_agents, A);
  SMARL_REQUIRE(pol->state_size == S, "state_size=%d, the env's observation has %d rows", pol->state_size, S);
  SMARL_REQUIRE(pol->hidden == kPolHidden && pol->n_actions == 2,
                "only the reference's ContinuousPolicy shape (hidden 16, 2 actions) is built (got %d, %d)", pol->hidden,
                pol->n_actions);
  SMARL_REQUIRE(pol->w1 && pol->b1 && pol->w_mu && pol->b_mu && pol->w_var && pol->b_var, "null policy weight");
  return SMARL_OK;
}

// One agent's network on the observation (x: the 2A position inputs in registers, lobs: n_lobs further inputs, one
// every LSTRIDE floats), then the Gaussian head: mu and sigma^2 = relu(fc2_) + 1e-4 (agent.py:60-67).
template <int A, int LSTRIDE>
__device__ __forceinline__ void agent_heads(const float (&x)[2 * A], const float* __restrict__ lobs, int n_lobs,
                                            const float* __restrict__ w1, const float* __restrict__ hd, float2& mu,
                                            float& v0, float& v1) {
  constexpr int H = kPolHidden;
  const float* b1 = w1 + (2 * A + n_lobs) * H;
  float2 h2[H / 2];
#pragma unroll
  for (int p = 0; p < H / 2; ++p) h2[p] = *reinterpret_cast<const float2*>(b1 + 2 * p);
#pragma unroll
  for (int k = 0; k < 2 * A; ++k) {
    const float2 xx = make_float2(x[k], x[k]);
    const float4* wr = reinterpret_cast<const float4*>(w1 + k * H);
#pragma unroll
    for (int v = 0; v < H / 4; ++v) {
      const float4 w = wr[v];
      h2[2 * v] = tc::ffma2(xx, make_float2(w.x, w.y), h2[2 * v]);
      h2[2 * v + 1] = tc::ffma2(xx, make_float2(w.z, w.w), h2[2 * v + 1]);
    }
  }
  for (int k = 0; k < n_lobs; ++k) {                  // shuffle=True: the landmark rows follow the positions
    const float xk = lobs[k * LSTRIDE];
    const float2 xx = make_float2(xk, xk);
    const float4* wr = reinterpret_cast<const float4*>(w1 + (2 * A + k) * H);
#pragma unroll
    for (int v = 0; v < H / 4; ++v) {
      const float4 w = wr[v];
      h2[2 * v] = tc::ffma2(xx, make_float2(w.x, w.y), h2[2 * v]);
      h2[2 * v + 1] = tc::ffma2(xx, make_float2(w.z, w.w), h2[2 * v + 1]);
    }
  }
  mu = make_float2(hd[H * 4 + 0], hd[H * 4 + 1]);
  float2 var = make_float2(hd[H * 4 + 2], hd[H * 4 + 3]);
#pragma unroll
  for (int u = 0; u < H; ++u) {
    const float r = fmaxf((u & 1) ? h2[u >> 1].y : h2[u >> 1].x, 0.f);
    const float4 w = *reinterpret_cast<const float4*>(hd + 4 * u);
    mu = tc::ffma2(make_float2(r, r), make_float2(w.x, w.y), mu);
    var = tc::ffma2(make_float2(r, r), make_float2(w.z, w.w), var);
  }
  v0 = fmaxf(var.x, 0.f) + 1e-4f;
  v1 = fmaxf(var.y, 0.f) + 1e-4f;
}

// Box-Muller sample and log N(action; mu, sigma^2) from two Philox words, policy_gauss.cu's arithmetic with its
// contractions spelled out.
__device__ __forceinline__ void gauss_sample(uint32_t wa, uint32_t wb, float2 mu, float v0, float v1, float& a0,
                                             float& a1, float& lp) {
  const float u0 = ((float)(wa >> 9) + 0.5f) * (1.0f / 8388608.0f), u1 = ((float)(wb >> 9) + 0.5f) * (1.0f / 8388608.0f);
  const float rad = sqrtf(-2.0f * logf(u0));
  float sn, cs;
  sincospif(2.0f * u1, &sn, &cs);
  a0 = fmaf(sqrtf(v0), rad * cs, mu.x);
  a1 = fmaf(sqrtf(v1), rad * sn, mu.y);
  const float d0 = a0 - mu.x, d1 = a1 - mu.y;
  lp = fmaf(-0.5f, d0 * d0 / v0 + d1 * d1 / v1 + logf(v0) + logf(v1), -1.8378770664093453f);   // ln(2 pi)
}

}  // namespace smarl
