// Fused per-agent discrete policies for the grid envs (sm_100a): the caller of the env step.
//
// Replaces, for n_envs envs and all agents at once, DiscretePolicy.forward / act of the reference
// (safe_multi_agent_RL/agent.py:23-47, called per agent and step from main.py:30-35 through
// AbstractAgent.act :118-127): every agent a owns an MLP  obs[2A] -> relu(fc1) [16] -> fc2 [5] -> softmax  fed the
// JOINT state np.array(state).flatten() = (x0, y0, x1, y1, ...), samples an action from the Categorical and keeps
// its log-probability.
//
// The PyTorch glue (policy.py) materialises [A, E, 16] hiddens and [A, E, 5] logits in HBM and launches a dozen
// kernels per step; at 2^18 envs x 16 agents it takes 98 % of the closed loop.  Here one kernel reads the u8
// position rows the env step kernels maintain (2 B per agent, NOT the float observation), keeps every agent's
// weights in shared memory, and writes the u8 action row and the f32 log-prob row: ~7 B per agent-step of HBM
// traffic.  The work is 2A*16 + 16*5 multiply-adds per agent-step (592 at A = 16).  This file evaluates all of them on
// the FP32 pipes; policy_tc.cu (the default) runs fc1 as tcgen05 GEMMs with a 3-way bf16 split of the weights that
// keeps the 1e-5 log-prob parity, and is 3x faster at A = 16.
//
// Thread mapping: one thread = one agent x four consecutive envs (64 hidden accumulators in registers); a CTA =
// all A agents x QPT env quads, looping over tiles of 4*QPT envs (persistent grid), so the weights are staged once
// per CTA.  Per input k a thread issues one LDS.128 for the four envs' value and four LDS.128 for the 16 weights
// (both conflict-free broadcasts) against 64 FFMA.
//
// Sampling (policy.cuh, shared with the tensor-core build): Philox4x32-10 with counter (global env id lo, hi,
// t | episode << 16, agent >> 2 | (episode >> 16) << 3) and key seed ^ "PLCY"; agent a takes word a & 3,
// u = min(((w >> 8) + 0.5) * 2^-24, 1 - 2^-24) in float32; the action is the inverse CDF of the softmax, a = #{c : sum_{c' <= c} e_c' <= u * sum_c e_c}.  Streams do not depend
// on sharding, nor on which of the two builds runs.
//
// This file is the FP32-pipe build (all 592 multiply-adds as packed FFMA2, two per issue slot); policy_tc.cu puts fc1
// on the tensor cores.  smarl_set_kernel_variant(SMARL_KERNEL_POLICY, 0 / 1 / 2) forces one; by default the
// tensor-core build serves every shape it fits.
#include <math.h>

#include "policy.cuh"
#include "tc.cuh"

namespace smarl {

template <int A>
struct PolCfg {
  static constexpr int IN = 2 * A;
  // env quads per tile: all A agents x QPT quads = one CTA of 96..256 threads
  static constexpr int QPT = A >= 16 ? 8 : (A >= 8 ? 16 : (A >= 4 ? 32 : 64));
  static constexpr int THREADS = A * QPT;
  static constexpr int TE = 4 * QPT;                          // envs per tile
  static constexpr int W1S = IN * kPolHidden + 4;             // floats per agent (+4: agents land on different banks)
  static constexpr int W2S = kPolHidden * kPolActions + 4;
  static constexpr size_t kSmemFloats = (size_t)A * W1S + (size_t)A * W2S + (size_t)A * kPolHidden + (size_t)A * 8 +
                                        (size_t)IN * TE;
};

template <int A>
__global__ void __launch_bounds__(PolCfg<A>::THREADS) policy_act_discrete_kernel(const PolicyArgs a) {
  pdl_prologue();   // programmatic dependent launch: the previous grid has completed past this point (common.cuh)
  using C = PolCfg<A>;
  constexpr int IN = C::IN, QPT = C::QPT, TE = C::TE, H = kPolHidden, NA = kPolActions;
  extern __shared__ float s_mem[];
  float* s_w1 = s_mem;                               // [A][W1S]  w1[a][k][u]
  float* s_w2 = s_w1 + A * C::W1S;                   // [A][W2S]  w2[a][u][c]
  float* s_b1 = s_w2 + A * C::W2S;                   // [A][16]
  float* s_b2 = s_b1 + A * H;                        // [A][8]
  float* s_in = s_b2 + A * 8;                        // [IN][TE] the joint observation of the tile, as floats
  const int tid = threadIdx.x;
  for (int i = tid; i < A * IN * H; i += C::THREADS) s_w1[(i / (IN * H)) * C::W1S + i % (IN * H)] = __ldg(a.w1 + i);
  for (int i = tid; i < A * H * NA; i += C::THREADS) s_w2[(i / (H * NA)) * C::W2S + i % (H * NA)] = __ldg(a.w2 + i) * kLog2e;   // logits in log2 units (policy_head)
  for (int i = tid; i < A * H; i += C::THREADS) s_b1[i] = __ldg(a.b1 + i);
  for (int i = tid; i < A * NA; i += C::THREADS) s_b2[(i / NA) * 8 + i % NA] = __ldg(a.b2 + i) * kLog2e;
  const int ag = tid / QPT, quad = tid % QPT;
  const uint2 key = policy_key(a.seed);
  const uint32_t episode = a.episode + (a.episode_dev ? __ldg(a.episode_dev) : 0u);
  const uint32_t t_word = a.t | episode << 16, ep_hi = policy_episode_hi(episode);
  const float* w1 = s_w1 + ag * C::W1S;
  const float* w2 = s_w2 + ag * C::W2S;

  for (int64_t tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int64_t e_tile = tile * TE;
    if (tile != (int64_t)blockIdx.x) __syncthreads();   // previous tile fully consumed; the first tile's position loads
                                                        // go out right behind the weight loads (one barrier covers both)
    // stage the tile's positions as floats: row 2i = x_i, row 2i+1 = y_i (main.py:33: np.array(state).flatten())
    for (int i = tid; i < IN * QPT; i += C::THREADS) {
      const int row = i / QPT, qd = i % QPT;
      const int64_t e = e_tile + 4 * qd;
      const uint8_t* src = (row & 1) ? a.pos_y : a.pos_x;
      const uint32_t w = e < a.ld ? ld_stream_u32(src + (int64_t)(row >> 1) * a.ld + e) : 0u;
      *reinterpret_cast<float4*>(s_in + row * TE + 4 * qd) = bytes_to_float4(w);
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
    // relu, fc2 (agent.py:34), softmax (:35), Categorical sample + log_prob (:44-46)
    uint32_t act4 = 0u;
    float lp[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float l[NA];
#pragma unroll
      for (int c = 0; c < NA; ++c) l[c] = s_b2[ag * 8 + c];
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

}  // namespace smarl

using namespace smarl;

extern "C" int smarl_policy_act_discrete(const SmarlDiscretePolicy* p, const uint8_t* pos_x, const uint8_t* pos_y,
                                         uint8_t* actions, float* logp, int32_t t, int64_t n_envs, int64_t ld,
                                         smarl_stream_t stream) {
  SMARL_REQUIRE(p != nullptr, "policy params is NULL");
  if (int rc = check_layout(n_envs, ld)) return rc;
  SMARL_REQUIRE(p->n_agents >= 1 && p->n_agents <= SMARL_MAX_AGENTS, "n_agents=%d outside 1..32", p->n_agents);
  if (int rc = check_discrete_policy(p, p->n_agents)) return rc;
  SMARL_REQUIRE(pos_x && pos_y && actions, "null pointer");
  SMARL_REQUIRE(t >= 0 && t < 65536, "t=%d outside 0..65535", t);
  SMARL_REQUIRE(aligned16(pos_x) && aligned16(pos_y) && aligned16(actions) && aligned16(logp), "pointers must be 16-byte aligned");
  PolicyArgs a;
  a.pos_x = pos_x; a.pos_y = pos_y; a.actions = actions; a.logp = logp; a.w1 = p->w1; a.b1 = p->b1; a.w2 = p->w2;
  a.b2 = p->b2; a.seed = p->seed; a.env_offset = p->env_offset; a.n_envs = n_envs; a.ld = ld;
  a.t = (uint32_t)t; a.episode = p->episode; a.episode_dev = p->episode_dev;
  int dev = 0, sms = 148;
  SMARL_CUDA(cudaGetDevice(&dev));
  SMARL_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  cudaStream_t st = (cudaStream_t)stream;
  // fc1 on the tensor cores (policy_tc.cu) unless the FP32-pipe build is forced: -1 / 2 = groups of up to 8 agents and
  // two env tiles per CTA iteration, 1 = groups of up to 16 agents and one tile
  const int variant = kernel_variant(SMARL_KERNEL_POLICY);
  if (variant != 0) return launch_policy_tc(a, p->n_agents, variant == 1 ? 16 : 8, sms, st);
  return dispatch<1, 32>(p->n_agents, [&](auto kA) {
    using C = PolCfg<kA>;
    auto kern = policy_act_discrete_kernel<kA>;
    const size_t smem = C::kSmemFloats * sizeof(float);
    if (smem > 227 * 1024) {
      set_error("policy weights of %d agents need %zu bytes of shared memory", (int)kA, smem);
      return SMARL_EUNSUPPORTED;
    }
    if (smem > 48 * 1024) SMARL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 1;
    SMARL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, C::THREADS, smem));
    a.n_tiles = (ld + C::TE - 1) / C::TE;
    const int64_t grid = a.n_tiles < (int64_t)sms * per_sm ? a.n_tiles : (int64_t)sms * per_sm;
    SMARL_CUDA(launch_pdl(kern, (unsigned)grid, C::THREADS, smem, st, a));
    SMARL_CUDA(cudaGetLastError());
    return SMARL_OK;
  });
}
