// Fused per-agent discrete policies for CoverageDiscretized (sm_100a): the caller of its step kernel.
//
// Replaces, for n_envs envs and all agents at once, DiscretePolicy.forward / act of the reference
// (safe_multi_agent_RL/agent.py:23-47) on the env's 9 actions (coverage.py:210-241): every agent a owns an MLP
// obs[2A] -> relu(fc1) [16] -> fc2 [9] -> softmax fed the JOINT state np.array(state).flatten() = (x0, y0, x1, y1, ...),
// samples an action from the Categorical and keeps its log-probability.
//
// The positions of this env are f64 multiples of 1 / zoom, not u8 grid cells, so policy.cu's u8 input path does not
// serve it: like policy_gauss.cu this kernel reads the f32 observation rows the reset / step kernels maintain
// ([2A][ld]) and writes the u8 action row the step consumes and the f32 log-probability row.
//
// Thread mapping as in policy.cu / policy_gauss.cu: one thread = one agent x four consecutive envs, a CTA = all A
// agents x QPT env quads looping over tiles of 4 QPT envs (persistent grid), every agent's weights staged once per CTA
// in shared memory (dynamic, opted in above 48 KB: 158 KB at A = 32).
//
// Operation order (coverage_discretized_policy.cu reproduces it bit for bit, with explicit fmaf / ffma2 because it is
// compiled with -fmad=false):
//   h[u]  = b1[u];  h[u] = fma(x_k, w1[k][u], h[u]) for k = 0..2A-1 ascending (packed FFMA2 over unit pairs)
//   r[u]  = max(h[u], 0)
//   l2[c] = log2(e) b2[c];  l2[c] = fma(r[u], log2(e) w2[u][c], l2[c]) for u = 0..15 ascending (one fmaf chain per c)
//   policy_head<9> (policy.cuh) on l2: softmax, inverse-CDF sample, log-probability.
// fc2 / b2 are scaled by log2(e) once when they are staged (the logits in log2 units, as policy.cu).
//
// Sampling: policy.cu's discrete stream unchanged -- Philox4x32-10, counter (global env id lo, hi, t | episode << 16,
// agent >> 2 | (episode >> 16) << 3), key seed ^ "PLCY", agent a takes word a & 3, u = min(((w >> 8) + 0.5) * 2^-24,
// 1 - 2^-24) in float32, action = #{c < 8 : sum_{c' <= c} e_c' <= u * sum e} (oracle/philox.policy_uniforms_f32 /
// policy_sample restate it).
//
// One build, the FP32 pipes: a tensor-core fc1 on f32 observations would need a 3 x 3 bf16 piece split, which does not
// pay at these agent counts (policy_gauss.cu), so smarl_set_kernel_variant(SMARL_KERNEL_POLICY, ...) does not apply.
#include <math.h>

#include "policy.cuh"
#include "tc.cuh"

namespace smarl {

constexpr int kDiscretizedActions = 9;

struct DiscretizedPolicyArgs {
  const float* obs;
  uint8_t* actions;
  float* logp;
  const float* w1;     // [A][2A][16]
  const float* b1;     // [A][16]
  const float* w2;     // [A][16][9]
  const float* b2;     // [A][9]
  uint64_t seed;
  int64_t env_offset;
  int64_t n_envs;
  int64_t ld;
  int64_t n_tiles;
  uint32_t t;
  uint32_t episode;    // *episode_dev is added on the device
  const uint32_t* episode_dev;
};

template <int A>
struct DzCfg {
  static constexpr int IN = 2 * A;
  static constexpr int QPT = A >= 16 ? 8 : (A >= 8 ? 16 : (A >= 4 ? 32 : 64));   // env quads per tile
  static constexpr int THREADS = A * QPT;
  static constexpr int TE = 4 * QPT;                                             // envs per tile
  static constexpr int W1S = IN * kPolHidden + 4;              // floats per agent (+4: agents land on different banks)
  static constexpr int W2S = kPolHidden * kDiscretizedActions + 4;
  static constexpr int B2S = 12;                               // 9 biases, padded so that s_in stays 16-byte aligned
  static constexpr size_t kSmemFloats = (size_t)A * W1S + (size_t)A * W2S + (size_t)A * kPolHidden + (size_t)A * B2S +
                                        (size_t)IN * TE;
  static_assert(kSmemFloats * sizeof(float) <= 227 * 1024, "weights exceed the shared memory of one SM");
};

template <int A>
__global__ void __launch_bounds__(DzCfg<A>::THREADS) policy_act_discretized_kernel(const DiscretizedPolicyArgs a) {
  pdl_prologue();   // programmatic dependent launch: the previous grid has completed past this point (common.cuh)
  using C = DzCfg<A>;
  constexpr int IN = C::IN, QPT = C::QPT, TE = C::TE, H = kPolHidden, NA = kDiscretizedActions;
  extern __shared__ float s_mem[];
  float* s_w1 = s_mem;                               // [A][W1S]  w1[a][k][u]
  float* s_w2 = s_w1 + A * C::W1S;                   // [A][W2S]  log2(e) w2[a][u][c]
  float* s_b1 = s_w2 + A * C::W2S;                   // [A][16]
  float* s_b2 = s_b1 + A * H;                        // [A][B2S]  log2(e) b2[a][c]
  float* s_in = s_b2 + A * C::B2S;                   // [IN][TE]  the joint observation of the tile
  const int tid = threadIdx.x;
  for (int i = tid; i < A * IN * H; i += C::THREADS) s_w1[(i / (IN * H)) * C::W1S + i % (IN * H)] = __ldg(a.w1 + i);
  for (int i = tid; i < A * H * NA; i += C::THREADS) s_w2[(i / (H * NA)) * C::W2S + i % (H * NA)] = __ldg(a.w2 + i) * kLog2e;
  for (int i = tid; i < A * H; i += C::THREADS) s_b1[i] = __ldg(a.b1 + i);
  for (int i = tid; i < A * NA; i += C::THREADS) s_b2[(i / NA) * C::B2S + i % NA] = __ldg(a.b2 + i) * kLog2e;
  const int ag = tid / QPT, quad = tid % QPT;
  const uint2 key = policy_key(a.seed);
  const uint32_t episode = a.episode + (a.episode_dev ? __ldg(a.episode_dev) : 0u);
  const uint32_t t_word = a.t | episode << 16, ep_hi = policy_episode_hi(episode);
  const float* w1 = s_w1 + ag * C::W1S;
  const float* w2 = s_w2 + ag * C::W2S;

  for (int64_t tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int64_t e_tile = tile * TE;
    if (tile != (int64_t)blockIdx.x) __syncthreads();   // previous tile fully consumed; the first tile's observation loads
                                                        // go out right behind the weight loads (one barrier covers both)
    for (int i = tid; i < IN * QPT; i += C::THREADS) {
      const int row = i / QPT, qd = i % QPT;
      const int64_t e = e_tile + 4 * qd;
      const float4 v = e < a.ld ? ld_stream_f4(a.obs + (int64_t)row * a.ld + e) : make_float4(0.f, 0.f, 0.f, 0.f);
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
    // relu, fc2 (agent.py:34), softmax (:35), Categorical sample + log_prob (:44-46)
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

}  // namespace smarl

using namespace smarl;

extern "C" int smarl_policy_act_discretized(const SmarlDiscretePolicy* p, const float* obs, uint8_t* actions,
                                            float* logp, int32_t t, int64_t n_envs, int64_t ld,
                                            smarl_stream_t stream) {
  SMARL_REQUIRE(p != nullptr, "policy params is NULL");
  if (int rc = check_layout(n_envs, ld)) return rc;
  SMARL_REQUIRE(p->n_agents >= 1 && p->n_agents <= SMARL_MAX_AGENTS, "n_agents=%d outside 1..32", p->n_agents);
  if (int rc = check_discrete_policy(p, p->n_agents, kDiscretizedActions)) return rc;
  SMARL_REQUIRE(obs && actions, "null pointer");
  SMARL_REQUIRE(t >= 0 && t < 65536, "t=%d outside 0..65535", t);
  SMARL_REQUIRE(aligned16(obs) && aligned16(actions) && aligned16(logp), "pointers must be 16-byte aligned");
  DiscretizedPolicyArgs a;
  a.obs = obs; a.actions = actions; a.logp = logp; a.w1 = p->w1; a.b1 = p->b1; a.w2 = p->w2; a.b2 = p->b2;
  a.seed = p->seed; a.env_offset = p->env_offset; a.n_envs = n_envs; a.ld = ld;
  a.t = (uint32_t)t; a.episode = p->episode; a.episode_dev = p->episode_dev;
  int dev = 0, sms = 148;
  SMARL_CUDA(cudaGetDevice(&dev));
  SMARL_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  cudaStream_t st = (cudaStream_t)stream;
  return dispatch<1, 32>(p->n_agents, [&](auto kA) {
    using C = DzCfg<kA>;
    auto kern = policy_act_discretized_kernel<kA>;
    const size_t smem = C::kSmemFloats * sizeof(float);
    if (smem > 48 * 1024) SMARL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 1;
    SMARL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, C::THREADS, smem));
    if (per_sm < 1) per_sm = 1;
    a.n_tiles = (ld + C::TE - 1) / C::TE;
    const int64_t grid = a.n_tiles < (int64_t)sms * per_sm ? a.n_tiles : (int64_t)sms * per_sm;
    SMARL_CUDA(launch_pdl(kern, (unsigned)grid, C::THREADS, smem, st, a));
    SMARL_CUDA(cudaGetLastError());
    return SMARL_OK;
  });
}
