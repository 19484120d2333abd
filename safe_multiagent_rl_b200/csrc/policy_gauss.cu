// Fused per-agent Gaussian policies for the continuous envs (CollisionAvoidance, CoverageContinuous): the caller of
// their step kernels (sm_100a).
//
// Replaces, for n_envs envs and all agents at once, ContinuousPolicy.forward / get_dist / act of the reference
// (safe_multi_agent_RL/agent.py:48-76, called per agent and step from main.py:30-35 through AbstractAgent.act
// :118-127): every agent a owns an MLP  obs[S] -> relu(fc1) [16] -> (mu = fc2 [2], sigma^2 = relu(fc2_) [2] + 1e-4),
// fed the JOINT state np.array(state).flatten(), samples a ~ N(mu, diag(sigma^2)) (MultivariateNormal with a diagonal
// covariance) and keeps log N(a; mu, diag(sigma^2)).
//
// One kernel reads the f32 observation rows the step kernels maintain ([S][ld], S = 2A, or 2A + 2L with shuffled
// landmarks), keeps every agent's weights in shared memory and writes the f32 action rows the step consumes
// (dx0, dy0, dx1, ...: [2A][ld]) and the f32 log-probability row: 4 S / A + 12 B per agent-step of HBM traffic instead
// of the [A, E, 16] hiddens and three [A, E, 2] heads of the PyTorch glue.  Thread mapping as in policy.cu: one thread =
// one agent x four consecutive envs, fc1 as packed FFMA2, persistent CTAs.  (fc1 of the discrete policies runs on the
// tensor cores, policy_tc.cu, because u8 grid positions are exact in bf16; f32 observations would need a 3 x 3 piece
// split, and at the agent counts of the continuous envs' configs -- 3 to 8 -- the kernel is not fc1-bound.)
//
// Sampling: Philox4x32-10, counter (global env id lo, hi, t | episode << 16,
// agent >> 1 | (episode >> 16) << 4), key seed ^ "GAUS" (hi word):
// one block serves two agents, agent a takes words w[2 (a & 1)], w[2 (a & 1) + 1];  u_k = ((w_k >> 9) + 0.5) * 2^-23
// (23 bits: exact in f32, never 0 or 1),
// Box-Muller  r = sqrt(-2 ln u_0), z = (r cos(2 pi u_1), r sin(2 pi u_1)),  action_k = mu_k + sqrt(sigma_k^2) z_k,
// log_prob = -1/2 sum ((action_k - mu_k)^2 / sigma_k^2 + ln sigma_k^2) - ln(2 pi), evaluated on the ROUNDED action as
// dist.log_prob(action) is.  oracle/philox.py restates it.  Streams do not depend on sharding.
#include <math.h>

#include "policy.cuh"
#include "tc.cuh"

namespace smarl {

constexpr int kGaussActions = 2;

struct GaussArgs {
  const float* obs;
  float* actions;
  float* logp;
  const float* w1;     // [A][S][16]
  const float* b1;     // [A][16]
  const float* w_mu;   // [A][16][2]
  const float* b_mu;   // [A][2]
  const float* w_var;  // [A][16][2]
  const float* b_var;  // [A][2]
  uint64_t seed;
  int64_t env_offset;
  int64_t n_envs;
  int64_t ld;
  int64_t n_tiles;
  uint32_t t;
  uint32_t episode;    // *episode_dev is added on the device
  const uint32_t* episode_dev;
  int32_t S;
};

template <int A>
struct GaussCfg {
  static constexpr int QPT = A >= 16 ? 8 : (A >= 8 ? 16 : (A >= 4 ? 32 : 64));   // env quads per tile
  static constexpr int THREADS = A * QPT;
  static constexpr int TE = 4 * QPT;                                             // envs per tile
  static constexpr int HS = kPolHidden * 4 + 4;                                  // head floats per agent: [u][mu0 mu1 v0 v1]
  static size_t smem_floats(int S) {
    return (size_t)A * ((size_t)S * kPolHidden + 4) + (size_t)A * HS + (size_t)A * kPolHidden + (size_t)A * 4 + (size_t)S * TE;
  }
};

template <int A>
__global__ void __launch_bounds__(GaussCfg<A>::THREADS) policy_act_gaussian_kernel(const GaussArgs a) {
  pdl_prologue();   // programmatic dependent launch: the previous grid has completed past this point (common.cuh)
  using C = GaussCfg<A>;
  constexpr int QPT = C::QPT, TE = C::TE, H = kPolHidden;
  const int S = a.S, W1S = S * H + 4;
  extern __shared__ float s_mem[];
  float* s_w1 = s_mem;                               // [A][W1S]  w1[a][k][u]
  float* s_hd = s_w1 + A * W1S;                      // [A][HS]   heads[a][u][mu0 mu1 v0 v1]
  float* s_b1 = s_hd + A * C::HS;                    // [A][16]
  float* s_bh = s_b1 + A * H;                        // [A][4]    b_mu0 b_mu1 b_var0 b_var1
  float* s_in = s_bh + A * 4;                        // [S][TE]   the joint observation of the tile
  const int tid = threadIdx.x;
  for (int i = tid; i < A * S * H; i += C::THREADS) s_w1[(i / (S * H)) * W1S + i % (S * H)] = __ldg(a.w1 + i);
  for (int i = tid; i < A * H * 4; i += C::THREADS) {
    const int ag = i / (H * 4), u = (i / 4) % H, c = i % 4;
    s_hd[ag * C::HS + u * 4 + c] = c < 2 ? __ldg(a.w_mu + (ag * H + u) * 2 + c) : __ldg(a.w_var + (ag * H + u) * 2 + (c - 2));
  }
  for (int i = tid; i < A * H; i += C::THREADS) s_b1[i] = __ldg(a.b1 + i);
  for (int i = tid; i < A * 4; i += C::THREADS) s_bh[i] = (i & 3) < 2 ? __ldg(a.b_mu + (i >> 2) * 2 + (i & 3)) : __ldg(a.b_var + (i >> 2) * 2 + (i & 3) - 2);
  const int ag = tid / QPT, quad = tid % QPT;
  const uint2 key = make_uint2((uint32_t)a.seed, (uint32_t)(a.seed >> 32) ^ 0x47415553u);   // "GAUS"
  const uint32_t episode = a.episode + (a.episode_dev ? __ldg(a.episode_dev) : 0u);
  const uint32_t t_word = a.t | episode << 16, ep_hi = gauss_episode_hi(episode);
  const float* w1 = s_w1 + ag * W1S;
  const float* hd = s_hd + ag * C::HS;

  for (int64_t tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int64_t e_tile = tile * TE;
    if (tile != (int64_t)blockIdx.x) __syncthreads();   // previous tile fully consumed; the first tile's observation loads
                                                        // go out right behind the weight loads (one barrier covers both)
    for (int i = tid; i < S * QPT; i += C::THREADS) {
      const int row = i / QPT, qd = i % QPT;
      const int64_t e = e_tile + 4 * qd;
      const float4 v = e < a.ld ? ld_stream_f4(a.obs + (int64_t)row * a.ld + e) : make_float4(0.f, 0.f, 0.f, 0.f);
      *reinterpret_cast<float4*>(s_in + row * TE + 4 * qd) = v;
    }
    __syncthreads();
    const int64_t e0 = e_tile + 4 * quad;
    // fc1 (agent.py:60) as packed FFMA2: h2[k][p] = (h[k][2p], h[k][2p+1]) for the four envs k of this thread
    float2 h2[4][H / 2];
#pragma unroll
    for (int p = 0; p < H / 2; ++p) {
      const float2 b = *reinterpret_cast<const float2*>(s_b1 + ag * H + 2 * p);
      h2[0][p] = h2[1][p] = h2[2][p] = h2[3][p] = b;
    }
#pragma unroll 2
    for (int k = 0; k < S; ++k) {
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
    // relu, the two heads (agent.py:61-62), sample (:73) and log_prob (:74)
    float ax[4], ay[4], lp[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float2 mu = make_float2(s_bh[ag * 4 + 0], s_bh[ag * 4 + 1]), var = make_float2(s_bh[ag * 4 + 2], s_bh[ag * 4 + 3]);
#pragma unroll
      for (int u = 0; u < H; ++u) {
        const float r = fmaxf((u & 1) ? h2[k][u >> 1].y : h2[k][u >> 1].x, 0.f);
        const float4 w = *reinterpret_cast<const float4*>(hd + 4 * u);
        mu = tc::ffma2(make_float2(r, r), make_float2(w.x, w.y), mu);
        var = tc::ffma2(make_float2(r, r), make_float2(w.z, w.w), var);
      }
      const float v0 = fmaxf(var.x, 0.f) + 1e-4f, v1 = fmaxf(var.y, 0.f) + 1e-4f;      // relu(fc2_) + 1e-4 (:67)
      const uint64_t id = (uint64_t)(a.env_offset + e0 + k);
      const uint4 o = philox4x32_10(make_uint4((uint32_t)id, (uint32_t)(id >> 32), t_word, ep_hi | (uint32_t)(ag >> 1)), key);
      const uint32_t wa = (ag & 1) ? o.z : o.x, wb = (ag & 1) ? o.w : o.y;
      const float u0 = ((float)(wa >> 9) + 0.5f) * (1.0f / 8388608.0f), u1 = ((float)(wb >> 9) + 0.5f) * (1.0f / 8388608.0f);   // exact in f32, in (0, 1)
      const float rad = sqrtf(-2.0f * logf(u0));
      float sn, cs;
      sincospif(2.0f * u1, &sn, &cs);
      const float a0 = fmaf(sqrtf(v0), rad * cs, mu.x), a1 = fmaf(sqrtf(v1), rad * sn, mu.y);
      const float d0 = a0 - mu.x, d1 = a1 - mu.y;
      ax[k] = a0;
      ay[k] = a1;
      lp[k] = -0.5f * (d0 * d0 / v0 + d1 * d1 / v1 + logf(v0) + logf(v1)) - 1.8378770664093453f;   // ln(2 pi)
    }
    if (e0 < a.ld) {
      st_stream_f4(a.actions + (int64_t)(2 * ag) * a.ld + e0, make_float4(ax[0], ax[1], ax[2], ax[3]));
      st_stream_f4(a.actions + (int64_t)(2 * ag + 1) * a.ld + e0, make_float4(ay[0], ay[1], ay[2], ay[3]));
      if (a.logp) st_stream_f4(a.logp + (int64_t)ag * a.ld + e0, make_float4(lp[0], lp[1], lp[2], lp[3]));
    }
  }
}

}  // namespace smarl

using namespace smarl;

extern "C" int smarl_policy_act_gaussian(const SmarlGaussianPolicy* p, const float* obs, float* actions, float* logp,
                                         int32_t t, int64_t n_envs, int64_t ld, smarl_stream_t stream) {
  SMARL_REQUIRE(p != nullptr, "policy params is NULL");
  if (int rc = check_layout(n_envs, ld)) return rc;
  SMARL_REQUIRE(p->n_agents >= 1 && p->n_agents <= SMARL_MAX_AGENTS, "n_agents=%d outside 1..32", p->n_agents);
  SMARL_REQUIRE(p->state_size >= 1 && p->state_size <= 2 * SMARL_MAX_AGENTS + 128, "state_size=%d outside 1..%d",
                p->state_size, 2 * SMARL_MAX_AGENTS + 128);
  SMARL_REQUIRE(p->hidden == kPolHidden && p->n_actions == kGaussActions,
                "only the reference's ContinuousPolicy shape (hidden 16, 2 actions) is built (got %d, %d)", p->hidden,
                p->n_actions);
  SMARL_REQUIRE(p->w1 && p->b1 && p->w_mu && p->b_mu && p->w_var && p->b_var && obs && actions, "null pointer");
  SMARL_REQUIRE(t >= 0 && t < 65536, "t=%d outside 0..65535", t);
  SMARL_REQUIRE(aligned16(obs) && aligned16(actions) && aligned16(logp), "pointers must be 16-byte aligned");
  GaussArgs a;
  a.obs = obs; a.actions = actions; a.logp = logp; a.w1 = p->w1; a.b1 = p->b1; a.w_mu = p->w_mu; a.b_mu = p->b_mu;
  a.w_var = p->w_var; a.b_var = p->b_var; a.seed = p->seed; a.env_offset = p->env_offset; a.n_envs = n_envs; a.ld = ld;
  a.t = (uint32_t)t; a.episode = p->episode; a.episode_dev = p->episode_dev; a.S = p->state_size;
  int dev = 0, sms = 148;
  SMARL_CUDA(cudaGetDevice(&dev));
  SMARL_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  cudaStream_t st = (cudaStream_t)stream;
  return dispatch<1, 32>(p->n_agents, [&](auto kA) {
    using C = GaussCfg<kA>;
    auto kern = policy_act_gaussian_kernel<kA>;
    const size_t smem = C::smem_floats(a.S) * sizeof(float);
    if (smem > 227 * 1024) {
      set_error("policy weights of %d agents with %d inputs need %zu bytes of shared memory", (int)kA, a.S, smem);
      return SMARL_EUNSUPPORTED;
    }
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
