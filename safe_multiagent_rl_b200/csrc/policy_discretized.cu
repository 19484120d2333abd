// Fused per-agent discrete policies for CoverageDiscretized (sm_100a): the caller of its step kernel.
//
// Replaces, for n_envs envs and all agents at once, DiscretePolicy.forward / act of the reference
// (safe_multi_agent_RL/agent.py:23-47) on the env's 9 actions (coverage.py:210-241): every agent a owns an MLP
// obs[2A] -> relu(fc1) [16] -> fc2 [9] -> softmax fed the JOINT state np.array(state).flatten() = (x0, y0, x1, y1, ...),
// samples an action from the Categorical and keeps its log-probability.
//
// The kernel is policy.cu's FP32-pipe build, policy_act_discrete_kernel<A, 9> in policy.cuh: the positions of this env
// are f64 multiples of 1 / zoom, not u8 grid cells, so it reads the f32 observation rows the reset / step kernels
// maintain ([2A][ld]) instead of the u8 position rows, and writes the u8 action row the step consumes and the f32
// log-probability row.  Thread mapping and weight staging are policy.cu's (dynamic shared memory, opted in above 48 KB:
// 158 KB at A = 32).
//
// Operation order (coverage_discretized_policy.cu reproduces it bit for bit, with explicit fmaf / ffma2 because it is
// compiled with -fmad=false):
//   h[u]  = b1[u];  h[u] = fma(x_k, w1[k][u], h[u]) for k = 0..2A-1 ascending (packed FFMA2 over unit pairs)
//   r[u]  = max(h[u], 0)
//   l2[c] = log2(e) b2[c];  l2[c] = fma(r[u], log2(e) w2[u][c], l2[c]) for u = 0..15 ascending (one fmaf chain per c)
//   policy_head<9> (policy.cuh) on l2: softmax, inverse-CDF sample, log-probability.
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
  PolicyArgs a;
  a.pos_x = nullptr; a.pos_y = nullptr; a.actions = actions; a.logp = logp; a.w1 = p->w1; a.b1 = p->b1; a.w2 = p->w2;
  a.b2 = p->b2; a.seed = p->seed; a.env_offset = p->env_offset; a.n_envs = n_envs; a.ld = ld;
  a.t = (uint32_t)t; a.episode = p->episode; a.episode_dev = p->episode_dev; a.obs = obs;
  int dev = 0, sms = 148;
  SMARL_CUDA(cudaGetDevice(&dev));
  SMARL_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  return launch_policy_fp32<kDiscretizedActions>(a, p->n_agents, sms, (cudaStream_t)stream);
}
