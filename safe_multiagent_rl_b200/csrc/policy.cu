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
// The FP32-pipe kernel, policy_act_discrete_kernel<A, 5>, and its launcher live in policy.cuh, shared with the 9-action
// closed loop of CoverageDiscretized (policy_discretized.cu), which differs only in reading f32 observation rows.
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
  a.t = (uint32_t)t; a.episode = p->episode; a.episode_dev = p->episode_dev; a.obs = nullptr;
  int dev = 0, sms = 148;
  SMARL_CUDA(cudaGetDevice(&dev));
  SMARL_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  cudaStream_t st = (cudaStream_t)stream;
  // fc1 on the tensor cores (policy_tc.cu) unless the FP32-pipe build is forced: -1 / 2 = groups of up to 8 agents and
  // two env tiles per CTA iteration, 1 = groups of up to 16 agents and one tile
  const int variant = kernel_variant(SMARL_KERNEL_POLICY);
  if (variant != 0) return launch_policy_tc(a, p->n_agents, variant == 1 ? 16 : 8, sms, st);
  return launch_policy_fp32<kPolActions>(a, p->n_agents, sms, st);
}
