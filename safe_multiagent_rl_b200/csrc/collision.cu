// CollisionAvoidance on sm_100a (float64 state).  One thread owns one env: a warp moves
// 32 x 8 B = 256 contiguous bytes per f64 row and 128 B per f32 / i32 row, all agent-major SoA.
//
// This file restates the reference's float64 arithmetic operation by operation so that
// positions, done flags and collision counts are bit-exact; it is compiled with -fmad=false
// and uses the _rn intrinsics wherever a contraction would change a rounding.
#include <stdlib.h>

#include "collision.cuh"

// Built as three translation units (build.py compiles this file once per SMARL_TU value):
//   0 step kernel   1 fused rollout kernel   2 reset kernel + C entry points

namespace smarl {

#if SMARL_TU_IS(0)
// CAP: 64 registers (8 CTAs per SM) for A <= 4 on large batches, where occupancy pays (2^22 envs: closed loop +6.6 %,
// fused +9 %); a one-wave batch like config 1 (65 536 envs) is latency-bound per thread and loses 3 % to the spills.
template <int A, bool CAP>
__global__ void __launch_bounds__(kCollThreads, (CAP ? 8 : 0)) collision_step_kernel(const CollisionStepArgs a) {
  pdl_prologue();   // programmatic dependent launch: the previous grid has completed past this point (common.cuh)
  __shared__ double2 s_clip[A <= SMARL_COLL_COMPACT_MAX_A ? kCollThreads / 32 : 1][A <= SMARL_COLL_COMPACT_MAX_A ? kClipSlots : 1];   // 4 KB, or a dummy
  constexpr bool kCompact = A <= SMARL_COLL_COMPACT_MAX_A;
  const int64_t eg = (int64_t)blockIdx.x * kCollThreads + threadIdx.x;
  const bool live = eg < a.n_envs;
  if (!kCompact && !live) return;                             // compaction is warp-wide: there every lane stays
  const int64_t e = live ? eg : a.n_envs - 1;
  const int64_t ld = a.ld;
  double px[A], py[A];
  float adx[A], ady[A];
  uint32_t done_mask = 0u;
#pragma unroll
  for (int i = 0; i < A; ++i) {
    px[i] = a.pos_x[i * ld + e];
    py[i] = a.pos_y[i * ld + e];
    adx[i] = a.actions[(2 * i) * ld + e];
    ady[i] = a.actions[(2 * i + 1) * ld + e];
    done_mask |= a.done[i * ld + e] ? (1u << i) : 0u;
  }
  const double lx0 = a.landmarks[e], ly0 = a.landmarks[ld + e];
  const int32_t steps_before = a.episode_len ? a.episode_len[e] : 0;
  const uint32_t all = A == 32 ? 0xFFFFFFFFu : ((1u << A) - 1u);
  const bool active = live && done_mask != all;               // main.py:51: episode already over
  double reward = 0.0;
  int collisions = 0;
  if constexpr (kCompact) {
    collision_transition_compact<A>(px, py, done_mask, active, adx, ady, a.size, s_clip[threadIdx.x >> 5]);
    if (!live) return;
    if (active)
      collision_env_step<A, true>(px, py, done_mask, a.landmarks + e, ld, a.L, lx0, ly0, a.size, a.agents_size, reward, collisions);
  } else if (active) {
    collision_transition_inline<A>(px, py, done_mask, adx, ady, a.size);
    collision_env_step<A, true>(px, py, done_mask, a.landmarks + e, ld, a.L, lx0, ly0, a.size, a.agents_size, reward, collisions);
  }
  const float rf = (float)reward;
#pragma unroll
  for (int i = 0; i < A; ++i) {
    if (active) {
      a.pos_x[i * ld + e] = px[i];
      a.pos_y[i * ld + e] = py[i];
      a.done[i * ld + e] = (uint8_t)((done_mask >> i) & 1u);
    }
    if (a.done_out) a.done_out[i * ld + e] = (uint8_t)((done_mask >> i) & 1u);
    if (a.reward_rows != 1 || i == 0) a.reward[i * ld + e] = rf;
  }
  if (a.obs) {
    if (!a.normalize) {                                       // the common case stays free of float64 divisions
#pragma unroll
      for (int i = 0; i < A; ++i) {
        a.obs[(2 * i) * ld + e] = (float)px[i];
        a.obs[(2 * i + 1) * ld + e] = (float)py[i];
      }
      if (a.obs_landmarks)                                    // :141-142 (shuffle=True layout)
        for (int l = 0; l < 2 * a.L; ++l) a.obs[(2 * A + l) * ld + e] = (float)a.landmarks[l * ld + e];
    } else {                                                  // _normalize_state, :164-165
      // A rolled loop indexes px / py dynamically, which makes the compiler keep a local-memory shadow of the positions
      // for the whole kernel (also when normalize is off); unrolled, with the division out of line, they stay in
      // registers.  Measured closed loop, unrolled vs rolled: A=3 +6 %, A=8 +3.5 %, A=24 +31 %, A=32 +33 %, but A=16
      // -10 % (the shadow copy happens to relieve the register allocation there), hence the middle range stays rolled.
      if constexpr (A <= 10 || A >= 22) {
#pragma unroll
        for (int i = 0; i < A; ++i) {
          a.obs[(2 * i) * ld + e] = obs_normalized(px[i], a.size);
          a.obs[(2 * i + 1) * ld + e] = obs_normalized(py[i], a.size);
        }
      } else {
#pragma unroll 1
        for (int i = 0; i < A; ++i) {
          a.obs[(2 * i) * ld + e] = obs_value(px[i], a.size, 1);
          a.obs[(2 * i + 1) * ld + e] = obs_value(py[i], a.size, 1);
        }
      }
      if (a.obs_landmarks)
        for (int l = 0; l < 2 * a.L; ++l) a.obs[(2 * A + l) * ld + e] = obs_value(a.landmarks[l * ld + e], a.size, 1);
    }
  }
  a.cost[e] = collisions;
  if (a.episode_len && active) a.episode_len[e] = steps_before + 1;
  if (a.penalty) a.penalty[e] = (float)(__ldg(a.lambdas) * (double)collisions);   // meta_agent.py:21-22
}

int launch_collision_step(int A, const CollisionStepArgs& a, unsigned grid, cudaStream_t s) {
  if (A <= 4 && a.n_envs >= kCollCapMinEnvs)
    return dispatch<1, 4>(A, [&](auto kA) {
      SMARL_CUDA(launch_pdl(collision_step_kernel<kA, true>, grid, kCollThreads, 0, s, a));
      SMARL_CUDA(cudaGetLastError());
      return SMARL_OK;
    });
  return dispatch<1, 32>(A, [&](auto kA) {
    SMARL_CUDA(launch_pdl(collision_step_kernel<kA, false>, grid, kCollThreads, 0, s, a));
    SMARL_CUDA(cudaGetLastError());
    return SMARL_OK;
  });
}
#endif

#if SMARL_TU_IS(1)
template <int A, bool CAP>
// (second launch bound: 0 = unspecified -- 1 would lift the compiler's register heuristic to 255 and cost A = 8 10 %;
//  A = 5..8 is held to 5 CTAs per SM / 96 registers: fused A = 6 +13 %, A = 8 +7 % on 2^20..2^21 envs)
__global__ void __launch_bounds__(kCollThreads, (CAP ? 8 : (A >= 5 && A <= 8 ? 5 : 0))) collision_rollout_kernel(const CollisionRolloutArgs a) {
  __shared__ double s_red[kCollThreads / 32];
  __shared__ double2 s_clip[A <= SMARL_COLL_COMPACT_ROLLOUT_MAX_A ? kCollThreads / 32 : 1][A <= SMARL_COLL_COMPACT_ROLLOUT_MAX_A ? kClipSlots : 1];
  const int64_t eg = (int64_t)blockIdx.x * kCollThreads + threadIdx.x;
  const bool live = eg < a.n_envs;
  const int64_t e = live ? eg : 0;
  const int64_t ld = a.ld;
  const int T = a.n_steps;
  double px[A], py[A];
#pragma unroll
  for (int i = 0; i < A; ++i) {
    px[i] = a.start_x[i * ld + e];
    py[i] = a.start_y[i * ld + e];
  }
  const uint32_t all = A == 32 ? 0xFFFFFFFFu : ((1u << A) - 1u);
  const double lam = a.lambdas ? __ldg(a.lambdas) : 0.0;
  uint32_t done_mask = 0u;
  double s_rew = 0.0, s_pen = 0.0, disc = 1.0;
  int csum = 0, steps = 0;
  for (int t = 0; t < T; ++t) {
    double reward = 0.0;
    int collisions = 0;
    const bool active = done_mask != all;               // main.py:51 (lanes past n_envs replay env 0 and store nothing)
    if constexpr (A <= SMARL_COLL_COMPACT_ROLLOUT_MAX_A) {
      float adx[A], ady[A];
#pragma unroll
      for (int i = 0; i < A; ++i) {
        adx[i] = active ? a.actions[((int64_t)t * 2 * A + 2 * i) * ld + e] : 0.f;
        ady[i] = active ? a.actions[((int64_t)t * 2 * A + 2 * i + 1) * ld + e] : 0.f;
      }
      collision_transition_compact<A>(px, py, done_mask, active, adx, ady, a.size, s_clip[threadIdx.x >> 5]);
      if (active) {
        collision_env_step<A, false>(px, py, done_mask, a.landmarks + e, ld, a.L, 0.0, 0.0, a.size, a.agents_size, reward, collisions);
        ++steps;
      }
    } else if (active) {
      float adx[A], ady[A];
#pragma unroll
      for (int i = 0; i < A; ++i) {
        adx[i] = a.actions[((int64_t)t * 2 * A + 2 * i) * ld + e];
        ady[i] = a.actions[((int64_t)t * 2 * A + 2 * i + 1) * ld + e];
      }
      collision_transition_inline<A>(px, py, done_mask, adx, ady, a.size);
      collision_env_step<A, false>(px, py, done_mask, a.landmarks + e, ld, a.L, 0.0, 0.0, a.size, a.agents_size, reward, collisions);
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
    const double bc = block_sum<kCollThreads>(live ? (double)csum : 0.0, s_red);
    const double bv = block_sum<kCollThreads>((live && a.thresholds && (double)csum > thr) ? 1.0 : 0.0, s_red);
    const double br = block_sum<kCollThreads>(live ? s_rew : 0.0, s_red);
    const double bm = block_sum<kCollThreads>(live ? s_rew - s_pen : 0.0, s_red);
    if (threadIdx.x == 0) {
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

int launch_collision_rollout(int A, const CollisionRolloutArgs& a, unsigned grid, cudaStream_t s) {
  if (A <= 4 && a.n_envs >= kCollCapMinEnvs)
    return dispatch<1, 4>(A, [&](auto kA) {
      collision_rollout_kernel<kA, true><<<grid, kCollThreads, 0, s>>>(a);
      SMARL_CUDA(cudaGetLastError());
      return SMARL_OK;
    });
  return dispatch<1, 32>(A, [&](auto kA) {
    collision_rollout_kernel<kA, false><<<grid, kCollThreads, 0, s>>>(a);
    SMARL_CUDA(cudaGetLastError());
    return SMARL_OK;
  });
}
#endif

#if SMARL_TU_IS(2)
__global__ void collision_reset_kernel(const double* __restrict__ start_x, const double* __restrict__ start_y,
                                       const double* __restrict__ landmarks, double* __restrict__ pos_x,
                                       double* __restrict__ pos_y, uint8_t* __restrict__ done,
                                       int32_t* __restrict__ episode_len, float* __restrict__ obs, int A, int L,
                                       int obs_landmarks, int normalize, double size, int64_t n_envs, int64_t ld) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_envs) return;
  if (episode_len) episode_len[e] = 0;
  for (int i = 0; i < A; ++i) {
    const double x = start_x[i * ld + e], y = start_y[i * ld + e];
    pos_x[i * ld + e] = x;
    pos_y[i * ld + e] = y;
    done[i * ld + e] = 0;
    if (obs) {
      obs[(2 * i) * ld + e] = obs_value(x, size, normalize);
      obs[(2 * i + 1) * ld + e] = obs_value(y, size, normalize);
    }
  }
  if (obs && obs_landmarks)
    for (int l = 0; l < 2 * L; ++l) obs[(2 * A + l) * ld + e] = obs_value(landmarks[l * ld + e], size, normalize);
}

// Lanes per env: 0 = one thread per env (collision.cu), 2 / 4 = lane-cooperative kernels (collision_coop.cu).
// Crossover measured on B200 (profiles/r02): see DESIGN.md section 3.3.  smarl_set_kernel_variant overrides it.
int collision_coop_lanes(int A, int L, int64_t ld, bool rollout) {
  if (A < 9) return 0;
  if ((int64_t)(2 * A + 2 * L + 2) * ld >= (1ll << 32)) return 0;   // the cooperative kernels use 32-bit element offsets
  const int forced = kernel_variant(SMARL_ENV_COLLISION);
  if (forced >= 0) return forced;
  // 2^20 envs, T = 20, one thread / 2 lanes (profiles/r02/crossover_a9_11.md): step A = 9 3.38 / 3.66 ms, A = 10 3.76 / 3.72,
  // A = 11 6.13 / 4.19; fused rollout A = 9 2.08 / 1.80, A = 10 3.26 / 1.80, A = 11 3.62 / 2.17
  if (A < (rollout ? 9 : 11)) return 0;
  return A <= 16 ? 2 : 4;
}

#endif

}  // namespace smarl

using namespace smarl;

#if SMARL_TU_IS(2)
extern "C" int smarl_collision_reset(const SmarlCollisionParams* p, const double* start_x,
                                     const double* start_y, const double* landmarks, double* pos_x,
                                     double* pos_y, uint8_t* done, int32_t* episode_len, float* obs,
                                     int64_t n_envs, int64_t ld, smarl_stream_t stream) {
  if (int rc = check_collision(p)) return rc;
  if (int rc = check_layout(n_envs, ld)) return rc;
  SMARL_REQUIRE(start_x && start_y && landmarks && pos_x && pos_y && done, "null required pointer");
  SMARL_REQUIRE(p->n_agents >= 1 && p->n_agents <= SMARL_MAX_AGENTS, "n_agents=%d outside 1..32", p->n_agents);
  const unsigned grid = (unsigned)((n_envs + 255) / 256);
  collision_reset_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(start_x, start_y, landmarks, pos_x, pos_y,
                                                                 done, episode_len, obs, p->n_agents, p->n_landmarks,
                                                                 p->obs_landmarks, p->normalize_state, (double)p->size,
                                                                 n_envs, ld);
  SMARL_CUDA(cudaGetLastError());
  return SMARL_OK;
}

extern "C" int smarl_collision_step(const SmarlCollisionParams* p, double* pos_x, double* pos_y,
                                    uint8_t* done, const float* actions, const double* landmarks,
                                    float* obs, float* reward, int32_t* cost, uint8_t* done_out,
                                    int32_t* episode_len, const double* lambdas, float* penalty,
                                    int64_t n_envs, int64_t ld, smarl_stream_t stream) {
  if (int rc = check_collision(p)) return rc;
  if (int rc = check_layout(n_envs, ld)) return rc;
  SMARL_REQUIRE(pos_x && pos_y && done && actions && landmarks && reward && cost, "null required pointer");
  SMARL_REQUIRE((lambdas == nullptr) == (penalty == nullptr), "lambdas and penalty go together");
  CollisionStepArgs a;
  a.pos_x = pos_x; a.pos_y = pos_y; a.done = done; a.actions = actions; a.landmarks = landmarks;
  a.obs = obs; a.reward = reward; a.cost = cost; a.done_out = done_out; a.episode_len = episode_len;
  a.lambdas = lambdas;
  a.penalty = penalty; a.n_envs = n_envs; a.ld = ld; a.size = (double)p->size;
  a.agents_size = p->agents_size; a.L = p->n_landmarks; a.obs_landmarks = p->obs_landmarks;
  a.normalize = p->normalize_state;
  a.reward_rows = p->reward_rows == 1 ? 1 : 0;
  if (const int lanes = collision_coop_lanes(p->n_agents, p->n_landmarks, ld, false))
    return launch_collision_coop_step(p->n_agents, lanes, a, (cudaStream_t)stream);
  const unsigned grid = (unsigned)((n_envs + kCollThreads - 1) / kCollThreads);
  if (int rc = launch_collision_step(p->n_agents, a, grid, (cudaStream_t)stream)) return rc;
  return SMARL_OK;
}

extern "C" int smarl_collision_rollout(const SmarlCollisionParams* p, const SmarlAccounting* acc,
                                       const double* start_x, const double* start_y,
                                       const double* landmarks, const float* actions,
                                       const double* lambdas, double* final_x, double* final_y,
                                       uint8_t* final_done, int32_t* n_active, float* R, float* modR,
                                       int32_t* C, float* G, float* g_scratch, double* stats,
                                       double* stats_scratch, int64_t n_envs, int64_t ld,
                                       smarl_stream_t stream) {
  if (int rc = check_collision(p)) return rc;
  if (int rc = check_layout(n_envs, ld)) return rc;
  if (int rc = check_accounting(acc, INT32_MAX, 2, G, stats, stats_scratch)) return rc;
  SMARL_REQUIRE(start_x && start_y && landmarks && actions && R && modR && C, "null required pointer");
  SMARL_REQUIRE(acc->g_mode != 1 || g_scratch, "g_mode 1 needs g_scratch [2][T][ld]");
  CollisionRolloutArgs a;
  a.start_x = start_x; a.start_y = start_y; a.landmarks = landmarks; a.actions = actions;
  a.lambdas = lambdas; a.final_x = final_x; a.final_y = final_y; a.final_done = final_done;
  a.n_active = n_active; a.R = R; a.modR = modR; a.C = C; a.G = G; a.g_scratch = g_scratch;
  a.partials = stats_scratch; a.thresholds = acc->thresholds; a.gamma = acc->gamma; a.n_envs = n_envs;
  a.ld = ld; a.size = (double)p->size; a.agents_size = p->agents_size; a.L = p->n_landmarks;
  a.n_steps = acc->n_steps; a.g_mode = acc->g_mode;
  unsigned grid = (unsigned)((n_envs + kCollThreads - 1) / kCollThreads);
  if (const int lanes = collision_coop_lanes(p->n_agents, p->n_landmarks, ld, true)) {
    const int64_t envs_per_cta = kCollThreads / lanes;     // the cooperative kernels run 128 / lanes envs per CTA
    grid = (unsigned)((n_envs + envs_per_cta - 1) / envs_per_cta);
    if (int rc = launch_collision_coop_rollout(p->n_agents, lanes, a, (cudaStream_t)stream)) return rc;
  } else if (int rc = launch_collision_rollout(p->n_agents, a, grid, (cudaStream_t)stream)) {
    return rc;
  }
  if (stats)
    return launch_stats_finalize(stats_scratch, grid, p->n_agents, 1, n_envs, stats, (cudaStream_t)stream);
  return SMARL_OK;
}
#endif
