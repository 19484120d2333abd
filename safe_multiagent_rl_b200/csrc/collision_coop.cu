// CollisionAvoidance, lane-cooperative kernels for large agent counts (sm_100a).
//
// One env is split over S = 2 or 4 lanes of a warp ("group"): lane s owns agents i = j*S + s, j = 0..B-1,
// B = ceil(A/S), so that the float64 state of an env (16 B per agent) never has to fit one thread's
// registers -- the one-thread-per-env kernels of collision.cu need 168-255 registers from A = 16 and run
// 2-3 CTAs per SM with a local-memory shadow of the positions.  A warp holds 32/S envs; lane = s*(32/S) + q
// with q the env inside the warp, so every load / store instruction of the agent-major SoA arrays touches S
// rows x (32/S) consecutive envs: full 32-byte sectors for every f64 / f32 row.
//
//   transition, landmark reach, per-agent minima   own agents only, same per-agent code as collision.cu
//   reward = -np.sum(minima)                       numpy's pairwise association: the 8 running accumulators
//                                                  r_k (k = i mod 8) are lane-local because S divides 8, the
//                                                  combining tree runs over xor-shuffles, the tail over broadcasts
//   collisions                                     every lane publishes its agents' new positions to shared
//                                                  memory (exact f64 + an f32 copy stored twice so that the
//                                                  circular partner index needs no modulo); agent i screens the
//                                                  partners i+1 .. i+A/2 (mod A) in f32 -- each unordered pair once,
//                                                  balanced over the lanes -- and only pairs inside the screen get
//                                                  the exact f64 test; the per-lane counts meet in a shuffle sum.
//
// Bit-exactness: the per-agent arithmetic is shared with collision.cu (collision.cuh); the reward uses the very
// association numpy_sum<A> uses; the collision count is an integer.  Compiled with -fmad=false.
#include <stdlib.h>

#include "collision.cuh"

// Built as two translation units (build.py compiles this file once per SMARL_TU value): 0 step, 1 rollout.

namespace smarl {

constexpr int kCoopThreads = 128;

template <int A, int S>
struct CollCoop {
  static constexpr int B = (A + S - 1) / S;          // agents per lane
  static constexpr int EPW = 32 / S;                 // envs per warp
  static constexpr int EPC = kCoopThreads / S;       // envs per CTA
  static constexpr int H = A / 2;                    // circular partner window (the last offset halved for even A)
  static constexpr bool kGhost = (A % S) != 0;       // some lanes own a padding agent at j = B-1
  static constexpr int PA = A | 1;                   // double2 stride per env: odd => conflict-free STS.128 / LDS.128
  static constexpr int FS = S == 2 ? (A | 1) : (((A + 3) & ~3) | 2);   // float2 stride per env (LDS.64)
  static constexpr int NS = A | 1;                   // float stride per env of the squared norms (LDS.32)
  static constexpr size_t kSmem = (size_t)EPC * (PA * sizeof(double2) + FS * sizeof(float2) + NS * sizeof(float)) +
                                  (size_t)(kCoopThreads / 32) * kClipSlots * sizeof(double2);
};

// (clip_action and kClipSlots live in collision.cuh: the one-thread kernels compact their clips the same way)

// Exact test of one pair (the arithmetic of pair_collides in collision.cuh) on values instead of arrays.
static __device__ __noinline__ int pair_collides_xy(double xi, double yi, double xj, double yj, double lim2_lo,
                                                    double lim2_hi, double lim) {
  const double dx = __dadd_rn(xi, -xj), dy = __dadd_rn(yi, -yj);
  const double q = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
  if (q < lim2_lo) return 1;
  return (q < lim2_hi && __dsqrt_rn(q) < lim) ? 1 : 0;
}

__device__ __forceinline__ double shfl_xor_f64(double v, int lane_mask) {
  return __shfl_xor_sync(0xffffffffu, v, lane_mask);
}
__device__ __forceinline__ double shfl_f64(double v, int src_lane) { return __shfl_sync(0xffffffffu, v, src_lane); }

// -np.sum of the A per-agent minima held as v[j] (agent j*S + s) in numpy's pairwise association
// (numpy_sum<A> in collision.cuh): identical on all S lanes of the group.  A >= 8.
template <int A, int S>
__device__ __forceinline__ double coop_numpy_sum(const double (&v)[CollCoop<A, S>::B], int q) {
  constexpr int EPW = CollCoop<A, S>::EPW;
  constexpr int NK = 8 / S;                 // accumulators r_k, k = kk*S + s, owned by this lane
  constexpr int kFull = A - (A % 8);
  double acc[NK];
  // agent 8m + k lives at j = (8m + k) / S = NK*m + kk on lane s = k % S
#pragma unroll
  for (int kk = 0; kk < NK; ++kk) acc[kk] = v[kk];
#pragma unroll
  for (int m = 1; m < kFull / 8; ++m) {
#pragma unroll
    for (int kk = 0; kk < NK; ++kk) acc[kk] = __dadd_rn(acc[kk], v[NK * m + kk]);
  }
  // ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)): the first log2(S) levels pair lanes (a + b == b + a exactly) ...
#pragma unroll
  for (int off = 1; off < S; off <<= 1) {
#pragma unroll
    for (int kk = 0; kk < NK; ++kk) acc[kk] = __dadd_rn(acc[kk], shfl_xor_f64(acc[kk], off * EPW));
  }
  // ... the rest is local
  double s;
  if constexpr (NK == 4) s = __dadd_rn(__dadd_rn(acc[0], acc[1]), __dadd_rn(acc[2], acc[3]));
  else s = __dadd_rn(acc[0], acc[1]);
  // tail agents kFull .. A-1, sequentially, each broadcast from its owner lane
#pragma unroll
  for (int i = kFull; i < A; ++i) s = __dadd_rn(s, shfl_f64(v[i / S], (i % S) * EPW + q));
  return s;
}

// One CollisionAvoidance.step of the group's env.  px/py/done_bits (bit j = own agent j) are updated in place;
// reward (identical on every lane of the group) and the group's collision count are returned.  Must be called by
// all 32 lanes (shuffles, __syncwarp); envs past their episode end simply have all agents done.
template <int A, int S, bool COMPACT>
__device__ __forceinline__ void collision_coop_env_step(double (&px)[CollCoop<A, S>::B], double (&py)[CollCoop<A, S>::B],
                                                        uint32_t& done_bits, const float (&adx)[CollCoop<A, S>::B],
                                                        const float (&ady)[CollCoop<A, S>::B],
                                                        const double* __restrict__ lm, int64_t ld, int L, double size,
                                                        double agents_size, int s, int q, double2* __restrict__ sp,
                                                        float2* __restrict__ sf, float* __restrict__ sn,
                                                        double2* __restrict__ clip, double& reward, int& collisions) {
  using C = CollCoop<A, S>;
  constexpr int B = C::B, H = C::H, EPW = C::EPW;
  // transition (collision_avoidance.py:103-121); padding agents carry a set done bit.
  // The clip to unit norm (:113-117) costs an f64 sqrt and two f64 divisions (~100 instructions) for the agents whose
  // action is longer than 1 -- a minority, but in practice some lane of every warp has one for every agent slot j, so
  // inlined per slot the whole warp pays it B times.  Instead the clips of a warp are COMPACTED: every agent that
  // needs one gets a rank (ballot + popc), posts its f32 action to shared memory, the lanes work the posted list
  // off round-robin (ceil(n / 32) rounds instead of B) and the owners pick their f64 result up.  Ranks beyond the
  // kClipSlots slots (an unusually clip-heavy warp) are evaluated in place.  Same arithmetic, same bits.
  if constexpr (!COMPACT) {
#pragma unroll
    for (int j = 0; j < B; ++j) {
      if ((done_bits >> j) & 1u) continue;
      collision_move_agent(px[j], py[j], adx[j], ady[j], size);
    }
  } else {
    const unsigned lane = threadIdx.x & 31u, lt = (1u << lane) - 1u;
    uint32_t need = 0u;
    int rank[B];
    int n_clip = 0;
#pragma unroll
    for (int j = 0; j < B; ++j) {
      const double dx = (double)adx[j], dy = (double)ady[j];
      const double q = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));   // :113 (dx**2 == dx*dx for fp32-origin values)
      const bool nd = !((done_bits >> j) & 1u) && q > 1.0;     // sqrt_rn is monotonic with sqrt_rn(1) == 1: norm > 1 needs q > 1
      const unsigned b = __ballot_sync(0xffffffffu, nd);
      rank[j] = n_clip + __popc(b & lt);
      n_clip += __popc(b);
      need |= nd ? (1u << j) : 0u;
      if (nd && rank[j] < kClipSlots) *reinterpret_cast<float2*>(clip + rank[j]) = make_float2(adx[j], ady[j]);
    }
    __syncwarp();
    for (int r = (int)lane; r < min(n_clip, kClipSlots); r += 32) {
      const float2 in = *reinterpret_cast<const float2*>(clip + r);
      clip[r] = clip_action(in.x, in.y);
    }
    __syncwarp();
#pragma unroll
    for (int j = 0; j < B; ++j) {
      double2 d = make_double2((double)adx[j], (double)ady[j]);
      if ((need >> j) & 1u) d = rank[j] < kClipSlots ? clip[rank[j]] : clip_action(adx[j], ady[j]);
      if (!((done_bits >> j) & 1u)) {
        px[j] = fmax(0.0, fmin(size, __dadd_rn(px[j], d.x)));      // :118
        py[j] = fmax(0.0, fmin(size, __dadd_rn(py[j], d.y)));      // :119
      }
    }
    __syncwarp();                       // the slots are reused by the next step
  }
  // landmark reach (:122-124) and per-agent minimum landmark distance (:158-161)
  double minq[B];
  uint32_t reach = 0u;
  const double as2 = agents_size * agents_size;
  const double as2_lo = as2 * 0.999999999, as2_hi = as2 * 1.000000001;
#pragma unroll
  for (int j = 0; j < B; ++j) minq[j] = 1.0e300;
  for (int l = 0; l < L; ++l) {
    const double lx = lm[(2 * l) * ld], ly = lm[(2 * l + 1) * ld];
#pragma unroll
    for (int j = 0; j < B; ++j)
      reach |= collision_landmark(px[j], py[j], lx, ly, agents_size, as2_lo, as2_hi, minq[j]) ? (1u << j) : 0u;
  }
  double mind[B];
#pragma unroll
  for (int j = 0; j < B; ++j) {
    mind[j] = __dsqrt_rn(minq[j]);
    if (C::kGhost && j == B - 1 && (j * S + s >= A)) mind[j] = 0.0;
  }
  done_bits |= reach & ~done_bits;   // only agents that moved this step are tested; done ones stay done
  reward = -coop_numpy_sum<A, S>(mind, q);   // :127-130, all agents incl. done ones

  // collisions among agents not done after this step (:150-156)
  const double lim = 2.0 * agents_size;
  const double lim2 = lim * lim;
  const double lim2_lo = lim2 * 0.999999, lim2_hi = lim2 * 1.000001;
  // f32 screen in expanded form, 4 instructions per pair (FFMA, FFMA, FSETP, predicated OR):
  //   |p_j - p_o|^2 < T   <=>   fma(-2 x_j, x_o, fma(-2 y_j, y_o, n_o)) < T - n_j,     n = x^2 + y^2,
  // with the partner's (x, y, n) read from shared memory.  Seven f32 roundings of magnitude <= 4 size^2 bound the
  // error by 28 * 2^-24 size^2 < size^2 * 2^-19; the threshold adds twice that to the coordinate-rounding margin
  // of collision_screen_q, so no pair inside the exact test's reach is ever screened out.
  const float T = (float)((double)collision_screen_q(lim, size) + size * size * (1.0 / 262144.0)) * 1.000001f;
  const float inf = __int_as_float(0x7f800000);
  float mx2[B], my2[B], thr[B];
#pragma unroll
  for (int j = 0; j < B; ++j) {
    const int i = j * S + s;
    const bool alive = !((done_bits >> j) & 1u);
    // done (and padding) agents never collide (:150-156 counts agents not done): as partners they publish a squared
    // norm of +inf, which makes every screen value they enter +inf (the two products are finite), on any field; as
    // owners their threshold is -inf.  (Their f32 coordinates stay parked at (4096 (i + 1), 0), which was the whole
    // exclusion once and missed partners near that point on fields >= 4096; they no longer decide anything.)
    const float fx = alive ? (float)px[j] : 4096.0f * (float)(i + 1);
    const float fy = alive ? (float)py[j] : 0.0f;
    const float n = fmaf(fy, fy, fx * fx);
    mx2[j] = -2.0f * fx;
    my2[j] = -2.0f * fy;
    thr[j] = alive ? T - n : -inf;
    if (!C::kGhost || j < B - 1 || i < A) {
      sp[i] = make_double2(px[j], py[j]);
      sf[i] = make_float2(fx, fy);
      sn[i] = alive ? n : inf;
    }
  }
  __syncwarp();
  // agent i screens partners (i + k) mod A, k = 1..H; for even A the offset k = H pairs each couple twice, so
  // only the lower half (i < H) counts it.  One LDS.64 + LDS.32 per partner offset c = j*S + k serves every own agent.
  uint32_t near[B];
#pragma unroll
  for (int j = 0; j < B; ++j) {
    near[j] = 0u;
  }
  const float2* sfs = sf + s;
  const float* sns = sn + s;
#pragma unroll
  for (int c = 1; c <= (B - 1) * S + H; ++c) {
    // partner index (s + c) mod A: known at compile time except for the S-1 offsets around the wrap
    const int cw = (c + S - 1 < A) ? c : (c >= A ? c - A : ((s + c >= A) ? c - A : c));
    const float2 p = sfs[cw];
    const float pn = sns[cw];
#pragma unroll
    for (int j = 0; j < B; ++j) {
      const int k = c - j * S;
      if (k >= 1 && k <= H) {
        const float v = fmaf(mx2[j], p.x, fmaf(my2[j], p.y, pn));
        if (A % 2 == 0 && k == H) {
          if (v < thr[j] && (j * S + s < H)) near[j] |= 1u << k;
        } else {
          asm("{\n\t.reg .pred q;\n\tsetp.lt.f32 q, %1, %2;\n\t@q or.b32 %0, %0, %3;\n\t}"
              : "+r"(near[j])
              : "f"(v), "f"(thr[j]), "r"(1u << k));
        }
      }
    }
  }
  int n = 0;
#pragma unroll
  for (int j = 0; j < B; ++j) {
    uint32_t m = near[j];
    while (m) {
      const int k = __ffs((int)m) - 1;
      m &= m - 1u;
      int ip = j * S + s + k;
      ip = ip >= A ? ip - A : ip;
      const double2 o = sp[ip];
      n += pair_collides_xy(px[j], py[j], o.x, o.y, lim2_lo, lim2_hi, lim);
    }
  }
#pragma unroll
  for (int off = 1; off < S; off <<= 1) n += __shfl_xor_sync(0xffffffffu, n, off * EPW);
  collisions = n;
  __syncwarp();                      // the next step's stores must not overtake this step's partner loads
}

#if SMARL_TU_IS(0)
template <int A, int S, bool COMPACT>
__global__ void __launch_bounds__(kCoopThreads, 5) collision_coop_step_kernel(const CollisionStepArgs a) {
  pdl_prologue();   // programmatic dependent launch: the previous grid has completed past this point (common.cuh)
  using C = CollCoop<A, S>;
  constexpr int B = C::B, EPW = C::EPW, EPC = C::EPC;
  extern __shared__ double2 s_pos[];                                  // [EPC][PA]
  float2* s_f = reinterpret_cast<float2*>(s_pos + EPC * C::PA);       // [EPC][FS]
  float* s_n = reinterpret_cast<float*>(s_f + EPC * C::FS);           // [EPC][NS]
  double2* s_clip = reinterpret_cast<double2*>(reinterpret_cast<char*>(s_pos) + C::kSmem) - (kCoopThreads / 32) * kClipSlots +
                    (threadIdx.x >> 5) * kClipSlots;                   // [warps][kClipSlots]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int q = lane % EPW, s = lane / EPW;
  const int el = warp * EPW + q;
  const int64_t eg = (int64_t)blockIdx.x * EPC + el;
  const bool live = eg < a.n_envs;
  const int64_t e = live ? eg : 0;
  const int64_t ld = a.ld;

  // 32-bit element offsets (the dispatcher checks (2A + 2L + 2) * ld < 2^32): one add per row, one wide
  // multiply-add per access
  const uint32_t ld32 = (uint32_t)ld;
  const uint32_t row0 = (uint32_t)s * ld32 + (uint32_t)e;      // agent s, this env
  double px[B], py[B];
  float adx[B], ady[B];
  uint32_t done_bits = 0u;
#pragma unroll
  for (int j = 0; j < B; ++j) {
    const uint32_t off = row0 + (uint32_t)(j * S) * ld32;       // agent i = j*S + s
    if (!C::kGhost || j < B - 1 || j * S + s < A) {
      px[j] = a.pos_x[off];
      py[j] = a.pos_y[off];
      adx[j] = a.actions[2u * off - (uint32_t)e];              // row 2i:   2*i*ld + e
      ady[j] = a.actions[2u * off - (uint32_t)e + ld32];       // row 2i+1
      done_bits |= a.done[off] ? (1u << j) : 0u;
    } else {
      px[j] = py[j] = 0.0;
      adx[j] = ady[j] = 0.f;
      done_bits |= 1u << j;
    }
  }
  const int32_t steps_before = (a.episode_len && s == 0) ? a.episode_len[e] : 0;
  // main.py:51: the episode is over once every agent of the env is done
  const uint32_t gmask = (S == 2 ? 0x00010001u : 0x01010101u) << q;
  const bool all_done = done_bits == ((1u << B) - 1u);
  const bool active = (__ballot_sync(0xffffffffu, all_done) & gmask) != gmask;

  double reward = 0.0;
  int collisions = 0;
  collision_coop_env_step<A, S, COMPACT>(px, py, done_bits, adx, ady, a.landmarks + e, ld, a.L, a.size, a.agents_size, s, q,
                                s_pos + el * C::PA, s_f + el * C::FS, s_n + el * C::NS, s_clip, reward, collisions);
  if (!live) return;
  const float rf = active ? (float)reward : 0.f;
  const bool all_rows = a.reward_rows != 1;
#pragma unroll
  for (int j = 0; j < B; ++j) {
    if (C::kGhost && j == B - 1 && j * S + s >= A) continue;
    const uint32_t off = row0 + (uint32_t)(j * S) * ld32;
    const uint8_t d = (uint8_t)((done_bits >> j) & 1u);
    if (active) {
      a.pos_x[off] = px[j];
      a.pos_y[off] = py[j];
      a.done[off] = d;
    }
    if (a.done_out) a.done_out[off] = d;
    if (all_rows || (j == 0 && s == 0)) a.reward[off] = rf;
  }
  if (a.obs) {
    if (!a.normalize) {
#pragma unroll
      for (int j = 0; j < B; ++j) {
        if (C::kGhost && j == B - 1 && j * S + s >= A) continue;
        const uint32_t o2 = 2u * (row0 + (uint32_t)(j * S) * ld32) - (uint32_t)e;
        a.obs[o2] = (float)px[j];
        a.obs[o2 + ld32] = (float)py[j];
      }
    } else {                                                    // _normalize_state, :164-165
#pragma unroll
      for (int j = 0; j < B; ++j) {
        if (C::kGhost && j == B - 1 && j * S + s >= A) continue;
        const uint32_t o2 = 2u * (row0 + (uint32_t)(j * S) * ld32) - (uint32_t)e;
        a.obs[o2] = obs_normalized(px[j], a.size);
        a.obs[o2 + ld32] = obs_normalized(py[j], a.size);
      }
    }
    if (a.obs_landmarks)                                        // :141-142 (shuffle=True layout)
      for (int l = s; l < 2 * a.L; l += S) a.obs[(2 * A + l) * ld + e] = obs_value(a.landmarks[l * ld + e], a.size, a.normalize);
  }
  if (s == 0) {
    a.cost[e] = collisions;
    if (a.episode_len && active) a.episode_len[e] = steps_before + 1;
    if (a.penalty) a.penalty[e] = (float)(__ldg(a.lambdas) * (double)collisions);   // meta_agent.py:21-22
  }
}

template <int S, bool COMPACT>
static int launch_step_s(int A, const CollisionStepArgs& a, cudaStream_t st) {
  return dispatch<9, 32>(A, [&](auto kA) {
    using C = CollCoop<kA, S>;
    auto kern = collision_coop_step_kernel<kA, S, COMPACT>;
    if (C::kSmem > 48 * 1024)
      SMARL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::kSmem));
    const unsigned grid = (unsigned)((a.n_envs + C::EPC - 1) / C::EPC);
    SMARL_CUDA(launch_pdl(kern, grid, kCoopThreads, C::kSmem, st, a));
    SMARL_CUDA(cudaGetLastError());
    return SMARL_OK;
  }, "cooperative Collision kernels cover n_agents 9..32 (got %d)");
}

int launch_collision_coop_step(int A, int S, const CollisionStepArgs& a, cudaStream_t st) {
  // compacting the action clips pays in the fused rollout (-7..17 %) but not in the one-step kernel, whose front of
  // global loads the ballots serialise (measured: A = 32 closed loop 14.4 -> 17.4 ms); SMARL_COLL_COMPACT=1 forces it
  static const char* env = getenv("SMARL_COLL_COMPACT");
  const bool compact = env && atoi(env) != 0;
  if (compact) return S == 2 ? launch_step_s<2, true>(A, a, st) : launch_step_s<4, true>(A, a, st);
  return S == 2 ? launch_step_s<2, false>(A, a, st) : launch_step_s<4, false>(A, a, st);
}
#endif

#if SMARL_TU_IS(1)
// Fused open-loop episode (main.py:28-57 minus the policy nets, incl. the early break at :51): the group's
// positions / done bits / discounted sums stay in registers for all T steps.
template <int A, int S, bool COMPACT>
__global__ void __launch_bounds__(kCoopThreads, 5) collision_coop_rollout_kernel(const CollisionRolloutArgs a) {
  using C = CollCoop<A, S>;
  constexpr int B = C::B, EPW = C::EPW, EPC = C::EPC;
  extern __shared__ double2 s_pos[];
  float2* s_f = reinterpret_cast<float2*>(s_pos + EPC * C::PA);
  float* s_n = reinterpret_cast<float*>(s_f + EPC * C::FS);
  double2* s_clip = reinterpret_cast<double2*>(reinterpret_cast<char*>(s_pos) + C::kSmem) - (kCoopThreads / 32) * kClipSlots +
                    (threadIdx.x >> 5) * kClipSlots;
  __shared__ double s_red[kCoopThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int q = lane % EPW, s = lane / EPW;
  const int el = warp * EPW + q;
  const int64_t eg = (int64_t)blockIdx.x * EPC + el;
  const bool live = eg < a.n_envs;
  const int64_t e = live ? eg : 0;
  const int64_t ld = a.ld;
  const int T = a.n_steps;
  const uint32_t gmask = (S == 2 ? 0x00010001u : 0x01010101u) << q;

  double px[B], py[B];
  uint32_t done_bits = 0u;
  bool own[B];
#pragma unroll
  for (int j = 0; j < B; ++j) {
    const int i = j * S + s;
    own[j] = !C::kGhost || j < B - 1 || i < A;
    px[j] = own[j] ? a.start_x[i * ld + e] : 0.0;
    py[j] = own[j] ? a.start_y[i * ld + e] : 0.0;
    done_bits |= own[j] ? 0u : (1u << j);
  }
  const double lam = a.lambdas ? __ldg(a.lambdas) : 0.0;
  double s_rew = 0.0, s_pen = 0.0, disc = 1.0;
  int csum = 0, steps = 0;
  for (int t = 0; t < T; ++t) {
    const bool all_done = done_bits == ((1u << B) - 1u);
    const bool active = (__ballot_sync(0xffffffffu, all_done) & gmask) != gmask;
    float adx[B], ady[B];
    const float* act_t = a.actions + (int64_t)t * 2 * A * ld;    // uniform; per-lane offsets stay 32-bit
#pragma unroll
    for (int j = 0; j < B; ++j) {
      const uint32_t o2 = 2u * (uint32_t)(j * S + s) * (uint32_t)ld + (uint32_t)e;
      const bool ldok = own[j] && active;
      adx[j] = ldok ? act_t[o2] : 0.f;
      ady[j] = ldok ? act_t[o2 + (uint32_t)ld] : 0.f;
    }
    double reward = 0.0;
    int collisions = 0;
    collision_coop_env_step<A, S, COMPACT>(px, py, done_bits, adx, ady, a.landmarks + e, ld, a.L, a.size, a.agents_size, s, q,
                                  s_pos + el * C::PA, s_f + el * C::FS, s_n + el * C::NS, s_clip, reward, collisions);
    if (!active) reward = 0.0;                 // collisions is 0 by itself: every agent is done
    steps += active ? 1 : 0;
    const float rf = (float)reward;
    const float pf = (float)(lam * (double)collisions);
    s_rew += disc * (double)rf;
    s_pen += disc * (double)pf;
    csum += collisions;
    if (a.g_mode == 1 && live && s == 0) {
      a.g_scratch[(int64_t)t * ld + e] = rf;
      a.g_scratch[((int64_t)T + t) * ld + e] = pf;
    } else if (a.g_mode == 2 && live) {
      const float o = (float)(disc * ((double)rf - (double)pf));
#pragma unroll
      for (int j = 0; j < B; ++j)
        if (own[j]) a.G[((int64_t)t * A + j * S + s) * ld + e] = o;
    }
    disc *= a.gamma;
  }
  if (live) {
    const float r = (float)s_rew, m = (float)(s_rew - s_pen);
#pragma unroll
    for (int j = 0; j < B; ++j) {
      const int i = j * S + s;
      if (!own[j]) continue;
      if (a.final_x) a.final_x[i * ld + e] = px[j];
      if (a.final_y) a.final_y[i * ld + e] = py[j];
      if (a.final_done) a.final_done[i * ld + e] = (uint8_t)((done_bits >> j) & 1u);
      a.R[i * ld + e] = r;
      a.modR[i * ld + e] = m;
    }
    if (s == 0) {
      a.C[e] = csum;
      if (a.n_active) a.n_active[e] = steps;
    }
  }
  if (a.partials) {
    double* out = a.partials + (int64_t)blockIdx.x * stats_len(A, 1);
    const bool mine = live && s == 0;
    const double thr = a.thresholds ? __ldg(a.thresholds) : 0.0;
    const double bc = block_sum<kCoopThreads>(mine ? (double)csum : 0.0, s_red);
    const double bv = block_sum<kCoopThreads>((mine && a.thresholds && (double)csum > thr) ? 1.0 : 0.0, s_red);
    const double br = block_sum<kCoopThreads>(mine ? s_rew : 0.0, s_red);
    const double bm = block_sum<kCoopThreads>(mine ? s_rew - s_pen : 0.0, s_red);
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
      for (int j = 0; j < B; ++j)
        if (own[j]) a.G[((int64_t)t * A + j * S + s) * ld + e] = o;
    }
  }
}

template <int S, bool COMPACT>
static int launch_rollout_s(int A, const CollisionRolloutArgs& a, cudaStream_t st) {
  return dispatch<9, 32>(A, [&](auto kA) {
    using C = CollCoop<kA, S>;
    auto kern = collision_coop_rollout_kernel<kA, S, COMPACT>;
    if (C::kSmem + 64 > 48 * 1024)
      SMARL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::kSmem));
    const unsigned grid = (unsigned)((a.n_envs + C::EPC - 1) / C::EPC);
    kern<<<grid, kCoopThreads, C::kSmem, st>>>(a);
    SMARL_CUDA(cudaGetLastError());
    return SMARL_OK;
  }, "cooperative Collision kernels cover n_agents 9..32 (got %d)");
}

int launch_collision_coop_rollout(int A, int S, const CollisionRolloutArgs& a, cudaStream_t st) {
  static const char* env = getenv("SMARL_COLL_COMPACT");
  const bool compact = !env || atoi(env) != 0;
  if (compact) return S == 2 ? launch_rollout_s<2, true>(A, a, st) : launch_rollout_s<4, true>(A, a, st);
  return S == 2 ? launch_rollout_s<2, false>(A, a, st) : launch_rollout_s<4, false>(A, a, st);
}
#endif

}  // namespace smarl
