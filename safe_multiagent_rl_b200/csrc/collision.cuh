// CollisionAvoidance device code shared by the one-thread-per-env kernels (collision.cu, collision_policy.cu) and the
// lane-cooperative kernels (collision_coop.cu).  Everything here restates the reference's float64
// arithmetic operation by operation; all three files are compiled with -fmad=false.
#pragma once
#include "common.cuh"
#include "stats.cuh"

namespace smarl {

struct CollisionStepArgs {
  double* pos_x;
  double* pos_y;
  uint8_t* done;
  const float* actions;       // [2A][ld]
  const double* landmarks;    // [2L][ld]
  float* obs;
  float* reward;
  int32_t* cost;
  uint8_t* done_out;
  int32_t* episode_len;
  const double* lambdas;
  float* penalty;
  int64_t n_envs;
  int64_t ld;
  double size;
  double agents_size;
  int32_t L;
  int32_t obs_landmarks;
  int32_t normalize;
  int32_t reward_rows;
};

constexpr int kCollThreads = 128;
constexpr int64_t kCollCapMinEnvs = 1 << 18;   // batches from which the A <= 4 kernels run register-capped (see below)

// observation value of a coordinate: the state itself, or state / size with normalize_state
// (collision_avoidance.py:164-165, a float64 division), rounded once to f32.
__device__ __forceinline__ float obs_value(double v, double size, int normalize) {
  return (float)(normalize ? __ddiv_rn(v, size) : v);
}

static __device__ __noinline__ float obs_normalized(double v, double size) { return (float)__ddiv_rn(v, size); }

// numpy's pairwise float64 sum of n <= 128 contiguous values (what np.sum does to the A
// per-agent minima at collision_avoidance.py:161): n < 8 sequential; otherwise 8 running
// accumulators over blocks of 8, combined as ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), then the tail.
template <int N>
__device__ __forceinline__ double numpy_sum(const double (&v)[N]) {
  if (N < 8) {
    double s = 0.0;   // np.sum starts from the first element; 0.0 + v0 == v0 exactly (v0 >= 0)
#pragma unroll
    for (int i = 0; i < N; ++i) s = __dadd_rn(s, v[i]);
    return s;
  }
  double r[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) r[j] = v[j < N ? j : 0];
  constexpr int kFull = N - (N % 8);
#pragma unroll
  for (int i = 8; i < kFull; i += 8) {
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = __dadd_rn(r[j], v[(i + j) < N ? (i + j) : 0]);
  }
  double s = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                       __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
#pragma unroll
  for (int i = kFull; i < N; ++i) s = __dadd_rn(s, v[i]);
  return s;
}

// sqrt_rn(q) < lim, out of line: only ever reached inside the 1e-9 / 1e-6 bands around lim^2 (practically
// never), so the call sites stay three instructions instead of an inlined f64 square root each.
static __device__ __noinline__ bool sqrt_below(double q, double lim) { return __dsqrt_rn(q) < lim; }

// Exact recount of the colliding pairs (sqrt on every pair) for the rare env with a pair inside the
// 1e-6 band around (2 agents_size)^2; rolled loops over a local-memory copy keep it out of the hot code.
static __device__ __noinline__ int collisions_exact(const double* x, const double* y, int A, uint32_t alive,
                                                    double lim) {
  int n = 0;
  for (int i = 0; i < A; ++i)
    for (int j = i + 1; j < A; ++j) {
      const double dx = __dadd_rn(x[i], -x[j]), dy = __dadd_rn(y[i], -y[j]);
      const double q = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
      n += (__dsqrt_rn(q) < lim && ((alive >> i) & (alive >> j) & 1u)) ? 1 : 0;
    }
  return n;
}

// Exact test of one pair (the f64 arithmetic of the pair loop below) for the f32-screened path.
static __device__ __noinline__ int pair_collides(const double* x, const double* y, int i, int j, double lim2_lo,
                                                 double lim2_hi, double lim) {
  const double dx = __dadd_rn(x[i], -x[j]), dy = __dadd_rn(y[i], -y[j]);
  const double q = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
  if (q < lim2_lo) return 1;
  return (q < lim2_hi && __dsqrt_rn(q) < lim) ? 1 : 0;
}

// ---------------------------------------------------------------------------------------
// Fused open-loop episode: positions / done mask / discounted sums in registers for all T
// steps (main.py:28-57 minus the policy nets, incl. the early break at :51).  The env reward
// is shared by all agents, so one (S_rew, S_pen) pair per env serves every agent.
// ---------------------------------------------------------------------------------------
struct CollisionRolloutArgs {
  const double* start_x;
  const double* start_y;
  const double* landmarks;
  const float* actions;      // [T][2A][ld]
  const double* lambdas;
  double* final_x;
  double* final_y;
  uint8_t* final_done;
  int32_t* n_active;
  float* R;
  float* modR;
  int32_t* C;
  float* G;
  float* g_scratch;          // [2][T][ld]
  double* partials;
  const double* thresholds;
  double gamma;
  int64_t n_envs;
  int64_t ld;
  double size;
  double agents_size;
  int32_t L;
  int32_t n_steps;
  int32_t g_mode;
};


// One agent's move (collision_avoidance.py:111-119): clip the action to unit norm, add, clamp to [0,size].
__device__ __forceinline__ void collision_move_agent(double& px, double& py, float adx, float ady, double size) {
  double dx = (double)adx, dy = (double)ady;
  // :113  fp32-origin components: dx**2 == dx*dx exactly, so this is the reference's norm.
  // sqrt_rn is monotonic with sqrt_rn(1) == 1, so norm > 1 needs q > 1: the sqrt (and the two
  // divisions) are only evaluated for actions that can actually be clipped.
  const double q = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
  if (q > 1.0) {
    const double norm = __dsqrt_rn(q);
    if (norm > 1.0) {                                     // :114-117
      dx = __ddiv_rn(dx, norm);
      dy = __ddiv_rn(dy, norm);
    }
  }
  px = fmax(0.0, fmin(size, __dadd_rn(px, dx)));         // :118
  py = fmax(0.0, fmin(size, __dadd_rn(py, dy)));         // :119
}

// The transition of all agents of one env (collision_avoidance.py:103-121), clips inline per agent slot.
template <int A>
__device__ __forceinline__ void collision_transition_inline(double (&px)[A], double (&py)[A], uint32_t done_mask,
                                                            const float (&adx)[A], const float (&ady)[A], double size) {
#pragma unroll
  for (int i = 0; i < A; ++i) {
    if ((done_mask >> i) & 1u) continue;
    collision_move_agent(px[i], py[i], adx[i], ady[i], size);
  }
}

// Agent counts up to which the one-thread STEP kernel compacts its clips over the warp (measured on B200, closed loop,
// ms per 2^20 envs x T = 50, inline -> compacted: A = 3 2.63 -> 2.35, A = 4 3.20 -> 2.87, A = 5 4.57 -> 3.75, A = 6
// 5.18 -> 4.75, A = 7 5.94 -> 5.56, A = 8 6.78 -> 7.82: the rank bookkeeping lifts the step kernel from ~100 to 140
// registers there).  The fused rollout gains up to A = 8 (3.71 -> 3.35 ms per 2^20 x 8 x 50) and loses from A = 12
// (one-thread rollout, T = 20: A = 16 4.73 -> 5.85 ms), where the lane-cooperative kernels take over anyway.
#ifndef SMARL_COLL_COMPACT_MAX_A
#define SMARL_COLL_COMPACT_MAX_A 7
#endif
#ifndef SMARL_COLL_COMPACT_ROLLOUT_MAX_A
#define SMARL_COLL_COMPACT_ROLLOUT_MAX_A 8
#endif

constexpr int kClipSlots = 64;        // compacted action clips per warp and step (two rounds of 32 lanes)

// The action clip of collision_move_agent (collision_avoidance.py:113-117) for one agent whose squared norm exceeds 1,
// out of line: norm = sqrt(dx^2 + dy^2); if norm > 1 both components are divided by it.
static __device__ __noinline__ double2 clip_action(float adx, float ady) {
  double dx = (double)adx, dy = (double)ady;
  const double q = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
  const double norm = __dsqrt_rn(q);
  if (norm > 1.0) {
    dx = __ddiv_rn(dx, norm);
    dy = __ddiv_rn(dy, norm);
  }
  return make_double2(dx, dy);
}

// The transition of all A agents of one env per thread (collision_avoidance.py:103-121) with the action clips of the
// WARP compacted.  The clip costs an f64 square root and two f64 divisions (a dependent chain of ~110 instructions);
// only actions longer than 1 need it (13 % with N(0, 0.5^2) components), but some lane of every warp does for every
// agent slot, so inlined per slot the whole warp runs the chain A times per step, one after the other.  Here every
// agent that needs a clip gets a rank (ballot + popc), posts its f32 action to shared memory, the lanes work the
// posted list off round-robin (ceil(n / 32) rounds instead of A) and the owners pick their f64 result up.  Ranks beyond
// the kClipSlots slots (an unusually clip-heavy warp) are evaluated in place.  Same arithmetic, same bits.
// Must be called by all 32 lanes of the warp; `active` = this lane's env takes the step at all.  clip: kClipSlots
// double2 slots of this warp.
template <int A>
__device__ __forceinline__ void collision_transition_compact(double (&px)[A], double (&py)[A], uint32_t done_mask,
                                                             bool active, const float (&adx)[A], const float (&ady)[A],
                                                             double size, double2* __restrict__ clip) {
  const unsigned lane = threadIdx.x & 31u, lt = (1u << lane) - 1u;
  uint32_t need = 0u;
  uint32_t rk[(A + 3) / 4];                             // rank per agent, one byte each (>= kClipSlots: in place)
#pragma unroll
  for (int w = 0; w < (A + 3) / 4; ++w) rk[w] = 0u;
  int n_clip = 0;
#pragma unroll
  for (int i = 0; i < A; ++i) {
    const double dx = (double)adx[i], dy = (double)ady[i];
    // :113  fp32-origin components: dx**2 == dx*dx exactly, so this is the reference's norm; sqrt_rn is monotonic
    // with sqrt_rn(1) == 1, so norm > 1 needs q > 1
    const double q = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
    const bool nd = active && !((done_mask >> i) & 1u) && q > 1.0;
    const unsigned b = __ballot_sync(0xffffffffu, nd);
    const int r = min(n_clip + __popc(b & lt), kClipSlots);
    n_clip += __popc(b);
    need |= nd ? (1u << i) : 0u;
    rk[i >> 2] |= (uint32_t)r << (8 * (i & 3));
    if (nd && r < kClipSlots) *reinterpret_cast<float2*>(clip + r) = make_float2(adx[i], ady[i]);
  }
  __syncwarp();
  for (int r = (int)lane; r < min(n_clip, kClipSlots); r += 32) {
    const float2 in = *reinterpret_cast<const float2*>(clip + r);
    clip[r] = clip_action(in.x, in.y);
  }
  __syncwarp();
#pragma unroll
  for (int i = 0; i < A; ++i) {
    double2 d = make_double2((double)adx[i], (double)ady[i]);
    if ((need >> i) & 1u) {
      const int r = (int)((rk[i >> 2] >> (8 * (i & 3))) & 0xFFu);
      d = r < kClipSlots ? clip[r] : clip_action(adx[i], ady[i]);
    }
    if (active && !((done_mask >> i) & 1u)) {
      px[i] = fmax(0.0, fmin(size, __dadd_rn(px[i], d.x)));      // :118
      py[i] = fmax(0.0, fmin(size, __dadd_rn(py[i], d.y)));      // :119
    }
  }
  __syncwarp();                         // the slots are reused by the next step
}

// One (agent, landmark) pair: landmark reach (:122-124, np.linalg.norm = sqrt(fma(ay, ay, ax*ax)), probed on OpenBLAS)
// decided on the squared norm outside a 1e-9 band around agents_size^2, and the running minimum of the squared
// distance_matrix entry (:158-161; sqrt_rn is monotonic, so min_l sqrt(q_l) = sqrt(min_l q_l)).
__device__ __forceinline__ bool collision_landmark(double px, double py, double lx, double ly, double agents_size,
                                                   double as2_lo, double as2_hi, double& minq) {
  const double ax = __dadd_rn(px, -lx), ay = __dadd_rn(py, -ly);
  const double axx = __dmul_rn(ax, ax);
  const double qn = __fma_rn(ay, ay, axx);
  bool hit = qn < as2_lo;
  if (!hit && qn < as2_hi) hit = sqrt_below(qn, agents_size);
  minq = fmin(minq, __dadd_rn(axx, __dmul_rn(ay, ay)));
  return hit;
}

// f32 screen threshold of the colliding-pair test: coordinates <= size carry an absolute f32 rounding error
// <= size * 2^-24 each, so an f32 pair distance is off by < size * 2^-22; the screen keeps (lim + size * 2^-21)^2
// plus the rounding of the squared sum itself, which is rigorous for any agents_size (the 1 % relative margin used
// before missed pairs for agents_size <~ 1e-3 on large fields).
__host__ __device__ inline float collision_screen_q(double lim, double size) {
  const double d = lim + size * (1.0 / 2097152.0);
  return (float)(d * d * 1.000001) * 1.000001f;
}

constexpr int kPairPrefilterA = 12;   // agent count from which the pair loop is screened in f32

// One CollisionAvoidance.step for one env held in registers.  Returns the env reward (same for
// every agent) and the collision count; updates px/py/done_mask in place.
// MOVED: the transition (collision_avoidance.py:103-121) was already applied by collision_transition_compact.
template <int A, bool LM0>
__device__ __forceinline__ void collision_env_step(double (&px)[A], double (&py)[A], uint32_t& done_mask,
                                                   const double* __restrict__ lm, int64_t ld, int L,
                                                   double lx0, double ly0, double size, double agents_size,
                                                   double& reward, int& collisions) {
  // landmark reach (:122-124) and per-agent min landmark distance (:158-161).  Both compare / minimise
  // square roots; sqrt_rn is monotonic, so the reach test is decided on the squared norm outside a
  // 1e-9 band around agents_size^2 and the minimum is taken over the squared distances, leaving ONE
  // sqrt per agent (instead of two per agent and landmark).
  double minq[A];
  uint32_t reach = 0u;
  const double as2 = agents_size * agents_size;
  const double as2_lo = as2 * 0.999999999, as2_hi = as2 * 1.000000001;
#pragma unroll
  for (int i = 0; i < A; ++i) minq[i] = 1.0e300;
  for (int l = 0; l < L; ++l) {
    // LM0: landmark 0 was loaded by the caller together with the positions (the step kernel): loaded here, after the
    // transition, its memory latency sat on every thread's critical path (A = 3 on 2^22 envs: 9.00 -> 8.16 ms closed
    // loop).  The fused rollout keeps the load here (hoisted or held across the loop it measured 4-7 % slower).
    const double lx = (LM0 && l == 0) ? lx0 : lm[(2 * l) * ld], ly = (LM0 && l == 0) ? ly0 : lm[(2 * l + 1) * ld];
#pragma unroll
    for (int i = 0; i < A; ++i) {
      const double ax = __dadd_rn(px[i], -lx), ay = __dadd_rn(py[i], -ly);
      const double axx = __dmul_rn(ax, ax);
      // np.linalg.norm(state - land) = sqrt(ddot) = sqrt(fma(ay, ay, ax*ax))   [probed, OpenBLAS]
      const double qn = __fma_rn(ay, ay, axx);
      bool hit = qn < as2_lo;
      if (!hit && qn < as2_hi) hit = sqrt_below(qn, agents_size);
      reach |= hit ? (1u << i) : 0u;
      // distance_matrix(states, landmarks): sqrt((lx-px)^2 + (ly-py)^2); (lx-px)^2 == (px-lx)^2 exactly
      minq[i] = fmin(minq[i], __dadd_rn(axx, __dmul_rn(ay, ay)));
    }
  }
  double mind[A];
#pragma unroll
  for (int i = 0; i < A; ++i) mind[i] = __dsqrt_rn(minq[i]);
  done_mask |= reach & ~done_mask;   // only agents that moved this step are tested; done ones stay done
  reward = -numpy_sum<A>(mind);      // :127-130, all agents incl. done ones
  // collisions among agents not done after this step (:150-156)
  int n = 0;
  const double lim = 2.0 * agents_size;
  const double lim2 = lim * lim;
  const double lim2_lo = lim2 * 0.999999, lim2_hi = lim2 * 1.000001;
  const uint32_t alive = ~done_mask;
  if constexpr (A >= kPairPrefilterA) {
    // Many agents: the A(A-1)/2 pair tests dominate and almost all pairs are far apart.  Screen them in f32
    // (full-rate pipe, half the registers) against collision_screen_q, whose margin covers the f32 rounding of
    // coordinates up to size on any field.  Only pairs of two alive agents that pass the screen are evaluated in
    // f64, out of line, from a local-memory copy of the positions.
    double cx[A], cy[A];
    float fx[A], fy[A];
#pragma unroll
    for (int i = 0; i < A; ++i) {
      cx[i] = px[i];
      cy[i] = py[i];
      fx[i] = (float)px[i];
      fy[i] = (float)py[i];
    }
    const float screen = collision_screen_q(lim, size);
#pragma unroll
    for (int i = 0; i < A; ++i) {
      uint32_t near = 0u;
#pragma unroll
      for (int j = i + 1; j < A; ++j) {
        const float dx = fx[i] - fx[j], dy = fy[i] - fy[j];
        near |= (fmaf(dy, dy, dx * dx) < screen) ? (1u << j) : 0u;
      }
      near &= ((alive >> i) & 1u) ? alive : 0u;
      while (near) {
        const int j = __ffs((int)near) - 1;
        near &= near - 1u;
        n += pair_collides(cx, cy, i, j, lim2_lo, lim2_hi, lim);
      }
    }
  } else {
    bool band = false;
#pragma unroll
    for (int i = 0; i < A; ++i) {
#pragma unroll
      for (int j = i + 1; j < A; ++j) {
        const double dx = __dadd_rn(px[i], -px[j]), dy = __dadd_rn(py[i], -py[j]);
        const double q = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
        const bool below_lo = q < lim2_lo, below_hi = q < lim2_hi;
        n += (below_lo && ((alive >> i) & (alive >> j) & 1u)) ? 1 : 0;
        band |= below_lo != below_hi;
      }
    }
    if (band) {
      double cx[A], cy[A];
#pragma unroll
      for (int i = 0; i < A; ++i) {
        cx[i] = px[i];
        cy[i] = py[i];
      }
      n = collisions_exact(cx, cy, A, alive, lim);
    }
  }
  collisions = n;
}

// The env parameters every CollisionAvoidance entry point checks.
inline int check_collision(const SmarlCollisionParams* p) {
  SMARL_REQUIRE(p != nullptr, "params is NULL");
  SMARL_REQUIRE(p->size >= 1, "size=%d must be >= 1", p->size);
  SMARL_REQUIRE(p->n_landmarks >= 1 && p->n_landmarks <= 64, "n_landmarks=%d outside 1..64", p->n_landmarks);
  SMARL_REQUIRE(p->agents_size > 0.0, "agents_size must be positive");
  // The reach and pair tests compare squared distances with agents_size^2 (1 -+ 1e-9) and (2 agents_size)^2 (1 -+ 1e-6)
  // and take the square root only inside those bands.  Below 2^-511 the square is subnormal or zero, the bands collapse
  // to nothing and the squared test alone would decide wrong (an agent exactly on its landmark: 0 < 0 is false).
  SMARL_REQUIRE(p->agents_size >= 0x1p-511, "agents_size=%g below 2^-511: its square is not a normal double",
                p->agents_size);
  return SMARL_OK;
}

int launch_collision_step(int A, const CollisionStepArgs& a, unsigned grid, cudaStream_t s);
int launch_collision_rollout(int A, const CollisionRolloutArgs& a, unsigned grid, cudaStream_t s);
int launch_collision_coop_step(int A, int S, const CollisionStepArgs& a, cudaStream_t s);
int launch_collision_coop_rollout(int A, int S, const CollisionRolloutArgs& a, cudaStream_t s);
// lanes per env of the lane-cooperative kernels for this agent count / batch (0 = one thread per env)
int collision_coop_lanes(int A, int L, int64_t ld, bool rollout);

}  // namespace smarl
