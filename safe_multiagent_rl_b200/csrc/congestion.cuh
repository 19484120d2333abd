// Congestion device code shared by the step kernel and the fused rollout kernel.
#pragma once
#include "common.cuh"

namespace smarl {

// envs/congestion.py:7-10
#define SMARL_HOURLY_COMPENSATION 30.0
#define SMARL_AVERAGE_RIDE_COMPENSATION 7.5
#define SMARL_AVERAGE_RIDE_COST 4.0
#define SMARL_CONGESTION_COST 2.0

// Effective (post-noise) moves of four envs for every agent, from Philox4x32-10:
//   counter = (env_id lo, env_id hi, t, agent >> 2 | episode << 3), key = seed; agent a reads word w = out[a & 3];
//   move = action if w < keep_threshold else w mod 5,
// the integer form of congestion.py:64-67 (u1 < 1 - noise ? a : int(u2 * 5)) with u1 = w * 2^-32 and
// u2 = (w mod 5 + 0.5) / 5.  Given w >= keep_threshold, w mod 5 is uniform on 0..4 up to one count in
// 2^32 per outcome -- the same resolution as drawing a second 32-bit word -- so one generator call serves
// four agents.  The episode index (low 29 bits) sits above the agent-quad index, so every episode of every
// env draws a fresh realisation, as the reference's random() does (congestion.py:64-67).
template <int A>
__device__ __forceinline__ void congestion_noise_moves(const uint32_t (&aw)[A], uint32_t (&mw)[A],
                                                       uint64_t seed, uint64_t keep_threshold,
                                                       int64_t env0, uint32_t t, uint32_t episode) {
  const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
#pragma unroll
  for (int i = 0; i < A; ++i) mw[i] = 0u;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const uint64_t id = (uint64_t)(env0 + k);
#pragma unroll
    for (int j = 0; j < (A + 3) / 4; ++j) {
      const uint4 o = philox4x32_10(make_uint4((uint32_t)id, (uint32_t)(id >> 32), t, (uint32_t)j | (episode << 3)), key);
      const uint32_t w[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        if (4 * j + q < A) {
          const uint32_t act = (aw[4 * j + q] >> (8 * k)) & 0xFFu;
          const uint32_t mv = ((uint64_t)w[q] < keep_threshold) ? act : w[q] % 5u;
          mw[4 * j + q] |= mv << (8 * k);
        }
      }
    }
  }
}

// One Congestion transition for four envs (congestion.py:49-75): applies the effective moves,
// leaves the new positions in xw/yw and the displacement codes in dcw.
template <int A>
__device__ __forceinline__ void congestion_transition(uint32_t (&xw)[A], uint32_t (&yw)[A],
                                                      const uint32_t (&mw)[A], uint32_t (&dcw)[A],
                                                      uint32_t size4) {
  const uint32_t k1 = 0x01010101u;
#pragma unroll
  for (int i = 0; i < A; ++i) {
    const uint32_t ox = xw[i], oy = yw[i];
    grid_move4(xw[i], yw[i], mw[i], size4);
    dcw[i] = ((xw[i] + k1) - ox) | (((yw[i] + k1) - oy) << 2);
  }
}

// 0x01 in every byte of v that is zero (carry-free: the low 7 bits are tested by an add that cannot leave the byte).
__device__ __forceinline__ uint32_t zero_bytes01(uint32_t v) {
  const uint32_t k7f = 0x7F7F7F7Fu;
  return (~(((v & k7f) + k7f) | v) & 0x80808080u) >> 7;
}

// Congestion._congestions (congestion.py:113-137) for the four envs of the packed words at once, in the
// closed form proved equivalent in tests/test_oracle_vs_reference.py: agents sharing the same directed edge
// form a class; with L = lowest index in the class whose INTENDED action is a move (<4), members >= L
// ("active") get (#members >= L) - 1, everything else 0.
//   xw,yw  new positions   dcw  displacement code (nx-ox+1) | (ny-oy+1) << 2   aw intended (0..4)
// The edge (ox,oy,nx,ny) is identified by the three bytes (nx, ny, dcode); every quantity below is a byte
// per env lane (flags 0/1, counts <= 31), so one pass over the A(A-1)/2 pairs serves all four envs:
//   e(i,j)  = [key_i == key_j]
//   act_j   = mov_j | OR_{i<j} e(i,j) & mov_i          (some member k <= j of j's class intends to move)
//   con_i   = act_i ? sum_{j != i} e(i,j) & act_j : 0
// Row j's e(.,j) are kept in registers until act_j is final, then added to both counters.
// Writes conw[i]; returns the per-lane number of agents standing on node (0,0) (congestion.py:97).
template <int A>
__device__ __forceinline__ uint32_t congestion_env4(const uint32_t (&xw)[A], const uint32_t (&yw)[A],
                                                    const uint32_t (&dcw)[A], const uint32_t (&aw)[A],
                                                    uint32_t (&conw)[A]) {
  const uint32_t k01 = 0x01010101u;
  uint32_t mov[A], act[A], cnt[A];
  uint32_t at_origin = 0u;
#pragma unroll
  for (int i = 0; i < A; ++i) {
    mov[i] = ((aw[i] >> 2) & k01) ^ k01;              // a < 4 for a in 0..4
    at_origin += zero_bytes01(xw[i] | yw[i]);
    cnt[i] = 0u;
  }
#pragma unroll
  for (int j = 0; j < A; ++j) {
    uint32_t e[A];
    uint32_t a_j = mov[j];
#pragma unroll
    for (int i = 0; i < j; ++i) {
      e[i] = zero_bytes01((xw[i] ^ xw[j]) | (yw[i] ^ yw[j]) | (dcw[i] ^ dcw[j]));
      a_j |= e[i] & mov[i];
    }
    act[j] = a_j;
#pragma unroll
    for (int i = 0; i < j; ++i) {
      cnt[i] += e[i] & a_j;
      cnt[j] += e[i] & act[i];
    }
  }
#pragma unroll
  for (int i = 0; i < A; ++i) conw[i] = cnt[i] & (act[i] * 0xFFu);
  return at_origin;
}

// The same closed form for ONE env lane k of the packed words, with per-agent class bitmasks and popc.  Used
// for larger agent counts (thresholds below), where the byte-SIMD form's unrolled pair loop over all four lanes runs out
// of registers (measured: A = 16 -2 %, A = 32 -5 % with the SIMD form; A = 3..8 +12..26 %).
//   xw,yw  new positions   dcw  displacement code (nx-ox+1) | (ny-oy+1) << 2   aw intended
// The edge (ox,oy,nx,ny) is identified by the 3-byte key (nx, ny, dcode).
// Writes byte k of conw[i]; returns the number of agents standing on node (0,0).
template <int A>
__device__ __forceinline__ int congestion_env(const uint32_t (&xw)[A], const uint32_t (&yw)[A],
                                              const uint32_t (&dcw)[A], const uint32_t (&aw)[A],
                                              uint32_t (&conw)[A], int k) {
  const uint32_t sel_xy = (uint32_t)k | ((uint32_t)(k + 4) << 4);          // (x_k, y_k, ., .)
  const uint32_t sel_key = 0x0010u | ((uint32_t)(k + 4) << 8) | (4u << 12); // (b0, b1, dcode_k, dc byte0)
  uint32_t key[A], same[A];
  uint32_t movers = 0u;
  int at_origin = 0;
#pragma unroll
  for (int i = 0; i < A; ++i) {
    const uint32_t xy = __byte_perm(xw[i], yw[i], sel_xy);
    key[i] = __byte_perm(xy, dcw[i], sel_key) & 0x00FFFFFFu;
    same[i] = 0u;
    movers |= (((aw[i] >> (8 * k)) & 0xFFu) < 4u) ? (1u << i) : 0u;
    at_origin += ((key[i] & 0xFFFFu) == 0u) ? 1 : 0;                       // congestion.py:97
  }
#pragma unroll
  for (int i = 0; i < A; ++i) {
#pragma unroll
    for (int j = i + 1; j < A; ++j) {
      // one compare + two predicated ORs (the select form costs two more instructions per pair)
      asm("{\n\t.reg .pred q;\n\tsetp.eq.u32 q, %2, %3;\n\t@q or.b32 %0, %0, %4;\n\t@q or.b32 %1, %1, %5;\n\t}"
          : "+r"(same[i]), "+r"(same[j])
          : "r"(key[i]), "r"(key[j]), "r"(1u << j), "r"(1u << i));
    }
  }
  uint32_t active = 0u;
#pragma unroll
  for (int i = 0; i < A; ++i) {
    const uint32_t below_or_self = (same[i] & ((1u << i) - 1u)) | (1u << i);
    active |= (below_or_self & movers) ? (1u << i) : 0u;
  }
#pragma unroll
  for (int i = 0; i < A; ++i) {
    const uint32_t cls = (same[i] | (1u << i)) & active;
    const uint32_t con = ((active >> i) & 1u) ? (uint32_t)__popc(cls) - 1u : 0u;
    conw[i] |= con << (8 * k);
  }
  return at_origin;
}

// Largest agent count served by the byte-SIMD form, per kernel (measured on 2^20 envs: the step kernel gains up to
// A = 10 and loses 12 % at A = 12, where it needs 180 registers; the fused rollout still gains 9 % at A = 12).
constexpr int kSimdClassAgentsStep = 10;
constexpr int kSimdClassAgentsRollout = 12;

// Congestions of the four envs of a thread + per-lane count of agents on node (0,0) (bytes of the result).
template <int A, int MAX_SIMD_A>
__device__ __forceinline__ uint32_t congestion_classes(const uint32_t (&xw)[A], const uint32_t (&yw)[A],
                                                       const uint32_t (&dcw)[A], const uint32_t (&aw)[A],
                                                       uint32_t (&conw)[A]) {
  if constexpr (A <= MAX_SIMD_A) {
    return congestion_env4<A>(xw, yw, dcw, aw, conw);
  } else {
#pragma unroll
    for (int i = 0; i < A; ++i) conw[i] = 0u;
    uint32_t org = 0u;
#pragma unroll 1
    for (int k = 0; k < 4; ++k) org |= (uint32_t)congestion_env<A>(xw, yw, dcw, aw, conw, k) << (8 * k);
    return org;
  }
}

struct CongestionStepArgs {
  uint8_t* pos_x;
  uint8_t* pos_y;
  const uint8_t* actions;
  uint8_t* moves;
  float* obs;
  float* reward;
  int32_t* cost;
  uint8_t* done;
  const double* lambdas;
  float* penalty;
  const double* demand;
  const float* wait_reward;
  uint64_t keep_threshold;
  uint64_t seed;
  int64_t env_offset;
  int64_t n_groups;
  int64_t ld;
  int32_t size;
  int32_t t;
  uint32_t episode;
  const uint32_t* episode_dev;
};

struct CongestionRolloutArgs {
  const uint8_t* start_x;
  const uint8_t* start_y;
  const uint8_t* actions;   // [T][A][ld]
  const uint8_t* moves;     // [T][A][ld] (MODE 1)
  const double* lambdas;
  uint8_t* final_x;
  uint8_t* final_y;
  float* R;
  float* modR;
  int32_t* C;
  float* G;                 // [T][A][ld]
  float* g_scratch;         // [T][ld] penalties (g_mode 1)
  double* partials;
  const double* thresholds;
  const double* demand;
  const float* wait_reward;
  double gamma;
  uint64_t keep_threshold;
  uint64_t seed;
  int64_t env_offset;
  int64_t n_groups;
  int64_t n_envs;
  int64_t ld;
  int32_t size;
  int32_t n_steps;
  int32_t g_mode;
  uint32_t episode;
  const uint32_t* episode_dev;
};

// CTA size of the fused rollouts that keep the per-agent sums in shared memory (congestion_rollout_kernel and
// congestion_policy_rollout_kernel): the block summation tree of their stats partials depends on it.
constexpr int kCongRollThreads = 64;

inline int check_congestion(const SmarlCongestionParams* p) {
  SMARL_REQUIRE(p != nullptr, "params is NULL");
  SMARL_REQUIRE(p->size >= 1 && p->size <= 254, "size=%d outside 1..254", p->size);
  SMARL_REQUIRE(p->demand != nullptr, "demand table is NULL");
  SMARL_REQUIRE(p->noise_mode >= 0 && p->noise_mode <= 2, "bad noise_mode %d", p->noise_mode);
  SMARL_REQUIRE(p->keep_threshold <= (1ull << 32), "keep_threshold must be <= 2^32");
  return SMARL_OK;
}

// Launchers of noise mode M = 0..2 (congestion.cu, congestion_coop.cu), each mode instantiated in its own translation unit
template <int M> int launch_congestion_step(int A, const CongestionStepArgs& a, unsigned grid, cudaStream_t s);
template <int M> int launch_congestion_rollout(int A, const CongestionRolloutArgs& a, unsigned grid, cudaStream_t s);
template <int M> int launch_congestion_coop_step(int A, int S, const CongestionStepArgs& a, cudaStream_t st);
// fused rollout, four lanes per env quad (congestion_coop.cu); *grid returns the CTA count (= rows of stats partials)
template <int M> int launch_congestion_coop_rollout(int A, const CongestionRolloutArgs& a, unsigned* grid, cudaStream_t st);

// Waiting-branch reward in f64, the reference's operation order (congestion.py:86-87).
__device__ __forceinline__ double congestion_reward_f64(uint32_t con, uint32_t nx, uint32_t ny,
                                                        const double* __restrict__ demand, int W) {
  const double d = __ldg(demand + nx * W + ny);
  const double q = __ddiv_rn(-SMARL_HOURLY_COMPENSATION * (double)(con + 1u), d);
  return __dadd_rn(__dadd_rn(q, SMARL_AVERAGE_RIDE_COMPENSATION), -SMARL_AVERAGE_RIDE_COST);
}

// Waiting-branch reward from the demand table, out of line: only reached when the caller passed no host-built
// waiting table.  (Inlined at every (agent, env lane) the float64 division was a third of the step kernels' code.)
static __device__ __noinline__ float congestion_wait_reward_slow(uint32_t con, uint32_t nx, uint32_t ny,
                                                                 const double* __restrict__ demand, int W) {
  return (float)congestion_reward_f64(con, nx, ny, demand, W);
}

// Congestion.reward (congestion.py:82-87) for the agent in env lane k of the packed words, rounded to f32 exactly
// once.  Movers (intended action < 4) get -4 - 2 con (exact: small integers); the waiting branch comes from the
// host-built table wait[con][cell] (the reference's f64 expression, rounded once) through ONE predicated load --
// no branch: the branchy form cost ~35 instructions per (agent, env) and 43 % of the A = 8 step kernel -- or,
// without a table, from the out-of-line float64 evaluation.
template <bool TABLE>
__device__ __forceinline__ float congestion_reward_lane(uint32_t aw, uint32_t conw, uint32_t xw, uint32_t yw, int k,
                                                        const double* __restrict__ demand, int W,
                                                        const float* __restrict__ wait) {
  const uint32_t sel = 0x4440u | (uint32_t)k;                      // byte k, zero-extended
  const uint32_t act = __byte_perm(aw, 0u, sel), con = __byte_perm(conw, 0u, sel);
  const uint32_t nx = __byte_perm(xw, 0u, sel), ny = __byte_perm(yw, 0u, sel);
  float r = fmaf(-2.0f, (float)con, -4.0f);
  if (TABLE) {
    const float* p = wait + (con * (uint32_t)W + nx) * (uint32_t)W + ny;
    asm("{\n\t.reg .pred q;\n\tsetp.ge.u32 q, %1, 4;\n\t@q ld.global.nc.f32 %0, [%2];\n\t}" : "+f"(r) : "r"(act), "l"(p));
  } else if (act >= 4u) {
    r = congestion_wait_reward_slow(con, nx, ny, demand, W);
  }
  return r;
}

// The four env lanes of one agent (TABLE: the host-built waiting table is present -- decided once per kernel, not
// per reward).
template <bool TABLE>
__device__ __forceinline__ float4 congestion_reward4(uint32_t aw, uint32_t conw, uint32_t xw, uint32_t yw,
                                                     const double* __restrict__ demand, int W,
                                                     const float* __restrict__ wait) {
  return make_float4(congestion_reward_lane<TABLE>(aw, conw, xw, yw, 0, demand, W, wait),
                     congestion_reward_lane<TABLE>(aw, conw, xw, yw, 1, demand, W, wait),
                     congestion_reward_lane<TABLE>(aw, conw, xw, yw, 2, demand, W, wait),
                     congestion_reward_lane<TABLE>(aw, conw, xw, yw, 3, demand, W, wait));
}

// Same for already extracted fields (kept for callers that hold them).
__device__ __forceinline__ float congestion_reward(uint32_t act, uint32_t con, uint32_t nx, uint32_t ny,
                                                   const double* __restrict__ demand, int W,
                                                   const float* __restrict__ wait) {
  if (act < 4u) return -4.0f - 2.0f * (float)con;                   // exact: small integers
  if (wait) return __ldg(wait + (con * W + nx) * W + ny);
  return congestion_wait_reward_slow(con, nx, ny, demand, W);
}

}  // namespace smarl
