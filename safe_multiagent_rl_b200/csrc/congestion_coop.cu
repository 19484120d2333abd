// Congestion, lane-cooperative step kernel for large agent counts (sm_100a).
//
// congestion.cu keeps all A agents of four envs in one thread; from A = 16 that is 168-255 registers (2-3 CTAs per
// SM, spills at A = 32) and the kernel falls to 0.55 / 0.31 of the HBM roofline at A = 16 / 32.  Here a group of
// S = 2 or 4 lanes shares one quad of four envs, lane s owning agents i = j*S + s as byte-SIMD words.  A warp covers
// 32/S quads (lane = s*(32/S) + q), so every load / store instruction touches S rows x (32/S) consecutive words
// or 16-byte vectors of the agent-major SoA arrays: whole 32-byte sectors.
//
// _congestions (congestion.py:113-137) is order dependent, so its A(A-1)/2 pair tests cannot be shared between
// the two partners' lanes without sending partial results back.  Instead every agent SCANS all agents in index
// order, as the reference's sequential loop does, over records published to shared memory:
//     r      running number of agents on the same directed edge           (class members so far, incl. self)
//     seen   an INTENDED mover with index <= own was on the edge          (= "active" in the closed form)
//     z      r at the moment the first such mover appears                 (= inactive members before the leader)
//     con = seen ? r_final - z - 1 : 0                                    (#members >= leader, minus self)
// which is the closed form proved against the literal loop in tests/test_oracle_vs_reference.py: members below
// the lowest-index intended mover L of a class get 0, members >= L get #{members >= L} - 1.  Lower partners cost
// 12 integer ops for the four envs, higher ones 8; nothing flows back between lanes.
//
// Philox noise (MODE 2): one generator block serves four agents of one env, so the 4 * ceil(A/4) blocks of a
// quad are spread over the S lanes and handed out through shared memory (no lane evaluates a block twice).
#include "congestion.cuh"
#include "stats.cuh"

// Built as six translation units (build.py passes -DSMARL_TU=k): step kernels of noise mode k = 0..2, fused rollout
// kernels of noise mode k - 3 = 0..2.

namespace smarl {

constexpr int kCongCoopThreads = 128;

template <int A, int S>
struct CongCoop {
  static constexpr int B = (A + S - 1) / S;          // agents per lane
  static constexpr int EPW = 32 / S;                 // env quads per warp
  static constexpr int EPC = kCongCoopThreads / S;   // env quads per CTA
  static constexpr int NQ = (A + 3) / 4;             // Philox blocks per env (four agents each)
  static constexpr bool kGhost = (A % S) != 0;
  static constexpr int PR = (B * S) | 1;             // uint4 records per quad (incl. padding agents): odd => conflict-free LDS.128
  static constexpr int PW = (4 * NQ) | 1;            // uint4 Philox blocks per quad
  static constexpr int PQ = PR > PW ? PR : PW;       // the Philox blocks are consumed before the records are written: one buffer
  static constexpr size_t kSmem = (size_t)EPC * PQ * sizeof(uint4);
};

// r = (e80 >> 7) + r per env byte as ONE multiply-add on the FMA pipe (the kernel is bound by the integer ALU
// pipe; written in C, ptxas turns the same expression into LEA.HI, an ALU-pipe instruction).
__device__ __forceinline__ uint32_t add_flags80(uint32_t e80, uint32_t r) {
  uint32_t o;
  // multiplier 2^25 + 1, not 2^25: the low 7 bits of e80 are clear, so e80 * 2^25 has a zero low word and the
  // extra e80 cannot carry into the high word -- same result, but not a shift ptxas would strength-reduce
  asm("mad.hi.u32 %0, %1, 33554433, %2;" : "=r"(o) : "r"(e80), "r"(r));
  return o;
}
// 0xFF in every env byte whose bit 7 is set in f80 (FMA pipe).
__device__ __forceinline__ uint32_t expand_flags80(uint32_t f80) { return __umulhi(f80, 0xFFu << 25); }

// The scan: all agents in index order against every own agent (see the file header).  Flags live in bit 7 of
// each env byte (0x80), so equality needs no final shift and counting / mask expansion are IMAD.HI.  The loop
// over partner ROWS (S partners each) is rolled -- fully unrolled, the scan alone was ~3000 instructions and the
// kernel stalled 3.6 cycles per issue on instruction fetch -- with the own agents unrolled inside; "partner <= own"
// is uniform per (row, own agent) except on the own row, where a per-lane mask decides.
//   KW    words of the edge key compared (2: the (x_old + 2 x', y_old + 2 y') encoding; 3: (x', y', dcode))
//   LOW7  every key byte is <= 0x7F, which saves two instructions of the zero-byte test
template <int A, int S, int KW, bool LOW7>
__device__ __forceinline__ void congestion_scan(const uint4* __restrict__ rec, const uint32_t (&k0)[CongCoop<A, S>::B],
                                                const uint32_t (&k1)[CongCoop<A, S>::B],
                                                const uint32_t (&k2)[CongCoop<A, S>::B], int s,
                                                uint32_t (&r)[CongCoop<A, S>::B], uint32_t (&seen)[CongCoop<A, S>::B],
                                                uint32_t (&z)[CongCoop<A, S>::B]) {
  constexpr int B = CongCoop<A, S>::B;
  const uint32_t k7f = 0x7F7F7F7Fu, k80 = 0x80808080u;
  uint32_t le80[S];
#pragma unroll
  for (int j = 0; j < B; ++j) r[j] = seen[j] = z[j] = 0u;
#pragma unroll
  for (int t = 0; t < S; ++t) le80[t] = (t <= s) ? k80 : 0u;
#pragma unroll 1
  for (int jr = 0; jr < B; ++jr) {
    uint4 p[S];
#pragma unroll
    for (int t = 0; t < S; ++t) p[t] = rec[jr * S + t];
#pragma unroll
    for (int j = 0; j < B; ++j) {
      uint32_t e[S];
#pragma unroll
      for (int t = 0; t < S; ++t) {
        uint32_t v = (p[t].x ^ k0[j]) | (p[t].y ^ k1[j]);
        if (KW == 3) v |= p[t].z ^ k2[j];
        // 0x80 in every env byte whose edge keys are equal
        e[t] = LOW7 ? (~(v + k7f) & k80) : (~(((v & k7f) + k7f) | v) & k80);
      }
      if (jr <= j) {                                                // uniform: this row holds partners <= own (or the own row)
#pragma unroll
        for (int t = 0; t < S; ++t) {
          const uint32_t w = jr < j ? p[t].w : (p[t].w & le80[t]);  // intended movers with index <= own
          const uint32_t first = e[t] & w & ~seen[j];
          z[j] |= expand_flags80(first) & r[j];                     // r before this partner: members below the leader
          seen[j] |= e[t] & w;
          r[j] = add_flags80(e[t], r[j]);
        }
      } else {
#pragma unroll
        for (int t = 0; t < S; ++t) r[j] = add_flags80(e[t], r[j]);
      }
    }
  }
}

template <int A, int S, int MODE>
__global__ void __launch_bounds__(kCongCoopThreads, 4) congestion_coop_step_kernel(const CongestionStepArgs a) {
  pdl_prologue();   // programmatic dependent launch: the previous grid has completed past this point (common.cuh)
  using C = CongCoop<A, S>;
  constexpr int B = C::B, EPW = C::EPW, EPC = C::EPC, NQ = C::NQ;
  extern __shared__ uint4 s_rec[];                                 // [EPC][PQ]: Philox blocks (MODE 2), then the
                                                                   // (x', y', dcode, intended mover) records
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int q = lane % EPW, s = lane / EPW;
  const int ql = warp * EPW + q;
  const int64_t gq = (int64_t)blockIdx.x * EPC + ql;
  const bool live = gq < a.n_groups;
  const uint32_t ld = (uint32_t)a.ld;
  const uint32_t e0 = (uint32_t)(live ? gq : 0) * 4u;
  const uint32_t row0 = (uint32_t)s * ld + e0;                     // 32-bit element offsets (host-checked)
  const uint32_t k01 = 0x01010101u;

  uint32_t xw[B], yw[B], aw[B], mw[B];
#pragma unroll
  for (int j = 0; j < B; ++j) {
    const uint32_t off = row0 + (uint32_t)(j * S) * ld;
    if (!C::kGhost || j < B - 1 || j * S + s < A) {
      xw[j] = ld_stream_u32(a.pos_x + off);
      yw[j] = ld_stream_u32(a.pos_y + off);
      aw[j] = ld_stream_u32(a.actions + off);
      mw[j] = MODE == 1 ? ld_stream_u32(a.moves + off) : aw[j];
    } else {
      xw[j] = yw[j] = 0xFFFFFFFFu;
      aw[j] = mw[j] = 0x04040404u;
    }
  }
  if (MODE == 2) {
    // blocks b = jq*4 + k (agent quad jq, env lane k) of this env quad, b = s, s + S, ...: counter and key as in
    // congestion_noise_moves (congestion.cuh)
    const uint2 key = make_uint2((uint32_t)a.seed, (uint32_t)(a.seed >> 32));
    const uint32_t episode = a.episode + (a.episode_dev ? __ldg(a.episode_dev) : 0u);
    const int64_t env0 = a.env_offset + (int64_t)(live ? gq : 0) * 4;
    uint4* wq = s_rec + ql * C::PQ;
#pragma unroll
    for (int m = 0; m * S < 4 * NQ; ++m) {
      const int b = m * S + s;
      if (4 * NQ % S == 0 || b < 4 * NQ) {
        const uint64_t id = (uint64_t)(env0 + (b & 3));
        wq[b] = philox4x32_10(make_uint4((uint32_t)id, (uint32_t)(id >> 32), (uint32_t)a.t,
                                         (uint32_t)(b >> 2) | (episode << 3)), key);
      }
    }
    __syncwarp();
    const uint32_t* ww = reinterpret_cast<const uint32_t*>(wq);
#pragma unroll
    for (int j = 0; j < B; ++j) {
      const int i = j * S + s;                                      // word (i & 3) of block (i >> 2, k)
      uint32_t m4 = 0u;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const uint32_t w = ww[(((i >> 2) * 4 + k) << 2) + (i & 3)];
        const uint32_t act = (aw[j] >> (8 * k)) & 0xFFu;
        const uint32_t mv = ((uint64_t)w < a.keep_threshold) ? act : w % 5u;
        m4 |= mv << (8 * k);
      }
      if (!C::kGhost || j < B - 1 || i < A) mw[j] = m4;
    }
    __syncwarp();                                                   // the records below reuse the block buffer
  }

  // transition (congestion.py:49-75) and the records every lane of the group scans
  const uint32_t size4 = (uint32_t)a.size * k01;
  // edge key (x_old, y_old, x', y') per env byte: up to size 84 the two bytes (x_old + 2 x', y_old + 2 y') identify
  // the directed edge (3 x' - dx with dx in {-1, 0, 1} determines both); larger grids compare (x', y', dcode)
  const bool small_key = a.size <= 84;
  uint32_t k0[B], k1[B], k2[B];
  uint32_t at_origin = 0u;
  uint4* rec = s_rec + ql * C::PQ;
#pragma unroll
  for (int j = 0; j < B; ++j) {
    const bool own = !C::kGhost || j < B - 1 || j * S + s < A;
    const uint32_t ox = xw[j], oy = yw[j];
    grid_move4(xw[j], yw[j], mw[j], size4);
    k0[j] = small_key ? ox + 2u * xw[j] : xw[j];
    k1[j] = small_key ? oy + 2u * yw[j] : yw[j];
    k2[j] = small_key ? 0u : (((xw[j] + k01) - ox) | (((yw[j] + k01) - oy) << 2));
    if (!own) {                                                      // a padding agent's record matches no real edge:
      const uint32_t never = (a.size <= 42 || (a.size > 84 && a.size <= 127)) ? 0x7F7F7F7Fu : 0xFFFFFFFFu;
      if (small_key) k0[j] = never;                                 // real bytes are <= 126 (size <= 42) / <= 252
      else k2[j] = never;                                           // real displacement codes are <= 0x0A
    }
    // record: edge key words, intended mover (action < 4) as 0x80 per env byte
    rec[j * S + s] = make_uint4(k0[j], k1[j], k2[j], own ? ((((aw[j] >> 2) & k01) ^ k01) << 7) : 0u);
    if (own) {
      at_origin += zero_bytes01(xw[j] | yw[j]);                    // congestion.py:97
      if (live) {
        const uint32_t off = row0 + (uint32_t)(j * S) * ld;
        st_stream_u32(a.pos_x + off, xw[j]);
        st_stream_u32(a.pos_y + off, yw[j]);
        if (MODE != 1 && a.moves) st_stream_u32(a.moves + off, mw[j]);
        if (a.done) st_stream_u32(a.done + off, 0u);                // congestion.py:103-104
        if (a.obs) {
          const uint32_t o2 = 2u * off - e0;
          st_stream_f4(a.obs + o2, bytes_to_float4(xw[j]));
          st_stream_f4(a.obs + (o2 + ld), bytes_to_float4(yw[j]));
        }
      }
    }
  }
  __syncwarp();

  // the scan (congestion_scan above), specialised on the width of the edge key
  uint32_t r[B], seen[B], z[B];
  if (a.size <= 42) congestion_scan<A, S, 2, true>(rec, k0, k1, k2, s, r, seen, z);
  else if (a.size <= 84) congestion_scan<A, S, 2, false>(rec, k0, k1, k2, s, r, seen, z);
  else if (a.size <= 127) congestion_scan<A, S, 3, true>(rec, k0, k1, k2, s, r, seen, z);
  else congestion_scan<A, S, 3, false>(rec, k0, k1, k2, s, r, seen, z);
#pragma unroll
  for (int off = 1; off < S; off <<= 1) at_origin += __shfl_xor_sync(0xffffffffu, at_origin, off * EPW);
  if (!live) return;

  // congestion.py:93-100: cost = max(0, A // 3 - #agents on node (0,0)) per env lane
  const int c0 = max(0, A / 3 - (int)(at_origin & 0xFFu)), c1 = max(0, A / 3 - (int)((at_origin >> 8) & 0xFFu)),
            c2 = max(0, A / 3 - (int)((at_origin >> 16) & 0xFFu)), c3 = max(0, A / 3 - (int)(at_origin >> 24));
  if (s == 0) {
    st_stream_i4(a.cost + e0, make_int4(c0, c1, c2, c3));
    if (a.penalty) {                                                // meta_agent.py:21-22
      const double lam = __ldg(a.lambdas);
      st_stream_f4(a.penalty + e0, make_float4((float)(lam * c0), (float)(lam * c1), (float)(lam * c2), (float)(lam * c3)));
    }
  }
  const int W = a.size + 1;
#pragma unroll
  for (int j = 0; j < B; ++j) {
    if (C::kGhost && j == B - 1 && j * S + s >= A) continue;
    const uint32_t conw = (r[j] - z[j] - k01) & __umulhi(seen[j], 0xFFu << 25);
    const float4 rw = a.wait_reward ? congestion_reward4<true>(aw[j], conw, xw[j], yw[j], a.demand, W, a.wait_reward)
                                    : congestion_reward4<false>(aw[j], conw, xw[j], yw[j], a.demand, W, nullptr);
    st_stream_f4(a.reward + (row0 + (uint32_t)(j * S) * ld), rw);
  }
}

// ---------------------------------------------------------------------------------------
// Fused open-loop episode on the same lane mapping (S = 4): T steps of the kernel above with the positions in
// registers, plus the accounting of congestion_rollout_kernel (congestion.cu) -- per-agent discounted sums in f64
// (shared memory, [own agent][env lane][thread]: conflict-free), the shared constraint's cost / penalty sums (every
// lane of a group carries them redundantly), G in g_mode 1 / 2, block partials of the stats vector.  The one-thread
// rollout needs 255 registers plus spills from A ~ 20 and falls BEHIND the closed loop of cooperative step launches
// (A = 32, 2^20 envs, T = 50: 22.9 ms fused against 14.4 ms closed); this one keeps the fused path ahead.
// Same per-(agent, env) accumulation order as the one-thread kernel: R, modR, C, G are bit-identical to it.
// ---------------------------------------------------------------------------------------
template <int A, int S>
struct CongCoopRoll {
  using C = CongCoop<A, S>;
  static constexpr size_t kRec = (size_t)C::EPC * C::PQ * sizeof(uint4);
  static constexpr size_t kSmem = kRec + (size_t)C::B * 4 * kCongCoopThreads * sizeof(double);
};

// Sum of v over the CTA separately for every lane slot s (lanes of one slot are EPW consecutive lanes of each warp);
// the result for slot s' is valid on thread s' < S.  s_red: (threads / 32) * S doubles.  Fixed order.
template <int S>
__device__ __forceinline__ double slot_block_sum(double v, double* s_red, int s, int q) {
  constexpr int EPW = 32 / S;
#pragma unroll
  for (int o = EPW / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if (q == 0) s_red[(threadIdx.x >> 5) * S + s] = v;
  __syncthreads();
  double r = 0.0;
  if (threadIdx.x < S) {
#pragma unroll
    for (int w = 0; w < kCongCoopThreads / 32; ++w) r += s_red[w * S + threadIdx.x];
  }
  __syncthreads();
  return r;
}

template <int A, int S, int MODE>
__global__ void __launch_bounds__(kCongCoopThreads, 3) congestion_coop_rollout_kernel(const CongestionRolloutArgs a) {
  using C = CongCoop<A, S>;
  constexpr int B = C::B, EPW = C::EPW, EPC = C::EPC, NQ = C::NQ;
  extern __shared__ uint4 s_rec[];                                 // [EPC][PQ] records / Philox blocks, then the sums
  double* s_acc = reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(s_rec) + CongCoopRoll<A, S>::kRec);
  __shared__ double s_red[(kCongCoopThreads / 32) * S];
  const int tid = threadIdx.x;
  const int lane = tid & 31, warp = tid >> 5;
  const int q = lane % EPW, s = lane / EPW;
  const int ql = warp * EPW + q;
  const int64_t gq = (int64_t)blockIdx.x * EPC + ql;
  const bool live = gq < a.n_groups;
  const uint32_t ld = (uint32_t)a.ld;
  const uint32_t e0 = (uint32_t)(live ? gq : 0) * 4u;
  const uint32_t row0 = (uint32_t)s * ld + e0;                     // 32-bit element offsets (host-checked: A * ld < 2^32)
  const uint32_t k01 = 0x01010101u;
  const int T = a.n_steps, W = a.size + 1;
  const uint32_t size4 = (uint32_t)a.size * k01;
  const bool small_key = a.size <= 84;
  const uint32_t never = (a.size <= 42 || (a.size > 84 && a.size <= 127)) ? 0x7F7F7F7Fu : 0xFFFFFFFFu;
  const double lam = a.lambdas ? __ldg(a.lambdas) : 0.0;
  const uint2 key = make_uint2((uint32_t)a.seed, (uint32_t)(a.seed >> 32));
  const uint32_t episode = a.episode + ((MODE == 2 && a.episode_dev) ? __ldg(a.episode_dev) : 0u);
  const int64_t env0 = a.env_offset + (int64_t)e0;
  uint4* rec = s_rec + ql * C::PQ;

  uint32_t xw[B], yw[B];
#pragma unroll
  for (int j = 0; j < B; ++j) {
    const bool own = !C::kGhost || j < B - 1 || j * S + s < A;
    const uint32_t off = row0 + (uint32_t)(j * S) * ld;
    xw[j] = own ? ld_stream_u32(a.start_x + off) : 0xFFFFFFFFu;
    yw[j] = own ? ld_stream_u32(a.start_y + off) : 0xFFFFFFFFu;
#pragma unroll
    for (int k = 0; k < 4; ++k) s_acc[(j * 4 + k) * kCongCoopThreads + tid] = 0.0;
  }
  double s_pen[4] = {0, 0, 0, 0};
  int csum[4] = {0, 0, 0, 0};
  double disc = 1.0;

#pragma unroll 1
  for (int t = 0; t < T; ++t) {
    uint32_t aw[B], mw[B];
    {
      const uint8_t* act_t = a.actions + (int64_t)t * A * a.ld;      // uniform; per-thread offsets stay 32-bit
      const uint8_t* mov_t = MODE == 1 ? a.moves + (int64_t)t * A * a.ld : nullptr;
#pragma unroll
      for (int j = 0; j < B; ++j) {
        const uint32_t off = row0 + (uint32_t)(j * S) * ld;
        if (!C::kGhost || j < B - 1 || j * S + s < A) {
          aw[j] = ld_stream_u32(act_t + off);
          mw[j] = MODE == 1 ? ld_stream_u32(mov_t + off) : aw[j];
        } else {
          aw[j] = mw[j] = 0x04040404u;
        }
      }
    }
    if (MODE == 2) {                                                // as in the step kernel, with this step's t
      uint4* wq = rec;
#pragma unroll
      for (int m = 0; m * S < 4 * NQ; ++m) {
        const int b = m * S + s;
        if (4 * NQ % S == 0 || b < 4 * NQ) {
          const uint64_t id = (uint64_t)(env0 + (b & 3));
          wq[b] = philox4x32_10(make_uint4((uint32_t)id, (uint32_t)(id >> 32), (uint32_t)t,
                                           (uint32_t)(b >> 2) | (episode << 3)), key);
        }
      }
      __syncwarp();
      const uint32_t* ww = reinterpret_cast<const uint32_t*>(wq);
#pragma unroll
      for (int j = 0; j < B; ++j) {
        const int i = j * S + s;
        uint32_t m4 = 0u;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const uint32_t w = ww[(((i >> 2) * 4 + k) << 2) + (i & 3)];
          const uint32_t act = (aw[j] >> (8 * k)) & 0xFFu;
          const uint32_t mv = ((uint64_t)w < a.keep_threshold) ? act : w % 5u;
          m4 |= mv << (8 * k);
        }
        if (!C::kGhost || j < B - 1 || i < A) mw[j] = m4;
      }
      __syncwarp();                                                 // the records below reuse the block buffer
    }

    // transition (congestion.py:49-75) and the records every lane of the group scans
    uint32_t k0[B], k1[B], k2[B];
    uint32_t at_origin = 0u;
#pragma unroll
    for (int j = 0; j < B; ++j) {
      const bool own = !C::kGhost || j < B - 1 || j * S + s < A;
      const uint32_t ox = xw[j], oy = yw[j];
      grid_move4(xw[j], yw[j], mw[j], size4);
      k0[j] = small_key ? ox + 2u * xw[j] : xw[j];
      k1[j] = small_key ? oy + 2u * yw[j] : yw[j];
      k2[j] = small_key ? 0u : (((xw[j] + k01) - ox) | (((yw[j] + k01) - oy) << 2));
      if (!own) {
        if (small_key) k0[j] = never;
        else k2[j] = never;
        xw[j] = yw[j] = 0xFFFFFFFFu;                                // a padding agent stays off the grid
      }
      rec[j * S + s] = make_uint4(k0[j], k1[j], k2[j], own ? ((((aw[j] >> 2) & k01) ^ k01) << 7) : 0u);
      if (own) at_origin += zero_bytes01(xw[j] | yw[j]);           // congestion.py:97
    }
    __syncwarp();
    uint32_t r[B], seen[B], z[B];
    if (a.size <= 42) congestion_scan<A, S, 2, true>(rec, k0, k1, k2, s, r, seen, z);
    else if (a.size <= 84) congestion_scan<A, S, 2, false>(rec, k0, k1, k2, s, r, seen, z);
    else if (a.size <= 127) congestion_scan<A, S, 3, true>(rec, k0, k1, k2, s, r, seen, z);
    else congestion_scan<A, S, 3, false>(rec, k0, k1, k2, s, r, seen, z);
#pragma unroll
    for (int off = 1; off < S; off <<= 1) at_origin += __shfl_xor_sync(0xffffffffu, at_origin, off * EPW);

    // congestion.py:93-100 and meta_agent.py:21-22; identical on every lane of the group
    const int cost[4] = {max(0, A / 3 - (int)(at_origin & 0xFFu)), max(0, A / 3 - (int)((at_origin >> 8) & 0xFFu)),
                         max(0, A / 3 - (int)((at_origin >> 16) & 0xFFu)), max(0, A / 3 - (int)(at_origin >> 24))};
    float pen[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      pen[k] = (float)(lam * cost[k]);                              // the step kernel publishes the penalty as f32
      s_pen[k] += disc * (double)pen[k];
      csum[k] += cost[k];
    }
    if (a.g_mode == 1 && live && s == 0)
      st_stream_f4(a.g_scratch + (int64_t)t * a.ld + e0, make_float4(pen[0], pen[1], pen[2], pen[3]));
    float* G_t = a.G + (int64_t)t * A * a.ld;
#pragma unroll
    for (int j = 0; j < B; ++j) {
      if (C::kGhost && j == B - 1 && j * S + s >= A) continue;
      const uint32_t conw = (r[j] - z[j] - k01) & __umulhi(seen[j], 0xFFu << 25);
      const float4 r4 = a.wait_reward ? congestion_reward4<true>(aw[j], conw, xw[j], yw[j], a.demand, W, a.wait_reward)
                                      : congestion_reward4<false>(aw[j], conw, xw[j], yw[j], a.demand, W, nullptr);
      const float rr[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) s_acc[(j * 4 + k) * kCongCoopThreads + tid] += disc * (double)rr[k];
      const uint32_t off = row0 + (uint32_t)(j * S) * ld;
      if (a.g_mode == 1 && live) {
        st_stream_f4(G_t + off, r4);
      } else if (a.g_mode == 2 && live) {                           // agent.py:129-132
        st_stream_f4(G_t + off,
                     make_float4((float)(disc * ((double)rr[0] - (double)pen[0])), (float)(disc * ((double)rr[1] - (double)pen[1])),
                                 (float)(disc * ((double)rr[2] - (double)pen[2])), (float)(disc * ((double)rr[3] - (double)pen[3]))));
      }
    }
    disc *= a.gamma;
    __syncwarp();                                                   // the next step overwrites the records
  }

  bool valid[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) valid[k] = live && ((int64_t)e0 + k < a.n_envs);
  double* out = a.partials ? a.partials + (int64_t)blockIdx.x * stats_len(A, 1) : nullptr;
  if (live && s == 0) st_stream_i4(a.C + e0, make_int4(csum[0], csum[1], csum[2], csum[3]));
#pragma unroll
  for (int j = 0; j < B; ++j) {
    const bool own = !C::kGhost || j < B - 1 || j * S + s < A;
    const uint32_t off = row0 + (uint32_t)(j * S) * ld;
    double raw[4], mod[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      raw[k] = s_acc[(j * 4 + k) * kCongCoopThreads + tid];
      mod[k] = raw[k] - s_pen[k];
    }
    if (live && own) {
      if (a.final_x) st_stream_u32(a.final_x + off, xw[j]);
      if (a.final_y) st_stream_u32(a.final_y + off, yw[j]);
      st_stream_f4(a.R + off, make_float4((float)raw[0], (float)raw[1], (float)raw[2], (float)raw[3]));
      st_stream_f4(a.modR + off, make_float4((float)mod[0], (float)mod[1], (float)mod[2], (float)mod[3]));
    }
    if (out) {                                                      // uniform
      double v_raw = 0.0, v_mod = 0.0;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        v_raw += (valid[k] && own) ? raw[k] : 0.0;
        v_mod += (valid[k] && own) ? mod[k] : 0.0;
      }
      const double b_raw = slot_block_sum<S>(v_raw, s_red, s, q);
      const double b_mod = slot_block_sum<S>(v_mod, s_red, s, q);
      if (tid < S && j * S + tid < A) {
        out[2 + j * S + tid] = b_raw;
        out[2 + A + j * S + tid] = b_mod;
      }
    }
  }
  if (out) {
    const double thr = a.thresholds ? __ldg(a.thresholds) : 0.0;
    double c = 0.0, viol = 0.0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      c += (valid[k] && s == 0) ? (double)csum[k] : 0.0;
      viol += (valid[k] && s == 0 && a.thresholds && (double)csum[k] > thr) ? 1.0 : 0.0;
    }
    const double bc = slot_block_sum<S>(c, s_red, s, q);
    const double bv = slot_block_sum<S>(viol, s_red, s, q);
    if (tid == 0) {
      out[0] = bc;
      out[1] = bv;
      out[2 + 2 * A] = 0.0;
    }
  }

  if (a.g_mode == 1) {                                              // agent.py:200-206, in place over the stored rewards
    __threadfence_block();                                          // lane s = 0 wrote the penalties all lanes read back
    __syncwarp();
    if (live) {
#pragma unroll
      for (int j = 0; j < B; ++j)
#pragma unroll
        for (int k = 0; k < 4; ++k) s_acc[(j * 4 + k) * kCongCoopThreads + tid] = 0.0;
      for (int t = T - 1; t >= 0; --t) {
        const float4 qv = ld_f4(a.g_scratch + (int64_t)t * a.ld + e0);
        const float qq[4] = {qv.x, qv.y, qv.z, qv.w};
        float* G_t = a.G + (int64_t)t * A * a.ld;
#pragma unroll
        for (int j = 0; j < B; ++j) {
          if (C::kGhost && j == B - 1 && j * S + s >= A) continue;
          float* gp = G_t + (row0 + (uint32_t)(j * S) * ld);
          const float4 rv = ld_f4(gp);
          const float rr[4] = {rv.x, rv.y, rv.z, rv.w};
          float o[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            double& run = s_acc[(j * 4 + k) * kCongCoopThreads + tid];
            run = ((double)rr[k] - (double)qq[k]) + a.gamma * run;
            o[k] = (float)run;
          }
          st_stream_f4(gp, make_float4(o[0], o[1], o[2], o[3]));
        }
      }
    }
  }
}

template <int MODE>
int launch_congestion_coop_rollout(int A, const CongestionRolloutArgs& a, unsigned* grid_out, cudaStream_t st) {
  return dispatch<9, 32>(A, [&](auto kA) {
    using C = CongCoop<kA, 4>;
    auto kern = congestion_coop_rollout_kernel<kA, 4, MODE>;
    const size_t smem = CongCoopRoll<kA, 4>::kSmem;
    if (smem + 256 > 48 * 1024)
      SMARL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const unsigned grid = (unsigned)((a.n_groups + C::EPC - 1) / C::EPC);
    kern<<<grid, kCongCoopThreads, smem, st>>>(a);
    *grid_out = grid;
    SMARL_CUDA(cudaGetLastError());
    return SMARL_OK;
  }, "cooperative Congestion kernels cover n_agents 9..32 (got %d)");
}

template <int S, int MODE>
static int launch_sm(int A, const CongestionStepArgs& a, cudaStream_t st) {
  return dispatch<9, 32>(A, [&](auto kA) {
    using C = CongCoop<kA, S>;
    auto kern = congestion_coop_step_kernel<kA, S, MODE>;
    const size_t smem = C::kSmem;
    if (smem > 48 * 1024)
      SMARL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const unsigned grid = (unsigned)((a.n_groups + C::EPC - 1) / C::EPC);
    SMARL_CUDA(launch_pdl(kern, grid, kCongCoopThreads, smem, st, a));
    SMARL_CUDA(cudaGetLastError());
    return SMARL_OK;
  }, "cooperative Congestion kernels cover n_agents 9..32 (got %d)");
}

template <int MODE>
int launch_congestion_coop_step(int A, int S, const CongestionStepArgs& a, cudaStream_t st) {
  return S == 2 ? launch_sm<2, MODE>(A, a, st) : launch_sm<4, MODE>(A, a, st);
}

#if SMARL_TU_IS(0)
template int launch_congestion_coop_step<0>(int, int, const CongestionStepArgs&, cudaStream_t);
#endif
#if SMARL_TU_IS(1)
template int launch_congestion_coop_step<1>(int, int, const CongestionStepArgs&, cudaStream_t);
#endif
#if SMARL_TU_IS(2)
template int launch_congestion_coop_step<2>(int, int, const CongestionStepArgs&, cudaStream_t);
#endif
#if SMARL_TU_IS(3)
template int launch_congestion_coop_rollout<0>(int, const CongestionRolloutArgs&, unsigned*, cudaStream_t);
#endif
#if SMARL_TU_IS(4)
template int launch_congestion_coop_rollout<1>(int, const CongestionRolloutArgs&, unsigned*, cudaStream_t);
#endif
#if SMARL_TU_IS(5)
template int launch_congestion_coop_rollout<2>(int, const CongestionRolloutArgs&, unsigned*, cudaStream_t);
#endif

}  // namespace smarl
