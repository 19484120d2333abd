// Fused per-agent discrete policies, tensor-core build (sm_100a: tcgen05.mma + tensor memory).
//
// Same contract as policy.cu (DiscretePolicy of safe_multi_agent_RL/agent.py:23-47 for all envs and agents, called
// from main.py:30-35): u8 position rows in, u8 action rows + f32 log-probabilities out.  Of the 2A*16 + 80
// multiply-adds per agent-step, fc1 (2A*16: 512 of 592 at A = 16) is ONE GEMM per tile of envs,
//
//     H[128 envs x 16*GA] = X[128 envs x 2A] * W1[2A x 16*GA]          (all agents of a group side by side along N)
//
// because every agent reads the same joint observation X.  It runs on the tensor cores with f32-grade accuracy:
//   * X holds grid coordinates 0..254: exact in bf16.
//   * every fp32 weight is split into three bf16 pieces w = hi + mid + lo (8 + 8 + 8 mantissa bits: the split is exact
//     for normal weights), so X*W1 = X*hi + X*mid + X*lo with exact products and f32 accumulation in tensor memory --
//     three passes over the same A operand with three B operands, smallest pieces first.
//   * the bias rides along as one more K step: X gets a constant block (1,1,1,0,...) and W1 the rows (b_hi, b_mid, b_lo).
// Measured error of the pre-activations against float64: ~5e-8 relative (tools/umma_probe.cu pins the descriptor layout
// and the accuracy on B200; tests/test_gpu_policy_fused.py holds the log-probabilities to 1e-5 against PyTorch).
// relu, fc2 (80 multiply-adds as 40 packed FFMA2), softmax, the Philox inverse-CDF sample and log_prob run on the FP32
// pipes straight out of tensor memory: a thread owns one TMEM lane = one env row of each of the R tiles of the CTA
// iteration and walks over its warpgroup's agents, 16 accumulator columns (tcgen05.ld.32x32b.x16) per agent and tile,
// the next agent's columns in flight while it computes.  Every fc2 weight it loads from shared memory (a 512-byte
// broadcast per LDS.128: tools/fma_probe.cu measures ~8 cycles of the SM's load path each when all four
// sub-partitions ask) therefore serves R = 2 envs.
//
// CTA = NWG warpgroups (the same 128 lanes, different agents); a CTA iteration = R tiles of 128 envs for one group of
// GA <= 8 agents: R * 16 * GA accumulator columns (256 of the SM's 512 at GA = 8, so two CTAs per SM overlap one
// CTA's staging + MMA with the other's epilogue).  Persistent over the env tiles; the raw u8 position rows of the
// next iteration travel global -> shared with cp.async during the epilogue and are converted to the bf16 K-major image
// (canonical no-swizzle layout: [K chunk of 8][row group of 8][8 rows][16 B]) before the MMAs; the bf16 images of the
// group's weights are built once per CTA from the fp32 parameters (no prepared buffers in the ABI).
// Measured (B200, 2^20 envs): A = 16: 168 us per launch against 509 us for the FP32-pipe build (policy.cu) and
// ~1960 us for the PyTorch glue; A = 32: 366 against 1810 us; A = 8: 80 against 175 us; A = 3: 39 against 50 us.
// The epilogue is what bounds it: ~190 issued instructions per (agent, env) pair of 32 lanes at 54 % issue
// utilisation (ncu, profiles/r02); the tensor pipe is 7 % busy.
#include <cuda_bf16.h>

#include "policy.cuh"
#include "tc.cuh"

namespace smarl {

template <int A, int GMAX, int R, int RT>
struct TcCfg {
  static constexpr int H = kPolHidden, NA = kPolActions;
  static constexpr int NGROUPS = (A + GMAX - 1) / GMAX;                    // agent groups; a CTA serves one
  static constexpr int GA = NGROUPS == 1 ? A : (((A + NGROUPS - 1) / NGROUPS + 3) & ~3);   // agents per group (multiple of 4 when split)
  static constexpr bool RAGGED = NGROUPS * GA != A;                        // the last group holds fewer agents
  static constexpr int NWG = GA > 4 ? 2 : 1;                               // warpgroups sharing the accumulator tiles
  static constexpr int AW = NWG == 1 ? GA : ((((GA + NWG - 1) / NWG) + 3) & ~3);   // agents per warpgroup
  static constexpr bool FULL = !RAGGED && NWG * AW == GA;                  // every (warpgroup, agent slot) exists
  static constexpr int N = H * GA;                                         // accumulator columns per tile = MMA N
  static constexpr int COLS = R * N <= 32 ? 32 : (R * N <= 64 ? 64 : (R * N <= 128 ? 128 : (R * N <= 256 ? 256 : 512)));
  static constexpr int KIN = 2 * A;                                        // observation components
  static constexpr int KST = (KIN + 15) / 16;                              // K steps (16 inputs each) per weight piece
  static constexpr int ACH = 2 * KST + 2;                                  // K chunks of one X image (+ the bias step)
  static constexpr int BCH = 6 * KST + 2;                                  // K chunks of the W1 image: 3 pieces + bias step
  static constexpr int NWR = R / RT;                                       // warpgroup sets along the tiles: a thread owns RT of the R tiles
  static constexpr int THREADS = 128 * NWG * NWR;
  static constexpr int ROWS = 128 * R;                                     // envs per CTA iteration
  static constexpr int W2S = H * NA + 8;                                   // floats per agent: w2t[c][u], b2[5], pad
  static constexpr uint32_t A_CHUNK = 128 * 16, B_CHUNK = N * 16;          // bytes per K chunk
  static constexpr uint32_t A_TILE = ACH * A_CHUNK;
  static constexpr size_t kSmemA = (size_t)R * A_TILE;
  static constexpr size_t kSmemB = (size_t)BCH * B_CHUNK;
  static constexpr size_t kSmemRaw = (size_t)16 * KST * ROWS;              // u8 [16 KST][ROWS]: the raw position rows
  static constexpr size_t kSmemW2 = (size_t)GA * W2S * sizeof(float);
  static constexpr size_t kSmem = kSmemA + kSmemB + kSmemRaw + kSmemW2 + 128;
  static_assert(N % 16 == 0 && N >= 16 && N <= 256, "MMA N out of range");
  static_assert(R * N <= 512, "accumulators exceed tensor memory");
  static_assert(R % RT == 0, "tiles per thread must divide the tiles per CTA");
};

__device__ __forceinline__ uint16_t bf16_bits(float x) { return __bfloat16_as_ushort(__float2bfloat16_rn(x)); }

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src, bool valid) {
  const uint32_t n = valid ? 16u : 0u;                              // 0 source bytes: the 16 destination bytes are zero-filled
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(tc::smem_u32(smem_dst)), "l"(gmem_src), "r"(n) : "memory");
}
__device__ __forceinline__ void st_u8_if(uint8_t* p, uint32_t v, bool on) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %2, 0;\n\t@p st.global.u8 [%0], %1;\n\t}" ::"l"(p), "r"(v), "r"((uint32_t)on) : "memory");
}
__device__ __forceinline__ void st_f32_if(float* p, float v, bool on) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %2, 0;\n\t@p st.global.f32 [%0], %1;\n\t}" ::"l"(p), "f"(v), "r"((uint32_t)on) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

template <int A, int GMAX, int R, int RT>
__global__ void __launch_bounds__(TcCfg<A, GMAX, R, RT>::THREADS, TcCfg<A, GMAX, R, RT>::THREADS >= 512 ? 2 : 0)
    policy_act_discrete_tc_kernel(const PolicyArgs a) {
  pdl_prologue();   // programmatic dependent launch: the previous grid has completed past this point (common.cuh)
  using C = TcCfg<A, GMAX, R, RT>;
  constexpr int NWG = C::NWG, H = C::H, NA = C::NA, N = C::N, KST = C::KST, GA = C::GA, AW = C::AW, ROWS = C::ROWS;
  extern __shared__ __align__(128) uint8_t s_raw[];
  uint8_t* s_a = s_raw;                                             // X images  [R][ACH][16 row groups][8][16 B]
  uint8_t* s_b = s_a + C::kSmemA;                                   // W1 image  [BCH][N / 8][8][16 B]
  uint8_t* s_pos = s_b + C::kSmemB;                                 // raw u8    [16 KST][ROWS]
  float* s_w2 = reinterpret_cast<float*>(s_pos + C::kSmemRaw);      // [GA][W2S], scaled by log2(e)
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(s_w2) + C::kSmemW2);
  uint32_t* s_slot = reinterpret_cast<uint32_t*>(s_bar + 1);
  const int tid = threadIdx.x;
  const int a0 = blockIdx.y * GA;                                   // first agent of this CTA's group
  const int n_real = C::RAGGED ? ((A - a0) < GA ? (A - a0) : GA) : GA;   // agents of the group that exist

  // ---- one-time setup: barrier, tensor memory, the bf16 images of the group's weights ---------------------------
  if (tid == 0) tc::mbar_init(s_bar, 1);
  if (tid < 32) tc::tmem_alloc(s_slot, C::COLS);
  {
    // W1 pieces: column n = (local agent, unit), K chunk = piece * 2 KST + k / 8
    constexpr int KP = 16 * KST;
    for (int i = tid; i < GA * KP * H; i += C::THREADS) {
      const int u = i % H, k = (i / H) % KP, j = i / (H * KP);
      float w = (j < n_real && k < C::KIN) ? __ldg(a.w1 + ((size_t)(a0 + j) * C::KIN + k) * H + u) : 0.f;
      const int n = j * H + u;
      uint8_t* dst = s_b + (size_t)(k >> 3) * C::B_CHUNK + (n >> 3) * 128 + (n & 7) * 16 + (k & 7) * 2;
#pragma unroll
      for (int piece = 0; piece < 3; ++piece) {
        const __nv_bfloat16 p = __float2bfloat16_rn(w);
        *reinterpret_cast<uint16_t*>(dst + (size_t)piece * 2 * KST * C::B_CHUNK) = __bfloat16_as_ushort(p);
        w -= __bfloat162float(p);                                   // exact: the remainder of an fp32 value
      }
    }
    // bias step: K chunk 6 KST holds (b_hi, b_mid, b_lo, 0, ...) per column, chunk 6 KST + 1 zeros
    for (int i = tid; i < N * 16; i += C::THREADS) {
      const int kk = i % 16, n = i / 16, j = n / H, u = n % H;
      float v = 0.f;
      if (kk < 3 && j < n_real) {
        float w = __ldg(a.b1 + (size_t)(a0 + j) * H + u);
        for (int piece = 0; piece < kk; ++piece) w -= __bfloat162float(__float2bfloat16_rn(w));
        v = w;
      }
      uint8_t* dst = s_b + (size_t)(6 * KST + (kk >> 3)) * C::B_CHUNK + (n >> 3) * 128 + (n & 7) * 16 + (kk & 7) * 2;
      *reinterpret_cast<uint16_t*>(dst) = bf16_bits(v);
    }
    // X images, constant part: chunk 2 KST = (1, 1, 1, 0, ...) for every env row, chunk 2 KST + 1 zeros
    for (int i = tid; i < R * 2 * 128; i += C::THREADS) {
      const int r = i / 256, q = i % 256;
      const uint32_t one2 = 0x3F803F80u;                            // two bf16 ones
      const uint4 v = q < 128 ? make_uint4(one2, 0x00003F80u, 0u, 0u) : make_uint4(0u, 0u, 0u, 0u);
      *reinterpret_cast<uint4*>(s_a + (size_t)r * C::A_TILE + (size_t)2 * KST * C::A_CHUNK + (size_t)q * 16) = v;
    }
    // raw position rows beyond the 2A real ones stay zero (K padding)
    for (int i = tid; i < (int)(C::kSmemRaw / 16); i += C::THREADS) reinterpret_cast<uint4*>(s_pos)[i] = make_uint4(0u, 0u, 0u, 0u);
    // fc2 in log2 units (policy_head): w2t[c][u] * log2(e) (pairs along u feed FFMA2), then b2 * log2(e)
    for (int i = tid; i < GA * C::W2S; i += C::THREADS) {
      const int j = i / C::W2S, r = i % C::W2S;
      float v = 0.f;
      if (j < n_real) {
        if (r < H * NA) v = __ldg(a.w2 + ((size_t)(a0 + j) * H + r % H) * NA + r / H);
        else if (r < H * NA + NA) v = __ldg(a.b2 + (size_t)(a0 + j) * NA + (r - H * NA));
      }
      s_w2[i] = v * kLog2e;
    }
  }
  tc::fence_async_smem();
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem = *s_slot;

  const int wg = (tid >> 7) % NWG, row = tid & 127;                 // agent warpgroup, TMEM lane
  const int r_lo = ((tid >> 7) / NWG) * RT;                         // first of this thread's RT tiles
  const uint32_t t_lane = tmem + ((uint32_t)(row & ~31) << 16);     // this warp's 32 TMEM lanes
  const uint2 key = policy_key(a.seed);
  const uint32_t episode = a.episode + (a.episode_dev ? __ldg(a.episode_dev) : 0u);
  const uint32_t t_word = a.t | episode << 16, ep_hi = policy_episode_hi(episode);
  const uint32_t idesc = tc::idesc_bf16_f32(128, N);
  const uint32_t sa_addr = tc::smem_u32(s_a), sb_addr = tc::smem_u32(s_b);
  const int j_lo = wg * AW;                                         // first local agent of this warpgroup
  const float* w2_lo = s_w2 + j_lo * C::W2S;
  const uint32_t ld32 = (uint32_t)a.ld;
  const bool want_logp = a.logp != nullptr;
  uint32_t phase = 0;

  // The raw u8 position rows of the next ROWS envs travel global -> shared with cp.async (16 envs per copy) while the
  // current envs are in the epilogue; rows past ld are zero-filled.
  auto fetch = [&](int64_t st) {
    const int64_t e_base = st * ROWS;
    for (int i = tid; i < C::KIN * (ROWS / 16); i += C::THREADS) {
      const int k = i / (ROWS / 16), q = i % (ROWS / 16);
      const int64_t e = e_base + 16 * q;
      const bool valid = e < a.ld;
      const uint8_t* src = ((k & 1) ? a.pos_y : a.pos_x) + (valid ? (int64_t)(k >> 1) * a.ld + e : 0);
      cp_async16(s_pos + (size_t)k * ROWS + 16 * q, src, valid);
    }
    cp_async_commit();
  };
  if ((int64_t)blockIdx.x < a.n_tiles) fetch(blockIdx.x);

  for (int64_t st = blockIdx.x; st < a.n_tiles; st += gridDim.x) {
    cp_async_wait_all();
    __syncthreads();
    // ---- the joint observation as bf16 K-major images: element k = 2 i is x_i, k = 2 i + 1 is y_i (main.py:33) ----
    // u8 -> bf16 without the conversion unit: 0x4B000000 | b is the float 2^23 + b, minus 2^23 gives b exactly, and the
    // upper halves of two such floats are the bf16 pair (PRMT).  All loads of a thread's items are issued first.
    {
      constexpr int ITEMS = (ROWS * 2 * KST + C::THREADS - 1) / C::THREADS;
      uint32_t b[ITEMS][8];
#pragma unroll
      for (int it = 0; it < ITEMS; ++it) {
        const int i = tid + it * C::THREADS;
        const int rr = i % ROWS, c = i / ROWS;
#pragma unroll
        for (int q = 0; q < 8; ++q) b[it][q] = (i < ROWS * 2 * KST) ? s_pos[(size_t)(8 * c + q) * ROWS + rr] : 0u;
      }
#pragma unroll
      for (int it = 0; it < ITEMS; ++it) {
        const int i = tid + it * C::THREADS;
        const int rr = i % ROWS, c = i / ROWS;
        uint32_t w[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float x = __uint_as_float(0x4B000000u | b[it][2 * q]) - 8388608.0f;
          const float y = __uint_as_float(0x4B000000u | b[it][2 * q + 1]) - 8388608.0f;
          w[q] = __byte_perm(__float_as_uint(x), __float_as_uint(y), 0x7632);
        }
        if (i < ROWS * 2 * KST)
          *reinterpret_cast<uint4*>(s_a + (size_t)(rr >> 7) * C::A_TILE + (size_t)c * C::A_CHUNK + (size_t)(rr & 127) * 16) =
              make_uint4(w[0], w[1], w[2], w[3]);
      }
    }
    tc::fence_async_smem();
    tc::fence_before_sync();              // also orders the previous epilogue's tcgen05.ld before the MMAs that overwrite it
    __syncthreads();
    // ---- fc1 on the tensor cores: one elected thread issues, pieces lo -> mid -> hi, then the bias step ---------
    if (tid == 0) {
      tc::fence_after_sync();
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const uint32_t sa_r = sa_addr + r * C::A_TILE, d_r = tmem + r * N;
#pragma unroll
        for (int piece = 2; piece >= 0; --piece)
#pragma unroll
          for (int ks = 0; ks < KST; ++ks)
            tc::mma_bf16(d_r, tc::smem_desc(sa_r + 2 * ks * C::A_CHUNK, C::A_CHUNK, 128),
                         tc::smem_desc(sb_addr + (piece * 2 * KST + 2 * ks) * C::B_CHUNK, C::B_CHUNK, 128), idesc,
                         !(piece == 2 && ks == 0));
        tc::mma_bf16(d_r, tc::smem_desc(sa_r + 2 * KST * C::A_CHUNK, C::A_CHUNK, 128),
                     tc::smem_desc(sb_addr + 6 * KST * C::B_CHUNK, C::B_CHUNK, 128), idesc, true);
      }
      tc::mma_commit(s_bar);
    }
    if (st + gridDim.x < a.n_tiles) fetch(st + gridDim.x);
    // the Philox blocks of this iteration (one per tile row and four agents) are computed while the MMAs run
    const int64_t e0 = st * ROWS + 128 * r_lo + row;
    uint4 rnd_all[(AW + 3) / 4][RT];
#pragma unroll
    for (int g4 = 0; g4 < (AW + 3) / 4; ++g4)
#pragma unroll
      for (int r = 0; r < RT; ++r)
        rnd_all[g4][r] = policy_words((uint64_t)(a.env_offset + e0 + 128 * r), t_word, ep_hi,
                                       (a0 + j_lo + 4 * g4) >> 2, key);
    tc::mbar_wait(s_bar, phase);
    phase ^= 1u;
    tc::fence_after_sync();
    // ---- epilogue out of tensor memory: relu, fc2, softmax, sample, log_prob; a thread owns row `row` of each of the
    //      R tiles, so every fc2 weight it loads serves R envs ---------------------------------------------------
    uint32_t idx[RT];                                                // element index of (agent, env) in actions / logp
    bool live[RT], live_lp[RT];
#pragma unroll
    for (int r = 0; r < RT; ++r) {
      live[r] = e0 + 128 * r < a.ld;
      live_lp[r] = live[r] && want_logp;
      idx[r] = (uint32_t)(a0 + j_lo) * ld32 + (uint32_t)(e0 + 128 * r);
    }
    uint4 rnd[RT];
    uint32_t hbuf[2][RT][16];                                        // the next agent's columns load while this one computes
    if (C::FULL || j_lo < n_real) {
#pragma unroll
      for (int r = 0; r < RT; ++r) tc::tmem_ld16_raw(t_lane + (uint32_t)((r_lo + r) * N + j_lo * H), hbuf[0][r]);
    }
#pragma unroll
    for (int jj = 0; jj < AW; ++jj) {
      if (C::FULL || j_lo + jj < n_real) {
        uint32_t (&hr)[RT][16] = hbuf[jj & 1];
        if ((jj & 3) == 0) {
#pragma unroll
          for (int r = 0; r < RT; ++r) rnd[r] = rnd_all[jj / 4][r];
        }
        const float* w2 = w2_lo + jj * C::W2S;
        float2 acc[RT][NA];
#pragma unroll
        for (int c = 0; c < NA; ++c) {
          const float b = w2[H * NA + c];
#pragma unroll
          for (int r = 0; r < RT; ++r) acc[r][c] = make_float2(b, 0.f);
        }
#pragma unroll
        for (int r = 0; r < RT; ++r) tc::tmem_ld_wait_regs(hr[r]);
        if (jj + 1 < AW && (C::FULL || j_lo + jj + 1 < n_real)) {
#pragma unroll
          for (int r = 0; r < RT; ++r) tc::tmem_ld16_raw(t_lane + (uint32_t)((r_lo + r) * N + (j_lo + jj + 1) * H), hbuf[(jj + 1) & 1][r]);
        }
#pragma unroll
        for (int p4 = 0; p4 < H / 4; ++p4) {
          float2 ra[RT], rb[RT];
#pragma unroll
          for (int r = 0; r < RT; ++r) {
            ra[r] = make_float2(fmaxf(__uint_as_float(hr[r][4 * p4 + 0]), 0.f), fmaxf(__uint_as_float(hr[r][4 * p4 + 1]), 0.f));
            rb[r] = make_float2(fmaxf(__uint_as_float(hr[r][4 * p4 + 2]), 0.f), fmaxf(__uint_as_float(hr[r][4 * p4 + 3]), 0.f));
          }
#pragma unroll
          for (int c = 0; c < NA; ++c) {
            const float4 w = *reinterpret_cast<const float4*>(w2 + c * H + 4 * p4);
#pragma unroll
            for (int r = 0; r < RT; ++r) {
              acc[r][c] = tc::ffma2(ra[r], make_float2(w.x, w.y), acc[r][c]);
              acc[r][c] = tc::ffma2(rb[r], make_float2(w.z, w.w), acc[r][c]);
            }
          }
        }
#pragma unroll
        for (int r = 0; r < RT; ++r) {
          float l2[NA];
#pragma unroll
          for (int c = 0; c < NA; ++c) l2[c] = acc[r][c].x + acc[r][c].y;
          int pick;
          float lp;
          policy_head(l2, word_of(rnd[r], jj & 3), pick, lp);
          // predicated stores, no branch: the whole epilogue of an iteration stays one basic block, so the softmax /
          // sampling chain of one agent is scheduled under the next agent's fc2
          st_u8_if(a.actions + idx[r], (uint32_t)pick, live[r]);
          st_f32_if(a.logp + idx[r], lp, live_lp[r]);
          idx[r] += ld32;
        }
      }
    }
  }
  tc::fence_before_sync();
  __syncthreads();
  if (tid < 32) tc::tmem_dealloc(tmem, C::COLS);
}

template <int A, int GMAX, int R, int RT>
static int launch_tc(const PolicyArgs& a_in, int sms, cudaStream_t st) {
  using C = TcCfg<A, GMAX, R, RT>;
  PolicyArgs a = a_in;
  auto kern = policy_act_discrete_tc_kernel<A, GMAX, R, RT>;
  // At most 512 / COLS CTAs of tensor memory fit an SM: size the shared-memory request so that no more than that
  // become resident (a surplus CTA would spin in tcgen05.alloc until a resident one exits).
  const int tmem_ctas = 512 / C::COLS;
  size_t smem = C::kSmem;
  const size_t floor_smem = (size_t)(227 * 1024) / (tmem_ctas + 1) + 1;
  if (smem < floor_smem) smem = floor_smem;
  if (smem > 227 * 1024) {
    set_error("tensor-core policy: %d agents need %zu bytes of shared memory", A, smem);
    return SMARL_EUNSUPPORTED;
  }
  if ((uint64_t)A * (uint64_t)a.ld >= (1ull << 32)) {
    set_error("tensor-core policy: n_agents * ld = %llu does not fit 32-bit element indices", (unsigned long long)A * a.ld);
    return SMARL_EUNSUPPORTED;
  }
  // per-kernel launch setup, once per device (the attribute calls cost host time on every step otherwise)
  static int cached_dev = -1, cached_per_sm = 1;
  int dev = 0;
  SMARL_CUDA(cudaGetDevice(&dev));
  if (dev != cached_dev) {
    SMARL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    SMARL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    // resident CTAs per SM: tensor memory (by construction of the shared-memory request) and registers; the occupancy
    // calculator is not asked because it assumes the default carveout and reported 1 where 2 CTAs run
    cudaFuncAttributes fa;
    SMARL_CUDA(cudaFuncGetAttributes(&fa, kern));
    int per_sm = tmem_ctas;
    const int by_regs = 65536 / (((fa.numRegs + 7) & ~7) * C::THREADS);
    if (per_sm > by_regs) per_sm = by_regs;
    if (per_sm > 2048 / C::THREADS) per_sm = 2048 / C::THREADS;
    if (per_sm < 1) per_sm = 1;
    cached_per_sm = per_sm;
    cached_dev = dev;
  }
  const int per_sm = cached_per_sm;
  a.n_tiles = (a.n_envs + C::ROWS - 1) / C::ROWS;                   // CTA iterations of ROWS envs
  int64_t gx = (int64_t)sms * per_sm / C::NGROUPS;
  if (gx < 1) gx = 1;
  if (gx > a.n_tiles) gx = a.n_tiles;
  SMARL_CUDA(launch_pdl(kern, dim3((unsigned)gx, C::NGROUPS), C::THREADS, smem, st, a));
  SMARL_CUDA(cudaGetLastError());
  return SMARL_OK;
}

// group_max: 16 = groups of up to 16 agents (256 accumulator columns, two warpgroups per CTA), 8 = groups of up to 8
// (128 columns, one warpgroup, more CTAs per SM; the tile's observation is staged once per group).
template <int A>
static int launch_tc_any(const PolicyArgs& a, int group_max, int sms, cudaStream_t st) {
  if (group_max == 16) return launch_tc<A, 8, 2, 1>(a, sms, st);     // variant 1: one tile per thread, twice the warps
  return launch_tc<A, 8, 2, 2>(a, sms, st);
}

int launch_policy_tc(const PolicyArgs& a, int n_agents, int group_max, int sms, cudaStream_t st) {
  return dispatch<1, 32>(n_agents, [&](auto kA) { return launch_tc_any<kA>(a, group_max, sms, st); });
}

}  // namespace smarl
