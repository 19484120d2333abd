// The learner's gradient of the DiscretePolicy over recorded episodes (sm_100a).
//
// Replaces the learner side of an agent cycle of the reference (loss agent.py:134-157 on the network of
// agent.py:23-47), which in PyTorch is T log_prob forwards, the loss and an autograd backward: for every agent a,
// step t < T and env e < n_envs, with x = obs_rec[t][:, e] (the joint state, 2A floats), c = actions[t][a][e] and the
// constant advantage psi = psi[t][a][e],
//   h = b1 + W1^T x    r = relu(h)    l = b2 + W2^T r    p = softmax(l)
//   L   += -scale psi log p_c
//   g_l  = -scale psi (onehot(c) - p)        dW2 += r (x) g_l     db2 += g_l
//   g_h  = (W2 g_l) * [h > 0]                dW1 += x (x) g_h     db1 += g_h     (relu backward: zero at h == 0)
// all in one kernel that reads the record slabs the on-policy rollouts write.
//
// Mapping.  One CTA = one agent x one chunk of (t, 256-env block) tiles; the chunks of an agent split its
// T * ceil(E / 256) tiles evenly, and their number P (policy_grad_chunks) comes from A, T and E only.  Per tile:
//   1. forward + backward, one sample per thread (FP32 pipes, the agent's weights in shared memory, exact expf / logf):
//      the thread writes its x, r, g_h and (g_l, psi log p_c) columns to shared memory.  -scale is applied at the end,
//      in f64, so the tile holds psi (onehot - p) and psi log p_c.
//   2. the weight-gradient contractions over the tile's samples as outer products [x; 1] (x) g_h (fc1 and b1) and
//      [r; 1] (x) [g_l, psi log p_c] (fc2, b2 and the loss): every thread owns a 4 x 4 register block of one of them
//      and a fixed slice of the tile's samples, and accumulates it with FFMA2 over sample pairs (even / odd samples in
//      the two halves).  Shared-memory rows are 260 floats apart, so consecutive rows start on different banks.
// Reduction order (no floating-point atomics): a thread's f32 block over its slice of one tile (<= 256 samples) is
// added into its f64 block after every tile; at the end of the chunk the slices' f64 blocks are summed in slice order
// and written to scratch as the chunk's partial; the last CTA of an agent to finish (an integer counter in scratch)
// sums the P partials in chunk order in f64, scales them by -scale and writes the f32 gradients; the last agent sums
// the agents' losses in agent order.  So the bits depend on the inputs and (A, NA, T, E) only, not on the device, the
// stream or the launch history.
//
// No tensor cores: fc1's inputs are not exact in bf16 on CoverageDiscretized, and an f32-grade three-piece bf16 split
// costs more than it saves at widths of 2A x 16 (policy_gauss.cu, DESIGN 3.9 / 3.15).
#include <math.h>

#include "policy.cuh"
#include "tc.cuh"

namespace smarl {

constexpr int kPgThreads = 256;
constexpr int kPgTile = 256;              // envs of one step per tile: one sample per thread in the forward
constexpr int kPgCtas = 1184;             // CTAs to aim for over all agents (P = kPgCtas / A chunks, at most n_tiles)
constexpr int kPgHeader = 64;             // doubles before the partials: 33 u32 counters, then the agents' losses

template <int A, int NA>
struct PgCfg {
  static constexpr int IN = 2 * A, H = kPolHidden, TE = kPgTile;
  static constexpr int SS = TE + 4;                              // row stride of the per-sample arrays
  static constexpr int RB = 4, CB = 4;                           // register block of a contraction item
  // fc1 items: rows [x (IN); 1] x columns g_h (16).  fc2 items: rows [r (16); 1] x columns [g_l (NA); psi log p_c].
  // Item (rb, cb) owns rows rb + k NRB (k < RB) and columns cb + j NCB (j < CB); rows and columns past the real ones
  // are zero in shared memory.
  static constexpr int NRB1 = (IN + 1 + RB - 1) / RB, NCB1 = H / CB;
  static constexpr int NRB2 = (H + 1 + RB - 1) / RB, NAP = (NA + 1 + CB - 1) / CB * CB, NCB2 = NAP / CB;
  static constexpr int I1 = NRB1 * NCB1, NI = I1 + NRB2 * NCB2;
  static constexpr int spl() {
    int s = 1;
    while (2 * s * NI <= kPgThreads && 8 * s <= TE) s *= 2;
    return s;
  }
  static constexpr int SPL = spl();                              // sample slices of a tile
  static constexpr int XR = NRB1 * RB, RR = NRB2 * RB;           // rows of s_x and s_r
  static constexpr int NOUT = IN * H + H + H * NA + NA + 1;      // gradients of one agent, then its loss
  static constexpr int WF = IN * H + H + H * NA + NA;            // floats of one agent's weights
  static constexpr int WFP = (WF + 3) / 4 * 4;
  static constexpr size_t kSampleFloats = (size_t)(XR + RR + H + NAP) * SS;
  static constexpr size_t kSmemBytes = (WFP + kSampleFloats) * sizeof(float);
  static_assert((size_t)SPL * NI * RB * CB * sizeof(double) <= kSampleFloats * sizeof(float),
                "the slice reduction reuses the sample arrays");
  static_assert(kSmemBytes <= 227 * 1024, "shared memory of one SM");
};

struct PolicyGradArgs {
  const float* obs;          // [T][2A][ld]
  const uint8_t* actions;    // [T][A][ld]
  const float* psi;          // [T][A][ld]
  const float* w1;
  const float* b1;
  const float* w2;
  const float* b2;
  float* dw1;
  float* db1;
  float* dw2;
  float* db2;
  double* loss;
  double* scratch;
  double scale;
  int64_t n_envs;
  int64_t ld;
  int64_t n_etiles;          // env blocks per step
  int64_t n_tiles;           // T * n_etiles
  int32_t n_chunks;          // P
};

// Chunks per agent: from the shape alone, so that the reduction tree does not depend on the device.
inline int64_t policy_grad_chunks(int A, int64_t n_steps, int64_t n_envs) {
  const int64_t n_tiles = n_steps * ((n_envs + kPgTile - 1) / kPgTile);
  const int64_t want = kPgCtas / A > 0 ? kPgCtas / A : 1;
  return n_tiles < want ? n_tiles : want;
}

template <int A, int NA>
__global__ void __launch_bounds__(kPgThreads, 1) policy_grad_kernel(const PolicyGradArgs a) {
  using C = PgCfg<A, NA>;
  constexpr int IN = C::IN, H = C::H, TE = C::TE, SS = C::SS, RB = C::RB, CB = C::CB;
  extern __shared__ __align__(16) float s_mem[];
  float* s_w1 = s_mem;                       // [IN][16]
  float* s_b1 = s_w1 + IN * H;               // [16]
  float* s_w2 = s_b1 + H;                    // [16][NA]
  float* s_b2 = s_w2 + H * NA;               // [NA]
  float* s_x = s_mem + C::WFP;               // [XR][SS]   x, ones, zeros
  float* s_r = s_x + C::XR * SS;             // [RR][SS]   r, ones, zeros
  float* s_gh = s_r + C::RR * SS;            // [16][SS]
  float* s_gl = s_gh + H * SS;               // [NAP][SS]  psi (onehot - p), psi log p_c, zeros
  __shared__ int s_last;

  const int tid = threadIdx.x;
  const int ag = (int)(blockIdx.x % A);
  const int64_t chunk = blockIdx.x / A;
  for (int i = tid; i < IN * H; i += kPgThreads) s_w1[i] = __ldg(a.w1 + (int64_t)ag * IN * H + i);
  for (int i = tid; i < H * NA; i += kPgThreads) s_w2[i] = __ldg(a.w2 + (int64_t)ag * H * NA + i);
  if (tid < H) s_b1[tid] = __ldg(a.b1 + ag * H + tid);
  if (tid < NA) s_b2[tid] = __ldg(a.b2 + ag * NA + tid);
  for (int s = tid; s < TE; s += kPgThreads) {
    for (int k = IN; k < C::XR; ++k) s_x[k * SS + s] = k == IN ? 1.f : 0.f;
    for (int k = H; k < C::RR; ++k) s_r[k * SS + s] = k == H ? 1.f : 0.f;
    for (int k = NA + 1; k < C::NAP; ++k) s_gl[k * SS + s] = 0.f;
  }

  // this thread's contraction item and sample slice
  const int slice = tid / C::NI, item = tid % C::NI;
  const bool fc1_item = item < C::I1;
  const int nrb = fc1_item ? C::NRB1 : C::NRB2, ncb = fc1_item ? C::NCB1 : C::NCB2;
  const int it = fc1_item ? item : item - C::I1;
  const int rb = it % nrb, cb = it / nrb;
  const float* lrow = (fc1_item ? s_x : s_r) + rb * SS;
  const float* rcol = (fc1_item ? s_gh : s_gl) + cb * SS;
  const int lstep = nrb * SS, rstep = ncb * SS;
  constexpr int SLICE = TE / C::SPL;
  const int s_begin = slice * SLICE;
  const bool contracts = slice < C::SPL;
  double acc64[RB][CB];
#pragma unroll
  for (int k = 0; k < RB; ++k)
#pragma unroll
    for (int j = 0; j < CB; ++j) acc64[k][j] = 0.0;

  const int64_t tile_lo = chunk * a.n_tiles / a.n_chunks, tile_hi = (chunk + 1) * a.n_tiles / a.n_chunks;
  for (int64_t tile = tile_lo; tile < tile_hi; ++tile) {
    const int64_t t = tile / a.n_etiles;
    const int64_t e = (tile - t * a.n_etiles) * TE + tid;
    const bool valid = e < a.n_envs;                     // padding columns up to ld are never read
    __syncthreads();                                     // the previous tile's contraction is done (and the staging)
    // 1. forward and backward of sample tid
    const float* xg = a.obs + t * IN * a.ld + e;
    for (int k = 0; k < IN; ++k) s_x[k * SS + tid] = valid ? __ldg(xg + (int64_t)k * a.ld) : 0.f;
    const int64_t ra = (t * A + ag) * a.ld + e;
    const int c = valid ? (int)__ldg(a.actions + ra) : 0;
    const float psi = valid ? __ldg(a.psi + ra) : 0.f;
    float2 h2[H / 2];
#pragma unroll
    for (int q = 0; q < H / 2; ++q) h2[q] = make_float2(s_b1[2 * q], s_b1[2 * q + 1]);
#pragma unroll 4
    for (int k = 0; k < IN; ++k) {
      const float xk = s_x[k * SS + tid];
      const float2 xx = make_float2(xk, xk);
      const float4* wr = reinterpret_cast<const float4*>(s_w1 + k * H);
#pragma unroll
      for (int v = 0; v < H / 4; ++v) {
        const float4 w = wr[v];
        h2[2 * v] = tc::ffma2(xx, make_float2(w.x, w.y), h2[2 * v]);
        h2[2 * v + 1] = tc::ffma2(xx, make_float2(w.z, w.w), h2[2 * v + 1]);
      }
    }
    float h[H];
#pragma unroll
    for (int q = 0; q < H / 2; ++q) {
      h[2 * q] = h2[q].x;
      h[2 * q + 1] = h2[q].y;
    }
    float l[NA];
#pragma unroll
    for (int j = 0; j < NA; ++j) l[j] = s_b2[j];
#pragma unroll
    for (int u = 0; u < H; ++u) {
      const float r = fmaxf(h[u], 0.f);
      s_r[u * SS + tid] = r;
#pragma unroll
      for (int j = 0; j < NA; ++j) l[j] = fmaf(r, s_w2[u * NA + j], l[j]);
    }
    float m = l[0];
#pragma unroll
    for (int j = 1; j < NA; ++j) m = fmaxf(m, l[j]);
    float ex[NA], sum = 0.f;
#pragma unroll
    for (int j = 0; j < NA; ++j) {
      ex[j] = expf(l[j] - m);
      sum += ex[j];
    }
    const float inv = 1.f / sum, log_sum = logf(sum);
    // the action selects by comparison, never as an index: a byte >= NA reads nothing out of bounds
    float l_pick = m, gl[NA];
#pragma unroll
    for (int j = 0; j < NA; ++j) {
      const bool hit = j == c;
      if (hit) l_pick = l[j];
      gl[j] = psi * ((hit ? 1.f : 0.f) - ex[j] * inv);
      s_gl[j * SS + tid] = gl[j];
    }
    s_gl[NA * SS + tid] = psi * ((l_pick - m) - log_sum);
#pragma unroll
    for (int u = 0; u < H; ++u) {
      float g = 0.f;
#pragma unroll
      for (int j = 0; j < NA; ++j) g = fmaf(s_w2[u * NA + j], gl[j], g);
      s_gh[u * SS + tid] = h[u] > 0.f ? g : 0.f;
    }
    __syncthreads();
    // 2. this thread's 4 x 4 block of the outer products over its slice of the tile
    if (contracts) {
      float2 acc[RB][CB];
#pragma unroll
      for (int k = 0; k < RB; ++k)
#pragma unroll
        for (int j = 0; j < CB; ++j) acc[k][j] = make_float2(0.f, 0.f);
#pragma unroll 2
      for (int s = s_begin; s < s_begin + SLICE; s += 4) {
        float4 lv[RB], rv[CB];
#pragma unroll
        for (int k = 0; k < RB; ++k) lv[k] = *reinterpret_cast<const float4*>(lrow + k * lstep + s);
#pragma unroll
        for (int j = 0; j < CB; ++j) rv[j] = *reinterpret_cast<const float4*>(rcol + j * rstep + s);
#pragma unroll
        for (int k = 0; k < RB; ++k)
#pragma unroll
          for (int j = 0; j < CB; ++j) {
            acc[k][j] = tc::ffma2(make_float2(lv[k].x, lv[k].y), make_float2(rv[j].x, rv[j].y), acc[k][j]);
            acc[k][j] = tc::ffma2(make_float2(lv[k].z, lv[k].w), make_float2(rv[j].z, rv[j].w), acc[k][j]);
          }
      }
#pragma unroll
      for (int k = 0; k < RB; ++k)
#pragma unroll
        for (int j = 0; j < CB; ++j) acc64[k][j] += (double)(acc[k][j].x + acc[k][j].y);
    }
  }

  // the chunk's partial: the slices' f64 blocks summed in slice order (the sample arrays are free from here on)
  __syncthreads();
  double* s_red = reinterpret_cast<double*>(s_x);      // [SPL][NI][RB * CB]
  if (contracts) {
#pragma unroll
    for (int k = 0; k < RB; ++k)
#pragma unroll
      for (int j = 0; j < CB; ++j) s_red[((size_t)slice * C::NI + item) * (RB * CB) + k * CB + j] = acc64[k][j];
  }
  __syncthreads();
  double* part = a.scratch + kPgHeader + ((int64_t)ag * a.n_chunks + chunk) * C::NOUT;
  for (int idx = tid; idx < C::NI * RB * CB; idx += kPgThreads) {
    const int i = idx / (RB * CB), k = (idx / CB) % RB, j = idx % CB;
    double v = 0.0;
    for (int sl = 0; sl < C::SPL; ++sl) v += s_red[((size_t)sl * C::NI + i) * (RB * CB) + k * CB + j];
    int o = -1;
    if (i < C::I1) {
      const int row = i % C::NRB1 + k * C::NRB1, col = i / C::NRB1 + j * C::NCB1;
      if (row <= IN) o = row * H + col;                                   // dw1 rows, then db1
    } else {
      const int i2 = i - C::I1;
      const int row = i2 % C::NRB2 + k * C::NRB2, col = i2 / C::NRB2 + j * C::NCB2;
      if (row < H && col < NA) o = IN * H + H + row * NA + col;           // dw2
      else if (row == H && col <= NA) o = IN * H + H + H * NA + col;      // db2, then the loss
    }
    if (o >= 0) part[o] = v;
  }

  // the last CTA of this agent sums the P partials in chunk order
  uint32_t* counters = reinterpret_cast<uint32_t*>(a.scratch);            // [0, A): agents, [32]: agents finished
  double* agent_loss = a.scratch + 32;
  __threadfence();
  __syncthreads();
  if (tid == 0) s_last = atomicAdd(counters + ag, 1u) == (uint32_t)a.n_chunks - 1u;
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  const double* parts = a.scratch + kPgHeader + (int64_t)ag * a.n_chunks * C::NOUT;
  for (int o = tid; o < C::NOUT; o += kPgThreads) {
    double v = 0.0;
    for (int p = 0; p < a.n_chunks; ++p) v += __ldcg(parts + (int64_t)p * C::NOUT + o);
    v *= -a.scale;
    if (o < IN * H) a.dw1[(int64_t)ag * IN * H + o] = (float)v;
    else if (o < IN * H + H) a.db1[ag * H + o - IN * H] = (float)v;
    else if (o < IN * H + H + H * NA) a.dw2[ag * H * NA + o - IN * H - H] = (float)v;
    else if (o < C::NOUT - 1) a.db2[ag * NA + o - IN * H - H - H * NA] = (float)v;
    else agent_loss[ag] = v;
  }
  if (!a.loss) return;
  __threadfence();
  __syncthreads();
  if (tid == 0 && atomicAdd(counters + 32, 1u) == (uint32_t)A - 1u) {
    __threadfence();
    double L = 0.0;
    for (int i = 0; i < A; ++i) L += __ldcg(agent_loss + i);
    *a.loss = L;
  }
}

template <int NA>
int launch_policy_grad(int n_agents, PolicyGradArgs& a, cudaStream_t st);
extern template int launch_policy_grad<kPolActions>(int, PolicyGradArgs&, cudaStream_t);   // unit 0
extern template int launch_policy_grad<9>(int, PolicyGradArgs&, cudaStream_t);             // unit 1

#if SMARL_TU_IS(0) || SMARL_TU_IS(1)
template <int NA>
int launch_policy_grad(int n_agents, PolicyGradArgs& a, cudaStream_t st) {
  return dispatch<1, 32>(n_agents, [&](auto kA) {
    using C = PgCfg<kA, NA>;
    auto kern = policy_grad_kernel<kA, NA>;
    const size_t smem = C::kSmemBytes;
    if (smem > 48 * 1024) SMARL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<(unsigned)((int64_t)kA * a.n_chunks), kPgThreads, smem, st>>>(a);
    SMARL_CUDA(cudaGetLastError());
    return SMARL_OK;
  });
}
#endif
#if SMARL_TU_IS(0)
template int launch_policy_grad<kPolActions>(int, PolicyGradArgs&, cudaStream_t);
#endif
#if SMARL_TU_IS(1)
template int launch_policy_grad<9>(int, PolicyGradArgs&, cudaStream_t);
#endif

}  // namespace smarl

using namespace smarl;

#if SMARL_TU_IS(0)
extern "C" int64_t smarl_policy_grad_scratch_len(int32_t n_agents, int32_t n_actions, int32_t n_steps, int64_t n_envs) {
  if (n_agents < 1 || n_agents > SMARL_MAX_AGENTS || (n_actions != 5 && n_actions != 9) || n_steps < 1 ||
      n_steps > 65536 || n_envs < 1)
    return -1;
  const int64_t nout = 2 * n_agents * kPolHidden + kPolHidden + kPolHidden * n_actions + n_actions + 1;
  return kPgHeader + (int64_t)n_agents * policy_grad_chunks(n_agents, n_steps, n_envs) * nout;
}

extern "C" int smarl_policy_grad_discrete(const SmarlDiscretePolicy* p, const float* obs_rec, const uint8_t* actions,
                                          const float* psi, int32_t n_steps, double scale, float* dw1, float* db1,
                                          float* dw2, float* db2, double* loss, double* scratch, int64_t n_envs,
                                          int64_t ld, smarl_stream_t stream) {
  SMARL_REQUIRE(p != nullptr, "policy params is NULL");
  SMARL_REQUIRE(p->n_agents >= 1 && p->n_agents <= SMARL_MAX_AGENTS, "n_agents=%d outside 1..32", p->n_agents);
  SMARL_REQUIRE(p->hidden == kPolHidden && (p->n_actions == 5 || p->n_actions == 9),
                "the DiscretePolicy gradient is built for hidden 16 and 5 or 9 actions (got %d, %d)", p->hidden,
                p->n_actions);
  SMARL_REQUIRE(p->w1 && p->b1 && p->w2 && p->b2 && obs_rec && actions && psi && dw1 && db1 && dw2 && db2 && scratch,
                "null pointer");
  SMARL_REQUIRE(n_steps >= 1 && n_steps <= 65536, "n_steps=%d outside 1..65536", n_steps);
  if (int rc = check_layout(n_envs, ld)) return rc;
  SMARL_REQUIRE(aligned16(obs_rec) && aligned16(actions) && aligned16(psi), "records must be 16-byte aligned");
  SMARL_REQUIRE(isfinite(scale), "scale is not finite");
  PolicyGradArgs a;
  a.obs = obs_rec; a.actions = actions; a.psi = psi; a.w1 = p->w1; a.b1 = p->b1; a.w2 = p->w2; a.b2 = p->b2;
  a.dw1 = dw1; a.db1 = db1; a.dw2 = dw2; a.db2 = db2; a.loss = loss; a.scratch = scratch; a.scale = scale;
  a.n_envs = n_envs; a.ld = ld;
  a.n_etiles = (n_envs + kPgTile - 1) / kPgTile;
  a.n_tiles = (int64_t)n_steps * a.n_etiles;
  a.n_chunks = (int32_t)policy_grad_chunks(p->n_agents, n_steps, n_envs);
  cudaStream_t st = (cudaStream_t)stream;
  SMARL_CUDA(cudaMemsetAsync(scratch, 0, 33 * sizeof(uint32_t), st));     // the completion counters
  return p->n_actions == 5 ? launch_policy_grad<5>(p->n_agents, a, st) : launch_policy_grad<9>(p->n_agents, a, st);
}
#endif
