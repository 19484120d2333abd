// Rollout accounting over a device rollout buffer + library plumbing (errors, device info).
//
// Replaces, for n_envs episodes at once: Buffer.step (safe_multi_agent_RL/buffer.py:30-39),
// MetaAgent.act's penalty and MetaAgent.step/update (meta_agent.py:18-39) and the learners'
// compute_returns (agent.py:129-132, :200-206).  All sums are carried in f64 like the
// reference; only the stored products are f32.
#include <stdarg.h>
#include <stdlib.h>

#include "mbarrier.cuh"
#include "stats.cuh"

namespace smarl {

static thread_local char g_error[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_error, sizeof(g_error), fmt, ap);
  va_end(ap);
}

static int g_variant[4] = {-1, -1, -1, -1};
int kernel_variant(int env_kind) { return (env_kind >= 0 && env_kind < 4) ? g_variant[env_kind] : -1; }

static int g_pdl = -1;                  // -1: not read yet (SMARL_PDL=0 in the environment turns it off)
bool pdl_enabled() {
  if (g_pdl < 0) {
    const char* e = getenv("SMARL_PDL");
    g_pdl = (e && e[0] == '0') ? 0 : 1;
  }
  return g_pdl != 0;
}

int check_layout(int64_t n_envs, int64_t ld) {
  SMARL_REQUIRE(n_envs >= 1, "n_envs=%lld must be >= 1", (long long)n_envs);
  SMARL_REQUIRE(ld >= n_envs && ld % 16 == 0, "ld=%lld must be a multiple of 16 and >= n_envs=%lld",
                (long long)ld, (long long)n_envs);
  return SMARL_OK;
}

constexpr int kAccThreads = 128;
constexpr int kReturnsThreads = 128;   // default CTA size of returns_kernel (>= 64: stats scratch rows are sized for 64)
constexpr int kReturnsStages = 6;      // returns_kernel's ring depth: up to kReturnsStages - 1 steps in flight per CTA

template <typename CT> struct CostVec;
template <> struct CostVec<float> {   // float costs are summed in f64 like the reference and stored as f32
  typedef double acc_t;
  static __device__ __forceinline__ void load(const float* p, double (&c)[4]) {
    const float4 f = ld_stream_f4(p);
    c[0] = f.x; c[1] = f.y; c[2] = f.z; c[3] = f.w;
  }
  static __device__ __forceinline__ void load_shared(const float* p, double (&c)[4]) {
    const float4 f = *reinterpret_cast<const float4*>(p);
    c[0] = f.x; c[1] = f.y; c[2] = f.z; c[3] = f.w;
  }
  static __device__ __forceinline__ int4 pack(const double (&s)[4]) {
    return make_int4(__float_as_int((float)s[0]), __float_as_int((float)s[1]), __float_as_int((float)s[2]),
                     __float_as_int((float)s[3]));
  }
};
template <> struct CostVec<uint8_t> {
  typedef int acc_t;
  static __device__ __forceinline__ int4 pack(const int (&s)[4]) { return make_int4(s[0], s[1], s[2], s[3]); }
  static __device__ __forceinline__ void load(const uint8_t* p, int (&c)[4]) {
    const uint32_t w = ld_stream_u32(p);
    c[0] = w & 0xFF; c[1] = (w >> 8) & 0xFF; c[2] = (w >> 16) & 0xFF; c[3] = w >> 24;
  }
  static __device__ __forceinline__ void load_shared(const uint8_t* p, int (&c)[4]) {
    const uint32_t w = *reinterpret_cast<const uint32_t*>(p);
    c[0] = w & 0xFF; c[1] = (w >> 8) & 0xFF; c[2] = (w >> 16) & 0xFF; c[3] = w >> 24;
  }
};
template <> struct CostVec<int32_t> {
  typedef int acc_t;
  static __device__ __forceinline__ int4 pack(const int (&s)[4]) { return make_int4(s[0], s[1], s[2], s[3]); }
  static __device__ __forceinline__ void load(const int32_t* p, int (&c)[4]) {
    const float4 f = ld_stream_f4(p);
    c[0] = __float_as_int(f.x); c[1] = __float_as_int(f.y); c[2] = __float_as_int(f.z); c[3] = __float_as_int(f.w);
  }
  static __device__ __forceinline__ void load_shared(const int32_t* p, int (&c)[4]) {
    const int4 v = *reinterpret_cast<const int4*>(p);
    c[0] = v.x; c[1] = v.y; c[2] = v.z; c[3] = v.w;
  }
};

// penalty[t][e] = sum_k lambda_k * cost[t][k][e]          (meta_agent.py:21-22)
template <typename CT>
__global__ void __launch_bounds__(kAccThreads)
penalty_kernel(const CT* __restrict__ cost, const double* __restrict__ lambdas, float* __restrict__ penalty,
               int K, int64_t n_groups, int64_t ld) {
  const int64_t g = (int64_t)blockIdx.x * kAccThreads + threadIdx.x;
  if (g >= n_groups) return;
  const int64_t e0 = g * 4;
  const int64_t t = blockIdx.y;
  double pen[4] = {0, 0, 0, 0};
  for (int k = 0; k < K; ++k) {
    typename CostVec<CT>::acc_t c[4];
    CostVec<CT>::load(cost + (t * K + k) * ld + e0, c);
    const double lam = __ldg(lambdas + k);
#pragma unroll
    for (int j = 0; j < 4; ++j) pen[j] += lam * (double)c[j];
  }
  st_stream_f4(penalty + t * ld + e0, make_float4((float)pen[0], (float)pen[1], (float)pen[2], (float)pen[3]));
}

struct ReturnsArgs {
  const float* reward;     // [T][A][ld]
  const void* cost;        // [T][K][ld]
  const float* penalty;    // [T][ld] or NULL
  const int32_t* n_active; // [ld] or NULL
  float* R;
  float* modR;
  int32_t* C;
  float* G;
  double* partials;        // [n_chunks][stats_len] or NULL
  const double* thresholds;
  double gamma;
  int64_t n_groups;
  int64_t n_envs;
  int64_t ld;
  int32_t A, K, T, g_mode;
  int32_t cost_rows_only;  // 1: only the K constraint rows (the shared-reward kernel handles the agents)
  const float* weights;    // shared-reward kernel: [A] or NULL
};

// Per-step input tiles of one returns_kernel CTA: an agent row's reward and penalty tiles, or kCostSteps consecutive
// time steps of a constraint row's cost tiles (so that a u8 row keeps as many bytes in flight as an agent row).
// Thread 0 fills the stages with cp.async.bulk; `full` counts the bytes landed, `empty` the THREADS threads that
// have read the stage.  Bytes in flight sit in shared memory, not in registers, so the depth of the
// ring does not cost occupancy.
template <typename CT, int THREADS, int S>
struct ReturnsRing {
  static constexpr int kCostSteps = 8 / (int)sizeof(CT);
  union Stage {
    struct {
      float4 reward[THREADS];
      float4 penalty[THREADS];
    } agent;
    CT cost[kCostSteps][4 * THREADS];
  };
  Stage stage[S];
  uint64_t full[S], empty[S];
};

// One CTA = one row (agent a, or constraint k) x 512 envs.  Rows of the same env chunk get
// consecutive block ids so that they run together and share the chunk's penalty rows in L2.
// GM = 1 serves g_mode 0 and 1 (backward Horner, G written iff g_mode == 1), 2 and 3 their own paths;
// a template parameter so that the PPO path's extra registers do not cut the occupancy of the others.
// The CTA walks a sequence of steps i (an agent row's time steps in the order the path visits them, GM 3 visits
// them twice; a constraint row's groups of kCostSteps time steps) and reads step i's tiles from ring stage i % S.
// The minimum of 4 CTAs per SM is what lets ptxas give the GM 3 instance the registers it needs without spilling
// (it spills at the 80 it picks unasked).
template <typename CT, int THREADS, int GM>
__global__ void __launch_bounds__(THREADS, 4) returns_kernel(const ReturnsArgs a) {
  constexpr int S = kReturnsStages;
  __shared__ double s_red[THREADS / 32];
  __shared__ alignas(128) ReturnsRing<CT, THREADS, S> ring;
  constexpr int CS = ReturnsRing<CT, THREADS, S>::kCostSteps;
  const int rows = (a.cost_rows_only ? 0 : a.A) + a.K;
  const int row = (int)(blockIdx.x % rows) + (a.cost_rows_only ? a.A : 0);
  const int64_t chunk = blockIdx.x / rows;
  const int64_t g = chunk * THREADS + threadIdx.x;
  const bool live = g < a.n_groups;
  const int64_t e0 = (live ? g : 0) * 4;
  const int64_t ld = a.ld;
  const int T = a.T;
  bool valid[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) valid[k] = live && (e0 + k < a.n_envs);
  double* out = a.partials ? a.partials + chunk * stats_len(a.A, a.K) : nullptr;

  const bool agent = row < a.A;
  const int n_steps = agent ? (GM == 3 ? 2 * T : T) : (T + CS - 1) / CS;
  // The chunk's envs rounded up to 16 (a multiple of 16 bytes for every element type) and never past ld.
  const int64_t c0 = chunk * 4 * THREADS;
  const uint32_t tile_envs = (uint32_t)min((int64_t)4 * THREADS, (a.n_envs - c0 + 15) & ~(int64_t)15);
  auto issue = [&](int i) {
    const int slot = i % S;
    const uint64_t read_once = l2_evict_first_policy();
    if (agent) {
      const int t = GM == 2 ? i : T - 1 - (i < T ? i : i - T);
      const uint32_t bytes = tile_envs * 4;
      mbar_arrive_expect_tx(&ring.full[slot], a.penalty ? 2 * bytes : bytes);
      bulk_load(ring.stage[slot].agent.reward, a.reward + ((int64_t)t * a.A + row) * ld + c0, bytes, &ring.full[slot],
                read_once);
      // the penalty row is shared by the chunk's A agent CTAs: left to L2's default policy
      if (a.penalty)
        bulk_load(ring.stage[slot].agent.penalty, a.penalty + (int64_t)t * ld + c0, bytes, &ring.full[slot],
                  l2_evict_normal_policy());
    } else {
      const uint32_t bytes = tile_envs * (uint32_t)sizeof(CT);
      const int t0 = i * CS, nt = min(CS, T - t0);
      mbar_arrive_expect_tx(&ring.full[slot], nt * bytes);
      for (int j = 0; j < nt; ++j)
        bulk_load(ring.stage[slot].cost[j], static_cast<const CT*>(a.cost) + ((int64_t)(t0 + j) * a.K + (row - a.A)) * ld + c0,
                  bytes, &ring.full[slot], read_once);
    }
  };
  if (threadIdx.x == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(&ring.full[s], 1);
      mbar_init(&ring.empty[s], THREADS);
    }
    for (int i = 0; i < min(S, n_steps); ++i) issue(i);
  }
  __syncthreads();
  auto wait_full = [&](int i) { mbar_wait(&ring.full[i % S], (uint32_t)(i / S) & 1u); };
  // Done reading step i.  Thread 0 then refills the stage of step i - 1 (which the other threads have most
  // likely left by now) with step i - 1 + S.
  auto release = [&](int i) {
    mbar_arrive(&ring.empty[i % S]);
    if (threadIdx.x == 0 && i >= 1 && i - 1 + S < n_steps) {
      mbar_wait(&ring.empty[(i - 1) % S], (uint32_t)((i - 1) / S) & 1u);
      issue(i - 1 + S);
    }
  };
  auto load_agent = [&](int i, float4& r, float4& p) {
    wait_full(i);
    r = ring.stage[i % S].agent.reward[threadIdx.x];
    p = make_float4(0.f, 0.f, 0.f, 0.f);
    if (a.penalty) p = ring.stage[i % S].agent.penalty[threadIdx.x];
    release(i);
  };

  if (agent) {
    double raw[4] = {0, 0, 0, 0}, mod[4] = {0, 0, 0, 0};
    const double gamma = a.gamma;
    if (GM == 3) {
      // PPO (agent.py:276-281; PPOAgent extends ACAgent, so compute_returns is the reward-to-go of
      // :200-206): x_t = G_t over the episode's T' steps, then (x - mean) / (std_unbiased + 1e-7).
      // Sweep 1 (backward Horner): G_t, their sum and sum of squares (G_0 = modR); sweep 2: write.
      int n_act[4] = {T, T, T, T};
      if (a.n_active) {
        int c[4];
        CostVec<int32_t>::load(a.n_active + e0, c);
#pragma unroll
        for (int k = 0; k < 4; ++k) n_act[k] = min(max(c[k], 0), T);
      }
      double sum[4] = {0, 0, 0, 0}, sq[4] = {0, 0, 0, 0};
      for (int t = T - 1; t >= 0; --t) {
        float4 r, p;
        load_agent(T - 1 - t, r, p);
        const float rr[4] = {r.x, r.y, r.z, r.w}, pp[4] = {p.x, p.y, p.z, p.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          raw[k] = (double)rr[k] + gamma * raw[k];
          mod[k] = ((double)rr[k] - (double)pp[k]) + gamma * mod[k];
          if (t < n_act[k]) {
            sum[k] += mod[k];
            sq[k] += mod[k] * mod[k];
          }
        }
      }
      double mean[4], inv[4], run[4] = {0, 0, 0, 0};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const double n = (double)n_act[k];
        mean[k] = sum[k] / n;
        const double var = (sq[k] - n * mean[k] * mean[k]) / (n - 1.0);
        inv[k] = 1.0 / (sqrt(fmax(var, 0.0)) + 1e-7);
        if (n_act[k] < 2) inv[k] = __longlong_as_double(0x7ff8000000000000ll);   // torch: std of one sample is nan
      }
      for (int t = T - 1; t >= 0; --t) {
        float4 r, p;
        load_agent(2 * T - 1 - t, r, p);
        const float rr[4] = {r.x, r.y, r.z, r.w}, pp[4] = {p.x, p.y, p.z, p.w};
        float o[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          run[k] = ((double)rr[k] - (double)pp[k]) + gamma * run[k];
          o[k] = t < n_act[k] ? (float)((run[k] - mean[k]) * inv[k]) : 0.f;
        }
        if (live) st_stream_f4(a.G + ((int64_t)t * a.A + row) * ld + e0, make_float4(o[0], o[1], o[2], o[3]));
      }
    } else if (GM != 2) {
      // Backward Horner: G_t = m_t + gamma G_{t+1} (agent.py:200-206); G_0 is the discounted
      // episode return of buffer.py:31-35.
      for (int t = T - 1; t >= 0; --t) {
        float4 r, p;
        load_agent(T - 1 - t, r, p);
        const float rr[4] = {r.x, r.y, r.z, r.w}, pp[4] = {p.x, p.y, p.z, p.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          raw[k] = (double)rr[k] + gamma * raw[k];
          mod[k] = ((double)rr[k] - (double)pp[k]) + gamma * mod[k];
        }
        if (a.g_mode == 1 && live)
          st_stream_f4(a.G + ((int64_t)t * a.A + row) * ld + e0,
                       make_float4((float)mod[0], (float)mod[1], (float)mod[2], (float)mod[3]));
      }
    } else {
      // Forward: gamma^t * m_t per step (agent.py:129-132) and their running sums.
      double disc = 1.0;
      for (int t = 0; t < T; ++t) {
        float4 r, p;
        load_agent(t, r, p);
        const float rr[4] = {r.x, r.y, r.z, r.w}, pp[4] = {p.x, p.y, p.z, p.w};
        double term[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          raw[k] += disc * (double)rr[k];
          term[k] = disc * ((double)rr[k] - (double)pp[k]);
          mod[k] += term[k];
        }
        if (live)
          st_stream_f4(a.G + ((int64_t)t * a.A + row) * ld + e0,
                       make_float4((float)term[0], (float)term[1], (float)term[2], (float)term[3]));
        disc *= gamma;
      }
    }
    if (live) {
      st_stream_f4(a.R + (int64_t)row * ld + e0, make_float4((float)raw[0], (float)raw[1], (float)raw[2], (float)raw[3]));
      st_stream_f4(a.modR + (int64_t)row * ld + e0, make_float4((float)mod[0], (float)mod[1], (float)mod[2], (float)mod[3]));
    }
    if (out) {
      double v_raw = 0.0, v_mod = 0.0;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        v_raw += valid[k] ? raw[k] : 0.0;
        v_mod += valid[k] ? mod[k] : 0.0;
      }
      const double b_raw = block_sum<THREADS>(v_raw, s_red);
      const double b_mod = block_sum<THREADS>(v_mod, s_red);
      if (threadIdx.x == 0) {
        out[2 * a.K + row] = b_raw;
        out[2 * a.K + a.A + row] = b_mod;
        if (row == 0) out[2 * a.K + 2 * a.A] = 0.0;
      }
    }
  } else {
    // C_k = sum_t c[t,k]  (buffer.py:39, meta_agent.py:28)
    const int k = row - a.A;
    typename CostVec<CT>::acc_t sum[4] = {0, 0, 0, 0};
    for (int i = 0; i < n_steps; ++i) {
      wait_full(i);
      const int nt = min(CS, T - i * CS);
      for (int s = 0; s < nt; ++s) {
        typename CostVec<CT>::acc_t c[4];
        CostVec<CT>::load_shared(ring.stage[i % S].cost[s] + 4 * threadIdx.x, c);
#pragma unroll
        for (int j = 0; j < 4; ++j) sum[j] += c[j];
      }
      release(i);
    }
    if (live) st_stream_i4(a.C + (int64_t)k * ld + e0, CostVec<CT>::pack(sum));
    if (out) {
      const double thr = a.thresholds ? __ldg(a.thresholds + k) : 0.0;
      double c = 0.0, viol = 0.0;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        c += valid[j] ? (double)sum[j] : 0.0;
        viol += (valid[j] && a.thresholds && (double)sum[j] > thr) ? 1.0 : 0.0;
      }
      const double bc = block_sum<THREADS>(c, s_red);
      const double bv = block_sum<THREADS>(viol, s_red);
      if (threadIdx.x == 0) {
        out[k] = bc;
        out[a.K + k] = bv;
      }
    }
  }
}

// Shared-reward accounting: one reward row per env and step, reward_a[t] = w_a * rew[t].  One CTA per
// 512-env chunk runs ONE backward Horner pair (G_rew, G_pen) per env and emits all A agents' rows:
//   G[t][a] = w_a * G_rew[t] - G_pen[t],  R_a = w_a * G_rew[0],  modR_a = w_a * G_rew[0] - G_pen[0].
template <int GM>
__global__ void __launch_bounds__(kAccThreads) returns_shared_kernel(const ReturnsArgs a) {
  __shared__ double s_red[kAccThreads / 32];
  __shared__ float s_w[SMARL_MAX_AGENTS];
  if (threadIdx.x < SMARL_MAX_AGENTS) s_w[threadIdx.x] = (a.weights && threadIdx.x < a.A) ? a.weights[threadIdx.x] : 1.0f;
  __syncthreads();
  const int64_t chunk = blockIdx.x;
  const int64_t g = chunk * kAccThreads + threadIdx.x;
  const bool live = g < a.n_groups;
  const int64_t e0 = (live ? g : 0) * 4;
  const int64_t ld = a.ld;
  const int T = a.T, A = a.A;
  const double gamma = a.gamma;
  double g_rew[4] = {0, 0, 0, 0}, g_pen[4] = {0, 0, 0, 0};
  if (GM == 3) {
    // PPO standardisation (agent.py:276-281) of x_t = w G_rew[t] - G_pen[t] per agent and env.  Its mean and
    // unbiased variance over t follow from five sums of the one Horner pair:
    //   sum x = w S_r - S_p,   sum x^2 = w^2 S_rr - 2 w S_rp + S_pp.
    double s_r[4] = {0, 0, 0, 0}, s_p[4] = {0, 0, 0, 0}, s_rr[4] = {0, 0, 0, 0}, s_rp[4] = {0, 0, 0, 0},
           s_pp[4] = {0, 0, 0, 0};
    // episodes that ended early (Collision, main.py:51) standardise over their own T' steps; later steps get 0
    int n_act[4] = {T, T, T, T};
    if (a.n_active) {
      int c[4];
      CostVec<int32_t>::load(a.n_active + e0, c);
#pragma unroll
      for (int k = 0; k < 4; ++k) n_act[k] = min(max(c[k], 0), T);
    }
    for (int t = T - 1; t >= 0; --t) {
      const float4 r = ld_stream_f4(a.reward + (int64_t)t * ld + e0);
      float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
      if (a.penalty) p = ld_stream_f4(a.penalty + (int64_t)t * ld + e0);
      const float rr[4] = {r.x, r.y, r.z, r.w}, pp[4] = {p.x, p.y, p.z, p.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        g_rew[k] = (double)rr[k] + gamma * g_rew[k];
        g_pen[k] = (double)pp[k] + gamma * g_pen[k];
        if (t < n_act[k]) {
          s_r[k] += g_rew[k];
          s_p[k] += g_pen[k];
          s_rr[k] += g_rew[k] * g_rew[k];
          s_rp[k] += g_rew[k] * g_pen[k];
          s_pp[k] += g_pen[k] * g_pen[k];
        }
      }
    }
    double h_rew[4] = {0, 0, 0, 0}, h_pen[4] = {0, 0, 0, 0};
    for (int t = T - 1; t >= 0; --t) {
      const float4 r = ld_stream_f4(a.reward + (int64_t)t * ld + e0);
      float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
      if (a.penalty) p = ld_stream_f4(a.penalty + (int64_t)t * ld + e0);
      const float rr[4] = {r.x, r.y, r.z, r.w}, pp[4] = {p.x, p.y, p.z, p.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        h_rew[k] = (double)rr[k] + gamma * h_rew[k];
        h_pen[k] = (double)pp[k] + gamma * h_pen[k];
      }
      if (live) {
        for (int i = 0; i < A; ++i) {
          const double w = (double)s_w[i];
          float o[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const double n = (double)n_act[k];
            const double mean = (w * s_r[k] - s_p[k]) / n;
            const double sq = w * w * s_rr[k] - 2.0 * w * s_rp[k] + s_pp[k];
            const double var = (sq - n * mean * mean) / (n - 1.0);
            double inv = 1.0 / (sqrt(fmax(var, 0.0)) + 1e-7);
            if (n_act[k] < 2) inv = __longlong_as_double(0x7ff8000000000000ll);   // torch: std of one sample is nan
            o[k] = t < n_act[k] ? (float)(((w * h_rew[k] - h_pen[k]) - mean) * inv) : 0.f;
          }
          st_stream_f4(a.G + ((int64_t)t * A + i) * ld + e0, make_float4(o[0], o[1], o[2], o[3]));
        }
      }
    }
  } else if (GM != 2) {
#pragma unroll 2
    for (int t = T - 1; t >= 0; --t) {
      const float4 r = ld_stream_f4(a.reward + (int64_t)t * ld + e0);
      float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
      if (a.penalty) p = ld_stream_f4(a.penalty + (int64_t)t * ld + e0);
      const float rr[4] = {r.x, r.y, r.z, r.w}, pp[4] = {p.x, p.y, p.z, p.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        g_rew[k] = (double)rr[k] + gamma * g_rew[k];
        g_pen[k] = (double)pp[k] + gamma * g_pen[k];
      }
      if (a.g_mode == 1 && live) {
        for (int i = 0; i < A; ++i) {
          const double w = (double)s_w[i];
          st_stream_f4(a.G + ((int64_t)t * A + i) * ld + e0,
                       make_float4((float)(w * g_rew[0] - g_pen[0]), (float)(w * g_rew[1] - g_pen[1]),
                                   (float)(w * g_rew[2] - g_pen[2]), (float)(w * g_rew[3] - g_pen[3])));
        }
      }
    }
  } else {
    double disc = 1.0;
    for (int t = 0; t < T; ++t) {
      const float4 r = ld_stream_f4(a.reward + (int64_t)t * ld + e0);
      float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
      if (a.penalty) p = ld_stream_f4(a.penalty + (int64_t)t * ld + e0);
      const float rr[4] = {r.x, r.y, r.z, r.w}, pp[4] = {p.x, p.y, p.z, p.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        g_rew[k] += disc * (double)rr[k];
        g_pen[k] += disc * (double)pp[k];
      }
      if (live) {
        for (int i = 0; i < A; ++i) {
          const double w = (double)s_w[i];
          st_stream_f4(a.G + ((int64_t)t * A + i) * ld + e0,
                       make_float4((float)(disc * (w * rr[0] - pp[0])), (float)(disc * (w * rr[1] - pp[1])),
                                   (float)(disc * (w * rr[2] - pp[2])), (float)(disc * (w * rr[3] - pp[3]))));
        }
      }
      disc *= gamma;
    }
  }
  if (live) {
    for (int i = 0; i < A; ++i) {
      const double w = (double)s_w[i];
      st_stream_f4(a.R + (int64_t)i * ld + e0, make_float4((float)(w * g_rew[0]), (float)(w * g_rew[1]),
                                                           (float)(w * g_rew[2]), (float)(w * g_rew[3])));
      st_stream_f4(a.modR + (int64_t)i * ld + e0,
                   make_float4((float)(w * g_rew[0] - g_pen[0]), (float)(w * g_rew[1] - g_pen[1]),
                               (float)(w * g_rew[2] - g_pen[2]), (float)(w * g_rew[3] - g_pen[3])));
    }
  }
  if (a.partials) {
    double* out = a.partials + chunk * stats_len(a.A, a.K);
    double v_rew = 0.0, v_pen = 0.0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const bool valid = live && (e0 + k < a.n_envs);
      v_rew += valid ? g_rew[k] : 0.0;
      v_pen += valid ? g_pen[k] : 0.0;
    }
    const double b_rew = block_sum<kAccThreads>(v_rew, s_red);
    const double b_pen = block_sum<kAccThreads>(v_pen, s_red);
    if (threadIdx.x == 0) {
      for (int i = 0; i < A; ++i) {
        out[2 * a.K + i] = (double)s_w[i] * b_rew;
        out[2 * a.K + A + i] = (double)s_w[i] * b_rew - b_pen;
      }
      out[2 * a.K + 2 * A] = 0.0;
    }
  }
}

// stats[j] = sum over rows of partials[row][j], fixed order; the count slot is n_envs.
__global__ void __launch_bounds__(256)
stats_finalize_kernel(const double* __restrict__ partials, int64_t n_rows, int n_stats, double count,
                      double* __restrict__ stats) {
  __shared__ double s_red[256 / 32];
  const int j = blockIdx.x;
  if (j == n_stats - 1) {
    if (threadIdx.x == 0) stats[j] = count;
    return;
  }
  double v = 0.0;
  for (int64_t r = threadIdx.x; r < n_rows; r += 256) v += partials[r * n_stats + j];
  const double b = block_sum<256>(v, s_red);
  if (threadIdx.x == 0) stats[j] = b;
}

int launch_stats_finalize(const double* partials, int64_t n_rows, int n_agents, int n_constraints,
                          int64_t n_envs, double* stats, cudaStream_t stream) {
  const int n = stats_len(n_agents, n_constraints);
  stats_finalize_kernel<<<n, 256, 0, stream>>>(partials, n_rows, n, (double)n_envs, stats);
  SMARL_CUDA(cudaGetLastError());
  return SMARL_OK;
}

// lambda_k <- max(0, lambda_k + lr * (mean C_k - thr_k))      (meta_agent.py:32-36)
__global__ void lambda_update_kernel(double* lambdas, const double* __restrict__ stats,
                                     const double* __restrict__ thresholds, double lr, int A, int K) {
  const int k = threadIdx.x;
  if (k >= K) return;
  const double count = stats[2 * K + 2 * A];
  const double mean = stats[k] / count;
  lambdas[k] = fmax(lambdas[k] + lr * (mean - thresholds[k]), 0.0);
}

}  // namespace smarl

using namespace smarl;

extern "C" int smarl_abi_version(void) { return SMARL_ABI_VERSION; }
extern "C" const char* smarl_last_error(void) { return g_error; }

extern "C" int smarl_set_kernel_variant(int32_t env_kind, int32_t lanes) {
  if (env_kind < 0 || env_kind >= 4) return -1;
  const int prev = g_variant[env_kind];
  if (env_kind == SMARL_KERNEL_POLICY) g_variant[env_kind] = (lanes >= 0 && lanes <= 2) ? lanes : -1;
  else g_variant[env_kind] = (lanes == 0 || lanes == 2 || lanes == 4) ? lanes : -1;
  return prev;
}

extern "C" int smarl_set_pdl(int32_t on) {
  const int prev = pdl_enabled() ? 1 : 0;
  g_pdl = on ? 1 : 0;
  return prev;
}

extern "C" int smarl_device_info(int* sm, int* major, int* minor) {
  int dev = 0;
  SMARL_CUDA(cudaGetDevice(&dev));
  if (sm) SMARL_CUDA(cudaDeviceGetAttribute(sm, cudaDevAttrMultiProcessorCount, dev));
  if (major) SMARL_CUDA(cudaDeviceGetAttribute(major, cudaDevAttrComputeCapabilityMajor, dev));
  if (minor) SMARL_CUDA(cudaDeviceGetAttribute(minor, cudaDevAttrComputeCapabilityMinor, dev));
  return SMARL_OK;
}

extern "C" int32_t smarl_stats_len(int32_t n_agents, int32_t n_constraints) {
  return stats_len(n_agents, n_constraints);
}

extern "C" int64_t smarl_stats_scratch_len(int32_t n_agents, int32_t n_constraints, int64_t n_envs) {
  // one row of block partials per CTA; the smallest CTA any producer uses covers 32 envs (cooperative kernels, 4 lanes per env)
  const int64_t n_chunks = (n_envs + 31) / 32;
  return n_chunks * stats_len(n_agents, n_constraints);
}

extern "C" int smarl_rollout_penalty(const void* cost, int32_t cost_dtype, const double* lambdas,
                                     float* penalty, int32_t K, int32_t T, int64_t n_envs, int64_t ld,
                                     smarl_stream_t stream) {
  if (int rc = check_layout(n_envs, ld)) return rc;
  SMARL_REQUIRE(cost && lambdas && penalty, "null pointer");
  SMARL_REQUIRE(K >= 1 && K <= SMARL_MAX_AGENTS && T >= 1 && T <= 65535, "bad K=%d or T=%d", K, T);
  SMARL_REQUIRE(aligned16(cost) && aligned16(penalty), "pointers must be 16-byte aligned");
  const int64_t n_groups = (n_envs + 3) / 4;
  dim3 grid((unsigned)((n_groups + kAccThreads - 1) / kAccThreads), (unsigned)T);
  if (cost_dtype == SMARL_COST_U8)
    penalty_kernel<uint8_t><<<grid, kAccThreads, 0, (cudaStream_t)stream>>>(
        static_cast<const uint8_t*>(cost), lambdas, penalty, K, n_groups, ld);
  else if (cost_dtype == SMARL_COST_I32)
    penalty_kernel<int32_t><<<grid, kAccThreads, 0, (cudaStream_t)stream>>>(
        static_cast<const int32_t*>(cost), lambdas, penalty, K, n_groups, ld);
  else if (cost_dtype == SMARL_COST_F32)
    penalty_kernel<float><<<grid, kAccThreads, 0, (cudaStream_t)stream>>>(
        static_cast<const float*>(cost), lambdas, penalty, K, n_groups, ld);
  else
    SMARL_REQUIRE(false, "bad cost_dtype %d", cost_dtype);
  SMARL_CUDA(cudaGetLastError());
  return SMARL_OK;
}

extern "C" int smarl_rollout_returns(const SmarlAccounting* acc, const float* reward, const void* cost,
                                     int32_t cost_dtype, const float* penalty, const int32_t* n_active,
                                     float* R, float* modR, int32_t* C, float* G, double* stats,
                                     double* stats_scratch,
                                     int32_t n_agents, int32_t n_constraints, int64_t n_envs,
                                     int64_t ld, smarl_stream_t stream) {
  if (int rc = check_layout(n_envs, ld)) return rc;
  SMARL_REQUIRE(acc != nullptr, "accounting params is NULL");
  SMARL_REQUIRE(acc->n_steps >= 1, "n_steps=%d must be >= 1", acc->n_steps);
  SMARL_REQUIRE(acc->g_mode >= 0 && acc->g_mode <= 3, "bad g_mode %d", acc->g_mode);
  SMARL_REQUIRE(n_agents >= 1 && n_agents <= SMARL_MAX_AGENTS, "n_agents=%d outside 1..32", n_agents);
  SMARL_REQUIRE(n_constraints >= 1 && n_constraints <= SMARL_MAX_AGENTS, "n_constraints=%d outside 1..32",
                n_constraints);
  SMARL_REQUIRE(reward && cost && R && modR && C, "null required pointer");
  SMARL_REQUIRE(acc->g_mode == 0 || G, "g_mode != 0 needs G");
  SMARL_REQUIRE((stats == nullptr) == (stats_scratch == nullptr), "stats and stats_scratch go together");
  SMARL_REQUIRE(aligned16(reward) && aligned16(cost) && aligned16(penalty) && aligned16(R) &&
                    aligned16(modR) && aligned16(C) && aligned16(G), "pointers must be 16-byte aligned");
  ReturnsArgs a;
  a.reward = reward; a.cost = cost; a.penalty = penalty; a.n_active = n_active; a.R = R; a.modR = modR; a.C = C; a.G = G;
  a.partials = stats_scratch; a.thresholds = acc->thresholds; a.gamma = acc->gamma;
  a.n_groups = (n_envs + 3) / 4; a.n_envs = n_envs; a.ld = ld;
  a.A = n_agents; a.K = n_constraints; a.T = acc->n_steps; a.g_mode = acc->g_mode;
  a.cost_rows_only = 0; a.weights = nullptr;
  constexpr int threads = kReturnsThreads;
  const int64_t n_chunks = (a.n_groups + threads - 1) / threads;
  const int64_t blocks = n_chunks * (n_agents + n_constraints);
  SMARL_REQUIRE(blocks <= 0x7fffffffLL, "too many blocks");
  cudaStream_t st = (cudaStream_t)stream;
#define SMARL_LAUNCH_RETURNS(CT_)                                                                     \
  switch (acc->g_mode) {                                                                              \
    case 2: returns_kernel<CT_, threads, 2><<<(unsigned)blocks, threads, 0, st>>>(a); break;          \
    case 3: returns_kernel<CT_, threads, 3><<<(unsigned)blocks, threads, 0, st>>>(a); break;          \
    default: returns_kernel<CT_, threads, 1><<<(unsigned)blocks, threads, 0, st>>>(a); break;         \
  }
  if (cost_dtype == SMARL_COST_U8) {
    SMARL_LAUNCH_RETURNS(uint8_t)
  } else if (cost_dtype == SMARL_COST_I32) {
    SMARL_LAUNCH_RETURNS(int32_t)
  } else if (cost_dtype == SMARL_COST_F32) {
    SMARL_LAUNCH_RETURNS(float)
  } else {
    SMARL_REQUIRE(false, "bad cost_dtype %d", cost_dtype);
  }
#undef SMARL_LAUNCH_RETURNS
  SMARL_CUDA(cudaGetLastError());
  if (stats)
    return launch_stats_finalize(stats_scratch, n_chunks, n_agents, n_constraints, n_envs, stats,
                                 (cudaStream_t)stream);
  return SMARL_OK;
}

extern "C" int smarl_rollout_returns_shared(const SmarlAccounting* acc, const float* reward_env,
                                            const float* weights, const void* cost, int32_t cost_dtype,
                                            const float* penalty, const int32_t* n_active, float* R, float* modR,
                                            int32_t* C, float* G,
                                            double* stats, double* stats_scratch, int32_t n_agents,
                                            int32_t n_constraints, int64_t n_envs, int64_t ld,
                                            smarl_stream_t stream) {
  if (int rc = check_layout(n_envs, ld)) return rc;
  SMARL_REQUIRE(acc != nullptr, "accounting params is NULL");
  SMARL_REQUIRE(acc->n_steps >= 1, "n_steps=%d must be >= 1", acc->n_steps);
  SMARL_REQUIRE(acc->g_mode >= 0 && acc->g_mode <= 3, "bad g_mode %d", acc->g_mode);
  SMARL_REQUIRE(n_agents >= 1 && n_agents <= SMARL_MAX_AGENTS, "n_agents=%d outside 1..32", n_agents);
  SMARL_REQUIRE(n_constraints >= 1 && n_constraints <= SMARL_MAX_AGENTS, "n_constraints=%d outside 1..32",
                n_constraints);
  SMARL_REQUIRE(reward_env && cost && R && modR && C, "null required pointer");
  SMARL_REQUIRE(acc->g_mode == 0 || G, "g_mode != 0 needs G");
  SMARL_REQUIRE((stats == nullptr) == (stats_scratch == nullptr), "stats and stats_scratch go together");
  SMARL_REQUIRE(aligned16(reward_env) && aligned16(cost) && aligned16(penalty) && aligned16(R) && aligned16(modR) &&
                    aligned16(C) && aligned16(G), "pointers must be 16-byte aligned");
  ReturnsArgs a;
  a.reward = reward_env; a.cost = cost; a.penalty = penalty; a.n_active = n_active; a.R = R; a.modR = modR; a.C = C;
  a.G = G; a.partials = stats_scratch; a.thresholds = acc->thresholds; a.gamma = acc->gamma;
  a.n_groups = (n_envs + 3) / 4; a.n_envs = n_envs; a.ld = ld;
  a.A = n_agents; a.K = n_constraints; a.T = acc->n_steps; a.g_mode = acc->g_mode;
  a.cost_rows_only = 1; a.weights = weights;
  const int64_t n_chunks = (a.n_groups + kAccThreads - 1) / kAccThreads;
  cudaStream_t st = (cudaStream_t)stream;
  if (acc->g_mode == 2)
    returns_shared_kernel<2><<<(unsigned)n_chunks, kAccThreads, 0, st>>>(a);
  else if (acc->g_mode == 3)
    returns_shared_kernel<3><<<(unsigned)n_chunks, kAccThreads, 0, st>>>(a);
  else
    returns_shared_kernel<1><<<(unsigned)n_chunks, kAccThreads, 0, st>>>(a);
  const int64_t blocks = n_chunks * n_constraints;      // the K constraint rows: C_k, violation counts
  if (cost_dtype == SMARL_COST_U8)
    returns_kernel<uint8_t, kReturnsThreads, 1><<<(unsigned)blocks, kReturnsThreads, 0, st>>>(a);
  else if (cost_dtype == SMARL_COST_I32)
    returns_kernel<int32_t, kReturnsThreads, 1><<<(unsigned)blocks, kReturnsThreads, 0, st>>>(a);
  else if (cost_dtype == SMARL_COST_F32)
    returns_kernel<float, kReturnsThreads, 1><<<(unsigned)blocks, kReturnsThreads, 0, st>>>(a);
  else
    SMARL_REQUIRE(false, "bad cost_dtype %d", cost_dtype);
  SMARL_CUDA(cudaGetLastError());
  if (stats)
    return launch_stats_finalize(stats_scratch, n_chunks, n_agents, n_constraints, n_envs, stats, st);
  return SMARL_OK;
}

extern "C" int smarl_lambda_update(double* lambdas, const double* stats, const double* thresholds,
                                   double lr, int32_t n_agents, int32_t n_constraints,
                                   smarl_stream_t stream) {
  SMARL_REQUIRE(lambdas && stats && thresholds, "null pointer");
  SMARL_REQUIRE(n_constraints >= 1 && n_constraints <= SMARL_MAX_AGENTS, "n_constraints=%d outside 1..32",
                n_constraints);
  lambda_update_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(lambdas, stats, thresholds, lr, n_agents,
                                                          n_constraints);
  SMARL_CUDA(cudaGetLastError());
  return SMARL_OK;
}
