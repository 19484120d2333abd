// Host-buffer entry points: what a caller holding numpy arrays binds (INTEGRATION.md).
// The env dimension is cut into chunks that are pipelined over two streams so that the
// host->device copy of chunk c+1, the fused rollout of chunk c and the device->host copy of
// chunk c-1 overlap (PCIe is full duplex; the kernel is far shorter than either copy).
#include <stdlib.h>
#include <string.h>
#include <sys/syscall.h>
#include <unistd.h>

#include <new>

#include "coverage.cuh"
#include "stats.cuh"

struct SmarlHostSession {
  int32_t kind, A, K, T, L;
  int64_t n_envs, ld;
  int n_chunks;
  int64_t chunk;            // envs per chunk (multiple of 16)
  cudaStream_t streams[2];
  void* d_start_x;          // u8 (grid envs) or f64 (Collision) [A][ld]
  void* d_start_y;
  void* d_actions;          // u8 [T][A][ld] or f32 [T][2A][ld]
  uint8_t* d_packed;        // Coverage 4-bit packed actions [T][A][ld/2], allocated on first use
  uint8_t* d_packed5;       // Coverage base-5 packed actions [T][A][pitch5], allocated on first use
  int64_t pitch5;           // bytes per base-5 packed row
  uint8_t* d_moves;         // Congestion recorded moves, allocated on first use
  double* d_landmarks;      // Collision f64 [2L][ld]
  float* d_R;
  float* d_modR;
  int32_t* d_C;
  int32_t* d_n_active;
  double* d_stats;          // [n_chunks][stats_len]
  double* d_scratch;        // [n_chunks][scratch_len(chunk)]
  int64_t scratch_per_chunk;
  float* d_lut;
  float* d_weights;
  double* d_lambdas;
  double* d_thresholds;
  double* d_demand;
  double* h_stats;          // pinned [n_chunks][stats_len]
  uint8_t* d_stage_in[2];   // env-major entry points: per-stream staging of one chunk's inputs / outputs,
  uint8_t* d_stage_out[2];  // allocated on first use
};

using namespace smarl;

static void free_session(SmarlHostSession* s) {
  if (!s) return;
  for (auto st : s->streams)
    if (st) cudaStreamDestroy(st);
  cudaFree(s->d_start_x); cudaFree(s->d_start_y); cudaFree(s->d_actions); cudaFree(s->d_moves); cudaFree(s->d_packed); cudaFree(s->d_packed5);
  cudaFree(s->d_landmarks); cudaFree(s->d_R); cudaFree(s->d_modR); cudaFree(s->d_C); cudaFree(s->d_n_active);
  cudaFree(s->d_stats); cudaFree(s->d_scratch); cudaFree(s->d_lut); cudaFree(s->d_weights);
  cudaFree(s->d_lambdas); cudaFree(s->d_thresholds); cudaFree(s->d_demand);
  for (int i = 0; i < 2; ++i) { cudaFree(s->d_stage_in[i]); cudaFree(s->d_stage_out[i]); }
  if (s->h_stats) cudaFreeHost(s->h_stats);
  delete s;
}

extern "C" int smarl_host_session_create(SmarlHostSession** out, int32_t kind, int32_t A, int32_t T,
                                         int64_t n_envs, int32_t n_landmarks) {
  SMARL_REQUIRE(out != nullptr, "out is NULL");
  SMARL_REQUIRE(kind >= SMARL_ENV_COVERAGE && kind <= SMARL_ENV_COLLISION, "bad env kind %d", kind);
  SMARL_REQUIRE(A >= 1 && A <= SMARL_MAX_AGENTS, "n_agents=%d outside 1..32", A);
  SMARL_REQUIRE(T >= 1 && n_envs >= 1, "bad T=%d or n_envs=%lld", T, (long long)n_envs);
  SMARL_REQUIRE(kind != SMARL_ENV_COVERAGE || T <= 255, "Coverage fused rollout needs T <= 255");
  SMARL_REQUIRE(kind != SMARL_ENV_COLLISION || (n_landmarks >= 1 && n_landmarks <= 64), "bad n_landmarks");
  SmarlHostSession* s = new (std::nothrow) SmarlHostSession();
  SMARL_REQUIRE(s != nullptr, "out of host memory");
  s->kind = kind; s->A = A; s->K = kind == SMARL_ENV_COVERAGE ? A : 1; s->T = T; s->L = n_landmarks;
  s->n_envs = n_envs;
  s->ld = (n_envs + 15) / 16 * 16;
  // ~32 chunks (SMARL_HOST_CHUNKS overrides), each a multiple of 16 envs and at least 64Ki envs so launches stay
  // large.  What is not overlapped is the last chunk's kernel + download: measured on the bench shape 67.6 ms with 8
  // chunks, 66.7 with 16, 66.1 with 32, 65.8 with 64.
  const char* env_chunks = getenv("SMARL_HOST_CHUNKS");
  const int64_t n_target = env_chunks && atoll(env_chunks) > 0 ? atoll(env_chunks) : 32;
  int64_t chunk = (s->ld / n_target + 47) / 48 * 48;     // multiple of 16 (vector width) and of 3 (base-5 action triples)
  if (chunk < 65520) chunk = 65520;
  if (chunk > s->ld) chunk = s->ld;
  s->pitch5 = ((s->ld + 2) / 3 + 15) / 16 * 16;
  s->chunk = chunk;
  s->n_chunks = (int)((n_envs + chunk - 1) / chunk);
  const int sl = stats_len(A, s->K);
  s->scratch_per_chunk = smarl_stats_scratch_len(A, s->K, chunk);
  const size_t pos_elem = kind == SMARL_ENV_COLLISION ? 8 : 1;
  const size_t act_bytes = kind == SMARL_ENV_COLLISION ? (size_t)T * 2 * A * s->ld * 4 : (size_t)T * A * s->ld;
#define SMARL_TRY(call)                                                              \
  do {                                                                               \
    cudaError_t e__ = (call);                                                        \
    if (e__ != cudaSuccess) {                                                        \
      set_error("%s failed: %s", #call, cudaGetErrorString(e__));                   \
      free_session(s);                                                               \
      return SMARL_ECUDA;                                                            \
    }                                                                                \
  } while (0)
  for (auto& st : s->streams) SMARL_TRY(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  SMARL_TRY(cudaMalloc(&s->d_start_x, pos_elem * A * s->ld));
  SMARL_TRY(cudaMalloc(&s->d_start_y, pos_elem * A * s->ld));
  SMARL_TRY(cudaMalloc(&s->d_actions, act_bytes));
  if (kind == SMARL_ENV_COLLISION) {
    SMARL_TRY(cudaMalloc(&s->d_landmarks, sizeof(double) * 2 * n_landmarks * s->ld));
    SMARL_TRY(cudaMalloc(&s->d_n_active, sizeof(int32_t) * s->ld));
  }
  if (kind == SMARL_ENV_CONGESTION) SMARL_TRY(cudaMalloc(&s->d_demand, sizeof(double) * 255 * 255));
  SMARL_TRY(cudaMalloc(&s->d_R, sizeof(float) * A * s->ld));
  SMARL_TRY(cudaMalloc(&s->d_modR, sizeof(float) * A * s->ld));
  SMARL_TRY(cudaMalloc(&s->d_C, sizeof(int32_t) * s->K * s->ld));
  SMARL_TRY(cudaMalloc(&s->d_stats, sizeof(double) * sl * s->n_chunks));
  SMARL_TRY(cudaMalloc(&s->d_scratch, sizeof(double) * s->scratch_per_chunk * s->n_chunks));
  SMARL_TRY(cudaMalloc(&s->d_lut, sizeof(float) * kCoverageMaxLut));
  SMARL_TRY(cudaMalloc(&s->d_weights, sizeof(float) * SMARL_MAX_AGENTS));
  SMARL_TRY(cudaMalloc(&s->d_lambdas, sizeof(double) * SMARL_MAX_AGENTS));
  SMARL_TRY(cudaMalloc(&s->d_thresholds, sizeof(double) * SMARL_MAX_AGENTS));
  SMARL_TRY(cudaMallocHost(&s->h_stats, sizeof(double) * sl * s->n_chunks));
#undef SMARL_TRY
  *out = s;
  return SMARL_OK;
}

extern "C" void smarl_host_session_destroy(SmarlHostSession* s) { free_session(s); }

extern "C" int64_t smarl_host_session_ld(const SmarlHostSession* s) { return s ? s->ld : 0; }

extern "C" int64_t smarl_host_session_pitch5(const SmarlHostSession* s) { return s ? s->pitch5 : 0; }

namespace {

// 4-bit packed actions -> one byte per action.  Byte j of a packed row holds env 2j (low nibble) and
// env 2j+1 (high nibble); a thread expands 8 packed bytes into 16 action bytes (one 16-byte store).
__global__ void unpack4_kernel(const uint8_t* __restrict__ packed, uint8_t* __restrict__ actions, int64_t rows,
                               int64_t ld, int64_t e0, int64_t w) {
  const int64_t per_row = w / 16;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * per_row) return;
  const int64_t row = i / per_row, col = (i % per_row) * 16;
  const uint2 v = *reinterpret_cast<const uint2*>(packed + row * (ld / 2) + (e0 + col) / 2);
  auto spread = [](uint32_t h) {          // 4 nibbles in the low 16 bits -> 4 bytes
    uint32_t x = (h | (h << 8)) & 0x00FF00FFu;
    return (x | (x << 4)) & 0x0F0F0F0Fu;
  };
  uint4 o;
  o.x = spread(v.x & 0xFFFFu); o.y = spread(v.x >> 16); o.z = spread(v.y & 0xFFFFu); o.w = spread(v.y >> 16);
  *reinterpret_cast<uint4*>(actions + row * ld + e0 + col) = o;
}

// Base-5 packed actions (actions are 0..4, so three fit one byte: b = a0 + 5 a1 + 25 a2 for envs 3j, 3j+1, 3j+2)
// -> one byte per action.  A thread expands 16 packed bytes into 48 action bytes (three 16-byte stores); e0 is a
// multiple of 48, so every access is aligned.  Stores beyond the row's ld (last chunk) are dropped.
__global__ void unpack5_kernel(const uint8_t* __restrict__ packed, uint8_t* __restrict__ actions, int64_t rows,
                               int64_t ld, int64_t pitch5, int64_t e0, int64_t groups) {
  __shared__ uint32_t s_dec[256];
  for (int b = threadIdx.x; b < 256; b += blockDim.x) s_dec[b] = (uint32_t)(b % 5) | ((uint32_t)((b / 5) % 5) << 8) | ((uint32_t)(b / 25) << 16);
  __syncthreads();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * groups) return;
  const int64_t row = i / groups, g = i % groups;
  const uint4 v = *reinterpret_cast<const uint4*>(packed + row * pitch5 + e0 / 3 + g * 16);
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
  uint8_t out[48];
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    const uint32_t d = s_dec[(w[k >> 2] >> (8 * (k & 3))) & 0xFFu];
    out[3 * k] = (uint8_t)d;
    out[3 * k + 1] = (uint8_t)(d >> 8);
    out[3 * k + 2] = (uint8_t)(d >> 16);
  }
  const int64_t col = e0 + g * 48;
#pragma unroll
  for (int q = 0; q < 3; ++q) {
    if (col + 16 * q < ld) {
      uint4 o;
      memcpy(&o, out + 16 * q, 16);
      *reinterpret_cast<uint4*>(actions + row * ld + col + 16 * q) = o;
    }
  }
}

// Layout converters for callers that keep the reference's env-major arrays ([.., env, agent], what
// np.array(actions) gives there).  A CTA stages kTileEnvs envs x R rows in shared memory so that both the
// env-major side (contiguous [env][R]) and the agent-major side ([R][ld], 128 consecutive envs of a row) are
// read / written in full lines.  Rows r of an interleaved pair layout (x0,y0,x1,y1,..) go to out0 / out1.
constexpr int kTileEnvs = 128;   // envs per CTA tile; halved until the tile fits the default 48 KB of shared memory

template <typename T>
static int tile_envs(int R) {
  int te = kTileEnvs;
  while (sizeof(T) * (size_t)te * (R + 1) > 48 * 1024) te /= 2;
  return te;
}

template <typename T>
__global__ void __launch_bounds__(256) envmajor_to_agentmajor(const T* __restrict__ in, T* __restrict__ out0,
                                                              T* __restrict__ out1, int R, int64_t n, int64_t in_outer,
                                                              int64_t out_outer, int64_t ld, int te) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* tile = reinterpret_cast<T*>(smem_raw);                    // [kTileEnvs][R + 1]
  const int RP = R + 1;
  const int64_t e_base = (int64_t)blockIdx.x * te;
  const int m = (int)min((int64_t)te, n - e_base);
  const T* src = in + (int64_t)blockIdx.y * in_outer + e_base * R;
  for (int idx = threadIdx.x; idx < m * R; idx += 256) tile[(idx / R) * RP + idx % R] = src[idx];
  __syncthreads();
  for (int idx = threadIdx.x; idx < R * te; idx += 256) {
    const int r = idx / te, e = idx % te;
    if (e >= m) continue;
    T* row = out1 ? ((r & 1) ? out1 : out0) + (int64_t)(r >> 1) * ld : out0 + (int64_t)r * ld;
    row[(int64_t)blockIdx.y * out_outer + e_base + e] = tile[e * RP + r];
  }
}

template <typename T>
__global__ void __launch_bounds__(256) agentmajor_to_envmajor(const T* __restrict__ in, T* __restrict__ out, int R,
                                                              int64_t n, int64_t ld, int te) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* tile = reinterpret_cast<T*>(smem_raw);
  const int RP = R + 1;
  const int64_t e_base = (int64_t)blockIdx.x * te;
  const int m = (int)min((int64_t)te, n - e_base);
  for (int idx = threadIdx.x; idx < R * te; idx += 256) {
    const int r = idx / te, e = idx % te;
    if (e < m) tile[e * RP + r] = in[(int64_t)r * ld + e_base + e];
  }
  __syncthreads();
  T* dst = out + e_base * R;
  for (int idx = threadIdx.x; idx < m * R; idx += 256) dst[idx] = tile[(idx / R) * RP + idx % R];
}

template <typename T>
int to_env_major(const T* in, T* out, int R, int64_t n, int64_t ld, cudaStream_t st) {
  const int te = tile_envs<T>(R);
  agentmajor_to_envmajor<T><<<(unsigned)((n + te - 1) / te), 256, sizeof(T) * te * (R + 1), st>>>(in, out, R, n, ld, te);
  SMARL_CUDA(cudaGetLastError());
  return SMARL_OK;
}

struct Chunk {
  int index;
  int64_t e0, n, w;   // first env, envs in the chunk, envs copied per row (n rounded up to 16)
  cudaStream_t st;
  double* stats;      // this chunk's additive stats and their scratch
  double* scratch;
};

// rows x w elements of `elem` bytes between pitched [rows][ld] arrays, starting at env e0
int copy_rows(void* dst, const void* src, size_t elem, int64_t rows, int64_t ld, const Chunk& c, cudaMemcpyKind kind) {
  SMARL_CUDA(cudaMemcpy2DAsync(static_cast<char*>(dst) + c.e0 * elem, ld * elem,
                               static_cast<const char*>(src) + c.e0 * elem, ld * elem, c.w * elem, (size_t)rows, kind,
                               c.st));
  return SMARL_OK;
}

// One input array of a rollout.  On the device it is agent-major, [outer][R][ld] elements of `elem` bytes at `dev`,
// except that with `dev_y` the R values of an env are interleaved (x, y) pairs (outer = 1): x to the R/2 rows of
// `dev`, y to those of `dev_y`.  The host array is agent-major like the device (x and y of a pair as two arrays,
// `host` and `host_y`) or env-major [outer][E][R] (`host` only).
struct Input {
  const void* host;
  const void* host_y;
  void* dev;
  void* dev_y;
  int elem, R, outer;
  size_t stage_off = 0;   // env-major: byte offset of this input's chunk in d_stage_in, set by ensure_staging
};

// Places the env-major staging of a chunk's inputs back to back in d_stage_in, and allocates it and the staging of
// the products (R, modR, C: 3 A rows of 4 bytes) for both streams on first use.
int ensure_staging(SmarlHostSession* s, Input* in, int n_in) {
  size_t bytes = 0;
  for (int i = 0; i < n_in; ++i) {
    in[i].stage_off = bytes;
    bytes += (size_t)in[i].elem * in[i].R * in[i].outer * s->chunk;
  }
  for (int i = 0; i < 2; ++i) {
    if (!s->d_stage_in[i]) SMARL_CUDA(cudaMalloc(&s->d_stage_in[i], bytes));
    if (!s->d_stage_out[i]) SMARL_CUDA(cudaMalloc(&s->d_stage_out[i], (size_t)3 * s->A * s->chunk * 4));
  }
  return SMARL_OK;
}

template <typename T>
int to_agent_major(const Input& x, const uint8_t* stage, int64_t chunk, int64_t ld, const Chunk& c) {
  const int te = tile_envs<T>(x.R);
  dim3 grid((unsigned)((c.n + te - 1) / te), (unsigned)x.outer);
  envmajor_to_agentmajor<T><<<grid, 256, sizeof(T) * te * (x.R + 1), c.st>>>(
      reinterpret_cast<const T*>(stage + x.stage_off), static_cast<T*>(x.dev) + c.e0,
      x.dev_y ? static_cast<T*>(x.dev_y) + c.e0 : nullptr, x.R, c.n, chunk * x.R, (int64_t)x.R * ld, ld, te);
  SMARL_CUDA(cudaGetLastError());
  return SMARL_OK;
}

// A chunk of each input into its agent-major device rows: agent-major host rows are copied as they are; env-major
// ones go to the stream's staging, all copies before the first transpose, then to the rows.
int to_device(SmarlHostSession* s, const Chunk& c, bool env_major, const Input* in, int n_in) {
  const int64_t ld = s->ld, chunk = s->chunk;
  uint8_t* stage = s->d_stage_in[c.index & 1];
  for (int i = 0; i < n_in; ++i) {
    const Input& x = in[i];
    if (!env_major) {
      const int64_t rows = x.dev_y ? x.R / 2 : (int64_t)x.outer * x.R;
      if (int rc = copy_rows(x.dev, x.host, x.elem, rows, ld, c, cudaMemcpyHostToDevice)) return rc;
      if (x.dev_y)
        if (int rc = copy_rows(x.dev_y, x.host_y, x.elem, rows, ld, c, cudaMemcpyHostToDevice)) return rc;
    } else {
      // the env-major host rows of this chunk are contiguous per step: [e0, e0+n) x R
      const size_t row = (size_t)x.elem * x.R;
      const char* src = static_cast<const char*>(x.host) + c.e0 * row;
      if (x.outer == 1)
        SMARL_CUDA(cudaMemcpyAsync(stage + x.stage_off, src, c.n * row, cudaMemcpyHostToDevice, c.st));
      else
        SMARL_CUDA(cudaMemcpy2DAsync(stage + x.stage_off, chunk * row, src, s->n_envs * row, c.n * row,
                                     (size_t)x.outer, cudaMemcpyHostToDevice, c.st));
    }
  }
  for (int i = 0; env_major && i < n_in; ++i) {
    const int rc = in[i].elem == 1 ? to_agent_major<uint8_t>(in[i], stage, chunk, ld, c)
                   : in[i].elem == 4 ? to_agent_major<float>(in[i], stage, chunk, ld, c)
                                     : to_agent_major<double>(in[i], stage, chunk, ld, c);
    if (rc) return rc;
  }
  return SMARL_OK;
}

// A chunk's products back to the host: R, modR [A] and C [K] rows, n_active when asked for, then the chunk's stats.
// Agent-major host arrays take the rows as they are; env-major ones ([E][A], [E][K], [E]) through a transpose into
// the stream's product staging.
int from_device(SmarlHostSession* s, const Chunk& c, bool env_major, float* R_h, float* modR_h, int32_t* C_h,
                int32_t* n_active_h) {
  const int A = s->A, K = s->K, sl = stats_len(A, K);
  const int64_t ld = s->ld, chunk = s->chunk;
  if (!env_major) {
    if (int rc = copy_rows(R_h, s->d_R, 4, A, ld, c, cudaMemcpyDeviceToHost)) return rc;
    if (int rc = copy_rows(modR_h, s->d_modR, 4, A, ld, c, cudaMemcpyDeviceToHost)) return rc;
    if (n_active_h)
      if (int rc = copy_rows(n_active_h, s->d_n_active, 4, 1, ld, c, cudaMemcpyDeviceToHost)) return rc;
    if (int rc = copy_rows(C_h, s->d_C, 4, K, ld, c, cudaMemcpyDeviceToHost)) return rc;
  } else {
    if (n_active_h)
      SMARL_CUDA(cudaMemcpyAsync(n_active_h + c.e0, s->d_n_active + c.e0, (size_t)c.n * 4, cudaMemcpyDeviceToHost, c.st));
    float* st_R = reinterpret_cast<float*>(s->d_stage_out[c.index & 1]);
    float* st_M = st_R + (size_t)A * chunk;
    int32_t* st_C = reinterpret_cast<int32_t*>(st_M + (size_t)A * chunk);
    if (int rc = to_env_major<float>(s->d_R + c.e0, st_R, A, c.n, ld, c.st)) return rc;
    if (int rc = to_env_major<float>(s->d_modR + c.e0, st_M, A, c.n, ld, c.st)) return rc;
    if (int rc = to_env_major<int32_t>(s->d_C + c.e0, st_C, K, c.n, ld, c.st)) return rc;
    SMARL_CUDA(cudaMemcpyAsync(R_h + c.e0 * A, st_R, (size_t)c.n * A * 4, cudaMemcpyDeviceToHost, c.st));
    SMARL_CUDA(cudaMemcpyAsync(modR_h + c.e0 * A, st_M, (size_t)c.n * A * 4, cudaMemcpyDeviceToHost, c.st));
    SMARL_CUDA(cudaMemcpyAsync(C_h + c.e0 * K, st_C, (size_t)c.n * K * 4, cudaMemcpyDeviceToHost, c.st));
  }
  SMARL_CUDA(cudaMemcpyAsync(s->h_stats + (int64_t)c.index * sl, c.stats, sizeof(double) * sl, cudaMemcpyDeviceToHost,
                             c.st));
  return SMARL_OK;
}

// What every rollout entry does first: checks that the call fits the session, then the env's own parameters
// (`check`), and only then queues the uploads of lambdas and thresholds, so that a call these checks reject has
// queued nothing.  *dacc is acc with its thresholds on the device.
template <class Params, class Check>
int begin_rollout(SmarlHostSession* s, int kind, const Params* p, const SmarlAccounting* acc, bool have_buffers,
                  const double* lambdas_h, SmarlAccounting* dacc, Check check) {
  SMARL_REQUIRE(s && p && acc, "null session / params");
  SMARL_REQUIRE(s->kind == kind && p->n_agents == s->A && acc->n_steps == s->T,
                "session was created for kind=%d A=%d T=%d", s->kind, s->A, s->T);
  SMARL_REQUIRE(acc->g_mode == 0, "host rollout returns episode products only (g_mode 0)");
  SMARL_REQUIRE(have_buffers, "null host buffer");
  if (int rc = check()) return rc;
  cudaStream_t s0 = s->streams[0];
  if (lambdas_h) SMARL_CUDA(cudaMemcpyAsync(s->d_lambdas, lambdas_h, sizeof(double) * s->K, cudaMemcpyHostToDevice, s0));
  if (acc->thresholds)
    SMARL_CUDA(cudaMemcpyAsync(s->d_thresholds, acc->thresholds, sizeof(double) * s->K, cudaMemcpyHostToDevice, s0));
  *dacc = *acc;
  dacc->thresholds = acc->thresholds ? s->d_thresholds : nullptr;
  return SMARL_OK;
}

// Waits for the first n_streams streams and returns rc, or the first failure to wait if rc is SMARL_OK.
int sync_streams(SmarlHostSession* s, int n_streams, int rc) {
  for (int i = 0; i < n_streams; ++i) {
    const cudaError_t e = cudaStreamSynchronize(s->streams[i]);
    if (e != cudaSuccess && rc == SMARL_OK) {
      set_error("cudaStreamSynchronize failed: %s", cudaGetErrorString(e));
      rc = SMARL_ECUDA;
    }
  }
  return rc;
}

// Runs `body(chunk)` for every env chunk on alternating streams, then gathers the additive stats.  Both streams are
// drained before it returns, after an error too, since copies already queued read and write the caller's arrays;
// the first error is the one reported.
template <class Body>
int pipeline(SmarlHostSession* s, double* stats_h, Body body) {
  const int sl = stats_len(s->A, s->K);
  int rc = sync_streams(s, 1, SMARL_OK);                   // small parameter uploads are visible to both streams
  for (int c = 0; c < s->n_chunks && rc == SMARL_OK; ++c) {
    Chunk ch;
    ch.index = c;
    ch.st = s->streams[c & 1];
    ch.e0 = (int64_t)c * s->chunk;
    ch.n = (ch.e0 + s->chunk <= s->n_envs) ? s->chunk : (s->n_envs - ch.e0);
    ch.w = (ch.n + 15) / 16 * 16;
    ch.stats = s->d_stats + (int64_t)c * sl;
    ch.scratch = s->d_scratch + (int64_t)c * s->scratch_per_chunk;
    rc = body(ch);
  }
  if (int e = sync_streams(s, 2, rc)) return e;
  if (stats_h) {
    for (int j = 0; j < sl; ++j) {
      double v = 0.0;
      for (int c = 0; c < s->n_chunks; ++c) v += s->h_stats[(int64_t)c * sl + j];
      stats_h[j] = v;
    }
  }
  return SMARL_OK;
}

// CoverageDiscrete episodes.  Agent-major host arrays (start_y_h given) carry one byte per action or, by `packing`,
// two 4-bit (4) or three base-5 (5) actions per byte; env-major arrays (start_y_h unused) one byte per action.
int coverage_rollout(SmarlHostSession* s, const SmarlCoverageParams* p, const SmarlAccounting* acc, bool env_major,
                     int packing /* 0 bytes, 4 nibbles, 5 base-5 triples */, const uint8_t* starts_h,
                     const uint8_t* start_y_h, const uint8_t* actions_h, const double* lambdas_h, float* R_h,
                     float* modR_h, int32_t* C_h, double* stats_h) {
  SmarlAccounting dacc;
  const bool have_buffers = starts_h && (env_major || start_y_h) && actions_h && R_h && modR_h && C_h;
  if (int rc = begin_rollout(s, SMARL_ENV_COVERAGE, p, acc, have_buffers, lambdas_h, &dacc, [&]() -> int {
        SMARL_REQUIRE(p->lut_len >= 0, "lut_len=%d is negative", p->lut_len);
        if (p->lut_len > kCoverageMaxLut) {
          set_error("lut_len=%d exceeds the shared-memory table limit %d", p->lut_len, kCoverageMaxLut);
          return SMARL_EUNSUPPORTED;
        }
        return SMARL_OK;
      }))
    return rc;
  const int A = s->A, T = s->T;
  const int64_t ld = s->ld;
  uint8_t* dx = static_cast<uint8_t*>(s->d_start_x);
  uint8_t* dy = static_cast<uint8_t*>(s->d_start_y);
  uint8_t* da = static_cast<uint8_t*>(s->d_actions);
  Input in[] = {{starts_h, start_y_h, dx, dy, 1, 2 * A, 1}, {actions_h, nullptr, da, nullptr, 1, A, T}};
  if (env_major)
    if (int rc = ensure_staging(s, in, 2)) return rc;
  if (packing == 4 && !s->d_packed) SMARL_CUDA(cudaMalloc(&s->d_packed, (size_t)T * A * ld / 2));
  if (packing == 5 && !s->d_packed5) SMARL_CUDA(cudaMalloc(&s->d_packed5, (size_t)T * A * s->pitch5));
  cudaStream_t s0 = s->streams[0];
  if (p->lut_len) SMARL_CUDA(cudaMemcpyAsync(s->d_lut, p->lut, sizeof(float) * p->lut_len, cudaMemcpyHostToDevice, s0));
  if (p->weights) SMARL_CUDA(cudaMemcpyAsync(s->d_weights, p->weights, sizeof(float) * A, cudaMemcpyHostToDevice, s0));
  SmarlCoverageParams dp = *p;
  dp.lut = s->d_lut;
  dp.weights = p->weights ? s->d_weights : nullptr;
  return pipeline(s, stats_h, [&](const Chunk& c) -> int {
    if (int rc = to_device(s, c, env_major, in, packing ? 1 : 2)) return rc;
    if (packing == 4) {                 // half the PCIe bytes: copy nibbles, expand on the device
      const int64_t rows = (int64_t)T * A;
      SMARL_CUDA(cudaMemcpy2DAsync(s->d_packed + c.e0 / 2, ld / 2, actions_h + c.e0 / 2, ld / 2, c.w / 2, (size_t)rows,
                                   cudaMemcpyHostToDevice, c.st));
      const int64_t n = rows * (c.w / 16);
      unpack4_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c.st>>>(s->d_packed, da, rows, ld, c.e0, c.w);
      SMARL_CUDA(cudaGetLastError());
    } else if (packing == 5) {          // a third of the PCIe bytes: copy base-5 triples, expand on the device
      const int64_t rows = (int64_t)T * A, groups = (c.w + 47) / 48;       // 16 packed bytes = 48 envs per group
      int64_t w5 = groups * 16;
      if (c.e0 / 3 + w5 > s->pitch5) w5 = s->pitch5 - c.e0 / 3;
      SMARL_CUDA(cudaMemcpy2DAsync(s->d_packed5 + c.e0 / 3, s->pitch5, actions_h + c.e0 / 3, s->pitch5, (size_t)w5,
                                   (size_t)rows, cudaMemcpyHostToDevice, c.st));
      const int64_t n = rows * groups;
      unpack5_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c.st>>>(s->d_packed5, da, rows, ld, s->pitch5, c.e0, groups);
      SMARL_CUDA(cudaGetLastError());
    }
    if (int rc = smarl_coverage_rollout(&dp, &dacc, dx + c.e0, dy + c.e0, da + c.e0, lambdas_h ? s->d_lambdas : nullptr,
                                        nullptr, nullptr, s->d_R + c.e0, s->d_modR + c.e0, s->d_C + c.e0, nullptr,
                                        nullptr, c.stats, c.scratch, c.n, ld, c.st))
      return rc;
    return from_device(s, c, env_major, R_h, modR_h, C_h, nullptr);
  });
}

// Congestion episodes; the host arrays are agent-major (start_y_h given) or env-major.
int congestion_rollout(SmarlHostSession* s, const SmarlCongestionParams* p, const SmarlAccounting* acc, bool env_major,
                       const uint8_t* starts_h, const uint8_t* start_y_h, const uint8_t* actions_h,
                       const uint8_t* moves_h, const double* lambdas_h, float* R_h, float* modR_h, int32_t* C_h,
                       double* stats_h) {
  SmarlAccounting dacc;
  const bool have_buffers = starts_h && (env_major || start_y_h) && actions_h && R_h && modR_h && C_h;
  if (int rc = begin_rollout(s, SMARL_ENV_CONGESTION, p, acc, have_buffers, lambdas_h, &dacc, [&]() -> int {
        SMARL_REQUIRE(p->size >= 1 && p->size <= 254 && p->demand, "bad size or demand table");
        SMARL_REQUIRE(p->noise_mode != 1 || moves_h, "noise_mode 1 needs the recorded moves");
        return SMARL_OK;
      }))
    return rc;
  const int A = s->A, T = s->T, W = p->size + 1;
  const int64_t ld = s->ld;
  if (moves_h && !s->d_moves) SMARL_CUDA(cudaMalloc(&s->d_moves, (size_t)T * A * ld));
  uint8_t* dx = static_cast<uint8_t*>(s->d_start_x);
  uint8_t* dy = static_cast<uint8_t*>(s->d_start_y);
  uint8_t* da = static_cast<uint8_t*>(s->d_actions);
  Input in[] = {{starts_h, start_y_h, dx, dy, 1, 2 * A, 1}, {actions_h, nullptr, da, nullptr, 1, A, T},
                {moves_h, nullptr, s->d_moves, nullptr, 1, A, T}};
  if (env_major)
    if (int rc = ensure_staging(s, in, 3)) return rc;
  SMARL_CUDA(cudaMemcpyAsync(s->d_demand, p->demand, sizeof(double) * W * W, cudaMemcpyHostToDevice, s->streams[0]));
  SmarlCongestionParams dp = *p;
  dp.episode_dev = nullptr;                 // host callers pass the episode by value
  dp.demand = s->d_demand;
  dp.wait_reward = nullptr;                 // host callers pass the demand table only; the kernel divides
  return pipeline(s, stats_h, [&](const Chunk& c) -> int {
    if (int rc = to_device(s, c, env_major, in, 2)) return rc;
    if (moves_h)
      if (int rc = to_device(s, c, env_major, in + 2, 1)) return rc;
    SmarlCongestionParams cp = dp;
    cp.env_offset = dp.env_offset + c.e0;                 // Philox streams are keyed by the global env id
    if (int rc = smarl_congestion_rollout(&cp, &dacc, dx + c.e0, dy + c.e0, da + c.e0, moves_h ? s->d_moves + c.e0 : nullptr,
                                          lambdas_h ? s->d_lambdas : nullptr, nullptr, nullptr, s->d_R + c.e0,
                                          s->d_modR + c.e0, s->d_C + c.e0, nullptr, nullptr, c.stats, c.scratch, c.n, ld,
                                          c.st))
      return rc;
    return from_device(s, c, env_major, R_h, modR_h, C_h, nullptr);
  });
}

// CollisionAvoidance episodes; the host arrays are agent-major (start_y_h given) or env-major.
int collision_rollout(SmarlHostSession* s, const SmarlCollisionParams* p, const SmarlAccounting* acc, bool env_major,
                      const double* starts_h, const double* start_y_h, const double* landmarks_h, const float* actions_h,
                      const double* lambdas_h, float* R_h, float* modR_h, int32_t* C_h, int32_t* n_active_h,
                      double* stats_h) {
  SmarlAccounting dacc;
  const bool have_buffers = starts_h && (env_major || start_y_h) && landmarks_h && actions_h && R_h && modR_h && C_h;
  if (int rc = begin_rollout(s, SMARL_ENV_COLLISION, p, acc, have_buffers, lambdas_h, &dacc, [&]() -> int {
        SMARL_REQUIRE(p->n_landmarks == s->L, "session was created for n_landmarks=%d", s->L);
        return SMARL_OK;
      }))
    return rc;
  const int A = s->A, T = s->T, L = s->L;
  const int64_t ld = s->ld;
  double* dx = static_cast<double*>(s->d_start_x);
  double* dy = static_cast<double*>(s->d_start_y);
  float* da = static_cast<float*>(s->d_actions);
  Input in[] = {{starts_h, start_y_h, dx, dy, 8, 2 * A, 1}, {landmarks_h, nullptr, s->d_landmarks, nullptr, 8, 2 * L, 1},
                {actions_h, nullptr, da, nullptr, 4, 2 * A, T}};
  if (env_major)
    if (int rc = ensure_staging(s, in, 3)) return rc;
  return pipeline(s, stats_h, [&](const Chunk& c) -> int {
    if (int rc = to_device(s, c, env_major, in, 3)) return rc;
    if (int rc = smarl_collision_rollout(p, &dacc, dx + c.e0, dy + c.e0, s->d_landmarks + c.e0, da + c.e0,
                                         lambdas_h ? s->d_lambdas : nullptr, nullptr, nullptr, nullptr,
                                         s->d_n_active + c.e0, s->d_R + c.e0, s->d_modR + c.e0, s->d_C + c.e0, nullptr,
                                         nullptr, c.stats, c.scratch, c.n, ld, c.st))
      return rc;
    return from_device(s, c, env_major, R_h, modR_h, C_h, n_active_h);
  });
}

}  // namespace

extern "C" int smarl_host_coverage_rollout(SmarlHostSession* s, const SmarlCoverageParams* p,
                                           const SmarlAccounting* acc, const uint8_t* start_x_h,
                                           const uint8_t* start_y_h, const uint8_t* actions_h,
                                           const double* lambdas_h, float* R_h, float* modR_h,
                                           int32_t* C_h, double* stats_h) {
  return coverage_rollout(s, p, acc, false, 0, start_x_h, start_y_h, actions_h, lambdas_h, R_h, modR_h, C_h, stats_h);
}

extern "C" int smarl_host_coverage_rollout_packed4(SmarlHostSession* s, const SmarlCoverageParams* p,
                                                   const SmarlAccounting* acc, const uint8_t* start_x_h,
                                                   const uint8_t* start_y_h, const uint8_t* actions4_h,
                                                   const double* lambdas_h, float* R_h, float* modR_h,
                                                   int32_t* C_h, double* stats_h) {
  return coverage_rollout(s, p, acc, false, 4, start_x_h, start_y_h, actions4_h, lambdas_h, R_h, modR_h, C_h, stats_h);
}

extern "C" int smarl_host_coverage_rollout_packed5(SmarlHostSession* s, const SmarlCoverageParams* p,
                                                   const SmarlAccounting* acc, const uint8_t* start_x_h,
                                                   const uint8_t* start_y_h, const uint8_t* actions5_h,
                                                   const double* lambdas_h, float* R_h, float* modR_h,
                                                   int32_t* C_h, double* stats_h) {
  return coverage_rollout(s, p, acc, false, 5, start_x_h, start_y_h, actions5_h, lambdas_h, R_h, modR_h, C_h, stats_h);
}

extern "C" int smarl_host_coverage_rollout_envmajor(SmarlHostSession* s, const SmarlCoverageParams* p,
                                                    const SmarlAccounting* acc, const uint8_t* starts_h,
                                                    const uint8_t* actions_h, const double* lambdas_h, float* R_h,
                                                    float* modR_h, int32_t* C_h, double* stats_h) {
  return coverage_rollout(s, p, acc, true, 0, starts_h, nullptr, actions_h, lambdas_h, R_h, modR_h, C_h, stats_h);
}

extern "C" int smarl_host_congestion_rollout(SmarlHostSession* s, const SmarlCongestionParams* p,
                                             const SmarlAccounting* acc, const uint8_t* start_x_h,
                                             const uint8_t* start_y_h, const uint8_t* actions_h,
                                             const uint8_t* moves_h, const double* lambdas_h, float* R_h,
                                             float* modR_h, int32_t* C_h, double* stats_h) {
  return congestion_rollout(s, p, acc, false, start_x_h, start_y_h, actions_h, moves_h, lambdas_h, R_h, modR_h, C_h,
                            stats_h);
}

extern "C" int smarl_host_congestion_rollout_envmajor(SmarlHostSession* s, const SmarlCongestionParams* p,
                                                      const SmarlAccounting* acc, const uint8_t* starts_h,
                                                      const uint8_t* actions_h, const uint8_t* moves_h,
                                                      const double* lambdas_h, float* R_h, float* modR_h,
                                                      int32_t* C_h, double* stats_h) {
  return congestion_rollout(s, p, acc, true, starts_h, nullptr, actions_h, moves_h, lambdas_h, R_h, modR_h, C_h, stats_h);
}

extern "C" int smarl_host_collision_rollout(SmarlHostSession* s, const SmarlCollisionParams* p,
                                            const SmarlAccounting* acc, const double* start_x_h,
                                            const double* start_y_h, const double* landmarks_h,
                                            const float* actions_h, const double* lambdas_h, float* R_h,
                                            float* modR_h, int32_t* C_h, int32_t* n_active_h, double* stats_h) {
  return collision_rollout(s, p, acc, false, start_x_h, start_y_h, landmarks_h, actions_h, lambdas_h, R_h, modR_h, C_h,
                           n_active_h, stats_h);
}

extern "C" int smarl_host_collision_rollout_envmajor(SmarlHostSession* s, const SmarlCollisionParams* p,
                                                     const SmarlAccounting* acc, const double* starts_h,
                                                     const double* landmarks_h, const float* actions_h,
                                                     const double* lambdas_h, float* R_h, float* modR_h,
                                                     int32_t* C_h, int32_t* n_active_h, double* stats_h) {
  return collision_rollout(s, p, acc, true, starts_h, nullptr, landmarks_h, actions_h, lambdas_h, R_h, modR_h, C_h,
                           n_active_h, stats_h);
}

// ---------------------------------------------------------------------------------------
// Pinned host staging on the NUMA node the current GPU hangs off.  With several ranks on one box, pinned buffers
// that all sit on one node make every GPU of the other socket pull its PCIe traffic across the inter-socket link;
// this binds the allocation (first touch) to the GPU's own node when the kernel lets it.
// ---------------------------------------------------------------------------------------
static int gpu_numa_node() {
  int dev = 0;
  char bus[32] = "";
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetPCIBusId(bus, sizeof(bus), dev) != cudaSuccess) return -1;
  for (char* c = bus; *c; ++c)
    if (*c >= 'A' && *c <= 'F') *c = (char)(*c - 'A' + 'a');     // sysfs spells the address in lower case
  char path[128];
  snprintf(path, sizeof(path), "/sys/bus/pci/devices/%s/numa_node", bus);
  FILE* f = fopen(path, "r");
  if (!f) return -1;
  int node = -1;
  if (fscanf(f, "%d", &node) != 1) node = -1;
  fclose(f);
  return node;
}

extern "C" int smarl_host_alloc_pinned(void** out, size_t bytes, int32_t* numa_node_out) {
  SMARL_REQUIRE(out != nullptr && bytes > 0, "bad arguments");
  const int node = gpu_numa_node();
  bool bound = false;
#ifdef SYS_set_mempolicy
  if (node >= 0 && node < 1024) {
    unsigned long mask[16] = {0};
    mask[node / (8 * sizeof(unsigned long))] |= 1ul << (node % (8 * sizeof(unsigned long)));
    // MPOL_PREFERRED = 1: fall back to other nodes instead of failing when the node is full or not in cpuset.mems
    bound = syscall(SYS_set_mempolicy, 1, mask, (unsigned long)(8 * sizeof(mask) + 1)) == 0;
  }
#endif
  void* p = nullptr;
  cudaError_t err = cudaHostAlloc(&p, bytes, cudaHostAllocPortable);
  if (err == cudaSuccess) memset(p, 0, bytes);                   // first touch under the policy
#ifdef SYS_set_mempolicy
  if (bound) syscall(SYS_set_mempolicy, 0 /* MPOL_DEFAULT */, nullptr, 0ul);
#endif
  if (err != cudaSuccess) {
    set_error("cudaHostAlloc(%zu) failed: %s", bytes, cudaGetErrorString(err));
    return SMARL_ECUDA;
  }
  if (numa_node_out) *numa_node_out = bound ? node : -1;
  *out = p;
  return SMARL_OK;
}

extern "C" void smarl_host_free_pinned(void* p) {
  if (p) cudaFreeHost(p);
}
