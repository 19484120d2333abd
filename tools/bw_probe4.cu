// Bandwidth probe with returns_kernel's exact traffic at the bench shape (A = K = 16, T = 50, E = ld = 2^22),
// no arithmetic beyond what keeps the loads live.  Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o bw_probe4 bw_probe4.cu
//
// One CTA of 128 threads per (row, 512-env chunk), the A + K rows of a chunk on consecutive block ids, t walked
// from high to low.  Agent rows read a 2 KB f32 reward tile and the chunk's 2 KB penalty tile (an L2 hit for all
// but the first of the A CTAs) and write a 2 KB G tile per step, then R and modR; constraint rows read a 512 B u8
// cost tile per step, then write C.  Variants:
//   regs     per-thread ld.global.nc, unroll 4 (how returns_kernel loaded before the ring)
//   ring S   cp.async.bulk into an S-stage shared-memory ring, mbarrier full/empty, thread 0 refills
//   ringK S  the same, but one CTA takes all K constraint rows of a chunk (grid = A + 1 CTAs per chunk)
//   read S / copy S   the reward slab alone through the ring: read-only, and read + st.global.cs of G
// GB/s are algorithmic bytes over CUDA-event time (the returns variants move 31.8 GB per launch).
#include <cstdint>
#include <cstdio>
#include <cuda_runtime.h>

#include "../safe_multiagent_rl_b200/csrc/mbarrier.cuh"

using namespace smarl;

constexpr int A = 16, K = 16, T = 50, TH = 128, CH = 4 * TH;
constexpr int64_t E = 1 << 22, LD = E;

__device__ __forceinline__ float4 ldnc4(const void* p) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ uint32_t ldnc1(const void* p) {
  uint32_t v;
  asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ void stcs4(void* p, float4 v) {
  asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ float4 sub4(float4 r, float4 p) { return make_float4(r.x - p.x, r.y - p.y, r.z - p.z, r.w - p.w); }
__device__ __forceinline__ float4 add4(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
__device__ __forceinline__ uint32_t addb(uint32_t s, uint32_t w) { return s + (w & 0xFF) + ((w >> 8) & 0xFF) + ((w >> 16) & 0xFF) + (w >> 24); }

struct Bufs {
  const float* rew;
  const uint8_t* cost;
  const float* pen;
  float *G, *R, *M;
  int32_t* C;
};

__global__ void __launch_bounds__(TH) regs_kernel(Bufs b) {
  const int row = blockIdx.x % (A + K);
  const int64_t chunk = blockIdx.x / (A + K);
  const int64_t e0 = chunk * CH + 4 * threadIdx.x;
  if (row < A) {
    float4 acc = make_float4(0, 0, 0, 0);
#pragma unroll 4
    for (int t = T - 1; t >= 0; --t) {
      const float4 r = ldnc4(b.rew + ((int64_t)t * A + row) * LD + e0);
      const float4 p = ldnc4(b.pen + (int64_t)t * LD + e0);
      acc = add4(acc, r);
      stcs4(b.G + ((int64_t)t * A + row) * LD + e0, sub4(acc, p));
    }
    stcs4(b.R + row * LD + e0, acc);
    stcs4(b.M + row * LD + e0, acc);
  } else {
    uint32_t s = 0;
#pragma unroll 4
    for (int t = 0; t < T; ++t) s = addb(s, ldnc1(b.cost + ((int64_t)t * K + row - A) * LD + e0));
    stcs4(b.C + (row - A) * LD + e0, make_float4(__int_as_float(s), 0, 0, 0));
  }
}

// Ring of S stages of STAGE bytes in dynamic shared memory, barriers after it.
template <int S>
struct Ring {
  uint8_t* base;
  uint64_t* full;
  uint64_t* empty;
  int stage_bytes;
  __device__ void* stage(int i) { return base + (i % S) * stage_bytes; }
  __device__ void wait(int i) { mbar_wait(&full[i % S], (uint32_t)(i / S) & 1u); }
};

// MODE 0: returns traffic, one CTA per row.  MODE 1: returns traffic, one CTA for all K constraint rows.
// MODE 2: read the reward slab only.  MODE 3: copy reward -> G.
template <int S, int MODE>
__global__ void __launch_bounds__(TH) ring_kernel(Bufs b, int stage_bytes) {
  extern __shared__ __align__(128) uint8_t smem[];
  Ring<S> ring{smem, reinterpret_cast<uint64_t*>(smem + S * stage_bytes), reinterpret_cast<uint64_t*>(smem + S * stage_bytes) + S,
               stage_bytes};
  const int rows = MODE == 0 ? A + K : MODE == 1 ? A + 1 : A;
  const int row = blockIdx.x % rows;
  const int64_t chunk = blockIdx.x / rows;
  const int64_t c0 = chunk * CH;
  const bool agent = row < A;
  const int kr = MODE == 1 ? K : 1;
  const uint64_t pol = l2_evict_first_policy();
  auto issue = [&](int i) {
    uint64_t* f = &ring.full[i % S];
    uint8_t* st = (uint8_t*)ring.stage(i);
    if (agent) {
      const int t = T - 1 - i;
      const bool pen = MODE < 2;
      mbar_arrive_expect_tx(f, pen ? 2 * CH * 4 : CH * 4);
      bulk_load(st, b.rew + ((int64_t)t * A + row) * LD + c0, CH * 4, f, pol);
      if (pen) bulk_load(st + CH * 4, b.pen + (int64_t)t * LD + c0, CH * 4, f, l2_evict_normal_policy());
    } else {
      mbar_arrive_expect_tx(f, kr * CH);
      for (int k = 0; k < kr; ++k)
        bulk_load(st + k * CH, b.cost + ((int64_t)i * K + (row - A) + k) * LD + c0, CH, f, pol);
    }
  };
  if (threadIdx.x == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(&ring.full[s], 1);
      mbar_init(&ring.empty[s], TH);
    }
    for (int i = 0; i < (S < T ? S : T); ++i) issue(i);
  }
  __syncthreads();
  auto release = [&](int i) {
    mbar_arrive(&ring.empty[i % S]);
    if (threadIdx.x == 0 && i >= 1 && i - 1 + S < T) {
      mbar_wait(&ring.empty[(i - 1) % S], (uint32_t)((i - 1) / S) & 1u);
      issue(i - 1 + S);
    }
  };
  const int64_t e0 = c0 + 4 * threadIdx.x;
  if (agent) {
    float4 acc = make_float4(0, 0, 0, 0);
    for (int i = 0; i < T; ++i) {
      const int t = T - 1 - i;
      ring.wait(i);
      const float4 r = reinterpret_cast<const float4*>(ring.stage(i))[threadIdx.x];
      const float4 p = MODE < 2 ? reinterpret_cast<const float4*>(ring.stage(i))[TH + threadIdx.x] : make_float4(0, 0, 0, 0);
      release(i);
      acc = add4(acc, r);
      if (MODE != 2) stcs4(b.G + ((int64_t)t * A + row) * LD + e0, sub4(acc, p));
    }
    if (MODE < 2) {
      stcs4(b.R + row * LD + e0, acc);
      stcs4(b.M + row * LD + e0, acc);
    } else if (MODE == 2 && acc.x == 12345.f) {
      b.R[0] = acc.y;   // keeps the reads live
    }
  } else {
    uint32_t s[kr];
    for (int k = 0; k < kr; ++k) s[k] = 0;
    for (int i = 0; i < T; ++i) {
      ring.wait(i);
      for (int k = 0; k < kr; ++k) s[k] = addb(s[k], reinterpret_cast<const uint32_t*>((uint8_t*)ring.stage(i) + k * CH)[threadIdx.x]);
      release(i);
    }
    for (int k = 0; k < kr; ++k) stcs4(b.C + (row - A + k) * LD + e0, make_float4(__int_as_float(s[k]), 0, 0, 0));
  }
}

#define CK(x)                                                                      \
  do {                                                                             \
    cudaError_t e_ = (x);                                                          \
    if (e_ != cudaSuccess) {                                                       \
      printf("%s failed: %s (line %d)\n", #x, cudaGetErrorString(e_), __LINE__);   \
      return 1;                                                                    \
    }                                                                              \
  } while (0)

template <typename F>
static float time_ms(F launch, int reps) {
  cudaEvent_t a, b;
  cudaEventCreate(&a);
  cudaEventCreate(&b);
  launch();
  cudaEventRecord(a);
  for (int i = 0; i < reps; ++i) launch();
  cudaEventRecord(b);
  cudaEventSynchronize(b);
  float ms = 0;
  cudaEventElapsedTime(&ms, a, b);
  cudaEventDestroy(a);
  cudaEventDestroy(b);
  return ms / reps;
}

template <int S, int MODE>
static int run_ring(const Bufs& b, const char* name, double bytes) {
  const int stage = MODE == 1 ? K * CH : 2 * CH * 4;
  const int smem = S * stage + 2 * S * 8;
  CK(cudaFuncSetAttribute(ring_kernel<S, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  int occ = 0;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, ring_kernel<S, MODE>, TH, smem));
  const int rows = MODE == 0 ? A + K : MODE == 1 ? A + 1 : A;
  const unsigned grid = (unsigned)(E / CH * rows);
  const float ms = time_ms([&] { ring_kernel<S, MODE><<<grid, TH, smem>>>(b, stage); }, 5);
  CK(cudaGetLastError());
  CK(cudaDeviceSynchronize());
  printf("%-8s S=%-2d smem %6d B  %2d CTAs/SM  %8.3f ms  %7.0f GB/s\n", name, S, smem, occ, ms, bytes / ms / 1e6);
  return 0;
}

int main() {
  const double n_rew = (double)T * A * LD, n_cost = (double)T * K * LD, n_pen = (double)T * LD;
  const double returns_bytes = n_rew * 4 + n_cost + n_pen * 4 + n_rew * 4 + 2.0 * A * LD * 4 + K * LD * 4;
  Bufs b;
  float *rew, *pen, *G, *R, *M;
  uint8_t* cost;
  int32_t* C;
  CK(cudaMalloc(&rew, (size_t)n_rew * 4));
  CK(cudaMalloc(&G, (size_t)n_rew * 4));
  CK(cudaMalloc(&cost, (size_t)n_cost));
  CK(cudaMalloc(&pen, (size_t)n_pen * 4));
  CK(cudaMalloc(&R, (size_t)A * LD * 4));
  CK(cudaMalloc(&M, (size_t)A * LD * 4));
  CK(cudaMalloc(&C, (size_t)K * LD * 4));
  CK(cudaMemset(rew, 0, (size_t)n_rew * 4));
  CK(cudaMemset(cost, 1, (size_t)n_cost));
  CK(cudaMemset(pen, 0, (size_t)n_pen * 4));
  b = Bufs{rew, cost, pen, G, R, M, C};
  printf("returns traffic: %.2f GB per launch (A=%d K=%d T=%d E=%lld)\n", returns_bytes / 1e9, A, K, T, (long long)E);
  {
    int occ = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, regs_kernel, TH, 0));
    const float ms = time_ms([&] { regs_kernel<<<(unsigned)(E / CH * (A + K)), TH>>>(b); }, 5);
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    printf("%-8s      smem %6d B  %2d CTAs/SM  %8.3f ms  %7.0f GB/s\n", "regs", 0, occ, ms, returns_bytes / ms / 1e6);
  }
  if (run_ring<4, 0>(b, "ring", returns_bytes) || run_ring<6, 0>(b, "ring", returns_bytes) ||
      run_ring<8, 0>(b, "ring", returns_bytes) || run_ring<16, 0>(b, "ring", returns_bytes) ||
      run_ring<4, 1>(b, "ringK", returns_bytes) || run_ring<8, 1>(b, "ringK", returns_bytes) ||
      run_ring<6, 2>(b, "read", n_rew * 4) || run_ring<6, 3>(b, "copy", n_rew * 8))
    return 1;
  cudaFree(rew); cudaFree(G); cudaFree(cost); cudaFree(pen); cudaFree(R); cudaFree(M); cudaFree(C);
  return 0;
}
