// CoverageContinuous / CoverageDiscretized code shared by the open-loop kernels (coverage_float.cu) and the on-policy
// rollout (coverage_float_policy.cu): the kernels' arguments and the env step of one env held in registers.  Both
// files are compiled with -fmad=false.
#pragma once
#include "common.cuh"

namespace smarl {

struct CoverageFloatArgs {
  double* pos_x;
  double* pos_y;
  const void* actions;
  float* obs;
  float* reward;
  float* cost;
  uint8_t* done;
  const double* lambdas;
  float* penalty;
  const float* weights;
  int64_t n_envs;
  int64_t ld;
  double size, fieldview, max_norm, zoom, hi, cost_axis, cost_diag;
  double m4_lo, m4_hi;        // max_norm^4 * (1 -+ 1e-9): outside this band q decides sqrt(sqrt(q)) > max_norm
  double rzoom;               // RN(1 / zoom)
  int32_t has_coarseness;
};

constexpr int kCovFThreads = 128;

// Host side of every entry point: the kernel's view of the env parameters, derived constants included.  The caller
// sets the state, action and output pointers, n_envs and ld.
inline void coverage_float_args(const SmarlCoverageFloatParams* p, CoverageFloatArgs& a) {
  a = CoverageFloatArgs{};
  a.weights = p->weights; a.size = (double)p->size; a.fieldview = p->fieldview; a.max_norm = p->max_norm;
  a.zoom = p->zoom; a.hi = p->hi; a.cost_axis = p->cost_axis; a.cost_diag = p->cost_diag;
  a.has_coarseness = p->has_coarseness;
  const double m4 = (a.max_norm * a.max_norm) * (a.max_norm * a.max_norm);
  a.m4_lo = m4 * (1.0 - 1e-9);
  a.m4_hi = m4 * (1.0 + 1e-9);
  a.rzoom = 1.0 / a.zoom;
}

// x / zoom, correctly rounded, for the kernel-invariant divisor zoom with rzoom = RN(1 / zoom) from the host: a
// multiply and two exact-residual corrections (5 instructions) instead of the ~45 of a float64 division, of which
// CoverageDiscretized.transition needs two per agent-step (coverage.py:230).  q1 is a faithful quotient, and a faithful
// quotient corrected once through the exact FMA residual with a correctly rounded reciprocal IS the rounded quotient
// (Markstein); x is 0 or a normal number of magnitude >= ~1e-16 here, so nothing underflows.  tools/div_probe.cu checked
// 3.3e10 operands of exactly this shape against __ddiv_rn bit for bit (profiles/r02/div_probe.txt).
__device__ __forceinline__ double div_by_zoom(double x, double zoom, double rzoom) {
  const double q0 = __dmul_rn(x, rzoom);
  const double q1 = __fma_rn(__fma_rn(-q0, zoom, x), rzoom, q0);
  return __fma_rn(__fma_rn(-q1, zoom, x), rzoom, q1);
}

// One step of one env held in registers: moves every agent by the actions fa (mode 0: dx0, dy0, dx1, ...) or ma
// (mode 1: 0..8), returns the per-agent costs (f64) and the unweighted env reward.
template <int A, int MODE>
__device__ __forceinline__ void coverage_float_env_step_regs(double (&px)[A], double (&py)[A],
    const float (&fa)[MODE == 0 ? 2 * A : 1], const uint32_t (&ma)[MODE == 1 ? A : 1],
    const CoverageFloatArgs& a, double (&cost)[A], double& rew) {
#pragma unroll
  for (int i = 0; i < A; ++i) {
    if (MODE == 0) {                                   // CoverageContinuous.transition, coverage.py:54-74
      double dx = (double)fa[2 * i], dy = (double)fa[2 * i + 1];
      cost[i] = __dsqrt_rn(__fma_rn(dy, dy, __dmul_rn(dx, dx)));       // :94 np.linalg.norm(action)
      if (a.has_coarseness) {
        // :65-69  norm = sqrt(dx^2 + dy^2); if sqrt(norm) > max_norm (sic: sqrt of the norm) rescale.  sqrt_rn is
        // monotonic, so sqrt(sqrt(q)) > max_norm is decided on q outside a 1e-9 band around max_norm^4 and the two
        // square roots are only evaluated for the few actions that are rescaled (or fall inside the band).
        const double q = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
        if (q > a.m4_lo) {
          const double norm = __dsqrt_rn(q);
          if (q > a.m4_hi || __dsqrt_rn(norm) > a.max_norm) {
            dx = __dmul_rn(__ddiv_rn(dx, norm), a.max_norm);
            dy = __dmul_rn(__ddiv_rn(dy, norm), a.max_norm);
          }
        }
      }
      px[i] = fmax(0.0, fmin(a.size, __dadd_rn(px[i], dx)));            // :70
      py[i] = fmax(0.0, fmin(a.size, __dadd_rn(py[i], dy)));
    } else {                                           // CoverageDiscretized.transition, coverage.py:219-234
      const uint32_t m = ma[i];
      // directions (:221): x +1,-1,0,0,+1,+1,-1,-1,0 ; y 0,0,-1,+1,+1,-1,+1,-1,0  -- two bits per action, value + 1
      const int dxi = (int)((0x10A52u >> (2 * m)) & 3u) - 1;
      const int dyi = (int)((0x12285u >> (2 * m)) & 3u) - 1;
      px[i] = div_by_zoom(fmax(0.0, fmin(a.hi, __dadd_rn(__dmul_rn(px[i], a.zoom), (double)dxi))), a.zoom, a.rzoom);   // :230
      py[i] = div_by_zoom(fmax(0.0, fmin(a.hi, __dadd_rn(__dmul_rn(py[i], a.zoom), (double)dyi))), a.zoom, a.rzoom);
      cost[i] = m < 4 ? a.cost_axis : (m < 8 ? a.cost_diag : 0.0);     // :237
    }
  }
  // reward, coverage.py:76-89: i-major sequential f64 sum over overlapping pairs
  rew = 0.0;
#pragma unroll
  for (int i = 0; i < A; ++i) {
#pragma unroll
    for (int j = i + 1; j < A; ++j) {
      const double dx = __dadd_rn(px[j], -px[i]), dy = __dadd_rn(py[j], -py[i]);
      const double gap = __dadd_rn(a.fieldview, -__dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy))));
      if (gap > 0.0) rew = __dadd_rn(rew, -__dmul_rn(gap, gap));
    }
  }
}

// The same, the actions loaded from global memory: `act` points at this env's lane of step t's action rows.
template <int A, int MODE>
__device__ __forceinline__ void coverage_float_env_step(double (&px)[A], double (&py)[A], const void* act, int64_t ld,
                                                        const CoverageFloatArgs& a, double (&cost)[A], double& rew) {
  // all action loads first: issued back to back with the caller's position loads, one memory latency per step
  // instead of one per agent (ncu on the A = 3 step kernel: 6.9 of 13 stall cycles per issue were long_scoreboard)
  float fa[MODE == 0 ? 2 * A : 1];
  uint32_t ma[MODE == 1 ? A : 1];
#pragma unroll
  for (int i = 0; i < A; ++i) {
    if (MODE == 0) {
      fa[2 * i] = static_cast<const float*>(act)[(2 * i) * ld];
      fa[2 * i + 1] = static_cast<const float*>(act)[(2 * i + 1) * ld];
    } else {
      ma[i] = static_cast<const uint8_t*>(act)[i * ld];
    }
  }
  coverage_float_env_step_regs<A, MODE>(px, py, fa, ma, a, cost, rew);
}

struct CoverageFloatRolloutArgs {
  CoverageFloatArgs env;      // env.pos_x/pos_y = start positions (read only), env.actions = [T][rows][ld]
  double* final_x;
  double* final_y;
  float* R;
  float* modR;
  float* C;                   // [A][ld] f32 cost sums
  float* G;
  float* g_scratch;           // [2][T][ld]
  double* partials;
  const double* thresholds;
  double gamma;
  int32_t n_steps;
  int32_t g_mode;
};

// Launchers of mode M (0 = Continuous, 1 = Discretized), in coverage_float.cu
template <int M> int launch_coverage_float_step(int A, const CoverageFloatArgs& a, unsigned grid, cudaStream_t s);
template <int M> int launch_coverage_float_rollout(int A, const CoverageFloatRolloutArgs& a, unsigned grid, cudaStream_t s);

}  // namespace smarl
