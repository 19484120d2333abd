/*
 * smarl.h -- C ABI of the B200-native batched env-step hot path (libsmarl.so).
 *
 * The reference (advilema/safe_multiagent_RL) is pure Python and has no FFI; the
 * boundary it offers for this path is the duck-typed env protocol
 * reset()/step(actions) -> (state, reward, constraint, done) consumed by main.py:28-57,
 * plus MetaAgent.act / Buffer.append / Buffer.step / *.compute_returns.  Each entry
 * point below names the reference function(s) it replaces (paths relative to the
 * reference root).  INTEGRATION.md shows the ctypes binding a maintainer would add.
 *
 * Conventions
 * -----------
 *  - Every pointer is a DEVICE pointer unless the name ends in _h (then pageable or
 *    pinned HOST memory).  The caller owns all buffers; nothing here allocates except
 *    the smarl_host_* staging helpers, which say so.
 *  - All batched arrays are agent-major SoA: element (row r, env e) lives at
 *    base[r * ld + e].  `ld` (row stride in ELEMENTS, shared by every array of a call)
 *    must be a multiple of 16 and >= n_envs; every base pointer must be 16-byte
 *    aligned.  Lanes n_envs..ld-1 of a row are padding: they may be read and written
 *    with garbage, never fault, and never enter a reduction.
 *  - Calls enqueue work on `stream` (a cudaStream_t passed as void*) and return
 *    without synchronising.  They are re-entrant; distinct state buffers may be driven
 *    from different host threads / streams.
 *  - Return value: SMARL_OK or a negative error; smarl_last_error() gives a
 *    thread-local message.  There is no CPU fallback.
 *  - n_agents is limited to 1..32; grid size to 1..127 (Coverage: doubled uint8 coordinates
 *    index the penalty table) and 1..254 (Congestion); per call (2*n_agents+1)*ld < 2^32.
 */
#ifndef SMARL_H_
#define SMARL_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SMARL_ABI_VERSION 2
#define SMARL_MAX_AGENTS 32

enum {
  SMARL_OK = 0,
  SMARL_EINVAL = -1,        /* bad shape / alignment / null pointer */
  SMARL_ECUDA = -2,         /* a CUDA runtime call failed (see smarl_last_error) */
  SMARL_EUNSUPPORTED = -3   /* valid request outside the compiled envelope */
};

typedef void* smarl_stream_t;   /* cudaStream_t */
enum { SMARL_ENV_COVERAGE = 0, SMARL_ENV_CONGESTION = 1, SMARL_ENV_COLLISION = 2, SMARL_KERNEL_POLICY = 3 };

int smarl_abi_version(void);
const char* smarl_last_error(void);
/* SM count and compute capability of the current device. */
int smarl_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* Kernel-variant knob (profiling and tests; results never depend on it).  Large agent counts are served by
 * lane-cooperative kernels that split one env over 2 or 4 lanes of a warp; by default the library picks the
 * measured-fastest mapping per (env kind, n_agents).  lanes: -1 = automatic (default), 0 = one thread per env
 * (Collision) / per four envs (grid envs), 2 or 4 = force the cooperative kernels where they exist (n_agents >= 9).
 * env_kind is SMARL_ENV_COVERAGE / _CONGESTION / _COLLISION.  With env_kind = SMARL_KERNEL_POLICY the knob picks the
 * build of smarl_policy_act_discrete: -1 = automatic (tensor cores), 0 = FP32 pipes only (packed FFMA2), 1 = fc1 on
 * the tensor cores (tcgen05.mma, accumulators in tensor memory) with groups of up to 16 agents per CTA, 2 = the same
 * with groups of up to 8.  smarl_policy_act_discretized has one build (FP32 pipes) and ignores the knob.
 * Process-wide; returns the previous setting. */
int smarl_set_kernel_variant(int32_t env_kind, int32_t lanes);

/* Programmatic dependent launch of the per-step kernels (the *_step and policy_act_* entry points): the next step's
 * CTAs are scheduled while the current kernel drains and block in griddepcontrol.wait until it has completed, which
 * hides most of the kernel-to-kernel launch gap of a closed loop (main.py:28-57 is T x (act, step) on one stream) --
 * in plain streams and inside captured CUDA graphs alike.  Results never depend on it.  On by default (SMARL_PDL=0 in
 * the environment turns it off); process-wide; returns the previous setting. */
int smarl_set_pdl(int32_t on);

/* ------------------------------------------------------------------------------------
 * Grid envs share start/reset: replaces CoverageContinuous.reset/_restart
 * (envs/coverage.py:28-52) and Congestion.reset/_restart (envs/congestion.py:34-47) for
 * shuffle=False: state <- start, and the float observation the policies read
 * (np.array(state).flatten(), main.py:33) is rebuilt.
 *   start_x,start_y,pos_x,pos_y  u8 [A][ld]      obs  f32 [2A][ld] rows x0,y0,x1,y1,... (may be NULL)
 * ---------------------------------------------------------------------------------- */
int smarl_grid_reset(const uint8_t* start_x, const uint8_t* start_y, uint8_t* pos_x,
                     uint8_t* pos_y, float* obs, int32_t n_agents, int64_t n_envs, int64_t ld,
                     smarl_stream_t stream);

/* ------------------------------------------------------------------------------------
 * shuffle=True: per-episode re-randomised starts / landmarks (Agent.reset: envs/coverage.py:266-273,
 * envs/congestion.py:211-217, envs/collision_avoidance.py:178-179; landmarks :100-101).  The reference
 * draws from numpy's global MT19937 stream; here each (x,y) pair comes from Philox4x32-10 with counter
 * (global env id, episode, row) and key seed, as 53-bit uniforms u (numpy's random_sample formula),
 * so draws do not depend on sharding.  Fill the start arrays, then call the env's reset.
 *   kind 0: floor(u*size) u8           kind 1: same, row 0 pinned to (0,0) (Congestion agent 0)
 *   kind 2: u*size f64                 kind 3: floor((u*size)*zoom)/zoom f64 (CoverageDiscretized)
 * The f64 variant addresses row r at x[r*row_stride + e] (row_stride = ld for starts, 2*ld with
 * y = x + ld for Collision's interleaved landmark rows); row_offset separates counter domains.
 * ---------------------------------------------------------------------------------- */
int smarl_random_starts_u8(int32_t kind, int32_t size, uint64_t seed, int64_t episode, int64_t env_offset,
                           uint8_t* start_x, uint8_t* start_y, int32_t n_agents, int64_t n_envs, int64_t ld,
                           smarl_stream_t stream);
int smarl_random_starts_f64(int32_t kind, int32_t size, double zoom, uint64_t seed, int64_t episode,
                            int64_t env_offset, int32_t row_offset, double* x, double* y, int64_t row_stride,
                            int32_t n_rows, int64_t n_envs, smarl_stream_t stream);

/* ------------------------------------------------------------------------------------
 * CoverageDiscrete ("Explore")
 * ---------------------------------------------------------------------------------- */
typedef struct {
  int32_t size;         /* coordinates clamp to [0,size]                 coverage.py:185-186 */
  int32_t n_agents;     /* A; also K = A constraints                     coverage.py:22      */
  int32_t lut_len;      /* penalties for squared distance q >= lut_len are 0                 */
  int32_t reward_rows;  /* step only: 0 (= A) per-agent weighted rewards [A][ld]; 1: ONE row with the
                           unweighted env reward -- reward_a = w_a * rew is linear, so the accounting
                           (smarl_rollout_returns_shared) can apply the weights; saves 4 - 4/A B per
                           agent-step of HBM traffic                                              */
  const float* lut;     /* [lut_len] pen(q) = (fv - sqrt(q))^2 if sqrt(q) < fv else 0, f32
                           rounding of the reference's f64 value         coverage.py:80-83   */
  const float* weights; /* [A] per-agent reward weight, NULL = 1         coverage.py:86-87   */
} SmarlCoverageParams;

/* One CoverageDiscrete.step (coverage.py:100-106 = transition :174-189 + reward :76-89 +
 * constraint :191-196 + check_done :97-98) for n_envs environments, with MetaAgent.act's
 * penalty <lambda, c> (safe_multi_agent_RL/meta_agent.py:21-22) fused in.
 *   pos_x,pos_y u8 [A][ld] in/out     actions u8 [A][ld] in 0..4
 *   obs     f32 [2A][ld]  out, NULL to skip
 *   reward  f32 [A][ld]   out   w_a * -(sum of pair penalties)   ([1][ld] unweighted if p->reward_rows == 1)
 *   cost    u8  [A][ld]   out   1 for a non-stay action
 *   done    u8  [A][ld]   out, NULL to skip (always 0 for Coverage)
 *   lambdas f64 [A]  in, penalty f32 [ld] out = sum_k lambda_k c_k; both NULL to skip
 * For a rollout buffer pass reward/cost/done/penalty offset to step t's slab. */
int smarl_coverage_step(const SmarlCoverageParams* p, uint8_t* pos_x, uint8_t* pos_y,
                        const uint8_t* actions, float* obs, float* reward, uint8_t* cost,
                        uint8_t* done, const double* lambdas, float* penalty, int64_t n_envs,
                        int64_t ld, smarl_stream_t stream);

/* Parameters of the per-episode accounting shared by every *_rollout / returns call. */
typedef struct {
  double gamma;           /* discount                              buffer.py:31             */
  int32_t n_steps;        /* T = max_t                             main.py:29               */
  int32_t g_mode;         /* what G holds: 0 none, 1 reward-to-go G_t = m_t + gamma G_{t+1}
                             (ACAgent.compute_returns agent.py:200-206), 2 gamma^t m_t
                             (AbstractAgent.compute_returns agent.py:129-132), 3 (returns kernel
                             only) PPO's per-episode standardisation of mode 1,
                             (G - mean) / (std_unbiased + 1e-7) over the episode's steps
                             (PPOAgent.step agent.py:276-281; PPOAgent extends ACAgent)     */
  const double* thresholds; /* [K] device, for violation counts; NULL = skip  buffer.py:47  */
} SmarlAccounting;

/* Number of f64 slots in a stats vector for (A agents, K constraints):
 *   [0,K) sum_e C_k   [K,2K) #{e : C_k > thr_k}   [2K,2K+A) sum_e R_a
 *   [2K+A,2K+2A) sum_e modR_a   [2K+2A] episode count. */
int32_t smarl_stats_len(int32_t n_agents, int32_t n_constraints);
/* Scratch (in f64 elements) the accounting kernels need for deterministic block partials. */
int64_t smarl_stats_scratch_len(int32_t n_agents, int32_t n_constraints, int64_t n_envs);

/* Whole open-loop episode in one launch: reset + T x (step + MetaAgent.act) + Buffer.step
 * + compute_returns, state register-resident (main.py:28-57 without the policy nets).
 *   start_x,start_y u8 [A][ld]     actions u8 [T][A][ld]     lambdas f64 [A] (NULL = 0)
 *   final_x,final_y u8 [A][ld] out (NULL to skip)
 *   R, modR f32 [A][ld] out        C i32 [A][ld] out
 *   G f32 [T][A][ld] out if acc->g_mode != 0    g_scratch f32 [2][T][ld] then required
 *   stats f64 [smarl_stats_len] out (NULL to skip), stats_scratch f64 [smarl_stats_scratch_len] */
int smarl_coverage_rollout(const SmarlCoverageParams* p, const SmarlAccounting* acc,
                           const uint8_t* start_x, const uint8_t* start_y,
                           const uint8_t* actions, const double* lambdas, uint8_t* final_x,
                           uint8_t* final_y, float* R, float* modR, int32_t* C, float* G,
                           float* g_scratch, double* stats, double* stats_scratch,
                           int64_t n_envs, int64_t ld, smarl_stream_t stream);

/* ------------------------------------------------------------------------------------
 * CoverageContinuous / CoverageDiscretized (float64 positions; the "ExploreContinuous" family the
 * paper's launchers use, experiments_run/AC_explore_constr_1.bat)
 * ---------------------------------------------------------------------------------- */
typedef struct {
  int32_t size;           /* positions clamp to [0,size]                       coverage.py:70-71    */
  int32_t n_agents;       /* A; K = A float costs                              coverage.py:22       */
  int32_t mode;           /* 0 CoverageContinuous (:54-74,:91-95), 1 CoverageDiscretized (:219-241) */
  int32_t has_coarseness; /* mode 0: rescale long moves (:64-69)                                    */
  double fieldview;       /* fv = size / sqrt(A) unless overridden             coverage.py:15-18    */
  double max_norm;        /* mode 0: sqrt(2)*size/coarseness                   coverage.py:66       */
  double zoom;            /* mode 1: coarseness/size                           coverage.py:215      */
  double hi;              /* mode 1: size*zoom                                 coverage.py:230      */
  double cost_axis;       /* mode 1: 1*(size/coarseness)                       coverage.py:237      */
  double cost_diag;       /* mode 1: sqrt(2)*(size/coarseness)                                      */
  const float* weights;   /* [A] or NULL                                       coverage.py:86-87    */
} SmarlCoverageFloatParams;

/* state <- start (f64 [A][ld]) and obs rebuild, for the float-position Coverage envs
 * (CoverageContinuous.reset/_restart, coverage.py:28-52). */
int smarl_coverage_float_reset(const double* start_x, const double* start_y, double* pos_x,
                               double* pos_y, float* obs, int32_t n_agents, int64_t n_envs,
                               int64_t ld, smarl_stream_t stream);

/* One CoverageContinuous.step / CoverageDiscretized.step (coverage.py:100-106) + MetaAgent.act.
 *   pos_x,pos_y f64 [A][ld] in/out
 *   actions: mode 0 f32 [2A][ld] rows dx0,dy0,dx1,...; mode 1 u8 [A][ld] in 0..8
 *   obs f32 [2A][ld], reward f32 [A][ld], cost f32 [A][ld] (norm of the action / lattice step length),
 *   done u8 [A][ld] (NULL ok, always 0), lambdas f64 [A] + penalty f32 [ld] (both NULL to skip) */
int smarl_coverage_float_step(const SmarlCoverageFloatParams* p, double* pos_x, double* pos_y,
                              const void* actions, float* obs, float* reward, float* cost,
                              uint8_t* done, const double* lambdas, float* penalty, int64_t n_envs,
                              int64_t ld, smarl_stream_t stream);

/* Fused open-loop episode of the float-position Coverage envs (as smarl_coverage_rollout).
 *   start_x,start_y f64 [A][ld]; actions f32 [T][2A][ld] (mode 0) or u8 [T][A][ld] (mode 1)
 *   final_x,final_y f64 [A][ld] (NULL ok); R, modR f32 [A][ld]; C f32 [A][ld] (float cost sums);
 *   G f32 [T][A][ld] per g_mode (0..2); g_scratch f32 [2][T][ld] for g_mode 1. */
int smarl_coverage_float_rollout(const SmarlCoverageFloatParams* p, const SmarlAccounting* acc,
                                 const double* start_x, const double* start_y, const void* actions,
                                 const double* lambdas, double* final_x, double* final_y, float* R, float* modR,
                                 float* C, float* G, float* g_scratch, double* stats, double* stats_scratch,
                                 int64_t n_envs, int64_t ld, smarl_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Congestion
 * ---------------------------------------------------------------------------------- */
typedef struct {
  int32_t size;          /* coordinates clamp to [0,size]                 congestion.py:70-71 */
  int32_t n_agents;      /* A; K = 1                                      congestion.py:26    */
  const double* demand;  /* [(size+1)*(size+1)] row-major [x][y], f64     congestion.py:28,86 */
  /* action noise (congestion.py:64-67): move = a if u1 < 1-noise else int(u2*5)              */
  int32_t noise_mode;    /* 0 = none, 1 = recorded effective moves, 2 = on-device Philox      */
  uint32_t episode;      /* mode 2: episode index mixed into the Philox counter (low 29 bits), so that every
                            episode draws fresh noise like the reference's random(); see episode_dev   */
  uint64_t keep_threshold; /* mode 2: keep action iff w < keep_threshold, = ceil((1-noise)*2^32);
                              otherwise the move is w mod 5 (w = word a&3 of the Philox output)    */
  uint64_t seed;         /* mode 2: Philox4x32-10 key                                         */
  int64_t env_offset;    /* mode 2: global id of env 0 (counter = (id, t, agent>>2 | episode<<3)), so the
                            stream does not depend on how envs are sharded over GPUs          */
  const float* wait_reward; /* optional [A][(size+1)^2]: f32(-30*(con+1)/demand[x][y] + 7.5 - 4) for
                            con = 0..A-1, i.e. the waiting-branch reward (congestion.py:86-87)
                            evaluated in f64 on the host and rounded once; replaces a float64
                            division per agent-step in the kernels.  NULL = compute from demand.  */
  const uint32_t* episode_dev; /* optional DEVICE scalar added to `episode` when the kernel runs: lets a captured
                            CUDA graph draw fresh noise on every replay (bump it between replays).  NULL = 0;
                            must be NULL in the smarl_host_* calls.                                    */
} SmarlCongestionParams;

/* One Congestion.step (congestion.py:106-111 = transition :49-75 + reward :77-90 with
 * _congestions :113-137 + constraint :93-100 + check_done :103-104) with MetaAgent.act fused.
 *   pos_x,pos_y u8 [A][ld] in/out    actions u8 [A][ld] intended 0..4
 *   moves u8 [A][ld]: noise_mode 1 in (recorded), else NULL or out (the effective move taken)
 *   obs f32 [2A][ld], reward f32 [A][ld], cost i32 [ld], done u8 [A][ld] (NULL ok)
 *   lambdas f64 [1], penalty f32 [ld];  t = step index (Philox counter). */
int smarl_congestion_step(const SmarlCongestionParams* p, uint8_t* pos_x, uint8_t* pos_y,
                          const uint8_t* actions, uint8_t* moves, float* obs, float* reward,
                          int32_t* cost, uint8_t* done, const double* lambdas, float* penalty,
                          int32_t t, int64_t n_envs, int64_t ld, smarl_stream_t stream);

/* Fused open-loop episode, as smarl_coverage_rollout.  moves u8 [T][A][ld] (mode 1) or NULL.
 * C i32 [1][ld]. */
int smarl_congestion_rollout(const SmarlCongestionParams* p, const SmarlAccounting* acc,
                             const uint8_t* start_x, const uint8_t* start_y,
                             const uint8_t* actions, const uint8_t* moves,
                             const double* lambdas, uint8_t* final_x, uint8_t* final_y, float* R,
                             float* modR, int32_t* C, float* G, float* g_scratch, double* stats,
                             double* stats_scratch, int64_t n_envs, int64_t ld,
                             smarl_stream_t stream);

/* ------------------------------------------------------------------------------------
 * CollisionAvoidance (continuous, float64 state)
 * ---------------------------------------------------------------------------------- */
typedef struct {
  int32_t size;          /* positions clamp to [0,size]          collision_avoidance.py:118-119 */
  int32_t n_agents;      /* A; K = 1                             collision_avoidance.py:69      */
  int32_t n_landmarks;   /* L >= 1                               collision_avoidance.py:62,101  */
  int32_t obs_landmarks; /* 1: obs has 2L extra rows (shuffle=True layout, :65-68,:141-142)    */
  double agents_size;    /* 0.25: reach radius, 2x = collision distance   :49,:123,:155        */
  int32_t normalize_state; /* 1: obs = state / size (_normalize_state, :87-88,:146-147,:164-165)  */
  int32_t reward_rows;     /* step only: 0 (= A) identical per-agent rows (:130); 1: one row [1][ld]
                              for smarl_rollout_returns_shared                                    */
} SmarlCollisionParams;

/* CollisionAvoidance.reset/_restart (:72-98) for shuffle=False: state <- start, done <- 0.
 *   start_x,start_y,pos_x,pos_y f64 [A][ld]   done u8 [A][ld]   landmarks f64 [2L][ld] rows
 *   lx0,ly0,lx1,...   obs f32 [2A(+2L)][ld] (NULL ok) */
int smarl_collision_reset(const SmarlCollisionParams* p, const double* start_x,
                          const double* start_y, const double* landmarks, double* pos_x,
                          double* pos_y, uint8_t* done, int32_t* episode_len, float* obs, int64_t n_envs,
                          int64_t ld, smarl_stream_t stream);

/* One CollisionAvoidance.step (:139-148 = transition :103-125 + reward :127-130/:158-162 +
 * constraint :132-133/:150-156 + check_done :135-136) with MetaAgent.act fused.  Envs whose
 * agents were all done before the call are past their episode end (main.py:51): frozen,
 * reward/cost/penalty 0.
 *   pos_x,pos_y f64 [A][ld] in/out   done u8 [A][ld] in/out
 *   actions f32 [2A][ld] rows dx0,dy0,dx1,... (the reference's policies emit fp32, agent.py:124-125)
 *   landmarks f64 [2L][ld]   obs f32 [2A(+2L)][ld]   reward f32 [A][ld]   cost i32 [ld]
 *   done_out u8 [A][ld]: this step's done flags for a rollout buffer (NULL ok)
 *   episode_len i32 [ld] in/out (NULL ok): incremented for envs that were still running (reset zeroes it) */
int smarl_collision_step(const SmarlCollisionParams* p, double* pos_x, double* pos_y,
                         uint8_t* done, const float* actions, const double* landmarks, float* obs,
                         float* reward, int32_t* cost, uint8_t* done_out, int32_t* episode_len,
                         const double* lambdas, float* penalty, int64_t n_envs, int64_t ld,
                         smarl_stream_t stream);

/* Fused open-loop episode.  actions f32 [T][2A][ld].  n_active i32 [ld] out = episode length
 * T' (steps until all agents done, NULL ok).  C i32 [1][ld]. */
int smarl_collision_rollout(const SmarlCollisionParams* p, const SmarlAccounting* acc,
                            const double* start_x, const double* start_y, const double* landmarks,
                            const float* actions, const double* lambdas, double* final_x,
                            double* final_y, uint8_t* final_done, int32_t* n_active, float* R,
                            float* modR, int32_t* C, float* G, float* g_scratch, double* stats,
                            double* stats_scratch, int64_t n_envs, int64_t ld,
                            smarl_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Rollout accounting over a device rollout buffer filled by the *_step calls
 * (closed-loop mode: a policy chooses actions between steps).
 * ---------------------------------------------------------------------------------- */
enum { SMARL_COST_U8 = 0, SMARL_COST_I32 = 1, SMARL_COST_F32 = 2 };   /* F32: C is written as f32 */

/* MetaAgent.act's penalty for rewards/costs that did not come from a *_step call
 * (meta_agent.py:21-22): penalty[t][e] = sum_k lambda_k cost[t][k][e].
 *   cost [T][K][ld] u8, i32 or f32, lambdas f64 [K], penalty f32 [T][ld] */
int smarl_rollout_penalty(const void* cost, int32_t cost_dtype, const double* lambdas,
                          float* penalty, int32_t n_constraints, int32_t n_steps, int64_t n_envs,
                          int64_t ld, smarl_stream_t stream);

/* Buffer.step (safe_multi_agent_RL/buffer.py:30-39), MetaAgent.step (meta_agent.py:25-30)
 * and compute_returns (agent.py:129-132, :200-206) for n_envs episodes at once:
 *   R_a = sum_t gamma^t r[t,a]   modR_a = sum_t gamma^t (r[t,a] - pen[t])   C_k = sum_t c[t,k]
 *   reward f32 [T][A][ld]   cost [T][K][ld]   penalty f32 [T][ld] (NULL = 0)
 *   n_active i32 [ld]: episode lengths T' (NULL = T); only g_mode 3 needs them (steps >= T' get 0)
 *   R, modR f32 [A][ld]     C i32 [K][ld]     G f32 [T][A][ld] per acc->g_mode
 *   stats/stats_scratch as above (NULL to skip). */
int smarl_rollout_returns(const SmarlAccounting* acc, const float* reward, const void* cost,
                          int32_t cost_dtype, const float* penalty, const int32_t* n_active, float* R,
                          float* modR, int32_t* C, float* G, double* stats, double* stats_scratch,
                          int32_t n_agents, int32_t n_constraints, int64_t n_envs, int64_t ld,
                          smarl_stream_t stream);

/* Same accounting for a rollout buffer that stores ONE reward row per env and step (Coverage with
 * reward_rows = 1; Collision, whose reward is identical for all agents): reward_a[t] = w_a * reward_env[t].
 *   reward_env f32 [T][ld]   weights f32 [A] (NULL = 1)   everything else as smarl_rollout_returns
 *   (g_mode 0..3; n_active i32 [ld] episode lengths, NULL = T, honoured by g_mode 3 exactly as there).
 *   Reads 8/A instead of 4 + 4/A reward/penalty bytes per agent-step. */
int smarl_rollout_returns_shared(const SmarlAccounting* acc, const float* reward_env, const float* weights,
                                 const void* cost, int32_t cost_dtype, const float* penalty,
                                 const int32_t* n_active, float* R,
                                 float* modR, int32_t* C, float* G, double* stats, double* stats_scratch,
                                 int32_t n_agents, int32_t n_constraints, int64_t n_envs, int64_t ld,
                                 smarl_stream_t stream);

/* MetaAgent.update (meta_agent.py:32-39, leq=True) from an (all-reduced) stats vector:
 *   lambda_k <- max(0, lambda_k + lr * (stats[k] / stats[count] - thr_k)).
 * stats may be the sum of several GPUs' / rollouts' vectors (every slot is additive). */
int smarl_lambda_update(double* lambdas, const double* stats, const double* thresholds, double lr,
                        int32_t n_agents, int32_t n_constraints, smarl_stream_t stream);

/* ------------------------------------------------------------------------------------
 * The caller of the env step: the reference's per-agent discrete policies, fused for all envs and agents.
 * DiscretePolicy (safe_multi_agent_RL/agent.py:23-47): fc1 = Linear(state_space, 16), relu, fc2 = Linear(16, action_space),
 * softmax, Categorical.sample / log_prob; one network per agent, each fed the joint state
 * np.array(state).flatten() = (x0, y0, x1, y1, ...) (main.py:30-35, AbstractAgent.act agent.py:118-127).
 * For the grid envs (CoverageDiscrete, Congestion: state_space = 2 n_agents, action_space = 5) the kernel reads the
 * u8 position rows the step kernels maintain -- so the step may run with obs = NULL -- and writes the u8 action row
 * the step consumes plus the f32 log-probability of the sampled action.
 *   w1 f32 [A][2A][16] (fc1.weight transposed: [in][out]), b1 f32 [A][16], w2 f32 [A][16][5], b2 f32 [A][5]: DEVICE
 *   pos_x,pos_y u8 [A][ld] in    actions u8 [A][ld] out    logp f32 [A][ld] out (NULL to skip)
 * Sampling: Philox4x32-10, counter (global env id lo, hi, t | episode << 16, agent >> 2 | (episode >> 16) << 3), key
 * seed ^ "PLCY" (hi word), episode = p->episode + *p->episode_dev: one block serves four consecutive agents, agent a
 * takes word w[a & 3]; u = min(fl32((w >> 8) + 0.5) * 2^-24, 1 - 2^-24) (the float32 sum rounds to 2^24 for the top
 * word; the clamp keeps u * sum below sum, so an action of probability 0 is never drawn);
 * action = #{c < 4 : sum_{c' <= c} e_c' <= u * sum e}, e_c = exp(logit_c - max).
 * Streams depend on the global env id, not on sharding or on the kernel build.  t in 0..65535.
 * Two builds (smarl_set_kernel_variant(SMARL_KERNEL_POLICY, ...)): all multiply-adds on the FP32 pipes, or fc1 as one
 * tcgen05 GEMM per 128-env tile (bf16 positions are exact, every fp32 weight enters as three bf16 pieces, f32
 * accumulation in tensor memory); log-probabilities of the two agree to ~1e-6.
 * ---------------------------------------------------------------------------------- */
typedef struct {
  int32_t n_agents;        /* A; the observation has 2A components                                   */
  int32_t hidden;          /* 16 (agent.py:24)                                                       */
  int32_t n_actions;       /* 5  (env.action_space of the grid envs)                                 */
  uint32_t episode;        /* mixed into the Philox counter (all 32 bits) so that episodes draw independent samples */
  const float* w1;
  const float* b1;
  const float* w2;
  const float* b2;
  uint64_t seed;
  int64_t env_offset;      /* global id of env 0 (sharding)                                          */
  const uint32_t* episode_dev; /* optional device scalar added to `episode` (CUDA-graph replays); NULL = 0 */
} SmarlDiscretePolicy;
int smarl_policy_act_discrete(const SmarlDiscretePolicy* p, const uint8_t* pos_x, const uint8_t* pos_y,
                              uint8_t* actions, float* logp, int32_t t, int64_t n_envs, int64_t ld,
                              smarl_stream_t stream);

/* The same for the continuous envs: ContinuousPolicy (safe_multi_agent_RL/agent.py:48-76): fc1 = Linear(state_space, 16),
 * relu, mu = fc2 (2 outputs), sigma^2 = relu(fc2_) + 1e-4, action ~ MultivariateNormal(mu, diag(sigma^2)), log_prob of
 * it; one network per agent, each fed the joint state (main.py:30-35).  The kernel reads the f32 observation rows the
 * step / reset kernels maintain and writes the f32 action rows the step consumes plus the log-probabilities.
 *   w1 f32 [A][S][16] ([in][out]), b1 [A][16], w_mu / w_var f32 [A][16][2], b_mu / b_var [A][2]: DEVICE
 *   obs f32 [S][ld] in    actions f32 [2A][ld] out (rows dx0, dy0, dx1, ...)    logp f32 [A][ld] out (NULL to skip)
 * Sampling: Philox4x32-10, counter (global env id lo, hi, t | episode << 16, agent >> 1 | (episode >> 16) << 4), key
 * seed ^ "GAUS" (hi word), episode = p->episode + *p->episode_dev (all 32 bits): one block serves two agents, agent a takes w[2 (a & 1)], w[2 (a & 1) + 1]; u_k = ((w_k >> 9) + 0.5) * 2^-23;
 * Box-Muller r = sqrt(-2 ln u_0), z = (r cos 2 pi u_1, r sin 2 pi u_1); action_k = mu_k + sigma_k z_k;
 * log_prob = -1/2 sum_k ((action_k - mu_k)^2 / sigma_k^2 + ln sigma_k^2) - ln 2 pi.  t in 0..65535. */
typedef struct {
  int32_t n_agents;        /* A                                                                      */
  int32_t state_size;      /* S = env.state_space: 2A, or 2A + 2L with shuffled landmarks (Collision) */
  int32_t hidden;          /* 16 (agent.py:49)                                                       */
  int32_t n_actions;       /* 2  (env.action_space of the continuous envs)                           */
  uint32_t episode;
  int32_t reserved;
  const float* w1;
  const float* b1;
  const float* w_mu;
  const float* b_mu;
  const float* w_var;
  const float* b_var;
  uint64_t seed;
  int64_t env_offset;
  const uint32_t* episode_dev;
} SmarlGaussianPolicy;
int smarl_policy_act_gaussian(const SmarlGaussianPolicy* p, const float* obs, float* actions, float* logp, int32_t t,
                              int64_t n_envs, int64_t ld, smarl_stream_t stream);

/* The DiscretePolicy (agent.py:23-47) of CoverageDiscretized (9 actions, coverage.py:210-241), whose positions are f64
 * multiples of 1 / zoom rather than u8 cells: the kernel reads the f32 observation rows the reset / step kernels
 * maintain (as smarl_policy_act_gaussian) and writes the u8 action row the step consumes plus the log-probabilities.
 *   w1 f32 [A][2A][16] ([in][out]), b1 [A][16], w2 f32 [A][16][9], b2 [A][9]: DEVICE
 *   obs f32 [2A][ld] in    actions u8 [A][ld] out    logp f32 [A][ld] out (NULL to skip)
 *   p->n_agents in 1..32, hidden 16, n_actions 9; t in 0..65535; obs, actions and logp 16-byte aligned
 * Sampling: smarl_policy_act_discrete's Philox stream and inverse-CDF head over the 9 actions
 * (action = #{c < 8 : sum_{c' <= c} e_c' <= u * sum e}).  One build, all multiply-adds on the FP32 pipes
 * (smarl_set_kernel_variant(SMARL_KERNEL_POLICY, ...) does not apply): h = b1, then fma(x_k, w1[k], h) for
 * k = 0..2A-1; logits2 = log2(e) b2, then fma(relu(h_u), log2(e) w2[u], logits2) for u = 0..15. */
int smarl_policy_act_discretized(const SmarlDiscretePolicy* p, const float* obs, uint8_t* actions, float* logp,
                                 int32_t t, int64_t n_envs, int64_t ld, smarl_stream_t stream);

/* REINFORCE / actor loss of the DiscretePolicy (agent.py:23-47, loss agent.py:134-157) over recorded episodes, and
 * its gradients with respect to every agent's fc1 / fc2, in one kernel.  For every agent a, step t < n_steps and env
 * e < n_envs, with x = obs_rec[t][:, e] (2A floats), c = actions[t][a][e] and psi = psi[t][a][e]:
 *   h = b1 + W1^T x,  r = relu(h),  l = b2 + W2^T r,  p = softmax(l)
 *   loss += -scale psi log p_c
 *   g_l = -scale psi (onehot(c) - p);   dW2 += r (x) g_l,  db2 += g_l
 *   g_h = (W2 g_l) * [h > 0];           dW1 += x (x) g_h,  db1 += g_h   (zero gradient at h == 0, as torch's relu)
 *   p: n_agents 1..32, hidden 16, n_actions 5 or 9, weights w1 [A][2A][16], b1 [A][16], w2 [A][16][NA], b2 [A][NA]
 *      (DEVICE; seed, episode, episode_dev and env_offset are ignored)
 *   obs_rec f32 [T][2A][ld], actions u8 [T][A][ld], psi f32 [T][A][ld]: what the on-policy rollouts record; 16-byte
 *      aligned.  Only env columns e < n_envs are read.  An action >= NA is a caller error: its sample's contribution is
 *      unspecified, but nothing is read or written out of bounds.
 *   dw1, db1, dw2, db2 f32 out, the layouts of the weights (overwritten, not accumulated); loss f64 [1] out (NULL = skip)
 *   scratch f64 [smarl_policy_grad_scratch_len(A, NA, T, n_envs)], DEVICE, caller-owned (its contents are overwritten)
 * Deterministic: no floating-point atomics; tile partials are f32 over at most 256 samples, the sums across tiles and
 * CTAs are f64 in a fixed order, and the number of partials depends on (A, T, n_envs) only, so the result bits depend
 * on the inputs and the shape, not on the device, the stream or earlier launches.  Computed in f32 with exact expf /
 * logf; scale is applied in f64 at the end.  A 132-byte memset of the scratch's counters precedes the kernel (both are
 * stream-ordered and CUDA-graph capturable).  Scratch is 64 + A * P * (32A + 17 NA + 17) doubles with
 * P = min(T * ceil(n_envs / 256), max(1, 1184 / A)): 11.3 MB at A = 32, NA = 9, T = 50, 2^20 envs.
 * smarl_policy_grad_scratch_len returns -1 for arguments the entry point rejects (n_agents, n_actions, n_steps,
 * n_envs < 1). */
int64_t smarl_policy_grad_scratch_len(int32_t n_agents, int32_t n_actions, int32_t n_steps, int64_t n_envs);
int smarl_policy_grad_discrete(const SmarlDiscretePolicy* p, const float* obs_rec, const uint8_t* actions,
                               const float* psi, int32_t n_steps, double scale, float* dw1, float* db1, float* dw2,
                               float* db2, double* loss, double* scratch, int64_t n_envs, int64_t ld,
                               smarl_stream_t stream);

/* Whole ON-POLICY CollisionAvoidance episodes in one launch: main.py:28-57 with the policies inside, i.e. per step
 * every agent's ContinuousPolicy (agent.py:48-76) on the current observation, the sample, CollisionAvoidance.step,
 * MetaAgent.act, and Buffer.step + compute_returns as in smarl_collision_rollout.  Bit-identical to the closed loop
 * reset + T x (smarl_policy_act_gaussian(t) + smarl_collision_step) on the same starts, weights and stream; actions
 * and log-probabilities are sampled for every (t, agent, env), also for done agents and envs past their episode end.
 *   p, acc, start_x .. lambdas and final_x .. stats_scratch as in smarl_collision_rollout (acc->g_mode 0..2)
 *   pol: weights, seed, episode, episode_dev and env_offset as in smarl_policy_act_gaussian;
 *        pol->state_size = 2A (+ 2L with p->obs_landmarks), hidden 16, 2 actions
 *   obs_rec f32 [T][S][ld]  the observation the policy saw at step t      (NULL = skip)
 *   actions f32 [T][2A][ld] the sampled rows dx0, dy0, dx1, ... (smarl_collision_rollout's layout; NULL = skip)
 *   logp    f32 [T][A][ld]  log N(action; mu, sigma^2)                    (NULL = skip)
 * A in 1..8 (one thread per env; A >= 9 returns SMARL_EUNSUPPORTED), T in 1..65536 (16 bits of the Philox counter). */
int smarl_collision_policy_rollout(const SmarlCollisionParams* p, const SmarlGaussianPolicy* pol,
                                   const SmarlAccounting* acc, const double* start_x, const double* start_y,
                                   const double* landmarks, const double* lambdas, float* obs_rec, float* actions,
                                   float* logp, double* final_x, double* final_y, uint8_t* final_done,
                                   int32_t* n_active, float* R, float* modR, int32_t* C, float* G, float* g_scratch,
                                   double* stats, double* stats_scratch, int64_t n_envs, int64_t ld,
                                   smarl_stream_t stream);

/* Whole ON-POLICY CoverageContinuous episodes in one launch: main.py:28-57 with the policies inside, i.e. per step
 * every agent's ContinuousPolicy (agent.py:48-76) on the current observation (x0, y0, x1, ...: what the reset / step
 * kernels write to env.obs), the sample, CoverageContinuous.step, MetaAgent.act, and Buffer.step + compute_returns as in
 * smarl_coverage_float_rollout.  Records and final positions are bit-identical to the closed loop reset +
 * T x (smarl_policy_act_gaussian(t) + smarl_coverage_float_step) on the same starts, weights and stream; the products
 * are bit-identical to smarl_coverage_float_rollout fed the recorded actions (the closed loop's returns kernel sums the
 * f32-rounded rewards, so its R, modR and C agree to ~1e-6 relative).
 *   p (mode 0), acc, start_x .. lambdas and final_x .. stats_scratch as in smarl_coverage_float_rollout (acc->g_mode 0..2)
 *   pol: weights, seed, episode, episode_dev and env_offset as in smarl_policy_act_gaussian;
 *        pol->state_size = 2A, hidden 16, 2 actions
 *   obs_rec f32 [T][2A][ld] the observation the policy saw at step t      (NULL = skip)
 *   actions f32 [T][2A][ld] the sampled rows dx0, dy0, dx1, ... (smarl_coverage_float_rollout's layout; NULL = skip)
 *   logp    f32 [T][A][ld]  log N(action; mu, sigma^2)                    (NULL = skip)
 * A in 1..8 (one thread per env; A >= 9 or mode 1 returns SMARL_EUNSUPPORTED), T in 1..65536 (16 bits of the Philox
 * counter). */
int smarl_coverage_float_policy_rollout(const SmarlCoverageFloatParams* p, const SmarlGaussianPolicy* pol,
                                        const SmarlAccounting* acc, const double* start_x, const double* start_y,
                                        const double* lambdas, float* obs_rec, float* actions, float* logp,
                                        double* final_x, double* final_y, float* R, float* modR, float* C, float* G,
                                        float* g_scratch, double* stats, double* stats_scratch, int64_t n_envs,
                                        int64_t ld, smarl_stream_t stream);

/* Whole ON-POLICY CoverageDiscrete episodes in one launch: main.py:28-57 with the policies inside, i.e. per step
 * every agent's DiscretePolicy (agent.py:23-47) on the joint state (x0, y0, x1, ...: what the reset / step kernels write
 * to env.obs), the sample, CoverageDiscrete.step, MetaAgent.act, and Buffer.step + compute_returns as in
 * smarl_coverage_rollout.  Records and final positions are bit-identical to the closed loop reset +
 * T x (smarl_policy_act_discrete(t) + smarl_coverage_step) on the same starts, weights and stream with the FP32-pipe
 * policy build (smarl_set_kernel_variant(SMARL_KERNEL_POLICY, 0)); the default tensor-core build agrees on all but a few
 * samples in 10^4, and an episode diverges from the step where one sample differs.  The products are bit-identical to
 * smarl_coverage_rollout fed the recorded actions (the closed loop's returns kernel sums the f32-rounded rewards, so its
 * R, modR and stats agree to 1e-5 relative and C is equal).
 *   p, acc, start_x .. lambdas and final_x .. stats_scratch as in smarl_coverage_rollout (acc->g_mode 0..2)
 *   pol: weights, seed, episode, episode_dev and env_offset as in smarl_policy_act_discrete;
 *        pol->n_agents = p->n_agents, hidden 16, 5 actions
 *   obs_rec f32 [T][2A][ld] the observation the policy saw at step t      (NULL = skip)
 *   actions u8  [T][A][ld]  the sampled actions (smarl_coverage_rollout's layout; NULL = skip)
 *   logp    f32 [T][A][ld]  log-probability of the sampled action        (NULL = skip)
 * A in 1..8 (one thread per four envs; A >= 9 returns SMARL_EUNSUPPORTED), T in 1..255 (byte cost counters). */
int smarl_coverage_policy_rollout(const SmarlCoverageParams* p, const SmarlDiscretePolicy* pol,
                                  const SmarlAccounting* acc, const uint8_t* start_x, const uint8_t* start_y,
                                  const double* lambdas, float* obs_rec, uint8_t* actions, float* logp,
                                  uint8_t* final_x, uint8_t* final_y, float* R, float* modR, int32_t* C, float* G,
                                  float* g_scratch, double* stats, double* stats_scratch, int64_t n_envs, int64_t ld,
                                  smarl_stream_t stream);

/* Whole ON-POLICY Congestion episodes in one launch: main.py:28-57 with the policies inside, i.e. per step every agent's
 * DiscretePolicy (agent.py:23-47) on the joint state (x0, y0, x1, ...: what the reset / step kernels write to env.obs),
 * the sample, Congestion.step with its action noise, MetaAgent.act, and Buffer.step + compute_returns as in
 * smarl_congestion_rollout.  Records and final positions are bit-identical to the closed loop reset +
 * T x (smarl_policy_act_discrete(t) + smarl_congestion_step(t)) on the same starts, weights, policy stream and noise
 * episode with the FP32-pipe policy build (smarl_set_kernel_variant(SMARL_KERNEL_POLICY, 0)); the default tensor-core
 * build agrees on all but a few samples in 10^4, and an episode diverges from the step where one sample differs.  The
 * products are bit-identical to smarl_congestion_rollout fed the recorded actions with the same noise episode (the
 * closed loop's returns kernel sums the f32-rounded rewards, so its R, modR and stats agree to 1e-5 relative and C is
 * equal).
 *   p (noise_mode 0 or 2), acc, start_x .. lambdas and final_x .. stats_scratch as in smarl_congestion_rollout
 *   (acc->g_mode 0..2; g_scratch [T][ld] with g_mode 1)
 *   pol: weights, seed, episode, episode_dev and env_offset as in smarl_policy_act_discrete;
 *        pol->n_agents = p->n_agents, hidden 16, 5 actions
 *   obs_rec f32 [T][2A][ld] the observation the policy saw at step t      (NULL = skip)
 *   actions u8  [T][A][ld]  the sampled actions (smarl_congestion_rollout's layout; NULL = skip)
 *   logp    f32 [T][A][ld]  log-probability of the sampled action        (NULL = skip)
 * A in 1..8 (one thread per four envs; A >= 9 or noise_mode 1 returns SMARL_EUNSUPPORTED), T in 1..65536 (16 bits of
 * the Philox counter). */
int smarl_congestion_policy_rollout(const SmarlCongestionParams* p, const SmarlDiscretePolicy* pol,
                                    const SmarlAccounting* acc, const uint8_t* start_x, const uint8_t* start_y,
                                    const double* lambdas, float* obs_rec, uint8_t* actions, float* logp,
                                    uint8_t* final_x, uint8_t* final_y, float* R, float* modR, int32_t* C, float* G,
                                    float* g_scratch, double* stats, double* stats_scratch, int64_t n_envs, int64_t ld,
                                    smarl_stream_t stream);

/* Whole ON-POLICY CoverageDiscretized episodes in one launch: main.py:28-57 with the policies inside, i.e. per step
 * every agent's DiscretePolicy (agent.py:23-47, 9 actions) on the current observation (x0, y0, x1, ...: what the
 * reset / step kernels write to env.obs), the sample, CoverageDiscretized.step, MetaAgent.act, and Buffer.step +
 * compute_returns as in smarl_coverage_float_rollout.  Records and final positions are bit-identical to the closed loop
 * reset + T x (smarl_policy_act_discretized(t) + smarl_coverage_float_step) on the same starts, weights and stream; the
 * products are bit-identical to smarl_coverage_float_rollout fed the recorded actions (the closed loop's returns kernel
 * sums the f32-rounded rewards, so its R, modR and stats agree to 1e-5 relative and C is equal).
 *   p (mode 1), acc, start_x .. lambdas and final_x .. stats_scratch as in smarl_coverage_float_rollout (acc->g_mode 0..2)
 *   pol: weights, seed, episode, episode_dev and env_offset as in smarl_policy_act_discretized;
 *        pol->n_agents = p->n_agents, hidden 16, 9 actions
 *   obs_rec f32 [T][2A][ld] the observation the policy saw at step t      (NULL = skip)
 *   actions u8  [T][A][ld]  the sampled actions (smarl_coverage_float_rollout's layout; NULL = skip)
 *   logp    f32 [T][A][ld]  log-probability of the sampled action        (NULL = skip)
 * A in 1..8 (one thread per env; A >= 9 or mode 0 returns SMARL_EUNSUPPORTED: smarl_coverage_float_policy_rollout
 * runs mode 0), T in 1..65536 (16 bits of the Philox counter). */
int smarl_coverage_discretized_policy_rollout(const SmarlCoverageFloatParams* p, const SmarlDiscretePolicy* pol,
                                              const SmarlAccounting* acc, const double* start_x, const double* start_y,
                                              const double* lambdas, float* obs_rec, uint8_t* actions, float* logp,
                                              double* final_x, double* final_y, float* R, float* modR, float* C,
                                              float* G, float* g_scratch, double* stats, double* stats_scratch,
                                              int64_t n_envs, int64_t ld, smarl_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Multi-GPU: env instances are independent (envs/coverage.py:19, congestion.py:22,
 * collision_avoidance.py:60), so ranks own contiguous ranges of global env ids and the data path has no
 * collective.  The only exchange is the sum of the stats vectors before MetaAgent.update
 * (meta_agent.py:32-39, called once per meta cycle at main.py:65-68).  NCCL is loaded at run time
 * (libnccl.so.2); single-GPU hosts never need it.
 *   rank 0: smarl_comm_get_unique_id(id)  ->  ship the SMARL_COMM_ID_BYTES bytes to every rank by any means
 *   all ranks, current device set: smarl_comm_init_from_unique_id(&comm, id, rank, world)   (collective)
 *   per batch:  smarl_stats_allreduce(comm, stats, smarl_stats_len(A, K), stream)  then  smarl_lambda_update
 * The all-reduce is enqueued on `stream` (no host sync, CUDA-graph capturable) and works in place.
 * ---------------------------------------------------------------------------------- */
#define SMARL_COMM_ID_BYTES 128
typedef struct SmarlComm SmarlComm;   /* opaque: one NCCL communicator */
int smarl_comm_get_unique_id(void* id_out /* [SMARL_COMM_ID_BYTES] host */);
int smarl_comm_init_from_unique_id(SmarlComm** out, const void* id, int32_t rank, int32_t world_size);
void smarl_comm_destroy(SmarlComm* comm);
/* NCCL version code of the library in use (e.g. 22809), 0 if NCCL cannot be loaded. */
int smarl_comm_nccl_version(void);
int smarl_stats_allreduce(SmarlComm* comm, double* stats, int32_t n, smarl_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Host-buffer entry points (what a host-side caller with numpy arrays binds).  Inputs are
 * HOST arrays (pageable, or pinned for full PCIe speed) in the same agent-major layout with
 * ld = smarl_host_session_ld(); the call pipelines env chunks over two streams (H2D copy,
 * fused rollout, D2H copy overlap) on the current device and returns when the episode
 * products are in the host arrays.  Synchronous; one call at a time per session.
 * ---------------------------------------------------------------------------------- */
typedef struct SmarlHostSession SmarlHostSession;   /* opaque: streams + device buffers */

/* One session per (env kind, n_agents, n_steps, n_envs[, n_landmarks]); K follows the env. */
int smarl_host_session_create(SmarlHostSession** out, int32_t env_kind, int32_t n_agents, int32_t n_steps,
                              int64_t n_envs, int32_t n_landmarks);
void smarl_host_session_destroy(SmarlHostSession* s);
/* ld (= padded n_envs) the host arrays of this session must use. */
int64_t smarl_host_session_ld(const SmarlHostSession* s);

/* CoverageDiscrete episodes from host buffers (main.py:28-57 for recorded actions).  p->lut /
 * p->weights, acc->thresholds and lambdas_h are HOST pointers here.  start_x_h,start_y_h u8 [A][ld];
 * actions_h u8 [T][A][ld]; R_h, modR_h f32 [A][ld]; C_h i32 [A][ld]; stats_h f64 [smarl_stats_len]
 * (NULL ok). */
int smarl_host_coverage_rollout(SmarlHostSession* s, const SmarlCoverageParams* p,
                                const SmarlAccounting* acc, const uint8_t* start_x_h,
                                const uint8_t* start_y_h, const uint8_t* actions_h,
                                const double* lambdas_h, float* R_h, float* modR_h, int32_t* C_h,
                                double* stats_h);

/* Same with 4-bit packed actions (actions are 0..4): actions4_h u8 [T][A][ld/2], byte j of a row holds
 * env 2j in its low and env 2j+1 in its high nibble.  Halves the PCIe bytes of this PCIe-bound call; the
 * nibbles are expanded on the device. */
int smarl_host_coverage_rollout_packed4(SmarlHostSession* s, const SmarlCoverageParams* p,
                                        const SmarlAccounting* acc, const uint8_t* start_x_h,
                                        const uint8_t* start_y_h, const uint8_t* actions4_h,
                                        const double* lambdas_h, float* R_h, float* modR_h, int32_t* C_h,
                                        double* stats_h);

/* Same with base-5 packed actions, three per byte: byte j of a row holds envs 3j, 3j+1, 3j+2 as a0 + 5 a1 + 25 a2
 * (0.33 B per action); actions5_h u8 [T][A][smarl_host_session_pitch5()].  A third of the action bytes on PCIe. */
int64_t smarl_host_session_pitch5(const SmarlHostSession* s);
int smarl_host_coverage_rollout_packed5(SmarlHostSession* s, const SmarlCoverageParams* p,
                                        const SmarlAccounting* acc, const uint8_t* start_x_h,
                                        const uint8_t* start_y_h, const uint8_t* actions5_h,
                                        const double* lambdas_h, float* R_h, float* modR_h, int32_t* C_h,
                                        double* stats_h);

/* Pinned (page-locked) host memory for the arrays of the smarl_host_* calls, placed on the NUMA node the current
 * GPU is attached to (sysfs numa_node of its PCI address, set_mempolicy(MPOL_PREFERRED) around the first touch) when
 * the kernel allows it; *numa_node_out (may be NULL) receives that node, or -1 if no binding was applied.  With one
 * rank per GPU this keeps every rank's PCIe traffic on its own socket.  Free with smarl_host_free_pinned. */
int smarl_host_alloc_pinned(void** out, size_t bytes, int32_t* numa_node_out);
void smarl_host_free_pinned(void* p);

/* Same for callers that keep the reference's env-major arrays (what np.array(actions) gives there): no
 * padding, no ld.  starts_h u8 [E][A][2] (x, y per agent, coverage.py:45-49); actions_h u8 [T][E][A];
 * R_h, modR_h f32 [E][A]; C_h i32 [E][A].  The layout change runs on the device inside the pipeline, so
 * the PCIe traffic equals smarl_host_coverage_rollout's. */
int smarl_host_coverage_rollout_envmajor(SmarlHostSession* s, const SmarlCoverageParams* p,
                                         const SmarlAccounting* acc, const uint8_t* starts_h,
                                         const uint8_t* actions_h, const double* lambdas_h, float* R_h,
                                         float* modR_h, int32_t* C_h, double* stats_h);

/* Congestion episodes from host buffers.  p->demand is a HOST table; moves_h u8 [T][A][ld] only for
 * noise_mode 1; C_h i32 [1][ld]. */
int smarl_host_congestion_rollout(SmarlHostSession* s, const SmarlCongestionParams* p,
                                  const SmarlAccounting* acc, const uint8_t* start_x_h,
                                  const uint8_t* start_y_h, const uint8_t* actions_h,
                                  const uint8_t* moves_h, const double* lambdas_h, float* R_h,
                                  float* modR_h, int32_t* C_h, double* stats_h);

/* CollisionAvoidance episodes from host buffers.  start_x_h,start_y_h f64 [A][ld]; landmarks_h f64
 * [2L][ld]; actions_h f32 [T][2A][ld]; C_h i32 [1][ld]; n_active_h i32 [ld] (NULL ok). */
int smarl_host_collision_rollout(SmarlHostSession* s, const SmarlCollisionParams* p,
                                 const SmarlAccounting* acc, const double* start_x_h,
                                 const double* start_y_h, const double* landmarks_h,
                                 const float* actions_h, const double* lambdas_h, float* R_h, float* modR_h,
                                 int32_t* C_h, int32_t* n_active_h, double* stats_h);

/* Env-major forms of the two calls above (arrays as a user of the reference holds them, no padding):
 * Congestion  starts_h u8 [E][A][2]; actions_h, moves_h u8 [T][E][A]; R_h, modR_h f32 [E][A]; C_h i32 [E].
 * Collision   starts_h f64 [E][A][2]; landmarks_h f64 [E][L][2]; actions_h f32 [T][E][A][2];
 *             R_h, modR_h f32 [E][A]; C_h, n_active_h i32 [E]. */
int smarl_host_congestion_rollout_envmajor(SmarlHostSession* s, const SmarlCongestionParams* p,
                                           const SmarlAccounting* acc, const uint8_t* starts_h,
                                           const uint8_t* actions_h, const uint8_t* moves_h,
                                           const double* lambdas_h, float* R_h, float* modR_h, int32_t* C_h,
                                           double* stats_h);
int smarl_host_collision_rollout_envmajor(SmarlHostSession* s, const SmarlCollisionParams* p,
                                          const SmarlAccounting* acc, const double* starts_h,
                                          const double* landmarks_h, const float* actions_h,
                                          const double* lambdas_h, float* R_h, float* modR_h, int32_t* C_h,
                                          int32_t* n_active_h, double* stats_h);

#ifdef __cplusplus
}
#endif
#endif /* SMARL_H_ */
