"""BatchedCoverageDiscrete -- n_envs instances of the reference's CoverageDiscrete ("Explore",
envs/coverage.py:166-196 on top of CoverageContinuous :8-106) stepped by one CUDA launch."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from .. import _lib
from ..rollout import G_NONE
from .base import BatchedEnv, PolicyRollout


MAX_LUT = 12279      # kCoverageMaxLut (csrc/coverage.cuh): the table + the rollout kernel's reduction buffer fill 48 KB


def penalty_table(size, n_agents, fieldview_size=None):
    """(fv, table) with table[q] = (fv - sqrt(q))**2 for integer squared distances q whose
    distance is inside the field of view, truncated after the last non-zero entry.

    Same numpy *scalar* expression as the reference (coverage.py:15-18, :82-83) so the f64 values
    are the reference's; the kernel reads their f32 rounding.
    """
    fv = size / (np.sqrt(n_agents)) if fieldview_size is None else fieldview_size
    vals = []
    for q in range(2 * size * size + 1):
        d = np.sqrt(np.float64(q))
        if fv - d > 0:
            vals.append(float((fv - d) ** 2))
        else:
            break                      # sqrt is monotone: every later q is outside the field of view
    return fv, np.asarray(vals, dtype=np.float64)


def default_starts(size, n_agents, n_envs):
    """Start positions [n_envs, n_agents, 2] drawn from the global ``np.random`` stream exactly as constructing
    n_envs reference ``CoverageDiscrete`` envs one after another does: each ctor first builds and discards
    n_agents continuous agents (coverage.py:19 via super().__init__, 2 rand values each), then draws the kept ones
    as ``floor(rand(2) * size)`` in agent order (:170, :267-269)."""
    draws = np.random.rand(n_envs, 2 * n_agents, 2)
    return np.floor(draws[:, n_agents:, :] * size)


class BatchedCoverageDiscrete(PolicyRollout, BatchedEnv):
    """Constructor mirrors ``CoverageDiscrete(size, n_agents, shuffle, agents_size, fieldview_size,
    weights)`` (coverage.py:167) plus ``n_envs`` / ``device``.

    starts  optional ``[n_envs, n_agents, 2]`` integer array.  By default they are drawn from the
            global ``np.random`` stream exactly as constructing n_envs reference envs one after
            another would (each ctor first builds and discards n_agents continuous agents,
            coverage.py:19,:170, then floors ``rand(2) * size``, :267-269).
    """

    action_space = 5
    cost_dtype = torch.uint8
    action_dtype = torch.uint8
    never_done = True          # check_done is all-False (coverage.py:97-98)
    supports_lean = True       # reward_a = w_a * rew: one env-reward row is enough (DESIGN.md section 3.6)
    rollout_policy, reference_policy, rollout_threads = "FusedDiscretePolicy", "DiscretePolicy", "one thread per four envs"

    def __init__(self, size, n_agents, n_envs=1, shuffle=False, agents_size=0.5, fieldview_size=None,
                 weights=None, device="cuda", starts=None, env_offset=0, seed=0):
        self._init_common(size, n_agents, n_envs, device, env_offset)
        if not (1 <= self.size <= 127):
            raise ValueError("size must be in 1..127 (doubled uint8 coordinates index the penalty table)")
        self.shuffle, self.seed = bool(shuffle), int(seed)
        self.agents_size = agents_size
        A, E = self.n_agents, self.n_envs
        self.state_space = 2 * A
        self.constraint_space = [1 for _ in range(A)]
        self.n_constraints = A
        self.action_rows = A
        self.fieldview_size, table = penalty_table(self.size, A, fieldview_size)
        if A == 1:
            table = table[:0]
        if len(table) > MAX_LUT:
            raise NotImplementedError("fieldview_size > 110 needs a penalty table larger than shared memory")
        self.weights = None if weights is None else list(weights)
        if self.weights is not None and len(self.weights) < A:
            # the reference zips rewards with weights and silently returns fewer rewards than agents
            # (coverage.py:86-87); that breaks its own driver, so it is rejected here
            raise ValueError("need at least n_agents weights")
        dev = self.device
        self._lut = torch.as_tensor(table, dtype=torch.float32).to(dev) if len(table) else None
        self._weights = None if self.weights is None else \
            torch.as_tensor(np.asarray(self.weights[:A], dtype=np.float64), dtype=torch.float32).to(dev)
        self._params = _lib.CoverageParams(self.size, A, len(table), 0, _lib.ptr(self._lut),
                                           _lib.ptr(self._weights))
        self._params_shared = _lib.CoverageParams(self.size, A, len(table), 1, _lib.ptr(self._lut),
                                                  _lib.ptr(self._weights))
        if starts is None:
            starts = default_starts(self.size, A, E)
        starts = np.asarray(starts)
        assert starts.shape == (E, A, 2)
        if starts.min() < 0 or starts.max() > self.size:
            raise ValueError("start coordinates must lie in [0, size]")
        self.start_x, self.start_y = self._alloc(A, torch.uint8), self._alloc(A, torch.uint8)
        self.start_x[:, :E] = torch.as_tensor(starts[:, :, 0].T.astype(np.uint8)).to(dev)
        self.start_y[:, :E] = torch.as_tensor(starts[:, :, 1].T.astype(np.uint8)).to(dev)
        self.pos_x, self.pos_y = self.start_x.clone(), self.start_y.clone()
        self.action_buffer = self._alloc(A, torch.uint8)
        self.obs = self._alloc(2 * A, torch.float32)
        self.reward = self._alloc(A, torch.float32)
        self.cost = self._alloc(A, torch.uint8)
        self.done = self._alloc(A, torch.uint8)
        self.penalty = self._alloc(1, torch.float32)[0]

    def _draw_starts(self, episode):
        self._draw_grid_starts(episode, 0)

    def state(self):
        """[n_envs, n_agents, 2] integer positions (a copy)."""
        E = self.n_envs
        return torch.stack([self.pos_x[:, :E].t(), self.pos_y[:, :E].t()], dim=-1)

    def _reset_impl(self):
        _lib.check(self.lib.smarl_grid_reset(_lib.ptr(self.start_x), _lib.ptr(self.start_y),
                                             _lib.ptr(self.pos_x), _lib.ptr(self.pos_y), _lib.ptr(self.obs),
                                             self.n_agents, self.n_envs, self.ld, _lib.stream_ptr()))

    def _step_impl(self, act, reward, cost, done, lambdas, penalty):
        params = self._params
        if reward.shape[0] == 1 and self.n_agents > 1:        # lean rollout buffer: one unweighted env-reward row
            params = self._params_shared
        _lib.check(self.lib.smarl_coverage_step(
            C.byref(params), _lib.ptr(self.pos_x), _lib.ptr(self.pos_y), _lib.ptr(act),
            _lib.ptr(self.obs if self.emit_obs else None), _lib.ptr(reward), _lib.ptr(cost), _lib.ptr(done), _lib.ptr(lambdas),
            _lib.ptr(penalty), self.n_envs, self.ld, _lib.stream_ptr()))

    def rollout(self, actions, lambdas=None, gamma=0.99, thresholds=None, g_mode=G_NONE, out=None):
        """Open-loop fused episode (one launch): reset + T steps + accounting, state in registers.

        actions ``[T, n_agents, ld]`` uint8 device tensor (kernel layout).  Returns dict with
        R/modR [E,A], C [E,A] i32, G [T,E,A] or None, final positions, stats.
        """
        T = int(actions.shape[0])
        A, E = self.n_agents, self.n_envs
        assert actions.dtype == torch.uint8 and tuple(actions.shape) == (T, A, self.ld) and actions.is_contiguous()
        o, acc = self._begin_rollout(T, g_mode, out, 2 * T, gamma, thresholds)
        _lib.check(self.lib.smarl_coverage_rollout(
            C.byref(self._params), C.byref(acc), _lib.ptr(self.start_x), _lib.ptr(self.start_y),
            _lib.ptr(actions), _lib.ptr(lambdas), _lib.ptr(self.pos_x), _lib.ptr(self.pos_y), _lib.ptr(o["R_"]),
            _lib.ptr(o["modR_"]), _lib.ptr(o["C_"]), _lib.ptr(o["G_"]), _lib.ptr(o["gs_"]),
            _lib.ptr(o["stats_vec"]), _lib.ptr(o["stats_scratch"]), E, self.ld, _lib.stream_ptr()))
        return self._rollout_result(o)

    def _policy_rollout_impl(self, pol, acc, lambdas, rec, o):
        _lib.check(self.lib.smarl_coverage_policy_rollout(
            C.byref(self._params), C.byref(pol), C.byref(acc), _lib.ptr(self.start_x), _lib.ptr(self.start_y),
            _lib.ptr(lambdas), *[_lib.ptr(x) for x in rec], _lib.ptr(self.pos_x), _lib.ptr(self.pos_y),
            _lib.ptr(o["R_"]), _lib.ptr(o["modR_"]), _lib.ptr(o["C_"]), _lib.ptr(o["G_"]), _lib.ptr(o["gs_"]),
            _lib.ptr(o["stats_vec"]), _lib.ptr(o["stats_scratch"]), self.n_envs, self.ld, _lib.stream_ptr()))
