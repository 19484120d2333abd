"""BatchedCoverageContinuous / BatchedCoverageDiscretized -- the float-position Coverage envs
(envs/coverage.py:8-106 and :210-241; "ExploreContinuous" in the paper's launchers)."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from .. import _lib
from ..rollout import G_NONE
from .base import BatchedEnv, PolicyRollout


class _CoverageFloat(BatchedEnv):
    cost_dtype = torch.float32
    never_done = True

    def _setup(self, size, n_agents, n_envs, device, env_offset, shuffle, agents_size, fieldview_size, weights, starts,
               seed=0):
        self._init_common(size, n_agents, n_envs, device, env_offset)
        self.shuffle, self.agents_size, self.seed = bool(shuffle), agents_size, int(seed)
        A, E, dev = self.n_agents, self.n_envs, self.device
        self.fieldview_size = self.size / (np.sqrt(A)) if fieldview_size is None else fieldview_size   # coverage.py:15-18
        self.state_space = 2 * A
        self.constraint_space = [1 for _ in range(A)]
        self.n_constraints = A
        self.weights = None if weights is None else list(weights)
        if self.weights is not None and len(self.weights) < A:
            raise ValueError("need at least n_agents weights")
        self._weights = None if self.weights is None else \
            torch.as_tensor(np.asarray(self.weights[:A], dtype=np.float64), dtype=torch.float32).to(dev)
        starts = np.asarray(starts, dtype=np.float64)
        assert starts.shape == (E, A, 2)
        f64 = torch.float64
        self.start_x, self.start_y = self._alloc(A, f64), self._alloc(A, f64)
        self.start_x[:, :E] = torch.as_tensor(starts[:, :, 0].T.copy()).to(dev)
        self.start_y[:, :E] = torch.as_tensor(starts[:, :, 1].T.copy()).to(dev)
        self.pos_x, self.pos_y = self.start_x.clone(), self.start_y.clone()
        self.action_buffer = self._alloc(self.action_rows, self.action_dtype)
        self.obs = self._alloc(2 * A, torch.float32)
        self.reward = self._alloc(A, torch.float32)
        self.cost = self._alloc(A, torch.float32)
        self.done = self._alloc(A, torch.uint8)
        self.penalty = self._alloc(1, torch.float32)[0]

    def state(self):
        E = self.n_envs
        return torch.stack([self.pos_x[:, :E].t(), self.pos_y[:, :E].t()], dim=-1)

    def _reset_impl(self):
        _lib.check(self.lib.smarl_coverage_float_reset(
            _lib.ptr(self.start_x), _lib.ptr(self.start_y), _lib.ptr(self.pos_x), _lib.ptr(self.pos_y),
            _lib.ptr(self.obs), self.n_agents, self.n_envs, self.ld, _lib.stream_ptr()))

    def _step_impl(self, act, reward, cost, done, lambdas, penalty):
        _lib.check(self.lib.smarl_coverage_float_step(
            C.byref(self._params), _lib.ptr(self.pos_x), _lib.ptr(self.pos_y), _lib.ptr(act), _lib.ptr(self.obs),
            _lib.ptr(reward), _lib.ptr(cost), _lib.ptr(done), _lib.ptr(lambdas), _lib.ptr(penalty), self.n_envs,
            self.ld, _lib.stream_ptr()))


    def rollout(self, actions, lambdas=None, gamma=0.99, thresholds=None, g_mode=G_NONE, out=None):
        """Open-loop fused episode (one launch).  actions in the kernel layout: float32 ``[T, 2*n_agents, ld]``
        (Continuous) or uint8 ``[T, n_agents, ld]`` (Discretized).  ``C`` holds float cost sums."""
        T = int(actions.shape[0])
        assert actions.dtype == self.action_dtype and tuple(actions.shape) == (T, self.action_rows, self.ld) \
            and actions.is_contiguous()
        o, acc = self._begin_rollout(T, g_mode, out, 2 * T, gamma, thresholds)
        _lib.check(self.lib.smarl_coverage_float_rollout(
            C.byref(self._params), C.byref(acc), _lib.ptr(self.start_x), _lib.ptr(self.start_y), _lib.ptr(actions),
            _lib.ptr(lambdas), _lib.ptr(self.pos_x), _lib.ptr(self.pos_y), _lib.ptr(o["R_"]), _lib.ptr(o["modR_"]),
            _lib.ptr(o["C_"]), _lib.ptr(o["G_"]), _lib.ptr(o["gs_"]), _lib.ptr(o["stats_vec"]),
            _lib.ptr(o["stats_scratch"]), self.n_envs, self.ld, _lib.stream_ptr()))
        return self._rollout_result(o)

    def _draw_starts(self, episode):
        zoom = getattr(self, "zoom_fac", None)
        self._draw_float_starts(episode, 3 if zoom is not None else 2, zoom or 0.0)


class BatchedCoverageContinuous(PolicyRollout, _CoverageFloat):
    """``CoverageContinuous(size, n_agents, shuffle, agents_size, fieldview_size, weights, coarseness)``
    (coverage.py:11) + ``n_envs``/``device``.  Actions are ``[n_envs, n_agents, 2]`` float32."""

    action_space = 2
    action_dtype = torch.float32
    rollout_policy, reference_policy, rollout_threads = "FusedGaussianPolicy", "ContinuousPolicy", "one thread per env"

    def __init__(self, size, n_agents, n_envs=1, shuffle=False, agents_size=0.5, fieldview_size=None, weights=None,
                 coarseness=None, device="cuda", starts=None, env_offset=0, seed=0):
        self.action_rows = 2 * int(n_agents)
        if starts is None:
            starts = np.random.rand(int(n_envs), int(n_agents), 2) * size          # coverage.py:267
        self._setup(size, n_agents, n_envs, device, env_offset, shuffle, agents_size, fieldview_size, weights, starts,
                    seed)
        self.coarseness = coarseness
        max_norm = float(np.sqrt(2) * self.size / coarseness) if coarseness is not None else 0.0   # coverage.py:66
        self._params = _lib.CoverageFloatParams(self.size, self.n_agents, 0, int(coarseness is not None),
                                                float(self.fieldview_size), max_norm, 0.0, 0.0, 0.0, 0.0,
                                                _lib.ptr(self._weights))

    def _policy_rollout_impl(self, pol, acc, lambdas, rec, o):
        _lib.check(self.lib.smarl_coverage_float_policy_rollout(
            C.byref(self._params), C.byref(pol), C.byref(acc), _lib.ptr(self.start_x), _lib.ptr(self.start_y),
            _lib.ptr(lambdas), *[_lib.ptr(x) for x in rec], _lib.ptr(self.pos_x), _lib.ptr(self.pos_y),
            _lib.ptr(o["R_"]), _lib.ptr(o["modR_"]), _lib.ptr(o["C_"]), _lib.ptr(o["G_"]), _lib.ptr(o["gs_"]),
            _lib.ptr(o["stats_vec"]), _lib.ptr(o["stats_scratch"]), self.n_envs, self.ld, _lib.stream_ptr()))


class BatchedCoverageDiscretized(_CoverageFloat):
    """``CoverageDiscretized(size, n_agents, coarseness=20, shuffle, agents_size, fieldview_size, weights)``
    (coverage.py:211) + ``n_envs``/``device``.  Actions are ``[n_envs, n_agents]`` in 0..8."""

    action_space = 9
    action_dtype = torch.uint8

    def __init__(self, size, n_agents, n_envs=1, coarseness=20, shuffle=False, agents_size=0.5, fieldview_size=None,
                 weights=None, device="cuda", starts=None, env_offset=0, seed=0):
        self.action_rows = int(n_agents)
        self.coarseness = coarseness
        self.zoom_fac = coarseness / size                                           # coverage.py:215
        if starts is None:
            # the ctor builds (and discards) n_agents continuous agents first, coverage.py:19,:216
            draws = np.random.rand(int(n_envs), 2 * int(n_agents), 2)[:, int(n_agents):] * size
            starts = np.floor(draws * self.zoom_fac) / self.zoom_fac                # coverage.py:270-272
        self._setup(size, n_agents, n_envs, device, env_offset, shuffle, agents_size, fieldview_size, weights, starts,
                    seed)
        table = np.array([1, np.sqrt(2)]) * (self.size / coarseness)                # coverage.py:237
        self._params = _lib.CoverageFloatParams(self.size, self.n_agents, 1, 0, float(self.fieldview_size), 0.0,
                                                float(self.zoom_fac), float(self.size * self.zoom_fac),
                                                float(table[0]), float(table[1]), _lib.ptr(self._weights))


class BatchedCoverageDiscretizedOnPolicy(PolicyRollout, BatchedCoverageDiscretized):
    """``BatchedCoverageDiscretized`` that also runs whole on-policy episodes in one launch: ``policy_rollout(policy, T,
    ...)`` with a ``FusedDiscretizedPolicy`` (``PolicyRollout``, DESIGN.md section 3.15).  Constructor, state,
    ``reset`` / ``step`` / ``rollout`` are those of ``BatchedCoverageDiscretized``, whose own interface stays as it
    was."""

    rollout_policy, reference_policy, rollout_threads = "FusedDiscretizedPolicy", "DiscretePolicy", "one thread per env"

    def _policy_rollout_impl(self, pol, acc, lambdas, rec, o):
        _lib.check(self.lib.smarl_coverage_discretized_policy_rollout(
            C.byref(self._params), C.byref(pol), C.byref(acc), _lib.ptr(self.start_x), _lib.ptr(self.start_y),
            _lib.ptr(lambdas), *[_lib.ptr(x) for x in rec], _lib.ptr(self.pos_x), _lib.ptr(self.pos_y),
            _lib.ptr(o["R_"]), _lib.ptr(o["modR_"]), _lib.ptr(o["C_"]), _lib.ptr(o["G_"]), _lib.ptr(o["gs_"]),
            _lib.ptr(o["stats_vec"]), _lib.ptr(o["stats_scratch"]), self.n_envs, self.ld, _lib.stream_ptr()))
