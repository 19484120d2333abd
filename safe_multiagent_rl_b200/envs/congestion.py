"""BatchedCongestion -- n_envs instances of the reference's Congestion env
(envs/congestion.py:13-137) stepped by one CUDA launch."""
from __future__ import annotations

import ctypes as C
import math
from fractions import Fraction

import numpy as np
import torch

from .. import _lib
from ..rollout import G_NONE
from .base import BatchedEnv, PolicyRollout

# congestion.py:28 -- the reference's hard-coded table (only valid for size <= 3)
REFERENCE_DEMAND = np.array([[2, 2, 4, 4], [3, 6, 10, 5], [3, 8, 3, 4], [4, 6, 7, 8]], dtype=np.float64)

NOISE_NONE, NOISE_RECORDED, NOISE_PHILOX = 0, 1, 2


def keep_threshold(noise: float) -> int:
    """Smallest integer thr with (w * 2**-32 < 1 - noise) <=> (w < thr) for a uint32 word w:
    the integer form of ``random() < 1 - self.noise`` (congestion.py:64)."""
    lim = Fraction(1 - noise) * (1 << 32)
    return min(1 << 32, max(0, math.ceil(lim)))


def default_starts(size, n_agents, n_envs):
    """Start positions [n_envs, n_agents, 2] in the reference ctor's RNG order (congestion.py:22, :215-217): agent 0
    sits at (0, 0) and draws nothing, agents 1.. draw ``floor(rand(2) * size)`` in index order, env after env."""
    starts = np.zeros((n_envs, n_agents, 2))
    if n_agents > 1:
        starts[:, 1:, :] = np.floor(np.random.rand(n_envs, n_agents - 1, 2) * size)
    return starts


class BatchedCongestion(BatchedEnv):
    """Constructor mirrors ``Congestion(size, n_agents, noise, shuffle)`` (congestion.py:19) plus
    ``n_envs`` / ``device``.

    demand_rate  ``[(size+1), (size+1)]`` table indexed [x][y] (congestion.py:86).  The reference
                 hard-codes a 4x4 table and raises IndexError beyond size 3; here the table is an
                 input, defaulting to the reference's when it fits.
    noise        action noise (congestion.py:64-67).  The reference draws it from Python's unseeded
                 ``random``; here ``seed`` keys an on-device Philox4x32-10 stream indexed by the
                 global env id, episode, step and agent, or recorded effective moves can be replayed
                 with ``step(actions, moves=...)``.  The episode index lives in a device scalar that
                 every ``reset()`` / ``rollout()`` after the first advances, so consecutive episodes
                 (and consecutive replays of a captured CUDA graph) draw independent noise like the
                 reference's ``random()``; ``set_noise_episode(n)`` pins it.
    starts       optional ``[n_envs, n_agents, 2]``; default as the reference: agent 0 at (0,0),
                 others ``floor(rand(2) * size)`` from the global np.random stream (:215-217).
    """

    action_space = 5
    cost_dtype = torch.int32
    action_dtype = torch.uint8
    never_done = True          # check_done is all-False (congestion.py:103-104)

    def __init__(self, size, n_agents, n_envs=1, noise=0.1, shuffle=False, device="cuda", starts=None,
                 demand_rate=None, seed=0, env_offset=0):
        self._init_common(size, n_agents, n_envs, device, env_offset)
        if not (1 <= self.size <= 254):
            raise ValueError("size must be in 1..254 (uint8 coordinates)")
        assert 0 <= noise <= 1                                    # congestion.py:30
        self.shuffle, self.noise, self.seed = bool(shuffle), float(noise), int(seed)
        A, E, dev = self.n_agents, self.n_envs, self.device
        self.state_space = 2 * A
        self.constraint_space = [1]
        self.n_constraints = 1
        self.action_rows = A
        self.landmark = [self.size, self.size]
        if demand_rate is None:
            if self.size > 3:
                raise ValueError("the reference's demand_rate table is 4x4 (congestion.py:28); pass "
                                 "demand_rate of shape (size+1, size+1) for size > 3")
            demand_rate = REFERENCE_DEMAND[: self.size + 1, : self.size + 1]
        demand_rate = np.asarray(demand_rate, dtype=np.float64)
        assert demand_rate.shape == (self.size + 1, self.size + 1)
        self.demand_rate = demand_rate
        self._demand = torch.as_tensor(np.ascontiguousarray(demand_rate)).to(dev)
        # waiting-branch reward (congestion.py:86-87) for every congestion level and cell, evaluated in f64 in the
        # reference's operation order and rounded once to f32: saves a float64 division per agent-step on the device
        con = np.arange(A, dtype=np.float64)[:, None, None]
        wait = -30.0 * (con + 1) / demand_rate[None] + 7.5 - 4.0
        self._wait_reward = torch.as_tensor(np.ascontiguousarray(wait.astype(np.float32))).to(dev)
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
        self.moves = self._alloc(A, torch.uint8)                  # effective (post-noise) moves of the last step
        self.obs = self._alloc(2 * A, torch.float32)
        self.reward = self._alloc(A, torch.float32)
        self.cost = self._alloc(1, torch.int32)
        self.done = self._alloc(A, torch.uint8)
        self.penalty = self._alloc(1, torch.float32)[0]
        self._recorded = None
        self._episode_dev = torch.zeros(1, dtype=torch.int32, device=dev)   # noise episode index (read as u32)
        self._noise_started = False

    def _params(self, mode):
        return _lib.CongestionParams(self.size, self.n_agents, _lib.ptr(self._demand), mode, 0,
                                     keep_threshold(self.noise), self.seed & (2 ** 64 - 1), self.env_offset,
                                     _lib.ptr(self._wait_reward), _lib.ptr(self._episode_dev))

    def set_noise_episode(self, n):
        """The next ``reset()`` / ``rollout()`` draws the noise of episode ``n`` (then counting on from there).
        A captured CUDA graph that contains the reset advances the device counter before it draws, so pin
        ``n - 1`` before replaying it for episode ``n``."""
        self._episode_dev.fill_(int(n))
        self._noise_started = False

    def _next_noise_episode(self):
        # a device-side increment: capturable, so every replay of a CUDA graph that contains this reset advances too
        if self._noise_started:
            self._episode_dev.add_(1)
        self._noise_started = True

    def _draw_starts(self, episode):
        self._draw_grid_starts(episode, 1)        # agent 0 restarts at (0,0), congestion.py:215-216

    def state(self):
        E = self.n_envs
        return torch.stack([self.pos_x[:, :E].t(), self.pos_y[:, :E].t()], dim=-1)

    def _reset_impl(self):
        self._next_noise_episode()
        _lib.check(self.lib.smarl_grid_reset(_lib.ptr(self.start_x), _lib.ptr(self.start_y),
                                             _lib.ptr(self.pos_x), _lib.ptr(self.pos_y), _lib.ptr(self.obs),
                                             self.n_agents, self.n_envs, self.ld, _lib.stream_ptr()))

    def step(self, actions, lambdas=None, out=None, agent_major=False, moves=None):
        """As BatchedEnv.step; ``moves`` ``[n_envs, n_agents]`` replays recorded effective moves
        instead of drawing noise."""
        if moves is not None:
            m = torch.as_tensor(np.asarray(moves) if not isinstance(moves, torch.Tensor) else moves).to(self.device)
            self.moves[:, : self.n_envs].copy_(m.reshape(self.n_envs, self.n_agents).t())
            self._recorded = True
        else:
            self._recorded = False
        return super().step(actions, lambdas=lambdas, out=out, agent_major=agent_major)

    def _step_impl(self, act, reward, cost, done, lambdas, penalty):
        mode = NOISE_RECORDED if self._recorded else (NOISE_PHILOX if self.noise > 0 else NOISE_NONE)
        p = self._params(mode)
        _lib.check(self.lib.smarl_congestion_step(
            C.byref(p), _lib.ptr(self.pos_x), _lib.ptr(self.pos_y), _lib.ptr(act), _lib.ptr(self.moves),
            _lib.ptr(self.obs if self.emit_obs else None), _lib.ptr(reward), _lib.ptr(cost), _lib.ptr(done), _lib.ptr(lambdas),
            _lib.ptr(penalty), self.t, self.n_envs, self.ld, _lib.stream_ptr()))

    def rollout(self, actions, lambdas=None, gamma=0.99, thresholds=None, g_mode=G_NONE, out=None, moves=None):
        """Open-loop fused episode (one launch).  actions ``[T, n_agents, ld]`` uint8 (kernel layout);
        ``moves`` of the same shape replays recorded effective moves, otherwise noise comes from the
        Philox stream (same stream as T calls of ``step``)."""
        T = int(actions.shape[0])
        A, E = self.n_agents, self.n_envs
        assert actions.dtype == torch.uint8 and tuple(actions.shape) == (T, A, self.ld) and actions.is_contiguous()
        if moves is not None:
            assert moves.dtype == torch.uint8 and tuple(moves.shape) == (T, A, self.ld) and moves.is_contiguous()
        mode = NOISE_RECORDED if moves is not None else (NOISE_PHILOX if self.noise > 0 else NOISE_NONE)
        o, acc = self._begin_rollout(T, g_mode, out, T, gamma, thresholds)
        p = self._params(mode)
        self._next_noise_episode()
        _lib.check(self.lib.smarl_congestion_rollout(
            C.byref(p), C.byref(acc), _lib.ptr(self.start_x), _lib.ptr(self.start_y), _lib.ptr(actions),
            _lib.ptr(moves), _lib.ptr(lambdas), _lib.ptr(self.pos_x), _lib.ptr(self.pos_y), _lib.ptr(o["R_"]),
            _lib.ptr(o["modR_"]), _lib.ptr(o["C_"]), _lib.ptr(o["G_"]), _lib.ptr(o["gs_"]),
            _lib.ptr(o["stats_vec"]), _lib.ptr(o["stats_scratch"]), E, self.ld, _lib.stream_ptr()))
        self.t = T
        return self._rollout_result(o)


class BatchedCongestionOnPolicy(PolicyRollout, BatchedCongestion):
    """``BatchedCongestion`` that also runs whole on-policy episodes in one launch: ``policy_rollout(policy, T, ...)``
    with a ``FusedDiscretePolicy`` (``PolicyRollout``, DESIGN.md section 3.14).  Constructor, state, ``reset`` / ``step`` /
    ``rollout`` and the noise stream are those of ``BatchedCongestion``, whose own interface stays as it was."""

    rollout_policy, reference_policy, rollout_threads = "FusedDiscretePolicy", "DiscretePolicy", "one thread per four envs"

    def _policy_rollout_impl(self, pol, acc, lambdas, rec, o):
        p = self._params(NOISE_PHILOX if self.noise > 0 else NOISE_NONE)
        self._next_noise_episode()                 # as rollout(): the same noise as the closed loop after its reset
        _lib.check(self.lib.smarl_congestion_policy_rollout(
            C.byref(p), C.byref(pol), C.byref(acc), _lib.ptr(self.start_x), _lib.ptr(self.start_y), _lib.ptr(lambdas),
            *[_lib.ptr(x) for x in rec], _lib.ptr(self.pos_x), _lib.ptr(self.pos_y), _lib.ptr(o["R_"]),
            _lib.ptr(o["modR_"]), _lib.ptr(o["C_"]), _lib.ptr(o["G_"]), _lib.ptr(o["gs_"]), _lib.ptr(o["stats_vec"]),
            _lib.ptr(o["stats_scratch"]), self.n_envs, self.ld, _lib.stream_ptr()))
