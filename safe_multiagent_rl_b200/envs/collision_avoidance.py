"""BatchedCollisionAvoidance -- n_envs instances of the reference's CollisionAvoidance env
(envs/collision_avoidance.py:6-165) stepped by one CUDA launch.  State is float64 like the
reference; actions are float32, which is what its policies emit (agent.py:124-125)."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from .. import _lib
from ..layout import env_major
from ..rollout import G_NONE
from .base import BatchedEnv, PolicyRollout


def default_starts(size, n_agents, n_envs, n_landmarks=1):
    """(starts [n_envs, n_agents, 2], landmarks [n_envs, n_landmarks, 2]) in the reference ctor's RNG order
    (collision_avoidance.py:60-62): per env the agents' ``rand(2) * size`` in index order, then the landmark(s).
    The ctor itself draws a single landmark; with shuffle every reset redraws n_landmarks (:100-101)."""
    draws = np.random.rand(n_envs, n_agents + n_landmarks, 2) * size
    return draws[:, :n_agents], draws[:, n_agents:]


class BatchedCollisionAvoidance(PolicyRollout, BatchedEnv):
    """Constructor mirrors ``CollisionAvoidance(size, n_agents, n_landmarks, shuffle, agents_size,
    normalize_state)`` (collision_avoidance.py:49) plus ``n_envs`` / ``device``.

    starts / landmarks  optional ``[n_envs, n_agents, 2]`` / ``[n_envs, n_landmarks, 2]`` float64.
        Defaults follow the reference ctor per env: agents ``rand(2) * size`` in index order, then
        ONE landmark (:60-62; n_landmarks only matters on shuffle, :100-101).
    """

    action_space = 2
    cost_dtype = torch.int32
    action_dtype = torch.float32
    supports_lean = True       # the reward is one value shared by all agents (collision_avoidance.py:129-130)
    rollout_policy, reference_policy, rollout_threads = "FusedGaussianPolicy", "ContinuousPolicy", "one thread per env"

    def __init__(self, size, n_agents, n_envs=1, n_landmarks=1, shuffle=False, agents_size=0.25,
                 normalize_state=False, device="cuda", starts=None, landmarks=None, env_offset=0, seed=0):
        assert type(size) == int and type(n_agents) == int and type(n_landmarks) == int   # :51-53
        assert type(agents_size) in (float, int)
        self._init_common(size, n_agents, n_envs, device, env_offset)
        self.shuffle, self.normalize_state, self.seed = bool(shuffle), bool(normalize_state), int(seed)
        self.agents_size = float(agents_size)
        A, E, dev = self.n_agents, self.n_envs, self.device
        self.n_landmarks = int(n_landmarks)
        self.state_space = 2 * A
        self.constraint_space = [1]
        self.n_constraints = 1
        self.action_rows = 2 * A
        if starts is None or landmarks is None:
            d_starts, d_landmarks = default_starts(self.size, A, E, self.n_landmarks if self.shuffle else 1)
            if starts is None:
                starts = d_starts
            if landmarks is None:
                landmarks = d_landmarks
        starts = np.asarray(starts, dtype=np.float64)
        landmarks = np.asarray(landmarks, dtype=np.float64)
        assert starts.shape == (E, A, 2) and landmarks.shape[0] == E and landmarks.shape[2] == 2
        self.L = landmarks.shape[1]
        f64 = torch.float64
        self.start_x, self.start_y = self._alloc(A, f64), self._alloc(A, f64)
        self.start_x[:, :E] = torch.as_tensor(starts[:, :, 0].T.copy()).to(dev)
        self.start_y[:, :E] = torch.as_tensor(starts[:, :, 1].T.copy()).to(dev)
        self.landmarks = self._alloc(2 * self.L, f64)           # rows lx0, ly0, lx1, ...
        self.landmarks[:, :E] = torch.as_tensor(landmarks.reshape(E, 2 * self.L).T.copy()).to(dev)
        self.pos_x, self.pos_y = self.start_x.clone(), self.start_y.clone()
        self.agent_done = self._alloc(A, torch.uint8)
        self.episode_len = self._alloc(1, torch.int32)[0]          # steps taken before all agents were done
        self.action_buffer = self._alloc(2 * A, torch.float32)  # rows dx0, dy0, dx1, ...
        if self.shuffle:
            self.state_space += 2 * self.L                       # landmarks are part of the state (:65-68)
        self.obs = self._alloc(2 * A + (2 * self.L if self.shuffle else 0), torch.float32)
        self.reward = self._alloc(A, torch.float32)
        self.cost = self._alloc(1, torch.int32)
        self.done = self._alloc(A, torch.uint8)
        self.penalty = self._alloc(1, torch.float32)[0]
        self._params = _lib.CollisionParams(self.size, A, self.L, int(self.shuffle), self.agents_size,
                                            int(self.normalize_state), 0)
        self._params_shared = _lib.CollisionParams(self.size, A, self.L, int(self.shuffle), self.agents_size,
                                                   int(self.normalize_state), 1)

    def _draw_starts(self, episode):
        self._draw_float_starts(episode, 2)                      # agents (:82-84) ...
        _lib.check(self.lib.smarl_random_starts_f64(               # ... then the landmarks (:85, :100-101)
            2, self.size, 0.0, self.seed & (2 ** 64 - 1), episode, self.env_offset, self.n_agents,
            _lib.ptr(self.landmarks), self.landmarks.data_ptr() + 8 * self.ld, 2 * self.ld, self.L, self.n_envs,
            _lib.stream_ptr()))

    def state(self):
        """[n_envs, n_agents, 2] float64 positions (a copy)."""
        E = self.n_envs
        return torch.stack([self.pos_x[:, :E].t(), self.pos_y[:, :E].t()], dim=-1)

    def _reset_impl(self):
        _lib.check(self.lib.smarl_collision_reset(
            C.byref(self._params), _lib.ptr(self.start_x), _lib.ptr(self.start_y), _lib.ptr(self.landmarks),
            _lib.ptr(self.pos_x), _lib.ptr(self.pos_y), _lib.ptr(self.agent_done), _lib.ptr(self.episode_len),
            _lib.ptr(self.obs), self.n_envs, self.ld, _lib.stream_ptr()))

    def _step_impl(self, act, reward, cost, done, lambdas, penalty):
        params = self._params_shared if (reward.shape[0] == 1 and self.n_agents > 1) else self._params
        _lib.check(self.lib.smarl_collision_step(
            C.byref(params), _lib.ptr(self.pos_x), _lib.ptr(self.pos_y), _lib.ptr(self.agent_done),
            _lib.ptr(act), _lib.ptr(self.landmarks), _lib.ptr(self.obs), _lib.ptr(reward), _lib.ptr(cost),
            _lib.ptr(done), _lib.ptr(self.episode_len), _lib.ptr(lambdas), _lib.ptr(penalty), self.n_envs, self.ld,
            _lib.stream_ptr()))

    def _rollout_outputs(self, T, g_mode, out, g_scratch_rows):
        # both fused rollouts also return the episode lengths, n_active
        o = super()._rollout_outputs(T, g_mode, out, g_scratch_rows)
        if "n_active_" not in o:
            o["n_active_"] = self._alloc(1, torch.int32)
        return o

    def rollout(self, actions, lambdas=None, gamma=0.99, thresholds=None, g_mode=G_NONE, out=None):
        """Open-loop fused episode (one launch).  actions ``[T, 2*n_agents, ld]`` float32 (kernel layout,
        rows dx0, dy0, dx1, ...).  Adds ``n_active`` [E]: the episode length T' (main.py:51)."""
        T = int(actions.shape[0])
        A, E = self.n_agents, self.n_envs
        assert actions.dtype == torch.float32 and tuple(actions.shape) == (T, 2 * A, self.ld) and actions.is_contiguous()
        o, acc = self._begin_rollout(T, g_mode, out, 2 * T, gamma, thresholds)
        _lib.check(self.lib.smarl_collision_rollout(
            C.byref(self._params), C.byref(acc), _lib.ptr(self.start_x), _lib.ptr(self.start_y),
            _lib.ptr(self.landmarks), _lib.ptr(actions), _lib.ptr(lambdas), _lib.ptr(self.pos_x), _lib.ptr(self.pos_y),
            _lib.ptr(self.agent_done), _lib.ptr(o["n_active_"]), _lib.ptr(o["R_"]), _lib.ptr(o["modR_"]),
            _lib.ptr(o["C_"]), _lib.ptr(o["G_"]), _lib.ptr(o["gs_"]), _lib.ptr(o["stats_vec"]),
            _lib.ptr(o["stats_scratch"]), E, self.ld, _lib.stream_ptr()))
        o["n_active"] = o["n_active_"][0, :E]
        return self._rollout_result(o)

    def _policy_rollout_impl(self, pol, acc, lambdas, rec, o):
        _lib.check(self.lib.smarl_collision_policy_rollout(
            C.byref(self._params), C.byref(pol), C.byref(acc), _lib.ptr(self.start_x), _lib.ptr(self.start_y),
            _lib.ptr(self.landmarks), _lib.ptr(lambdas), *[_lib.ptr(x) for x in rec], _lib.ptr(self.pos_x),
            _lib.ptr(self.pos_y), _lib.ptr(self.agent_done), _lib.ptr(o["n_active_"]), _lib.ptr(o["R_"]),
            _lib.ptr(o["modR_"]), _lib.ptr(o["C_"]), _lib.ptr(o["G_"]), _lib.ptr(o["gs_"]), _lib.ptr(o["stats_vec"]),
            _lib.ptr(o["stats_scratch"]), self.n_envs, self.ld, _lib.stream_ptr()))
        o["n_active"] = o["n_active_"][0, :self.n_envs]
