"""Shared host logic of the batched envs: buffers in the agent-major SoA layout, action ingest,
reference-oriented views, closed-loop and fused rollout helpers, the one-launch on-policy rollout
and the single-env list adaptor."""
from __future__ import annotations

import numpy as np
import torch

from .. import _lib
from ..layout import alloc, env_major, pad_ld, require_cuda
from ..rollout import G_NONE, G_REWARD_TO_GO, RolloutBuffer, device_thresholds, make_accounting


class BatchedEnv:
    """Base of the batched drop-ins.  Subclasses set ``n_constraints``, ``cost_dtype``,
    ``action_rows``/``action_dtype`` and implement ``_reset_impl`` / ``_step_impl``."""

    cost_dtype = torch.uint8
    action_dtype = torch.uint8

    def _init_common(self, size, n_agents, n_envs, device, env_offset):
        if not (1 <= int(n_agents) <= 32):
            raise ValueError("n_agents must be in 1..32")
        self.size, self.n_agents, self.n_envs = int(size), int(n_agents), int(n_envs)
        self.device = require_cuda(device)
        if self.device.index != torch.cuda.current_device():
            # libsmarl launches on the current device; one process drives one GPU (torchrun model)
            raise ValueError(f"env device {self.device} is not the current CUDA device; call "
                             "torch.cuda.set_device() first")
        self.ld = pad_ld(self.n_envs)
        self.env_offset = int(env_offset)       # global id of env 0 when sharded over GPUs
        self.lib = _lib.load()
        self.t = 0
        self.shuffle = False
        self.seed = 0
        self._episode = 0          # shuffle=True: index of the next episode's start draw
        self.validate_actions = False   # True: also range-check discrete actions handed over as DEVICE tensors (syncs)
        self.emit_obs = True            # False: the step kernels skip the float observation rows (8 of Coverage's 19
                                        # bytes per agent-step); for consumers that read the u8 position rows pos_x /
                                        # pos_y directly, e.g. a fused policy kernel.  env.step then returns obs=None.

    # ---- buffers --------------------------------------------------------------------------------
    def _alloc(self, rows, dtype, lead=()):
        return alloc(rows, self.n_envs, dtype, self.device, lead)

    def _ingest_actions(self, actions, agent_major):
        """Return an ``[action_rows, ld]`` device tensor in the kernel layout (zero-copy when the
        caller already hands one over, e.g. ``env.action_buffer`` filled by the policies)."""
        rows = self.action_rows
        if actions is self.action_buffer:                       # policies wrote the env's own buffer in place
            return actions
        kernel_shape = isinstance(actions, torch.Tensor) and tuple(actions.shape) == (rows, self.ld)
        if kernel_shape and (agent_major or (rows, self.ld) != (self.n_envs, rows)):
            # already in the kernel layout (unambiguous shape, or the caller said so): zero-copy
            if actions.device == self.device and actions.dtype == self.action_dtype and actions.is_contiguous():
                return actions
            self.action_buffer.copy_(actions)
            return self.action_buffer
        a = torch.as_tensor(np.asarray(actions) if not isinstance(actions, torch.Tensor) else actions)
        if self.action_dtype == torch.uint8 and (not a.is_cuda or self.validate_actions) and a.numel():
            # the reference indexes its direction / cost tables with the action (coverage.py:176-196,
            # congestion.py:55-69) and raises IndexError beyond them; the kernels' bit tricks would decode such a
            # byte as some other move.  Host arrays are checked for free; device tensors only on request (a sync).
            lo, hi = int(a.min()), int(a.max())
            if lo < 0 or hi >= self.action_space:
                raise IndexError(f"discrete action outside 0..{self.action_space - 1} (got {lo if lo < 0 else hi})")
        a = a.to(self.device)
        if not agent_major:                                   # reference orientation: [E, A(, 2)]
            a = a.reshape(self.n_envs, rows).t()
        else:
            a = a.reshape(rows, -1)[:, : self.n_envs]
        self.action_buffer[:, : self.n_envs].copy_(a)
        return self.action_buffer

    def _views(self, reward, cost, done):
        E = self.n_envs
        return (env_major(self.obs, E), env_major(reward, E), env_major(cost, E), env_major(done, E))

    # ---- reference protocol ---------------------------------------------------------------------
    def reset(self):
        """``env.reset()`` for every env: returns the observation ``[n_envs, state_space]`` (a view;
        row e is ``np.array(state).flatten()`` of env e, main.py:33)."""
        self.t = 0
        self._maybe_shuffle()
        self._reset_impl()
        return env_major(self.obs, self.n_envs)

    def _maybe_shuffle(self):
        """shuffle=True (coverage.py:31-43, congestion.py:42-43, collision_avoidance.py:75-89): draw
        this episode's starts on the device before the reset / fused rollout reads them."""
        if self.shuffle:
            self._draw_starts(self._episode)
            self._episode += 1

    def _draw_grid_starts(self, episode, kind):
        _lib.check(self.lib.smarl_random_starts_u8(kind, self.size, self.seed & (2 ** 64 - 1), episode, self.env_offset,
                                                   _lib.ptr(self.start_x), _lib.ptr(self.start_y), self.n_agents,
                                                   self.n_envs, self.ld, _lib.stream_ptr()))

    def _draw_float_starts(self, episode, kind, zoom=0.0):
        _lib.check(self.lib.smarl_random_starts_f64(kind, self.size, float(zoom), self.seed & (2 ** 64 - 1), episode,
                                                    self.env_offset, 0, _lib.ptr(self.start_x), _lib.ptr(self.start_y),
                                                    self.ld, self.n_agents, self.n_envs, _lib.stream_ptr()))

    def step(self, actions, lambdas=None, out=None, agent_major=False):
        """``env.step(actions)`` for every env.

        actions  ``[n_envs, n_agents(, 2)]`` (reference orientation) or, with ``agent_major=True``
                 / the env's own ``action_buffer``, the kernel layout.
        lambdas  optional f64 device tensor [K]: fuses MetaAgent.act's penalty <lambda, c> into the
                 step (written to ``out.penalty[t]`` / ``self.penalty``).
        out      optional (RolloutBuffer, t): write reward/cost/done/penalty into slab t.
        Returns (obs [E, S], reward [E, A], cost [E, K], done [E, A]) -- views, valid until the
        next step.
        """
        act = self._ingest_actions(actions, agent_major)
        if out is not None:
            reward, cost, done, penalty, reward_v, cost_v, done_v = out[0].slot(out[1])
        else:
            own = self.__dict__.get("_own_slot")
            if own is None:
                E = self.n_envs
                own = self._own_slot = (self.reward, self.cost, self.done, self.penalty, env_major(self.reward, E),
                                        env_major(self.cost, E), env_major(self.done, E))
            reward, cost, done, penalty, reward_v, cost_v, done_v = own
        self._step_impl(act, reward, cost, done, lambdas, penalty if lambdas is not None else None)
        self.t += 1
        if done_v is None:                     # not stored per step: this env's agents never finish
            done_v = self.__dict__.get("_done_zeros_v")
            if done_v is None:
                done_v = self._done_zeros_v = env_major(self._zero_done(), self.n_envs)
        if not self.emit_obs:
            return None, reward_v, cost_v, done_v
        obs_v = self.__dict__.get("_obs_v")
        if obs_v is None:
            obs_v = self._obs_v = env_major(self.obs, self.n_envs)
        return obs_v, reward_v, cost_v, done_v

    def _zero_done(self):
        if not hasattr(self, "_done_zeros"):
            self._done_zeros = self._alloc(self.n_agents, torch.uint8)
        return self._done_zeros

    def _rollout_outputs(self, T, g_mode, out, g_scratch_rows):
        """Allocate (or reuse from ``out``) the product buffers of a fused rollout."""
        from ..rollout import G_NONE
        A, K, E, dev = self.n_agents, self.n_constraints, self.n_envs, self.device
        o = out if out is not None else {}

        def buf(name, rows, dtype, lead=()):
            # a buffer reused from a caller's dict must fit THIS call (a longer T or another g_mode than the call that
            # created it would let the kernels write past its end): wrong shape or dtype => allocate afresh
            want = tuple(lead) + (rows, self.ld)
            have = o.get(name)
            if have is None or tuple(have.shape) != want or have.dtype != dtype:
                o[name] = self._alloc(rows, dtype, lead)
            return o[name]
        buf("R_", A, torch.float32), buf("modR_", A, torch.float32)
        buf("C_", K, torch.float32 if self.cost_dtype == torch.float32 else torch.int32)
        o["G_"] = buf("G_buf", A, torch.float32, (T,)) if g_mode != G_NONE else None
        o["gs_"] = buf("g_scratch", 1, torch.float32, (g_scratch_rows,)) if g_mode == G_REWARD_TO_GO else None
        n_stats, n_scratch = self.lib.smarl_stats_len(A, K), self.lib.smarl_stats_scratch_len(A, K, E)
        if o.get("stats_vec") is None or o["stats_vec"].numel() != n_stats or o["stats_scratch"].numel() < n_scratch:
            o["stats_vec"] = torch.zeros(n_stats, dtype=torch.float64, device=dev)
            o["stats_scratch"] = torch.zeros(n_scratch, dtype=torch.float64, device=dev)
        return o

    def _begin_rollout(self, T, g_mode, out, g_scratch_rows, gamma, thresholds):
        """What every fused rollout does before its launch: the product buffers (``_rollout_outputs``), the
        accounting block and, with shuffle=True, this episode's start draw.  Returns (o, acc)."""
        o = self._rollout_outputs(T, g_mode, out, g_scratch_rows)
        thr = device_thresholds(thresholds, self.device, self.n_constraints)
        acc = make_accounting(gamma, T, g_mode, thr)
        self._maybe_shuffle()
        return o, acc

    def _policy_records(self, o, T, S, record):
        """The record slabs of an on-policy rollout in ``o``: ``obs_`` [T, S, ld], ``actions_`` [T, action_rows, ld]
        of ``action_dtype`` and ``logp_`` [T, A, ld] (allocated unless ``o`` holds them in this shape and dtype), and
        their views ``obs`` [T, E, S], ``actions`` [T, A, E, 2] (continuous actions) or [T, A, E] (discrete) and
        ``logp`` [T, A, E].  Returns the three slabs the kernel writes, or three ``None`` with ``record=False``, which
        also drops the records ``o`` held from an earlier call."""
        if not record:
            for name in ("obs_", "actions_", "logp_", "obs", "actions", "logp"):
                o.pop(name, None)
            return [None, None, None]
        A, E = self.n_agents, self.n_envs
        for name, rows, dtype in (("obs_", S, torch.float32), ("actions_", self.action_rows, self.action_dtype),
                                  ("logp_", A, torch.float32)):
            have = o.get(name)
            if have is None or tuple(have.shape) != (T, rows, self.ld) or have.dtype != dtype:
                o[name] = self._alloc(rows, dtype, (T,))
        o["obs"] = o["obs_"][:, :, :E].permute(0, 2, 1)
        o["actions"] = o["actions_"][:, :, :E]
        if self.action_rows != A:                                        # rows dx0, dy0, dx1, ...
            o["actions"] = o["actions"].view(T, A, 2, E).permute(0, 1, 3, 2)
        o["logp"] = o["logp_"][:, :, :E]
        return [o["obs_"], o["actions_"], o["logp_"]]

    def _rollout_result(self, o):
        from ..rollout import Stats
        A, K, E = self.n_agents, self.n_constraints, self.n_envs
        o.update(R=env_major(o["R_"], E), modR=env_major(o["modR_"], E), C=env_major(o["C_"], E),
                 G=None if o["G_"] is None else env_major(o["G_"], E), stats=Stats(o["stats_vec"], A, K))
        return o

    def new_rollout_buffer(self, n_steps, g_mode=G_REWARD_TO_GO, lean=False, store_done=None):
        """Device slabs for one batch of episodes.  Envs whose agents never finish (check_done is constant
        False: coverage.py:97-98, congestion.py:103-104) do not store per-step done flags unless
        ``store_done=True``: ``env.step`` still returns the all-False done array (one cached zero view), but the
        step kernel writes one byte per agent-step less.  ``lean=True`` (envs that support it) also replaces the
        n_agents weighted reward rows by one env-reward row; ``env.step`` then returns the ``[E, 1]`` env reward
        and per-agent rewards are ``buffer.rewards()``."""
        if lean and not getattr(self, "supports_lean", False):
            raise ValueError(f"{type(self).__name__} has no lean rollout buffer")
        if store_done is None:
            store_done = not getattr(self, "never_done", False)
        return RolloutBuffer(n_steps, self.n_agents, self.n_constraints, self.n_envs, self.cost_dtype,
                             self.device, g_mode, shared_reward=lean, weights=getattr(self, "_weights", None) if lean else None,
                             store_done=store_done)

    def rollout_closed_loop(self, policy, n_steps, lambdas, gamma, thresholds=None, buffer=None,
                            g_mode=G_REWARD_TO_GO):
        """main.py:28-57 for all envs: ``policy(obs, t) -> actions`` is called between steps (it may
        write ``env.action_buffer`` in place and return it).  Returns RolloutBuffer.finish()."""
        buf = buffer if buffer is not None else self.new_rollout_buffer(n_steps, g_mode)
        obs = self.reset()
        for t in range(n_steps):
            actions = policy(obs, t)
            agent_major = isinstance(actions, torch.Tensor) and actions.data_ptr() == self.action_buffer.data_ptr()
            obs, _, _, _ = self.step(actions, lambdas=lambdas, out=(buf, t), agent_major=agent_major)
        out = buf.finish(gamma, thresholds, g_mode, n_active=getattr(self, "episode_len", None))
        out["buffer"] = buf
        return out


class PolicyRollout:
    """``policy_rollout`` of the envs that run a whole on-policy episode in one launch (BatchedEnv subclasses).  The env
    supplies ``rollout_policy`` (the name of the fused policy class it samples, in ``policy.py``),
    ``reference_policy`` (the reference's policy that class implements), ``rollout_threads`` (how its kernel maps
    envs to threads, up to 8 agents) and ``_policy_rollout_impl(pol, acc, lambdas, rec, o)``, its C entry point's
    call."""

    def policy_rollout(self, policy, n_steps, lambdas=None, gamma=0.99, thresholds=None, g_mode=G_NONE, record=True,
                       out=None):
        """Whole on-policy episode in one launch: every step samples ``policy`` (a ``FusedGaussianPolicy`` for the
        continuous envs, a ``FusedDiscretePolicy`` for CoverageDiscrete and Congestion (``BatchedCongestionOnPolicy``),
        a ``FusedDiscretizedPolicy`` for CoverageDiscretized (``BatchedCoverageDiscretizedOnPolicy``): its weights,
        seed and episode) on the current observation, steps the env and accumulates what ``rollout``
        returns (CollisionAvoidance's ``n_active`` included).  The records and the final state are the bits of the closed loop reset + T x
        (``policy.act(t=t)``, ``env.step``) (for the discrete envs with the FP32-pipe policy build,
        ``_lib.kernel_variant(_lib.KERNEL_POLICY, 0)``), the products those of ``rollout`` fed the recorded actions.
        Congestion draws its action noise as the closed loop does: the call advances the noise episode like ``reset``
        and ``rollout``, so after ``set_noise_episode(n)`` both draw the noise of episode ``n``.
        The episode index of ``policy`` is not advanced: call ``policy.next_episode()`` for fresh samples.  With
        ``record`` it adds views of the kernel-layout slabs ``obs_`` [T, S, ld], ``actions_`` [T, action_rows, ld]
        (what ``rollout`` takes) and ``logp_`` [T, A, ld]: ``obs`` [T, E, S], ``actions`` [T, A, E, 2] (continuous)
        or [T, A, E] (discrete) and ``logp`` [T, A, E], so that ``policy.log_prob(out["obs"][t], out["actions"][t])``
        is the learner's differentiable side.  With ``record=False`` the returned dict holds no records, also when
        ``out`` held some.  With ``out`` reused the call allocates nothing (CUDA-graph capturable)."""
        from .. import policy as policies
        if not isinstance(policy, getattr(policies, self.rollout_policy)):
            raise NotImplementedError(f"policy_rollout runs the reference's {self.reference_policy}: pass a "
                                      f"{self.rollout_policy}")
        if self.n_agents > 8:
            raise NotImplementedError(f"policy_rollout runs {self.rollout_threads}, for n_agents up to 8")
        pol = policy.c_params(self)
        T = int(n_steps)
        o = out if out is not None else {}
        rec = self._policy_records(o, T, self.obs.shape[0], record)
        o, acc = self._begin_rollout(T, g_mode, o, 2 * T, gamma, thresholds)
        self._policy_rollout_impl(pol, acc, lambdas, rec, o)
        return self._rollout_result(o)


class SingleEnvAdapter:
    """Wrap a batched env with n_envs == 1 so the reference's unmodified driver loop
    (main.py:28-57) can drive it: Python lists in, Python lists out."""

    def __init__(self, env):
        if env.n_envs != 1:
            raise ValueError("SingleEnvAdapter needs n_envs == 1")
        self.env = env

    def __getattr__(self, name):
        return getattr(self.env, name)

    def reset(self):
        self.env.reset()
        return self.env.state()[0].cpu().numpy().astype(np.float64).tolist()

    def step(self, action):
        a = np.asarray(action, dtype=np.float64).reshape(1, self.env.n_agents, -1)
        if self.env.action_dtype == torch.uint8:
            a = a.reshape(1, self.env.n_agents).astype(np.uint8)
        else:
            a = a.astype(np.float32)
        obs, r, c, d = self.env.step(a)
        state = self.env.state()[0].cpu().numpy().astype(np.float64).tolist()
        return (state, r[0].cpu().numpy().astype(np.float64).tolist(),
                c[0].cpu().numpy().astype(np.float64).tolist(), d[0].cpu().numpy().astype(bool).tolist())
