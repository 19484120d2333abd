"""Batched policy glue (SURVEY.md section 8f-1): the n_agents independent policies of the reference
(one DiscretePolicy / ContinuousPolicy per agent, safe_multi_agent_RL/agent.py:23-76, each fed the
joint state ``np.array(state).flatten()``, main.py:32-35) evaluated for ALL envs at once.

This is plain PyTorch on purpose -- 16-unit MLPs are not the hot path -- but it closes the loop
without a host round trip: ``obs`` is the env's own ``[E, S]`` view (no copy), the per-agent
weights are stacked so one batched matmul serves all agents, and sampled actions are written
straight into ``env.action_buffer`` (the kernel layout ``[rows, ld]``), which ``env.step`` takes
zero-copy with ``agent_major=True``.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn
import torch.nn.functional as F


class _Stacked(nn.Module):
    """A independent ``nn.Linear(in, out)`` layers as one [A, in, out] parameter (default Linear init)."""

    def __init__(self, n, fan_in, fan_out):
        super().__init__()
        bound = 1.0 / math.sqrt(fan_in)
        self.weight = nn.Parameter(torch.empty(n, fan_in, fan_out).uniform_(-bound, bound))
        self.bias = nn.Parameter(torch.empty(n, 1, fan_out).uniform_(-bound, bound))

    def forward(self, x):            # x [A, E, in] or [E, in] (shared input)
        return torch.matmul(x, self.weight) + self.bias


class BatchedDiscretePolicy(nn.Module):
    """``DiscretePolicy`` (agent.py:23-47) x n_agents: fc1 -> relu -> fc2 -> softmax -> Categorical."""

    def __init__(self, env, hidden_size=16):
        super().__init__()
        self.env = env
        self.fc1 = _Stacked(env.n_agents, env.state_space, hidden_size)
        self.fc2 = _Stacked(env.n_agents, hidden_size, env.action_space)
        self.to(env.device)

    def logits(self, obs):           # obs [E, S] -> [A, E, n_actions]
        return self.fc2(F.relu(self.fc1(obs)))

    def dist(self, obs):
        return torch.distributions.Categorical(logits=self.logits(obs), validate_args=False)   # no host sync: graph-capturable

    @torch.no_grad()
    def act(self, obs):
        """Sample one action per (agent, env); writes ``env.action_buffer`` in place and returns
        (action_buffer, actions [A, E] int64, log_prob [A, E])."""
        d = self.dist(obs)
        a = d.sample()
        self.env.action_buffer[:, : self.env.n_envs].copy_(a)
        return self.env.action_buffer, a, d.log_prob(a)

    def log_prob(self, obs, actions):
        return self.dist(obs).log_prob(actions)


class _PolicyGradLoss(torch.autograd.Function):
    """The loss of ``_FusedDiscreteSampler.policy_gradient_loss``: the forward makes the one launch and keeps the
    gradients, the backward scales them by ``grad_output``."""

    @staticmethod
    def forward(ctx, w1, b1, w2, b2, call):
        import ctypes as C
        pol, obs_, act_, psi, T, scale, scratch = call
        env, L = pol.env, pol._lib_mod
        p = pol.c_params(env)
        grads = [torch.empty_like(w) for w in (w1, b1, w2, b2)]
        loss = torch.empty((), dtype=torch.float64, device=env.device)
        L.check(pol.lib.smarl_policy_grad_discrete(C.byref(p), L.ptr(obs_), L.ptr(act_), L.ptr(psi), T, scale,
                                                   *[L.ptr(g) for g in grads], L.ptr(loss), L.ptr(scratch),
                                                   env.n_envs, env.ld, L.stream_ptr()))
        ctx.save_for_backward(*grads)
        return loss.float()

    @staticmethod
    def backward(ctx, grad_output):
        return (*[grad_output * g for g in ctx.saved_tensors], None)


class _FusedDiscreteSampler(BatchedDiscretePolicy):
    """What the fused DiscretePolicy kernels share: the Philox sampling stream (``seed`` and a device episode index),
    the log-probability row and the ``SmarlDiscretePolicy`` block of the weights.  Subclasses set ``n_actions``, the
    action count their kernel is built for."""

    n_actions = None

    def __init__(self, env, hidden_size=16, seed=0):
        super().__init__(env, hidden_size)
        from . import _lib
        self._lib_mod, self.lib = _lib, _lib.load()
        self.seed = int(seed)
        self.logp = torch.zeros(env.n_agents, env.ld, dtype=torch.float32, device=env.device)
        self._episode_dev = torch.zeros(1, dtype=torch.int32, device=env.device)

    def next_episode(self):
        """Advance the sampling stream's episode index (a device-side increment: CUDA-graph capturable)."""
        self._episode_dev.add_(1)

    def c_params(self, env):
        """The ``SmarlDiscretePolicy`` of these weights and this sampling stream for ``env`` (its env_offset).  Raises
        ValueError when the weights are not those of ``env``'s agent count: the kernels read ``env.n_agents`` agents'
        networks of ``env.state_space`` inputs."""
        L = self._lib_mod
        w = [t_.detach() for t_ in (self.fc1.weight, self.fc1.bias, self.fc2.weight, self.fc2.bias)]
        assert all(x.is_contiguous() and x.dtype == torch.float32 for x in w)
        A, S = self.fc1.weight.shape[:2]
        if (A, S) != (env.n_agents, env.state_space):
            raise ValueError(f"the policy holds {A} agents' networks of {S} inputs; the env has {env.n_agents} agents "
                             f"and {env.state_space} inputs")
        return L.DiscretePolicyParams(A, 16, self.n_actions, 0, L.ptr(w[0]), L.ptr(w[1]), L.ptr(w[2]), L.ptr(w[3]),
                                      self.seed & (2 ** 64 - 1), env.env_offset, L.ptr(self._episode_dev))

    def policy_gradient_loss(self, records, psi, scale=None):
        """The REINFORCE / actor loss ``-(psi * log pi(a|s)).sum() * scale`` (agent.py:134-157) of the episodes a
        ``policy_rollout`` recorded, as ONE libsmarl kernel (smarl_policy_grad_discrete) that reads the record slabs
        ``records["obs_"]`` / ``records["actions_"]`` and computes the loss and its gradients with respect to fc1 / fc2
        at once.  ``psi`` [T, A, E] float32 is the constant advantage (no gradient flows into it); the
        ``[:, :, :E]`` view of a contiguous [T, A, ld] slab is read in place, anything else is copied into one.
        ``scale`` defaults to 1 / (T A E), i.e. ``.mean()``.  Returns a 0-dim float32 loss whose ``backward()``
        accumulates ``grad_output x`` the kernel's gradients into ``fc1`` / ``fc2``'s ``.grad`` as the PyTorch loss
        does."""
        env = self.env
        self.c_params(env)                                # the weights are this env's agent count and input width
        A, E, ld = env.n_agents, env.n_envs, env.ld
        obs_, act_ = records.get("obs_"), records.get("actions_")
        if obs_ is None or act_ is None:
            raise ValueError("records hold no obs_ / actions_ slabs: call policy_rollout with record=True")
        T = obs_.shape[0]
        if (tuple(obs_.shape) != (T, 2 * A, ld) or tuple(act_.shape) != (T, A, ld) or obs_.dtype != torch.float32
                or act_.dtype != torch.uint8 or not obs_.is_contiguous() or not act_.is_contiguous()):
            raise ValueError(f"records of shape {tuple(obs_.shape)} / {tuple(act_.shape)} are not those of this env "
                             f"({A} agents, ld {ld})")
        if not isinstance(psi, torch.Tensor) or tuple(psi.shape) != (T, A, E) or psi.dtype != torch.float32:
            raise ValueError(f"psi must be a float32 tensor of shape {(T, A, E)}")
        if psi.requires_grad:
            raise ValueError("psi requires grad: it is a constant advantage and the kernel has no gradient for it; "
                             "pass psi.detach()")
        if psi.device != env.device:
            raise ValueError(f"psi is on {psi.device}, the records on {env.device}")
        if psi.stride() != (A * ld, ld, 1) or psi.data_ptr() % 16:
            slab = self.__dict__.get("_psi_slab")
            if slab is None or tuple(slab.shape) != (T, A, ld):
                slab = self._psi_slab = torch.zeros(T, A, ld, dtype=torch.float32, device=env.device)
            slab[:, :, :E].copy_(psi)
            psi = slab
        scale = 1.0 / (T * A * E) if scale is None else float(scale)
        n = int(self.lib.smarl_policy_grad_scratch_len(A, self.n_actions, T, E))
        if n < 0:
            raise ValueError(f"no policy gradient for {A} agents, {self.n_actions} actions, T = {T}, E = {E}")
        scratch = self.__dict__.get("_grad_scratch")
        if scratch is None or scratch.numel() < n:
            scratch = self._grad_scratch = torch.empty(n, dtype=torch.float64, device=env.device)
        return _PolicyGradLoss.apply(self.fc1.weight, self.fc1.bias, self.fc2.weight, self.fc2.bias,
                                     (self, obs_, act_, psi, T, scale, scratch))


class FusedDiscretePolicy(_FusedDiscreteSampler):
    """``BatchedDiscretePolicy`` whose ``act`` is ONE libsmarl kernel (smarl_policy_act_discrete): it reads the env's u8
    position rows (not the float observation: the env may run with ``emit_obs = False``), evaluates every agent's
    2A -> 16 -> 5 MLP -- fc1 as tcgen05 tensor-core GEMMs over 256-env tiles with f32-grade accuracy (exact bf16
    positions x three bf16 pieces per fp32 weight, f32 accumulators in tensor memory), the rest on the FP32 pipes out of
    tensor memory -- samples the Categorical with a Philox stream keyed by (global env id, episode, step, agent) and
    writes ``env.action_buffer`` and the log-probabilities: about 7 bytes of HBM traffic per agent-step instead of the
    [A, E, 16] / [A, E, 5] intermediates of the PyTorch forward.  ``_lib.kernel_variant(_lib.KERNEL_POLICY, 0)`` forces
    the FP32-pipe build of the kernel.
    ``log_prob`` / ``dist`` (the differentiable path the learners train through) stay the parent's."""

    n_actions = 5

    def __init__(self, env, hidden_size=16, seed=0):
        if hidden_size != 16 or env.action_space != 5 or env.state_space != 2 * env.n_agents:
            raise NotImplementedError("the fused kernel is built for the reference's DiscretePolicy on the grid envs: "
                                      "state_space = 2 n_agents, hidden 16, 5 actions")
        super().__init__(env, hidden_size, seed)

    @torch.no_grad()
    def act(self, obs=None, t=None):
        """Sample actions for step ``t`` (default: the env's step counter) into ``env.action_buffer``; returns
        (action_buffer, actions [A, E] uint8 view, log_prob [A, E] view).  ``obs`` is ignored: the kernel reads
        ``env.pos_x`` / ``env.pos_y``."""
        import ctypes as C
        env, L = self.env, self._lib_mod
        p = self.c_params(env)
        L.check(self.lib.smarl_policy_act_discrete(C.byref(p), L.ptr(env.pos_x), L.ptr(env.pos_y),
                                                   L.ptr(env.action_buffer), L.ptr(self.logp),
                                                   int(env.t if t is None else t), env.n_envs, env.ld, L.stream_ptr()))
        E = env.n_envs
        return env.action_buffer, env.action_buffer[:, :E], self.logp[:, :E]


class FusedDiscretizedPolicy(_FusedDiscreteSampler):
    """``BatchedDiscretePolicy`` on CoverageDiscretized (9 actions) whose ``act`` is ONE libsmarl kernel
    (smarl_policy_act_discretized): it reads the env's f32 observation rows ``env.obs`` (the positions are float64
    multiples of 1 / zoom, not u8 cells), evaluates every agent's 2A -> 16 -> 9 MLP on the FP32 pipes with the weights in
    shared memory, samples the Categorical from ``FusedDiscretePolicy``'s Philox stream (global env id, episode, step,
    agent) and writes ``env.action_buffer`` and the log-probabilities.  A sibling of ``FusedDiscretePolicy``, not a
    subclass: each env's ``policy_rollout`` takes exactly one of the two.
    ``log_prob`` / ``dist`` (the differentiable path the learners train through) stay the parent's."""

    n_actions = 9

    def __init__(self, env, hidden_size=16, seed=0):
        if (hidden_size != 16 or env.action_space != 9 or env.state_space != 2 * env.n_agents
                or getattr(env, "obs", None) is None or env.obs.dtype != torch.float32):
            raise NotImplementedError("the fused kernel is built for the reference's DiscretePolicy on "
                                      "CoverageDiscretized: state_space = 2 n_agents, hidden 16, 9 actions, f32 "
                                      "observation rows")
        super().__init__(env, hidden_size, seed)

    @torch.no_grad()
    def act(self, obs=None, t=None):
        """Sample actions for step ``t`` (default: the env's step counter) into ``env.action_buffer``; returns
        (action_buffer, actions [A, E] uint8 view, log_prob [A, E] view).  ``obs`` is ignored: the kernel reads
        ``env.obs``."""
        import ctypes as C
        env, L = self.env, self._lib_mod
        p = self.c_params(env)
        L.check(self.lib.smarl_policy_act_discretized(C.byref(p), L.ptr(env.obs), L.ptr(env.action_buffer),
                                                      L.ptr(self.logp), int(env.t if t is None else t), env.n_envs,
                                                      env.ld, L.stream_ptr()))
        E = env.n_envs
        return env.action_buffer, env.action_buffer[:, :E], self.logp[:, :E]


class BatchedGaussianPolicy(nn.Module):
    """``ContinuousPolicy`` (agent.py:50-76) x n_agents: diagonal Gaussian with variance relu(.) + 1e-4."""

    def __init__(self, env, hidden_size=16):
        super().__init__()
        self.env = env
        self.fc1 = _Stacked(env.n_agents, env.state_space, hidden_size)
        self.fc2 = _Stacked(env.n_agents, hidden_size, env.action_space)
        self.fc2_ = _Stacked(env.n_agents, hidden_size, env.action_space)
        self.to(env.device)

    def dist(self, obs):
        h = F.relu(self.fc1(obs))
        mu, var = self.fc2(h), F.relu(self.fc2_(h)) + 1e-4
        return torch.distributions.Independent(torch.distributions.Normal(mu, var.sqrt(), validate_args=False), 1,
                                              validate_args=False)

    @torch.no_grad()
    def act(self, obs):
        """actions [A, E, 2] float32 -> ``env.action_buffer`` rows dx0, dy0, dx1, ... in place."""
        d = self.dist(obs)
        base = d.base_dist
        # mu + sigma * eps instead of d.sample(): torch.normal(mean, std) checks std >= 0 on the host, which a CUDA-graph
        # capture does not allow
        a = base.loc + base.scale * torch.randn_like(base.loc)
        A, E = self.env.n_agents, self.env.n_envs
        self.env.action_buffer[:, :E].view(A, 2, E).copy_(a.permute(0, 2, 1))
        return self.env.action_buffer, a, d.log_prob(a)

    def log_prob(self, obs, actions):
        return self.dist(obs).log_prob(actions)


class FusedGaussianPolicy(BatchedGaussianPolicy):
    """``BatchedGaussianPolicy`` whose ``act`` is ONE libsmarl kernel (smarl_policy_act_gaussian): it reads the env's
    f32 observation rows, evaluates every agent's ``S -> 16 -> (mu, sigma^2)`` network with the weights in shared
    memory, samples ``a ~ N(mu, diag(sigma^2))`` by Box-Muller from a Philox stream keyed by (global env id, episode,
    step, agent) and writes ``env.action_buffer`` (rows dx0, dy0, dx1, ...) and the log-probabilities.
    ``log_prob`` / ``dist`` (the differentiable path) stay the parent's."""

    def __init__(self, env, hidden_size=16, seed=0):
        if hidden_size != 16 or env.action_space != 2 or not hasattr(env, "obs"):
            raise NotImplementedError("the fused kernel is built for the reference's ContinuousPolicy on the continuous "
                                      "envs: hidden 16, 2 actions, f32 observation rows")
        super().__init__(env, hidden_size)
        from . import _lib
        self._lib_mod, self.lib = _lib, _lib.load()
        self.seed = int(seed)
        self.logp = torch.zeros(env.n_agents, env.ld, dtype=torch.float32, device=env.device)
        self._episode_dev = torch.zeros(1, dtype=torch.int32, device=env.device)

    def next_episode(self):
        self._episode_dev.add_(1)

    def c_params(self, env):
        """The ``SmarlGaussianPolicy`` of these weights and this sampling stream for ``env`` (its env_offset)."""
        L = self._lib_mod
        w = [t_.detach() for t_ in (self.fc1.weight, self.fc1.bias, self.fc2.weight, self.fc2.bias, self.fc2_.weight,
                                    self.fc2_.bias)]
        assert all(x.is_contiguous() and x.dtype == torch.float32 for x in w)
        S = env.obs.shape[0]
        assert S == env.state_space == self.fc1.weight.shape[1]
        return L.GaussianPolicyParams(env.n_agents, S, 16, 2, 0, 0, *[L.ptr(x) for x in w], self.seed & (2 ** 64 - 1),
                                      env.env_offset, L.ptr(self._episode_dev))

    @torch.no_grad()
    def act(self, obs=None, t=None):
        """Sample actions for step ``t`` into ``env.action_buffer``; returns (action_buffer, actions [A, E, 2] view,
        log_prob [A, E] view).  ``obs`` is ignored: the kernel reads ``env.obs``."""
        import ctypes as C
        env, L = self.env, self._lib_mod
        p = self.c_params(env)
        L.check(self.lib.smarl_policy_act_gaussian(C.byref(p), L.ptr(env.obs), L.ptr(env.action_buffer), L.ptr(self.logp),
                                                   int(env.t if t is None else t), env.n_envs, env.ld, L.stream_ptr()))
        A, E = env.n_agents, env.n_envs
        return env.action_buffer, env.action_buffer[:, :E].view(A, 2, E).permute(0, 2, 1), self.logp[:, :E]
