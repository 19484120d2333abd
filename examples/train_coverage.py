#!/usr/bin/env python
"""Constrained policy-gradient training on the batched CoverageDiscrete env: the reference's loop
(main.py:25-68: meta cycles x agent cycles x batch of episodes) with the batch dimension on the GPU.

    python examples/train_coverage.py --n_envs 4096 --meta_cycles 5 --agent_cycles 10 [--fused]

Per agent cycle: one closed-loop batch of n_envs episodes (policies -> env.step with the penalty
<lambda, c> fused -> rollout buffer), one accounting launch (returns, cost sums, reward-to-go,
stats), a REINFORCE-with-reward-to-go update of the n_agents policies; per meta cycle the
lambda update from the (all-reduced) cost statistics (meta_agent.py:32-39).

--fused: the batch is ONE launch instead (env.policy_rollout with a FusedDiscretePolicy: policies, sampling, steps
and accounting in one kernel, DESIGN.md section 3.13); the same loss is computed from its records, and
policy.next_episode() moves the sampling stream on so that the next batch draws fresh samples.

--fused_grad (with --fused): the loss and its gradients come from ONE kernel too (policy.policy_gradient_loss on the
records, DESIGN.md section 3.16) instead of T log_prob forwards and an autograd backward; Adam stays torch.optim."""
import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import safe_multiagent_rl_b200 as smarl  # noqa: E402
from safe_multiagent_rl_b200.policy import BatchedDiscretePolicy, FusedDiscretePolicy  # noqa: E402


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=5)
    ap.add_argument("--n_agents", type=int, default=3)
    ap.add_argument("--n_envs", type=int, default=4096)
    ap.add_argument("--max_t", type=int, default=50)
    ap.add_argument("--gamma", type=float, default=0.999)
    ap.add_argument("--meta_cycles", type=int, default=5)
    ap.add_argument("--agent_cycles", type=int, default=10)
    ap.add_argument("--actor_lr", type=float, default=0.01)
    ap.add_argument("--meta_lr", type=float, default=0.02)
    ap.add_argument("--thresholds", type=float, nargs="*", default=[25.0, 25.0, 25.0])
    ap.add_argument("--weights", type=float, nargs="*", default=[1.0, 2.0, 3.0])
    ap.add_argument("--fused", action="store_true", help="one launch per batch (env.policy_rollout)")
    ap.add_argument("--fused_grad", action="store_true",
                    help="with --fused: loss and gradients in one launch (policy.policy_gradient_loss)")
    a = ap.parse_args(argv)
    if a.fused_grad and not a.fused:
        ap.error("--fused_grad needs --fused")
    return a


def train(a):
    """The training loop; returns the policy."""
    torch.manual_seed(0)
    A, E, T = a.n_agents, a.n_envs, a.max_t
    env = smarl.BatchedCoverageDiscrete(a.size, A, n_envs=E, weights=a.weights, shuffle=True, seed=0)
    meta = smarl.BatchedMetaAgent(env.constraint_space, a.gamma, a.meta_lr, a.thresholds,
                                  start_learning_cycle=max(0, a.agent_cycles - 4), n_agents=A)
    policy = FusedDiscretePolicy(env) if a.fused else BatchedDiscretePolicy(env)
    opt = torch.optim.Adam(policy.parameters(), lr=a.actor_lr)
    buf = env.new_rollout_buffer(T)
    hist = smarl.BatchedBuffer(argparse.Namespace(gamma=a.gamma, thresholds=a.thresholds))
    obs_log = torch.empty(T, E, env.state_space, device=env.device)
    act_log = torch.empty(T, A, E, dtype=torch.long, device=env.device)
    out = None                      # --fused: the product and record buffers, reused by every batch
    for mc in range(a.meta_cycles):
        for ac in range(a.agent_cycles):
            if a.fused:
                out = env.policy_rollout(policy, T, lambdas=meta.lambdas, gamma=a.gamma, thresholds=a.thresholds,
                                         g_mode=smarl.G_REWARD_TO_GO, out=out)
                obs_log, act_log = out["obs"], out["actions"].long()
            else:
                obs = env.reset()
                for t in range(T):
                    obs_log[t].copy_(obs)
                    act_buf, act, _ = policy.act(obs)
                    act_log[t] = act
                    obs, _, _, _ = env.step(act_buf, lambdas=meta.lambdas, out=(buf, t), agent_major=True)
                out = buf.finish(a.gamma, a.thresholds)
            hist.extend(out["R"], out["modR"], out["C"])
            meta.step(out["stats"])
            G = out["G"].permute(0, 2, 1)                                   # [T, A, E] reward-to-go of r - <lambda, c>
            adv = (G - G.mean(dim=2, keepdim=True)) / (G.std(dim=2, keepdim=True) + 1e-6)
            if a.fused_grad:
                loss = policy.policy_gradient_loss(out, adv)
            else:
                logp = torch.stack([policy.log_prob(obs_log[t], act_log[t]) for t in range(T)])
                loss = -(logp * adv).mean()
            opt.zero_grad()
            loss.backward()
            opt.step()
            if a.fused:
                policy.next_episode()
            meta.increment_learning_cycle()
        meta.update()
        hist.append_lambdas(meta.lambdas)
        s, ms, viol = hist.mean_score(n=E)
        print(f"meta {mc}: score {s.round(2)}  cost - thr {[round(float(v), 2) for v in viol]}  "
              f"lambda {meta.lambdas.cpu().numpy().round(3)}")
    return policy


if __name__ == "__main__":
    train(parse_args())
