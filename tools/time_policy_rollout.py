"""Time the on-policy episode in one launch (``policy_rollout`` of BatchedCollisionAvoidance, BatchedCoverageContinuous,
BatchedCoverageDiscrete, BatchedCongestionOnPolicy or BatchedCoverageDiscretizedOnPolicy) against the closed loop it replaces: T x (fused policy act + env.step) + the returns
kernel, replayed from one CUDA graph (for CollisionAvoidance exactly as bench.py's config2_collision_gaussian_graphed
builds it, for CoverageDiscrete as its config1_graphed.fused).

    python tools/time_policy_rollout.py [--env collision|coverage_continuous|coverage_discrete|congestion|
                                               coverage_discretized] [--iters 20] [--rounds 5] [--out FILE]

Shapes: 65 536 envs at 3 agents (BASELINE configs[1] for collision) and 2^20 envs at 3 and 8 agents, size 5, T = 50,
lambda = 0.1, reward-to-go G.  collision: one landmark, thresholds [2].  coverage_continuous: lambda and threshold 25
per agent, weights [1, 2, 3] at 3 agents.  coverage_discrete: BASELINE configs[0] (50 envs x 3 agents) and the same
setup at 65 536 x 3, 2^20 x 3 and 2^20 x 8; there --iters rises per shape until every timed window lasts at least
--min-window-ms (150 ms).  congestion: the paper's setup (size 3, the reference's demand table, noise 0.1, lambda 0.1,
threshold 1.5, gamma 0.9, T = 10, reward-to-go G) at 50 x 3, 65 536 x 3 and 2^20 x 3, and bench.py's
c3_congestion_1M_T100 shape (size 10, 2^20 x 8, T = 100, its seeded demand table); the windows rise as for
coverage_discrete.  coverage_discretized: the paper's runs (size 5, coarseness 6, lambda 0.1, threshold 25 per agent,
weights [1, 2, 3] at 3 agents, T = 50, reward-to-go G) at 50 x 3, 65 536 x 3, 2^20 x 3 and 2^20 x 8, the closed loop
graphed with the PyTorch BatchedDiscretePolicy and with FusedDiscretizedPolicy; the windows rise as for
coverage_discrete.  A --shapes entry is E x A, or E x A x T x size for congestion.
The arms alternate within one process, each timed with CUDA events over --iters calls per round; the products of the
paths are compared on the timed inputs.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def event_ms(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip()}


def shape(E, A, T, iters, rounds):
    import safe_multiagent_rl_b200 as s
    from safe_multiagent_rl_b200.policy import FusedGaussianPolicy
    rng = np.random.default_rng(2)
    starts, lms = rng.random((E, A, 2)) * 5, rng.random((E, 1, 2)) * 5
    mk = lambda: s.BatchedCollisionAvoidance(5, A, n_envs=E, n_landmarks=1, starts=starts, landmarks=lms)
    lam = torch.full((1,), 0.1, dtype=torch.float64, device="cuda")
    thr = torch.tensor([2.0], dtype=torch.float64, device="cuda")
    gamma = 0.999
    env_c = mk()
    pol_c = FusedGaussianPolicy(env_c, seed=7)                     # as bench.py builds config2_collision_gaussian_graphed
    loop = s.GraphedClosedLoop(env_c, T, lambda obs, t: pol_c.act(t=t), lam, gamma, thresholds=[2.0])
    env_p = mk()
    pol_p = FusedGaussianPolicy(env_p, seed=7)
    pol_p.load_state_dict(pol_c.state_dict())
    kw = dict(lambdas=lam, gamma=gamma, thresholds=thr, g_mode=1)
    out = env_p.policy_rollout(pol_p, T, **kw)
    out_nr = env_p.policy_rollout(pol_p, T, record=False, **kw)
    torch.cuda.synchronize()
    graphs = {}
    for tag, o, rec in (("fused_graphed", out, True), ("fused_graphed_no_record", out_nr, False)):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            env_p.policy_rollout(pol_p, T, out=o, record=rec, **kw)
        graphs[tag] = g
    arms = {"closed_loop_graphed": loop.replay,
            "fused_eager": lambda: env_p.policy_rollout(pol_p, T, out=out, **kw),
            "fused_graphed": graphs["fused_graphed"].replay,
            "fused_graphed_no_record": graphs["fused_graphed_no_record"].replay}
    for fn in arms.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            times[k].append(event_ms(fn, iters))
    # the products on the timed inputs: one more call of each path
    ref = loop.replay()
    graphs["fused_graphed"].replay()
    torch.cuda.synchronize()
    same = {k: bool(torch.equal(out[k], ref[k])) for k in ("R", "modR", "C", "G")}
    same["n_active"] = bool(torch.equal(out["n_active"], env_c.episode_len[:E]))
    same["final_state"] = all(bool(torch.equal(a[:, :E], b[:, :E])) for a, b in
                              ((env_p.pos_x, env_c.pos_x), (env_p.pos_y, env_c.pos_y), (env_p.agent_done, env_c.agent_done)))
    same["last_step_actions"] = bool(torch.equal(out["actions_"][T - 1, :, :E], env_c.action_buffer[:, :E]))
    same["last_step_logp"] = bool(torch.equal(out["logp_"][T - 1, :, :E], pol_c.logp[:, :E]))
    sv, rv = out["stats_vec"], ref["stats"].vec
    res = {"n_envs": E, "n_agents": A, "T": T, "iters": iters, "rounds": rounds,
           "ms_per_batch": {k: {"min": min(v), "median": statistics.median(v), "all": v} for k, v in times.items()},
           "identical": same, "stats_identical": bool(torch.equal(sv, rv)),
           "stats_max_rel_diff": float(((sv - rv).abs() / rv.abs().clamp_min(1e-300)).max())}
    c, f = res["ms_per_batch"]["closed_loop_graphed"]["median"], res["ms_per_batch"]["fused_graphed"]["median"]
    res["speedup_fused_graphed_vs_closed_loop"] = c / f
    del loop, graphs, out, out_nr
    torch.cuda.empty_cache()
    return res


def shape_coverage(E, A, T, iters, rounds):
    import safe_multiagent_rl_b200 as s
    from safe_multiagent_rl_b200.policy import FusedGaussianPolicy
    starts = np.random.default_rng(2).random((E, A, 2)) * 5
    weights = [1.0, 2.0, 3.0] if A == 3 else None
    mk = lambda: s.BatchedCoverageContinuous(5, A, n_envs=E, weights=weights, starts=starts)
    lam = torch.full((A,), 0.1, dtype=torch.float64, device="cuda")
    thr = torch.full((A,), 25.0, dtype=torch.float64, device="cuda")
    gamma = 0.999
    env_c = mk()
    pol_c = FusedGaussianPolicy(env_c, seed=7)
    loop = s.GraphedClosedLoop(env_c, T, lambda obs, t: pol_c.act(t=t), lam, gamma, thresholds=[25.0] * A)
    env_p = mk()
    pol_p = FusedGaussianPolicy(env_p, seed=7)
    pol_p.load_state_dict(pol_c.state_dict())
    kw = dict(lambdas=lam, gamma=gamma, thresholds=thr, g_mode=1)
    out = env_p.policy_rollout(pol_p, T, **kw)
    out_nr = env_p.policy_rollout(pol_p, T, record=False, **kw)
    torch.cuda.synchronize()
    graphs = {}
    for tag, o, rec in (("fused_graphed", out, True), ("fused_graphed_no_record", out_nr, False)):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            env_p.policy_rollout(pol_p, T, out=o, record=rec, **kw)
        graphs[tag] = g
    arms = {"closed_loop_graphed": loop.replay,
            "fused_eager": lambda: env_p.policy_rollout(pol_p, T, out=out, **kw),
            "fused_graphed": graphs["fused_graphed"].replay,
            "fused_graphed_no_record": graphs["fused_graphed_no_record"].replay}
    for fn in arms.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            times[k].append(event_ms(fn, iters))
    # the products on the timed inputs: one more call of each path, then the open-loop rollout of the recorded actions
    ref = loop.replay()
    graphs["fused_graphed"].replay()
    torch.cuda.synchronize()
    same = {"final_state": all(bool(torch.equal(a[:, :E], b[:, :E])) for a, b in
                               ((env_p.pos_x, env_c.pos_x), (env_p.pos_y, env_c.pos_y))),
            "last_step_actions": bool(torch.equal(out["actions_"][T - 1, :, :E], env_c.action_buffer[:, :E])),
            "last_step_logp": bool(torch.equal(out["logp_"][T - 1, :, :E], pol_c.logp[:, :E]))}
    fused = {k: out[k].clone() for k in ("R", "modR", "C", "G", "stats_vec")}
    env_r = mk()
    open_loop = env_r.rollout(out["actions_"], **kw)
    torch.cuda.synchronize()
    same_open = {k: bool(torch.equal(fused[k], open_loop[k])) for k in fused}
    same_open["final_state"] = all(bool(torch.equal(a[:, :E], b[:, :E])) for a, b in
                                   ((env_p.pos_x, env_r.pos_x), (env_p.pos_y, env_r.pos_y)))

    def rel(a, b):
        a, b = a.double(), b.double()
        return float(((a - b).abs() / b.abs().clamp_min(1e-300)).max())
    res = {"env": "coverage_continuous", "n_envs": E, "n_agents": A, "T": T, "iters": iters, "rounds": rounds,
           "ms_per_batch": {k: {"min": min(v), "median": statistics.median(v), "all": v} for k, v in times.items()},
           "identical_to_closed_loop": same, "identical_to_open_loop_rollout": same_open,
           "max_rel_diff_vs_closed_loop": {k: rel(fused[k], ref[k]) for k in ("R", "modR", "C")} |
                                          {"stats": rel(fused["stats_vec"], ref["stats"].vec)}}
    c, f = res["ms_per_batch"]["closed_loop_graphed"]["median"], res["ms_per_batch"]["fused_graphed"]["median"]
    res["speedup_fused_graphed_vs_closed_loop"] = c / f
    del loop, graphs, out, out_nr
    torch.cuda.empty_cache()
    return res


def shape_coverage_discrete(E, A, T, iters, rounds, min_window_ms):
    """BASELINE configs[0] at every batch size: size 5, weights [1, 2, 3] at 3 agents, lambda 0.1, thresholds 25,
    gamma 0.999, reward-to-go G.  Closed loops with FusedDiscretePolicy in its default (tensor-core) build, as bench.py
    builds config1_graphed.fused, and in its FP32-pipe build, whose samples the one launch reproduces bit for bit."""
    import safe_multiagent_rl_b200 as s
    from safe_multiagent_rl_b200 import _lib
    from safe_multiagent_rl_b200.policy import FusedDiscretePolicy
    starts = np.random.default_rng(1).integers(0, 5, (E, A, 2))
    weights = [1.0, 2.0, 3.0] if A == 3 else None
    mk = lambda: s.BatchedCoverageDiscrete(5, A, n_envs=E, weights=weights, starts=starts)
    lam = torch.full((A,), 0.1, dtype=torch.float64, device="cuda")
    thr = torch.full((A,), 25.0, dtype=torch.float64, device="cuda")
    gamma = 0.999
    env_tc = mk()
    pol_tc = FusedDiscretePolicy(env_tc, seed=7)
    loop_tc = s.GraphedClosedLoop(env_tc, T, lambda obs, t: pol_tc.act(t=t), lam, gamma, thresholds=[25.0] * A)
    env_c = mk()
    pol_c = FusedDiscretePolicy(env_c, seed=7)
    pol_c.load_state_dict(pol_tc.state_dict())
    with _lib.kernel_variant(_lib.KERNEL_POLICY, 0):       # the kernel is chosen when the graph is captured
        loop_c = s.GraphedClosedLoop(env_c, T, lambda obs, t: pol_c.act(t=t), lam, gamma, thresholds=[25.0] * A)
    env_p = mk()
    pol_p = FusedDiscretePolicy(env_p, seed=7)
    pol_p.load_state_dict(pol_tc.state_dict())
    kw = dict(lambdas=lam, gamma=gamma, thresholds=thr, g_mode=1)
    out = env_p.policy_rollout(pol_p, T, **kw)
    out_nr = env_p.policy_rollout(pol_p, T, record=False, **kw)
    torch.cuda.synchronize()
    graphs = {}
    for tag, o, rec in (("fused_graphed", out, True), ("fused_graphed_no_record", out_nr, False)):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            env_p.policy_rollout(pol_p, T, out=o, record=rec, **kw)
        graphs[tag] = g
    arms = {"closed_loop_graphed": loop_tc.replay,
            "closed_loop_graphed_fp32_policy": loop_c.replay,
            "fused_eager": lambda: env_p.policy_rollout(pol_p, T, out=out, **kw),
            "fused_graphed": graphs["fused_graphed"].replay,
            "fused_graphed_no_record": graphs["fused_graphed_no_record"].replay}
    for fn in arms.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    # enough calls per window that even the fastest arm's window lasts min_window_ms
    iters = max(iters, math.ceil(min_window_ms / min(event_ms(fn, 5) for fn in arms.values())))
    times = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            times[k].append(event_ms(fn, iters))
    # the products on the timed inputs: one more call of each path, then the open-loop rollout of the recorded actions
    ref = loop_c.replay()
    graphs["fused_graphed"].replay()
    torch.cuda.synchronize()
    same = {"final_state": all(bool(torch.equal(a[:, :E], b[:, :E])) for a, b in
                               ((env_p.pos_x, env_c.pos_x), (env_p.pos_y, env_c.pos_y))),
            "last_step_actions": bool(torch.equal(out["actions_"][T - 1, :, :E], env_c.action_buffer[:, :E])),
            "last_step_logp": bool(torch.equal(out["logp_"][T - 1, :, :E], pol_c.logp[:, :E])),
            "C": bool(torch.equal(out["C"].long(), ref["C"].long()))}
    fused = {k: out[k].clone() for k in ("R", "modR", "C", "G", "stats_vec")}
    env_r = mk()
    open_loop = env_r.rollout(out["actions_"], **kw)
    torch.cuda.synchronize()
    same_open = {k: bool(torch.equal(fused[k], open_loop[k])) for k in fused}
    same_open["final_state"] = all(bool(torch.equal(a[:, :E], b[:, :E])) for a, b in
                                   ((env_p.pos_x, env_r.pos_x), (env_p.pos_y, env_r.pos_y)))
    # the default build at t = 0 (same observation): share of equal samples, log-prob gap where they agree
    env_tc.reset()
    _, a0, lp0 = pol_tc.act(t=0)
    agree = a0 == out["actions"][0]
    tc = {"actions_agree": float(agree.float().mean()),
          "max_logp_diff_where_equal": float((lp0 - out["logp"][0]).abs()[agree].max())}

    def rel(a, b):
        a, b = a.double(), b.double()
        return float(((a - b).abs() / b.abs().clamp_min(1e-300)).max())
    res = {"env": "coverage_discrete", "n_envs": E, "n_agents": A, "T": T, "iters": iters, "rounds": rounds,
           "ms_per_batch": {k: {"min": min(v), "median": statistics.median(v), "all": v} for k, v in times.items()},
           "identical_to_fp32_closed_loop": same, "identical_to_open_loop_rollout": same_open,
           "max_rel_diff_vs_fp32_closed_loop": {k: rel(fused[k], ref[k]) for k in ("R", "modR")} |
                                               {"stats": rel(fused["stats_vec"], ref["stats"].vec)},
           "tensor_core_build_t0": tc}
    m = {k: v["median"] for k, v in res["ms_per_batch"].items()}
    res["speedup_fused_graphed_vs_closed_loop"] = m["closed_loop_graphed"] / m["fused_graphed"]
    res["speedup_fused_graphed_vs_fp32_closed_loop"] = m["closed_loop_graphed_fp32_policy"] / m["fused_graphed"]
    del loop_tc, loop_c, graphs, out, out_nr
    torch.cuda.empty_cache()
    return res


def shape_congestion(E, A, T, size, iters, rounds, min_window_ms):
    """The paper's Congestion setup (BASELINE section 2) or bench.py's c3 shape: noise 0.1, lambda 0.1, threshold 1.5,
    gamma 0.9, reward-to-go G.  Size 3 takes the reference's demand table, size 10 bench.py's seeded one.  Closed loops
    with FusedDiscretePolicy in its default (tensor-core) build and in its FP32-pipe build, whose samples the one launch
    reproduces bit for bit.  Every captured reset / policy_rollout advances the noise episode, so the comparison pins it
    in every env before its call."""
    import safe_multiagent_rl_b200 as s
    from safe_multiagent_rl_b200 import _lib
    from safe_multiagent_rl_b200.policy import FusedDiscretePolicy
    demand = None if size == 3 else np.random.default_rng(0).random((size + 1, size + 1)) * 8 + 2
    starts = np.random.default_rng(1).integers(0, size, (E, A, 2))
    starts[:, 0] = 0                                       # agent 0 starts at the origin (congestion.py:215-216)
    mk = lambda cls=s.BatchedCongestion: cls(size, A, n_envs=E, noise=0.1, starts=starts, demand_rate=demand, seed=1)
    lam = torch.full((1,), 0.1, dtype=torch.float64, device="cuda")
    thr = torch.full((1,), 1.5, dtype=torch.float64, device="cuda")
    gamma = 0.9
    env_tc = mk()
    pol_tc = FusedDiscretePolicy(env_tc, seed=7)
    loop_tc = s.GraphedClosedLoop(env_tc, T, lambda obs, t: pol_tc.act(t=t), lam, gamma, thresholds=[1.5])
    env_c = mk()
    pol_c = FusedDiscretePolicy(env_c, seed=7)
    pol_c.load_state_dict(pol_tc.state_dict())
    with _lib.kernel_variant(_lib.KERNEL_POLICY, 0):       # the kernel is chosen when the graph is captured
        loop_c = s.GraphedClosedLoop(env_c, T, lambda obs, t: pol_c.act(t=t), lam, gamma, thresholds=[1.5])
    env_p = mk(s.BatchedCongestionOnPolicy)
    pol_p = FusedDiscretePolicy(env_p, seed=7)
    pol_p.load_state_dict(pol_tc.state_dict())
    kw = dict(lambdas=lam, gamma=gamma, thresholds=thr, g_mode=1)
    out = env_p.policy_rollout(pol_p, T, **kw)
    out_nr = env_p.policy_rollout(pol_p, T, record=False, **kw)
    torch.cuda.synchronize()
    graphs = {}
    for tag, o, rec in (("fused_graphed", out, True), ("fused_graphed_no_record", out_nr, False)):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            env_p.policy_rollout(pol_p, T, out=o, record=rec, **kw)
        graphs[tag] = g
    arms = {"closed_loop_graphed": loop_tc.replay,
            "closed_loop_graphed_fp32_policy": loop_c.replay,
            "fused_eager": lambda: env_p.policy_rollout(pol_p, T, out=out, **kw),
            "fused_graphed": graphs["fused_graphed"].replay,
            "fused_graphed_no_record": graphs["fused_graphed_no_record"].replay}
    for fn in arms.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    # enough calls per window that even the fastest arm's window lasts min_window_ms
    iters = max(iters, math.ceil(min_window_ms / min(event_ms(fn, 5) for fn in arms.values())))
    times = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            times[k].append(event_ms(fn, iters))
    # the products on the timed inputs, all for noise episode 1: both graphs hold the increment of their reset /
    # policy_rollout, so they are pinned to 0; the open-loop rollout below draws the pinned episode itself
    episode = 1
    env_c.set_noise_episode(episode - 1)
    env_p.set_noise_episode(episode - 1)
    ref = loop_c.replay()
    graphs["fused_graphed"].replay()
    torch.cuda.synchronize()
    same = {"final_state": all(bool(torch.equal(a[:, :E], b[:, :E])) for a, b in
                               ((env_p.pos_x, env_c.pos_x), (env_p.pos_y, env_c.pos_y))),
            "last_step_actions": bool(torch.equal(out["actions_"][T - 1, :, :E], env_c.action_buffer[:, :E])),
            "last_step_logp": bool(torch.equal(out["logp_"][T - 1, :, :E], pol_c.logp[:, :E])),
            "C": bool(torch.equal(out["C"].long(), ref["C"].long()))}
    fused = {k: out[k].clone() for k in ("R", "modR", "C", "G", "stats_vec")}
    env_r = mk()
    env_r.set_noise_episode(episode)
    open_loop = env_r.rollout(out["actions_"], **kw)
    torch.cuda.synchronize()
    same_open = {k: bool(torch.equal(fused[k], open_loop[k])) for k in fused}
    same_open["final_state"] = all(bool(torch.equal(a[:, :E], b[:, :E])) for a, b in
                                   ((env_p.pos_x, env_r.pos_x), (env_p.pos_y, env_r.pos_y)))
    # the default build at t = 0 (same observation): share of equal samples, log-prob gap where they agree
    env_tc.reset()
    _, a0, lp0 = pol_tc.act(t=0)
    agree = a0 == out["actions"][0]
    tc = {"actions_agree": float(agree.float().mean()),
          "max_logp_diff_where_equal": float((lp0 - out["logp"][0]).abs()[agree].max())}

    def rel(a, b):
        a, b = a.double(), b.double()
        return float(((a - b).abs() / b.abs().clamp_min(1e-300)).max())
    res = {"env": "congestion", "n_envs": E, "n_agents": A, "T": T, "size": size, "iters": iters, "rounds": rounds,
           "ms_per_batch": {k: {"min": min(v), "median": statistics.median(v), "all": v} for k, v in times.items()},
           "identical_to_fp32_closed_loop": same, "identical_to_open_loop_rollout": same_open,
           "max_rel_diff_vs_fp32_closed_loop": {k: rel(fused[k], ref[k]) for k in ("R", "modR")} |
                                               {"stats": rel(fused["stats_vec"], ref["stats"].vec)},
           "tensor_core_build_t0": tc}
    m = {k: v["median"] for k, v in res["ms_per_batch"].items()}
    res["speedup_fused_graphed_vs_closed_loop"] = m["closed_loop_graphed"] / m["fused_graphed"]
    res["speedup_fused_graphed_vs_fp32_closed_loop"] = m["closed_loop_graphed_fp32_policy"] / m["fused_graphed"]
    del loop_tc, loop_c, graphs, out, out_nr
    torch.cuda.empty_cache()
    return res


def shape_coverage_discretized(E, A, T, iters, rounds, min_window_ms):
    """The paper's CoverageDiscretized runs (size 5, coarseness 6, as tools/sweep.py): weights [1, 2, 3] at 3 agents,
    lambda 0.1, threshold 25 per agent, gamma 0.999, reward-to-go G.  Closed loops with the PyTorch glue
    BatchedDiscretePolicy (sampled by torch; its own stream) and with FusedDiscretizedPolicy, whose samples the one
    launch reproduces bit for bit; the one launch eager, graphed, and graphed without records."""
    import safe_multiagent_rl_b200 as s
    from safe_multiagent_rl_b200.policy import BatchedDiscretePolicy, FusedDiscretizedPolicy
    size, coarseness = 5, 6
    zoom = coarseness / size
    starts = np.floor(np.random.default_rng(1).random((E, A, 2)) * size * zoom) / zoom
    weights = [1.0, 2.0, 3.0] if A == 3 else None
    mk = lambda cls=s.BatchedCoverageDiscretized: cls(size, A, n_envs=E, coarseness=coarseness, weights=weights,
                                                      starts=starts)
    lam = torch.full((A,), 0.1, dtype=torch.float64, device="cuda")
    thr = torch.full((A,), 25.0, dtype=torch.float64, device="cuda")
    gamma = 0.999
    env_g = mk()
    pol_g = BatchedDiscretePolicy(env_g)
    loop_g = s.GraphedClosedLoop(env_g, T, lambda obs, t: pol_g.act(obs), lam, gamma, thresholds=[25.0] * A)
    env_c = mk()
    pol_c = FusedDiscretizedPolicy(env_c, seed=7)
    pol_c.load_state_dict(pol_g.state_dict())
    loop_c = s.GraphedClosedLoop(env_c, T, lambda obs, t: pol_c.act(t=t), lam, gamma, thresholds=[25.0] * A)
    env_p = mk(s.BatchedCoverageDiscretizedOnPolicy)
    pol_p = FusedDiscretizedPolicy(env_p, seed=7)
    pol_p.load_state_dict(pol_g.state_dict())
    kw = dict(lambdas=lam, gamma=gamma, thresholds=thr, g_mode=1)
    out = env_p.policy_rollout(pol_p, T, **kw)
    out_nr = env_p.policy_rollout(pol_p, T, record=False, **kw)
    torch.cuda.synchronize()
    graphs = {}
    for tag, o, rec in (("fused_graphed", out, True), ("fused_graphed_no_record", out_nr, False)):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            env_p.policy_rollout(pol_p, T, out=o, record=rec, **kw)
        graphs[tag] = g
    arms = {"closed_loop_graphed_pytorch_policy": loop_g.replay,
            "closed_loop_graphed": loop_c.replay,
            "fused_eager": lambda: env_p.policy_rollout(pol_p, T, out=out, **kw),
            "fused_graphed": graphs["fused_graphed"].replay,
            "fused_graphed_no_record": graphs["fused_graphed_no_record"].replay}
    for fn in arms.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    # enough calls per window that even the fastest arm's window lasts min_window_ms
    iters = max(iters, math.ceil(min_window_ms / min(event_ms(fn, 5) for fn in arms.values())))
    times = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            times[k].append(event_ms(fn, iters))
    # the products on the timed inputs: one more call of each path, then the open-loop rollout of the recorded actions
    ref = loop_c.replay()
    graphs["fused_graphed"].replay()
    torch.cuda.synchronize()
    same = {"final_state": all(bool(torch.equal(a[:, :E], b[:, :E])) for a, b in
                               ((env_p.pos_x, env_c.pos_x), (env_p.pos_y, env_c.pos_y))),
            "last_step_actions": bool(torch.equal(out["actions_"][T - 1, :, :E], env_c.action_buffer[:, :E])),
            "last_step_logp": bool(torch.equal(out["logp_"][T - 1, :, :E], pol_c.logp[:, :E])),
            "C": bool(torch.equal(out["C"], ref["C"]))}
    fused = {k: out[k].clone() for k in ("R", "modR", "C", "G", "stats_vec")}
    env_r = mk()
    open_loop = env_r.rollout(out["actions_"], **kw)
    torch.cuda.synchronize()
    same_open = {k: bool(torch.equal(fused[k], open_loop[k])) for k in fused}
    same_open["final_state"] = all(bool(torch.equal(a[:, :E], b[:, :E])) for a, b in
                                   ((env_p.pos_x, env_r.pos_x), (env_p.pos_y, env_r.pos_y)))

    def rel(a, b):
        a, b = a.double(), b.double()
        return float(((a - b).abs() / b.abs().clamp_min(1e-300)).max())
    res = {"env": "coverage_discretized", "n_envs": E, "n_agents": A, "T": T, "size": size, "coarseness": coarseness,
           "iters": iters, "rounds": rounds,
           "ms_per_batch": {k: {"min": min(v), "median": statistics.median(v), "all": v} for k, v in times.items()},
           "identical_to_closed_loop": same, "identical_to_open_loop_rollout": same_open,
           "max_rel_diff_vs_closed_loop": {k: rel(fused[k], ref[k]) for k in ("R", "modR")} |
                                          {"stats": rel(fused["stats_vec"], ref["stats"].vec)}}
    m = {k: v["median"] for k, v in res["ms_per_batch"].items()}
    res["speedup_fused_graphed_vs_pytorch_closed_loop"] = m["closed_loop_graphed_pytorch_policy"] / m["fused_graphed"]
    res["speedup_fused_graphed_vs_closed_loop"] = m["closed_loop_graphed"] / m["fused_graphed"]
    del loop_g, loop_c, graphs, out, out_nr
    torch.cuda.empty_cache()
    return res


SHAPES = {"collision": "65536x3,1048576x3,1048576x8", "coverage_continuous": "65536x3,1048576x3,1048576x8",
          "coverage_discrete": "50x3,65536x3,1048576x3,1048576x8",
          "coverage_discretized": "50x3,65536x3,1048576x3,1048576x8",
          "congestion": "50x3x10x3,65536x3x10x3,1048576x3x10x3,1048576x8x100x10"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--env", choices=tuple(SHAPES), default="collision")
    ap.add_argument("--iters", type=int, default=20,
                    help="calls per timed window (coverage_discrete, coverage_discretized, congestion: at least)")
    ap.add_argument("--min-window-ms", type=float, default=150.0,
                    help="coverage_discrete, coverage_discretized, congestion: raise the calls per window until the "
                         "fastest arm's window lasts this long")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--shapes", default=None, help="ExA list (default: per env)")
    ap.add_argument("--out", default=None, help="also write the JSON lines here")
    a = ap.parse_args()
    lines = [json.dumps({"gpu": gpu_info(), "lib": os.path.basename(os.environ.get("SMARL_LIB", "libsmarl.so"))})]
    print(lines[-1], flush=True)
    run = {"collision": shape, "coverage_continuous": shape_coverage, "coverage_discrete": shape_coverage_discrete,
           "coverage_discretized": shape_coverage_discretized, "congestion": shape_congestion}[a.env]
    for sh in (a.shapes or SHAPES[a.env]).split(","):
        dims = [int(x) for x in sh.split("x")]
        if a.env == "congestion":
            E, A, T, size = dims
            lines.append(json.dumps(run(E, A, T, size, a.iters, a.rounds, a.min_window_ms)))
        else:
            E, A = dims
            extra = (a.min_window_ms,) if a.env in ("coverage_discrete", "coverage_discretized") else ()
            lines.append(json.dumps(run(E, A, 50, a.iters, a.rounds, *extra)))
        print(lines[-1], flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
