#!/usr/bin/env python
"""Headline benchmark: agent-steps/sec (env step + cost + returns) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR writes what the last timed step of `value` returned (a fixed sample of envs, see
dump_closed_loop) as DIR/<name>.npy, so that two builds can be compared output for output.

One "step" = one batch of episodes of the named workload (default: BASELINE.json configs[3],
CoverageDiscrete 32x32 / 16 agents / T=50 with 2^22 envs PER GPU, weak scaling):

  value   closed-loop mode, inputs resident in HBM: reset + T x smarl_coverage_step (each writes
          obs / reward / cost / done / penalty, the true drop-in for env.step with a policy in the
          loop) + smarl_rollout_returns (R, modR, C, reward-to-go G, stats) + stats all-reduce over
          ranks + smarl_lambda_update.  Timed with CUDA events, max over ranks.
  e2e     the same workload through the host-buffer C-ABI call smarl_host_coverage_rollout:
          pinned HOST actions/starts in, HOST R/modR/C/stats out, copies inside the timed region.
  roofline  dominant kernel (coverage_step_kernel): algorithmic bytes per launch (19 B per
          agent-step x A x E) / its CUDA-event launch duration, against MEASURED_PEAKS.json.
  fused   extra: the open-loop fused rollout kernel (state in registers for all T steps).
  cpu_baseline  oracle/scalar_port.py (reference-structure Python loop) on all host cores.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "agent-steps/sec (env step+cost+returns)"
UNIT = "agent-steps/s"

# The contract is ONE JSON line on stdout.  Libraries (NCCL's version banner, torchrun notices) also
# write to fd 1, so keep a private handle on the real stdout for the result line and point fd 1 at
# stderr for everything else.
_RESULT_OUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(obj):
    _RESULT_OUT.write(json.dumps(obj) + "\n")
    _RESULT_OUT.flush()


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps (batches) of the headline closed loop and of its policy-path, lean, fused, "
                         "strong-scaled and host-buffer variants; the extra named configs and the policy loops "
                         "size their own repeat counts")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n_envs", type=int, default=1 << 22, help="envs per GPU")
    ap.add_argument("--size", type=int, default=32)
    ap.add_argument("--n_agents", type=int, default=16)
    ap.add_argument("--max_t", type=int, default=50)
    ap.add_argument("--gamma", type=float, default=0.999)
    ap.add_argument("--cpu_seconds", type=float, default=12.0, help="CPU-baseline sample length")
    ap.add_argument("--no_cpu_baseline", action="store_true")
    ap.add_argument("--no_e2e", action="store_true")
    ap.add_argument("--no_fused", action="store_true")
    ap.add_argument("--no_configs", action="store_true", help="skip the extra named configs (c2, c3, c4_strong)")
    ap.add_argument("--no_policy", action="store_true", help="skip the policy-in-the-loop timing")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (rank 0's envs)")
    a = ap.parse_args()
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs needs --impl ours: the reference arm times CPU episodes and returns no arrays")
    return a


def workload_name(a):
    return (f"CoverageDiscrete size={a.size} n_agents={a.n_agents} max_t={a.max_t} "
            f"n_envs={a.n_envs}/GPU weights=1+(a%3) thresholds=25 gamma={a.gamma} (BASELINE configs[3] shape)")


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's execution model (one env per process, Python loop) on all host cores
# ------------------------------------------------------------------------------------------------
def cpu_impl():
    """(module, kind): the unmodified reference classes when their copy travelled with the repo (oracle/_ref, made
    by __graft_entry__.build() from /root/reference) or the tree is mounted, else the pinned port."""
    from oracle import ref_timing as rt
    if rt.root() is not None:
        try:
            rt.load()
            return rt, "reference"
        except Exception as ex:                     # e.g. a dependency of the reference missing on this box
            sys.stderr.write(f"reference arm: falling back to the port ({ex})\n")
    from oracle import scalar_port as sp
    return sp, "port"


def cpu_rate(a, seconds):
    mod, _ = cpu_impl()
    procs = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    rate, used = mod.time_all_cores("coverage", a.size, a.n_agents, a.max_t, a.gamma, seconds, procs)
    return rate, used


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    for _ in range(a.warmup):
        cpu_rate(a, 1.0)
    per_step = max(1.0, min(a.cpu_seconds, 120.0 / max(1, a.steps)))
    rates, cores = [], 1
    t0 = time.perf_counter()
    for _ in range(a.steps):
        r, cores = cpu_rate(a, per_step)
        rates.append(r)
    wall = time.perf_counter() - t0
    v = statistics.mean(rates)
    kind = cpu_impl()[1]
    what = ("the unmodified reference classes (oracle/_ref copy of envs/ + safe_multi_agent_RL/)" if kind == "reference"
            else "oracle/scalar_port.py (reference-structured port; the reference copy is absent)")
    sample = (f"{a.steps} x {per_step:.1f}s of whole episodes (env.step + MetaAgent.act + Buffer.append/step + "
              f"reward-to-go) of {what} on {cores} processes, one env each, recorded random actions")
    emit({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1e3 * wall / a.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(a), "note": "CPU arm ignores n_envs: it steps one env per core"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })


# ------------------------------------------------------------------------------------------------
# clocks sampled DURING the timed region
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "25", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, p in zip(names, parts[2:6]):
                if p.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return None
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except (KeyError, ValueError):
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel, a):
    """Per-launch DRAM bytes of `kernel` from the committed ncu --set full summary, if it was
    captured on this workload shape."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(path):
        return None
    try:
        d = json.load(open(path)).get(kernel)
        if d and d["n_envs"] == a.n_envs and d["n_agents"] == a.n_agents and d["size"] == a.size:
            return d["dram_bytes_per_launch"]
    except (ValueError, KeyError):
        pass
    return None


# ------------------------------------------------------------------------------------------------
# extras of the result line: the other named configs, the strong-scaled config, the policy loop
# ------------------------------------------------------------------------------------------------
def _event_ms(fn, iters, warmup=3):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def bench_named_config(s, _lib, env_name, S, A, E, T, gamma, peak, graph):
    """Closed loop (reset + T step launches + returns kernel) of one named config on this GPU; `graph` replays the
    whole batch from one CUDA graph (small batches are launch-bound otherwise).  The roofline block is the step
    kernel's: algorithmic bytes per launch (DESIGN.md section 3) / its average duration inside the batch."""
    import numpy as np
    import torch
    g = torch.Generator(device="cuda"); g.manual_seed(7)
    rng = np.random.default_rng(0)
    if env_name == "collision":
        env = s.BatchedCollisionAvoidance(S, A, n_envs=E, starts=np.zeros((E, A, 2)), landmarks=np.zeros((E, 1, 2)))
        env.start_x[:, :E] = torch.rand((A, E), generator=g, device="cuda", dtype=torch.float64) * S
        env.start_y[:, :E] = torch.rand((A, E), generator=g, device="cuda", dtype=torch.float64) * S
        env.landmarks[:, :E] = torch.rand((2, E), generator=g, device="cuda", dtype=torch.float64) * S
        actions = torch.randn((T, 2 * A, env.ld), generator=g, device="cuda") * 0.5
        K, kernel = 1, "collision_step_kernel"
        bytes_step = 55.0 + 24.0 / A           # pos r/w 32, action 8, done r/w/out 3, obs 8, reward 4 + (landmarks 16, cost 4, penalty 4)/A
    else:
        env = s.BatchedCongestion(S, A, n_envs=E, noise=0.1, starts=np.zeros((E, A, 2), np.uint8),
                                  demand_rate=rng.random((S + 1, S + 1)) * 8 + 2, seed=1)
        env.start_x[1:, :E] = torch.randint(0, S, (A - 1, E), generator=g, device="cuda", dtype=torch.uint8)
        env.start_y[1:, :E] = torch.randint(0, S, (A - 1, E), generator=g, device="cuda", dtype=torch.uint8)
        actions = torch.randint(0, 5, (T, A, env.ld), generator=g, device="cuda", dtype=torch.uint8)
        K, kernel = 1, "congestion_step_kernel"
        bytes_step = 18.0 + 8.0 / A            # pos r/w 4, action 1, effective move 1, obs 8, reward 4 + (cost 4, penalty 4)/A
    lam = torch.full((K,), 0.1, dtype=torch.float64, device="cuda")
    buf = env.new_rollout_buffer(T)
    thr = [1.5] * K

    def steps_only():
        env.reset()
        for t in range(T):
            env.step(actions[t], lambdas=lam, out=(buf, t), agent_major=True)

    def closed():
        steps_only()
        buf.finish(gamma, thr, n_active=getattr(env, "episode_len", None))
    closed()
    torch.cuda.synchronize()
    iters = max(5, min(200, int(4e9 / (float(E) * A * T))))
    if graph:
        g_all, g_steps = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        with torch.cuda.graph(g_all):
            closed()
        with torch.cuda.graph(g_steps):
            steps_only()
        ms = _event_ms(g_all.replay, iters)
        ms_steps = _event_ms(g_steps.replay, iters)
    else:
        ms = _event_ms(closed, iters)
        ms_steps = _event_ms(steps_only, iters)
    n = float(E) * A * T
    launch_ms = ms_steps / T
    achieved = bytes_step * A * E / (launch_ms * 1e-3) / 1e9
    return {"value": n / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "n_envs": E, "n_agents": A, "size": S, "max_t": T,
            "mode": "closed loop: reset + T step launches + returns kernel" + (", one CUDA graph" if graph else ""),
            "roofline": {"bound": "hbm", "kernel": kernel, "bytes_per_launch": bytes_step * A * E, "launch_ms": launch_ms,
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "note": "launch_ms = (reset + T steps) / T" + (", incl. graph-node launch gaps" if graph else "")}}


def bench_strong(s, _lib, lib, sd, comm, a, rank, world, dev, peak, timed):
    """BASELINE.json configs[3] literally: n_envs TOTAL (default 2^22) sharded over the ranks by contiguous global env
    ids, stats all-reduce (C ABI) + lambda update inside the timed region.  At world = 1 this is the headline workload."""
    import numpy as np
    import torch
    A, T, S = a.n_agents, a.max_t, a.size
    total = a.n_envs
    off, E = sd.shard_range(total, rank, world)
    g = torch.Generator(device=dev); g.manual_seed(4321 + rank)
    env = s.BatchedCoverageDiscrete(S, A, n_envs=E, weights=[1.0 + (i % 3) for i in range(A)], device=dev, env_offset=off,
                                    starts=np.zeros((E, A, 2), dtype=np.uint8))
    ld = env.ld
    env.start_x[:, :E] = torch.randint(0, S, (A, E), generator=g, device=dev, dtype=torch.uint8)
    env.start_y[:, :E] = torch.randint(0, S, (A, E), generator=g, device=dev, dtype=torch.uint8)
    actions = torch.randint(0, 5, (T, A, ld), generator=g, device=dev, dtype=torch.uint8)
    thr = torch.full((A,), 25.0, dtype=torch.float64, device=dev)
    lam = torch.full((A,), 0.1, dtype=torch.float64, device=dev)
    buf = env.new_rollout_buffer(T, g_mode=s.G_REWARD_TO_GO)
    from safe_multiagent_rl_b200.rollout import make_accounting
    acc = make_accounting(a.gamma, T, s.G_REWARD_TO_GO, thr)
    P, stream, params = _lib.ptr, torch.cuda.current_stream().cuda_stream, env._params
    # per-step argument lists built once: at 2^19 envs per rank a step kernel runs ~27 us, about what slicing four tensors
    # and reading ten data pointers costs in Python per step -- the launch queue must not run dry
    pr, px, py, po, pl = C.byref(params), P(env.pos_x), P(env.pos_y), P(env.obs), P(lam)
    step_args = [(pr, px, py, P(actions[t]), po, P(buf.reward[t]), P(buf.cost[t]), None, pl, P(buf.penalty[t]), E, ld, stream)
                 for t in range(T)]
    step = lib.smarl_coverage_step

    def loop():
        _lib.check(lib.smarl_grid_reset(P(env.start_x), P(env.start_y), px, py, po, A, E, ld, stream))
        for args in step_args:
            if step(*args):
                _lib.check(-1)
        _lib.check(lib.smarl_rollout_returns(C.byref(acc), P(buf.reward), P(buf.cost), buf.cost_code, P(buf.penalty), None,
                                             P(buf.R), P(buf.modR), P(buf.Csum), P(buf.G), P(buf.stats_vec),
                                             P(buf.stats_scratch), A, A, E, ld, stream))
        comm.allreduce(buf.stats_vec)
        _lib.check(lib.smarl_lambda_update(P(lam), P(buf.stats_vec), P(thr), 0.002, A, A, stream))
    ms, _ = timed(loop, a.steps, a.warmup)
    ms /= a.steps
    count = float(buf.stats_vec[-1].item())
    return {"value": float(total) * A * T / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "scaling": "strong",
            "n_envs_total": total, "n_envs_per_rank": E, "world": world, "episodes_reduced": count,
            "count_ok": bool(count == float(total)),
            "mode": "configs[3] as written: the env batch sharded over the ranks, stats all-reduce + lambda update timed"}


def bench_policy_loop(s, a, dev):
    """main.py:28-57 WITH the reference's policy networks (agent.py:23-47: per-agent 2A -> 16 -> 5 MLP + Categorical
    sampling, here the stacked PyTorch glue of policy.py) between the steps: ms per batch split into policy and env."""
    import numpy as np
    import torch
    A, T, S = a.n_agents, a.max_t, a.size
    E = min(a.n_envs, 1 << 18)                 # the stacked forward materialises [A, E, 16] / [A, E, 5] f32 per step
    env = s.BatchedCoverageDiscrete(S, A, n_envs=E, weights=[1.0 + (i % 3) for i in range(A)], device=dev,
                                    starts=np.random.default_rng(0).integers(0, S, (E, A, 2)))
    from safe_multiagent_rl_b200.policy import BatchedDiscretePolicy
    pol = BatchedDiscretePolicy(env)
    lam = torch.full((A,), 0.1, dtype=torch.float64, device=dev)
    buf = env.new_rollout_buffer(T)
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(T)]

    def batch(record):
        obs = env.reset()
        for t in range(T):
            if record:
                ev[t][0].record()
            pol.act(obs)
            if record:
                ev[t][1].record()
            obs, _, _, _ = env.step(env.action_buffer, lambdas=lam, out=(buf, t), agent_major=True)
            if record:
                ev[t][2].record()
        buf.finish(a.gamma, [25.0] * A)
    for _ in range(2):
        batch(False)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    batch(True)
    e1.record()
    torch.cuda.synchronize()
    total = e0.elapsed_time(e1)
    pol_ms = sum(x[0].elapsed_time(x[1]) for x in ev)
    env_ms = sum(x[1].elapsed_time(x[2]) for x in ev)
    n = float(E) * A * T
    out = {"n_envs": E, "ms_per_batch": total, "policy_ms": pol_ms, "env_step_ms": env_ms,
           "value_with_policy": n / (total * 1e-3), "value_env_only": n / ((total - pol_ms) * 1e-3), "unit": UNIT,
           "policy_share": pol_ms / total,
           "policy": "BatchedDiscretePolicy (PyTorch: stacked per-agent 2A->16->5 MLPs, Categorical sampling into env.action_buffer)"}
    # the same loop with the fused policy kernel (smarl_policy_act_discrete) reading the u8 position rows: no float
    # observation rows, no [A, E, 16] / [A, E, 5] intermediates
    from safe_multiagent_rl_b200.policy import FusedDiscretePolicy
    del pol, buf, env
    torch.cuda.empty_cache()
    from safe_multiagent_rl_b200 import _lib as L_
    # policy_fused / policy_fused_full: the default build (fc1 on the tensor cores, tcgen05 + TMEM);
    # policy_fused_fp32_pipes: the FP32-pipe build of the same kernel, for comparison
    for tag, Ef, variant in (("policy_fused", E, -1), ("policy_fused_full", a.n_envs, -1), ("policy_fused_fp32_pipes", E, 0)):
        envf = s.BatchedCoverageDiscrete(S, A, n_envs=Ef, weights=[1.0 + (i % 3) for i in range(A)], device=dev,
                                         starts=np.zeros((Ef, A, 2), dtype=np.uint8))
        g = torch.Generator(device=dev); g.manual_seed(99)
        envf.start_x[:, :Ef] = torch.randint(0, S, (A, Ef), generator=g, device=dev, dtype=torch.uint8)
        envf.start_y[:, :Ef] = torch.randint(0, S, (A, Ef), generator=g, device=dev, dtype=torch.uint8)
        envf.emit_obs = False
        polf = FusedDiscretePolicy(envf, seed=5)
        buff = envf.new_rollout_buffer(T)

        def batchf(record):
            envf.reset()
            for t in range(T):
                if record:
                    ev[t][0].record()
                polf.act(t=t)
                if record:
                    ev[t][1].record()
                envf.step(envf.action_buffer, lambdas=lam, out=(buff, t), agent_major=True)
                if record:
                    ev[t][2].record()
            buff.finish(a.gamma, [25.0] * A)
        with L_.kernel_variant(L_.KERNEL_POLICY, variant):
            for _ in range(2):
                batchf(False)
            torch.cuda.synchronize()
            e0.record()
            batchf(True)
            e1.record()
            torch.cuda.synchronize()
        tot = e0.elapsed_time(e1)
        pm = sum(x[0].elapsed_time(x[1]) for x in ev)
        em = sum(x[1].elapsed_time(x[2]) for x in ev)
        nf = float(Ef) * A * T
        macs = 2.0 * A * 16 + 16 * 5                        # multiply-adds per agent-step of the 2A -> 16 -> 5 MLP
        out[tag] = {"n_envs": Ef, "ms_per_batch": tot, "policy_ms": pm, "env_step_ms": em,
                    "value_with_policy": nf / (tot * 1e-3), "unit": UNIT, "policy_share": pm / tot,
                    "policy_tflops_fp32_equivalent": 2.0 * macs * nf / (pm * 1e-3) / 1e12,
                    "slowdown_vs_env_only": tot / (tot - pm),
                    "policy": "FusedDiscretePolicy (smarl_policy_act_discrete: u8 positions in, u8 actions + f32 log-probs out, "
                              "Philox inverse-CDF sampling; " +
                              ("all multiply-adds on the FP32 pipes (packed FFMA2)" if variant == 0 else
                               "fc1 as tcgen05.mma GEMMs per 256-env tile -- exact bf16 positions x three bf16 pieces per "
                               "fp32 weight, f32 accumulators in tensor memory -- relu / fc2 / softmax / sampling out of TMEM") +
                              "); env steps run with obs = NULL"}
        del envf, polf, buff
        torch.cuda.empty_cache()
    # BASELINE configs[0] (50 envs) with the policy in the loop, replayed from one CUDA graph
    env1 = s.BatchedCoverageDiscrete(5, 3, n_envs=50, weights=[1.0, 2.0, 3.0], device=dev,
                                     starts=np.random.default_rng(1).integers(0, 5, (50, 3, 2)))
    pol1 = BatchedDiscretePolicy(env1)
    lam1 = torch.full((3,), 0.1, dtype=torch.float64, device=dev)
    loop = s.GraphedClosedLoop(env1, 50, lambda obs, t: pol1.act(obs), lam1, 0.999, thresholds=[25.0] * 3)
    ms1 = _event_ms(loop.replay, 50)
    out["config1_graphed"] = {"n_envs": 50, "n_agents": 3, "max_t": 50, "ms_per_batch": ms1,
                              "value_with_policy": 50 * 3 * 50 / (ms1 * 1e-3), "unit": UNIT,
                              "policy": "BatchedDiscretePolicy (PyTorch glue)"}
    del loop
    polf1 = FusedDiscretePolicy(env1, seed=3)
    loopf = s.GraphedClosedLoop(env1, 50, lambda obs, t: polf1.act(t=t), lam1, 0.999, thresholds=[25.0] * 3)
    msf = _event_ms(loopf.replay, 50)
    out["config1_graphed"]["fused"] = {"ms_per_batch": msf, "value_with_policy": 50 * 3 * 50 / (msf * 1e-3),
                                       "policy": "FusedDiscretePolicy (smarl_policy_act_discrete)"}
    del loopf
    # BASELINE configs[1] (CollisionAvoidance 5x5, 3 agents, 65 536 envs, T = 50: the reference's default environment) with
    # the reference's ContinuousPolicy (agent.py:48-76) in the loop, one CUDA graph per batch: the fused Gaussian policy
    # kernel (smarl_policy_act_gaussian) against the PyTorch glue
    from safe_multiagent_rl_b200.policy import BatchedGaussianPolicy, FusedGaussianPolicy
    E2 = 65536
    rng2 = np.random.default_rng(2)
    env2 = s.BatchedCollisionAvoidance(5, 3, n_envs=E2, n_landmarks=1, device=dev, starts=rng2.random((E2, 3, 2)) * 5,
                                       landmarks=rng2.random((E2, 1, 2)) * 5)
    lam2 = torch.full((1,), 0.1, dtype=torch.float64, device=dev)
    polg, polt = FusedGaussianPolicy(env2, seed=7), BatchedGaussianPolicy(env2)
    c2 = {"n_envs": E2, "n_agents": 3, "max_t": 50, "unit": UNIT}
    for tag, fn in (("fused", lambda obs, t: polg.act(t=t)), ("pytorch_glue", lambda obs, t: polt.act(obs))):
        lp = s.GraphedClosedLoop(env2, 50, fn, lam2, 0.999, thresholds=[2.0])
        ms2 = _event_ms(lp.replay, 20)
        c2[tag] = {"ms_per_batch": ms2, "value_with_policy": E2 * 3 * 50 / (ms2 * 1e-3)}
        del lp
    out["config2_collision_gaussian_graphed"] = c2
    return out


DUMP_BYTES = 48 << 20


def dump_closed_loop(out_dir, env, buf, lambdas, n_envs):
    """--dump-outputs: what the last timed closed-loop step handed its caller.  Per-env arrays keep a fixed, seeded,
    sorted sample of env columns sized to stay under DUMP_BYTES (the full per-step slabs of 2^22 envs are GBs):
    per-step rewards / costs / penalties and reward-to-go G [T, rows, n], the final observations and positions,
    episode returns R / modR and cost sums C [rows, n].  The reduced stats vector and the updated lambdas are whole.
    Integer outputs are written as float32 (exact), f64 outputs as float64."""
    import numpy as np
    import torch
    per_env = {"reward": buf.reward, "cost": buf.cost, "penalty": buf.penalty, "G": buf.G, "obs": env.obs,
               "pos_x": env.pos_x, "pos_y": env.pos_y, "R": buf.R, "modR": buf.modR, "C": buf.Csum}
    col_bytes = sum(4 * t[..., 0].numel() for t in per_env.values())
    n = min(n_envs, DUMP_BYTES // col_bytes)
    cols = torch.as_tensor(np.sort(np.random.default_rng(0).choice(n_envs, n, replace=False)), device=buf.R.device)
    os.makedirs(out_dir, exist_ok=True)
    whole = {"stats": buf.stats_vec, "lambdas": lambdas}
    for name, t in [*((k, v.index_select(-1, cols)) for k, v in per_env.items()), *whole.items()]:
        t = t.double() if t.dtype == torch.float64 else t.float()
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


# ------------------------------------------------------------------------------------------------
def run_ours(a):
    import numpy as np
    import torch
    import torch.distributed as dist
    import safe_multiagent_rl_b200 as s
    from safe_multiagent_rl_b200 import _lib
    from safe_multiagent_rl_b200 import dist as sd
    from safe_multiagent_rl_b200.rollout import make_accounting

    rank, world, local_rank = sd.init_from_env()
    if world > 1:
        sd.bind_to_gpu_numa(local_rank)
    if world != a.gpus and world > 1:
        a.gpus = world
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    lib = _lib.load()
    A, E, T, S = a.n_agents, a.n_envs, a.max_t, a.size
    K = A

    # ---- synthetic workload (seeded; per-rank shard of the global env range) ----------------------
    g = torch.Generator(device=dev)
    g.manual_seed(1234 + rank)
    weights = [1.0 + (i % 3) for i in range(A)]
    env = s.BatchedCoverageDiscrete(S, A, n_envs=E, weights=weights, device=dev, env_offset=rank * E,
                                    starts=np.zeros((E, A, 2), dtype=np.uint8))
    ld = env.ld
    env.start_x[:, :E] = torch.randint(0, S, (A, E), generator=g, device=dev, dtype=torch.uint8)
    env.start_y[:, :E] = torch.randint(0, S, (A, E), generator=g, device=dev, dtype=torch.uint8)
    actions = torch.randint(0, 5, (T, A, ld), generator=g, device=dev, dtype=torch.uint8)
    thr = torch.full((K,), 25.0, dtype=torch.float64, device=dev)
    meta = s.BatchedMetaAgent([1] * K, a.gamma, 0.002, [25.0] * K, start_learning_cycle=0, lambda_0=0.1,
                              n_agents=A, device=dev)
    buf = env.new_rollout_buffer(T, g_mode=s.G_REWARD_TO_GO)     # Coverage agents never finish: no per-step done slab
    assert buf.done is None
    acc = make_accounting(a.gamma, T, s.G_REWARD_TO_GO, thr)
    params = env._params
    stream = torch.cuda.current_stream().cuda_stream
    P = _lib.ptr
    launches_per_step = 1 + T + 2 + 1 + 1     # reset, T steps, returns + stats finalize, all-reduce, lambda update
    comm = sd.StatsComm.from_process_group()  # libsmarl's own NCCL binding (smarl_comm_* / smarl_stats_allreduce)
    local_stats = torch.zeros_like(buf.stats_vec)

    def closed_loop(ev_a=None, ev_b=None, obs=env.obs):
        _lib.check(lib.smarl_grid_reset(P(env.start_x), P(env.start_y), P(env.pos_x), P(env.pos_y), P(obs),
                                        A, E, ld, stream))
        if ev_a is not None:
            ev_a.record()
        for t in range(T):
            _lib.check(lib.smarl_coverage_step(C.byref(params), P(env.pos_x), P(env.pos_y), P(actions[t]),
                                               P(obs), P(buf.reward[t]), P(buf.cost[t]), None,
                                               P(meta.lambdas), P(buf.penalty[t]), E, ld, stream))
        if ev_b is not None:
            ev_b.record()
        _lib.check(lib.smarl_rollout_returns(C.byref(acc), P(buf.reward), P(buf.cost), buf.cost_code,
                                             P(buf.penalty), None, P(buf.R), P(buf.modR), P(buf.Csum), P(buf.G),
                                             P(buf.stats_vec), P(buf.stats_scratch), A, K, E, ld, stream))
        local_stats.copy_(buf.stats_vec)                        # this rank's shard (kept for the post-run check)
        comm.allreduce(buf.stats_vec)                           # the only inter-GPU traffic, through the C ABI
        _lib.check(lib.smarl_lambda_update(P(meta.lambdas), P(buf.stats_vec), P(thr), 0.002, A, K, stream))

    def timed(fn, steps, warmup, per_step_events=False):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            if per_step_events:
                fn(*evs[i])
            else:
                fn()
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = e0.elapsed_time(e1)
        inner = sum(x.elapsed_time(y) for x, y in evs) if per_step_events else None
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), inner

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    total_ms, step_kernel_ms = timed(closed_loop, a.steps, a.warmup, per_step_events=True)
    clocks = sampler.stop() if sampler else None
    if a.dump_outputs and rank == 0:
        dump_closed_loop(a.dump_outputs, env, buf, meta.lambdas, E)

    agent_steps = float(E) * A * T
    ms_per_step = total_ms / a.steps
    value = world * agent_steps / (ms_per_step * 1e-3)

    # ---- roofline of the dominant kernel ----------------------------------------------------------
    peak, peak_src = measured_peak()
    launch_ms = step_kernel_ms / (a.steps * T)
    # pos read + write 4, action 1, obs 8, reward 4, cost 1 (done is constant False for Coverage, coverage.py:97-98,
    # and no longer stored per step; the 4/A penalty bytes are left out of the numerator)
    bytes_per_launch = 18.0 * A * E
    achieved = bytes_per_launch / (launch_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "coverage_step_kernel", "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak, "traffic": ncu_traffic("coverage_step_kernel", a),
                "bytes_per_launch": bytes_per_launch, "launch_ms": launch_ms, "peak_source": peak_src,
                "share_of_step": step_kernel_ms / total_ms}

    # ---- N-rank check of the reduced vector (not timed): count, integer cost sums, identical lambda --------
    n_stats = buf.stats_vec.numel()
    glob = buf.stats_vec.clone()
    via_torch = local_stats.clone()
    lam_all = [meta.lambdas.clone() for _ in range(world)]
    if world > 1:
        dist.all_reduce(via_torch, op=dist.ReduceOp.SUM)        # the same sum through torch.distributed
        dist.all_gather(lam_all, meta.lambdas)
    gl = glob.cpu()
    stats_check = {
        "count_ok": bool(gl[-1].item() == float(world) * E),
        "cost_sum_int": bool(torch.equal(gl[:K], gl[:K].round()) and float(gl[:K].min()) >= 0),
        # integer-valued slots (cost sums, violation counts, episode count) must agree exactly, the f64 return
        # sums up to the association of the two communicators' reduction trees
        "abi_allreduce_matches_torch": bool(torch.equal(glob[:2 * K], via_torch[:2 * K]) and glob[-1] == via_torch[-1]
                                            and torch.allclose(glob, via_torch, rtol=1e-12, atol=0.0)),
        "lambda_equal_across_ranks": bool(all(torch.equal(x, lam_all[0]) for x in lam_all)),
        "world": world, "episodes": float(gl[-1].item()), "nccl": int(lib.smarl_comm_nccl_version()),
    }

    # ---- the same closed loop for a consumer of the u8 position rows (a fused policy): obs = NULL -----------------
    def policy_path_loop(ev_a=None, ev_b=None):
        closed_loop(ev_a, ev_b, obs=None)
    pp_ms, pp_step_ms = timed(policy_path_loop, a.steps, a.warmup, per_step_events=True)
    pp_ms /= a.steps
    pp_launch = pp_step_ms / (a.steps * T)
    pp_bytes = 10.0 * A * E                                     # pos read + write 4, action 1, reward 4, cost 1
    value_policy_path = {"value": world * agent_steps / (pp_ms * 1e-3), "unit": UNIT, "ms_per_step": pp_ms,
                         "mode": "closed loop without the float observation rows (obs = NULL): for policies that read "
                                 "the u8 position rows directly; rewards, costs, penalties and returns unchanged",
                         "roofline": {"bound": "hbm", "kernel": "coverage_step_kernel (obs=NULL, done=NULL)",
                                      "achieved": pp_bytes / (pp_launch * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                      "frac": pp_bytes / (pp_launch * 1e-3) / 1e9 / peak, "bytes_per_launch": pp_bytes,
                                      "launch_ms": pp_launch}}

    # ---- lean closed loop (extra): one env-reward row + no done flags in the rollout buffer ---------------
    lean = None
    if not a.no_fused:
        lbuf = env.new_rollout_buffer(T, g_mode=s.G_REWARD_TO_GO, lean=True)
        pshared = env._params_shared

        def lean_loop(ev_a=None, ev_b=None):
            _lib.check(lib.smarl_grid_reset(P(env.start_x), P(env.start_y), P(env.pos_x), P(env.pos_y), P(env.obs),
                                            A, E, ld, stream))
            if ev_a is not None:
                ev_a.record()
            for t in range(T):
                _lib.check(lib.smarl_coverage_step(C.byref(pshared), P(env.pos_x), P(env.pos_y), P(actions[t]),
                                                   P(env.obs), P(lbuf.reward[t]), P(lbuf.cost[t]), None,
                                                   P(meta.lambdas), P(lbuf.penalty[t]), E, ld, stream))
            if ev_b is not None:
                ev_b.record()
            _lib.check(lib.smarl_rollout_returns_shared(C.byref(acc), P(lbuf.reward), P(env._weights), P(lbuf.cost),
                                                        lbuf.cost_code, P(lbuf.penalty), None, P(lbuf.R), P(lbuf.modR),
                                                        P(lbuf.Csum), P(lbuf.G), P(lbuf.stats_vec),
                                                        P(lbuf.stats_scratch), A, K, E, ld, stream))
            comm.allreduce(lbuf.stats_vec)
            _lib.check(lib.smarl_lambda_update(P(meta.lambdas), P(lbuf.stats_vec), P(thr), 0.002, A, K, stream))
        l_ms, l_step_ms = timed(lean_loop, a.steps, a.warmup, per_step_events=True)
        l_ms /= a.steps
        l_launch = l_step_ms / (a.steps * T)
        l_bytes = (2 + 1 + 2 + 8 + 1 + 8.0 / A) * A * E        # pos in/out, action, obs, cost, (reward + penalty)/A
        lean = {"value": world * agent_steps / (l_ms * 1e-3), "unit": UNIT, "ms_per_step": l_ms,
                "mode": "closed loop, lean rollout buffer: one env-reward row (weights applied by "
                        "smarl_rollout_returns_shared), no per-step done flags",
                "roofline": {"bound": "hbm", "kernel": "coverage_step_kernel (reward_rows=1, done=NULL)",
                             "achieved": l_bytes / (l_launch * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                             "frac": l_bytes / (l_launch * 1e-3) / 1e9 / peak, "bytes_per_launch": l_bytes,
                             "launch_ms": l_launch}}
        del lbuf

    # ---- fused open-loop rollout (extra) ------------------------------------------------------------
    fused = None
    if not a.no_fused:
        out = {}
        def fused_fn():
            env.rollout(actions, lambdas=meta.lambdas, gamma=a.gamma, thresholds=thr, g_mode=s.G_NONE, out=out)
        f_ms, _ = timed(fused_fn, a.steps, a.warmup)
        f_ms /= a.steps
        f_bytes = (1.0 + 16.0 / T) * A * E * T                 # SURVEY 8d: 1 + 16/T B per agent-step
        fused = {"value": world * agent_steps / (f_ms * 1e-3), "unit": UNIT, "ms_per_step": f_ms,
                 "kernel": "coverage_rollout_kernel (open loop, g_mode 0)",
                 "roofline": {"bound": "hbm", "achieved": f_bytes / (f_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                              "frac": f_bytes / (f_ms * 1e-3) / 1e9 / peak,
                              "note": "issue-bound by design: 1.32 algorithmic B per agent-step"}}
        del out

    # ---- the other named configs (BASELINE.json configs[1], [2]) and the literal sharded configs[3] ---------------
    configs = None
    if not a.no_configs:
        configs = {}
        try:
            configs["c2_collision_65536"] = bench_named_config(s, _lib, "collision", 5, 3, 65536, 50, 0.99, peak, graph=True)
            configs["c3_congestion_1M_T100"] = bench_named_config(s, _lib, "congestion", 10, 8, 1 << 20, 100, 0.9, peak,
                                                                  graph=False)
            configs["c4_strong"] = bench_strong(s, _lib, lib, sd, comm, a, rank, world, dev, peak, timed)
        except Exception as ex:                                 # an extra must never cost the headline line
            configs["error"] = str(ex)[:300]
        torch.cuda.empty_cache()

    # ---- the loop with the reference's policy networks in it (not part of `value`) ------------------------------------
    policy_loop = None
    if not a.no_policy:
        try:
            policy_loop = bench_policy_loop(s, a, dev)
        except Exception as ex:
            policy_loop = {"error": str(ex)[:300]}
        torch.cuda.empty_cache()

    # ---- end to end through the host-buffer C-ABI call -----------------------------------------------
    e2e = None
    if not a.no_e2e:
        del buf
        torch.cuda.empty_cache()
        sess = C.c_void_p()
        _lib.check(lib.smarl_host_session_create(C.byref(sess), _lib.ENV_COVERAGE, A, T, E, 0))
        assert lib.smarl_host_session_ld(sess) == ld
        pin = dict(pin_memory=True)
        pinned_nodes, pinned_raw = [], []

        def pinned(shape, dtype):
            """Pinned host array from smarl_host_alloc_pinned: placed on the NUMA node of this rank's GPU when the
            kernel allows it (matters once several ranks share the box)."""
            n = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
            raw, node = C.c_void_p(), C.c_int32(-1)
            _lib.check(lib.smarl_host_alloc_pinned(C.byref(raw), n, C.byref(node)))
            pinned_raw.append(raw)
            pinned_nodes.append(int(node.value))
            arr = np.ctypeslib.as_array((C.c_uint8 * n).from_address(raw.value))
            return torch.from_numpy(arr).view(dtype).reshape(shape)
        actions_h = pinned((T, A, ld), torch.uint8).copy_(actions)
        sx_h = pinned((A, ld), torch.uint8).copy_(env.start_x)
        sy_h = pinned((A, ld), torch.uint8).copy_(env.start_y)
        R_h = pinned((A, ld), torch.float32)
        M_h = pinned((A, ld), torch.float32)
        C_h = pinned((K, ld), torch.int32)
        st_h = torch.zeros(lib.smarl_stats_len(A, K), dtype=torch.float64)
        lut_h = env._lut.cpu()
        w_h = torch.tensor(weights, dtype=torch.float32)
        lam_h = meta.lambdas.cpu()
        thr_h = thr.cpu()
        hp = _lib.CoverageParams(S, A, lut_h.numel(), 0, lut_h.data_ptr(), w_h.data_ptr())
        hacc = _lib.Accounting(a.gamma, T, 0, thr_h.data_ptr())

        def host_call():
            _lib.check(lib.smarl_host_coverage_rollout(sess, C.byref(hp), C.byref(hacc), sx_h.data_ptr(),
                                                       sy_h.data_ptr(), actions_h.data_ptr(), lam_h.data_ptr(),
                                                       R_h.data_ptr(), M_h.data_ptr(), C_h.data_ptr(),
                                                       st_h.data_ptr()))
        e2e_steps = a.steps
        for _ in range(2):
            host_call()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            host_call()                                         # synchronous: returns with host results ready
        el = time.perf_counter() - t0
        el_local = el
        tt = torch.tensor([el], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        el = float(tt.item())
        h2d_b, d2h_b = int(T * A * ld + 2 * A * ld), int(3 * A * ld * 4 + 8 * lib.smarl_stats_len(A, K))
        mine = torch.tensor([h2d_b * e2e_steps / el_local / 1e9], dtype=torch.float64, device=dev)
        per_rank = [mine.clone() for _ in range(world)]
        if world > 1:
            dist.all_gather(per_rank, mine)
        e2e = {"value": world * agent_steps * e2e_steps / el, "unit": UNIT,
               "per_rank_h2d_gbs": [round(float(x.item()), 2) for x in per_rank],
               "pinned_numa_node": sorted(set(pinned_nodes)),
               "h2d_bytes_per_step": int(T * A * ld + 2 * A * ld),
               "d2h_bytes_per_step": int(3 * A * ld * 4 + 8 * lib.smarl_stats_len(A, K)),
               "ms_per_step": 1e3 * el / e2e_steps, "steps": e2e_steps,
               "api": "smarl_host_coverage_rollout (pinned host buffers, fused rollout, chunked 2-stream pipeline)",
               "check": {"mean_cost_agent0": float(st_h[0] / st_h[-1]), "episodes": float(st_h[-1])}}
        # extra: the same call with 4-bit packed actions (half the PCIe bytes; expanded on the device)
        try:
            packed_h = torch.empty((T, A, ld // 2), dtype=torch.uint8, **pin)
            packed_h.copy_(actions[:, :, 0::2] | (actions[:, :, 1::2] << 4))
            R_ref = R_h.clone()

            def host_call4():
                _lib.check(lib.smarl_host_coverage_rollout_packed4(sess, C.byref(hp), C.byref(hacc), sx_h.data_ptr(),
                                                                   sy_h.data_ptr(), packed_h.data_ptr(), lam_h.data_ptr(),
                                                                   R_h.data_ptr(), M_h.data_ptr(), C_h.data_ptr(),
                                                                   st_h.data_ptr()))
            for _ in range(2):
                host_call4()
            same = bool(torch.equal(R_h, R_ref))
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                host_call4()
            el4 = time.perf_counter() - t0
            tt = torch.tensor([el4], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            el4 = float(tt.item())
            e2e["packed4"] = {"value": world * agent_steps * e2e_steps / el4, "unit": UNIT,
                              "h2d_bytes_per_step": int(T * A * ld // 2 + 2 * A * ld), "ms_per_step": 1e3 * el4 / e2e_steps,
                              "api": "smarl_host_coverage_rollout_packed4 (two 4-bit actions per byte)",
                              "same_results_as_u8": same}
        except Exception as ex:
            e2e["packed4"] = {"error": str(ex)[:200]}
        # extra: base-5 packed actions, three per byte (a third of the action bytes on PCIe; expanded on the device)
        try:
            pitch5 = int(lib.smarl_host_session_pitch5(sess))
            pad = torch.zeros((T, A, 3 * pitch5), dtype=torch.uint8, device=dev)
            pad[:, :, :ld] = actions
            packed5_h = pinned((T, A, pitch5), torch.uint8)
            packed5_h.copy_(pad[:, :, 0::3] + 5 * pad[:, :, 1::3] + 25 * pad[:, :, 2::3])
            del pad

            def host_call5():
                _lib.check(lib.smarl_host_coverage_rollout_packed5(sess, C.byref(hp), C.byref(hacc), sx_h.data_ptr(),
                                                                   sy_h.data_ptr(), packed5_h.data_ptr(), lam_h.data_ptr(),
                                                                   R_h.data_ptr(), M_h.data_ptr(), C_h.data_ptr(),
                                                                   st_h.data_ptr()))
            for _ in range(2):
                host_call5()
            same5 = bool(torch.equal(R_h, R_ref))
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                host_call5()
            el5 = time.perf_counter() - t0
            tt = torch.tensor([el5], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            el5 = float(tt.item())
            e2e["packed5"] = {"value": world * agent_steps * e2e_steps / el5, "unit": UNIT,
                              "h2d_bytes_per_step": int(T * A * pitch5 + 2 * A * ld), "ms_per_step": 1e3 * el5 / e2e_steps,
                              "api": "smarl_host_coverage_rollout_packed5 (three base-5 actions per byte)",
                              "same_results_as_u8": same5}
        except Exception as ex:
            e2e["packed5"] = {"error": str(ex)[:200]}
        # extra: the same call on the reference's env-major arrays ([T][E][A] actions, [E][A] results); the layout
        # change runs on the device inside the pipeline
        try:
            del packed_h
            act_em = torch.empty((T, E, A), dtype=torch.uint8, **pin)
            act_em.copy_(actions[:, :, :E].permute(0, 2, 1))
            st_em = torch.empty((E, A, 2), dtype=torch.uint8, **pin)
            st_em.copy_(torch.stack([env.start_x[:, :E].t(), env.start_y[:, :E].t()], dim=2))
            R_em = torch.empty((E, A), dtype=torch.float32, **pin)
            M_em = torch.empty((E, A), dtype=torch.float32, **pin)
            C_em = torch.empty((E, A), dtype=torch.int32, **pin)

            def host_call_em():
                _lib.check(lib.smarl_host_coverage_rollout_envmajor(sess, C.byref(hp), C.byref(hacc), st_em.data_ptr(),
                                                                    act_em.data_ptr(), lam_h.data_ptr(), R_em.data_ptr(),
                                                                    M_em.data_ptr(), C_em.data_ptr(), st_h.data_ptr()))
            for _ in range(2):
                host_call_em()
            same = bool(torch.equal(R_em, R_ref[:, :E].t()))
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                host_call_em()
            el_em = time.perf_counter() - t0
            tt = torch.tensor([el_em], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            el_em = float(tt.item())
            e2e["envmajor"] = {"value": world * agent_steps * e2e_steps / el_em, "unit": UNIT,
                               "h2d_bytes_per_step": int(T * A * E + 2 * A * E), "d2h_bytes_per_step": int(3 * A * E * 4),
                               "ms_per_step": 1e3 * el_em / e2e_steps,
                               "api": "smarl_host_coverage_rollout_envmajor (reference orientation: actions [T][E][A], "
                                      "results [E][A]; transposed on the device)",
                               "same_results_as_agent_major": same}
        except Exception as ex:
            e2e["envmajor"] = {"error": str(ex)[:200]}
        lib.smarl_host_session_destroy(sess)

    # ---- CPU baseline (rank 0, N=1 only) ---------------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        rate, cores = cpu_rate(a, a.cpu_seconds)
        cmod, ckind = cpu_impl()
        one_steps, one_el = cmod.time_episodes("coverage", a.size, a.n_agents, a.max_t, a.gamma, 2.0)
        cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": ckind, "one_core": one_steps / one_el,
               "sample": f"{a.cpu_seconds:.0f}s of whole episodes of the same env config, one env per process on "
                         f"{cores} processes ({'the unmodified reference classes, oracle/_ref' if ckind == 'reference' else 'oracle/scalar_port.py'}"
                         f": env.step + MetaAgent.act + Buffer + reward-to-go)"}
        try:                                       # extra: the plain-C oracle (pthreads) on a 2^16-env slice
            from oracle import c_oracle as co
            from oracle import numpy_oracle as no
            n = 1 << 16
            lut64 = no.coverage_penalty_lut(S, no.coverage_fieldview(S, A))
            sx, sy = env.start_x[:, :n].cpu().numpy(), env.start_y[:, :n].cpu().numpy()
            act = actions[:, :, :n].cpu().numpy()
            t0 = time.perf_counter()
            co.coverage_rollout(S, sx, sy, act, lut64, np.asarray(weights), np.full(A, 0.1), a.gamma, n)
            cpu["c_oracle"] = {"value": n * A * T / (time.perf_counter() - t0), "unit": UNIT, "threads": co.num_threads(),
                               "sample": "oracle/c/oracle.c fused rollout of 65536 envs (batched C, not the reference's execution model)"}
        except Exception as ex:                    # the C oracle is optional test infrastructure
            cpu["c_oracle"] = {"error": str(ex)[:200]}

    if rank == 0:
        emit({
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": workload_name(a), "mode": "closed-loop step API + returns kernel",
                       "l2": "inputs larger than L2: each step launch streams 1.2 GB (18 B x 16 x 2^22)",
                       "agent_steps_per_step": world * agent_steps,
                       "protocol": "per agent-step: pos r/w, action, obs f32 x2, reward f32, cost u8; done is constant "
                                   "False for Coverage and returned as a cached zero view, not stored per step"},
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches_per_step * a.steps,
            "roofline": roofline, "cpu_baseline": cpu, "fused": fused, "lean": lean,
            "value_policy_path": value_policy_path, "configs": configs, "stats_check": stats_check,
            "policy_loop": policy_loop,
        })
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
