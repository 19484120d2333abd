"""Time the learner's loss and gradient of the DiscretePolicy: the PyTorch path (T ``log_prob`` forwards, the loss and
autograd) against ``policy_gradient_loss`` (one kernel, smarl_policy_grad_discrete), and a whole agent cycle both ways.

    python tools/time_policy_grad.py [--rounds 5] [--min-window-ms 150] [--shapes cov:50:3:50 ...] [--out FILE]

Arms, alternated in one process, each timed with CUDA events over windows of at least --min-window-ms, median of
--rounds rounds:
  pytorch        zero_grad, the log_prob stack, -(logp * psi).mean(), backward
  fused          zero_grad, policy_gradient_loss(records, psi), backward
  kernel         smarl_policy_grad_discrete alone on preallocated outputs (the counters' memset and the kernel)
  cycle_pytorch  policy_rollout, psi standardisation, the pytorch loss and backward, Adam.step
  cycle_fused    the same with the fused loss
Shapes (kind:E:A:T): CoverageDiscrete (size 5) at 50 / 65 536 / 2^20 envs x 3 agents and 2^20 x 8, T = 50; Congestion
(size 3, noise 0.1) at 50 / 65 536 x 3, T = 10; CoverageDiscretized (5, coarseness 6) at 50 / 65 536 x 3, T = 50;
synthetic records (uniform positions and actions, 5 actions) at 2^18 x 16 and 2^18 x 32, T = 50, which have no
agent cycle.  The kernel's FMA rate counts 2 (2A) 16 + 3 16 NA FMAs per agent-sample; its share of peak is against
148 SMs x 128 FMA/clk x the SM clock nvidia-smi reports while the kernel runs.  The fused gradients and loss are
checked on the timed inputs against a float64 autograd: max|g - g64| <= max(4 max|g_torch32 - g64|, 1e-6 max|g64|).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import statistics
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

SHAPES = ["cov:50:3:50", "cov:65536:3:50", "cov:1048576:3:50", "cov:1048576:8:50", "cong:50:3:10",
          "cong:65536:3:10", "dz:50:3:50", "dz:65536:3:50", "syn:262144:16:50", "syn:262144:32:50"]


def event_ms(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def smi(fields):
    q = subprocess.run(["nvidia-smi", f"--query-gpu={fields}", "--format=csv,noheader,nounits", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return q.stdout.strip()


def setup(kind, E, A, T):
    import safe_multiagent_rl_b200 as s
    from safe_multiagent_rl_b200.policy import FusedDiscretePolicy, FusedDiscretizedPolicy
    torch.manual_seed(0)
    if kind == "cov":
        env = s.BatchedCoverageDiscrete(5, A, n_envs=E, shuffle=True, seed=1)
        pol = FusedDiscretePolicy(env, seed=7)
    elif kind == "cong":
        env = s.BatchedCongestionOnPolicy(3, A, n_envs=E, noise=0.1, shuffle=True, seed=1)
        pol = FusedDiscretePolicy(env, seed=7)
    elif kind == "dz":
        env = s.BatchedCoverageDiscretizedOnPolicy(5, A, n_envs=E, coarseness=6, shuffle=True, seed=1)
        pol = FusedDiscretizedPolicy(env, seed=7)
    else:
        env = s.BatchedCoverageDiscrete(5, A, n_envs=E)
        pol = FusedDiscretePolicy(env, seed=7)
    lam = torch.full((env.n_constraints,), 0.1, dtype=torch.float64, device="cuda")
    if kind == "syn":
        g = torch.Generator(device="cuda").manual_seed(0)
        obs_ = torch.zeros(T, 2 * A, env.ld, device="cuda")
        obs_[:, :, :E] = torch.randint(0, 6, (T, 2 * A, E), generator=g, device="cuda").float()
        act_ = torch.zeros(T, A, env.ld, dtype=torch.uint8, device="cuda")
        act_[:, :, :E] = torch.randint(0, 5, (T, A, E), generator=g, device="cuda", dtype=torch.uint8)
        out = {"obs_": obs_, "actions_": act_, "obs": obs_[:, :, :E].permute(0, 2, 1), "actions": act_[:, :, :E],
               "G": torch.randn(T, E, A, generator=g, device="cuda")}
        rollout = None
    else:
        out = env.policy_rollout(pol, T, lambdas=lam, g_mode=1)
        rollout = lambda: env.policy_rollout(pol, T, lambdas=lam, g_mode=1, out=out)
    return env, pol, out, rollout


def standardise(out):
    G = out["G"].permute(0, 2, 1)
    return (G - G.mean(dim=2, keepdim=True)) / (G.std(dim=2, keepdim=True) + 1e-6)


def pytorch_loss(pol, out, psi):
    T = psi.shape[0]
    logp = torch.stack([pol.log_prob(out["obs"][t], out["actions"][t].long()) for t in range(T)])
    return -(logp * psi).mean()


def reference64(pol, out, psi, scale):
    params = [p.detach().double().requires_grad_() for p in (pol.fc1.weight, pol.fc1.bias, pol.fc2.weight,
                                                              pol.fc2.bias)]
    grads, loss, mag = [torch.zeros_like(p) for p in params], 0.0, 0.0
    step = max(1, (1 << 22) // (psi.shape[1] * psi.shape[2]))
    for t0 in range(0, psi.shape[0], step):
        h = F.relu(torch.matmul(out["obs"][t0:t0 + step].double()[:, None], params[0]) + params[1])
        lp = F.log_softmax(torch.matmul(h, params[2]) + params[3], -1)
        lp = lp.gather(-1, out["actions"][t0:t0 + step].long()[..., None]).squeeze(-1)
        term = psi[t0:t0 + step].double() * lp
        chunk = -scale * term.sum()
        for g, d in zip(grads, torch.autograd.grad(chunk, params)):
            g += d
        loss, mag = loss + float(chunk), mag + float(term.abs().sum())
    return grads, loss, mag / psi.numel()


def grads_of(pol):
    return [p.grad.clone() for p in (pol.fc1.weight, pol.fc1.bias, pol.fc2.weight, pol.fc2.bias)]


def run_shape(kind, E, A, T, rounds, min_window_ms):
    from safe_multiagent_rl_b200 import _lib
    env, pol, out, rollout = setup(kind, E, A, T)
    psi = standardise(out).contiguous()
    NA = pol.n_actions
    opt = torch.optim.Adam(pol.parameters(), lr=1e-9)      # a tiny step: the timed inputs stay what was checked
    n = pol.lib.smarl_policy_grad_scratch_len(A, NA, T, E)
    outs = [torch.empty_like(p) for p in (pol.fc1.weight, pol.fc1.bias, pol.fc2.weight, pol.fc2.bias)]
    outs += [torch.empty((), dtype=torch.float64, device="cuda"), torch.empty(n, dtype=torch.float64, device="cuda")]
    psi_slab = torch.zeros(T, A, env.ld, device="cuda")
    psi_slab[:, :, :E] = psi

    def kernel():
        p = pol.c_params(env)
        _lib.check(pol.lib.smarl_policy_grad_discrete(C.byref(p), _lib.ptr(out["obs_"]), _lib.ptr(out["actions_"]),
                                                      _lib.ptr(psi_slab), T, 1.0 / (T * A * E),
                                                      *[_lib.ptr(o) for o in outs], E, env.ld, _lib.stream_ptr()))

    def pytorch():
        pol.zero_grad()
        pytorch_loss(pol, out, psi).backward()

    def fused():
        pol.zero_grad()
        pol.policy_gradient_loss(out, psi).backward()

    arms = {"pytorch": pytorch, "fused": fused, "kernel": kernel}
    if rollout is not None:
        def cycle(loss_fn):
            def fn():
                rollout()
                adv = standardise(out)
                opt.zero_grad()
                loss_fn(adv).backward()
                opt.step()
            return fn
        arms["cycle_pytorch"] = cycle(lambda adv: pytorch_loss(pol, out, adv))
        arms["cycle_fused"] = cycle(lambda adv: pol.policy_gradient_loss(out, adv))
    for fn in arms.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    iters = {k: max(1, math.ceil(min_window_ms / event_ms(fn, 3))) for k, fn in arms.items()}
    times = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            times[k].append(event_ms(fn, iters[k]))
    med = {k: statistics.median(v) for k, v in times.items()}
    # the SM clock while the kernel runs: enqueue about 0.5 s of it, read the clock, then wait
    for _ in range(max(1, int(500 / med["kernel"]))):
        kernel()
    clock = smi("clocks.sm")
    torch.cuda.synchronize()
    # check the timed inputs (the cycles moved the weights by at most 1e-9 per step: recheck on the current ones)
    if rollout is not None:
        rollout()
        psi.copy_(standardise(out))
    pol.zero_grad()
    loss = pol.policy_gradient_loss(out, psi)
    loss.backward()
    got = grads_of(pol)
    pol.zero_grad()
    pytorch_loss(pol, out, psi).backward()
    g32 = grads_of(pol)
    g64, l64, mag = reference64(pol, out, psi, 1.0 / (T * A * E))
    check = {}
    for name, g, base, want in zip(("w1", "b1", "w2", "b2"), got, g32, g64):
        err, err32 = float((g.double() - want).abs().max()), float((base.double() - want).abs().max())
        check[name] = {"err": err, "err_torch32": err32, "ok": err <= max(4 * err32, 1e-6 * float(want.abs().max()))}
    check["loss"] = {"err": abs(float(loss.detach()) - l64), "tol": 1e-5 * mag, "ok": abs(float(loss.detach()) - l64) <= 1e-5 * mag}
    fmas = (2 * (2 * A) * 16 + 3 * 16 * NA) * A * T * E
    rate = fmas / (med["kernel"] * 1e-3)
    peak = 148 * 128 * float(clock) * 1e6
    res = {"kind": kind, "n_envs": E, "n_agents": A, "n_actions": NA, "T": T, "iters": iters, "rounds": rounds,
           "ms": {k: {"median": med[k], "all": v} for k, v in times.items()},
           "speedup_fused_vs_pytorch": med["pytorch"] / med["fused"],
           "kernel_fma_per_s": rate, "sm_clock_mhz": float(clock), "share_of_fp32_fma_peak": rate / peak,
           "check_vs_float64": check, "all_ok": all(v["ok"] for v in check.values())}
    if rollout is not None:
        res["speedup_cycle_fused_vs_pytorch"] = med["cycle_pytorch"] / med["cycle_fused"]
    del env, pol, out, outs, opt, arms
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--min-window-ms", type=float, default=150.0)
    ap.add_argument("--shapes", nargs="*", default=SHAPES, help="kind:E:A:T, kind in cov, cong, dz, syn")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool times the GPU and has no CPU mode")
    info = {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": smi("name,power.limit,clocks.max.sm")}
    lines = [json.dumps({"gpu": info})]
    print(lines[-1], flush=True)
    for sh in a.shapes:
        kind, E, A, T = sh.split(":")
        lines.append(json.dumps(run_shape(kind, int(E), int(A), int(T), a.rounds, a.min_window_ms)))
        print(lines[-1], flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
