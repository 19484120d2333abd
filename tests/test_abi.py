"""CPU checks of the drop-in boundary: libsmarl.so loads, exports every symbol that
include/smarl.h declares, the ctypes prototypes cover the header, argument validation
fails loudly before any CUDA work, and the product has no CPU / oracle fallback."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "smarl.h")


def declared_symbols():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(smarl_[a-z0-9_]+)\s*\(", text)))


@pytest.fixture(scope="module")
def lib():
    from safe_multiagent_rl_b200 import _lib, build
    build.build()
    return _lib.load()


def test_header_symbols_exported_and_bound(lib):
    from safe_multiagent_rl_b200 import _lib
    syms = declared_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in smarl.h but not exported"
    assert sorted(_lib.PROTOTYPES) == syms, "ctypes prototypes and header disagree"


def test_every_declared_symbol_cites_the_reference():
    text = open(HEADER).read()
    for needle in ["coverage.py:", "congestion.py:", "collision_avoidance.py:", "meta_agent.py:", "buffer.py:",
                   "agent.py:", "main.py:"]:
        assert needle in text


def test_abi_struct_sizes():
    from safe_multiagent_rl_b200 import _lib
    assert C.sizeof(_lib.CoverageParams) == 32
    assert C.sizeof(_lib.Accounting) == 24
    assert C.sizeof(_lib.CongestionParams) == 64      # ABI v2: + episode_dev
    assert C.sizeof(_lib.CollisionParams) == 32


def agent_count_call(lib, env, kind, n_agents, n_envs):
    """One open-loop step or rollout of `env` with `n_agents` agents over n_envs = ld envs, every other argument valid.
    The state pointers are fake: the call must be rejected before it touches them."""
    from safe_multiagent_rl_b200 import _lib
    f = C.c_void_p(0x1000)
    acc = C.byref(_lib.Accounting(0.9, 4, 0, None))
    if env == "coverage":
        p = C.byref(_lib.CoverageParams(5, n_agents, 0, 0, None, None))
        if kind == "step":
            return lib.smarl_coverage_step(p, f, f, f, None, f, f, None, None, None, n_envs, n_envs, None)
        return lib.smarl_coverage_rollout(p, acc, f, f, f, None, f, f, f, f, f, None, None, None, None, n_envs, n_envs,
                                          None)
    if env == "congestion":
        p = C.byref(_lib.CongestionParams(5, n_agents, f, 0, 0, 0, 0, 0, None, None))
        if kind == "step":
            return lib.smarl_congestion_step(p, f, f, f, None, None, f, f, None, None, None, 0, n_envs, n_envs, None)
        return lib.smarl_congestion_rollout(p, acc, f, f, f, None, None, f, f, f, f, f, None, None, None, None, n_envs,
                                            n_envs, None)
    if env == "collision":
        p = C.byref(_lib.CollisionParams(5, n_agents, 3, 0, 0.25, 0, 0))
        if kind == "step":
            return lib.smarl_collision_step(p, f, f, f, f, f, None, f, f, None, None, None, None, n_envs, n_envs, None)
        return lib.smarl_collision_rollout(p, acc, f, f, f, f, None, f, f, f, f, f, f, f, None, None, None, None, n_envs,
                                           n_envs, None)
    p = C.byref(_lib.CoverageFloatParams(5, n_agents, 0, 0, 2.0, 0.0, 0.0, 0.0, 0.0, 0.0, None))
    if kind == "step":
        return lib.smarl_coverage_float_step(p, f, f, f, None, f, f, None, None, None, n_envs, n_envs, None)
    return lib.smarl_coverage_float_rollout(p, acc, f, f, f, None, f, f, f, f, f, None, None, None, None, n_envs, n_envs,
                                            None)


def test_validation_errors_before_any_cuda_work(lib):
    from safe_multiagent_rl_b200 import _lib
    p = _lib.CoverageParams(5, 3, 0, 0, None, None)
    fake = C.c_void_p(0x1000)   # never dereferenced: validation rejects the call first
    rc = lib.smarl_coverage_step(C.byref(p), fake, fake, fake, None, fake, fake, None, None, None, 10, 10, None)
    assert rc == -1 and b"multiple of 16" in lib.smarl_last_error()
    p = _lib.CoverageParams(300, 3, 0, 0, None, None)
    rc = lib.smarl_coverage_step(C.byref(p), fake, fake, fake, None, fake, fake, None, None, None, 16, 16, None)
    assert rc == -1 and b"size=300" in lib.smarl_last_error()
    p = _lib.CoverageParams(5, 3, 0, 0, None, None)
    rc = lib.smarl_coverage_step(C.byref(p), C.c_void_p(0x1001), fake, fake, None, fake, fake, None, None, None,
                                 16, 16, None)
    assert rc == -1 and b"aligned" in lib.smarl_last_error()
    with pytest.raises(_lib.SmarlError):
        _lib.check(rc)
    # The accounting arguments of the open-loop rollouts and the returns entry points: each call below fails on them
    f = fake
    cov = _lib.CoverageParams(5, 3, 0, 0, None, None)
    cong = _lib.CongestionParams(5, 3, f, 0, 0, 0, 0, 0, None, None)
    coll = _lib.CollisionParams(5, 3, 1, 0, 0.25, 0, 0)
    covf = _lib.CoverageFloatParams(5, 3, 0, 0, 2.0, 0.0, 0.0, 0.0, 0.0, 0.0, None)

    def acc(n_steps=4, g_mode=0):
        return C.byref(_lib.Accounting(0.9, n_steps, g_mode, None))
    entry_points = [   # (call(acc, G, g_scratch, stats, stats_scratch), longest episode, largest g_mode, takes g_scratch)
        (lambda a, G, gs, s, ss: lib.smarl_coverage_rollout(C.byref(cov), a, f, f, f, None, f, f, f, f, f, G, gs, s, ss,
                                                            16, 16, None), 255, 2, True),
        (lambda a, G, gs, s, ss: lib.smarl_congestion_rollout(C.byref(cong), a, f, f, f, None, None, f, f, f, f, f, G, gs,
                                                              s, ss, 16, 16, None), 2 ** 31 - 1, 2, True),
        (lambda a, G, gs, s, ss: lib.smarl_collision_rollout(C.byref(coll), a, f, f, f, f, None, f, f, f, f, f, f, f, G,
                                                             gs, s, ss, 16, 16, None), 2 ** 31 - 1, 2, True),
        (lambda a, G, gs, s, ss: lib.smarl_coverage_float_rollout(C.byref(covf), a, f, f, f, None, f, f, f, f, f, G, gs,
                                                                  s, ss, 16, 16, None), 2 ** 31 - 1, 2, True),
        (lambda a, G, gs, s, ss: lib.smarl_rollout_returns(a, f, f, 0, f, None, f, f, f, G, s, ss, 3, 3, 16, 16, None),
         2 ** 31 - 1, 3, False),
        (lambda a, G, gs, s, ss: lib.smarl_rollout_returns_shared(a, f, f, f, 0, f, None, f, f, f, G, s, ss, 3, 3, 16, 16,
                                                                  None), 2 ** 31 - 1, 3, False),
    ]
    for call, max_steps, max_g, takes_gs in entry_points:
        cases = [((None, f, f, None, None), b"accounting params is NULL"),
                 ((acc(n_steps=0), f, f, None, None), b"n_steps=0 outside"),
                 ((acc(g_mode=-1), f, f, None, None), b"bad g_mode -1"),
                 ((acc(g_mode=max_g + 1), f, f, None, None), b"bad g_mode %d" % (max_g + 1)),
                 ((acc(g_mode=2), None, f, None, None), b"needs G"),
                 ((acc(), f, f, f, None), b"stats and stats_scratch go together")]
        if max_steps < 2 ** 31 - 1:
            cases.append(((acc(n_steps=max_steps + 1), f, f, None, None), b"outside 1..%d" % max_steps))
        if takes_gs:
            cases.append(((acc(g_mode=1), f, None, None, None), b"needs g_scratch"))
        for args, needle in cases:
            assert call(*args) == -1 and needle in lib.smarl_last_error(), (needle, lib.smarl_last_error())
    # Agent counts no kernel is built for: the open-loop steps and rollouts leave them to the launchers' dispatch
    for env in ("coverage", "congestion", "collision", "coverage_float"):
        for kind in ("step", "rollout"):
            rc = agent_count_call(lib, env, kind, 0, 16)
            assert rc == -3 and b"n_agents=0 outside 1..32" in lib.smarl_last_error(), (env, kind)
    coop = b"cooperative %s kernels cover n_agents 9..32 (got 33)"
    for env, kind, needle in [("coverage", "step", coop % b"Coverage"), ("coverage", "rollout", b"n_agents=33 outside 1..32"),
                              ("congestion", "step", coop % b"Congestion"), ("congestion", "rollout", coop % b"Congestion"),
                              ("collision", "step", coop % b"Collision"), ("collision", "rollout", coop % b"Collision"),
                              ("coverage_float", "step", b"n_agents=33 outside 1..32"),
                              ("coverage_float", "rollout", b"n_agents=33 outside 1..32")]:
        rc = agent_count_call(lib, env, kind, 33, 16)
        assert rc == -3 and needle in lib.smarl_last_error(), (env, kind, rc, lib.smarl_last_error())
    assert lib.smarl_stats_len(16, 16) == 65
    assert lib.smarl_stats_scratch_len(3, 3, 50) == 26      # one row of partials per 32 envs


def test_register_capped_launchers_reject_bad_agent_counts(lib):
    """From 2^18 envs the A <= 4 kernels of these entry points run register-capped; a count below 1 must still be
    rejected before any launch, not run through the A = 4 kernel."""
    for env, kind in [("collision", "step"), ("collision", "rollout"), ("coverage_float", "rollout")]:
        for A in (0, -1):
            rc = agent_count_call(lib, env, kind, A, 1 << 18)
            assert rc == -3 and b"n_agents=%d outside 1..32" % A in lib.smarl_last_error(), (env, kind, A, rc)


def test_collision_rejects_agents_size_without_a_normal_square(lib):
    """The Collision kernels compare squared distances with agents_size^2 and (2 agents_size)^2 and take the square
    root only in a relative band around them.  Below 2^-511 that square is subnormal or zero and the band collapses
    (an agent exactly on its landmark would not reach it: qn = 0 < 0 is false), so every Collision entry point rejects
    such an agents_size before any CUDA work."""
    from safe_multiagent_rl_b200 import _lib
    f = C.c_void_p(0x1000)   # never dereferenced
    acc = C.byref(_lib.Accounting(0.9, 4, 0, None))
    pol = C.byref(_lib.GaussianPolicyParams(3, 6, 16, 2, 0, 0, f, f, f, f, f, f, 1, 0, None))
    tiny = 2.0 ** -511
    for agents_size in (1e-170, np.nextafter(tiny, 0), 2.0 ** -600, 5e-324):
        p = C.byref(_lib.CollisionParams(5, 3, 1, 0, float(agents_size), 0, 0))
        calls = {
            "reset": lambda: lib.smarl_collision_reset(p, f, f, f, f, f, f, None, None, 16, 16, None),
            "step": lambda: lib.smarl_collision_step(p, f, f, f, f, f, None, f, f, None, None, None, None, 16, 16, None),
            "rollout": lambda: lib.smarl_collision_rollout(p, acc, f, f, f, f, None, f, f, f, f, f, f, f, None, None,
                                                           None, None, 16, 16, None),
            "policy_rollout": lambda: lib.smarl_collision_policy_rollout(p, pol, acc, f, f, f, None, None, None, None,
                                                                         f, f, f, f, f, f, f, None, None, None, None,
                                                                         16, 16, None),
        }
        for name, call in calls.items():
            assert call() == -1 and b"below 2^-511" in lib.smarl_last_error(), (name, agents_size)
    for agents_size in (0.0, -0.25, float("nan")):
        p = C.byref(_lib.CollisionParams(5, 3, 1, 0, agents_size, 0, 0))
        assert lib.smarl_collision_step(p, f, f, f, f, f, None, f, f, None, None, None, None, 16, 16, None) == -1
        assert b"agents_size must be positive" in lib.smarl_last_error()


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback():
    import safe_multiagent_rl_b200 as s
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        s.BatchedCoverageDiscrete(5, 3, n_envs=4)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        s.BatchedCongestion(3, 3, n_envs=4)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        s.BatchedCollisionAvoidance(5, 3, n_envs=4)


def test_missing_library_fails_loudly(tmp_path):
    code = ("import os; os.environ['SMARL_LIB']=%r; from safe_multiagent_rl_b200 import _lib\n"
            "try:\n    _lib.load()\nexcept _lib.SmarlError as e:\n    print('RAISED', e)\n") % str(tmp_path / "nope.so")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT)
    assert "RAISED" in out.stdout and "no CPU fallback" in out.stdout


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "safe_multiagent_rl_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f
                assert "/root/reference" not in text, f
    code = "import sys, safe_multiagent_rl_b200; print(any(m == 'oracle' or m.startswith('oracle.') for m in sys.modules))"
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT)
    assert out.stdout.strip() == "False", out.stderr


def test_host_parameter_helpers_match_oracle():
    """Host-side parameter setup (penalty table, Philox keep threshold) against the oracle."""
    import numpy as np
    from oracle import numpy_oracle as no
    from oracle import philox
    from safe_multiagent_rl_b200.envs.congestion import keep_threshold
    from safe_multiagent_rl_b200.envs.coverage import penalty_table
    for size, A, fv in [(5, 3, None), (32, 16, None), (64, 32, None), (3, 2, 10.0), (10, 7, 2.5)]:
        f, table = penalty_table(size, A, fv)
        want = no.coverage_penalty_lut(size, no.coverage_fieldview(size, A, fv))
        assert f == no.coverage_fieldview(size, A, fv)
        n = len(table)
        assert np.array_equal(table, want[:n]) and not want[n:].any() and (n == 0 or table[-1] > 0)
    for noise in [0.0, 0.1, 0.5, 1.0, 0.3333]:
        assert keep_threshold(noise) == philox.keep_threshold(noise)
