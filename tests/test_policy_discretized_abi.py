"""CPU checks of the argument validation of smarl_policy_act_discretized and smarl_coverage_discretized_policy_rollout:
every rejected input returns its code and message before any CUDA work, so the pointers below are fake and never
dereferenced."""
import ctypes as C

import pytest

FAKE = C.c_void_p(0x1000)
ODD = C.c_void_p(0x1008)          # 8-byte aligned, not 16
SHAPE9 = b"CoverageDiscretized runs the reference's DiscretePolicy of hidden 16 and 9 actions"


@pytest.fixture(scope="module")
def lib():
    from safe_multiagent_rl_b200 import _lib, build
    build.build()
    return _lib.load()


def policy(A=3, hidden=16, n_actions=9, null_weight=False):
    from safe_multiagent_rl_b200 import _lib
    return _lib.DiscretePolicyParams(A, hidden, n_actions, 0, None if null_weight else FAKE, FAKE, FAKE, FAKE, 1, 0,
                                     None)


def act(lib, A=3, hidden=16, n_actions=9, null_weight=False, null=(), odd=(), t=0, n_envs=16, ld=16, params=True):
    p = policy(A, hidden, n_actions, null_weight)
    ptrs = {k: (None if k in null else ODD if k in odd else FAKE) for k in ("obs", "actions", "logp")}
    return lib.smarl_policy_act_discretized(C.byref(p) if params else None, ptrs["obs"], ptrs["actions"],
                                            ptrs["logp"], t, n_envs, ld, None)


def rollout(lib, A=3, mode=1, size=6, zoom=1.0, pol_agents=None, hidden=16, n_actions=9, null_weight=False, n_steps=4,
            g_mode=0, null=(), stats=False, stats_scratch=False, params=True, pol=True, accounting=True, n_envs=16,
            ld=16):
    """One call with every argument valid unless a keyword says otherwise; `null` names pointer arguments to pass as
    NULL."""
    from safe_multiagent_rl_b200 import _lib
    p = _lib.CoverageFloatParams(size, A, mode, 0, 2.0, 0.0, zoom, size * zoom, 1.0, 1.4, None)
    pp = policy(A if pol_agents is None else pol_agents, hidden, n_actions, null_weight)
    acc = _lib.Accounting(0.9, n_steps, g_mode, None)
    names = ["start_x", "start_y", "lambdas", "obs_rec", "actions", "logp", "final_x", "final_y", "R", "modR", "C",
             "G", "g_scratch"]
    ptrs = {k: (None if k in null else FAKE) for k in names}
    return lib.smarl_coverage_discretized_policy_rollout(
        C.byref(p) if params else None, C.byref(pp) if pol else None, C.byref(acc) if accounting else None,
        *[ptrs[k] for k in names], FAKE if stats else None, FAKE if stats_scratch else None, n_envs, ld, None)


def expect(lib, fn, rc_want, needle, **kw):
    rc = fn(lib, **kw)
    assert rc == rc_want and needle in lib.smarl_last_error(), (kw, rc, lib.smarl_last_error())


def test_policy_act_rejections(lib):
    assert act(lib, params=False) == -1 and b"policy params is NULL" in lib.smarl_last_error()
    expect(lib, act, -1, b"n_agents=0 outside 1..32", A=0)
    expect(lib, act, -1, b"n_agents=33 outside 1..32", A=33)
    expect(lib, act, -1, SHAPE9 + b" (got 8, 9)", hidden=8)
    expect(lib, act, -1, SHAPE9 + b" (got 16, 5)", n_actions=5)
    expect(lib, act, -1, b"null pointer", null_weight=True)
    for name in ("obs", "actions"):
        expect(lib, act, -1, b"null pointer", null=(name,))
    expect(lib, act, -1, b"t=-1 outside 0..65535", t=-1)
    expect(lib, act, -1, b"t=65536 outside 0..65535", t=65536)
    for name in ("obs", "actions", "logp"):
        expect(lib, act, -1, b"pointers must be 16-byte aligned", odd=(name,))
    expect(lib, act, -1, b"multiple of 16", n_envs=10, ld=10)


def test_policy_act_discrete_still_rejects_nine_actions(lib):
    """The grid envs' entry point keeps its 5-action shape and its message."""
    p = policy(n_actions=9)
    assert lib.smarl_policy_act_discrete(C.byref(p), FAKE, FAKE, FAKE, None, 0, 16, 16, None) == -1
    assert (b"only the reference's DiscretePolicy shape (hidden 16, 5 actions) is built (got 16, 9)"
            in lib.smarl_last_error())


def test_rollout_agent_counts_and_mode(lib):
    expect(lib, rollout, -1, b"n_agents=0 outside 1..32", A=0)
    expect(lib, rollout, -1, b"n_agents=33 outside 1..32", A=33)
    for A in (9, 32):
        expect(lib, rollout, -3, b"runs one thread per env: n_agents=%d above 8" % A, A=A)
    expect(lib, rollout, -3, b"runs the discretized env (mode 1), not mode 0", mode=0)
    expect(lib, rollout, -1, b"bad mode 2", mode=2)
    expect(lib, rollout, -1, b"mode 1 needs zoom > 0", zoom=0.0)


def test_rollout_policy_shape(lib):
    expect(lib, rollout, -1, b"policy has 2 agents, the env 3", pol_agents=2)
    expect(lib, rollout, -1, SHAPE9 + b" (got 8, 9)", hidden=8)
    expect(lib, rollout, -1, SHAPE9 + b" (got 16, 5)", n_actions=5)
    expect(lib, rollout, -1, b"null pointer", null_weight=True)


def test_rollout_accounting(lib):
    expect(lib, rollout, -1, b"n_steps=0 outside 1..65536", n_steps=0)
    expect(lib, rollout, -1, b"n_steps=65537 outside 1..65536", n_steps=65537)
    expect(lib, rollout, -1, b"bad g_mode -1", g_mode=-1)
    expect(lib, rollout, -1, b"bad g_mode 3", g_mode=3)
    expect(lib, rollout, -1, b"needs G", g_mode=2, null=("G",))
    expect(lib, rollout, -1, b"g_mode 1 needs g_scratch", g_mode=1, null=("g_scratch",))
    expect(lib, rollout, -1, b"stats and stats_scratch go together", stats=True)


def test_rollout_pointers(lib):
    for kw in (dict(params=False), dict(pol=False), dict(accounting=False)):
        assert rollout(lib, **kw) == -1 and b"params is NULL" in lib.smarl_last_error()
    for name in ("start_x", "start_y", "R", "modR", "C"):
        expect(lib, rollout, -1, b"null required pointer", null=(name,))
    expect(lib, rollout, -1, b"multiple of 16", n_envs=10, ld=10)
