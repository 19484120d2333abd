"""CPU checks of smarl_coverage_policy_rollout's argument validation: every rejected input returns its code and message
before any CUDA work, so the pointers below are fake and never dereferenced."""
import ctypes as C

import pytest

FAKE = C.c_void_p(0x1000)
ODD = C.c_void_p(0x1008)          # 8-byte aligned, not 16


@pytest.fixture(scope="module")
def lib():
    from safe_multiagent_rl_b200 import _lib, build
    build.build()
    return _lib.load()


def call(lib, A=3, size=5, lut_len=0, lut=None, pol_agents=None, hidden=16, n_actions=5, null_weight=False,
         n_steps=4, g_mode=0, null=(), odd=(), stats=False, stats_scratch=False, params=True, policy=True,
         accounting=True, n_envs=16, ld=16):
    """One call with every argument valid unless a keyword says otherwise; `null` / `odd` name pointer arguments to
    pass as NULL / misaligned."""
    from safe_multiagent_rl_b200 import _lib
    p = _lib.CoverageParams(size, A, lut_len, 0, lut, None)
    pol = _lib.DiscretePolicyParams(A if pol_agents is None else pol_agents, hidden, n_actions, 0,
                                    None if null_weight else FAKE, FAKE, FAKE, FAKE, 1, 0, None)
    acc = _lib.Accounting(0.9, n_steps, g_mode, None)
    names = ["start_x", "start_y", "lambdas", "obs_rec", "actions", "logp", "final_x", "final_y", "R", "modR", "C",
             "G", "g_scratch"]
    ptrs = {k: (None if k in null else ODD if k in odd else FAKE) for k in names}
    return lib.smarl_coverage_policy_rollout(
        C.byref(p) if params else None, C.byref(pol) if policy else None, C.byref(acc) if accounting else None,
        *[ptrs[k] for k in names], FAKE if stats else None, FAKE if stats_scratch else None, n_envs, ld, None)


def expect(lib, rc_want, needle, **kw):
    rc = call(lib, **kw)
    assert rc == rc_want and needle in lib.smarl_last_error(), (kw, rc, lib.smarl_last_error())


def test_agent_counts(lib):
    expect(lib, -1, b"n_agents=0 outside 1..32", A=0)
    expect(lib, -1, b"n_agents=33 outside 1..32", A=33)
    for A in (9, 32):
        expect(lib, -3, b"runs one thread per four envs: n_agents=%d above 8" % A, A=A)


def test_policy_shape(lib):
    expect(lib, -1, b"policy has 2 agents, the env 3", pol_agents=2)
    shape = b"only the reference's DiscretePolicy shape (hidden 16, 5 actions) is built"
    expect(lib, -1, shape + b" (got 8, 5)", hidden=8)
    expect(lib, -1, shape + b" (got 16, 9)", n_actions=9)
    expect(lib, -1, b"null pointer", null_weight=True)


def test_accounting(lib):
    expect(lib, -1, b"n_steps=0 outside 1..255", n_steps=0)
    expect(lib, -1, b"n_steps=256 outside 1..255", n_steps=256)
    expect(lib, -1, b"bad g_mode -1", g_mode=-1)
    expect(lib, -1, b"bad g_mode 3", g_mode=3)
    expect(lib, -1, b"needs G", g_mode=2, null=("G",))
    expect(lib, -1, b"g_mode 1 needs g_scratch", g_mode=1, null=("g_scratch",))
    expect(lib, -1, b"stats and stats_scratch go together", stats=True)
    assert call(lib, accounting=False) == -1 and b"params is NULL" in lib.smarl_last_error()


def test_pointers(lib):
    assert call(lib, params=False) == -1 and b"params is NULL" in lib.smarl_last_error()
    assert call(lib, policy=False) == -1 and b"params is NULL" in lib.smarl_last_error()
    for name in ("start_x", "start_y", "R", "modR", "C"):
        expect(lib, -1, b"null required pointer", null=(name,))
    for name in ("start_x", "start_y", "obs_rec", "actions", "logp", "final_x", "final_y", "R", "modR", "C", "G",
                 "g_scratch"):
        expect(lib, -1, b"pointers must be 16-byte aligned", odd=(name,))
    expect(lib, -1, b"multiple of 16", n_envs=10, ld=10)


def test_env_params(lib):
    expect(lib, -1, b"size=0 outside 1..127", size=0)
    expect(lib, -1, b"size=128 outside 1..127", size=128)
    expect(lib, -1, b"bad penalty table", lut_len=4, lut=None)
    expect(lib, -3, b"lut_len=12280 exceeds the shared-memory table limit 12279", lut_len=12280, lut=FAKE)


def test_policy_act_discrete_keeps_its_checks(lib):
    """smarl_policy_act_discrete shares the policy checks: same codes and messages as before."""
    from safe_multiagent_rl_b200 import _lib

    def act(A=3, hidden=16, n_actions=5, null_weight=False, null_pos=False):
        p = _lib.DiscretePolicyParams(A, hidden, n_actions, 0, None if null_weight else FAKE, FAKE, FAKE, FAKE, 1, 0,
                                      None)
        return lib.smarl_policy_act_discrete(C.byref(p), None if null_pos else FAKE, FAKE, FAKE, None, 0, 16, 16, None)
    assert lib.smarl_policy_act_discrete(None, FAKE, FAKE, FAKE, None, 0, 16, 16, None) == -1
    assert b"policy params is NULL" in lib.smarl_last_error()
    assert act(A=0) == -1 and b"n_agents=0 outside 1..32" in lib.smarl_last_error()
    assert act(hidden=8) == -1 and b"DiscretePolicy shape (hidden 16, 5 actions) is built (got 8, 5)" in lib.smarl_last_error()
    assert act(null_weight=True) == -1 and b"null pointer" in lib.smarl_last_error()
    assert act(null_pos=True) == -1 and b"null pointer" in lib.smarl_last_error()
