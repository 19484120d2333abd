"""CPU checks of smarl_congestion_policy_rollout's argument validation: every rejected input returns its code and
message before any CUDA work, so the pointers below are fake and never dereferenced.  Also checks that the open-loop
Congestion entry points keep their own parameter checks, which they share with it."""
import ctypes as C

import pytest

FAKE = C.c_void_p(0x1000)
ODD = C.c_void_p(0x1008)          # 8-byte aligned, not 16


@pytest.fixture(scope="module")
def lib():
    from safe_multiagent_rl_b200 import _lib, build
    build.build()
    return _lib.load()


def params(A=3, size=3, demand=True, noise_mode=2, keep_threshold=1 << 31):
    from safe_multiagent_rl_b200 import _lib
    return _lib.CongestionParams(size, A, FAKE if demand else None, noise_mode, 0, keep_threshold, 7, 0, None, None)


def call(lib, A=3, size=3, demand=True, noise_mode=2, keep_threshold=1 << 31, pol_agents=None, hidden=16,
         n_actions=5, null_weight=False, n_steps=4, g_mode=0, null=(), odd=(), stats=False, stats_scratch=False,
         has_params=True, policy=True, accounting=True, n_envs=16, ld=16):
    """One call with every argument valid unless a keyword says otherwise; `null` / `odd` name pointer arguments to
    pass as NULL / misaligned."""
    from safe_multiagent_rl_b200 import _lib
    p = params(A, size, demand, noise_mode, keep_threshold)
    pol = _lib.DiscretePolicyParams(A if pol_agents is None else pol_agents, hidden, n_actions, 0,
                                    None if null_weight else FAKE, FAKE, FAKE, FAKE, 1, 0, None)
    acc = _lib.Accounting(0.9, n_steps, g_mode, None)
    names = ["start_x", "start_y", "lambdas", "obs_rec", "actions", "logp", "final_x", "final_y", "R", "modR", "C",
             "G", "g_scratch"]
    ptrs = {k: (None if k in null else ODD if k in odd else FAKE) for k in names}
    return lib.smarl_congestion_policy_rollout(
        C.byref(p) if has_params else None, C.byref(pol) if policy else None, C.byref(acc) if accounting else None,
        *[ptrs[k] for k in names], FAKE if stats else None, FAKE if stats_scratch else None, n_envs, ld, None)


def expect(lib, rc_want, needle, **kw):
    rc = call(lib, **kw)
    assert rc == rc_want and needle in lib.smarl_last_error(), (kw, rc, lib.smarl_last_error())


def test_agent_counts(lib):
    expect(lib, -1, b"n_agents=0 outside 1..32", A=0)
    expect(lib, -1, b"n_agents=33 outside 1..32", A=33)
    for A in (9, 32):
        expect(lib, -3, b"runs one thread per four envs: n_agents=%d above 8" % A, A=A)


def test_noise_modes(lib):
    expect(lib, -3, b"noise_mode 1 replays recorded moves", noise_mode=1)
    expect(lib, -1, b"bad noise_mode 3", noise_mode=3)
    expect(lib, -1, b"bad noise_mode -1", noise_mode=-1)
    expect(lib, -1, b"keep_threshold must be <= 2^32", keep_threshold=(1 << 32) + 1)


def test_policy_shape(lib):
    expect(lib, -1, b"policy has 2 agents, the env 3", pol_agents=2)
    shape = b"only the reference's DiscretePolicy shape (hidden 16, 5 actions) is built"
    expect(lib, -1, shape + b" (got 8, 5)", hidden=8)
    expect(lib, -1, shape + b" (got 16, 9)", n_actions=9)
    expect(lib, -1, b"null pointer", null_weight=True)


def test_accounting(lib):
    expect(lib, -1, b"n_steps=0 outside 1..65536", n_steps=0)
    expect(lib, -1, b"n_steps=65537 outside 1..65536", n_steps=65537)
    expect(lib, -1, b"bad g_mode -1", g_mode=-1)
    expect(lib, -1, b"bad g_mode 3", g_mode=3)
    expect(lib, -1, b"needs G", g_mode=2, null=("G",))
    expect(lib, -1, b"g_mode 1 needs g_scratch", g_mode=1, null=("g_scratch",))
    expect(lib, -1, b"stats and stats_scratch go together", stats=True)
    assert call(lib, accounting=False) == -1 and b"params is NULL" in lib.smarl_last_error()


def test_pointers(lib):
    assert call(lib, has_params=False) == -1 and b"params is NULL" in lib.smarl_last_error()
    assert call(lib, policy=False) == -1 and b"params is NULL" in lib.smarl_last_error()
    for name in ("start_x", "start_y", "R", "modR", "C"):
        expect(lib, -1, b"null required pointer", null=(name,))
    for name in ("start_x", "start_y", "obs_rec", "actions", "logp", "final_x", "final_y", "R", "modR", "C", "G",
                 "g_scratch"):
        expect(lib, -1, b"pointers must be 16-byte aligned", odd=(name,))
    expect(lib, -1, b"multiple of 16", n_envs=10, ld=10)
    expect(lib, -1, b"A*ld = 4294967296 exceeds 32-bit element offsets", A=8, n_envs=1 << 29, ld=1 << 29)


def test_env_params(lib):
    expect(lib, -1, b"size=0 outside 1..254", size=0)
    expect(lib, -1, b"size=255 outside 1..254", size=255)
    expect(lib, -1, b"demand table is NULL", demand=False)


def test_open_loop_entry_points_keep_their_checks(lib):
    """smarl_congestion_step / smarl_congestion_rollout share check_congestion: same codes and messages as before."""
    def step(**kw):
        p = params(**kw)
        return lib.smarl_congestion_step(C.byref(p), FAKE, FAKE, FAKE, FAKE, None, FAKE, FAKE, None, None, None, 0, 16,
                                         16, None)

    def rollout(**kw):
        from safe_multiagent_rl_b200 import _lib
        p = params(**kw)
        acc = _lib.Accounting(0.9, 4, 0, None)
        return lib.smarl_congestion_rollout(C.byref(p), C.byref(acc), FAKE, FAKE, FAKE, FAKE, None, None, None, FAKE,
                                            FAKE, FAKE, None, None, None, None, 16, 16, None)
    for f in (step, rollout):
        assert f(size=0) == -1 and b"size=0 outside 1..254" in lib.smarl_last_error()
        assert f(demand=False) == -1 and b"demand table is NULL" in lib.smarl_last_error()
        assert f(noise_mode=3) == -1 and b"bad noise_mode 3" in lib.smarl_last_error()
        assert f(keep_threshold=(1 << 32) + 1) == -1 and b"keep_threshold must be <= 2^32" in lib.smarl_last_error()
    assert lib.smarl_congestion_step(None, FAKE, FAKE, FAKE, FAKE, None, FAKE, FAKE, None, None, None, 0, 16, 16,
                                     None) == -1
    assert b"params is NULL" in lib.smarl_last_error()
