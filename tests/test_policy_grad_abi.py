"""CPU checks of the argument validation of smarl_policy_grad_discrete and of smarl_policy_grad_scratch_len: every
rejected input returns -1 and its message before any CUDA work, so the pointers below are fake and never
dereferenced."""
import ctypes as C
import math

import pytest

FAKE = C.c_void_p(0x1000)
ODD = C.c_void_p(0x1008)          # 8-byte aligned, not 16
SHAPE = b"the DiscretePolicy gradient is built for hidden 16 and 5 or 9 actions"
POINTERS = ("w1", "b1", "w2", "b2", "obs_rec", "actions", "psi", "dw1", "db1", "dw2", "db2", "scratch")


@pytest.fixture(scope="module")
def lib():
    from safe_multiagent_rl_b200 import _lib, build
    build.build()
    return _lib.load()


def grad(lib, A=3, hidden=16, n_actions=5, null=(), odd=(), n_steps=50, scale=0.01, n_envs=16, ld=16, params=True,
         loss=True):
    """One call with every argument valid unless a keyword says otherwise; `null` names pointer arguments to pass as
    NULL, `odd` record pointers to pass 8- but not 16-byte aligned."""
    from safe_multiagent_rl_b200 import _lib
    ptrs = {k: (None if k in null else ODD if k in odd else FAKE) for k in POINTERS}
    p = _lib.DiscretePolicyParams(A, hidden, n_actions, 0, ptrs["w1"], ptrs["b1"], ptrs["w2"], ptrs["b2"], 1, 0, None)
    return lib.smarl_policy_grad_discrete(C.byref(p) if params else None, ptrs["obs_rec"], ptrs["actions"],
                                          ptrs["psi"], n_steps, scale, ptrs["dw1"], ptrs["db1"], ptrs["dw2"],
                                          ptrs["db2"], FAKE if loss else None, ptrs["scratch"], n_envs, ld, None)


def expect(lib, needle, **kw):
    rc = grad(lib, **kw)
    assert rc == -1 and needle in lib.smarl_last_error(), (kw, rc, lib.smarl_last_error())


def test_params_and_shape(lib):
    expect(lib, b"policy params is NULL", params=False)
    expect(lib, b"n_agents=0 outside 1..32", A=0)
    expect(lib, b"n_agents=33 outside 1..32", A=33)
    expect(lib, SHAPE + b" (got 8, 5)", hidden=8)
    for na in (4, 6, 10):
        expect(lib, SHAPE + b" (got 16, %d)" % na, n_actions=na)


def test_null_pointers(lib):
    for name in POINTERS:
        expect(lib, b"null pointer", null=(name,))


def test_steps_layout_alignment_scale(lib):
    expect(lib, b"n_steps=0 outside 1..65536", n_steps=0)
    expect(lib, b"n_steps=65537 outside 1..65536", n_steps=65537)
    expect(lib, b"multiple of 16", n_envs=10, ld=10)
    expect(lib, b"multiple of 16", n_envs=17, ld=16)
    for name in ("obs_rec", "actions", "psi"):
        expect(lib, b"records must be 16-byte aligned", odd=(name,))
    for s in (math.inf, -math.inf, math.nan):
        expect(lib, b"scale is not finite", scale=s)


def test_rejections_come_in_order(lib):
    """The first failing check names the error: a NULL weight is reported before a bad n_steps, which is reported
    before the layout, the alignment and the scale."""
    expect(lib, b"null pointer", null=("w1",), n_steps=0, n_envs=10, ld=10, scale=math.nan)
    expect(lib, b"n_steps=0", n_steps=0, n_envs=10, ld=10, scale=math.nan)
    expect(lib, b"multiple of 16", n_envs=10, ld=10, odd=("psi",), scale=math.nan)
    expect(lib, b"16-byte aligned", odd=("psi",), scale=math.nan)


def test_scratch_len(lib):
    f = lib.smarl_policy_grad_scratch_len
    for args in ((0, 5, 50, 64), (33, 5, 50, 64), (3, 6, 50, 64), (3, 5, 0, 64), (3, 5, 65537, 64), (3, 5, 50, 0)):
        assert f(*args) == -1, args
    # 64 header doubles + A chunks-per-agent x (32 A + 17 NA + 17) outputs, P = min(T ceil(E / 256), 1184 // A)
    assert f(3, 5, 1, 1) == 64 + 3 * 1 * (96 + 85 + 17)
    assert f(3, 5, 50, 50) == 64 + 3 * 50 * (96 + 85 + 17)
    assert f(3, 9, 50, 65536) == 64 + 3 * 394 * (96 + 153 + 17)
    assert f(32, 9, 50, 2 ** 20) == 64 + 32 * 37 * (1024 + 153 + 17)
    assert f(32, 9, 50, 2 ** 20) * 8 < 12e6
    assert f(1, 5, 65536, 2 ** 20) == 64 + 1184 * (32 + 85 + 17)
