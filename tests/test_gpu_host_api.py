"""The host-buffer C-ABI entry points (numpy arrays in / out, chunked 2-stream pipeline inside)
against the oracle, for all three envs, with more envs than one chunk so the pipeline is exercised."""
import numpy as np
import pytest

from oracle import numpy_oracle as no
from oracle import philox

pytestmark = pytest.mark.gpu


def close(got, want, scale, rtol=1e-5):
    np.testing.assert_allclose(np.asarray(got, np.float64), want, rtol=rtol, atol=rtol * scale)


@pytest.mark.parametrize("size,A,E,T", [(7, 4, 150_001, 6),      # 3 chunks of 65536, ragged tail
                                         (9, 16, 70_003, 3),      # the bench's agent count
                                         (5, 3, 77, 5)])          # less than one transpose tile
def test_host_coverage_rollout_multi_chunk(size, A, E, T):
    """Default wrapper path = smarl_host_coverage_rollout_envmajor (env-major arrays as they are, layout change
    on the device); packed4 = the agent-major entry point.  Both against the oracle / each other."""
    from safe_multiagent_rl_b200.host import HostRollout
    gamma = 0.99
    rng = np.random.default_rng(0)
    starts = rng.integers(0, size, (E, A, 2))
    actions = rng.integers(0, 5, (T, E, A))
    w, lam, thr = [1.0 + (i % 3) for i in range(A)], np.linspace(0.1, 0.4, A), [3.0] * A
    lut = no.coverage_penalty_lut(size, no.coverage_fieldview(size, A))
    pos = starts.copy()

    def step_fn(t):
        nonlocal pos
        pos, r, c, _ = no.coverage_discrete_step(pos, actions[t], size, lut, w)
        return r, c
    want = no.rollout(step_fn, T, gamma, lam)
    h = HostRollout("coverage", A, T, E)
    out = h.coverage(size, starts, actions, weights=w, lambdas=lam, gamma=gamma, thresholds=thr)
    scale = np.abs(want["modR"]).max()
    assert np.array_equal(out["C"], want["C"])
    close(out["R"], want["R"], scale); close(out["modR"], want["modR"], scale)
    st = out["stats"]
    assert np.array_equal(st[:A], want["C"].sum(0)) and st[-1] == E
    assert np.array_equal(st[A:2 * A], (want["C"] > 3.0).sum(0))
    close(st[2 * A:3 * A], want["R"].sum(0), scale * E)
    packed = h.coverage(size, starts, actions, weights=w, lambdas=lam, gamma=gamma, thresholds=thr, packed4=True)
    for k in ("R", "modR", "C"):
        assert np.array_equal(packed[k], out[k]), k                     # 4-bit packed actions: identical products
    assert np.array_equal(packed["stats"], st)
    h.close()


def test_host_congestion_rollout_multi_chunk():
    from safe_multiagent_rl_b200.host import HostRollout
    size, A, E, T, gamma, noise, seed, off = 6, 5, 70_000, 8, 0.9, 0.2, 31, 12345
    rng = np.random.default_rng(1)
    demand = rng.random((size + 1, size + 1)) * 8 + 2
    starts = rng.integers(0, size, (E, A, 2)); starts[:, 0] = 0
    actions = rng.integers(0, 5, (T, E, A))
    pos = starts.copy()
    ids = np.arange(off, off + E)

    def step_fn(t):
        nonlocal pos
        u1, u2 = philox.congestion_uniforms(seed, ids, t, A)
        mv = no.congestion_noise_moves(actions[t], u1, u2, noise)
        pos, r, c, _, _ = no.congestion_step(pos, actions[t], mv, size, demand)
        return r.astype(np.float32).astype(np.float64), c
    want = no.rollout(step_fn, T, gamma, [0.4])
    h = HostRollout("congestion", A, T, E)
    out = h.congestion(size, starts, actions, demand, noise=noise, seed=seed, env_offset=off, lambdas=[0.4], gamma=gamma,
                       thresholds=[2.0])
    scale = np.abs(want["modR"]).max()
    assert np.array_equal(out["C"], want["C"])                 # same Philox stream across chunk boundaries
    close(out["R"], want["R"], scale); close(out["modR"], want["modR"], scale)
    assert out["stats"][0] == want["C"].sum() and out["stats"][-1] == E
    h.close()


def test_host_collision_rollout_multi_chunk():
    from safe_multiagent_rl_b200.host import HostRollout
    size, A, L, E, T, gamma = 5, 3, 2, 66_000, 10, 0.99
    rng = np.random.default_rng(2)
    starts, lm = rng.random((E, A, 2)) * size, rng.random((E, L, 2)) * size
    actions = rng.normal(0, 0.5, (T, E, A, 2)).astype(np.float32)
    q = E // 4
    actions[:, :q] = ((lm[:q, :1] - starts[:q]) / 3).astype(np.float32)[None]
    pos, done = starts.copy(), np.zeros((E, A), bool)
    n_active = np.zeros(E, np.int64)

    def step_fn(t):
        nonlocal pos, done, n_active
        pos, r, c, done, active = no.collision_step(pos, done, actions[t].astype(np.float64), lm, size)
        n_active += active
        return r.astype(np.float32).astype(np.float64), c
    want = no.rollout(step_fn, T, gamma, [0.5])
    h = HostRollout("collision", A, T, E, n_landmarks=L)
    out = h.collision(size, starts, lm, actions, lambdas=[0.5], gamma=gamma, thresholds=[1.0])
    scale = np.abs(want["modR"]).max()
    assert np.array_equal(out["C"], want["C"].astype(np.int64)) and np.array_equal(out["n_active"], n_active)
    close(out["R"], want["R"], scale); close(out["modR"], want["modR"], scale)
    assert (n_active < T).any()
    h.close()


def test_host_agent_major_entries_equal_env_major():
    """The padded agent-major entry points (what bench.py's e2e binds) and the env-major ones the numpy wrapper
    uses must produce identical arrays, for Congestion (Philox noise and recorded moves), Collision and Coverage
    (one byte per action and base-5 packed)."""
    import ctypes as C
    from safe_multiagent_rl_b200 import _lib
    from safe_multiagent_rl_b200.envs.congestion import keep_threshold
    from safe_multiagent_rl_b200.envs.coverage import penalty_table
    from safe_multiagent_rl_b200.host import HostRollout, _am, _p
    rng = np.random.default_rng(5)
    # ---- Congestion
    size, A, E, T, gamma, noise, seed, off = 7, 6, 66_001, 5, 0.95, 0.3, 9, 77
    demand = rng.random((size + 1, size + 1)) * 8 + 2
    starts = rng.integers(0, size, (E, A, 2)); starts[:, 0] = 0
    actions = rng.integers(0, 5, (T, E, A))
    moves = rng.integers(0, 5, (T, E, A))
    h = HostRollout("congestion", A, T, E)
    ld = h.ld
    for mv in (None, moves):
        em = h.congestion(size, starts, actions, demand, noise=noise, seed=seed, env_offset=off, moves=mv, lambdas=[0.4],
                          gamma=gamma, thresholds=[2.0])
        sx, sy = _am(starts[:, :, 0], ld, np.uint8), _am(starts[:, :, 1], ld, np.uint8)
        act, mva = _am(actions, ld, np.uint8), (None if mv is None else _am(mv, ld, np.uint8))
        R, M = np.zeros((A, ld), np.float32), np.zeros((A, ld), np.float32)
        Cs, st = np.zeros((1, ld), np.int32), np.zeros(h.lib.smarl_stats_len(A, 1))
        dem, lam, thr = np.ascontiguousarray(demand), np.array([0.4]), np.array([2.0])
        p = _lib.CongestionParams(size, A, _p(dem), 1 if mv is not None else 2, 0, keep_threshold(noise), seed, off, None, None)
        acc = _lib.Accounting(gamma, T, 0, _p(thr))
        _lib.check(h.lib.smarl_host_congestion_rollout(h._sess, C.byref(p), C.byref(acc), _p(sx), _p(sy), _p(act), _p(mva),
                                                       _p(lam), _p(R), _p(M), _p(Cs), _p(st)))
        assert np.array_equal(R[:, :E].T, em["R"]) and np.array_equal(M[:, :E].T, em["modR"])
        assert np.array_equal(Cs[:, :E].T, em["C"]) and np.array_equal(st, em["stats"])
    h.close()
    # ---- Collision (A = 24: the f64 transpose tile has to shrink to fit shared memory)
    size, A, L, E, T = 6, 24, 2, 65_600, 4
    starts, lm = rng.random((E, A, 2)) * size, rng.random((E, L, 2)) * size
    actions = rng.normal(0, 0.5, (T, E, A, 2)).astype(np.float32)
    h = HostRollout("collision", A, T, E, n_landmarks=L)
    ld = h.ld
    em = h.collision(size, starts, lm, actions, lambdas=[0.5], gamma=0.99, thresholds=[1.0])
    sx, sy = _am(starts[:, :, 0], ld, np.float64), _am(starts[:, :, 1], ld, np.float64)
    lma = _am(lm.reshape(E, 2 * L), ld, np.float64)
    act = _am(actions.reshape(T, E, 2 * A), ld, np.float32)
    R, M = np.zeros((A, ld), np.float32), np.zeros((A, ld), np.float32)
    Cs, na, st = np.zeros((1, ld), np.int32), np.zeros((1, ld), np.int32), np.zeros(h.lib.smarl_stats_len(A, 1))
    lam, thr = np.array([0.5]), np.array([1.0])
    p = _lib.CollisionParams(size, A, L, 0, 0.25, 0, 0)
    acc = _lib.Accounting(0.99, T, 0, _p(thr))
    _lib.check(h.lib.smarl_host_collision_rollout(h._sess, C.byref(p), C.byref(acc), _p(sx), _p(sy), _p(lma), _p(act), _p(lam),
                                                  _p(R), _p(M), _p(Cs), _p(na), _p(st)))
    assert np.array_equal(R[:, :E].T, em["R"]) and np.array_equal(M[:, :E].T, em["modR"])
    assert np.array_equal(Cs[:, :E].T, em["C"]) and np.array_equal(na[0, :E], em["n_active"])
    assert np.array_equal(st, em["stats"])
    h.close()
    # ---- Coverage (3 chunks, ragged tail); base-5 packing as bench.py does it: rows padded to 3 * pitch5
    size, A, E, T, gamma = 7, 4, 150_001, 6, 0.99
    rng = np.random.default_rng(6)
    starts = rng.integers(0, size, (E, A, 2))
    actions = rng.integers(0, 5, (T, E, A))
    w, lam, thr = np.array([1.0, 2.0, 3.0, 1.5], np.float32), np.linspace(0.1, 0.4, A), np.array([3.0] * A)
    h = HostRollout("coverage", A, T, E)
    ld, pitch5 = h.ld, int(h.lib.smarl_host_session_pitch5(h._sess))
    em = h.coverage(size, starts, actions, weights=w, lambdas=lam, gamma=gamma, thresholds=thr)
    lut = np.ascontiguousarray(penalty_table(size, A)[1], dtype=np.float32)
    p = _lib.CoverageParams(size, A, len(lut), 0, _p(lut), _p(w))
    acc = _lib.Accounting(gamma, T, 0, _p(thr))
    sx, sy = _am(starts[:, :, 0], ld, np.uint8), _am(starts[:, :, 1], ld, np.uint8)
    act = _am(actions, ld, np.uint8)                                                   # [T, A, ld]
    pad = np.zeros((T, A, 3 * pitch5), np.uint8)
    pad[:, :, :ld] = act
    act5 = np.ascontiguousarray(pad[..., 0::3] + 5 * pad[..., 1::3] + 25 * pad[..., 2::3])   # [T, A, pitch5]
    for fn, a in ((h.lib.smarl_host_coverage_rollout, act), (h.lib.smarl_host_coverage_rollout_packed5, act5)):
        R, M = np.zeros((A, ld), np.float32), np.zeros((A, ld), np.float32)
        Cs, st = np.zeros((A, ld), np.int32), np.zeros(h.lib.smarl_stats_len(A, A))
        _lib.check(fn(h._sess, C.byref(p), C.byref(acc), _p(sx), _p(sy), _p(a), _p(lam), _p(R), _p(M), _p(Cs), _p(st)))
        assert np.array_equal(R[:, :E].T, em["R"]) and np.array_equal(M[:, :E].T, em["modR"])
        assert np.array_equal(Cs[:, :E].T, em["C"]) and np.array_equal(st, em["stats"])
    h.close()


def test_host_errors_leave_the_session_usable():
    """Parameters that only the device entry point checks (Coverage size, every Collision field) fail with the
    parameter named, an oversized Coverage table fails as unsupported, and after each failure the same session gives
    what a fresh session gives."""
    import ctypes as C
    from safe_multiagent_rl_b200 import _lib
    from safe_multiagent_rl_b200.envs.coverage import MAX_LUT, penalty_table
    from safe_multiagent_rl_b200.host import HostRollout, _p
    rng = np.random.default_rng(8)
    # ---- Coverage
    size, A, E, T, gamma = 6, 3, 140_000, 4, 0.99
    starts = rng.integers(0, size, (E, A, 2)).astype(np.uint8)
    actions = rng.integers(0, 5, (T, E, A)).astype(np.uint8)
    w, lam, thr = np.array([1.0, 2.0, 3.0], np.float32), np.array([0.1, 0.2, 0.3]), np.array([2.0] * A)
    kw = dict(weights=w, lambdas=lam, gamma=gamma, thresholds=thr)
    fresh = HostRollout("coverage", A, T, E)
    want = fresh.coverage(size, starts, actions, **kw)
    fresh.close()
    lut = np.ascontiguousarray(penalty_table(size, A)[1], dtype=np.float32)
    acc = _lib.Accounting(gamma, T, 0, _p(thr))
    h = HostRollout("coverage", A, T, E)
    for bad_size, table, rc, name in ((200, lut, -1, "size"), (size, np.zeros(MAX_LUT + 1, np.float32), -3, "lut_len"),
                                      (size, np.zeros(12288, np.float32), -3, "lut_len")):
        p = _lib.CoverageParams(bad_size, A, len(table), 0, _p(table), _p(w))
        R, M, Cs = np.zeros((E, A), np.float32), np.zeros((E, A), np.float32), np.zeros((E, A), np.int32)
        st = np.zeros(h.lib.smarl_stats_len(A, A))
        got = h.lib.smarl_host_coverage_rollout_envmajor(h._sess, C.byref(p), C.byref(acc), _p(starts), _p(actions),
                                                         _p(lam), _p(R), _p(M), _p(Cs), _p(st))
        assert got == rc and name in h.lib.smarl_last_error().decode(), (bad_size, len(table))
        out = h.coverage(size, starts, actions, **kw)
        for k in ("R", "modR", "C", "stats"):
            assert np.array_equal(out[k], want[k]), k
    h.close()
    # ---- Collision
    size, A, L, E, T = 5, 3, 2, 66_000, 4
    starts, lm = rng.random((E, A, 2)) * size, rng.random((E, L, 2)) * size
    actions = rng.normal(0, 0.5, (T, E, A, 2)).astype(np.float32)
    kw = dict(lambdas=[0.5], gamma=gamma, thresholds=[1.0])
    fresh = HostRollout("collision", A, T, E, n_landmarks=L)
    want = fresh.collision(size, starts, lm, actions, **kw)
    fresh.close()
    h = HostRollout("collision", A, T, E, n_landmarks=L)
    p = _lib.CollisionParams(size, A, L, 0, 0.0, 0, 0)                                  # agents_size = 0
    thr1, lam1 = np.array([1.0]), np.array([0.5])
    acc = _lib.Accounting(gamma, T, 0, _p(thr1))
    R, M = np.zeros((E, A), np.float32), np.zeros((E, A), np.float32)
    Cs, na, st = np.zeros(E, np.int32), np.zeros(E, np.int32), np.zeros(h.lib.smarl_stats_len(A, 1))
    got = h.lib.smarl_host_collision_rollout_envmajor(h._sess, C.byref(p), C.byref(acc), _p(starts), _p(lm), _p(actions),
                                                      _p(lam1), _p(R), _p(M), _p(Cs), _p(na), _p(st))
    assert got == -1 and "agents_size" in h.lib.smarl_last_error().decode()
    out = h.collision(size, starts, lm, actions, **kw)
    for k in ("R", "modR", "C", "n_active", "stats"):
        assert np.array_equal(out[k], want[k]), k
    h.close()
