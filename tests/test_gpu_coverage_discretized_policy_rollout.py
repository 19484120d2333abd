"""smarl_coverage_discretized_policy_rollout / BatchedCoverageDiscretizedOnPolicy.policy_rollout: whole on-policy
CoverageDiscretized episodes (main.py:28-57 with the 9-action DiscretePolicy of agent.py:23-47 inside) in one launch,
against the closed loop it replaces (FusedDiscretizedPolicy.act + env.step per step) and against the open-loop fused
rollout of the recorded actions.  Every comparison is bit-exact unless it says otherwise."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
GUARD = 4096


def make(A, E, size=5, coarseness=6, weights=None, shuffle=False, seed=0, env_offset=0, starts=None):
    """One env and its FusedDiscretizedPolicy; calling it twice with the same arguments gives identical pairs."""
    import safe_multiagent_rl_b200 as s
    from safe_multiagent_rl_b200.policy import FusedDiscretizedPolicy
    if starts is None:
        zoom = coarseness / size
        starts = np.floor(np.random.default_rng(seed).random((E, A, 2)) * size * zoom) / zoom
    env = s.BatchedCoverageDiscretizedOnPolicy(size, A, n_envs=E, coarseness=coarseness, shuffle=shuffle,
                                               weights=weights, starts=starts, env_offset=env_offset, seed=seed + 5)
    torch.manual_seed(seed)
    pol = FusedDiscretizedPolicy(env, seed=1234 + seed)
    with torch.no_grad():
        pol.fc2.weight.mul_(4.0)
    return env, pol


def closed_loop(env, pol, T, lam, **finish):
    """reset + T x (act, step), recording what the policy saw and sampled; then the returns kernel."""
    E = env.n_envs
    buf = env.new_rollout_buffer(T)
    obs, act, logp = [], [], []
    env.reset()
    for t in range(T):
        obs.append(env.obs[:, :E].clone())
        pol.act(t=t)
        act.append(env.action_buffer[:, :E].clone())
        logp.append(pol.logp[:, :E].clone())
        env.step(env.action_buffer, lambdas=lam, out=(buf, t), agent_major=True)
    return torch.stack(obs), torch.stack(act), torch.stack(logp), buf.finish(finish.get("gamma", 0.99),
                                                                             finish.get("thresholds"), 0)


def assert_close_rel(got, want, rel=1e-5):
    got, want = got.double(), want.double()
    assert bool(((got - want).abs() <= rel * want.abs().clamp_min(1e-6)).all()), float((got - want).abs().max())


CASES = [  # A, E, T, (size, coarseness), weights, shuffle, env_offset
    (1, 1, 1, (5, 6), None, False, 0),
    (2, 37, 50, (32, 20), None, False, 0),
    (3, 50, 50, (5, 6), [1.0, 2.0, 3.0], False, 0),         # the paper's shape
    (3, 65536, 50, (5, 6), [1.0, 2.0, 3.0], False, 0),
    (4, 4099, 300, (127, 200), None, True, 0),
    (5, 37, 300, (5, 6), [0.5, 1.5, 1.0, 2.0, 1.0], True, 0),
    (6, 4099, 50, (32, 20), [1.0] * 6, False, 3 * 2 ** 32 + 17),
    (7, 1, 50, (127, 200), None, True, 2 ** 33),
    (8, 4099, 50, (5, 6), [2.0, 1.0] * 4, True, 0),
    (8, 65536, 1, (32, 20), None, False, 0),
]


@pytest.mark.parametrize("A,E,T,sc,weights,shuffle,env_offset", CASES)
def test_matches_the_closed_loop(A, E, T, sc, weights, shuffle, env_offset):
    kw = dict(size=sc[0], coarseness=sc[1], weights=weights, shuffle=shuffle, env_offset=env_offset, seed=A + E + T)
    env_c, pol_c = make(A, E, **kw)
    env_p, pol_p = make(A, E, **kw)
    lam = torch.full((A,), 0.1, dtype=torch.float64, device="cuda")
    thr = [2.0] * A
    obs, act, logp, ref = closed_loop(env_c, pol_c, T, lam, thresholds=thr)
    out = env_p.policy_rollout(pol_p, T, lambdas=lam, thresholds=thr)
    assert torch.equal(out["obs_"][:, :, :E], obs)
    assert torch.equal(out["actions_"][:, :, :E], act)
    assert torch.equal(out["logp_"][:, :, :E], logp)
    assert torch.equal(out["obs"], obs.permute(0, 2, 1))
    assert torch.equal(out["actions"], act)
    assert torch.equal(env_p.pos_x[:, :E], env_c.pos_x[:, :E]) and torch.equal(env_p.pos_y[:, :E], env_c.pos_y[:, :E])
    # against the closed loop's returns kernel, which sums the f32-rounded rewards
    for k in ("R", "modR"):
        assert_close_rel(out[k], ref[k])
    assert torch.equal(out["C"], ref["C"])
    assert_close_rel(out["stats"].vec, ref["stats"].vec)


@pytest.mark.parametrize("g_mode", [0, 1, 2])
@pytest.mark.parametrize("with_extras", [False, True])
def test_accounting_matches_the_open_loop_rollout(g_mode, with_extras):
    """The recorded actions, replayed by smarl_coverage_float_rollout from the same starts: the same products; and
    the same again with the records switched off on the reused dict."""
    A, E, T = 4, 1001, 40
    w = [1.0, 2.0, 0.5, 3.0] if with_extras else None
    env_p, pol = make(A, E, size=32, coarseness=20, weights=w)
    env_r, _ = make(A, E, size=32, coarseness=20, weights=w)
    lam = torch.tensor([0.3, 0.1, 0.2, 0.05], dtype=torch.float64, device="cuda") if with_extras else None
    thr = [20.0, 25.0, 30.0, 35.0] if with_extras else None
    out = env_p.policy_rollout(pol, T, lambdas=lam, gamma=0.97, thresholds=thr, g_mode=g_mode)
    got = {k: v.clone() for k, v in out.items() if isinstance(v, torch.Tensor)}
    final = [t.clone() for t in (env_p.pos_x, env_p.pos_y)]
    ref = env_r.rollout(out["actions_"], lambdas=lam, gamma=0.97, thresholds=thr, g_mode=g_mode)
    keys = ["R", "modR", "C", "stats_vec"] + (["G"] if g_mode else [])
    for k in keys:
        assert torch.equal(got[k], ref[k]), k
    for a, b in zip(final, (env_r.pos_x, env_r.pos_y)):
        assert torch.equal(a[:, :E], b[:, :E])
    lean = env_p.policy_rollout(pol, T, lambdas=lam, gamma=0.97, thresholds=thr, g_mode=g_mode, record=False, out=out)
    assert not any(k in lean for k in ("obs", "actions", "logp", "obs_", "actions_", "logp_"))   # no stale records
    for k in keys:
        assert torch.equal(lean[k], got[k]), k
    for a, b in zip(final, (env_p.pos_x, env_p.pos_y)):
        assert torch.equal(a[:, :E], b[:, :E])


def test_stays_in_bounds():
    """Every buffer carved out of a sentinel-filled allocation, the records sentinel-filled too: nothing outside
    the declared rows x [0, n_envs) is written."""
    from safe_multiagent_rl_b200 import _lib
    lib = _lib.load()
    A, E, T, size, coarseness = 3, 37, 5, 6, 12
    zoom = coarseness / size
    ld = 48
    S = 2 * A
    bufs = []
    f32, f64, u8 = torch.float32, torch.float64, torch.uint8

    def make_buf(rows, dtype, fill):
        item = torch.empty((), dtype=dtype).element_size()
        raw = torch.full((rows * ld * item + 2 * GUARD,), 0xA5, dtype=torch.uint8, device="cuda")
        view = raw[GUARD:GUARD + rows * ld * item].view(dtype).view(rows, ld)
        view.copy_(fill)
        bufs.append(raw)
        return view
    g = torch.Generator(device="cuda")
    g.manual_seed(3)
    sx = make_buf(A, f64, torch.floor(torch.rand(A, ld, generator=g, device="cuda", dtype=f64) * coarseness) / zoom)
    sy = make_buf(A, f64, torch.floor(torch.rand(A, ld, generator=g, device="cuda", dtype=f64) * coarseness) / zoom)
    w1 = make_buf(A * S, f32, torch.randn(A * S, ld, generator=g, device="cuda") * 0.3)   # >= [A][S][16]
    b1 = make_buf(1, f32, torch.randn(1, ld, generator=g, device="cuda"))                # >= [A][16], [A][9]
    w2 = make_buf(A * 4, f32, torch.randn(A * 4, ld, generator=g, device="cuda"))        # >= [A][16][9]
    wts = make_buf(1, f32, torch.full((1, ld), 1.5, device="cuda"))
    lam = make_buf(1, f64, torch.full((1, ld), 0.5, device="cuda", dtype=f64))
    thr = make_buf(1, f64, torch.full((1, ld), 1.0, device="cuda", dtype=f64))
    sentinel = 12345.0
    obs = make_buf(T * S, f32, sentinel)
    act = make_buf(T * A, u8, 200)
    logp = make_buf(T * A, f32, sentinel)
    fx, fy = make_buf(A, f64, sentinel), make_buf(A, f64, sentinel)
    R, M, Cs = make_buf(A, f32, sentinel), make_buf(A, f32, sentinel), make_buf(A, f32, sentinel)
    G, gs = make_buf(T * A, f32, sentinel), make_buf(2 * T, f32, sentinel)
    stats = make_buf(1, f64, 0.0)
    scratch = make_buf(max(1, lib.smarl_stats_scratch_len(A, A, E) // ld + 1), f64, 0.0)
    P = _lib.ptr
    pol = _lib.DiscretePolicyParams(A, 16, 9, 0, P(w1), P(b1), P(w2), P(b1), 77, 0, None)
    table = np.array([1, np.sqrt(2)]) * (size / coarseness)
    kp = _lib.CoverageFloatParams(size, A, 1, 0, size / np.sqrt(A), 0.0, zoom, size * zoom, float(table[0]),
                                  float(table[1]), P(wts))
    acc = _lib.Accounting(0.9, T, 1, P(thr))
    _lib.check(lib.smarl_coverage_discretized_policy_rollout(
        C.byref(kp), C.byref(pol), C.byref(acc), P(sx), P(sy), P(lam), P(obs), P(act), P(logp), P(fx), P(fy), P(R),
        P(M), P(Cs), P(G), P(gs), P(stats), P(scratch), E, ld, torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    for i, raw in enumerate(bufs):
        assert bool((raw[:GUARD] == 0xA5).all()) and bool((raw[-GUARD:] == 0xA5).all()), f"buffer {i} overrun"
    for name, b in dict(obs=obs, logp=logp, fx=fx, fy=fy, R=R, M=M, C=Cs, G=G, gs=gs).items():
        assert bool((b[:, E:] == sentinel).all()), name
        assert not bool((b[:, :E] == sentinel).any()), name
    assert bool((act[:, E:] == 200).all()) and bool((act[:, :E] < 9).all())
    assert float(stats[0, 4 * A]) == E


def test_null_stats_and_records_through_the_abi():
    """stats / stats_scratch and the three records NULL: the episode products are those of the full call."""
    from safe_multiagent_rl_b200 import _lib
    A, E, T = 3, 300, 25
    env, pol = make(A, E, weights=[1.0, 2.0, 3.0])
    lam = torch.tensor([0.2, 0.1, 0.3], dtype=torch.float64, device="cuda")
    want = {k: v.clone() for k, v in env.policy_rollout(pol, T, lambdas=lam, gamma=0.95, g_mode=1).items()
            if isinstance(v, torch.Tensor)}
    P = _lib.ptr
    f32 = torch.float32
    R, M, Cs, G = env._alloc(A, f32), env._alloc(A, f32), env._alloc(A, f32), env._alloc(A, f32, (T,))
    gs = env._alloc(1, f32, (2 * T,))
    fx, fy = torch.empty_like(env.pos_x), torch.empty_like(env.pos_y)
    acc = _lib.Accounting(0.95, T, 1, None)
    pp = pol.c_params(env)
    _lib.check(env.lib.smarl_coverage_discretized_policy_rollout(
        C.byref(env._params), C.byref(pp), C.byref(acc), P(env.start_x), P(env.start_y), P(lam), None, None, None,
        P(fx), P(fy), P(R), P(M), P(Cs), P(G), P(gs), None, None, E, env.ld, _lib.stream_ptr()))
    torch.cuda.synchronize()
    assert torch.equal(R[:, :E].t(), want["R"]) and torch.equal(M[:, :E].t(), want["modR"])
    assert torch.equal(Cs[:, :E].t(), want["C"])
    assert torch.equal(G[:, :, :E].permute(0, 2, 1), want["G"])
    assert torch.equal(fx[:, :E], env.pos_x[:, :E]) and torch.equal(fy[:, :E], env.pos_y[:, :E])


def test_shards_reproduce_the_full_batch():
    A, E, T = 3, 400, 30
    starts = np.floor(np.random.default_rng(9).random((E, A, 2)) * 6) / 1.2
    env, pol = make(A, E, starts=starts)
    full = {k: v.clone() for k, v in env.policy_rollout(pol, T, g_mode=1).items() if isinstance(v, torch.Tensor)}
    h = E // 2
    for lo, hi in ((0, h), (h, E)):
        sub, sub_pol = make(A, hi - lo, starts=starts[lo:hi], env_offset=lo)
        sub_pol.load_state_dict(pol.state_dict())
        sub_pol.seed = pol.seed
        part = sub.policy_rollout(sub_pol, T, g_mode=1)
        assert torch.equal(part["obs"], full["obs"][:, lo:hi])
        assert torch.equal(part["actions"], full["actions"][..., lo:hi])
        assert torch.equal(part["logp"], full["logp"][..., lo:hi])
        assert torch.equal(part["G"], full["G"][:, lo:hi]), "G"
        for k in ("R", "modR", "C"):
            assert torch.equal(part[k], full[k][lo:hi]), k
        assert torch.equal(sub.pos_x[:, :hi - lo], env.pos_x[:, lo:hi])


def test_cuda_graph_replay_and_episodes():
    A, E, T = 3, 1000, 20
    env, pol = make(A, E)
    lam = torch.full((A,), 0.1, dtype=torch.float64, device="cuda")
    thr = torch.full((A,), 5.0, dtype=torch.float64, device="cuda")
    out = env.policy_rollout(pol, T, lambdas=lam, thresholds=thr, g_mode=1)
    eager = {k: v.clone() for k, v in out.items() if isinstance(v, torch.Tensor)}
    ptrs = {k: v.data_ptr() for k, v in out.items() if isinstance(v, torch.Tensor)}
    out = env.policy_rollout(pol, T, lambdas=lam, thresholds=thr, g_mode=1, out=out)
    assert all(out[k].data_ptr() == p for k, p in ptrs.items())      # reused, nothing allocated
    for k in eager:
        out[k].zero_()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        env.policy_rollout(pol, T, lambdas=lam, thresholds=thr, g_mode=1, out=out)
    g.replay()
    torch.cuda.synchronize()
    for k, v in eager.items():
        assert torch.equal(out[k], v), k
    pol.next_episode()
    g.replay()
    torch.cuda.synchronize()
    assert not torch.equal(out["actions"], eager["actions"])
    assert torch.equal(out["obs"][0], eager["obs"][0])          # same starts, other samples


def test_rejected_inputs():
    import safe_multiagent_rl_b200 as s
    from safe_multiagent_rl_b200.policy import BatchedDiscretePolicy, FusedDiscretizedPolicy
    E, T = 16, 4
    env = s.BatchedCoverageDiscretizedOnPolicy(5, 3, n_envs=E, coarseness=6)
    with pytest.raises(NotImplementedError, match="DiscretePolicy: pass a FusedDiscretizedPolicy"):
        env.policy_rollout(BatchedDiscretePolicy(env), T)
    env9 = s.BatchedCoverageDiscretizedOnPolicy(5, 9, n_envs=E, coarseness=6)
    with pytest.raises(NotImplementedError, match="one thread per env"):
        env9.policy_rollout(FusedDiscretizedPolicy(env9), T)
    # a policy of another agent count: rejected before the start draw or any launch
    env_s = s.BatchedCoverageDiscretizedOnPolicy(5, 3, n_envs=E, coarseness=6, shuffle=True)
    other = FusedDiscretizedPolicy(s.BatchedCoverageDiscretizedOnPolicy(5, 2, n_envs=E, coarseness=6))
    episode, pos = env_s._episode, env_s.pos_x.clone()
    with pytest.raises(ValueError):
        env_s.policy_rollout(other, T)
    torch.cuda.synchronize()
    assert env_s._episode == episode and torch.equal(env_s.pos_x, pos)
    assert issubclass(s.BatchedCoverageDiscretizedOnPolicy, s.BatchedCoverageDiscretized)
    assert not hasattr(s.BatchedCoverageDiscretized(5, 3, n_envs=E), "policy_rollout")


@pytest.mark.parametrize("size,coarseness", [(5, 6), (32, 20)])
def test_log_prob_of_the_records_matches_the_learner_side(size, coarseness):
    """policy.log_prob on the recorded observations and actions (the PyTorch path a learner differentiates) against the
    kernel's log-probabilities: within 1e-5 on the paper's (5, 6); on (32, 20) the inputs reach 32 and the f32 rounding
    of the log-softmax grows with |log p|, so the bound there is 1e-5 (1 + |log p|)."""
    A, E, T = 5, 3000, 12
    env, pol = make(A, E, size=size, coarseness=coarseness, shuffle=True)
    out = env.policy_rollout(pol, T)
    for t in (0, 5, T - 1):
        with torch.no_grad():
            want = pol.log_prob(out["obs"][t], out["actions"][t].long())
        bound = 1e-5 if size == 5 else 1e-5 * (1.0 + want.abs())
        assert bool(((out["logp"][t] - want).abs() <= bound).all()), float((out["logp"][t] - want).abs().max())
