"""smarl_collision_policy_rollout / BatchedCollisionAvoidance.policy_rollout: whole on-policy CollisionAvoidance
episodes (main.py:28-57 with the ContinuousPolicy of agent.py:48-76 inside) in one launch, against the closed loop it
replaces (FusedGaussianPolicy.act + env.step per step) and against the open-loop fused rollout of the recorded
actions.  Every comparison is bit-exact unless it says otherwise."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
GUARD = 4096


def make(A, E, size=6, L=1, shuffle=False, normalize=False, agents_size=0.25, seed=0, env_offset=0, starts=None,
         landmarks=None):
    """One env and its FusedGaussianPolicy; calling it twice with the same arguments gives identical pairs."""
    import safe_multiagent_rl_b200 as s
    from safe_multiagent_rl_b200.policy import FusedGaussianPolicy
    rng = np.random.default_rng(seed)
    if starts is None:
        starts = rng.random((E, A, 2)) * size
        landmarks = rng.random((E, L, 2)) * size
    env = s.BatchedCollisionAvoidance(size, A, n_envs=E, n_landmarks=L, shuffle=shuffle, agents_size=agents_size,
                                      normalize_state=normalize, starts=starts, landmarks=landmarks,
                                      env_offset=env_offset, seed=seed + 5)
    torch.manual_seed(seed)
    pol = FusedGaussianPolicy(env, seed=1234 + seed)
    with torch.no_grad():
        pol.fc2_.bias.add_(1.0)        # sigma around 1: many actions longer than 1 take the clip path
    return env, pol


def closed_loop(env, pol, T, lam):
    """reset + T x (act, step), recording what the policy saw and sampled."""
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
    return torch.stack(obs), torch.stack(act), torch.stack(logp)


CASES = [  # A, E, T, shuffle, normalize, L, size, agents_size
    (1, 1, 1, False, False, 1, 6, 0.25),
    (3, 37, 50, False, False, 1, 5, 0.25),
    (3, 65536, 50, False, False, 1, 5, 0.25),       # BASELINE configs[1]
    (5, 4099, 300, True, False, 3, 6, 0.25),
    (8, 4099, 50, True, True, 3, 8, 0.25),
    (8, 37, 300, False, True, 3, 6, 0.25),
    (5, 65536, 1, False, True, 1, 6, 0.25),
    (3, 4099, 50, True, True, 1, 3, 1.2),           # most envs end early: post-episode steps
    (8, 1, 50, True, False, 1, 4, 1.0),
    # dynamic shared memory within 48 KB but over 48 KB with the static part: needs the opt-in
    (8, 4099, 50, True, False, 17, 8, 0.25),
    (3, 37, 20, True, True, 32, 6, 0.25),
]


@pytest.mark.parametrize("A,E,T,shuffle,normalize,L,size,agents_size", CASES)
def test_matches_the_closed_loop(A, E, T, shuffle, normalize, L, size, agents_size):
    kw = dict(size=size, L=L, shuffle=shuffle, normalize=normalize, agents_size=agents_size, seed=A + E + T)
    env_c, pol_c = make(A, E, **kw)
    env_p, pol_p = make(A, E, **kw)
    lam = torch.tensor([0.1], dtype=torch.float64, device="cuda")
    obs, act, logp = closed_loop(env_c, pol_c, T, lam)
    out = env_p.policy_rollout(pol_p, T, lambdas=lam)
    assert torch.equal(out["obs_"][:, :, :E], obs)
    assert torch.equal(out["actions_"][:, :, :E], act)
    assert torch.equal(out["logp_"][:, :, :E], logp)
    assert torch.equal(out["obs"], obs.permute(0, 2, 1))
    assert torch.equal(out["actions"], act.view(T, A, 2, E).permute(0, 1, 3, 2))
    assert torch.equal(env_p.pos_x[:, :E], env_c.pos_x[:, :E]) and torch.equal(env_p.pos_y[:, :E], env_c.pos_y[:, :E])
    assert torch.equal(env_p.agent_done[:, :E], env_c.agent_done[:, :E])
    assert torch.equal(out["n_active"], env_c.episode_len[:E])
    if agents_size >= 1.0 and E > 1:
        assert (out["n_active"] < T).float().mean() > 0.5


@pytest.mark.parametrize("g_mode", [0, 1, 2])
@pytest.mark.parametrize("with_extras", [False, True])
def test_accounting_matches_the_open_loop_rollout(g_mode, with_extras):
    """The recorded actions, replayed by smarl_collision_rollout from the same starts: the same products; and the
    same again with the records switched off."""
    A, E, T = 4, 1001, 40
    env_p, pol = make(A, E, size=5, agents_size=0.6, L=2)
    env_r, _ = make(A, E, size=5, agents_size=0.6, L=2)
    lam = torch.tensor([0.3], dtype=torch.float64, device="cuda") if with_extras else None
    thr = [2.0] if with_extras else None
    out = env_p.policy_rollout(pol, T, lambdas=lam, gamma=0.97, thresholds=thr, g_mode=g_mode)
    got = {k: v.clone() for k, v in out.items() if isinstance(v, torch.Tensor)}
    final = [t.clone() for t in (env_p.pos_x, env_p.pos_y, env_p.agent_done)]
    ref = env_r.rollout(out["actions_"], lambdas=lam, gamma=0.97, thresholds=thr, g_mode=g_mode)
    keys = ["R", "modR", "C", "n_active", "stats_vec"] + (["G"] if g_mode else [])
    for k in keys:
        assert torch.equal(got[k], ref[k]), k
    for a, b in zip(final, (env_r.pos_x, env_r.pos_y, env_r.agent_done)):
        assert torch.equal(a[:, :E], b[:, :E])
    lean = env_p.policy_rollout(pol, T, lambdas=lam, gamma=0.97, thresholds=thr, g_mode=g_mode, record=False, out=out)
    assert not any(k in lean for k in ("obs", "actions", "logp", "obs_", "actions_", "logp_"))   # no stale records
    for k in keys:
        assert torch.equal(lean[k], got[k]), k


def test_stays_in_bounds():
    """Every buffer carved out of a sentinel-filled allocation, the records sentinel-filled too: nothing outside
    the declared rows x [0, n_envs) is written."""
    from safe_multiagent_rl_b200 import _lib
    lib = _lib.load()
    A, E, T, L, S_ = 3, 37, 5, 2, 6
    ld = 48
    S = 2 * A + 2 * L
    bufs = []
    f32, f64, u8, i32 = torch.float32, torch.float64, torch.uint8, torch.int32

    def make_buf(rows, dtype, fill):
        item = torch.empty((), dtype=dtype).element_size()
        raw = torch.full((rows * ld * item + 2 * GUARD,), 0xA5, dtype=torch.uint8, device="cuda")
        view = raw[GUARD:GUARD + rows * ld * item].view(dtype).view(rows, ld)
        view.copy_(fill)
        bufs.append(raw)
        return view
    g = torch.Generator(device="cuda")
    g.manual_seed(3)
    sx = make_buf(A, f64, torch.rand(A, ld, generator=g, device="cuda", dtype=f64) * S_)
    sy = make_buf(A, f64, torch.rand(A, ld, generator=g, device="cuda", dtype=f64) * S_)
    lm = make_buf(2 * L, f64, torch.rand(2 * L, ld, generator=g, device="cuda", dtype=f64) * S_)
    w1 = make_buf(A * S, f32, torch.randn(A * S, ld, generator=g, device="cuda") * 0.3)   # >= [A][S][16]
    b1 = make_buf(1, f32, torch.randn(1, ld, generator=g, device="cuda"))                # >= [A][16], [A][2]
    hw = make_buf(4, f32, torch.randn(4, ld, generator=g, device="cuda"))                # 2 x [A][16][2]
    lam = make_buf(1, f64, torch.full((1, ld), 0.5, device="cuda", dtype=f64))
    thr = make_buf(1, f64, torch.full((1, ld), 1.0, device="cuda", dtype=f64))
    sentinel = 12345.0
    obs = make_buf(T * S, f32, sentinel)
    act = make_buf(T * 2 * A, f32, sentinel)
    logp = make_buf(T * A, f32, sentinel)
    fx, fy, fd = make_buf(A, f64, sentinel), make_buf(A, f64, sentinel), make_buf(A, u8, 7)
    nact, Cs = make_buf(1, i32, -9), make_buf(1, i32, -9)
    R, M, G, gs = make_buf(A, f32, sentinel), make_buf(A, f32, sentinel), make_buf(T * A, f32, sentinel), make_buf(2 * T, f32, sentinel)
    stats = make_buf(1, f64, 0.0)
    scratch = make_buf(max(1, lib.smarl_stats_scratch_len(A, 1, E) // ld + 1), f64, 0.0)
    P = _lib.ptr
    pol = _lib.GaussianPolicyParams(A, S, 16, 2, 0, 0, P(w1), P(b1), P(hw), P(b1), P(hw[2:]), P(b1), 77, 0, None)
    kp = _lib.CollisionParams(S_, A, L, 1, 0.25, 1, 0)
    acc = _lib.Accounting(0.9, T, 1, P(thr))
    _lib.check(lib.smarl_collision_policy_rollout(C.byref(kp), C.byref(pol), C.byref(acc), P(sx), P(sy), P(lm), P(lam),
                                                  P(obs), P(act), P(logp), P(fx), P(fy), P(fd), P(nact), P(R), P(M),
                                                  P(Cs), P(G), P(gs), P(stats), P(scratch), E, ld,
                                                  torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    for i, raw in enumerate(bufs):
        assert bool((raw[:GUARD] == 0xA5).all()) and bool((raw[-GUARD:] == 0xA5).all()), f"buffer {i} overrun"
    for name, b in dict(obs=obs, act=act, logp=logp, fx=fx, fy=fy, R=R, M=M, G=G, gs=gs).items():
        assert bool((b[:, E:] == sentinel).all()), name
        assert not bool((b[:, :E] == sentinel).any()), name
    assert bool((fd[:, E:] == 7).all()) and bool((nact[:, E:] == -9).all()) and bool((Cs[:, E:] == -9).all())
    assert float(stats[0, 2 + 2 * A]) == E


def test_null_stats_and_records_through_the_abi():
    """stats / stats_scratch and the three records NULL: the episode products are those of the full call."""
    from safe_multiagent_rl_b200 import _lib
    A, E, T = 3, 300, 25
    env, pol = make(A, E, agents_size=0.5)
    lam = torch.tensor([0.2], dtype=torch.float64, device="cuda")
    want = {k: v.clone() for k, v in env.policy_rollout(pol, T, lambdas=lam, gamma=0.95, g_mode=1).items()
            if isinstance(v, torch.Tensor)}
    P = _lib.ptr
    f32 = torch.float32
    R, M, G = env._alloc(A, f32), env._alloc(A, f32), env._alloc(A, f32, (T,))
    Cs, nact, gs = env._alloc(1, torch.int32), env._alloc(1, torch.int32), env._alloc(1, f32, (2 * T,))
    fx, fy, fd = torch.empty_like(env.pos_x), torch.empty_like(env.pos_y), torch.empty_like(env.agent_done)
    acc = _lib.Accounting(0.95, T, 1, None)
    pp = pol.c_params(env)
    _lib.check(env.lib.smarl_collision_policy_rollout(
        C.byref(env._params), C.byref(pp), C.byref(acc), P(env.start_x), P(env.start_y), P(env.landmarks), P(lam),
        None, None, None, P(fx), P(fy), P(fd), P(nact), P(R), P(M), P(Cs), P(G), P(gs), None, None, E, env.ld,
        _lib.stream_ptr()))
    torch.cuda.synchronize()
    assert torch.equal(R[:, :E].t(), want["R"]) and torch.equal(M[:, :E].t(), want["modR"])
    assert torch.equal(Cs[:, :E].t(), want["C"]) and torch.equal(nact[0, :E], want["n_active"])
    assert torch.equal(G[:, :, :E].permute(0, 2, 1), want["G"])
    assert torch.equal(fx[:, :E], env.pos_x[:, :E]) and torch.equal(fd[:, :E], env.agent_done[:, :E])


def test_shards_reproduce_the_full_batch():
    A, E, T = 3, 400, 30
    rng = np.random.default_rng(9)
    starts, lms = rng.random((E, A, 2)) * 6, rng.random((E, 1, 2)) * 6
    env, pol = make(A, E, starts=starts, landmarks=lms)
    full = {k: v.clone() for k, v in env.policy_rollout(pol, T, g_mode=1).items() if isinstance(v, torch.Tensor)}
    h = E // 2
    for lo, hi in ((0, h), (h, E)):
        sub, sub_pol = make(A, hi - lo, starts=starts[lo:hi], landmarks=lms[lo:hi], env_offset=lo)
        sub_pol.load_state_dict(pol.state_dict())
        sub_pol.seed = pol.seed
        part = sub.policy_rollout(sub_pol, T, g_mode=1)
        for k in ("obs", "actions", "logp"):
            assert torch.equal(part[k], full[k][..., lo:hi, :] if k != "logp" else full[k][..., lo:hi]), k
        assert torch.equal(part["G"], full["G"][:, lo:hi]), "G"
        for k in ("R", "modR", "C", "n_active"):
            assert torch.equal(part[k], full[k][lo:hi]), k


def test_cuda_graph_replay_and_episodes():
    A, E, T = 3, 1000, 20
    env, pol = make(A, E)
    lam = torch.tensor([0.1], dtype=torch.float64, device="cuda")
    thr = torch.tensor([1.0], dtype=torch.float64, device="cuda")
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


def test_rejected_inputs_queue_no_work():
    from safe_multiagent_rl_b200 import _lib
    lib = _lib.load()
    E, ld, T = 16, 16, 4
    P = _lib.ptr
    st = torch.cuda.current_stream().cuda_stream

    def call(A, S, hidden=16, g_mode=0, n_steps=T, null_start=False, null_weight=False, null_g=False, null_gs=False,
             stats_only=False):
        big = torch.zeros(4096, ld, dtype=torch.float64, device="cuda")
        out = torch.full((4096, ld), 5.0, dtype=torch.float32, device="cuda")
        kp = _lib.CollisionParams(6, A, 1, 0, 0.25, 0, 0)
        pol = _lib.GaussianPolicyParams(A, S, hidden, 2, 0, 0, None if null_weight else P(out), P(out), P(out), P(out),
                                        P(out), P(out), 1, 0, None)
        acc = _lib.Accounting(0.9, n_steps, g_mode, None)
        rc = lib.smarl_collision_policy_rollout(C.byref(kp), C.byref(pol), C.byref(acc), None if null_start else P(big),
                                                P(big), P(big), None, P(out), P(out), P(out), P(big), P(big), P(big),
                                                P(big), P(out), P(out), P(big), None if null_g else P(out),
                                                None if null_gs else P(out), P(big) if stats_only else None, None, E, ld,
                                                st)
        torch.cuda.synchronize()
        assert bool((out == 5.0).all()) and not bool(big.any())       # nothing ran
        return rc
    assert call(9, 18) == -3
    assert call(3, 6, g_mode=3) == -1
    assert call(3, 8) == -1
    assert call(3, 6, hidden=8) == -1
    assert call(3, 6, null_start=True) == -1
    assert call(3, 6, n_steps=0) == -1
    assert call(3, 6, n_steps=65537) == -1
    assert call(3, 6, null_weight=True) == -1
    assert call(3, 6, g_mode=2, null_g=True) == -1
    assert call(3, 6, g_mode=1, null_gs=True) == -1
    assert call(3, 6, stats_only=True) == -1
    import safe_multiagent_rl_b200 as s
    from safe_multiagent_rl_b200.policy import BatchedGaussianPolicy, FusedGaussianPolicy
    env = s.BatchedCollisionAvoidance(6, 3, n_envs=E)
    with pytest.raises(NotImplementedError):
        env.policy_rollout(BatchedGaussianPolicy(env), T)
    env9 = s.BatchedCollisionAvoidance(6, 9, n_envs=E)
    with pytest.raises(NotImplementedError):
        env9.policy_rollout(FusedGaussianPolicy(env9), T)


def test_log_prob_of_the_records_matches_the_learner_side():
    """policy.log_prob on the recorded observations and actions (the PyTorch path a learner differentiates) against
    the kernel's log-probabilities, within test_gpu_policy_gauss.py's bound."""
    A, E, T = 5, 3000, 12
    env, pol = make(A, E, L=2, shuffle=True)
    out = env.policy_rollout(pol, T)
    for t in (0, 5, T - 1):
        obs, act = out["obs"][t], out["actions"][t]
        with torch.no_grad():
            h = torch.relu(pol.fc1(obs))
            mu = pol.fc2(h).double().cpu().numpy()
            var = (torch.relu(pol.fc2_(h)) + 1e-4).double().cpu().numpy()
            want = pol.log_prob(obs, act).double().cpu().numpy()
        lp = out["logp"][t].double().cpu().numpy()
        z = (act.double().cpu().numpy() - mu) / np.sqrt(var)
        tol = 2e-5 * (1.0 + np.abs(lp)) + (4e-6 * (1.0 + np.abs(mu)) * np.abs(z) / np.sqrt(var) +
                                           4e-6 * (1.0 + var) / var * 0.5 * (z ** 2 + 1.0)).sum(axis=-1)
        assert np.all(np.abs(lp - want) <= tol), np.abs(lp - want).max()
