"""smarl_congestion_policy_rollout / BatchedCongestionOnPolicy.policy_rollout: whole on-policy Congestion episodes
(main.py:28-57 with the DiscretePolicy of agent.py:23-47 inside, action noise included) in one launch, against the closed loop it
replaces (FusedDiscretePolicy.act + env.step per step, FP32-pipe policy build) and against the open-loop fused rollout
of the recorded actions with the same noise episode.  Every comparison is bit-exact unless it says otherwise."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
GUARD = 4096


def make(A, E, size=3, noise=0.1, shuffle=False, seed=0, env_offset=0, starts=None, on_policy=True):
    """One env and its FusedDiscretePolicy; calling it twice with the same arguments gives identical pairs.  Size 3 takes
    the reference's demand table, other sizes a seeded one.  ``on_policy=False`` builds the plain BatchedCongestion, which
    the closed loop and the open-loop rollout run on."""
    import safe_multiagent_rl_b200 as s
    from safe_multiagent_rl_b200.policy import FusedDiscretePolicy
    rng = np.random.default_rng(seed)
    if starts is None:
        starts = rng.integers(0, size + 1, (E, A, 2))
    demand = None if size == 3 else rng.random((size + 1, size + 1)) * 8 + 2
    cls = s.BatchedCongestionOnPolicy if on_policy else s.BatchedCongestion
    env = cls(size, A, n_envs=E, noise=noise, shuffle=shuffle, starts=starts, demand_rate=demand, env_offset=env_offset,
              seed=seed + 5)
    torch.manual_seed(seed)
    pol = FusedDiscretePolicy(env, seed=1234 + seed)
    with torch.no_grad():
        pol.fc1.weight.mul_(4.0 / size)            # inputs of order 1 at every size: no action dominates
    return env, pol


def closed_loop(env, pol, T, lam, gamma=0.9, thresholds=None):
    """reset + T x (act, step) with the FP32-pipe policy build, recording what the policy saw and sampled; then the
    returns kernel."""
    from safe_multiagent_rl_b200 import _lib
    E = env.n_envs
    buf = env.new_rollout_buffer(T)
    obs, act, logp = [], [], []
    env.reset()
    with _lib.kernel_variant(_lib.KERNEL_POLICY, 0):
        for t in range(T):
            obs.append(env.obs[:, :E].clone())
            pol.act(t=t)
            act.append(env.action_buffer[:, :E].clone())
            logp.append(pol.logp[:, :E].clone())
            env.step(env.action_buffer, lambdas=lam, out=(buf, t), agent_major=True)
    return torch.stack(obs), torch.stack(act), torch.stack(logp), buf.finish(gamma, thresholds, 0)


def assert_close_rel(got, want, rel=1e-5):
    """|got - want| <= rel * max(|want|, 1): a discounted sum of rewards of either sign can cancel to near zero."""
    got, want = got.double(), want.double()
    assert bool(((got - want).abs() <= rel * want.abs().clamp_min(1.0)).all()), float((got - want).abs().max())


def tensors(out):
    return {k: v.clone() for k, v in out.items() if isinstance(v, torch.Tensor)}


CASES = [  # A, E, T, size, noise, shuffle, env_offset
    (1, 1, 1, 3, 0.1, False, 0),
    (2, 37, 50, 10, 0.0, False, 0),
    (3, 50, 10, 3, 0.1, False, 0),                      # the paper's setup
    (3, 65536, 10, 3, 0.1, False, 0),
    (4, 4099, 300, 10, 1.0, True, 0),
    (5, 37, 100, 254, 0.1, True, 0),
    (6, 4099, 50, 10, 0.1, False, 3 * 2 ** 32 + 17),
    (7, 1, 50, 254, 0.0, True, 2 ** 33),
    (8, 4099, 50, 3, 0.1, True, 0),
    (8, 65536, 2, 10, 1.0, False, 0),
]


@pytest.mark.parametrize("A,E,T,size,noise,shuffle,env_offset", CASES)
def test_matches_the_closed_loop(A, E, T, size, noise, shuffle, env_offset):
    kw = dict(size=size, noise=noise, shuffle=shuffle, env_offset=env_offset, seed=A + E + T)
    env_c, pol_c = make(A, E, on_policy=False, **kw)
    env_p, pol_p = make(A, E, **kw)
    lam = torch.full((1,), 0.1, dtype=torch.float64, device="cuda")
    thr = [float(T) / 2]
    obs, act, logp, ref = closed_loop(env_c, pol_c, T, lam, thresholds=thr)
    out = env_p.policy_rollout(pol_p, T, lambdas=lam, gamma=0.9, thresholds=thr)
    assert torch.equal(out["obs_"][:, :, :E], obs)
    assert torch.equal(out["actions_"][:, :, :E], act)
    assert torch.equal(out["logp_"][:, :, :E], logp)
    assert torch.equal(out["obs"], obs.permute(0, 2, 1))
    assert torch.equal(out["actions"], act) and torch.equal(out["logp"], logp)
    assert torch.equal(env_p.pos_x[:, :E], env_c.pos_x[:, :E]) and torch.equal(env_p.pos_y[:, :E], env_c.pos_y[:, :E])
    for k in ("R", "modR"):
        assert_close_rel(out[k], ref[k])
    assert torch.equal(out["C"].long(), ref["C"].long())
    assert_close_rel(out["stats_vec"], ref["stats"].vec)
    if E >= 37 and T > 1:                                       # the policy moves the agents
        assert bool((act != 4).any()) and bool((act == 4).any())


@pytest.mark.parametrize("g_mode", [0, 1, 2])
@pytest.mark.parametrize("with_extras", [False, True])
def test_accounting_matches_the_open_loop_rollout(g_mode, with_extras):
    """The recorded actions, replayed by smarl_congestion_rollout from the same starts and noise episode: the same
    products; and the same again with the records switched off on the reused dict."""
    A, E, T = 4, 1001, 40
    env_p, pol = make(A, E, size=10, noise=0.2)
    env_r, _ = make(A, E, size=10, noise=0.2, on_policy=False)
    lam = torch.tensor([0.3], dtype=torch.float64, device="cuda") if with_extras else None
    thr = [12.0] if with_extras else None
    out = env_p.policy_rollout(pol, T, lambdas=lam, gamma=0.97, thresholds=thr, g_mode=g_mode)
    got = tensors(out)
    final = [t.clone() for t in (env_p.pos_x, env_p.pos_y)]
    ref = env_r.rollout(out["actions_"], lambdas=lam, gamma=0.97, thresholds=thr, g_mode=g_mode)
    keys = ["R", "modR", "C", "stats_vec"] + (["G"] if g_mode else [])
    for k in keys:
        assert torch.equal(got[k], ref[k]), k
    for a, b in zip(final, (env_r.pos_x, env_r.pos_y)):
        assert torch.equal(a[:, :E], b[:, :E])
    env_p.set_noise_episode(0)                                  # the first call's noise again
    lean = env_p.policy_rollout(pol, T, lambdas=lam, gamma=0.97, thresholds=thr, g_mode=g_mode, record=False, out=out)
    assert not any(k in lean for k in ("obs", "actions", "logp", "obs_", "actions_", "logp_"))   # no stale records
    for k in keys:
        assert torch.equal(lean[k], got[k]), k


def test_accounting_without_the_waiting_table_through_the_abi():
    """wait_reward = NULL on both sides (the waiting reward evaluated from the demand table on the device): the one
    launch and smarl_congestion_rollout fed its recorded actions give the same products."""
    from safe_multiagent_rl_b200 import _lib
    A, E, T = 5, 777, 30
    env, pol = make(A, E, size=10, noise=0.3, seed=4)
    P, f32, i32 = _lib.ptr, torch.float32, torch.int32
    lam = torch.tensor([0.2], dtype=torch.float64, device="cuda")
    thr = torch.tensor([8.0], dtype=torch.float64, device="cuda")
    st = _lib.stream_ptr()

    def products():
        return [env._alloc(A, f32), env._alloc(A, f32), env._alloc(1, i32), env._alloc(A, f32, (T,)),
                env._alloc(1, f32, (T,)), torch.empty_like(env.pos_x), torch.empty_like(env.pos_y),
                torch.zeros(env.lib.smarl_stats_len(A, 1), dtype=torch.float64, device="cuda"),
                torch.zeros(env.lib.smarl_stats_scratch_len(A, 1, E), dtype=torch.float64, device="cuda")]
    p = env._params(2)
    p.wait_reward = None
    acc = _lib.Accounting(0.9, T, 1, P(thr))
    obs, act, logp = env._alloc(2 * A, f32, (T,)), env._alloc(A, torch.uint8, (T,)), env._alloc(A, f32, (T,))
    R, M, Cs, G, gs, fx, fy, stats, scratch = got = products()
    _lib.check(env.lib.smarl_congestion_policy_rollout(
        C.byref(p), C.byref(pol.c_params(env)), C.byref(acc), P(env.start_x), P(env.start_y), P(lam), P(obs), P(act),
        P(logp), P(fx), P(fy), P(R), P(M), P(Cs), P(G), P(gs), P(stats), P(scratch), E, env.ld, st))
    R, M, Cs, G, gs, fx, fy, stats, scratch = want = products()
    _lib.check(env.lib.smarl_congestion_rollout(
        C.byref(p), C.byref(acc), P(env.start_x), P(env.start_y), P(act), None, P(lam), P(fx), P(fy), P(R), P(M),
        P(Cs), P(G), P(gs), P(stats), P(scratch), E, env.ld, st))
    torch.cuda.synchronize()
    for i in (0, 1, 2, 3, 5, 6, 7):                             # R, modR, C, G, final positions, stats
        a, b = got[i], want[i]
        assert torch.equal(a[..., :E] if a.dim() > 1 else a, b[..., :E] if b.dim() > 1 else b), i
    assert bool((act[:, :, :E] != 4).any())
    # the same episode with the host-built table: the actions do not depend on it, and the rewards round alike
    out = env.policy_rollout(pol, T, lambdas=lam, gamma=0.9, thresholds=thr, g_mode=1)
    assert torch.equal(out["actions_"][:, :, :E], act[:, :, :E])
    assert torch.equal(out["R"], want[0][:, :E].t()) and torch.equal(out["C"], want[2][:, :E].t())


def test_stays_in_bounds():
    """Every buffer carved out of a sentinel-filled allocation, the records sentinel-filled too: nothing outside the
    declared rows x [0, 4 ceil(n_envs / 4)) is written (a thread writes its four envs as one word)."""
    from safe_multiagent_rl_b200 import _lib
    lib = _lib.load()
    A, E, T, size = 3, 37, 5, 6
    ld, E4 = 48, 40
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
    sx = make_buf(A, u8, torch.randint(0, size + 1, (A, ld), generator=g, device="cuda"))
    sy = make_buf(A, u8, torch.randint(0, size + 1, (A, ld), generator=g, device="cuda"))
    w1 = make_buf(6, f32, torch.randn(6, ld, generator=g, device="cuda") * 0.3)     # >= [A][2A][16]
    b1 = make_buf(1, f32, torch.randn(1, ld, generator=g, device="cuda"))           # [A][16]
    w2 = make_buf(5, f32, torch.randn(5, ld, generator=g, device="cuda"))           # [A][16][5]
    b2 = make_buf(1, f32, torch.randn(1, ld, generator=g, device="cuda"))           # >= [A][5]
    demand = make_buf(2, f64, torch.rand(2, ld, generator=g, device="cuda", dtype=f64) * 8 + 2)   # >= [7][7]
    lam = make_buf(1, f64, torch.full((1, ld), 0.5, device="cuda", dtype=f64))
    thr = make_buf(1, f64, torch.full((1, ld), 1.0, device="cuda", dtype=f64))
    sentinel = 12345.0
    obs = make_buf(T * 2 * A, f32, sentinel)
    act = make_buf(T * A, u8, 200)
    logp = make_buf(T * A, f32, sentinel)
    fx, fy = make_buf(A, u8, 200), make_buf(A, u8, 200)
    R, M, Cs = make_buf(A, f32, sentinel), make_buf(A, f32, sentinel), make_buf(1, i32, 12345)
    G, gs = make_buf(T * A, f32, sentinel), make_buf(T, f32, sentinel)
    stats = make_buf(1, f64, 0.0)
    scratch = make_buf(max(1, lib.smarl_stats_scratch_len(A, 1, E) // ld + 1), f64, 0.0)
    P = _lib.ptr
    pol = _lib.DiscretePolicyParams(A, 16, 5, 0, P(w1), P(b1), P(w2), P(b2), 77, 0, None)
    kp = _lib.CongestionParams(size, A, P(demand), 2, 0, 1 << 31, 9, 0, None, None)
    acc = _lib.Accounting(0.9, T, 1, P(thr))
    _lib.check(lib.smarl_congestion_policy_rollout(C.byref(kp), C.byref(pol), C.byref(acc), P(sx), P(sy), P(lam),
                                                   P(obs), P(act), P(logp), P(fx), P(fy), P(R), P(M), P(Cs), P(G),
                                                   P(gs), P(stats), P(scratch), E, ld,
                                                   torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    for i, raw in enumerate(bufs):
        assert bool((raw[:GUARD] == 0xA5).all()) and bool((raw[-GUARD:] == 0xA5).all()), f"buffer {i} overrun"
    for name, b, sent in (("obs", obs, sentinel), ("act", act, 200), ("logp", logp, sentinel), ("fx", fx, 200),
                          ("fy", fy, 200), ("R", R, sentinel), ("M", M, sentinel), ("C", Cs, 12345),
                          ("G", G, sentinel), ("gs", gs, sentinel)):
        assert bool((b[:, E4:] == sent).all()), name
        assert not bool((b[:, :E] == sent).any()), name
    assert bool((act[:, :E] <= 4).all())
    assert float(stats[0, 2 + 2 * A]) == E


def test_null_stats_and_records_through_the_abi():
    """stats / stats_scratch and the three records NULL: the episode products are those of the full call."""
    from safe_multiagent_rl_b200 import _lib
    A, E, T = 3, 300, 25
    env, pol = make(A, E, size=10, noise=0.1)
    lam = torch.tensor([0.2], dtype=torch.float64, device="cuda")
    want = tensors(env.policy_rollout(pol, T, lambdas=lam, gamma=0.95, g_mode=1))
    P = _lib.ptr
    f32 = torch.float32
    R, M, Cs, G = env._alloc(A, f32), env._alloc(A, f32), env._alloc(1, torch.int32), env._alloc(A, f32, (T,))
    gs = env._alloc(1, f32, (T,))
    fx, fy = torch.empty_like(env.pos_x), torch.empty_like(env.pos_y)
    acc = _lib.Accounting(0.95, T, 1, None)
    pp = pol.c_params(env)
    p = env._params(2)                                          # the noise episode of the call above
    _lib.check(env.lib.smarl_congestion_policy_rollout(
        C.byref(p), C.byref(pp), C.byref(acc), P(env.start_x), P(env.start_y), P(lam), None, None, None,
        P(fx), P(fy), P(R), P(M), P(Cs), P(G), P(gs), None, None, E, env.ld, _lib.stream_ptr()))
    torch.cuda.synchronize()
    assert torch.equal(R[:, :E].t(), want["R"]) and torch.equal(M[:, :E].t(), want["modR"])
    assert torch.equal(Cs[:, :E].t(), want["C"])
    assert torch.equal(G[:, :, :E].permute(0, 2, 1), want["G"])
    assert torch.equal(fx[:, :E], env.pos_x[:, :E]) and torch.equal(fy[:, :E], env.pos_y[:, :E])


def test_shards_reproduce_the_full_batch():
    A, E, T = 3, 400, 30
    starts = np.random.default_rng(9).integers(0, 4, (E, A, 2))
    env, pol = make(A, E, size=3, noise=0.3, starts=starts)
    full = tensors(env.policy_rollout(pol, T, g_mode=1))
    h = 202                                                     # a multiple of two, not of four
    for lo, hi in ((0, h), (h, E)):
        sub, sub_pol = make(A, hi - lo, size=3, noise=0.3, starts=starts[lo:hi], env_offset=lo)
        sub_pol.load_state_dict(pol.state_dict())
        sub_pol.seed = pol.seed
        part = sub.policy_rollout(sub_pol, T, g_mode=1)
        assert torch.equal(part["obs"], full["obs"][:, lo:hi]), "obs"
        for k in ("actions", "logp"):
            assert torch.equal(part[k], full[k][..., lo:hi]), k
        assert torch.equal(part["G"], full["G"][:, lo:hi]), "G"
        for k in ("R", "modR", "C"):
            assert torch.equal(part[k], full[k][lo:hi]), k
        assert torch.equal(sub.pos_x[:, :hi - lo], env.pos_x[:, lo:hi])


def test_cuda_graph_replay_and_episodes():
    """A captured policy_rollout bakes in the noise-episode increment: pinned to n - 1 it replays episode n, and after
    policy.next_episode() and another bump it draws what the eager call draws for those episodes."""
    A, E, T = 3, 1000, 20
    env, pol = make(A, E, size=3, noise=0.2)
    lam = torch.full((1,), 0.1, dtype=torch.float64, device="cuda")
    thr = torch.full((1,), 5.0, dtype=torch.float64, device="cuda")
    kw = dict(lambdas=lam, thresholds=thr, g_mode=1)
    out = env.policy_rollout(pol, T, **kw)                      # noise episode 0
    ptrs = {k: v.data_ptr() for k, v in out.items() if isinstance(v, torch.Tensor)}
    out = env.policy_rollout(pol, T, out=out, **kw)             # noise episode 1
    assert all(out[k].data_ptr() == p for k, p in ptrs.items())      # reused, nothing allocated
    eager1 = tensors(out)
    for k in eager1:
        out[k].zero_()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        env.policy_rollout(pol, T, out=out, **kw)
    env.set_noise_episode(0)
    g.replay()                                                  # bumps to 1
    torch.cuda.synchronize()
    for k, v in eager1.items():
        assert torch.equal(out[k], v), k
    pol.next_episode()
    g.replay()                                                  # noise episode 2, policy episode 1
    torch.cuda.synchronize()
    replayed = tensors(out)
    assert not torch.equal(replayed["actions"], eager1["actions"])
    assert torch.equal(replayed["obs"][0], eager1["obs"][0])    # same starts, other samples
    env.set_noise_episode(2)
    eager2 = tensors(env.policy_rollout(pol, T, **kw))
    for k, v in eager2.items():
        assert torch.equal(replayed[k], v), k


def test_noise_episode_follows_the_closed_loop():
    """set_noise_episode(n) then policy_rollout draws the noise that set_noise_episode(n) then the closed loop draws;
    noise 1.0 makes every move random, so the final positions depend on the noise alone."""
    A, E, T = 4, 2000, 12
    env_c, pol_c = make(A, E, size=10, noise=1.0, seed=2, on_policy=False)
    env_p, pol_p = make(A, E, size=10, noise=1.0, seed=2)
    finals = []
    for n in (5, 6):
        env_c.set_noise_episode(n)
        env_p.set_noise_episode(n)
        _, act, _, _ = closed_loop(env_c, pol_c, T, None)
        out = env_p.policy_rollout(pol_p, T)
        assert torch.equal(out["actions"], act)
        assert torch.equal(env_p.pos_x[:, :E], env_c.pos_x[:, :E]) and torch.equal(env_p.pos_y[:, :E], env_c.pos_y[:, :E])
        finals.append(env_p.pos_x[:, :E].clone())
    assert not torch.equal(finals[0], finals[1])


def test_rejected_inputs_queue_no_work():
    from safe_multiagent_rl_b200 import _lib
    lib = _lib.load()
    E, ld, T = 16, 16, 4
    P = _lib.ptr
    st = torch.cuda.current_stream().cuda_stream

    def call(A, pol_agents=None, hidden=16, n_actions=5, g_mode=0, n_steps=T, size=6, noise_mode=2, null_start=False,
             null_weight=False, null_g=False, null_gs=False, stats_only=False):
        big = torch.zeros(4096, ld, dtype=torch.float64, device="cuda")
        out = torch.full((4096, ld), 5.0, dtype=torch.float32, device="cuda")
        kp = _lib.CongestionParams(size, A, P(big), noise_mode, 0, 1 << 31, 1, 0, None, None)
        pol = _lib.DiscretePolicyParams(A if pol_agents is None else pol_agents, hidden, n_actions, 0,
                                        None if null_weight else P(out), P(out), P(out), P(out), 1, 0, None)
        acc = _lib.Accounting(0.9, n_steps, g_mode, None)
        rc = lib.smarl_congestion_policy_rollout(
            C.byref(kp), C.byref(pol), C.byref(acc), None if null_start else P(big), P(big), None, P(out), P(out),
            P(out), P(big), P(big), P(out), P(out), P(out), None if null_g else P(out), None if null_gs else P(out),
            P(big) if stats_only else None, None, E, ld, st)
        torch.cuda.synchronize()
        assert bool((out == 5.0).all()) and not bool(big.any())       # nothing ran
        return rc
    assert call(9) == -3
    assert call(32) == -3
    assert call(33) == -1
    assert call(3, noise_mode=1) == -3
    assert call(3, g_mode=3) == -1
    assert call(3, g_mode=-1) == -1
    assert call(3, hidden=8) == -1
    assert call(3, n_actions=9) == -1
    assert call(3, n_steps=0) == -1
    assert call(3, n_steps=65537) == -1
    assert call(3, size=255) == -1
    assert call(3, null_start=True) == -1
    assert call(3, null_weight=True) == -1
    assert call(3, g_mode=2, null_g=True) == -1
    assert call(3, g_mode=1, null_gs=True) == -1
    assert call(3, pol_agents=2) == -1
    assert call(3, stats_only=True) == -1
    import safe_multiagent_rl_b200 as s
    from safe_multiagent_rl_b200.policy import BatchedDiscretePolicy, FusedDiscretePolicy, FusedGaussianPolicy
    env = s.BatchedCongestionOnPolicy(3, 3, n_envs=E)
    with pytest.raises(NotImplementedError, match="DiscretePolicy: pass a FusedDiscretePolicy"):
        env.policy_rollout(BatchedDiscretePolicy(env), T)
    env9 = s.BatchedCongestionOnPolicy(10, 9, n_envs=E, demand_rate=np.full((11, 11), 3.0))
    with pytest.raises(NotImplementedError, match="one thread per four envs"):
        env9.policy_rollout(FusedDiscretePolicy(env9), T)
    envc = s.BatchedCoverageContinuous(6, 3, n_envs=E)       # the continuous envs keep their messages
    with pytest.raises(NotImplementedError, match="ContinuousPolicy: pass a FusedGaussianPolicy"):
        envc.policy_rollout(FusedDiscretePolicy(env), T)
    assert not hasattr(s.BatchedCoverageDiscretized(6, 3, n_envs=E), "policy_rollout")
    assert not hasattr(s.BatchedCongestion(3, 3, n_envs=E), "policy_rollout")   # the on-policy episode is opt-in
    assert issubclass(s.BatchedCongestionOnPolicy, s.BatchedCongestion)
    assert isinstance(FusedGaussianPolicy, type)


def test_policy_of_another_agent_count_is_rejected_before_any_launch():
    """A FusedDiscretePolicy holds the networks of the env it was built for; handed to an env of another agent count
    its weights would be read with that env's shapes.  policy_rollout raises before it draws starts, advances the
    noise episode or launches."""
    import safe_multiagent_rl_b200 as s
    from safe_multiagent_rl_b200.policy import FusedDiscretePolicy
    for A_pol, A_env in ((3, 4), (4, 3)):
        _, pol = make(A_pol, 64)
        env = s.BatchedCongestionOnPolicy(3, A_env, n_envs=64, shuffle=True, seed=3)
        env.set_noise_episode(7)
        before = [t.clone() for t in (env.start_x, env.start_y, env.pos_x, env.pos_y, env._episode_dev)]
        torch.cuda.synchronize()
        with pytest.raises(ValueError, match=f"policy holds {A_pol} agents' networks"):
            env.policy_rollout(pol, 10, g_mode=1)
        torch.cuda.synchronize()
        assert env._episode == 0 and not env._noise_started
        for a, b in zip(before, (env.start_x, env.start_y, env.pos_x, env.pos_y, env._episode_dev)):
            assert torch.equal(a, b)
        assert FusedDiscretePolicy(env).c_params(env).n_agents == A_env      # the env's own policy is accepted


def test_default_tensor_core_build_agrees_at_the_first_step():
    """At t = 0 the observation is the same for both paths: the default (tensor-core) build of FusedDiscretePolicy.act
    draws the one-launch rollout's actions except where the uniform sits within f32 rounding of a CDF step, with
    log-probabilities within test_tensor_core_and_fp32_builds_agree's bound.  Later steps diverge once one action
    differs (DESIGN.md section 3.14)."""
    for A, size in ((3, 3), (8, 10)):
        E = 65536
        env, pol = make(A, E, size=size, env_offset=123)
        out = env.policy_rollout(pol, 1)
        env.reset()
        _, act, logp = pol.act(t=0)
        same = act == out["actions"][0]
        assert same.float().mean().item() > 0.9995
        d = (logp - out["logp"][0]).abs()[same]
        assert d.max().item() < 2e-5 * max(1.0, size / 16), d.max().item()


def test_log_prob_of_the_records_matches_the_learner_side():
    """policy.log_prob on the recorded observations and actions (the PyTorch path a learner differentiates) against the
    kernel's log-probabilities."""
    A, E, T = 5, 3000, 12
    env, pol = make(A, E, size=10, shuffle=True)
    out = env.policy_rollout(pol, T)
    for t in (0, 5, T - 1):
        with torch.no_grad():
            want = pol.log_prob(out["obs"][t], out["actions"][t].long())
        assert torch.allclose(out["logp"][t], want, rtol=0, atol=1e-5), (out["logp"][t] - want).abs().max().item()
