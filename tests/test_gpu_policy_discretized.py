"""smarl_policy_act_discretized / FusedDiscretizedPolicy: the reference's DiscretePolicy (agent.py:23-47) on
CoverageDiscretized's 9 actions, against float64 logits and the Philox stream restated in oracle/philox.py."""
import numpy as np
import pytest
import torch

from oracle import philox

pytestmark = pytest.mark.gpu


def make(A, E, size=5, coarseness=6, seed=0, env_offset=0, starts=None):
    import safe_multiagent_rl_b200 as s
    from safe_multiagent_rl_b200.policy import FusedDiscretizedPolicy
    if starts is None:
        zoom = coarseness / size
        starts = np.floor(np.random.default_rng(seed).random((E, A, 2)) * size * zoom) / zoom
    env = s.BatchedCoverageDiscretized(size, A, n_envs=E, coarseness=coarseness, starts=starts, env_offset=env_offset)
    torch.manual_seed(seed)
    pol = FusedDiscretizedPolicy(env, seed=4321 + seed)
    with torch.no_grad():                  # wider logits than the default init: every action gets real probability mass
        pol.fc2.weight.mul_(4.0)
    return env, pol


def logits64(pol, obs):
    """[E, A, 9] float64 logits of the f32 observation [E, 2A]."""
    x = obs.double()
    w1, b1 = pol.fc1.weight.detach().double(), pol.fc1.bias.detach().double()
    w2, b2 = pol.fc2.weight.detach().double(), pol.fc2.bias.detach().double()
    h = torch.relu(torch.matmul(x, w1) + b1)               # [A, E, 16]
    return (torch.matmul(h, w2) + b2).permute(1, 0, 2).cpu().numpy()


@pytest.mark.parametrize("A", [1, 3, 5, 8, 12, 17, 32])
@pytest.mark.parametrize("E,env_offset", [(1, 0), (37, 2 ** 33), (4099, 0)])
def test_matches_the_oracle(A, E, env_offset):
    env, pol = make(A, E, seed=A + E, env_offset=env_offset)
    env.reset()
    for t in (0, 1, 7):
        obs = env.obs[:, :E].t().contiguous()
        _, act, lp = pol.act(t=t)
        act, lp = act.long(), lp.clone()
        with torch.no_grad():
            want_lp = pol.log_prob(obs, act)
        assert float((lp - want_lp).abs().max()) <= 1e-5
        u = philox.policy_uniforms(pol.seed, env_offset + np.arange(E), t, A)
        a_ref, _, margin = philox.policy_sample(logits64(pol, obs), u)
        got = act.t().cpu().numpy()
        sure = margin > 1e-5
        assert sure.mean() > 0.99 or sure.size < 100
        assert np.array_equal(got[sure], a_ref[sure])
        env.step(env.action_buffer, agent_major=True)


def test_every_action_occurs():
    A, E = 3, 65536
    env, pol = make(A, E, size=32, coarseness=20)
    env.reset()
    _, act, _ = pol.act(t=0)
    counts = torch.bincount(act.reshape(-1).long(), minlength=9)
    assert counts.numel() == 9 and bool((counts > 0).all()), counts.tolist()


def test_streams_follow_global_env_ids_and_episodes():
    A, E = 5, 400
    zoom = 6 / 5
    starts = np.floor(np.random.default_rng(3).random((E, A, 2)) * 5 * zoom) / zoom
    env, pol = make(A, E, starts=starts)
    env.reset()
    _, act, lp = pol.act(t=3)
    act, lp = act.clone(), lp.clone()
    h = E // 2
    for lo, hi in ((0, h), (h, E)):
        sub, sub_pol = make(A, hi - lo, starts=starts[lo:hi], env_offset=lo)
        sub_pol.load_state_dict(pol.state_dict())
        sub_pol.seed = pol.seed
        sub.reset()
        _, a_s, l_s = sub_pol.act(t=3)
        assert torch.equal(a_s, act[:, lo:hi]) and torch.equal(l_s, lp[:, lo:hi])
    pol.next_episode()
    _, act2, _ = pol.act(t=3)
    assert not torch.equal(act2, act)
    u0 = philox.policy_uniforms(pol.seed, np.arange(E), 3, A)
    u1 = philox.policy_uniforms(pol.seed, np.arange(E), 3, A, episode=1)
    a_ref, _, margin = philox.policy_sample(logits64(pol, env.obs[:, :E].t()), u1)
    sure = margin > 1e-5
    assert not np.array_equal(u0, u1)
    assert np.array_equal(act2.t().cpu().numpy()[sure], a_ref[sure])


def test_graphed_closed_loop():
    import safe_multiagent_rl_b200 as s
    A, E, T = 3, 50, 50
    env, pol = make(A, E)
    lam = torch.full((A,), 0.1, dtype=torch.float64, device="cuda")
    loop = s.GraphedClosedLoop(env, T, lambda obs, t: pol.act(t=t), lam, 0.99, thresholds=[2.0] * A)
    final = env.pos_x.clone()                      # the eager warm-up's episode (the capture itself runs nothing)
    env.pos_x.zero_()
    out = loop.replay()
    torch.cuda.synchronize()
    assert torch.equal(env.pos_x, final)
    want = {k: v.clone() for k, v in out.items() if isinstance(v, torch.Tensor)}
    out = loop.replay()
    torch.cuda.synchronize()
    for k, v in want.items():
        assert torch.equal(out[k], v), k
    pol.next_episode()
    loop.replay()
    torch.cuda.synchronize()
    assert not torch.equal(env.pos_x[:, :E], final[:, :E])


def test_rejections():
    import safe_multiagent_rl_b200 as s
    from safe_multiagent_rl_b200.policy import FusedDiscretePolicy, FusedDiscretizedPolicy
    with pytest.raises(NotImplementedError):
        FusedDiscretizedPolicy(s.BatchedCoverageDiscrete(5, 3, n_envs=16))
    with pytest.raises(NotImplementedError):
        FusedDiscretizedPolicy(s.BatchedCoverageContinuous(5, 3, n_envs=16))
    env = s.BatchedCoverageDiscretized(5, 3, n_envs=16, coarseness=6)
    with pytest.raises(NotImplementedError):
        FusedDiscretizedPolicy(env, hidden_size=8)
    with pytest.raises(NotImplementedError):
        FusedDiscretePolicy(env)
    other = FusedDiscretizedPolicy(s.BatchedCoverageDiscretized(5, 2, n_envs=16, coarseness=6))
    with pytest.raises(ValueError):
        other.c_params(env)
