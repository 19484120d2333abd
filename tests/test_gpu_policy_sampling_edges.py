"""Every fused policy sampler at its extreme Philox draws: the seven discrete ones (smarl_policy_act_discrete in its
FP32-pipe and two tensor-core builds, smarl_policy_act_discretized, and the one-launch rollouts of CoverageDiscrete,
Congestion and CoverageDiscretized) and the three Gaussian ones (smarl_policy_act_gaussian and the Collision and
CoverageContinuous rollouts).

The other tests compare samples with oracle/philox.py only where the uniform is clear of float32 rounding at a CDF
step; these put the env ids whose words sit at the extremes (oracle/philox.py's tables, re-derived on the CPU by
tests/test_policy_sampling_draws.py) inside batches through env_offset, at a first tile, the second 128-row tile of a
tensor-core CTA iteration, a later tile of a persistent CTA and the ragged tail, and check:
  * an action of probability 0 (logit -200, first or last) is never drawn, also at the top word u = 1 - 2**-24, and
    every log-probability is the float64 log_softmax of the same observation at the drawn action;
  * an action of probability ~8e-7 is drawn by exactly the top words of its CDF interval;
  * episode 65 536 draws other samples than episode 0, and episodes 65 535 / 65 536 match the oracle;
  * the Gaussian samples at u0, u1 = 2**-24 and 1 - 2**-24 match the float64 Box-Muller to 1e-6."""
import math

import numpy as np
import pytest
import torch

from oracle import philox

pytestmark = pytest.mark.gpu

SEED = philox.EDGE_SEED
E = 300_007                  # not a multiple of 16, and more tiles than one wave of persistent CTAs holds
PLACES = (5, 128 + 9, 200_003, E - 3)   # first tile, second 128-row tile, a later tile of a persistent CTA, the tail
DISCRETE = ["act_fp32", "act_tc16", "act_tc8", "act_discretized", "rollout_coverage", "rollout_congestion",
            "rollout_discretized"]
GAUSSIAN = ["act_gaussian", "rollout_collision", "rollout_coverage_continuous"]


def place(i, env_id):
    """Where hit i lands in the batch (cycling over PLACES; ids below a placement take the first tile)."""
    j = PLACES[i % len(PLACES)]
    return j if j <= env_id else PLACES[0]


# ---- discrete -------------------------------------------------------------------------------------------------------
def discrete_setup(path, A, n_envs):
    import safe_multiagent_rl_b200 as s
    from safe_multiagent_rl_b200.policy import FusedDiscretePolicy, FusedDiscretizedPolicy
    rng = np.random.default_rng(A + n_envs)
    if path in ("act_discretized", "rollout_discretized"):
        zoom = 6 / 5
        starts = np.floor(rng.random((n_envs, A, 2)) * 5 * zoom) / zoom
        env = s.BatchedCoverageDiscretizedOnPolicy(5, A, n_envs=n_envs, coarseness=6, starts=starts)
        cls = FusedDiscretizedPolicy
    elif path == "rollout_congestion":
        env = s.BatchedCongestionOnPolicy(3, A, n_envs=n_envs, noise=0.0, starts=rng.integers(0, 4, (n_envs, A, 2)))
        cls = FusedDiscretePolicy
    else:
        env = s.BatchedCoverageDiscrete(5, A, n_envs=n_envs, starts=rng.integers(0, 6, (n_envs, A, 2)))
        cls = FusedDiscretePolicy
    torch.manual_seed(A)
    pol = cls(env, seed=SEED)
    with torch.no_grad():
        pol.fc1.weight.mul_(0.8)                   # inputs of order 1: no action dominates
        pol.fc2.weight.mul_(4.0)
    return env, pol


def discrete_draws(path, env, pol, env_offset, T=2):
    """[(obs [E, S] f32, actions [A, E] int64, logp [A, E] f32)] of steps t = 0..T-1, all on the device."""
    from safe_multiagent_rl_b200 import _lib
    env.env_offset = int(env_offset)
    E_ = env.n_envs
    if path.startswith("rollout"):
        out = env.policy_rollout(pol, T, record=True)
        return [(out["obs"][t], out["actions"][t].long(), out["logp"][t]) for t in range(T)]
    variant = {"act_fp32": 0, "act_tc16": 1, "act_tc8": 2}.get(path, 0)
    obs = env.reset().clone()
    res = []
    for t in range(T):
        with _lib.kernel_variant(_lib.KERNEL_POLICY, variant):
            pol.act(t=t)
        res.append((obs, env.action_buffer[:, :E_].long(), pol.logp[:, :E_].clone()))
    return res


def logits64(pol, obs):
    """[A, E, NA] float64 logits of the f32 observation [E, S], on the device."""
    w1, b1, w2, b2 = (p.detach().double() for p in (pol.fc1.weight, pol.fc1.bias, pol.fc2.weight, pol.fc2.bias))
    return torch.matmul(torch.relu(torch.matmul(obs.double(), w1) + b1), w2) + b2


def check_logp(pol, obs, act, logp):
    """Every log-probability is the float64 log_softmax of the same observation at the drawn action."""
    want = torch.log_softmax(logits64(pol, obs), dim=-1).gather(-1, act[..., None])[..., 0]
    err = (logp.double() - want).abs() / (1 + want.abs())
    assert err.max().item() <= 1e-5, err.max().item()


@pytest.mark.parametrize("path", DISCRETE)
def test_actions_of_probability_zero_are_never_drawn(path):
    """Logits of -200 on the first and last actions (fc2 column 0, bias -200): their e_c flush to 0.  At the top word
    the unclamped float32 uniform was 1, u * sum == sum, and the last action was drawn with a log-probability near -200;
    at the bottom word the first action must not be drawn either."""
    A = 8
    env, pol = discrete_setup(path, A, E)
    NA = pol.n_actions
    with torch.no_grad():
        for c in (0, NA - 1):
            pol.fc2.weight[:, :, c] = 0.0
            pol.fc2.bias[:, :, c] = -200.0
    hits = [(i, h, NA - 1) for i, h in enumerate(philox.DISCRETE_TOP)]
    hits += [(i, h, 0) for i, h in enumerate(philox.DISCRETE_BOTTOM)]
    for i, (env_id, agent, t), impossible in hits:
        j = place(i, env_id)
        steps = discrete_draws(path, env, pol, env_id - j)
        obs, act, logp = steps[t]
        assert int(act[agent, j]) != impossible, (path, env_id, agent, t, j)
        for obs_s, act_s, logp_s in steps:
            assert int(act_s.min()) >= 1 and int(act_s.max()) <= NA - 2, (path, env_id)
            check_logp(pol, obs_s, act_s, logp_s)


@pytest.mark.parametrize("path", DISCRETE)
def test_rare_last_action_is_drawn_at_the_top_of_its_interval(path):
    """The last action 14 nats below the first (p ~ 8e-7, some 14 words at the top of the 2**24), the middle ones 40
    below: the top words draw the last action, the words below its CDF interval the first, with the float64
    log-probability.  Words within 2e-7 of the CDF step (float32 rounding of u * sum) are not judged."""
    A = 8
    env, pol = discrete_setup(path, A, E)
    NA = pol.n_actions
    with torch.no_grad():
        pol.fc2.weight[:, :, 1:] = 0.0
        pol.fc2.weight[:, :, 0] *= 0.005                   # the gap stays within 14 +- 0.03 nats
        pol.fc2.bias[:, :, 0] = 0.0
        pol.fc2.bias[:, :, 1:NA - 1] = -40.0
        pol.fc2.bias[:, :, NA - 1] = -14.0
    drawn = judged = 0
    for i, (env_id, agent, t, _) in enumerate(philox.DISCRETE_NEAR_TOP):
        j = place(i, env_id)
        steps = discrete_draws(path, env, pol, env_id - j)
        obs, act, logp = steps[t]
        u = philox.policy_uniforms_f32(SEED, [env_id], t, A)[0, agent]
        l64 = logits64(pol, obs[j:j + 1])[agent, 0].cpu().numpy()
        a_o, lp_o, margin = philox.policy_sample(l64, np.float64(u))
        if margin > 2e-7:
            judged += 1
            drawn += int(a_o == NA - 1)
            assert int(act[agent, j]) == int(a_o), (path, env_id, agent, t, j, float(margin))
            assert abs(float(logp[agent, j]) - float(lp_o)) <= 1e-5 * (1 + abs(float(lp_o)))
        for obs_s, act_s, logp_s in steps:
            assert bool(((act_s == 0) | (act_s == NA - 1)).all())
            check_logp(pol, obs_s, act_s, logp_s)
    assert drawn >= 3 and judged - drawn >= 3, (drawn, judged)


def discrete_oracle_match(pol, obs, act, logp, env_ids, t, episode):
    A = act.shape[0]
    u = philox.policy_uniforms_f32(SEED, env_ids, t, A, episode).T                        # [A, E]
    a_o, lp_o, margin = philox.policy_sample(logits64(pol, obs).cpu().numpy(), u)
    clear = margin > 1e-5
    assert clear.mean() > 0.99
    act_np, logp_np = act.cpu().numpy(), logp.cpu().numpy()
    assert np.array_equal(act_np[clear], a_o[clear]), (episode, t)
    np.testing.assert_allclose(logp_np[clear], lp_o[clear], rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("path", DISCRETE)
def test_discrete_streams_do_not_repeat_after_65536_episodes(path):
    A, n = 6, 4099
    env, pol = discrete_setup(path, A, n)
    ids = 7_000_000_000 + np.arange(n)
    draws = {}
    for episode in (0, 65535, 65536):
        pol._episode_dev.fill_(episode)
        draws[episode] = [(o.clone(), a.clone(), lp.clone()) for o, a, lp in discrete_draws(path, env, pol, ids[0])]
    for t in range(2):
        assert not torch.equal(draws[65536][t][1], draws[0][t][1]), (path, t)
        for episode in (65535, 65536):
            discrete_oracle_match(pol, *draws[episode][t], ids, t, episode)


# ---- Gaussian -------------------------------------------------------------------------------------------------------
MU = (0.25, -0.5)
VAR_BIAS = 0.5


def gaussian_setup(path, A, n_envs):
    """fc2 / fc2_ weights zeroed: mu = (0.25, -0.5) and sigma^2 = 0.5 + 1e-4 for every observation, so the samples
    measure the sampler alone."""
    import safe_multiagent_rl_b200 as s
    from safe_multiagent_rl_b200.policy import FusedGaussianPolicy
    rng = np.random.default_rng(A + n_envs)
    if path == "rollout_collision":
        env = s.BatchedCollisionAvoidance(6, A, n_envs=n_envs, n_landmarks=1, starts=rng.random((n_envs, A, 2)) * 6,
                                          landmarks=rng.random((n_envs, 1, 2)) * 6)
    else:
        env = s.BatchedCoverageContinuous(8, A, n_envs=n_envs, starts=rng.random((n_envs, A, 2)) * 8)
    torch.manual_seed(A)
    pol = FusedGaussianPolicy(env, seed=SEED)
    with torch.no_grad():
        pol.fc2.weight.zero_()
        pol.fc2_.weight.zero_()
        pol.fc2.bias[:, :, 0] = MU[0]
        pol.fc2.bias[:, :, 1] = MU[1]
        pol.fc2_.bias.fill_(VAR_BIAS)
    return env, pol


def gaussian_draws(path, env, pol, env_offset, T=2):
    """[(actions [A, E, 2], logp [A, E])] of steps t = 0..T-1, on the device."""
    env.env_offset = int(env_offset)
    E_ = env.n_envs
    if path.startswith("rollout"):
        out = env.policy_rollout(pol, T, record=True)
        return [(out["actions"][t], out["logp"][t]) for t in range(T)]
    env.reset()
    res = []
    for t in range(T):
        _, a, lp = pol.act(t=t)
        res.append((a.clone(), lp.clone()))
    return res


def gauss_moments():
    mu = torch.tensor(MU, dtype=torch.float64, device="cuda")
    var = torch.tensor(float(np.float32(VAR_BIAS) + np.float32(1e-4)), dtype=torch.float64, device="cuda")
    return mu, var


def gauss_logp64(a):
    """float64 log N(a; mu, diag var) of actions [..., 2] (the kernel evaluates it on its rounded action)."""
    mu, var = gauss_moments()
    d = a.double() - mu
    return -0.5 * ((d * d / var).sum(-1) + 2 * torch.log(var)) - math.log(2 * math.pi)


def check_gauss_logp(act, logp, rel):
    want = gauss_logp64(act)
    err = (logp.double() - want).abs() / (1 + want.abs())
    assert err.max().item() <= rel, err.max().item()


@pytest.mark.parametrize("path", GAUSSIAN)
def test_gaussian_samples_at_the_extreme_uniforms(path):
    A = 4
    env, pol = gaussian_setup(path, A, E)
    mu, var = (x.cpu().numpy() for x in gauss_moments())
    i = 0
    for (which, v), hits in philox.GAUSS_EDGES.items():
        for env_id, agent, t in hits:
            j = place(i, env_id)
            i += 1
            steps = gaussian_draws(path, env, pol, env_id - j)
            act, logp = steps[t]
            z = philox.gaussian_normals(SEED, [env_id], t, A)[0, agent]
            a_o = mu + math.sqrt(var) * z
            a_k = act[agent, j].double().cpu().numpy()
            assert np.all(np.abs(a_k - a_o) <= 1e-6 * (1 + np.abs(a_o))), (path, which, v, env_id, a_k, a_o)
            lp_want = float(gauss_logp64(act[agent, j]))
            assert abs(float(logp[agent, j]) - lp_want) <= 1e-6 * (1 + abs(lp_want)), (path, which, v, env_id)
            if (which, v) == ("u0", 0):                     # the largest radius: |z| = sqrt(-2 ln 2**-24)
                r = math.hypot(*((a_k - mu) / math.sqrt(var)))
                assert math.isclose(r, math.sqrt(48 * math.log(2)), rel_tol=2e-6), (path, env_id, r)
            for act_s, logp_s in steps:
                assert bool(torch.isfinite(act_s).all())
                check_gauss_logp(act_s, logp_s, 1e-5)


@pytest.mark.parametrize("path", GAUSSIAN)
def test_gaussian_streams_do_not_repeat_after_65536_episodes(path):
    A, n = 4, 4099
    env, pol = gaussian_setup(path, A, n)
    mu, var = (x.cpu().numpy() for x in gauss_moments())
    ids = 7_000_000_000 + np.arange(n)
    draws = {}
    for episode in (0, 65535, 65536):
        pol._episode_dev.fill_(episode)
        draws[episode] = [(a.clone(), lp.clone()) for a, lp in gaussian_draws(path, env, pol, ids[0])]
    for t in range(2):
        assert not torch.equal(draws[65536][t][0], draws[0][t][0]), (path, t)
        for episode in (65535, 65536):
            act, logp = draws[episode][t]
            z = philox.gaussian_normals(SEED, ids, t, A, episode)                              # [E, A, 2]
            a_o = mu + math.sqrt(var) * z.transpose(1, 0, 2)                                    # [A, E, 2]
            a_k = act.double().cpu().numpy()
            assert np.all(np.abs(a_k - a_o) <= 1e-5 * (1 + np.abs(a_o))), (path, episode, t)
            check_gauss_logp(act, logp, 1e-5)
