"""The policy samplers' Philox draws at their extremes, on the CPU (oracle/philox.py): the env ids that
tests/test_gpu_policy_sampling_edges.py places inside batches really draw the extreme words, the float32 uniform of the
discrete head stays below 1 so that an action of probability 0 is never drawn, and the episode index reaches the
counter with all its 32 bits while the streams of episodes below 65 536 stay what they were."""
import math

import numpy as np
import pytest

from oracle import philox

SEED = philox.EDGE_SEED
TOP, ONE_BELOW = 2 ** 24 - 1, np.float32(1.0 - 2.0 ** -24)


def k_of(env_id, agent, t, n_agents=8, episode=0):
    return int(philox.policy_words(SEED, [env_id], t, n_agents, episode)[0, agent] >> np.uint32(8))


def test_discrete_edge_ids_draw_the_extreme_words():
    for env_id, agent, t in philox.DISCRETE_TOP:
        assert k_of(env_id, agent, t) == TOP, (env_id, agent, t)
    for env_id, agent, t in philox.DISCRETE_BOTTOM:
        assert k_of(env_id, agent, t) == 0, (env_id, agent, t)
    for env_id, agent, t, j in philox.DISCRETE_NEAR_TOP:
        assert k_of(env_id, agent, t) == 2 ** 24 - j, (env_id, agent, t)
    # what the GPU tests cover: every word slot of both agent quads, and two steps, at the top and bottom words
    for table in (philox.DISCRETE_TOP, philox.DISCRETE_BOTTOM):
        assert {a & 3 for _, a, _ in table} == {0, 1, 2, 3}
        assert {a >> 2 for _, a, _ in table} == {0, 1} and {t for _, _, t in table} == {0, 1}
    # a hit draws its extreme word in its own slot only: the word is a function of (env id, t, agent quad)
    env_id, agent, t = philox.DISCRETE_TOP[0]
    assert k_of(env_id, agent, t, n_agents=agent + 1) == TOP


def test_gaussian_edge_ids_draw_the_extreme_words():
    for (which, v), hits in philox.GAUSS_EDGES.items():
        assert {a >> 1 for _, a, _ in hits} == {0, 1}
        for env_id, agent, t in hits:
            wa, wb = philox.gaussian_words(SEED, [env_id], t, 4)
            w = (wa if which == "u0" else wb)[0, agent]
            assert int(w >> np.uint32(9)) == v, (which, v, env_id, agent, t)
    # u0's floor 2**-24 is the largest radius the sampler can draw: |z| = sqrt(-2 ln 2**-24) = sqrt(48 ln 2)
    env_id, agent, t = philox.GAUSS_EDGES[("u0", 0)][0]
    u0, u1 = philox.gaussian_uniforms(SEED, [env_id], t, 4)
    assert u0[0, agent] == 2.0 ** -24 and 0.0 < u1[0, agent] < 1.0
    z = philox.gaussian_normals(SEED, [env_id], t, 4)[0, agent]
    assert math.isclose(math.hypot(*z), math.sqrt(48 * math.log(2)), rel_tol=1e-12)
    env_id, agent, t = philox.GAUSS_EDGES[("u1", 2 ** 23 - 1)][0]
    assert philox.gaussian_uniforms(SEED, [env_id], t, 4)[1][0, agent] == 1.0 - 2.0 ** -24


def test_float32_uniform_rounds_as_the_kernel_and_stays_below_one():
    k = np.arange(2 ** 24, dtype=np.uint32)
    u = philox.policy_u_f32(k)
    assert u.dtype == np.float32
    exact = (k.astype(np.float64) + 0.5) / 2.0 ** 24
    # below 2**23, k + 0.5 is exact; above it rounds to even, off by 2**-25; the top word is clamped to 1 - 2**-24
    assert np.array_equal(u[: 2 ** 23], exact[: 2 ** 23].astype(np.float32))
    assert np.abs(u[:-1].astype(np.float64) - exact[:-1]).max() == 2.0 ** -25
    assert u[TOP] == ONE_BELOW and u.max() == ONE_BELOW and bool(np.all(np.diff(u) >= 0))
    # without the clamp the top word would be 1 exactly: u * sum == sum picks the last action whatever its probability
    assert (np.float32(TOP) + np.float32(0.5)) * np.float32(2.0 ** -24) == np.float32(1.0)


def test_clamped_uniform_keeps_the_target_below_every_sum():
    """policy_head draws action #{c < NA-1 : cum_c <= u * sum} with the partial sums cum formed in the order of sum,
    so a trailing action whose e_c is 0 has cum_{NA-2} == sum: it is never drawn iff fl(u * sum) < sum.  The max term
    alone contributes 1, so sum >= 1; it is at most NA = 9.  Every float32 sum in [1, 16) is checked."""
    s = (np.arange(4 * 2 ** 23, dtype=np.uint32) + np.uint32(0x3F800000)).view(np.float32)     # [1, 16)
    assert s[0] == 1.0 and s[-1] == np.nextafter(np.float32(16.0), np.float32(0.0))
    assert bool(np.all(ONE_BELOW * s < s))
    assert bool(np.all(np.float32(1.0) * s == s))


def head_f32(l2, u):
    """policy_head in numpy float32 (ex2 flushed to 0 below 2**-126 as ex2.approx.ftz does): the pick of u."""
    l2 = np.asarray(l2, dtype=np.float32)
    m = l2.max()
    ex = np.exp2((l2 - m).astype(np.float64)).astype(np.float32)
    ex[ex < np.float32(2.0 ** -126)] = 0
    tot = np.float32(0)
    for e in ex:
        tot = np.float32(tot + e)
    target, cum, pick = np.float32(u * tot), np.float32(0), 0
    for c in range(len(l2) - 1):
        cum = np.float32(cum + ex[c])
        if cum <= target:
            pick = c + 1
    return pick


@pytest.mark.parametrize("l2", [(10.0, 0.0, -3.0, 1.0, -200.0), (0.5, -1.0, 2.0, 0.0, 3.0, 1.0, -2.0, 0.25, -300.0)])
def test_top_word_never_draws_a_zero_probability_last_action(l2):
    assert head_f32(l2, np.float32(1.0)) == len(l2) - 1                  # the unclamped top draw
    assert head_f32(l2, philox.policy_u_f32(TOP)) == len(l2) - 2
    assert head_f32(l2, philox.policy_u_f32(0)) == 0                    # the bottom draw takes the first action


def old_words(seed, env_ids, t, n_agents, episode, key_xor, per_block):
    """The counter before the episode's high bits were carried: (id, t | episode << 16, agent // per_block)."""
    env_ids = np.asarray(env_ids, dtype=np.uint64)
    tw = (t | (episode << 16)) & 0xFFFFFFFF
    ag = np.arange(n_agents, dtype=np.uint64) // np.uint64(per_block)
    return philox.philox4x32_10((env_ids & philox.MASK)[:, None], (env_ids >> np.uint64(32))[:, None],
                                np.full((1, 1), tw, dtype=np.uint64), ag[None, :], seed & 0xFFFFFFFF,
                                ((seed >> 32) & 0xFFFFFFFF) ^ key_xor)


@pytest.mark.parametrize("episode", [0, 1, 777, 65535])
def test_streams_below_episode_65536_are_unchanged(episode):
    ids = np.arange(5_000_000_000, 5_000_000_000 + 300, dtype=np.uint64)
    A = 32
    o = np.stack(old_words(SEED, ids, 9, A, episode, 0x504C4359, 4), axis=0)
    want = o[np.arange(A) & 3, :, np.arange(A)].T
    assert np.array_equal(philox.policy_words(SEED, ids, 9, A, episode), want)
    o = np.stack(old_words(SEED, ids, 9, A, episode, 0x47415553, 2), axis=0)
    ag = np.arange(A)
    wa, wb = philox.gaussian_words(SEED, ids, 9, A, episode)
    assert np.array_equal(wa, o[2 * (ag & 1), :, ag].T) and np.array_equal(wb, o[2 * (ag & 1) + 1, :, ag].T)


@pytest.mark.parametrize("base", [0, 3, 65535])
def test_episodes_65536_apart_draw_different_streams(base):
    ids = np.arange(1000, 1400, dtype=np.uint64)
    A = 32
    streams = {}
    for ep in (base, base + 65536, base + 2 * 65536, base + (2 ** 32 - 65536)):
        streams[ep] = (philox.policy_words(SEED, ids, 5, A, ep), *philox.gaussian_words(SEED, ids, 5, A, ep))
    eps = list(streams)
    for i in range(len(eps)):
        for j in range(i + 1, len(eps)):
            for x, y in zip(streams[eps[i]], streams[eps[j]]):
                assert (x == y).mean() < 0.01, (eps[i], eps[j])
    # and different agent quads / pairs of one episode still draw different blocks at the highest episodes
    w = philox.policy_words(SEED, ids, 5, A, 2 ** 32 - 1)
    assert (w[:, 0] == w[:, 4]).mean() < 0.01
