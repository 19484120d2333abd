"""oracle/threshold_cases.py builds inputs on the decision thresholds of the CollisionAvoidance and CoverageContinuous
env steps.  These CPU checks hold each family to its claim: the values sit where the family says (recomputed from the
laid-out env inputs with the oracle's arithmetic), every band holds cases on both sides of the reference's decision,
and some cases are ones the squared comparison alone would decide wrong."""
import numpy as np
import pytest

from oracle import numpy_oracle as no
from oracle import threshold_cases as tc


def sides(p):
    return int((p.in_band & p.decision).sum()), int((p.in_band & ~p.decision).sum())


@pytest.mark.parametrize("agents_size", tc.REACH_SIZES)
def test_reach_probes_sit_on_the_threshold(agents_size):
    p = tc.reach_probes(agents_size)
    a = agents_size
    as2 = a * a
    qn = tc.reach_qn(p.pts[:, 0, 0], p.pts[:, 0, 1], p.lms[:, 0, 0], p.lms[:, 0, 1])
    assert np.array_equal(qn, p.value)
    assert np.array_equal(np.sqrt(qn) < a, p.decision) and np.array_equal(qn < as2, p.squared)
    assert np.array_equal((qn >= as2 * 0.999999999) & (qn < as2 * 1.000000001), p.in_band)
    for t in (as2, np.nextafter(as2, 0), np.nextafter(as2, 1)):          # on it and one ulp either side
        assert (qn == t).any()
    inside, outside = sides(p)
    assert inside >= 10 and outside >= 10
    assert (~p.in_band & p.decision).any() and (~p.in_band & ~p.decision).any()
    if a in (0.1, 0.3):        # no exact square: qn < agents_size^2 and sqrt(qn) < agents_size disagree
        assert (p.squared != p.decision).sum() >= 5
        assert (p.in_band[p.squared != p.decision]).all()


@pytest.mark.parametrize("agents_size", [0.25, 0.1, 0.3])
def test_pair_probes_sit_on_the_threshold(agents_size):
    p = tc.pair_probes(agents_size)
    lim = 2 * agents_size
    lim2 = lim * lim
    q = tc.pair_q(p.pts[:, 0, 0], p.pts[:, 0, 1], p.pts[:, 1, 0], p.pts[:, 1, 1])
    assert np.array_equal(q, p.value) and np.array_equal(np.sqrt(q) < lim, p.decision)
    assert np.array_equal((q >= lim2 * 0.999999) & (q < lim2 * 1.000001), p.in_band)
    for t in (lim2, np.nextafter(lim2, 0), np.nextafter(lim2, 1)):
        assert (q == t).any()
    inside, outside = sides(p)
    assert inside >= 10 and outside >= 10
    if agents_size != 0.25:
        assert (p.squared != p.decision).sum() >= 5


@pytest.mark.parametrize("size", [200, 5000])
def test_screen_probes_are_near_the_far_corner(size):
    p = tc.pair_probes(1e-3, size=size, near=(size, size), park=(10.0, 10.0))
    assert p.pts.min() > size - 1 and p.pts.max() <= size
    inside, outside = sides(p)
    assert inside >= 10 and outside >= 10
    q = tc.pair_q(p.pts[:, 0, 0], p.pts[:, 0, 1], p.pts[:, 1, 0], p.pts[:, 1, 1])
    assert np.array_equal(np.sqrt(q) < 2e-3, p.decision)


def test_special_pairs_count_only_alive_agents():
    """Through the oracle itself: the reach-and-collide pairs count exactly when the probe does not reach its landmark,
    the corner pairs are clamped onto (0, 0) and always count."""
    p = tc.pair_special_probes(0.25)
    c = tc.layout(p, 5, seed=1)
    pos, _, cost, done, _ = no.collision_step(c.starts, np.zeros(c.starts.shape[:2], bool), c.actions[0], c.landmarks,
                                              c.size, c.agents_size)
    assert np.array_equal(cost[:, 0] == 1, p.decision)
    corner = p.kind == "corner"
    e = np.flatnonzero(corner)
    assert np.all(pos[e[:, None], c.probe_idx[e]] == 0.0)
    rp = ~corner
    assert (p.in_band[rp] & p.decision[rp]).any() and (p.in_band[rp] & ~p.decision[rp]).any()


def test_clip_probes():
    p = tc.clip_probes()
    q = (p.act[:, 0].astype(np.float64) ** 2).sum(1)
    assert np.array_equal(q, p.value)
    kinds = dict(zip(*np.unique(p.kind, return_counts=True)))
    assert kinds["q_eq_1"] >= 4 and kinds["q_gt_1_norm_eq_1"] >= 4 and kinds["first_clip"] >= 4
    assert np.all(np.sqrt(q[p.kind == "q_gt_1_norm_eq_1"]) == 1.0)          # q > 1 and no division
    assert np.all(np.sqrt(q[p.kind == "first_clip"]) > 1.0)
    assert np.all(q[p.kind == "first_clip"] == 1 + 2.0 ** -51)                # smallest q with sqrt_rn(q) > 1
    assert (q < 1).any()


def test_clip_overflow_posts_more_clips_than_slots():
    for A in (3, 7, 9, 16):
        c = tc.clip_overflow_cases(A)
        q = (c.actions.astype(np.float64) ** 2).sum(-1)
        assert (q > 1).all() and 32 * A > 64


@pytest.mark.parametrize("size,coarseness", [(5, 6), (10, 7)])
def test_rescale_cases_straddle_the_decision(size, coarseness):
    act, q, dec, band = tc.rescale_actions(size, coarseness)
    mn = np.sqrt(2) * size / coarseness
    assert np.array_equal((act.astype(np.float64) ** 2).sum(1), q)
    assert np.array_equal(np.sqrt(np.sqrt(q)) > mn, dec)
    assert (band & dec).sum() >= 20 and (band & ~dec).sum() >= 20
    assert (~band & dec).any() and (~band & ~dec).any()
    m4 = (mn * mn) * (mn * mn)
    assert np.all(np.abs(q[band] / m4 - 1) <= 1e-9 * (1 + 1e-6))


@pytest.mark.parametrize("A", [3, 7, 8, 12, 16, 31])
def test_layout_keeps_the_probes_and_parks_the_rest(A):
    p = tc.reach_probes(0.1)
    c = tc.layout(p, A, T=2, seed=A)
    E = len(p.value)
    assert c.starts.shape == (E, A, 2) and c.landmarks.shape == (E, 2, 2) and c.actions.shape == (2, E, A, 2)
    assert np.array_equal(c.starts[np.arange(E), c.probe_idx[:, 0]], p.pts[:, 0])
    pos, _, _, done, _ = no.collision_step(c.starts, np.zeros((E, A), bool), c.actions[0], c.landmarks, c.size,
                                           c.agents_size)
    assert np.array_equal(pos, c.starts)                                     # zero actions: starts unchanged
    assert np.array_equal(done[np.arange(E), c.probe_idx[:, 0]], p.decision)
    parked = np.ones((E, A), bool)
    parked[np.arange(E), c.probe_idx[:, 0]] = False
    assert done[1::2][parked[1::2]].all() and not done[0::2][parked[0::2]].any()


def test_sentinel_geometry():
    for A, size, d, a in [(16, 5000, 0, 15), (32, 90000, 20, 5), (16, 1000, 0, 15)]:
        c = tc.sentinel_cases(A, size, d, a)
        pos, done = c.starts, np.zeros((2, A), bool)
        pos, _, cost, done, _ = no.collision_step(pos, done, c.actions[0], c.landmarks, size, 0.25)
        assert done[:, d].all() and not done[:, a].any() and (cost == 0).all()
        assert np.hypot(*(c.starts[0, d] - c.starts[0, a])) < 0.5
        if size > 4096:
            assert c.starts[0, d, 0] == 4096.0 * (d + 1)
