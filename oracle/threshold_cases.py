"""Inputs that put the CollisionAvoidance and CoverageContinuous env steps on their decision thresholds.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  The kernels decide the reference's square-root comparisons on
the squared value and take the square root only inside a narrow band around the threshold:

    action clip      collision_avoidance.py:113-117  norm > 1             q > 1, then sqrt
    landmark reach   :122-124   sqrt(qn) < agents_size                    qn against agents_size^2 (1 -+ 1e-9)
    colliding pair   :150-156   sqrt(q) < 2 agents_size                   q against (2 agents_size)^2 (1 -+ 1e-6)
    rescale          coverage.py:65-69  sqrt(sqrt(q)) > max_norm          q against max_norm^4 (1 -+ 1e-9)

Random inputs essentially never land in those bands.  The builders here search np.nextafter neighbourhoods and keep
the inputs whose float64 intermediates, computed with the oracle's own arithmetic (numpy_oracle), land where each
family needs them: on the threshold, one ulp either side, spread through the band on both sides of the reference's
decision, and where the squared comparison alone would decide wrong.  Every case carries what it claims
(``value``, ``decision``, ``squared``, ``in_band``) so that tests/test_threshold_cases.py can check the claim.

Collision families are built as probes (one to three agents per env and their landmarks) and laid out for any agent
count A >= 3 by ``layout``: the probe agents get random indices, the others are parked away from everything -- on a
grid (they stay alive) in half of the envs and exactly on an extra landmark (done after the first step, so that
episodes end early) in the other half.  Zero f32 actions leave float64 starts unchanged, so the geometry is placed
through the starts; the first step is the one on the thresholds.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

from .numpy_oracle import _fma

REACH_BAND = (0.999999999, 1.000000001)      # agents_size^2 * (1 -+ 1e-9), collision.cuh collision_env_step
PAIR_BAND = (0.999999, 1.000001)             # (2 agents_size)^2 * (1 -+ 1e-6)
RESCALE_BAND = (1.0 - 1e-9, 1.0 + 1e-9)      # max_norm^4 * (1 -+ 1e-9), coverage_float.cuh coverage_float_args
REACH_SIZES = (0.25, 0.1, 0.3, 1e-3)         # 0.25 has an exact square, the others do not


@dataclass
class Probes:
    """Per-env probe geometry of one family, independent of the agent count.

    pts [E, P, 2] f64 probe agent starts, act [E, P, 2] f32 their first actions, lms [E, Lp, 2] f64 the family's
    landmarks.  value / decision / squared / in_band [E]: the compared quantity of the env's probe, the reference's
    decision on it, the decision of the squared comparison alone and whether it lies inside the kernel's band.
    kind [E]: a label per env."""
    family: str
    size: int
    agents_size: float
    pts: np.ndarray
    act: np.ndarray
    lms: np.ndarray
    value: np.ndarray
    decision: np.ndarray
    squared: np.ndarray
    in_band: np.ndarray
    kind: np.ndarray
    park: tuple = (6.0, 6.0)       # parking landmark; the grid starts one gap up and right of it
    gap: float = 0.75


@dataclass
class Cases:
    """One batch of envs ready for BatchedCollisionAvoidance / numpy_oracle.collision_step."""
    family: str
    size: int
    agents_size: float
    starts: np.ndarray            # [E, A, 2] f64
    landmarks: np.ndarray         # [E, L, 2] f64
    actions: np.ndarray           # [T, E, A, 2] f32: the probes' actions at t = 0, zero afterwards
    probe_idx: np.ndarray = field(default=None)   # [E, P] agent index of each probe


def _neighbours(v, k, dtype=np.float64):
    """[..., 2k+1]: v and its k nextafter neighbours on either side."""
    v = np.asarray(v, dtype=dtype)
    out, up, dn = [v], v, v
    for _ in range(k):
        up = np.nextafter(up, dtype(np.inf))
        dn = np.nextafter(dn, dtype(-np.inf))
        out += [up, dn]
    return np.stack(out, axis=-1)


def _grid2(x, y, k, dtype=np.float64):
    """All (x', y') with x' among the 2k+1 neighbours of x and y' among those of y, flattened."""
    gx, gy = _neighbours(x, k, dtype), _neighbours(y, k, dtype)
    gx, gy = np.broadcast_arrays(gx[..., :, None], gy[..., None, :])
    return gx.reshape(-1), gy.reshape(-1)


def reach_qn(px, py, lx, ly):
    """numpy_oracle.collision_step's reach operand: fma(ay, ay, ax*ax), ax = px - lx, ay = py - ly."""
    ax, ay = np.subtract(px, lx), np.subtract(py, ly)
    return _fma(ay, ay, ax * ax)


def pair_q(xi, yi, xj, yj):
    """numpy_oracle.collision_step's pair operand: dx*dx + dy*dy (no fma)."""
    dx, dy = np.subtract(xi, xj), np.subtract(yi, yj)
    return dx * dx + dy * dy


def _select(value, decision, squared, lo, hi, thr, n_band):
    """Indices of a spread: every distinct value equal to thr and one ulp either side, the disagreements of the
    squared comparison, and up to n_band values inside [lo, hi) on each side of the decision (spread by rank)."""
    keep = []
    for t in (thr, np.nextafter(thr, -np.inf), np.nextafter(thr, np.inf)):
        keep += list(np.flatnonzero(value == t)[:6])
    keep += list(np.flatnonzero(squared != decision)[:2 * n_band])
    band = (value >= lo) & (value < hi)
    for side in (True, False):
        idx = np.flatnonzero(band & (decision == side))
        idx = idx[np.argsort(value[idx], kind="stable")]
        if len(idx):
            keep += list(idx[np.unique(np.linspace(0, len(idx) - 1, n_band).astype(int))])
    # just outside the band, where the squared comparison decides alone
    for edge, side in ((lo, True), (hi, False)):
        idx = np.flatnonzero((decision == side) & ~band)
        if len(idx):
            keep += list(idx[np.argsort(np.abs(value[idx] - edge), kind="stable")[:3]])
    return np.unique(np.asarray(keep, dtype=np.int64))


def reach_probes(agents_size, seed=0, n_band=12):
    """Landmark reach: one probe agent per env, qn on agents_size^2, one ulp either side and spread through the 1e-9
    band.  Landmarks at the origin give the probe's coordinates full resolution (ax = px exactly), so qn hits single
    ulps; landmarks at generic positions add the subtraction's rounding."""
    rng = np.random.default_rng(seed)
    a = float(agents_size)
    as2 = a * a
    lo, hi = as2 * REACH_BAND[0], as2 * REACH_BAND[1]
    pts, lms = [], []
    for origin in (True, False):
        n_dir = 60
        th = rng.uniform(0.05, np.pi / 2 - 0.05, n_dir)
        r = a * (1.0 + np.concatenate([[0.0], np.linspace(-0.7e-9, 0.7e-9, 9)]))
        th, r = np.broadcast_arrays(th[:, None], r[None, :])
        l = np.zeros((th.size, 2)) if origin else np.stack([1.5 + rng.random(th.size), 2.5 + rng.random(th.size)], 1)
        px, py = _grid2(l[:, 0] + r.reshape(-1) * np.cos(th.reshape(-1)),
                        l[:, 1] + r.reshape(-1) * np.sin(th.reshape(-1)), 2)
        lx = np.repeat(l[:, 0], 25)
        ly = np.repeat(l[:, 1], 25)
        pts.append(np.stack([px, py], 1))
        lms.append(np.stack([lx, ly], 1))
    pts, lms = np.concatenate(pts), np.concatenate(lms)
    qn = reach_qn(pts[:, 0], pts[:, 1], lms[:, 0], lms[:, 1])
    decision = np.sqrt(qn) < a
    squared = qn < as2
    k = _select(qn, decision, squared, lo, hi, as2, n_band)
    E = len(k)
    return Probes("reach", 12, a, pts[k, None], np.zeros((E, 1, 2), np.float32), lms[k, None], qn[k], decision[k],
                  squared[k], (qn[k] >= lo) & (qn[k] < hi), np.array(["reach"] * E))


def pair_probes(agents_size, seed=0, n_band=12, size=12, near=None, park=(6.0, 6.0)):
    """Colliding pairs: two probe agents per env at distance 2 agents_size: q on lim^2, one ulp either side and
    spread through the 1e-6 band.  ``near`` places the pairs at generic coordinates around that point (the f32
    screen's worst case near the field's far corner); otherwise half sit with one agent at the origin (full
    resolution) and half at generic coordinates."""
    rng = np.random.default_rng(seed)
    a = float(agents_size)
    lim = 2.0 * a
    lim2 = lim * lim
    lo, hi = lim2 * PAIR_BAND[0], lim2 * PAIR_BAND[1]
    base = []
    n = 600
    if near is None:
        base.append(np.zeros((n, 2)))
        base.append(np.stack([2.3 + rng.random(n), 1.7 + rng.random(n)], 1))
    else:
        base.append(np.asarray(near, dtype=np.float64)[None] - rng.random((2 * n, 2)) * 0.5)
    base = np.concatenate(base)
    th = rng.uniform(0.05, np.pi / 2 - 0.05, len(base)) + (0.0 if near is None else np.pi)   # towards the inside
    r = lim * (1.0 + rng.choice(np.concatenate([[0.0] * 4, np.linspace(-0.8e-6, 0.8e-6, 17)]), len(base)))
    xj, yj = _grid2(base[:, 0] + r * np.cos(th), base[:, 1] + r * np.sin(th), 2)
    xi, yi = np.repeat(base[:, 0], 25), np.repeat(base[:, 1], 25)
    q = pair_q(xi, yi, xj, yj)
    decision = np.sqrt(q) < lim
    squared = q < lim2
    k = _select(q, decision, squared, lo, hi, lim2, n_band)
    E = len(k)
    pts = np.stack([np.stack([xi[k], yi[k]], 1), np.stack([xj[k], yj[k]], 1)], 1)
    lms = np.repeat(np.asarray(park, dtype=np.float64)[None, None], E, 0)[:, :0]    # no probe landmark
    return Probes("pair", size, a, pts, np.zeros((E, 2, 2), np.float32), lms, q[k], decision[k], squared[k],
                  (q[k] >= lo) & (q[k] < hi), np.array(["pair"] * E), park=park)


def pair_special_probes(agents_size, seed=0):
    """Pairs that collide unless one agent is done, with a landmark each: (a) two agents clamped into the same
    corner (zero distance), (b) a pair 1.2 agents_size apart of which one agent sits on the reach threshold of its
    landmark (both sides of it), so the pair counts exactly when that agent is not done after the step."""
    rng = np.random.default_rng(seed)
    a = float(agents_size)
    reach = reach_probes(a, seed + 1, n_band=6)
    E = len(reach.value)
    p = reach.pts[:, 0]
    l = reach.lms[:, 0]
    d = (p - l) / np.maximum(np.linalg.norm(p - l, axis=1, keepdims=True), 1e-300)
    partner = p + 1.2 * a * d                          # further from the landmark than a, closer to p than 2a
    pts = np.stack([p, partner], 1)
    lms = l[:, None]
    q = pair_q(p[:, 0], p[:, 1], partner[:, 0], partner[:, 1])
    # corner: both agents clipped to unit moves towards (0, 0), clamped onto it (distance 0); their landmark is far
    n_c = 8
    c0 = rng.random((n_c, 2, 2)) * 0.3
    cact = (-(0.9 + rng.random((n_c, 2, 2))) * 1.3).astype(np.float32)
    clm = np.tile(np.array([[[3.0, 4.0]]]), (n_c, 1, 1))
    return Probes("pair_special", 12, a, np.concatenate([pts, c0]),
                  np.concatenate([np.zeros((E, 2, 2), np.float32), cact]), np.concatenate([lms, clm]),
                  np.concatenate([q, np.zeros(n_c)]), np.concatenate([~reach.decision, np.ones(n_c, bool)]),
                  np.concatenate([~reach.squared, np.ones(n_c, bool)]), np.concatenate([reach.in_band, np.zeros(n_c, bool)]),
                  np.array(["reach_pair"] * E + ["corner"] * n_c))


def clip_probes(seed=0):
    """Action clips: one probe agent per env with an f32 action whose q = dx^2 + dy^2 is exactly 1 (no clip), 1 + 2^-52
    (q > 1 but sqrt_rn(q) == 1: no division), 1 + 2^-51 (the smallest q whose norm exceeds 1), just below 1, and a
    few ulps around those, in all four quadrants and both component orders."""
    rng = np.random.default_rng(seed)
    big = [np.float32(1.0), np.float32(1.0 - 2.0 ** -24), np.float32(1.0 - 2.0 ** -23)]
    small = np.concatenate([[0.0, 2.0 ** -27, 2.0 ** -26, 1.2 * 2.0 ** -26, 1.5 * 2.0 ** -26, 2.0 ** -25],
                            np.sqrt(2.0 ** -23) * (1 + np.arange(-3, 4) * 2.0 ** -23),
                            np.sqrt(2.0 ** -22) * (1 + np.arange(-3, 4) * 2.0 ** -23)]).astype(np.float32)
    a, b = np.meshgrid(np.array(big, np.float32), small, indexing="ij")
    a, b = a.reshape(-1), b.reshape(-1)
    # a handful of generic directions too: f32 rounding of (cos, sin) around the unit circle
    th = rng.uniform(0, np.pi / 2, 400)
    ga, gb = _grid2(np.cos(th).astype(np.float32), np.sin(th).astype(np.float32), 1, np.float32)
    a, b = np.concatenate([a, ga]), np.concatenate([b, gb])
    q = a.astype(np.float64) ** 2 + b.astype(np.float64) ** 2
    keep = (np.abs(q - 1.0) <= 4 * 2.0 ** -52) | (np.arange(len(q)) < len(big) * len(small))
    keep &= np.abs(q - 1.0) < 1e-6
    a, b, q = a[keep], b[keep], q[keep]
    _, u = np.unique(np.stack([a, b], 1), axis=0, return_index=True)
    a, b, q = a[u], b[u], q[u]
    # quadrants and component order
    acts = []
    for sx, sy, swap in [(1, 1, False), (-1, 1, True), (-1, -1, False), (1, -1, True)]:
        x, y = (b, a) if swap else (a, b)
        acts.append(np.stack([sx * x, sy * y], 1))
    act = np.concatenate(acts).astype(np.float32)
    q = np.tile(q, 4)
    E = len(act)
    norm = np.sqrt(q)
    pts = np.stack([5.0 + rng.random(E), 2.0 + rng.random(E)], 1)[:, None]
    lms = np.broadcast_to(np.array([3.0, 0.5]), (E, 1, 2)).copy()
    kind = np.where(q == 1.0, "q_eq_1", np.where(q == 1 + 2.0 ** -52, "q_gt_1_norm_eq_1",
                    np.where(q == 1 + 2.0 ** -51, "first_clip", "near_1")))
    return Probes("clip", 12, 0.25, pts, act[:, None], lms, q, norm > 1, q > 1, q > 1, kind, park=(7.0, 6.0))


def rescale_actions(size, coarseness, n=300000, seed=0):
    """CoverageContinuous rescale (coverage.py:65-69): f32 action pairs whose q = dx^2 + dy^2 falls inside the kernel's
    max_norm^4 (1 -+ 1e-9) band, on both sides of sqrt(sqrt(q)) > max_norm, plus some just outside the band.
    Returns (act [n_cases, 2] f32, q, decision, in_band)."""
    rng = np.random.default_rng(seed)
    mn = np.sqrt(2) * size / coarseness             # coverage.py:66, as BatchedCoverageContinuous computes it
    m4 = (mn * mn) * (mn * mn)
    lo, hi = m4 * RESCALE_BAND[0], m4 * RESCALE_BAND[1]
    th = rng.uniform(0, 2 * np.pi, n)
    R = mn * mn
    a = (R * np.cos(th)).astype(np.float32)
    b = (R * np.sin(th)).astype(np.float32)
    q = a.astype(np.float64) ** 2 + b.astype(np.float64) ** 2
    decision = np.sqrt(np.sqrt(q)) > mn
    band = (q > lo) & (q <= hi)                    # the kernel evaluates the square roots for lo < q <= hi
    out = []
    for side in (True, False):
        idx = np.flatnonzero(band & (decision == side))
        idx = idx[np.argsort(q[idx], kind="stable")]
        out += list(idx[np.unique(np.linspace(0, len(idx) - 1, min(len(idx), 48)).astype(int))])
    for edge in (lo, hi):
        idx = np.flatnonzero(~band)
        out += list(idx[np.argsort(np.abs(q[idx] - edge), kind="stable")[:6]])
    k = np.unique(np.asarray(out, dtype=np.int64))
    return np.stack([a[k], b[k]], 1), q[k], decision[k], band[k]


def rescale_cases(size, coarseness, A, seed=0):
    """(starts [E, A, 2], actions [E, A, 2] f32, q [E, A], decision [E, A], in_band [E, A]) for CoverageContinuous:
    every agent of every env takes one band action, from the middle of the field so that no move is clamped."""
    act, q, dec, band = rescale_actions(size, coarseness, seed=seed)
    E = -(-len(act) // A)
    idx = np.arange(E * A) % len(act)
    rng = np.random.default_rng(seed + 1)
    starts = size / 2 + (rng.random((E, A, 2)) - 0.5) * 0.2
    return (starts, act[idx].reshape(E, A, 2), q[idx].reshape(E, A), dec[idx].reshape(E, A),
            band[idx].reshape(E, A))


def layout(pr: Probes, A, T=1, seed=0):
    """Cases for A agents: the probes at random distinct indices per env, the other agents parked (see the module
    docstring).  Landmarks: the family's, then the parking landmark."""
    rng = np.random.default_rng(seed)
    E, P, _ = pr.pts.shape
    assert A >= max(P, 3) and A <= 32
    park = np.asarray(pr.park, dtype=np.float64)
    gx, gy = np.meshgrid(np.arange(6), np.arange(6), indexing="ij")
    grid = park + pr.gap * (1 + np.stack([gx.reshape(-1), gy.reshape(-1)], 1))
    starts = np.empty((E, A, 2))
    actions = np.zeros((T, E, A, 2), np.float32)
    idx = np.stack([rng.permutation(A)[:P] for _ in range(E)])
    for e in range(E):
        starts[e] = park if e % 2 else grid[:A]
        starts[e, idx[e]] = pr.pts[e]
        actions[0, e, idx[e]] = pr.act[e]
    landmarks = np.concatenate([pr.lms, np.broadcast_to(park, (E, 1, 2))], 1)
    assert np.all((starts >= 0) & (starts <= pr.size))
    return Cases(pr.family, pr.size, pr.agents_size, starts, landmarks, actions, idx)


def clip_overflow_cases(A, E=256, T=3, seed=0):
    """Every action of every env and step longer than 1: a warp posts 32 x A clips per step, more than the 64
    compaction slots from A = 3 on."""
    rng = np.random.default_rng(seed)
    size = 40
    starts = 10 + rng.random((E, A, 2)) * 20
    landmarks = rng.random((E, 1, 2)) * size
    th = rng.uniform(0, 2 * np.pi, (T, E, A))
    r = 1.0 + 1e-6 + rng.random((T, E, A)) * 2
    actions = np.stack([r * np.cos(th), r * np.sin(th)], -1).astype(np.float32)
    assert (actions.astype(np.float64) ** 2).sum(-1).min() > 1
    return Cases("clip_overflow", size, 0.25, starts, landmarks, actions)


def sentinel_cases(A, size, done_agent, alive_agent, T=2):
    """A done agent and an alive one 0.4 apart (< 2 agents_size = 0.5) at the point (4096 (done_agent + 1), 0) -- where
    a done agent once sat as a partner in the lane-cooperative f32 screen -- or at the same relative geometry on a
    smaller field.  The done agent sits on a landmark (done after the first step), the alive one 0.4 from it (not
    done); every other agent is parked far apart.  The reference counts no collision: the pair has a done agent."""
    x = 4096.0 * (done_agent + 1)
    if x + 1 > size:
        x = size / 2
    starts = np.stack([100.0 + 10.0 * np.arange(A), np.full(A, 100.0)], 1)
    starts[done_agent] = (x, 0.0)
    starts[alive_agent] = (x + 0.4, 0.0)
    starts = np.stack([starts, starts[::1]])
    starts[1, alive_agent] = (x + 0.6, 0.0)          # a control env: the pair never collides
    landmarks = np.array([[[x, 0.0]]] * 2)
    return Cases("sentinel", size, 0.25, starts, landmarks, np.zeros((T, 2, A, 2), np.float32))
