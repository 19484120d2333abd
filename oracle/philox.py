"""Philox4x32-10 (Salmon et al., SC'11) in numpy.  TEST INFRASTRUCTURE ONLY.

The reference draws Congestion's action noise from Python's unseeded ``random``
(envs/congestion.py:4,64,67), so it has no reproducible stream to match.  The B200
path uses a counter-based generator keyed by the *global* env id, so results do not
depend on how envs are sharded over GPUs:

    out = philox4x32_10(counter=(env_lo, env_hi, t, agent >> 2 | episode << 3), key=(seed_lo, seed_hi))
    agent a uses the word w = out[a & 3]
    u1 = w * 2**-32,  u2 = (w mod 5 + 0.5) / 5     (both exact enough in f64: int(u2 * 5) == w mod 5)
    move = action if u1 < 1 - noise else int(u2 * 5)      (congestion.py:64-67)

In integers:  keep <=> w < ceil((1-noise) * 2**32);  replacement = w mod 5.  Conditional on the move
being replaced (w >= threshold), w mod 5 is uniform on 0..4 up to one count in 2**32 per outcome, the
same resolution a second 32-bit word would give, so one generator call serves four agents.
This file restates the generator so the test-suite can replay the very same
uniforms through the reference's ``random()`` hook and through the oracle.
"""
from __future__ import annotations

import numpy as np

M0 = np.uint64(0xD2511F53)
M1 = np.uint64(0xCD9E8D57)
W0 = 0x9E3779B9
W1 = 0xBB67AE85
MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """All arguments broadcastable integer arrays holding uint32 values; returns 4 uint32 arrays."""
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint64) & MASK for c in (c0, c1, c2, c3))
    c0, c1, c2, c3 = np.broadcast_arrays(c0, c1, c2, c3)
    k0 = int(k0) & 0xFFFFFFFF
    k1 = int(k1) & 0xFFFFFFFF
    for _ in range(10):
        p0 = M0 * c0
        p1 = M1 * c2
        hi0, lo0 = p0 >> np.uint64(32), p0 & MASK
        hi1, lo1 = p1 >> np.uint64(32), p1 & MASK
        c0, c1, c2, c3 = (hi1 ^ c1 ^ np.uint64(k0)), lo1, (hi0 ^ c3 ^ np.uint64(k1)), lo0
        k0 = (k0 + W0) & 0xFFFFFFFF
        k1 = (k1 + W1) & 0xFFFFFFFF
    return tuple(c.astype(np.uint32) for c in (c0, c1, c2, c3))


def congestion_words(seed, env_ids, t, n_agents, episode=0):
    """uint32 word w, [E, A], for global env ids ``env_ids`` at step ``t`` of episode ``episode``."""
    env_ids = np.asarray(env_ids, dtype=np.uint64)
    E = env_ids.shape[0]
    quads = (n_agents + 3) // 4
    c0 = (env_ids & MASK)[:, None]
    c1 = (env_ids >> np.uint64(32))[:, None]
    c2 = np.full((1, 1), t, dtype=np.uint64)
    c3 = np.arange(quads, dtype=np.uint64)[None, :] | np.uint64((int(episode) << 3) & 0xFFFFFFFF)
    o = philox4x32_10(c0, c1, c2, c3, seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)   # 4 x [E, quads]
    w = np.empty((E, 4 * quads), dtype=np.uint32)
    for q in range(4):
        w[:, q::4] = o[q]
    return w[:, :n_agents]


def congestion_uniforms(seed, env_ids, t, n_agents, episode=0):
    """The f64 uniforms (u1, u2) in [0,1) equivalent to the device's integer tests: feeding them to the
    reference's two ``random()`` calls (congestion.py:64,67) reproduces the device's moves."""
    w = congestion_words(seed, env_ids, t, n_agents, episode)
    return w.astype(np.float64) * 2.0 ** -32, ((w % np.uint32(5)).astype(np.float64) + 0.5) / 5.0


def keep_threshold(noise):
    """Smallest integer thr with  (w * 2**-32 < 1 - noise)  <=>  (w < thr)  for uint32 w."""
    import math
    from fractions import Fraction
    lim = Fraction(1 - noise) * (1 << 32)        # exact value of the f64 ``1 - noise`` times 2**32
    return min(1 << 32, max(0, math.ceil(lim)))


def start_uniforms(seed, env_ids, episode, rows):
    """53-bit uniforms (ux, uy), each [E, len(rows)], of the shuffle=True start draws: counter
    (env id, episode, row), key (seed lo, seed hi ^ "RSET"), numpy's random_sample bit recipe."""
    env_ids = np.asarray(env_ids, dtype=np.uint64)
    rows = np.asarray(rows, dtype=np.uint64)
    o = philox4x32_10((env_ids & MASK)[:, None], (env_ids >> np.uint64(32))[:, None],
                      np.full((1, 1), episode, dtype=np.uint64), rows[None, :],
                      seed & 0xFFFFFFFF, ((seed >> 32) & 0xFFFFFFFF) ^ 0x52534554)

    def u53(a, b):
        return ((a >> np.uint32(5)).astype(np.float64) * 67108864.0 + (b >> np.uint32(6)).astype(np.float64)) \
            * (1.0 / 9007199254740992.0)
    return u53(o[0], o[1]), u53(o[2], o[3])


def random_starts(kind, size, seed, env_ids, episode, n_rows, zoom=None, row_offset=0):
    """[E, n_rows, 2] starts: kind 0 floor(u*size); 1 same with row 0 at (0,0); 2 u*size;
    3 floor((u*size)*zoom)/zoom  (Agent.reset in the reference envs)."""
    ux, uy = start_uniforms(seed, env_ids, episode, np.arange(n_rows) + row_offset)
    xy = np.stack([ux * size, uy * size], axis=-1)
    if kind in (0, 1):
        xy = np.floor(xy)
        if kind == 1:
            xy[:, 0] = 0
    elif kind == 3:
        xy = np.floor(xy * zoom) / zoom
    return xy


def policy_words(seed, env_ids, t, n_agents, episode=0):
    """uint32 word w [E, A] of the discrete policy stream: Philox counter (env id lo, hi, t | episode << 16,
    agent >> 2 | (episode >> 16) << 3), key (seed lo, seed hi ^ "PLCY"); agent a takes word a & 3 of its block.  The
    episode's bits above 16 sit above the agent quad (at most 8 quads for 32 agents), so episode 65 536 does not repeat
    the stream of episode 0."""
    env_ids = np.asarray(env_ids, dtype=np.uint64)
    episode = int(episode)
    tw = (int(t) | (episode << 16)) & 0xFFFFFFFF
    ag = np.arange(n_agents, dtype=np.uint64)
    c3 = (ag >> np.uint64(2)) | np.uint64(((episode >> 16) << 3) & 0xFFFFFFFF)
    o = philox4x32_10((env_ids & MASK)[:, None], (env_ids >> np.uint64(32))[:, None], np.full((1, 1), tw, dtype=np.uint64),
                      c3[None, :], seed & 0xFFFFFFFF, ((seed >> 32) & 0xFFFFFFFF) ^ 0x504C4359)
    return np.stack(o, axis=0)[np.arange(n_agents) & 3, :, np.arange(n_agents)].T             # [E, A]: word a & 3


def policy_uniforms(seed, env_ids, t, n_agents, episode=0):
    """u [E, A] of smarl_policy_act_discrete in float64: u = ((w >> 8) + 0.5) * 2**-24 of the words of policy_words.
    The kernel forms u in float32 (policy_uniforms_f32), where k + 0.5 rounds to even for k = w >> 8 >= 2**23: off by
    2**-25 there, below the margin the tests allow, except at k = 2**24 - 1, where the kernel's u is 1 - 2**-24."""
    k = policy_words(seed, env_ids, t, n_agents, episode) >> np.uint32(8)
    return (k.astype(np.float64) + 0.5) / 16777216.0


def policy_uniforms_f32(seed, env_ids, t, n_agents, episode=0):
    """u [E, A] exactly as the kernel's float32 arithmetic forms it: fl(k + 0.5) * 2**-24 (k = w >> 8; k + 0.5 rounds
    to even for k >= 2**23 and to 2**24 at k = 2**24 - 1), clamped to at most 1 - 2**-24 so that u * sum stays below
    sum and a zero-probability last action is never drawn."""
    return policy_u_f32(policy_words(seed, env_ids, t, n_agents, episode) >> np.uint32(8))


def policy_u_f32(k):
    """The kernel's float32 uniform of k = w >> 8 (policy_uniforms_f32)."""
    u = (np.asarray(k).astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -24)
    return np.minimum(u, np.float32(1.0 - 2.0 ** -24))


def policy_sample(logits, u):
    """Inverse-CDF Categorical sample as the kernel draws it: logits [..., C] (float64), u [...]:
    a = #{c < C-1 : cumsum(e)[c] <= u * sum(e)}, e = exp(logits - max).  Returns (actions, log_prob of them,
    margin) where margin is the relative distance of u * sum(e) to the nearest CDF step (ties are measure-zero; the
    float32 kernel may legitimately differ where margin is below its rounding)."""
    logits = np.asarray(logits, dtype=np.float64)
    m = logits.max(axis=-1, keepdims=True)
    e = np.exp(logits - m)
    s = e.sum(axis=-1)
    cum = np.cumsum(e, axis=-1)[..., :-1]
    target = (np.asarray(u, dtype=np.float64) * s)[..., None]
    a = (cum <= target).sum(axis=-1)
    logp = np.take_along_axis(logits - m - np.log(s)[..., None], a[..., None], axis=-1)[..., 0]
    margin = np.abs(cum - target).min(axis=-1) / s
    return a, logp, margin


def gaussian_words(seed, env_ids, t, n_agents, episode=0):
    """uint32 words (wa, wb), each [E, A], of the Gaussian policy stream: Philox counter (env id lo, hi,
    t | episode << 16, agent >> 1 | (episode >> 16) << 4), key (seed lo, seed hi ^ "GAUS"); agent a takes words
    2 (a & 1) and 2 (a & 1) + 1.  The episode's bits above 16 sit above the agent pair (at most 16 pairs for 32 agents),
    so episode 65 536 does not repeat the stream of episode 0."""
    env_ids = np.asarray(env_ids, dtype=np.uint64)
    episode = int(episode)
    tw = (int(t) | (episode << 16)) & 0xFFFFFFFF
    ag = np.arange(n_agents)
    c3 = (ag.astype(np.uint64) >> np.uint64(1)) | np.uint64(((episode >> 16) << 4) & 0xFFFFFFFF)
    o = philox4x32_10((env_ids & MASK)[:, None], (env_ids >> np.uint64(32))[:, None], np.full((1, 1), tw, dtype=np.uint64),
                      c3[None, :], seed & 0xFFFFFFFF, ((seed >> 32) & 0xFFFFFFFF) ^ 0x47415553)
    w = np.stack(o, axis=0)                                                              # [4, E, A]
    return w[2 * (ag & 1), :, ag].T, w[2 * (ag & 1) + 1, :, ag].T


def gaussian_uniforms(seed, env_ids, t, n_agents, episode=0):
    """(u0, u1), each [E, A]: u = ((w >> 9) + 0.5) * 2**-23 of the words of gaussian_words (24 significant bits:
    exact in float32, so the kernel forms the same values; never 0 or 1)."""
    wa, wb = gaussian_words(seed, env_ids, t, n_agents, episode)
    return tuple(((w >> np.uint32(9)).astype(np.float64) + 0.5) / 8388608.0 for w in (wa, wb))


def gaussian_normals(seed, env_ids, t, n_agents, episode=0):
    """z [E, A, 2] of smarl_policy_act_gaussian from the uniforms of gaussian_uniforms;
    Box-Muller r = sqrt(-2 ln u0), z = (r cos 2 pi u1, r sin 2 pi u1) (float64 here)."""
    u0, u1 = gaussian_uniforms(seed, env_ids, t, n_agents, episode)
    r = np.sqrt(-2.0 * np.log(u0))
    return np.stack([r * np.cos(2.0 * np.pi * u1), r * np.sin(2.0 * np.pi * u1)], axis=-1)


def gaussian_sample(mu, var, z):
    """actions and log-probabilities as the kernel forms them: a = mu + sqrt(var) z, log N(a; mu, diag(var))."""
    mu, var, z = (np.asarray(x, dtype=np.float64) for x in (mu, var, z))
    a = mu + np.sqrt(var) * z
    logp = -0.5 * (((a - mu) ** 2 / var) + np.log(var)).sum(axis=-1) - np.log(2.0 * np.pi)
    return a, logp


# Global env ids whose policy words sit at the extremes of the uniforms, for seed EDGE_SEED and episode 0, found by a
# search over the first 2**25 ids (tests/test_policy_sampling_draws.py re-derives every entry; the GPU tests place them
# inside batches through env_offset).  Entries are (env id, agent, t).
EDGE_SEED = 77
# discrete stream (policy_words, 8 agents: both agent quads, every word slot): k = w >> 8
DISCRETE_TOP = [(14399409, 0, 0), (5068164, 1, 0), (13308236, 2, 0), (11493987, 4, 0), (12665387, 5, 0),
                (2342586, 7, 0), (16214439, 0, 1), (1484137, 3, 1), (14008471, 5, 1), (28475229, 6, 1)]   # k = 2**24 - 1
DISCRETE_BOTTOM = [(28550453, 0, 0), (11866442, 2, 0), (2229929, 4, 0), (4043212, 7, 0), (11228756, 1, 1),
                   (13522544, 3, 1), (7472350, 5, 1), (7714371, 6, 1)]                                     # k = 0
# (env id, agent, t, j): k = 2**24 - j, the top of the CDF where an action of probability ~1e-6 is drawn
DISCRETE_NEAR_TOP = [(3983378, 6, 0, 2), (1278034, 7, 1, 4), (179760, 1, 0, 6), (2403015, 2, 1, 8), (2811240, 0, 0, 10),
                     (6355444, 3, 1, 12), (4532832, 4, 0, 14), (8541136, 5, 1, 17), (1388300, 0, 0, 20),
                     (1982424, 7, 1, 26), (805129, 5, 0, 32), (169398, 5, 1, 38)]
# Gaussian stream (gaussian_words, 4 agents: both agent pairs), keyed by the uniform and w >> 9: 0 or 2**23 - 1
GAUSS_EDGES = {
    ("u0", 0): [(125380, 0, 0), (2698502, 1, 0), (3012936, 2, 0), (7978842, 3, 0), (7030430, 0, 1), (2871920, 1, 1)],
    ("u0", 2 ** 23 - 1): [(1246992, 0, 0), (2289924, 1, 0), (12656889, 2, 0), (3390058, 3, 0), (2160676, 3, 1)],
    ("u1", 0): [(208835, 0, 0), (415691, 1, 0), (16037746, 2, 0), (3081717, 3, 0), (7881140, 0, 1)],
    ("u1", 2 ** 23 - 1): [(209714, 0, 0), (4525523, 2, 0), (9812806, 3, 0), (8933202, 1, 1)],
}
