"""The CollisionAvoidance and CoverageContinuous env steps on inputs at their decision thresholds (built by
oracle/threshold_cases.py), through every kernel instantiation, against numpy_oracle.

The kernels decide the reference's square-root comparisons (action clip, landmark reach, colliding pair, rescale) on
squared values and take the square root only inside narrow bands; random inputs never reach those bands.  Bars as in
test_gpu_parity.py: positions, done flags, costs and episode lengths bit-exact, step rewards == the oracle's float64
reward rounded to f32, fused-rollout sums within 1e-5.

Instantiations forced through smarl_set_kernel_variant (lanes 0 = one thread per env):
    A = 3, 7        one-thread step kernel, clips compacted over the warp (SMARL_COLL_COMPACT_MAX_A = 7)
    A = 8, 11       one-thread step kernel, clips inline
    A = 12, 16      one-thread step kernel, pair loop screened in f32 (kPairPrefilterA = 12)
    A = 9..32       lane-cooperative step (lanes 2, 4), including A not divisible by the lane count
    A = 3, 8 / 12   one-thread fused rollout with compacted / inline clips, g_mode 0-2
    A = 9..31       lane-cooperative fused rollout (lanes 2, 4), g_mode 0-2
The cooperative kernels pick compacted or inline clips from SMARL_COLL_COMPACT once per process; a child process runs
them again with the instantiation the default does not use."""
import functools
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import test_gpu_parity as tp
import test_gpu_policy_rollout as tpr
from oracle import numpy_oracle as no
from oracle import threshold_cases as tc
from safe_multiagent_rl_b200 import _lib

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

STEP_PATHS = [(3, 0), (7, 0), (8, 0), (11, 0), (12, 0), (16, 0), (9, 2), (13, 2), (16, 2), (32, 2), (13, 4), (16, 4),
              (22, 4), (31, 4)]
ROLLOUT_PATHS = [(3, 0), (8, 0), (12, 0), (9, 2), (13, 2), (16, 4), (31, 4)]
COOP_STEP = [p for p in STEP_PATHS if p[1]]
COOP_ROLLOUT = [p for p in ROLLOUT_PATHS if p[1]]


@functools.lru_cache(maxsize=None)
def families(A, T):
    """Every Collision family laid out for A agents, T steps (the probes act at t = 0)."""
    fs = [tc.layout(tc.reach_probes(a), A, T, seed=A) for a in tc.REACH_SIZES]
    fs += [tc.layout(tc.pair_probes(a), A, T, seed=A + 1) for a in (0.25, 0.1, 0.3)]
    fs += [tc.layout(tc.pair_special_probes(a), A, T, seed=A + 2) for a in (0.25, 0.1)]
    fs += [tc.layout(tc.clip_probes(), A, T, seed=A + 3)]
    fs += [tc.layout(tc.pair_probes(1e-3, size=s, near=(s, s), park=(10.0, 10.0)), A, T, seed=A + 4) for s in (200, 5000)]
    fs.append(tc.clip_overflow_cases(A, T=T, seed=A))
    return fs


def make_env(c):
    s = tp.smarl()
    E, A, _ = c.starts.shape
    return s.BatchedCollisionAvoidance(c.size, A, n_envs=E, n_landmarks=c.landmarks.shape[1], starts=c.starts,
                                       landmarks=c.landmarks, agents_size=c.agents_size)


def check_steps(c):
    T, E, A, _ = c.actions.shape
    env = make_env(c)
    env.reset()
    pos, done = c.starts.copy(), np.zeros((E, A), dtype=bool)
    for t in range(T):
        _, r, cost, d = env.step(c.actions[t])
        pos, r_o, c_o, done, _ = no.collision_step(pos, done, c.actions[t].astype(np.float64), c.landmarks, c.size,
                                                   c.agents_size)
        where = (c.family, c.agents_size, c.size, t)
        assert np.array_equal(env.state().cpu().numpy(), pos), where
        assert np.array_equal(d.cpu().numpy().astype(bool), done), where
        assert np.array_equal(cost.cpu().numpy(), c_o.astype(np.int64)), where
        assert np.array_equal(r.cpu().numpy(), r_o.astype(np.float32)), where


def check_rollout(c, g_mode):
    T, E, A, _ = c.actions.shape
    env = make_env(c)
    gamma, lam_np, thr = 0.97, np.array([0.5]), np.array([1.0])
    pos, done = c.starts.copy(), np.zeros((E, A), dtype=bool)
    n_active = np.zeros(E, dtype=np.int64)

    def step_fn(t):
        nonlocal pos, done
        pos, r, cost, done, active = no.collision_step(pos, done, c.actions[t].astype(np.float64), c.landmarks, c.size,
                                                       c.agents_size)
        n_active[:] += active
        return r.astype(np.float32).astype(np.float64), cost
    want = no.rollout(step_fn, T, gamma, lam_np)
    want_G = {0: None, 1: want["G"], 2: no.discounted_terms(want["mod_reward"], gamma)}[g_mode]
    act_k = tp.kernel_layout(c.actions.reshape(T, E, 2 * A), env.ld)
    out = env.rollout(act_k, lambdas=torch.as_tensor(lam_np, device="cuda"), gamma=gamma, thresholds=thr,
                      g_mode=g_mode)
    where = (c.family, c.agents_size, c.size)
    assert np.array_equal(env.state().cpu().numpy(), pos), where
    assert np.array_equal(env.agent_done[:, :E].t().cpu().numpy().astype(bool), done), where
    assert np.array_equal(out["n_active"].cpu().numpy(), n_active), where
    tp.check_products(out, want, want_G, thr, E, np.max(np.abs(want["modR"])))


def run_steps(A, lanes):
    with _lib.kernel_variant(_lib.ENV_COLLISION, lanes):
        for c in families(A, 2):
            check_steps(c)


def run_rollouts(A, lanes, g_modes=(0, 1, 2)):
    with _lib.kernel_variant(_lib.ENV_COLLISION, lanes):
        for g_mode in g_modes:
            for c in families(A, 3):
                check_rollout(c, g_mode)


@pytest.mark.parametrize("A,lanes", STEP_PATHS)
def test_collision_step_at_thresholds(A, lanes):
    run_steps(A, lanes)


@pytest.mark.parametrize("A,lanes", ROLLOUT_PATHS)
@pytest.mark.parametrize("g_mode", [0, 1, 2])
def test_collision_fused_rollout_at_thresholds(A, lanes, g_mode):
    run_rollouts(A, lanes, (g_mode,))


@pytest.mark.parametrize("compact,kind", [("1", "step"), ("0", "rollout")])
def test_collision_coop_other_clip_instantiation(compact, kind):
    """SMARL_COLL_COMPACT is read once per process: 1 compacts the cooperative step's clips (off by default), 0 keeps
    the cooperative rollout's inline (compacted by default)."""
    paths = COOP_STEP if kind == "step" else COOP_ROLLOUT
    fn = "run_steps" if kind == "step" else "run_rollouts"
    code = (f"import sys; sys.path[:0] = [{ROOT!r}, {os.path.join(ROOT, 'tests')!r}]\n"
            "import test_gpu_thresholds as t\n"
            f"for A, lanes in {paths!r}:\n    t.{fn}(A, lanes)\n"
            "print('threshold cases ok')\n")
    env = dict(os.environ, SMARL_COLL_COMPACT=compact)
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=ROOT, timeout=3000)
    assert out.returncode == 0 and "threshold cases ok" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]


@pytest.mark.parametrize("lanes", [0, 2, 4])
@pytest.mark.parametrize("A,size,done_agent,alive_agent", [(16, 5000, 0, 15), (32, 90000, 20, 5), (16, 1000, 0, 15),
                                                            (13, 5000, 0, 12)])
def test_done_partner_is_never_counted(lanes, A, size, done_agent, alive_agent):
    """A done agent and an alive one 0.4 apart (inside 2 agents_size): the reference counts no collision for a pair
    with a done agent (collision_avoidance.py:150-156).  On fields of 4096 and more the pair sits where the
    lane-cooperative screen once put done partners, (4096 (i + 1), 0); the field of 1000 is the control."""
    c = tc.sentinel_cases(A, size, done_agent, alive_agent, T=3)
    with _lib.kernel_variant(_lib.ENV_COLLISION, lanes):
        env = make_env(c)
        env.reset()
        for t in range(3):
            _, _, cost, d = env.step(c.actions[t])
            assert int(cost.abs().sum()) == 0, (t, cost.cpu().numpy().ravel())
            assert bool(d[:, done_agent].all()) and not bool(d[:, alive_agent].any())
        check_steps(c)
        for g_mode in (0, 1, 2):
            check_rollout(c, g_mode)


def threshold_landmarks(p1, agents_size, seed):
    """Landmarks [E, A, 2], landmark i on the reach threshold of agent i's position p1 [E, A, 2]: in the 1e-9 band,
    alternately below and above the reference decision, or as close to it as the coordinates allow."""
    rng = np.random.default_rng(seed)
    E, A, _ = p1.shape
    a = agents_size
    as2 = a * a
    lo, hi = as2 * tc.REACH_BAND[0], as2 * tc.REACH_BAND[1]
    px = np.repeat(p1.reshape(-1, 2), 25 * 9, 0)
    th = rng.uniform(0, 2 * np.pi, (E * A, 9))
    r = a * (1 + np.linspace(-0.5e-9, 0.5e-9, 9))[None]
    lx, ly = tc._grid2((p1.reshape(-1, 1, 2)[..., 0] - r * np.cos(th)).reshape(-1),
                       (p1.reshape(-1, 1, 2)[..., 1] - r * np.sin(th)).reshape(-1), 2)
    qn = tc.reach_qn(px[:, 0], px[:, 1], lx, ly).reshape(E * A, -1)
    lx, ly = lx.reshape(E * A, -1), ly.reshape(E * A, -1)
    want = (np.arange(E * A) % 2 == 0)
    dec = np.sqrt(qn) < a
    band = (qn >= lo) & (qn < hi)
    score = np.where(band & (dec == want[:, None]), 0.0, 1.0) + np.abs(qn / as2 - 1)
    k = np.argmin(score, axis=1)
    rows = np.arange(E * A)
    lms = np.stack([lx[rows, k], ly[rows, k]], 1).reshape(E, A, 2)
    return lms, band[rows, k].reshape(E, A), dec[rows, k].reshape(E, A)


@pytest.mark.parametrize("A", [3, 8])
def test_policy_rollout_reach_at_thresholds(A):
    """The on-policy Collision rollout samples its actions itself.  With shuffle=False the landmarks are not observed
    and policy_rollout does not advance the policy's episode, so a first run gives the post-step positions, landmarks
    are then placed on the reach thresholds of those positions, and a second run lands the same samples on them."""
    E, T, size, agents_size = 257, 4, 6, 0.25
    rng = np.random.default_rng(A)
    starts = 1 + rng.random((E, A, 2)) * (size - 2)
    lm0 = np.full((E, A, 2), 100.0)
    env, pol = tpr.make(A, E, size=size, L=A, agents_size=agents_size, seed=A, starts=starts, landmarks=lm0)
    env.policy_rollout(pol, 1)
    p1 = env.state().cpu().numpy()
    lms, band, dec = threshold_landmarks(p1, agents_size, A)
    assert band.mean() > 0.9 and dec[band].any() and (~dec[band]).any()
    env_p, pol_p = tpr.make(A, E, size=size, L=A, agents_size=agents_size, seed=A, starts=starts, landmarks=lms)
    env_c, pol_c = tpr.make(A, E, size=size, L=A, agents_size=agents_size, seed=A, starts=starts, landmarks=lms)
    lam = torch.tensor([0.5], dtype=torch.float64, device="cuda")
    out = env_p.policy_rollout(pol_p, T, lambdas=lam, gamma=0.97, thresholds=[1.0], g_mode=1)
    _, act, _ = tpr.closed_loop(env_c, pol_c, T, lam)
    assert torch.equal(out["actions_"][:, :, :E], act)
    assert torch.equal(env_p.pos_x[:, :E], env_c.pos_x[:, :E]) and torch.equal(env_p.pos_y[:, :E], env_c.pos_y[:, :E])
    assert torch.equal(env_p.agent_done[:, :E], env_c.agent_done[:, :E])
    assert torch.equal(out["n_active"], env_c.episode_len[:E])
    # the oracle on the recorded actions
    actions = out["actions"].cpu().numpy().transpose(0, 2, 1, 3)           # [T, E, A, 2]
    # the second run's first samples are the first run's: its post-step positions are the ones the landmarks fit
    assert np.array_equal(no.collision_step(starts, np.zeros((E, A), bool), actions[0].astype(np.float64), lm0, size,
                                            agents_size)[0], p1)
    pos, done, n_active, C = starts.copy(), np.zeros((E, A), bool), np.zeros(E, np.int64), np.zeros(E, np.int64)
    for t in range(T):
        pos, _, c_o, new_done, active = no.collision_step(pos, done, actions[t].astype(np.float64), lms, size, agents_size)
        if t == 0:
            # the reach decisions of the thresholds, for the agents no other landmark is near
            d_other = np.linalg.norm(p1[:, :, None] - lms[:, None], axis=-1) + np.where(np.eye(A, dtype=bool), 1e9, 0)
            clean = d_other.min(-1) > 2 * agents_size
            assert clean.mean() > 0.5 and np.array_equal(new_done[clean], dec[clean])
        done = new_done
        n_active += active
        C += c_o[:, 0].astype(np.int64)
    assert np.array_equal(env_p.state().cpu().numpy(), pos)
    assert np.array_equal(env_p.agent_done[:, :E].t().cpu().numpy().astype(bool), done)
    assert np.array_equal(out["n_active"].cpu().numpy(), n_active)
    assert np.array_equal(out["C"].cpu().numpy().reshape(-1), C)


# ----------------------------------------------------------------------------- CoverageContinuous rescale
@pytest.mark.parametrize("size,coarseness", [(5, 6), (10, 7)])
@pytest.mark.parametrize("A", [3, 8])
def test_coverage_continuous_rescale_at_thresholds(size, coarseness, A):
    s = tp.smarl()
    starts, act, q, dec, band = tc.rescale_cases(size, coarseness, A)
    E = starts.shape[0]
    assert (band & dec).any() and (band & ~dec).any()
    T = 2
    actions = np.zeros((T, E, A, 2), np.float32)
    actions[0] = act
    w = (1.0 + (np.arange(A) % 3)).tolist()
    fv = no.coverage_fieldview(size, A)
    env = s.BatchedCoverageContinuous(size, A, n_envs=E, weights=w, coarseness=coarseness, starts=starts)
    env.reset()
    pos = starts.copy()
    for t in range(T):
        _, r, c, _ = env.step(actions[t])
        pos, r_o, c_o, _ = no.coverage_continuous_step(pos, actions[t].astype(np.float64), size, fv, w, coarseness,
                                                       exact_pow=False)
        assert np.array_equal(env.state().cpu().numpy(), pos), t
        assert np.array_equal(r.cpu().numpy(), r_o.astype(np.float32)), t
        assert np.array_equal(c.cpu().numpy(), c_o.astype(np.float32)), t
    # the rescaled moves really differ from the unscaled ones: the decision is visible in the positions
    moved = (pos - starts)
    assert np.all((np.hypot(moved[..., 0], moved[..., 1]) < np.hypot(act[..., 0], act[..., 1]) - 1e-3) == dec)
    for g_mode in (0, 1, 2):
        env2 = s.BatchedCoverageContinuous(size, A, n_envs=E, weights=w, coarseness=coarseness, starts=starts)
        lam_np, gamma = np.linspace(0.1, 0.3, A), 0.99
        pos2 = starts.copy()

        def step_fn(t):
            nonlocal pos2
            pos2, r_, c_, _ = no.coverage_continuous_step(pos2, actions[t].astype(np.float64), size, fv, w, coarseness,
                                                          exact_pow=False)
            return r_.astype(np.float32).astype(np.float64), c_.astype(np.float32).astype(np.float64)
        want = no.rollout(step_fn, T, gamma, lam_np)
        out = env2.rollout(tp.kernel_layout(actions.reshape(T, E, 2 * A), env2.ld),
                           lambdas=torch.as_tensor(lam_np, device="cuda"), gamma=gamma, thresholds=[1.0] * A,
                           g_mode=g_mode)
        assert np.array_equal(env2.state().cpu().numpy(), pos2)
        scale = np.abs(want["modR"]).max()
        tp.close(out["R"].cpu().numpy(), want["R"], scale)
        tp.close(out["modR"].cpu().numpy(), want["modR"], scale)
        tp.close(out["C"].cpu().numpy(), want["C"], np.abs(want["C"]).max())
