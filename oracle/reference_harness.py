"""Drive the UNMODIFIED reference (/root/reference) on injected states and recorded actions.

TEST INFRASTRUCTURE ONLY.  The run_* functions need the reference tree; where it is
absent, reference_side() serves the differential tests the reference outputs recorded in
tests/golden/reference_record.npz.  The ``-m gpu`` tests, smoke() and bench.py use
tests/golden/*.npz produced from these functions by tests/golden/make_golden.py.

The reference is imported read-only (no bytecode written).  ``matplotlib`` is absent
in this image and only needed by Buffer.save_results, so an empty stub module is
registered before importing safe_multi_agent_RL.buffer (buffer.py:2).
"""
from __future__ import annotations

import os
import sys
import types
import warnings

import numpy as np

REFERENCE_ROOT = os.environ.get("SMARL_REFERENCE_ROOT", "/root/reference")


def available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "envs", "coverage.py"))


_ns = None


def load():
    """Import the reference modules once; returns a namespace of its classes."""
    global _ns
    if _ns is not None:
        return _ns
    if not available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    sys.dont_write_bytecode = True
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    for name in ("matplotlib", "matplotlib.pyplot"):
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    warnings.filterwarnings("ignore", category=DeprecationWarning)
    import envs.coverage as coverage
    import envs.congestion as congestion
    import envs.collision_avoidance as collision
    from safe_multi_agent_RL.meta_agent import MetaAgent
    from safe_multi_agent_RL.buffer import Buffer
    from safe_multi_agent_RL.agent import ACAgent, AbstractAgent, PPOAgent
    _ns = types.SimpleNamespace(coverage=coverage, congestion=congestion, collision=collision,
                                MetaAgent=MetaAgent, Buffer=Buffer, ACAgent=ACAgent,
                                AbstractAgent=AbstractAgent, PPOAgent=PPOAgent)
    return _ns


RECORD = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden",
                      "reference_record.npz")
_record = None


def reference_side(key, live, e=None):
    """The reference's outputs for one test case: ``live()`` where the reference tree is present, else the entries
    ``<key>/<name>`` of tests/golden/reference_record.npz (made by tests/golden/make_reference_record.py, which states
    their provenance).  ``e`` selects one env of a case recorded per env."""
    global _record
    if available():
        return live()
    if _record is None:
        with np.load(RECORD) as g:
            _record = {k: g[k] for k in g.files}
    rec = {k[len(key) + 1:]: v for k, v in _record.items() if k.startswith(key + "/")}
    if not rec:
        raise KeyError(f"no recorded reference outputs for {key}")
    return rec if e is None else {k: v[e] for k, v in rec.items()}


def _f64(x):
    return np.asarray(x, dtype=np.float64)


def run_coverage_discrete(size, n_agents, starts, actions, weights=None, fieldview_size=None):
    """starts [A,2] ints, actions [T,A] ints -> dict of per-step traces (one env instance)."""
    ref = load()
    env = ref.coverage.CoverageDiscrete(size, n_agents, shuffle=False, weights=weights,
                                        fieldview_size=fieldview_size)
    for ag, s in zip(env.agents, starts):
        ag.start = [float(s[0]), float(s[1])]
    s0 = env.reset()
    T = len(actions)
    pos = np.zeros((T, n_agents, 2)); rew = np.zeros((T, n_agents))
    cost = np.zeros((T, n_agents)); done = np.zeros((T, n_agents), dtype=bool)
    for t in range(T):
        st, r, c, d = env.step([int(a) for a in actions[t]])
        pos[t] = _f64(st); rew[t] = _f64(r); cost[t] = _f64(c); done[t] = np.asarray(d, dtype=bool)
    return dict(state0=_f64(s0), pos=pos, reward=rew, cost=cost, done=done,
                fieldview=float(env.fieldview_size))


def run_coverage_float(kind, size, n_agents, starts, actions, weights=None, fieldview_size=None, coarseness=None):
    """kind 'continuous' (actions [T,A,2] floats) or 'discretized' (actions [T,A] ints 0..8)."""
    ref = load()
    np_state = np.random.get_state()
    if kind == "continuous":
        env = ref.coverage.CoverageContinuous(size, n_agents, shuffle=False, weights=weights,
                                              fieldview_size=fieldview_size, coarseness=coarseness)
    else:
        env = ref.coverage.CoverageDiscretized(size, n_agents, coarseness=coarseness, shuffle=False, weights=weights,
                                               fieldview_size=fieldview_size)
    np.random.set_state(np_state)
    for ag, s in zip(env.agents, starts):
        ag.start = [float(s[0]), float(s[1])]
    s0 = env.reset()
    T = len(actions)
    pos = np.zeros((T, n_agents, 2)); rew = np.zeros((T, n_agents)); cost = np.zeros((T, n_agents))
    for t in range(T):
        if kind == "continuous":
            act = [[[float(a[0]), float(a[1])]] for a in actions[t]]
        else:
            act = [int(a) for a in actions[t]]
        st, r, c, d = env.step(act)
        pos[t] = _f64(st); rew[t] = _f64(r); cost[t] = _f64(c)
        assert not any(d)
    return dict(state0=_f64(s0), pos=pos, reward=rew, cost=cost, fieldview=float(env.fieldview_size))


def run_congestion(size, n_agents, starts, actions, demand, noise=0.0, uniforms=None):
    """starts [A,2] ints (agent 0 is forced to (0,0) by the reference ctor; we inject all),
    actions [T,A] intended, uniforms [T,A,2] in [0,1) replayed through the env's
    ``random()`` (congestion.py:64,67: second draw consumed only when the first fails).
    Returns traces incl. the effective moves recovered from agent.edge."""
    ref = load()
    env = ref.congestion.Congestion(size, n_agents, noise=noise, shuffle=False)
    env.demand_rate = np.asarray(demand)
    for ag, s in zip(env.agents, starts):
        ag.start = [float(s[0]), float(s[1])]
    s0 = env.reset()
    T = len(actions)
    pos = np.zeros((T, n_agents, 2)); rew = np.zeros((T, n_agents))
    cost = np.zeros((T, 1)); done = np.zeros((T, n_agents), dtype=bool)
    con = np.zeros((T, n_agents)); edges = np.zeros((T, n_agents, 4))
    saved = ref.congestion.random
    try:
        for t in range(T):
            if uniforms is not None:
                # the env draws per agent in index order: u1, then u2 only if u1 >= 1-noise
                queue = []
                for a in range(n_agents):
                    u1, u2 = float(uniforms[t, a, 0]), float(uniforms[t, a, 1])
                    queue.append(u1)
                    if not (u1 < 1 - noise):
                        queue.append(u2)
                it = iter(queue)
                ref.congestion.random = lambda it=it: next(it)
            acts = [int(a) for a in actions[t]]
            st, r, c, d = env.step(acts)
            pos[t] = _f64(st); rew[t] = _f64(r); cost[t] = _f64(c); done[t] = np.asarray(d, dtype=bool)
            edges[t] = _f64([list(map(float, ag.edge)) for ag in env.agents])
            con[t] = _f64(env._congestions(acts))
    finally:
        ref.congestion.random = saved
    return dict(state0=_f64([list(map(float, s)) for s in s0]), pos=pos, reward=rew, cost=cost,
                done=done, congestions=con, edges=edges)


def run_collision(size, n_agents, starts, landmarks, actions, n_landmarks=1):
    """starts [A,2] f64, landmarks [L,2] f64, actions [T,A,2] (fp32-origin values as the
    reference's policies emit, agent.py:124-125) -> traces.  Follows main.py:29-52: stops
    after the step at which all agents are done; later steps are zero-filled, positions frozen."""
    ref = load()
    np_state = np.random.get_state()
    env = ref.collision.CollisionAvoidance(int(size), int(n_agents), n_landmarks=int(n_landmarks),
                                           shuffle=False)
    np.random.set_state(np_state)
    for ag, s in zip(env.agents, starts):
        ag.start = [float(s[0]), float(s[1])]
    env.landmarks = [[float(l[0]), float(l[1])] for l in landmarks]
    s0 = env.reset()
    T = len(actions)
    pos = np.zeros((T, n_agents, 2)); rew = np.zeros((T, n_agents))
    cost = np.zeros((T, 1)); done = np.zeros((T, n_agents), dtype=bool)
    active = np.zeros(T, dtype=bool)
    last_pos, last_done = _f64(s0), np.zeros(n_agents, dtype=bool)
    finished = False
    for t in range(T):
        if finished:
            pos[t] = last_pos; done[t] = last_done
            continue
        act = [[[float(a[0]), float(a[1])]] for a in actions[t]]   # [[dx,dy]] as agent.py emits
        st, r, c, d = env.step(act)
        pos[t] = _f64(st); rew[t] = _f64(r); cost[t] = _f64(c); done[t] = np.asarray(d, dtype=bool)
        active[t] = True
        last_pos, last_done = pos[t], done[t]
        if np.all(d):
            finished = True
    return dict(state0=_f64(s0), pos=pos, reward=rew, cost=cost, done=done, active=active)


class _Params:
    def __init__(self, gamma, thresholds):
        self.gamma = gamma
        self.thresholds = thresholds


def run_accounting(rewards, costs, lambdas0, gamma, thresholds, meta_lr, n_steps=None):
    """Feed per-step rewards [T][A] and costs [T][K] of ONE episode through the reference's
    MetaAgent.act / Buffer.append / Buffer.step / MetaAgent.step / MetaAgent.update and
    ACAgent/AbstractAgent.compute_returns (main.py:36-57,66).  ``n_steps`` truncates the
    episode (early break).  lambdas0 [K] is injected after construction."""
    ref = load()
    K = len(lambdas0)
    meta = ref.MetaAgent([1] * K, gamma, meta_lr, list(thresholds), start_learning_cycle=0)
    meta.lambdas = np.array(lambdas0, dtype=np.float64)
    buf = ref.Buffer(_Params(gamma, list(thresholds)), constrained=True)
    T = len(rewards) if n_steps is None else n_steps
    A = len(rewards[0])
    mods = []
    for t in range(T):
        r = [float(v) for v in rewards[t]]
        c = [float(v) for v in costs[t]]
        m = meta.act(c, r)
        mods.append(m)
        buf.append(r, m, c)
    buf.step()
    meta.step()
    G = np.zeros((T, A)); disc = np.zeros((T, A))
    for a in range(A):
        holder = types.SimpleNamespace(rewards=[m[a] for m in mods], gamma=gamma)
        G[:, a] = _f64(ref.ACAgent.compute_returns(holder))
        disc[:, a] = _f64(ref.AbstractAgent.compute_returns(holder))
    mean_sc = buf.mean_score()
    meta.update()
    return dict(mod_reward=_f64(mods), R=_f64(buf.scores[-1]), modR=_f64(buf.modified_scores[-1]),
                C=_f64(buf.constraints[-1]), G=G, disc=disc, lambdas_after=_f64(meta.lambdas),
                mean_violation=_f64(mean_sc[2]))


def run_ppo_returns(mod_rewards, gamma):
    """The reference's PPOAgent.step (agent.py:276-281) on one agent's modified rewards [T'] ->
    standardised discounted terms [T'] (torch float32).  The agent object is created without
    __init__ (no networks needed): step() only touches rewards / gamma / returns."""
    ref = load()
    agent = object.__new__(ref.PPOAgent)
    agent.rewards = [float(v) for v in mod_rewards]
    agent.gamma = gamma
    agent.returns = []
    agent.step()
    return np.asarray([float(v) for v in agent.returns], dtype=np.float64)
