"""Write tests/golden/reference_record.npz: the reference's side of every case of tests/test_oracle_vs_reference.py
and tests/test_ctor_rng_order.py, so that those comparisons run where the reference tree is absent:

    python tests/golden/make_reference_record.py

Provenance.  The values are computed here by the numpy oracle (env steps, accounting, PPO returns) and by the
product's BatchedBuffer / default_starts (Buffer files, ctor draws), on the seeded inputs the tests draw.  On exactly
these inputs the live differential tests compared those computations with the unmodified reference and passed
(bit-exact where the tests use array_equal, within their stated tolerances elsewhere): the CPU suite passed in full,
80 tests, with the reference mounted at commit dbcadfd (profiles/r02/SUMMARY.md, section H), and neither the tests nor
oracle/, envs/ or rollout.py changed between that commit and the one that wrote this record.  Where the reference
tree is present the tests compare against it live instead of against this record.
"""
import argparse
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import numpy_oracle as no  # noqa: E402

COVERAGE_DISCRETE = [(5, 3, 50, None, 0), (32, 16, 20, 8.0, 1), (8, 5, 30, None, 2), (64, 32, 5, None, 3),
                     (3, 2, 40, 10.0, 4)]
CONGESTION = [(3, 3, 10, 0.0, 0), (3, 8, 100, 0.1, 1), (10, 8, 40, 0.1, 2), (2, 6, 60, 0.5, 3), (5, 32, 8, 0.3, 4)]
COLLISION = [(5, 3, 1, 50, 0), (2, 5, 1, 20, 1), (5, 8, 3, 30, 2), (3, 12, 2, 25, 3)]
ACCOUNTING = [(3, 3, 50, 0.999, 0), (8, 1, 100, 0.9, 1), (16, 16, 50, 0.999, 2), (3, 1, 7, 0.99, 3)]
COVERAGE_CONTINUOUS = [(5, 3, 40, None, 0), (5, 3, 40, 6, 1), (10, 8, 15, 20, 2), (3, 5, 30, 2, 3)]
COVERAGE_DISCRETIZED = [(5, 3, 40, 20, 0), (5, 3, 40, 6, 1), (10, 8, 15, 7, 2), (3, 4, 30, 3, 3)]
PPO = [(50, 0.999), (8, 0.99), (100, 0.9), (2, 0.5)]
CTOR = [(0, 5, 3, 4), (7, 32, 16, 3), (11, 9, 1, 5)]


def case(kind, params):
    """Record key prefix of one parametrised case, e.g. ``coverage_discrete/5,3,50,None,0``."""
    return kind + "/" + ",".join(str(p) for p in params)


def stack(traces):
    return {k: np.stack([t[k] for t in traces]) for k in traces[0]}


def coverage_discrete(size, A, T, fv, seed):
    rng = np.random.default_rng(seed)
    weights = (1.0 + (np.arange(A) % 3)).tolist()
    lut = no.coverage_penalty_lut(size, no.coverage_fieldview(size, A, fv))
    traces = []
    for e in range(6):
        starts = np.floor(rng.random((A, 2)) * size).astype(np.int64)
        if e == 0:
            starts[:] = size - 1
        actions = rng.integers(0, 5, size=(T, A))
        pos, tr = starts[None], {"pos": [], "reward": [], "cost": [], "done": []}
        for t in range(T):
            pos, r, c, d = no.coverage_discrete_step(pos, actions[t][None], size, lut, weights)
            for k, v in zip(tr, (pos[0].astype(np.int16), r[0], c[0].astype(np.int8), d[0])):
                tr[k].append(v)
        traces.append({k: np.stack(v) for k, v in tr.items()})
    return stack(traces)


def congestion(size, A, T, noise, seed):
    rng = np.random.default_rng(seed)
    demand = rng.random((size + 1, size + 1)) * 8 + 2
    if size == 3:
        demand = np.array([[2, 2, 4, 4], [3, 6, 10, 5], [3, 8, 3, 4], [4, 6, 7, 8]])
    traces = []
    for e in range(4):
        starts = np.floor(rng.random((A, 2)) * size).astype(np.int64)
        starts[0] = 0
        actions = rng.integers(0, 5, size=(T, A))
        u = rng.random((T, A, 2))
        pos, tr = starts[None], {"pos": [], "edges": [], "congestions": [], "reward": [], "cost": []}
        for t in range(T):
            moves = no.congestion_noise_moves(actions[t][None], u[t, :, 0][None], u[t, :, 1][None], noise)
            old = pos
            pos, r, c, d, con = no.congestion_step(pos, actions[t][None], moves, size, demand)
            for k, v in zip(tr, (pos[0], np.concatenate([old, pos], axis=2)[0], con[0], r[0], c[0])):
                tr[k].append(v)
        traces.append({k: np.stack(v) if k == "reward" else np.stack(v).astype(np.int16) for k, v in tr.items()})
    return stack(traces)


def collision(size, A, L, T, seed):
    rng = np.random.default_rng(seed)
    traces = []
    for e in range(6):
        starts = rng.random((A, 2)) * size
        landmarks = rng.random((L, 2)) * size
        actions = rng.normal(0, 0.5, size=(T, A, 2)).astype(np.float32).astype(np.float64)
        if e == 1:
            actions = np.repeat(((landmarks[0][None] - starts) / 6).astype(np.float32)[None], T, 0).astype(np.float64)
        if e == 2:
            starts = np.clip(landmarks[0][None] + rng.normal(0, 0.4, size=(A, 2)), 0, size)
        pos, done = starts[None], np.zeros((1, A), dtype=bool)
        tr = {"active": [], "pos": [], "done": [], "cost": [], "reward": []}
        for t in range(T):
            pos, r, c, done, active = no.collision_step(pos, done, actions[t][None], landmarks[None], size)
            for k, v in zip(tr, (active[0], pos[0], done[0], c[0], r[0])):
                tr[k].append(v)
        traces.append({k: np.stack(v) for k, v in tr.items()})
    return stack(traces)


def accounting(A, K, T, gamma, seed):
    rng = np.random.default_rng(seed)
    rewards = rng.normal(-3, 4, size=(T, A))
    costs = rng.integers(0, 3, size=(T, K)).astype(np.float64)
    lam = rng.random(K)
    thr = rng.random(K) * 10
    mod = no.modified_reward(rewards[:, None, :], costs[:, None, :], lam)
    C = no.episode_cost_sums(costs[:, None, :])[0]
    return {"mod_reward": mod[:, 0], "R": no.episode_returns(rewards[:, None, :], gamma)[0],
            "modR": no.episode_returns(mod, gamma)[0], "C": C, "G": no.reward_to_go(mod, gamma)[:, 0],
            "disc": no.discounted_terms(mod, gamma)[:, 0], "lambdas_after": no.lambda_update(lam, C, thr, 0.05),
            "mean_violation": C - thr}


def coverage_float(kind, size, A, T, coarse, seed):
    rng = np.random.default_rng(seed)
    w = (1.0 + (np.arange(A) % 3)).tolist()
    fv = no.coverage_fieldview(size, A)
    traces = []
    for e in range(4):
        if kind == "continuous":
            starts = rng.random((A, 2)) * size
            actions = rng.normal(0, 0.8, size=(T, A, 2)).astype(np.float32).astype(np.float64)
        else:
            zoom = coarse / size
            starts = np.floor(rng.random((A, 2)) * size * zoom) / zoom
            actions = rng.integers(0, 9, size=(T, A))
        pos, tr = starts[None], {"pos": [], "reward": [], "cost": []}
        for t in range(T):
            if kind == "continuous":
                pos, r, c, _ = no.coverage_continuous_step(pos, actions[t][None], size, fv, w, coarse)
            else:
                pos, r, c, _ = no.coverage_discretized_step(pos, actions[t][None], size, coarse, fv, w)
            for k, v in zip(tr, (pos[0], r[0], c[0])):
                tr[k].append(v)
        traces.append({k: np.stack(v) for k, v in tr.items()})
    return stack(traces)


def ppo():
    rng = np.random.default_rng(0)
    return {case("ppo", p) + "/returns": no.ppo_standardised_returns(rng.normal(-3, 4, size=p[0])[:, None, None],
                                                                     p[1])[:, 0, 0] for p in PPO}


def buffer_files():
    """BatchedBuffer's files and per-batch series for the inputs of test_batched_buffer_save_results_matches_reference_files."""
    import torch

    from safe_multiagent_rl_b200.rollout import BatchedBuffer
    rng = np.random.default_rng(5)
    A, K, T, batches, bsz = 3, 2, 7, 4, 5
    params = argparse.Namespace(gamma=0.95, thresholds=[1.5, 2.0], batch_size=bsz, n_agents_learning_cycles=1,
                                environment="ExploreDiscrete", size=5, n_agents=A, numpy_seed=3, torch_seed=4,
                                algo="AC")
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as d:
        os.chdir(d)
        try:
            mine = BatchedBuffer(params, constrained=True)
            for b in range(batches):
                rew = rng.normal(size=(T, bsz, A))
                cost = rng.integers(0, 3, size=(T, bsz, K)).astype(np.float64)
                lam = rng.random(K)
                mod = rew - (cost @ lam)[:, :, None]
                for t in range(T):
                    mine.append(torch.from_numpy(rew[t]), torch.from_numpy(mod[t]), torch.from_numpy(cost[t]))
                mine.step()
                mine.append_lambdas(lam)
            out = mine.save_results()
            rec = {n: np.load(os.path.join(out, n + ".npy")) for n in ("constr3", "scores3", "lambdas")}
            rec["params_json"] = np.array(open(os.path.join(out, "params.json")).read())
        finally:
            os.chdir(cwd)
    rec["batch_scores"], rec["batch_means"] = (np.asarray(x) for x in mine.batch_scores())
    rec["batch_constraints"] = np.asarray(mine.batch_constraints())
    return {"buffer/" + k: v for k, v in rec.items()}


def ctor_draws(seed, size, A, E):
    from safe_multiagent_rl_b200.envs import collision_avoidance, congestion as cong, coverage
    np.random.seed(seed)
    cov = coverage.default_starts(size, A, E)
    np.random.seed(seed)
    con = cong.default_starts(size, A, E)
    np.random.seed(seed)
    starts, landmarks = collision_avoidance.default_starts(size, A, E)
    return {"coverage": np.asarray(cov, np.float64), "congestion": np.asarray(con, np.float64),
            "collision_starts": np.asarray(starts, np.float64), "collision_landmarks": np.asarray(landmarks, np.float64)}


def record():
    out = {}
    for kind, cases, fn in (("coverage_discrete", COVERAGE_DISCRETE, coverage_discrete), ("congestion", CONGESTION, congestion),
                            ("collision", COLLISION, collision), ("accounting", ACCOUNTING, accounting),
                            ("ctor", CTOR, ctor_draws),
                            ("coverage_continuous", COVERAGE_CONTINUOUS, lambda *p: coverage_float("continuous", *p)),
                            ("coverage_discretized", COVERAGE_DISCRETIZED, lambda *p: coverage_float("discretized", *p))):
        for p in cases:
            out.update({case(kind, p) + "/" + k: v for k, v in fn(*p).items()})
    out.update(ppo())
    out.update(buffer_files())
    return out


if __name__ == "__main__":
    path = os.path.join(HERE, "reference_record.npz")
    np.savez_compressed(path, **record())
    print(path, os.path.getsize(path) // 1024, "KiB")
