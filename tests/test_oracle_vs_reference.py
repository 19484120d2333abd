"""Pin the numpy oracle against the unmodified reference.

The reference ships no tests (SURVEY.md section 4), so these differential runs -- and the
golden fixtures generated from the same harness -- are what pins parity.  Integer
dynamics and f64 rewards are compared bit-exactly (the oracle restates the reference's
own f64 arithmetic in the same order); only BLAS-ordered reductions get a tolerance.
Every test runs everywhere: the differential cases take the reference's side from the live
reference tree where it is present and from tests/golden/reference_record.npz elsewhere
(``rh.reference_side``); the known answers (SURVEY.md 4.2) are the reference's own outputs.
"""
import numpy as np
import pytest

from oracle import numpy_oracle as no
from oracle import reference_harness as rh


# ------------------------------------------------------------------ the reference's known answers (SURVEY.md 4.2)
def test_kat_coverage_discrete():
    fv = no.coverage_fieldview(5, 3)
    assert fv == 2.886751345948129
    lut = no.coverage_penalty_lut(5, fv)
    pos, r, c, _ = no.coverage_discrete_step([[[2, 2]] * 3], [[0, 4, 4]], 5, lut, [1, 2, 3])
    assert pos[0].tolist() == [[3, 2], [2, 2], [2, 2]]
    assert c[0].tolist() == [1, 0, 0]
    assert r[0].tolist() == [-15.452994616207489, -30.905989232414978, -46.358983848622465]
    _, r, _, _ = no.coverage_discrete_step([[[2, 2]] * 3], [[4, 4, 4]], 5, lut, [1, 2, 3])
    assert r[0].tolist() == [-25.000000000000007, -50.000000000000014, -75.00000000000003]


def test_kat_congestion():
    dem = np.array([[2, 2, 4, 4], [3, 6, 10, 5], [3, 8, 3, 4], [4, 6, 7, 8]])

    def step(starts, actions):                                  # noise 0: the moves are the intended actions
        _, r, c, _, con = no.congestion_step([starts], [actions], [actions], 3, dem)
        return r[0].tolist(), c[0].tolist(), con[0].tolist()
    r, c, con = step([[0, 0], [0, 0]], [1, 4])
    assert r == [-6.0, -26.5] and con == [1, 1] and c == [0]
    r, c, con = step([[0, 0], [0, 0]], [4, 1])
    assert r == [-11.5, -4.0] and con == [0, 0]
    r, c, con = step([[1, 1]] * 3, [0, 0, 0])
    assert r == [-8, -8, -8] and c == [1]
    r, c, con = step([[1, 1], [2, 1]], [0, 1])
    assert r == [-4, -4]


def test_kat_accounting():
    rew = np.array([[-1, -2], [-3, -4], [-5, -6]], dtype=np.float64)[:, None]      # [T, E=1, A]
    cost = np.array([[1, 0], [1, 1], [0, 1]], dtype=np.float64)[:, None]
    lam = np.array([0.5, 0.5])
    mod = no.modified_reward(rew, cost, lam)
    assert mod[:, 0].tolist() == [[-1.5, -2.5], [-4, -5], [-5.5, -6.5]]
    assert no.episode_returns(rew, 0.9)[0].tolist() == [-7.750000000000001, -10.46]
    np.testing.assert_allclose(no.episode_returns(mod, 0.9)[0], [-9.555, -12.265], rtol=1e-14)
    C = no.episode_cost_sums(cost)[0]
    assert C.tolist() == [2, 2]
    assert no.lambda_update(lam, C, [1, 1], 0.5).tolist() == [1, 1]
    np.testing.assert_allclose(no.reward_to_go(mod, 0.9)[:, 0, 0], [-9.555, -8.95, -5.5], rtol=1e-14)


# ------------------------------------------------------------------ differential: Coverage
@pytest.mark.parametrize("size,A,T,fv,seed", [(5, 3, 50, None, 0), (32, 16, 20, 8.0, 1),
                                              (8, 5, 30, None, 2), (64, 32, 5, None, 3),
                                              (3, 2, 40, 10.0, 4)])
def test_coverage_discrete_matches_reference(size, A, T, fv, seed):
    rng = np.random.default_rng(seed)
    E = 6
    weights = (1.0 + (np.arange(A) % 3)).tolist()
    fvv = no.coverage_fieldview(size, A, fv)
    lut = no.coverage_penalty_lut(size, fvv)
    for e in range(E):
        starts = np.floor(rng.random((A, 2)) * size).astype(np.int64)
        if e == 0:
            starts[:] = size - 1                      # everyone stacked near the wall
        actions = rng.integers(0, 5, size=(T, A))
        tr = rh.reference_side(f"coverage_discrete/{size},{A},{T},{fv},{seed}", lambda: rh.run_coverage_discrete(
            size, A, starts, actions, weights=weights, fieldview_size=fv), e)
        pos = starts[None].copy()
        for t in range(T):
            pos, r, c, d = no.coverage_discrete_step(pos, actions[t][None], size, lut, weights)
            assert np.array_equal(pos[0], tr["pos"][t])
            assert np.array_equal(r[0], tr["reward"][t])          # bit-exact f64
            assert np.array_equal(c[0], tr["cost"][t])
            assert np.array_equal(d[0], tr["done"][t])


# ------------------------------------------------------------------ differential: Congestion
def test_congestion_closed_form_vs_literal():
    rng = np.random.default_rng(5)
    for _ in range(4000):
        A = int(rng.integers(1, 9))
        S = int(rng.integers(1, 3))
        pos = rng.integers(0, S + 1, size=(1, A, 2))
        actions = rng.integers(0, 5, size=(1, A))
        moves = np.where(rng.random((1, A)) < 0.7, actions, rng.integers(0, 5, size=(1, A)))
        new = pos.copy()
        new[:, :, 0] = np.clip(pos[:, :, 0] + no.DIR_X[moves], 0, S)
        new[:, :, 1] = np.clip(pos[:, :, 1] + no.DIR_Y[moves], 0, S)
        edges = np.concatenate([pos, new], axis=2)[0]
        W = S + 1
        key = ((pos[:, :, 0] * W + pos[:, :, 1]) * W + new[:, :, 0]) * W + new[:, :, 1]
        lit = no.congestions_literal(actions[0].tolist(), edges.tolist())
        assert no.congestions_closed_form(actions, key)[0].tolist() == lit


@pytest.mark.parametrize("size,A,T,noise,seed", [(3, 3, 10, 0.0, 0), (3, 8, 100, 0.1, 1),
                                                 (10, 8, 40, 0.1, 2), (2, 6, 60, 0.5, 3),
                                                 (5, 32, 8, 0.3, 4)])
def test_congestion_matches_reference(size, A, T, noise, seed):
    rng = np.random.default_rng(seed)
    demand = rng.random((size + 1, size + 1)) * 8 + 2          # congestion.py:27 (commented)
    if size == 3:
        demand = np.array([[2, 2, 4, 4], [3, 6, 10, 5], [3, 8, 3, 4], [4, 6, 7, 8]])  # :28
    for e in range(4):
        starts = np.floor(rng.random((A, 2)) * size).astype(np.int64)
        starts[0] = 0                                           # congestion.py:215-216
        actions = rng.integers(0, 5, size=(T, A))
        u = rng.random((T, A, 2))
        tr = rh.reference_side(f"congestion/{size},{A},{T},{noise},{seed}", lambda: rh.run_congestion(
            size, A, starts, actions, demand, noise=noise, uniforms=u), e)
        pos = starts[None].copy()
        for t in range(T):
            moves = no.congestion_noise_moves(actions[t][None], u[t, :, 0][None], u[t, :, 1][None], noise)
            old = pos
            pos, r, c, d, con = no.congestion_step(pos, actions[t][None], moves, size, demand)
            assert np.array_equal(pos[0], tr["pos"][t])
            assert np.array_equal(np.concatenate([old, pos], axis=2)[0], tr["edges"][t])
            assert np.array_equal(con[0], tr["congestions"][t])
            assert np.array_equal(r[0], tr["reward"][t])          # bit-exact f64
            assert np.array_equal(c[0], tr["cost"][t])


# ------------------------------------------------------------------ differential: Collision
@pytest.mark.parametrize("size,A,L,T,seed", [(5, 3, 1, 50, 0), (2, 5, 1, 20, 1), (5, 8, 3, 30, 2),
                                             (3, 12, 2, 25, 3)])
def test_collision_matches_reference(size, A, L, T, seed):
    rng = np.random.default_rng(seed)
    for e in range(6):
        starts = rng.random((A, 2)) * size
        landmarks = rng.random((L, 2)) * size
        # fp32-origin actions as torch policies emit (agent.py:124-125); ~30% exceed unit norm
        actions = rng.normal(0, 0.5, size=(T, A, 2)).astype(np.float32).astype(np.float64)
        if e == 1:   # steer everyone to the first landmark so agents finish and the episode ends early
            for t in range(T):
                pass
            actions = np.repeat(((landmarks[0][None] - starts) / 6).astype(np.float32)[None], T, 0).astype(np.float64)
        if e == 2:   # crowd the agents to provoke collisions
            starts = landmarks[0][None] + rng.normal(0, 0.4, size=(A, 2))
            starts = np.clip(starts, 0, size)
        tr = rh.reference_side(f"collision/{size},{A},{L},{T},{seed}", lambda: rh.run_collision(
            size, A, starts, landmarks, actions, n_landmarks=L), e)
        pos = starts[None].copy()
        done = np.zeros((1, A), dtype=bool)
        for t in range(T):
            pos, r, c, done, active = no.collision_step(pos, done, actions[t][None], landmarks[None], size)
            assert active[0] == tr["active"][t]
            assert np.array_equal(pos[0], tr["pos"][t]), (e, t)                   # bit-exact f64
            assert np.array_equal(done[0], tr["done"][t])
            assert np.array_equal(c[0], tr["cost"][t])
            assert np.array_equal(r[0], tr["reward"][t]), (e, t)                  # bit-exact f64


# ------------------------------------------------------------------ differential: accounting
@pytest.mark.parametrize("A,K,T,gamma,seed", [(3, 3, 50, 0.999, 0), (8, 1, 100, 0.9, 1), (16, 16, 50, 0.999, 2),
                                              (3, 1, 7, 0.99, 3)])
def test_accounting_matches_reference(A, K, T, gamma, seed):
    rng = np.random.default_rng(seed)
    rewards = rng.normal(-3, 4, size=(T, A))
    costs = rng.integers(0, 3, size=(T, K)).astype(np.float64)
    lam = rng.random(K)
    thr = rng.random(K) * 10
    out = rh.reference_side(f"accounting/{A},{K},{T},{gamma},{seed}",
                            lambda: rh.run_accounting(rewards, costs, lam, gamma, thr, 0.05))
    mod = no.modified_reward(rewards[:, None, :], costs[:, None, :], lam)      # [T,1,A]
    np.testing.assert_allclose(mod[:, 0], out["mod_reward"], rtol=1e-13, atol=1e-13)
    assert np.array_equal(no.episode_returns(rewards[:, None, :], gamma)[0], out["R"])   # same order => exact
    np.testing.assert_allclose(no.episode_returns(mod, gamma)[0], out["modR"], rtol=1e-12)
    assert np.array_equal(no.episode_cost_sums(costs[:, None, :])[0], out["C"])
    np.testing.assert_allclose(no.reward_to_go(mod, gamma)[:, 0], out["G"], rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(no.discounted_terms(mod, gamma)[:, 0], out["disc"], rtol=1e-12, atol=1e-12)
    lam2 = no.lambda_update(lam, out["C"], thr, 0.05)
    np.testing.assert_allclose(lam2, out["lambdas_after"], rtol=1e-14)
    np.testing.assert_allclose(out["C"] - thr, out["mean_violation"], rtol=1e-14)


# ------------------------------------------------------------------ differential: float Coverage variants
@pytest.mark.parametrize("size,A,T,coarse,seed", [(5, 3, 40, None, 0), (5, 3, 40, 6, 1), (10, 8, 15, 20, 2), (3, 5, 30, 2, 3)])
def test_coverage_continuous_matches_reference(size, A, T, coarse, seed):
    rng = np.random.default_rng(seed)
    w = (1.0 + (np.arange(A) % 3)).tolist()
    fv = no.coverage_fieldview(size, A)
    for e in range(4):
        starts = rng.random((A, 2)) * size
        actions = rng.normal(0, 0.8, size=(T, A, 2)).astype(np.float32).astype(np.float64)
        tr = rh.reference_side(f"coverage_continuous/{size},{A},{T},{coarse},{seed}", lambda: rh.run_coverage_float(
            "continuous", size, A, starts, actions, weights=w, coarseness=coarse), e)
        pos = starts[None].copy()
        for t in range(T):
            pos, r, c, d = no.coverage_continuous_step(pos, actions[t][None], size, fv, w, coarse)
            assert np.array_equal(pos[0], tr["pos"][t])                   # bit-exact f64
            assert np.array_equal(r[0], tr["reward"][t])                  # bit-exact f64 (libm pow path)
            assert np.array_equal(c[0], tr["cost"][t])
            fast = no.coverage_float_reward(pos, fv, w, exact_pow=False)  # the multiply the CUDA kernel uses
            np.testing.assert_allclose(fast[0], tr["reward"][t], rtol=1e-14)


@pytest.mark.parametrize("size,A,T,coarse,seed", [(5, 3, 40, 20, 0), (5, 3, 40, 6, 1), (10, 8, 15, 7, 2), (3, 4, 30, 3, 3)])
def test_coverage_discretized_matches_reference(size, A, T, coarse, seed):
    rng = np.random.default_rng(seed)
    w = (1.0 + (np.arange(A) % 3)).tolist()
    fv = no.coverage_fieldview(size, A)
    zoom = coarse / size
    for e in range(4):
        starts = np.floor(rng.random((A, 2)) * size * zoom) / zoom        # coverage.py:270-272
        actions = rng.integers(0, 9, size=(T, A))
        tr = rh.reference_side(f"coverage_discretized/{size},{A},{T},{coarse},{seed}", lambda: rh.run_coverage_float(
            "discretized", size, A, starts, actions, weights=w, coarseness=coarse), e)
        pos = starts[None].copy()
        for t in range(T):
            pos, r, c, d = no.coverage_discretized_step(pos, actions[t][None], size, coarse, fv, w)
            assert np.array_equal(pos[0], tr["pos"][t])
            assert np.array_equal(r[0], tr["reward"][t])
            assert np.array_equal(c[0], tr["cost"][t])


def test_ppo_standardised_returns_match_reference():
    rng = np.random.default_rng(0)
    for T, gamma in [(50, 0.999), (8, 0.99), (100, 0.9), (2, 0.5)]:
        m = rng.normal(-3, 4, size=T)
        want = rh.reference_side(f"ppo/{T},{gamma}", lambda: {"returns": rh.run_ppo_returns(m, gamma)})["returns"]
        got = no.ppo_standardised_returns(m[:, None, None], gamma)[:, 0, 0]
        np.testing.assert_allclose(got, want, rtol=2e-5, atol=2e-5)


# ------------------------------------------------------------------ Buffer persistence (buffer.py:50-65,141-177)
def test_batched_buffer_save_results_matches_reference_files(tmp_path, monkeypatch):
    """The .npy / params.json files and the per-batch series of BatchedBuffer equal the reference Buffer's
    (its matplotlib calls are replaced by a recording no-op: figures are out of scope)."""
    import argparse
    import json
    import sys
    from unittest import mock

    import torch

    from safe_multiagent_rl_b200.rollout import BatchedBuffer

    rng = np.random.default_rng(5)
    A, K, T, batches, bsz = 3, 2, 7, 4, 5
    params = argparse.Namespace(gamma=0.95, thresholds=[1.5, 2.0], batch_size=bsz, n_agents_learning_cycles=1,
                                environment="ExploreDiscrete", size=5, n_agents=A, numpy_seed=3, torch_seed=4,
                                algo="AC")
    monkeypatch.chdir(tmp_path)
    mine = BatchedBuffer(params, constrained=True)            # default path: results/<name>_<i>
    fed = []
    for b in range(batches):
        rew = rng.normal(size=(T, bsz, A))
        cost = rng.integers(0, 3, size=(T, bsz, K)).astype(np.float64)
        lam = rng.random(K)
        mod = rew - (cost @ lam)[:, :, None]
        fed.append((rew, mod, cost, lam))
        for t in range(T):                                     # compat path: per-step [E, A] / [E, K] tensors
            mine.append(torch.from_numpy(rew[t]), torch.from_numpy(mod[t]), torch.from_numpy(cost[t]))
        mine.step()
        mine.append_lambdas(lam)

    def live():
        ref = rh.load()
        rb = ref.Buffer(params, constrained=True, save_path=str(tmp_path / "ref"))
        (tmp_path / "ref").mkdir()
        for rew, mod, cost, lam in fed:
            for e in range(bsz):
                for t in range(T):
                    rb.append(list(rew[t, e]), list(mod[t, e]), list(cost[t, e]))
                rb.step()
            rb.append_lambdas(lam)
        plt = mock.MagicMock()
        with mock.patch.object(sys.modules[ref.Buffer.__module__], "plt", plt), mock.patch("builtins.print"):
            rb.save_results()
        out = {n: np.load(tmp_path / "ref" / (n + ".npy")) for n in ("constr3", "scores3", "lambdas")}
        out["params_json"] = (tmp_path / "ref" / "params.json").read_text()
        bs, bm = rb._get_batch_scores()
        return dict(out, batch_scores=np.array(bs), batch_means=np.array(bm),
                    batch_constraints=np.array(rb._get_batch_constraints()))
    want = rh.reference_side("buffer", live)
    out = mine.save_results()
    assert out == "results/ExploreDiscrete_s5_n3_3-4_AC_0" and mine.save_results() == out
    for name in ("constr3", "scores3", "lambdas"):
        np.testing.assert_allclose(np.load(tmp_path / out / (name + ".npy")), want[name], rtol=1e-13, atol=0)
    assert json.load(open(tmp_path / out / "params.json")) == json.loads(str(want["params_json"]))
    ms, mm = mine.batch_scores()
    np.testing.assert_allclose(ms, want["batch_scores"], rtol=1e-13)
    np.testing.assert_allclose(mm, want["batch_means"], rtol=1e-13)
    np.testing.assert_allclose(mine.batch_constraints(), want["batch_constraints"], rtol=1e-13)
    # unconstrained runs get their own directory stem and no lambdas file (buffer.py:56-57,152-153)
    un = BatchedBuffer(params, constrained=False)
    un.extend(torch.zeros(2, A), torch.zeros(2, A), torch.zeros(2, K))
    p = un.save_results()
    assert p.endswith("_AC_unconstr_0") and not (tmp_path / p / "lambdas.npy").exists()
