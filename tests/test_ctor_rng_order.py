"""The batched ctors' default starts follow the reference ctors' RNG order: constructing n_envs reference envs one
after another under ``np.random.seed(k)`` gives the same starts / landmarks as one batched draw (A1, B1, C1 of
SURVEY.md section 8a).  The SURVEY section 4 known answer (np.random.seed(0); CollisionAvoidance(5, 3)) needs no
reference tree; the differential part takes the reference ctors' draws live where the reference tree is present and
from tests/golden/reference_record.npz elsewhere."""
import numpy as np
import pytest

from oracle import reference_harness as rh
from safe_multiagent_rl_b200.envs import collision_avoidance, congestion, coverage


def test_collision_seed0_known_answer():
    """envs/collision_avoidance.py:60-62 with np.random.seed(0), size 5, 3 agents (SURVEY.md 4.2)."""
    np.random.seed(0)
    starts, landmarks = collision_avoidance.default_starts(5, 3, 1)
    assert starts[0].tolist() == [[2.7440675196366238, 3.5759468318620975], [3.0138168803582195, 2.724415914984484],
                                  [2.1182739966945237, 3.2294705653332807]]
    assert landmarks[0].tolist() == [[2.1879360563134624, 4.4588650039103985]]


@pytest.mark.parametrize("seed,size,A,E", [(0, 5, 3, 4), (7, 32, 16, 3), (11, 9, 1, 5)])
def test_ctor_draws_match_the_live_reference(seed, size, A, E):
    def live():
        ref = rh.load()
        np.random.seed(seed)       # Coverage (coverage.py:19, :170, :267-269)
        cov = [[list(ag.start) for ag in ref.coverage.CoverageDiscrete(size, A).agents] for _ in range(E)]
        np.random.seed(seed)       # Congestion (congestion.py:22, :215-217)
        con = [[np.asarray(ag.start, dtype=np.float64).tolist() for ag in ref.congestion.Congestion(size, A).agents]
               for _ in range(E)]
        np.random.seed(seed)       # Collision (collision_avoidance.py:60-62)
        envs = [ref.collision.CollisionAvoidance(size, A) for _ in range(E)]
        return {"coverage": np.asarray(cov, dtype=np.float64), "congestion": np.asarray(con, dtype=np.float64),
                "collision_starts": np.asarray([[list(ag.start) for ag in e.agents] for e in envs]),
                "collision_landmarks": np.asarray([np.asarray(e.landmarks, dtype=np.float64).reshape(-1, 2)
                                                   for e in envs])}
    want = rh.reference_side(f"ctor/{seed},{size},{A},{E}", live)
    np.random.seed(seed)
    assert np.array_equal(coverage.default_starts(size, A, E), want["coverage"])
    np.random.seed(seed)
    assert np.array_equal(congestion.default_starts(size, A, E), want["congestion"])
    np.random.seed(seed)
    starts, landmarks = collision_avoidance.default_starts(size, A, E)
    assert np.array_equal(starts, want["collision_starts"])
    assert np.array_equal(landmarks, want["collision_landmarks"])
