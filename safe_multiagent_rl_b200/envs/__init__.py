from .base import BatchedEnv, SingleEnvAdapter
from .collision_avoidance import BatchedCollisionAvoidance
from .congestion import BatchedCongestion, BatchedCongestionOnPolicy
from .coverage import BatchedCoverageDiscrete
from .coverage_float import BatchedCoverageContinuous, BatchedCoverageDiscretized, BatchedCoverageDiscretizedOnPolicy

__all__ = ["BatchedEnv", "SingleEnvAdapter", "BatchedCoverageDiscrete", "BatchedCongestion", "BatchedCongestionOnPolicy",
           "BatchedCollisionAvoidance", "BatchedCoverageContinuous", "BatchedCoverageDiscretized",
           "BatchedCoverageDiscretizedOnPolicy"]
