"""safe_multiagent_rl_b200 -- B200-native batched env-step hot path of safe_multiagent_RL.

Host side: Python mirrors of the reference's env / Buffer / MetaAgent protocol.  Compute:
hand-written sm_100a CUDA kernels behind the C ABI in include/smarl.h (libsmarl.so, loaded
with ctypes).  There is no CPU fallback: constructing an env without CUDA raises.
"""
from .envs import (BatchedCollisionAvoidance, BatchedCongestion, BatchedCongestionOnPolicy, BatchedCoverageContinuous,
                   BatchedCoverageDiscrete, BatchedCoverageDiscretized, BatchedCoverageDiscretizedOnPolicy, BatchedEnv,
                   SingleEnvAdapter)
from .graph import GraphedClosedLoop
from .meta_agent import BatchedMetaAgent
from .policy import FusedDiscretizedPolicy
from .rollout import (G_DISCOUNTED_TERMS, G_NONE, G_PPO_STANDARDISED, G_REWARD_TO_GO, BatchedBuffer, RolloutBuffer,
                      Stats)
from .util import make_env

__all__ = ["BatchedCoverageDiscrete", "BatchedCoverageContinuous", "BatchedCoverageDiscretized",
           "BatchedCoverageDiscretizedOnPolicy", "FusedDiscretizedPolicy", "BatchedCongestion", "BatchedCongestionOnPolicy",
           "BatchedCollisionAvoidance", "BatchedEnv",
           "SingleEnvAdapter", "BatchedMetaAgent", "GraphedClosedLoop", "BatchedBuffer", "RolloutBuffer", "Stats", "make_env",
           "G_NONE", "G_REWARD_TO_GO", "G_DISCOUNTED_TERMS", "G_PPO_STANDARDISED"]
