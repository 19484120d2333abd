"""ctypes binding of libsmarl.so (include/smarl.h).  No CPU fallback: if the library is
missing or a call fails, this raises."""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

c_ptr = C.c_void_p


class CoverageParams(C.Structure):
    _fields_ = [("size", C.c_int32), ("n_agents", C.c_int32), ("lut_len", C.c_int32),
                ("reward_rows", C.c_int32), ("lut", c_ptr), ("weights", c_ptr)]


class Accounting(C.Structure):
    _fields_ = [("gamma", C.c_double), ("n_steps", C.c_int32), ("g_mode", C.c_int32),
                ("thresholds", c_ptr)]


class CoverageFloatParams(C.Structure):
    _fields_ = [("size", C.c_int32), ("n_agents", C.c_int32), ("mode", C.c_int32), ("has_coarseness", C.c_int32),
                ("fieldview", C.c_double), ("max_norm", C.c_double), ("zoom", C.c_double), ("hi", C.c_double),
                ("cost_axis", C.c_double), ("cost_diag", C.c_double), ("weights", c_ptr)]


class CongestionParams(C.Structure):
    _fields_ = [("size", C.c_int32), ("n_agents", C.c_int32), ("demand", c_ptr),
                ("noise_mode", C.c_int32), ("episode", C.c_uint32),
                ("keep_threshold", C.c_uint64), ("seed", C.c_uint64), ("env_offset", C.c_int64),
                ("wait_reward", c_ptr), ("episode_dev", c_ptr)]


class CollisionParams(C.Structure):
    _fields_ = [("size", C.c_int32), ("n_agents", C.c_int32), ("n_landmarks", C.c_int32),
                ("obs_landmarks", C.c_int32), ("agents_size", C.c_double), ("normalize_state", C.c_int32),
                ("reward_rows", C.c_int32)]


class DiscretePolicyParams(C.Structure):
    _fields_ = [("n_agents", C.c_int32), ("hidden", C.c_int32), ("n_actions", C.c_int32), ("episode", C.c_uint32),
                ("w1", c_ptr), ("b1", c_ptr), ("w2", c_ptr), ("b2", c_ptr), ("seed", C.c_uint64),
                ("env_offset", C.c_int64), ("episode_dev", c_ptr)]


class GaussianPolicyParams(C.Structure):
    _fields_ = [("n_agents", C.c_int32), ("state_size", C.c_int32), ("hidden", C.c_int32), ("n_actions", C.c_int32),
                ("episode", C.c_uint32), ("reserved", C.c_int32),
                ("w1", c_ptr), ("b1", c_ptr), ("w_mu", c_ptr), ("b_mu", c_ptr), ("w_var", c_ptr), ("b_var", c_ptr),
                ("seed", C.c_uint64), ("env_offset", C.c_int64), ("episode_dev", c_ptr)]


P = C.POINTER
i32, i64, f64 = C.c_int32, C.c_int64, C.c_double

# name -> (restype, argtypes); every symbol include/smarl.h declares.
PROTOTYPES = {
    "smarl_abi_version": (C.c_int, []),
    "smarl_last_error": (C.c_char_p, []),
    "smarl_device_info": (C.c_int, [P(C.c_int), P(C.c_int), P(C.c_int)]),
    "smarl_set_kernel_variant": (C.c_int, [i32, i32]),
    "smarl_set_pdl": (C.c_int, [i32]),
    "smarl_grid_reset": (C.c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, i32, i64, i64, c_ptr]),
    "smarl_random_starts_u8": (C.c_int, [i32, i32, C.c_uint64, i64, i64, c_ptr, c_ptr, i32, i64, i64, c_ptr]),
    "smarl_random_starts_f64": (C.c_int, [i32, i32, f64, C.c_uint64, i64, i64, i32, c_ptr, c_ptr, i64, i32, i64, c_ptr]),
    "smarl_coverage_step": (C.c_int, [P(CoverageParams), c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                      c_ptr, c_ptr, i64, i64, c_ptr]),
    "smarl_stats_len": (i32, [i32, i32]),
    "smarl_stats_scratch_len": (i64, [i32, i32, i64]),
    "smarl_coverage_rollout": (C.c_int, [P(CoverageParams), P(Accounting), c_ptr, c_ptr, c_ptr, c_ptr,
                                         c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                         i64, i64, c_ptr]),
    "smarl_coverage_float_reset": (C.c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, i32, i64, i64, c_ptr]),
    "smarl_coverage_float_step": (C.c_int, [P(CoverageFloatParams), c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                            c_ptr, c_ptr, i64, i64, c_ptr]),
    "smarl_coverage_float_rollout": (C.c_int, [P(CoverageFloatParams), P(Accounting), c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                               c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, i64, i64, c_ptr]),
    "smarl_congestion_step": (C.c_int, [P(CongestionParams), c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                        c_ptr, c_ptr, c_ptr, c_ptr, i32, i64, i64, c_ptr]),
    "smarl_congestion_rollout": (C.c_int, [P(CongestionParams), P(Accounting), c_ptr, c_ptr, c_ptr, c_ptr,
                                           c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                           c_ptr, i64, i64, c_ptr]),
    "smarl_collision_reset": (C.c_int, [P(CollisionParams), c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                        c_ptr, c_ptr, i64, i64, c_ptr]),
    "smarl_collision_step": (C.c_int, [P(CollisionParams), c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                       c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, i64, i64, c_ptr]),
    "smarl_collision_rollout": (C.c_int, [P(CollisionParams), P(Accounting), c_ptr, c_ptr, c_ptr, c_ptr,
                                          c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                          c_ptr, c_ptr, c_ptr, i64, i64, c_ptr]),
    "smarl_rollout_penalty": (C.c_int, [c_ptr, i32, c_ptr, c_ptr, i32, i32, i64, i64, c_ptr]),
    "smarl_rollout_returns": (C.c_int, [P(Accounting), c_ptr, c_ptr, i32, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                        c_ptr, c_ptr, c_ptr, i32, i32, i64, i64, c_ptr]),
    "smarl_rollout_returns_shared": (C.c_int, [P(Accounting), c_ptr, c_ptr, c_ptr, i32, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                               c_ptr, c_ptr, c_ptr, i32, i32, i64, i64, c_ptr]),
    "smarl_lambda_update": (C.c_int, [c_ptr, c_ptr, c_ptr, f64, i32, i32, c_ptr]),
    "smarl_policy_act_discrete": (C.c_int, [P(DiscretePolicyParams), c_ptr, c_ptr, c_ptr, c_ptr, i32, i64, i64, c_ptr]),
    "smarl_policy_act_gaussian": (C.c_int, [P(GaussianPolicyParams), c_ptr, c_ptr, c_ptr, i32, i64, i64, c_ptr]),
    "smarl_policy_act_discretized": (C.c_int, [P(DiscretePolicyParams), c_ptr, c_ptr, c_ptr, i32, i64, i64, c_ptr]),
    "smarl_policy_grad_scratch_len": (i64, [i32, i32, i32, i64]),
    "smarl_policy_grad_discrete": (C.c_int, [P(DiscretePolicyParams), c_ptr, c_ptr, c_ptr, i32, f64, c_ptr, c_ptr,
                                             c_ptr, c_ptr, c_ptr, c_ptr, i64, i64, c_ptr]),
    "smarl_collision_policy_rollout": (C.c_int, [P(CollisionParams), P(GaussianPolicyParams), P(Accounting), c_ptr,
                                                 c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                                 c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, i64, i64, c_ptr]),
    "smarl_coverage_float_policy_rollout": (C.c_int, [P(CoverageFloatParams), P(GaussianPolicyParams), P(Accounting),
                                                      c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                                      c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, i64, i64, c_ptr]),
    "smarl_coverage_policy_rollout": (C.c_int, [P(CoverageParams), P(DiscretePolicyParams), P(Accounting), c_ptr, c_ptr,
                                                c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                                c_ptr, c_ptr, c_ptr, i64, i64, c_ptr]),
    "smarl_congestion_policy_rollout": (C.c_int, [P(CongestionParams), P(DiscretePolicyParams), P(Accounting), c_ptr,
                                                  c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                                  c_ptr, c_ptr, c_ptr, c_ptr, i64, i64, c_ptr]),
    "smarl_coverage_discretized_policy_rollout": (C.c_int, [P(CoverageFloatParams), P(DiscretePolicyParams),
                                                            P(Accounting), c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                                            c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                                            c_ptr, i64, i64, c_ptr]),
    "smarl_comm_get_unique_id": (C.c_int, [c_ptr]),
    "smarl_comm_init_from_unique_id": (C.c_int, [P(c_ptr), c_ptr, i32, i32]),
    "smarl_comm_destroy": (None, [c_ptr]),
    "smarl_comm_nccl_version": (C.c_int, []),
    "smarl_stats_allreduce": (C.c_int, [c_ptr, c_ptr, i32, c_ptr]),
    "smarl_host_session_create": (C.c_int, [P(c_ptr), i32, i32, i32, i64, i32]),
    "smarl_host_session_destroy": (None, [c_ptr]),
    "smarl_host_session_ld": (i64, [c_ptr]),
    "smarl_host_coverage_rollout": (C.c_int, [c_ptr, P(CoverageParams), P(Accounting), c_ptr, c_ptr, c_ptr,
                                              c_ptr, c_ptr, c_ptr, c_ptr, c_ptr]),
    "smarl_host_coverage_rollout_packed4": (C.c_int, [c_ptr, P(CoverageParams), P(Accounting), c_ptr, c_ptr, c_ptr,
                                                      c_ptr, c_ptr, c_ptr, c_ptr, c_ptr]),
    "smarl_host_session_pitch5": (i64, [c_ptr]),
    "smarl_host_coverage_rollout_packed5": (C.c_int, [c_ptr, P(CoverageParams), P(Accounting), c_ptr, c_ptr, c_ptr,
                                                      c_ptr, c_ptr, c_ptr, c_ptr, c_ptr]),
    "smarl_host_alloc_pinned": (C.c_int, [P(c_ptr), C.c_size_t, P(i32)]),
    "smarl_host_free_pinned": (None, [c_ptr]),
    "smarl_host_coverage_rollout_envmajor": (C.c_int, [c_ptr, P(CoverageParams), P(Accounting), c_ptr, c_ptr, c_ptr,
                                                       c_ptr, c_ptr, c_ptr, c_ptr]),
    "smarl_host_congestion_rollout_envmajor": (C.c_int, [c_ptr, P(CongestionParams), P(Accounting), c_ptr, c_ptr, c_ptr,
                                                         c_ptr, c_ptr, c_ptr, c_ptr, c_ptr]),
    "smarl_host_collision_rollout_envmajor": (C.c_int, [c_ptr, P(CollisionParams), P(Accounting), c_ptr, c_ptr, c_ptr,
                                                        c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr]),
    "smarl_host_congestion_rollout": (C.c_int, [c_ptr, P(CongestionParams), P(Accounting), c_ptr, c_ptr, c_ptr,
                                                c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr]),
    "smarl_host_collision_rollout": (C.c_int, [c_ptr, P(CollisionParams), P(Accounting), c_ptr, c_ptr, c_ptr, c_ptr,
                                               c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr]),
}

COST_U8, COST_I32, COST_F32 = 0, 1, 2
ENV_COVERAGE, ENV_CONGESTION, ENV_COLLISION = 0, 1, 2
KERNEL_POLICY = 3          # smarl_set_kernel_variant: 0 = FP32 pipes, 1 / 2 = tensor cores (groups of <= 16 / <= 8 agents)
_lib = None


class SmarlError(RuntimeError):
    pass


def lib_path() -> str:
    return os.environ.get("SMARL_LIB", _build.LIB_PATH)


def load():
    """Load libsmarl.so and bind every prototype.  Raises if the library is absent."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise SmarlError(f"{path} not found: build it with `python -m safe_multiagent_rl_b200.build` "
                         "(there is no CPU fallback)")
    lib = C.CDLL(path)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)       # AttributeError here = header/library mismatch
        fn.restype = res
        fn.argtypes = args
    if lib.smarl_abi_version() != 2:
        raise SmarlError("libsmarl ABI version mismatch")
    _lib = lib
    return lib


class kernel_variant:
    """Context manager: force the thread mapping of one env kind's kernels (smarl_set_kernel_variant)."""

    def __init__(self, env_kind: int, lanes: int):
        self.env_kind, self.lanes = env_kind, lanes

    def __enter__(self):
        self.prev = load().smarl_set_kernel_variant(self.env_kind, self.lanes)
        return self

    def __exit__(self, *exc):
        load().smarl_set_kernel_variant(self.env_kind, self.prev)
        return False


def check(rc: int) -> None:
    if rc != 0:
        msg = load().smarl_last_error().decode()
        raise SmarlError(f"libsmarl error {rc}: {msg}")


def ptr(t):
    """Device/host pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


_torch = None


def stream_ptr():
    global _torch
    if _torch is None:
        import torch
        _torch = torch
    return _torch.cuda.current_stream().cuda_stream
