"""ctypes binding of libmbpo_b200.so (include/mbpo_b200.h).

The library is the product: there is no Python/PyTorch fallback.  If the shared object is
missing this module raises at import time with the command that builds it.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

MBPO_ABI_VERSION = 1
MBPO_MAX_HORIZON = 128
MBPO_MAX_FREQ = MBPO_MAX_HORIZON // 2 + 1

MBPO_OK = 0
MBPO_EINVAL = -1
MBPO_EUNSUPPORTED = -2
MBPO_ECUDA = -3
MBPO_EWORKSPACE = -4

PRNG_LEGACY, PRNG_PARTITIONABLE = 0, 1
SUMMARIZE_MEAN, SUMMARIZE_MAX = 0, 1
SYSTEM_PENDULUM, SYSTEM_MLP_ENSEMBLE, SYSTEM_NOISY_PENDULUM, SYSTEM_POINT_MASS = 0, 1, 2, 3
MATH_REFERENCE, MATH_THETA_CARRY = 0, 1

_HERE = os.path.dirname(os.path.abspath(__file__))
# MBPO_B200_LIB: another build of the same ABI (A/B measurements of kernel variants); default = the in-tree library
LIB_PATH = os.environ.get("MBPO_B200_LIB") or os.path.join(_HERE, "libmbpo_b200.so")


class MbpoError(RuntimeError):
    """Non-zero return code from libmbpo_b200 (message from mbpo_last_error())."""

    def __init__(self, code: int, message: str):
        super().__init__("libmbpo_b200 error %d: %s" % (code, message))
        self.code = code


class MbpoUnsupported(MbpoError, NotImplementedError):
    """MBPO_EUNSUPPORTED: the configuration has no CUDA kernel (there is no fallback)."""


class PendulumParamsC(C.Structure):
    _fields_ = [(n, C.c_float) for n in ("max_speed", "max_torque", "dt", "g", "m", "l",
                                         "control_cost", "angle_cost", "target_angle")]


class PointMassParamsC(C.Structure):
    _fields_ = [(n, C.c_float) for n in ("dt", "max_accel", "max_speed", "target_x", "target_y", "speed_cost",
                                         "control_cost")]


class GeneralSystemParamsC(C.Structure):
    _fields_ = [("pendulum", PendulumParamsC), ("noise_std", C.c_float), ("point_mass", PointMassParamsC)]


class MlpEnsembleParamsC(C.Structure):
    _fields_ = [("num_members", C.c_int32), ("hidden", C.c_int32), ("x_dim", C.c_int32), ("u_dim", C.c_int32),
                ("w_in", C.c_void_p), ("b_in", C.c_void_p), ("w_h", C.c_void_p), ("b_h", C.c_void_p),
                ("w_out", C.c_void_p), ("b_out", C.c_void_p), ("reward", PendulumParamsC)]


class IcemCfgC(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("horizon", "action_dim", "x_dim", "num_samples", "num_elites",
                                         "num_prev_elites", "num_particles", "num_steps", "warm_start",
                                         "prng_mode", "summarize", "system_kind", "math_mode")] + \
               [(n, C.c_float) for n in ("init_std", "alpha", "exponent", "u_min", "u_max", "lambda_constraint",
                                         "sigma")] + [("s_scale", C.c_float * MBPO_MAX_FREQ)]


class PolicyParamsC(C.Structure):
    """MbpoPolicyParams."""
    _fields_ = [("num_hidden", C.c_int32), ("hidden", C.c_int32), ("obs_dim", C.c_int32), ("action_dim", C.c_int32),
                ("w", C.c_void_p * 5), ("b", C.c_void_p * 5), ("min_std", C.c_float),
                ("head", C.c_int32), ("shared_noise", C.c_int32), ("normalize", C.c_int32),
                ("sig_bias", C.c_float), ("sig_min", C.c_float), ("sig_max", C.c_float), ("action_clip", C.c_float),
                ("obs_mean", C.c_float * 4), ("obs_std", C.c_float * 4),
                ("obs_mean_dev", C.c_void_p), ("obs_std_dev", C.c_void_p), ("kernel", C.c_int32),
                ("draw_offset", C.c_int32), ("draw_total", C.c_int32)]


KEYS_SAC, KEYS_UNROLL, KEYS_AS_IS = 0, 1, 2
HEAD_NORMAL_TANH, HEAD_BPTT_ACTOR = 0, 1
ACTOR_AUTO, ACTOR_CUDA_CORES, ACTOR_TCGEN05, ACTOR_TCGEN05_WIDE = 0, 1, 2, 3


class IcemTraceC(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("actions", "values", "elite_idx", "mean", "std", "best_value")]


MBPO_REPLAY_MAX_FIELDS = 8


class ReplayStateC(C.Structure):
    """MbpoReplayState."""
    _fields_ = [("data", C.c_void_p), ("capacity", C.c_longlong), ("row_width", C.c_int32), ("reserved", C.c_int32),
                ("head", C.c_longlong), ("insert_position", C.c_longlong), ("sample_position", C.c_longlong)]


class ReplayFieldsC(C.Structure):
    """MbpoReplayFields."""
    _fields_ = [("num_fields", C.c_int32), ("width", C.c_int32 * MBPO_REPLAY_MAX_FIELDS),
                ("ptr", C.c_void_p * MBPO_REPLAY_MAX_FIELDS)]


# name -> (restype, argtypes); every symbol include/mbpo_b200.h declares
_P, _I, _F, _SZ, _LL = C.c_void_p, C.c_int, C.c_float, C.c_size_t, C.c_longlong
SIGNATURES = {
    "mbpo_abi_version": (_I, []),
    "mbpo_last_error": (C.c_char_p, []),
    "mbpo_struct_size": (_SZ, [_I]),
    "mbpo_icem_cfg_init": (_I, [C.POINTER(IcemCfgC), _I, _I, _I, _I, _I, _I, _F, _F, _I, _F, _F, _F, _F, _I, _F]),
    "mbpo_prng_split": (_I, [_P, _I, _I, _I, _P, _P]),
    "mbpo_prng_random_bits": (_I, [_P, _I, _I, _I, _P, _P]),
    "mbpo_prng_uniform": (_I, [_P, _I, _I, _I, _F, _F, _P, _P]),
    "mbpo_prng_normal": (_I, [_P, _I, _I, _I, _P, _P]),
    "mbpo_powerlaw_noise": (_I, [C.POINTER(IcemCfgC), _P, _I, _P, _P, _P]),
    "mbpo_powerlaw_noise_rolled": (_I, [C.POINTER(IcemCfgC), _P, _I, _P, _P, _P]),
    "mbpo_icem_sample_actions": (_I, [C.POINTER(IcemCfgC), _P, _P, _P, _I, _P, _P, _P, _P]),
    "mbpo_system_step": (_I, [_I, _P, _I, _P, _P, _I, _P, _P, _P]),
    "mbpo_rollout_actions": (_I, [_I, _P, _I, _I, _I, _I, _P, _P, _I, _I, _P, _P, _P, _P, _P]),
    "mbpo_system_step_general": (_I, [_I, C.POINTER(GeneralSystemParamsC), _I, _P, _P, _P, _I, _P, _P, _P, _P]),
    "mbpo_system_objective": (_I, [_I, C.POINTER(GeneralSystemParamsC), _I, _I, _P, _P, _P, _I, _I, _I, _I, _P, _P, _P,
                                   _P, _P]),
    "mbpo_icem_elite_refit": (_I, [C.POINTER(IcemCfgC), _P, _P, _P, _P, _P, _P, _I, _P, _P, _P, _P, _P, _P]),
    "mbpo_icem_plan": (_I, [C.POINTER(IcemCfgC), _P, _P, _P, _P, _I, _P, _P, _P, C.POINTER(IcemTraceC), _P]),
    "mbpo_icem_plan_clustered": (_I, [C.POINTER(IcemCfgC), _P, _P, _P, _P, _I, _P, _P, _P, C.POINTER(IcemTraceC), _I,
                                      _P]),
    "mbpo_icem_plan_cluster_size": (_I, [C.POINTER(IcemCfgC), _I]),
    "mbpo_icem_plan_cluster_capacity": (_I, [C.POINTER(IcemCfgC), _I]),
    "mbpo_icem_plan_is_fused": (_I, [C.POINTER(IcemCfgC)]),
    "mbpo_icem_workspace_bytes": (_SZ, [C.POINTER(IcemCfgC), _I]),
    "mbpo_icem_plan_staged": (_I, [C.POINTER(IcemCfgC), _P, _P, _P, _P, _I, _P, _P, _P, _P, _SZ, _P]),
    "mbpo_icem_penalize": (_I, [_P, _P, C.c_longlong, _I, _I, _I, _F, _P]),
    "mbpo_icem_penalize_particles": (_I, [_P, _P, _I, _P, C.c_longlong, _I, _I, _I, _F, _P]),
    "mbpo_icem_clip_actions": (_I, [_P, _P, _P, _I, _I, _I, _I, _P]),
    "mbpo_icem_mpc_closed_loop": (_I, [C.POINTER(IcemCfgC), _P, _P, _P, _P, _I, _I, _P, _P, _P, _P, _P, _P]),
    "mbpo_icem_mpc_closed_loop_clustered": (_I, [C.POINTER(IcemCfgC), _P, _P, _P, _P, _I, _I, _P, _P, _P, _P, _P, _I,
                                                 _P]),
    "mbpo_env_rollout": (_I, [_I, _P, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P, _I, _I, _P, _P, _P, _P, _P, _P]),
    "mbpo_env_unroll": (_I, [_I, _P, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _P, _P, _P, _P, _P, _P]),
    "mbpo_actor_rollout": (_I, [_I, _P, _I, _I, C.POINTER(PolicyParamsC), _I, _I, _P, _I, _I, _P, _P, _P, _P, _I, _I,
                                _P, _P, _P, _P, _P, _P, _P]),
    "mbpo_actor_rollout_extras": (_I, [_I, _P, _I, _I, C.POINTER(PolicyParamsC), _I, _I, _P, _I, _I, _P, _P, _P, _P, _I,
                                       _I, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "mbpo_env_unroll_general": (_I, [_I, C.POINTER(GeneralSystemParamsC), _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P,
                                     _P, _P, _I, _I, _P, _P, _P, _P, _P, _P]),
    "mbpo_actor_rollout_general": (_I, [_I, C.POINTER(GeneralSystemParamsC), _I, C.POINTER(PolicyParamsC), _I, _I, _P,
                                        _I, _I, _P, _P, _P, _P, _P, _P, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "mbpo_rollout_policy_general": (_I, [_I, C.POINTER(GeneralSystemParamsC), _I, C.POINTER(PolicyParamsC), _I, _I,
                                         _P, _P, _I, _P, _I, _I, _P, _P, _P, _P, _P, _P]),
    "mbpo_rollout_adjoint": (_I, [_I, _P, _I, _I, _I, _I, _LL, _LL, _LL, _LL, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "mbpo_rollout_adjoint_general": (_I, [_I, C.POINTER(GeneralSystemParamsC), _I, _I, _LL, _LL, _LL, _LL, _LL, _LL,
                                          _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "mbpo_lambda_return": (_I, [_P, _P, _I, _I, _LL, _LL, C.c_double, C.c_double, _P, _P]),
    "mbpo_lambda_return_vjp": (_I, [_P, _I, _I, _LL, _LL, C.c_double, C.c_double, _P, _P, _P]),
    "mbpo_mlp_dynamics_forward": (_I, [C.POINTER(MlpEnsembleParamsC), _P, _P, _I, _P, _P]),
    "mbpo_ensemble_rollout": (_I, [C.POINTER(MlpEnsembleParamsC), _I, _P, _P, _I, _I, _I, _P, _P]),
    "mbpo_ensemble_rollout_transitions": (_I, [C.POINTER(MlpEnsembleParamsC), _I, _P, _P, _I, _I, _P, _P, _P]),
    "mbpo_ensemble_env_rollout": (_I, [C.POINTER(MlpEnsembleParamsC), _I, C.POINTER(PolicyParamsC), _I, _I, _P, _I,
                                       _I, _P, _P, _P, _P, _P, _P, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "mbpo_prng_randint": (_I, [_P, _I, _I, _I, _I, _I, _P, _P]),
    "mbpo_replay_insert": (_I, [C.POINTER(ReplayStateC), C.POINTER(ReplayFieldsC), _LL, _P]),
    "mbpo_replay_sample": (_I, [C.POINTER(ReplayStateC), _P, _I, _I, _P, _P, _P, _P]),
    "mbpo_replay_read": (_I, [C.POINTER(ReplayStateC), _LL, _LL, _P, _P]),
    "mbpo_running_statistics_workspace_bytes": (_SZ, [_I]),
    "mbpo_running_statistics_accumulate": (_I, [_P, _LL, _I, _P, _P, _SZ, _P, _P]),
    "mbpo_running_statistics_finalize": (_I, [_P, _I, _P, _P, _P, _F, _F, _P, _P, _P, _P, _P]),
    "mbpo_running_statistics_normalize": (_I, [_P, _LL, _I, _P, _P, _F, _P, _P]),
    "mbpo_normalizer_finalize": (_I, [_P, _I, _P, _P, _P, _F, _P, _P, _P, _P]),
    "mbpo_normalizer_inverse": (_I, [_P, _LL, _I, _P, _P, _P, _P]),
    "mbpo_replay_take": (_I, [C.POINTER(ReplayStateC), _P, _LL, _P, _P]),
    "mbpo_compute_gae": (_I, [_P, _P, _P, _P, _P, _I, _I, _LL, _LL, C.c_double, C.c_double, _P, _P, _P]),
    "mbpo_eval_metrics": (_I, [_P, _P, _P, _P, _I, _I, _I, _LL, _LL, _P, _P, _P, _P]),
    "mbpo_env_reset_from_buffer": (_I, [C.POINTER(ReplayStateC), _P, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P]),
}


def _load() -> C.CDLL:
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "libmbpo_b200.so is not built (%s).  Build it with `python model-based-policy-optimizers_b200/build.py` "
            "or `python -c 'import __graft_entry__ as g; g.build()'`.  There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    got = lib.mbpo_abi_version()
    if got != MBPO_ABI_VERSION:
        raise ImportError("libmbpo_b200.so ABI version %d != binding version %d; rebuild" % (got, MBPO_ABI_VERSION))
    for which, struct in enumerate((IcemCfgC, PendulumParamsC, MlpEnsembleParamsC, IcemTraceC, PolicyParamsC, ReplayStateC,
                                    ReplayFieldsC)):
        if lib.mbpo_struct_size(which) != C.sizeof(struct):
            raise ImportError("struct layout mismatch for %s: C %d vs ctypes %d" % (
                struct.__name__, lib.mbpo_struct_size(which), C.sizeof(struct)))
    return lib


lib = _load()


def check(rc: int) -> None:
    if rc == MBPO_OK:
        return
    msg = (lib.mbpo_last_error() or b"").decode("utf-8", "replace")
    if rc == MBPO_EUNSUPPORTED:
        raise MbpoUnsupported(rc, msg)
    raise MbpoError(rc, msg)


def ptr(t: torch.Tensor | None) -> int | None:
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise MbpoError(MBPO_EINVAL, "expected a CUDA tensor, got device %s (there is no CPU path)" % t.device)
    if not t.is_contiguous():
        raise MbpoError(MBPO_EINVAL, "expected a contiguous tensor")
    return t.data_ptr()


def stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def require_cuda(device=None) -> torch.device:
    if not torch.cuda.is_available():
        raise MbpoError(MBPO_ECUDA, "no CUDA device is available: mbpo_b200 has no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)


def cuda_guard(t: torch.Tensor):
    """Context manager making t's device current; raises for CPU tensors (no CPU path)."""
    if not t.is_cuda:
        raise MbpoError(MBPO_EINVAL, "expected a CUDA tensor, got device %s (there is no CPU path)" % t.device)
    return torch.cuda.device(t.device)
