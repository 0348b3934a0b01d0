"""ctypes binding of libsatb200.so (include/satb200.h). No torch types cross the boundary: tensors
are passed as raw device pointers plus the current CUDA stream handle.

There is NO CPU fallback: if the library is missing or no CUDA device is present every entry point
raises. Build it with `python ppo-rl-satellite_b200/build.py` (nvcc cross-compiles without a GPU).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libsatb200.so")

SAT_STATE_COLS = 16
SAT_ISTATE_COLS = 4
COL_P, COL_PV, COL_E, COL_EV, COL_FUEL_C, COL_FUEL_T, COL_DIS, COL_RET = 0, 3, 6, 9, 12, 13, 14, 15
ICOL_DZ, ICOL_COUNT, ICOL_INTSTATE, ICOL_ERR = 0, 1, 2, 3
MODE_CW, MODE_RK4 = 0, 1
ACT_F32, ACT_F64 = 0, 1
ACTOR_PACKED_FLOATS = 18 * 256 + 256 + 256 * 256 + 256 + 4 * 256 + 4 + 4
ACTOR_TC_IMAGE_FLOATS = 2 * 256 * 256


class SatEnvState(C.Structure):
    _fields_ = [("state", C.c_void_p), ("istate", C.c_void_p), ("n", C.c_int64), ("ld", C.c_int64)]


class SatEnvParams(C.Structure):
    _fields_ = [("mode", C.c_int32), ("flag", C.c_int32), ("max_episode_steps", C.c_int32),
                ("auto_reset", C.c_int32), ("action_dtype", C.c_int32), ("substeps", C.c_int32),
                ("skip_danger_zone", C.c_int32), ("fast_libm", C.c_int32),
                ("d_capture", C.c_double), ("d_range", C.c_double), ("gamma", C.c_double),
                ("stm", C.c_double * 36),
                ("h", C.c_double), ("mu", C.c_double), ("re", C.c_double), ("j2", C.c_double),
                ("r_cw", C.c_double * 3), ("v_cw", C.c_double * 3), ("u_grav", C.c_double),
                ("reset_p", C.c_double * 3), ("reset_e", C.c_double * 3)]


class SatActorWeights(C.Structure):
    _fields_ = [("w1", C.c_void_p), ("b1", C.c_void_p), ("w2", C.c_void_p), ("b2", C.c_void_p),
                ("w3", C.c_void_p), ("b3", C.c_void_p), ("log_std", C.c_void_p), ("packed", C.c_void_p),
                ("in_dim", C.c_int32), ("hidden", C.c_int32), ("act_dim", C.c_int32),
                ("use_tanh", C.c_int32), ("max_action", C.c_float)]


# name -> (restype, argtypes); kept in one table so tests can check it against include/satb200.h
class SatPpoNet(C.Structure):
    _fields_ = [("params", C.c_void_p), ("packed", C.c_void_p), ("grads", C.c_void_p), ("exp_avg", C.c_void_p),
                ("exp_avg_sq", C.c_void_p), ("workspace", C.c_void_p), ("heads", C.c_int32), ("use_tanh", C.c_int32),
                ("max_action", C.c_float), ("reserved", C.c_int32)]


PPO_OFF_W1, PPO_OFF_B1, PPO_OFF_W2, PPO_OFF_B2, PPO_OFF_W3 = 0, 4608, 4864, 70400, 70656


def ppo_param_floats(heads: int) -> int:
    return 70656 + 257 * heads + (3 if heads == 3 else 0)


def ppo_grad_floats_stats(heads: int) -> int:
    """SAT_PPO_GRAD_FLOATS_STATS: flat gradient, loss slot, one spare float and the four-float diagnostics tail"""
    return ppo_param_floats(heads) + 6


# fp64 record of sat_ppo_adam_stats (SAT_PPO_STAT_*): sums over the minibatches added, COUNT of them
(PPO_STAT_LOSS, PPO_STAT_SURROGATE, PPO_STAT_ENTROPY, PPO_STAT_APPROX_KL, PPO_STAT_CLIP_FRAC, PPO_STAT_GRAD_NORM,
 PPO_STAT_CLIP_COEF, PPO_STAT_COUNT) = range(8)
PPO_STATS_DOUBLES = 8


_P, _I64, _I32, _D, _F, _U64 = C.c_void_p, C.c_int64, C.c_int, C.c_double, C.c_float, C.c_uint64
SIGNATURES = {
    "sat_abi_version": (C.c_int, []),
    "sat_strerror": (C.c_char_p, [C.c_int]),
    "sat_rk4_propagate": (C.c_int, [_P, _I64, _I64, _D, _I32, _D, _D, _D, _P]),
    "sat_rk4_propagate_host": (C.c_int, [_P, _I64, _P, _I64, _D, _I32, _D, _D, _D, _P]),
    "sat_state_eq": (C.c_int, [_P, _P, _I64, _I64, _D, _D, _D, _P]),
    "sat_cw_propagate": (C.c_int, [_P, _I64, _I64, C.POINTER(C.c_double), _P]),
    "sat_cw_ode_rk45": (C.c_int, [_P, _I64, _I64, _D, _D, _D, _D, _D, _D, _P, _P]),
    "sat_ppo_use_tensor_cores": (C.c_int, [C.c_int]),
    "sat_ppo_workspace_floats": (C.c_int64, [_I64]),
    "sat_ppo_pack": (C.c_int, [_P, _P]),
    "sat_ppo_actor_grad": (C.c_int, [_P, _P, _P, _P, _P, _P, _I64, _F, _F, _P]),
    "sat_ppo_critic_grad": (C.c_int, [_P, _P, _P, _P, _I64, _P]),
    "sat_ppo_adam": (C.c_int, [_P, _P, _F, _F, _F, _F, _F, _P, _P]),
    "sat_ppo_adam_peers": (C.c_int, [_P, _P, _F, _F, _F, _F, _F, _P, _P, _I32, _I64, _P]),
    "sat_ppo_actor_grad_stats": (C.c_int, [_P, _P, _P, _P, _P, _P, _I64, _F, _F, _P]),
    "sat_ppo_adam_stats": (C.c_int, [_P, _P, _F, _F, _F, _F, _F, _P, _P, _P]),
    "sat_ppo_adam_peers_stats": (C.c_int, [_P, _P, _F, _F, _F, _F, _F, _P, _P, _I32, _I64, _P, _P]),
    "sat_reachable_domain": (C.c_int, [_P, _P, _I64, _I32, _I32, _D, _P, _P, _P, _P]),
    "sat_orbital_elements": (C.c_int, [_P, _I64, _D, _P, _P, _P]),
    "sat_state_from_elements": (C.c_int, [_P, _I64, _D, _P, _P]),
    "sat_workspace_bytes": (_I64, [_I64]),
    "sat_env_default_params": (None, [C.POINTER(SatEnvParams)]),
    "sat_env_init": (C.c_int, [C.POINTER(SatEnvState), _D, _D, C.POINTER(SatEnvParams), _P]),
    "sat_env_reset": (C.c_int, [C.POINTER(SatEnvState), _P, C.POINTER(SatEnvParams), _P]),
    "sat_env_observe": (C.c_int, [C.POINTER(SatEnvState), _P, _P, _P]),
    "sat_env_observe_norm": (C.c_int, [C.POINTER(SatEnvState), _P, _P, _P]),
    "sat_env_step": (C.c_int, [C.POINTER(SatEnvState), _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                               C.POINTER(SatEnvParams), _P]),
    "sat_env_step_timed": (C.c_int, [C.POINTER(SatEnvState), _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                                     C.POINTER(SatEnvParams), _P, _P]),
    "sat_danger_zone_count": (C.c_int, [_P, _P, _I64, _D, _P, _P, _P]),
    "sat_fsolve_pfai": (C.c_int, [_P, _P, _P, _P, _P, _P, _I64, _D, _P, _P, _P]),
    "sat_libm_eval": (C.c_int, [_I32, _P, _P, _I64, _P]),
    "sat_env_step_host_bytes": (_I64, [_I64]),
    "sat_env_step_host": (C.c_int, [C.POINTER(SatEnvState), _P, _P, _P, _P, _P, _P, C.POINTER(SatEnvParams), _P, _P, _I32]),
    "sat_norm_update": (C.c_int, [_P, _P, _I64, _I32, _I32, _P, _P, _P, _P]),
    "sat_actor_pack": (C.c_int, [C.POINTER(SatActorWeights), _P, _P]),
    "sat_actor_sample": (C.c_int, [C.POINTER(SatActorWeights), _P, C.POINTER(SatEnvState), _P, _I64, _I64,
                                   _U64, _U64, _P, _P, _P, _P, _P, _P, _P]),
    "sat_actor_sample_tc": (C.c_int, [C.POINTER(SatActorWeights), _P, _P, C.POINTER(SatEnvState), _P, _I64, _I64,
                                      _U64, _U64, _P, _P, _P, _P, _P, _P, _P]),
    "sat_actor_sample_pair_tc": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _I64, _I64, _U64, _U64, _U64, _P, _P, _P, _P, _P, _P]),
    "sat_critic_forward": (C.c_int, [C.POINTER(SatActorWeights), _P, _I64, _P, _P]),
    "sat_actor_sample_pair": (C.c_int, [_P, _P, _P, _P, _P, _I64, _I64, _U64, _U64, _U64, _P, _P, _P, _P, _P, _P]),
    "sat_gae": (C.c_int, [_P, _P, _P, _P, _I64, _I64, _F, _F, _P, _P, _P]),
    "sat_gae_flat": (C.c_int, [_P, _P, _P, _P, _P, _I64, _F, _F, _P, _P, _P]),
    "sat_adv_moments": (C.c_int, [_P, _I64, _P, _P, _P]),
    "sat_adv_normalize": (C.c_int, [_P, _I64, _P, _P]),
    "sat_peak_fp64": (C.c_int, [_P, _I32, _I32, _I32, C.POINTER(C.c_double), _P]),
    "sat_peak_fp32": (C.c_int, [_P, _I32, _I32, _I32, C.POINTER(C.c_double), _P]),
}

_lib = None


class SatError(RuntimeError):
    pass


def load():
    """dlopen the CUDA library; raises (never falls back) if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not found: the CUDA extension is not built and there is no CPU fallback. "
                "Run `python ppo-rl-satellite_b200/build.py` (or __graft_entry__.build()).")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)     # AttributeError if the .so does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        if lib.sat_abi_version() != 1:
            raise ImportError("libsatb200.so ABI version mismatch")
        _lib = lib
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().sat_strerror(rc).decode()
        raise SatError(f"{what or 'libsatb200'} failed: {msg} (code {rc})")


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise SatError("no CUDA device: libsatb200 has no CPU fallback (the CPU restatement lives in oracle/ "
                       "and is test infrastructure only)")
    return torch


def stream_ptr() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream


def guard_device(device) -> None:
    """kernels launch on the CURRENT device: refuse to run when it is not the one that owns the buffers"""
    import torch
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if torch.cuda.current_device() != idx:
        raise SatError(f"current CUDA device is {torch.cuda.current_device()} but the buffers live on cuda:{idx}; "
                       "wrap the call in `with torch.cuda.device(...)` or call torch.cuda.set_device first")


def ptr(t) -> int:
    """device pointer of a CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise SatError("expected a CUDA tensor")
    if not t.is_contiguous():
        raise SatError("expected a contiguous tensor")
    return t.data_ptr()


def default_params() -> SatEnvParams:
    p = SatEnvParams()
    load().sat_env_default_params(C.byref(p))
    return p
