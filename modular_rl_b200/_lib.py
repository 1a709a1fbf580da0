"""ctypes binding of libmrl_b200.so (include/mrl_b200.h).

There is no CPU fallback: if the shared library is missing or cannot be loaded every
entry point raises.  Build it with ``python -c "import __graft_entry__ as g; g.build()"``
(or ``modular_rl_b200/csrc/build.sh``).
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HOST, DEVICE = 0, 1
F32, F64, I32, I64 = 0, 1, 2, 3
GAUSS, CATEGORICAL, VALUE = 0, 1, 2
ACTIVATIONS = {"tanh": 0, "relu": 1, "sigmoid": 2}
# envs.py device_kind -> MRL_ENV_CARTPOLE, MRL_ENV_PENDULUM, MRL_ENV_ACROBOT, MRL_ENV_MOUNTAIN_CAR,
# MRL_ENV_MOUNTAIN_CAR_CONTINUOUS (user environments, envs.DeviceEnv, get ids >= 64 from mrl_rollout_env_compile)
DEVICE_ENVS = {"cartpole": 0, "pendulum": 1, "acrobot": 2, "mountaincar": 3, "mountaincar_continuous": 4}

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MRL_LIB") or os.path.join(_HERE, "libmrl_b200.so")   # MRL_LIB: kernel experiments only

_DT = {np.dtype(np.float32): F32, np.dtype(np.float64): F64, np.dtype(np.int32): I32,
       np.dtype(np.int64): I64}


class TrpoCfg(C.Structure):
    _fields_ = [("cg_damping", C.c_double), ("max_kl", C.c_double), ("residual_tol", C.c_double),
                ("accept_ratio", C.c_double), ("cg_iters", C.c_int), ("max_backtracks", C.c_int)]


class ZFilterCfg(C.Structure):
    _fields_ = [("enabled", C.c_int), ("demean", C.c_int), ("destd", C.c_int), ("clip", C.c_double)]


_lib = None

_P, _I, _LL, _D = C.c_void_p, C.c_int, C.c_longlong, C.c_double
_SIGS = {
    "mrl_last_error": (C.c_char_p, []),
    "mrl_version": (_I, []),
    "mrl_launch_count": (_LL, []),
    "mrl_profile_enable": (_I, [_I]),
    "mrl_profile_kinds": (_I, []),
    "mrl_profile_kind_name": (C.c_char_p, [_I]),
    "mrl_profile_read": (_I, [_P, _P]),
    "mrl_measure_fp32_tflops": (_I, [_I, _P]),
    "mrl_measure_mma_tf32_tflops": (_I, [_I, _P]),
    "mrl_measure_tcgen05_tf32_tflops": (_I, [_I, _P]),
    "mrl_batch_refresh_advantages": (_I, [_P, _P]),
    "mrl_batch_create": (_I, [C.POINTER(_P), _I, _I, _I]),
    "mrl_batch_destroy": (_I, [_P]),
    "mrl_batch_set_obs": (_I, [_P, _P, _I, _LL, _LL, _I, _P]),
    "mrl_batch_set_paths": (_I, [_P, _P, _P, _I, _D, _I, _P]),
    "mrl_batch_set_policy_inputs": (_I, [_P, _I, _I, _P, _I, _P, _I, _P, _I, _I, _P]),
    "mrl_batch_set_vf_target": (_I, [_P, _P, _I, _I, _P]),
    "mrl_batch_mix_vf_target": (_I, [_P, _D, _P]),
    "mrl_batch_set_global_n": (_I, [_P, _LL]),
    "mrl_batch_size": (_LL, [_P]),
    "mrl_batch_get_time_index": (_I, [_P, _P, _I, _P]),
    "mrl_batch_gae": (_I, [_P, _P, _I, _P, _I, _D, _D, _I, _P, _P, _P, _I, _P]),
    "mrl_gae": (_I, [_P, _I, _P, _I, _P, _P, _I, _LL, _D, _D, _P, _P, _I, _P]),
    "mrl_standardize": (_I, [_P, _LL, _P, _I, _P]),
    "mrl_zfilter_scan": (_I, [_P, _I, _LL, _I, _P, _P, _P, _I, _I, _D, _P, _I, _I, _P]),
    "mrl_net_create": (_I, [C.POINTER(_P), _I, _I, C.POINTER(_I), _I, _I]),
    "mrl_net_destroy": (_I, [_P]),
    "mrl_net_num_params": (_LL, [_P]),
    "mrl_net_set_params": (_I, [_P, _P, _I, _I, _P]),
    "mrl_net_get_params": (_I, [_P, _P, _I, _P]),
    "mrl_net_set_comm": (_I, [_P, _P]),
    "mrl_net_forward": (_I, [_P, _P, _P, _I, _P]),
    "mrl_net_predict_into_baseline": (_I, [_P, _P, _P]),
    "mrl_net_losses": (_I, [_P, _P, _P, _P]),
    "mrl_net_policy_gradient": (_I, [_P, _P, _P, _I, _P, _P]),
    "mrl_net_fvp": (_I, [_P, _P, _P, _P, _I, _P]),
    "mrl_net_ppo_lossgrad": (_I, [_P, _P, _D, _D, _I, _P, _P, _P, _P]),
    "mrl_net_vf_lossgrad": (_I, [_P, _P, _D, _P, _P, _P]),
    "mrl_net_trpo_step": (_I, [_P, _P, C.POINTER(TrpoCfg), _P, _P, _P]),
    "mrl_net_get_trpo_vectors": (_I, [_P, _P, _P, _P]),
    "mrl_batch_gather": (_I, [_P, _P, _P, _I, _I, _P]),
    "mrl_net_ppo_sgd_step": (_I, [_P, _P, _D, _D, _I, _D, _D, _D, _D, _P]),
    "mrl_net_ppo_sgd_read": (_I, [_P, _P, _P, _P]),
    "mrl_net_adam_reset": (_I, [_P, _P]),
    "mrl_net_ppo_clip_lossgrad": (_I, [_P, _P, _D, _P, _P, _P]),
    "mrl_net_ppo_clip_sgd_step": (_I, [_P, _P, _D, _D, _D, _D, _D, _P]),
    "mrl_population_forward": (_I, [_I, _I, C.POINTER(_I), _I, _P, _LL, _P, _I, _P, _I, _P]),
    "mrl_comm_unique_id": (_I, [_P]),
    "mrl_comm_create": (_I, [C.POINTER(_P), _P, _I, _I, _I]),
    "mrl_comm_destroy": (_I, [_P]),
    "mrl_comm_allreduce_f64": (_I, [_P, _P, _LL, _P]),
    "mrl_comm_p2p_export": (_I, [_P, _LL, _P]),
    "mrl_comm_p2p_connect": (_I, [_P, _P]),
    "mrl_comm_p2p_enable": (_I, [_P, _I]),
    "mrl_rollout_max_envs": (_I, []),
    "mrl_rollout_env_info": (_I, [_I, C.POINTER(_I), C.POINTER(_I), C.POINTER(_I), C.POINTER(_I)]),
    "mrl_rollout_create": (_I, [C.POINTER(_P), _I, _I, _I, _I]),
    "mrl_rollout_destroy": (_I, [_P]),
    "mrl_rollout_run": (_I, [_P, _P, C.c_ulonglong, _I, C.POINTER(ZFilterCfg), _P, _P, C.POINTER(ZFilterCfg), _P, _P,
                             _I, C.POINTER(_LL), _P]),
    "mrl_rollout_run_population": (_I, [_P, _I, C.POINTER(_I), _I, _P, _LL, _I, _I, C.c_ulonglong,
                                        C.POINTER(ZFilterCfg), _P, _P, C.POINTER(ZFilterCfg), _P, _P,
                                        _P, _I, _I, C.POINTER(_LL), _P]),
    "mrl_rollout_read": (_I, [_P, _P, _P, _P, _P, _P, _P, _P]),
    "mrl_rollout_env_compile": (_I, [C.c_char_p, C.c_char_p, _I, _I, _I, _I, C.POINTER(_I)]),
    "mrl_rollout_env_log": (_I, [_I, C.c_char_p, _I]),
    "mrl_cem_search_create": (_I, [C.POINTER(_P), _I, _LL, _I, _LL]),
    "mrl_cem_search_destroy": (_I, [_P]),
    "mrl_cem_search_set_mean": (_I, [_P, _P, _I, _P]),
    "mrl_cem_search_set_var": (_I, [_P, _P, _I, _P]),
    "mrl_cem_search_get_mean": (_I, [_P, _P, _I, _P]),
    "mrl_cem_search_get_var": (_I, [_P, _P, _I, _P]),
    "mrl_cem_search_draw": (_I, [_P, C.c_ulonglong, _D, _D, _P, _I, _P]),
    "mrl_cem_search_rows": (_I, [_P, C.POINTER(_P), C.POINTER(_LL)]),
    "mrl_cem_search_refit": (_I, [_P, _P, _I, _I, _P]),
}


def lib():
    """The loaded library; raises if it is not built (no fallback by design)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: the CUDA extension is not built "
                "(run __graft_entry__.build()); modular_rl_b200 has no CPU fallback")
        L = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        for name, (res, args) in _SIGS.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def exported_symbols():
    return sorted(_SIGS)


def check(rc):
    if rc:
        raise RuntimeError("mrl_b200: " + lib().mrl_last_error().decode(errors="replace"))


def dtype_code(a: np.ndarray) -> int:
    try:
        return _DT[a.dtype]
    except KeyError:
        raise TypeError(f"unsupported dtype {a.dtype}") from None


def as_c(a, dtypes=None) -> np.ndarray:
    """C-contiguous ndarray with one of the supported dtypes (no copy when already so)."""
    a = np.asarray(a)
    if dtypes is not None and a.dtype not in dtypes:
        a = a.astype(dtypes[0])
    if a.dtype not in _DT:
        a = a.astype(np.float64 if a.dtype.kind == "f" else np.int64)
    return np.ascontiguousarray(a)


def ptr(a):
    if a is None:
        return None
    return a.ctypes.data_as(C.c_void_p)
