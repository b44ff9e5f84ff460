"""ctypes binding of libbayesrul_b200.so (the C ABI in include/bayesrul_b200.h).

There is deliberately NO fallback: if the CUDA library is missing or fails to load, every entry
point raises.  (The reference surfaces extension failures as RuntimeError, which is what its Optuna
loop catches: tasks/hpsearch.py:93.)
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BRL_LIB_PATH") or os.path.join(HERE, "lib", "libbayesrul_b200.so")

BRL_MAX_LAYERS = 16

NET_IDS = {"inception": 0, "conv": 1, "linear": 2}
MODE_IDS = {"det": 0, "ws": 1, "lrt": 2, "flipout": 3}
GUIDE_IDS = {"normal": 0, "radial": 1}
ENGINE_IDS = {"simt": 0, "tc": 1}

_fp = C.POINTER(C.c_float)


class BrlNoise(C.Structure):
    _fields_ = [
        ("seed", C.c_uint64),
        ("sample0", C.c_int64),
        ("window0", C.c_int64),
        ("weight_eps", C.c_void_p),
        ("radial_r", C.c_void_p),
        ("lrt_eps", C.c_void_p * BRL_MAX_LAYERS),
        ("flip_in", C.c_void_p * BRL_MAX_LAYERS),
        ("flip_out", C.c_void_p * BRL_MAX_LAYERS),
        ("drop_mask", C.c_void_p * BRL_MAX_LAYERS),
    ]


# name -> (restype, argtypes); the single source of truth for tests/test_cabi.py too
_vp, _i, _i64, _f, _d, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_double, C.c_size_t
_np = C.POINTER(BrlNoise)
SIGNATURES = {
    "brl_version": (_i, []),
    "brl_last_error": (C.c_char_p, []),
    "brl_launch_count": (_i64, []),
    "brl_net_num_params": (_i, [_i]),
    "brl_net_num_layers": (_i, [_i]),
    "brl_net_num_sites": (_i, [_i]),
    "brl_net_site": (_i, [_i, _i, C.POINTER(_i64), C.POINTER(_i), C.POINTER(_i64 * 4)]),
    "brl_net_layer": (_i, [_i, _i, C.POINTER(_i), C.POINTER(_i), C.POINTER(_i), C.POINTER(_f)]),
    "brl_net_flops_fwd": (_i64, [_i]),
    "brl_create": (_i, [C.POINTER(_vp), _i, _i]),
    "brl_destroy": (_i, [_vp]),
    "brl_engine_available": (_i, [_vp, _i]),
    "brl_tc_status": (_i, [_vp]),
    "brl_set_gemm_backend": (_i, [_vp, _i]),
    "brl_set_step_graph": (_i, [_vp, _i]),
    "brl_gemm_status": (_i, []),
    "brl_tc_timing": (_i, [_vp, _i]),
    "brl_tc_timing_read": (_i, [_vp, C.POINTER(C.c_double), C.POINTER(_i64)]),  # double[2], int64[2]
    "brl_tc_trace": (_i, [_vp, _vp]),
    "brl_tt_trace": (_i, [_vp, _vp]),
    "brl_workspace_bytes": (_i64, [_vp, _i64, _i64, _i, _i]),
    "brl_sample_weights": (_i, [_vp, _vp, _vp, _i, _i64, _np, _vp, _vp, _vp, _sz, _vp]),
    "brl_forward": (_i, [_vp, _vp, _i64, _i64, _i, _vp, _vp, _vp, _f, _np, _vp, _i, _vp, _sz, _vp]),
    "brl_predict_moments": (_i, [_vp, _vp, _i64, _i64, _i, _vp, _vp, _f, _np, _vp, _vp, _vp, _vp, _i, _vp, _sz, _vp]),
    "brl_predict_moments_ensemble": (_i, [_vp, _vp, _i64, _i64, _i64, _i, _vp, _vp, _f, _np, _vp, _i, _vp, _sz, _vp]),
    "brl_workspace_bytes_host": (_i64, [_vp, _i64, _i64, _i]),
    "brl_predict_moments_host": (_i, [_vp, _vp, _i64, _i64, _i, _vp, _vp, _f, _np, _vp, _i, _vp, _sz, _vp]),
    "brl_moments": (_i, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "brl_aggregate_predictions": (_i, [_vp, _i64, _i64, _vp, _vp]),
    "brl_elbo_step": (_i, [_vp, _vp, _vp, _i64, _vp, _vp, _i, _i, _i, _f, _f, _i64, _np, _i, _vp, _vp, _vp, _vp, _vp,
                           _vp, _sz, _vp]),
    "brl_elbo_step_ensemble": (_i, [_vp, _vp, _vp, _i64, _i64, _vp, _vp, _i, _i, _i, _f, _f, _i64, _np, _i, _vp, _vp, _vp, _vp,
                                    _vp, _vp, _sz, _vp]),
    "brl_hnn_step": (_i, [_vp, _vp, _vp, _i64, _vp, _f, _np, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "brl_hnn_step_ensemble": (_i, [_vp, _vp, _vp, _i64, _i64, _vp, _f, _np, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "brl_elbo_train_steps": (_i, [_vp, _vp, _vp, _i64, _vp, _i64, _i64, _i64] + [_vp] * 7 + [_i64] + [_f] * 7 + [_i, _i, _i, _f, _f, _i64,
                                 C.c_uint64, _i64, _i64, _vp, _vp, _vp, _sz, _vp]),
    "brl_hnn_train_steps": (_i, [_vp, _vp, _vp, _i64, _vp, _i64, _i64, _i64] + [_vp] * 3 + [_i64] + [_f] * 8 + [C.c_uint64, _i64, _i64,
                                _vp, _vp, _vp, _sz, _vp]),
    "brl_hnn_train_steps_adam": (_i, [_vp, _vp, _vp, _i64, _vp, _i64, _i64, _i64] + [_vp] * 3 + [_i64] + [_d] * 5 + [_f, C.c_uint64, _i64,
                                     _i64, _vp, _vp, _vp, _sz, _vp]),
    "brl_elbo_val_steps": (_i, [_vp, _vp, _vp, _i64, _vp, _i64, _i64, _vp, _vp, _i, _i, _i64, _i, _f, _f, _i64, C.c_uint64, _i64, _i64,
                               _vp, _vp, _vp, _sz, _vp]),
    "brl_mixture_moments": (_i, [_vp, _vp, _i64, _i64, _vp, _vp, _vp]),
    "brl_step_metrics": (_i, [_vp, _vp, _vp, _i64, _vp, _vp, _sz, _vp]),
    "brl_step_metrics_ensemble": (_i, [_vp, _vp, _vp, _i64, _i64, _vp, _vp, _sz, _vp]),
    "brl_clipped_adam_vi_scaled": (_i, [_vp] * 9 + [_i64, _i64] + [_f] * 8 + [_vp]),
    "brl_test_metrics": (_i, [_vp, _vp, _vp, _i64, _vp, _vp, _sz, _vp]),
    "brl_clipped_adam": (_i, [_vp, _vp, _vp, _vp, _i64, _i64, _f, _f, _f, _f, _f, _f, _f, _vp]),
    "brl_clipped_adam_vi": (_i, [_vp] * 9 + [_i64, _i64, _f, _f, _f, _f, _f, _f, _f, _vp]),
    "brl_adam": (_i, [_vp, _vp, _vp, _vp, _i64, _i64, _d, _d, _d, _d, _d, _vp]),
}

_lib = None


def load() -> C.CDLL:
    """Load the shared library (built by bayesrul_b200.build / __graft_entry__.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"bayesrul_b200: CUDA library not built ({LIB_PATH} missing). Run `python -m bayesrul_b200.build` "
            "(nvcc, sm_100a). There is no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing: fail loudly
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        raise RuntimeError(load().brl_last_error().decode() or f"bayesrul_b200 error {rc}")
