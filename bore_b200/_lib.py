"""ctypes binding of libbore_b200.so -- the C ABI declared in include/bore_b200.h.

This is the only place the host layer touches native code.  There is NO CPU fallback: if the
library cannot be built/loaded, or no CUDA device is visible, the product path raises.
"""
import ctypes as C
import os
import threading

from . import build as _build

_lock = threading.Lock()
_lib = None

c_int_p = C.POINTER(C.c_int)
c_float_p = C.POINTER(C.c_float)
c_double_p = C.POINTER(C.c_double)
vp = C.c_void_p

# name -> (restype, argtypes); mirrors include/bore_b200.h one to one
SIGNATURES = {
    "bore_abi_version": (C.c_int, []),
    "bore_last_error": (C.c_char_p, []),
    "bore_device_count": (C.c_int, []),
    "bore_mlp_create": (C.c_int, [C.c_int, c_int_p, c_int_p, C.c_int, C.c_int, C.POINTER(vp)]),
    "bore_mlp_destroy": (C.c_int, [vp]),
    "bore_mlp_num_params": (C.c_int, [vp]),
    "bore_mlp_num_models": (C.c_int, [vp]),
    "bore_mlp_set_weights": (C.c_int, [vp, C.c_int, vp]),
    "bore_mlp_get_weights": (C.c_int, [vp, C.c_int, vp]),
    "bore_mlp_set_adam_state": (C.c_int, [vp, C.c_int, vp, vp, C.c_int64]),
    "bore_mlp_get_adam_state": (C.c_int, [vp, C.c_int, vp, vp, C.POINTER(C.c_int64)]),
    "bore_mlp_reset_optimizer": (C.c_int, [vp, C.c_int, C.c_int, vp]),
    "bore_mlp_set_optimizer": (C.c_int, [vp, C.c_float, C.c_float, C.c_float, C.c_float]),
    "bore_mlp_set_optimizer_kind": (C.c_int, [vp, C.c_int, vp]),
    "bore_mlp_get_nadam_cache": (C.c_int, [vp, C.c_int, C.POINTER(C.c_float)]),
    "bore_mlp_set_nadam_cache": (C.c_int, [vp, C.c_int, C.c_float]),
    "bore_mlp_set_fit_mode": (C.c_int, [vp, C.c_int]),
    "bore_mlp_params_dev": (C.c_int, [vp, C.POINTER(vp)]),
    "bore_mlp_predict": (C.c_int, [vp, C.c_int, vp, C.c_int, vp, vp]),
    "bore_mlp_value_and_grad": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, vp, C.c_int, vp, vp, vp]),
    "bore_mlp_fit": (C.c_int, [vp, C.c_int, C.c_int, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int,
                               vp, C.c_int, vp, vp]),
    "bore_mlp_evaluate": (C.c_int, [vp, C.c_int, vp, vp, C.c_int, vp, vp]),
    "bore_mlp_fit_weighted": (C.c_int, [vp, C.c_int, C.c_int, vp, vp, vp, C.c_int, C.c_int, C.c_float,
                                        C.c_float, C.c_int, C.c_int, vp, C.c_int, vp, vp]),
    "bore_mlp_evaluate_weighted": (C.c_int, [vp, C.c_int, vp, vp, vp, C.c_float, C.c_float, C.c_int,
                                             vp, vp]),
    "bore_mlp_fit_ragged": (C.c_int, [vp, C.c_int, C.c_int, vp, vp, vp, vp, vp, C.c_float, C.c_float, C.c_int,
                                      vp, vp, vp]),
    "bore_mlp_set_regularizers": (C.c_int, [vp, vp, vp]),
    "bore_lbfgsb_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "bore_lbfgsb_minimize_workspace_bytes": (C.c_size_t, [vp, C.c_int, C.c_int]),
    "bore_lbfgsb_set_mode": (C.c_int, [C.c_int]),
    "bore_lbfgsb_minimize": (C.c_int, [vp, C.c_int, C.c_int, vp, C.c_int, vp, vp, C.c_int,
                                       C.c_double, C.c_double, C.c_int, C.c_int, C.c_int,
                                       vp, C.c_size_t, vp, vp, vp, vp, vp, vp,
                                       c_int_p, C.POINTER(C.c_longlong), vp]),
    "bore_lbfgsb_profile": (C.c_int, [C.c_int]),
    "bore_lbfgsb_last_profile": (C.c_int, [c_double_p]),
    "bore_lbfgsb_init": (C.c_int, [vp, C.c_int, C.c_int, vp, vp, C.c_int, C.c_double, C.c_double,
                                   C.c_int, C.c_int, C.c_int, vp, C.c_size_t, vp, vp, C.c_int, vp]),
    "bore_lbfgsb_step": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, vp, vp, vp, c_int_p,
                                   C.c_int, vp]),
    "bore_lbfgsb_results": (C.c_int, [C.c_int, C.c_int, vp, vp, vp, vp, vp, vp, vp, C.c_int, vp]),
    "bore_topk_smallest": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, vp, vp, C.c_size_t, C.c_int, vp]),
    "bore_topk_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "bore_select_best": (C.c_int, [vp, vp, vp, C.c_int, C.c_int64, vp, C.c_int, vp]),
    "bore_mlp_predict_multi": (C.c_int, [vp, C.c_int, C.c_int, vp, C.c_int, vp, vp]),
    "bore_topk_smallest_groups": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, C.c_int, vp]),
    "bore_lbfgsb_minimize_multi": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, C.c_int,
                                             C.c_double, C.c_double, C.c_int, C.c_int, C.c_int,
                                             vp, C.c_size_t, vp, vp, vp, vp, vp, vp,
                                             c_int_p, C.POINTER(C.c_longlong), vp]),
    "bore_select_best_groups": (C.c_int, [vp, vp, vp, C.c_int, C.c_int, vp, C.c_int, vp]),
    "bore_allreduce_maxloc": (C.c_int, [vp, vp, vp]),
    "bore_quantile_labels": (C.c_int, [vp, C.c_int, C.c_int, C.c_double, vp, vp, vp, C.c_int, vp]),
    "bore_is_duplicate": (C.c_int, [vp, C.c_int, C.c_int, vp, C.c_int, C.c_int, C.c_double, C.c_double,
                                    vp, vp, C.c_int, vp]),
    "bore_quantile_labels_ragged": (C.c_int, [vp, C.c_int, vp, C.c_double, vp, vp, vp, C.c_int, vp]),
    "bore_is_duplicate_ragged": (C.c_int, [vp, C.c_int, C.c_int, vp, vp, C.c_int, C.c_double, C.c_double,
                                           vp, vp, C.c_int, vp]),
    "bore_truncnorm_distort": (C.c_int, [vp, C.c_int, C.c_int, C.c_double, vp, vp, vp, vp, C.c_int, vp]),
    "bore_svgd_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "bore_svgd_maximize": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, vp, C.c_int, vp, vp, C.c_double, C.c_int,
                                     C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double,
                                     vp, C.c_size_t, vp]),
    "bore_svgd_step": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, vp, vp, C.c_int, vp, vp, C.c_double, C.c_int,
                                 C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double,
                                 vp, vp, C.c_int, vp]),
    "bore_svgd_kernel_value_and_grad": (C.c_int, [vp, C.c_int, C.c_int, C.c_double, vp, vp, C.c_int, vp]),
    "bore_lstm_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(vp)]),
    "bore_lstm_destroy": (C.c_int, [vp]),
    "bore_lstm_num_params": (C.c_int, [vp]),
    "bore_lstm_set_weights": (C.c_int, [vp, vp]),
    "bore_lstm_get_weights": (C.c_int, [vp, vp]),
    "bore_lstm_set_adam_state": (C.c_int, [vp, vp, vp, C.c_int64]),
    "bore_lstm_get_adam_state": (C.c_int, [vp, vp, vp, C.POINTER(C.c_int64)]),
    "bore_lstm_set_optimizer_kind": (C.c_int, [vp, C.c_int, vp]),
    "bore_lstm_get_nadam_cache": (C.c_int, [vp, C.POINTER(C.c_float)]),
    "bore_lstm_set_nadam_cache": (C.c_int, [vp, C.c_float]),
    "bore_lstm_set_regularizers": (C.c_int, [vp, vp]),
    "bore_lstm_predict_sequences": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_float, C.c_int, vp, vp]),
    "bore_lstm_predict": (C.c_int, [vp, vp, C.c_int, C.c_int, vp, vp]),
    "bore_lstm_value_and_grad": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, vp, C.c_int, C.c_int, vp, vp, vp, vp]),
    "bore_lstm_fit": (C.c_int, [vp, vp, vp, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, vp, vp, vp]),
    "bore_lstm_evaluate": (C.c_int, [vp, vp, vp, C.c_int, C.c_int, C.c_float, vp, vp]),
    "bore_bench_ffma_peak": (C.c_int, [C.c_int, C.c_int, c_double_p]),
    "bore_mt19937_uniform": (C.c_int, [vp, c_int_p, vp, vp, C.c_int, C.c_longlong, vp]),
}


class BoreNativeError(RuntimeError):
    pass


def lib_path():
    return _build.LIB_PATH


def load(build_if_missing=True):
    """Load (building first if the .so is absent) and type every exported symbol."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = _build.LIB_PATH
        if not os.path.exists(path) or _build.needs_build():
            # a library older than csrc/ or the header is never loaded silently
            if not build_if_missing:
                raise BoreNativeError(f"{path} is missing or stale; run `python -m bore_b200.build`")
            _build.build_library()
        lib = C.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError => header/library drift: fail loudly
            fn.restype = res
            fn.argtypes = args
        if lib.bore_abi_version() != 1:
            raise BoreNativeError("libbore_b200.so ABI version mismatch")
        _lib = lib
        return lib


def check(rc):
    if rc != 0:
        msg = load().bore_last_error()
        raise BoreNativeError(msg.decode() if msg else f"native call failed ({rc})")


def require_cuda():
    """The product path has no CPU fallback: fail loudly when no GPU is visible."""
    lib = load()
    if lib.bore_device_count() <= 0:
        raise BoreNativeError("bore_b200: no CUDA device visible; the BORE-MLP hot path has no "
                              "CPU fallback (build: sm_100a only)")
    return lib
