"""ctypes binding of csrc/libmxprune.so (the C ABI declared in include/mxprune.h).

There is no fallback: if the library is missing, or a call returns an error code, this raises.
"""
import ctypes
import os
from ctypes import c_float, c_int, c_int64, c_size_t, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
# MXPRUNE_LIB: developer override (e.g. the phase-accounting build csrc/libmxprune_timing.so, `make timing`)
LIB_PATH = os.environ.get("MXPRUNE_LIB") or os.path.join(_HERE, "csrc", "libmxprune.so")
ABI_VERSION = 8

MXP_OK, MXP_E_BADARG, MXP_E_UNSUPPORTED, MXP_E_CUDA = 0, -1, -2, -3
MXP_DT_F32, MXP_DT_BF16, MXP_DT_F16 = 0, 1, 2
MXP_ACT_GELU, MXP_ACT_GELU_TANH = 0, 1

_VIEW = [c_void_p, c_int64, c_int64, c_int64]          # ptr, sB, sH, sN
_ADALN = [c_int] + [c_void_p, c_int64] * 4              # tokens, shift, scale, residual, gate (each with its row stride)
_NORM = [c_int, c_void_p, c_void_p, c_float]            # layer_norm, ln_weight, ln_bias, ln_eps

_SIGNATURES = {
    "mxp_abi_version": (c_int, []),
    "mxp_last_error": (ctypes.c_char_p, []),
    "mxp_last_launch_count": (c_int, []),
    "mxp_set_attention_path": (c_int, [c_int]),
    "mxp_set_predict_path": (c_int, [c_int]),
    "mxp_set_fused_path": (c_int, [c_int]),
    "mxp_debug_fused_timing": (c_int, [c_void_p]),
    "mxp_debug_fused_pingpong": (c_int, [c_int]),
    "mxp_limits": (None, [ctypes.POINTER(c_int), ctypes.POINTER(c_int)]),
    "mxp_quantize_mxint8": (c_int, _VIEW + [c_int] * 6 + [c_void_p] * 4),
    "mxp_quantize_mxint8_dt": (c_int, [c_void_p, c_int, c_int64, c_int64, c_int64] + [c_int] * 6 + [c_void_p] * 4),
    "mxp_exp_sign_approx": (c_int, _VIEW + [c_int] * 6 + [c_void_p] * 2),
    "mxp_predict_scores": (c_int, _VIEW + _VIEW + [c_int] * 7 + [c_void_p] * 2),
    "mxp_predict_topk_workspace_bytes": (c_size_t, [c_int] * 5),
    "mxp_predict_topk": (c_int, _VIEW + _VIEW + [c_int] * 8 + [c_void_p] * 7 + [c_size_t, c_void_p]),
    "mxp_predict_topk_dt": (c_int, _VIEW + _VIEW + [c_int] * 9 + [c_void_p] * 7 + [c_size_t, c_void_p]),
    "mxp_sparse_attention_workspace_bytes": (c_size_t, [c_int] * 5),
    "mxp_sparse_attention": (c_int, [c_void_p] * 4 + _VIEW + [c_void_p] + [c_int] * 5 + [c_float, c_int, c_int]
                             + _VIEW + [c_void_p, c_size_t, c_void_p]),
    "mxp_sparse_attention_dt": (c_int, [c_void_p] * 4 + _VIEW + [c_int, c_void_p] + [c_int] * 5 + [c_float, c_int, c_int]
                                + _VIEW + [c_int, c_void_p, c_size_t, c_void_p]),
    "mxp_pruned_attention_workspace_bytes": (c_size_t, [c_int] * 5),
    "mxp_pruned_attention": (c_int, _VIEW * 3 + [c_int] * 6 + [c_float, c_int, c_int] + _VIEW
                             + [c_void_p, c_void_p, c_size_t, c_void_p]),
    "mxp_pruned_attention_biased": (c_int, _VIEW * 3 + [c_int] * 6 + [c_float, c_int, c_int] + _VIEW
                                    + [c_void_p, ctypes.c_int64, c_void_p, c_void_p, c_size_t, c_void_p]),
    "mxp_pruned_attention_dt": (c_int, _VIEW * 3 + [c_int] * 7 + [c_float, c_int, c_int] + _VIEW
                                + [c_int, c_void_p, c_int64, c_void_p, c_void_p, c_size_t, c_void_p]),
    "mxp_pruned_attention_mode": (c_int, _VIEW * 3 + [c_int] * 7 + [c_float, c_int, c_int] + _VIEW
                                  + [c_void_p, c_int64, c_void_p, c_void_p, c_size_t, c_void_p]),
    "mxp_predict_topk_mode": (c_int, _VIEW * 2 + [c_int] * 7 + [c_float, c_int, c_int]
                              + [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "mxp_pruned_attention_elsa": (c_int, _VIEW * 3 + [c_int] * 5 + [c_void_p, c_float] + [c_float, c_int, c_int] + _VIEW
                                  + [c_void_p, c_void_p, c_size_t, c_void_p]),
    "mxp_predict_topk_elsa": (c_int, _VIEW * 2 + [c_int] * 5 + [c_void_p, c_float] + [c_int, c_int]
                              + [c_void_p, c_void_p, c_void_p]),
    "mxp_mx_linear_weight_bytes": (c_size_t, [c_int, c_int]),
    "mxp_mx_linear_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "mxp_mx_linear_prepare_weight": (c_int, [c_void_p, c_int64, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "mxp_mx_linear": (c_int, [c_void_p, c_int64, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_void_p,
                              c_int64, c_void_p, c_size_t, c_void_p]),
    "mxp_mx_linear_prepare_weight_dt": (c_int, [c_void_p, c_int, c_int64, c_int, c_int, c_int, c_int, c_void_p,
                                                c_void_p]),
    "mxp_mx_linear_dt": (c_int, [c_void_p, c_int, c_int64, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int,
                                 c_void_p, c_int64, c_void_p, c_size_t, c_void_p]),
    "mxp_mx_mlp_workspace_bytes": (c_size_t, [c_int] * 4),
    "mxp_mx_mlp_dt": (c_int, [c_void_p, c_int, c_int64, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_void_p,
                              c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_int64, c_void_p, c_size_t, c_void_p]),
    "mxp_activation_dt": (c_int, [c_void_p, c_int, c_int64, c_int, c_void_p, c_void_p]),
    "mxp_mx_linear_adaln_dt": (c_int, [c_void_p, c_int, c_int64, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_int,
                                       c_int, c_void_p, c_int64] + _ADALN + [c_void_p, c_size_t, c_void_p]),
    "mxp_mx_mlp_adaln_dt": (c_int, [c_void_p, c_int, c_int64, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_int,
                                    c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_int64] + _ADALN
                            + [c_void_p, c_size_t, c_void_p]),
    "mxp_mx_linear_ex_workspace_bytes": (c_size_t, [c_int] * 3),
    "mxp_mx_mlp_ex_workspace_bytes": (c_size_t, [c_int] * 4),
    "mxp_mx_linear_ex_dt": (c_int, [c_void_p, c_int, c_int64, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_int,
                                    c_int, c_void_p, c_int64] + _NORM + _ADALN + [c_void_p, c_size_t, c_void_p]),
    "mxp_mx_mlp_ex_dt": (c_int, [c_void_p, c_int, c_int64, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_int,
                                 c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_int64] + _NORM + _ADALN
                         + [c_void_p, c_size_t, c_void_p]),
    "mxp_layer_norm_dt": (c_int, [c_void_p, c_int, c_int64, c_int, c_int, c_void_p, c_void_p, c_float, c_void_p,
                                  c_void_p, c_void_p, c_void_p]),
    "mxp_pruned_attention_profile": (c_int, _VIEW * 3 + [c_int] * 6 + [c_float, c_int, c_int] + _VIEW
                                     + [c_void_p, c_void_p, c_size_t, c_void_p, ctypes.POINTER(c_float)]),
}

_lib = None


class MxpError(RuntimeError):
    pass


def exported_symbols():
    return sorted(_SIGNATURES)


def load():
    """Load the shared library once; raise loudly if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MxpError(
            f"{LIB_PATH} not found: the CUDA extension is not built. Run "
            "`python -m mx_quantization_b200.build` (needs nvcc; targets sm_100a). "
            "There is no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in _SIGNATURES.items():
        fn = getattr(lib, name)            # AttributeError if the symbol is missing
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.mxp_abi_version() != ABI_VERSION:
        raise MxpError(f"libmxprune ABI {lib.mxp_abi_version()} != binding ABI {ABI_VERSION}; rebuild")
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc == MXP_OK:
        return
    msg = load().mxp_last_error().decode("utf-8", "replace")
    if rc in (MXP_E_BADARG, MXP_E_UNSUPPORTED):
        raise ValueError(f"{what}: {msg}")
    raise MxpError(f"{what}: {msg} (code {rc})")
