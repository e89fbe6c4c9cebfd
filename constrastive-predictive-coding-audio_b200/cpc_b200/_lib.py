"""ctypes binding of ``libcpc_b200.so`` (the C-ABI in ``include/cpc_b200.h``).

There is no CPU implementation behind any of these calls: when the shared library is missing the import
of an op raises, and when a tensor is not on a B200 the call raises.  PyTorch only provides device
memory and the stream.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "lib", "libcpc_b200.so")

CQT_MAX_GROUPS = 16
CQT_COMPLEX, CQT_LOGPOW, CQT_LOGPOW_PHASE = 0, 1, 2
SCORE_LINEAR, SCORE_SOFTPLUS, SCORE_DIFFERENCE = 0, 1, 2
CQT_FLAG_NO_TENSOR = 1
CQT_FLAG_HALF_OPERANDS = 2
CONV_FLAG_CUDA_CORE, CONV_FLAG_NO_TALL, CONV_FLAG_NO_SMALLK, CONV_FLAG_NO_FUSED_DGRAD = 1, 2, 4, 8
CONV_FLAG_NO_MMA_SMALL_WGRAD = 16
INFONCE_FLAG_NO_TENSOR = 1
INFONCE_OUT_FLOATS = 4
ABI_VERSION = 7


class CqtParams(ctypes.Structure):
    _fields_ = [("batch", ctypes.c_int32), ("n_samples", ctypes.c_int32), ("x_pitch", ctypes.c_int32),
                ("n_bins", ctypes.c_int32), ("hop", ctypes.c_int32), ("n_frames", ctypes.c_int32),
                ("n_groups", ctypes.c_int32),
                ("kernel_size", ctypes.c_int32 * CQT_MAX_GROUPS), ("bin_lo", ctypes.c_int32 * CQT_MAX_GROUPS),
                ("bin_hi", ctypes.c_int32 * CQT_MAX_GROUPS), ("weight_offset", ctypes.c_int64 * CQT_MAX_GROUPS),
                ("mode", ctypes.c_int32), ("pool_t", ctypes.c_int32),
                ("eps", ctypes.c_float), ("log_offset", ctypes.c_float), ("norm", ctypes.c_float),
                ("power", ctypes.c_float), ("flags", ctypes.c_int32)]


class ConvParams(ctypes.Structure):
    _fields_ = [("batch", ctypes.c_int32), ("c_in", ctypes.c_int32), ("h_in", ctypes.c_int32),
                ("w_in", ctypes.c_int32), ("c_out", ctypes.c_int32), ("h_out", ctypes.c_int32),
                ("w_out", ctypes.c_int32), ("kh", ctypes.c_int32), ("kw", ctypes.c_int32),
                ("stride_h", ctypes.c_int32), ("stride_w", ctypes.c_int32), ("pad_top", ctypes.c_int32),
                ("pad_left", ctypes.c_int32), ("relu", ctypes.c_int32), ("precision", ctypes.c_int32),
                ("flags", ctypes.c_int32)]


class BnParams(ctypes.Structure):
    _fields_ = [("batch", ctypes.c_int32), ("channels", ctypes.c_int32), ("height", ctypes.c_int32),
                ("width", ctypes.c_int32), ("res_height", ctypes.c_int32), ("res_width", ctypes.c_int32),
                ("res_off_h", ctypes.c_int32), ("res_off_w", ctypes.c_int32), ("relu", ctypes.c_int32),
                ("outer_relu", ctypes.c_int32), ("training", ctypes.c_int32), ("eps", ctypes.c_float),
                ("momentum", ctypes.c_float), ("packed_planes", ctypes.c_int32)]


class PoolParams(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in ("batch", "channels", "h_in", "w_in", "h_out", "w_out", "kernel",
                                              "ceil_mode")]


class InfoNceParams(ctypes.Structure):
    _fields_ = [("batch", ctypes.c_int32), ("steps", ctypes.c_int32), ("enc", ctypes.c_int32),
                ("all_steps", ctypes.c_int32), ("score_kind", ctypes.c_int32), ("regularization", ctypes.c_float),
                ("tgt_stride_b", ctypes.c_int64), ("tgt_stride_e", ctypes.c_int64), ("tgt_stride_k", ctypes.c_int64),
                ("precision", ctypes.c_int32), ("flags", ctypes.c_int32)]


class AdamParams(ctypes.Structure):
    _fields_ = [("lr", ctypes.c_double), ("beta1", ctypes.c_double), ("beta2", ctypes.c_double), ("eps", ctypes.c_double),
                ("weight_decay", ctypes.c_double), ("grad_scale", ctypes.c_float), ("maximize", ctypes.c_int32)]


# name -> (restype, argtypes); exactly the symbols include/cpc_b200.h declares
_P = ctypes.c_void_p
SIGNATURES = {
    "cpc_status_string": (ctypes.c_char_p, [ctypes.c_int]),
    "cpc_abi_version": (ctypes.c_int, []),
    "cpc_runtime_check": (ctypes.c_int, []),
    "cpc_launch_count": (ctypes.c_uint64, []),
    "cpc_launch_count_reset": (None, []),
    "cpc_cqt_workspace_bytes": (ctypes.c_size_t, [ctypes.POINTER(CqtParams)]),
    "cpc_cqt_fwd": (ctypes.c_int, [_P, _P, _P, _P, _P, ctypes.POINTER(CqtParams), _P, ctypes.c_size_t, _P]),
    "cpc_cqt_packed_filter_bytes": (ctypes.c_size_t, [ctypes.POINTER(CqtParams)]),
    "cpc_cqt_pack_filters": (ctypes.c_int, [_P, _P, ctypes.POINTER(CqtParams), _P]),
    "cpc_cqt_fwd_ex": (ctypes.c_int, [_P, _P, _P, _P, _P, _P, ctypes.POINTER(CqtParams), _P, ctypes.c_size_t, _P]),
    "cpc_conv_workspace_bytes": (ctypes.c_size_t, [ctypes.POINTER(ConvParams), ctypes.c_int]),
    "cpc_conv_fwd": (ctypes.c_int, [_P, _P, _P, _P, ctypes.POINTER(ConvParams), _P, ctypes.c_size_t, _P]),
    "cpc_conv_dgrad": (ctypes.c_int, [_P, _P, _P, ctypes.POINTER(ConvParams), _P, ctypes.c_size_t, _P]),
    "cpc_conv_wgrad": (ctypes.c_int, [_P, _P, _P, _P, ctypes.POINTER(ConvParams), _P, ctypes.c_size_t, _P]),
    "cpc_dwconv_fwd": (ctypes.c_int, [_P, _P, _P, ctypes.POINTER(ConvParams), _P]),
    "cpc_dwconv_dgrad": (ctypes.c_int, [_P, _P, _P, ctypes.POINTER(ConvParams), _P]),
    "cpc_dwconv_wgrad": (ctypes.c_int, [_P, _P, _P, ctypes.POINTER(ConvParams), _P]),
    "cpc_conv_kernel_family": (ctypes.c_int, [ctypes.POINTER(ConvParams), ctypes.c_int]),
    "cpc_conv_packed_bytes": (ctypes.c_size_t, [ctypes.POINTER(ConvParams), ctypes.c_int]),
    "cpc_conv_pack": (ctypes.c_int, [_P, _P, ctypes.POINTER(ConvParams), ctypes.c_int, _P]),
    "cpc_conv_pack_dy": (ctypes.c_int, [_P, _P, _P, ctypes.POINTER(ConvParams), _P]),
    "cpc_conv_fwd_ex": (ctypes.c_int, [_P, _P, _P, _P, ctypes.POINTER(ConvParams), _P, _P, ctypes.c_size_t, _P]),
    "cpc_conv_dgrad_ex": (ctypes.c_int, [_P, _P, _P, ctypes.POINTER(ConvParams), _P, _P, ctypes.c_size_t, _P]),
    "cpc_conv_wgrad_ex": (ctypes.c_int, [_P, _P, _P, _P, ctypes.POINTER(ConvParams), _P, _P, _P, ctypes.c_size_t, _P]),
    "cpc_bn_relu_workspace_bytes": (ctypes.c_size_t, [ctypes.POINTER(BnParams)]),
    "cpc_bn_relu_fwd": (ctypes.c_int, [_P] * 9 + [ctypes.POINTER(BnParams), _P, ctypes.c_size_t, _P]),
    "cpc_bn_relu_bwd": (ctypes.c_int, [_P] * 11 + [ctypes.POINTER(BnParams), _P, ctypes.c_size_t, _P]),
    "cpc_bn_packed_bytes": (ctypes.c_size_t, [ctypes.POINTER(BnParams)]),
    "cpc_bn_relu_fwd_packed": (ctypes.c_int, [_P] * 9 + [ctypes.POINTER(BnParams), _P, ctypes.c_size_t, _P]),
    "cpc_bn_relu_bwd_packed": (ctypes.c_int, [_P] * 12 + [ctypes.POINTER(BnParams), _P, ctypes.c_size_t, _P]),
    "cpc_bn_mask_bytes": (ctypes.c_size_t, [ctypes.POINTER(BnParams)]),
    "cpc_bn_relu_fwd_mask": (ctypes.c_int, [_P] * 10 + [ctypes.POINTER(BnParams), _P, ctypes.c_size_t, _P]),
    "cpc_bn_relu_bwd_mask": (ctypes.c_int, [_P] * 12 + [ctypes.POINTER(BnParams), _P, ctypes.c_size_t, _P]),
    "cpc_bn_relu_bwd_packed_mask": (ctypes.c_int, [_P] * 13 + [ctypes.POINTER(BnParams), _P, ctypes.c_size_t, _P]),
    "cpc_maxpool_fwd": (ctypes.c_int, [_P, _P, ctypes.POINTER(PoolParams), _P]),
    "cpc_maxpool_bwd": (ctypes.c_int, [_P, _P, _P, ctypes.POINTER(PoolParams), _P]),
    "cpc_maxpool_bwd_accumulate": (ctypes.c_int, [_P, _P, _P, ctypes.POINTER(PoolParams), _P]),
    "cpc_infonce_workspace_bytes": (ctypes.c_size_t, [ctypes.POINTER(InfoNceParams), ctypes.c_int]),
    "cpc_infonce_fwd": (ctypes.c_int, [_P, _P, _P, _P, ctypes.POINTER(InfoNceParams), _P, ctypes.c_size_t, _P]),
    "cpc_infonce_bwd": (ctypes.c_int, [_P, _P, _P, _P, _P, _P, ctypes.POINTER(InfoNceParams), _P, ctypes.c_size_t, _P]),
    "cpc_infonce_validate": (ctypes.c_int, [_P, _P, _P, ctypes.POINTER(InfoNceParams), _P, ctypes.c_size_t, _P]),
    "cpc_adam_step": (ctypes.c_int, [ctypes.c_int32, _P, _P, _P, _P, _P, _P, ctypes.POINTER(AdamParams), _P]),
}

_lib = None


class CpcError(RuntimeError):
    pass


def load():
    """Load the shared library (once).  Raises CpcError when it has not been built -- there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CpcError("libcpc_b200.so not found at %s -- run `python __graft_entry__.py` (build()) first; "
                       "cpc_b200 has no CPU/PyTorch fallback" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.cpc_abi_version() != ABI_VERSION:
        raise CpcError("libcpc_b200.so ABI version %d != expected %d; rebuild" % (lib.cpc_abi_version(), ABI_VERSION))
    _lib = lib
    return lib


def check(status, what):
    if status != 0:
        raise CpcError("%s failed: %s (%d)" % (what, load().cpc_status_string(status).decode(), status))


def launch_count():
    return int(load().cpc_launch_count())


def reset_launch_count():
    load().cpc_launch_count_reset()
