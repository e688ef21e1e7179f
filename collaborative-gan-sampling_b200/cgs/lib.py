"""ctypes binding of libcgs.so (include/cgs.h).  No torch types cross this boundary: plain pointers and sizes.

The library is sm_100a-only and has no CPU fallback: if the shared object is missing the import fails loudly,
and every compute entry point returns CGS_ERR_CUDA on a machine without a B200.
"""
from __future__ import annotations

import contextlib
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CGS_LIB_PATH") or os.path.join(_HERE, "libcgs.so")   # override: A/B experiments only

CGS_OK, CGS_ERR_INVALID, CGS_ERR_UNSUPPORTED, CGS_ERR_CUDA, CGS_ERR_WORKSPACE = 0, -1, -2, -3, -4
POLICY_SGD, POLICY_MOMENTUM, POLICY_LADAM = 0, 1, 2
POLICY_IDS = {"sgd": POLICY_SGD, "momentum": POLICY_MOMENTUM, "ladam": POLICY_LADAM}
F32, F64 = 0, 1
LAYER_CONV, LAYER_DECONV, LAYER_FC = 0, 1, 2
LAYER_IDS = {"conv": LAYER_CONV, "deconv": LAYER_DECONV, "fc": LAYER_FC}
ACT_IDS = {"none": 0, "relu": 1, "lrelu": 2, "tanh": 3}
MODE_DETERMINISTIC, MODE_PROBABILISTIC = 0, 1
MATH_TF32_TENSOR, MATH_FP32_SIMT = 0, 1
MATH_IDS = {"tf32": MATH_TF32_TENSOR, "fp32": MATH_FP32_SIMT}
MLP_MAX_LAYERS = 8
MAX_LAYERS = 8

# developer knobs, enum cgs_debug_flag of include/cgs.h (the comments there say what each one does)
DEBUG_SKIP_A_GATHER = 1
DEBUG_SKIP_WEIGHT_TMA = 2
DEBUG_SKIP_MMA = 4
DEBUG_SKIP_A_TMA = 8
DEBUG_SKIP_EPILOGUE = 16
DEBUG_TRACE = 256
DEBUG_GATHER_A = 512
DEBUG_SKIP_STORES = 1024
DEBUG_NO_PREFETCH = 2048
DEBUG_EDGE_GENERAL = 4096
DEBUG_NO_FC_SPLIT = 16384
DEBUG_PDL_ON = 32768
DEBUG_NO_EDGE_PAIR = 65536
DEBUG_NO_HEAD_PARTIALS = 131072
DEBUG_NO_FUSION = 524288
DEBUG_FORCE_FUSION = 1048576
DEBUG_NO_MTILE_PAIRS = 4194304
DEBUG_FORCE_MTILE_PAIRS = 8388608
DEBUG_NO_CTA_PAIRS = 16777216
DEBUG_FORCE_CTA_PAIRS = 33554432
DEBUG_MLP2D_ONE_THREAD = 134217728
DEBUG_MLP2D_CLUSTER = 268435456
DEBUG_PDL_OFF = 536870912
DEBUG_TF32_OPERANDS = 1073741824


class PolicyCfg(C.Structure):
    _fields_ = [("method", C.c_int), ("degree", C.c_int), ("step_size", C.c_double), ("alpha", C.c_double),
                ("beta1", C.c_double), ("beta2", C.c_double), ("beta3", C.c_double), ("eps", C.c_double)]


class MlpDesc(C.Structure):
    _fields_ = [("nlayers", C.c_int), ("nhidden", C.c_int),
                ("weights", C.c_void_p * MLP_MAX_LAYERS), ("biases", C.c_void_p * MLP_MAX_LAYERS)]


class Refine2dCfg(C.Structure):
    _fields_ = [("steps", C.c_int), ("policy", PolicyCfg), ("n_mean", C.c_int64), ("real_sigmoid_mean", C.c_float)]


class LayerDesc(C.Structure):
    _fields_ = [("type", C.c_int), ("k", C.c_int), ("cin", C.c_int), ("cout", C.c_int), ("hin", C.c_int),
                ("win", C.c_int), ("act", C.c_int),
                ("w_fwd", C.c_void_p), ("rows_fwd", C.c_int), ("kcols_fwd", C.c_int),
                ("w_bwd", C.c_void_p), ("rows_bwd", C.c_int), ("kcols_bwd", C.c_int),
                ("bias", C.c_void_p), ("w16_fwd", C.c_void_p), ("w16_bwd", C.c_void_p)]


class NetDesc(C.Structure):
    _fields_ = [("n_layers", C.c_int), ("layers", LayerDesc * MAX_LAYERS)]


class BatchnormDesc(C.Structure):
    _fields_ = [("n_layers", C.c_int), ("gamma", C.c_void_p * MAX_LAYERS), ("beta", C.c_void_p * MAX_LAYERS)]


class RefineCfg(C.Structure):
    _fields_ = [("steps", C.c_int), ("rate", C.c_double), ("method", C.c_int), ("alpha", C.c_double),
                ("mode", C.c_int), ("clip", C.c_int), ("vmin", C.c_float), ("vmax", C.c_float),
                ("math", C.c_int), ("early_exit", C.c_int), ("exit_logit", C.c_float)]


class CgsError(RuntimeError):
    def __init__(self, status, message):
        super().__init__("libcgs status %d: %s" % (status, message))
        self.status = status


_SIGNATURES = {
    "cgs_version": (C.c_int, []),
    "cgs_last_error": (C.c_char_p, []),
    "cgs_launch_count": (C.c_longlong, []),
    "cgs_policy_step": (C.c_int, [C.POINTER(PolicyCfg), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_void_p]),
    "cgs_drs_workspace_bytes": (C.c_size_t, [C.c_int64]),
    "cgs_drs_accept": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p,
                                 C.c_double, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_size_t, C.c_void_p]),
    "cgs_drs_set_score_max": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "cgs_mh_workspace_bytes": (C.c_size_t, [C.c_int64]),
    "cgs_mh_accept": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p,
                                C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_void_p, C.c_size_t, C.c_void_p]),
    "cgs_gather_rows": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "cgs_mlp2d_score": (C.c_int, [C.POINTER(MlpDesc), C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_void_p]),
    "cgs_refine_mlp2d": (C.c_int, [C.POINTER(MlpDesc), C.POINTER(Refine2dCfg), C.c_void_p, C.c_int64, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cgs_refine_max_batch": (C.c_int64, [C.POINTER(NetDesc), C.POINTER(NetDesc)]),
    "cgs_refine_workspace_bytes": (C.c_size_t, [C.POINTER(NetDesc), C.POINTER(NetDesc), C.c_int64]),
    "cgs_refine_conv": (C.c_int, [C.POINTER(NetDesc), C.POINTER(NetDesc), C.POINTER(RefineCfg), C.c_int64,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "cgs_forward_logits_and_grad": (C.c_int, [C.POINTER(NetDesc), C.POINTER(NetDesc), C.c_int, C.c_int64,
                                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.c_size_t, C.c_void_p]),
    "cgs_refine_workspace_bytes_bn": (C.c_size_t, [C.POINTER(NetDesc), C.POINTER(NetDesc), C.POINTER(BatchnormDesc),
                                                   C.c_int64]),
    "cgs_refine_conv_bn": (C.c_int, [C.POINTER(NetDesc), C.POINTER(NetDesc), C.POINTER(BatchnormDesc),
                                     C.POINTER(RefineCfg), C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "cgs_forward_logits_and_grad_bn": (C.c_int, [C.POINTER(NetDesc), C.POINTER(NetDesc), C.POINTER(BatchnormDesc),
                                                 C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                 C.c_void_p, C.c_size_t, C.c_void_p]),
    "cgs_batchnorm_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int]),
    "cgs_batchnorm_forward": (C.c_int, [C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "cgs_batchnorm_backward": (C.c_int, [C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_size_t, C.c_void_p]),
    "cgs_pack_map": (C.c_int64, [C.POINTER(LayerDesc), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]),
    "cgs_debug_gemm_params": (C.c_int64, [C.POINTER(LayerDesc), C.c_int, C.c_int64, C.c_void_p, C.c_int64]),
    "cgs_debug_fusion_plan": (C.c_int64, [C.POINTER(LayerDesc), C.c_int, C.c_int64, C.c_void_p, C.c_int64]),
    "cgs_debug_chain_layout": (C.c_int64, [C.POINTER(NetDesc), C.POINTER(NetDesc), C.c_int, C.c_void_p, C.c_int64]),
    "cgs_debug_chain_pass": (C.c_int, [C.POINTER(NetDesc), C.POINTER(NetDesc), C.c_int, C.c_int64, C.c_int, C.c_int,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(RefineCfg),
                                       C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "cgs_pass_layout": (C.c_int, [C.POINTER(LayerDesc), C.c_int]),
    "cgs_layer_workspace_bytes": (C.c_size_t, [C.POINTER(LayerDesc), C.c_int64]),
    "cgs_layer_forward": (C.c_int, [C.POINTER(LayerDesc), C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_size_t, C.c_void_p]),
    "cgs_layer_backward": (C.c_int, [C.POINTER(LayerDesc), C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "cgs_debug_trace": (C.c_int, [C.c_void_p, C.c_int]),
    "cgs_debug_trace_tc": (C.c_int, [C.c_void_p]),
    "cgs_debug_set_flags": (C.c_int, [C.c_int]),
}

EXPORTED_SYMBOLS = tuple(sorted(_SIGNATURES))

_lib = None


def load():
    """Load libcgs.so (built in-tree by collaborative-gan-sampling_b200/build.py).  Fails loudly if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("libcgs.so not found at %s -- run `python collaborative-gan-sampling_b200/build.py` "
                          "(there is no CPU fallback)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.cgs_version() != 1:
        raise ImportError("libcgs ABI version mismatch")
    _lib = lib
    return lib


@contextlib.contextmanager
def debug_flags(flags):
    """Run the body with the CGS_DEBUG knobs set to `flags` (process-wide), then restore the previous value."""
    lib = load()
    old = lib.cgs_debug_set_flags(flags)
    try:
        yield
    finally:
        lib.cgs_debug_set_flags(old)


def last_error():
    return load().cgs_last_error().decode("utf-8", "replace")


def check(status):
    """Map a cgs_status to the exception the reference would raise at the same spot."""
    if status >= 0:
        return status
    msg = last_error()
    if status == CGS_ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    if status == CGS_ERR_INVALID:
        raise ValueError(msg)
    raise CgsError(status, msg)


def ptr(t):
    """Device (or host) address of a torch tensor / None."""
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr(stream=None):
    import torch
    s = stream if stream is not None else torch.cuda.current_stream()
    return C.c_void_p(s.cuda_stream)
