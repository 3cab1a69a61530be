"""ctypes binding of libgbnf_b200.so -- the C ABI declared in include/gbnf.h.

There is no CPU fallback anywhere in this package: if the shared library cannot be loaded the import of the
compute entry points raises, and gbnf_create itself refuses to run without a CUDA device.
"""
import ctypes as C
import os

from . import build as _build

GBNF_MAX_LAYERS = 6

KIND = {"realnvp": 0, "glow": 1}
ACT = {"tanh": 0, "relu": 1, "mixed": 2, "residual": 3}
COUPLING = {"affine": 0, "additive": 1}
BASE_STD_NORMAL, BASE_DIAG_NORMAL = 0, 1
GEMM = {"fp32": 0, "f16": 1, "f16fast": 2}
WEIGHTS = {"density": 0, "toy": 1}
MIX_SIMPLEX, MIX_RAW_RHO, MIX_GEOMETRIC = 0, 1, 2


class GbnfError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"gbnf error {code}: {msg}")
        self.code = code


class Config(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("kind", "D", "h", "K", "C", "depth", "act", "coupling", "base", "gemm_mode",
                                         "device", "glow_invconv")]


class StepParams(C.Structure):
    _fields_ = [("an_bias", C.c_void_p), ("an_logs", C.c_void_p), ("perm", C.c_void_p),
                ("bn_log_gamma", C.c_void_p), ("bn_beta", C.c_void_p), ("bn_mean", C.c_void_p), ("bn_var", C.c_void_p),
                ("W", (C.c_void_p * GBNF_MAX_LAYERS) * 2), ("b", (C.c_void_p * GBNF_MAX_LAYERS) * 2),
                ("invconv_w", C.c_void_p), ("invconv_winv", C.c_void_p), ("invconv_logdet", C.c_void_p)]


class StepGrads(C.Structure):
    _fields_ = [("an_bias", C.c_void_p), ("an_logs", C.c_void_p),
                ("W", (C.c_void_p * GBNF_MAX_LAYERS) * 2), ("b", (C.c_void_p * GBNF_MAX_LAYERS) * 2)]


class ComponentParams(C.Structure):
    _fields_ = [("flip_init", C.c_int32), ("n_steps", C.c_int32), ("steps", C.POINTER(StepParams))]


class Info(C.Structure):
    _fields_ = [("gemm_mode", C.c_int32), ("rows_per_cta", C.c_int32), ("smem_bytes", C.c_int32), ("tmem_cols", C.c_int32),
                ("num_sms", C.c_int32), ("grid", C.c_int32), ("packed_bytes", C.c_int64), ("launches", C.c_int64),
                ("pipelined", C.c_int32), ("two_chain", C.c_int32)]


# name -> (restype, argtypes); mirrors include/gbnf.h one to one (tests/test_abi.py checks the two stay in sync)
_vp, _i32, _i64, _f32, _f64 = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_double
SIGNATURES = {
    "gbnf_create": (C.c_int, [C.POINTER(_vp), C.POINTER(Config)]),
    "gbnf_destroy": (None, [_vp]),
    "gbnf_last_error": (C.c_char_p, []),
    "gbnf_abi_version": (C.c_int, []),
    "gbnf_pack_component": (C.c_int, [_vp, _i32, C.POINTER(ComponentParams), _vp]),
    "gbnf_set_base": (C.c_int, [_vp, _vp, _vp, _vp]),
    "gbnf_component_logq": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _vp, _vp, _vp, _vp]),
    "gbnf_component_inverse": (C.c_int, [_vp, _vp, _i64, _i32, _vp, _vp, _vp]),
    "gbnf_mixture_inverse": (C.c_int, [_vp, _vp, _i64, _vp, _i32, _vp, _vp, _vp]),
    "gbnf_mixture_logdensity": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _vp, _i32, _i32, _vp, _vp]),
    "gbnf_fused_eval": (C.c_int, [_vp, _vp, _i64, _i32, _vp, _i32, _i32, _vp, _vp, _vp]),
    "gbnf_boost_weights": (C.c_int, [_vp, _vp, _i64, _f32, _f32, _i32, _vp, _vp, _vp]),
    "gbnf_weight_stats": (C.c_int, [_vp, _vp, _i64, _vp, _vp]),
    "gbnf_weight_apply": (C.c_int, [_vp, _vp, _i64, _vp, _f32, _f32, _i32, _vp, _vp, _vp]),
    "gbnf_weight_renorm": (C.c_int, [_vp, _vp, _i64, _vp, _i32, _vp]),
    "gbnf_component_backward": (C.c_int, [_vp, _i32, C.POINTER(ComponentParams), _vp, _i64, _vp, _vp, C.POINTER(StepGrads), _vp, _vp]),
    "gbnf_component_inverse_backward": (C.c_int, [_vp, _i32, C.POINTER(ComponentParams), _vp, _i64, _vp, _vp, C.POINTER(StepGrads),
                                                  _vp, _vp]),
    "gbnf_mixture_inverse_backward": (C.c_int, [_vp, C.POINTER(ComponentParams), _vp, _i64, _vp, _i32, _vp, _vp,
                                                C.POINTER(C.POINTER(StepGrads)), _vp, _vp]),
    "gbnf_comm_local_handle": (C.c_int, [_vp, _i64, _vp]),
    "gbnf_comm_init": (C.c_int, [_vp, _i32, _i32, _vp]),
    "gbnf_comm_destroy": (C.c_int, [_vp]),
    "gbnf_boost_weights_dist": (C.c_int, [_vp, _vp, _i64, _f32, _f32, _i32, _vp, _vp, _vp]),
    "gbnf_mixture_component_parallel": (C.c_int, [_vp, _vp, _i64, _i32, _vp, _i32, _i32, _vp, _vp]),
    "gbnf_resample": (C.c_int, [_vp, _vp, _i64, _vp, _i64, _vp, _vp]),
    "gbnf_gather_rows": (C.c_int, [_vp, _vp, _i32, _vp, _i64, _vp, _vp]),
    "gbnf_actnorm_init": (C.c_int, [_vp, _i64, _i32, C.c_float, _vp, _vp, _vp]),
    "gbnf_sample_component": (C.c_int, [C.POINTER(_f32), _i32, _f64, _i32, C.POINTER(_i32)]),
    "gbnf_get_info": (C.c_int, [_vp, C.POINTER(Info)]),
    "gbnf_check_status": (C.c_int, [_vp, _vp]),
    "gbnf_get_profile": (C.c_int, [_vp, C.POINTER(C.c_int64)]),
    "gbnf_get_trace": (C.c_int, [_vp, C.POINTER(C.c_int64)]),
}

_LIB = None


def lib_path():
    return _build.LIB_PATH


def load(rebuild_if_stale=True):
    """Load (building first when the in-tree .so is missing or older than its sources and nvcc is present)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = _build.LIB_PATH
    if rebuild_if_stale and _build.is_stale():
        try:
            _build.build()
        except Exception as e:  # no nvcc on the box and no prebuilt library: nothing can run
            if not os.path.exists(path):
                raise RuntimeError(f"libgbnf_b200.so is missing and could not be built ({e}); "
                                   "this package has no CPU or PyTorch fallback") from e
    if not os.path.exists(path):
        raise RuntimeError("libgbnf_b200.so is missing; run `python __graft_entry__.py build` (no CPU fallback exists)")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError here == ABI drift, fail loudly
        fn.restype = res
        fn.argtypes = args
    if lib.gbnf_abi_version() != 2:
        raise RuntimeError("libgbnf_b200.so ABI version mismatch")
    _LIB = lib
    return lib


def check(code):
    if code != 0:
        raise GbnfError(code, load().gbnf_last_error().decode("utf-8", "replace"))
