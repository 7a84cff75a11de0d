"""ctypes binding of libscd_b200.so (the C ABI declared in include/scd_b200.h).

There is no CPU fallback: if the shared library is missing, cannot be loaded or
a call fails, a RuntimeError is raised.
"""
import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
# SCD_B200_LIB selects another build of the same library (the debug build with time stamps, tools/timeline.py)
LIB_PATH = os.environ.get("SCD_B200_LIB") or os.path.join(_HERE, "_lib", "libscd_b200.so")

SCD_E_INVALID = -10001
SCD_E_NODEVICE = -10002
SCD_E_WORKSPACE = -10003

SCD_GEOM_MATCHED_ADJOINT = 0x1     # scd_geom_create_ex flag: A* is the exact transpose of A


class GeomDesc(C.Structure):
    _fields_ = [
        ("n0", C.c_int32), ("n1", C.c_int32),
        ("x_min", C.c_double), ("y_min", C.c_double), ("dx", C.c_double),
        ("n_angles", C.c_int32), ("angles", C.POINTER(C.c_double)),
        ("n_det", C.c_int32), ("s_min", C.c_double), ("ds", C.c_double),
        ("adj_scale", C.c_double),
    ]


# name -> (restype, argtypes); kept in one place so the tests can check that
# every symbol declared in the header is exported.
_F = C.c_void_p   # device float*
SIGNATURES = {
    "scd_geom_create": (C.c_int, [C.POINTER(GeomDesc), C.POINTER(C.c_void_p)]),
    "scd_geom_create_weighted": (C.c_int, [C.POINTER(GeomDesc), C.POINTER(C.c_double), C.POINTER(C.c_void_p)]),
    "scd_geom_create_ex": (C.c_int, [C.POINTER(GeomDesc), C.POINTER(C.c_double), C.c_uint32, C.POINTER(C.c_void_p)]),
    "scd_geom_destroy": (C.c_int, [C.c_void_p]),
    "scd_fp_scratch_bytes": (C.c_size_t, [C.c_void_p, C.c_int]),
    "scd_fp": (C.c_int, [C.c_void_p, _F, _F, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "scd_bp_scratch_bytes": (C.c_size_t, [C.c_void_p, C.c_int]),
    "scd_bp": (C.c_int, [C.c_void_p, _F, _F, C.c_int, C.c_int, C.c_int, C.c_float, _F, C.c_float,
                         C.c_void_p, C.c_size_t, C.c_void_p]),
    "scd_sino_il_buffer_bytes": (C.c_size_t, [C.c_void_p, C.c_int]),
    "scd_fp_il": (C.c_int, [C.c_void_p, _F, _F, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "scd_bp_il": (C.c_int, [C.c_void_p, _F, _F, C.c_int, C.c_int, C.c_int, C.c_float, _F, C.c_float, C.c_void_p]),
    "scd_img_il_bytes": (C.c_size_t, [C.c_void_p, C.c_int]),
    "scd_img_il_pack": (C.c_int, [C.c_void_p, _F, _F, C.c_int, C.c_void_p]),
    "scd_img_il_unpack": (C.c_int, [C.c_void_p, _F, _F, C.c_int, C.c_void_p]),
    "scd_fp_ilimg": (C.c_int, [C.c_void_p, _F, _F, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "scd_bp_ilimg": (C.c_int, [C.c_void_p, _F, _F, C.c_int, C.c_int, C.c_int, C.c_float, _F, C.c_float, C.c_void_p]),
    "scd_sino_weights_pack": (C.c_int, [C.c_void_p, _F, _F, C.c_int, C.c_void_p]),
    "scd_fp_il_w": (C.c_int, [C.c_void_p, _F, _F, _F, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "scd_fp_ilimg_w": (C.c_int, [C.c_void_p, _F, _F, _F, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "scd_cg_workspace_bytes": (C.c_size_t, [C.c_void_p, C.c_int]),
    "scd_cg": (C.c_int, [C.c_void_p, _F, _F, C.c_double, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "scd_cg_w": (C.c_int, [C.c_void_p, _F, _F, _F, C.c_double, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "scd_tweedie_rhs": (C.c_int, [_F, _F, _F, _F, _F, C.c_int, C.c_double, _F, _F, C.c_int, C.c_int64, C.c_void_p]),
    "scd_ddim": (C.c_int, [_F, _F, _F, _F, _F, _F, C.c_int, C.c_double, _F, C.c_int, C.c_int64, C.c_void_p]),
    "scd_dds_step": (C.c_int, [C.c_void_p, _F, _F, _F, _F, _F, _F, _F, C.c_int, C.c_double, C.c_double,
                               C.c_int, _F, _F, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "scd_dds_step_w": (C.c_int, [C.c_void_p, _F, _F, _F, _F, _F, _F, _F, _F, C.c_int, C.c_double, C.c_double,
                                 C.c_int, _F, _F, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "scd_residual_sq_blocks": (C.c_int, [C.c_int64]),
    "scd_residual_sq": (C.c_int, [_F, _F, _F, _F, C.c_int64, C.c_void_p]),
    "scd_residual_sq_w": (C.c_int, [_F, _F, _F, _F, _F, C.c_int64, C.c_void_p]),
    "scd_tv_blocks": (C.c_int, [C.c_int, C.c_int]),
    "scd_tv_loss": (C.c_int, [_F, _F, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "scd_tv_grad": (C.c_int, [_F, _F, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "scd_adapt_workspace_bytes": (C.c_size_t, [C.c_void_p, C.c_int, C.c_int]),
    "scd_adapt_fwd": (C.c_int, [C.c_void_p, _F, _F, _F, _F, _F, _F, C.c_int, C.c_double, C.c_int, C.c_int, C.c_double,
                                _F, _F, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "scd_adapt_bwd": (C.c_int, [C.c_void_p, _F, _F, _F, C.c_int, C.c_double, C.c_int, C.c_int, C.c_double, C.c_double,
                                _F, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "scd_adapt_fwd_w": (C.c_int, [C.c_void_p, _F, _F, _F, _F, _F, _F, _F, _F, C.c_int, C.c_double, C.c_int, C.c_int,
                                  C.c_double, _F, _F, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "scd_adapt_bwd_w": (C.c_int, [C.c_void_p, _F, _F, _F, _F, C.c_int, C.c_double, C.c_int, C.c_int, C.c_double,
                                  C.c_double, _F, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "scd_ramp_filter": (C.c_int, [C.c_void_p, _F, _F, C.c_int, C.c_void_p]),
    "scd_bp_banded": (C.c_int, [C.c_void_p, _F, C.c_int, C.c_int, C.c_int, C.c_float, C.POINTER(C.c_void_p), C.c_int, C.c_int,
                                C.c_void_p, C.c_size_t, C.c_void_p]),
    "scd_bp_il_banded": (C.c_int, [C.c_void_p, _F, C.c_int, C.c_int, C.c_int, C.c_float, C.POINTER(C.c_void_p), C.c_int, C.c_int,
                                   C.c_void_p]),
    "scd_band_reduce": (C.c_int, [_F, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                  C.POINTER(C.c_void_p), C.c_int, C.c_int, _F, C.c_float, C.c_float, C.c_void_p]),
    "scd_fp_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "scd_bp_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "scd_geom_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "scd_launch_count": (C.c_int64, []),
    "scd_launch_count_reset": (None, []),
    "scd_set_tuning": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int]),
    "scd_last_error_string": (C.c_char_p, []),
    "scd_version": (C.c_char_p, []),
}

_lib = None
_lock = threading.Lock()


def load():
    """Load (once) and return the ctypes handle of libscd_b200.so."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found. Build it with `python -m diffusion_models_dev_project_b200.build` "
                "(needs nvcc). This package has no CPU or PyTorch fallback for the ray transform.")
        try:
            lib = C.CDLL(LIB_PATH)
        except OSError as e:  # pragma: no cover
            raise RuntimeError(f"cannot load {LIB_PATH}: {e}") from e
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError if a symbol is missing
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def last_error():
    s = load().scd_last_error_string()
    return s.decode() if s else ""


def check(rc, what):
    if rc != 0:
        raise RuntimeError(f"{what} failed (code {rc}): {last_error()}")
