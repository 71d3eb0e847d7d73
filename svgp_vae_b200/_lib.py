"""ctypes binding of libsvgp_b200.so (the C ABI declared in include/svgp_b200.h).

There is no CPU fallback: if the library is missing or the device is not sm_100 the
product path raises.  Build the library with ``python -m svgp_vae_b200.build`` (or
``__graft_entry__.build()``); the .so stays in-tree so that it travels to the GPU box.
"""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsvgp_b200.so")

SVGP_K_NONE, SVGP_K_SE, SVGP_K_EXPSIN, SVGP_K_LINEAR, SVGP_K_COSINE = 0, 1, 2, 3, 4
SVGP_K_MATERN12, SVGP_K_MATERN32, SVGP_K_MATERN52 = 5, 6, 7
IMPL_AUTO, IMPL_SIMT, IMPL_TC, IMPL_TC_I8, IMPL_TC_I8_D3, IMPL_TC_I8_O4 = 0, 1, 2, 3, 4, 5


class KopStruct(ctypes.Structure):
    """struct svgp_kop (include/svgp_b200.h)."""
    _fields_ = [("K", c_void_p), ("Kh", c_void_p), ("Kl", c_void_p), ("Kth", c_void_p), ("Ktl", c_void_p),
                ("kscale", c_void_p), ("N", c_int64), ("M", c_int64), ("ldk", c_int64), ("ldkh", c_int64),
                ("ldkt", c_int64), ("Kr", c_void_p), ("rscale", c_void_p), ("Kc", c_void_p), ("cscale", c_void_p),
                ("ldkr", c_int64)]


class SvgpLibraryError(RuntimeError):
    pass


_P = c_void_p
# name -> argtypes (restype is int unless listed in _RESTYPE); mirrors include/svgp_b200.h one to one
SIGNATURES = {
    "svgp_version": [],
    "svgp_last_error": [],
    "svgp_device_ok": [],
    "svgp_kernel_fwd": [_P, c_int64, c_int64, _P, c_int64, c_int64, c_int, c_int, c_int, c_int, _P,
                        _P, c_int64, _P, _P, c_int64, _P, _P, c_int64, _P, _P],
    "svgp_kernel_bwd": [_P, c_int64, c_int64, _P, c_int64, c_int64, c_int, c_int, c_int, c_int, _P,
                        _P, c_int64, _P, _P, _P, _P],
    "svgp_kernel_diag_fwd": [_P, c_int64, _P, c_int64, c_int64, c_int, c_int, c_int, c_int, _P, _P, _P],
    "svgp_kernel_diag_bwd": [_P, c_int64, _P, c_int64, c_int64, c_int, c_int, c_int, c_int, _P, _P, _P, _P, _P, _P],
    "svgp_gather_rows": [_P, c_int64, c_int64, _P, c_int64, c_int64, _P, c_int64, _P],
    "svgp_scatter_add_rows": [_P, c_int64, _P, c_int64, c_int64, c_int64, _P, c_int64, _P],
    "svgp_syrk_ws_floats": [c_int64, c_int64, c_int64],
    "svgp_syrk": [POINTER(KopStruct), _P, c_int64, c_int64, _P, c_int, c_int64, _P, _P],
    "svgp_gemm_tn": [POINTER(KopStruct), _P, c_int64, c_int64, _P, _P],
    "svgp_gemm_nn": [POINTER(KopStruct), _P, c_int64, c_int64, _P, c_int64, _P],
    "svgp_gemm_nn_tc": [POINTER(KopStruct), _P, _P, _P, c_int64, _P, c_int64, _P],
    "svgp_rowquad": [POINTER(KopStruct), _P, _P, _P, c_int64, c_int, _P, c_int64, c_int, _P],
    "svgp_scaled_gemm": [POINTER(KopStruct), _P, c_int64, _P, _P, _P, c_int64, _P, c_int64, c_int, _P, c_int64, c_int64,
                         c_int, _P],
    "svgp_gemm_f32": [c_int64, c_int64, c_int64, _P, c_int64, _P, c_int64, _P, c_int64, c_int, _P],
    "svgp_split_f16": [_P, c_int64, c_int64, _P, _P, _P, _P],
    "svgp_i8_ldkr": [c_int64],
    "svgp_i8_nblk": [c_int64],
    "svgp_kernel_fwd_f64": [_P, c_int64, c_int64, _P, c_int64, c_int64, c_int, c_int, c_int, c_int, _P, _P, c_int64, _P],
    "svgp_kernel_fwd_i8": [_P, c_int64, c_int64, _P, c_int64, c_int64, c_int, c_int, c_int, c_int, _P,
                           _P, _P, c_int64, _P, c_int64, _P, _P, _P, _P, _P, _P],
    "svgp_split_i8": [_P, c_int64, c_int64, c_int64, c_int, _P, c_int64, _P, _P],
    "svgp_scaled_gemm_i8": [POINTER(KopStruct), _P, c_int64, _P, c_int64, _P, c_int64, c_int64, _P, c_int64, c_int, _P, c_int64,
                            c_int64, c_int64, _P, _P, _P],
    "svgp_i8_pair_bias": [_P, c_int64, c_int64, _P, _P],
    "svgp_chol_f64": [_P, c_int64, c_int64, c_int64, c_int64, _P, _P, _P],
    "svgp_trinv_f64": [_P, _P, c_int64, c_int64, c_int64, c_int64, _P, _P],
    "svgp_ltl_f64": [_P, _P, c_int64, c_int64, c_int64, c_int64, _P],
    "svgp_gemm_f64": [c_int, c_int, c_int64, c_int64, c_int64, c_double, _P, c_int64, c_int64, _P, c_int64,
                      c_int64, c_double, _P, c_int64, c_int64, c_int64, _P],
    "svgp_rowstats_fwd": [_P, _P, _P, c_int64, c_int64, _P, _P, _P, _P],
    "svgp_predictive_fwd": [_P, _P, _P, _P, c_int64, c_int64, c_int, c_float, c_float, _P, _P, _P],
    "svgp_rowterms_bwd_pre": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, c_int64, c_int64, _P, _P, _P, _P, _P, _P],
    "svgp_rowterms_bwd_post": [_P, _P, _P, _P, _P, _P, _P, _P, c_int64, c_int64, _P, _P, _P, _P],
}
_RESTYPE = {"svgp_last_error": c_char_p, "svgp_syrk_ws_floats": c_int64, "svgp_i8_ldkr": c_int64, "svgp_i8_nblk": c_int64}

_lib = None


def load():
    """Load the shared library (once).  Raises SvgpLibraryError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SvgpLibraryError(
            "%s not found: build it with `python -m svgp_vae_b200.build` (nvcc, sm_100a). "
            "svgp_vae_b200 has no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, args in SIGNATURES.items():
        fn = getattr(lib, name)            # AttributeError here == header / library mismatch
        fn.argtypes = args
        fn.restype = _RESTYPE.get(name, c_int)
    _lib = lib
    return lib


def call(name, *args):
    """Call an int-returning entry point and raise on a non-zero status."""
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        msg = lib.svgp_last_error()
        raise SvgpLibraryError("%s failed (%d): %s" % (name, rc, msg.decode() if msg else ""))
    return rc
