"""ctypes binding of libpioran_b200.so (include/pioran_b200.h).  Fails loudly when the library is missing:
there is no CPU fallback in this package."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# PIORAN_B200_LIB: another build of the same library (kernel-variant timing, tools/variants_gpu.py); never a fallback
LIB_PATH = os.environ.get("PIORAN_B200_LIB") or os.path.join(HERE, "libpioran_b200.so")

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)


class ApproxSpec(C.Structure):
    """struct pioran_approx_spec"""
    _fields_ = [("psd_model", C.c_int32), ("n_components", C.c_int32), ("basis", C.c_int32),
                ("is_integrated_power", C.c_int32), ("f_min", C.c_double), ("f_max", C.c_double),
                ("S_low", C.c_double), ("S_high", C.c_double)]


class PriorSpec(C.Structure):
    """struct pioran_prior_spec"""
    _fields_ = [("kind", C.c_int32), ("ref_col", C.c_int32), ("p0", C.c_double), ("p1", C.c_double)]


# every symbol include/pioran_b200.h declares: name → (restype, argtypes)
SYMBOLS = {
    "pioran_last_error": (C.c_char_p, []),
    "pioran_version": (C.c_int, []),
    "pioran_ctx_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "pioran_ctx_destroy": (C.c_int, [C.c_void_p]),
    "pioran_ctx_create_multi": (C.c_int, [_ip, C.c_int, C.POINTER(C.c_void_p)]),
    "pioran_ctx_device_count": (C.c_int, [C.c_void_p]),
    "pioran_ctx_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "pioran_ctx_synchronize": (C.c_int, [C.c_void_p]),
    "pioran_ctx_launch_count": (C.c_int64, [C.c_void_p]),
    "pioran_ctx_last_kernel_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_double)]),
    "pioran_ctx_last_kernel_name": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int]),
    "pioran_series_upload": (C.c_int, [C.c_void_p, C.c_int64, _dp, _dp, _dp, _ip]),
    "pioran_series_free": (C.c_int, [C.c_void_p, C.c_int]),
    "pioran_series_length": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int64)]),
    "pioran_approx_coeffs": (C.c_int, [C.c_void_p, C.POINTER(ApproxSpec), C.c_int, _dp, _dp, _dp, _dp, _dp]),
    "pioran_approx_coeffs_features": (C.c_int, [C.c_void_p, C.POINTER(ApproxSpec), C.c_int, C.c_int, _dp, _dp, _dp, _dp, _dp]),
    "pioran_approx_features_logl": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(ApproxSpec), C.c_int, C.c_int, _dp, _dp]),
    "pioran_celerite_logl": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, _dp, _dp, _dp, _dp, _dp, _dp, _dp, _dp, _dp]),
    "pioran_approx_logl": (C.c_int, [C.c_void_p, C.c_int, _ip, C.POINTER(ApproxSpec), C.c_int, _dp, C.c_int, _dp]),
    "pioran_approx_logl_logshift": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(ApproxSpec), C.c_int, _dp, _dp]),
    "pioran_approx_logl_dev": (C.c_int, [C.c_void_p, C.c_int, _ip, C.POINTER(ApproxSpec), C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "pioran_approx_logl_grad": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(ApproxSpec), C.c_int, _dp, _dp, _dp]),
    "pioran_approx_logl_logshift_grad": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(ApproxSpec), C.c_int, _dp, _dp, _dp]),
    "pioran_approx_logl_sine": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(ApproxSpec), C.c_int, _dp, _dp]),
    "pioran_approx_logl_sine_grad": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(ApproxSpec), C.c_int, _dp, _dp, _dp]),
    "pioran_approx_logl_grad_dev": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(ApproxSpec), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pioran_celerite_logl_jvp": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int] + [_dp] * 18),
    "pioran_approx_features_logl_grad": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(ApproxSpec), C.c_int, C.c_int, _dp, _dp, _dp]),
    "pioran_celerite_logl_vjp": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int] + [_dp] * 17),
    "pioran_approx_features_logl_grad_reverse": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(ApproxSpec), C.c_int, C.c_int, _dp, _dp, _dp]),
    "pioran_ctx_set_vjp_workspace": (C.c_int, [C.c_void_p, C.c_longlong]),
    "pioran_ctx_set_auto_scan": (C.c_int, [C.c_void_p, C.c_int]),
    "pioran_ctx_set_sweep_kernel": (C.c_int, [C.c_void_p, C.c_int]),
    "pioran_ctx_set_scan_chunks": (C.c_int, [C.c_void_p, C.c_int]),
    "pioran_ctx_set_scan_tolerance": (C.c_int, [C.c_void_p, C.c_double]),
    "pioran_celerite_scan_range_check": (C.c_int, [C.c_void_p, _dp]),
    "pioran_ctx_last_scan_check": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "pioran_ctx_set_scan_floor_cap": (C.c_int, [C.c_void_p, C.c_double]),
    "pioran_ctx_last_scan_history": (C.c_int, [C.c_void_p, C.c_int, C.c_int, _dp, _dp, C.POINTER(C.c_int)]),
    "pioran_prior_transform": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(PriorSpec), C.c_int, _dp, _dp]),
    "pioran_prior_transform_logl": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(ApproxSpec), C.c_int, C.POINTER(PriorSpec), C.c_int, _dp, _dp, _dp]),
    "pioran_celerite_logl_scan": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, _dp, _dp, _dp, _dp, _dp, _dp, _dp]),
    "pioran_scan_composite_doubles": (C.c_int, []),
    "pioran_celerite_scan_range_begin": (C.c_int, [C.c_void_p, C.c_int, C.c_int, _dp, _dp, _dp, _dp, _dp, _dp, C.c_int64, C.c_int64, C.c_int, _dp]),
    "pioran_celerite_scan_range_end": (C.c_int, [C.c_void_p, C.c_int, _dp, _dp]),
    "pioran_direct_logl": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, _dp, _dp, _dp, _dp, _dp, _dp, _dp, _ip]),
    "pioran_celerite_predict": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, _dp, _dp, _dp, _dp, _dp, _dp, C.c_int64, _dp, _dp]),
    "pioran_celerite_simulate": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, _dp, _dp, _dp, _dp, _dp, _dp, _dp]),
    "pioran_celerite_predict_var": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, _dp, _dp, _dp, _dp, _dp, _dp, C.c_int64,
                                              _dp, _dp, _dp]),
    "pioran_celerite_posterior_draws": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, _dp, _dp, _dp, _dp, _dp, _dp, _dp,
                                                  C.c_int64, _dp, C.c_double, C.c_int, _dp, _dp]),
    "pioran_celerite_predict_cov": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, _dp, _dp, _dp, _dp, _dp, _dp, C.c_int64,
                                              _dp, _dp, _dp]),
    "pioran_ctx_set_postcov_workspace": (C.c_int, [C.c_void_p, C.c_longlong]),
    "pioran_lombscargle": (C.c_int, [C.c_void_p, C.c_int, C.c_int, _dp, C.c_int, C.c_int64, _dp, _dp]),
    "pioran_ctx_set_lsp_workspace": (C.c_int, [C.c_void_p, C.c_longlong]),
}

_lib = None


class PioranError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libpioran_b200 error {code}: {msg}")
        self.code = code


def load():
    """Loads the shared library (never builds it, never falls back)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). The pioran B200 backend has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the ABI is incomplete
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise PioranError(rc, load().pioran_last_error().decode("utf-8", "replace"))
