"""ctypes binding of libbioen_b200.so -- every symbol declared in include/bioen_b200.h.

This is the only place the shared library is loaded.  There is no fallback: if the library is missing or no
sm_100 GPU is usable, calls raise (RuntimeError with the library's own error text).
"""
import ctypes as C
import os

import numpy as np

from . import build as _build

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)


class params_t(C.Structure):  # include/bioen_b200.h, reference c_bioen_common.h:44-60
    _fields_ = [
        ("forces", _dp), ("w0", _dp), ("g", _dp), ("G", _dp), ("yTilde", _dp), ("YTilde", _dp), ("w", _dp),
        ("result", _dp), ("theta", C.c_double), ("yTildeT", _dp), ("caching", C.c_int), ("tmp_n", _dp),
        ("tmp_m", _dp), ("m", C.c_int), ("n", C.c_int),
    ]


class gsl_config_params(C.Structure):  # c_bioen_common.h:62-67
    _fields_ = [("step_size", C.c_double), ("tol", C.c_double), ("max_iterations", C.c_int),
                ("algorithm", C.c_int)]


class lbfgs_config_params(C.Structure):  # c_bioen_common.h:69-79
    _fields_ = [
        ("linesearch", C.c_int), ("max_iterations", C.c_int), ("delta", C.c_double), ("epsilon", C.c_double),
        ("ftol", C.c_double), ("gtol", C.c_double), ("wolfe", C.c_double), ("past", C.c_int),
        ("max_linesearch", C.c_int),
    ]


class visual_params(C.Structure):  # c_bioen_common.h:89-92
    _fields_ = [("debug", C.c_size_t), ("verbose", C.c_size_t)]


class bioen_b200_batch(C.Structure):  # include/bioen_b200.h: per-problem inputs of a batch (NULL = shared vector)
    _fields_ = [("K", C.c_int), ("thetas", _dp), ("YTilde", _dp), ("row_weights", _dp), ("w0", _dp)]


# name -> (restype, argtypes); mirrors include/bioen_b200.h one to one (tests/test_abi.py checks the set)
_vp = C.c_void_p
SIGNATURES = {
    # part 1
    "_get_weights": (C.c_double, [_dp, _dp, C.c_size_t]),
    "_bioen_log_posterior_logw": (C.c_double, [_dp, _dp, _dp, _dp, _dp, _dp, C.c_double, C.c_int, _dp, _dp, _dp,
                                               C.c_int, C.c_int, C.c_double]),
    "_grad_bioen_log_posterior_logw": (None, [_dp, _dp, _dp, _dp, _dp, _dp, C.c_double, C.c_int, _dp, _dp, _dp,
                                              C.c_int, C.c_int, C.c_double]),
    "_opt_bfgs_logw": (C.c_double, [params_t, gsl_config_params, visual_params, _ip]),
    "_opt_lbfgs_logw": (C.c_double, [params_t, lbfgs_config_params, visual_params, _ip]),
    "_get_weights_from_forces": (None, [_dp, _dp, _dp, _dp, C.c_int, _dp, _dp, C.c_size_t, C.c_size_t]),
    "_bioen_log_posterior_forces": (C.c_double, [_dp, _dp, _dp, _dp, _dp, C.c_double, C.c_int, _dp, _dp, _dp,
                                                 C.c_int, C.c_int]),
    "_grad_bioen_log_posterior_forces": (None, [_dp, _dp, _dp, _dp, _dp, C.c_double, C.c_int, _dp, _dp, _dp,
                                                C.c_int, C.c_int]),
    "_opt_bfgs_forces": (C.c_double, [params_t, gsl_config_params, visual_params, _ip]),
    "_opt_lbfgs_forces": (C.c_double, [params_t, lbfgs_config_params, visual_params, _ip]),
    "_library_gsl": (C.c_int, []),
    "_library_lbfgs": (C.c_int, []),
    "_omp_set_num_threads": (None, [C.c_int]),
    "_set_fast_openmp_flag": (None, [C.c_int]),
    "_get_fast_openmp_flag": (C.c_int, []),
    "bioen_gsl_error": (C.c_char_p, [C.c_int]),
    "lbfgs_strerror": (C.c_char_p, [C.c_int]),
    # part 2
    "bioen_b200_last_error": (C.c_char_p, []),
    "bioen_b200_error_pending": (C.c_int, []),
    "bioen_b200_device_count": (C.c_int, []),
    "bioen_b200_create": (_vp, [C.c_int, C.c_int, C.c_int]),
    "bioen_b200_destroy": (None, [_vp]),
    "bioen_b200_upload_ytilde": (C.c_int, [_vp, _dp, C.c_size_t]),
    "bioen_b200_adopt_ytilde": (C.c_int, [_vp, _vp, C.c_size_t]),
    "bioen_b200_upload_rows": (C.c_int, [_vp, C.c_int, C.c_int, _dp, C.c_size_t]),
    "bioen_b200_host_alloc": (_vp, [C.c_size_t]),
    "bioen_b200_host_free": (None, [_vp]),
    "bioen_b200_alloc_ytilde": (C.c_int, [_vp]),
    "bioen_b200_download_ytilde": (C.c_int, [_vp, C.c_int, C.c_int, C.c_longlong, C.c_longlong, _dp]),
    "bioen_b200_set_logw": (C.c_int, [_vp, _dp, _dp, C.c_double]),
    "bioen_b200_set_forces": (C.c_int, [_vp, _dp, _dp, C.c_double]),
    "bioen_b200_set_theta": (C.c_int, [_vp, C.c_double]),
    "bioen_b200_set_option": (C.c_int, [_vp, C.c_int, C.c_int]),
    "bioen_b200_eval": (C.c_int, [_vp, C.c_int, _dp, _dp, _dp]),
    "bioen_b200_grad_continue": (C.c_int, [_vp, C.c_int, _dp]),
    "bioen_b200_weights": (C.c_int, [_vp, C.c_int, _dp, _dp, _dp]),
    "bioen_b200_average": (C.c_int, [_vp, _dp, _dp]),
    "bioen_b200_affine_rows": (C.c_int, [_vp, _dp, _dp]),
    "bioen_b200_forces_from_weights": (C.c_int, [_vp, _dp, _dp, _dp]),
    "bioen_b200_opt_lbfgs": (C.c_int, [_vp, C.c_int, _dp, _dp, lbfgs_config_params, visual_params, _dp, _ip]),
    "bioen_b200_opt_gsl": (C.c_int, [_vp, C.c_int, _dp, _dp, gsl_config_params, visual_params, _dp, _ip]),
    "bioen_b200_theta_scan": (C.c_int, [_vp, C.c_int, C.c_int, _dp, _dp, _dp, lbfgs_config_params, visual_params, _dp,
                                        _ip, _ip, _dp]),
    "bioen_b200_time_scan_evals": (C.c_int, [_vp, C.c_int, C.c_int, _dp, _dp, C.c_int, C.c_int, C.POINTER(C.c_float),
                                             C.POINTER(C.c_float), C.POINTER(C.c_longlong)]),
    "bioen_b200_batch_minimize": (C.c_int, [_vp, C.c_int, C.POINTER(bioen_b200_batch), _dp, _dp, lbfgs_config_params,
                                            visual_params, _dp, _ip, _ip, _dp, _dp, _dp, _dp]),
    "bioen_b200_batch_eval": (C.c_int, [_vp, C.c_int, C.POINTER(bioen_b200_batch), _dp, _dp, _dp, _dp, _dp, _dp]),
    "bioen_b200_time_batch_evals": (C.c_int, [_vp, C.c_int, C.POINTER(bioen_b200_batch), _dp, C.c_int, C.c_int,
                                              C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_longlong)]),
    "bioen_b200_dmma_peak": (C.c_int, [C.c_int, _dp]),
    "bioen_b200_read_stream_peak": (C.c_int, [_vp, C.c_int, _dp]),
    "bioen_b200_selftest_linesearch": (C.c_int, [lbfgs_config_params, C.c_double, C.c_double, C.c_double,
                                                 C.CFUNCTYPE(None, C.c_double, _dp, _dp), _dp, _dp, _ip]),
    "bioen_b200_selftest_interpolate": (C.c_double, [C.c_double] * 8 + [C.c_int]),
    "bioen_b200_selftest_tilewalk": (C.c_longlong, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_longlong, C.c_int, C.c_int,
                                                   C.c_longlong, _ip, _ip, C.POINTER(C.c_longlong), _ip]),
    "bioen_b200_selftest_num_slots": (C.c_int, [C.c_longlong, C.c_longlong, C.c_longlong]),
    "bioen_b200_selftest_slice_plan": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_longlong, C.POINTER(C.c_longlong)]),
    "bioen_b200_selftest_twoloop_schedule": (C.c_int, [C.c_int, C.c_int, C.c_int, _ip]),
    "bioen_b200_selftest_lbfgs_update": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, _ip, _ip, _dp, _dp, _dp, _dp, _dp,
                                                   _dp, _dp, _dp, _dp]),
    "bioen_b200_nccl_unique_id": (C.c_int, [C.c_char_p]),
    "bioen_b200_comm_init": (C.c_int, [_vp, C.c_char_p, C.c_int, C.c_int, C.c_longlong]),
    "bioen_b200_comm_init_local": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.c_longlong]),
    "bioen_b200_comm_mode": (C.c_int, [_vp]),
    "bioen_b200_set_logw_dev": (C.c_int, [_vp, _vp, _dp, C.c_double]),
    "bioen_b200_set_forces_dev": (C.c_int, [_vp, _vp, _dp, C.c_double]),
    "bioen_b200_eval_dev": (C.c_int, [_vp, C.c_int, _vp, _vp]),
    "bioen_b200_fetch": (C.c_int, [_vp, _dp, _dp]),
    "bioen_b200_opt_lbfgs_dev": (C.c_int, [_vp, C.c_int, _vp, lbfgs_config_params, visual_params, _dp, _ip]),
    "bioen_b200_time_evals": (C.c_int, [_vp, C.c_int, _vp, _vp, C.c_int, C.c_int, C.POINTER(C.c_float),
                                        C.POINTER(C.c_float), C.POINTER(C.c_longlong)]),
    "bioen_b200_generate_ytilde": (C.c_int, [_vp, C.c_ulonglong, C.c_longlong, _dp, C.c_double]),
    "bioen_b200_kernels_launched": (C.c_longlong, [_vp]),
    "bioen_b200_query": (C.c_longlong, [_vp, C.c_int]),
    "bioen_b200_debug_read": (C.c_int, [_vp, C.c_int, _dp, C.c_size_t]),
    "bioen_b200_stream": (_vp, [_vp]),
}

_lib = None


def library_path():
    # BIOEN_B200_LIB: load another build of the library (kernel experiments); default = the in-tree build
    return os.environ.get("BIOEN_B200_LIB") or _build.LIB


def load(build_if_missing=True):
    """Load (building first if the .so is absent and nvcc is available) and type the library."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        if not build_if_missing:
            raise ImportError("bioen_b200: %s is missing -- run `python -m bioen_b200.build`" % path)
        _build.build_library()
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = header / library out of sync: fail loudly
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error():
    return load().bioen_b200_last_error().decode("utf-8", "replace")


def check(status, what="bioen_b200"):
    """Raise for a non-zero status of a part-2 call (and consume the thread's pending-error flag, which is meant
    for the part-1 entry points that have no status of their own)."""
    if status:
        msg = last_error()
        load().bioen_b200_error_pending()
        raise RuntimeError("%s failed: %s" % (what, msg))


def clear_pending():
    """Forget an error that was already reported through a status code (call before a part-1 entry point)."""
    load().bioen_b200_error_pending()


def check_pending(what):
    """Raise if a part-1 call (no status in its signature) failed since the last clear_pending()."""
    if load().bioen_b200_error_pending():
        raise RuntimeError("%s failed: %s" % (what, last_error()))


def vec(a):
    """C-contiguous float64 1-D view/copy of a vector-like (accepts (n,), (n,1), (1,n), np.matrix)."""
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64).ravel())


def mat(a):
    """C-contiguous float64 2-D array (np.matrix accepted)."""
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64))


def ptr(a):
    return a.ctypes.data_as(_dp)
