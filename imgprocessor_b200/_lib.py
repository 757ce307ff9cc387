"""ctypes binding of libimgcorr.so (include/imgcorr.h).  There is no CPU fallback: if the library
is missing it is built with nvcc, and if that is impossible importing this module's `lib()` raises."""
import ctypes
import os

from . import build as _build

_LIB = None

U8, U16, F32, F64 = 0, 1, 2, 3
COND_GT, COND_LT = 0, 1
DO_DARK, DO_FLAT, DO_NAN_TO_NUM, DO_PERSPECTIVE = 1, 2, 4, 8
OPT_K1_VARIANT, OPT_K2_VARIANT, OPT_HOST_SLOTS, OPT_K1_SEG_ROWS, OPT_PROFILE, OPT_CHAIN_GROUP = 1, 2, 3, 4, 5, 6
OPT_RAW_BIG_ENDIAN, OPT_RAW_FRAME_GAP, OPT_K3_VARIANT, OPT_CHAIN_OVERLAP, OPT_K2_COORD_CACHE = 7, 8, 9, 10, 11
INTER_CUBIC, INTER_LANCZOS4 = 2, 4
OK, ERR_INVALID, ERR_CUDA, ERR_STATE, ERR_NOMEM = 0, -1, -2, -3, -4

c_void_p, c_int, c_double, c_size_t = ctypes.c_void_p, ctypes.c_int, ctypes.c_double, ctypes.c_size_t

# name -> (restype, argtypes): every symbol include/imgcorr.h declares
SIGNATURES = {
    'imgcorr_last_error': (ctypes.c_char_p, []),
    'imgcorr_version': (c_int, []),
    'imgcorr_device_count': (c_int, []),
    'imgcorr_ctx_create': (c_int, [c_int, c_int, c_int, ctypes.POINTER(c_void_p)]),
    'imgcorr_ctx_destroy': (c_int, [c_void_p]),
    'imgcorr_set_option': (c_int, [c_void_p, c_int, c_int]),
    'imgcorr_launch_count': (ctypes.c_longlong, [c_void_p]),
    'imgcorr_profile_read': (c_int, [c_void_p, ctypes.POINTER(c_double)]),
    'imgcorr_set_dark': (c_int, [c_void_p, c_void_p, c_void_p, c_double, c_int, c_int]),
    'imgcorr_set_dark_exposures': (c_int, [c_void_p, c_void_p, c_int]),
    'imgcorr_set_flat': (c_int, [c_void_p, c_void_p, c_int]),
    'imgcorr_set_lens': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    'imgcorr_set_lens_model': (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    'imgcorr_pointwise_median': (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_double,
                                         c_int, c_int, c_int, c_void_p]),
    'imgcorr_undistort': (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_double, c_int, c_int, c_int,
                                  c_int, c_void_p]),
    'imgcorr_remap': (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_void_p, c_void_p, c_double,
                              c_void_p]),
    'imgcorr_undistort_maps': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    'imgcorr_correct_batch': (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_double, c_int, c_int, c_int,
                                      c_double, c_int, c_int, c_int, c_int, c_void_p]),
    'imgcorr_correct_host': (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_double, c_int, c_int, c_int,
                                     c_double, c_int, c_int, c_int, c_int]),
    'imgcorr_correct_batch_bg': (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_double, c_int,
                                         c_int, c_int, c_double, c_int, c_int, c_int, c_int, c_void_p]),
    'imgcorr_correct_host_bg': (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_double, c_int,
                                        c_int, c_int, c_double, c_int, c_int, c_int, c_int]),
    'imgcorr_set_output_scale': (c_int, [c_void_p, c_double, c_double]),
    'imgcorr_set_perspective': (c_int, [c_void_p, c_void_p, c_int, c_int, c_double, c_void_p, c_int, c_int, c_int]),
    'imgcorr_set_perspective_frames': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_double]),
    'imgcorr_warp_perspective': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_int, c_int, c_void_p,
                                         c_int, c_int, c_double, c_void_p]),
    'imgcorr_divide_f64': (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_size_t, c_int, c_void_p]),
    'imgcorr_ste_average': (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_double, c_void_p]),
    'imgcorr_ste_average_thr': (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    'imgcorr_stack_mean': (c_int, [c_void_p, c_void_p, c_int, c_int, c_size_t, c_void_p, c_double, c_int, c_int, c_void_p, c_void_p]),
    'imgcorr_scale_f64': (c_int, [c_void_p, c_void_p, c_size_t, c_double, c_void_p]),
    'imgcorr_subsample_f64': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    'imgcorr_linear_fit': (c_int, [c_void_p, c_void_p, c_int, c_int, c_size_t, c_void_p, c_double, c_double, c_void_p, c_void_p, c_void_p,
                                   c_void_p]),
    'imgcorr_selftest_division': (c_int, [c_void_p, c_int, ctypes.c_ulonglong, ctypes.POINTER(c_double)]),
    'imgcorr_host_fingerprint': (c_int, [c_void_p, c_size_t, ctypes.POINTER(ctypes.c_ulonglong)]),
    'imgcorr_host_alloc': (c_int, [c_size_t, ctypes.POINTER(c_void_p)]),
    'imgcorr_host_free': (c_int, [c_void_p]),
}


class ImgcorrError(RuntimeError):
    def __init__(self, status, message):
        RuntimeError.__init__(self, 'libimgcorr status %d: %s' % (status, message))
        self.status = status


def lib_path():
    return os.environ.get('IMGCORR_LIB') or _build.LIB      # IMGCORR_LIB: development override (kernel variants)


def lib():
    """Load (building first if needed) libimgcorr.so.  Raises if it cannot be had."""
    global _LIB
    if _LIB is None:
        path = lib_path()
        if not os.path.exists(path):
            _build.build()
        handle = ctypes.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)          # AttributeError if the .so lacks a declared symbol
            fn.restype = res
            fn.argtypes = args
        _LIB = handle
    return _LIB


def check(status):
    if status != OK:
        raise ImgcorrError(status, lib().imgcorr_last_error().decode('utf-8', 'replace'))
    return status
