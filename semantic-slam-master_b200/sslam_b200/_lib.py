"""ctypes binding of libsslam_b200.so (the C ABI declared in include/sslam_b200.h)."""

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SSLAM_B200_LIB") or os.path.join(_HERE, "libsslam_b200.so")   # (override: tools / experiments)

c_int, c_float, c_size_t, c_void_p = ctypes.c_int, ctypes.c_float, ctypes.c_size_t, ctypes.c_void_p

# name -> (restype, argtypes); must list every symbol of include/sslam_b200.h
SIGNATURES = {
    "sslam_abi_version": (c_int, []),
    "sslam_last_error": (c_int, [ctypes.c_char_p, c_size_t]),
    "sslam_device_check": (c_int, []),
    "sslam_launch_count": (ctypes.c_uint64, []),
    "sslam_profile_enable": (c_int, [c_int]),
    "sslam_profile_kinds": (c_int, []),
    "sslam_profile_kind_name": (ctypes.c_char_p, [c_int]),
    "sslam_profile_read": (c_int, [c_int, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_uint64)]),
    "sslam_decode_workspace_bytes": (c_size_t, [c_int] * 4),
    "sslam_decode_topk_f32": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_float,
                                      c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t,
                                      c_void_p]),
    "sslam_nms_f32": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "sslam_gather_bilinear_f32": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                          c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "sslam_l2norm_rows": (c_int, [c_void_p, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_void_p]),
    "sslam_refiner_packed_bytes": (c_size_t, [c_int] * 4),
    "sslam_refiner_pack_weights": (c_int, [ctypes.POINTER(c_void_p), c_int, c_int, c_int, c_int, c_void_p,
                                           c_size_t, c_void_p]),
    "sslam_refiner_workspace_bytes": (c_size_t, [c_int] * 5),
    "sslam_refiner_forward_f32": (c_int, [ctypes.POINTER(c_void_p), c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                          c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p, c_void_p,
                                          c_void_p, c_size_t, c_void_p]),
    "sslam_refiner_range_check": (c_int, [c_void_p]),
    "sslam_match_workspace_bytes": (c_size_t, [c_int] * 7),
    "sslam_match_top2": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p, c_int, c_int,
                                 c_int, c_int, c_int,
                                 c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                 c_size_t, c_void_p]),
    "sslam_match_finalize": (c_int, [c_int, ctypes.POINTER(ctypes.c_double), c_void_p, c_int, c_int, c_int,
                                     c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_void_p]),
    "sslam_nn_points": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int,
                                c_void_p, c_void_p, c_void_p]),
    "sslam_gt_matches": (c_int, [c_void_p, c_void_p, c_int, ctypes.c_double, c_int, c_int, c_void_p, c_void_p,
                                 c_void_p]),
    "sslam_eval_matches": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int,
                                   c_void_p, c_void_p, c_void_p]),
    "sslam_selector_packed_bytes": (c_size_t, [c_int, c_int]),
    "sslam_selector_pack_weights": (c_int, [c_void_p, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "sslam_selector_workspace_bytes": (c_size_t, [c_int] * 4),
    "sslam_selector_head_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                        c_int, c_int, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "sslam_heatmap_from_cells_f32": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "sslam_ransac_workspace_bytes": (c_size_t, [c_int] * 3),
    "sslam_ransac_homography": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int,
                                        c_void_p, c_void_p, c_void_p, c_int, c_int, ctypes.c_double, ctypes.c_uint64,
                                        c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t,
                                        c_void_p]),
    "sslam_ransac_fundamental_workspace_bytes": (c_size_t, [c_int] * 3),
    "sslam_ransac_fundamental": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int,
                                         c_void_p, c_void_p, c_void_p, c_int, c_int, ctypes.c_double,
                                         ctypes.c_uint64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                         c_void_p, c_size_t, c_void_p]),
}

# include/sslam_b200_debug.h (tools only)
DEBUG_SIGNATURES = {
    "sslam_debug_watchdog_gemm": (c_int, [c_void_p]),
    "sslam_debug_decode_stream": (None, [c_int]),
    "sslam_debug_refiner_fused": (None, [c_int]),
    "sslam_debug_decode_tune": (None, [c_int, c_int]),
}

ERROR_NAMES = {-1: "SSLAM_EINVAL", -2: "SSLAM_EUNSUPPORTED", -3: "SSLAM_EWORKSPACE",
               -4: "SSLAM_ECUDA", -5: "SSLAM_ENODEVICE", -6: "SSLAM_ERANGE"}

_lib = None
ABI_VERSION = 4


class SslamError(RuntimeError):
    def __init__(self, code, text):
        super().__init__(f"{ERROR_NAMES.get(code, code)}: {text}")
        self.code = code


def load():
    """Load the shared library (once).  Raises if it has not been built — there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; "
                "g.build()'` or `make -C semantic-slam-master_b200/csrc`. There is no CPU fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in list(SIGNATURES.items()) + list(DEBUG_SIGNATURES.items()):
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        if lib.sslam_abi_version() != ABI_VERSION:
            raise ImportError("libsslam_b200.so ABI version mismatch; rebuild")
        _lib = lib
    return _lib


def last_error():
    buf = ctypes.create_string_buffer(512)
    load().sslam_last_error(buf, 512)
    return buf.value.decode(errors="replace")


def check(code):
    if code != 0:
        raise SslamError(code, last_error())
