"""ctypes binding of the C ABI declared in include/sstem_b200.h.

This is the only way the package computes anything: if the shared library is
missing (or was not built for this GPU) every call raises -- there is no CPU,
PyTorch-eager or oracle fallback.
"""
from __future__ import annotations

import ctypes
import os
import threading

from ._build import LIB_PATH as _DEFAULT_LIB_PATH, needs_build as _needs_build

#: must equal SSTEM_ABI_VERSION of include/sstem_b200.h (checked against the loaded library in load())
ABI_VERSION = 7

#: SSTEM_LIB_PATH selects another build of the same library (kernel-tuning experiments)
LIB_PATH = os.environ.get("SSTEM_LIB_PATH") or _DEFAULT_LIB_PATH

_c_i64 = ctypes.c_int64
_c_i32 = ctypes.c_int32
_c_u32 = ctypes.c_uint32
_c_p = ctypes.c_void_p

SEPCONV_DEFAULT = 0
SEPCONV_STRICT_ORDER = 1
SEPCONV_GRAY_REPLICATED = 2
SEPCONV_ACCUMULATE = 4
TAPCONV_UPSAMPLE2X = 1
TAPCONV_TILED = 2
BRANCH_RELU = 1
BRANCH_IN_CHUNKED = 2
BRANCH_OUT_CHUNKED = 4
LAYOUT_NCHW = 0
LAYOUT_NHWC = 1
PIX_U8 = 0
PIX_F32 = 1
WARP_BILINEAR = 0
WARP_NEAREST = 1

#: every symbol include/sstem_b200.h declares (tests check the library exports all of them)
EXPORTED_SYMBOLS = (
    "sstem_sepconv_forward", "sstem_sepconv_backward", "sstem_interp_tail_forward", "sstem_interp_tail_backward",
    "sstem_warp_forward", "sstem_warp_backward", "sstem_image_warp", "sstem_sff_degrade", "sstem_sff_contrast",
    "sstem_sections_to_input", "sstem_prediction_to_u8", "sstem_warp_stitch_u8", "sstem_warp_stitch_forward",
    "sstem_taps_tiled_elems", "sstem_taps_to_tiled", "sstem_sepconv_forward_tiled", "sstem_frame_mean_pad",
    "sstem_sepconv_backward_tiled", "sstem_taps_from_tiled",
    "sstem_sepconv_forward_detect", "sstem_sepconv_backward_detect",
    "sstem_tap_conv3x3_packed_elems", "sstem_tap_conv3x3_pack_weights", "sstem_tap_conv3x3",
    "sstem_tap_conv3x3_pack_weights_adjoint", "sstem_tap_conv3x3_backward",
    "sstem_branch_conv3x3_packed_elems", "sstem_branch_conv3x3_pack_weights", "sstem_chunked_elems", "sstem_branch_conv3x3",
    "sstem_branch_conv3x3_pack_weights_adjoint", "sstem_branch_conv3x3_backward",
    "sstem_fp32_peak_probe", "sstem_launch_count", "sstem_abi_version", "sstem_error_string",
)

_lock = threading.Lock()
_lib = None


class SstemError(RuntimeError):
    pass


def load() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise SstemError(
                f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  sstem_restoration_b200 has no CPU fallback."
            )
        lib = ctypes.CDLL(LIB_PATH)
        lib.sstem_sepconv_forward.argtypes = [_c_p, _c_p, _c_p, _c_p, _c_i64, _c_i64, _c_i64, _c_i64, _c_i32, _c_u32, _c_p]
        lib.sstem_sepconv_forward.restype = ctypes.c_int
        lib.sstem_sepconv_backward.argtypes = [_c_p] * 7 + [_c_i64] * 4 + [_c_i32, _c_u32, _c_p]
        lib.sstem_sepconv_backward.restype = ctypes.c_int
        lib.sstem_interp_tail_forward.argtypes = [_c_p, _c_p, _c_i64] + [_c_p] * 5 + [_c_i64] * 4 + [_c_i32, _c_u32, _c_p]
        lib.sstem_interp_tail_forward.restype = ctypes.c_int
        lib.sstem_interp_tail_backward.argtypes = [_c_p, _c_p, _c_p, _c_i64] + [_c_p] * 8 + [_c_i64] * 4 + [_c_i32, _c_u32, _c_p]
        lib.sstem_interp_tail_backward.restype = ctypes.c_int
        lib.sstem_warp_forward.argtypes = [_c_p, _c_p, ctypes.POINTER(_c_i64), _c_p, _c_i64, _c_i64, _c_i64, _c_i64, _c_i32, _c_p]
        lib.sstem_warp_forward.restype = ctypes.c_int
        lib.sstem_warp_backward.argtypes = [_c_p, _c_p, ctypes.POINTER(_c_i64), _c_p, _c_p, _c_p, _c_i64, _c_i64, _c_i64, _c_i64, _c_p]
        lib.sstem_warp_backward.restype = ctypes.c_int
        lib.sstem_image_warp.argtypes = [_c_p, _c_i32, _c_p, _c_p, _c_p, _c_i64, _c_i64, _c_i64, _c_i64, _c_i32, _c_p]
        lib.sstem_image_warp.restype = ctypes.c_int
        lib.sstem_sff_degrade.argtypes = [_c_p] * 7 + [_c_i64] * 4 + [_c_p]
        lib.sstem_sff_degrade.restype = ctypes.c_int
        lib.sstem_sff_contrast.argtypes = [_c_p] * 3 + [_c_i64] * 5 + [_c_p]
        lib.sstem_sff_contrast.restype = ctypes.c_int
        lib.sstem_sections_to_input.argtypes = [_c_p] * 3 + [_c_i64] * 3 + [_c_i32, _c_p]
        lib.sstem_sections_to_input.restype = ctypes.c_int
        lib.sstem_prediction_to_u8.argtypes = [_c_p] * 2 + [_c_i64] * 3 + [_c_i32, _c_p]
        lib.sstem_prediction_to_u8.restype = ctypes.c_int
        lib.sstem_warp_stitch_u8.argtypes = [_c_p] * 4 + [_c_i64] * 4 + [_c_p]
        lib.sstem_warp_stitch_u8.restype = ctypes.c_int
        lib.sstem_warp_stitch_forward.argtypes = [_c_p, _c_p, ctypes.POINTER(_c_i64), _c_p, _c_p, _c_p, _c_i64, _c_i64, _c_i64, _c_i64, _c_p]
        lib.sstem_warp_stitch_forward.restype = ctypes.c_int
        lib.sstem_taps_tiled_elems.argtypes = [_c_i64] * 3
        lib.sstem_taps_tiled_elems.restype = _c_i64
        lib.sstem_taps_to_tiled.argtypes = [_c_p, _c_p, _c_i64, _c_i64, _c_i64, _c_p]
        lib.sstem_taps_to_tiled.restype = ctypes.c_int
        lib.sstem_sepconv_forward_tiled.argtypes = [_c_p, _c_p, _c_p, _c_p, _c_i64, _c_i64, _c_i64, _c_i64, _c_i32, _c_u32, _c_p]
        lib.sstem_sepconv_forward_tiled.restype = ctypes.c_int
        lib.sstem_sepconv_backward_tiled.argtypes = [_c_p] * 7 + [_c_i64] * 4 + [_c_i32, _c_u32, _c_p]
        lib.sstem_sepconv_backward_tiled.restype = ctypes.c_int
        lib.sstem_taps_from_tiled.argtypes = [_c_p, _c_p, _c_i64, _c_i64, _c_i64, _c_p]
        lib.sstem_taps_from_tiled.restype = ctypes.c_int
        lib.sstem_frame_mean_pad.argtypes = [_c_p, _c_i64, _c_p, _c_i64, _c_i64, _c_i64, _c_i64, _c_i32, _c_u32, _c_p]
        lib.sstem_frame_mean_pad.restype = ctypes.c_int
        lib.sstem_sepconv_forward_detect.argtypes = [_c_p, _c_p, _c_p, _c_p, _c_i64, _c_i64, _c_i64, _c_i64, _c_i32, _c_u32, _c_p, _c_p]
        lib.sstem_sepconv_forward_detect.restype = ctypes.c_int
        lib.sstem_sepconv_backward_detect.argtypes = [_c_p] * 7 + [_c_i64] * 4 + [_c_i32, _c_u32, _c_p, _c_p]
        lib.sstem_sepconv_backward_detect.restype = ctypes.c_int
        lib.sstem_tap_conv3x3_packed_elems.argtypes = []
        lib.sstem_tap_conv3x3_packed_elems.restype = _c_i64
        lib.sstem_tap_conv3x3_pack_weights.argtypes = [_c_p, _c_p, _c_i32, _c_i32, _c_p]
        lib.sstem_tap_conv3x3_pack_weights.restype = ctypes.c_int
        lib.sstem_tap_conv3x3.argtypes = [_c_p, _c_p, _c_p, _c_p, _c_i64, _c_i32, _c_i32, _c_i64, _c_i64, _c_u32, _c_p]
        lib.sstem_tap_conv3x3.restype = ctypes.c_int
        lib.sstem_tap_conv3x3_pack_weights_adjoint.argtypes = [_c_p, _c_p, _c_i32, _c_i32, _c_p]
        lib.sstem_tap_conv3x3_pack_weights_adjoint.restype = ctypes.c_int
        lib.sstem_tap_conv3x3_backward.argtypes = [_c_p] * 6 + [_c_i64, _c_i32, _c_i32, _c_i64, _c_i64, _c_u32, _c_p]
        lib.sstem_tap_conv3x3_backward.restype = ctypes.c_int
        lib.sstem_branch_conv3x3_packed_elems.argtypes = []
        lib.sstem_branch_conv3x3_packed_elems.restype = _c_i64
        lib.sstem_branch_conv3x3_pack_weights.argtypes = [_c_p, _c_p, _c_i32, _c_i32, _c_p]
        lib.sstem_branch_conv3x3_pack_weights.restype = ctypes.c_int
        lib.sstem_chunked_elems.argtypes = [_c_i64] * 4
        lib.sstem_chunked_elems.restype = _c_i64
        lib.sstem_branch_conv3x3.argtypes = [_c_p, _c_p, _c_p, _c_p, _c_i64, _c_i32, _c_i32, _c_i64, _c_i64, _c_u32, _c_p]
        lib.sstem_branch_conv3x3.restype = ctypes.c_int
        lib.sstem_branch_conv3x3_pack_weights_adjoint.argtypes = [_c_p, _c_p, _c_i32, _c_i32, _c_p]
        lib.sstem_branch_conv3x3_pack_weights_adjoint.restype = ctypes.c_int
        lib.sstem_branch_conv3x3_backward.argtypes = [_c_p] * 7 + [_c_i64, _c_i32, _c_i32, _c_i64, _c_i64, _c_u32, _c_p]
        lib.sstem_branch_conv3x3_backward.restype = ctypes.c_int
        lib.sstem_fp32_peak_probe.argtypes = [ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]
        lib.sstem_fp32_peak_probe.restype = ctypes.c_int
        lib.sstem_launch_count.argtypes = []
        lib.sstem_launch_count.restype = _c_i64
        lib.sstem_abi_version.argtypes = []
        lib.sstem_abi_version.restype = ctypes.c_int
        lib.sstem_error_string.argtypes = [ctypes.c_int]
        lib.sstem_error_string.restype = ctypes.c_char_p
        got = int(lib.sstem_abi_version())
        if got != ABI_VERSION:
            raise SstemError(f"{LIB_PATH} exports ABI version {got}, this package binds version {ABI_VERSION}: "
                             "stale library -- rebuild with `python -c 'import __graft_entry__ as g; g.build()'`")
        if LIB_PATH == _DEFAULT_LIB_PATH and _needs_build(LIB_PATH):
            import warnings
            warnings.warn(f"{LIB_PATH} is older than its sources (csrc/ or include/sstem_b200.h): rebuild it", RuntimeWarning)
        _lib = lib
    return _lib


def check(code: int, what: str) -> None:
    if code != 0:
        msg = load().sstem_error_string(code).decode()
        raise SstemError(f"{what} failed with code {code}: {msg}")


def launch_count() -> int:
    return int(load().sstem_launch_count())


def fp32_peak_probe():
    """(TFLOP/s, SM MHz) of a register-resident FFMA loop on the current device."""
    t = ctypes.c_double(0.0)
    m = ctypes.c_double(0.0)
    check(load().sstem_fp32_peak_probe(ctypes.byref(t), ctypes.byref(m)), "sstem_fp32_peak_probe")
    return t.value, m.value
