"""ctypes binding of include/dvc_b200.h.  There is no CPU fallback: if libdvc_b200.so is missing or a
call fails, this raises."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# tools/ that A/B kernel variants set DVC_LIB_FLAVOUR=measure to load the -DDVC_MEASURE build (build.py --measure);
# that file does not exist unless such a tool built it
LIB_PATH = os.path.join(HERE, "libdvc_b200_measure.so" if os.environ.get("DVC_LIB_FLAVOUR") == "measure" else "libdvc_b200.so")

DVC_MODE_FD, DVC_MODE_WINDOW, DVC_MODE_FLOW = 0, 1, 2
DVC_MORPH_ERODE, DVC_MORPH_DILATE, DVC_MORPH_OPEN, DVC_MORPH_CLOSE = 0, 1, 2, 3
DVC_SHAPE_RECT, DVC_SHAPE_ELLIPSE = 0, 1
DVC_DEGRADE_FD, DVC_DEGRADE_MCO = 0, 1
PROF_KERNELS = ("front", "diff", "vote", "ema", "morph", "ccl", "degrade", "misc")
DVC_ERR_INVALID, DVC_ERR_UNSUPPORTED, DVC_ERR_CUDA, DVC_ERR_NOMEM = -1, -2, -3, -4


class DvcConfig(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("mode", C.c_int32), ("block_size", C.c_int32),
                ("motion_threshold", C.c_float), ("min_area", C.c_double), ("kernel_size", C.c_int32),
                ("release_factor", C.c_double), ("quantization_level", C.c_float), ("window_size", C.c_int32),
                ("alpha_fraction", C.c_double), ("morph_kernel", C.c_int32), ("morph_shape", C.c_int32),
                ("max_batch", C.c_int32), ("device", C.c_int32), ("src_width", C.c_int32), ("src_height", C.c_int32), ("n_streams", C.c_int32)]


class DvcCounters(C.Structure):
    _fields_ = [("frames", C.c_uint64), ("pixels", C.c_uint64), ("motion_pixels", C.c_uint64),
                ("blocks", C.c_uint64), ("static_blocks", C.c_uint64)]


class DvcError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"dvc_b200 error {code}: {message}")
        self.code = code


class DvcUnsupported(DvcError, NotImplementedError):
    """The reference accepts this configuration; the GPU path does not implement it (no CPU fallback)."""


# every symbol include/dvc_b200.h declares: (name, restype, argtypes)
_P, _I, _F, _D, _L = C.c_void_p, C.c_int32, C.c_float, C.c_double, C.c_int64
SYMBOLS = {
    "dvc_abi_version": (C.c_int, []),
    "dvc_measure_build": (C.c_int, []),
    "dvc_last_error": (C.c_char_p, [_P]),
    "dvc_default_config": (None, [C.POINTER(DvcConfig)]),
    "dvc_create": (C.c_int, [C.POINTER(DvcConfig), C.POINTER(_P)]),
    "dvc_destroy": (C.c_int, [_P]),
    "dvc_begin_stream": (C.c_int, [_P, _P]),
    "dvc_begin_stream_frames": (C.c_int, [_P, _P]),
    "dvc_state_bytes": (C.c_size_t, [_P]),
    "dvc_get_state": (C.c_int, [_P, _P, C.c_size_t]),
    "dvc_set_state": (C.c_int, [_P, _P, C.c_size_t]),
    "dvc_get_counters": (C.c_int, [_P, C.POINTER(DvcCounters)]),
    "dvc_reset_counters": (C.c_int, [_P]),
    "dvc_set_flow_params": (C.c_int, [_P, _F, _D, _I, _I, _I, _I, _D, _I]),
    "dvc_process_batch": (C.c_int, [_P, _P, _I, _P, _P, _P, _P]),
    "dvc_set_overlap": (C.c_int, [_P, _I]),
    "dvc_flush": (C.c_int, [_P, _P]),
    "dvc_process_host": (C.c_int, [_P, _P, _L, _P, _P, _P]),
    "dvc_profile_enable": (C.c_int, [_P, _I]),
    "dvc_profile_read": (C.c_int, [_P, C.POINTER(C.c_double), C.POINTER(C.c_int64), _I]),
    "dvc_launch_count": (C.c_int64, [_P]),
    "dvc_bgr2gray_u8": (C.c_int, [_P, _P, _I, _I, _I, _P]),
    "dvc_gray_absdiff_thresh_u8": (C.c_int, [_P, _P, _P, _P, _I, _I, _I, _F, _I, _P]),
    "dvc_temporal_ring_u8": (C.c_int, [_P, _P, _I, _I, _I, _I, _D, _P]),
    "dvc_temporal_ema_u8": (C.c_int, [_P, _P, _P, _I, _I, _I, _D, _P]),
    "dvc_morph_u8": (C.c_int, [_P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "dvc_contour_filter_u8": (C.c_int, [_P, _P, _I, _I, _I, _D, _P]),
    "dvc_mask_rectangles_u8": (C.c_int, [_P, _P, _I, _I, _I, _P]),
    "dvc_resize_linear_u8": (C.c_int, [_P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "dvc_degrade_blend_u8": (C.c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _F, _I, _P, _P]),
    "dvc_dct_blocks_f32": (C.c_int, [_P, _P, _L, _I, _I, _I, _P]),
    "dvc_gaussian_blur_u8": (C.c_int, [_P, _P, _I, _I, _I, _I, _D, _P]),
    "dvc_farneback_flow_f32": (C.c_int, [_P, _P, _P, _I, _I, _I, _D, _I, _I, _I, _I, _D, _I, _P]),
    "dvc_flow_masks_u8": (C.c_int, [_P, _P, _I, _I, _I, _D, _I, _I, _I, _I, _D, _I, _F, _P]),
}

_lib = None


def load() -> C.CDLL:
    """Load libdvc_b200.so (built in-tree by build.py / __graft_entry__.build())."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: run `python -m dynamic_video_compression_surveillance_b200.build` "
                              "(there is no CPU fallback for this path)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def last_error(handle=None) -> str:
    msg = load().dvc_last_error(handle)
    return msg.decode("utf-8", "replace") if msg else ""


def check(rc: int, handle=None) -> None:
    if rc != 0:
        cls = DvcUnsupported if rc == DVC_ERR_UNSUPPORTED else DvcError
        raise cls(rc, last_error(handle))
