"""ctypes binding of libpadel_b200.so (the C ABI declared in include/padel_b200.h).

There is no CPU fallback: if the library is missing or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import os

_HERE = Path(__file__).resolve().parent
# PADEL_B200_LIB: load another build of the same ABI (bring-up A/B of experimental kernels); default = the product lib
LIB_PATH = Path(os.environ["PADEL_B200_LIB"]).resolve() if os.environ.get("PADEL_B200_LIB") else _HERE / "libpadel_b200.so"


class PbError(RuntimeError):
    pass


class ConvDesc(C.Structure):
    _fields_ = [
        ("in_", C.c_void_p),
        ("N", C.c_int), ("H", C.c_int), ("W", C.c_int), ("C", C.c_int),
        ("c_in_off", C.c_int), ("cin", C.c_int),
        ("weight", C.c_void_p), ("bias", C.c_void_p),
        ("cout_pad", C.c_int), ("ksize", C.c_int), ("stride", C.c_int), ("act", C.c_int),
        ("res", C.c_void_p), ("res_C", C.c_int), ("res_coff", C.c_int),
        ("out", C.c_void_p), ("out_C", C.c_int), ("out_coff", C.c_int), ("out_mode", C.c_int),
        ("cout_store", C.c_int),
        ("head_weight", C.c_void_p), ("head_bias", C.c_void_p), ("head_n", C.c_int), ("head_out", C.c_void_p),
        ("in_layout", C.c_int),
        ("res_before_act", C.c_int),
        ("out2", C.c_void_p), ("out2_C", C.c_int), ("out2_coff", C.c_int), ("out2_mode", C.c_int),
    ]


class YoloLevel(C.Structure):
    _fields_ = [("feat", C.c_void_p), ("h", C.c_int), ("w", C.c_int), ("stride", C.c_int)]


ACT_NONE, ACT_RELU, ACT_SILU, ACT_SIGMOID = 0, 1, 2, 3
OUT_F16_NHWC, OUT_F16_NHWC_UP2, OUT_F32_NHWC, OUT_F32_NCHW, OUT_NONE = 0, 1, 2, 3, 4
IN_NHWC, IN_STEM4 = 0, 1
OUT2_NONE, OUT2_UP2, OUT2_POOL2 = 0, 1, 2

# name -> (restype, argtypes); must list every symbol of include/padel_b200.h (tests check this)
_i, _p, _f = C.c_int, C.c_void_p, C.c_float
SIGNATURES = {
    "pb_last_error": (C.c_char_p, []),
    "pb_version": (_i, []),
    "pb_launch_count": (C.c_longlong, []),
    "pb_conv2d": (_i, [C.POINTER(ConvDesc), _p]),
    "pb_conv2d_reference": (_i, [C.POINTER(ConvDesc), _p]),
    "pb_program_create": (_p, []),
    "pb_program_destroy": (None, [_p]),
    "pb_program_add_conv": (_i, [_p, C.POINTER(ConvDesc)]),
    "pb_program_add_maxpool2": (_i, [_p, _p, _i, _i, _i, _i, _i, _i, _p, _i, _i]),
    "pb_program_add_sppf_pool": (_i, [_p, _p, _i, _i, _i, _i, _i]),
    "pb_program_num_ops": (_i, [_p]),
    "pb_program_op_kernel": (_i, [_p, _i]),
    "pb_program_run": (_i, [_p, _p]),
    "pb_program_run_range": (_i, [_p, _i, _i, _p]),
    "pb_letterbox_u8_f16": (_i, [_p, _i, _i, _i, _p, _i, _i, _i, _i, _i, _i, _p, _p, _p, _p, _i, _i, _i, _i, _p]),
    "pb_pil_resize_u8": (_i, [_p, _i, _i, _i, _p, _p, _i, _i, _p, _p, _i, _p, _p, _i, _i, _p, _i, _p]),
    "pb_u8_to_f16_nhwc16": (_i, [_p, _i, _i, _i, _p, _i, _i, _i, _i, _p]),
    "pb_tracknet_pack_windows": (_i, [_p, _i, _i, _p, _i, _i, _i, _p, _p]),
    "pb_yolo_decode": (_i, [C.POINTER(YoloLevel), _i, _i, _i, _i, _i, _i, _i, _i, _f, C.POINTER(C.c_int), _i, _p, _p, _p,
                             _i, _p]),
    "pb_yolo_nms_scratch_bytes": (C.c_size_t, [_i, _i]),
    "pb_yolo_nms": (_i, [_p, _p, _p, _i, _i, _i, _f, _i, _p, _p, _p, _p]),
    "pb_u8_normalize_f16": (_i, [_p, C.c_longlong, C.POINTER(C.c_float), C.POINTER(C.c_float), _p, _p]),
    "pb_resnet_stem7x7": (_i, [_p, _i, _i, _i, _p, _p, _p, _p]),
    "pb_maxpool3x3s2": (_i, [_p, _i, _i, _i, _i, _p, _p]),
    "pb_avgpool_fc_sigmoid": (_i, [_p, _i, _i, _i, _p, _p, _i, _p, _p]),
    "pb_bytetrack_create": (_p, [C.c_double, _i, C.c_double, C.c_double]),
    "pb_bytetrack_destroy": (None, [_p]),
    "pb_bytetrack_reset": (None, [_p]),
    "pb_bytetrack_update": (_i, [_p, _p, _p, _i, _p]),
    "pb_bytetrack_update_many": (_i, [_p, _p, _p, _p, _i, _p]),
    "pb_inpaintnet_forward": (_i, [_p, _p, _i, _i, _p, _p, _p]),
    "pb_median_u8": (_i, [_p, _i, C.c_longlong, _p, _i, _p]),
    "pb_tracknet_ensemble": (_i, [_p, _i, _i, _i, _i, _i, _i, _i, _f, _p, _p, _p]),
    "pb_ccl_bbox": (_i, [_p, _i, _i, _i, _p, _p, _p]),
}

_lib = None


def lib() -> C.CDLL:
    """Load the shared library (once). Raises PbError if it has not been built."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise PbError(
                f"{LIB_PATH} not found: build it with `python -m padel_analytics_b200.build` "
                "(no CPU fallback exists)")
        l = C.CDLL(str(LIB_PATH))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        raise PbError(lib().pb_last_error().decode())


def ptr(t) -> int:
    """Device/host pointer of a torch tensor (or None)."""
    return 0 if t is None else t.data_ptr()


def stream_ptr() -> int:
    import torch

    return torch.cuda.current_stream().cuda_stream
