"""ctypes binding of libtuatara_b200.so (include/tuatara_c.h).

Fails loudly when the library is missing: there is no Python or CPU fallback for any
GPU stage.  Build with ``python -m tuatara_b200.build`` (or ``__graft_entry__.build()``).
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

LIB_PATH = Path(__file__).resolve().parent / "lib" / "libtuatara_b200.so"


class TuataraError(RuntimeError):
    pass


class tt_image(C.Structure):
    _fields_ = [("data", C.c_void_p), ("rows", C.c_int), ("cols", C.c_int), ("channels", C.c_int),
                ("step", C.c_size_t)]


class tt_config(C.Structure):
    _fields_ = [("canvas_size", C.c_float), ("mag_ratio", C.c_float), ("text_threshold", C.c_float),
                ("link_threshold", C.c_float), ("low_text", C.c_float), ("min_area", C.c_int),
                ("max_batch_pages", C.c_int), ("slots_per_gpu", C.c_int), ("rectify", C.c_int)]


class tt_ocr_options(C.Structure):
    _fields_ = [("pages_on_device", C.c_int), ("override_on_device", C.c_int),
                ("score_override", C.POINTER(C.c_void_p)), ("detect_only", C.c_int), ("with_scores", C.c_int)]


class tt_char_filter(C.Structure):
    _fields_ = [("allow", C.c_char_p), ("block", C.c_char_p)]


class tt_item(C.Structure):
    _fields_ = [("text", C.c_char_p), ("bbox", C.c_float * 4)]


class tt_page_result(C.Structure):
    _fields_ = [("n_items", C.c_int), ("items", C.POINTER(tt_item))]


class tt_result(C.Structure):
    _fields_ = [("n_pages", C.c_int), ("pages", C.POINTER(tt_page_result))]


_P = C.c_void_p
_I = C.c_int
_F = C.c_float
_PI = C.POINTER(C.c_int)
_PF = C.POINTER(C.c_float)

# name -> (restype, argtypes); every symbol include/tuatara_c.h declares
SIGNATURES = {
    "tt_config_default": (None, [C.POINTER(tt_config)]),
    "tt_last_error": (C.c_char_p, []),
    "tt_engine_create": (_I, [C.c_char_p, _PI, _I, C.POINTER(tt_config), C.POINTER(_P)]),
    "tt_engine_destroy": (None, [_P]),
    "tt_device_count": (_I, []),
    "tt_ocr_pages": (_I, [_P, C.POINTER(tt_image), _I, C.POINTER(C.POINTER(tt_result))]),
    "tt_ocr_pages_ex": (_I, [_P, C.POINTER(tt_image), _I, C.POINTER(tt_ocr_options), C.POINTER(C.POINTER(tt_result))]),
    "tt_result_free": (None, [C.POINTER(tt_result)]),
    "tt_char_filter_mask": (_I, [C.POINTER(tt_char_filter), _P]),
    "tt_ocr_pages_filtered": (_I, [_P, C.POINTER(tt_image), _I, C.POINTER(tt_ocr_options), C.POINTER(tt_char_filter), _I,
                                   C.POINTER(C.POINTER(tt_result))]),
    "tt_ocr_pages_oriented": (_I, [_P, C.POINTER(tt_image), _I, C.POINTER(tt_ocr_options), C.POINTER(tt_char_filter), _I,
                                   _P, _I, C.POINTER(C.POINTER(tt_result))]),
    "tt_lexicon_create": (_I, [C.POINTER(C.c_char_p), _I, C.POINTER(_P)]),
    "tt_lexicon_destroy": (None, [_P]),
    "tt_lexicon_info": (_I, [_P, _PI, _PI]),
    "tt_ocr_pages_lexicon": (_I, [_P, C.POINTER(tt_image), _I, C.POINTER(tt_ocr_options), C.POINTER(tt_char_filter), _I,
                                  _P, _I, C.POINTER(_P), _I, C.POINTER(C.POINTER(tt_result))]),
    "tt_ocr_pages_contrast": (_I, [_P, C.POINTER(tt_image), _I, C.POINTER(tt_ocr_options), C.POINTER(tt_char_filter), _I,
                                   _P, _I, C.POINTER(_P), _I, _F, _F, C.POINTER(C.POINTER(tt_result))]),
    "tt_item_angle": (_I, [C.POINTER(tt_result), _I, _I, _PI]),
    "tt_item_scores": (_I, [C.POINTER(tt_result), _I, _I, _PF, _PF, C.POINTER(_PF), _PI]),
    "tt_launch_count": (C.c_ulonglong, []),
    "tt_engine_set_slots": (None, [_P, _I]),
    "tt_engine_stream": (_P, [_P, _I]),
    "tt_io_bytes": (None, [C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong)]),
    "tt_profile_enable": (None, [_I]),
    "tt_profile_collect": (None, [C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_ulonglong)]),
    "tt_profile_dump": (None, [C.c_char_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_ulonglong)]),
    "tt_profile_stages": (_I, [C.c_char_p, _I]),
    "tt_debug_trace_report": (_I, [C.c_char_p, _I]),
    "tt_resize_plan": (_I, [_I, _I, _F, _F, _PI, _PI, _PI, _PI, _PF]),
    "tt_preprocess": (_I, [C.POINTER(tt_image), _F, _F, _P]),
    "tt_craft_forward": (_I, [_P, _P, _I, _I, _P]),
    "tt_postprocess": (_I, [_P, _I, _I, C.POINTER(tt_config), _P, _P, _I, _PI, _P, _P, _I, _PI]),
    "tt_crop_resize": (_I, [C.POINTER(tt_image), _P, _I, _P]),
    "tt_crop_resize_rotated": (_I, [C.POINTER(tt_image), _P, _P, _I, _P]),
    "tt_contrast_adjust": (_I, [_P, _I, _F, _P, _P]),
    "tt_craft_tap": (_I, [_P, C.c_char_p, _P, C.c_longlong, _P]),
    "tt_crop_warp": (_I, [C.POINTER(tt_image), _P, _I, _P]),
    "tt_rect_to_quad": (_I, [_P, _P]),
    "tt_parseq_forward": (_I, [_P, _P, _I, _P, _P, _P]),
    "tt_parseq_forward_scores": (_I, [_P, _P, _I, _P, _P]),
    "tt_parseq_forward_masked": (_I, [_P, _P, _I, _P, _P, _P, _P, _P]),
    "tt_parseq_forward_lexicon": (_I, [_P, _P, _I, _P, _P, _P, _P, _P]),
    "tt_decode": (_I, [_P, _I, _I, _P, _I]),
    "tt_decode_scores": (_I, [_P, _P, _I, _I, _P, _I, _P, _P]),
    "tt_tokenizer_table": (_I, [C.c_char_p, _PI, _PI, _PI]),
    "tt_convex_hull_i32": (_I, [_P, _I, _P, _PI]),
    "tt_convex_hull_f32": (_I, [_P, _I, _P, _PI]),
    "tt_min_area_rect_i32": (_I, [_P, _I, _P]),
    "tt_min_area_rect_f32": (_I, [_P, _I, _P]),
    "tt_rect_points": (_I, [_P, _P]),
    "tt_rect_bounding": (_I, [_P, _P]),
    "tt_adjust_rect": (_I, [_P, _F, _F, _F, _P]),
    "tt_rect_to_bbox": (_I, [_P, _P]),
    "tt_linear_dev": (_I, [_P, _I, _I, _I, _P, _I, _P, _I, _P, _I, _I, _P, _I, _I, _I, _I, _P]),
    "tt_linear_ln_pair_dev": (_I, [_P, _I, _I, _P, _P, _I, _P, _P, _P, _P, _P, _P, _I, _I, C.c_float, _P, _P]),
    "tt_linear_ln_dev": (_I, [_P, _I, _I, _P, _P, _P, _I, _P, _I, C.c_float, _P, _P]),
    "tt_enc_mlp_dev": (_I, [_P, _P, _P, C.c_longlong, _P, _P, _P, _P, _P, _P, _P, _P, C.c_float, _P]),
    "tt_enc_qkv_attn_dev": (_I, [_P, _P, _I, _P, _P, _P, _P, _I, _I, _I, C.c_float, _P]),
    "tt_conv_dev": (_I, [_P, _I, _P, _I, _I, _I, _I, _I, _I, _P, _P, _I, _I, _P, _I, _I, _P]),
    "tt_attn_enc_dev": (_I, [_P, _P, _I, _I, _I, _I, _P]),
    "tt_dec_score_table_dev": (_I, [_P, _P, _I, _I, _I, _I, _P, _P]),
    "tt_dec_self_attn_dev": (_I, [_I, _I, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _I, _I, _P, _P]),
    "tt_dec_cross_attn_dev": (_I, [_I, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P]),
    "tt_orient_select_dev": (_I, [_P, _P, _I, _P, _I, _P, _P, _P, _P]),
    "tt_contrast_select_dev": (_I, [_P, _P, _P, _I, _P, _P, _P]),
    "tt_lexicon_walk_dev": (_I, [_P, _P, _I, _P, _P, _P]),
    "tt_postprocess_dev": (_I, [_P, _P, _I, _I, _I, _PI, _P]),
}

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise TuataraError(f"{LIB_PATH} is missing: run `python -m tuatara_b200.build` "
                               "(there is no CPU fallback for this path)")
        _lib = C.CDLL(str(LIB_PATH))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(_lib, name)
            fn.restype, fn.argtypes = res, args
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise TuataraError(f"{what}: {lib().tt_last_error().decode(errors='replace')}")


def ptr(a) -> int | None:
    """Address of a numpy array / torch tensor / None as a void*."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    return a.data_ptr()  # torch tensor


def image_struct(img: np.ndarray) -> tt_image:
    if img.dtype != np.uint8 or img.ndim != 3:
        raise RuntimeError("Input array should have 3 dimensions")  # bindings/python.cpp:15-17
    if not img.flags.c_contiguous:
        img = np.ascontiguousarray(img)
    s = tt_image(img.ctypes.data, img.shape[0], img.shape[1], img.shape[2], img.strides[0])
    s._keepalive = img
    return s
