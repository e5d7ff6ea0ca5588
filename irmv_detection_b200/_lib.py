"""ctypes binding of libirmv_b200.so (include/irmv_cabi.h).  No fallback: if the CUDA library is
missing or fails to load, importing the product path raises."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libirmv_b200.so")

NET = 640
NUM_CLASSES = 14
CLASS_UNKNOWN = 14
NUM_ANCHORS = 8400

CH_PASSTHROUGH, CH_SWAP_RB, CH_BAYER_RGGB, CH_BAYER_BGGR, CH_BAYER_GRBG, CH_BAYER_GBRG = range(6)
RESIZE_STRETCH, RESIZE_LETTERBOX, RESIZE_STRETCH_HALF_PIXEL = 0, 1, 2
CONV_TCGEN05, CONV_DIRECT = 0, 1
RAW_8, RAW_10, RAW_12, RAW_12_PACKED = range(4)


class Bbox(C.Structure):
    _fields_ = [("xyxy", C.c_float * 4), ("score", C.c_float), ("class_id", C.c_int32)]


class Armor(C.Structure):
    _fields_ = [("pts", C.c_float * 8), ("center", C.c_float * 2), ("score", C.c_float), ("class_id", C.c_int32),
                ("size", C.c_int32), ("valid", C.c_int32)]


class Pose(C.Structure):
    _fields_ = [("position", C.c_double * 3), ("orientation", C.c_double * 4), ("rvec", C.c_double * 3),
                ("distance_to_image_center", C.c_float), ("ok", C.c_int32)]


class ArmorParams(C.Structure):
    _fields_ = [("binary_threshold", C.c_int32), ("light_min_ratio", C.c_float), ("light_max_ratio", C.c_float),
                ("light_max_angle", C.c_float), ("min_small_center_distance", C.c_double),
                ("max_small_center_distance", C.c_double), ("min_large_center_distance", C.c_double),
                ("max_large_center_distance", C.c_double)]


class AwbParams(C.Structure):
    _fields_ = [("dark_level", C.c_int32), ("clip_level", C.c_int32), ("min_quads", C.c_int32),
                ("gain_max_q10", C.c_int32)]


class EngineConfig(C.Structure):
    _fields_ = [
        ("src_width", C.c_int32), ("src_height", C.c_int32), ("chan_order", C.c_int32),
        ("rotate180", C.c_int32), ("resize_mode", C.c_int32), ("quantize_u8", C.c_int32),
        ("max_batch", C.c_int32), ("sub_batch", C.c_int32), ("num_lanes", C.c_int32),
        ("num_slots", C.c_int32), ("device", C.c_int32), ("conv_impl", C.c_int32),
        ("max_det", C.c_int32), ("score_thr", C.c_float), ("iou_thr", C.c_float),
        ("use_graph", C.c_int32), ("reserved", C.c_int32 * 7), ("raw_format", C.c_int32),
    ]


# every symbol include/irmv_cabi.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "irmv_last_error": (C.c_char_p, []),
    "irmv_version": (C.c_int, []),
    "irmv_chan_order_from_media_type": (C.c_int, [C.c_uint32]),
    "irmv_source_format_from_media_type": (C.c_int, [C.c_uint32, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "irmv_engine_config_default": (C.c_int, [C.POINTER(EngineConfig)]),
    "irmv_engine_create": (C.c_int, [C.c_char_p, C.POINTER(EngineConfig), C.POINTER(_P)]),
    "irmv_engine_destroy": (None, [_P]),
    "irmv_engine_src_buffer": (_P, [_P, C.c_int]),
    "irmv_engine_rotated_image": (C.c_int, [_P, C.c_int, _P]),
    "irmv_engine_rotated_view": (C.c_int, [_P, C.c_int, C.POINTER(_P)]),
    "irmv_debug_alloc_count": (C.c_longlong, []),
    "irmv_debug_check_padding": (C.c_int, [C.c_void_p, C.POINTER(C.c_longlong)]),
    "irmv_debug_stem_ctas": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "irmv_engine_fetch_armor_poses": (C.c_int, [_P, C.c_int, C.c_int, _P]),
    "irmv_engine_detect": (C.c_int, [_P, C.c_int, C.POINTER(Bbox), C.c_int, C.POINTER(C.c_int)]),
    "irmv_engine_detect_batch": (C.c_int, [_P, _P, C.c_int, C.c_int, C.POINTER(Bbox), C.POINTER(C.c_int)]),
    "irmv_engine_enqueue_batch": (C.c_int, [_P, _P, C.c_int]),
    "irmv_engine_sync": (C.c_int, [_P]),
    "irmv_engine_fetch": (C.c_int, [_P, C.c_int, C.POINTER(Bbox), C.POINTER(C.c_int)]),
    "irmv_engine_profile_ms": (C.c_double, [_P]),
    "irmv_engine_copy_bytes": (C.c_int, [_P, C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong)]),
    "irmv_engine_last_device_ms": (C.c_double, [_P]),
    "irmv_engine_kernel_launches": (C.c_int, [_P, C.c_int]),
    "irmv_engine_stream": (_P, [_P]),
    "irmv_engine_enable_pnp": (C.c_int, [_P, C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_float, C.c_float]),
    "irmv_engine_fetch_poses": (C.c_int, [_P, C.c_int, _P, _P, _P]),
    "irmv_engine_has_keypoints": (C.c_int, [_P]),
    "irmv_engine_fetch_keypoints": (C.c_int, [_P, C.c_int, C.c_int, _P]),
    "irmv_armor_params_default": (C.c_int, [C.POINTER(ArmorParams)]),
    "irmv_extract_armors": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, C.c_int,
                                      C.POINTER(ArmorParams), C.c_int, _P]),
    "irmv_extract_armors_last_device_ms": (C.c_double, []),
    "irmv_extract_armors_last_profile": (C.c_int, [C.POINTER(C.c_uint64 * 8)]),
    "irmv_engine_enable_armors": (C.c_int, [_P, C.POINTER(ArmorParams)]),
    "irmv_engine_fetch_armors": (C.c_int, [_P, C.c_int, C.c_int, _P]),
    "irmv_engine_set_raw_lut": (C.c_int, [_P, _P]),
    "irmv_engine_set_color_matrix": (C.c_int, [_P, _P, _P]),
    "irmv_awb_params_default": (C.c_int, [C.POINTER(AwbParams)]),
    "irmv_engine_set_auto_white_balance": (C.c_int, [_P, C.POINTER(AwbParams)]),
    "irmv_engine_fetch_white_balance": (C.c_int, [_P, C.c_int, C.c_int, _P]),
    "irmv_engine_profile_stages": (C.c_int, [_P, _P, C.c_int, C.POINTER(C.c_float * 5)]),
    "irmv_engine_submit_batch": (C.c_int, [_P, _P, C.c_int, C.POINTER(C.c_int)]),
    "irmv_engine_collect": (C.c_int, [_P, C.c_int, _P, _P, _P, _P, _P]),
    "irmv_engine_describe_ops": (C.c_int, [_P, _P, C.c_int]),
    "irmv_engine_describe_plans": (C.c_int, [_P, C.c_int, _P, C.c_int]),
    "irmv_engine_profile_ops": (C.c_int, [_P, _P, C.c_int, _P, C.c_int]),
    "irmv_engine_trace_conv": (C.c_int, [_P, C.c_int, C.c_int, _P, C.c_int, C.POINTER(C.c_float)]),
    "irmv_engine_read_tensor": (C.c_int, [_P, C.c_char_p, _P, C.c_int64, C.POINTER(C.c_int32 * 5)]),
    "irmv_engine_read_kept_indices": (C.c_int, [_P, C.c_int, _P, C.c_int, C.POINTER(C.c_int)]),
    "irmv_preprocess": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, C.c_int]),
    "irmv_nms": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int, _P, _P, _P, _P, _P, C.c_int]),
    "irmv_decode": (C.c_int, [_P, _P, C.c_int, _P, _P, C.c_int]),
    "irmv_pnp_create": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_int, C.POINTER(_P)]),
    "irmv_pnp_destroy": (None, [_P]),
    "irmv_pnp_solve": (C.c_int, [_P, C.POINTER(C.c_float), C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int)]),
    "irmv_pnp_solve_batch": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "irmv_pnp_solve_batch_ex": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P, _P, _P, _P]),
    "irmv_pnp_last_device_ms": (C.c_double, [_P]),
    "irmv_pnp_set_refine_lm": (C.c_int, [_P, C.c_int]),
    "irmv_pnp_distance_to_center": (C.c_float, [_P, C.c_float, C.c_float]),
}

_lib = None


class IrmvError(RuntimeError):
    pass


def lib() -> C.CDLL:
    """Load the CUDA library (once).  Raises if it is not built -- there is no CPU path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise IrmvError(
                f"{LIB_PATH} is missing: build it with `python -m irmv_detection_b200.build` "
                "(nvcc, sm_100a).  irmv_detection_b200 has no CPU fallback.")
        l = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(l, name)     # AttributeError if the library does not export it
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().irmv_last_error()
        raise IrmvError(f"{what} failed (code {rc}): {msg.decode() if msg else ''}")
