"""Python mirror of the reference's YoloEngine / PnPSolver interfaces over the C ABI.

Names, argument meaning and error behaviour follow the reference classes
(/root/reference/include/irmv_detection/yolo_engine.hpp:16-73, pnp_solver.hpp:12-38); the
arithmetic is entirely in libirmv_b200.so (CUDA, sm_100a).  numpy is used for host buffers only.
"""
from __future__ import annotations

import ctypes as C
import enum
import os
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import _lib as L


class ArmorClass(enum.IntEnum):
    """/root/reference/include/irmv_detection/armor.hpp:7"""
    B1 = 0; B2 = 1; B3 = 2; B4 = 3; B5 = 4; BO = 5; BS = 6
    R1 = 7; R2 = 8; R3 = 9; R4 = 10; R5 = 11; RO = 12; RS = 13
    UNKNOWN = 14


@dataclass
class bbox:
    """YoloEngine::bbox, /root/reference/include/irmv_detection/yolo_engine.hpp:19-26"""
    xyxy: Tuple[float, float, float, float]
    score: float
    class_id: ArmorClass


def weights_path_for(onnx_file_path: str) -> str:
    """The reference swaps the .onnx extension for .engine (src/yolo_engine.cpp:28-31); the
    B200 engine swaps it for .irmw."""
    root, _ = os.path.splitext(onnx_file_path)
    return root + ".irmw"


class YoloEngine:
    """YoloEngine(onnx_file_path, src_image_size=(W,H), enable_profiling=False)

    Extra keyword arguments expose what the reference hard-codes: channel order, rotation,
    batch size and the bring-up convolution kernel.
    """

    def __init__(self, onnx_file_path: str, src_image_size: Tuple[int, int] = (1280, 1024),
                 enable_profiling: bool = False, *, chan_order: int = L.CH_PASSTHROUGH,
                 rotate180: bool = True, quantize_u8: bool = True, half_pixel: bool = False, letterbox: bool = False,
                 max_batch: int = 1,
                 sub_batch: int = 0, num_lanes: int = 0, num_slots: int = 3, device: int = 0,
                 conv_impl: int = L.CONV_TCGEN05, score_thr: float = 0.25, iou_thr: float = 0.45,
                 max_det: int = 100, use_graph: bool = True, fused_stem: bool = True, fuse_tails: bool = True,
                 fuse_units: bool = True, split_upsample_convs: bool = True, raw_format: int = L.RAW_8):
        lib = L.lib()
        wpath = onnx_file_path if onnx_file_path.endswith(".irmw") else weights_path_for(onnx_file_path)
        if not os.path.exists(wpath):
            # reference: prints and exit(0)s (src/yolo_engine.cpp:37-40); raising is the Python form
            raise FileNotFoundError(f"weight file {wpath} not found (build it with "
                                    "irmv_detection_b200.weights.write_random or convert a checkpoint)")
        cfg = L.EngineConfig()
        L.check(lib.irmv_engine_config_default(C.byref(cfg)), "irmv_engine_config_default")
        cfg.src_width, cfg.src_height = int(src_image_size[0]), int(src_image_size[1])
        cfg.chan_order = chan_order
        cfg.rotate180 = int(rotate180)
        cfg.quantize_u8 = int(quantize_u8)
        cfg.resize_mode = L.RESIZE_LETTERBOX if letterbox else (L.RESIZE_STRETCH_HALF_PIXEL if half_pixel else L.RESIZE_STRETCH)
        cfg.max_batch, cfg.sub_batch, cfg.num_lanes, cfg.num_slots = max_batch, sub_batch, num_lanes, num_slots
        cfg.device, cfg.conv_impl = device, conv_impl
        cfg.score_thr, cfg.iou_thr, cfg.max_det = score_thr, iou_thr, max_det
        cfg.use_graph = int(use_graph)
        cfg.reserved[0] = 0 if fused_stem else 1
        cfg.reserved[1] = 0 if fuse_tails else 1
        cfg.reserved[2] = 0 if fuse_units else 1          # ShuffleNetV2 variant: one kernel per unit (default) or one per conv
        cfg.reserved[3] = 0 if split_upsample_convs else 1   # neck cv1 over concat(upsample(a), b): two raster launches or one gather launch
        cfg.raw_format = raw_format
        self._cfg = cfg
        self._h = C.c_void_p()
        self._lib = lib
        L.check(lib.irmv_engine_create(wpath.encode(), C.byref(cfg), C.byref(self._h)), "irmv_engine_create")
        self.src_image_size = (cfg.src_width, cfg.src_height)
        self.enable_profiling = enable_profiling
        self.channels = 1 if chan_order >= L.CH_BAYER_RGGB else 3
        self.raw_format = raw_format
        W, H = cfg.src_width, cfg.src_height
        # one frame as the engine takes it: dtype and shape (RAW_8: [H, W] Bayer or [H, W, 3] packed RGB)
        if raw_format in (L.RAW_10, L.RAW_12):
            self.frame_dtype, self.frame_shape = np.dtype(np.uint16), (H, W)
        elif raw_format == L.RAW_12_PACKED:
            self.frame_dtype, self.frame_shape = np.dtype(np.uint8), (H, W * 3 // 2)
        else:
            self.frame_dtype, self.frame_shape = np.dtype(np.uint8), (H, W) + ((3,) if self.channels == 3 else ())
        self.raw_bits = {L.RAW_10: 10, L.RAW_12: 12, L.RAW_12_PACKED: 12}.get(raw_format, 8)
        self.frame_bytes = int(np.prod(self.frame_shape)) * self.frame_dtype.itemsize
        self.max_batch, self.max_det = max_batch, max_det
        self._slot = 0
        self._out = (L.Bbox * (max_batch * max_det))()
        self._counts = (C.c_int * max_batch)()
        self._ticket_n = [0, 0, 0]

    # -- reference surface ---------------------------------------------------------------
    def get_src_image_buffer(self, slot: int = 0) -> np.ndarray:
        """Pinned-host frame slot as a writable numpy view (reference returns uint8_t*): u8 [H, W, 3] or [H, W] for
        8-bit sources, u16 [H, W] for RAW_10 / RAW_12, u8 [H, 3W/2] for RAW_12_PACKED."""
        p = self._lib.irmv_engine_src_buffer(self._h, slot)
        if not p:
            raise L.IrmvError("bad slot")
        buf = (C.c_uint8 * self.frame_bytes).from_address(p)
        return np.frombuffer(buf, self.frame_dtype).reshape(self.frame_shape)

    def detect(self, slot: int = 0) -> List[bbox]:
        n = C.c_int(0)
        L.check(self._lib.irmv_engine_detect(self._h, slot, self._out, self.max_det, C.byref(n)), "irmv_engine_detect")
        self._slot = slot
        return self._to_list(0, n.value)

    def get_rotated_image(self, slot: Optional[int] = None) -> np.ndarray:
        slot = self._slot if slot is None else slot
        out = np.empty((self.src_image_size[1], self.src_image_size[0], 3), np.uint8)
        L.check(self._lib.irmv_engine_rotated_image(self._h, slot, out.ctypes.data), "irmv_engine_rotated_image")
        return out

    def get_rotated_view(self, slot: Optional[int] = None) -> np.ndarray:
        """Zero-copy form of get_rotated_image(): a read-only view of the engine's pinned, address-stable
        rotated-frame buffer of `slot`, refreshed by every detect() once this has been called."""
        slot = self._slot if slot is None else slot
        p = C.c_void_p()
        L.check(self._lib.irmv_engine_rotated_view(self._h, slot, C.byref(p)), "irmv_engine_rotated_view")
        n = self.src_image_size[0] * self.src_image_size[1] * 3
        buf = (C.c_uint8 * n).from_address(p.value)
        return np.frombuffer(buf, np.uint8).reshape(self.src_image_size[1], self.src_image_size[0], 3)

    def get_profiling_time(self) -> float:
        return float(self._lib.irmv_engine_profile_ms(self._h))

    # -- batch extension -----------------------------------------------------------------
    def detect_batch(self, frames: np.ndarray) -> List[List[bbox]]:
        """frames u8 [n,H,W,3] (or [n,H,W] Bayer) in host memory; 10/12-bit engines: [n] frames of exactly
        get_src_image_buffer()'s dtype and shape."""
        if self.raw_format != L.RAW_8:
            frames = self._raw_frames(frames)
        else:
            frames = np.ascontiguousarray(frames, np.uint8)
        n = frames.shape[0]
        if frames[0].size != self.frame_bytes // self.frame_dtype.itemsize:
            raise ValueError("frame size does not match the engine's src_image_size")
        L.check(self._lib.irmv_engine_detect_batch(self._h, frames.ctypes.data, 0, n, self._out, self._counts),
                "irmv_engine_detect_batch")
        return [self._to_list(f, self._counts[f]) for f in range(n)]

    def detect_batch_arrays(self, frames: np.ndarray):
        """Same call as detect_batch, results as arrays (no per-detection Python objects):
        counts i32[n] and a structured view {xyxy f32[4], score f32, class_id i32}[n, max_det]."""
        frames = self._raw_frames(frames) if self.raw_format != L.RAW_8 else np.ascontiguousarray(frames, np.uint8)
        n = frames.shape[0]
        L.check(self._lib.irmv_engine_detect_batch(self._h, frames.ctypes.data, 0, n, self._out, self._counts),
                "irmv_engine_detect_batch")
        dt = np.dtype([("xyxy", np.float32, 4), ("score", np.float32), ("class_id", np.int32)])
        dets = np.frombuffer(self._out, dtype=dt, count=n * self.max_det).reshape(n, self.max_det)
        return np.frombuffer(self._counts, dtype=np.int32, count=n), dets

    # -- pipelined hand-off (copy of batch k+1 under the kernels of batch k) ---------------
    def submit_batch(self, frames: np.ndarray) -> int:
        """Queue H2D + pipeline + D2H for host frames and return a ticket; at most three batches in
        flight, collect in order.  `frames` must stay alive and unchanged until collected (pinned
        memory makes the copy asynchronous)."""
        if self.raw_format != L.RAW_8:
            frames = self._raw_frames(frames, copy=False)
        elif not frames.flags.c_contiguous or frames.dtype != np.uint8:
            raise ValueError("submit_batch needs a C-contiguous uint8 array")
        n = frames.shape[0]
        if frames[0].size != self.frame_bytes // self.frame_dtype.itemsize:
            raise ValueError("frame size does not match the engine's src_image_size")
        t = C.c_int(0)
        L.check(self._lib.irmv_engine_submit_batch(self._h, frames.ctypes.data, n, C.byref(t)), "irmv_engine_submit_batch")
        self._ticket_n[t.value % 3] = n
        return t.value

    def _raw_frames(self, frames: np.ndarray, copy: bool = True) -> np.ndarray:
        """Host frames of a 10/12-bit engine: exactly [n] + frame_shape of frame_dtype, never cast (a cast would
        truncate or reinterpret the samples).  copy=False: they must already be C-contiguous."""
        frames = np.asarray(frames)
        if frames.dtype != self.frame_dtype or frames.ndim != 1 + len(self.frame_shape) or \
                tuple(frames.shape[1:]) != self.frame_shape or frames.shape[0] < 1:
            raise ValueError(f"this engine takes {self.frame_dtype.name} frames of shape [n, "
                             f"{', '.join(map(str, self.frame_shape))}], got {frames.dtype.name} {list(frames.shape)}")
        if not frames.flags.c_contiguous:
            if not copy:
                raise ValueError("submit_batch needs a C-contiguous array")
            frames = np.ascontiguousarray(frames)
        return frames

    def collect_arrays(self, ticket: int, poses: bool = False):
        """Wait for a submitted batch: (counts i32[n], dets structured [n, max_det]) and, with
        poses=True, (rvec f64[n,max_det,3], tvec, ok).  The arrays are views that the next collect
        of the same parity overwrites."""
        n = self._ticket_n[ticket % 3]
        rv = tv = ok = None
        if poses:
            rv = np.empty((n, self.max_det, 3)); tv = np.empty((n, self.max_det, 3))
            ok = np.empty((n, self.max_det), np.uint8)
        L.check(self._lib.irmv_engine_collect(self._h, ticket, self._out, self._counts,
                                              rv.ctypes.data if poses else None, tv.ctypes.data if poses else None,
                                              ok.ctypes.data if poses else None), "irmv_engine_collect")
        dt = np.dtype([("xyxy", np.float32, 4), ("score", np.float32), ("class_id", np.int32)])
        dets = np.frombuffer(self._out, dtype=dt, count=n * self.max_det).reshape(n, self.max_det)
        counts = np.frombuffer(self._counts, dtype=np.int32, count=n)
        return (counts, dets, rv, tv, ok.astype(bool)) if poses else (counts, dets)

    def detect_batch_device(self, dev_ptr: int, n: int) -> List[List[bbox]]:
        L.check(self._lib.irmv_engine_detect_batch(self._h, C.c_void_p(dev_ptr), 1, n, self._out, self._counts),
                "irmv_engine_detect_batch")
        return [self._to_list(f, self._counts[f]) for f in range(n)]

    def enqueue_batch_device(self, dev_ptr: int, n: int) -> None:
        L.check(self._lib.irmv_engine_enqueue_batch(self._h, C.c_void_p(dev_ptr), n), "irmv_engine_enqueue_batch")

    def sync(self) -> float:
        L.check(self._lib.irmv_engine_sync(self._h), "irmv_engine_sync")
        return float(self._lib.irmv_engine_last_device_ms(self._h))

    def fetch(self, n: int) -> List[List[bbox]]:
        L.check(self._lib.irmv_engine_fetch(self._h, n, self._out, self._counts), "irmv_engine_fetch")
        return [self._to_list(f, self._counts[f]) for f in range(n)]

    def last_device_ms(self) -> float:
        return float(self._lib.irmv_engine_last_device_ms(self._h))

    def copy_bytes(self) -> Tuple[int, int]:
        """(host->device, device->host) bytes of every copy the engine has queued since creation."""
        a, b = C.c_ulonglong(0), C.c_ulonglong(0)
        L.check(self._lib.irmv_engine_copy_bytes(self._h, C.byref(a), C.byref(b)), "irmv_engine_copy_bytes")
        return int(a.value), int(b.value)

    def kernel_launches(self, n: int) -> int:
        return int(self._lib.irmv_engine_kernel_launches(self._h, n))

    def enable_pnp(self, camera_matrix, dist_coeffs, corner_scale=(1.0, 1.0)) -> None:
        """Fuse the pose stage (box corners -> IPPE) into every replay."""
        K = (C.c_double * 9)(*[float(v) for v in camera_matrix])
        D = (C.c_double * 5)(*[float(v) for v in list(dist_coeffs)[:5]])
        L.check(self._lib.irmv_engine_enable_pnp(self._h, K, D, float(corner_scale[0]), float(corner_scale[1])),
                "irmv_engine_enable_pnp")

    def fetch_poses(self, n: int):
        rv = np.empty((n, self.max_det, 3)); tv = np.empty((n, self.max_det, 3))
        ok = np.empty((n, self.max_det), np.uint8)
        L.check(self._lib.irmv_engine_fetch_poses(self._h, n, rv.ctypes.data, tv.ctypes.data, ok.ctypes.data),
                "irmv_engine_fetch_poses")
        return rv, tv, ok.astype(bool)

    def fetch_armor_poses(self, n: int, ticket: int = -1) -> np.ndarray:
        """Per-armor message payload of IrmDetector::message_callback (position, tf2 quaternion x y z w,
        distance_to_image_center, ok) from the fused replay: structured POSE_DTYPE [n, max_det]."""
        out = np.zeros((n, self.max_det), POSE_DTYPE)
        L.check(self._lib.irmv_engine_fetch_armor_poses(self._h, ticket, n, out.ctypes.data), "irmv_engine_fetch_armor_poses")
        return out

    def has_keypoints(self) -> bool:
        """True when the weight file carries the keypoint branch (72 convolutions)."""
        return bool(self._lib.irmv_engine_has_keypoints(self._h))

    def fetch_keypoints(self, n: int, ticket: int = -1) -> np.ndarray:
        """Keypoints (armor corners LB, LT, RT, RB) of the kept detections, source pixels: f32[n, max_det, 4, 2]."""
        out = np.zeros((n, self.max_det, 4, 2), np.float32)
        L.check(self._lib.irmv_engine_fetch_keypoints(self._h, ticket, n, out.ctypes.data), "irmv_engine_fetch_keypoints")
        return out

    def enable_armors(self, **params) -> None:
        """Fuse IrmDetector::extract_armors (light bars -> armors) into every replay, between NMS and
        PnP; keyword arguments override the node-parameter defaults (see armor_params)."""
        prm = armor_params(**params)
        L.check(self._lib.irmv_engine_enable_armors(self._h, C.byref(prm)), "irmv_engine_enable_armors")

    def set_raw_lut(self, lut: Optional[np.ndarray]) -> None:
        """Raw-domain colour stage of a Bayer engine: `lut` is a (3, 2^b) uint8 table (rows: red, green, blue
        sites; b = 8, 10 or 12 bits per raw sample) that every raw sample goes through before the demosaic, or None.
        8-bit engines: None switches the table off, and the engine with table L on frames F returns what it returns
        without a table on raw_lut.apply_raw_lut(F, L).  10/12-bit engines: None restores the default shift
        s >> (b - 8); the engine returns what an 8-bit engine without a table returns on raw_lut.decode_raw(F, ...)."""
        if lut is None:
            L.check(self._lib.irmv_engine_set_raw_lut(self._h, None), "irmv_engine_set_raw_lut")
            return
        lut = np.asarray(lut)
        n = 1 << self.raw_bits
        if lut.shape != (3, n) or lut.dtype != np.uint8:
            raise ValueError(f"set_raw_lut needs a (3, {n}) uint8 table or None")
        lut = np.ascontiguousarray(lut)
        L.check(self._lib.irmv_engine_set_raw_lut(self._h, lut.ctypes.data), "irmv_engine_set_raw_lut")

    def set_color_matrix(self, m: Optional[np.ndarray], tone: Optional[np.ndarray] = None) -> None:
        """Colour-correction stage of a Bayer engine: `m` is a (3, 3) int16 matrix in units of 1/1024 and `tone` a
        (3, 256) uint8 output tone table or None (identity), applied to every demosaiced pixel after the raw table
        (or the 10/12-bit decode) and before rot180 and resize; m None switches the stage off (tone must be None
        then).  The engine with M and T on Bayer frames F returns what a PASSTHROUGH engine returns on the packed
        frames raw_lut.apply_color_matrix(demosaic_bilinear(F), M, T).  raw_lut.color_matrix_q10 builds M from a
        colour-correction matrix and a saturation gain; raw_lut.make_raw_lut(0, (1, 1, 1), gamma) is a tone table."""
        from . import raw_lut as R
        mp = tp = None
        if m is not None:
            m = np.ascontiguousarray(R._check_matrix(m))
            mp = m.ctypes.data
        if tone is not None:
            tone = np.ascontiguousarray(R._check_tone(tone))
            tp = tone.ctypes.data
        L.check(self._lib.irmv_engine_set_color_matrix(self._h, mp, tp), "irmv_engine_set_color_matrix")

    def set_auto_white_balance(self, params: Optional[dict] = None) -> None:
        """Automatic white balance of a Bayer engine, per frame: `params` is None (off, the default) or a dict
        overriding raw_lut.AWB_DEFAULTS (dark_level, clip_level, min_quads, gain_max_q10).  Every frame is then
        demosaiced with the colour-correction matrix raw_lut.awb_matrix(g, M) and the tone table T of
        set_color_matrix (M = 1024 * I and identity tone when none is set), g = raw_lut.awb_gains of
        raw_lut.awb_statistics of the frame's 8-bit mosaic.  fetch_white_balance returns what was applied; with AWB
        off, set_color_matrix(raw_lut.awb_matrix(g, M), T) reproduces it exactly (locks the white balance)."""
        if params is None:
            L.check(self._lib.irmv_engine_set_auto_white_balance(self._h, None), "irmv_engine_set_auto_white_balance")
            return
        from . import raw_lut as R
        p = R.awb_params(params)
        prm = L.AwbParams(p["dark_level"], p["clip_level"], p["min_quads"], p["gain_max_q10"])
        L.check(self._lib.irmv_engine_set_auto_white_balance(self._h, C.byref(prm)), "irmv_engine_set_auto_white_balance")

    def fetch_white_balance(self, n: int, ticket: int = -1) -> np.ndarray:
        """Auto white balance records of the last synchronous call (or of a collected ticket): structured AWB_DTYPE
        [n] (sum = SR, SG, SB over the counted quads; counted, dark, clipped quads; valid; gain_q10)."""
        out = np.zeros(n, AWB_DTYPE)
        L.check(self._lib.irmv_engine_fetch_white_balance(self._h, ticket, n, out.ctypes.data),
                "irmv_engine_fetch_white_balance")
        return out

    def fetch_armors(self, n: int, ticket: int = -1) -> np.ndarray:
        """Armors of the last synchronous call (or of a collected ticket): structured [n, max_det]."""
        out = np.zeros((n, self.max_det), ARMOR_DTYPE)
        L.check(self._lib.irmv_engine_fetch_armors(self._h, ticket, n, out.ctypes.data), "irmv_engine_fetch_armors")
        return out

    def check_padding(self) -> int:
        """Debug: number of padding pixels of the activation tensors that are not zero (0 unless a kernel stored out of bounds)."""
        bad = C.c_longlong(-1)
        L.check(self._lib.irmv_debug_check_padding(self._h, C.byref(bad)), "irmv_debug_check_padding")
        return int(bad.value)

    def stem_camera_ctas(self) -> int:
        """Debug: CTAs per SM of the camera-case stem kernel (csrc/stem_bayer.cu) as the engine launches it now, with
        its raw table when one is set; 0 when the frames go to the generic stem kernel instead."""
        n = C.c_int(-1)
        L.check(self._lib.irmv_debug_stem_ctas(self._h, C.byref(n)), "irmv_debug_stem_ctas")
        return int(n.value)

    def describe_ops(self):
        """Kernels of the network stage in issue order: dicts {kind, k, s, cin, cout, hw, raster, tail_cout}."""
        buf = C.create_string_buffer(16384)
        if self._lib.irmv_engine_describe_ops(self._h, buf, 16384) < 0:
            L.check(1, "irmv_engine_describe_ops")
        ops = []
        for line in buf.value.decode().splitlines():
            f = line.split()
            if f[0] == "pool":
                ops.append({"kind": "pool"})
            elif f[0] == "dw":
                ops.append({"kind": "dw", "s": int(f[1]), "c": int(f[2]), "hw": int(f[3])})
            elif f[0] == "unit":
                ops.append({"kind": "unit", "down": bool(int(f[1])), "cin": int(f[2]), "h": int(f[3]), "hw": int(f[4]), "rows_per_cta": int(f[5])})
            else:
                k, s, cin, cout, hw, raster, tail = (int(v) for v in f[1:])
                ops.append({"kind": "conv", "k": k, "s": s, "cin": cin, "cout": cout, "hw": hw, "raster": bool(raster),
                            "tail_cout": tail})
        return ops

    def describe_plans(self, n: int):
        """Tiling plan / kernel instantiation of every network-stage launch for a replay of n frames:
        list of tuples ("raster", k, s, cin, cout, hw, R, nepi, b_stream, ctas_per_sm, stages, b_stages, tail,
        act, res, tiles) | ("gather", k, s, cin, cout, hw) | ("pool",)."""
        buf = C.create_string_buffer(32768)
        if self._lib.irmv_engine_describe_plans(self._h, n, buf, 32768) < 0:
            L.check(1, "irmv_engine_describe_plans")
        out = []
        for line in buf.value.decode().splitlines():
            f = line.split()
            out.append((f[0],) + tuple(int(v) for v in f[1:]))
        return out

    def profile_stages(self, dev_ptr: int, n: int):
        ms = (C.c_float * 5)()
        k = self._lib.irmv_engine_profile_stages(self._h, C.c_void_p(dev_ptr), n, C.byref(ms))
        if k <= 0:
            L.check(1, "irmv_engine_profile_stages")
        return k, dict(zip(("preprocess", "conv", "decode_nms", "pnp", "total"), [float(v) for v in ms]))

    # -- parity taps ---------------------------------------------------------------------
    def read_tensor(self, name: str) -> np.ndarray:
        dims = (C.c_int32 * 5)()
        L.check(self._lib.irmv_engine_read_tensor(self._h, name.encode(), None, 0, C.byref(dims)), "read_tensor")
        b, h, w, c, es = list(dims)
        out = np.empty((b, h, w, c), np.float32 if es == 4 else np.float16)
        L.check(self._lib.irmv_engine_read_tensor(self._h, name.encode(), out.ctypes.data, out.nbytes, C.byref(dims)),
                "read_tensor")
        return out

    def kept_indices(self, frame: int = 0) -> np.ndarray:
        idx = np.empty(self.max_det, np.int32)
        n = C.c_int(0)
        L.check(self._lib.irmv_engine_read_kept_indices(self._h, frame, idx.ctypes.data, self.max_det, C.byref(n)),
                "read_kept_indices")
        return idx[: n.value].copy()

    def _to_list(self, frame: int, k: int) -> List[bbox]:
        out = []
        base = frame * self.max_det
        for i in range(k):
            b = self._out[base + i]
            out.append(bbox(tuple(b.xyxy), float(b.score), ArmorClass(int(b.class_id))))
        return out

    def close(self) -> None:
        if getattr(self, "_h", None) and self._h.value:
            self._lib.irmv_engine_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class PnPSolver:
    """PnPSolver(camera_matrix[9], dist_coeffs[>=5]); solvePnP(points) -> (ok, rvec, tvec).

    `points` stands for the reference's Armor: the four image points in the order
    left_light.bottom, left_light.top, right_light.top, right_light.bottom
    (/root/reference/src/pnp_solver.cpp:41-44).
    """

    def __init__(self, camera_matrix: Sequence[float], dist_coeffs: Sequence[float], device: int = 0):
        self._lib = L.lib()
        K = (C.c_double * 9)(*[float(v) for v in camera_matrix])
        D = (C.c_double * 5)(*[float(v) for v in list(dist_coeffs)[:5]])
        self._h = C.c_void_p()
        L.check(self._lib.irmv_pnp_create(K, D, device, C.byref(self._h)), "irmv_pnp_create")

    def solvePnP(self, points) -> Tuple[bool, np.ndarray, np.ndarray]:
        pts = (C.c_float * 8)(*np.asarray(points, np.float32).reshape(8))
        r = (C.c_double * 3)()
        t = (C.c_double * 3)()
        ok = C.c_int(0)
        L.check(self._lib.irmv_pnp_solve(self._h, pts, r, t, C.byref(ok)), "irmv_pnp_solve")
        return bool(ok.value), np.array(r[:]).reshape(3, 1), np.array(t[:]).reshape(3, 1)

    def solve_batch(self, points: np.ndarray, large_armor: bool = False, extended: bool = False):
        pts = np.ascontiguousarray(points, np.float32).reshape(-1, 8)
        n = pts.shape[0]
        rv = np.empty((n, 3)); tv = np.empty((n, 3)); ok = np.empty(n, np.uint8)
        if not extended:
            L.check(self._lib.irmv_pnp_solve_batch(self._h, pts.ctypes.data, n, 0, int(large_armor),
                                                   rv.ctypes.data, tv.ctypes.data, ok.ctypes.data), "irmv_pnp_solve_batch")
            return rv, tv, ok.astype(bool)
        q = np.empty((n, 4)); rv2 = np.empty((n, 3)); tv2 = np.empty((n, 3)); e = np.empty((n, 2))
        L.check(self._lib.irmv_pnp_solve_batch_ex(self._h, pts.ctypes.data, n, 0, int(large_armor), rv.ctypes.data,
                                                  tv.ctypes.data, ok.ctypes.data, q.ctypes.data, rv2.ctypes.data,
                                                  tv2.ctypes.data, e.ctypes.data), "irmv_pnp_solve_batch_ex")
        return rv, tv, ok.astype(bool), q, rv2, tv2, e

    def solve_batch_device(self, dev_ptr: int, n: int, rv: np.ndarray, tv: np.ndarray, ok: np.ndarray,
                           large_armor: bool = False) -> float:
        L.check(self._lib.irmv_pnp_solve_batch(self._h, C.c_void_p(dev_ptr), n, 1, int(large_armor),
                                               rv.ctypes.data, tv.ctypes.data, ok.ctypes.data), "irmv_pnp_solve_batch")
        return float(self._lib.irmv_pnp_last_device_ms(self._h))

    def last_device_ms(self) -> float:
        return float(self._lib.irmv_pnp_last_device_ms(self._h))

    def set_refine_lm(self, max_iters: int = 20) -> None:
        """Optional Levenberg-Marquardt refinement after IPPE (0 = off = reference behaviour)."""
        L.check(self._lib.irmv_pnp_set_refine_lm(self._h, int(max_iters)), "irmv_pnp_set_refine_lm")

    def calculateDistanceToCenter(self, image_point) -> float:
        return float(self._lib.irmv_pnp_distance_to_center(self._h, float(image_point[0]), float(image_point[1])))

    def close(self) -> None:
        if getattr(self, "_h", None) and self._h.value:
            self._lib.irmv_pnp_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


ARMOR_DTYPE = np.dtype([("pts", np.float32, (4, 2)), ("center", np.float32, 2), ("score", np.float32),
                        ("class_id", np.int32), ("size", np.int32), ("valid", np.int32)])
POSE_DTYPE = np.dtype([("position", np.float64, 3), ("orientation", np.float64, 4), ("rvec", np.float64, 3),
                       ("distance_to_image_center", np.float32), ("ok", np.int32)])
AWB_DTYPE = np.dtype([("sum", np.uint64, 3), ("counted", np.uint32), ("dark", np.uint32), ("clipped", np.uint32),
                      ("valid", np.int32), ("gain_q10", np.int32, 3), ("reserved", np.int32)])   # == irmv_awb
BBOX_DTYPE = np.dtype([("xyxy", np.float32, 4), ("score", np.float32), ("class_id", np.int32)])


def armor_params(**kw) -> "L.ArmorParams":
    """Node parameters of the light / armor filters (reference src/irm_detector.cpp:152,162-173)."""
    prm = L.ArmorParams()
    L.check(L.lib().irmv_armor_params_default(C.byref(prm)), "irmv_armor_params_default")
    for k, v in kw.items():
        if not hasattr(prm, k):
            raise TypeError(f"unknown armor parameter {k}")
        setattr(prm, k, v)
    return prm


# ---- stage-level wrappers (parity tests) ------------------------------------------------------
def extract_armors(frames: np.ndarray, boxes: np.ndarray, counts: np.ndarray, chan_order: int = L.CH_PASSTHROUGH,
                   rotate180: bool = True, device: int = 0, **params) -> np.ndarray:
    """IrmDetector::extract_armors on the GPU.  frames u8 [n,H,W,3] or [n,H,W] as the camera wrote
    them; boxes structured BBOX_DTYPE [n, max_det] (source pixels) with counts[n] valid entries.
    Returns ARMOR_DTYPE [n, max_det], slot-aligned with boxes."""
    frames = np.ascontiguousarray(frames, np.uint8)
    n, H, W = frames.shape[:3]
    return extract_armors_ptr(frames.ctypes.data, False, n, W, H, boxes, counts, chan_order, rotate180, device, **params)


def extract_armors_ptr(ptr: int, on_device: bool, n: int, W: int, H: int, boxes: np.ndarray, counts: np.ndarray,
                       chan_order: int = L.CH_PASSTHROUGH, rotate180: bool = True, device: int = 0, **params) -> np.ndarray:
    """Same stage on n frames at a raw host or device address (device: no copy of the frames)."""
    boxes = np.ascontiguousarray(boxes, BBOX_DTYPE)
    counts = np.ascontiguousarray(counts, np.int32)
    max_det = boxes.shape[1]
    out = np.zeros((n, max_det), ARMOR_DTYPE)
    prm = armor_params(**params)
    L.check(L.lib().irmv_extract_armors(C.c_void_p(ptr), int(on_device), n, W, H, chan_order, int(rotate180),
                                        boxes.ctypes.data, counts.ctypes.data, max_det, C.byref(prm), device,
                                        out.ctypes.data), "irmv_extract_armors")
    return out


def extract_armors_last_device_ms() -> float:
    return float(L.lib().irmv_extract_armors_last_device_ms())



def preprocess(frames: np.ndarray, chan_order: int = L.CH_PASSTHROUGH, rotate180: bool = True,
               quantize_u8: bool = True, want_rotated: bool = False, device: int = 0,
               half_pixel: bool = False, letterbox: bool = False):
    """frames u8 [n,H,W,3] or [n,H,W] -> FP16 [n,640,640,8] NHWC (+ rotated u8 [n,H,W,3])."""
    frames = np.ascontiguousarray(frames, np.uint8)
    n, H, W = frames.shape[:3]
    out = np.empty((n, L.NET, L.NET, 8), np.float16)
    rot = np.empty((n, H, W, 3), np.uint8) if want_rotated else None
    L.check(L.lib().irmv_preprocess(frames.ctypes.data, n, W, H, chan_order, int(rotate180),
                                    L.RESIZE_LETTERBOX if letterbox else
                                    (L.RESIZE_STRETCH_HALF_PIXEL if half_pixel else L.RESIZE_STRETCH),
                                    int(quantize_u8), out.ctypes.data, rot.ctypes.data if want_rotated else None,
                                    device), "irmv_preprocess")
    return (out, rot) if want_rotated else out


def nms(boxes: np.ndarray, scores: np.ndarray, score_thr: float = 0.25, iou_thr: float = 0.45,
        max_det: int = 100, device: int = 0):
    """boxes f32 [n,A,4], scores f32 [n,A,nc] -> per frame (index, boxes, scores, classes)."""
    boxes = np.ascontiguousarray(boxes, np.float32)
    scores = np.ascontiguousarray(scores, np.float32)
    n, A, nc = scores.shape
    num = np.zeros(n, np.int32)
    db = np.zeros((n, max_det, 4), np.float32); ds = np.zeros((n, max_det), np.float32)
    dc = np.zeros((n, max_det), np.int32); di = np.zeros((n, max_det), np.int32)
    L.check(L.lib().irmv_nms(boxes.ctypes.data, scores.ctypes.data, n, A, nc, score_thr, iou_thr, max_det,
                             num.ctypes.data, db.ctypes.data, ds.ctypes.data, dc.ctypes.data, di.ctypes.data, device),
            "irmv_nms")
    return [(di[f, :num[f]].copy(), db[f, :num[f]].copy(), ds[f, :num[f]].copy(), dc[f, :num[f]].copy())
            for f in range(n)]


def decode(box: np.ndarray, cls: np.ndarray, device: int = 0):
    """box f16 [n,8400,64], cls f16 [n,8400,16] -> boxes f32 [n,8400,4], scores f32 [n,8400,14]."""
    box = np.ascontiguousarray(box, np.float16)
    cls = np.ascontiguousarray(cls, np.float16)
    n = box.shape[0]
    boxes = np.empty((n, L.NUM_ANCHORS, 4), np.float32)
    scores = np.empty((n, L.NUM_ANCHORS, L.NUM_CLASSES), np.float32)
    L.check(L.lib().irmv_decode(box.ctypes.data, cls.ctypes.data, n, boxes.ctypes.data, scores.ctypes.data, device),
            "irmv_decode")
    return boxes, scores
