"""Synthetic camera frames for tests and benches (there is no camera and no dataset offline).

SURVEY.md section 8d: frames are derived from the reference's only fixture, test/rm_test.jpg
(a dark 1280x1024 arena frame, copied to tests/golden/rm_test.jpg), with per-frame seeded
shifts, gain and sensor noise so that detections differ from frame to frame.
"""
from __future__ import annotations

import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
BASE_IMAGE = os.path.join(os.path.dirname(_HERE), "tests", "golden", "rm_test.jpg")


def load_base(path: str = BASE_IMAGE) -> np.ndarray:
    """BGR u8 [1024,1280,3] as cv::imread returns it (/root/reference/test/yolo_test.cpp:24,63)."""
    import cv2
    img = cv2.imread(path)
    if img is None:
        raise FileNotFoundError(path)
    return img


def frames_from_base(base: np.ndarray, n: int, seed: int = 0) -> np.ndarray:
    """n frames u8 [n,H,W,3]: circular shift (|dx|,|dy| <= 96), gain 0.9..1.2, N(0,3) noise."""
    rng = np.random.default_rng(seed)
    out = np.empty((n,) + base.shape, np.uint8)
    for i in range(n):
        dx, dy = rng.integers(-96, 97, 2)
        gain = rng.uniform(0.9, 1.2)
        f = np.roll(base, (int(dy), int(dx)), (0, 1)).astype(np.float32) * np.float32(gain)
        f += rng.normal(0.0, 3.0, base.shape).astype(np.float32)
        out[i] = np.clip(np.rint(f), 0, 255).astype(np.uint8)
    return out


def bayer_from_rgb(rgb: np.ndarray, pattern: str = "RGGB") -> np.ndarray:
    """Sample an RGB frame [.., H, W, 3] onto an 8-bit Bayer mosaic [.., H, W]."""
    ry, rx = {"RGGB": (0, 0), "BGGR": (1, 1), "GRBG": (0, 1), "GBRG": (1, 0)}[pattern]
    out = rgb[..., 1].copy()
    out[..., ry::2, rx::2] = rgb[..., ry::2, rx::2, 0]
    out[..., (ry ^ 1)::2, (rx ^ 1)::2] = rgb[..., (ry ^ 1)::2, (rx ^ 1)::2, 2]
    return out


# Camera intrinsics the reference ships (config/camera_info.yaml:4-12, a 640 x 480 calibration)
K_CAMERA = (957.669211, 0.0, 345.943891, 0.0, 969.127115, 284.057302, 0.0, 0.0, 1.0)
D_CAMERA = (-0.405274, 0.126058, -0.026939, -0.006503, 0.0)


def armor_object_points(large: bool = False) -> np.ndarray:
    """Armor corners LB, LT, RT, RB in the model frame (x forward, y left, z up), metres
    (/root/reference/src/pnp_solver.cpp:18-33, include/irmv_detection/pnp_solver.hpp:30-33)."""
    hw, hh = ((225.0 if large else 135.0) / 2.0 / 1000.0, 55.0 / 2.0 / 1000.0)
    return np.array([[0, hw, -hh], [0, hw, hh], [0, -hw, hh], [0, -hw, -hh]], np.float64)


def armor_quads(n: int, seed: int = 0, noise_px: float = 0.5, K=K_CAMERA, D=D_CAMERA, img_w: int = 640, img_h: int = 480,
                dist=(0.5, 8.0), yaw: float = 60.0, pitch: float = 30.0, roll: float = 15.0, margin: float = 0.15,
                large: bool = False):
    """SURVEY.md section 8d config 5 input: seeded armor poses (distance uniform in `dist` metres, yaw, pitch and roll
    uniform in +-`yaw`, +-`pitch`, +-`roll` degrees) projected through K/D with N(0, noise_px) pixel noise, kept inside
    the image: f32 [n, 4, 2].  The armor centre aims at a pixel drawn at least `margin` (a fraction of the frame)
    from each edge; `large` selects the large armor.  The defaults are the survey's envelope, and the same seed
    gives the same quads as before these arguments existed.

    Model frame is x-forward/y-left/z-up; the camera looks along +z, so the base rotation maps model x ->
    camera z, model y -> camera -x, model z -> camera -y."""
    import cv2
    rng = np.random.default_rng(seed)
    Km = np.asarray(K, np.float64).reshape(3, 3)
    Dm = np.asarray(D, np.float64).reshape(1, 5)
    base = np.array([[0.0, -1.0, 0.0], [0.0, 0.0, -1.0], [1.0, 0.0, 0.0]])
    obj = armor_object_points(large)
    out = np.empty((n, 4, 2), np.float32)
    i = 0
    while i < n:
        d = rng.uniform(dist[0], dist[1])
        ya, pi, ro = (np.deg2rad(rng.uniform(-yaw, yaw)), np.deg2rad(rng.uniform(-pitch, pitch)),
                      np.deg2rad(rng.uniform(-roll, roll)))
        cy, sy = np.cos(ya), np.sin(ya)
        cp, sp = np.cos(pi), np.sin(pi)
        cr, sr = np.cos(ro), np.sin(ro)
        Ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
        Rx = np.array([[1, 0, 0], [0, cp, -sp], [0, sp, cp]])
        Rz = np.array([[cr, -sr, 0], [sr, cr, 0], [0, 0, 1]])
        R = Rz @ Rx @ Ry @ base
        u = rng.uniform(margin, 1.0 - margin) * img_w
        v = rng.uniform(margin, 1.0 - margin) * img_h
        t = np.array([(u - Km[0, 2]) / Km[0, 0] * d, (v - Km[1, 2]) / Km[1, 1] * d, d])
        rvec, _ = cv2.Rodrigues(R)
        p, _ = cv2.projectPoints(obj, rvec, t, Km, Dm)
        p = p.reshape(4, 2) + rng.normal(0.0, noise_px, (4, 2))
        if (p[:, 0].min() < 0 or p[:, 0].max() >= img_w or p[:, 1].min() < 0 or p[:, 1].max() >= img_h):
            continue
        out[i] = p.astype(np.float32)
        i += 1
    return out


def armor_scene(n_armors: int = 6, seed: int = 0, w: int = 1280, h: int = 1024, noise: bool = True):
    """A dark arena frame (rotated view) with bright light-bar pairs and the boxes a detector would put
    around them; returns (image u8[h,w,3], boxes[n,4], scores[n], classes[n])."""
    import cv2
    rng = np.random.default_rng(seed)
    img = rng.integers(0, 60, (h, w, 3), dtype=np.uint8) if noise else np.zeros((h, w, 3), np.uint8)
    boxes, scores, classes = [], [], []
    for k in range(n_armors):
        cx, cy = rng.uniform(120, w - 120), rng.uniform(100, h - 100)
        L = rng.uniform(18, 70)                       # light length, px
        large = rng.random() < 0.3
        sep = L * (rng.uniform(3.5, 5.0) if large else rng.uniform(1.2, 2.8))
        tilt = rng.uniform(-20, 20)
        wd = L * rng.uniform(0.15, 0.3)
        for sgn in (-1, 1):
            c = (cx + sgn * sep / 2, cy + rng.uniform(-2, 2))
            box = cv2.boxPoints((c, (wd, L), tilt + rng.uniform(-4, 4)))
            cv2.fillConvexPoly(img, np.round(box).astype(np.int32), (int(rng.integers(200, 256)),) * 3)
        if rng.random() < 0.5:                        # a number sticker between the lights (dim or bright)
            v = int(rng.integers(100, 256))
            cv2.putText(img, str(int(rng.integers(1, 6))), (int(cx - L / 4), int(cy + L / 4)), cv2.FONT_HERSHEY_SIMPLEX,
                        L / 40, (v, v, v), max(1, int(L / 15)))
        m = rng.uniform(0.05, 0.3)
        boxes.append([cx - sep / 2 - wd - m * sep, cy - L * (0.6 + m), cx + sep / 2 + wd + m * sep, cy + L * (0.6 + m)])
        scores.append(rng.uniform(0.3, 0.95))
        classes.append(int(rng.integers(0, 14)))
    return img, np.array(boxes, np.float32), np.array(scores, np.float32), np.array(classes, np.int32)
