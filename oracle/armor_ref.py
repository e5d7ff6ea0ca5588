"""CPU oracle for the light/armor extraction that feeds PnP (TEST INFRASTRUCTURE ONLY: imported by
tests/, __graft_entry__.smoke() and bench.py's CPU legs, never by the product path).

Restates `IrmDetector::extract_armors` (/root/reference/src/irm_detector.cpp:292-355) and the
`Light` / `Armor` constructors (/root/reference/include/irmv_detection/armor.hpp:11-77).  The
arithmetic of the OpenCV calls it makes lives in OpenCV (system dependency, version unpinned by
the reference's package.xml); the binary oracle here is cv2 4.13:

  cv::cvtColor(BGR2GRAY)   -> gray_bgr2gray()          pinned bit-exact against cv2.cvtColor
  cv::threshold(BINARY)    -> gray > thr
  cv::findContours(RETR_EXTERNAL, CHAIN_APPROX_SIMPLE)
                           -> find_external_contours() pinned point-for-point against cv2.findContours
                              (Suzuki-Abe border following, 8-connected foreground, top-level outer
                              borders only, contours returned in reverse raster order of their start)
  cv::minAreaRect          -> min_area_rect()          pinned against cv2.minAreaRect/boxPoints
                              (same rectangle; corner coordinates agree to float rounding; shapes
                              with two different rectangles of equal area are reported as ambiguous)

`extract_armors_cv2` is the reference's function written with the cv2 calls themselves;
`extract_armors` is the restatement the CUDA kernel follows (csrc/armors.cu).

The image the reference hands to extract_armors is `get_rotated_image()`: the 180-degree rotated
source in the buffer's own channel order (src/irm_detector.cpp:183, src/yolo_engine.cpp:182-184).
It calls COLOR_BGR2GRAY on it whatever that order is, so memory channel 0 gets the blue weight.
For a Bayer source the vendor ISP writes RGB8 (src/mv_camera.cpp:64,96), i.e. channel 0 = R.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

from . import preprocess_ref as PR

# OpenCV's 8-bit BGR2GRAY: 15-bit fixed point (imgproc/src/color_yuv / color_rgb: BY15, GY15, RY15)
BY15, GY15, RY15, GRAY_SHIFT = 3735, 19235, 9798, 15

SMALL, LARGE = 0, 1


@dataclass
class ArmorParams:
    """Node parameters, /root/reference/src/irm_detector.cpp:152,162-173."""
    binary_threshold: int = 150
    light_min_ratio: float = 0.1
    light_max_ratio: float = 0.4
    light_max_angle: float = 40.0
    min_small_center_distance: float = 0.8
    max_small_center_distance: float = 3.2
    min_large_center_distance: float = 3.2
    max_large_center_distance: float = 5.5


@dataclass
class Light:
    center: np.ndarray
    top: np.ndarray
    bottom: np.ndarray
    length: float
    width: float
    tilt_angle: float


@dataclass
class Armor:
    """pts = the PnP image points in the order PnPSolver::solvePnP builds them
    (/root/reference/src/pnp_solver.cpp:41-44): left.bottom, left.top, right.top, right.bottom."""
    pts: np.ndarray
    center: np.ndarray
    size: int
    class_id: int
    score: float
    bbox_index: int
    ambiguous: bool = field(default=False)


def rotated_image(frame: np.ndarray, chan: int = PR.CH_PASSTHROUGH, rotate: bool = True) -> np.ndarray:
    """The frame as `get_rotated_image()` exposes it: packed sources keep their byte order, Bayer
    sources are demosaiced to RGB first (the ISP's job in the reference)."""
    if chan >= PR.CH_BAYER_RGGB:
        img = PR.demosaic_bilinear(frame, chan)
    else:
        img = frame
    return PR.rot180(img) if rotate else np.ascontiguousarray(img)


def gray_bgr2gray(img: np.ndarray) -> np.ndarray:
    c = img.astype(np.int64)
    return ((c[..., 0] * BY15 + c[..., 1] * GY15 + c[..., 2] * RY15 + (1 << (GRAY_SHIFT - 1))) >> GRAY_SHIFT).astype(np.uint8)


# 8 directions, OpenCV's chain code: 0 = E, 1 = NE, 2 = N, 3 = NW, 4 = W, 5 = SW, 6 = S, 7 = SE (y down)
_DX = (1, 1, 0, -1, -1, -1, 0, 1)
_DY = (0, -1, -1, -1, 0, 1, 1, 1)


def trace_outer_border(fg: np.ndarray, x0: int, y0: int):
    """Suzuki-Abe border following from an outer-border start pixel (left neighbour is background),
    CHAIN_APPROX_SIMPLE point selection: a pixel is emitted when the outgoing direction differs from
    the previous outgoing direction.  fg is a bool array padded by one background pixel all round;
    (x0, y0) are padded coordinates.  Returns the points in unpadded coordinates."""
    s = 4
    while True:
        s = (s - 1) & 7
        if fg[y0 + _DY[s], x0 + _DX[s]] or s == 4:
            break
    if s == 4:
        return [(x0 - 1, y0 - 1)]
    x1, y1 = x0 + _DX[s], y0 + _DY[s]
    pts = []
    x3, y3 = x0, y0
    prev_s = s ^ 4
    while True:
        while True:
            s = (s + 1) & 7
            x4, y4 = x3 + _DX[s], y3 + _DY[s]
            if fg[y4, x4]:
                break
        if s != prev_s:
            pts.append((x3 - 1, y3 - 1))
        prev_s = s
        if x4 == x0 and y4 == y0 and x3 == x1 and y3 == y1:
            break
        x3, y3 = x4, y4
        s = (s + 4) & 7
    return pts


def exterior_background(fg: np.ndarray) -> np.ndarray:
    """Background pixels 4-connected to the outside of the (padded) image."""
    h, w = fg.shape
    ext = np.zeros_like(fg)
    ext[0, :] = ext[-1, :] = ext[:, 0] = ext[:, -1] = True
    ext &= ~fg
    stack = list(zip(*np.nonzero(ext)))
    while stack:
        y, x = stack.pop()
        for dy, dx in ((1, 0), (-1, 0), (0, 1), (0, -1)):
            yy, xx = y + dy, x + dx
            if 0 <= yy < h and 0 <= xx < w and not fg[yy, xx] and not ext[yy, xx]:
                ext[yy, xx] = True
                stack.append((yy, xx))
    return ext


def find_external_contours(binary: np.ndarray):
    """cv2.findContours(binary, RETR_EXTERNAL, CHAIN_APPROX_SIMPLE): list of (n, 2) int arrays (x, y).

    Formulated the way the CUDA kernel does it, without a serial raster scan: a component is top
    level iff the background left of its first pixel (raster order) reaches the image frame; a
    start candidate is a foreground pixel whose W neighbour is exterior background and whose NW, N,
    NE neighbours are background; the candidate owns the border iff no pixel of the traced border
    precedes it in raster order."""
    h, w = binary.shape
    fg = np.zeros((h + 2, w + 2), bool)
    fg[1:-1, 1:-1] = binary != 0
    ext = exterior_background(fg)
    cand = fg[1:-1, 1:-1] & ext[1:-1, :-2] & ~fg[:-2, :-2] & ~fg[:-2, 1:-1] & ~fg[:-2, 2:]
    out = []
    ys, xs = np.nonzero(cand)
    for y, x in zip(ys.tolist(), xs.tolist()):
        pts = trace_outer_border_full(fg, x + 1, y + 1)
        if pts is None:
            continue
        out.append(np.array(pts, np.int32).reshape(-1, 2))
    return out[::-1]


def trace_outer_border_full(fg, x0, y0):
    """trace_outer_border with the ownership test: None if the border visits a pixel that precedes
    (x0, y0) in raster order (the border then belongs to that earlier start, or is a hole border)."""
    s = 4
    while True:
        s = (s - 1) & 7
        if fg[y0 + _DY[s], x0 + _DX[s]] or s == 4:
            break
    if s == 4:
        return [(x0 - 1, y0 - 1)]
    x1, y1 = x0 + _DX[s], y0 + _DY[s]
    pts = []
    x3, y3 = x0, y0
    prev_s = s ^ 4
    while True:
        while True:
            s = (s + 1) & 7
            x4, y4 = x3 + _DX[s], y3 + _DY[s]
            if fg[y4, x4]:
                break
        if y4 < y0 or (y4 == y0 and x4 < x0):
            return None
        if s != prev_s:
            pts.append((x3 - 1, y3 - 1))
        prev_s = s
        if x4 == x0 and y4 == y0 and x3 == x1 and y3 == y1:
            break
        x3, y3 = x4, y4
        s = (s + 4) & 7
    return pts


def convex_hull(points: np.ndarray) -> np.ndarray:
    """Andrew monotone chain on integer points; strictly convex vertices, counter-clockwise in a
    y-up frame (any consistent order serves min_area_rect)."""
    p = sorted(set(map(tuple, points.tolist())))
    if len(p) <= 2:
        return np.array(p, np.int64).reshape(-1, 2)

    def cross(o, a, b):
        return (a[0] - o[0]) * (b[1] - o[1]) - (a[1] - o[1]) * (b[0] - o[0])

    lo = []
    for q in p:
        while len(lo) >= 2 and cross(lo[-2], lo[-1], q) <= 0:
            lo.pop()
        lo.append(q)
    up = []
    for q in reversed(p):
        while len(up) >= 2 and cross(up[-2], up[-1], q) <= 0:
            up.pop()
        up.append(q)
    return np.array(lo[:-1] + up[:-1], np.int64).reshape(-1, 2)


def min_area_rect(points: np.ndarray):
    """Minimum-area enclosing rectangle of an integer point set (cv::minAreaRect = convex hull +
    rotating calipers; a minimum-area rectangle has a side on a hull edge, so scanning the hull edges
    finds the same rectangle).  FP32 arithmetic like OpenCV's.  Returns (corners[4,2] float32,
    center[2] float32, ambiguous): `ambiguous` is set when a different rectangle has the same area
    to 1e-3 relative (OpenCV's choice then depends on rounding inside its calipers walk)."""
    hull = convex_hull(points)
    n = len(hull)
    f = np.float32
    if n == 0:
        raise ValueError("empty contour")
    if n == 1:
        c = hull[0].astype(f)
        return np.tile(c, (4, 1)), c, False
    org = hull[0]                       # project relative to a hull vertex: small numbers, exact in FP32
    hp = (hull - org).astype(f)
    best = None
    cands = []
    for i in range(n if n > 2 else 1):
        a, b = hp[i], hp[(i + 1) % n]
        e = b - a
        ln = f(np.sqrt(e[0] * e[0] + e[1] * e[1]))
        u = e / ln
        v = np.array([-u[1], u[0]], f)
        pu = hp[:, 0] * u[0] + hp[:, 1] * u[1]        # two FP32 products, one FP32 sum (no FMA), like the kernel
        pv = hp[:, 0] * v[0] + hp[:, 1] * v[1]
        u0, u1, v0, v1 = pu.min(), pu.max(), pv.min(), pv.max()
        area = f((u1 - u0) * (v1 - v0))
        corners = np.stack([u * u0 + v * v0, u * u1 + v * v0, u * u1 + v * v1, u * u0 + v * v1]).astype(f)
        cands.append((area, corners))
        if best is None or area < best[0]:
            best = (area, corners)
    area, corners = best
    corners = (corners + org.astype(f)).astype(f)
    center = ((corners[0] + corners[2]) * f(0.5)).astype(f)
    ambiguous = False
    key = np.sort(np.ascontiguousarray(corners).view(np.complex64).ravel())
    for a2, c2 in cands:
        if abs(float(a2) - float(area)) <= 1e-3 * max(float(area), 1e-12):
            k2 = np.sort(np.ascontiguousarray((c2 + org.astype(f)).astype(f)).view(np.complex64).ravel())
            if np.abs(k2 - key).max() > 1e-2:
                ambiguous = True
    return corners, center, ambiguous


def make_light(corners: np.ndarray, center: np.ndarray) -> Light:
    """Light::Light, armor.hpp:15-29: corners sorted by y; top/bottom = midpoints of the two upper /
    two lower corners; length = |top - bottom|; width = |p0 - p1|; tilt from the vertical in degrees."""
    p = corners[np.argsort(corners[:, 1], kind="stable")].astype(np.float32)
    top = ((p[0] + p[1]) / np.float32(2)).astype(np.float32)
    bottom = ((p[2] + p[3]) / np.float32(2)).astype(np.float32)
    d = (top - bottom).astype(np.float64)
    length = float(np.hypot(d[0], d[1]))
    w = (p[0] - p[1]).astype(np.float64)
    width = float(np.hypot(w[0], w[1]))
    # std::atan2(float, float) is the float overload; the division by CV_PI happens in double
    tilt = float(np.arctan2(np.abs(top[0] - bottom[0]), np.abs(top[1] - bottom[1]))) / np.pi * 180.0
    return Light(center.astype(np.float32), top, bottom, length, width, tilt)


def light_is_unstable(corners: np.ndarray, eps: float = 1e-3) -> bool:
    """Light::Light pairs the corners by sorted y (armor.hpp:19-21).  When the second and third corner
    have the same y to rounding (a rectangle whose short and long side project equally, common for
    small lattice shapes), which pair is "top" is decided by float noise inside cv::minAreaRect and by
    std::sort: the reference's own answer is not stable there."""
    y = np.sort(corners[:, 1].astype(np.float64))
    return bool(abs(y[1] - y[2]) < eps and (abs(y[0] - y[1]) > eps or abs(y[2] - y[3]) > eps))


def is_light(l: Light, prm: ArmorParams) -> bool:
    """Light::is_light, armor.hpp:31-38 (float parameters, double ratio; NaN compares false)."""
    if l.length == 0.0:
        ratio = float("nan") if l.width == 0.0 else float("inf")
    else:
        ratio = l.width / l.length
    mn, mx, ma = (float(np.float32(prm.light_min_ratio)), float(np.float32(prm.light_max_ratio)),
                  float(np.float32(prm.light_max_angle)))
    return (mn < ratio < mx) and (l.tilt_angle < ma)


def roi_of(bbox_xyxy, cols: int, rows: int):
    """src/irm_detector.cpp:299-304: float clamp, then cv::Rect's float -> int truncation."""
    f = np.float32
    min_x, min_y = max(f(bbox_xyxy[0]), f(0)), max(f(bbox_xyxy[1]), f(0))
    max_x, max_y = min(f(bbox_xyxy[2]), f(cols)), min(f(bbox_xyxy[3]), f(rows))
    if not (min_x < max_x and min_y < max_y):       # also drops NaN boxes
        return None
    rx, ry, rw, rh = int(min_x), int(min_y), int(f(max_x - min_x)), int(f(max_y - min_y))
    if rw <= 0 or rh <= 0:
        return None                                  # (the reference would throw inside cvtColor)
    return rx, ry, rw, rh, f(min_x), f(min_y)


def _armor_from(l0: Light, l1: Light, cls: int, score: float, idx: int, prm: ArmorParams, amb: bool):
    """Armor::Armor (armor.hpp:58-68) + the size / centre-distance filter (irm_detector.cpp:333-350)."""
    left, right = (l0, l1) if l0.center[0] < l1.center[0] else (l1, l0)
    center = ((left.center + right.center) / np.float32(2)).astype(np.float32)
    avg_len = (l0.length + l1.length) / 2
    d = (left.center - right.center).astype(np.float64)
    cd = float(np.hypot(d[0], d[1])) / avg_len if avg_len != 0 else float("inf")
    size = LARGE if cd > prm.min_large_center_distance else SMALL
    if size == SMALL and (prm.min_small_center_distance > cd or prm.max_small_center_distance < cd):
        return None
    if size == LARGE and (prm.min_large_center_distance > cd or prm.max_large_center_distance < cd):
        return None
    pts = np.stack([left.bottom, left.top, right.top, right.bottom]).astype(np.float32)
    return Armor(pts, center, size, int(cls), float(score), idx, amb)


def _offset(l: Light, min_x, min_y) -> Light:
    o = np.array([min_x, min_y], np.float32)
    return Light(l.center + o, l.top + o, l.bottom + o, l.length, l.width, l.tilt_angle)


def extract_armors(image: np.ndarray, boxes: np.ndarray, scores, classes, prm: ArmorParams = ArmorParams(),
                   ambiguous: dict | None = None):
    """Restatement the CUDA kernel follows.  image: rotated packed u8x3; boxes: [n,4] xyxy source pixels.
    `ambiguous` (optional) receives {box index: True} for boxes where a contour that was looked at has
    two different minimum-area rectangles (see min_area_rect)."""
    rows, cols = image.shape[:2]
    out = []
    for i, b in enumerate(np.asarray(boxes, np.float32).reshape(-1, 4)):
        roi = roi_of(b, cols, rows)
        if roi is None:
            continue
        rx, ry, rw, rh, min_x, min_y = roi
        binary = gray_bgr2gray(image[ry:ry + rh, rx:rx + rw]) > prm.binary_threshold
        lights, amb = [], False
        for c in find_external_contours(binary):
            if len(c) < 5:
                continue
            corners, center, a = min_area_rect(c)
            amb |= a or light_is_unstable(corners)
            l = make_light(corners, center)
            if not is_light(l, prm):
                continue
            lights.append(_offset(l, min_x, min_y))
            if len(lights) == 2:
                break
        if amb and ambiguous is not None:
            ambiguous[i] = True
        if len(lights) < 2:
            continue
        arm = _armor_from(lights[0], lights[1], classes[i], scores[i], i, prm, amb)
        if arm is not None:
            out.append(arm)
    return out


def extract_armors_cv2(image: np.ndarray, boxes: np.ndarray, scores, classes, prm: ArmorParams = ArmorParams()):
    """The reference's function with the cv2 calls themselves (binary oracle)."""
    import cv2
    rows, cols = image.shape[:2]
    out = []
    for i, b in enumerate(np.asarray(boxes, np.float32).reshape(-1, 4)):
        roi = roi_of(b, cols, rows)
        if roi is None:
            continue
        rx, ry, rw, rh, min_x, min_y = roi
        gray = cv2.cvtColor(np.ascontiguousarray(image[ry:ry + rh, rx:rx + rw]), cv2.COLOR_BGR2GRAY)
        _, binary = cv2.threshold(gray, prm.binary_threshold, 255, cv2.THRESH_BINARY)
        contours, _ = cv2.findContours(binary, cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_SIMPLE)
        lights = []
        for c in contours:
            if len(c) < 5:
                continue
            rect = cv2.minAreaRect(c)
            corners = cv2.boxPoints(rect).astype(np.float32)
            l = make_light(corners, np.array(rect[0], np.float32))
            if not is_light(l, prm):
                continue
            lights.append(_offset(l, min_x, min_y))
        if len(lights) < 2:
            continue
        arm = _armor_from(lights[0], lights[1], classes[i], scores[i], i, prm, False)
        if arm is not None:
            out.append(arm)
    return out


ARMOR_TOL_PX = 1e-2     # corner / centre agreement of the CUDA stage with cv2 (FP32 rectangle arithmetic on both sides)


def check_armors(got, image, boxes, scores, classes, prm: ArmorParams = ArmorParams()):
    """The GPU stage's armors of one frame against the reference's function written with the cv2 calls.

    got: ARMOR_DTYPE[max_det] (irmv_detection_b200.ARMOR_DTYPE), slot-aligned with `boxes` [n, 4] (rotated-view
    pixels); image: the rotated view.  Valid flags, size class, class and score must be identical and corners and
    centre within ARMOR_TOL_PX; every slot from n on must be invalid.  A box may only differ where the restatement
    `extract_armors` reports an ambiguous minimum-area rectangle (two different rectangles of equal area: OpenCV's pick
    depends on rounding inside its calipers).  The restatement is pure Python and runs on the mismatched boxes only.
    Returns (number of armors of the reference, indices of the excused boxes)."""
    ref = {a.bbox_index: a for a in extract_armors_cv2(image, boxes, scores, classes, prm)}
    bad = []
    for i in range(len(boxes)):
        g = got[i]
        if bool(g["valid"]) != (i in ref):
            bad.append(i)
            continue
        if i in ref:
            r = ref[i]
            if (int(g["size"]) != r.size or np.abs(g["pts"] - r.pts).max() > ARMOR_TOL_PX or
                    np.abs(g["center"] - r.center).max() > ARMOR_TOL_PX):
                bad.append(i)
            else:
                assert int(g["class_id"]) == r.class_id and abs(float(g["score"]) - r.score) < 1e-7, f"box {i}"
    assert not got[len(boxes):]["valid"].any(), "an armor in a slot past the frame's detection count"
    if bad:
        amb = {}
        sub = np.asarray(boxes)[bad]
        extract_armors(image, sub, np.asarray(scores)[bad], np.asarray(classes)[bad], prm, ambiguous=amb)
        not_excused = [bad[k] for k in range(len(bad)) if k not in amb]
        assert not not_excused, f"armor mismatch on boxes {not_excused}"
    return len(ref), bad


def boxes_struct(boxes, scores, classes, max_det: int):
    """One frame's detections as the stage takes them: BBOX_DTYPE [1, max_det], the first len(boxes) slots filled."""
    from irmv_detection_b200 import BBOX_DTYPE
    b = np.zeros((1, max_det), BBOX_DTYPE)
    b["xyxy"][0, :len(boxes)] = boxes
    b["score"][0, :len(boxes)] = scores
    b["class_id"][0, :len(boxes)] = classes
    return b


def blob_scene(seed: int, h: int = 1024, w: int = 1280, n_blobs: int = 260):
    """Speckle (sparse bright pixels and tiny components), filled rotated rectangles and rings (components inside a
    ring are not external): with permissive light filters most contours with >= 5 vertices become lights, so contour
    order, the vertex count and the external-only rule all decide the answer."""
    import cv2
    rng = np.random.default_rng(seed)
    img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    img[rng.random((h, w)) < 0.97] //= 3
    for _ in range(n_blobs):
        c = (float(rng.uniform(0, w)), float(rng.uniform(0, h)))
        size = (float(rng.uniform(2, 14)), float(rng.uniform(4, 60)))
        box = cv2.boxPoints((c, size, float(rng.uniform(-60, 60))))
        v = int(rng.integers(150, 256))
        if rng.random() < 0.3:
            cv2.ellipse(img, (int(c[0]), int(c[1])), (int(size[1]), int(size[1] * 0.6) + 2), 0, 0, 360, (v, v, v), 2)
        else:
            cv2.fillConvexPoly(img, np.round(box).astype(np.int32), (v, v, v))
    return img


def synth_armor_scene(n_armors: int = 6, seed: int = 0, w: int = 1280, h: int = 1024, noise: bool = True):
    """A dark arena frame (rotated view) with bright light-bar pairs and the boxes a detector would put
    around them (generator: irmv_detection_b200/synth.py armor_scene)."""
    from irmv_detection_b200 import synth
    return synth.armor_scene(n_armors, seed, w, h, noise)
