"""Raw-domain colour stage of Bayer sources (YoloEngine.set_raw_lut, irmv_engine_set_raw_lut), on the host.

apply_raw_lut is the definition the engine's kernels are checked against: the engine with table L on
frames F returns, bit for bit, what it returns without a table on apply_raw_lut(F, L, pattern).
make_raw_lut builds such a table from the black level, white-balance gains and gamma a caller would set
on the camera's ISP.
"""
from __future__ import annotations

from typing import Sequence

import numpy as np

from . import _lib as L

# (red_y, red_x): the red site of each Bayer pattern, as bayer_rgb (csrc/preprocess.cu) and gray_at (csrc/armors.cu)
RED_SITE = {L.CH_BAYER_RGGB: (0, 0), L.CH_BAYER_BGGR: (1, 1), L.CH_BAYER_GRBG: (0, 1), L.CH_BAYER_GBRG: (1, 0)}


def site_colours(h: int, w: int, pattern: int) -> np.ndarray:
    """u8 [h, w]: colour of every sensor position (0 red, 1 green, 2 blue) under `pattern`."""
    ry, rx = RED_SITE[pattern]
    py = (np.arange(h) & 1)[:, None]
    px = (np.arange(w) & 1)[None, :]
    red = (py == ry) & (px == rx)
    blue = (py != ry) & (px != rx)
    return np.where(red, 0, np.where(blue, 2, 1)).astype(np.uint8)


def apply_raw_lut(raw: np.ndarray, lut: np.ndarray, pattern: int) -> np.ndarray:
    """raw u8 [..., H, W] Bayer mosaic(s) as the camera wrote them (before rot180), lut u8 [3, 256]:
    sample s at sensor position (y, x) becomes lut[colour of (y, x)][s].  Returns a new array."""
    raw = np.asarray(raw, np.uint8)
    lut = np.asarray(lut, np.uint8)
    if lut.shape != (3, 256):
        raise ValueError("lut must be (3, 256) uint8")
    c = site_colours(raw.shape[-2], raw.shape[-1], pattern)
    return lut[c, raw]


def make_raw_lut(black_level: int = 0, gains: Sequence[float] = (1.0, 1.0, 1.0), gamma: float = 1.0) -> np.ndarray:
    """u8 [3, 256] table of the usual ISP chain per colour site: subtract the black level, rescale to the
    full range, apply the channel's white-balance gain, clip, apply the tone curve x ** gamma, round half up."""
    v = np.arange(256, dtype=np.float64)
    x = np.clip(v - black_level, 0.0, None) / (255.0 - black_level)
    out = np.empty((3, 256), np.uint8)
    for c in range(3):
        y = np.clip(x * float(gains[c]), 0.0, 1.0) ** float(gamma)
        out[c] = np.floor(y * 255.0 + 0.5).astype(np.uint8)
    return out
