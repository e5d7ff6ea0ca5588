"""TEST INFRASTRUCTURE ONLY -- read the fused stem's network input back through conv0.

The fused stem (csrc/preprocess.cu stem_kernel, csrc/stem_bayer.cu stem_bayer2x_kernel) never stores the 640 x 640
network input: it only exists in shared memory, where conv0 (3x3, stride 2, pad 1, 3 -> 16, SiLU) consumes it.
Probe weights make conv0 copy it out instead.  In a probe file, output channel 3i + c has weight 1 at (input
channel c, tap TAP_FILES[f][i]) and bias 0, so m0[y, x, 3i + c] = SiLU(xp[c, 2y + ky, 2x + kx]) with tap
t = 3 ky + kx and xp the input with one zero row / column of conv padding on top and on the left.  The two files
of TAP_FILES cover all nine taps: every input pixel is read through every tap that reaches it (odd rows and
columns twice), and the top / left padding through ky = 0 and kx = 0.

With the 8-bit intermediate every input value is k / 255 in FP16 and SiLU is increasing on [0, 1] with slope
>= 0.5, so each output decodes to exactly one 8-bit code (neighbouring codes are >= 1.9e-3 apart after SiLU;
tanh.approx and the FP16 store move an output by < 4e-4).  Without it, the outputs are compared with
SiLU(x_ref) to FLOAT_TOL: tanh.approx (about 1.2e-4) plus half an FP16 ulp below 1 (2.4e-4).

Only tests/ may import this module.
"""
from __future__ import annotations

from typing import Optional, Sequence, Tuple

import numpy as np

TAP_FILES: Tuple[Tuple[int, ...], ...] = ((0, 1, 2, 3, 4), (5, 6, 7, 8))
FLOAT_TOL = 4e-4
NET = 640


def probe_conv0(taps: Sequence[int]) -> Tuple[np.ndarray, np.ndarray]:
    """conv0 weights [16, 3, 3, 3] (out, in, ky, kx) and bias [16] of one probe file."""
    w = np.zeros((16, 3, 3, 3), np.float32)
    for i, t in enumerate(taps):
        for c in range(3):
            w[3 * i + c, c, t // 3, t % 3] = 1.0
    return w, np.zeros(16, np.float32)


def tap_views(xp: np.ndarray) -> np.ndarray:
    """xp [N, 3, 641, 641] (input with its top / left padding) -> [N, 9, 3, 320, 320]: what conv0 reads through
    each tap t = 3 ky + kx at output pixel (y, x), namely xp[:, c, 2y + ky, 2x + kx]."""
    return np.stack([xp[:, :, t // 3:t // 3 + NET:2, t % 3:t % 3 + NET:2] for t in range(9)], 1)


def pad_input(x: np.ndarray, value=0) -> np.ndarray:
    """x [N, 3, 640, 640] -> [N, 3, 641, 641] with `value` in the top row and left column."""
    return np.pad(x, ((0, 0), (0, 0), (1, 0), (1, 0)), constant_values=value)


def engine_views(m0s: Sequence[np.ndarray]) -> np.ndarray:
    """The m0 tensors [N, 320, 320, 16] of the engines running the probe files of TAP_FILES, in that order ->
    [N, 9, 3, 320, 320] float64 in the layout of tap_views."""
    out = np.empty((m0s[0].shape[0], 9, 3, NET // 2, NET // 2))
    for m0, taps in zip(m0s, TAP_FILES):
        for i, t in enumerate(taps):
            out[:, t] = m0[..., 3 * i:3 * i + 3].astype(np.float64).transpose(0, 3, 1, 2)
    return out


def silu(v):
    v = np.asarray(v, np.float64)
    return v / (1.0 + np.exp(-v))


_CODE_SILU = silu(np.float16(np.arange(256) / 255.0).astype(np.float64))
_CODE_MID = (_CODE_SILU[1:] + _CODE_SILU[:-1]) / 2


def decode_codes(v: np.ndarray) -> np.ndarray:
    """SiLU outputs of 8-bit input values -> the nearest code 0..255 (-1 for NaN or for values more than half a
    step outside the table)."""
    v = np.asarray(v, np.float64)
    k = np.searchsorted(_CODE_MID, v).astype(np.int64)
    step = _CODE_SILU[1] - _CODE_SILU[0]
    bad = np.isnan(v) | (v < _CODE_SILU[0] - step / 2) | (v > _CODE_SILU[-1] + step / 2)
    return np.where(bad, -1, k)


def _where(idx, shape) -> dict:
    f, t, c, y, x = np.unravel_index(idx, shape)
    ky, kx = int(t) // 3, int(t) % 3
    # input coordinates of the read; -1 is the conv padding
    return {"frame": int(f), "channel": int(c), "y": 2 * int(y) + ky - 1, "x": 2 * int(x) + kx - 1, "tap": (ky, kx)}


def compare_codes(got: np.ndarray, codes: np.ndarray) -> Optional[str]:
    """got: engine_views() of a run with the 8-bit intermediate; codes: the oracle's 8-bit input [N, 3, 640, 640].
    None when every read decodes to the oracle's code (padding reads to 0), else the first mismatch."""
    want = tap_views(pad_input(codes.astype(np.int64)))
    dec = decode_codes(got)
    if np.array_equal(dec, want):
        return None
    i = int(np.flatnonzero(dec != want)[0])
    w = _where(i, want.shape)
    return (f"first mismatch at (frame, channel, y, x) = ({w['frame']}, {w['channel']}, {w['y']}, {w['x']}) through "
            f"tap {w['tap']}: code {int(dec.flat[i])}, oracle {int(want.flat[i])}; "
            f"{int((dec != want).sum())} reads differ")


def float_deviation(got: np.ndarray, x: np.ndarray) -> Tuple[float, dict]:
    """got: engine_views() of a run without the 8-bit intermediate; x: the oracle's FP16 input [N, 3, 640, 640].
    Largest |got - SiLU(x)| over all reads (NaN counts as infinite) and where it is."""
    d = np.abs(got - silu(tap_views(pad_input(x.astype(np.float64)))))
    d = np.where(np.isnan(d), np.inf, d)
    i = int(np.argmax(d))
    return float(d.flat[i]), _where(i, d.shape)
