"""Raw-domain colour stage of Bayer sources (YoloEngine.set_raw_lut, irmv_engine_set_raw_lut), on the host.

apply_raw_lut is the definition the engine's kernels are checked against: the engine with table L on
frames F returns, bit for bit, what it returns without a table on apply_raw_lut(F, L, pattern).
make_raw_lut builds such a table from the black level, white-balance gains and gamma a caller would set
on the camera's ISP.

decode_raw is the same definition for 10- and 12-bit sources (raw_format RAW_10, RAW_12, RAW_12_PACKED): a b-bit
engine with table T on frames F returns, bit for bit, what an otherwise identical 8-bit engine without a table
returns on decode_raw(F, raw_format, T, pattern).

apply_color_matrix is the definition of the colour-correction stage that follows the demosaic (set_color_matrix):
a 3x3 integer matrix and an output tone table; color_matrix_q10 builds the matrix from a colour-correction matrix and
a saturation gain.

awb_statistics, awb_gains and awb_matrix are the definition of automatic white balance (set_auto_white_balance):
per frame, grey-world gains from the unclipped, not-too-dark 2x2 quads of the 8-bit mosaic, applied as a diagonal
matrix composed with the colour-correction stage's matrix.
"""
from __future__ import annotations

from typing import Optional, Sequence

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


RAW_BITS = {L.RAW_8: 8, L.RAW_10: 10, L.RAW_12: 12, L.RAW_12_PACKED: 12}


def apply_raw_lut(raw: np.ndarray, lut: np.ndarray, pattern: int) -> np.ndarray:
    """raw [..., H, W] Bayer mosaic(s) as the camera wrote them (before rot180), lut u8 [3, 2^b] (b = 8, 10, 12):
    sample s at sensor position (y, x) becomes lut[colour of (y, x)][s & (2^b - 1)].  With a (3, 256) table raw is
    taken as u8; wider tables take unsigned integer samples (u16).  Returns a new u8 array."""
    lut = np.asarray(lut, np.uint8)
    if lut.shape == (3, 256):
        raw = np.asarray(raw, np.uint8)
    elif lut.shape in ((3, 1 << 10), (3, 1 << 12)):
        raw = np.asarray(raw)
        if raw.dtype.kind != "u":
            raise ValueError("samples for a 10/12-bit table must be unsigned integers")
        raw = raw & np.asarray(lut.shape[1] - 1, raw.dtype)
    else:
        raise ValueError("lut must be (3, 256), (3, 1024) or (3, 4096) uint8")
    c = site_colours(raw.shape[-2], raw.shape[-1], pattern)
    return lut[c, raw]


def unpack_raw12_packed(packed: np.ndarray) -> np.ndarray:
    """u8 [..., H, 3W/2] 12-bit packed rows -> u16 [..., H, W].  Two horizontally adjacent samples p0, p1 in three
    bytes (GigE Vision BayerXX12Packed): B0 = p0[11:4], B1 = p1[3:0] << 4 | p0[3:0], B2 = p1[11:4]."""
    packed = np.asarray(packed, np.uint8)
    if packed.shape[-1] % 3:
        raise ValueError("a 12-bit packed row holds a multiple of 3 bytes")
    b = packed.reshape(packed.shape[:-1] + (-1, 3)).astype(np.uint16)
    p0 = b[..., 0] << 4 | (b[..., 1] & 15)
    p1 = b[..., 2] << 4 | b[..., 1] >> 4
    return np.stack([p0, p1], -1).reshape(packed.shape[:-1] + (-1,))


def pack_raw12_packed(raw: np.ndarray) -> np.ndarray:
    """u16 [..., H, W] (W even; the low 12 bits of each sample) -> u8 [..., H, 3W/2], the inverse of
    unpack_raw12_packed."""
    raw = np.asarray(raw)
    if raw.shape[-1] % 2:
        raise ValueError("12-bit packed rows need an even width")
    s = (raw.astype(np.uint16) & 0xFFF).reshape(raw.shape[:-1] + (-1, 2))
    p0, p1 = s[..., 0], s[..., 1]
    out = np.stack([p0 >> 4, (p1 & 15) << 4 | (p0 & 15), p1 >> 4], -1).astype(np.uint8)
    return out.reshape(raw.shape[:-1] + (-1,))


def default_raw_lut(bits: int) -> np.ndarray:
    """u8 [3, 2^bits]: the table a b-bit engine runs with until set_raw_lut, s -> s >> (bits - 8)."""
    return np.tile((np.arange(1 << bits) >> (bits - 8)).astype(np.uint8), (3, 1))


def decode_raw(frames: np.ndarray, raw_format: int, lut: Optional[np.ndarray], pattern: int) -> np.ndarray:
    """Frames as a raw_format engine takes them (u16 [..., H, W] for RAW_10 / RAW_12, u8 [..., H, 3W/2] for
    RAW_12_PACKED) -> the u8 [..., H, W] mosaics an 8-bit engine without a table must see: unpack, mask each sample
    to b bits, map it through lut[colour of its sensor site] (lut None: default_raw_lut(b))."""
    bits = RAW_BITS[raw_format]
    if bits == 8:
        raise ValueError("decode_raw takes 10/12-bit formats; 8-bit frames go through apply_raw_lut")
    raw = unpack_raw12_packed(frames) if raw_format == L.RAW_12_PACKED else np.asarray(frames, np.uint16)
    lut = default_raw_lut(bits) if lut is None else np.asarray(lut, np.uint8)
    if lut.shape != (3, 1 << bits):
        raise ValueError(f"a {bits}-bit format takes a (3, {1 << bits}) table")
    return apply_raw_lut(raw, lut, pattern)


def make_raw_lut(black_level: int = 0, gains: Sequence[float] = (1.0, 1.0, 1.0), gamma: float = 1.0,
                 bits: int = 8) -> np.ndarray:
    """u8 [3, 2^bits] table of the usual ISP chain per colour site, from bits-bit samples to 8-bit values: subtract
    the black level (in units of that bit depth), rescale to the full range 2^bits - 1 - black, apply the channel's
    white-balance gain, clip, apply the tone curve x ** gamma, round half up.

    make_raw_lut(0, (1, 1, 1), gamma) is also the output tone table of the colour-correction stage
    (apply_color_matrix, set_color_matrix): an ISP applies black level and gains before the matrix and gamma after
    it, so the raw table then keeps gamma 1."""
    top = (1 << bits) - 1
    v = np.arange(top + 1, dtype=np.float64)
    x = np.clip(v - black_level, 0.0, None) / (float(top) - black_level)
    out = np.empty((3, top + 1), np.uint8)
    for c in range(3):
        y = np.clip(x * float(gains[c]), 0.0, 1.0) ** float(gamma)
        out[c] = np.floor(y * 255.0 + 0.5).astype(np.uint8)
    return out


# BT.601 luma weights of R, G, B: the grey axis a saturation gain keeps fixed
LUMA_BT601 = (0.299, 0.587, 0.114)


def apply_color_matrix(rgb: np.ndarray, m: np.ndarray, tone: Optional[np.ndarray] = None) -> np.ndarray:
    """Colour-correction stage of Bayer sources (YoloEngine.set_color_matrix, irmv_engine_set_color_matrix).
    rgb u8 [..., 3] is the demosaiced frame (oracle.preprocess_ref.demosaic_bilinear, after the raw table or the
    10/12-bit decode, before rot180 and resize); m is int16 [3, 3], row-major, in units of 1/1024; tone is u8
    [3, 256] or None (identity).  For every pixel and output channel c:
        v_c = sum_k m[c][k] * in_k                     (int32)
        o_c = clamp(floor((v_c + 512) / 1024), 0, 255)
        out_c = tone[c][o_c]
    The engine with matrix M and tone T on Bayer frames F returns, bit for bit, what a PASSTHROUGH engine returns
    on the packed frames apply_color_matrix(demosaic_bilinear(F), M, T).  Returns a new u8 array."""
    rgb = np.asarray(rgb)
    if rgb.dtype != np.uint8 or rgb.ndim < 1 or rgb.shape[-1] != 3:
        raise ValueError("rgb must be uint8 [..., 3]")
    m = _check_matrix(m)
    tone = _check_tone(tone)
    v = rgb.astype(np.int32) @ m.astype(np.int32).T
    o = np.clip((v + 512) >> 10, 0, 255)
    if tone is None:
        return o.astype(np.uint8)
    return tone[np.arange(3), o]


def color_matrix_q10(ccm: Optional[np.ndarray] = None, saturation: float = 1.0) -> np.ndarray:
    """int16 [3, 3] matrix of the colour-correction stage: rint(1024 * S @ ccm), clipped to the int16 range, with
    ccm a float [3, 3] colour-correction matrix (None: identity) and S = s*I + (1 - s) * 1 * luma^T the saturation
    gain s about the BT.601 grey axis (s = 0 maps every pixel to its luma, s > 1 pushes colours apart)."""
    c = np.eye(3) if ccm is None else np.asarray(ccm, np.float64)
    if c.shape != (3, 3):
        raise ValueError("ccm must be 3 x 3")
    s = float(saturation)
    S = s * np.eye(3) + (1.0 - s) * np.outer(np.ones(3), LUMA_BT601)
    return np.clip(np.rint(1024.0 * (S @ c)), -32768, 32767).astype(np.int16)


def _check_matrix(m) -> np.ndarray:
    m = np.asarray(m)
    if m.shape != (3, 3) or m.dtype != np.int16:
        raise ValueError("the colour matrix must be a (3, 3) int16 array")
    return m


def _check_tone(tone) -> Optional[np.ndarray]:
    if tone is None:
        return None
    tone = np.asarray(tone)
    if tone.shape != (3, 256) or tone.dtype != np.uint8:
        raise ValueError("the tone table must be a (3, 256) uint8 array or None")
    return tone


# Automatic white balance (YoloEngine.set_auto_white_balance, irmv_engine_set_auto_white_balance, irmv_awb_params)
AWB_DEFAULTS = {"dark_level": 8, "clip_level": 250, "min_quads": 4096, "gain_max_q10": 4096}


def awb_params(params: Optional[dict] = None) -> dict:
    """AWB_DEFAULTS updated with `params`, checked as the engine checks them: 0 <= dark_level <= clip_level <= 255,
    min_quads >= 1, 1024 <= gain_max_q10 <= 32767."""
    p = dict(AWB_DEFAULTS)
    if params:
        unknown = set(params) - set(p)
        if unknown:
            raise ValueError(f"unknown auto white balance parameters: {sorted(unknown)}")
        p.update({k: int(v) for k, v in params.items()})
    if not 0 <= p["dark_level"] <= p["clip_level"] <= 255:
        raise ValueError("auto white balance needs 0 <= dark_level <= clip_level <= 255")
    if p["min_quads"] < 1:
        raise ValueError("auto white balance needs min_quads >= 1")
    if not 1024 <= p["gain_max_q10"] <= 32767:
        raise ValueError("auto white balance needs 1024 <= gain_max_q10 <= 32767")
    return p


def awb_statistics(mosaic8: np.ndarray, pattern: int, params: Optional[dict] = None) -> dict:
    """Statistics of one frame.  mosaic8 is the u8 [H, W] mosaic the demosaic reads (RAW_8: after the raw table when
    one is set, apply_raw_lut; 10/12-bit: decode_raw), in sensor coordinates (before rot180).  Quad (i, j) covers rows
    2i, 2i + 1 and columns 2j, 2j + 1 (i < H // 2, j < W // 2: an odd last row or column is not used); its samples are
    R, Gr, Gb, B under `pattern`.  A quad is clipped if a sample is > clip_level, else dark if a sample is
    < dark_level, else counted.  Returns {"sum": (SR, SG, SB), "counted", "dark", "clipped"}: SR = sum of R,
    SG = sum of Gr + Gb, SB = sum of B over the counted quads (Python ints)."""
    p = awb_params(params)
    m = np.asarray(mosaic8)
    if m.dtype != np.uint8 or m.ndim != 2:
        raise ValueError("mosaic8 must be a uint8 [H, W] mosaic")
    h2, w2 = m.shape[0] // 2, m.shape[1] // 2
    q = m[:2 * h2, :2 * w2].reshape(h2, 2, w2, 2).astype(np.int64)
    s = [[q[:, py, :, px] for px in range(2)] for py in range(2)]
    ry, rx = RED_SITE[pattern]
    r, b = s[ry][rx], s[1 - ry][1 - rx]
    g = s[ry][1 - rx] + s[1 - ry][rx]
    hi = np.maximum(np.maximum(s[0][0], s[0][1]), np.maximum(s[1][0], s[1][1]))
    lo = np.minimum(np.minimum(s[0][0], s[0][1]), np.minimum(s[1][0], s[1][1]))
    clipped = hi > p["clip_level"]
    dark = ~clipped & (lo < p["dark_level"])
    counted = ~clipped & ~dark
    return {"sum": (int(r[counted].sum()), int(g[counted].sum()), int(b[counted].sum())),
            "counted": int(counted.sum()), "dark": int(dark.sum()), "clipped": int(clipped.sum())}


def awb_gains(stats: dict, params: Optional[dict] = None) -> tuple:
    """Q10 gains (gR, gG, gB) and validity of a frame from its statistics.  With the comparable channel sums
    A = (2 SR, SG, 2 SB) and Amax = max(A): g_c = min((1024 Amax + A_c // 2) // A_c, gain_max_q10), so the brightest
    channel gets exactly 1024 and no gain is below 1024.  A frame with fewer than min_quads counted quads or an
    empty channel is invalid: gains (1024, 1024, 1024).  Returns ((gR, gG, gB), valid)."""
    p = awb_params(params)
    sr, sg, sb = (int(v) for v in stats["sum"])
    a = (2 * sr, sg, 2 * sb)
    if stats["counted"] < p["min_quads"] or min(a) == 0:
        return (1024, 1024, 1024), False
    amax = max(a)
    return tuple(min((1024 * amax + c // 2) // c, p["gain_max_q10"]) for c in a), True


def awb_matrix(gains: Sequence[int], m: Optional[np.ndarray] = None) -> np.ndarray:
    """int16 [3, 3] matrix the colour-correction stage applies to a frame with AWB gains g under the user's matrix m
    (None: 1024 * I): M_F[r][k] = clamp_int16((m[r][k] * g_k + 512) >> 10) (arithmetic shift).  With AWB off,
    set_color_matrix(awb_matrix(g, m), tone) reproduces exactly what AWB with gains g produced: that locks the white
    balance."""
    mm = (1024 * np.eye(3)).astype(np.int16) if m is None else _check_matrix(m)
    g = np.asarray(gains, np.int64)
    if g.shape != (3,):
        raise ValueError("gains must be three Q10 integers")
    v = (mm.astype(np.int64) * g[None, :] + 512) >> 10
    return np.clip(v, -32768, 32767).astype(np.int16)


def awb_record(mosaic8: np.ndarray, pattern: int, params: Optional[dict] = None) -> dict:
    """What the engine reports for one frame (irmv_awb, YoloEngine.fetch_white_balance): the statistics of
    awb_statistics, the gains of awb_gains and their validity."""
    st = awb_statistics(mosaic8, pattern, params)
    g, valid = awb_gains(st, params)
    return {**st, "valid": int(valid), "gain_q10": g}
