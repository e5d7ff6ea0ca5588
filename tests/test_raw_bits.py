"""10- and 12-bit raw sources on the host: the 12-bit packed layout, the default and ISP tables of a b-bit engine,
masking of the container bits, decode_raw (the definition the engine is checked against), the media-type mapping
and the C layout of irmv_engine_config.raw_format."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from irmv_detection_b200 import _lib as L, raw_lut as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PATTERNS = [L.CH_BAYER_RGGB, L.CH_BAYER_BGGR, L.CH_BAYER_GRBG, L.CH_BAYER_GBRG]


def test_packed_known_answer_and_round_trip():
    raw = np.array([[0xABC, 0xDEF]], np.uint16)
    packed = R.pack_raw12_packed(raw)
    assert packed.tolist() == [[0xAB, 0xFC, 0xDE]]
    assert np.array_equal(R.unpack_raw12_packed(packed), raw)
    rng = np.random.default_rng(0)
    frames = rng.integers(0, 4096, (3, 5, 14), dtype=np.uint16)
    p = R.pack_raw12_packed(frames)
    assert p.shape == (3, 5, 21) and p.dtype == np.uint8
    assert np.array_equal(R.unpack_raw12_packed(p), frames)
    b = rng.integers(0, 256, (4, 9), dtype=np.uint8)
    assert np.array_equal(R.pack_raw12_packed(R.unpack_raw12_packed(b)), b)
    with pytest.raises(ValueError):
        R.pack_raw12_packed(np.zeros((2, 3), np.uint16))


@pytest.mark.parametrize("bits", [8, 10, 12])
def test_default_table_is_the_shift(bits):
    t = R.default_raw_lut(bits)
    assert t.shape == (3, 1 << bits) and t.dtype == np.uint8
    for c in range(3):
        assert np.array_equal(t[c], (np.arange(1 << bits) >> (bits - 8)).astype(np.uint8))


def test_make_raw_lut_bits():
    assert np.array_equal(R.make_raw_lut(bits=8), R.make_raw_lut())
    assert np.array_equal(R.make_raw_lut(8, (1.9, 1.0, 1.6), 1 / 2.2, bits=8), R.make_raw_lut(8, (1.9, 1.0, 1.6), 1 / 2.2))
    lut = R.make_raw_lut(128, (1.9, 1.0, 1.6), 1 / 2.2, bits=12)
    assert lut.shape == (3, 4096) and lut.dtype == np.uint8
    assert (np.diff(lut.astype(int), axis=1) >= 0).all()
    assert (lut[:, :129] == 0).all() and (lut[:, 4095] == 255).all()
    assert (lut[0] >= lut[2]).all() and (lut[2] >= lut[1]).all()
    assert lut[0, 2300] == 255 and lut[1, 2300] < 255              # red saturates first (gain 1.9), then clips
    ident = R.make_raw_lut(bits=12)
    assert ident[1, 0] == 0 and ident[1, 4095] == 255 and ident[1, 2048] == 128
    # the tone curve lifts the bottom codes of a 12-bit sample apart where an 8-bit sample has one code
    g = R.make_raw_lut(0, (1.0, 1.0, 1.0), 1 / 2.2, bits=12)[1]
    assert len(set(g[:16].tolist())) > 8


@pytest.mark.parametrize("bits", [10, 12])
def test_high_container_bits_are_masked(bits):
    rng = np.random.default_rng(bits)
    lut = rng.integers(0, 256, (3, 1 << bits), dtype=np.uint8)
    raw = rng.integers(0, 1 << bits, (2, 6, 8), dtype=np.uint16)
    dirty = raw | (rng.integers(0, 1 << (16 - bits), raw.shape, dtype=np.uint16) << bits).astype(np.uint16)
    assert not np.array_equal(dirty, raw)
    fmt = L.RAW_10 if bits == 10 else L.RAW_12
    for pattern in PATTERNS:
        assert np.array_equal(R.apply_raw_lut(dirty, lut, pattern), R.apply_raw_lut(raw, lut, pattern))
        assert np.array_equal(R.decode_raw(dirty, fmt, lut, pattern), R.decode_raw(raw, fmt, lut, pattern))
    sites = R.site_colours(6, 8, L.CH_BAYER_GRBG)
    assert np.array_equal(R.apply_raw_lut(raw, lut, L.CH_BAYER_GRBG), lut[sites, raw])


@pytest.mark.parametrize("fmt", [L.RAW_10, L.RAW_12, L.RAW_12_PACKED])
def test_decode_raw_default_table_recovers_8bit(fmt):
    rng = np.random.default_rng(fmt)
    v8 = rng.integers(0, 256, (2, 6, 10), dtype=np.uint8)
    b = R.RAW_BITS[fmt]
    raw = (v8.astype(np.uint16) << (b - 8)) | rng.integers(0, 1 << (b - 8), v8.shape, dtype=np.uint16)
    frames = R.pack_raw12_packed(raw) if fmt == L.RAW_12_PACKED else raw
    for pattern in PATTERNS:
        assert np.array_equal(R.decode_raw(frames, fmt, None, pattern), v8)
    # and with a table: each sample goes through the table of its site
    lut = rng.integers(0, 256, (3, 1 << b), dtype=np.uint8)
    sites = R.site_colours(6, 10, L.CH_BAYER_BGGR)
    assert np.array_equal(R.decode_raw(frames, fmt, lut, L.CH_BAYER_BGGR), lut[sites, raw])
    with pytest.raises(ValueError):
        R.decode_raw(frames, fmt, np.zeros((3, 256), np.uint8), L.CH_BAYER_BGGR)


def test_apply_raw_lut_rejects_bad_tables():
    with pytest.raises(ValueError):
        R.apply_raw_lut(np.zeros((4, 4), np.uint16), np.zeros((3, 2048), np.uint8), L.CH_BAYER_RGGB)
    with pytest.raises(ValueError):
        R.apply_raw_lut(np.zeros((4, 4), np.int16), np.zeros((3, 4096), np.uint8), L.CH_BAYER_RGGB)


MONO, COLOR, O8, O12, O16, O24 = 0x01000000, 0x02000000, 0x00080000, 0x000C0000, 0x00100000, 0x00180000
# vendor name -> (code from the header's MONO | occupancy | id formula, chan_order, raw_format)
INGESTED = {
    "BAYGR8": (MONO | O8 | 0x08, L.CH_BAYER_GRBG, L.RAW_8), "BAYRG8": (MONO | O8 | 0x09, L.CH_BAYER_RGGB, L.RAW_8),
    "BAYGB8": (MONO | O8 | 0x0A, L.CH_BAYER_GBRG, L.RAW_8), "BAYBG8": (MONO | O8 | 0x0B, L.CH_BAYER_BGGR, L.RAW_8),
    "RGB8": (COLOR | O24 | 0x14, L.CH_PASSTHROUGH, L.RAW_8), "BGR8": (COLOR | O24 | 0x15, L.CH_SWAP_RB, L.RAW_8),
    "BAYGR10": (MONO | O16 | 0x0C, L.CH_BAYER_GRBG, L.RAW_10), "BAYRG10": (MONO | O16 | 0x0D, L.CH_BAYER_RGGB, L.RAW_10),
    "BAYGB10": (MONO | O16 | 0x0E, L.CH_BAYER_GBRG, L.RAW_10), "BAYBG10": (MONO | O16 | 0x0F, L.CH_BAYER_BGGR, L.RAW_10),
    "BAYGR12": (MONO | O16 | 0x10, L.CH_BAYER_GRBG, L.RAW_12), "BAYRG12": (MONO | O16 | 0x11, L.CH_BAYER_RGGB, L.RAW_12),
    "BAYGB12": (MONO | O16 | 0x12, L.CH_BAYER_GBRG, L.RAW_12), "BAYBG12": (MONO | O16 | 0x13, L.CH_BAYER_BGGR, L.RAW_12),
    "BAYGR12_PACKED": (MONO | O12 | 0x2A, L.CH_BAYER_GRBG, L.RAW_12_PACKED),
    "BAYRG12_PACKED": (MONO | O12 | 0x2B, L.CH_BAYER_RGGB, L.RAW_12_PACKED),
    "BAYGB12_PACKED": (MONO | O12 | 0x2C, L.CH_BAYER_GBRG, L.RAW_12_PACKED),
    "BAYBG12_PACKED": (MONO | O12 | 0x2D, L.CH_BAYER_BGGR, L.RAW_12_PACKED),
}
NOT_INGESTED = {"MONO8": MONO | O8 | 0x01, "MONO12": MONO | O16 | 0x05, "BAYGR10_PACKED": MONO | O12 | 0x26,
                "BAYBG10_PACKED": MONO | O12 | 0x29, "BAYRG16": MONO | O16 | 0x2F, "YUV422_8": COLOR | O16 | 0x32,
                "BGR10": COLOR | 0x00300000 | 0x19, "zero": 0}


def test_source_format_from_media_type():
    f = L.lib().irmv_source_format_from_media_type
    old = L.lib().irmv_chan_order_from_media_type
    for name, (code, chan, fmt) in INGESTED.items():
        co, rf = C.c_int32(-7), C.c_int32(-7)
        assert f(code, C.byref(co), C.byref(rf)) == 0, name
        assert (co.value, rf.value) == (chan, fmt), name
        assert old(code) == (chan if fmt == L.RAW_8 else -1), name     # the 8-bit mapping is unchanged
    hdr = open(os.path.join(ROOT, "include", "irmv_cabi.h")).read()
    for name, (code, _, _) in INGESTED.items():
        assert f"#define IRMV_MV_MEDIA_TYPE_{name} 0x{code:08X}u" in hdr, name
    for name, code in NOT_INGESTED.items():
        co, rf = C.c_int32(-7), C.c_int32(-7)
        assert f(code, C.byref(co), C.byref(rf)) != 0, name
    assert f(INGESTED["BAYRG12"][0], None, None) != 0


def test_engine_config_layout_matches_the_header(tmp_path):
    exe = tmp_path / "cabi_config_probe"
    subprocess.run(["g++", "-std=c++17", "-O2", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "cpp", "cabi_config_probe.cpp"), "-o", str(exe)], check=True)
    size, reserved, raw_format = (int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True,
                                                                 check=True).stdout.split())
    assert C.sizeof(L.EngineConfig) == size == 96                    # unchanged by raw_format
    assert L.EngineConfig.reserved.offset == reserved == 64
    assert L.EngineConfig.raw_format.offset == raw_format == reserved + 7 * 4
    cfg = L.EngineConfig()
    assert L.lib().irmv_engine_config_default(C.byref(cfg)) == 0 and cfg.raw_format == L.RAW_8
