"""Definition of automatic white balance (raw_lut.awb_statistics / awb_gains / awb_matrix): known answers on hand-built
mosaics for every pattern, the classification boundaries, the fallback, the gain rounding and clamp, the composition
with the user's matrix, odd frame sizes and parameter validation.  No GPU."""
import ctypes as C

import numpy as np
import pytest

from irmv_detection_b200 import _lib as L, raw_lut as R

PATTERNS = [L.CH_BAYER_RGGB, L.CH_BAYER_BGGR, L.CH_BAYER_GRBG, L.CH_BAYER_GBRG]
ANY = {"min_quads": 1}


def _mosaic(h, w, pattern, r, gr, gb, b):
    """Constant value per site: r on red, gr on the green of the red row, gb on the green of the blue row, b on blue."""
    ry, rx = R.RED_SITE[pattern]
    m = np.empty((h, w), np.uint8)
    m[ry::2, rx::2] = r
    m[ry::2, 1 - rx::2] = gr
    m[1 - ry::2, rx::2] = gb
    m[1 - ry::2, 1 - rx::2] = b
    return m


@pytest.mark.parametrize("pattern", PATTERNS)
def test_constant_sites_give_known_sums(pattern):
    h, w = 12, 20
    st = R.awb_statistics(_mosaic(h, w, pattern, 100, 60, 70, 40), pattern, ANY)
    q = (h // 2) * (w // 2)
    assert st == {"sum": (100 * q, 130 * q, 40 * q), "counted": q, "dark": 0, "clipped": 0}
    g, valid = R.awb_gains(st, ANY)
    # A = (200 q, 130 q, 80 q): red is the brightest channel
    assert valid and g == (1024, (1024 * 200 + 65) // 130, (1024 * 200 + 40) // 80)


@pytest.mark.parametrize("pattern", PATTERNS)
def test_pattern_decides_which_site_is_red(pattern):
    """The same mosaic read under another pattern puts other sites on R and B."""
    m = _mosaic(4, 4, L.CH_BAYER_RGGB, 10, 20, 30, 40)        # (0,0)=10 (0,1)=20 (1,0)=30 (1,1)=40
    ry, rx = R.RED_SITE[pattern]
    site = {(0, 0): 10, (0, 1): 20, (1, 0): 30, (1, 1): 40}
    st = R.awb_statistics(m, pattern, ANY)
    r, b = site[(ry, rx)], site[(1 - ry, 1 - rx)]
    assert st["sum"] == (4 * r, 4 * (100 - r - b), 4 * b)


def test_dark_and_clip_boundaries():
    p = {"dark_level": 8, "clip_level": 250, "min_quads": 1}
    rg = L.CH_BAYER_RGGB
    at = _mosaic(2, 8, rg, 8, 250, 100, 100)                   # exactly at both levels: counted
    assert R.awb_statistics(at, rg, p)["counted"] == 4
    below = _mosaic(2, 8, rg, 7, 100, 100, 100)
    assert R.awb_statistics(below, rg, p) == {"sum": (0, 0, 0), "counted": 0, "dark": 4, "clipped": 0}
    above = _mosaic(2, 8, rg, 100, 100, 100, 251)
    assert R.awb_statistics(above, rg, p) == {"sum": (0, 0, 0), "counted": 0, "dark": 0, "clipped": 4}
    both = _mosaic(2, 8, rg, 0, 255, 100, 100)                 # clipped wins over dark
    assert R.awb_statistics(both, rg, p)["clipped"] == 4
    one = np.full((2, 8), 100, np.uint8)
    one[1, 7] = 251                                            # a single sample clips its quad only
    st = R.awb_statistics(one, rg, p)
    assert (st["counted"], st["clipped"]) == (3, 1) and st["sum"] == (300, 600, 300)


@pytest.mark.parametrize("value", [255, 0])
def test_all_clipped_or_all_dark_frames_fall_back(value):
    st = R.awb_statistics(np.full((64, 64), value, np.uint8), L.CH_BAYER_BGGR)
    assert st["counted"] == 0 and st["clipped" if value else "dark"] == 32 * 32
    assert R.awb_gains(st) == ((1024, 1024, 1024), False)
    rec = R.awb_record(np.full((64, 64), value, np.uint8), L.CH_BAYER_BGGR)
    assert rec["valid"] == 0 and rec["gain_q10"] == (1024, 1024, 1024)


def test_min_quads_boundary_and_empty_channel():
    st = {"sum": (100, 300, 200), "counted": 4096, "dark": 0, "clipped": 0}
    assert R.awb_gains(st)[1]
    assert R.awb_gains({**st, "counted": 4095}) == ((1024, 1024, 1024), False)
    assert R.awb_gains({**st, "counted": 4096}, {"min_quads": 4097}) == ((1024, 1024, 1024), False)
    assert R.awb_gains({**st, "sum": (0, 300, 200)}) == ((1024, 1024, 1024), False)


def test_gain_rounding():
    # A = (2 SR, SG, 2 SB) = (2048, 2049, 2048): 1024 * 2049 / 2048 = 1024.5 rounds up
    assert R.awb_gains({"sum": (1024, 2049, 1024), "counted": 1}, ANY) == ((1025, 1024, 1025), True)
    # A = (6, 7, 4): 1194.67 -> 1195, 1792 exactly
    assert R.awb_gains({"sum": (3, 7, 2), "counted": 1}, ANY) == ((1195, 1024, 1792), True)
    # every gain is the exact quotient rounded half up
    from fractions import Fraction
    rng = np.random.default_rng(1)
    for sr, sg, sb in rng.integers(1, 1 << 40, (200, 3)):
        a = (2 * int(sr), int(sg), 2 * int(sb))
        g, ok = R.awb_gains({"sum": (int(sr), int(sg), int(sb)), "counted": 1}, {**ANY, "gain_max_q10": 32767})
        want = tuple(min(int(Fraction(1024 * max(a), c) + Fraction(1, 2)), 32767) for c in a)
        assert ok and g == want and min(g) >= 1024 and 1024 in g


def test_gain_max_clamp():
    st = {"sum": (1, 1000, 500), "counted": 1}
    assert R.awb_gains(st, ANY)[0] == (4096, 1024, 1024)
    assert R.awb_gains(st, {**ANY, "gain_max_q10": 32767})[0] == (min((1024 * 1000 + 1) // 2, 32767), 1024, 1024)
    assert R.awb_gains(st, {**ANY, "gain_max_q10": 1024})[0] == (1024, 1024, 1024)


def test_matrix_composition_and_int16_clamp():
    assert np.array_equal(R.awb_matrix((1024, 1024, 1024)), (1024 * np.eye(3)).astype(np.int16))
    assert np.array_equal(R.awb_matrix((2048, 1024, 1536)), np.diag([2048, 1024, 1536]).astype(np.int16))
    m = np.array([[32767, -1, -300], [-20000, 1024, 511], [-1, 0, -32768]], np.int16)
    g = (4096, 1025, 1536)
    got = R.awb_matrix(g, m)
    want = np.array([[max(-32768, min(32767, (int(m[r, k]) * g[k] + 512) >> 10)) for k in range(3)] for r in range(3)])
    assert got.dtype == np.int16 and np.array_equal(got, want)
    assert got[0, 0] == 32767 and got[1, 0] == -32768 and got[2, 2] == -32768       # both ends of the clamp
    assert got[0, 1] == -1 and got[0, 2] == -450 and got[1, 2] == 767              # arithmetic shift floors
    with pytest.raises(ValueError):
        R.awb_matrix(g, m.astype(np.int32))
    with pytest.raises(ValueError):
        R.awb_matrix((1024, 1024))


@pytest.mark.parametrize("h,w", [(5, 7), (4, 7), (5, 8), (1, 8), (6, 1)])
def test_odd_sizes_drop_the_last_row_or_column(h, w):
    m = np.full((h, w), 100, np.uint8)
    m[-1, :] = 255 if h % 2 else 100
    m[:, -1] = 255 if w % 2 else m[:, -1]
    st = R.awb_statistics(m, L.CH_BAYER_GRBG, ANY)
    q = (h // 2) * (w // 2)
    assert st["counted"] == q and st["clipped"] == 0 and st["sum"] == (100 * q, 200 * q, 100 * q)


def test_parameter_validation():
    assert R.awb_params() == R.AWB_DEFAULTS
    assert R.awb_params({"dark_level": 0, "clip_level": 0})["clip_level"] == 0
    assert R.awb_params({"clip_level": 255, "gain_max_q10": 32767, "min_quads": 1})["gain_max_q10"] == 32767
    for bad in ({"dark_level": -1}, {"clip_level": 256}, {"dark_level": 9, "clip_level": 8}, {"min_quads": 0},
                {"gain_max_q10": 1023}, {"gain_max_q10": 32768}, {"gain": 2}):
        with pytest.raises(ValueError):
            R.awb_params(bad)
    with pytest.raises(ValueError):
        R.awb_statistics(np.zeros((4, 4), np.uint16), L.CH_BAYER_RGGB)
    with pytest.raises(ValueError):
        R.awb_statistics(np.zeros((2, 4, 4), np.uint8), L.CH_BAYER_RGGB)


def test_c_defaults_and_record_layout_match():
    from irmv_detection_b200 import engine as E
    p = L.AwbParams()
    assert L.lib().irmv_awb_params_default(C.byref(p)) == 0
    assert {k: getattr(p, k) for k in R.AWB_DEFAULTS} == R.AWB_DEFAULTS
    assert E.AWB_DTYPE.itemsize == 56 and E.AWB_DTYPE.fields["gain_q10"][1] == 40
