"""The raw-domain colour stage's host definition (irmv_detection_b200.raw_lut): which table each sensor
position uses, for the four Bayer patterns, and that rot180 does not move a position to another table."""
import numpy as np
import pytest

from irmv_detection_b200 import raw_lut as R
from oracle import preprocess_ref as PR

PATTERNS = [PR.CH_BAYER_RGGB, PR.CH_BAYER_BGGR, PR.CH_BAYER_GRBG, PR.CH_BAYER_GBRG]


def _random_lut(seed):
    return np.random.default_rng(seed).integers(0, 256, (3, 256), dtype=np.uint8)


@pytest.mark.parametrize("pattern", PATTERNS)
def test_constant_colour_maps_through_its_site_tables(pattern):
    lut = _random_lut(pattern)
    for a, b, c in [(0, 0, 0), (255, 255, 255), (10, 128, 250), (200, 3, 77)]:
        img = np.empty((6, 8, 3), np.uint8)
        img[...] = (a, b, c)
        got = R.apply_raw_lut(PR.mosaic_from_rgb(img, pattern), lut, pattern)
        img[...] = (lut[0, a], lut[1, b], lut[2, c])
        assert np.array_equal(got, PR.mosaic_from_rgb(img, pattern))


@pytest.mark.parametrize("pattern", PATTERNS)
def test_table_is_chosen_by_sensor_position_before_rot180(pattern):
    rng = np.random.default_rng(1)
    raw = rng.integers(0, 256, (2, 10, 12), dtype=np.uint8)
    lut = _random_lut(10 + pattern)
    out = R.apply_raw_lut(raw, lut, pattern)
    sites = R.site_colours(10, 12, pattern)
    for y in range(10):
        for x in range(12):
            assert (out[:, y, x] == lut[sites[y, x], raw[:, y, x]]).all()
    # the rotated view of a corrected frame keeps each sample's own table: at rotated position (y, x) the
    # sample of sensor position (H-1-y, W-1-x), whose site is red where the rotated pattern has blue
    rot = out[:, ::-1, ::-1]
    assert np.array_equal(rot, lut[sites[::-1, ::-1], raw[:, ::-1, ::-1]])
    assert not np.array_equal(rot, R.apply_raw_lut(raw[:, ::-1, ::-1], lut, pattern))


def test_make_raw_lut():
    ident = R.make_raw_lut()
    assert np.array_equal(ident, np.tile(np.arange(256, dtype=np.uint8), (3, 1)))
    lut = R.make_raw_lut(8, (1.9, 1.0, 1.6), 1 / 2.2)
    assert lut.shape == (3, 256) and lut.dtype == np.uint8
    assert (lut[:, :9] == 0).all() and (lut[:, 255] == 255).all()
    assert (np.diff(lut.astype(int), axis=1) >= 0).all()
    assert (lut[0] >= lut[2]).all() and (lut[2] >= lut[1]).all()
    with pytest.raises(ValueError):
        R.apply_raw_lut(np.zeros((4, 4), np.uint8), lut[:2], PR.CH_BAYER_RGGB)
