"""Colour-correction stage (raw_lut.apply_color_matrix, raw_lut.color_matrix_q10): the definition the engine's
kernels are checked against, on the host."""
import numpy as np
import pytest

from irmv_detection_b200 import raw_lut as R

I1024 = (1024 * np.eye(3)).astype(np.int16)


def _px(r, g, b):
    return np.array([[r, g, b]], np.uint8)


def test_identity_without_tone_returns_the_input():
    rgb = np.random.default_rng(0).integers(0, 256, (7, 5, 3), dtype=np.uint8)
    out = R.apply_color_matrix(rgb, I1024)
    assert out.dtype == np.uint8 and out.shape == rgb.shape
    assert np.array_equal(out, rgb)


def test_rounding_boundaries():
    m = np.zeros((3, 3), np.int16)
    m[0, 0] = 511                                       # v = 511: (511 + 512) >> 10 = 0
    m[1, 0] = 512                                       # v = 512: (512 + 512) >> 10 = 1
    m[2, 0] = 1535                                      # v = 1535: 1
    assert R.apply_color_matrix(_px(1, 0, 0), m).tolist() == [[0, 1, 1]]
    m[2, 0] = 1536                                      # v = 1536: 2 (half rounds up)
    assert R.apply_color_matrix(_px(1, 0, 0), m)[0, 2] == 2


def test_clamping():
    m = np.zeros((3, 3), np.int16)
    m[0] = (-1024, 0, 0)                                # negative sum: 0
    m[1] = (1026, 0, 0)                                 # 255 * 1026 = 261630 < 255.5 * 1024: 255
    m[2] = (0, 0, 0)
    assert R.apply_color_matrix(_px(10, 0, 0), m).tolist() == [[0, 10, 0]]
    assert R.apply_color_matrix(_px(255, 0, 0), m)[0, 1] == 255
    m[1] = (1024, 1, 0)                                 # 255 * 1024 + 512 = 255.5 * 1024: 256 before the clamp
    m[2] = (1024, 1024, 1024)                           # far above
    assert R.apply_color_matrix(_px(255, 255, 0), m)[0, 1:].tolist() == [255, 255]
    m[0] = (-32768, -32768, -32768)                     # the most negative sum the int16 matrix allows
    assert R.apply_color_matrix(_px(255, 255, 255), m)[0, 0] == 0


def test_floor_of_negative_sums():
    m = np.zeros((3, 3), np.int16)
    m[0] = (-513, 0, 0)                                 # v = -513: (-1) >> 10 = -1 -> 0, never a truncation to 0
    m[1] = (2048, -512, 0)                              # v = 2048 - 512 = 1536: 2
    assert R.apply_color_matrix(_px(1, 1, 0), m).tolist() == [[0, 2, 0]]


def test_tone_is_per_output_channel():
    tone = np.stack([np.arange(256), 255 - np.arange(256), np.full(256, 7)]).astype(np.uint8)
    out = R.apply_color_matrix(_px(10, 20, 30), I1024, tone)
    assert out.tolist() == [[10, 235, 7]]


def test_matches_a_scalar_loop():
    rng = np.random.default_rng(3)
    rgb = rng.integers(0, 256, (40, 3), dtype=np.uint8)
    m = rng.integers(-3000, 3000, (3, 3)).astype(np.int16)
    tone = rng.integers(0, 256, (3, 256), dtype=np.uint8)
    out = R.apply_color_matrix(rgb, m, tone)
    for p, o in zip(rgb.tolist(), out.tolist()):
        for c in range(3):
            v = sum(int(m[c, k]) * p[k] for k in range(3))
            assert o[c] == tone[c, min(max((v + 512) // 1024, 0), 255)]


def test_q10_identity_and_saturation():
    q = R.color_matrix_q10()
    assert q.dtype == np.int16 and np.array_equal(q, I1024)
    z = R.color_matrix_q10(saturation=0.0)
    luma = np.rint(1024 * np.array(R.LUMA_BT601)).astype(np.int16)
    for row in z:
        assert np.array_equal(row, luma)
    s = R.color_matrix_q10(saturation=1.5)
    assert (s[~np.eye(3, dtype=bool)] < 0).all() and (np.diag(s) > 1024).all()


def test_q10_applies_ccm_and_clips():
    ccm = np.array([[1.5, -0.3, -0.2], [-0.2, 1.4, -0.2], [-0.1, -0.4, 1.5]])
    assert np.array_equal(R.color_matrix_q10(ccm), np.rint(1024 * ccm).astype(np.int16))
    big = R.color_matrix_q10(np.full((3, 3), 100.0))
    assert (big == 32767).all()


@pytest.mark.parametrize("m,tone", [
    (np.eye(3, dtype=np.int32) * 1024, None),
    (np.eye(3) * 1024, None),
    (I1024[:2], None),
    (I1024, np.zeros((3, 255), np.uint8)),
    (I1024, np.zeros((3, 256), np.int16)),
])
def test_shape_and_dtype_errors(m, tone):
    with pytest.raises(ValueError):
        R.apply_color_matrix(_px(1, 2, 3), m, tone)


def test_input_errors():
    with pytest.raises(ValueError):
        R.apply_color_matrix(np.zeros((2, 2, 4), np.uint8), I1024)
    with pytest.raises(ValueError):
        R.apply_color_matrix(np.zeros((2, 2, 3), np.int32), I1024)
    with pytest.raises(ValueError):
        R.color_matrix_q10(np.eye(2))
