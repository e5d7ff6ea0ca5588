"""Colour-correction stage of Bayer sources (YoloEngine.set_color_matrix).  Every test rests on one identity: the
Bayer engine with raw table L, matrix M and tone T on frames F returns, bit for bit, what the otherwise identical
PASSTHROUGH engine without any stage returns on the packed frames
apply_color_matrix(demosaic_bilinear(apply_raw_lut(F, L)), M, T) -- detections, kept indices, head tensors, network
input, detect(0), the rotated view, armors and poses -- on every kernel that demosaics the raw frame: the camera-case
stem, the generic stem (sampled and column-walk forms), the unfused preprocess, the rotate kernel and the fused armor
stage.  Both kinds of engine are pinned to the same preprocess oracle, and a Bayer rotated view stores R, G, B in the
byte order of a packed one."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PATTERN_NAME = {2: "RGGB", 3: "BGGR", 4: "GRBG", 5: "GBRG"}
HEADS = [f"{t}{i}" for t in ("box", "cls") for i in range(3)]
PATHS = {"camera": {}, "letterbox": {"letterbox": True}, "float_input": {"quantize_u8": False},
         "unfused": {"fused_stem": False}}


def _cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _lut():
    from irmv_detection_b200 import raw_lut as R
    return R.make_raw_lut(8, (1.9, 1.0, 1.6), 1.0)


def _matrix():
    """Negative off-diagonal entries and a saturation gain above 1: both ends of the clamp are reached."""
    from irmv_detection_b200 import raw_lut as R
    ccm = np.array([[1.55, -0.35, -0.20], [-0.25, 1.45, -0.20], [-0.05, -0.45, 1.50]])
    return R.color_matrix_q10(ccm, saturation=1.4)


def _tone():
    from irmv_detection_b200 import raw_lut as R
    return R.make_raw_lut(0, (1, 1, 1), 1 / 2.2)


def _scaled_rgb(base_image, n, seed, w, h):
    from irmv_detection_b200 import synth
    rgb = synth.frames_from_base(base_image, n, seed=seed)[..., ::-1]
    if (w, h) != (rgb.shape[2], rgb.shape[1]):
        ys, xs = np.arange(h) * rgb.shape[1] // h, np.arange(w) * rgb.shape[2] // w
        rgb = rgb[:, ys][:, :, xs]
    return np.ascontiguousarray(rgb)


def _bayer_frames(base_image, n, chan, seed, w=1280, h=1024):
    from irmv_detection_b200 import synth
    return np.ascontiguousarray(synth.bayer_from_rgb(_scaled_rgb(base_image, n, seed, w, h), PATTERN_NAME[chan]))


def _packed(mosaics, chan, m, tone, lut=None):
    """The definition: 8-bit mosaics -> raw table -> demosaic -> colour stage -> packed u8 RGB frames."""
    from irmv_detection_b200 import raw_lut as R
    from oracle import preprocess_ref as PR
    if lut is not None:
        mosaics = R.apply_raw_lut(mosaics, lut, chan)
    rgb = np.stack([PR.demosaic_bilinear(f, chan) for f in mosaics])
    return np.ascontiguousarray(rgb if m is None else R.apply_color_matrix(rgb, m, tone))


def _same_bits(a, b):
    return a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()


def _run(eng, frames, read_input=False):
    """Everything a synchronous batch call and a detect() on slot 0 expose."""
    out = {}
    counts, dets = eng.detect_batch_arrays(frames)
    out["counts"], out["dets"] = counts.copy(), dets.copy()
    out["kept"] = [eng.kept_indices(f) for f in range(len(frames))]
    out["heads"] = [eng.read_tensor(h) for h in HEADS]
    if read_input:
        out["input"] = eng.read_tensor("input")
    eng.get_src_image_buffer(0)[...] = frames[0]
    out["det0"] = eng.detect(0)
    out["rot"] = eng.get_rotated_image(0)
    return out


def _assert_same(got, want, what=""):
    assert np.array_equal(got["counts"], want["counts"]), what
    for f, k in enumerate(want["counts"]):
        assert np.array_equal(got["dets"][f, :k], want["dets"][f, :k]), f"{what} frame {f}: detections"
        assert np.array_equal(got["kept"][f], want["kept"][f]), f"{what} frame {f}: kept indices"
    for h, a, b in zip(HEADS, got["heads"], want["heads"]):
        assert _same_bits(a, b), f"{what} {h}"
    if "input" in want:
        assert _same_bits(got["input"], want["input"]), f"{what} network input"
    assert got["det0"] == want["det0"], what
    assert np.array_equal(got["rot"], want["rot"]), f"{what} rotated view"


def test_stage_reaches_both_clamps(base_image):
    """The chosen matrix and tone clamp on both sides on the test frames (otherwise the clamp is untested)."""
    from irmv_detection_b200 import raw_lut as R
    from oracle import preprocess_ref as PR
    raw = _bayer_frames(base_image, 1, 2, seed=1)
    rgb = PR.demosaic_bilinear(R.apply_raw_lut(raw, _lut(), 2)[0], 2).astype(np.int64)
    v = rgb @ _matrix().astype(np.int64).T
    assert ((v + 512) >> 10).min() < 0 and ((v + 512) >> 10).max() > 255


@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("chan", [2, 3, 4, 5])
@pytest.mark.parametrize("rotate", [True, False])
def test_stage_equals_packed_engine_on_corrected_frames(base_image, weights_seed0, path, chan, rotate):
    import irmv_detection_b200 as irmv
    _cuda()
    lut, m, tone = _lut(), _matrix(), _tone()
    raw = _bayer_frames(base_image, 2, chan, seed=60 + chan)
    kw = dict(rotate180=rotate, max_batch=2, sub_batch=2, **PATHS[path])
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=chan, **kw)
    ref = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=irmv.CH_PASSTHROUGH, **kw)
    eng.set_raw_lut(lut)
    eng.set_color_matrix(m, tone)
    read_input = path == "unfused"
    _assert_same(_run(eng, raw, read_input), _run(ref, _packed(raw, chan, m, tone, lut), read_input))
    assert np.array_equal(eng.get_src_image_buffer(0), raw[0]), "the pinned slot must keep the raw frame"
    assert eng.check_padding() == 0 and ref.check_padding() == 0
    eng.close(); ref.close()


def test_bench_shape_device_and_pipelined_host(base_image, weights_seed0):
    """bench.py's configuration: 256 device-resident 1280 x 1024 RGGB frames as one replay with fused PnP, and the
    same engine's pipelined host path (128-frame chunks through the copy stream)."""
    import torch
    import irmv_detection_b200 as irmv
    from oracle import pnp_ref as P
    _cuda()
    lut, m, tone = _lut(), _matrix(), _tone()
    raw16 = _bayer_frames(base_image, 16, 2, seed=78)
    raw = np.ascontiguousarray(np.tile(raw16, (16, 1, 1)))
    pre = np.ascontiguousarray(np.tile(_packed(raw16, 2, m, tone, lut), (16, 1, 1, 1)))
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=irmv.CH_BAYER_RGGB, max_batch=256)
    ref = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=irmv.CH_PASSTHROUGH, max_batch=256)
    for e in (eng, ref):
        e.enable_pnp(P.K_DEFAULT, P.D_DEFAULT, (0.5, 480 / 1024))
    eng.set_raw_lut(lut)
    eng.set_color_matrix(m, tone)
    assert eng.stem_camera_ctas() == 2, "the colour stage must keep two CTAs per SM at 1024 rows"
    raw_dev, pre_dev = torch.from_numpy(raw).cuda(), torch.from_numpy(pre).cuda()
    got = eng.detect_batch_device(raw_dev.data_ptr(), 256)
    want = ref.detect_batch_device(pre_dev.data_ptr(), 256)
    assert got == want
    assert sum(len(d) for d in want) > 0
    for a, b in zip(eng.fetch_poses(256), ref.fetch_poses(256)):
        assert np.array_equal(a, b)
    for h in HEADS:
        assert _same_bits(eng.read_tensor(h), ref.read_tensor(h)), h
    assert torch.equal(raw_dev.cpu(), torch.from_numpy(raw)), "the device batch must keep the raw frames"
    pin_raw = torch.from_numpy(raw).pin_memory().numpy()
    pin_pre = torch.from_numpy(pre).pin_memory().numpy()
    cg, dg, rvg, tvg, okg = eng.collect_arrays(eng.submit_batch(pin_raw), poses=True)
    cg, dg, rvg, tvg, okg = cg.copy(), dg.copy(), rvg.copy(), tvg.copy(), okg.copy()
    cw, dw, rvw, tvw, okw = ref.collect_arrays(ref.submit_batch(pin_pre), poses=True)
    assert np.array_equal(cg, cw)
    for f in range(256):
        k = int(cw[f])
        assert np.array_equal(dg[f, :k], dw[f, :k]), f"pipelined frame {f}"
        assert np.array_equal(rvg[f, :k], rvw[f, :k]) and np.array_equal(tvg[f, :k], tvw[f, :k])
        assert np.array_equal(okg[f, :k], okw[f, :k])
    assert np.array_equal(pin_raw, raw), "the caller's host frames must stay raw"
    assert eng.check_padding() == 0 and ref.check_padding() == 0
    eng.close(); ref.close()


@pytest.mark.parametrize("chan,rotate", [(2, True), (3, False), (5, True)])
def test_fused_armors_and_poses_on_light_bar_scenes(weights_seed0, chan, rotate):
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import synth
    from oracle import pnp_ref as P, preprocess_ref as PR
    _cuda()
    lut, m, tone = _lut(), _matrix(), _tone()
    scenes = [synth.armor_scene(10, s)[0] for s in (7, 8, 9)]
    cam = [PR.rot180(s) if rotate else s for s in scenes]           # frames as the camera wrote them
    raw = np.ascontiguousarray(np.stack([synth.bayer_from_rgb(c, PATTERN_NAME[chan]) for c in cam]))
    prm = dict(light_min_ratio=0.01, light_max_ratio=10.0, light_max_angle=90.0, min_small_center_distance=0.0,
               max_large_center_distance=1e9)

    def run(eng, frames):
        counts, dets = eng.detect_batch_arrays(frames)
        return counts.copy(), dets.copy(), eng.fetch_armors(3), eng.fetch_armor_poses(3)

    engines = []
    for c in (chan, irmv.CH_PASSTHROUGH, chan):
        e = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=c, rotate180=rotate, max_batch=3)
        e.enable_armors(**prm)
        e.enable_pnp(P.K_DEFAULT, P.D_DEFAULT, (0.5, 480 / 1024))
        engines.append(e)
    eng, ref, plain = engines
    eng.set_raw_lut(lut)
    eng.set_color_matrix(m, tone)
    plain.set_raw_lut(lut)
    got, want, untouched = run(eng, raw), run(ref, _packed(raw, chan, m, tone, lut)), run(plain, raw)
    assert np.array_equal(got[0], want[0])
    assert int(want[0].sum()) > 0, "no detections: the armor stage had nothing to work on"
    for f, k in enumerate(want[0]):
        assert np.array_equal(got[1][f, :k], want[1][f, :k])
    assert _same_bits(got[2], want[2]), "armors"
    assert _same_bits(got[3], want[3]), "armor poses"
    # a stage that changes nothing would pass the comparison above: it must change what the detector sees
    changed = not np.array_equal(untouched[0], want[0]) or not _same_bits(untouched[2], want[2]) or \
        any(not np.array_equal(untouched[1][f, :k], want[1][f, :k]) for f, k in enumerate(want[0]))
    assert changed, "the colour stage changed neither detections nor armors"
    print("armors:", int(want[2]["valid"].sum()), "without the stage:", int(untouched[2]["valid"].sum()))
    for e in engines:
        assert e.check_padding() == 0
        e.close()


@pytest.mark.parametrize("fmt", [3, 1])                     # RAW_12_PACKED, RAW_10
@pytest.mark.parametrize("size", [(1280, 1024), (1920, 1200)])
def test_wide_formats_after_the_decode(base_image, weights_seed0, fmt, size):
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import raw_lut as R
    _cuda()
    W, H = size
    chan = irmv.CH_BAYER_GBRG
    b = R.RAW_BITS[fmt]
    v8 = _bayer_frames(base_image, 2, chan, seed=90 + fmt, w=W, h=H)
    rng = np.random.default_rng(fmt)
    wide = (v8.astype(np.uint16) << (b - 8)) | rng.integers(0, 1 << (b - 8), v8.shape, dtype=np.uint16)
    frames = np.ascontiguousarray(R.pack_raw12_packed(wide) if fmt == irmv.RAW_12_PACKED else wide)
    dlut = R.make_raw_lut(8 << (b - 8), (1.9, 1.0, 1.6), 1.0, bits=b)
    m, tone = _matrix(), _tone()
    kw = dict(max_batch=2, sub_batch=2)
    eng = irmv.YoloEngine(weights_seed0, (W, H), chan_order=chan, raw_format=fmt, **kw)
    ref = irmv.YoloEngine(weights_seed0, (W, H), chan_order=irmv.CH_PASSTHROUGH, **kw)
    eng.set_raw_lut(dlut)
    eng.set_color_matrix(m, tone)
    pre = _packed(R.decode_raw(frames, fmt, dlut, chan), chan, m, tone)
    _assert_same(_run(eng, frames), _run(ref, pre), f"fmt {fmt} {W}x{H}")
    assert eng.check_padding() == 0 and ref.check_padding() == 0
    eng.close(); ref.close()


@pytest.fixture(scope="module")
def probe_weights(tmp_path_factory):
    """Weight files whose conv0 exposes every network-input pixel of the fused stem (oracle/stem_probe.py)."""
    from irmv_detection_b200 import weights
    from oracle import stem_probe as SP
    paths = []
    for i, taps in enumerate(SP.TAP_FILES):
        tens = weights.random_init(0)
        tens[0] = SP.probe_conv0(taps)
        p = str(tmp_path_factory.mktemp("probe") / f"probe{i}.irmw")
        weights.save(p, tens)
        paths.append(p)
    return paths


@pytest.mark.parametrize("h", [720, 1024, 1200, 760])
def test_stem_heights(base_image, weights_seed0, probe_weights, h):
    """Camera-kernel heights.  At 760 rows the tables would cost the camera kernel a CTA per SM, so the Bayer frames go
    to stem_kernel while the packed reference stays on the camera kernel; the two kernels accumulate conv0 in different
    orders, so there the fused stem's input is compared exactly through the probe weights instead of bit for bit after
    conv0 -- either way the result is the definition."""
    import irmv_detection_b200 as irmv
    from oracle import preprocess_ref as PR, stem_probe as SP
    _cuda()
    chan = irmv.CH_BAYER_BGGR
    lut, m, tone = _lut(), _matrix(), _tone()
    raw = _bayer_frames(base_image, 2, chan, seed=h, h=h)
    pre = _packed(raw, chan, m, tone, lut)
    kw = dict(max_batch=2, sub_batch=2)

    def staged(wpath):
        e = irmv.YoloEngine(wpath, (1280, h), chan_order=chan, **kw)
        e.set_raw_lut(lut)
        e.set_color_matrix(m, tone)
        return e

    m0s = []
    for wp in probe_weights:
        e = staged(wp)
        e.detect_batch(raw)
        m0s.append(e.read_tensor("m0"))
        assert e.check_padding() == 0
        e.close()
    x = np.stack([PR.preprocess_fp16(f, irmv.CH_PASSTHROUGH, True, True, False)[0] for f in pre])
    msg = SP.compare_codes(SP.engine_views(m0s), np.rint(x.astype(np.float64) * 255).astype(np.int64))
    assert msg is None, f"{h} rows, fused stem input: {msg}"

    eng = irmv.YoloEngine(weights_seed0, (1280, h), chan_order=chan, **kw)
    off = eng.stem_camera_ctas()
    eng.close()
    eng = staged(weights_seed0)
    on = eng.stem_camera_ctas()
    print(f"{h} rows: camera-kernel CTAs per SM {off} without tables, {on} with raw table + colour stage")
    if h == 1024:
        assert on == 2
    assert on in (0, off), "the tables may send the frames to stem_kernel, never run the camera kernel at fewer CTAs"
    if on:                                  # both engines on the camera kernel: bit for bit through the whole pipeline
        ref = irmv.YoloEngine(weights_seed0, (1280, h), chan_order=irmv.CH_PASSTHROUGH, **kw)
        _assert_same(_run(eng, raw), _run(ref, pre), f"{h} rows")
        assert ref.check_padding() == 0
        ref.close()
    else:                                   # the rotated view does not depend on the stem kernel
        eng.detect_batch(raw)
        eng.get_src_image_buffer(0)[...] = raw[0]
        eng.detect(0)
        assert np.array_equal(eng.get_rotated_image(0), PR.rot180(pre[0])), f"{h} rows rotated view"
    assert eng.check_padding() == 0
    eng.close()


def test_identity_clear_and_never_set(base_image, weights_seed0):
    import irmv_detection_b200 as irmv
    _cuda()
    chan = irmv.CH_BAYER_GRBG
    raw = _bayer_frames(base_image, 2, chan, seed=5)
    ident = (1024 * np.eye(3)).astype(np.int16)
    kw = dict(chan_order=chan, max_batch=2, sub_batch=2)
    never = irmv.YoloEngine(weights_seed0, (1280, 1024), **kw)
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), **kw)
    want = _run(never, raw)
    eng.set_color_matrix(ident)
    _assert_same(_run(eng, raw), want, "identity matrix")
    eng.set_color_matrix(ident, np.tile(np.arange(256, dtype=np.uint8), (3, 1)))
    _assert_same(_run(eng, raw), want, "identity matrix and tone")
    never.set_raw_lut(_lut())
    eng.set_raw_lut(_lut())
    _assert_same(_run(eng, raw), _run(never, raw), "identity matrix with a raw table")
    never.set_raw_lut(None)
    eng.set_raw_lut(None)
    eng.set_color_matrix(_matrix(), _tone())
    changed = _run(eng, raw)
    assert not all(_same_bits(a, b) for a, b in zip(changed["heads"], want["heads"]))
    eng.set_color_matrix(None)
    _assert_same(_run(eng, raw), want, "cleared")
    assert eng.check_padding() == 0 and never.check_padding() == 0
    eng.close(); never.close()


def test_update_in_place_without_allocation(base_image, weights_seed0):
    import torch
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import _lib, raw_lut as R
    _cuda()
    lib = _lib.lib()
    chan = irmv.CH_BAYER_RGGB
    raw = _bayer_frames(base_image, 2, chan, seed=9)
    m1, t1 = _matrix(), _tone()
    m2, t2 = R.color_matrix_q10(saturation=0.3), R.make_raw_lut(0, (1, 1, 1), 0.7)
    kw = dict(max_batch=2, sub_batch=2)
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=chan, **kw)
    ref = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=irmv.CH_PASSTHROUGH, **kw)
    raw_dev = torch.from_numpy(raw).cuda()
    eng.set_color_matrix(m1, t1)
    _assert_same(_run(eng, raw), _run(ref, _packed(raw, chan, m1, t1)), "first matrix")
    eng.detect_batch_device(raw_dev.data_ptr(), 2)
    before = lib.irmv_debug_alloc_count()
    eng.set_color_matrix(m2, t2)
    got = _run(eng, raw)
    got_dev = eng.detect_batch_device(raw_dev.data_ptr(), 2)
    eng.set_color_matrix(m1, t1)
    eng.set_color_matrix(m2, t2)
    eng.detect(0)
    assert lib.irmv_debug_alloc_count() == before
    pre2 = _packed(raw, chan, m2, t2)
    _assert_same(got, _run(ref, pre2), "updated matrix")
    assert got_dev == ref.detect_batch(pre2)
    assert np.array_equal(eng.get_src_image_buffer(0), raw[0]) and torch.equal(raw_dev.cpu(), torch.from_numpy(raw))
    assert eng.check_padding() == 0 and ref.check_padding() == 0
    eng.close(); ref.close()


def test_set_color_matrix_errors(base_image, weights_seed0):
    import torch
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import _lib
    _cuda()
    m, tone = _matrix(), _tone()
    for chan in (irmv.CH_PASSTHROUGH, irmv.CH_SWAP_RB):
        rgb = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=chan, max_batch=1)
        with pytest.raises(irmv.IrmvError):
            rgb.set_color_matrix(m, tone)
        with pytest.raises(irmv.IrmvError):
            rgb.set_color_matrix(None)
        assert rgb.check_padding() == 0
        rgb.close()
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=irmv.CH_BAYER_RGGB, max_batch=2, sub_batch=2)
    for bad_m, bad_t in ((m.astype(np.int32), None), (m[:2], None), (m.astype(np.float32), None), (m, tone[:2]),
                         (m, tone.astype(np.int16))):
        with pytest.raises(ValueError):
            eng.set_color_matrix(bad_m, bad_t)
    with pytest.raises(irmv.IrmvError):
        eng.set_color_matrix(None, tone)                  # a tone table without a matrix
    lib = _lib.lib()
    assert lib.irmv_engine_set_color_matrix(eng._h, None, tone.ctypes.data) != 0
    host = torch.from_numpy(_bayer_frames(base_image, 2, 2, seed=3)).pin_memory().numpy()
    t = eng.submit_batch(host)
    with pytest.raises(irmv.IrmvError):
        eng.set_color_matrix(m, tone)                     # a batch is in flight
    eng.collect_arrays(t)
    eng.set_color_matrix(m, tone)
    assert eng.check_padding() == 0
    eng.close()
