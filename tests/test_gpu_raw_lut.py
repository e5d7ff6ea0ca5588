"""Raw-domain colour stage of Bayer sources (YoloEngine.set_raw_lut): an engine with table L on frames F must
return, bit for bit, what the same engine without a table returns on apply_raw_lut(F, L) -- detections, kept
indices, head tensors, network input, armors, poses and the rotated view -- on every kernel that reads the raw
frame: the camera-case stem, the generic stem (sampled and column-walk forms), the unfused preprocess, the
rotate kernel and the fused armor stage."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PATTERN_NAME = {2: "RGGB", 3: "BGGR", 4: "GRBG", 5: "GBRG"}
HEADS = [f"{t}{i}" for t in ("box", "cls") for i in range(3)]


def _cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _lut():
    from irmv_detection_b200 import raw_lut as R
    return R.make_raw_lut(8, (1.9, 1.0, 1.6), 1 / 2.2)


def _bayer_frames(base_image, n, chan, seed):
    from irmv_detection_b200 import synth
    rgb = synth.frames_from_base(base_image, n, seed=seed)[..., ::-1]
    return np.ascontiguousarray(synth.bayer_from_rgb(rgb, PATTERN_NAME[chan]))


def _pre(frames, lut, chan):
    from irmv_detection_b200 import raw_lut as R
    return np.ascontiguousarray(R.apply_raw_lut(frames, lut, chan))


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


def _assert_same(got, want):
    assert np.array_equal(got["counts"], want["counts"])
    for f, k in enumerate(want["counts"]):
        assert np.array_equal(got["dets"][f, :k], want["dets"][f, :k]), f"frame {f}: detections"
        assert np.array_equal(got["kept"][f], want["kept"][f]), f"frame {f}: kept indices"
    for h, a, b in zip(HEADS, got["heads"], want["heads"]):
        assert _same_bits(a, b), h
    if "input" in want:
        assert _same_bits(got["input"], want["input"]), "network input"
    assert got["det0"] == want["det0"]
    assert np.array_equal(got["rot"], want["rot"]), "rotated view"


# camera: 1280 x 1024 stretch, 8-bit intermediate (stem_bayer.cu); letterbox: stem_kernel's sampled path;
# float_input: no 8-bit intermediate, so stem_kernel's column walk; unfused: preprocess_kernel + conv0
PATHS = {"camera": {}, "letterbox": {"letterbox": True}, "float_input": {"quantize_u8": False},
         "unfused": {"fused_stem": False}}


@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("chan", [2, 3, 4, 5])
@pytest.mark.parametrize("rotate", [True, False])
def test_table_equals_preapplied_frames(base_image, weights_seed0, path, chan, rotate):
    import irmv_detection_b200 as irmv
    _cuda()
    lut = _lut()
    raw = _bayer_frames(base_image, 2, chan, seed=20 + chan)
    kw = dict(chan_order=chan, rotate180=rotate, max_batch=2, sub_batch=2, **PATHS[path])
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), **kw)
    ref = irmv.YoloEngine(weights_seed0, (1280, 1024), **kw)
    eng.set_raw_lut(lut)
    got = _run(eng, raw, read_input=path == "unfused")
    want = _run(ref, _pre(raw, lut, chan), read_input=path == "unfused")
    _assert_same(got, want)
    assert np.array_equal(eng.get_src_image_buffer(0), raw[0]), "the pinned slot must keep the raw frame"
    assert eng.check_padding() == 0
    eng.close(); ref.close()


def test_bench_shape_device_and_pipelined_host(base_image, weights_seed0):
    """bench.py's configuration: 256 device-resident Bayer frames as one replay with fused PnP, and the same
    engine's pipelined host path (128-frame chunks through the copy stream)."""
    import torch
    import irmv_detection_b200 as irmv
    from oracle import pnp_ref as P
    _cuda()
    lut = _lut()
    raw16 = _bayer_frames(base_image, 16, 2, seed=77)
    raw = np.ascontiguousarray(np.tile(raw16, (16, 1, 1)))
    pre = _pre(raw, lut, 2)
    engines = []
    for _ in range(2):
        e = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=irmv.CH_BAYER_RGGB, max_batch=256)
        e.enable_pnp(P.K_DEFAULT, P.D_DEFAULT, (0.5, 480 / 1024))
        engines.append(e)
    eng, ref = engines
    eng.set_raw_lut(lut)
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
    cg, dg = cg.copy(), dg.copy()
    cw, dw, rvw, tvw, okw = ref.collect_arrays(ref.submit_batch(pin_pre), poses=True)
    assert np.array_equal(cg, cw)
    for f in range(256):
        k = int(cw[f])
        assert np.array_equal(dg[f, :k], dw[f, :k]), f"pipelined frame {f}"
        assert np.array_equal(rvg[f, :k], rvw[f, :k]) and np.array_equal(tvg[f, :k], tvw[f, :k])
        assert np.array_equal(okg[f, :k], okw[f, :k])
    assert np.array_equal(pin_raw, raw), "the caller's host frames must stay raw"
    assert eng.check_padding() == 0
    eng.close(); ref.close()


@pytest.mark.parametrize("chan,rotate", [(2, True), (3, False), (5, True)])
def test_fused_armors_and_poses_on_light_bar_scenes(weights_seed0, chan, rotate):
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import synth
    from oracle import pnp_ref as P, preprocess_ref as PR
    _cuda()
    lut = _lut()
    scenes = [synth.armor_scene(10, s)[0] for s in (7, 8, 9)]
    cam = [PR.rot180(s) if rotate else s for s in scenes]           # frames as the camera wrote them
    raw = np.ascontiguousarray(np.stack([synth.bayer_from_rgb(c, PATTERN_NAME[chan]) for c in cam]))
    prm = dict(light_min_ratio=0.01, light_max_ratio=10.0, light_max_angle=90.0, min_small_center_distance=0.0,
               max_large_center_distance=1e9)

    def run(eng, frames):
        counts, dets = eng.detect_batch_arrays(frames)
        return counts.copy(), dets.copy(), eng.fetch_armors(3), eng.fetch_armor_poses(3)

    engines = []
    for _ in range(3):
        e = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=chan, rotate180=rotate, max_batch=3)
        e.enable_armors(**prm)
        e.enable_pnp(P.K_DEFAULT, P.D_DEFAULT, (0.5, 480 / 1024))
        engines.append(e)
    eng, ref, plain = engines
    eng.set_raw_lut(lut)
    got, want, untouched = run(eng, raw), run(ref, _pre(raw, lut, chan)), run(plain, raw)
    assert np.array_equal(got[0], want[0])
    assert int(want[0].sum()) > 0, "no detections: the armor stage had nothing to work on"
    for f, k in enumerate(want[0]):
        assert np.array_equal(got[1][f, :k], want[1][f, :k])
    assert _same_bits(got[2], want[2]), "armors"
    assert _same_bits(got[3], want[3]), "armor poses"
    # a table that changes nothing would pass the comparison above: it must change what the stage sees
    changed = not np.array_equal(untouched[0], want[0]) or not _same_bits(untouched[2], want[2]) or \
        any(not np.array_equal(untouched[1][f, :k], want[1][f, :k]) for f, k in enumerate(want[0]))
    assert changed, "the table changed neither detections nor armors"
    print("armors:", int(want[2]["valid"].sum()), "without table:", int(untouched[2]["valid"].sum()))
    for e in engines:
        assert e.check_padding() == 0
        e.close()


def test_identity_and_cleared_tables_match_no_table(base_image, weights_seed0):
    import irmv_detection_b200 as irmv
    _cuda()
    raw = _bayer_frames(base_image, 2, 3, seed=5)
    kw = dict(chan_order=irmv.CH_BAYER_BGGR, max_batch=2, sub_batch=2)
    never = irmv.YoloEngine(weights_seed0, (1280, 1024), **kw)
    want = _run(never, raw)
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), **kw)
    eng.set_raw_lut(np.tile(np.arange(256, dtype=np.uint8), (3, 1)))
    _assert_same(_run(eng, raw), want)
    eng.set_raw_lut(_lut())
    changed = _run(eng, raw)
    assert not all(_same_bits(a, b) for a, b in zip(changed["heads"], want["heads"]))
    eng.set_raw_lut(None)
    _assert_same(_run(eng, raw), want)
    eng.close(); never.close()


def test_table_update_in_place_without_allocation(base_image, weights_seed0):
    import torch
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import _lib, raw_lut as R
    _cuda()
    lib = _lib.lib()
    chan = irmv.CH_BAYER_GRBG
    raw = _bayer_frames(base_image, 2, chan, seed=9)
    l1 = _lut()
    l2 = R.make_raw_lut(16, (1.2, 0.9, 2.1), 0.8)
    kw = dict(chan_order=chan, max_batch=2, sub_batch=2)
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), **kw)
    ref = irmv.YoloEngine(weights_seed0, (1280, 1024), **kw)
    raw_dev = torch.from_numpy(raw).cuda()
    eng.set_raw_lut(l1)
    _assert_same(_run(eng, raw), _run(ref, _pre(raw, l1, chan)))
    eng.detect_batch_device(raw_dev.data_ptr(), 2)
    before = lib.irmv_debug_alloc_count()
    eng.set_raw_lut(l2)
    got = _run(eng, raw)
    got_dev = eng.detect_batch_device(raw_dev.data_ptr(), 2)
    eng.set_raw_lut(l1)
    eng.set_raw_lut(l2)
    eng.detect(0)
    assert lib.irmv_debug_alloc_count() == before
    want = _run(ref, _pre(raw, l2, chan))
    _assert_same(got, want)
    assert got_dev == ref.detect_batch(_pre(raw, l2, chan))
    assert np.array_equal(eng.get_src_image_buffer(0), raw[0]) and torch.equal(raw_dev.cpu(), torch.from_numpy(raw))
    assert eng.check_padding() == 0
    eng.close(); ref.close()


def test_set_raw_lut_errors(base_image, weights_seed0):
    import torch
    import irmv_detection_b200 as irmv
    _cuda()
    rgb = irmv.YoloEngine(weights_seed0, (1280, 1024), max_batch=1)
    with pytest.raises(irmv.IrmvError):
        rgb.set_raw_lut(_lut())
    with pytest.raises(irmv.IrmvError):
        rgb.set_raw_lut(None)
    rgb.close()
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=irmv.CH_BAYER_RGGB, max_batch=2, sub_batch=2)
    with pytest.raises(ValueError):
        eng.set_raw_lut(_lut()[:2])
    host = torch.from_numpy(_bayer_frames(base_image, 2, 2, seed=3)).pin_memory().numpy()
    t = eng.submit_batch(host)
    with pytest.raises(irmv.IrmvError):
        eng.set_raw_lut(_lut())                            # a batch is in flight
    eng.collect_arrays(t)
    eng.set_raw_lut(_lut())
    eng.close()
