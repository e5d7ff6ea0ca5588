"""10- and 12-bit raw sources (raw_format RAW_10, RAW_12, RAW_12_PACKED): a b-bit engine with table T on frames F
must return, bit for bit, what an otherwise identical 8-bit engine without a table returns on
raw_lut.decode_raw(F, raw_format, T, pattern) -- detections, kept indices, head tensors, network input, rotated view,
armors, poses -- on every path that reads the raw frame.  The 10/12-bit frames are built as (bayer8 << (b - 8)) |
seeded noise, so the default table reproduces the 8-bit synthetic frames and the detections are not empty."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PATTERN_NAME = {2: "RGGB", 3: "BGGR", 4: "GRBG", 5: "GBRG"}
HEADS = [f"{t}{i}" for t in ("box", "cls") for i in range(3)]
FORMATS = {"raw10": 1, "raw12": 2, "raw12_packed": 3}          # irmv.RAW_10, RAW_12, RAW_12_PACKED
# camera: 1280 x 1024 stretch, 8-bit intermediate (stem_bayer.cu); letterbox: stem_kernel's sampled path;
# float_input: no 8-bit intermediate, so stem_kernel's column walk; unfused: preprocess_kernel + conv0
PATHS = {"camera": {}, "letterbox": {"letterbox": True}, "float_input": {"quantize_u8": False},
         "unfused": {"fused_stem": False}}


def _cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _bayer_frames(base_image, n, chan, seed):
    from irmv_detection_b200 import synth
    rgb = synth.frames_from_base(base_image, n, seed=seed)[..., ::-1]
    return np.ascontiguousarray(synth.bayer_from_rgb(rgb, PATTERN_NAME[chan]))


def _widen(v8, fmt, seed, garbage=False):
    """u8 mosaics -> frames of `fmt`: (v8 << (b - 8)) | noise, packed for RAW_12_PACKED; garbage: random upper
    container bits (u16 formats)."""
    from irmv_detection_b200 import raw_lut as R
    b = R.RAW_BITS[fmt]
    rng = np.random.default_rng(seed)
    raw = (v8.astype(np.uint16) << (b - 8)) | rng.integers(0, 1 << (b - 8), v8.shape, dtype=np.uint16)
    if fmt == 3:
        return np.ascontiguousarray(R.pack_raw12_packed(raw))
    if garbage:
        raw |= (rng.integers(0, 1 << (16 - b), v8.shape, dtype=np.uint16) << b).astype(np.uint16)
    return np.ascontiguousarray(raw)


def _gamma(fmt):
    from irmv_detection_b200 import raw_lut as R
    b = R.RAW_BITS[fmt]
    return R.make_raw_lut(8 << (b - 8), (1.9, 1.0, 1.6), 1 / 2.2, bits=b)


def _decode(frames, fmt, lut, chan):
    from irmv_detection_b200 import raw_lut as R
    return np.ascontiguousarray(R.decode_raw(frames, fmt, lut, chan))


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


@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("chan", [2, 3, 4, 5])
@pytest.mark.parametrize("rotate", [True, False])
def test_bits_equal_8bit_engine_on_decoded_frames(base_image, weights_seed0, path, chan, rotate):
    import irmv_detection_b200 as irmv
    _cuda()
    v8 = _bayer_frames(base_image, 2, chan, seed=40 + chan)
    kw = dict(chan_order=chan, rotate180=rotate, max_batch=2, sub_batch=2, **PATHS[path])
    read_input = path == "unfused"
    ref = irmv.YoloEngine(weights_seed0, (1280, 1024), **kw)
    for name, fmt in FORMATS.items():
        frames = _widen(v8, fmt, seed=chan)
        keep = frames.copy()
        eng = irmv.YoloEngine(weights_seed0, (1280, 1024), raw_format=fmt, **kw)
        for lut in (None, _gamma(fmt)):
            if lut is not None:
                eng.set_raw_lut(lut)
            got = _run(eng, frames, read_input)
            want = _run(ref, _decode(frames, fmt, lut, chan), read_input)
            _assert_same(got, want, f"{name} {'gamma' if lut is not None else 'default'}")
        assert np.array_equal(frames, keep), "the caller's frames must not be written"
        assert np.array_equal(eng.get_src_image_buffer(0), frames[0]), "the pinned slot must keep the raw frame"
        assert eng.check_padding() == 0
        eng.close()
    assert ref.check_padding() == 0
    ref.close()


@pytest.mark.parametrize("fmt", [3, 1])
def test_generic_geometry_unaligned_frames(base_image, weights_seed0, fmt):
    """1300 x 970: a 12-bit packed frame is 1891500 bytes (not a multiple of 16), rows of 1300 samples do not split
    into 16-sample groups, and the batch ends on a ragged group.  Device batches at the caller's alignment (16-byte
    aligned and not) and host frames."""
    import torch
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import synth
    _cuda()
    W, H, chan = 1300, 970, irmv.CH_BAYER_GBRG
    ys, xs = np.arange(H) * 1024 // H, np.arange(W) * 1280 // W
    rgb = synth.frames_from_base(base_image, 3, seed=11)[:, ys][:, :, xs][..., ::-1]
    v8 = np.ascontiguousarray(synth.bayer_from_rgb(rgb, PATTERN_NAME[chan]))
    frames = _widen(v8, fmt, seed=12)
    lut = _gamma(fmt)
    kw = dict(chan_order=chan, max_batch=3, sub_batch=3)
    eng = irmv.YoloEngine(weights_seed0, (W, H), raw_format=fmt, **kw)
    ref = irmv.YoloEngine(weights_seed0, (W, H), **kw)
    eng.set_raw_lut(lut)
    pre = _decode(frames, fmt, lut, chan)
    want = _run(ref, pre)
    _assert_same(_run(eng, frames), want, "host frames")
    want_dev = ref.detect_batch(pre)
    raw_bytes = frames.view(np.uint8).reshape(-1)
    for off in (0, 1, 2, 6):                               # byte offset of the batch from a 256-byte boundary
        buf = torch.zeros(raw_bytes.size + 16, dtype=torch.uint8, device="cuda")
        buf[off:off + raw_bytes.size] = torch.from_numpy(raw_bytes).cuda()
        got = eng.detect_batch_device(buf.data_ptr() + off, 3)
        assert got == want_dev, f"device batch at offset {off}"
        for h in HEADS:
            assert _same_bits(eng.read_tensor(h), ref.read_tensor(h)), f"offset {off}: {h}"
        assert torch.equal(buf[off:off + raw_bytes.size].cpu(), torch.from_numpy(raw_bytes)), "device frames written"
    assert eng.check_padding() == 0 and ref.check_padding() == 0
    eng.close(); ref.close()


@pytest.mark.parametrize("fmt", [1, 2])
def test_upper_container_bits_are_ignored(base_image, weights_seed0, fmt):
    import irmv_detection_b200 as irmv
    _cuda()
    v8 = _bayer_frames(base_image, 2, 2, seed=31)
    from irmv_detection_b200 import raw_lut as R
    clean, dirty = _widen(v8, fmt, seed=5), _widen(v8, fmt, seed=5, garbage=True)
    assert not np.array_equal(clean, dirty) and np.array_equal(clean, dirty & ((1 << R.RAW_BITS[fmt]) - 1))
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=irmv.CH_BAYER_RGGB, raw_format=fmt, max_batch=2,
                          sub_batch=2, letterbox=True)
    eng.set_raw_lut(_gamma(fmt))
    want = _run(eng, clean)
    _assert_same(_run(eng, dirty), want, "garbage bits")
    assert eng.check_padding() == 0
    eng.close()


def test_bench_shape_packed_device_and_pipelined_host(base_image, weights_seed0):
    """bench.py's configuration at 12-bit packed: 256 device-resident frames as one replay with fused PnP, and the
    same engine's pipelined host path (128-frame chunks through the copy stream)."""
    import torch
    import irmv_detection_b200 as irmv
    from oracle import pnp_ref as P
    _cuda()
    W, H, fmt = 1280, 1024, irmv.RAW_12_PACKED
    v8 = _bayer_frames(base_image, 16, 2, seed=77)
    raw16 = _widen(v8, fmt, seed=78)
    raw = np.ascontiguousarray(np.tile(raw16, (16, 1, 1)))
    lut = _gamma(fmt)
    pre = _decode(raw, fmt, lut, 2)
    eng = irmv.YoloEngine(weights_seed0, (W, H), chan_order=irmv.CH_BAYER_RGGB, max_batch=256, raw_format=fmt)
    ref = irmv.YoloEngine(weights_seed0, (W, H), chan_order=irmv.CH_BAYER_RGGB, max_batch=256)
    for e in (eng, ref):
        e.enable_pnp(P.K_DEFAULT, P.D_DEFAULT, (0.5, 480 / 1024))
    eng.set_raw_lut(lut)
    raw_dev, pre_dev = torch.from_numpy(raw).cuda(), torch.from_numpy(pre).cuda()
    h0 = eng.copy_bytes()[0]
    got = eng.detect_batch_device(raw_dev.data_ptr(), 256)
    assert eng.copy_bytes()[0] == h0, "device-resident frames are not copied"
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
    h0 = eng.copy_bytes()[0]
    cg, dg, rvg, tvg, okg = eng.collect_arrays(eng.submit_batch(pin_raw), poses=True)
    assert eng.copy_bytes()[0] - h0 == 256 * W * H * 3 // 2
    cg, dg = cg.copy(), dg.copy()
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


@pytest.mark.parametrize("chan,rotate,fmt", [(2, True, 3), (3, False, 2), (5, True, 1)])
def test_fused_armors_and_poses_on_light_bar_scenes(weights_seed0, chan, rotate, fmt):
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import synth
    from oracle import pnp_ref as P, preprocess_ref as PR
    _cuda()
    lut = _gamma(fmt)
    scenes = [synth.armor_scene(10, s)[0] for s in (7, 8, 9)]
    cam = [PR.rot180(s) if rotate else s for s in scenes]           # frames as the camera wrote them
    v8 = np.ascontiguousarray(np.stack([synth.bayer_from_rgb(c, PATTERN_NAME[chan]) for c in cam]))
    raw = _widen(v8, fmt, seed=chan)
    prm = dict(light_min_ratio=0.01, light_max_ratio=10.0, light_max_angle=90.0, min_small_center_distance=0.0,
               max_large_center_distance=1e9)

    def run(eng, frames):
        counts, dets = eng.detect_batch_arrays(frames)
        return counts.copy(), dets.copy(), eng.fetch_armors(3), eng.fetch_armor_poses(3)

    engines = []
    for f in (fmt, fmt, 0):
        e = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=chan, rotate180=rotate, max_batch=3, raw_format=f)
        e.enable_armors(**prm)
        e.enable_pnp(P.K_DEFAULT, P.D_DEFAULT, (0.5, 480 / 1024))
        engines.append(e)
    eng, plain, ref = engines
    eng.set_raw_lut(lut)
    got, want, untouched = run(eng, raw), run(ref, _decode(raw, fmt, lut, chan)), run(plain, raw)
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
    print("armors:", int(want[2]["valid"].sum()), "with the default table:", int(untouched[2]["valid"].sum()))
    for e in engines:
        assert e.check_padding() == 0
        e.close()


def test_no_allocation_and_cleared_table_restores_the_shift(base_image, weights_seed0):
    import torch
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import _lib, raw_lut as R
    _cuda()
    lib = _lib.lib()
    fmt, chan = irmv.RAW_12, irmv.CH_BAYER_GRBG
    frames = _widen(_bayer_frames(base_image, 2, chan, seed=9), fmt, seed=10)
    l1, l2 = _gamma(fmt), R.make_raw_lut(300, (1.2, 0.9, 2.1), 0.8, bits=12)
    kw = dict(chan_order=chan, max_batch=2, sub_batch=2)
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), raw_format=fmt, **kw)
    fresh = irmv.YoloEngine(weights_seed0, (1280, 1024), raw_format=fmt, **kw)
    ref = irmv.YoloEngine(weights_seed0, (1280, 1024), **kw)
    frames_dev = torch.from_numpy(frames).cuda()
    default = _run(fresh, frames)
    eng.set_raw_lut(l1)
    _run(eng, frames)                                       # warm-up: graphs, rotated view, staging buffers
    eng.detect_batch_device(frames_dev.data_ptr(), 2)
    before = lib.irmv_debug_alloc_count()
    eng.set_raw_lut(l2)
    got = _run(eng, frames)
    got_dev = eng.detect_batch_device(frames_dev.data_ptr(), 2)
    eng.set_raw_lut(l1)
    eng.set_raw_lut(l2)
    eng.detect(0)
    eng.set_raw_lut(None)
    cleared = _run(eng, frames)
    assert lib.irmv_debug_alloc_count() == before, "per-frame calls and table updates must not allocate"
    _assert_same(got, _run(ref, _decode(frames, fmt, l2, chan)), "l2")
    assert got_dev == ref.detect_batch(_decode(frames, fmt, l2, chan))
    _assert_same(cleared, default, "set_raw_lut(None)")
    _assert_same(default, _run(ref, _decode(frames, fmt, None, chan)), "default table")
    eng.set_raw_lut(R.default_raw_lut(12))
    _assert_same(_run(eng, frames), default, "explicit shift table")
    for e in (eng, fresh, ref):
        assert e.check_padding() == 0
        e.close()


def test_rotated_view_survives_a_batch_in_between(base_image, weights_seed0):
    """detect(slot) -> detect_batch(other frames) -> get_rotated_image(slot) is the slot's frame, both on the first
    call (decoded from the device copy of the slot) and once every detect() refreshes the view."""
    import irmv_detection_b200 as irmv
    _cuda()
    fmt, chan = irmv.RAW_12_PACKED, irmv.CH_BAYER_BGGR
    v8 = _bayer_frames(base_image, 4, chan, seed=50)
    frames = _widen(v8, fmt, seed=51)
    lut = _gamma(fmt)
    kw = dict(chan_order=chan, max_batch=2, sub_batch=2)
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), raw_format=fmt, **kw)
    ref = irmv.YoloEngine(weights_seed0, (1280, 1024), **kw)
    eng.set_raw_lut(lut)
    pre = _decode(frames, fmt, lut, chan)
    want = []
    for i in (0, 1):
        ref.get_src_image_buffer(i)[...] = pre[i]
        ref.detect(i)
        want.append(ref.get_rotated_image(i))
    assert not np.array_equal(want[0], want[1])
    eng.get_src_image_buffer(0)[...] = frames[0]
    eng.detect(0)
    eng.detect_batch(frames[2:4])
    assert np.array_equal(eng.get_rotated_image(0), want[0]), "first call after a batch"
    eng.get_src_image_buffer(1)[...] = frames[1]
    eng.detect(1)
    eng.detect_batch(frames[2:4])
    assert np.array_equal(eng.get_rotated_image(1), want[1]), "refreshed by detect()"
    assert np.array_equal(eng.get_rotated_image(0), want[0]), "slot 0 kept its view"
    eng.close(); ref.close()


def test_configuration_and_frame_errors(base_image, weights_seed0):
    import torch
    import irmv_detection_b200 as irmv
    _cuda()
    for bad in (4, -1, 12):
        with pytest.raises(irmv.IrmvError, match="raw_format"):
            irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=irmv.CH_BAYER_RGGB, raw_format=bad)
    for chan in (irmv.CH_PASSTHROUGH, irmv.CH_SWAP_RB):
        with pytest.raises(irmv.IrmvError, match="Bayer"):
            irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=chan, raw_format=irmv.RAW_12)
    with pytest.raises(irmv.IrmvError, match="even"):
        irmv.YoloEngine(weights_seed0, (1281, 1024), chan_order=irmv.CH_BAYER_RGGB, raw_format=irmv.RAW_12_PACKED)
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=irmv.CH_BAYER_RGGB, raw_format=irmv.RAW_12,
                          max_batch=2, sub_batch=2)
    assert eng.get_src_image_buffer(0).dtype == np.uint16 and eng.get_src_image_buffer(0).shape == (1024, 1280)
    for lut in (np.zeros((3, 256), np.uint8), np.zeros((3, 1024), np.uint8), np.zeros((2, 4096), np.uint8),
                np.zeros((3, 4096), np.uint16)):
        with pytest.raises(ValueError):
            eng.set_raw_lut(lut)
    v8 = _bayer_frames(base_image, 2, 2, seed=3)
    frames = _widen(v8, irmv.RAW_12, seed=4)
    for wrong in (v8, frames.astype(np.int32), frames.view(np.uint8), frames[:, :, :640], frames[0]):
        with pytest.raises(ValueError):
            eng.detect_batch(wrong)
        with pytest.raises(ValueError):
            eng.detect_batch_arrays(wrong)
        with pytest.raises(ValueError):
            eng.submit_batch(wrong)
    host = torch.from_numpy(frames).pin_memory().numpy()
    with pytest.raises(ValueError):
        eng.submit_batch(host[:, :, ::-1])                   # not C-contiguous: submit never copies
    t = eng.submit_batch(host)
    with pytest.raises(irmv.IrmvError):
        eng.set_raw_lut(_gamma(irmv.RAW_12))                 # a batch is in flight
    eng.collect_arrays(t)
    eng.set_raw_lut(_gamma(irmv.RAW_12))
    eng.close()
    packed = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=irmv.CH_BAYER_RGGB,
                             raw_format=irmv.RAW_12_PACKED, max_batch=2, sub_batch=2)
    assert packed.get_src_image_buffer(0).dtype == np.uint8 and packed.get_src_image_buffer(0).shape == (1024, 1920)
    with pytest.raises(ValueError):
        packed.detect_batch(frames)                          # u16 frames into a packed engine
    packed.detect_batch(_widen(v8, irmv.RAW_12_PACKED, seed=4))
    assert packed.check_padding() == 0
    packed.close()


def test_kernel_launches_one_more_for_decode(base_image, weights_seed0):
    import irmv_detection_b200 as irmv
    _cuda()
    v8 = _bayer_frames(base_image, 4, 2, seed=60)
    kw = dict(chan_order=irmv.CH_BAYER_RGGB, max_batch=4, sub_batch=2, num_lanes=2)
    e8 = irmv.YoloEngine(weights_seed0, (1280, 1024), **kw)
    e8.detect_batch(v8)
    for fmt in FORMATS.values():
        eb = irmv.YoloEngine(weights_seed0, (1280, 1024), raw_format=fmt, **kw)
        eb.detect_batch(_widen(v8, fmt, seed=61))
        for n in (1, 2, 3, 4):
            replays = (n + 1) // 2
            assert eb.kernel_launches(n) == e8.kernel_launches(n) + replays, (fmt, n)
        eb.close()
    e8.close()
