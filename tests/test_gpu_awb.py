"""Automatic white balance (YoloEngine.set_auto_white_balance).  Every test rests on one identity: the engine with AWB
on, user matrix M and tone T returns on a batch of Bayer frames F_i, bit for bit, what the same engine with AWB off
returns on each F_i alone after set_color_matrix(awb_matrix(g_i, M), T), g_i = the oracle's gains of F_i
(raw_lut.awb_statistics / awb_gains); and the records fetch_white_balance returns equal raw_lut.awb_record exactly.
Each frame gets its own seeded colour cast, so the gains differ inside a batch."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PATTERN_NAME = {2: "RGGB", 3: "BGGR", 4: "GRBG", 5: "GBRG"}
PATHS = {"camera": ((1280, 1024), {}), "generic": ((1920, 1200), {}), "generic760": ((1280, 760), {}),
         "unfused": ((1280, 1024), {"fused_stem": False})}


def _cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _lut():
    from irmv_detection_b200 import raw_lut as R
    return R.make_raw_lut(8, (1.0, 1.0, 1.0), 1.0)              # black level only: AWB does the gains


def _matrix():
    from irmv_detection_b200 import raw_lut as R
    return R.color_matrix_q10(np.array([[1.55, -0.35, -0.20], [-0.25, 1.45, -0.20], [-0.05, -0.45, 1.50]]), 1.3)


def _tone():
    from irmv_detection_b200 import raw_lut as R
    return R.make_raw_lut(0, (1, 1, 1), 1 / 2.2)


def _cast_rgb(base_image, n, seed, w, h):
    """n RGB frames, each under its own colour cast (channel gains 0.55 .. 1.0)."""
    from irmv_detection_b200 import synth
    rgb = synth.frames_from_base(base_image, n, seed=seed)[..., ::-1]
    if (w, h) != (rgb.shape[2], rgb.shape[1]):
        ys, xs = np.arange(h) * rgb.shape[1] // h, np.arange(w) * rgb.shape[2] // w
        rgb = rgb[:, ys][:, :, xs]
    gains = np.random.default_rng(seed).uniform(0.55, 1.0, (n, 1, 1, 3))
    return np.clip(rgb * gains + 0.5, 0, 255).astype(np.uint8)


def _bayer(rgb, chan):
    from irmv_detection_b200 import synth
    return np.ascontiguousarray(synth.bayer_from_rgb(rgb, PATTERN_NAME[chan]))


def _records(mosaics, chan, params=None):
    from irmv_detection_b200 import raw_lut as R
    return [R.awb_record(m, chan, params) for m in mosaics]


def _assert_records(got, want, what=""):
    assert len(got) >= len(want)
    for f, w in enumerate(want):
        g = got[f]
        assert tuple(int(v) for v in g["sum"]) == w["sum"], f"{what} frame {f} sums"
        assert (int(g["counted"]), int(g["dark"]), int(g["clipped"])) == (w["counted"], w["dark"], w["clipped"]), \
            f"{what} frame {f} quads"
        assert int(g["valid"]) == w["valid"] and tuple(int(v) for v in g["gain_q10"]) == w["gain_q10"], \
            f"{what} frame {f} gains"


def _same_bits(a, b):
    return a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()


def _lock(ref, rec, m, tone):
    from irmv_detection_b200 import raw_lut as R
    ref.set_color_matrix(R.awb_matrix(rec["gain_q10"], m), tone)


def _compare_batch(eng, ref, frames, want_recs, m, tone, read_input=False, what=""):
    """eng (AWB on) on the whole batch against ref (AWB off) on each frame alone with the locked matrix."""
    counts, dets = eng.detect_batch_arrays(frames)
    counts, dets = counts.copy(), dets.copy()
    kept = [eng.kept_indices(f) for f in range(len(frames))]
    x = eng.read_tensor("input") if read_input else None
    _assert_records(eng.fetch_white_balance(len(frames)), want_recs, what)
    for f, rec in enumerate(want_recs):
        _lock(ref, rec, m, tone)
        c1, d1 = ref.detect_batch_arrays(frames[f:f + 1])
        k = int(c1[0])
        assert int(counts[f]) == k, f"{what} frame {f}: count"
        assert np.array_equal(dets[f, :k], d1[0, :k]), f"{what} frame {f}: detections"
        assert np.array_equal(kept[f], ref.kept_indices(0)), f"{what} frame {f}: kept indices"
        if read_input:
            assert _same_bits(x[f], ref.read_tensor("input")[0]), f"{what} frame {f}: network input"
    # detect(0) and the rotated view of frame 0
    eng.get_src_image_buffer(0)[...] = frames[0]
    ref.get_src_image_buffer(0)[...] = frames[0]
    _lock(ref, want_recs[0], m, tone)
    assert eng.detect(0) == ref.detect(0), f"{what} detect(0)"
    assert np.array_equal(eng.get_rotated_image(0), ref.get_rotated_image(0)), f"{what} rotated view"
    _assert_records(eng.fetch_white_balance(1), want_recs[:1], what + " detect(0)")
    return int(counts.sum())


CASES = [("camera", 2, True, "lut+mt"), ("camera", 3, False, "plain"), ("camera", 4, True, "mt"),
         ("camera", 5, False, "lut"), ("camera", 2, False, "plain"), ("camera", 5, True, "lut+mt"),
         ("generic", 2, True, "lut+mt"), ("generic", 4, False, "plain"),
         ("generic760", 3, True, "mt"), ("generic760", 5, False, "lut"),
         ("unfused", 2, True, "mt"), ("unfused", 3, False, "lut+mt"), ("unfused", 4, True, "plain")]


@pytest.mark.parametrize("path,chan,rotate,stages", CASES)
def test_awb_equals_locked_matrix_per_frame(base_image, weights_seed0, path, chan, rotate, stages):
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import raw_lut as R
    _cuda()
    (w, h), extra = PATHS[path]
    lut = _lut() if "lut" in stages else None
    m, tone = (_matrix(), _tone()) if "mt" in stages else (None, None)
    frames = _bayer(_cast_rgb(base_image, 3, 100 + chan + 10 * rotate, w, h), chan)
    kw = dict(chan_order=chan, rotate180=rotate, max_batch=3, sub_batch=3, **extra)
    eng = irmv.YoloEngine(weights_seed0, (w, h), **kw)
    ref = irmv.YoloEngine(weights_seed0, (w, h), **kw)
    for e in (eng, ref):
        if lut is not None:
            e.set_raw_lut(lut)
    if m is not None:
        eng.set_color_matrix(m, tone)
    eng.set_auto_white_balance({})
    want = _records(frames if lut is None else R.apply_raw_lut(frames, lut, chan), chan)
    assert all(r["valid"] for r in want) and len({r["gain_q10"] for r in want}) == 3, "casts must give distinct gains"
    _compare_batch(eng, ref, frames, want, m, tone, read_input=path == "unfused", what=f"{path} {chan} {rotate}")
    assert np.array_equal(eng.get_src_image_buffer(0), frames[0]), "the pinned slot must keep the raw frame"
    assert eng.check_padding() == 0 and ref.check_padding() == 0
    eng.close(); ref.close()


@pytest.mark.parametrize("fmt", [2, 3])                     # RAW_12, RAW_12_PACKED
def test_wide_formats_measure_the_decoded_mosaic(base_image, weights_seed0, fmt):
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import raw_lut as R
    _cuda()
    chan = irmv.CH_BAYER_GBRG
    v8 = _bayer(_cast_rgb(base_image, 3, 40 + fmt, 1280, 1024), chan)
    rng = np.random.default_rng(fmt)
    wide = (v8.astype(np.uint16) << 4) | rng.integers(0, 16, v8.shape, dtype=np.uint16)
    frames = np.ascontiguousarray(R.pack_raw12_packed(wide) if fmt == irmv.RAW_12_PACKED else wide)
    dlut = R.make_raw_lut(64, (1, 1, 1), 1.0, bits=12)
    m, tone = _matrix(), _tone()
    kw = dict(chan_order=chan, raw_format=fmt, max_batch=3, sub_batch=3)
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), **kw)
    ref = irmv.YoloEngine(weights_seed0, (1280, 1024), **kw)
    for e in (eng, ref):
        e.set_raw_lut(dlut)
    eng.set_color_matrix(m, tone)
    eng.set_auto_white_balance({"dark_level": 4, "clip_level": 240})
    prm = {"dark_level": 4, "clip_level": 240}
    want = _records(R.decode_raw(frames, fmt, dlut, chan), chan, prm)
    assert len({r["gain_q10"] for r in want}) == 3
    _compare_batch(eng, ref, frames, want, m, tone, what=f"fmt {fmt}")
    assert eng.check_padding() == 0 and ref.check_padding() == 0
    eng.close(); ref.close()


def test_bench_shape_device_and_pipelined_host(base_image, weights_seed0):
    """256 device-resident 1280 x 1024 RGGB frames in one replay with fused PnP, and the pipelined host path
    (128-frame chunks): detections, poses and records equal a batch-1 engine's, frame by frame."""
    import torch
    import irmv_detection_b200 as irmv
    from oracle import pnp_ref as P
    _cuda()
    chan = irmv.CH_BAYER_RGGB
    raw16 = _bayer(_cast_rgb(base_image, 16, 7, 1280, 1024), chan)
    raw = np.ascontiguousarray(np.tile(raw16, (16, 1, 1)))
    m, tone = _matrix(), _tone()
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=chan, max_batch=256)
    one = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=chan, max_batch=1)
    for e in (eng, one):
        e.enable_pnp(P.K_DEFAULT, P.D_DEFAULT, (0.5, 480 / 1024))
        e.set_color_matrix(m, tone)
        e.set_auto_white_balance({})
    assert eng.stem_camera_ctas() == 2, "AWB must keep the camera stem at two CTAs per SM at 1024 rows"
    want16 = _records(raw16, chan)
    assert len({r["gain_q10"] for r in want16}) == 16
    per_frame = []
    for f in range(16):
        c, d = one.detect_batch_arrays(raw16[f:f + 1])
        rv, tv, ok = one.fetch_poses(1)
        per_frame.append((int(c[0]), d[0].copy(), rv.copy(), tv.copy(), one.fetch(1)[0]))
        _assert_records(one.fetch_white_balance(1), want16[f:f + 1], f"batch-1 frame {f}")
    want = [per_frame[f % 16] for f in range(256)]
    assert sum(p[0] for p in per_frame) > 0

    raw_dev = torch.from_numpy(raw).cuda()
    eng.detect_batch_device(raw_dev.data_ptr(), 256)
    got = eng.detect_batch_device(raw_dev.data_ptr(), 256)        # (a second replay of the captured graph)
    recs = eng.fetch_white_balance(256)
    _assert_records(recs, [want16[f % 16] for f in range(256)], "device batch")
    rv, tv, ok = eng.fetch_poses(256)
    for f in range(256):
        k = want[f][0]
        assert got[f] == want[f][4], f"device frame {f}"
        assert np.array_equal(rv[f, :k], want[f][2][0, :k]) and np.array_equal(tv[f, :k], want[f][3][0, :k])
    pin = torch.from_numpy(raw).pin_memory().numpy()
    t = eng.submit_batch(pin)
    cg, dg, rvg, tvg, okg = eng.collect_arrays(t, poses=True)
    cg, dg, rvg, tvg = cg.copy(), dg.copy(), rvg.copy(), tvg.copy()
    _assert_records(eng.fetch_white_balance(256, t), [want16[f % 16] for f in range(256)], "pipelined")
    for f in range(256):
        k = want[f][0]
        assert int(cg[f]) == k and np.array_equal(dg[f, :k], want[f][1][:k]), f"pipelined frame {f}"
        assert np.array_equal(rvg[f, :k], want[f][2][0, :k]) and np.array_equal(tvg[f, :k], want[f][3][0, :k])
    assert torch.equal(raw_dev.cpu(), torch.from_numpy(raw)) and np.array_equal(pin, raw), "frames must stay raw"
    assert eng.check_padding() == 0 and one.check_padding() == 0
    eng.close(); one.close()


@pytest.mark.parametrize("chan,rotate", [(2, True), (5, False)])
def test_fused_armors_and_poses(weights_seed0, chan, rotate):
    """The armor stage's result for a frame can depend on the other frames of its batch and on earlier calls (found with
    100 random-init detections a frame: the same frame and matrix give different armors at batch 1 and batch 3 without
    AWB), so both engines here see the same sequence of calls: each frame alone, then each frame three times in one
    batch (the per-frame block of frames 1 and 2 is then staged by index)."""
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import synth
    from oracle import pnp_ref as P, preprocess_ref as PR
    _cuda()
    rng = np.random.default_rng(chan)
    scenes = [synth.armor_scene(10, s)[0] for s in (7, 8, 9)]
    cast = [np.clip(s * rng.uniform(0.6, 1.0, 3) + 0.5, 0, 255).astype(np.uint8) for s in scenes]
    cam = [PR.rot180(s) if rotate else s for s in cast]
    raw = _bayer(np.stack(cam), chan)
    m, tone = _matrix(), _tone()
    prm = dict(light_min_ratio=0.01, light_max_ratio=10.0, light_max_angle=90.0, min_small_center_distance=0.0,
               max_large_center_distance=1e9)
    awb = {"min_quads": 64}
    engines = []
    for _ in range(2):
        e = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=chan, rotate180=rotate, max_batch=3)
        e.enable_armors(**prm)
        e.enable_pnp(P.K_DEFAULT, P.D_DEFAULT, (0.5, 480 / 1024))
        engines.append(e)
    eng, ref = engines
    eng.set_color_matrix(m, tone)
    eng.set_auto_white_balance(awb)
    want = _records(raw, chan, awb)
    assert all(r["valid"] for r in want) and len({r["gain_q10"] for r in want}) == 3

    def run(e, frames):
        c, d = e.detect_batch_arrays(frames)
        return c.copy(), d.copy(), e.fetch_armors(len(frames)), e.fetch_armor_poses(len(frames))

    valid = 0
    for batch in ([f] for f in range(3)), ([f] * 3 for f in range(3)):
        for idx in batch:
            f = idx[0]
            frames = np.ascontiguousarray(raw[idx])
            got = run(eng, frames)
            _assert_records(eng.fetch_white_balance(len(idx)), [want[f]] * len(idx), f"frames {idx}")
            _lock(ref, want[f], m, tone)
            exp = run(ref, frames)
            assert np.array_equal(got[0], exp[0]) and int(exp[0].sum()) > 0, f"frames {idx}: counts"
            for i, k in enumerate(exp[0]):
                assert np.array_equal(got[1][i, :k], exp[1][i, :k]), f"frames {idx}: detections"
            assert _same_bits(got[2], exp[2]), f"frames {idx}: armors"
            assert _same_bits(got[3], exp[3]), f"frames {idx}: armor poses"
            valid += int(exp[2]["valid"].sum())
    print("armors:", valid)
    assert valid > 0
    for e in engines:
        assert e.check_padding() == 0
        e.close()


def test_clipped_frame_falls_back_to_the_user_matrix(base_image, weights_seed0):
    import irmv_detection_b200 as irmv
    _cuda()
    chan = irmv.CH_BAYER_BGGR
    frames = _bayer(_cast_rgb(base_image, 2, 3, 1280, 1024), chan)
    frames[1] = np.maximum(frames[1], 251)                    # every quad clipped
    m, tone = _matrix(), _tone()
    kw = dict(chan_order=chan, max_batch=2, sub_batch=2)
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), **kw)
    ref = irmv.YoloEngine(weights_seed0, (1280, 1024), **kw)
    eng.set_color_matrix(m, tone)
    ref.set_color_matrix(m, tone)
    eng.set_auto_white_balance({})
    want = _records(frames, chan)
    assert want[0]["valid"] == 1 and want[1]["valid"] == 0 and want[1]["gain_q10"] == (1024, 1024, 1024)
    assert want[1]["clipped"] == 512 * 640
    counts, dets = eng.detect_batch_arrays(frames)
    _assert_records(eng.fetch_white_balance(2), want)
    c1, d1 = ref.detect_batch_arrays(frames[1:])
    k = int(c1[0])
    assert int(counts[1]) == k and np.array_equal(dets[1, :k], d1[0, :k])
    eng.close(); ref.close()


def test_off_on_off_and_updates_in_place(base_image, weights_seed0):
    import torch
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import _lib, raw_lut as R
    _cuda()
    lib = _lib.lib()
    chan = irmv.CH_BAYER_GRBG
    frames = _bayer(_cast_rgb(base_image, 2, 11, 1280, 1024), chan)
    kw = dict(chan_order=chan, max_batch=2, sub_batch=2)
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), **kw)
    never = irmv.YoloEngine(weights_seed0, (1280, 1024), **kw)
    dev = torch.from_numpy(frames).cuda()
    plain = never.detect_batch_device(dev.data_ptr(), 2)
    assert eng.detect_batch_device(dev.data_ptr(), 2) == plain
    eng.set_auto_white_balance({})
    on = eng.detect_batch_device(dev.data_ptr(), 2)
    _assert_records(eng.fetch_white_balance(2), _records(frames, chan))
    eng.set_auto_white_balance(None)
    assert eng.detect_batch_device(dev.data_ptr(), 2) == plain, "off again equals never on"
    with pytest.raises(irmv.IrmvError):
        eng.fetch_white_balance(2)                             # the stage is off
    before = lib.irmv_debug_alloc_count()
    eng.set_auto_white_balance({})
    assert eng.detect_batch_device(dev.data_ptr(), 2) == on
    # in-place updates: parameters and the user's matrix, no allocation, results follow
    prm = {"gain_max_q10": 1100, "dark_level": 20}
    eng.set_auto_white_balance(prm)
    got = eng.detect_batch_device(dev.data_ptr(), 2)
    want = _records(frames, chan, prm)
    _assert_records(eng.fetch_white_balance(2), want, "updated parameters")
    assert max(max(r["gain_q10"]) for r in want) == 1100, "the update must reach the gain clamp"
    assert lib.irmv_debug_alloc_count() == before, "off -> on and parameter updates must not allocate"
    m, tone = _matrix(), _tone()
    eng.set_color_matrix(m, tone)                              # (the first matrix allocates its block)
    before = lib.irmv_debug_alloc_count()
    eng.set_color_matrix(R.color_matrix_q10(saturation=0.5), None)
    got_m = eng.detect_batch_device(dev.data_ptr(), 2)
    eng.get_src_image_buffer(0)[...] = frames[0]
    eng.detect(0)
    assert lib.irmv_debug_alloc_count() == before, "matrix updates under AWB and detects must not allocate"
    for f, ds in enumerate((got, got_m)):
        mm, tt = (None, None) if f == 0 else (R.color_matrix_q10(saturation=0.5), None)
        for i in range(2):
            never.set_color_matrix(R.awb_matrix(want[i]["gain_q10"], mm), tt)
            assert never.detect_batch(frames[i:i + 1])[0] == ds[i], f"update {f} frame {i}"
    assert eng.check_padding() == 0 and never.check_padding() == 0
    eng.close(); never.close()


def test_errors(base_image, weights_seed0):
    import ctypes as C
    import torch
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import _lib
    _cuda()
    lib = _lib.lib()
    for chan in (irmv.CH_PASSTHROUGH, irmv.CH_SWAP_RB):
        rgb = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=chan, max_batch=1)
        with pytest.raises(irmv.IrmvError):
            rgb.set_auto_white_balance({})
        with pytest.raises(irmv.IrmvError):
            rgb.set_auto_white_balance(None)
        rgb.close()
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=irmv.CH_BAYER_RGGB, max_batch=2, sub_batch=2)
    frames = _bayer(_cast_rgb(base_image, 2, 5, 1280, 1024), 2)
    eng.detect_batch(frames)
    with pytest.raises(irmv.IrmvError):
        eng.fetch_white_balance(2)                             # never enabled
    for bad in ((-1, 250, 1, 4096), (9, 8, 1, 4096), (8, 256, 1, 4096), (8, 250, 0, 4096), (8, 250, 1, 1023),
                (8, 250, 1, 32768)):
        p = _lib.AwbParams(*bad)
        assert lib.irmv_engine_set_auto_white_balance(eng._h, C.byref(p)) == 1, bad
        with pytest.raises(ValueError):
            eng.set_auto_white_balance(dict(zip(("dark_level", "clip_level", "min_quads", "gain_max_q10"), bad)))
    eng.set_auto_white_balance({})
    with pytest.raises(irmv.IrmvError):
        eng.fetch_white_balance(2)                             # the last call ran without the stage
    host = torch.from_numpy(frames).pin_memory().numpy()
    t = eng.submit_batch(host)
    with pytest.raises(irmv.IrmvError):
        eng.set_auto_white_balance({"min_quads": 10})         # a batch is in flight
    with pytest.raises(irmv.IrmvError):
        eng.fetch_white_balance(2, t)                          # not collected yet
    eng.collect_arrays(t)
    _assert_records(eng.fetch_white_balance(2, t), _records(frames, 2))
    with pytest.raises(irmv.IrmvError):
        eng.fetch_white_balance(0)
    assert lib.irmv_engine_fetch_white_balance(eng._h, t, 2, None) != 0
    assert eng.check_padding() == 0
    eng.close()
