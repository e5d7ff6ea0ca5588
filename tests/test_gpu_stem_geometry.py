"""The fused stem against the preprocess oracle at every source geometry and on each of its kernel paths.

The engine takes any src_width x src_height >= 2 and sends a frame down one of three paths:
  camera       stem_bayer2x_kernel (csrc/stem_bayer.cu): width 1280, stretch, 8-bit intermediate, 640 <= H <= 4096,
               H / 640 = P / Q with Q <= 16, shared memory within a block's limit, and with a raw table only where
               the table keeps the kernel's CTAs per SM;
  column walk  stem_kernel (csrc/preprocess.cu) with fast_x: Bayer, W % 640 == 0, stretch, everything else;
  sampled      stem_kernel through sample_pixel: every other geometry, letterbox, half-pixel centres.
GEOMETRIES reaches each path and each sizing case of the camera kernel (one or two CTAs per SM, Q from 1 to 16,
H < 640, Q = 64).  Frames are seeded noise (every byte value at every colour site) and rm_test.jpg resampled to the
geometry.  Checks per geometry:
  * the stand-alone preprocess and its rotated view are bit-exact with the oracle (sample_pixel is shared with
    stem_kernel);
  * the fused stem's input, read back through conv0 with the probe weights of oracle/stem_probe.py (all 9 taps x
    3 channels, conv padding included), equals the oracle's 8-bit image (float path: within stem_probe.FLOAT_TOL);
  * conv0 with the seed-0 weights is within the FP64 hop bound of oracle/hop_ref.py, fed with the oracle's input;
  * with a raw table: the probe equals the oracle on raw_lut.apply_raw_lut (8-bit) or raw_lut.decode_raw
    (RAW_12, RAW_12_PACKED) of the frames;
  * boxes map back to source pixels by W / 640, H / 640 or the letterbox inverse;
  * the profiler sees stem_bayer2x_kernel on the camera rows and stem_kernel on the others.
Run with -s for one line per geometry: path, kernel and worst deviation.
"""
import functools
import re

import numpy as np
import pytest

from oracle import stem_probe as SP

pytestmark = pytest.mark.gpu

PATTERN_NAME = {2: "RGGB", 3: "BGGR", 4: "GRBG", 5: "GBRG"}


class Geo:
    def __init__(self, path, W, H, chan, rot, lut=False, **kw):
        self.path, self.W, self.H, self.chan, self.rot, self.lut = path, W, H, chan, rot, lut
        self.kw = kw                                          # letterbox / half_pixel / quantize_u8
        self.quant = kw.get("quantize_u8", True)
        extra = "".join(f"-{k}" for k, v in kw.items() if k != "quantize_u8" and v) + ("-float" if not self.quant else "")
        self.id = f"{W}x{H}-c{chan}{'-rot' if rot else ''}{'-lut' if lut else ''}{extra}"

    @property
    def bayer(self):
        return self.chan >= 2


CAMERA_H = (640, 720, 800, 960, 1024, 1080, 1200, 1280)
GEOMETRIES = (
    # camera kernel: every sizing case (Q = 1 .. 16; 2 CTAs per SM up to 1024 rows, 1 from 1080), the four Bayer
    # patterns and packed RGB / BGR, rot180 on and off
    [Geo("camera", 1280, h, c, r) for h, c, r in zip(CAMERA_H, (0, 2, 3, 4, 5, 1, 2, 5),
                                                         (True, False, True, False, True, False, False, True))]
    # camera-kernel edge cases: the raw table would cost a CTA per SM at 760 rows; packed rows from 3400 on do not
    # fit a block's shared memory.  Both run on stem_kernel's column walk / sampled path instead.
    + [Geo("column", 1280, 760, 3, True, lut=True), Geo("sampled", 1280, 3400, 0, True)]
    # column walk: x scale 3, x scale 1 with vertical upsampling, H < 640, Q = 64, float input
    + [Geo("column", 1920, 1080, 2, True), Geo("column", 1920, 1200, 5, False), Geo("column", 640, 480, 4, True),
       Geo("column", 1280, 600, 3, False), Geo("column", 1280, 1010, 2, True),
       Geo("column", 1280, 1024, 4, True, quantize_u8=False)]
    # sampled: non-integer x scale, odd W and H, upscale on both axes, letterbox, half-pixel centres
    + [Geo("sampled", 1440, 1080, 2, True), Geo("sampled", 2048, 1536, 0, False), Geo("sampled", 1001, 777, 5, True),
       Geo("sampled", 320, 240, 1, True),
       Geo("sampled", 1280, 1024, 2, True, letterbox=True), Geo("sampled", 1440, 1080, 0, True, letterbox=True),
       Geo("sampled", 1920, 1200, 3, False, letterbox=True), Geo("sampled", 640, 480, 1, True, letterbox=True),
       Geo("sampled", 1440, 1080, 4, False, half_pixel=True)]
)
BY_ID = {g.id: g for g in GEOMETRIES}
# the raw table at every camera-kernel height (Bayer patterns cycled); 760 rows is in GEOMETRIES
LUT_CAMERA = [Geo("camera", 1280, h, 2 + i % 4, i % 2 == 0, lut=True) for i, h in enumerate(CAMERA_H)]


def _cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


@pytest.fixture(scope="module")
def probe_weights(tmp_path_factory):
    from irmv_detection_b200 import weights
    paths = []
    for i, taps in enumerate(SP.TAP_FILES):
        tens = weights.random_init(0)
        tens[0] = SP.probe_conv0(taps)
        p = str(tmp_path_factory.mktemp("probe") / f"probe{i}.irmw")
        weights.save(p, tens)
        paths.append(p)
    return paths


def _gamma(bits=8):
    from irmv_detection_b200 import raw_lut as R
    return R.make_raw_lut(8 << (bits - 8), (1.9, 1.0, 1.6), 1 / 2.2, bits=bits)


@pytest.fixture(scope="module")
def frames_of(base_image):
    """g -> u8 [2, H, W] Bayer or [2, H, W, 3] packed: seeded noise, then rm_test.jpg resampled to W x H."""
    from irmv_detection_b200 import synth

    @functools.lru_cache(maxsize=4)
    def make(W, H, chan):
        rng = np.random.default_rng(W * 7919 + H * 31 + chan)
        ys, xs = np.arange(H) * base_image.shape[0] // H, np.arange(W) * base_image.shape[1] // W
        img = base_image[ys][:, xs]
        if chan >= 2:
            return np.stack([rng.integers(0, 256, (H, W), dtype=np.uint8),
                             synth.bayer_from_rgb(img[..., ::-1], PATTERN_NAME[chan])])
        return np.stack([rng.integers(0, 256, (H, W, 3), dtype=np.uint8), img])

    return lambda g: make(g.W, g.H, g.chan)


def _oracle(src, g):
    """The oracle's network input of the frames: FP16 [N, 3, 640, 640]."""
    from oracle import preprocess_ref as PR
    out = []
    for f in src:
        if g.kw.get("letterbox"):
            x, _ = PR.preprocess_letterbox(f, g.chan, g.rot, g.quant)
            out.append(x.astype(np.float16))
        else:
            out.append(PR.preprocess_fp16(f, g.chan, g.rot, g.quant, g.kw.get("half_pixel", False))[0])
    return np.stack(out)


def _engine(irmv, wpath, g, **kw):
    return irmv.YoloEngine(wpath, (g.W, g.H), chan_order=g.chan, rotate180=g.rot, max_batch=2, sub_batch=2,
                           **g.kw, **kw)


def _probe(irmv, probe_weights, g, frames, lut=None, **kw):
    """engine_views() of the probe engines on the frames; `lut` is set on the engines before the batch."""
    m0s = []
    for wp in probe_weights:
        eng = _engine(irmv, wp, g, **kw)
        if lut is not None:
            eng.set_raw_lut(lut)
        eng.detect_batch(frames)
        m0s.append(eng.read_tensor("m0"))
        assert eng.check_padding() == 0
        eng.close()
    return SP.engine_views(m0s)


def _check_probe(got, x, g, what=""):
    if g.quant:
        codes = np.rint(x.astype(np.float64) * 255).astype(np.int64)
        msg = SP.compare_codes(got, codes)
        print(f"{g.id}{what} [{g.path}] probe: {'all 9 taps x 3 channels exact' if msg is None else msg}")
        assert msg is None, f"{g.id}{what}: {msg}"
    else:
        d, at = SP.float_deviation(got, x)
        print(f"{g.id}{what} [{g.path}] probe: max |got - SiLU(x)| {d:.2e} at {at}")
        assert d <= SP.FLOAT_TOL, f"{g.id}{what}: {d:.3g} at {at}"


@pytest.mark.parametrize("gid", list(BY_ID))
def test_standalone_preprocess_and_rotated_view_bit_exact(frames_of, gid):
    import irmv_detection_b200 as irmv
    from oracle import preprocess_ref as PR
    _cuda()
    g = BY_ID[gid]
    src = frames_of(g)
    got, rot = irmv.preprocess(src, g.chan, g.rot, g.quant, want_rotated=True,
                               half_pixel=g.kw.get("half_pixel", False), letterbox=g.kw.get("letterbox", False))
    x = _oracle(src, g)
    for f in range(len(src)):
        assert np.array_equal(got[f, :, :, :3].view(np.uint16), x[f].transpose(1, 2, 0).view(np.uint16)), (gid, f)
        assert not got[f, :, :, 3:].any(), (gid, f)
        img = PR.to_rgb(src[f], g.chan)
        assert np.array_equal(rot[f], PR.rot180(img) if g.rot else img), (gid, f, "rotated view")


@pytest.mark.parametrize("gid", list(BY_ID))
def test_fused_stem_input_all_taps(frames_of, probe_weights, gid):
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import raw_lut as R
    _cuda()
    g = BY_ID[gid]
    src = frames_of(g)
    lut = _gamma() if g.lut else None
    ref_src = np.ascontiguousarray(R.apply_raw_lut(src, lut, g.chan)) if g.lut else src
    _check_probe(_probe(irmv, probe_weights, g, src, lut), _oracle(ref_src, g), g)


@pytest.mark.parametrize("H", CAMERA_H)
def test_raw_table_at_camera_heights(frames_of, probe_weights, H):
    """An 8-bit Bayer engine with a gamma table at every camera-kernel height: it runs (the camera kernel where the
    table keeps its CTAs per SM, stem_kernel elsewhere) and its input equals the oracle on apply_raw_lut(F, L)."""
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import raw_lut as R
    _cuda()
    g = LUT_CAMERA[CAMERA_H.index(H)]
    src = frames_of(g)
    lut = _gamma()
    _check_probe(_probe(irmv, probe_weights, g, src, lut), _oracle(R.apply_raw_lut(src, lut, g.chan), g), g)


@pytest.mark.parametrize("fmt", ["raw12", "raw12_packed"])
def test_raw12_formats_at_1920x1200(frames_of, probe_weights, fmt):
    """12-bit sources (the decode kernel applies the table, then the column walk reads its 8-bit mosaic): the input
    equals the oracle on decode_raw(F, format, L)."""
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import raw_lut as R
    _cuda()
    code = {"raw12": irmv.RAW_12, "raw12_packed": irmv.RAW_12_PACKED}[fmt]
    g = Geo("column", 1920, 1200, 3, True)
    v8 = frames_of(g)
    raw = (v8.astype(np.uint16) << 4) | np.random.default_rng(5).integers(0, 16, v8.shape, dtype=np.uint16)
    frames = np.ascontiguousarray(R.pack_raw12_packed(raw) if code == irmv.RAW_12_PACKED else raw)
    lut = _gamma(12)
    got = _probe(irmv, probe_weights, g, frames, lut, raw_format=code)
    _check_probe(got, _oracle(R.decode_raw(frames, code, lut, g.chan), g), g, f" {fmt}")


@pytest.mark.parametrize("gid", list(BY_ID))
def test_conv0_real_weights_within_hop_bound(frames_of, weights_seed0, gid):
    """conv0 of the seed-0 network after the fused stem against the FP64 hop reference fed with the ORACLE's input
    (the stem's input is exact, so the hop bound of tests/test_gpu_hops.py holds unchanged)."""
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import raw_lut as R
    from oracle import hop_ref as H, yolov8n_ref as Y
    _cuda()
    g = BY_ID[gid]
    src = frames_of(g)
    eng = _engine(irmv, weights_seed0, g)
    lut = _gamma() if g.lut else None
    if lut is not None:
        eng.set_raw_lut(lut)
    eng.detect_batch(src)
    m0 = eng.read_tensor("m0")
    eng.close()
    x = _oracle(np.ascontiguousarray(R.apply_raw_lut(src, lut, g.chan)) if g.lut else src, g)
    ref, mag = H.hop_ref(Y.build(weights_seed0), ("m0", ("input",)), [x.transpose(0, 2, 3, 1)])
    r, at = H.hop_ratio(m0[..., :ref.shape[3]], ref, mag)
    print(f"{gid} [{g.path}] conv0 hop ratio {r:.4f} at {at}")
    assert r <= 1.0, f"{gid}: ratio {r:.3g} at {at}"


@pytest.mark.parametrize("gid", ["1440x1080-c2-rot", "1440x1080-c0-rot-letterbox", "1920x1200-c5"])
def test_boxes_map_back_to_source_pixels(frames_of, weights_seed0, gid):
    """Detections are the engine's decoded boxes at kept_indices mapped from network to source pixels: by W / 640 and
    H / 640 when stretched, by unletterbox_boxes when letterboxed."""
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import _lib as L
    from oracle import preprocess_ref as PR
    _cuda()
    g = BY_ID[gid]
    src = frames_of(g)
    eng = _engine(irmv, weights_seed0, g)
    dets = eng.detect_batch(src)
    boxes = eng.read_tensor("boxes").reshape(len(src), -1, 4)
    assert sum(len(d) for d in dets) > 0
    for f in range(len(src)):
        kept = eng.kept_indices(f)                         # flat anchor * NUM_CLASSES + class
        assert len(dets[f]) == len(kept)
        assert [int(d.class_id) for d in dets[f]] == (kept % L.NUM_CLASSES).tolist(), f"{gid} frame {f}"
        nb = boxes[f, kept // L.NUM_CLASSES].astype(np.float32)
        if g.kw.get("letterbox"):
            want = PR.unletterbox_boxes(nb, g.W, g.H)
        else:
            want = nb * np.array([g.W / 640, g.H / 640, g.W / 640, g.H / 640], np.float32)
        got = np.array([d.xyxy for d in dets[f]], np.float32).reshape(-1, 4)
        np.testing.assert_allclose(got, want, rtol=1e-6, err_msg=f"{gid} frame {f}")
    eng.close()


def test_dispatch_reaches_both_stem_kernels(frames_of, weights_seed0):
    """torch.profiler over one detect_batch per geometry: the camera rows launch stem_bayer2x_kernel, every other row
    (the raw-table and packed edge cases included) stem_kernel.  Column walk versus sampled is a branch inside
    stem_kernel on its fast_x argument and has no runtime observable; the path column of GEOMETRIES names the branch
    the launch's arguments select.  Also: at the camera's 1280 x 1024 the raw table keeps the kernel's two CTAs
    per SM."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    import irmv_detection_b200 as irmv
    _cuda()
    for g in GEOMETRIES + LUT_CAMERA:
        src = frames_of(g)
        eng = _engine(irmv, weights_seed0, g, use_graph=False)
        if g.lut:
            eng.set_raw_lut(_gamma())
        ctas = eng.stem_camera_ctas()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            eng.detect_batch(src)
            torch.cuda.synchronize()
        names = {e.name for e in prof.events() if "stem" in e.name}
        camera = any("stem_bayer2x_kernel" in n for n in names)
        generic = any("stem_kernel<" in n for n in names)
        short = sorted({m.group(0) for n in names for m in [re.search(r"stem_\w+<[^>]*>", n)] if m})
        print(f"{g.id} [{g.path}] {short}, camera kernel CTAs/SM {ctas}")
        assert camera != generic, (g.id, names)
        assert camera == (g.path == "camera"), (g.id, g.path, names)
        assert (ctas > 0) == camera, (g.id, ctas)
        if g.path == "camera" and g.bayer and g.H == 1024:
            assert ctas == 2, (g.id, ctas)
        eng.close()
