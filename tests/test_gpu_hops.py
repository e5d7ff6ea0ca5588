"""Every network module of every engine program, one hop at a time, against the FP64 reference of
oracle/hop_ref.py fed with the engine's own FP16 input taps.

test_network_parity bounds each module tap end to end by 2e-2 * max(|ref|, 1): enough room for 20 modules of
FP16 drift, and enough to hide a kernel that zeroes a tenth of a tap's channels or gets one border wrong.  Here
each hop must satisfy max |got - ref| / (2^-8 * mag + ulp16(|ref|)) <= 1, where mag = conv(|x|, |W|) + |b| of
the module's last conv (tests/test_hop_ref.py: a faithful FP32-accumulate emulation uses at most a quarter of
that; per-channel, per-row and per-border mutations exceed it by 4x or more).  The programs cover every
conv kernel and its instantiations: the direct kernel, tcgen05 with and without fused tails, the gather neck,
batch 1 (output-channel split, branched schedule, small-replay plan), a 64-frame replay (other plan()
instantiations), the camera-case Bayer stem, the keypoint heads and both ShuffleNetV2 unit paths.

One line per hop: `program hop max_ratio at (frame, channel, y, x)`; run with -s to see the margins.
"""
import numpy as np
import pytest

from oracle import hop_ref as H

pytestmark = pytest.mark.gpu


def _cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


@pytest.fixture(scope="module")
def frames(base_image):
    from irmv_detection_b200 import synth
    _cuda()
    rnd = np.random.default_rng(0).integers(0, 256, base_image.shape, dtype=np.uint8)
    syn = synth.frames_from_base(base_image, 2, seed=11)
    return np.stack([base_image, rnd, syn[0], syn[1]])


@pytest.fixture(scope="module")
def weights_shuffle(tmp_path_factory):
    from irmv_detection_b200 import weights as W
    p = tmp_path_factory.mktemp("ws") / "shufflenetv2_pose_seed0.irmw"
    W.write_random(str(p), 0, arch="shufflenetv2-pose")
    return str(p)


@pytest.fixture(scope="module")
def weights_pose(tmp_path_factory):
    from irmv_detection_b200 import weights as W
    p = tmp_path_factory.mktemp("wp") / "pose_seed0.irmw"
    W.write_random(str(p), 0, pose=True)
    return str(p)


# program -> (weight file, engine keyword arguments, how frames are run, m1 / m3 fused into their consumers)
PROGRAMS = {
    "direct": ("yolo", {"conv_impl": "direct"}, "batch4", False),
    "tcgen05": ("yolo", {}, "batch4", True),
    "tcgen05_unfused": ("yolo", {"fuse_tails": False}, "batch4", False),
    "tcgen05_gather_neck": ("yolo", {"split_upsample_convs": False}, "batch4", True),
    "batch1": ("yolo", {}, "batch1", True),
    "batch64": ("yolo", {}, "batch64", True),
    "bayer_rggb": ("yolo", {"chan_order": "rggb"}, "batch4", True),
    "pose": ("pose", {}, "batch4", True),
    "shuffle_fused_units": ("shuffle", {"fuse_units": True}, "batch4", False),
    "shuffle_per_conv": ("shuffle", {"fuse_units": False}, "batch4", False),
}
B64_FRAMES = (0, 31, 63)


def _run_program(irmv, wpath, kw, mode, frames, base_image, names):
    """Run the engine; return (frame ids, network input FP16 NHWC, {tap: FP16 NHWC} for those frames)."""
    from irmv_detection_b200 import synth
    kw = dict(kw)
    if kw.get("conv_impl") == "direct":
        kw["conv_impl"] = irmv.CONV_DIRECT
    chan = irmv.CH_PASSTHROUGH
    src = frames
    if kw.get("chan_order") == "rggb":
        chan = kw["chan_order"] = irmv.CH_BAYER_RGGB
        src = synth.bayer_from_rgb(frames[..., ::-1], "RGGB")
    taps = {}
    if mode == "batch4":
        eng = irmv.YoloEngine(wpath, (1280, 1024), max_batch=4, sub_batch=4, **kw)
        eng.detect_batch(src)
        taps = {n: eng.read_tensor(n) for n in names}
        ids = list(range(len(src)))
    elif mode == "batch1":
        eng = irmv.YoloEngine(wpath, (1280, 1024), **kw)
        per = []
        for f in range(len(src)):
            eng.detect_batch(src[f:f + 1])
            per.append({n: eng.read_tensor(n) for n in names})
        taps = {n: np.concatenate([p[n] for p in per]) for n in names}
        ids = list(range(len(src)))
    else:
        fr = synth.frames_from_base(base_image, 64, seed=29)
        fr[list(B64_FRAMES)] = src[:3]
        src = fr
        eng = irmv.YoloEngine(wpath, (1280, 1024), max_batch=64, sub_batch=64, num_lanes=1, **kw)
        eng.detect_batch(src)
        for n in names:                                   # one tap at a time: 64 frames of m0 are 210 MB
            t = eng.read_tensor(n)
            assert t.shape[0] == 64, n
            taps[n] = t[list(B64_FRAMES)].copy()
            del t
        ids = list(B64_FRAMES)
        src = src[list(B64_FRAMES)]
    eng.close()
    return ids, irmv.preprocess(src, chan), taps


@pytest.mark.parametrize("program", list(PROGRAMS))
def test_every_hop_within_fp64_bound(frames, base_image, weights_seed0, weights_pose, weights_shuffle, program):
    import irmv_detection_b200 as irmv
    from oracle import yolov8n_ref as Y
    _cuda()
    which, kw, mode, fused = PROGRAMS[program]
    wpath = {"yolo": weights_seed0, "pose": weights_pose, "shuffle": weights_shuffle}[which]
    model = Y.build(wpath)
    hops = H.hops_for(model, fused_tails=fused)
    names = sorted({n for out, ins in hops for n in (out,) + ins} - {"input"})
    ids, x, taps = _run_program(irmv, wpath, kw, mode, frames, base_image, names)
    taps["input"] = x
    bad = []
    for hop in hops:
        ref, mag = H.hop_ref(model, hop, [taps[n] for n in hop[1]])
        got = taps[hop[0]]
        assert got.shape[:3] == ref.shape[:3] and got.shape[3] >= ref.shape[3], (hop, got.shape, ref.shape)
        if got.shape[3] > ref.shape[3]:
            assert hop[0][:3] in ("cls", "kpt"), hop     # padded head planes (test_activation_padding_stays_zero)
        r, at = H.hop_ratio(got[..., :ref.shape[3]], ref, mag)
        where = (ids[at["frame"]], at["channel"], at["y"], at["x"])
        print(f"{program} {H.hop_label(hop)} {r:.4f} at {where}")
        if not r <= 1.0:
            bad.append(f"{H.hop_label(hop)}: ratio {r:.3g} at (frame, channel, y, x) = {where}")
    assert not bad, f"{program}: " + "; ".join(bad)
