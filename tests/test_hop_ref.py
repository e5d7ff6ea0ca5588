"""The one-hop FP64 check (oracle/hop_ref.py) is tight for a faithful implementation and sensitive to subtly
wrong ones.  CPU only: an FP32-accumulate / FP16-store emulation of the engine stands in for the kernels.

The emulation stores FP16 at the engine's points, computes SiLU as h + h * tanh(h) with h = z / 2 in float32
(the tanh.approx form of the kernels) and runs the neck's cv1 over concat(upsample(a), b) the way the default
program does: W_a . a at half resolution rounded to FP16 without bias, upsampled and added before the activation
(conv_raster RES = 2).  Driven through both architectures (YOLOv8n with the keypoint heads, ShuffleNetV2), every
hop must stay at or below a quarter of the tolerance.  Each mutation of the table below models a kernel bug that
shows up as a per-channel, per-row or per-border error; each must exceed the tolerance by 4x on its hop.  Beside
each, the verdict of the old end-to-end gate (2e-2 * max(|ref|, 1) per tap) is recorded: the bias and the
border cases pass it, which is why the one-hop check exists.  No kernel is run or changed here.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import hop_ref as H
from oracle import yolov8n_ref as Y

FAITHFUL_MAX = 0.25
MUTATION_MIN = 4.0


class Emu32(H.Ref64):
    """What the kernels compute: FP32 accumulation, FP16 storage, tanh-form SiLU, split neck conv."""
    dtype = torch.float32
    want_mag = False

    def act(self, z):
        h = z * 0.5
        return h + h * torch.tanh(h)

    def cat_up_conv(self, c, a, b):
        w, bias = self.params(c)
        ca = a.shape[1]
        ya = self.store(self.conv2d(c, a, w[:, :ca], None))
        return self.conv2d(c, b, w[:, ca:], bias) + self.up(ya)


@pytest.fixture(scope="module")
def inputs(base_image):
    """Network inputs as the engine's "input" tap: FP16 NHWC with 8 channels (3 used), rm_test.jpg + one
    synthetic frame."""
    from irmv_detection_b200 import synth
    from oracle import preprocess_ref as PR
    frames = [base_image, synth.frames_from_base(base_image, 1, seed=11)[0]]
    x = np.zeros((2, 640, 640, 8), np.float16)
    for i, f in enumerate(frames):
        x[i, ..., :3] = PR.preprocess_fp16(f)[0].transpose(1, 2, 0)
    return x


@pytest.fixture(scope="module")
def models(tmp_path_factory):
    from irmv_detection_b200 import weights as W
    d = tmp_path_factory.mktemp("hopw")
    py, ps = str(d / "pose_seed0.irmw"), str(d / "shuffle_seed0.irmw")
    W.write_random(py, 0, pose=True)
    W.write_random(ps, 0, arch="shufflenetv2-pose")
    return {"yolov8n": Y.build(py), "shuffle": Y.build(ps)}


class Run:
    """One architecture driven through the emulation: its FP16 taps, and the reference of every hop."""

    def __init__(self, model, x):
        self.model = model
        self.taps = {"input": x}
        self.refs = {}
        with torch.no_grad():
            for hop in H.hops_for(model):
                y, _ = H.evaluate(model, hop, self.ins32(hop), Emu32())
                self.taps[hop[0]] = H.to_nhwc(y.half())

    def ins32(self, hop):
        return [H.to_nchw(self.taps[n], torch.float32) for n in hop[1]]

    def ref(self, hop):
        if hop not in self.refs:
            self.refs[hop] = H.hop_ref(self.model, hop, [self.taps[n] for n in hop[1]])
        return self.refs[hop]


@pytest.fixture(scope="module")
def runs(models, inputs):
    return {k: Run(m, inputs) for k, m in models.items()}


def _all_hops(model):
    hops = H.hops_for(model)
    if not isinstance(model, Y.ShuffleV2Kpt):
        hops = hops + [h for h in H.hops_for(model, fused_tails=True) if h not in hops]
    return hops


@pytest.mark.parametrize("arch", ["yolov8n", "shuffle"])
def test_faithful_emulation_passes_every_hop(runs, arch):
    run = runs[arch]
    worst = []
    for hop in _all_hops(run.model):
        ref, mag = run.ref(hop)
        r, at = H.hop_ratio(run.taps[hop[0]], ref, mag)
        print(f"faithful {arch:8s} {H.hop_label(hop):14s} ratio {r:.4f} at {at}")
        worst.append((r, H.hop_label(hop), at))
    assert len(worst) == (27 if arch == "yolov8n" else 21)
    bad = [w for w in worst if not w[0] <= FAITHFUL_MAX]
    assert not bad, bad


# ------------------------------------------------------------------------------------------- mutations
def _bias(get_conv, ch, tap):
    class M(Emu32):
        def params(self, c):
            w, b = super().params(c)
            if c is get_conv(self.model):
                b = b.clone()
                b[ch] += 0.01 * float(np.abs(self.taps[tap][..., ch].astype(np.float32)).max())
            return w, b
    return M


def _drop_k(get_conv, k0):
    class M(Emu32):
        def params(self, c):
            w, b = super().params(c)
            if c is get_conv(self.model):
                w = w.clone()
                w[:, k0:k0 + 8] = 0
            return w, b
    return M


def _replicate(get_conv, side):
    class M(Emu32):
        def conv2d(self, c, x, w, b):
            if c is not get_conv(self.model):
                return super().conv2d(c, x, w, b)
            xp = F.pad(x, (1, 1, 1, 1))
            if side == "last column":
                xp[..., 1:-1, -1] = x[..., :, -1]
            else:
                xp[..., 0, 1:-1] = x[..., 0, :]
            return F.conv2d(xp, w, b, c.stride, 0, 1, c.groups)
    return M


def _no_residual_last_row():
    class M(Emu32):
        def residual(self, o, r):
            r = r.clone()
            r[..., -1, :] = 0
            return o + r
    return M


def _upsample_off_by_one():
    class M(Emu32):
        def up(self, x):
            W = x.shape[3]
            src = torch.clamp((torch.arange(2 * W) + 1) // 2, max=W - 1)      # (x + 1) / 2 instead of x / 2
            return x.repeat_interleave(2, 2)[..., src]
    return M


def _neighbour_block(get_conv, n0):
    class M(Emu32):
        def params(self, c):
            w, b = super().params(c)
            if c is get_conv(self.model):
                w = w.clone()
                w[n0:n0 + 16] = w[n0 - 16:n0]
            return w, b
    return M


def _dw_transposed(get_conv):
    class M(Emu32):
        def params(self, c):
            w, b = super().params(c)
            if c is get_conv(self.model):
                w = w.transpose(2, 3).contiguous()
            return w, b
    return M


def _swap(a, b):
    def post(y):
        y = y.copy()
        y[..., [a, b]] = y[..., [b, a]]
        return y
    return post


# (id, arch, hop, emulation class, post-processing of the hop output or None, the old gate must pass it)
MUTATIONS = [
    ("bias_ch7_plus_1pct", "yolov8n", ("m2", ("m1",)), _bias(lambda m: m.m2.cv2.conv, 7, "m2"), None, True),
    ("drop_k_group_40", "yolov8n", ("m6", ("m5",)), _drop_k(lambda m: m.m6.cv2.conv, 40), None, False),
    ("replicate_last_column", "yolov8n", ("box0", ("m15",)), _replicate(lambda m: m.box[0][0].conv, "last column"),
     None, True),
    ("replicate_first_row", "yolov8n", ("m16", ("m15",)), _replicate(lambda m: m.m16.conv, "first row"), None, True),
    ("no_residual_last_row", "yolov8n", ("m4", ("m3",)), _no_residual_last_row(), None, False),
    ("upsample_src_off_by_one_column", "yolov8n", ("m15", ("m12", "m4")), _upsample_off_by_one(), None, False),
    ("neighbour_weights_block_16", "yolov8n", ("m8", ("m7",)), _neighbour_block(lambda m: m.m8.cv2.conv, 16), None,
     False),
    ("dw_kernel_transposed", "shuffle", ("d2", ("d1",)), _dw_transposed(lambda m: m.stages[1][1].dw.conv), None,
     False),
    ("stage_map_channels_swapped", "shuffle", ("d3", ("d2",)), Emu32, _swap(5, 70), False),
]


@pytest.mark.parametrize("name,arch,hop,emu,post,old_must_pass", MUTATIONS, ids=[m[0] for m in MUTATIONS])
def test_mutation_is_caught(runs, name, arch, hop, emu, post, old_must_pass):
    run = runs[arch]
    A = emu()
    A.model, A.taps = run.model, run.taps
    with torch.no_grad():
        y, _ = H.evaluate(run.model, hop, run.ins32(hop), A)
    got = H.to_nhwc(y.half())
    if post is not None:
        got = post(got)
    ref, mag = run.ref(hop)
    r, at = H.hop_ratio(got, ref, mag)
    old = H.old_gate_passes(got, ref)
    print(f"mutation {name:32s} {H.hop_label(hop):12s} ratio {r:9.2f} at {at}  old 2e-2 gate: "
          f"{'passes' if old else 'fails'}")
    assert r >= MUTATION_MIN, (name, r, at)
    if old_must_pass:
        assert old, f"{name}: the old gate was expected to miss this mutation"


def test_hop_ratio_reports_the_location():
    """A single wrong element is reported at its frame, row, column and channel, and NaN counts as a failure."""
    rng = np.random.default_rng(3)
    ref = rng.standard_normal((2, 5, 6, 16))
    mag = np.abs(ref) * 4 + 1
    got = ref.astype(np.float16)
    r0, _ = H.hop_ratio(got, ref, mag)
    assert r0 <= 0.5                                  # the final FP16 rounding is half an ulp
    got[1, 3, 5, 11] += np.float16(0.5)
    r, at = H.hop_ratio(got, ref, mag)
    assert r > 1 and at == {"frame": 1, "channel": 11, "y": 3, "x": 5}
    got[0, 0, 0, 0] = np.float16(np.nan)
    r, at = H.hop_ratio(got, ref, mag)
    assert r == np.inf and at == {"frame": 0, "channel": 0, "y": 0, "x": 0}
    with pytest.raises(ValueError):
        H.hop_ratio(got[..., :14], ref, mag)


def test_ulp16_matches_numpy_spacing():
    v = np.array([1.0, 1.5, 2.0, 1e-3, 6e-5, 3e-6, 0.0, -7.25, 1000.0])
    assert np.array_equal(H.ulp16(v), np.abs(np.spacing(np.abs(v).astype(np.float16))).astype(np.float64))
