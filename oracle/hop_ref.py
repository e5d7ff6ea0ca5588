"""TEST INFRASTRUCTURE ONLY -- one-hop FP64 reference of every network module.

The end-to-end network check (tests/test_gpu_parity.py::test_network_parity) runs the FP32 oracle from the
input frame and bounds each module tap by 2e-2 * max(|ref|, 1).  After 20 modules that bound has to absorb the
FP16 drift of everything upstream, and because it scales with the tap's absolute maximum it cannot see an error
confined to one channel, one border or one row.  A hop instead starts from the engine's own FP16 input tensors
(exactly as YoloEngine.read_tensor returns them) and computes ONE module in float64, rounding to FP16 exactly
where the engine stores FP16 inside the module:

  C2f       the cv1 output, each bottleneck's cv1 output, each bottleneck's output after the residual add
            (the residual joins the FP32 accumulator before a single rounding: conv_raster.cu epi_chunk);
  SPPF      the cv1 output (the max pools are exact);
  heads     the two intermediate 3x3 outputs of the box / cls / keypoint towers;
  ShuffleNetV2 units  the pw1 output, the depthwise output, the pw2 output (shuffle_unit.cu rounds the
            depthwise accumulator to FP16 before the second 1x1; the per-conv path stores T1 / T2 / Ta / Tb / Tc).

What is left between a faithful kernel and this reference is FP32 accumulation order, tanh.approx in SiLU, the
final FP16 rounding and the occasional one-ulp flip of an intermediate rounding.  All of it is bounded by the
natural scale of the module's last dot product, mag = conv(|x|, |W|) + |b| of its last conv on the reference's
own rounded input, so the per-element tolerance is

    tol = 2^-8 * mag + ulp16(|ref|)

and hop_ratio() = max |got - ref| / tol.  The weights and the architecture come from oracle/yolov8n_ref.py
(Y.build), so there is one source for both.

The module arithmetic is written against an `Arith` object (Ref64 here).  tests/test_hop_ref.py derives an
FP32 / FP16-storage emulation of the engine from it and mutates that emulation to show the check is tight for a
faithful implementation and fails for subtly wrong ones.

Only tests/ may import this module.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle import yolov8n_ref as Y

TOL_REL = 2.0 ** -8

Hop = Tuple[str, Tuple[str, ...]]        # (output tap, input taps)

# modules whose first input is upsampled (nearest x2) before the concat, as yolov8n_ref.features does it
_UP_FIRST = ("m12", "m15")
# fused-tail program: m1 / m3 are consumed inside the next module's launch and never materialised
_FUSED_CHAIN = {("m2", ("m0",)): ("m1", "m2"), ("m4", ("m2",)): ("m3", "m4")}


def yolo_hops(pose: bool = False, fused_tails: bool = False) -> List[Hop]:
    """Hops of the YOLOv8n program.  fused_tails: m1 and m3 are not taps, so m0 -> m2 and m2 -> m4 are one hop
    each (m1 / m3 rounded to FP16 inside the reference, as the fused launch keeps them in shared memory)."""
    back = [("m0", ("input",))]
    if fused_tails:
        back += [("m2", ("m0",)), ("m4", ("m2",))]
    else:
        back += [("m1", ("m0",)), ("m2", ("m1",)), ("m3", ("m2",)), ("m4", ("m3",))]
    back += [("m5", ("m4",)), ("m6", ("m5",)), ("m7", ("m6",)), ("m8", ("m7",)), ("m9", ("m8",))]
    return back + _neck_and_heads("m6", "m4", pose)


def shuffle_hops() -> List[Hop]:
    """Hops of the ShuffleNetV2-backbone keypoint program: a whole stage per hop (read_tensor returns the stage
    buffers in logical channel order), then SPPF, the neck (d3 / d2 in place of m6 / m4) and the heads."""
    back = [("m0", ("input",)), ("d1", ("m0",)), ("d2", ("d1",)), ("d3", ("d2",)), ("d4", ("d3",)),
            ("m9", ("d4",))]
    return back + _neck_and_heads("d3", "d2", True)


def _neck_and_heads(p4: str, p3: str, pose: bool) -> List[Hop]:
    hops = [("m12", ("m9", p4)), ("m15", ("m12", p3)), ("m16", ("m15",)), ("m18", ("m16", "m12")),
            ("m19", ("m18",)), ("m21", ("m19", "m9"))]
    for i, f in enumerate(("m15", "m18", "m21")):
        hops += [(f"box{i}", (f,)), (f"cls{i}", (f,))] + ([(f"kpt{i}", (f,))] if pose else [])
    return hops


def hops_for(model: nn.Module, fused_tails: bool = False) -> List[Hop]:
    if isinstance(model, Y.ShuffleV2Kpt):
        return shuffle_hops()
    return yolo_hops(model.pose, fused_tails)


def hop_label(hop: Hop) -> str:
    return f"{','.join(hop[1])}->{hop[0]}"


class Ref64:
    """FP64 arithmetic with FP16 storage: the reference.  tests/test_hop_ref.py overrides these methods to
    emulate the engine (FP32 accumulation, tanh-form SiLU, split neck conv) and to mutate that emulation."""

    dtype = torch.float64
    want_mag = True

    def __init__(self):
        self._cache: Dict[int, Tuple[torch.Tensor, torch.Tensor]] = {}

    def params(self, c: nn.Conv2d) -> Tuple[torch.Tensor, torch.Tensor]:
        k = id(c)
        if k not in self._cache:
            self._cache[k] = (c.weight.detach().to(self.dtype), c.bias.detach().to(self.dtype))
        return self._cache[k]

    def conv2d(self, c: nn.Conv2d, x, w, b):
        return F.conv2d(x, w, b, c.stride, c.padding, 1, c.groups)

    def conv(self, c: nn.Conv2d, x):
        w, b = self.params(c)
        return self.conv2d(c, x, w, b)

    def mag(self, c: nn.Conv2d, x) -> Optional[torch.Tensor]:
        """conv(|x|, |W|) + |b|: the scale of the dot product that produced each output element."""
        if not self.want_mag:
            return None
        w, b = self.params(c)
        return F.conv2d(x.abs(), w.abs(), b.abs(), c.stride, c.padding, 1, c.groups)

    def act(self, z):
        return F.silu(z)

    def store(self, t):
        return t.half().to(self.dtype)

    def up(self, x):
        return x.repeat_interleave(2, 2).repeat_interleave(2, 3)

    def residual(self, o, r):
        return o + r

    def cat_up_conv(self, c: nn.Conv2d, a, b):
        """1x1 conv over concat(upsample(a), b) (the cv1 of m12 / m15)."""
        return self.conv(c, torch.cat((self.up(a), b), 1))

    def maxpool(self, x):
        return F.max_pool2d(x, 5, 1, 2)


# ---------------------------------------------------------------------------------------------- modules
# Each returns (output before its final FP16 store, mag of its last conv or None).
def _conv(A: Ref64, m: Y.Conv, x):
    z = A.conv(m.conv, x)
    return (A.act(z) if m.act else z), A.mag(m.conv, x)


def _c2f(A: Ref64, mod: Y.C2f, xs: Sequence[torch.Tensor], up_first: bool):
    z = A.cat_up_conv(mod.cv1.conv, xs[0], xs[1]) if up_first else A.conv(mod.cv1.conv, torch.cat(list(xs), 1))
    ys = list(A.store(A.act(z)).chunk(2, 1))
    for b in mod.m:
        h = A.store(_conv(A, b.cv1, ys[-1])[0])
        o = _conv(A, b.cv2, h)[0]
        ys.append(A.store(A.residual(o, ys[-1]) if b.add else o))
    return _conv(A, mod.cv2, torch.cat(ys, 1))


def _sppf(A: Ref64, mod: Y.SPPF, x):
    y = A.store(_conv(A, mod.cv1, x)[0])
    p1 = A.maxpool(y)
    p2 = A.maxpool(p1)
    return _conv(A, mod.cv2, torch.cat((y, p1, p2, A.maxpool(p2)), 1))


def _tower(A: Ref64, seq: nn.Sequential, x):
    h = A.store(_conv(A, seq[0], x)[0])
    h = A.store(_conv(A, seq[1], h)[0])
    return _conv(A, seq[2], h)


def _shuffle(t):
    return None if t is None else Y.channel_shuffle(t)


def _dw(A: Ref64, d: Y.DWConv, x):
    return A.store(A.conv(d.conv, x))


def _shuffle_stage(A: Ref64, stage: nn.ModuleList, x):
    """A down unit and its basic units; mag is tracked per output channel through concat and shuffle (each
    channel's scale is that of the 1x1 that last wrote it)."""
    down = stage[0]
    left, ml = _conv(A, down.b1_pw, _dw(A, down.b1_dw, x))
    t = _dw(A, down.b2_dw, A.store(_conv(A, down.b2_pw1, x)[0]))
    right, mr = _conv(A, down.b2_pw2, t)
    y = _shuffle(torch.cat((left, right), 1))
    mag = _shuffle(torch.cat((ml, mr), 1)) if A.want_mag else None
    for u in stage[1:]:
        y = A.store(y)                                   # every unit's output is a stored stage buffer
        x1, x2 = y.chunk(2, 1)
        t = _dw(A, u.dw, A.store(_conv(A, u.pw1, x2)[0]))
        o, mo = _conv(A, u.pw2, t)
        y = _shuffle(torch.cat((x1, o), 1))
        if A.want_mag:
            mag = _shuffle(torch.cat((mag.chunk(2, 1)[0], mo), 1))
    return y, mag


def _module(model: nn.Module, name: str, xs: Sequence[torch.Tensor], A: Ref64):
    if name == "m0":
        return _conv(A, model.m0, xs[0][:, :3])
    if name[0] == "d":
        return _shuffle_stage(A, model.stages[int(name[1:]) - 1], xs[0])
    if name[:3] in ("box", "cls", "kpt"):
        return _tower(A, getattr(model, name[:3])[int(name[3:])], xs[0])
    mod = getattr(model, name)
    if isinstance(mod, Y.C2f):
        return _c2f(A, mod, xs, name in _UP_FIRST)
    if isinstance(mod, Y.SPPF):
        return _sppf(A, mod, xs[0])
    return _conv(A, mod, xs[0])


def evaluate(model: nn.Module, hop: Hop, xs: Sequence[torch.Tensor], A: Ref64):
    """Output of `hop` (before its final FP16 store) and its mag, from NCHW input tensors of A.dtype."""
    chain = _FUSED_CHAIN.get((hop[0], tuple(hop[1])), (hop[0],))
    for name in chain[:-1]:
        xs = [A.store(_module(model, name, xs, A)[0])]
    return _module(model, chain[-1], xs, A)


def to_nchw(a: np.ndarray, dtype=torch.float64) -> torch.Tensor:
    """FP16 NHWC (read_tensor layout) -> NCHW torch tensor of `dtype` (exact)."""
    return torch.from_numpy(np.ascontiguousarray(a.transpose(0, 3, 1, 2))).to(dtype)


def to_nhwc(t: torch.Tensor) -> np.ndarray:
    return np.ascontiguousarray(t.permute(0, 2, 3, 1).numpy())


def hop_ref(model: nn.Module, hop: Hop, inputs: Sequence[np.ndarray]) -> Tuple[np.ndarray, np.ndarray]:
    """(ref, mag) float64 NHWC for one hop, from its FP16 NHWC input taps.  `ref` has the module's logical
    channel count (cls: nc, kpt: 8); the engine's padded tensors are compared on those channels only."""
    with torch.no_grad():
        y, mag = evaluate(model, hop, [to_nchw(a) for a in inputs], Ref64())
    return to_nhwc(y), to_nhwc(mag)


def ulp16(a: np.ndarray) -> np.ndarray:
    """Spacing of FP16 numbers at |a| (subnormal spacing 2^-24 below 2^-14)."""
    e = np.floor(np.log2(np.maximum(np.abs(a), 2.0 ** -14)))
    return np.exp2(e - 10)


def hop_ratio(got: np.ndarray, ref: np.ndarray, mag: np.ndarray) -> Tuple[float, Dict[str, int]]:
    """max |got - ref| / (2^-8 * mag + ulp16(|ref|)) over NHWC arrays of one shape, and where it is:
    {"frame", "channel", "y", "x"}.  A failure then names the channel, row or border that is wrong."""
    if got.shape != ref.shape or mag.shape != ref.shape:
        raise ValueError(f"shape mismatch: got {got.shape}, ref {ref.shape}, mag {mag.shape}")
    r = np.abs(got.astype(np.float64) - ref) / (TOL_REL * mag + ulp16(ref))
    r = np.where(np.isnan(r), np.inf, r)                 # a NaN from the kernel is a failure, not a pass
    i = int(np.argmax(r))
    f, y, x, c = np.unravel_index(i, r.shape)
    return float(r.flat[i]), {"frame": int(f), "channel": int(c), "y": int(y), "x": int(x)}


def old_gate_passes(got: np.ndarray, ref: np.ndarray) -> bool:
    """The end-to-end per-tap bound of test_network_parity, max |got - ref| <= 2e-2 * max(|ref|, 1), applied to
    one hop: what that check would let through."""
    return bool(np.abs(got.astype(np.float64) - ref).max() <= 2e-2 * max(float(np.abs(ref).max()), 1.0))
