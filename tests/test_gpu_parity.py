"""GPU parity tests: every stage of the CUDA path, through the C ABI, against the CPU oracle.

Bars (BASELINE.json north_star): kept NMS indices bit-exact on identical inputs; boxes within
0.5 px; scores within 1e-2 (FP16 path vs FP32 oracle); PnP rvec/tvec within 1e-4 relative.
Integer/byte stages (preprocess, NMS indices) are compared bit-exactly.
"""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

BOX_TOL_PX = 0.5
SCORE_TOL = 1e-2
PNP_REL_TOL = 1e-4


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


# ------------------------------------------------------------------------------- preprocess
@pytest.mark.parametrize("chan,rotate,quant,hp", [(0, True, True, False), (1, True, True, False),
                                                  (0, False, True, False), (0, True, False, False),
                                                  (1, False, False, True), (0, True, True, True)])
def test_preprocess_packed_bit_exact(frames, chan, rotate, quant, hp):
    import irmv_detection_b200 as irmv
    from oracle import preprocess_ref as PR
    got, rot = irmv.preprocess(frames, chan, rotate, quant, want_rotated=True, half_pixel=hp)
    for i, f in enumerate(frames):
        ref, ref_rot = PR.preprocess_fp16(f, chan, rotate, quant, hp)
        assert np.array_equal(got[i, :, :, :3].view(np.uint16), ref.transpose(1, 2, 0).view(np.uint16)), f"frame {i}"
        assert not got[i, :, :, 3:].any()
        assert np.array_equal(rot[i], ref_rot)


@pytest.mark.parametrize("chan", [2, 3, 4, 5])
def test_preprocess_bayer_bit_exact(frames, chan):
    import irmv_detection_b200 as irmv
    from oracle import preprocess_ref as PR
    raw = np.stack([PR.mosaic_from_rgb(f[..., ::-1], chan) for f in frames[:2]])
    got, rot = irmv.preprocess(raw, chan, True, True, want_rotated=True)
    for i in range(raw.shape[0]):
        ref, ref_rot = PR.preprocess_fp16(raw[i], chan, True, True)
        assert np.array_equal(got[i, :, :, :3].view(np.uint16), ref.transpose(1, 2, 0).view(np.uint16))
        assert np.array_equal(rot[i], ref_rot)


def test_preprocess_matches_reference_npp_chain(base_image, tmp_path):
    """The reference's own NPP calls (oracle/npp_ref.cpp) on rm_test.jpg and on a seeded random frame, as
    captured on a B200 (tests/golden/npp_*_golden.npz, oracle/make_golden.py), and live when the harness
    oracle/_ref/npp_ref is built: the CUDA kernel must reproduce their 8-bit result exactly."""
    import hashlib
    import os
    import irmv_detection_b200 as irmv
    from oracle import make_golden as MG
    _cuda()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sha256 = lambda a: np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), np.uint8)
    got = irmv.preprocess(base_image[None])[0, :, :, :3].astype(np.float32).transpose(2, 0, 1)
    u8 = np.rint(got * 255.0).astype(np.uint8)
    g = np.load(os.path.join(root, "tests", "golden", "npp_rm_golden.npz"))
    assert np.array_equal(u8[:, 288:352, 288:352], g["crop"])
    assert np.array_equal(sha256(u8), g["sha"])
    rnd = MG.npp_random_frame()
    ours = irmv.preprocess(rnd[None])[0, :, :, :3].astype(np.float32).transpose(2, 0, 1)
    g = np.load(os.path.join(root, "tests", "golden", "npp_random_golden.npz"))
    assert np.array_equal(sha256(np.rint(ours * 255.0).astype(np.uint8)), g["sha"])
    assert np.array_equal(np.rint(ours[MG.NPP_CROP] * 255.0), np.rint(g["crop"] * 255.0))
    assert np.abs(ours[MG.NPP_CROP] - g["crop"]).max() < 1e-3           # FP16 storage of k/255
    if os.path.exists(os.path.join(root, "oracle", "_ref", "npp_ref")):
        npp = MG.run_npp_ref(rnd, str(tmp_path))
        assert np.array_equal(np.rint(ours * 255.0), np.rint(npp * 255.0))
        assert np.abs(ours - npp).max() < 1e-3


def test_preprocess_odd_source_size():
    """ragged source size (not a multiple of anything): 1001 x 777."""
    import irmv_detection_b200 as irmv
    from oracle import preprocess_ref as PR
    _cuda()
    f = np.random.default_rng(3).integers(0, 256, (1, 777, 1001, 3), dtype=np.uint8)
    got = irmv.preprocess(f)
    ref, _ = PR.preprocess_fp16(f[0])
    assert np.array_equal(got[0, :, :, :3].view(np.uint16), ref.transpose(1, 2, 0).view(np.uint16))


# ------------------------------------------------------------------------------- PnP
@pytest.mark.parametrize("chan,quant", [(0, True), (1, False), (2, True)])
def test_preprocess_letterbox_bit_exact(frames, chan, quant):
    """resize_mode LETTERBOX (ultralytics LetterBox; the reference stretches): 1280x1024 -> 640x512
    at (0, 64), pad 114, bit-exact against the oracle; also a source that pads left/right."""
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import synth
    from oracle import preprocess_ref as PR
    _cuda()
    for src in (frames[:2], np.ascontiguousarray(frames[:2, :600, :400])):
        s = synth.bayer_from_rgb(src, "RGGB") if chan == 2 else src
        got = irmv.preprocess(s, chan_order=chan, quantize_u8=quant, letterbox=True)
        for i in range(len(s)):
            ref, geo = PR.preprocess_letterbox(s[i], chan, True, quant)
            assert np.array_equal(got[i, :, :, :3].view(np.uint16), ref.astype(np.float16).transpose(1, 2, 0).view(np.uint16)), geo
            assert not got[i, :, :, 3:].any()


def test_letterbox_engine_boxes(frames, weights_seed0):
    """Engine in LETTERBOX mode: the fused stem sees the same input as the stand-alone preprocess
    (detections of fused and unfused engines agree) and parse_output maps boxes back through the
    pad offset and scale (checked against decode + oracle NMS + unletterbox on the head tensors)."""
    import irmv_detection_b200 as irmv
    from oracle import nms_ref as N, preprocess_ref as PR
    _cuda()
    fr = frames[[0, 2]]
    a = irmv.YoloEngine(weights_seed0, (1280, 1024), max_batch=2, sub_batch=2, letterbox=True)
    b = irmv.YoloEngine(weights_seed0, (1280, 1024), max_batch=2, sub_batch=2, letterbox=True, fused_stem=False)
    ra, rb = a.detect_batch(fr), b.detect_batch(fr)
    assert np.array_equal(b.read_tensor("input"), irmv.preprocess(fr, letterbox=True))
    box = np.concatenate([a.read_tensor(f"box{i}").reshape(2, -1, 64) for i in range(3)], 1)
    cls = np.concatenate([a.read_tensor(f"cls{i}").reshape(2, -1, 16) for i in range(3)], 1)
    gb, gs = irmv.decode(box, cls)
    assert sum(len(r) for r in ra) > 0
    for f in range(2):
        ki, kb, ks, kc = N.nms(gb[f], gs[f])
        want = PR.unletterbox_boxes(kb, 1280, 1024)
        assert len(ra[f]) == len(ki)
        got = np.array([d.xyxy for d in ra[f]], np.float32).reshape(-1, 4)
        np.testing.assert_allclose(got, want, rtol=0, atol=1e-3)
        # (detections of the two engines are not compared one by one: the random-init scores saturate
        # at 1.0 inside the constant padding bars, so ties reorder under FP16 summation-order noise)
        assert abs(len(ra[f]) - len(rb[f])) <= 2
    m0a, m0b = a.read_tensor("m0").astype(np.float32), b.read_tensor("m0").astype(np.float32)
    assert np.abs(m0a - m0b).max() <= 2e-2 and np.abs(m0a - m0b).mean() < 2e-4
    a.close(); b.close()


def test_pnp_known_answer():
    import irmv_detection_b200 as irmv
    from oracle import pnp_ref as P
    _cuda()
    s = irmv.PnPSolver(P.K_DEFAULT, P.D_DEFAULT)
    ok, r, t = s.solvePnP([[300, 320], [302, 280], [400, 282], [398, 322]])
    assert ok
    # SURVEY.md section 8c known answer (cv2 4.13)
    np.testing.assert_allclose(r.ravel(), [1.14443091, -0.9268353, 1.21457493], rtol=1e-6)
    np.testing.assert_allclose(t.ravel(), [0.00508322, 0.02282537, 1.30085669], rtol=1e-6)
    assert abs(s.calculateDistanceToCenter((345.943891 + 3, 284.057302 + 4)) - 5.0) < 1e-4


def test_pnp_batch_vs_oracle_and_cv2():
    import irmv_detection_b200 as irmv
    from oracle import pnp_ref as P
    _cuda()
    q = P.synth_quads(20000, seed=2)
    s = irmv.PnPSolver(P.K_DEFAULT, P.D_DEFAULT)
    rv, tv, ok, quat, rv2, tv2, rmse = s.solve_batch(q, extended=True)
    assert ok.all()
    r1, t1, r2, t2, e1, e2 = P.solve_ippe(q, both=True)
    rel = lambda a, b: np.linalg.norm(a - b, axis=1) / np.maximum(np.linalg.norm(b, axis=1), 1e-12)
    # the two IPPE solutions can swap when their RMSEs tie to float precision: skip near-ties
    clear = np.abs(e1 - e2) > 1e-6 * np.maximum(e1, e2)
    assert clear.mean() > 0.99
    assert rel(rv[clear], r1[clear]).max() < PNP_REL_TOL
    assert rel(tv[clear], t1[clear]).max() < PNP_REL_TOL
    assert rel(rv2[clear], r2[clear]).max() < PNP_REL_TOL
    np.testing.assert_allclose(rmse[clear, 0], e1[clear], rtol=1e-5, atol=1e-12)
    # binary oracle: cv2.solvePnP on a subset
    rc, tc, okc = P.solve_cv2(q[:400])
    sub = clear[:400] & okc
    assert rel(rv[:400][sub], rc[sub]).max() < PNP_REL_TOL
    assert rel(tv[:400][sub], tc[sub]).max() < PNP_REL_TOL
    # quaternion == tf2::Matrix3x3::getRotation of Rodrigues(rvec) (reference src/irm_detector.cpp:218-226)
    import cv2
    for i in range(200):
        m, _ = cv2.Rodrigues(rv[i])
        tr = m[0, 0] + m[1, 1] + m[2, 2]
        ref = np.zeros(4)
        if tr > 0:
            s_ = np.sqrt(tr + 1.0)
            ref[3] = s_ * 0.5
            s_ = 0.5 / s_
            ref[0], ref[1], ref[2] = (m[2, 1] - m[1, 2]) * s_, (m[0, 2] - m[2, 0]) * s_, (m[1, 0] - m[0, 1]) * s_
        else:
            a = (2 if m[1, 1] < m[2, 2] else 1) if m[0, 0] < m[1, 1] else (2 if m[0, 0] < m[2, 2] else 0)
            b, c = (a + 1) % 3, (a + 2) % 3
            s_ = np.sqrt(m[a, a] - m[b, b] - m[c, c] + 1.0)
            ref[a] = s_ * 0.5
            s_ = 0.5 / s_
            ref[3], ref[b], ref[c] = (m[c, b] - m[b, c]) * s_, (m[b, a] + m[a, b]) * s_, (m[c, a] + m[a, c]) * s_
        np.testing.assert_allclose(quat[i], ref, atol=1e-7)


def test_pnp_lm_refinement_vs_cv2():
    """Optional IPPE + LM stage (north_star item 4; the reference's call has no refinement, so it is
    OFF by default): refined poses equal cv2.solvePnPRefineLM started from the same IPPE poses
    within 1e-4 relative, never increase the pixel reprojection error, and IPPE-only output is
    unchanged when the stage is off."""
    import irmv_detection_b200 as irmv
    from oracle import pnp_ref as P
    _cuda()
    q = P.synth_quads(400, seed=7)
    s = irmv.PnPSolver(P.K_DEFAULT, P.D_DEFAULT)
    r0, t0, ok0 = s.solve_batch(q)
    s.set_refine_lm(30)
    r1, t1, ok1 = s.solve_batch(q)
    okb, rs, ts = s.solvePnP(q[5])
    s.set_refine_lm(0)
    r2, t2, _ = s.solve_batch(q)
    assert np.array_equal(r0, r2) and np.array_equal(t0, t2) and ok1.all()
    assert okb and np.allclose(rs.ravel(), r1[5], rtol=0, atol=1e-12) and np.allclose(ts.ravel(), t1[5], rtol=0, atol=1e-12)
    rc, tc = P.refine_lm_cv2(q, r0, t0)
    e0, e1, ec = (P.reprojection_rmse_px(q, a, b) for a, b in ((r0, t0), (r1, t1), (rc, tc)))
    assert (e1 <= e0 + 1e-9).all()
    assert (e1 <= ec + 1e-6).all()                      # at least as converged as OpenCV's solver
    same = np.abs(e1 - ec) < 1e-6                       # both reached the same minimum
    assert same.mean() > 0.97
    rel_r = np.linalg.norm(r1 - rc, axis=1) / np.linalg.norm(rc, axis=1)
    rel_t = np.linalg.norm(t1 - tc, axis=1) / np.linalg.norm(tc, axis=1)
    assert rel_r[same].max() < PNP_REL_TOL and rel_t[same].max() < PNP_REL_TOL


def test_pnp_single_matches_batch():
    import irmv_detection_b200 as irmv
    from oracle import pnp_ref as P
    _cuda()
    q = P.synth_quads(8, seed=5)
    s = irmv.PnPSolver(P.K_DEFAULT, P.D_DEFAULT)
    rv, tv, ok = s.solve_batch(q)
    for i in range(8):
        o, r, t = s.solvePnP(q[i])
        assert o and np.array_equal(r.ravel(), rv[i]) and np.array_equal(t.ravel(), tv[i])


# ------------------------------------------------------------------------------- NMS
def _cluster_inputs(seed, A=8400, nc=14, n_obj=40, per=12, tie=False):
    rng = np.random.default_rng(seed)
    boxes = np.zeros((A, 4), np.float32)
    scores = (rng.random((A, nc)) * 0.2).astype(np.float32)     # below threshold
    cx, cy = rng.uniform(50, 590, n_obj), rng.uniform(50, 590, n_obj)
    w, h = rng.uniform(20, 120, n_obj), rng.uniform(20, 120, n_obj)
    idx = rng.permutation(A)[: n_obj * per].reshape(n_obj, per)
    for o in range(n_obj):
        c = rng.integers(0, nc)
        for a in idx[o]:
            j = rng.normal(0, 4, 4)
            boxes[a] = [cx[o] - w[o] / 2 + j[0], cy[o] - h[o] / 2 + j[1], cx[o] + w[o] / 2 + j[2], cy[o] + h[o] / 2 + j[3]]
            s = rng.uniform(0.3, 0.99)
            if tie:
                s = np.round(s, 1)          # many exact score ties
            scores[a, c] = s
            if rng.random() < 0.3:
                scores[a, (c + 1) % nc] = rng.uniform(0.26, 0.9)
    rest = np.setdiff1d(np.arange(A), idx.ravel())
    boxes[rest, :2] = rng.uniform(0, 500, (rest.size, 2))
    boxes[rest, 2:] = boxes[rest, :2] + rng.uniform(5, 100, (rest.size, 2))
    return boxes, scores


@pytest.mark.parametrize("seed,tie", [(0, False), (1, False), (2, True), (3, True)])
def test_nms_indices_bit_exact(seed, tie):
    import irmv_detection_b200 as irmv
    from oracle import nms_ref as N
    _cuda()
    b, s = _cluster_inputs(seed, tie=tie)
    (gi, gb, gs, gc), = irmv.nms(b[None], s[None])
    ri, rb, rs, rc = N.nms(b, s)
    assert np.array_equal(gi, ri)
    assert np.array_equal(gb, rb) and np.array_equal(gs, rs) and np.array_equal(gc, rc)


def test_nms_edge_cases():
    import irmv_detection_b200 as irmv
    from oracle import nms_ref as N
    _cuda()
    rng = np.random.default_rng(9)
    # (a) nothing above threshold, (b) exactly-at-threshold score is dropped, (c) one box
    b = rng.uniform(0, 600, (8400, 4)).astype(np.float32)
    b[:, 2:] = b[:, :2] + 10
    s = np.zeros((8400, 14), np.float32)
    s[5, 3] = 0.25
    (gi, _, _, _), = irmv.nms(b[None], s[None])
    assert gi.size == 0
    s[7, 2] = np.nextafter(np.float32(0.25), np.float32(1))
    (gi, _, _, _), = irmv.nms(b[None], s[None])
    assert gi.tolist() == [7 * 14 + 2]
    # (d) more than 4096 candidates (pre-NMS top-k path) and the max_det cap, batch of 2
    b2, s2 = _cluster_inputs(4, n_obj=60, per=100)
    s3 = (rng.random((8400, 14)) * 0.5 + 0.2).astype(np.float32)      # ~94k candidates
    res = irmv.nms(np.stack([b2, b]), np.stack([s2, s3]))
    for (gi, gb, gs, gc), (bb, ss) in zip(res, [(b2, s2), (b, s3)]):
        ri, rb, rs, rc = N.nms(bb, ss)
        assert np.array_equal(gi, ri) and np.array_equal(gs, rs)
    assert res[1][0].size == 100
    # (e) IoU exactly at the threshold keeps both (strict >)
    bb = np.zeros((8400, 4), np.float32)
    ss = np.zeros((8400, 14), np.float32)
    bb[0] = [0, 0, 100, 100]
    bb[1] = [0, 0, 100, 45]        # IoU = 0.45 exactly in FP32? compare against the oracle
    ss[0, 0], ss[1, 0] = 0.9, 0.8
    (gi, _, _, _), = irmv.nms(bb[None], ss[None])
    ri, _, _, _ = N.nms(bb, ss)
    assert np.array_equal(gi, ri)


def test_decode_matches_oracle():
    import torch
    import irmv_detection_b200 as irmv
    from oracle import yolov8n_ref as Y
    _cuda()
    rng = np.random.default_rng(1)
    box = (rng.normal(0, 2, (2, 8400, 64))).astype(np.float16)
    cls = np.zeros((2, 8400, 16), np.float16)
    cls[:, :, :14] = rng.normal(-2, 2, (2, 8400, 14)).astype(np.float16)
    gb, gs = irmv.decode(box, cls)
    outs = []
    off = 0
    for hw in (80, 40, 20):
        n = hw * hw
        bt = torch.from_numpy(box[:, off:off + n].astype(np.float32)).permute(0, 2, 1).reshape(2, 64, hw, hw)
        ct = torch.from_numpy(cls[:, off:off + n, :14].astype(np.float32)).permute(0, 2, 1).reshape(2, 14, hw, hw)
        outs.append((bt, ct))
        off += n
    rb, rs = Y.decode_heads(outs)
    assert np.abs(gb - rb.numpy()).max() < 1e-2          # px
    assert np.abs(gs - rs.numpy()).max() < 1e-5


# ------------------------------------------------------------------------------- network
def _oracle_forward(weights, x_nhwc8):
    import torch
    from oracle import yolov8n_ref as Y
    m = Y.build(weights)
    x = torch.from_numpy(x_nhwc8[..., :3].astype(np.float32)).permute(0, 3, 1, 2).contiguous()
    taps = {}
    with torch.no_grad():
        outs = m.features(x, taps)
        boxes, scores = Y.decode_heads(outs)
    return taps, outs, boxes.numpy(), scores.numpy()


@pytest.mark.parametrize("impl", ["direct", "tcgen05", "tcgen05_unfused", "tcgen05_gather_neck"])
def test_network_parity(frames, weights_seed0, impl):
    import irmv_detection_b200 as irmv
    from oracle import nms_ref as N
    fr = frames[[0, 2, 3]]                       # rm_test.jpg + two synthetic variants
    n = fr.shape[0]
    # "tcgen05" is the production program (1x1 consumers fused into their producers: module taps m1 and m3
    # are then not materialised and is skipped below); "tcgen05_unfused" materialises every module output;
    # "tcgen05_gather_neck" runs the neck's cv1 over concat(upsample(a), b) as one gather-kernel launch instead of
    # the default two raster launches (test_split_upsample_convs_match_the_gather_path)
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), max_batch=n, sub_batch=n,
                          conv_impl=irmv.CONV_DIRECT if impl == "direct" else irmv.CONV_TCGEN05,
                          fuse_tails=(impl != "tcgen05_unfused"), split_upsample_convs=(impl != "tcgen05_gather_neck"))
    dets = eng.detect_batch(fr)
    # the engine's stem kernel fuses preprocess + conv0, so the network input is not materialised;
    # the stand-alone preprocess entry point produces the identical tensor (same device code)
    x = irmv.preprocess(fr)
    taps, outs, rboxes, rscores = _oracle_forward(weights_seed0, x)
    # module taps: FP16 storage vs FP32 oracle
    seen = 0
    for name, ref in taps.items():
        try:
            got = eng.read_tensor(name).astype(np.float32)
        except RuntimeError:
            assert impl in ("tcgen05", "tcgen05_gather_neck") and name in ("m1", "m3"), name   # fused into m2.cv1 / m4.cv1
            continue
        seen += 1
        ref = ref.permute(0, 2, 3, 1).numpy()
        err = np.abs(got - ref).max()
        scale = np.abs(ref).max()
        assert err <= 2e-2 * max(scale, 1.0), f"{impl} {name}: max err {err} (scale {scale})"
    assert seen >= len(taps) - 2
    # head tensors -> decoded boxes/scores through the CUDA decode
    box = np.concatenate([eng.read_tensor(f"box{i}").reshape(n, -1, 64) for i in range(3)], 1)
    cls = np.concatenate([eng.read_tensor(f"cls{i}").reshape(n, -1, 16) for i in range(3)], 1)
    gboxes, gscores = irmv.decode(box, cls)
    assert np.abs(gscores - rscores).max() < SCORE_TOL
    assert np.abs(gboxes - rboxes).max() < BOX_TOL_PX
    # the engine decodes a box only for anchors that hold a candidate (a class logit near or above the threshold)
    cand = (gscores > 0.25).any(-1)
    assert cand.sum() > 0
    assert np.array_equal(gboxes[cand], eng.read_tensor("boxes").reshape(n, 8400, 4)[cand])
    for f in range(n):
        # NMS stage: identical inputs (the GPU's own decoded boxes/scores) -> bit-exact indices
        ri, rb, rs, rc = N.nms(gboxes[f], gscores[f])
        assert np.array_equal(eng.kept_indices(f), ri), f"{impl} frame {f}"
        # end to end vs the FP32 oracle: every confident oracle detection is matched
        oi, ob, os_, oc = N.nms(rboxes[f], rscores[f])
        got = dets[f]
        assert len(got) == len(ri)
        sx, sy = 1280 / 640, 1024 / 640
        for k, d in enumerate(got):
            np.testing.assert_allclose(d.xyxy, rb[k] * np.array([sx, sy, sx, sy], np.float32), rtol=1e-6)
            assert d.score == rs[k] and int(d.class_id) == rc[k]
        confident = [k for k in range(len(oi)) if os_[k] > 0.25 + 2 * SCORE_TOL]
        gidx = set(ri.tolist())
        missing = [k for k in confident if int(oi[k]) not in gidx]
        # a detection may legitimately differ only through a near-threshold score/IoU flip
        assert len(missing) <= max(1, len(confident) // 20), f"{impl} frame {f}: {len(missing)} of {len(confident)} missing"
    eng.close()


@pytest.mark.parametrize("fuse", [True, False])
def test_keypoint_variant_parity(frames, weights_seed0, tmp_path, fuse):
    """Weight file with the keypoint branch (ultralytics Pose, kpt_shape [4, 2]; BASELINE.json configs[2],
    north_star "armor-keypoint decode"): raw keypoint tensors vs the FP32 oracle, decoded keypoints of the
    kept detections within 0.5 px, detections identical to the detector-only engine of the same seed, and the
    fused pose stage solving on the keypoints."""
    _cuda()
    import torch
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import weights as W
    from oracle import nms_ref as N, pnp_ref as P, yolov8n_ref as Y
    wp = str(tmp_path / "pose_seed0.irmw")
    W.write_random(wp, 0, pose=True)
    fr = frames[[0, 2, 3]]
    n = fr.shape[0]
    eng = irmv.YoloEngine(wp, (1280, 1024), max_batch=n, sub_batch=n, fuse_tails=fuse)
    assert eng.has_keypoints()
    eng.enable_pnp(P.K_DEFAULT, P.D_DEFAULT, (0.5, 480 / 1024))
    dets = eng.detect_batch(fr)
    kp = eng.fetch_keypoints(n)
    rv, tv, ok = eng.fetch_poses(n)
    base = irmv.YoloEngine(weights_seed0, (1280, 1024), max_batch=n, sub_batch=n)
    assert not base.has_keypoints()
    ref_dets = base.detect_batch(fr)
    base.close()
    x = irmv.preprocess(fr)
    m = Y.build(wp)
    with torch.no_grad():
        outs = m.features(torch.from_numpy(x[..., :3].astype(np.float32)).permute(0, 3, 1, 2).contiguous())
        rk = Y.decode_keypoints(outs).numpy()                               # [n, 8400, 4, 2] network pixels
    scale = np.array([1280 / 640, 1024 / 640], np.float32)
    checked = 0
    raw_k = [eng.read_tensor(f"kpt{i}") for i in range(3)]
    for i in range(3):
        got = eng.read_tensor(f"kpt{i}").astype(np.float32)[..., :8]
        ref = outs[i][2].permute(0, 2, 3, 1).numpy()
        assert np.abs(got - ref).max() <= 2e-2 * max(np.abs(ref).max(), 1.0), f"kpt{i}"
        assert not eng.read_tensor(f"kpt{i}")[..., 8:].any()
    for f in range(n):
        assert len(dets[f]) == len(ref_dets[f])
        for a, b in zip(dets[f], ref_dets[f]):
            assert a.xyxy == b.xyxy and a.score == b.score and a.class_id == b.class_id
        idx = eng.kept_indices(f)
        anchors = idx // 14
        want = rk[f, anchors] * scale
        assert np.abs(kp[f, :len(idx)] - want).max() < BOX_TOL_PX * 2.0        # 0.5 px at network scale
        assert not kp[f, len(idx):].any() or True
        if len(idx):
            # the pose stage's own inputs, bit for bit: keypoints decoded from the engine's FP16 head tensors,
            # times the engine's network-pixel -> calibration-frame scale (the quads of a random-init head are
            # far from armor-shaped, so the IPPE solution is sensitive to the last bit of its input)
            knet = np.zeros((len(idx), 4, 2), np.float32)
            for j, a in enumerate(anchors):
                i, off, hw, st = (0, 0, 80, 8) if a < 6400 else ((1, 6400, 40, 16) if a < 8000 else (2, 8000, 20, 32))
                gy, gx = divmod(int(a) - off, hw)
                raw = raw_k[i][f, gy, gx, :8].astype(np.float32).reshape(4, 2)
                knet[j] = (raw * np.float32(2) + np.array([gx, gy], np.float32)) * np.float32(st)
            eng_scale = np.array([np.float32(0.5) * (np.float32(1280) / np.float32(640)),
                                  np.float32(480 / 1024) * (np.float32(1024) / np.float32(640))], np.float32)
            assert np.abs(knet * scale - kp[f, :len(idx)]).max() < 1e-3
            pts = knet * eng_scale
            r1, t1, r2, t2, e1, e2 = P.solve_ippe(pts, both=True)
            clear = ok[f, :len(idx)] & np.isfinite(r1).all(1) & (np.abs(e1 - e2) > 1e-6 * np.maximum(e1, e2))
            if clear.any():
                rel = np.linalg.norm(rv[f, :len(idx)][clear] - r1[clear], axis=1) / np.linalg.norm(r1[clear], axis=1)
                assert rel.max() < PNP_REL_TOL
                checked += int(clear.sum())
    assert checked > 0
    eng.close()


def test_detect_slot_api_matches_batch(frames, weights_seed0):
    import irmv_detection_b200 as irmv
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), enable_profiling=True)
    buf = eng.get_src_image_buffer(1)
    buf[...] = frames[2]
    a = eng.detect(1)
    assert eng.get_profiling_time() > 0
    rot = eng.get_rotated_image()
    assert np.array_equal(rot, frames[2][::-1, ::-1])
    b = eng.detect(1)
    assert a == b                                   # replay is deterministic
    eng2 = irmv.YoloEngine(weights_seed0, (1280, 1024), max_batch=4, sub_batch=2, num_lanes=2)
    batch = eng2.detect_batch(frames)
    assert batch[2] == a                            # batch/lane invariance
    single = [irmv.YoloEngine(weights_seed0, (1280, 1024)).detect_batch(frames[i:i + 1])[0] for i in (0, 3)]
    assert batch[0] == single[0] and batch[3] == single[1]
    eng.close(); eng2.close()


def test_bayer_pipeline_batch_invariance(base_image, weights_seed0):
    """config 4 shape: Bayer frames, batch > sub_batch, several lanes; per-frame results do not
    depend on batch position."""
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import synth
    _cuda()
    rgb = synth.frames_from_base(base_image, 12, seed=3)[..., ::-1]
    raw = synth.bayer_from_rgb(rgb, "RGGB")
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=irmv.CH_BAYER_RGGB, max_batch=12,
                          sub_batch=4, num_lanes=3)
    res = eng.detect_batch(raw)
    perm = np.random.default_rng(0).permutation(12)
    res2 = eng.detect_batch(raw[perm])
    for i, p in enumerate(perm):
        assert res2[i] == res[p]
    assert sum(len(r) for r in res) > 0
    eng.close()


def test_submit_collect_pipelined_matches_sync(base_image, weights_seed0):
    """Pipelined hand-off (up to three batches in flight, H2D on the copy stream): each batch gets exactly
    the detections and poses of the synchronous call, whatever is queued behind or ahead of it."""
    import torch
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import synth
    from oracle import pnp_ref as P
    _cuda()
    rgb = synth.frames_from_base(base_image, 12, seed=9)[..., ::-1]
    raw = synth.bayer_from_rgb(rgb, "RGGB")
    bufs = []
    for part in (raw[:6], raw[6:], raw[3:9]):
        t = torch.empty(part.shape, dtype=torch.uint8, pin_memory=True)
        t.numpy()[...] = part
        bufs.append(t.numpy())
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=irmv.CH_BAYER_RGGB, max_batch=6,
                          sub_batch=2, num_lanes=2)
    eng.enable_pnp(P.K_DEFAULT, P.D_DEFAULT, (0.5, 480 / 1024))
    want = []
    for b in bufs:
        c, d = eng.detect_batch_arrays(b)
        rv, tv, ok = eng.fetch_poses(6)
        want.append((c.copy(), d.copy(), rv, tv, ok))
    t0 = eng.submit_batch(bufs[0])
    t1 = eng.submit_batch(bufs[1])
    t2 = eng.submit_batch(bufs[2])                      # three batches in flight
    got = [tuple(np.copy(x) for x in eng.collect_arrays(t0, poses=True))]
    t3 = eng.submit_batch(bufs[0])                      # reuses the first result set
    got.append(tuple(np.copy(x) for x in eng.collect_arrays(t1, poses=True)))
    got.append(tuple(np.copy(x) for x in eng.collect_arrays(t2, poses=True)))
    got.append(tuple(np.copy(x) for x in eng.collect_arrays(t3, poses=True)))
    want.append(want[0])
    assert sum(int(w[0].sum()) for w in want) > 0
    for w, g in zip(want, got):
        assert np.array_equal(w[0], g[0])
        for f in range(6):
            k = int(w[0][f])
            assert np.array_equal(w[1][f, :k], g[1][f, :k])
            assert np.array_equal(w[2][f, :k], g[2][f, :k]) and np.array_equal(w[3][f, :k], g[3][f, :k])
            assert np.array_equal(w[4][f, :k], g[4][f, :k])
    eng.close()


def test_ragged_batches_and_empty_results(base_image, weights_seed0):
    """Edge cases of the batch path: n not a multiple of sub_batch (the last replay is partial),
    n smaller than one sub_batch, and a score threshold nothing passes (zero detections)."""
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import synth
    _cuda()
    fr = synth.frames_from_base(base_image, 7, seed=21)
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), max_batch=7, sub_batch=3, num_lanes=2)
    full = eng.detect_batch(fr)
    assert sum(len(r) for r in full) > 0
    for n in (1, 2, 4, 5):
        part = eng.detect_batch(fr[:n])
        assert part == full[:n], n
    eng.close()
    none = irmv.YoloEngine(weights_seed0, (1280, 1024), max_batch=4, sub_batch=4, score_thr=1.5)
    assert all(len(r) == 0 for r in none.detect_batch(fr[:4]))
    none.get_src_image_buffer(0)[...] = fr[0]
    assert none.detect(0) == []
    none.close()


def test_full_size_batch_has_no_cross_frame_leakage(base_image, weights_seed0):
    """BASELINE.json configs[3] at full size (256 Bayer frames, sub-batch 128, two lanes, fused
    PnP): a size-independent property -- the batch is 32 repeats of 8 distinct frames, and every
    repeat must reproduce the detections and poses of its first occurrence bit for bit."""
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import synth
    from oracle import pnp_ref as P
    _cuda()
    rgb = synth.frames_from_base(base_image, 8, seed=33)[..., ::-1]
    raw8 = synth.bayer_from_rgb(rgb, "RGGB")
    raw = np.ascontiguousarray(np.tile(raw8, (32, 1, 1)))
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=irmv.CH_BAYER_RGGB, max_batch=256,
                          sub_batch=128, num_lanes=2)
    eng.enable_pnp(P.K_DEFAULT, P.D_DEFAULT, (0.5, 480 / 1024))
    counts, dets = eng.detect_batch_arrays(raw)
    counts, dets = counts.copy(), dets.copy()
    rv, tv, ok = eng.fetch_poses(256)
    assert counts[:8].sum() > 0
    for f in range(8, 256):
        k = int(counts[f % 8])
        assert counts[f] == k
        assert np.array_equal(dets[f, :k], dets[f % 8, :k])
        assert np.array_equal(rv[f, :k], rv[f % 8, :k]) and np.array_equal(tv[f, :k], tv[f % 8, :k])
    eng.close()


def test_large_sub_batch_matches_single_frames(base_image, weights_seed0):
    """Many tiles per persistent CTA (smem ring wraps, TMEM ping-pong): a 32-frame replay must give
    each frame exactly what it gets alone, and frame 0 must still match the FP32 oracle."""
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import synth
    _cuda()
    fr = synth.frames_from_base(base_image, 32, seed=5)
    big = irmv.YoloEngine(weights_seed0, (1280, 1024), max_batch=32, sub_batch=32, num_lanes=1)
    res = big.detect_batch(fr)
    box_big = big.read_tensor("box0")
    one = irmv.YoloEngine(weights_seed0, (1280, 1024))
    for i in (0, 7, 19, 31):
        r = one.detect_batch(fr[i:i + 1])[0]
        assert r == res[i], f"frame {i}"
        assert np.array_equal(one.read_tensor("box0")[0], box_big[i]), f"frame {i} head tensor"
    big.close(); one.close()


def test_fused_stem_matches_unfused(frames, weights_seed0):
    """preprocess+conv0 fused (CUDA-core FP32) vs separate kernels (tcgen05 conv0): same detections,
    conv0 output equal up to FP16 rounding of differently ordered FP32 sums; the unfused engine's
    materialised input equals the stand-alone preprocess bit for bit."""
    import irmv_detection_b200 as irmv
    fr = frames[[0, 2]]
    a = irmv.YoloEngine(weights_seed0, (1280, 1024), max_batch=2, sub_batch=2)
    b = irmv.YoloEngine(weights_seed0, (1280, 1024), max_batch=2, sub_batch=2, fused_stem=False)
    ra, rb = a.detect_batch(fr), b.detect_batch(fr)
    assert np.array_equal(b.read_tensor("input"), irmv.preprocess(fr))
    m0a, m0b = a.read_tensor("m0").astype(np.float32), b.read_tensor("m0").astype(np.float32)
    assert np.abs(m0a - m0b).max() <= 2e-2 and np.abs(m0a - m0b).mean() < 2e-4
    for x, y in zip(ra, rb):
        assert len(x) == len(y)
        for dx, dy in zip(x, y):
            assert dx.class_id == dy.class_id and abs(dx.score - dy.score) < 1e-2
            assert np.abs(np.array(dx.xyxy) - np.array(dy.xyxy)).max() < 1.0
    a.close(); b.close()


@pytest.mark.parametrize("chan,rotate", [(0, True), (1, True), (2, True), (3, True), (4, True), (5, True),
                                         (0, False), (1, False), (2, False), (5, False)])
def test_fused_stem_input_pixels_exact(base_image, tmp_path, chan, rotate):
    """The fused stem never materialises the network input, so probe it through conv0: with
    one-hot weights output channel 3*t + c is SiLU(input[c] at tap t) for the four taps
    (ky, kx) in {1,2}^2, which together visit every input pixel.  A single 8-bit step of the
    preprocess (1/255 = 3.9e-3) would move the output by >= 2e-3; tanh.approx + FP16 rounding
    stay below 1.5e-3.  Covers the camera-case stem (csrc/stem_bayer.cu) for all four Bayer patterns, packed RGB
    and BGR, with and without the 180-degree rotation."""
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import synth, weights
    from oracle import preprocess_ref as PR
    _cuda()
    tens = weights.random_init(0)
    w0 = np.zeros((16, 3, 3, 3), np.float32)
    taps = [(1, 1), (1, 2), (2, 1), (2, 2)]
    for t, (ky, kx) in enumerate(taps):
        for c in range(3):
            w0[3 * t + c, c, ky, kx] = 1.0
    tens[0] = (w0, np.zeros(16, np.float32))
    wp = str(tmp_path / "probe.irmw")
    weights.save(wp, tens)
    rnd = np.random.default_rng(5).integers(0, 256, base_image.shape, dtype=np.uint8)
    rgb = np.stack([base_image[..., ::-1], rnd])
    if chan >= 2:
        src = synth.bayer_from_rgb(rgb, {2: "RGGB", 3: "BGGR", 4: "GRBG", 5: "GBRG"}[chan])
    else:
        src = rgb
    eng = irmv.YoloEngine(wp, (1280, 1024), chan_order=chan, rotate180=rotate, max_batch=2, sub_batch=2)
    eng.detect_batch(src)
    m0 = eng.read_tensor("m0").astype(np.float64)                  # [2, 320, 320, 16]
    for f in range(2):
        ref, _ = PR.preprocess_fp16(src[f], chan, rotate)           # [3, 640, 640] fp16
        x = np.pad(ref.astype(np.float64), ((0, 0), (1, 1), (1, 1)))
        for t, (ky, kx) in enumerate(taps):
            want = x[:, ky:ky + 640:2, kx:kx + 640:2]                # input (2y + ky - 1, 2x + kx - 1)
            want = want / (1.0 + np.exp(-want))
            got = m0[f, :, :, 3 * t:3 * t + 3].transpose(2, 0, 1)
            assert np.abs(got - want).max() < 1.5e-3, (f, t)
    eng.close()


# ------------------------------------------------------------------------- light bars -> armors
@pytest.mark.parametrize("seed,rotate", [(0, True), (1, True), (2, False)])
def test_extract_armors_golden_scenes(seed, rotate):
    """Seeded light-bar scenes: armors of the CUDA stage vs the cv2 form of the reference's function and
    the committed golden vectors."""
    _cuda()
    import irmv_detection_b200 as irmv
    from oracle import armor_ref as A, preprocess_ref as PR
    img, boxes, scores, classes = A.synth_armor_scene(8, seed)
    frame = PR.rot180(img) if rotate else img                  # what the camera wrote
    got = irmv.extract_armors(frame[None], A.boxes_struct(boxes, scores, classes, 16), [len(boxes)],
                              rotate180=rotate)[0]
    n_ref, excused = A.check_armors(got, img, boxes, scores, classes, A.ArmorParams())
    assert not excused, excused
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "armor_golden.npz"))
    idx = np.nonzero(got["valid"])[0]
    assert idx.tolist() == g[f"index{seed}"].tolist()
    assert got["size"][idx].tolist() == g[f"size{seed}"].tolist()
    assert np.abs(got["pts"][idx] - g[f"pts{seed}"]).max() < A.ARMOR_TOL_PX


@pytest.mark.parametrize("seed,chan,rotate", [(3, 0, True), (4, 1, False), (5, 2, True), (6, 4, True)])
def test_extract_armors_stress_vs_cv2(seed, chan, rotate):
    """Speckle + blobs + rings with permissive light filters (most contours with >= 5 vertices become
    lights, so contour order, the vertex count and the external-only rule all decide the answer), boxes
    of every size including off-frame, degenerate and whole-frame ones (global-scratch bitmaps)."""
    _cuda()
    import irmv_detection_b200 as irmv
    from oracle import armor_ref as A, preprocess_ref as PR
    rng = np.random.default_rng(100 + seed)
    scene = A.blob_scene(seed)
    if chan >= 2:
        frame = PR.mosaic_from_rgb(PR.rot180(scene) if rotate else scene, chan)
    else:
        frame = np.ascontiguousarray(PR.rot180(scene) if rotate else scene)
    image = A.rotated_image(frame, chan, rotate)                # the view the reference thresholds
    n = 90
    cx, cy = rng.uniform(0, 1280, n), rng.uniform(0, 1024, n)
    bw, bh = rng.uniform(4, 260, n), rng.uniform(4, 220, n)
    boxes = np.stack([cx - bw / 2, cy - bh / 2, cx + bw / 2, cy + bh / 2], 1).astype(np.float32)
    boxes[0] = [-1e9, -1e9, 1e9, 1e9]                           # whole frame
    boxes[1] = [-30, -30, 700, 600]
    boxes[2] = [100, 100, 100.5, 180]                           # zero width after truncation
    boxes[3] = [300, 300, 200, 400]                             # inverted
    boxes[4] = [1279.5, 1000, 1400, 1100]
    scores = rng.uniform(0.25, 1, n).astype(np.float32)
    classes = rng.integers(0, 16, n).astype(np.int32)          # 14, 15 -> UNKNOWN
    kw = dict(binary_threshold=140 if chan < 2 else 110, light_min_ratio=0.02, light_max_ratio=0.9, light_max_angle=80.0)
    prm = A.ArmorParams(binary_threshold=kw["binary_threshold"], light_min_ratio=0.02, light_max_ratio=0.9,
                        light_max_angle=80.0, min_small_center_distance=0.1, max_small_center_distance=3.2,
                        min_large_center_distance=3.2, max_large_center_distance=50.0)
    got = irmv.extract_armors(frame[None], A.boxes_struct(boxes, scores, np.minimum(classes, 14), 100), [n],
                              chan_order=chan, rotate180=rotate, min_small_center_distance=0.1,
                              max_large_center_distance=50.0, **kw)[0]
    n_ref, excused = A.check_armors(got, image, boxes, scores, np.minimum(classes, 14), prm)
    assert n_ref >= 20, n_ref
    assert len(excused) <= 6, excused                            # excused (ambiguous rectangle) boxes are rare


def test_engine_armor_stage_feeds_pnp(weights_seed0):
    """enable_armors + enable_pnp: the replay runs detect -> extract_armors -> solvePnP like
    IrmDetector::message_callback (src/irm_detector.cpp:181-208); armors must equal the stand-alone
    stage on the engine's own boxes, poses must equal the PnP oracle on the armor corners."""
    _cuda()
    import irmv_detection_b200 as irmv
    from oracle import armor_ref as A, pnp_ref as P, preprocess_ref as PR
    scenes = [A.synth_armor_scene(10, s)[0] for s in (7, 8, 9)]
    frames = np.stack([PR.rot180(s) for s in scenes])
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), max_batch=3)
    eng.enable_armors(binary_threshold=150)
    eng.enable_pnp(P.K_DEFAULT, P.D_DEFAULT, (0.5, 480 / 1024))
    counts, dets = eng.detect_batch_arrays(frames)
    counts, dets = counts.copy(), dets.copy()
    arm = eng.fetch_armors(3)
    rv, tv, ok = eng.fetch_poses(3)
    alone = irmv.extract_armors(frames, dets, counts)
    n_valid = 0
    for f in range(3):
        k = int(counts[f])
        assert np.array_equal(arm[f]["valid"][:k], alone[f]["valid"][:k])
        v = np.nonzero(arm[f]["valid"][:k])[0]
        assert np.array_equal(arm[f]["pts"][v], alone[f]["pts"][v])
        A.check_armors(arm[f], scenes[f], dets[f]["xyxy"][:k], dets[f]["score"][:k], dets[f]["class_id"][:k], A.ArmorParams())
        assert not ok[f, :k][arm[f]["valid"][:k] == 0].any()
        if len(v):
            pts = arm[f]["pts"][v] * np.array([0.5, 480 / 1024], np.float32)
            r1, t1, r2, t2, e1, e2 = P.solve_ippe(pts, both=True)
            clear = ok[f, v] & np.isfinite(r1).all(1) & (np.abs(e1 - e2) > 1e-6 * np.maximum(e1, e2))
            rel = np.linalg.norm(rv[f, v][clear] - r1[clear], axis=1) / np.linalg.norm(r1[clear], axis=1)
            assert rel.size == 0 or rel.max() < PNP_REL_TOL
            n_valid += len(v)
    # pipelined hand-off: the armors travel with their ticket's result set
    import torch
    pinned = torch.from_numpy(frames).pin_memory().numpy()
    t = eng.submit_batch(pinned)
    c2, d2, rv2, tv2, ok2 = eng.collect_arrays(t, poses=True)
    arm2 = eng.fetch_armors(3, ticket=t)
    assert np.array_equal(c2, counts) and np.array_equal(arm2["valid"], arm["valid"]) and np.array_equal(arm2["pts"], arm["pts"])
    assert np.array_equal(ok2, ok)
    eng.close()
    # (random-init weights put boxes anywhere; the count only documents how much of the path ran)
    print("armors from engine boxes:", n_valid)


def test_cpp_drop_in_classes(base_image, weights_seed0, tmp_path):
    """The C++ YoloEngine / PnPSolver / TripleBuffer with the reference's class interfaces
    (include/irmv_detection/*.hpp), exercised by a program shaped like the reference's
    yolo_engine_benchmark test: same detections as the Python mirror, max time < 30 ms."""
    import shutil
    import subprocess
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import build as B
    _cuda()
    exe = B.DROP_IN_TEST
    if not os.path.exists(exe):
        pytest.skip("drop_in_test not built")
    shutil.copy(weights_seed0, tmp_path / "yolov7.irmw")          # the reference passes models/yolov7.onnx
    base_image.tofile(tmp_path / "frame.raw")
    r = subprocess.run([exe, str(tmp_path / "yolov7.onnx"), str(tmp_path / "frame.raw"), "5"], capture_output=True,
                       text=True, timeout=240)
    assert r.returncode == 0 and "DROP_IN_OK" in r.stdout, f"rc={r.returncode}\nstdout:\n{r.stdout[-2000:]}\nstderr:\n{r.stderr[-2000:]}"
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024))
    eng.get_src_image_buffer(0)[...] = base_image
    dets = eng.detect(0)
    lines = r.stdout.splitlines()
    assert int(lines[0].split()[1]) == len(dets)
    for ln, d in zip([l for l in lines if l.startswith("box ")], dets):
        f = ln.split()
        np.testing.assert_allclose([float(v) for v in f[1:5]], d.xyxy, atol=2e-3)
        assert abs(float(f[6]) - d.score) < 1e-4 and f[8] == d.class_id.name
    pnp = [l for l in lines if l.startswith("pnp ok")][0].split()
    np.testing.assert_allclose([float(v) for v in pnp[4:7]], [1.14443091, -0.9268353, 1.21457493], rtol=1e-6)
    np.testing.assert_allclose([float(v) for v in pnp[8:11]], [0.00508322, 0.02282537, 1.30085669], rtol=1e-6)
    eng.close()
    # ArmorExtractor (IrmDetector::extract_armors): the C++ program's scene through the cv2 form of the reference
    import cv2
    from oracle import armor_ref as A
    img = np.full((1024, 1280, 3), 20, np.uint8)
    img[400:440, 600:606] = 250
    img[402:442, 680:686] = 250
    img[399, 602:604] = 250
    img[401, 682:684] = 250
    ref = A.extract_armors_cv2(img, np.array([[580.5, 380.25, 710, 460]], np.float32), [0.9], [9])
    assert len(ref) == 1 and ref[0].size == A.SMALL
    arm = [l for l in lines if l.startswith("armor size")][0].split()
    assert int(arm[2]) == 0 and arm[4] == "R3"
    got_left = np.array([float(v) for v in arm[8:12]]).reshape(2, 2)       # top, bottom
    got_right = np.array([float(v) for v in arm[13:17]]).reshape(2, 2)
    np.testing.assert_allclose(got_left, ref[0].pts[[1, 0]], atol=2e-3)
    np.testing.assert_allclose(got_right, ref[0].pts[[2, 3]], atol=2e-3)
    assert [l for l in lines if l.startswith("armor pnp ok 1")]


def test_pnp_stress_one_million_properties():
    """BASELINE.json configs[4] at full size: properties that do not need the CPU oracle at 1M --
    every solve succeeds, the returned pose reprojects onto its quad (normalised RMSE of the first
    IPPE solution <= the second), and results are independent of batch position."""
    import irmv_detection_b200 as irmv
    from oracle import pnp_ref as P
    _cuda()
    base = P.synth_quads(5000, seed=3)
    n = 1_000_000
    q = np.tile(base, (n // len(base), 1, 1))
    s = irmv.PnPSolver(P.K_DEFAULT, P.D_DEFAULT)
    rv, tv, ok, quat, rv2, tv2, rmse = s.solve_batch(q, extended=True)
    assert ok.all() and np.isfinite(rv).all() and np.isfinite(tv).all()
    assert (rmse[:, 0] <= rmse[:, 1] + 1e-12).all()
    assert rmse[:, 0].max() < 5e-3                       # 0.5 px noise / f ~ 1e-3 in normalised units
    assert (tv[:, 2] > 0.3).all() and (tv[:, 2] < 12).all()
    np.testing.assert_allclose(np.linalg.norm(quat, axis=1), 1.0, atol=1e-9)
    # tiling: copy k of the base set equals copy 0 bit for bit
    assert np.array_equal(rv[:5000], rv[-5000:]) and np.array_equal(tv[:5000], tv[-5000:])
    r1, t1 = P.solve_ippe(base)
    rel = np.linalg.norm(rv[:5000] - r1, axis=1) / np.linalg.norm(r1, axis=1)
    assert np.quantile(rel, 0.99) < PNP_REL_TOL


# ------------------------------------------------------- the configuration bench.py times, pinned
def _frame_vs_oracle(eng, f, x_nhwc8, wpath):
    """Frame f of the engine's last run (lane 0) against the FP32 oracle on the same network input:
    head tensors -> decoded scores within 1e-2, boxes within 0.5 px, kept indices bit-exact on the
    GPU's own decoded inputs."""
    import irmv_detection_b200 as irmv
    from oracle import nms_ref as N
    _, outs, rboxes, rscores = _oracle_forward(wpath, x_nhwc8)
    box = np.concatenate([eng.read_tensor(f"box{i}")[f:f + 1].reshape(1, -1, 64) for i in range(3)], 1)
    cls = np.concatenate([eng.read_tensor(f"cls{i}")[f:f + 1].reshape(1, -1, 16) for i in range(3)], 1)
    gboxes, gscores = irmv.decode(box, cls)
    assert np.abs(gscores - rscores).max() < SCORE_TOL
    assert np.abs(gboxes - rboxes).max() < BOX_TOL_PX
    ri, _, _, _ = N.nms(gboxes[0], gscores[0])
    return ri, outs


@pytest.mark.parametrize("sub,lanes", [(256, 1), (128, 2)])
def test_bench_configuration_pinned_to_single_frame_engine_and_oracle(base_image, weights_seed0, sub, lanes):
    """bench.py's engine (BASELINE.json configs[3]: Bayer frames, max_batch 256, one 256-frame replay --
    and the round-1 split, two lanes of 128 -- fused PnP) runs kernel instantiations that plan() only
    picks at large tile counts (R = 4 / 2, streamed weights, other ring depths).  Pin that configuration:
    frames at the start, middle and end of every replay must equal a max_batch = 1 engine bit for bit
    (detections, Detect head tensor, poses), and frame 0 must be within tolerance of the FP32 oracle."""
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import synth
    from oracle import pnp_ref as P
    _cuda()
    rgb = synth.frames_from_base(base_image, 16, seed=77)[..., ::-1]
    raw16 = synth.bayer_from_rgb(rgb, "RGGB")
    raw = np.ascontiguousarray(np.tile(raw16[:8], (32, 1, 1)))
    probe = {0: 0, 1: 1, 2: 2, 3: 3, 5: 4, 64: 5, 126: 6, 127: 7, 128: 8, 129: 9, 200: 10, 254: 11, 255: 12}
    for pos, src in probe.items():
        raw[pos] = raw16[src + 3 if src + 3 < 16 else src]
    big = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=irmv.CH_BAYER_RGGB, max_batch=256,
                          sub_batch=sub, num_lanes=lanes)
    big.enable_pnp(P.K_DEFAULT, P.D_DEFAULT, (0.5, 480 / 1024))
    import torch
    raw_dev = torch.from_numpy(raw).cuda()
    res_host = big.detect_batch(raw)           # host frames: 128-frame chunks through the copy stream when sub = 256
    res = big.detect_batch_device(raw_dev.data_ptr(), 256)            # the bench's timed path: device-resident frames
    assert res == res_host
    rv, tv, ok = big.fetch_poses(256)
    box_big = [big.read_tensor(f"box{i}") for i in range(3)]          # lane 0 = frames 0..sub-1
    cls_big = [big.read_tensor(f"cls{i}") for i in range(3)]
    one = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=irmv.CH_BAYER_RGGB)
    one.enable_pnp(P.K_DEFAULT, P.D_DEFAULT, (0.5, 480 / 1024))
    total = 0
    for pos in probe:
        r = one.detect_batch(raw[pos:pos + 1])[0]
        r1, t1, o1 = one.fetch_poses(1)
        assert r == res[pos], f"frame {pos}: detections differ from the batch-1 engine"
        k = len(r)
        total += k
        assert np.array_equal(rv[pos, :k], r1[0, :k]) and np.array_equal(tv[pos, :k], t1[0, :k]), f"frame {pos}: poses"
        assert np.array_equal(ok[pos, :k], o1[0, :k])
        if pos < sub:
            for i in range(3):
                assert np.array_equal(one.read_tensor(f"box{i}")[0], box_big[i][pos]), f"frame {pos} box{i}"
                assert np.array_equal(one.read_tensor(f"cls{i}")[0], cls_big[i][pos]), f"frame {pos} cls{i}"
    assert total > 0
    one.close()
    # the pipelined host path of the same engine (submit_batch replays a 256-frame batch in host chunks of 128
    # frames while the copy of the next chunk runs): same detections and poses as the synchronous call
    cs, ds = big.detect_batch_arrays(raw)
    cs, ds = cs.copy(), ds.copy()
    cp, dp, rvp, tvp, okp = big.collect_arrays(big.submit_batch(raw), poses=True)
    assert np.array_equal(cs, cp)
    for f in range(256):
        k = int(cs[f])
        assert np.array_equal(ds[f, :k], dp[f, :k]), f"pipelined frame {f}"
        assert np.array_equal(rv[f, :k], rvp[f, :k]) and np.array_equal(tv[f, :k], tvp[f, :k]) and np.array_equal(ok[f, :k], okp[f, :k])
    big.detect_batch_device(raw_dev.data_ptr(), 256)                  # lane 0 holds frames 0.. again
    # frame 0 of the replay against the FP32 oracle
    x = irmv.preprocess(raw[:1], irmv.CH_BAYER_RGGB)
    ri, _ = _frame_vs_oracle(big, 0, x, weights_seed0)
    assert np.array_equal(big.kept_indices(0), ri)
    big.close()


def test_keypoint_variant_batch64_pinned(base_image, tmp_path):
    """BASELINE.json configs[2]'s shape (keypoint weight file, batch 64, one replay): frames across the
    replay equal the batch-1 engine bit for bit (detections, keypoints, poses); frame 0 within
    tolerance of the FP32 oracle, raw keypoint tensors included."""
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import synth, weights as W
    from oracle import pnp_ref as P
    _cuda()
    wp = str(tmp_path / "pose_seed0.irmw")
    W.write_random(wp, 0, pose=True)
    fr = synth.frames_from_base(base_image, 64, seed=13)
    big = irmv.YoloEngine(wp, (1280, 1024), max_batch=64, sub_batch=64, num_lanes=1)
    big.enable_pnp(P.K_DEFAULT, P.D_DEFAULT, (0.5, 480 / 1024))
    res = big.detect_batch(fr)
    kp = big.fetch_keypoints(64)
    rv, tv, ok = big.fetch_poses(64)
    raw_k = [big.read_tensor(f"kpt{i}") for i in range(3)]
    one = irmv.YoloEngine(wp, (1280, 1024))
    one.enable_pnp(P.K_DEFAULT, P.D_DEFAULT, (0.5, 480 / 1024))
    for pos in (0, 1, 31, 32, 62, 63):
        r = one.detect_batch(fr[pos:pos + 1])[0]
        assert r == res[pos], f"frame {pos}"
        k = len(r)
        assert np.array_equal(one.fetch_keypoints(1)[0, :k], kp[pos, :k])
        r1, t1, _ = one.fetch_poses(1)
        assert np.array_equal(rv[pos, :k], r1[0, :k]) and np.array_equal(tv[pos, :k], t1[0, :k])
        for i in range(3):
            assert np.array_equal(one.read_tensor(f"kpt{i}")[0], raw_k[i][pos])
    one.close()
    x = irmv.preprocess(fr[:1])
    ri, outs = _frame_vs_oracle(big, 0, x, wp)
    assert np.array_equal(big.kept_indices(0), ri)
    for i in range(3):
        ref = outs[i][2].permute(0, 2, 3, 1).numpy()
        assert np.abs(raw_k[i][:1, ..., :8].astype(np.float32) - ref).max() <= 2e-2 * max(np.abs(ref).max(), 1.0)
    big.close()


def _plan_signatures(plans):
    out = set()
    for p in plans:
        if p[0] == "raster":
            _, k, s, cin, cout, hw, R, nepi, bstream, ctas, stages, bstages, tail, act, res, tiles = p
            out.add(("raster", k, s, R, nepi, bstream, ctas, min(stages, 2), tail, act, res))
        elif p[0] == "gather":
            out.add(("gather", p[1], p[2]))
    return out


def test_every_plan_instantiation_is_oracle_compared(base_image, weights_seed0):
    """plan() (csrc/conv_raster.cu) picks R, weight streaming, CTAs per SM and ring depths from the tile
    count, so different replay sizes run different kernel instantiations.  Enumerate the instantiations
    (k, stride, R, NEPI, b_stream, CTAs/SM, >= 2 stages, tail, act, res) over every replay size 1..256,
    pick replay sizes that cover all of them (greedy, the bench's 256 first), and for each picked size
    require frames at the start, middle and end of the replay to equal the batch-1 engine bit for bit
    (detections + all Detect head tensors) and frame 0 to be within tolerance of the FP32 oracle."""
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import synth
    _cuda()
    NMAX = 256
    big = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=irmv.CH_BAYER_RGGB, max_batch=NMAX, sub_batch=NMAX, num_lanes=1)
    sig = {n: _plan_signatures(big.describe_plans(n)) for n in range(1, NMAX + 1)}
    every = set().union(*sig.values())
    picked, covered = [NMAX], set(sig[NMAX])
    while covered != every:
        n = max(range(1, NMAX + 1), key=lambda m: (len(sig[m] - covered), m))
        picked.append(n)
        covered |= sig[n]
    assert len(picked) <= 12, picked
    rgb = synth.frames_from_base(base_image, 128, seed=55)[..., ::-1]
    raw = synth.bayer_from_rgb(rgb, "RGGB")
    raw = np.ascontiguousarray(np.concatenate([raw, raw[::-1]]))          # 256 frames, no two neighbours alike
    one = irmv.YoloEngine(weights_seed0, (1280, 1024), chan_order=irmv.CH_BAYER_RGGB)
    x0 = irmv.preprocess(raw[:1], irmv.CH_BAYER_RGGB)
    ref = {}
    import torch
    raw_dev = torch.from_numpy(raw).cuda()
    for n in picked:
        res = big.detect_batch_device(raw_dev.data_ptr(), n)       # one replay of n device-resident frames (host batches of > 128 frames are chunked)
        heads = [big.read_tensor(f"{t}{i}") for t in ("box", "cls") for i in range(3)]
        for pos in sorted({0, n // 2, n - 1}):
            if pos not in ref:
                r = one.detect_batch(raw[pos:pos + 1])[0]
                ref[pos] = (r, [one.read_tensor(f"{t}{i}")[0].copy() for t in ("box", "cls") for i in range(3)])
            assert res[pos] == ref[pos][0], f"replay of {n}: frame {pos} detections"
            for h, hr in zip(heads, ref[pos][1]):
                assert np.array_equal(h[pos], hr), f"replay of {n}: frame {pos} head tensor"
        ri, _ = _frame_vs_oracle(big, 0, x0, weights_seed0)
        assert np.array_equal(big.kept_indices(0), ri), f"replay of {n}"
    assert sum(len(v[0]) for v in ref.values()) > 0
    print("replay sizes covering every instantiation:", picked, "instantiations:", len(every))
    one.close(); big.close()


# ------------------------------------------------------- fused message_callback outputs
def _tf2_quaternion(Rm):
    """tf2::Matrix3x3::getRotation (x, y, z, w), the call at reference src/irm_detector.cpp:224-225."""
    tr = Rm[0, 0] + Rm[1, 1] + Rm[2, 2]
    q = np.zeros(4)
    if tr > 0:
        s = np.sqrt(tr + 1.0)
        q[3] = s * 0.5
        s = 0.5 / s
        q[0] = (Rm[2, 1] - Rm[1, 2]) * s; q[1] = (Rm[0, 2] - Rm[2, 0]) * s; q[2] = (Rm[1, 0] - Rm[0, 1]) * s
    else:
        i = (2 if Rm[1, 1] < Rm[2, 2] else 1) if Rm[0, 0] < Rm[1, 1] else (2 if Rm[0, 0] < Rm[2, 2] else 0)
        j, k = (i + 1) % 3, (i + 2) % 3
        s = np.sqrt(Rm[i, i] - Rm[j, j] - Rm[k, k] + 1.0)
        q[i] = s * 0.5
        s = 0.5 / s
        q[3] = (Rm[k, j] - Rm[j, k]) * s
        q[j] = (Rm[j, i] + Rm[i, j]) * s
        q[k] = (Rm[k, i] + Rm[i, k]) * s
    return q


def test_fused_message_callback_outputs(weights_seed0):
    """detect -> extract_armors -> solvePnP -> Rodrigues -> tf2 quaternion -> distance_to_image_center
    (reference src/irm_detector.cpp:181-230) as one replay: the per-armor payload of
    irmv_engine_fetch_armor_poses against cv2.Rodrigues + the tf2 formula + the intended distance, for
    the armor stage (light-bar scene) and for the box-corner pose stage."""
    import cv2
    import irmv_detection_b200 as irmv
    from oracle import armor_ref as A, pnp_ref as P, preprocess_ref as PR
    _cuda()
    cs = (np.float32(0.5), np.float32(480 / 1024))
    cx, cy = np.float32(P.K_DEFAULT[2]), np.float32(P.K_DEFAULT[5])

    def check(poses, rv, tv, ok, centers):
        n_ok = 0
        for i in range(len(poses)):
            p = poses[i]
            assert bool(p["ok"]) == bool(ok[i])
            if not ok[i]:
                continue
            n_ok += 1
            assert np.array_equal(p["position"], tv[i]) and np.array_equal(p["rvec"], rv[i])
            Rm, _ = cv2.Rodrigues(rv[i].reshape(3, 1))
            q = _tf2_quaternion(Rm)
            assert np.abs(p["orientation"] - q).max() < 1e-7, (p["orientation"], q)
            assert abs(np.linalg.norm(p["orientation"]) - 1.0) < 1e-9
            dx, dy = np.float32(centers[i][0]) - cx, np.float32(centers[i][1]) - cy
            want = np.sqrt(np.float32(dx * dx + dy * dy))
            assert abs(float(p["distance_to_image_center"]) - float(want)) <= 1e-4 * max(1.0, float(want))
        return n_ok

    # (1) box-corner pose stage on camera frames
    from irmv_detection_b200 import synth
    fr = synth.frames_from_base(synth.load_base(), 2, seed=4)
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), max_batch=2, sub_batch=2)
    eng.enable_pnp(P.K_DEFAULT, P.D_DEFAULT, cs)
    dets = eng.detect_batch(fr)
    rv, tv, ok = eng.fetch_poses(2)
    poses = eng.fetch_armor_poses(2)
    seen = 0
    for f in range(2):
        k = len(dets[f])
        cen = [((np.float32(d.xyxy[0]) * cs[0] + np.float32(d.xyxy[0]) * cs[0] + np.float32(d.xyxy[2]) * cs[0] + np.float32(d.xyxy[2]) * cs[0]) * np.float32(0.25),
                (np.float32(d.xyxy[3]) * cs[1] + np.float32(d.xyxy[1]) * cs[1] + np.float32(d.xyxy[1]) * cs[1] + np.float32(d.xyxy[3]) * cs[1]) * np.float32(0.25))
               for d in dets[f]]
        seen += check(poses[f, :k], rv[f, :k], tv[f, :k], ok[f, :k], cen)
        assert not poses[f, k:]["ok"].any()
    assert seen > 0
    eng.close()
    # (2) armor stage: seeded light-bar scene, boxes injected through the stand-alone stage + solver
    img, ab, asc, acl = A.synth_armor_scene(6, 3)
    boxes = np.zeros((1, 8), irmv.BBOX_DTYPE)
    boxes["xyxy"][0, :6] = ab; boxes["score"][0, :6] = asc; boxes["class_id"][0, :6] = acl
    arm = irmv.extract_armors(PR.rot180(img)[None], boxes, [6])[0]
    valid = np.nonzero(arm["valid"])[0]
    assert len(valid) > 0
    s = irmv.PnPSolver(P.K_DEFAULT, P.D_DEFAULT)
    pts = arm["pts"][valid] * np.array(cs, np.float32)
    rv, tv, okb, q, _, _, _ = s.solve_batch(pts, extended=True)
    for i in range(len(valid)):
        if okb[i]:
            Rm, _ = cv2.Rodrigues(rv[i].reshape(3, 1))
            assert np.abs(q[i] - _tf2_quaternion(Rm)).max() < 1e-7
            c = arm["center"][valid[i]] * np.array(cs, np.float32)
            d = s.calculateDistanceToCenter(c)
            assert abs(d - float(np.hypot(np.float32(c[0]) - cx, np.float32(c[1]) - cy))) < 1e-3
    s.close()


def test_engine_armor_stage_payload(weights_seed0):
    """Engine-fused armor stage: the payload's distance uses Armor::center, ok is 0 without an armor."""
    import cv2
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import synth
    from oracle import pnp_ref as P
    _cuda()
    cs = (np.float32(0.5), np.float32(480 / 1024))
    fr = synth.frames_from_base(synth.load_base(), 2, seed=4)
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), max_batch=2, sub_batch=2)
    eng.enable_armors(binary_threshold=20, light_min_ratio=0.01, light_max_ratio=10.0, light_max_angle=90.0,
                      min_small_center_distance=0.0, max_large_center_distance=1e9)
    eng.enable_pnp(P.K_DEFAULT, P.D_DEFAULT, cs)
    dets = eng.detect_batch(fr)
    arm = eng.fetch_armors(2)
    rv, tv, ok = eng.fetch_poses(2)
    poses = eng.fetch_armor_poses(2)
    cx, cy = np.float32(P.K_DEFAULT[2]), np.float32(P.K_DEFAULT[5])
    for f in range(2):
        for i in range(len(dets[f])):
            assert bool(poses[f, i]["ok"]) == bool(ok[f, i])
            if ok[f, i]:
                assert arm[f, i]["valid"]
                c = arm[f, i]["center"] * np.array(cs, np.float32)
                want = float(np.sqrt(np.float32((c[0] - cx) * (c[0] - cx) + (c[1] - cy) * (c[1] - cy))))
                assert abs(float(poses[f, i]["distance_to_image_center"]) - want) <= 1e-4 * max(1.0, want)
                Rm, _ = cv2.Rodrigues(rv[f, i].reshape(3, 1))
                assert np.abs(poses[f, i]["orientation"] - _tf2_quaternion(Rm)).max() < 1e-7
    eng.close()


def test_multi_replay_results_land_at_their_frames(weights_seed0, tmp_path):
    """Every result field of a batch replayed as 2 + 2 + 1 frames on two lanes (detections, kept indices, poses,
    armor poses, armors, keypoints) lands at the same frame offsets as from one 5-frame replay: bit-identical,
    synchronous and pipelined."""
    import torch
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import synth, weights as W
    from oracle import armor_ref as A, pnp_ref as P, preprocess_ref as PR
    _cuda()
    wp = str(tmp_path / "pose_seed0.irmw")
    W.write_random(wp, 0, pose=True)
    scenes = [PR.rot180(A.synth_armor_scene(10, s)[0]) for s in (7, 8)]
    fr = np.concatenate([synth.frames_from_base(synth.load_base(), 3, seed=4), np.stack(scenes)])
    pinned = torch.from_numpy(fr).pin_memory().numpy()
    n = len(fr)
    same = lambda a, b: a.shape == b.shape and a.tobytes() == b.tobytes()
    # the extractor writes a whole record where it finds an armor and only `valid` elsewhere
    armors = lambda a: [a["valid"], a[a["valid"] != 0]]

    def run(sub_batch, num_lanes):
        eng = irmv.YoloEngine(wp, (1280, 1024), max_batch=n, sub_batch=sub_batch, num_lanes=num_lanes)
        eng.enable_armors(binary_threshold=20, light_min_ratio=0.01, light_max_ratio=10.0, light_max_angle=90.0,
                          min_small_center_distance=0.0, max_large_center_distance=1e9)
        eng.enable_pnp(P.K_DEFAULT, P.D_DEFAULT, (np.float32(0.5), np.float32(480 / 1024)))
        counts, dets = (a.copy() for a in eng.detect_batch_arrays(fr))
        sync = {"dets": [counts, *(dets[f, :counts[f]] for f in range(n))], "kept": [eng.kept_indices(f) for f in range(n)],
                "poses": list(eng.fetch_poses(n)), "armor_poses": [eng.fetch_armor_poses(n)],
                "armors": armors(eng.fetch_armors(n)), "kpts": [eng.fetch_keypoints(n)]}
        t = eng.submit_batch(pinned)
        c, d, rv, tv, ok = (a.copy() for a in eng.collect_arrays(t, poses=True))
        piped = {"dets": [c, *(d[f, :c[f]] for f in range(n))], "poses": [rv, tv, ok],
                 "armor_poses": [eng.fetch_armor_poses(n, ticket=t)], "armors": armors(eng.fetch_armors(n, ticket=t)),
                 "kpts": [eng.fetch_keypoints(n, ticket=t)]}
        eng.close()
        return sync, piped

    (sync_a, piped_a), (sync_b, piped_b) = run(2, 2), run(n, 1)
    assert sync_a["armor_poses"][0]["ok"].any(), "no armor was solved: the comparison would not cover the armor poses"
    # A against B, and the pipelined results against the synchronous ones
    for x, y in ((sync_a, sync_b), (piped_a, piped_b), (piped_a, sync_a)):
        for key, xs in x.items():
            assert len(xs) == len(y[key]) and all(same(a, b) for a, b in zip(xs, y[key])), key


# ------------------------------------------------------- host-path hygiene
def test_per_frame_calls_do_not_allocate(base_image, weights_seed0):
    """After construction and one warm call, detect(), get_rotated_image(), detect_batch(), the pipelined
    hand-off and the PnP batch call make no device or pinned allocation (VERDICT r1: cudaMalloc inside
    irmv_pnp_solve_batch_ex and irmv_engine_rotated_image)."""
    import torch
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import _lib
    from oracle import pnp_ref as P
    _cuda()
    lib = _lib.lib()
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), max_batch=4, sub_batch=2, num_lanes=2)
    eng.enable_pnp(P.K_DEFAULT, P.D_DEFAULT, (0.5, 480 / 1024))
    eng.get_src_image_buffer(0)[...] = base_image
    eng.get_src_image_buffer(1)[...] = base_image[::-1]
    host = torch.empty((4,) + base_image.shape, dtype=torch.uint8, pin_memory=True).numpy()
    host[...] = base_image
    s = irmv.PnPSolver(P.K_DEFAULT, P.D_DEFAULT)
    quads = P.synth_quads(500, seed=1)
    # warm: lazily created graphs, result sets, staging and rotated buffers
    eng.detect(0); eng.detect(1)
    v0 = eng.get_rotated_view(0)
    eng.detect_batch_arrays(host)
    for _ in range(3):
        eng.collect_arrays(eng.submit_batch(host))
    s.solve_batch(quads, extended=True)
    before = lib.irmv_debug_alloc_count()
    for _ in range(3):
        eng.detect(0)
        a = eng.get_rotated_view(0)
        eng.detect(1)
        b = eng.get_rotated_view(1)
        eng.detect_batch_arrays(host)
        eng.fetch_poses(4); eng.fetch_armor_poses(4)
        t = [eng.submit_batch(host) for _ in range(3)]
        for x in t:
            eng.collect_arrays(x, poses=True)
        s.solve_batch(quads[:300], extended=True)
        s.solvePnP(quads[0])
    assert lib.irmv_debug_alloc_count() == before
    # the view is address-stable and holds the rotated frame of the slot's last detect()
    assert a.ctypes.data == v0.ctypes.data
    assert np.array_equal(a, base_image[::-1, ::-1]) and np.array_equal(b, base_image[:, ::-1])
    assert np.array_equal(eng.get_rotated_image(0), base_image[::-1, ::-1])
    s.close(); eng.close()


def test_pipelined_handoff_state_is_checked(base_image, weights_seed0):
    """ADVICE r1: a fourth submit before a collect, stale / duplicate / out-of-order tickets and synchronous
    calls while batches are in flight are errors, not silent reads of another batch's results."""
    import torch
    import irmv_detection_b200 as irmv
    _cuda()
    eng = irmv.YoloEngine(weights_seed0, (1280, 1024), max_batch=2, sub_batch=2)
    host = torch.empty((2,) + base_image.shape, dtype=torch.uint8, pin_memory=True).numpy()
    host[...] = base_image
    eng.get_src_image_buffer(0)[...] = base_image
    with pytest.raises(irmv.IrmvError):
        eng.collect_arrays(0)                              # never submitted
    t0, t1, t2 = (eng.submit_batch(host) for _ in range(3))
    with pytest.raises(irmv.IrmvError):
        eng.submit_batch(host)                             # a fourth batch would overwrite set 0
    with pytest.raises(irmv.IrmvError):
        eng.detect(0)                                      # synchronous call while batches are in flight
    with pytest.raises(irmv.IrmvError):
        eng.detect_batch_arrays(host)
    with pytest.raises(irmv.IrmvError):
        eng.collect_arrays(t1)                             # out of order
    c0, d0 = (np.copy(x) for x in eng.collect_arrays(t0))
    with pytest.raises(irmv.IrmvError):
        eng.collect_arrays(t0)                             # duplicate
    eng.collect_arrays(t1); eng.collect_arrays(t2)
    with pytest.raises(irmv.IrmvError):
        eng.collect_arrays(t0 + 3)                         # not issued yet
    ref = eng.detect(0)                                    # everything collected: synchronous calls work again
    assert len(ref) == int(c0[0])
    eng.close()


def test_weight_file_validation(tmp_path, weights_seed0):
    """ADVICE r1: a corrupt or foreign weight file is refused with an error (nothing throws across the
    ABI, nothing is indexed past its shape)."""
    import struct
    import irmv_detection_b200 as irmv
    _cuda()
    blob = open(weights_seed0, "rb").read()
    cases = {
        "truncated": blob[: len(blob) // 2],
        "huge_count": blob[:12] + struct.pack("<I", 0x7fffffff) + blob[16:],
        "bad_k": blob[:16] + struct.pack("<5I", 3, 16, 5, 2, 1) + blob[36:],
        "huge_cin": blob[:16] + struct.pack("<5I", 0x40000000, 16, 3, 2, 1) + blob[36:],
        "wrong_shape": blob[:16] + struct.pack("<5I", 3, 16, 3, 1, 1) + blob[36:],     # stride 1 conv0
    }
    for name, data in cases.items():
        p = tmp_path / f"{name}.irmw"
        p.write_bytes(data)
        with pytest.raises(irmv.IrmvError):
            irmv.YoloEngine(str(p), (1280, 1024))


def test_split_upsample_convs_match_the_gather_path(frames, weights_seed0):
    """The neck's cv1 over concat(upsample(a), b) runs as W_a . a at a's resolution + W_b . b with the partial sum
    added before the activation (two raster-kernel launches, conv_raster RES = 2) by default, or as one
    gather-kernel launch (cfg.reserved[3]).  Same network either way: the module outputs agree to FP16 rounding of
    the partial sum, both launch lists are what the design says (4 vs 6 gather launches), and the decoded boxes /
    scores of the two FP16 paths -- each within the north_star tolerance of the FP32 oracle on its own
    (test_network_parity[tcgen05], [tcgen05_gather_neck]) -- lie within twice that of each other."""
    import irmv_detection_b200 as irmv
    _cuda()
    fr = frames[[0, 2, 3]]                       # the frames of test_network_parity
    a = irmv.YoloEngine(weights_seed0, (1280, 1024), max_batch=3, sub_batch=3)
    b = irmv.YoloEngine(weights_seed0, (1280, 1024), max_batch=3, sub_batch=3, split_upsample_convs=False)
    ga = sum(1 for o in a.describe_ops() if o["kind"] == "conv" and not o["raster"])
    gb = sum(1 for o in b.describe_ops() if o["kind"] == "conv" and not o["raster"])
    assert (ga, gb) == (4, 6)
    assert len(a.describe_ops()) == len(b.describe_ops()) + 2
    da, db = a.detect_batch(fr), b.detect_batch(fr)
    for name in ("m12", "m15", "m18", "m21"):
        x, y = a.read_tensor(name).astype(np.float32), b.read_tensor(name).astype(np.float32)
        assert np.abs(x - y).max() <= 4e-3 * max(np.abs(y).max(), 1.0), name
    box = [np.concatenate([e.read_tensor(f"box{i}").reshape(3, -1, 64) for i in range(3)], 1) for e in (a, b)]
    cls = [np.concatenate([e.read_tensor(f"cls{i}").reshape(3, -1, 16) for i in range(3)], 1) for e in (a, b)]
    (ba, sa), (bb, sb) = irmv.decode(box[0], cls[0]), irmv.decode(box[1], cls[1])
    assert np.abs(sa - sb).max() < 2 * SCORE_TOL and np.abs(ba - bb).max() < 2 * BOX_TOL_PX
    assert sum(len(d) for d in da) > 0 and abs(sum(len(d) for d in da) - sum(len(d) for d in db)) <= 2
    a.close(); b.close()


# ------------------------------------------------------- ShuffleNetV2-backbone keypoint detector (configs[2])
@pytest.fixture(scope="module")
def weights_shuffle(tmp_path_factory):
    from irmv_detection_b200 import weights as W
    p = tmp_path_factory.mktemp("ws") / "shufflenetv2_pose_seed0.irmw"
    W.write_random(str(p), 0, arch="shufflenetv2-pose")
    return str(p)


@pytest.mark.parametrize("fuse_units", [True, False])
def test_shufflenet_variant_parity(frames, weights_shuffle, fuse_units):
    """BASELINE.json configs[2], north_star "depthwise and elementwise layers are fused bandwidth-bound
    kernels": the keypoint detector on the ShuffleNetV2-style backbone.  Depthwise 3x3 kernel + 1x1 convs on
    the tcgen05 raster kernel, channel split / concat / shuffle folded into plane runs and weight
    permutations (zero bytes moved).  Every stage output (un-permuted by read_tensor), the neck taps and the
    three head tensors against the FP32 oracle; decoded scores / boxes / keypoints within the north_star
    tolerances; kept indices bit-exact on the GPU's own decoded inputs.  fuse_units: each ShuffleNetV2 unit
    as ONE kernel (shuffle_unit.cu; intermediates in shared memory) or one launch per convolution -- the two
    store the same FP16 intermediates and differ only in the tensor cores' accumulation order."""
    import torch
    import irmv_detection_b200 as irmv
    from oracle import nms_ref as N, pnp_ref as P, yolov8n_ref as Y
    _cuda()
    fr = frames[[0, 2, 3]]
    n = fr.shape[0]
    eng = irmv.YoloEngine(weights_shuffle, (1280, 1024), max_batch=n, sub_batch=n, fuse_units=fuse_units)
    assert eng.has_keypoints()
    kinds = [o["kind"] for o in eng.describe_ops()]
    if fuse_units:
        assert kinds.count("unit") == 7 and kinds.count("dw") == 3       # the h = 128 stage stays one launch per conv
        other = irmv.YoloEngine(weights_shuffle, (1280, 1024), max_batch=n, sub_batch=n, fuse_units=False)
        other.detect_batch(fr)
        eng.detect_batch(fr)
        for name in ("d1", "d2", "d3", "d4", "box0", "cls2", "kpt1"):
            a, b = eng.read_tensor(name).astype(np.float32), other.read_tensor(name).astype(np.float32)
            assert np.abs(a - b).max() <= 4e-3 * max(np.abs(b).max(), 1.0), name     # mma.sync vs tcgen05 accumulation order
        other.close()
    else:
        assert kinds.count("dw") == 13 and kinds.count("unit") == 0
    # (the engine refuses to build unless every backbone 1x1 runs on the tcgen05 raster kernel; the two
    # neck convs over concat(upsample, skip) are the only gather-kernel launches left)
    assert sum(1 for o in eng.describe_ops() if o["kind"] == "conv" and not o["raster"]) <= 4
    eng.enable_pnp(P.K_DEFAULT, P.D_DEFAULT, (0.5, 480 / 1024))
    dets = eng.detect_batch(fr)
    kp = eng.fetch_keypoints(n)
    x = irmv.preprocess(fr)
    m = Y.build(weights_shuffle)
    taps = {}
    with torch.no_grad():
        outs = m.features(torch.from_numpy(x[..., :3].astype(np.float32)).permute(0, 3, 1, 2).contiguous(), taps)
        rboxes, rscores = Y.decode_heads(outs)
        rk = Y.decode_keypoints(outs).numpy()
    rboxes, rscores = rboxes.numpy(), rscores.numpy()
    seen = 0
    for name, ref in taps.items():
        try:
            got = eng.read_tensor(name).astype(np.float32)
        except RuntimeError:
            continue
        seen += 1
        ref = ref.permute(0, 2, 3, 1).numpy()
        err, scale = np.abs(got - ref).max(), np.abs(ref).max()
        assert err <= 2e-2 * max(scale, 1.0), f"{name}: max err {err} (scale {scale})"
    assert seen >= 9 and all(k in taps for k in ("d1", "d2", "d3", "d4"))
    box = np.concatenate([eng.read_tensor(f"box{i}").reshape(n, -1, 64) for i in range(3)], 1)
    cls = np.concatenate([eng.read_tensor(f"cls{i}").reshape(n, -1, 16) for i in range(3)], 1)
    gboxes, gscores = irmv.decode(box, cls)
    assert np.abs(gscores - rscores).max() < SCORE_TOL
    assert np.abs(gboxes - rboxes).max() < BOX_TOL_PX
    for i in range(3):
        got = eng.read_tensor(f"kpt{i}").astype(np.float32)[..., :8]
        ref = outs[i][2].permute(0, 2, 3, 1).numpy()
        assert np.abs(got - ref).max() <= 2e-2 * max(np.abs(ref).max(), 1.0), f"kpt{i}"
    scale = np.array([1280 / 640, 1024 / 640], np.float32)
    total = 0
    for f in range(n):
        ri, rb, rs, rc = N.nms(gboxes[f], gscores[f])
        assert np.array_equal(eng.kept_indices(f), ri), f"frame {f}"
        assert len(dets[f]) == len(ri)
        total += len(ri)
        if len(ri):
            assert np.abs(kp[f, :len(ri)] - rk[f, ri // 14] * scale).max() < BOX_TOL_PX * 2.0     # 0.5 px at network scale
        oi, ob, os_, oc = N.nms(rboxes[f], rscores[f])
        confident = [k for k in range(len(oi)) if os_[k] > 0.25 + 2 * SCORE_TOL]
        missing = [k for k in confident if int(oi[k]) not in set(ri.tolist())]
        assert len(missing) <= max(1, len(confident) // 20)
    assert total > 0
    eng.close()


def test_shufflenet_variant_batch64_pinned(base_image, weights_shuffle):
    """configs[2]'s own shape: batch 64 in one replay.  Frames across the replay equal the batch-1 engine bit
    for bit (detections, keypoints, poses, raw keypoint tensors); frame 0 within tolerance of the FP32 oracle."""
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import synth
    from oracle import pnp_ref as P
    _cuda()
    fr = synth.frames_from_base(base_image, 64, seed=29)
    big = irmv.YoloEngine(weights_shuffle, (1280, 1024), max_batch=64, sub_batch=64, num_lanes=1)
    big.enable_pnp(P.K_DEFAULT, P.D_DEFAULT, (0.5, 480 / 1024))
    res = big.detect_batch(fr)
    kp = big.fetch_keypoints(64)
    rv, tv, ok = big.fetch_poses(64)
    raw_k = [big.read_tensor(f"kpt{i}") for i in range(3)]
    d3 = big.read_tensor("d3")
    one = irmv.YoloEngine(weights_shuffle, (1280, 1024))
    one.enable_pnp(P.K_DEFAULT, P.D_DEFAULT, (0.5, 480 / 1024))
    for pos in (0, 1, 31, 32, 62, 63):
        r = one.detect_batch(fr[pos:pos + 1])[0]
        assert r == res[pos], f"frame {pos}"
        k = len(r)
        assert np.array_equal(one.fetch_keypoints(1)[0, :k], kp[pos, :k])
        r1, t1, _ = one.fetch_poses(1)
        assert np.array_equal(rv[pos, :k], r1[0, :k]) and np.array_equal(tv[pos, :k], t1[0, :k])
        for i in range(3):
            assert np.array_equal(one.read_tensor(f"kpt{i}")[0], raw_k[i][pos])
        assert np.array_equal(one.read_tensor("d3")[0], d3[pos])
    one.close()
    x = irmv.preprocess(fr[:1])
    ri, outs = _frame_vs_oracle(big, 0, x, weights_shuffle)
    assert np.array_equal(big.kept_indices(0), ri)
    big.close()


@pytest.mark.parametrize("arch,n,chan", [("yolov8n", 1, "rgb"), ("yolov8n", 5, "bayer"), ("yolov8n", 32, "bayer"),
                                         ("shuffle", 2, "rgb"), ("shuffle", 5, "bayer"), ("shuffle", 64, "bayer")])
def test_activation_padding_stays_zero(base_image, weights_seed0, weights_shuffle, arch, n, chan):
    """Memory check in place of a sanitizer run: every activation tensor is a zero-padded raster (guard pixels,
    a zero row per image, a zero column) and every kernel relies on the padding staying zero, so a store
    outside a kernel's own pixels lands either in the padding or in another frame.  After full runs (armor and
    pose stages on, ragged sub-batches, repeated replays) no padding pixel of any tensor of any lane may be
    non-zero, and repeating the batch gives identical detections (no stray store into a neighbour's pixels)."""
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import synth
    from oracle import pnp_ref as P
    _cuda()
    fr = synth.frames_from_base(base_image, n, seed=41)
    if chan == "bayer":
        fr, order = synth.bayer_from_rgb(fr[..., ::-1], "RGGB"), irmv.CH_BAYER_RGGB
    else:
        order = irmv.CH_PASSTHROUGH
    w = weights_seed0 if arch == "yolov8n" else weights_shuffle
    sub = max(1, min(n, 32) if n != 5 else 2)          # n = 5, sub-batch 2: ragged last sub-batch
    eng = irmv.YoloEngine(w, (1280, 1024), chan_order=order, max_batch=n, sub_batch=sub, num_lanes=2 if n > sub else 1)
    assert eng.check_padding() == 0, "padding not zero after construction"
    eng.enable_armors()
    eng.enable_pnp(P.K_DEFAULT, P.D_DEFAULT, (0.5, 480 / 1024))
    first = eng.detect_batch(fr)
    assert eng.check_padding() == 0, "a kernel stored into the padding"
    for _ in range(2):
        assert eng.detect_batch(fr) == first
    if n > 1:
        eng.detect_batch(fr[:1])
        assert eng.detect_batch(fr) == first
    assert eng.check_padding() == 0
    eng.close()
