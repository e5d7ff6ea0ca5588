"""CPU suite: pins the oracles against the binary oracles available here (cv2 4.13) and the
committed golden vectors; checks host logic and that the C-ABI library exports every declared
symbol.  No GPU compute."""
import hashlib
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


# ----------------------------------------------------------------------------------- PnP
def test_pnp_oracle_known_answer():
    from oracle import pnp_ref as P
    q = np.array([[[300, 320], [302, 280], [400, 282], [398, 322]]], np.float32)
    r, t, r2, t2, e1, e2 = P.solve_ippe(q, both=True)
    # SURVEY.md section 8c, measured with cv2 4.13
    np.testing.assert_allclose(r[0], [1.14443091, -0.9268353, 1.21457493], rtol=2e-6)
    np.testing.assert_allclose(t[0], [0.00508322, 0.02282537, 1.30085669], rtol=2e-6)
    np.testing.assert_allclose(r2[0], [1.29618529, -1.43086736, 1.25301183], rtol=2e-6)


def test_pnp_oracle_matches_cv2_and_golden():
    from oracle import pnp_ref as P
    g = np.load(os.path.join(GOLD, "pnp_golden.npz"))
    r, t = P.solve_ippe(g["quads"])
    rel = lambda a, b: np.linalg.norm(a - b, axis=1) / np.linalg.norm(b, axis=1)
    assert rel(r, g["rvec"]).max() < 1e-9 and rel(t, g["tvec"]).max() < 1e-9
    q = P.synth_quads(300, seed=123)
    rc, tc, ok = P.solve_cv2(q)
    r, t = P.solve_ippe(q)
    assert ok.all() and rel(r, rc).max() < 1e-9 and rel(t, tc).max() < 1e-9


def test_pnp_oracle_noise_free_recovers_pose():
    from oracle import pnp_ref as P
    rv0, tv0 = np.array([1.2, -1.2, 1.2]), np.array([0.1, -0.05, 2.0])
    pts = P.project(rv0, tv0).astype(np.float32)[None]
    r, t = P.solve_ippe(pts)
    np.testing.assert_allclose(r[0], rv0, atol=2e-5)
    np.testing.assert_allclose(t[0], tv0, atol=2e-5)


def test_undistort_matches_cv2():
    import cv2
    from oracle import pnp_ref as P
    pts = np.random.default_rng(0).uniform(0, 640, (50, 1, 2))
    ref = cv2.undistortPoints(pts, P.K_DEFAULT.reshape(3, 3), P.D_DEFAULT.reshape(1, 5)).reshape(-1, 2)
    got = P.undistort_points(pts.reshape(-1, 2))
    np.testing.assert_allclose(got, ref, atol=1e-12)


# ----------------------------------------------------------------------------------- NMS
def test_nms_oracle_golden_and_cv2():
    import cv2
    from oracle import nms_ref as N
    g = np.load(os.path.join(GOLD, "nms_golden.npz"))
    boxes = np.zeros((8400, 4), np.float32)
    scores = np.zeros((8400, 14), np.float32)
    boxes[g["used"]] = g["boxes"]
    scores[g["used"]] = g["scores"]
    keep, kb, ks, kc = N.nms(boxes, scores)
    assert np.array_equal(keep, g["keep"]) and np.array_equal(ks, g["keep_scores"])
    # cross-check: class-aware OpenCV NMS on the same candidates
    a, c = np.nonzero(scores > 0.25)
    xywh = [[float(b[0]), float(b[1]), float(b[2] - b[0]), float(b[3] - b[1])] for b in boxes[a]]
    sel = cv2.dnn.NMSBoxesBatched(xywh, scores[a, c].tolist(), c.tolist(), 0.25, 0.45)
    got = sorted(int(a[i]) * 14 + int(c[i]) for i in np.asarray(sel).ravel())
    assert got == sorted(keep.tolist())


def test_nms_oracle_rules():
    from oracle import nms_ref as N
    b = np.zeros((4, 4), np.float32)
    s = np.zeros((4, 14), np.float32)
    b[0] = b[1] = b[2] = [0, 0, 10, 10]
    b[3] = [100, 100, 110, 110]
    s[0, 1] = s[1, 1] = 0.9          # tie: lower flat index wins, the other is suppressed
    s[2, 2] = 0.8                    # other class: kept
    s[3, 1] = 0.25                   # exactly at threshold: dropped
    keep, _, _, kc = N.nms(b, s)
    assert keep.tolist() == [0 * 14 + 1, 2 * 14 + 2]
    keep, _, _, _ = N.nms(b, s, max_det=1)
    assert keep.tolist() == [1]
    out, sc, cls = N.parse_output(np.array([[64, 64, 128, 128]], np.float32), np.array([0.5], np.float32),
                                  np.array([17]), 1280, 1024)
    assert out.tolist() == [[128.0, 102.4000015258789, 256.0, 204.8000030517578]] and cls.tolist() == [14]


# ----------------------------------------------------------------------------------- preprocess
def test_preprocess_oracle_golden(base_image):
    from oracle import preprocess_ref as PR
    g = np.load(os.path.join(GOLD, "pre_golden.npz"))
    for chan, rot, quant in [(0, True, True), (1, True, True), (0, False, True), (0, True, False)]:
        x, _ = PR.preprocess_fp16(base_image, chan, rot, quant)
        key = f"c{chan}_r{int(rot)}_q{int(quant)}"
        sha = np.frombuffer(hashlib.sha256(np.ascontiguousarray(x).tobytes()).digest(), np.uint8)
        assert np.array_equal(sha, g[key + "_sha"]), key
        assert np.array_equal(x[:, 300:316, 300:316], g[key + "_crop"])


def test_preprocess_oracle_matches_reference_npp_capture(base_image):
    """tests/golden/npp_rm_golden.npz = output of the reference's own NPP chain (oracle/npp_ref.cpp)
    for test/rm_test.jpg on a B200: the restatement must equal it bit for bit."""
    from oracle import preprocess_ref as PR
    g = np.load(os.path.join(GOLD, "npp_rm_golden.npz"))
    x, _ = PR.preprocess(base_image)
    u8 = np.rint(x * 255.0).astype(np.uint8)
    assert np.array_equal(u8[:, 288:352, 288:352], g["crop"])
    assert np.array_equal(np.frombuffer(hashlib.sha256(np.ascontiguousarray(u8).tobytes()).digest(), np.uint8), g["sha"])


def test_preprocess_oracle_vs_cv2(base_image):
    """BASELINE.md section 3 CPU form (cv2.flip + cv2.resize LINEAR): same half-pixel convention;
    OpenCV's 11-bit fixed-point lerp may differ by one 8-bit step."""
    from oracle import preprocess_ref as PR
    rnd = np.random.default_rng(1).integers(0, 256, base_image.shape, dtype=np.uint8)
    for img in (base_image, rnd):
        a, rot_a = PR.preprocess(img, half_pixel=True)
        b, rot_b = PR.preprocess_cv2(img)
        assert np.array_equal(rot_a, rot_b)
        d = np.abs(a - b) * 255.0
        assert d.max() <= 1.0 + 1e-3 and (d > 0.5).mean() < 0.15


def test_demosaic_oracle_vs_cv2_interior(base_image):
    import cv2
    from oracle import preprocess_ref as PR
    rgb = base_image[..., ::-1]
    codes = {PR.CH_BAYER_RGGB: cv2.COLOR_BayerRGGB2RGB, PR.CH_BAYER_BGGR: cv2.COLOR_BayerBGGR2RGB,
             PR.CH_BAYER_GRBG: cv2.COLOR_BayerGRBG2RGB, PR.CH_BAYER_GBRG: cv2.COLOR_BayerGBRG2RGB}
    for pat, code in codes.items():
        raw = PR.mosaic_from_rgb(rgb, pat)
        ours = PR.demosaic_bilinear(raw, pat)
        ref = cv2.cvtColor(raw, code)
        assert np.array_equal(ours[2:-2, 2:-2], ref[2:-2, 2:-2]), pat


def test_synth_bayer_matches_oracle_mosaic(base_image):
    from irmv_detection_b200 import synth
    from oracle import preprocess_ref as PR
    rgb = base_image[..., ::-1]
    for name, pat in (("RGGB", 2), ("BGGR", 3), ("GRBG", 4), ("GBRG", 5)):
        assert np.array_equal(synth.bayer_from_rgb(rgb, name), PR.mosaic_from_rgb(rgb, pat))


# ----------------------------------------------------------------------------------- network
def test_weights_inventory(tmp_path):
    from irmv_detection_b200 import weights as W
    specs = W.conv_specs()
    assert len(specs) == 63
    assert abs(W.total_flops() - 8.0956416e9) < 1e3                 # SURVEY.md section 8d
    params = sum(c.cout * c.cin * c.k * c.k + c.cout for c in specs)
    assert params == 3008362                                         # SURVEY.md section 8d
    p = tmp_path / "w.irmw"
    W.write_random(str(p), 0)
    nc, t = W.load(str(p))
    assert nc == 14 and len(t) == 63
    ref = W.random_init(0)
    assert all(np.array_equal(a[1], b[0]) and np.array_equal(a[2], b[1]) for a, b in zip(t, ref))
    assert all(np.array_equal(w.astype(np.float16).astype(np.float32), w) for _, w, _ in t)   # FP16-exact


def test_network_oracle_golden(base_image, weights_seed0):
    import torch
    from oracle import nms_ref as N, preprocess_ref as PR, yolov8n_ref as Y
    g = np.load(os.path.join(GOLD, "net_golden.npz"))
    sha = np.frombuffer(hashlib.sha256(open(weights_seed0, "rb").read()).digest(), np.uint8)
    assert np.array_equal(sha, g["weights_sha"])
    m = Y.build(weights_seed0)
    x, _ = PR.preprocess_fp16(base_image)
    with torch.no_grad():
        boxes, scores = m(torch.from_numpy(x.astype(np.float32))[None])
    boxes, scores = boxes[0].numpy(), scores[0].numpy()
    top = g["top_index"]
    np.testing.assert_allclose(scores.reshape(-1)[top], g["top_scores"], atol=1e-4)
    np.testing.assert_allclose(boxes[top // 14], g["top_boxes"], atol=1e-2)
    keep, kb, ks, kc = N.nms(boxes, scores)
    assert len(set(keep.tolist()) & set(g["keep"].tolist())) >= 0.9 * len(g["keep"])


def test_network_oracle_vs_opencv_dnn(base_image, weights_seed0, tmp_path):
    """Second opinion on the FP32 oracle: the same module through ONNX + OpenCV-DNN
    (the CPU baseline form of BASELINE.md section 3)."""
    import cv2
    import torch
    from oracle import export_onnx, preprocess_ref as PR, yolov8n_ref as Y
    m = Y.build(weights_seed0)
    path = str(tmp_path / "yolov8n.onnx")
    try:
        export_onnx.export(m, path)
    except Exception as e:          # exporter internals differ between torch builds
        pytest.skip(f"ONNX export unavailable: {e}")
    net = cv2.dnn.readNetFromONNX(path)
    x, _ = PR.preprocess(base_image)
    net.setInput(x[None])
    out = net.forward()
    with torch.no_grad():
        boxes, scores = m(torch.from_numpy(x)[None])
    ref = torch.cat((boxes, scores), 2).numpy()
    assert out.shape == ref.shape
    assert np.abs(out - ref).max() < 5e-3


def test_keypoint_variant_weights_and_decode(tmp_path):
    """72-conv weight file = the 63 detector convs of the same seed + the Pose branch; keypoint decode is
    (raw * 2 + grid) * stride in anchor order (ultralytics Pose.kpts_decode, kpt_shape [4, 2])."""
    import torch
    from irmv_detection_b200 import weights as W
    from oracle import yolov8n_ref as Y
    p = str(tmp_path / "pose.irmw")
    d = str(tmp_path / "det.irmw")
    W.write_random(p, 0, pose=True)
    W.write_random(d, 0)
    a, b = W.load(p)[1], W.load(d)[1]
    assert len(a) == 72 and len(b) == 63
    assert all(np.array_equal(x[1], y[1]) and np.array_equal(x[2], y[2]) for x, y in zip(a, b))
    assert [c.name for c, _, _ in a[63:66]] == ["m22.kpt0.0", "m22.kpt0.1", "m22.kpt0.2"] and a[65][0].cout == 8
    m = Y.build(p)
    assert m.pose
    outs = [(torch.zeros(1, 64, hw, hw), torch.zeros(1, 14, hw, hw), torch.zeros(1, 8, hw, hw)) for hw in (80, 40, 20)]
    outs[1][2][0, :, 3, 5] = torch.tensor([0.25, -0.5, 0.0, 0.0, 1.0, 1.0, -0.25, 0.125])
    k = Y.decode_keypoints(outs).numpy()
    a_idx = 6400 + 3 * 40 + 5
    np.testing.assert_allclose(k[0, a_idx], [[(0.5 + 5) * 16, (-1.0 + 3) * 16], [5 * 16, 3 * 16], [(2 + 5) * 16, (2 + 3) * 16],
                                             [(-0.5 + 5) * 16, (0.25 + 3) * 16]])
    np.testing.assert_allclose(k[0, 0], [[0, 0]] * 4)
    np.testing.assert_allclose(k[0, 8399], [[19 * 32, 19 * 32]] * 4)


# ----------------------------------------------------------------------------- light bars / armors
def test_armor_gray_is_cv2_bgr2gray():
    import cv2
    from oracle import armor_ref as A
    img = np.random.default_rng(3).integers(0, 256, (120, 200, 3), dtype=np.uint8)
    assert np.array_equal(A.gray_bgr2gray(img), cv2.cvtColor(img, cv2.COLOR_BGR2GRAY))


def test_armor_contours_match_cv2_point_for_point():
    """Top-level outer borders, CHAIN_APPROX_SIMPLE vertices and OpenCV's contour order, on noise,
    dilated noise, rings with nested blobs, single rows/columns and empty images."""
    import cv2
    from oracle import armor_ref as A
    rng = np.random.default_rng(1)
    total = 0
    for t in range(160):
        h, w = int(rng.integers(1, 40)), int(rng.integers(1, 50))
        b = rng.random((h, w)) < rng.choice([0.0, 0.1, 0.3, 0.5, 0.7, 0.9, 1.0])
        if t % 3 == 0:
            b = cv2.dilate(b.astype(np.uint8), np.ones((3, 3), np.uint8)) > 0
        if t % 5 == 0 and h > 10 and w > 10:
            b = np.zeros((h, w), bool)
            cv2.circle(b.view(np.uint8), (w // 2, h // 2), min(h, w) // 2 - 1, 1, 2)
            b[h // 2 - 1:h // 2 + 1, w // 2 - 1:w // 2 + 1] = True      # a blob inside the ring: not external
        ref, _ = cv2.findContours((b * 255).astype(np.uint8), cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_SIMPLE)
        mine = A.find_external_contours(b)
        assert len(ref) == len(mine), t
        for r, m in zip(ref, mine):
            assert np.array_equal(r.reshape(-1, 2), m), t
        total += len(ref)
    assert total > 500


def test_armor_min_area_rect_matches_cv2():
    import cv2
    from oracle import armor_ref as A
    rng = np.random.default_rng(2)
    n = amb = 0
    for _ in range(600):
        pts = rng.integers(0, rng.integers(3, 60), (int(rng.integers(3, 30)), 2)).astype(np.int32)
        c, cen, a = A.min_area_rect(pts)
        if a:
            amb += 1
            continue
        rect = cv2.minAreaRect(pts.reshape(-1, 1, 2))
        bp = cv2.boxPoints(rect)
        d = np.abs(c[:, None, :] - bp[None, :, :]).sum(-1)
        assert d.min(1).max() < 1e-3 and np.abs(cen - np.array(rect[0])).max() < 1e-3
        n += 1
    assert n > 500 and amb < 100


def test_extract_armors_restatement_matches_cv2_and_golden():
    from oracle import armor_ref as A
    g = np.load(os.path.join(ROOT, "tests", "golden", "armor_golden.npz"))
    for seed in (0, 1, 2):
        img, boxes, scores, classes = A.synth_armor_scene(8, seed)
        assert np.array_equal(boxes, g[f"boxes{seed}"])
        a1 = A.extract_armors(img, boxes, scores, classes)
        a2 = A.extract_armors_cv2(img, boxes, scores, classes)
        assert [a.bbox_index for a in a1] == [a.bbox_index for a in a2] == g[f"index{seed}"].tolist()
        assert [a.size for a in a1] == [a.size for a in a2] == g[f"size{seed}"].tolist()
        for k, (x, y) in enumerate(zip(a1, a2)):
            assert np.abs(x.pts - y.pts).max() < 1e-3 and np.abs(x.center - y.center).max() < 1e-3
            assert np.abs(y.pts - g[f"pts{seed}"][k]).max() < 1e-4
    assert len(g["index2"]) == 7          # one detection of scene 2 holds no valid light pair


def test_extract_armors_roi_edge_cases():
    """Boxes outside / across the frame, empty after truncation, and NaN (src/irm_detector.cpp:299-304)."""
    from oracle import armor_ref as A
    img, boxes, scores, classes = A.synth_armor_scene(2, 5)
    odd = np.array([[-50, -40, 30, 20], [1270, 1000, 1400, 1100], [100, 100, 100.5, 180], [300, 300, 200, 400],
                    [np.nan, 0, 50, 50], [-1e9, -1e9, 1e9, 1e9]], np.float32)
    b = np.concatenate([boxes, odd])
    s = np.concatenate([scores, np.full(len(odd), 0.5, np.float32)])
    c = np.concatenate([classes, np.zeros(len(odd), np.int32)])
    a1 = A.extract_armors(img, b, s, c)
    a2 = A.extract_armors_cv2(img, b, s, c)
    assert [a.bbox_index for a in a1] == [a.bbox_index for a in a2]
    assert A.roi_of(odd[2], 1280, 1024) is None and A.roi_of(odd[3], 1280, 1024) is None
    assert A.roi_of(odd[4], 1280, 1024) is None
    assert A.roi_of(odd[5], 1280, 1024)[:4] == (0, 0, 1280, 1024)


# ----------------------------------------------------------------------------------- boundary
def test_cabi_exports_every_declared_symbol():
    from irmv_detection_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "irmv_cabi.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(irmv_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    lib = _lib.lib()
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.irmv_version() >= 100
    import ctypes as C
    cfg = _lib.EngineConfig()
    assert lib.irmv_engine_config_default(C.byref(cfg)) == 0
    assert (cfg.src_width, cfg.src_height, cfg.rotate180, cfg.max_det) == (1280, 1024, 1, 100)
    assert abs(cfg.score_thr - 0.25) < 1e-7 and abs(cfg.iou_thr - 0.45) < 1e-7
    assert C.sizeof(_lib.Bbox) == 24 and C.sizeof(_lib.Armor) == 56 and C.sizeof(_lib.ArmorParams) == 48
    prm = _lib.ArmorParams()
    assert lib.irmv_armor_params_default(C.byref(prm)) == 0 and prm.binary_threshold == 150


def test_missing_weights_raises(tmp_path):
    import irmv_detection_b200 as irmv
    with pytest.raises(FileNotFoundError):
        irmv.YoloEngine(str(tmp_path / "nope.onnx"), (1280, 1024))


def test_weights_path_follows_reference_convention():
    from irmv_detection_b200.engine import weights_path_for
    assert weights_path_for("/a/b/models/yolov7.onnx") == "/a/b/models/yolov7.irmw"


# ----------------------------------------------------------------------------------- sharding
def test_shard_range_partitions():
    from irmv_detection_b200.sharding import shard_range
    for total in (0, 1, 7, 256, 1000):
        for world in (1, 2, 3, 8):
            spans = [shard_range(total, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == total
            assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
            sizes = [e - b for b, e in spans]
            assert max(sizes) - min(sizes) <= 1


def _gloo_worker(rank, world, port, q):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank),
                      MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    from irmv_detection_b200 import sharding
    import torch.distributed as dist
    sharding.init_process_group("gloo")
    b, e = sharding.shard_range(10, rank, world)
    sharding.barrier()
    mx, sm = sharding.reduce_max_sum(float(rank + 1), float(e - b))
    q.put((rank, mx, sm))
    dist.destroy_process_group()


def test_gloo_world2_reduction():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29600 + os.getpid() % 200
    ps = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    [p.start() for p in ps]
    res = sorted(q.get(timeout=120) for _ in ps)
    [p.join(60) for p in ps]
    assert res == [(0, 2.0, 10.0), (1, 2.0, 10.0)]


def test_triple_buffer_monotonic(tmp_path):
    """include/irmv_detection/triple_buffer.hpp under a full-speed producer: the consumer never
    steps back to an older frame (the reference's two-atomic protocol can; see the header)."""
    import subprocess
    exe = tmp_path / "tb_test"
    subprocess.run(["g++", "-std=c++20", "-O2", "-pthread", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "cpp", "triple_buffer_test.cpp"), "-o", str(exe)], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "FAIL" not in r.stdout, r.stdout[-500:]


def test_virtual_camera_handoff(tmp_path):
    """include/irmv_detection/camera.hpp: VirtualCamera streams into three caller-owned buffers through the
    TripleBuffer; a slow consumer drops frames but never sees a torn, repeated or reordered one."""
    import subprocess
    exe = tmp_path / "vc_test"
    subprocess.run(["g++", "-std=c++20", "-O2", "-pthread", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "cpp", "virtual_camera_test.cpp"), "-o", str(exe)], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "VIRTUAL_CAMERA_OK" in r.stdout, r.stdout[-500:]


def test_letterbox_oracle_vs_cv2(base_image):
    """LETTERBOX oracle vs the ultralytics recipe done with cv2 (resize INTER_LINEAR + copyMakeBorder
    114): same geometry, pixels within 1 grey level (cv2 resizes u8 in fixed point)."""
    import cv2
    from oracle import preprocess_ref as PR
    for img in (base_image, np.ascontiguousarray(base_image[:700, :900])):
        H, W = img.shape[:2]
        x, (px, py, nw, nh) = PR.preprocess_letterbox(img, rotate=False)
        r = min(640 / H, 640 / W)
        new_unpad = int(round(W * r)), int(round(H * r))
        dw, dh = (640 - new_unpad[0]) / 2, (640 - new_unpad[1]) / 2
        ref = cv2.resize(img, new_unpad, interpolation=cv2.INTER_LINEAR)
        top, bottom = int(round(dh - 0.1)), int(round(dh + 0.1))
        left, right = int(round(dw - 0.1)), int(round(dw + 0.1))
        ref = cv2.copyMakeBorder(ref, top, bottom, left, right, cv2.BORDER_CONSTANT, value=(114, 114, 114))
        assert ref.shape[:2] == (640, 640) and (px, py, nw, nh) == (left, top, new_unpad[0], new_unpad[1])
        got = np.rint(x.transpose(1, 2, 0) * 255).astype(np.int32)
        assert np.abs(got - ref.astype(np.int32)).max() <= 1


def test_stem_integer_lerp_equals_float_oracle():
    """csrc/stem_bayer.cu replaces the reference's FP32 vertical lerp + 8-bit rounding
    (floor(a*(1-f) + b*f + 0.5), oracle/preprocess_ref.resize_bilinear_u8) by the integer form
    (2(Q-k)*a + 2k*b + Q) // 2Q with f = k/Q, and the FP32 tap computation by i0 = (dy*P)//Q.
    Exhaustive over all 640 rows and all byte pairs for the camera height (1024 -> P/Q = 8/5) and
    sampled for the other heights the fast path accepts."""
    from math import gcd
    from oracle import preprocess_ref as PR
    one = np.float32(1)
    a = np.arange(256, dtype=np.float32)[:, None, None]
    b = np.arange(256, dtype=np.float32)[None, :, None]
    ai, bi = np.arange(256)[:, None, None], np.arange(256)[None, :, None]
    for H in (1024, 960, 720, 1080, 800, 640):
        g = gcd(H, 640)
        P, Q = H // g, 640 // g
        assert Q <= 16
        i0, i1, f = PR._axis_taps(640, H, False)
        dy = np.arange(640)
        assert np.array_equal((dy * P) // Q, i0) and np.array_equal(np.minimum((dy * P) // Q + 1, H - 1), i1)
        k = (dy * P) % Q
        step = 1 if H == 1024 else 7
        for d0 in range(0, 640, 64):
            sl = slice(d0, d0 + 64, step)
            ff = f[sl][None, None, :]
            v = a * (one - ff) + b * ff
            qf = np.clip(np.floor(v + np.float32(0.5)), 0, 255).astype(np.int64)
            kk = k[sl][None, None, :]
            qi = ((2 * (Q - kk)) * ai + 2 * kk * bi + Q) // (2 * Q)
            assert np.array_equal(qf, qi), (H, d0)


def _stem_fast_path_emulation(raw, chan, rot):
    """The sampling arithmetic of stem_bayer2x_kernel (csrc/stem_bayer.cu) in numpy, packed 2 x 16-bit
    lanes included: network-input pixels as 8-bit values [640, 640, 3]."""
    from math import gcd
    H, W = raw.shape
    g = gcd(H, 640)
    P, Q = H // g, 640 // g
    red_y = 1 if chan in (3, 5) else 0
    red_x = 1 if chan in (3, 4) else 0
    red_col = ((1 if rot else 0) == red_x)
    M, K1, K2, QQ = 0x00ff00ff, 0x00010001, 0x00020002, Q * 0x10001
    out = np.zeros((640, 640, 3), np.int64)
    j = np.arange(320)

    def refl(i):
        i = -i if i < 0 else i
        return 2 * H - 2 - i if i >= H else i

    for iy in range(640):
        tt = iy * P
        i0, k = tt // Q, tt % Q
        i1 = min(i0 + 1, H - 1)
        wA, wB = 2 * (Q - k), 2 * k
        if i1 == i0:
            wA, wB = wA + wB, 0
        sy0, sy1 = (H - 1 - i0, H - 1 - i1) if rot else (i0, i1)
        lo = min(sy0, sy1)
        w_lo, w_hi = (wA, wB) if sy0 <= sy1 else (wB, wA)
        lo_site = (((lo & 1) == red_y) == red_col)
        rows = []
        for d in range(-1, 3):
            r = raw[min(refl(lo + d), H - 1)].astype(np.int64)
            buf = np.zeros(16 + W + 16, np.int64)
            buf[16:16 + W] = r; buf[15] = r[1]; buf[16 + W] = r[W - 2]
            b4 = buf.reshape(-1, 4)
            w32 = b4[:, 0] | (b4[:, 1] << 8) | (b4[:, 2] << 16) | (b4[:, 3] << 24)
            C = w32[4 + j]
            if rot:
                N = w32[5 + j]
                rows.append((C & M, (C >> 8) & M, (((C >> 16) | (N << 16)) & 0xffffffff) & M))
            else:
                Pw = w32[3 + j]
                rows.append(((((Pw >> 24) | (C << 8)) & 0xffffffff) & M, C & M, (C >> 8) & M))
        r0, r1, r2, r3 = rows                      # (w, c, e) per row
        if lo_site:
            cross = ((r0[1] + r2[1] + r1[0] + r1[2] + K2) >> 2) & M
            diag = ((r0[0] + r0[2] + r2[0] + r2[2] + K2) >> 2) & M
            cS, cG = r1[1], r2[1]
            horiz = ((r2[0] + r2[2] + K1) >> 1) & M
            vert = ((r1[1] + r3[1] + K1) >> 1) & M
            wS, wG = w_lo, w_hi
        else:
            horiz = ((r1[0] + r1[2] + K1) >> 1) & M
            vert = ((r0[1] + r2[1] + K1) >> 1) & M
            cG, cS = r1[1], r2[1]
            cross = ((r1[1] + r3[1] + r2[0] + r2[2] + K2) >> 2) & M
            diag = ((r1[0] + r1[2] + r3[0] + r3[2] + K2) >> 2) & M
            wG, wS = w_lo, w_hi
        RS, BS = (cS, diag) if red_col else (diag, cS)
        RG, BG = (vert, horiz) if red_col else (horiz, vert)
        for ch, x in enumerate((RS * wS + RG * wG + QQ, cross * wS + cG * wG + QQ, BS * wS + BG * wG + QQ)):
            lo16, hi16 = (x & 0xffff) // (2 * Q), (x >> 16) // (2 * Q)
            if rot:
                out[iy, 638 - 2 * j, ch] = hi16; out[iy, 639 - 2 * j, ch] = lo16
            else:
                out[iy, 2 * j, ch] = lo16; out[iy, 2 * j + 1, ch] = hi16
    return out


@pytest.mark.parametrize("rot", [True, False])
@pytest.mark.parametrize("chan", [2, 3, 4, 5])
@pytest.mark.parametrize("H", [640, 720, 800, 960, 1024, 1080, 1200, 1280])
def test_stem_fast_path_arithmetic_matches_oracle(H, chan, rot):
    """The camera-case stem's packed-lane demosaic + integer lerp, restated in numpy, equals the oracle's
    demosaic -> rot180 -> NPP-convention resize -> 8-bit rounding for every pixel, at every height of the GPU
    geometry matrix (tests/test_gpu_stem_geometry.py), all four Bayer patterns, with and without rot180."""
    from oracle import preprocess_ref as PR
    raw = np.random.default_rng(H + chan).integers(0, 256, (H, 1280), dtype=np.uint8)
    x, _ = PR.preprocess(raw, chan, rot, True)
    ref = np.rint(x.transpose(1, 2, 0) * 255).astype(np.int64)
    assert np.array_equal(_stem_fast_path_emulation(raw, chan, rot), ref)


def _probe_m0(xp, taps_of=lambda t: t):
    """What a faithful engine stores in m0 for each probe file of oracle/stem_probe.py, from the padded input xp
    [N, 3, 641, 641] (FP16 values): FP16(SiLU(read)).  taps_of(t) is the tap actually read for tap t."""
    from oracle import stem_probe as SP
    views = SP.tap_views(xp.astype(np.float64))
    out = []
    for taps in SP.TAP_FILES:
        m0 = np.zeros(views.shape[:1] + (320, 320, 16), np.float16)
        for i, t in enumerate(taps):
            m0[..., 3 * i:3 * i + 3] = SP.silu(views[:, taps_of(t)]).transpose(0, 2, 3, 1).astype(np.float16)
        out.append(m0)
    return out


def test_stem_probe_helper_catches_single_errors():
    """The probe comparison of tests/test_gpu_stem_geometry.py (oracle/stem_probe.py) passes a faithful engine and
    fails each single error a fused stem could make: one pixel off by one 8-bit step, tap (0, 0) read from (0, 1),
    a non-zero top padding row, and on the float path one pixel off by two FP16 ulps."""
    from oracle import stem_probe as SP
    rng = np.random.default_rng(7)
    codes = rng.integers(0, 256, (2, 3, 640, 640))
    x16 = (codes / 255.0).astype(np.float16)
    got = lambda xp, **kw: SP.engine_views(_probe_m0(xp, **kw))
    assert SP.compare_codes(got(SP.pad_input(x16)), codes) is None
    for f, c, y, x in ((0, 0, 0, 0), (1, 2, 639, 639), (1, 1, 331, 12), (0, 1, 7, 400)):
        bad = codes.copy()
        bad[f, c, y, x] = bad[f, c, y, x] + 1 if bad[f, c, y, x] < 255 else 254
        msg = SP.compare_codes(got(SP.pad_input((bad / 255.0).astype(np.float16))), codes)
        assert msg is not None and f"({f}, {c}, {y}, {x})" in msg, msg
    msg = SP.compare_codes(got(SP.pad_input(x16), taps_of=lambda t: 1 if t == 0 else t), codes)
    assert msg is not None and "tap (0, 0)" in msg, msg
    top = SP.pad_input(x16)
    top[:, :, 0, 1:] = np.float16(1 / 255)                     # top padding row, left padding column kept zero
    msg = SP.compare_codes(got(top), codes)
    assert msg is not None and ", -1, " in msg and "tap (0, " in msg, msg
    # float path: values off the 8-bit grid, one pixel two FP16 ulps off at a value in [0.5, 1)
    xf = rng.uniform(0, 1, (1, 3, 640, 640)).astype(np.float16)
    xf[0, 1, 100, 200] = np.float16(0.75)
    assert SP.float_deviation(got(SP.pad_input(xf)), xf)[0] <= SP.FLOAT_TOL
    bad = xf.copy()
    bad[0, 1, 100, 200] = np.float16(0.75 + 2 * 2.0 ** -11)
    d, at = SP.float_deviation(got(SP.pad_input(bad)), xf)
    assert d > SP.FLOAT_TOL and (at["frame"], at["channel"], at["y"], at["x"]) == (0, 1, 100, 200), (d, at)


def test_shufflenet_variant_weights_and_oracle(base_image, tmp_path):
    """BASELINE.json configs[2]: the keypoint detector on the ShuffleNetV2-style backbone.  The weight file
    (IRMW v2: architecture id + groups per conv) round-trips, the inventory is what weights.py documents
    (83 convs, 13 of them depthwise), the units are the published ShuffleNetV2 ones (channel shuffle checked
    against its definition), and OpenCV-DNN running the ONNX export agrees with the torch oracle."""
    import cv2
    import torch
    from irmv_detection_b200 import weights as W
    from oracle import export_onnx, preprocess_ref as PR, yolov8n_ref as Y
    specs = W.shuffle_conv_specs()
    assert len(specs) == 83 and sum(1 for c in specs if c.groups > 1) == 13
    assert all(c.groups in (1, c.cin) and (c.groups == 1 or (c.k == 3 and c.act == 0 and c.cin == c.cout)) for c in specs)
    assert [c.name for c in specs[36:40]] == ["m9.cv1", "m9.cv2", "m12.cv1", "m12.m0.cv1"]
    p = str(tmp_path / "shuffle.irmw")
    W.write_random(p, 0, arch="shufflenetv2-pose")
    assert W.file_arch(p) == W.ARCH_SHUFFLE_KPT
    nc, t = W.load(p)
    assert nc == 14 and len(t) == 83
    assert all(np.array_equal(w.astype(np.float16).astype(np.float32), w) for _, w, _ in t)   # FP16-exact
    x = torch.arange(2 * 8 * 1 * 1, dtype=torch.float32).view(2, 8, 1, 1)
    assert Y.channel_shuffle(x)[0, :, 0, 0].tolist() == [0, 4, 1, 5, 2, 6, 3, 7]              # y[2i] = a[i], y[2i+1] = b[i]
    m = Y.build(p)
    assert isinstance(m, Y.ShuffleV2Kpt) and len(m.convs_in_order()) == 83
    xin, _ = PR.preprocess(base_image)
    taps = {}
    with torch.no_grad():
        outs = m.features(torch.from_numpy(xin)[None], taps)
        boxes, scores = Y.decode_heads(outs)
    assert [tuple(taps[k].shape[1:]) for k in ("d1", "d2", "d3", "d4")] == [(32, 160, 160), (64, 80, 80), (128, 40, 40), (256, 20, 20)]
    assert all(0.2 < float(taps[k].std()) < 3.0 for k in taps)            # calibrated init keeps activations O(1)
    assert outs[0][2].shape == (1, 8, 80, 80)
    path = str(tmp_path / "shuffle.onnx")
    try:
        export_onnx.export(m, path)
        net = cv2.dnn.readNetFromONNX(path)
    except Exception as e:          # exporter internals differ between torch builds
        pytest.skip(f"ONNX export / import unavailable: {e}")
    net.setInput(xin[None])
    out = net.forward()
    ref = torch.cat((boxes, scores), 2).numpy()
    assert out.shape == ref.shape and np.abs(out - ref).max() < 5e-3


def test_media_type_to_channel_order():
    """tSdkFrameHead.uiMediaType -> IRMV_CH_* (reference mvsdk/include/CameraDefine.h:693-705,733-736,771-772).
    The codes are rebuilt here from the vendor header's formula (MONO|COLOR base | bit occupancy | id)."""
    from irmv_detection_b200 import _lib as L
    MONO, COLOR, O8, O24, O16 = 0x01000000, 0x02000000, 0x00080000, 0x00180000, 0x00100000
    f = L.lib().irmv_chan_order_from_media_type
    assert f(MONO | O8 | 0x0009) == L.CH_BAYER_RGGB      # BAYRG8: R G / G B
    assert f(MONO | O8 | 0x0008) == L.CH_BAYER_GRBG      # BAYGR8
    assert f(MONO | O8 | 0x000A) == L.CH_BAYER_GBRG      # BAYGB8
    assert f(MONO | O8 | 0x000B) == L.CH_BAYER_BGGR      # BAYBG8
    assert f(COLOR | O24 | 0x0014) == L.CH_PASSTHROUGH   # RGB8: what CameraImageProcess emits (src/mv_camera.cpp:64)
    assert f(COLOR | O24 | 0x0015) == L.CH_SWAP_RB       # BGR8
    assert f(MONO | O8 | 0x0001) == -1                   # MONO8
    assert f(MONO | O16 | 0x000D) == -1                  # BAYRG10: not ingested


def test_bench_replay_split_and_config_are_shared_by_both_arms():
    """bench.py: the engine runs the 256-frame step as one replay on one lane by default; explicit flags win; the
    reference arm prints the same `config` object as the repo's arm (the driver compares them)."""
    import argparse
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench
    a = argparse.Namespace(batch=256, sub_batch=0, lanes=0)
    assert bench.replay_split(a) == (256, 1)
    assert bench.replay_split(argparse.Namespace(batch=512, sub_batch=0, lanes=0)) == (256, 2)
    assert bench.replay_split(argparse.Namespace(batch=64, sub_batch=0, lanes=0)) == (64, 1)
    assert bench.replay_split(argparse.Namespace(batch=256, sub_batch=128, lanes=2)) == (128, 2)
    cfg = bench.workload_config(256, *bench.replay_split(a))
    assert cfg["frames_per_gpu_per_step"] == 256 and cfg["sub_batch"] == 256 and cfg["lanes"] == 1
    assert "workload" in cfg and "model" not in cfg
