"""The armor stage (light bars -> armors, csrc/armors.cu) against the OpenCV chain at every source geometry and on each
of its kernel paths.

Every comparison is oracle.armor_ref.check_armors: the stage's armors against the reference's function written with
the cv2 calls, on armor_ref.rotated_image(frame, chan, rot180); identical valid flags, size class, class and score,
corners and centre within 1e-2 px, a mismatch excused only where the restatement armor_ref.extract_armors flags the
box's minimum-area rectangle as ambiguous.

  a. geometries: the stand-alone stage (irmv_extract_armors) from 320 x 240 to 1280 x 3400, every channel order, rot180
     on and off, ragged batches; light-bar pairs at each frame edge and a corner whose boxes run past the frame (Bayer:
     reflect-101 neighbours feed the threshold), whole-frame, off-frame, degenerate and inverted boxes; speckle / blob /
     ring scenes with permissive filters at three geometries;
  b. kernel paths: one pair of bars in boxes on both sides of each dispatch threshold of extract_armors_kernel (shared
     memory or global scratch bitmap; <= 64 or more start candidates), padded widths around the 32-bit word, borders
     on a word boundary and on the ROI's first and last row and column, a bar inside a ring;
  c. the stage fused into the engine replay at new geometries, with letterbox, with a raw table, and after a replay on
     black frames;
  d. the source sizes the stage refuses, refused when it is set up.
Run with -s for one line per case: the path each box takes and the excused boxes.
"""
import ctypes as C

import numpy as np
import pytest

from oracle import armor_ref as A, preprocess_ref as PR

pytestmark = pytest.mark.gpu

# filters that let most elongated contours through (contour order and the >= 5-vertex rule then decide the answer)
PERMISSIVE = dict(light_min_ratio=0.02, light_max_ratio=0.9, light_max_angle=80.0, min_small_center_distance=0.1,
                  max_large_center_distance=50.0)
# extract_armors_kernel's dispatch (csrc/armors.cu): bitmap words in shared memory, rows of the per-warp arrays in
# shared memory, start candidates the warps share out from a list
SMEM_WORDS, SMEM_ROWS, CAND_CAP = 2048, 256, 64
MAX_SIDE = 32766


def _cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _prm(**kw):
    return A.ArmorParams(**kw)


def roi_words(rw, rh):
    return (rh + 2) * ((rw + 2 + 31) // 32)


def is_large(rw, rh):
    """The ROI's bitmaps and per-warp arrays live in the CTA's global scratch slot instead of shared memory."""
    return roi_words(rw, rh) > SMEM_WORDS or rh > SMEM_ROWS


def start_candidates(image, box, thr):
    """Start candidates of the box's ROI by the kernel's rule: foreground with exterior background to the W and no
    foreground to the NW, N or NE (padded ROI, exterior = 4-connected to the padding)."""
    rows, cols = image.shape[:2]
    rx, ry, rw, rh = A.roi_of(box, cols, rows)[:4]
    fg = np.zeros((rh + 2, rw + 2), bool)
    fg[1:-1, 1:-1] = A.gray_bgr2gray(image[ry:ry + rh, rx:rx + rw]) > thr
    ext = A.exterior_background(fg)
    return int((fg[1:-1, 1:-1] & ext[1:-1, :-2] & ~fg[:-2, :-2] & ~fg[:-2, 1:-1] & ~fg[:-2, 2:]).sum())


def _camera_frame(view, chan, rot):
    """What the camera wrote, given the rotated view the reference thresholds (Bayer: a mosaic of the view's colours)."""
    img = PR.rot180(view) if rot else np.ascontiguousarray(view)
    return PR.mosaic_from_rgb(img, chan) if chan >= 2 else img


def _bar(img, c, length, width, tilt, colour):
    import cv2
    box = cv2.boxPoints(((float(c[0]), float(c[1])), (float(width), float(length)), float(tilt)))
    cv2.fillConvexPoly(img, np.round(box).astype(np.int32), tuple(int(v) for v in colour))


def _pair(img, cx, cy, length, width, sep, tilt, colour):
    for s in (-1, 1):
        _bar(img, (cx + s * sep / 2, cy), length, width, tilt + 2 * s, colour)


# the edge bars are green so that their gray value (~160) sits close to the threshold: a Bayer fetch that took the
# wrong colour site at the frame edge (clamped instead of mirrored neighbours) moves it across
EDGE_COLOUR = (60, 230, 60)


def _edge_pairs(img, rng):
    """Light-bar pairs cut by the left, right, top and bottom edges and by the bottom-right corner; their boxes run
    past the frame."""
    H, W = img.shape[:2]
    L, wd, sep = 32.0, 7.0, 44.0
    boxes = []
    places = [(sep / 2 - 2, rng.uniform(L, H - L)), (W - sep / 2 + 2, rng.uniform(L, H - L)),
              (rng.uniform(sep, W - sep), L / 2 - 3), (rng.uniform(sep, W - sep), H - L / 2 + 3),
              (W - sep / 2 + 2, H - L / 2 + 3)]
    for cx, cy in places:
        _pair(img, cx, cy, L, wd, sep, rng.uniform(-10, 10), EDGE_COLOUR)
        m = rng.uniform(8, 20)
        boxes.append([cx - sep / 2 - wd - m, cy - L * 0.8 - m, cx + sep / 2 + wd + m, cy + L * 0.8 + m])
    return np.array(boxes, np.float32)


def _special_boxes(W, H):
    return np.array([[-1e9, -1e9, 1e9, 1e9],                    # whole frame (global-scratch bitmaps, every row)
                     [W + 10, H + 10, W + 90, H + 70],          # off frame
                     [100.25, 50, 100.75, 90],                  # zero width after truncation
                     [60, 60, 20, 120]], np.float32)            # inverted


class Case:
    def __init__(self, W, H, chan, rot, blobs=False):
        self.W, self.H, self.chan, self.rot, self.blobs = W, H, chan, rot, blobs
        self.id = f"{W}x{H}-c{chan}{'-rot' if rot else ''}{'-blobs' if blobs else ''}"


_GEO = [(1280, 1024), (1280, 1200), (1280, 1280), (1920, 1080), (1920, 1200), (1440, 1080), (2048, 1536), (1280, 3400),
        (640, 480), (320, 240), (1001, 777)]
GEOMETRY_CASES = [Case(W, H, i % 6, i % 2 == 0) for i, (W, H) in enumerate(_GEO)]
BLOB_CASES = [Case(1920, 1200, 5, False, True), Case(1280, 3400, 0, True, True), Case(1001, 777, 3, True, True)]


def _scene_frames(case, n):
    """n rotated views: seeded light-bar scene + edge pairs; per frame its boxes, scores and classes."""
    from irmv_detection_b200 import synth
    W, H = case.W, case.H
    views, dets = [], []
    for f in range(n):
        seed = 1000 * f + W + H
        rng = np.random.default_rng(seed)
        img, boxes, scores, classes = synth.armor_scene(2 if W < 400 else 5, seed, W, H)
        eb = _edge_pairs(img, rng)
        boxes = np.concatenate([boxes, eb, _special_boxes(W, H)]).astype(np.float32)
        extra = len(boxes) - len(scores)
        scores = np.concatenate([scores, rng.uniform(0.3, 0.95, extra)]).astype(np.float32)
        classes = np.concatenate([classes, rng.integers(0, 15, extra)]).astype(np.int32)
        views.append(img)
        dets.append((boxes, scores, classes))
    return views, dets


def _blob_frames(case, n):
    W, H = case.W, case.H
    views, dets = [], []
    for f in range(n):
        seed = 2000 * f + W + H
        rng = np.random.default_rng(seed)
        views.append(A.blob_scene(seed, H, W, int(260 * W * H / (1280 * 1024))))
        m = 64
        cx, cy = rng.uniform(-20, W + 20, m), rng.uniform(-20, H + 20, m)
        bw, bh = rng.uniform(4, 260, m), rng.uniform(4, 220, m)
        boxes = np.stack([cx - bw / 2, cy - bh / 2, cx + bw / 2, cy + bh / 2], 1).astype(np.float32)
        boxes[:2] = [[40, 30, 460, 350], [W - 380, H - 420, W + 20, H + 30]]   # global-scratch bitmaps (> 2048 words)
        boxes[-3:] = _special_boxes(W, H)[1:]                   # no whole-frame box over speckle
        dets.append((boxes, rng.uniform(0.25, 1, m).astype(np.float32), rng.integers(0, 15, m).astype(np.int32)))
    return views, dets


def _run_stage(frames, dets, counts, max_det, chan, rot, **params):
    """The stand-alone stage on a ragged batch.  The slots past a frame's count hold live boxes (copies of the
    frame's first boxes), so a stage that read past the count would find armors there."""
    import irmv_detection_b200 as irmv
    b = np.zeros((len(frames), max_det), irmv.BBOX_DTYPE)
    for f, (boxes, scores, classes) in enumerate(dets):
        k = min(len(boxes), max_det)
        b["xyxy"][f, :k], b["score"][f, :k], b["class_id"][f, :k] = boxes[:k], scores[:k], classes[:k]
        for j in range(k, max_det):
            b[f, j] = b[f, j % max(k, 1)]
    return irmv.extract_armors(np.stack(frames), b, np.asarray(counts, np.int32), chan_order=chan, rotate180=rot,
                               **params)


def _path_summary(views, dets, counts):
    small = large = 0
    for img, (boxes, _, _), k in zip(views, dets, counts):
        for b in boxes[:k]:
            roi = A.roi_of(b, img.shape[1], img.shape[0])
            if roi is not None:
                large += is_large(roi[2], roi[3])
                small += not is_large(roi[2], roi[3])
    return f"small {small} large {large}"


# ------------------------------------------------------------------------------------------------ a. geometries
@pytest.mark.parametrize("case", GEOMETRY_CASES, ids=lambda c: c.id)
def test_stage_at_geometry(case):
    _cuda()
    n = 2 if case.H > 2000 else 3
    views, dets = _scene_frames(case, n)
    frames = [_camera_frame(v, case.chan, case.rot) for v in views]
    images = [A.rotated_image(fr, case.chan, case.rot) for fr in frames]
    counts = [len(d[0]) for d in dets]
    counts[-1] -= 3                                              # ragged: the last frame's last boxes are not counted
    prm = dict(binary_threshold=150, **PERMISSIVE)
    got = _run_stage(frames, dets, counts, max(len(d[0]) for d in dets) + 4, case.chan, case.rot, **prm)
    n_ref = 0
    excused = []
    for f in range(n):
        boxes, scores, classes = dets[f]
        k = counts[f]
        r, ex = A.check_armors(got[f], images[f], boxes[:k], scores[:k], classes[:k], _prm(**prm))
        n_ref += r
        excused += [(f, i) for i in ex]
    print(f"{case.id}: {_path_summary(images, dets, counts)}, armors {n_ref}, excused {excused}")
    assert n_ref >= n, "too few armors for the comparison to mean much"
    assert len(excused) <= 2, excused


@pytest.mark.parametrize("case", BLOB_CASES, ids=lambda c: c.id)
def test_stage_speckle_at_geometry(case):
    """Ragged counts: the first frame has no detection, the second max_det; every slot from the count on is invalid."""
    _cuda()
    views, dets = _blob_frames(case, 3)
    frames = [_camera_frame(v, case.chan, case.rot) for v in views]
    images = [A.rotated_image(fr, case.chan, case.rot) for fr in frames]
    max_det = len(dets[0][0])
    counts = [0, max_det, 40]
    thr = 140 if case.chan < 2 else 110
    prm = dict(binary_threshold=thr, **PERMISSIVE)
    got = _run_stage(frames, dets, counts, max_det, case.chan, case.rot, **prm)
    n_ref, excused = 0, []
    for f in range(3):
        boxes, scores, classes = dets[f]
        k = counts[f]
        assert not got[f][k:]["valid"].any(), f"frame {f}: armor past the count {k}"
        r, ex = A.check_armors(got[f], images[f], boxes[:k], scores[:k], classes[:k], _prm(**prm))
        n_ref += r
        excused += [(f, i) for i in ex]
    print(f"{case.id}: {_path_summary(images, dets, counts)}, armors {n_ref}, excused {excused}")
    assert n_ref >= 10, n_ref
    assert len(excused) <= 6, excused


# ---------------------------------------------------------------------------------------------- b. kernel paths
# One well-conditioned pair of bars (16 x 4 px, 8 degrees, centres 16 px apart: 23 px wide in all) at the centre of a
# 640 x 600 frame; the boxes around it sit on both sides of each threshold.
PAIR_W, PAIR_H = 640, 600
PAIR_C = (320.5, 300.5)
PAIR = dict(length=16.0, width=4.0, sep=16.0, tilt=8.0)
PATH_PRM = dict(binary_threshold=150)                          # the node's default filters


def _pair_view():
    img = np.zeros((PAIR_H, PAIR_W, 3), np.uint8)
    p = PAIR
    _pair(img, PAIR_C[0], PAIR_C[1], p["length"], p["width"], p["sep"], p["tilt"], (255, 255, 255))
    return img


def _centred(rw, rh, dx=0.0):
    """Box of rw x rh ROI pixels around the pair (centre shifted by dx)."""
    x0, y0 = int(PAIR_C[0] + dx) - rw // 2, int(PAIR_C[1]) - rh // 2
    return [x0, y0, x0 + rw, y0 + rh]


def _dots(img, box, k):
    """k isolated bright pixels (not 8-adjacent to anything) in the box's top rows, left to right."""
    x0, y0, x1, _ = (int(v) for v in box)
    placed = 0
    for y in range(y0 + 2, y0 + 40, 3):
        for x in range(x0 + 2, x1 - 2, 3):
            if placed == k:
                return
            if not img[y - 1:y + 2, x - 1:x + 2].any():
                img[y, x] = 255
                placed += 1
    assert placed == k, "box too small for the dots"


def _path_cases():
    """[(name, view, box, threshold group)]: each group is a pair of cases on both sides of one threshold."""
    cases = []
    base = _pair_view()
    for rh in (255, 256, 257):                                  # rows of the shared-memory per-warp arrays
        cases.append((f"rows{rh}", base, _centred(60, rh), "rows"))
    for rh in (254, 255):                                       # 8 words x 256 / 257 rows: 2048 / 2056 bitmap words
        cases.append((f"words{roi_words(254, rh)}", base, _centred(254, rh), "words"))
    for pw in (31, 32, 33, 63, 64, 65, 97):                     # padded width around the 32-bit word
        cases.append((f"pw{pw}", base, _centred(pw - 2, 40), None))
    # the left bar's border crosses padded column 32 (bit 31 of word 0 / bit 0 of word 1)
    cases.append(("word-boundary", base, [PAIR_C[0] - PAIR["sep"] / 2 - 31, 260, PAIR_C[0] + 60, 340], None))
    # the pair's own bounding box: bars on the ROI's first and last row and column
    ys, xs = np.nonzero(A.gray_bgr2gray(base) > PATH_PRM["binary_threshold"])
    cases.append(("tight", base, [xs.min(), ys.min(), xs.max() + 1, ys.max() + 1], None))
    # a third bar below the pair inside a ring: it is not external, so the pair stays the first two lights
    import cv2
    ring = base.copy()
    _bar(ring, (PAIR_C[0], PAIR_C[1] + 40), 16.0, 4.0, 5.0, (255, 255, 255))
    cv2.rectangle(ring, (int(PAIR_C[0]) - 12, int(PAIR_C[1]) + 24), (int(PAIR_C[0]) + 12, int(PAIR_C[1]) + 56),
                  (255, 255, 255), 2)
    cases.append(("ring", ring, [PAIR_C[0] - 40, PAIR_C[1] - 30, PAIR_C[0] + 40, PAIR_C[1] + 70], None))
    # start candidates 63 / 64 / 65 (isolated dots) in a shared-memory ROI and a global-scratch one
    for tag, rw, rh in (("smem", 200, 120), ("global", 200, 300)):
        box = _centred(rw, rh)
        own = start_candidates(base, box, PATH_PRM["binary_threshold"])
        for target in (63, 64, 65):
            v = base.copy()
            _dots(v, box, target - own)
            cases.append((f"cand{target}-{tag}", v, box, f"cand-{tag}"))
    return cases


def _profile_walks(frame, box, chan, rot, prm):
    """Run one box with the stage's cycle profile on: True when the list schedule (<= 64 candidates) walked borders."""
    import os
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import _lib
    old = os.environ.get("IRMV_ARMOR_PROF")
    os.environ["IRMV_ARMOR_PROF"] = "1"
    try:
        irmv.extract_armors(frame[None], A.boxes_struct(np.array([box], np.float32), [0.5], [1], 1), [1],
                            chan_order=chan, rotate180=rot, **prm)
    finally:
        if old is None:
            del os.environ["IRMV_ARMOR_PROF"]
        else:
            os.environ["IRMV_ARMOR_PROF"] = old
    buf = (C.c_uint64 * 8)()
    _lib.lib().irmv_extract_armors_last_profile(C.byref(buf))
    assert buf[4] == 1, "the profile did not see the ROI"
    return buf[6] > 0                                           # recording walks: only the list schedule counts them


@pytest.mark.parametrize("chan,rot", [(0, True), (1, False)])
def test_stage_kernel_paths(chan, rot):
    _cuda()
    cases = _path_cases()
    thr = PATH_PRM["binary_threshold"]
    info = {}
    for name, view, box, group in cases:
        rx, ry, rw, rh = A.roi_of(np.array(box, np.float32), PAIR_W, PAIR_H)[:4]
        info[name] = dict(rw=rw, rh=rh, large=is_large(rw, rh), ncand=start_candidates(view, box, thr))
    # the table must straddle every threshold, or a path would silently drop out of the test
    assert [info[f"rows{r}"]["large"] for r in (255, 256, 257)] == [False, False, True]
    assert info["rows257"]["rh"] == 257 and roi_words(info["rows257"]["rw"], 257) <= SMEM_WORDS
    assert [roi_words(info[n]["rw"], info[n]["rh"]) for n in ("words2048", "words2056")] == [2048, 2056]
    assert [info[n]["large"] for n in ("words2048", "words2056")] == [False, True]
    assert all(info[n]["rh"] <= SMEM_ROWS for n in ("words2048", "words2056"))
    assert [info[f"pw{p}"]["rw"] + 2 for p in (31, 32, 33, 63, 64, 65, 97)] == [31, 32, 33, 63, 64, 65, 97]
    for tag, large in (("smem", False), ("global", True)):
        assert [info[f"cand{t}-{tag}"]["ncand"] for t in (63, 64, 65)] == [63, 64, 65]
        assert all(info[f"cand{t}-{tag}"]["large"] == large for t in (63, 64, 65))
    frames = [_camera_frame(v, chan, rot) for _, v, _, _ in cases]
    images = [A.rotated_image(fr, chan, rot) for fr in frames]
    dets = [(np.array([b], np.float32), np.array([0.5 + 0.01 * i], np.float32), np.array([i % 15], np.int32))
            for i, (_, _, b, _) in enumerate(cases)]
    got = _run_stage(frames, dets, [1] * len(cases), 2, chan, rot, **PATH_PRM)
    n_valid = 0
    for f, (name, _, box, _) in enumerate(cases):
        n_ref, excused = A.check_armors(got[f], images[f], *dets[f], _prm(**PATH_PRM))
        assert not excused, f"{name}: excused {excused}"
        n_valid += n_ref
        d = info[name]
        print(f"{name}: roi {d['rw']}x{d['rh']} words {roi_words(d['rw'], d['rh'])} "
              f"{'global' if d['large'] else 'smem'} cand {d['ncand']} {'list' if d['ncand'] <= CAND_CAP else 'lanes'} "
              f"armor {n_ref} excused []")
    # the pair is an armor in every box that holds it whole (all but the narrowest widths)
    assert n_valid >= len(cases) - 3, n_valid
    # the schedule the kernel took for the candidate counts, read from its cycle profile
    for f, (name, _, box, group) in enumerate(cases):
        if group and group.startswith("cand"):
            assert _profile_walks(frames[f], box, chan, rot, PATH_PRM) == (info[name]["ncand"] <= CAND_CAP), name


# ----------------------------------------------------------------------------------------- c. fused in the engine
ENGINE_CASES = [  # (W, H, chan, rot180, letterbox)
    (1920, 1200, 5, True, False),
    (1280, 1280, 0, False, False),
    (1440, 1080, 0, True, True),                                # letterbox: rows padded (box_py)
    (1080, 1440, 1, True, True),                                # letterbox: columns padded (box_px)
    (640, 480, 2, True, False),
]
ENGINE_PRM = dict(binary_threshold=150, **PERMISSIVE)
# valid armors over all ENGINE_CASES with the seed-0 weights (random init: the boxes land anywhere); a B200 run
# (1000 W limit) compared 864: 245, 226, 82, 93 and 218 in the order above
MIN_ENGINE_ARMORS = 400


def _engine(weights, W, H, chan, rot, letterbox, n=3, armors=True):
    import irmv_detection_b200 as irmv
    from oracle import pnp_ref as P
    eng = irmv.YoloEngine(weights, (W, H), chan_order=chan, rotate180=rot, letterbox=letterbox, max_batch=n)
    if armors:
        eng.enable_armors(**ENGINE_PRM)
    eng.enable_pnp(P.K_DEFAULT, P.D_DEFAULT, (640 / W, 480 / H))
    return eng


def _engine_frames(W, H, chan, rot, n=3):
    from irmv_detection_b200 import synth
    views = [synth.armor_scene(12, 50 + s, W, H)[0] for s in range(n)]
    return np.ascontiguousarray(np.stack([_camera_frame(v, chan, rot) for v in views]))


def test_fused_stage_at_geometries(weights_seed0):
    import irmv_detection_b200 as irmv
    _cuda()
    n_valid = 0
    for W, H, chan, rot, lb in ENGINE_CASES:
        name = f"{W}x{H}-c{chan}{'-rot' if rot else ''}{'-letterbox' if lb else ''}"
        frames = _engine_frames(W, H, chan, rot)
        eng = _engine(weights_seed0, W, H, chan, rot, lb)
        counts, dets = eng.detect_batch_arrays(frames)
        counts, dets = counts.copy(), dets.copy()
        arm = eng.fetch_armors(3)
        _, _, ok = eng.fetch_poses(3)
        alone = irmv.extract_armors(frames, dets, counts, chan_order=chan, rotate180=rot, **ENGINE_PRM)
        valid, excused = 0, []
        for f in range(3):
            k = int(counts[f])
            assert np.array_equal(arm[f]["valid"][:k], alone[f]["valid"][:k]), f"{name} frame {f}: valid flags"
            v = np.nonzero(arm[f]["valid"][:k])[0]
            assert arm[f][v].tobytes() == alone[f][v].tobytes(), f"{name} frame {f}: armors"
            assert not arm[f]["valid"][k:].any()
            assert not ok[f, :k][arm[f]["valid"][:k] == 0].any(), f"{name} frame {f}: pose without an armor"
            image = A.rotated_image(frames[f], chan, rot)
            _, ex = A.check_armors(arm[f], image, dets[f]["xyxy"][:k], dets[f]["score"][:k], dets[f]["class_id"][:k],
                                   _prm(**ENGINE_PRM))
            excused += [(f, i) for i in ex]
            valid += len(v)
        # a replay on black frames: no light bar anywhere, so no slot may keep an armor of the replay before
        eng.detect_batch_arrays(np.zeros_like(frames))
        assert not eng.fetch_armors(3)["valid"].any(), f"{name}: armor after a replay on black frames"
        eng.close()
        print(f"{name}: detections {int(counts.sum())}, armors {valid}, excused {excused}")
        assert len(excused) <= 2, excused
        n_valid += valid
    assert n_valid >= MIN_ENGINE_ARMORS, n_valid


def test_fused_stage_raw_table_at_1920x1200(weights_seed0):
    """The engine with table L on frames F equals the engine without a table on apply_raw_lut(F, L): armors, poses."""
    from irmv_detection_b200 import raw_lut as R
    _cuda()
    W, H, chan, rot = 1920, 1200, 4, False
    lut = R.make_raw_lut(8, (1.9, 1.0, 1.6), 1 / 2.2)
    frames = _engine_frames(W, H, chan, rot)
    pre = np.ascontiguousarray(R.apply_raw_lut(frames, lut, chan))
    eng, ref = _engine(weights_seed0, W, H, chan, rot, False), _engine(weights_seed0, W, H, chan, rot, False)
    eng.set_raw_lut(lut)
    got_c, got_d = (a.copy() for a in eng.detect_batch_arrays(frames))
    want_c, want_d = (a.copy() for a in ref.detect_batch_arrays(pre))
    assert np.array_equal(got_c, want_c) and int(want_c.sum()) > 0
    for f, k in enumerate(want_c):
        assert np.array_equal(got_d[f, :k], want_d[f, :k])
    a, b = eng.fetch_armors(3), ref.fetch_armors(3)
    assert a.tobytes() == b.tobytes(), "armors"
    assert eng.fetch_armor_poses(3).tobytes() == ref.fetch_armor_poses(3).tobytes(), "armor poses"
    print(f"1920x1200-c{chan}-lut: detections {int(want_c.sum())}, armors {int(b['valid'].sum())}")
    eng.close(); ref.close()


# ------------------------------------------------------------------------------------------------------ d. limits
def test_stage_takes_the_largest_width():
    """A 32766-pixel-wide source: ROI columns up to the 16-bit limit (whole-frame box, pair at the right edge)."""
    _cuda()
    import irmv_detection_b200 as irmv
    W, H = MAX_SIDE, 64
    view = np.zeros((H, W, 3), np.uint8)
    _pair(view, W - 40.5, 32.5, 24.0, 5.0, 28.0, 6.0, (255, 255, 255))
    boxes = np.array([[-1e9, -1e9, 1e9, 1e9], [W - 90, 0, W + 50, H]], np.float32)
    for chan, rot in ((0, True), (3, False)):
        frame = _camera_frame(view, chan, rot)
        got = irmv.extract_armors(frame[None], A.boxes_struct(boxes, [0.9, 0.8], [3, 4], 2), [2], chan_order=chan,
                                  rotate180=rot)[0]
        n_ref, excused = A.check_armors(got, A.rotated_image(frame, chan, rot), boxes, [0.9, 0.8], [3, 4])
        assert n_ref == 2 and not excused, (n_ref, excused)


@pytest.mark.parametrize("W,H,chan,what", [(MAX_SIDE + 1, 8, 0, "32766"), (8, MAX_SIDE + 1, 2, "32766"),
                                           (16383, 16383, 2, "2^31")])
def test_stage_refuses_sizes_up_front(weights_seed0, W, H, chan, what):
    _cuda()
    import irmv_detection_b200 as irmv
    frames = np.zeros((1, H, W) + (() if chan >= 2 else (3,)), np.uint8)
    with pytest.raises(irmv.IrmvError, match=what.replace("^", r"\^")):
        irmv.extract_armors(frames, A.boxes_struct(np.array([[0, 0, 8, 8]], np.float32), [0.5], [0], 1), [1],
                            chan_order=chan)
    if H <= 8:                                                  # an engine of that size takes no armor stage
        eng = irmv.YoloEngine(weights_seed0, (W, H), chan_order=chan, max_batch=1)
        with pytest.raises(irmv.IrmvError, match=what):
            eng.enable_armors()
        eng.close()
