"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/*.npz from the oracles in THIS container
(cv2 4.13.0, torch 2.11 CPU).  The reference holds no golden vectors for this path
(SURVEY.md section 4), so these seeded known-answer vectors are the pins:

  pnp_golden.npz   64 seeded quads -> cv2.solvePnP(SOLVEPNP_IPPE) rvec/tvec (the binary oracle)
  nms_golden.npz   clustered boxes/scores -> kept flat indices (oracle/nms_ref.py, cross-checked
                   against cv2.dnn.NMSBoxesBatched)
  pre_golden.npz   rm_test.jpg -> sha256 of the FP16 preprocess output per mode + a 16x16 crop
  net_golden.npz   rm_test.jpg, seed-0 weights -> top-32 scores/boxes of the FP32 oracle
  armor_golden.npz seeded light-bar scenes -> armors of the reference's extract_armors written with
                   the cv2 calls themselves (oracle/armor_ref.extract_armors_cv2)
  npp_random_golden.npz  a seeded random 1280x1024 frame -> the reference's NPP chain (oracle/_ref/npp_ref,
                   needs a GPU): sha256 of the 8-bit output + a crop of the FP32 output

Run:  python -m oracle.make_golden            (npp_random_golden.npz: python -m oracle.make_golden npp)
"""
import hashlib
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden")


def clustered(seed, A=8400, nc=14, n_obj=30, per=10):
    rng = np.random.default_rng(seed)
    boxes = np.zeros((A, 4), np.float32)
    scores = np.zeros((A, nc), np.float32)
    idx = rng.permutation(A)[: n_obj * per].reshape(n_obj, per)
    for o in range(n_obj):
        cx, cy, w, h = rng.uniform(60, 580), rng.uniform(60, 580), rng.uniform(20, 120), rng.uniform(20, 120)
        c = rng.integers(0, nc)
        for a in idx[o]:
            j = rng.normal(0, 4, 4)
            boxes[a] = [cx - w / 2 + j[0], cy - h / 2 + j[1], cx + w / 2 + j[2], cy + h / 2 + j[3]]
            scores[a, c] = rng.uniform(0.3, 0.99)
    return boxes, scores, idx.ravel()


def main():
    import cv2
    import torch
    from irmv_detection_b200 import synth, weights
    from oracle import nms_ref as N, pnp_ref as P, preprocess_ref as PR, yolov8n_ref as Y
    os.makedirs(OUT, exist_ok=True)
    # PnP
    q = P.synth_quads(64, seed=42)
    rv, tv, ok = P.solve_cv2(q)
    assert ok.all()
    np.savez_compressed(os.path.join(OUT, "pnp_golden.npz"), quads=q, rvec=rv, tvec=tv,
                        K=P.K_DEFAULT, D=P.D_DEFAULT, cv2_version=cv2.__version__)
    # NMS
    b, s, used = clustered(7)
    keep, kb, ks, kc = N.nms(b, s)
    np.savez_compressed(os.path.join(OUT, "nms_golden.npz"), boxes=b[used], scores=s[used], used=used.astype(np.int32),
                        keep=keep, keep_scores=ks, keep_classes=kc)
    # preprocess
    img = synth.load_base()
    rec = {}
    for chan, rot, quant in [(0, True, True), (1, True, True), (0, False, True), (0, True, False)]:
        x, _ = PR.preprocess_fp16(img, chan, rot, quant)
        key = f"c{chan}_r{int(rot)}_q{int(quant)}"
        rec[key + "_sha"] = np.frombuffer(hashlib.sha256(np.ascontiguousarray(x).tobytes()).digest(), np.uint8)
        rec[key + "_crop"] = x[:, 300:316, 300:316].copy()
    raw = PR.mosaic_from_rgb(img[..., ::-1], PR.CH_BAYER_RGGB)
    x, _ = PR.preprocess_fp16(raw, PR.CH_BAYER_RGGB, True, True)
    rec["bayer_rggb_sha"] = np.frombuffer(hashlib.sha256(np.ascontiguousarray(x).tobytes()).digest(), np.uint8)
    np.savez_compressed(os.path.join(OUT, "pre_golden.npz"), **rec)
    # network
    wp = "/tmp/_golden_seed0.irmw"
    weights.write_random(wp, 0)
    m = Y.build(wp)
    x, _ = PR.preprocess_fp16(img)
    with torch.no_grad():
        boxes, scores = m(torch.from_numpy(x.astype(np.float32))[None])
    boxes, scores = boxes[0].numpy(), scores[0].numpy()
    flat = scores.reshape(-1)
    top = np.argsort(-flat, kind="stable")[:32]
    keep, kb, ks, kc = N.nms(boxes, scores)
    np.savez_compressed(os.path.join(OUT, "net_golden.npz"), top_index=top.astype(np.int32), top_scores=flat[top],
                        top_boxes=boxes[top // 14], keep=keep, keep_scores=ks, keep_boxes=kb,
                        weights_sha=np.frombuffer(hashlib.sha256(open(wp, "rb").read()).digest(), np.uint8))
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


def armor_golden():
    """Known answers for the light/armor extraction, produced by the cv2 form of the reference's
    function (oracle/armor_ref.extract_armors_cv2) on seeded synthetic scenes."""
    from oracle import armor_ref as A
    rec = {}
    for seed in (0, 1, 2):
        img, boxes, scores, classes = A.synth_armor_scene(8, seed)
        arms = A.extract_armors_cv2(img, boxes, scores, classes)
        rec[f"boxes{seed}"] = boxes
        rec[f"scores{seed}"] = scores
        rec[f"classes{seed}"] = classes
        rec[f"index{seed}"] = np.array([a.bbox_index for a in arms], np.int32)
        rec[f"size{seed}"] = np.array([a.size for a in arms], np.int32)
        rec[f"pts{seed}"] = np.stack([a.pts for a in arms]).astype(np.float32)
        rec[f"center{seed}"] = np.stack([a.center for a in arms]).astype(np.float32)
    np.savez_compressed(os.path.join(OUT, "armor_golden.npz"), **rec)


NPP_RANDOM_SEED = 21
NPP_CROP = (slice(None), slice(288, 352), slice(288, 352))


def npp_random_frame() -> np.ndarray:
    """The seeded random frame of tests/test_gpu_parity.py::test_preprocess_matches_reference_npp_chain."""
    return np.random.default_rng(NPP_RANDOM_SEED).integers(0, 256, (1024, 1280, 3), dtype=np.uint8)


def run_npp_ref(img: np.ndarray, work_dir: str) -> np.ndarray:
    """The reference's NPP chain (oracle/_ref/npp_ref, built by oracle/Makefile) on a GPU: f32 [3, 640, 640]."""
    import subprocess
    exe = os.path.join(ROOT, "oracle", "_ref", "npp_ref")
    src, dst = os.path.join(work_dir, "npp_in.raw"), os.path.join(work_dir, "npp_out.f32")
    img.tofile(src)
    r = subprocess.run([exe, src, str(img.shape[1]), str(img.shape[0]), dst], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"npp_ref failed: {r.stderr}")
    return np.fromfile(dst, np.float32).reshape(3, 640, 640)


def npp_golden(out_dir: str = OUT):
    """The NPP chain's output for npp_random_frame(): the full output is 4.9 MB, so the sha256 of its 8-bit
    values (which pins every pixel) and an FP32 crop are stored."""
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        npp = run_npp_ref(npp_random_frame(), d)
    u8 = np.rint(npp * 255.0).astype(np.uint8)
    np.savez_compressed(os.path.join(out_dir, "npp_random_golden.npz"),
                        sha=np.frombuffer(hashlib.sha256(np.ascontiguousarray(u8).tobytes()).digest(), np.uint8),
                        crop=npp[NPP_CROP].copy())


if __name__ == "__main__":
    import sys
    if sys.argv[1:] == ["npp"]:
        npp_golden()
    else:
        main()
        armor_golden()
