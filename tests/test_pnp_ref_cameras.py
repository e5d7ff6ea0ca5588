"""The PnP oracle (oracle/pnp_ref.py) against OpenCV beyond the default camera: every camera of CAMERAS,
both armor sizes, both pose envelopes, with and without pixel noise.  CPU only; the GPU kernels are
held to the oracle in tests/test_gpu_pnp_geometry.py."""
import hashlib

import numpy as np
import pytest

# Oracle vs cv2.solvePnP.  Measured worst over these cells: rotation 1.4e-11, translation 6.3e-11
# relative.  The FP32 rounding of the undistorted points alone moves the pose by 5e-6.
R_TOL = 1e-9
T_TOL = 1e-9


def test_undistort_matches_cv2_bit_for_bit():
    """cv2.undistortPoints on a sub-pixel grid over each camera's frame, corners and edges included, equals
    the oracle rounded to FP32 bit for bit.  Only the wide camera reaches the icdist < 0 exit, where OpenCV
    keeps the initial guess; an oracle that resets and iterates on differs from cv2 there."""
    import cv2
    from oracle import pnp_ref as P
    for name, (K, D, (w, h)) in P.CAMERAS.items():
        ys, xs = np.mgrid[0:h + 1:4, 0:w + 1:4]
        pts = np.stack([np.minimum(xs + 0.25, w - 0.5).ravel(), ys.ravel()], 1).astype(np.float32)
        pts = np.concatenate([pts, np.array([[0, 0], [w - 1, 0], [0, h - 1], [w - 1, h - 1]], np.float32)])
        want = cv2.undistortPoints(pts.reshape(-1, 1, 2), K.reshape(3, 3), D.reshape(1, 5)).reshape(-1, 2)
        got, stop = P.undistort_points(pts.astype(np.float64), K, D, with_stop=True)
        got = got.astype(np.float32)
        bad = (got != want).any(1)
        assert not bad.any(), f"{name}: {bad.sum()} points differ, first {pts[bad][0]}: {got[bad][0]} vs {want[bad][0]}"
        assert stop.any() == (name == "wide"), name
        if name == "wide":
            r = np.hypot(pts[stop, 0] - K[2], pts[stop, 1] - K[5])
            assert stop.mean() > 0.2 and r.min() > 450, (stop.mean(), r.min())


@pytest.mark.parametrize("camera", ["default", "k3_tangential", "pincushion", "strong_barrel", "wide",
                                    "no_distortion", "anisotropic_offcentre", "telephoto"])
def test_solve_ippe_matches_cv2(camera):
    """solve_ippe against cv2.solvePnP(IPPE) for one camera x both armor sizes x both envelopes x noise
    0 / 0.5 px.  Rotations are compared as matrices, translations relatively.  Where the two IPPE
    solutions tie (|e1 - e2| <= 1e-6 max), cv2 may return either, so the pose must match one of them."""
    import cv2
    from oracle import pnp_ref as P
    K, D, _ = P.CAMERAS[camera]
    for large in (False, True):
        for env in P.ENVELOPES:
            for noise in (0.0, 0.5):
                cell = f"{camera} large={large} {env} noise={noise}"
                q = P.camera_quads(camera, 150, seed=11, large=large, envelope=env, noise_px=noise)
                s = P.ippe_solutions(q, K, D, large)
                rc, tc, ok = P.solve_cv2(q, K, D, large)
                assert ok.all(), cell
                Rc = np.array([cv2.Rodrigues(r)[0] for r in rc])
                trel = lambda t: np.linalg.norm(t - tc, axis=1) / np.linalg.norm(tc, axis=1)
                dr1, dt1 = P.rotation_error(Rc, s["R1"]), trel(s["t1"])
                dr2, dt2 = P.rotation_error(Rc, s["R2"]), trel(s["t2"])
                tie = np.abs(s["e1"] - s["e2"]) <= 1e-6 * np.maximum(s["e1"], s["e2"])
                use2 = tie & (dr2 + dt2 < dr1 + dt1)
                dr, dt = np.where(use2, dr2, dr1), np.where(use2, dt2, dt1)
                assert dr.max() < R_TOL and dt.max() < T_TOL, (cell, dr.max(), dt.max(), int(tie.sum()))
                assert np.array_equal(s["r1"], P.solve_ippe(q, K, D, large)[0])


def test_armor_quads_defaults_unchanged():
    """synth.armor_quads' envelope arguments default to the survey's envelope: seeded quads stay bit for bit
    what they were before the arguments existed (these hashes were taken then)."""
    from irmv_detection_b200 import synth
    from oracle import pnp_ref as P
    cases = [(dict(n=2000, seed=0), "8b46e59999eb4032f206f61feaab28db0a0977cb488612d125bc854173801f5e"),
             (dict(n=500, seed=7, noise_px=0.0), "551b6787b2565e3e06c786ba509e85447d5fae9f421d3a1e8e18d18c71310bf1"),
             (dict(n=300, seed=3, K=P.K_DEFAULT, D=P.D_DEFAULT, img_w=1280, img_h=1024),
              "b1c2d0e7e43461ec8c9221bfe2116f0b84502f884aaee5e00359713e6e8d315e")]
    for args, want in cases:
        q = synth.armor_quads(**args)
        assert hashlib.sha256(q.tobytes()).hexdigest() == want, args


def test_armor_quads_envelope_arguments():
    """The envelope arguments do what they say: large armors are wider, the wide envelope reaches
    grazing yaw and the frame edge."""
    from oracle import pnp_ref as P
    K, D, (w, h) = P.CAMERAS["k3_tangential"]
    small = P.camera_quads("k3_tangential", 200, seed=5, noise_px=0.0)
    large = P.camera_quads("k3_tangential", 200, seed=5, large=True, noise_px=0.0)
    width = lambda q: np.linalg.norm(q[:, 0] - q[:, 3], axis=1)
    assert np.median(width(large) / width(small)) > 1.4
    wide = P.camera_quads("k3_tangential", 400, seed=5, envelope="wide", noise_px=0.0)
    assert (wide[..., 0] >= 0).all() and (wide[..., 0] < w).all() and (wide[..., 1] >= 0).all() and (wide[..., 1] < h).all()
    edge = np.minimum.reduce([wide[..., 0].min(1), w - wide[..., 0].max(1), wide[..., 1].min(1), h - wide[..., 1].max(1)])
    assert edge.min() < 0.05 * h
    s = P.ippe_solutions(wide, K, D)
    t = s["t1"][:, 2]
    assert t.min() < 1.0 and t.max() > 15.0
    ang = np.degrees(np.arccos(np.clip((np.trace(s["R1"], axis1=1, axis2=2) - 1) / 2, -1, 1)))
    assert ang.max() > 170.0
