"""The pose kernels (`pnp_kernel`, `pnp_refine_kernel`, csrc/pnp.cu) against the PnP oracle and cv2 beyond the
default camera: every camera of oracle.pnp_ref.CAMERAS, both armor sizes, two pose envelopes, pixel noise,
undistortion past the invertible radius, degenerate quads, batch edges, and the engine's fused pose stage with a
non-default camera.

Metric: rotations as matrices, ||Rodrigues(r_gpu) - R_ref||_F with R_ref straight from the oracle (scaled near a
half turn, see pnp_ref.rotation_error); translations relatively; quaternions against tf2 of R_ref.  Where the two
IPPE solutions tie (|e1 - e2| <= 1e-6 max) either may come first: the kernel must then match one of the oracle's two
poses.  Each cell prints its worst rotation and translation error and the number of excused near-ties.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

# Kernel vs oracle and kernel vs cv2.solvePnP.  Worst values over all cells of test_cameras_sizes_envelopes_noise,
# measured on an NVIDIA B200 at its 1000 W power limit: rotation 4.2e-11 (second solution; first 9.6e-12),
# translation 4.8e-12 relative (vs cv2 3.2e-11), quaternion 2.1e-12, rmse 5.9e-8 relative (noise-free quads, whose
# RMSE is ~1e-9).  Leaving out the FP32 rounding of the undistorted points alone moves the pose by 5e-6, 5000x
# above these bounds.
R_TOL = 1e-9
T_TOL = 1e-9
Q_TOL = 1e-10
RMSE_TOL = 1e-6          # relative, on the normalised reprojection RMSE of both solutions
LM_TOL = 1e-4            # refined pose vs cv2.solvePnPRefineLM where both reach the same minimum

CAMERAS = ["default", "k3_tangential", "pincushion", "strong_barrel", "wide", "no_distortion",
           "anisotropic_offcentre", "telephoto"]


def _cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _rodrigues(rv):
    import cv2
    return np.array([cv2.Rodrigues(np.asarray(r, np.float64).reshape(3, 1))[0] for r in rv]).reshape(-1, 3, 3)


def _trel(t, t_ref):
    return np.linalg.norm(t - t_ref, axis=1) / np.linalg.norm(t_ref, axis=1)


def _match(rv, tv, ref, tie):
    """Errors of the poses (rv, tv) against the oracle's first solution, or against whichever of its two
    solutions is nearer where they tie.  Returns (rotation error, translation error, took the second)."""
    from oracle import pnp_ref as P
    R = _rodrigues(rv)
    d1 = P.rotation_error(R, ref["R1"]), _trel(tv, ref["t1"])
    d2 = P.rotation_error(R, ref["R2"]), _trel(tv, ref["t2"])
    second = tie & (d2[0] + d2[1] < d1[0] + d1[1])
    return np.where(second, d2[0], d1[0]), np.where(second, d2[1], d1[1]), second


def _ties(ref):
    return np.abs(ref["e1"] - ref["e2"]) <= 1e-6 * np.maximum(ref["e1"], ref["e2"])


def _cv2_errors(rv, tv, rc, tc, tie):
    """Kernel pose vs cv2's, near-ties excused: there cv2 and the kernel may each take either solution
    (the comparison with the oracle covers both)."""
    from oracle import pnp_ref as P
    dr, dt = P.rotation_error(_rodrigues(rv), _rodrigues(rc)), _trel(tv, tc)
    return np.where(tie, 0.0, dr), np.where(tie, 0.0, dt)


# ------------------------------------------------------------------ 1. undistortion past the invertible radius
def _wide_stop_quads(n, seed):
    """Quads of the wide camera whose four corners all lie where undistortPoints takes its icdist < 0 exit
    (beyond ~500 px from the centre).  Its lens model cannot project there, so the armors are projected
    through the pinhole part of the camera."""
    from irmv_detection_b200 import synth
    from oracle import pnp_ref as P
    K, D, (w, h) = P.CAMERAS["wide"]
    q = synth.armor_quads(8 * n, seed, 0.3, K, np.zeros(5), w, h, dist=(1.0, 6.0), yaw=70.0, roll=180.0, margin=0.0)
    _, stop = P.undistort_points(q.astype(np.float64), K, D, with_stop=True)
    q = q[stop.all(1)][:n]
    assert len(q) == n
    return q


def test_undistort_stops_where_opencv_stops():
    """Wide camera, corners beyond the invertible radius: cv2.undistortPoints keeps the initial guess there.
    The stand-alone solver (single and batch call) returns cv2.solvePnP's pose and the oracle's."""
    import irmv_detection_b200 as irmv
    from oracle import pnp_ref as P
    _cuda()
    K, D, _ = P.CAMERAS["wide"]
    q = _wide_stop_quads(200, 21)
    s = irmv.PnPSolver(K, D)
    rv, tv, ok = s.solve_batch(q)
    ref = P.ippe_solutions(q, K, D)
    tie = _ties(ref)
    rc, tc, okc = P.solve_cv2(q, K, D)
    assert ok.all() and okc.all()
    dr, dt, _ = _match(rv, tv, ref, tie)
    cr, ct = _cv2_errors(rv, tv, rc, tc, tie)
    print(f"\n[icdist<0] n={len(q)} R={dr.max():.2e} t={dt.max():.2e} cv2 R={cr.max():.2e} t={ct.max():.2e} ties={int(tie.sum())}")
    assert dr.max() < R_TOL and dt.max() < T_TOL
    assert cr.max() < R_TOL and ct.max() < T_TOL
    for i in range(0, len(q), 25):
        o, r, t = s.solvePnP(q[i])
        assert o and np.array_equal(r.ravel(), rv[i]) and np.array_equal(t.ravel(), tv[i])
    s.close()


# ------------------------------------------------------------------ 2. cameras x armor size x envelope x noise
@pytest.mark.parametrize("camera", CAMERAS)
def test_cameras_sizes_envelopes_noise(camera):
    """solve_batch(extended=True) against the oracle (both solutions, rmse, quaternion = tf2 of the oracle's R,
    |q| = 1, ok) and the first solution against cv2.solvePnP, for one camera x both armor sizes x the survey
    and the wide envelope x noise 0 / 0.5 px."""
    import irmv_detection_b200 as irmv
    from oracle import pnp_ref as P
    _cuda()
    K, D, _ = P.CAMERAS[camera]
    s = irmv.PnPSolver(K, D)
    for large in (False, True):
        for env in P.ENVELOPES:
            for noise in (0.0, 0.5):
                cell = f"{camera} large={int(large)} {env} noise={noise}"
                q = P.camera_quads(camera, 300, seed=31, large=large, envelope=env, noise_px=noise)
                rv, tv, ok, quat, rv2, tv2, rmse = s.solve_batch(q, large_armor=large, extended=True)
                ref = P.ippe_solutions(q, K, D, large)
                tie = _ties(ref)
                assert ok.all(), cell
                dr, dt, second = _match(rv, tv, ref, tie)
                # the other solution: the oracle's pose that the first did not take
                other = {"R1": np.where(second[:, None, None], ref["R1"], ref["R2"]),
                         "t1": np.where(second[:, None], ref["t1"], ref["t2"])}
                dr2 = P.rotation_error(_rodrigues(rv2), other["R1"])
                dt2 = _trel(tv2, other["t1"])
                e_ref = np.where(second[:, None], np.stack([ref["e2"], ref["e1"]], 1), np.stack([ref["e1"], ref["e2"]], 1))
                de = np.abs(rmse - e_ref) / np.maximum(e_ref, 1e-300)
                q_ref = P.tf2_quaternion(np.where(second[:, None, None], ref["R2"], ref["R1"]))
                dq = np.abs(quat - q_ref).max(1)
                rc, tc, okc = P.solve_cv2(q[:100], K, D, large)
                cr, ct = _cv2_errors(rv[:100][okc], tv[:100][okc], rc[okc], tc[okc], tie[:100][okc])
                print(f"\n[{cell}] R={dr.max():.2e} t={dt.max():.2e} R2={dr2.max():.2e} t2={dt2.max():.2e} "
                      f"rmse={de.max():.2e} q={dq.max():.2e} cv2 R={cr.max():.2e} t={ct.max():.2e} ties={int(tie.sum())}")
                assert dr.max() < R_TOL and dt.max() < T_TOL, cell
                assert dr2.max() < R_TOL and dt2.max() < T_TOL, cell
                assert de.max() < RMSE_TOL, cell
                assert dq.max() < Q_TOL, cell
                np.testing.assert_allclose(np.linalg.norm(quat, axis=1), 1.0, rtol=0, atol=1e-12)
                assert okc.all() and cr.max() < R_TOL and ct.max() < T_TOL, cell
                # the plain batch call returns the first solution of the extended one bit for bit
                rvp, tvp, okp = s.solve_batch(q, large_armor=large)
                assert np.array_equal(rvp, rv) and np.array_equal(tvp, tv) and np.array_equal(okp, ok)
    s.close()


# ------------------------------------------------------------------ 3. degenerate and hostile inputs
def _hostile_quads():
    nan = np.nan
    return {
        "duplicate corner": [[300, 320], [300, 320], [400, 282], [398, 322]],
        "collinear 4": [[300, 300], [320, 300], [340, 300], [360, 300]],
        "collinear 3": [[300, 320], [302, 280], [304, 240], [398, 322]],
        "zero area": [[300, 300]] * 4,
        "self-crossing": [[300, 320], [400, 282], [302, 280], [398, 322]],
        "mirrored order": [[398, 322], [400, 282], [302, 280], [300, 320]],
        "nan corner": [[nan, 320], [302, 280], [400, 282], [398, 322]],
        "far off frame": [[3e4, 320], [3e4 + 2, 280], [3e4 + 100, 282], [3e4 + 98, 322]],
        "far off frame, negative": [[-3e4, -3e4 + 40], [-3e4 + 2, -3e4], [-3e4 + 100, -3e4 + 2], [-3e4 + 98, -3e4 + 42]],
    }


@pytest.mark.parametrize("camera", ["default", "wide"])
def test_degenerate_and_hostile_quads(camera):
    """Duplicate corner, collinear corners, zero area, self-crossing and mirrored order, a NaN corner, corners
    3e4 px off the frame: no error, ok <=> every output finite, a finite pose wherever cv2 returns one, and
    valid quads interleaved with these give bit for bit what they give without them."""
    import irmv_detection_b200 as irmv
    from oracle import pnp_ref as P
    _cuda()
    K, D, _ = P.CAMERAS[camera]
    hostile = _hostile_quads()
    names = list(hostile)
    bad = np.array([hostile[k] for k in names], np.float32)
    good = P.camera_quads(camera, 64, seed=41, envelope="wide")
    s = irmv.PnPSolver(K, D)
    for large in (False, True):
        rv, tv, ok, quat, rv2, tv2, rmse = s.solve_batch(bad, large_armor=large, extended=True)
        finite = np.isfinite(rv).all(1) & np.isfinite(tv).all(1) & np.isfinite(quat).all(1)
        assert np.array_equal(ok, finite), dict(zip(names, zip(ok, finite)))
        rc, tc, okc = P.solve_cv2(bad, K, D, large)
        cv_finite = okc & np.isfinite(rc).all(1) & np.isfinite(tc).all(1)
        print(f"\n[hostile {camera} large={int(large)}] " + ", ".join(f"{k}: ok={int(o)} cv2={int(c)}"
                                                                      for k, o, c in zip(names, ok, cv_finite)))
        assert ok[cv_finite].all(), [k for k, o, c in zip(names, ok, cv_finite) if c and not o]
        # interleave: good, bad, good, bad, ...
        mixed = np.empty((len(good) + len(bad) * 4, 4, 2), np.float32)
        slot = np.zeros(len(mixed), bool)
        gi = np.sort(np.random.default_rng(5).choice(len(mixed), len(good), replace=False))
        slot[gi] = True
        mixed[slot] = good
        mixed[~slot] = np.tile(bad, (4, 1, 1))
        a = s.solve_batch(good, large_armor=large, extended=True)
        b = s.solve_batch(mixed, large_armor=large, extended=True)
        for x, y in zip(a, b):
            assert np.array_equal(x, y[slot])
    s.close()


# ------------------------------------------------------------------ 4. LM refinement
@pytest.mark.parametrize("camera", ["k3_tangential", "anisotropic_offcentre", "telephoto"])
def test_lm_refinement_cameras(camera):
    """IPPE + LM with k3 and tangential terms, both armor sizes, against cv2.solvePnPRefineLM from the same IPPE
    poses: never a higher pixel reprojection error than the IPPE pose, at least as converged as OpenCV, and the
    same pose where both reach the same minimum."""
    import irmv_detection_b200 as irmv
    from oracle import pnp_ref as P
    _cuda()
    K, D, _ = P.CAMERAS[camera]
    s = irmv.PnPSolver(K, D)
    for large in (False, True):
        q = P.camera_quads(camera, 300, seed=51, large=large)
        s.set_refine_lm(0)
        r0, t0, _ = s.solve_batch(q, large_armor=large)
        s.set_refine_lm(30)
        r1, t1, ok1, quat, _, _, _ = s.solve_batch(q, large_armor=large, extended=True)
        assert ok1.all()
        rc, tc = P.refine_lm_cv2(q, r0, t0, K, D, large)
        e0, e1, ec = (P.reprojection_rmse_px(q, a, b, K, D, large) for a, b in ((r0, t0), (r1, t1), (rc, tc)))
        assert (e1 <= e0 + 1e-9).all()
        assert (e1 <= ec + 1e-6).all()
        same = np.abs(e1 - ec) < 1e-6
        R1 = _rodrigues(r1)
        dr, dt = P.rotation_error(R1, _rodrigues(rc)), _trel(t1, tc)
        dq = np.abs(quat - P.tf2_quaternion(R1)).max(1)
        print(f"\n[LM {camera} large={int(large)}] same={same.mean():.3f} R={dr[same].max():.2e} t={dt[same].max():.2e}")
        assert same.mean() > 0.97
        assert dr[same].max() < LM_TOL and dt[same].max() < LM_TOL
        assert dq.max() < 1e-9
    s.close()


# ------------------------------------------------------------------ 5. batch plumbing
def test_batch_edges_and_device_entry():
    """n = 1, 127, 128, 129 at two offsets, and the device-pointer entry: bit for bit one large batch."""
    import torch
    import irmv_detection_b200 as irmv
    from oracle import pnp_ref as P
    _cuda()
    K, D, _ = P.CAMERAS["k3_tangential"]
    q = P.camera_quads("k3_tangential", 600, seed=61, large=True, envelope="wide")
    s = irmv.PnPSolver(K, D)
    big = s.solve_batch(q, large_armor=True, extended=True)
    for n in (1, 127, 128, 129):
        for off in (0, 301):
            part = s.solve_batch(q[off:off + n], large_armor=True, extended=True)
            for x, y in zip(big, part):
                assert np.array_equal(x[off:off + n], y), (n, off)
            dev = torch.from_numpy(np.ascontiguousarray(q[off:off + n])).cuda()
            rv, tv, ok = np.empty((n, 3)), np.empty((n, 3)), np.empty(n, np.uint8)
            s.solve_batch_device(dev.data_ptr(), n, rv, tv, ok, large_armor=True)
            assert np.array_equal(rv, big[0][off:off + n]) and np.array_equal(tv, big[1][off:off + n])
            assert np.array_equal(ok.astype(bool), big[2][off:off + n])
    s.close()


# ------------------------------------------------------------------ 6. the engine's pose stage, non-default camera
ENGINE_CAMERA = "k3_tangential"     # 1280 x 1024 like the engine's frames, so corner_scale = (1, 1)


def _engine_vs_solver(eng, quads_of_frame, n, s, cx, cy, centers_of_frame=None):
    """The engine's fused poses (fetch_poses, fetch_armor_poses) of n frames against PnPSolver.solve_batch on
    the engine's own quads, bit for bit; distance_to_image_center against the camera's (cx, cy) in FP32."""
    rv, tv, ok = eng.fetch_poses(n)
    poses = eng.fetch_armor_poses(n)
    solved = 0
    for f in range(n):
        q, live = quads_of_frame(f)
        k = len(q)
        if k == 0:
            continue
        srv, stv, sok, squat, _, _, _ = s.solve_batch(q, extended=True)
        sok = sok & live
        assert np.array_equal(ok[f, :k], sok), f
        m = sok
        assert np.array_equal(rv[f, :k][m], srv[m]) and np.array_equal(tv[f, :k][m], stv[m]), f
        p = poses[f, :k]
        assert np.array_equal(p["ok"][m], np.ones(m.sum(), np.int32))
        assert np.array_equal(p["orientation"][m], squat[m]) and np.array_equal(p["position"][m], stv[m])
        if centers_of_frame is None:
            c = np.stack([(q[:, 0, 0] + q[:, 1, 0]) + (q[:, 2, 0] + q[:, 3, 0]),
                          (q[:, 0, 1] + q[:, 1, 1]) + (q[:, 2, 1] + q[:, 3, 1])], 1) * np.float32(0.25)
        else:
            c = centers_of_frame(f)
        dx, dy = c[:, 0] - np.float32(cx), c[:, 1] - np.float32(cy)
        want = np.sqrt(dx * dx + dy * dy)
        assert np.array_equal(p["distance_to_image_center"][m], want[m]), f
        solved += int(m.sum())
    return solved, (rv, tv, ok, poses)


def test_engine_pose_stage_non_default_camera(weights_seed0, tmp_path):
    """enable_pnp with a k3 / tangential camera on the box-corner path, the keypoint weight file and the fused
    armor stage: poses, quaternions and ok equal PnPSolver(K, D) on the engine's own FP32 quads bit for bit,
    distance_to_image_center uses that camera's (cx, cy), and a batch-1 engine gives what the replay gives."""
    import irmv_detection_b200 as irmv
    from irmv_detection_b200 import synth, weights as W
    from oracle import armor_ref as A, pnp_ref as P, preprocess_ref as PR
    _cuda()
    K, D, (w, h) = P.CAMERAS[ENGINE_CAMERA]
    cx, cy = K[2], K[5]
    s = irmv.PnPSolver(K, D)
    pose_w = str(tmp_path / "pose_seed0.irmw")
    W.write_random(pose_w, 0, pose=True)
    scenes = [PR.rot180(A.synth_armor_scene(10, sd)[0]) for sd in (7, 8)]
    frames = np.concatenate([synth.frames_from_base(synth.load_base(), 2, seed=4), np.stack(scenes)])
    n = len(frames)
    armor_kw = dict(binary_threshold=20, light_min_ratio=0.01, light_max_ratio=10.0, light_max_angle=90.0,
                    min_small_center_distance=0.0, max_large_center_distance=1e9)

    def engine(wpath, batch, armors):
        e = irmv.YoloEngine(wpath, (w, h), max_batch=batch, sub_batch=batch)
        if armors:
            e.enable_armors(**armor_kw)
        e.enable_pnp(K, D, (1.0, 1.0))
        return e

    for path, wpath, armors in (("boxes", weights_seed0, False), ("keypoints", pose_w, False), ("armors", pose_w, True)):
        eng = engine(wpath, n, armors)
        dets = eng.detect_batch(frames)
        kp = eng.fetch_keypoints(n) if path == "keypoints" else None
        arm = eng.fetch_armors(n) if armors else None

        def quads(f):
            k = len(dets[f])
            if path == "boxes":
                b = np.array([d.xyxy for d in dets[f]], np.float32).reshape(-1, 4)
                q = np.stack([b[:, [0, 3]], b[:, [0, 1]], b[:, [2, 1]], b[:, [2, 3]]], 1)
                return q, np.ones(k, bool)
            if path == "keypoints":
                return kp[f, :k].copy(), np.ones(k, bool)
            a = arm[f, :k]
            fill = np.array([[150, 160], [150, 140], [200, 140], [200, 160]], np.float32)
            q = np.where(a["valid"][:, None, None] != 0, a["pts"], fill)
            return q.astype(np.float32), a["valid"] != 0

        centers = (lambda f: arm[f, :len(dets[f])]["center"].astype(np.float32)) if armors else None
        solved, got = _engine_vs_solver(eng, quads, n, s, cx, cy, centers)
        print(f"\n[engine {path}] poses compared: {solved}")
        assert solved > 0, path
        eng.close()
        one = engine(wpath, 1, armors)
        for f in range(n):
            r = one.detect_batch(frames[f:f + 1])[0]
            assert r == dets[f], (path, f)
            k = len(r)
            rv1, tv1, ok1 = one.fetch_poses(1)
            assert np.array_equal(ok1[0, :k], got[2][f, :k]), (path, f)
            m = ok1[0, :k]
            assert np.array_equal(rv1[0, :k][m], got[0][f, :k][m]) and np.array_equal(tv1[0, :k][m], got[1][f, :k][m])
            p1 = one.fetch_armor_poses(1)[0, :k]
            assert np.array_equal(p1[m].tobytes(), got[3][f, :k][m].tobytes()), (path, f)
        one.close()
    s.close()
