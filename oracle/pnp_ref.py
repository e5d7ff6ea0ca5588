"""TEST INFRASTRUCTURE ONLY -- CPU oracle for PnPSolver::solvePnP.

Reference: /root/reference/src/pnp_solver.cpp:7-52 -- image points {left.bottom, left.top,
right.top, right.bottom} (:41-44), always the small-armor object points (:47-48, 23-28), then
cv::solvePnP(obj, img, K, D, rvec, tvec, false, SOLVEPNP_IPPE) (:49-51) with K/D from
/root/reference/config/camera_info.yaml:4-12.

The arithmetic lives in OpenCV calib3d (system dependency, version unpinned by package.xml:13);
the binary oracle in this image is cv2 4.13.0 (`solve_cv2`).  `solve_ippe` restates the
published algorithm (Collins & Bartoli, "Infinitesimal Plane-based Pose Estimation", IJCV 2014,
as implemented in OpenCV modules/calib3d/src/ippe.cpp and undistort.dispatch.cpp):
  1. undistortPoints: normalise with K, then exactly 5 fixed-point iterations of the
     plumb-bob inverse (TermCriteria default count 5); a point whose icdist turns negative
     stops at once with its initial guess, as OpenCV's does; result rounded to FP32 (the output
     array takes the Point2f input depth -- measured: without that rounding the restatement is
     5e-6 off cv2, with it 6e-11).  After the rounding it equals cv2.undistortPoints bit for bit
     on every pixel grid of CAMERAS (tests/test_pnp_ref_cameras.py);
  2. canonical object frame (centred, planar, z = 0) -- constant per armor size;
  3. exact homography canonical plane -> normalised image from the 4 correspondences;
  4. IPPE: Jacobian of the homography at the origin -> two rotations; translation by linear LSQ;
  5. back to the model frame, order the two poses by reprojection RMSE in normalised
     coordinates, return the lower;
  6. rotation matrix -> rvec with IPPE's rot2vec (axis from the skew part, angle = acos).
It is pinned against cv2.solvePnP on seeded quads in tests/test_oracle_cpu.py (<=1e-9 relative),
on the survey's known-answer vector (SURVEY.md section 8c), and across CAMERAS x both armor sizes x
both ENVELOPES x noise in tests/test_pnp_ref_cameras.py (rotation matrices and relative translations).

Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs may import this module.
"""
from __future__ import annotations

import numpy as np

# /root/reference/config/camera_info.yaml:4-12
K_DEFAULT = np.array([957.669211, 0.0, 345.943891, 0.0, 969.127115, 284.057302, 0.0, 0.0, 1.0])
D_DEFAULT = np.array([-0.405274, 0.126058, -0.026939, -0.006503, 0.0])

# /root/reference/include/irmv_detection/pnp_solver.hpp:30-33 (mm)
SMALL_W, SMALL_H, LARGE_W, LARGE_H = 135.0, 55.0, 225.0, 55.0

# The cameras the pose stage is checked with: name -> (K[9], D[5], (width, height)).  Only "wide" takes
# undistortPoints' icdist < 0 exit (pixels beyond ~500 px from its centre); tests/test_pnp_ref_cameras.py
# pins which camera does.
CAMERAS = {
    "default": (K_DEFAULT, D_DEFAULT, (640, 480)),
    "k3_tangential": (np.array([1200.0, 0.0, 640.0, 0.0, 1180.0, 512.0, 0.0, 0.0, 1.0]),
                      np.array([-0.3, 0.15, 0.001, -0.002, -0.05]), (1280, 1024)),
    "pincushion": (np.array([1200.0, 0.0, 640.0, 0.0, 1200.0, 512.0, 0.0, 0.0, 1.0]),
                   np.array([0.25, 0.05, 0.0, 0.0, 0.01]), (1280, 1024)),
    "strong_barrel": (np.array([1400.0, 0.0, 640.0, 0.0, 1400.0, 512.0, 0.0, 0.0, 1.0]),
                      np.array([-0.45, 0.0, 0.0, 0.0, 0.0]), (1280, 1024)),
    "wide": (np.array([800.0, 0.0, 640.0, 0.0, 800.0, 512.0, 0.0, 0.0, 1.0]),
             np.array([-0.5, 0.0, 0.0, 0.0, 0.0]), (1280, 1024)),
    "no_distortion": (np.array([1500.0, 0.0, 700.0, 0.0, 1500.0, 480.0, 0.0, 0.0, 1.0]), np.zeros(5), (1280, 1024)),
    "anisotropic_offcentre": (np.array([1100.0, 0.0, 702.3, 0.0, 1045.7, 431.9, 0.0, 0.0, 1.0]),
                              np.array([-0.21, 0.09, 0.0015, 0.0008, -0.02]), (1280, 1024)),
    "telephoto": (np.array([3000.0, 0.0, 960.0, 0.0, 3000.0, 600.0, 0.0, 0.0, 1.0]),
                  np.array([-0.08, 0.4, 0.0005, -0.0003, -1.2]), (1920, 1200)),
}

# Pose envelopes of synth.armor_quads: the survey's (its defaults) and a wide one -- grazing yaw, any roll,
# 0.3-25 m, armor centres up to 2 % from the frame edge.
ENVELOPES = {
    "survey": {},
    "wide": dict(dist=(0.3, 25.0), yaw=85.0, roll=180.0, margin=0.02),
}


def camera_quads(camera: str, n: int, seed: int, large: bool = False, envelope: str = "survey",
                 noise_px: float = 0.5) -> np.ndarray:
    """synth.armor_quads through CAMERAS[camera] on its own frame, poses drawn from ENVELOPES[envelope]."""
    from irmv_detection_b200 import synth
    K, D, (w, h) = CAMERAS[camera]
    return synth.armor_quads(n, seed, noise_px, K, D, w, h, large=large, **ENVELOPES[envelope])


def object_points(large: bool = False) -> np.ndarray:
    """/root/reference/src/pnp_solver.cpp:17-33: LB, LT, RT, RB; x forward, y left, z up (m)."""
    hy = (LARGE_W if large else SMALL_W) / 2.0 / 1000.0
    hz = (LARGE_H if large else SMALL_H) / 2.0 / 1000.0
    return np.array([[0, hy, -hz], [0, hy, hz], [0, -hy, hz], [0, -hy, -hz]], np.float64)


def undistort_points(pts: np.ndarray, K=K_DEFAULT, D=D_DEFAULT, iters: int = 5, with_stop: bool = False):
    """pts f64[...,2] pixel -> normalised undistorted coordinates (cv::undistortPoints, no R/P).

    Like OpenCV, a point whose icdist turns negative in an iteration (an iterate beyond the radius where the
    radial polynomial can be inverted) leaves the loop at once and keeps its initial guess (x0, y0).
    with_stop=True also returns the bool[...] mask of those points."""
    fx, fy, cx, cy = K[0], K[4], K[2], K[5]
    k1, k2, p1, p2, k3 = D[:5]
    x0 = (pts[..., 0] - cx) / fx
    y0 = (pts[..., 1] - cy) / fy
    x, y = x0.copy(), y0.copy()
    stop = np.zeros(x0.shape, bool)
    for _ in range(iters):
        r2 = x * x + y * y
        with np.errstate(divide="ignore", invalid="ignore"):
            icdist = 1.0 / (1.0 + ((k3 * r2 + k2) * r2 + k1) * r2)
        stop |= icdist < 0
        dx = 2.0 * p1 * x * y + p2 * (r2 + 2.0 * x * x)
        dy = p1 * (r2 + 2.0 * y * y) + 2.0 * p2 * x * y
        x = np.where(stop, x0, (x0 - dx) * icdist)
        y = np.where(stop, y0, (y0 - dy) * icdist)
    xy = np.stack((x, y), -1)
    return (xy, stop) if with_stop else xy


def _homography_rect_to_quad(a: float, b: float, q: np.ndarray) -> np.ndarray:
    """Exact homography taking the canonical rectangle corners to the 4 image points.

    Canonical corner order follows object_points(): (+a,-b), (+a,+b), (-a,+b), (-a,-b) with
    canonical X = model y, canonical Y = model z.  Square->quad closed form (Heckbert 1989)
    composed with the affine rectangle->unit-square map.  q f64[n,4,2].  Returns H f64[n,3,3],
    normalised so H[2,2] = 1.
    """
    x0, y0 = q[:, 0, 0], q[:, 0, 1]
    x1, y1 = q[:, 1, 0], q[:, 1, 1]
    x2, y2 = q[:, 2, 0], q[:, 2, 1]
    x3, y3 = q[:, 3, 0], q[:, 3, 1]
    dx1, dx2, sx = x1 - x2, x3 - x2, x0 - x1 + x2 - x3
    dy1, dy2, sy = y1 - y2, y3 - y2, y0 - y1 + y2 - y3
    det = dx1 * dy2 - dx2 * dy1
    g = (sx * dy2 - dx2 * sy) / det
    h = (dx1 * sy - sx * dy1) / det
    n = q.shape[0]
    Hs = np.empty((n, 3, 3))
    Hs[:, 0, 0] = x1 - x0 + g * x1
    Hs[:, 0, 1] = x3 - x0 + h * x3
    Hs[:, 0, 2] = x0
    Hs[:, 1, 0] = y1 - y0 + g * y1
    Hs[:, 1, 1] = y3 - y0 + h * y3
    Hs[:, 1, 2] = y0
    Hs[:, 2, 0] = g
    Hs[:, 2, 1] = h
    Hs[:, 2, 2] = 1.0
    # unit square (u,v): corner0=(0,0), corner1=(1,0), corner2=(1,1), corner3=(0,1)
    # canonical (X,Y): corner0=(+a,-b), corner1=(+a,+b), corner2=(-a,+b), corner3=(-a,-b)
    #   => u = (Y + b)/(2b), v = (a - X)/(2a)
    A = np.array([[0.0, 1.0 / (2 * b), 0.5], [-1.0 / (2 * a), 0.0, 0.5], [0.0, 0.0, 1.0]])
    H = Hs @ A
    return H / H[:, 2:3, 2:3]


def _rot_z_to(v: np.ndarray) -> np.ndarray:
    """Rotation Rv with Rv @ e_z = v/|v| (Rodrigues about e_z x v). v f64[n,3]."""
    a = v / np.linalg.norm(v, axis=1, keepdims=True)
    ax, ay, az = a[:, 0], a[:, 1], a[:, 2]
    n = v.shape[0]
    R = np.empty((n, 3, 3))
    k = 1.0 / (1.0 + az)
    R[:, 0, 0] = 1.0 - ax * ax * k
    R[:, 0, 1] = -ax * ay * k
    R[:, 0, 2] = ax
    R[:, 1, 0] = -ax * ay * k
    R[:, 1, 1] = 1.0 - ay * ay * k
    R[:, 1, 2] = ay
    R[:, 2, 0] = -ax
    R[:, 2, 1] = -ay
    R[:, 2, 2] = az
    return R


def _ippe_rotations(H: np.ndarray):
    j00 = H[:, 0, 0] - H[:, 2, 0] * H[:, 0, 2]
    j01 = H[:, 0, 1] - H[:, 2, 1] * H[:, 0, 2]
    j10 = H[:, 1, 0] - H[:, 2, 0] * H[:, 1, 2]
    j11 = H[:, 1, 1] - H[:, 2, 1] * H[:, 1, 2]
    p, q = H[:, 0, 2], H[:, 1, 2]
    n = H.shape[0]
    Rv = _rot_z_to(np.stack((p, q, np.ones(n)), 1))
    b00 = Rv[:, 0, 0] - p * Rv[:, 2, 0]
    b01 = Rv[:, 0, 1] - p * Rv[:, 2, 1]
    b10 = Rv[:, 1, 0] - q * Rv[:, 2, 0]
    b11 = Rv[:, 1, 1] - q * Rv[:, 2, 1]
    dtinv = 1.0 / (b00 * b11 - b01 * b10)
    bi00, bi01, bi10, bi11 = dtinv * b11, -dtinv * b01, -dtinv * b10, dtinv * b00
    a00 = bi00 * j00 + bi01 * j10
    a01 = bi00 * j01 + bi01 * j11
    a10 = bi10 * j00 + bi11 * j10
    a11 = bi10 * j01 + bi11 * j11
    ata00 = a00 * a00 + a01 * a01
    ata01 = a00 * a10 + a01 * a11
    ata11 = a10 * a10 + a11 * a11
    gamma = np.sqrt(0.5 * (ata00 + ata11 + np.sqrt((ata00 - ata11) ** 2 + 4.0 * ata01 * ata01)))
    r00, r01, r10, r11 = a00 / gamma, a01 / gamma, a10 / gamma, a11 / gamma
    b0 = np.sqrt(np.maximum(1.0 - r00 * r00 - r10 * r10, 0.0))
    b1 = np.sqrt(np.maximum(1.0 - r01 * r01 - r11 * r11, 0.0))
    sp = -(r00 * r01 + r10 * r11)
    b1 = np.where(sp < 0, -b1, b1)
    out = []
    for sgn in (1.0, -1.0):
        c1 = np.stack((r00, r10, sgn * b0), 1)
        c2 = np.stack((r01, r11, sgn * b1), 1)
        c3 = np.cross(c1, c2)
        Rt = np.stack((c1, c2, c3), 2)
        out.append(Rv @ Rt)
    return out


def _ippe_translation(X: np.ndarray, q: np.ndarray, R: np.ndarray) -> np.ndarray:
    """Linear least squares for t given R; X f64[4,2] canonical, q f64[n,4,2], R f64[n,3,3]."""
    Px = R[:, 0:1, 0] * X[None, :, 0] + R[:, 0:1, 1] * X[None, :, 1]
    Py = R[:, 1:2, 0] * X[None, :, 0] + R[:, 1:2, 1] * X[None, :, 1]
    Pz = R[:, 2:3, 0] * X[None, :, 0] + R[:, 2:3, 1] * X[None, :, 1]
    u, v = q[..., 0], q[..., 1]
    npts = X.shape[0]
    # normal equations of rows [1,0,-u | u*Pz-Px], [0,1,-v | v*Pz-Py]
    su, sv = u.sum(1), v.sum(1)
    suv2 = (u * u + v * v).sum(1)
    bx = (u * Pz - Px)
    by = (v * Pz - Py)
    r0, r1 = bx.sum(1), by.sum(1)
    r2 = -(u * bx + v * by).sum(1)
    n = q.shape[0]
    A = np.zeros((n, 3, 3))
    A[:, 0, 0] = npts
    A[:, 1, 1] = npts
    A[:, 0, 2] = A[:, 2, 0] = -su
    A[:, 1, 2] = A[:, 2, 1] = -sv
    A[:, 2, 2] = suv2
    rhs = np.stack((r0, r1, r2), 1)
    return np.linalg.solve(A, rhs[..., None])[..., 0]


def rot2vec(R: np.ndarray) -> np.ndarray:
    tr = R[:, 0, 0] + R[:, 1, 1] + R[:, 2, 2]
    w = np.arccos(np.clip((tr - 1.0) / 2.0, -1.0, 1.0))
    eps = np.finfo(np.float32).eps
    with np.errstate(divide="ignore", invalid="ignore"):
        d = w / (2.0 * np.sin(w))
    c = np.stack((R[:, 2, 1] - R[:, 1, 2], R[:, 0, 2] - R[:, 2, 0], R[:, 1, 0] - R[:, 0, 1]), 1)
    r = d[:, None] * c
    r[w < eps] = 0.0
    return r


def ippe_solutions(img_pts: np.ndarray, K=K_DEFAULT, D=D_DEFAULT, large: bool = False) -> dict:
    """Both IPPE poses of img_pts f32/f64[n,4,2] (LB,LT,RT,RB px), in OpenCV's order: the first is the one
    cv::solvePnP returns.  Keys: R1, R2 f64[n,3,3] rotation matrices (model -> camera), r1, r2 their rvecs,
    t1, t2 f64[n,3], e1, e2 f64[n] reprojection RMSE in normalised coordinates."""
    pts = np.asarray(img_pts, np.float32).astype(np.float64).reshape(-1, 4, 2)
    # cv::undistortPoints writes its result in the input depth (CV_32FC2 for Point2f input,
    # /root/reference/src/pnp_solver.cpp:37-44), so IPPE sees FP32-rounded normalised points.
    q = undistort_points(pts, K, D).astype(np.float32).astype(np.float64)
    obj = object_points(large)
    a, b = obj[0, 1], obj[1, 2]                      # half width (model y), half height (model z)
    Xc = np.stack((obj[:, 1], obj[:, 2]), 1)         # canonical X = model y, Y = model z
    H = _homography_rect_to_quad(a, b, q)
    Ra, Rb = _ippe_rotations(H)
    sols = []
    # canonical -> model: [X,Y,Z]_c = C @ [x,y,z]_m with rows (0,1,0),(0,0,1),(1,0,0), det = +1
    C = np.array([[0.0, 1.0, 0.0], [0.0, 0.0, 1.0], [1.0, 0.0, 0.0]])
    for R in (Ra, Rb):
        t = _ippe_translation(Xc, q, R)
        Rm = R @ C
        P = np.einsum("nij,kj->nki", Rm, obj) + t[:, None, :]
        proj = P[..., :2] / P[..., 2:3]
        err = np.sqrt(((proj - q) ** 2).sum((1, 2)) / (2.0 * 4))
        sols.append((Rm, t, err))
    first = sols[0][2].astype(np.float32) < sols[1][2].astype(np.float32)   # OpenCV compares floats
    # OpenCV: if (err1 < err2) keep order else swap  (ties -> second)
    out = {}
    for k, (i, j) in (("1", (0, 1)), ("2", (1, 0))):
        out["R" + k] = np.where(first[:, None, None], sols[i][0], sols[j][0])
        out["t" + k] = np.where(first[:, None], sols[i][1], sols[j][1])
        out["e" + k] = np.where(first, sols[i][2], sols[j][2])
        out["r" + k] = rot2vec(out["R" + k])
    return out


def solve_ippe(img_pts: np.ndarray, K=K_DEFAULT, D=D_DEFAULT, large: bool = False,
               both: bool = False):
    """img_pts f32/f64[n,4,2] (LB,LT,RT,RB px) -> rvec f64[n,3], tvec f64[n,3]; both=True:
    (r1, t1, r2, t2, e1, e2), see ippe_solutions."""
    s = ippe_solutions(img_pts, K, D, large)
    if not both:
        return s["r1"], s["t1"]
    return s["r1"], s["t1"], s["r2"], s["t2"], s["e1"], s["e2"]


def rotation_error(R: np.ndarray, R_ref: np.ndarray) -> np.ndarray:
    """||R - R_ref||_F per pose (f64[n,3,3] each), scaled by sin(theta_ref) past a quarter turn: near a
    half turn rot2vec (OpenCV's, the kernel's and ours) keeps only eps / sin(theta) of its precision, so
    the Rodrigues matrix of a returned rvec fixes the rotation no better than that."""
    d = np.linalg.norm(R - R_ref, axis=(1, 2))
    c = np.clip((np.trace(R_ref, axis1=1, axis2=2) - 1.0) / 2.0, -1.0, 1.0)
    return d * np.where(c < 0, np.sqrt(1.0 - c * c), 1.0)


def tf2_quaternion(R: np.ndarray) -> np.ndarray:
    """tf2::Matrix3x3::getRotation (x, y, z, w) of each R f64[n,3,3] (reference src/irm_detector.cpp:218-226)."""
    out = np.empty((R.shape[0], 4))
    for n, m in enumerate(R):
        tr = m[0, 0] + m[1, 1] + m[2, 2]
        q = np.zeros(4)
        if tr > 0:
            s = np.sqrt(tr + 1.0)
            q[3] = s * 0.5
            s = 0.5 / s
            q[0], q[1], q[2] = (m[2, 1] - m[1, 2]) * s, (m[0, 2] - m[2, 0]) * s, (m[1, 0] - m[0, 1]) * s
        else:
            i = (2 if m[1, 1] < m[2, 2] else 1) if m[0, 0] < m[1, 1] else (2 if m[0, 0] < m[2, 2] else 0)
            j, k = (i + 1) % 3, (i + 2) % 3
            s = np.sqrt(m[i, i] - m[j, j] - m[k, k] + 1.0)
            q[i] = s * 0.5
            s = 0.5 / s
            q[3], q[j], q[k] = (m[k, j] - m[j, k]) * s, (m[j, i] + m[i, j]) * s, (m[k, i] + m[i, k]) * s
        out[n] = q
    return out


def solve_cv2(img_pts: np.ndarray, K=K_DEFAULT, D=D_DEFAULT, large: bool = False):
    """The binary oracle: cv2.solvePnP(SOLVEPNP_IPPE) per quad, exactly the reference's call."""
    import cv2
    Km = np.asarray(K, np.float64).reshape(3, 3)
    Dm = np.asarray(D, np.float64).reshape(1, 5)
    obj = object_points(large)
    pts = np.asarray(img_pts, np.float32).reshape(-1, 4, 2)
    rv = np.empty((pts.shape[0], 3))
    tv = np.empty((pts.shape[0], 3))
    ok = np.zeros(pts.shape[0], bool)
    for i in range(pts.shape[0]):
        try:
            o, r, t = cv2.solvePnP(obj, pts[i], Km, Dm, flags=cv2.SOLVEPNP_IPPE)
        except cv2.error:
            o = False
        ok[i] = bool(o)
        if o:
            rv[i] = r.reshape(3)
            tv[i] = t.reshape(3)
    return rv, tv, ok


def project(rvec, tvec, K=K_DEFAULT, D=D_DEFAULT, large=False):
    import cv2
    Km = np.asarray(K, np.float64).reshape(3, 3)
    Dm = np.asarray(D, np.float64).reshape(1, 5)
    p, _ = cv2.projectPoints(object_points(large), np.asarray(rvec, np.float64),
                             np.asarray(tvec, np.float64), Km, Dm)
    return p.reshape(4, 2)


def synth_quads(n: int, seed: int = 0, noise_px: float = 0.5, K=K_DEFAULT, D=D_DEFAULT,
                img_w: int = 640, img_h: int = 480):
    """SURVEY.md section 8d config 5: seeded armor poses projected through K/D (+ pixel noise).  The
    generator lives with the other synthetic inputs (irmv_detection_b200/synth.py: armor_quads)."""
    from irmv_detection_b200 import synth
    return synth.armor_quads(n, seed, noise_px, K, D, img_w, img_h)


def refine_lm_cv2(img_pts: np.ndarray, rvecs: np.ndarray, tvecs: np.ndarray, K=K_DEFAULT, D=D_DEFAULT,
                  large: bool = False):
    """Oracle of the optional LM stage (NOT in the reference's call): cv2.solvePnPRefineLM with a
    tight termination criterion, started from the given poses."""
    import cv2
    obj = object_points(large)
    Km = np.asarray(K, np.float64).reshape(3, 3)
    Dm = np.asarray(D, np.float64).reshape(-1, 1)
    out_r, out_t = np.empty_like(rvecs), np.empty_like(tvecs)
    crit = (cv2.TERM_CRITERIA_EPS + cv2.TERM_CRITERIA_COUNT, 200, 1e-15)
    for i in range(len(img_pts)):
        r, t = cv2.solvePnPRefineLM(obj, np.asarray(img_pts[i], np.float64).reshape(4, 1, 2), Km, Dm,
                                    rvecs[i].reshape(3, 1).copy(), tvecs[i].reshape(3, 1).copy(), crit)
        out_r[i], out_t[i] = r.ravel(), t.ravel()
    return out_r, out_t


def reprojection_rmse_px(img_pts, rvecs, tvecs, K=K_DEFAULT, D=D_DEFAULT, large=False):
    import cv2
    obj = object_points(large)
    Km = np.asarray(K, np.float64).reshape(3, 3)
    Dm = np.asarray(D, np.float64).reshape(-1, 1)
    out = np.empty(len(img_pts))
    for i in range(len(img_pts)):
        pr, _ = cv2.projectPoints(obj, rvecs[i].reshape(3, 1), tvecs[i].reshape(3, 1), Km, Dm)
        out[i] = np.sqrt(np.mean((pr.reshape(4, 2) - np.asarray(img_pts[i], np.float64).reshape(4, 2)) ** 2))
    return out
