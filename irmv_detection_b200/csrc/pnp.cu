// Batched planar PnP (IPPE) for the 4 armor corners, FP64, sm_100a.
// Replaces the per-armor CPU cv::solvePnP(..., SOLVEPNP_IPPE) call of the reference
// (reference src/pnp_solver.cpp:36-52) and, optionally, the Rodrigues -> tf2 quaternion step of
// the caller (reference src/irm_detector.cpp:218-226).  Algorithm = oracle/pnp_ref.py:
// undistort (5 fixed-point iterations, stopping at the initial guess where icdist < 0, result
// rounded to FP32 like cv::undistortPoints with Point2f input), exact rectangle->quad
// homography, IPPE two-rotation solve, linear-LSQ translation, sort by normalised reprojection
// RMSE, rot2vec.  No LM refinement (the reference's call has none, SURVEY.md section 0.6).
//
// 80 algorithmic bytes per armor (32 in, 48 out) against ~2.5 kFLOP of dependent FP64 math:
// the kernel is FP64-latency bound, so the mapping is one armor per thread with enough
// resident warps to cover the dependent chains.
#include "common.cuh"

namespace irmv {
namespace {

struct M3 { double m[3][3]; };

__device__ __forceinline__ void solve_translation(const double R[3][3], const double X[4],
                                                  const double Y[4], const double u[4],
                                                  const double v[4], double t[3]) {
  double su = 0, sv = 0, suv2 = 0, r0 = 0, r1 = 0, r2 = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    double Px = R[0][0] * X[i] + R[0][1] * Y[i];
    double Py = R[1][0] * X[i] + R[1][1] * Y[i];
    double Pz = R[2][0] * X[i] + R[2][1] * Y[i];
    double bx = u[i] * Pz - Px, by = v[i] * Pz - Py;
    su += u[i]; sv += v[i]; suv2 += u[i] * u[i] + v[i] * v[i];
    r0 += bx; r1 += by; r2 -= u[i] * bx + v[i] * by;
  }
  // normal matrix [[4,0,-su],[0,4,-sv],[-su,-sv,suv2]]; eliminate tx,ty
  const double n = 4.0;
  double den = suv2 - (su * su + sv * sv) / n;
  double tz = (r2 + (su * r0 + sv * r1) / n) / den;
  t[0] = (r0 + su * tz) / n;
  t[1] = (r1 + sv * tz) / n;
  t[2] = tz;
}

__device__ __forceinline__ void rot2vec(const double R[3][3], double r[3]) {
  double tr = R[0][0] + R[1][1] + R[2][2];
  double c = fmin(fmax((tr - 1.0) * 0.5, -1.0), 1.0);
  double w = acos(c);
  if (w < 1.1920928955078125e-07) { r[0] = r[1] = r[2] = 0.0; return; }
  double d = w / (2.0 * sin(w));
  r[0] = d * (R[2][1] - R[1][2]);
  r[1] = d * (R[0][2] - R[2][0]);
  r[2] = d * (R[1][0] - R[0][1]);
}

// tf2::Matrix3x3::getRotation (x,y,z,w)
__device__ __forceinline__ void rot2quat(const double m[3][3], double q[4]) {
  double trace = m[0][0] + m[1][1] + m[2][2];
  if (trace > 0.0) {
    double s = sqrt(trace + 1.0);
    q[3] = s * 0.5;
    s = 0.5 / s;
    q[0] = (m[2][1] - m[1][2]) * s;
    q[1] = (m[0][2] - m[2][0]) * s;
    q[2] = (m[1][0] - m[0][1]) * s;
  } else {
    int i = m[0][0] < m[1][1] ? (m[1][1] < m[2][2] ? 2 : 1) : (m[0][0] < m[2][2] ? 2 : 0);
    int j = (i + 1) % 3, k = (i + 2) % 3;
    double s = sqrt(m[i][i] - m[j][j] - m[k][k] + 1.0);
    q[i] = s * 0.5;
    s = 0.5 / s;
    q[3] = (m[k][j] - m[j][k]) * s;
    q[j] = (m[j][i] + m[i][j]) * s;
    q[k] = (m[k][i] + m[i][k]) * s;
  }
}

__global__ void __launch_bounds__(128) pnp_kernel(PnpConsts C, const float *__restrict__ pts, int n,
                                                  int large, PnpOut out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 *pp = reinterpret_cast<const float4 *>(pts) + (size_t)i * 2;
  float4 a = __ldg(pp), b = __ldg(pp + 1);
  double px[4] = {a.x, a.z, b.x, b.z}, py[4] = {a.y, a.w, b.y, b.w};

  // 1. undistort -> normalised coordinates, rounded to FP32
  double u[4], v[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    double x0 = (px[k] - C.cx) / C.fx, y0 = (py[k] - C.cy) / C.fy;
    double x = x0, y = y0;
#pragma unroll
    for (int it = 0; it < 5; ++it) {
      double r2 = x * x + y * y;
      double icd = 1.0 / (1.0 + ((C.k3 * r2 + C.k2) * r2 + C.k1) * r2);
      // past the radius where the radial polynomial can be inverted: OpenCV stops and keeps (x0, y0)
      if (icd < 0.0) { x = x0; y = y0; break; }
      double dx = 2.0 * C.p1 * x * y + C.p2 * (r2 + 2.0 * x * x);
      double dy = C.p1 * (r2 + 2.0 * y * y) + 2.0 * C.p2 * x * y;
      x = (x0 - dx) * icd;
      y = (y0 - dy) * icd;
    }
    u[k] = (double)(float)x;
    v[k] = (double)(float)y;
  }

  // 2. canonical rectangle (X = model y, Y = model z): (+a,-b),(+a,+b),(-a,+b),(-a,-b)
  const double ha = C.half_w[large ? 1 : 0], hb = C.half_h[large ? 1 : 0];
  const double X[4] = {ha, ha, -ha, -ha}, Y[4] = {-hb, hb, hb, -hb};

  // 3. exact homography: unit square -> quad (Heckbert), composed with rectangle -> square
  double dx1 = u[1] - u[2], dx2 = u[3] - u[2], sx = u[0] - u[1] + u[2] - u[3];
  double dy1 = v[1] - v[2], dy2 = v[3] - v[2], sy = v[0] - v[1] + v[2] - v[3];
  double det = dx1 * dy2 - dx2 * dy1;
  double g = (sx * dy2 - dx2 * sy) / det, h = (dx1 * sy - sx * dy1) / det;
  double s00 = u[1] - u[0] + g * u[1], s01 = u[3] - u[0] + h * u[3], s02 = u[0];
  double s10 = v[1] - v[0] + g * v[1], s11 = v[3] - v[0] + h * v[3], s12 = v[0];
  // A = [[0, 1/(2b), .5], [-1/(2a), 0, .5], [0,0,1]];  H = S * A, then / H22
  double ia = -1.0 / (2.0 * ha), ib = 1.0 / (2.0 * hb);
  double H[3][3];
  H[0][0] = s01 * ia; H[0][1] = s00 * ib; H[0][2] = 0.5 * (s00 + s01) + s02;
  H[1][0] = s11 * ia; H[1][1] = s10 * ib; H[1][2] = 0.5 * (s10 + s11) + s12;
  H[2][0] = h * ia;   H[2][1] = g * ib;   H[2][2] = 0.5 * (g + h) + 1.0;
  double inv22 = 1.0 / H[2][2];
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) H[r][c] *= inv22;

  // 4. IPPE rotations
  double j00 = H[0][0] - H[2][0] * H[0][2], j01 = H[0][1] - H[2][1] * H[0][2];
  double j10 = H[1][0] - H[2][0] * H[1][2], j11 = H[1][1] - H[2][1] * H[1][2];
  double p = H[0][2], q = H[1][2];
  double nrm = 1.0 / sqrt(p * p + q * q + 1.0);
  double ax = p * nrm, ay = q * nrm, az = nrm;
  double kk = 1.0 / (1.0 + az);
  double Rv[3][3] = {{1.0 - ax * ax * kk, -ax * ay * kk, ax},
                     {-ax * ay * kk, 1.0 - ay * ay * kk, ay},
                     {-ax, -ay, az}};
  double b00 = Rv[0][0] - p * Rv[2][0], b01 = Rv[0][1] - p * Rv[2][1];
  double b10 = Rv[1][0] - q * Rv[2][0], b11 = Rv[1][1] - q * Rv[2][1];
  double dtinv = 1.0 / (b00 * b11 - b01 * b10);
  double bi00 = dtinv * b11, bi01 = -dtinv * b01, bi10 = -dtinv * b10, bi11 = dtinv * b00;
  double a00 = bi00 * j00 + bi01 * j10, a01 = bi00 * j01 + bi01 * j11;
  double a10 = bi10 * j00 + bi11 * j10, a11 = bi10 * j01 + bi11 * j11;
  double ata00 = a00 * a00 + a01 * a01, ata01 = a00 * a10 + a01 * a11, ata11 = a10 * a10 + a11 * a11;
  double dd = ata00 - ata11;
  double gamma = sqrt(0.5 * (ata00 + ata11 + sqrt(dd * dd + 4.0 * ata01 * ata01)));
  double r00 = a00 / gamma, r01 = a01 / gamma, r10 = a10 / gamma, r11 = a11 / gamma;
  double bb0 = sqrt(fmax(1.0 - r00 * r00 - r10 * r10, 0.0));
  double bb1 = sqrt(fmax(1.0 - r01 * r01 - r11 * r11, 0.0));
  if (-(r00 * r01 + r10 * r11) < 0.0) bb1 = -bb1;

  double Rm[2][3][3], tt[2][3], err[2];
#pragma unroll
  for (int sol = 0; sol < 2; ++sol) {
    double sg = sol == 0 ? 1.0 : -1.0;
    double c1[3] = {r00, r10, sg * bb0}, c2[3] = {r01, r11, sg * bb1};
    double c3[3] = {c1[1] * c2[2] - c1[2] * c2[1], c1[2] * c2[0] - c1[0] * c2[2],
                    c1[0] * c2[1] - c1[1] * c2[0]};
    double Rc[3][3];   // canonical-frame rotation = Rv * [c1 c2 c3]
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      Rc[r][0] = Rv[r][0] * c1[0] + Rv[r][1] * c1[1] + Rv[r][2] * c1[2];
      Rc[r][1] = Rv[r][0] * c2[0] + Rv[r][1] * c2[1] + Rv[r][2] * c2[2];
      Rc[r][2] = Rv[r][0] * c3[0] + Rv[r][1] * c3[1] + Rv[r][2] * c3[2];
    }
    solve_translation(Rc, X, Y, u, v, tt[sol]);
    // 5. reprojection RMSE in normalised coordinates
    double e = 0.0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      double Px = Rc[0][0] * X[k] + Rc[0][1] * Y[k] + tt[sol][0];
      double Py = Rc[1][0] * X[k] + Rc[1][1] * Y[k] + tt[sol][1];
      double Pz = Rc[2][0] * X[k] + Rc[2][1] * Y[k] + tt[sol][2];
      double du = Px / Pz - u[k], dv = Py / Pz - v[k];
      e += du * du + dv * dv;
    }
    err[sol] = sqrt(e / 8.0);
    // canonical -> model frame: Rm = Rc * C, C rows (0,1,0),(0,0,1),(1,0,0)
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      Rm[sol][r][0] = Rc[r][2];
      Rm[sol][r][1] = Rc[r][0];
      Rm[sol][r][2] = Rc[r][1];
    }
  }
  // OpenCV compares the two errors as floats; the first wins only if strictly smaller
  int best = ((float)err[0] < (float)err[1]) ? 0 : 1;
  int other = best ^ 1;
  double rv[3];
  rot2vec(Rm[best], rv);
  bool ok = isfinite(rv[0]) && isfinite(rv[1]) && isfinite(rv[2]) && isfinite(tt[best][0]) &&
            isfinite(tt[best][1]) && isfinite(tt[best][2]);
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    out.rvec[(size_t)i * 3 + k] = rv[k];
    out.tvec[(size_t)i * 3 + k] = tt[best][k];
  }
  out.ok[i] = ok ? 1 : 0;
  if (out.quat) {
    double qv[4];
    rot2quat(Rm[best], qv);
#pragma unroll
    for (int k = 0; k < 4; ++k) out.quat[(size_t)i * 4 + k] = qv[k];
  }
  if (out.dist) {
    float cxp, cyp;
    if (out.centers) { cxp = out.centers[(size_t)i * 2]; cyp = out.centers[(size_t)i * 2 + 1]; }
    else {
      const float4 *pq = reinterpret_cast<const float4 *>(pts) + (size_t)i * 2;
      const float4 qa = __ldg(pq), qb = __ldg(pq + 1);
      cxp = __fmul_rn(__fadd_rn(__fadd_rn(qa.x, qa.z), __fadd_rn(qb.x, qb.z)), 0.25f);
      cyp = __fmul_rn(__fadd_rn(__fadd_rn(qa.y, qa.w), __fadd_rn(qb.y, qb.w)), 0.25f);
    }
    const float dx = __fsub_rn(cxp, (float)C.cx), dy = __fsub_rn(cyp, (float)C.cy);
    out.dist[i] = __fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
  }
  if (out.rvec2) {
    double rv2[3];
    rot2vec(Rm[other], rv2);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      out.rvec2[(size_t)i * 3 + k] = rv2[k];
      out.tvec2[(size_t)i * 3 + k] = tt[other][k];
    }
    out.rmse[(size_t)i * 2 + 0] = err[best];
    out.rmse[(size_t)i * 2 + 1] = err[other];
  }
}

// ------------------------------------------------------------------ optional LM refinement
// Levenberg-Marquardt on the pixel reprojection error of the 4 corners (plumb-bob projection with
// K and D), 6 parameters, started from the IPPE pose.  NOT part of the reference's call
// (cv::solvePnP(..., SOLVEPNP_IPPE) has no refinement, SURVEY.md section 0.6): this is the
// north_star's "IPPE + LM" stage, oracle = cv2.solvePnPRefineLM.  The rotation is updated
// multiplicatively (R <- exp(dw) R), which has the same minimiser as OpenCV's rvec
// parametrisation; one armor per thread, FP64.
__device__ __forceinline__ void rodrigues(const double r[3], double R[3][3]) {
  const double th2 = r[0] * r[0] + r[1] * r[1] + r[2] * r[2];
  const double th = sqrt(th2);
  double a, b;                       // a = sin(th)/th, b = (1 - cos(th))/th^2
  if (th < 1e-8) { a = 1.0 - th2 / 6.0; b = 0.5 - th2 / 24.0; }
  else { a = sin(th) / th; b = (1.0 - cos(th)) / th2; }
  const double x = r[0], y = r[1], z = r[2];
  R[0][0] = 1.0 - b * (y * y + z * z); R[0][1] = -a * z + b * x * y;        R[0][2] = a * y + b * x * z;
  R[1][0] = a * z + b * x * y;         R[1][1] = 1.0 - b * (x * x + z * z); R[1][2] = -a * x + b * y * z;
  R[2][0] = -a * y + b * x * z;        R[2][1] = a * x + b * y * z;         R[2][2] = 1.0 - b * (x * x + y * y);
}

// residuals (8) and cost of pose (R, t); optionally the normal equations JtJ (upper, 21) and Jtf (6)
__device__ __forceinline__ double lm_eval(const PnpConsts &C, const double R[3][3], const double t[3], const double ha,
                                          const double hb, const double px[4], const double py[4], bool want_j,
                                          double JtJ[6][6], double Jtf[6]) {
  double cost = 0.0;
  if (want_j) {
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      Jtf[i] = 0.0;
#pragma unroll
      for (int j = 0; j < 6; ++j) JtJ[i][j] = 0.0;
    }
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    // model-frame corners LB, LT, RT, RB: (0, +-ha, -+hb)  (reference src/pnp_solver.cpp:23-28)
    const double Y = (k < 2) ? ha : -ha, Z = (k == 1 || k == 2) ? hb : -hb;
    const double a0 = R[0][1] * Y + R[0][2] * Z, a1 = R[1][1] * Y + R[1][2] * Z, a2 = R[2][1] * Y + R[2][2] * Z;
    const double Px = a0 + t[0], Py = a1 + t[1], Pz = a2 + t[2];
    const double iz = 1.0 / Pz, xn = Px * iz, yn = Py * iz;
    const double r2 = xn * xn + yn * yn;
    const double rad = 1.0 + ((C.k3 * r2 + C.k2) * r2 + C.k1) * r2;
    const double xd = xn * rad + 2.0 * C.p1 * xn * yn + C.p2 * (r2 + 2.0 * xn * xn);
    const double yd = yn * rad + C.p1 * (r2 + 2.0 * yn * yn) + 2.0 * C.p2 * xn * yn;
    const double fu = C.fx * xd + C.cx - px[k], fv = C.fy * yd + C.cy - py[k];
    cost += fu * fu + fv * fv;
    if (want_j) {
      const double g = (3.0 * C.k3 * r2 + 2.0 * C.k2) * r2 + C.k1;        // d rad / d r2
      const double dxx = rad + 2.0 * g * xn * xn + 2.0 * C.p1 * yn + 6.0 * C.p2 * xn;
      const double dxy = 2.0 * g * xn * yn + 2.0 * C.p1 * xn + 2.0 * C.p2 * yn;
      const double dyy = rad + 2.0 * g * yn * yn + 6.0 * C.p1 * yn + 2.0 * C.p2 * xn;
      // d(xn, yn)/dP
      const double nx[3] = {iz, 0.0, -xn * iz}, ny[3] = {0.0, iz, -yn * iz};
      double gu[3], gv[3];            // d(u, v)/dP
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        gu[c] = C.fx * (dxx * nx[c] + dxy * ny[c]);
        gv[c] = C.fy * (dxy * nx[c] + dyy * ny[c]);
      }
      // dP/d(dw) = -skew(a): columns (0, a2, -a1)... i.e. grad . (dw x a) = dw . (a x grad)
      const double Ju[6] = {a1 * gu[2] - a2 * gu[1], a2 * gu[0] - a0 * gu[2], a0 * gu[1] - a1 * gu[0], gu[0], gu[1], gu[2]};
      const double Jv[6] = {a1 * gv[2] - a2 * gv[1], a2 * gv[0] - a0 * gv[2], a0 * gv[1] - a1 * gv[0], gv[0], gv[1], gv[2]};
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        Jtf[i] += Ju[i] * fu + Jv[i] * fv;
#pragma unroll
        for (int j = i; j < 6; ++j) JtJ[i][j] += Ju[i] * Ju[j] + Jv[i] * Jv[j];
      }
    }
  }
  return cost;
}

__global__ void __launch_bounds__(64) pnp_refine_kernel(PnpConsts C, const float *__restrict__ pts, int n, int large,
                                                       int max_iters, double *rvec, double *tvec, double *quat) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 *pp = reinterpret_cast<const float4 *>(pts) + (size_t)i * 2;
  const float4 pa = __ldg(pp), pb = __ldg(pp + 1);
  const double px[4] = {pa.x, pa.z, pb.x, pb.z}, py[4] = {pa.y, pa.w, pb.y, pb.w};
  const double ha = C.half_w[large ? 1 : 0], hb = C.half_h[large ? 1 : 0];
  double r[3] = {rvec[(size_t)i * 3], rvec[(size_t)i * 3 + 1], rvec[(size_t)i * 3 + 2]};
  double t[3] = {tvec[(size_t)i * 3], tvec[(size_t)i * 3 + 1], tvec[(size_t)i * 3 + 2]};
  if (!(isfinite(r[0]) && isfinite(r[1]) && isfinite(r[2]) && isfinite(t[0]) && isfinite(t[1]) && isfinite(t[2]))) return;
  double R[3][3];
  rodrigues(r, R);
  double A[6][6], g[6];
  double lambda = 1e-3;
  double cost = lm_eval(C, R, t, ha, hb, px, py, true, A, g);
  for (int it = 0; it < max_iters; ++it) {
    // (JtJ + lambda diag) d = -Jtf, Cholesky
    double L[6][6], d[6];
    bool spd = true;
#pragma unroll
    for (int c = 0; c < 6; ++c) {
      double s = A[c][c] * (1.0 + lambda);
#pragma unroll
      for (int k = 0; k < c; ++k) s -= L[c][k] * L[c][k];
      if (!(s > 0.0)) spd = false;
      const double lc = sqrt(fmax(s, 1e-300));
      L[c][c] = lc;
#pragma unroll
      for (int rr = c + 1; rr < 6; ++rr) {
        double v = A[c][rr];
#pragma unroll
        for (int k = 0; k < c; ++k) v -= L[rr][k] * L[c][k];
        L[rr][c] = v / lc;
      }
    }
#pragma unroll
    for (int c = 0; c < 6; ++c) {              // forward: L y = -g
      double v = -g[c];
#pragma unroll
      for (int k = 0; k < c; ++k) v -= L[c][k] * d[k];
      d[c] = v / L[c][c];
    }
#pragma unroll
    for (int c = 5; c >= 0; --c) {             // backward: L^T d = y
      double v = d[c];
#pragma unroll
      for (int k = c + 1; k < 6; ++k) v -= L[k][c] * d[k];
      d[c] = v / L[c][c];
    }
    double dR[3][3], Rn[3][3], tn[3] = {t[0] + d[3], t[1] + d[4], t[2] + d[5]};
    const double dw[3] = {d[0], d[1], d[2]};
    rodrigues(dw, dR);
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
      for (int b = 0; b < 3; ++b) Rn[a][b] = dR[a][0] * R[0][b] + dR[a][1] * R[1][b] + dR[a][2] * R[2][b];
    double An[6][6], gn[6];
    const double cn = spd ? lm_eval(C, Rn, tn, ha, hb, px, py, true, An, gn) : cost;
    const double step2 = d[0] * d[0] + d[1] * d[1] + d[2] * d[2] + d[3] * d[3] + d[4] * d[4] + d[5] * d[5];
    if (spd && cn < cost) {                    // accept
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        t[a] = tn[a];
#pragma unroll
        for (int b = 0; b < 3; ++b) R[a][b] = Rn[a][b];
      }
#pragma unroll
      for (int a = 0; a < 6; ++a) {
        g[a] = gn[a];
#pragma unroll
        for (int b = 0; b < 6; ++b) A[a][b] = An[a][b];
      }
      const double rel = (cost - cn) / fmax(cost, 1e-300);
      cost = cn;
      lambda = fmax(lambda * 0.1, 1e-12);
      if (step2 < 1e-24 || rel < 1e-14) break;
    } else {
      lambda = fmin(lambda * 10.0, 1e12);
      if (step2 < 1e-24) break;
    }
  }
  rot2vec(R, r);
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    rvec[(size_t)i * 3 + k] = r[k];
    tvec[(size_t)i * 3 + k] = t[k];
  }
  if (quat) {
    double qv[4];
    rot2quat(R, qv);
#pragma unroll
    for (int k = 0; k < 4; ++k) quat[(size_t)i * 4 + k] = qv[k];
  }
}

}  // namespace

cudaError_t launch_pnp(const PnpConsts &c, const float *pts, int n, int large, PnpOut out,
                       cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  int blocks = (n + 127) / 128;
  pnp_kernel<<<blocks, 128, 0, s>>>(c, pts, n, large, out);
  return cudaGetLastError();
}

}  // namespace irmv

namespace irmv {
cudaError_t launch_pnp_refine_lm(const PnpConsts &c, const float *pts, int n, int large, int max_iters, double *rvec,
                                 double *tvec, double *quat, cudaStream_t s) {
  if (n <= 0 || max_iters <= 0) return cudaSuccess;
  pnp_refine_kernel<<<(n + 63) / 64, 64, 0, s>>>(c, pts, n, large, max_iters, rvec, tvec, quat);
  return cudaGetLastError();
}
}  // namespace irmv
