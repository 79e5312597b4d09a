// csrc/ekf_math.cuh — per-thread fp64 math of the EKF path (SURVEY.md §8(a) a3-a9), written so the
// order of operations inside every expression is the reference's (files are compiled with
// --fmad=false, so nothing here is contracted into FMAs).  Citations: V: = vslamRansac.cpp,
// C: = camModel.cpp.
#pragma once
#include "ekf_common.cuh"

// V:1408-1421 — R(q), w-first, un-normalised form.  R row-major 3x3.
__device__ __forceinline__ void d_quat2rot(const double q[4], double R[9]) {
  const double qr = q[0], qi = q[1], qj = q[2], qk = q[3];
  R[0] = qr * qr + qi * qi - qj * qj - qk * qk; R[1] = -2 * qr * qk + 2 * qi * qj; R[2] = 2 * qr * qj + 2 * qi * qk;
  R[3] = 2 * qr * qk + 2 * qi * qj; R[4] = qr * qr - qi * qi + qj * qj - qk * qk; R[5] = -2 * qr * qi + 2 * qj * qk;
  R[6] = -2 * qr * qj + 2 * qi * qk; R[7] = 2 * qr * qi + 2 * qj * qk; R[8] = qr * qr - qi * qi - qj * qj + qk * qk;
}
// V:1388-1400
__device__ __forceinline__ void d_vec2quat(const double v[3], double q[4]) {
  const double alpha = sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
  if (alpha != 0) {
    q[0] = cos(alpha / 2);
    const double s = sin(alpha / 2);
    for (int i = 0; i < 3; ++i) q[1 + i] = v[i] * s / alpha;
  } else {
    q[0] = 1; q[1] = 0; q[2] = 0; q[3] = 0;
  }
}
// V:1423-1438 (Y) and V:1441-1455 (Ybar), row-major 4x4
__device__ __forceinline__ void d_yupsilon(const double q[4], double Y[16]) {
  const double r1 = q[0], x1 = q[1], y1 = q[2], z1 = q[3];
  Y[0] = r1; Y[1] = -x1; Y[2] = -y1; Y[3] = -z1;
  Y[4] = x1; Y[5] = r1; Y[6] = -z1; Y[7] = y1;
  Y[8] = y1; Y[9] = z1; Y[10] = r1; Y[11] = -x1;
  Y[12] = z1; Y[13] = -y1; Y[14] = x1; Y[15] = r1;
}
__device__ __forceinline__ void d_yupsilon_c(const double q[4], double Y[16]) {
  const double r1 = q[0], x1 = q[1], y1 = q[2], z1 = q[3];
  Y[0] = r1; Y[1] = -x1; Y[2] = -y1; Y[3] = -z1;
  Y[4] = x1; Y[5] = r1; Y[6] = z1; Y[7] = -y1;
  Y[8] = y1; Y[9] = -z1; Y[10] = r1; Y[11] = x1;
  Y[12] = z1; Y[13] = y1; Y[14] = -x1; Y[15] = r1;
}
// V:1457-1460
__device__ __forceinline__ void d_quat_mul(const double a[4], const double b[4], double o[4]) {
  double Y[16];
  d_yupsilon(a, Y);
  for (int i = 0; i < 4; ++i) {
    double s = 0;
    for (int k = 0; k < 4; ++k) s += Y[i * 4 + k] * b[k];
    o[i] = s;
  }
}
// V:1492-1535 — F (13x13 row-major) = d g / d x at mu13 with w + ctrl (SURVEY §8(a) a3).
__device__ inline void d_system_jacobian(const double* mu13, double dT, const double ctrl[3], double F[169]) {
  for (int i = 0; i < 169; ++i) F[i] = 0;
  for (int i = 0; i < 13; ++i) F[i * 13 + i] = 1;
  const double* q = mu13 + 3;
  double wc[3], wdt[3], hq[4];
  for (int i = 0; i < 3; ++i) { wc[i] = mu13[10 + i] + ctrl[i]; wdt[i] = dT * wc[i]; }
  d_vec2quat(wdt, hq);
  double Yc[16];
  d_yupsilon_c(hq, Yc);
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 4; ++j) F[(3 + i) * 13 + 3 + j] = Yc[i * 4 + j];
  // Jacobian_qt_w(q, wc, dT) = Y(q) * t2
  const double n = sqrt(wc[0] * wc[0] + wc[1] * wc[1] + wc[2] * wc[2]);
  const double s = sin(dT * n / 2);
  const double c = cos(dT * n / 2);
  const double Sinc = (n == 0 ? 1.0 : 2 * sin(dT * n / 2) / (dT * n));
  double nw[3] = {0, 0, 0};  // reference leaves n_w uninitialised when n == 0 (V:1523); 0 here
  if (n > 0) for (int i = 0; i < 3; ++i) nw[i] = wc[i] / n;
  double t2[12];
  const double a0 = -dT * 0.5 * s;
  for (int j = 0; j < 3; ++j) t2[j] = a0 * nw[j];
  const double a1 = dT * 0.5;
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) t2[(1 + i) * 3 + j] = a1 * (Sinc * (i == j ? 1.0 : 0.0) + ((c - Sinc) * nw[i]) * nw[j]);
  double Y[16];
  d_yupsilon(q, Y);
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 3; ++j) {
      double acc = 0;
      for (int k = 0; k < 4; ++k) acc += Y[i * 4 + k] * t2[k * 3 + j];
      F[(3 + i) * 13 + 10 + j] = acc;
    }
  for (int i = 0; i < 3; ++i) F[i * 13 + 7 + i] = dT * 1.0;
}
// V:1575-1589
__device__ inline void d_predict_state(double* X, const double dv[3], const double dw[3], double dT) {
  double v[3], w[3], wdt[3], hq[4], qn[4];
  for (int i = 0; i < 3; ++i) { v[i] = X[7 + i] + dv[i]; w[i] = X[10 + i] + dw[i]; }
  for (int i = 0; i < 3; ++i) X[i] += dT * v[i];
  for (int i = 0; i < 3; ++i) wdt[i] = dT * w[i];
  d_vec2quat(wdt, hq);
  d_quat_mul(X + 3, hq, qn);
  for (int i = 0; i < 4; ++i) X[3 + i] = qn[i];
  for (int i = 0; i < 3; ++i) { X[7 + i] = v[i]; X[10 + i] = w[i]; }
}
// C:18-47 — 2x2 distortion Jacobian, row-major
__device__ __forceinline__ void d_diff_distort(const CamParams& cm, double hx, double hy, double J[4]) {
  const double r_2 = hx * hx + hy * hy;
  const double Lrn = 1 + cm.k1 * r_2 + cm.k2 * r_2 * r_2 + cm.k3 * r_2 * r_2 * r_2;
  const double f = cm.k1 + 2 * cm.k2 * r_2 + 3 * cm.k3 * r_2 * r_2;
  const double hn[2] = {hx, hy}, hc[2] = {hy, hx}, pv[2] = {cm.p1, cm.p2}, pc[2] = {cm.p2, cm.p1};
  const double jm[4] = {cm.p2 * hx, 0.0, 0.0, cm.p1 * hy};
  for (int a = 0; a < 2; ++a)
    for (int b = 0; b < 2; ++b) {
      double v = Lrn * (a == b ? 1.0 : 0.0);
      v = v + ((2 * f) * hn[a]) * hn[b];
      v = v + (2 * pv[a]) * hc[b];
      v = v + (2 * pc[a]) * hn[b];
      v = v + 4 * jm[a * 2 + b];
      J[a * 2 + b] = v;
    }
}
// C:113-138
__device__ __forceinline__ void d_cam_project(const CamParams& cm, const double h[3], double hd[2]) {
  const double x = h[0], y = h[1], z = h[2];
  const double x1 = x / z, y1 = y / z;
  const double r_2 = x1 * x1 + y1 * y1;
  const double l = 1 + cm.k1 * r_2 + cm.k2 * r_2 * r_2 + cm.k3 * r_2 * r_2 * r_2;
  const double x2 = x1 * l + 2 * cm.p1 * x1 * y1 + cm.p2 * (r_2 + 2 * x1 * x1);
  const double y2 = y1 * l + 2 * cm.p2 * x1 * y1 + cm.p1 * (r_2 + 2 * y1 * y1);
  hd[0] = cm.fx * x2 + cm.u0;
  hd[1] = cm.fy * y2 + cm.v0;
}
// C:68-111 — J is 2x3 row-major = (K * D) * Jn
__device__ __forceinline__ void d_cam_project_J(const CamParams& cm, const double h[3], double hd[2], double J[6]) {
  const double x = h[0], y = h[1], z = h[2];
  d_cam_project(cm, h, hd);
  const double x1 = x / z, y1 = y / z;
  double Jn[6];
  Jn[0] = 1 / z; Jn[1] = 0; Jn[2] = -x / z / z;
  Jn[3] = 0; Jn[4] = 1 / z; Jn[5] = -y / z / z;
  double D[4], KD[4];
  d_diff_distort(cm, x1, y1, D);
  const double Kp[4] = {cm.fx, 0.0, 0.0, cm.fy};
  for (int a = 0; a < 2; ++a)
    for (int b = 0; b < 2; ++b) {
      double s = 0;
      for (int k = 0; k < 2; ++k) s += Kp[a * 2 + k] * D[k * 2 + b];
      KD[a * 2 + b] = s;
    }
  for (int a = 0; a < 2; ++a)
    for (int b = 0; b < 3; ++b) {
      double s = 0;
      for (int k = 0; k < 2; ++k) s += KD[a * 2 + k] * Jn[k * 3 + b];
      J[a * 3 + b] = s;
    }
}
// C:140-192 — hC = (x1, y1, 1), J 3x2 row-major = (U * inv(D)) * diag(1/fx, 1/fy)
__device__ inline void d_cam_unproject_J(const CamParams& cm, const double hd[2], double hC[3], double J[6]) {
  const double x2 = (hd[0] - cm.u0) / cm.fx;
  const double y2 = (hd[1] - cm.v0) / cm.fy;
  double x1 = x2, y1 = y2;
  for (int i = 0; i < 50; ++i) {
    const double r_2 = x1 * x1 + y1 * y1;
    const double l = 1 + cm.k1 * r_2 + cm.k2 * r_2 * r_2 + cm.k3 * r_2 * r_2 * r_2;
    const double dx = 2 * cm.p1 * x1 * y1 + cm.p2 * (r_2 + 2 * x1 * x1);
    const double dy = 2 * cm.p2 * x1 * y1 + cm.p1 * (r_2 + 2 * y1 * y1);
    x1 = (x2 - dx) / l;
    y1 = (y2 - dy) / l;
  }
  hC[0] = x1; hC[1] = y1; hC[2] = 1;
  double D[4], Di[4];
  d_diff_distort(cm, x1, y1, D);
  const double det = D[0] * D[3] - D[2] * D[1];
  const double invdet = 1.0 / det;
  Di[0] = D[3] * invdet; Di[2] = -D[2] * invdet; Di[1] = -D[1] * invdet; Di[3] = D[0] * invdet;
  // U = [1 0; 0 1; 0 0]; (U*Di) rows 0,1 = Di (sums with exact zeros), row 2 = 0
  const double Jp[4] = {1 / cm.fx, 0.0, 0.0, 1 / cm.fy};
  for (int a = 0; a < 3; ++a)
    for (int b = 0; b < 2; ++b) {
      double s = 0;
      for (int k = 0; k < 2; ++k) {
        const double ud = (a < 2) ? Di[a * 2 + k] : 0.0;
        s += ud * Jp[k * 2 + b];
      }
      J[a * 2 + b] = s;
    }
}
// V:1537-1566 + V:1654-1661 — d(R(q) d)/dq, 3x4 row-major
__device__ inline void d_jac_hW_q(const double q[4], const double d[3], double J[12]) {
  const double q0 = 2 * q[0], qx = 2 * q[1], qy = 2 * q[2], qz = 2 * q[3];
  const double dR[4][9] = {
      {q0, -qz, qy, qz, q0, -qx, -qy, qx, q0},
      {qx, qy, qz, qy, -qx, -q0, qz, q0, -qx},
      {-qy, qx, q0, qx, qy, qz, -q0, qz, -qy},
      {-qz, -q0, qx, q0, -qz, qy, qx, qy, qz}};
  for (int j = 0; j < 4; ++j)
    for (int i = 0; i < 3; ++i) {
      double s = 0;
      for (int k = 0; k < 3; ++k) s += dR[j][i * 3 + k] * d[k];
      J[i * 4 + j] = s;
    }
}
// V:1462-1489 — d = rho (x - r) + m(theta, phi); optional J (3x6 row-major)
__device__ inline void d_inverse2xyz(const double f[6], const double r[3], double d[3], double* J) {
  const double theta = f[3], phi = f[4], ro = f[5];
  double st, ct, sp, cp;
  st = sin(theta); ct = cos(theta); sp = sin(phi); cp = cos(phi);
  const double m[3] = {st * cp, -sp, ct * cp};
  if (J) {
    for (int i = 0; i < 18; ++i) J[i] = 0;
    for (int i = 0; i < 3; ++i) J[i * 6 + i] = ro * 1.0;
    J[0 * 6 + 3] = ct * cp; J[1 * 6 + 3] = 0; J[2 * 6 + 3] = -st * cp;
    J[0 * 6 + 4] = -st * sp; J[1 * 6 + 4] = -cp; J[2 * 6 + 4] = -ct * sp;
    for (int i = 0; i < 3; ++i) J[i * 6 + 5] = f[i] - r[i];
  }
  for (int i = 0; i < 3; ++i) d[i] = ro * (f[i] - r[i]) + m[i];
}
// V:508-578 / V:1080-1112 — h and compact H (2 x 13) of one feature.
//   fs: feature state (6 inverse depth / 3 XYZ), r: camera position, qc: conj(q), Rcw = R(qc).
// Compact columns: [0,3) d/dr, [3,7) d/dq, [7,13) d/dfeature (XYZ: [7,10), rest 0).
__device__ inline void d_feature_hH(const CamParams& cm, const double* fs, int coding, const double r[3],
                                    const double qc[4], const double Rcw[9], double hi[2], double Hc[26],
                                    double* hCz) {
  double d[3], hC[3], Jh[6], Jf[18];
  if (!coding) d_inverse2xyz(fs, r, d, Jf);
  else for (int i = 0; i < 3; ++i) d[i] = fs[i] - r[i];
  for (int i = 0; i < 3; ++i) {
    double s = 0;
    for (int k = 0; k < 3; ++k) s += Rcw[i * 3 + k] * d[k];
    hC[i] = s;
  }
  d_cam_project_J(cm, hC, hi, Jh);
  *hCz = hC[2];
  double Jq[12];
  d_jac_hW_q(qc, d, Jq);
  // * d_qbar_q() = diag(1,-1,-1,-1): column sign flips (exact; the reference sums x*1 and x*0 terms)
  for (int i = 0; i < 3; ++i) { Jq[i * 4 + 1] = -Jq[i * 4 + 1]; Jq[i * 4 + 2] = -Jq[i * 4 + 2]; Jq[i * 4 + 3] = -Jq[i * 4 + 3]; }
  for (int i = 0; i < 26; ++i) Hc[i] = 0;
  // JR = Jh * Rcw (2x3), with the leading scalar applied to Jh first where the reference does
  const double sc = coding ? -1.0 : -fs[5];
  double JRs[6], JR[6];
  for (int a = 0; a < 2; ++a)
    for (int b = 0; b < 3; ++b) {
      double s0 = 0, s1 = 0;
      for (int k = 0; k < 3; ++k) { s0 += (sc * Jh[a * 3 + k]) * Rcw[k * 3 + b]; s1 += Jh[a * 3 + k] * Rcw[k * 3 + b]; }
      JRs[a * 3 + b] = s0; JR[a * 3 + b] = s1;
    }
  for (int a = 0; a < 2; ++a) {
    // XYZ: Hit.middleCols<3>(0) = -J*R is -(J*R) (unary minus on the product, V:568)
    for (int b = 0; b < 3; ++b) Hc[a * 13 + b] = coding ? -JR[a * 3 + b] : JRs[a * 3 + b];
    for (int b = 0; b < 4; ++b) {
      double s = 0;
      for (int k = 0; k < 3; ++k) s += Jh[a * 3 + k] * Jq[k * 4 + b];
      Hc[a * 13 + 3 + b] = s;
    }
    if (!coding) {
      for (int b = 0; b < 6; ++b) {
        double s = 0;
        for (int k = 0; k < 3; ++k) s += JR[a * 3 + k] * Jf[k * 6 + b];
        Hc[a * 13 + 7 + b] = s;
      }
    } else {
      for (int b = 0; b < 3; ++b) Hc[a * 13 + 7 + b] = JR[a * 3 + b];
    }
  }
}
// Reprojection without Jacobian (RANSAC consensus test, V:1010-1020).
__device__ inline void d_feature_h(const CamParams& cm, const double* fs, int coding, const double r[3],
                                   const double Rcw[9], double hi[2]) {
  double d[3], hC[3];
  if (!coding) d_inverse2xyz(fs, r, d, nullptr);
  else for (int i = 0; i < 3; ++i) d[i] = fs[i] - r[i];
  for (int i = 0; i < 3; ++i) {
    double s = 0;
    for (int k = 0; k < 3; ++k) s += Rcw[i * 3 + k] * d[k];
    hC[i] = s;
  }
  d_cam_project(cm, hC, hi);
}
// V:1599-1623 — rows 3 (theta) and 4 (phi) of the 6x3 d f / d hW; the other rows are zero.
__device__ inline void d_jac_f_hW(const double hW[3], double Jt[3], double Jp[3]) {
  const double hx = hW[0], hy = hW[1], hz = hW[2];
  const double normal = hx * hx + hz * hz;
  const double normal2 = hx * hx + hy * hy + hz * hz;
  Jt[0] = hz / normal; Jt[1] = 0; Jt[2] = -hx / normal;
  Jp[0] = hx * hy / sqrt(normal) / normal2;
  Jp[1] = -sqrt(normal) / normal2;
  Jp[2] = hz * hy / sqrt(normal) / normal2;
}
// Dynamic 2x2 inverse() = partial-pivot LU solve against I (see oracle inverse_pplu; V:995, P:223)
__host__ __device__ __forceinline__ void d_inv2_pplu(const double A[4], double X[4]) {
  double a00 = A[0], a01 = A[1], a10 = A[2], a11 = A[3];
  int swapped = 0;
  if (fabs(a10) > fabs(a00)) {
    double t = a00; a00 = a10; a10 = t;
    t = a01; a01 = a11; a11 = t;
    swapped = 1;
  }
  const double l = a10 / a00;
  const double u11 = a11 - l * a01;
  // rows of P*I: row0 = e_{perm0}, row1 = e_{perm1}
  double x0[2], x1[2];
  x0[0] = swapped ? 0.0 : 1.0; x0[1] = swapped ? 1.0 : 0.0;
  x1[0] = swapped ? 1.0 : 0.0; x1[1] = swapped ? 0.0 : 1.0;
  for (int j = 0; j < 2; ++j) if (l != 0.0) x1[j] -= l * x0[j];
  for (int j = 0; j < 2; ++j) x1[j] = x1[j] / u11;
  for (int j = 0; j < 2; ++j) { x0[j] -= a01 * x1[j]; x0[j] = x0[j] / a00; }
  X[0] = x0[0]; X[1] = x0[1]; X[2] = x1[0]; X[3] = x1[1];
}

// ---- addFeature (V:309-371) ---------------------------------------------------------------------------------------------
// Shared by the single filter (k_add_feature) and the batched filters (k_batch_add).  New state entries and the 6 new rows /
// columns of Sigma' = Js blkdiag(Sigma, sigma_px^2 I2, sigma_rho_0) Js^T, evaluated in the reference's association
// (Js*S)*Js^T with the exact-zero terms dropped (SURVEY.md §3.2):
//   rows  n+a, j<n : sum_{c<7} A[a,c] Sigma[c,j]          cols i<n, n+b : sum_{c<7} Sigma[i,c] A[b,c]
//   corner         : sum_{c<7} T[a,c] A[b,c] + sum_e (Ap[a,e] s_e) Ap[b,e]
// A = [I3 0 ; Jf*Jq (rows theta,phi) ; 0], Ap = [Jf*R*J2d | e6].
//
// A (6 x 7), Ap (6 x 3) and the new state entries fnew[6] from the camera r, q = mu[0:7] and the pixel.
__device__ inline void add_feature_jacobians(const CamParams& cam, const double* mu, float pfx, float pfy, double rho_0, double* A,
                                             double* Ap, double* fnew) {
  double r[3] = {mu[0], mu[1], mu[2]}, q[4] = {mu[3], mu[4], mu[5], mu[6]};
  const double hd[2] = {(double)pfx, (double)pfy};
  double hC[3], J2d[6], Rot[9], hW[3];
  d_cam_unproject_J(cam, hd, hC, J2d);
  d_quat2rot(q, Rot);
  for (int i = 0; i < 3; ++i) {
    double s = 0;
    for (int k = 0; k < 3; ++k) s += Rot[i * 3 + k] * hC[k];
    hW[i] = s;
  }
  const double hx = hW[0], hy = hW[1], hz = hW[2];
  fnew[0] = r[0]; fnew[1] = r[1]; fnew[2] = r[2];
  fnew[3] = atan2(hx, hz);
  fnew[4] = atan2(-hy, sqrt(hx * hx + hz * hz));
  fnew[5] = rho_0;
  double Jt[3], Jp[3], Jq[12];
  d_jac_f_hW(hW, Jt, Jp);
  d_jac_hW_q(q, hC, Jq);
  for (int i = 0; i < 42; ++i) A[i] = 0;
  for (int i = 0; i < 18; ++i) Ap[i] = 0;
  for (int i = 0; i < 3; ++i) A[i * 7 + i] = 1;
  // (Jf*Jq): rows 3,4 = Jt*Jq, Jp*Jq (other rows are sums of exact zeros)
  for (int b = 0; b < 4; ++b) {
    double s3 = 0, s4 = 0;
    for (int k = 0; k < 3; ++k) { s3 += Jt[k] * Jq[k * 4 + b]; s4 += Jp[k] * Jq[k * 4 + b]; }
    A[3 * 7 + 3 + b] = s3; A[4 * 7 + 3 + b] = s4;
  }
  // (Jf*Rot)*J2d
  double JR3[3], JR4[3];
  for (int b = 0; b < 3; ++b) {
    double s3 = 0, s4 = 0;
    for (int k = 0; k < 3; ++k) { s3 += Jt[k] * Rot[k * 3 + b]; s4 += Jp[k] * Rot[k * 3 + b]; }
    JR3[b] = s3; JR4[b] = s4;
  }
  for (int b = 0; b < 2; ++b) {
    double s3 = 0, s4 = 0;
    for (int k = 0; k < 3; ++k) { s3 += JR3[k] * J2d[k * 2 + b]; s4 += JR4[k] * J2d[k * 2 + b]; }
    Ap[3 * 3 + b] = s3; Ap[4 * 3 + b] = s4;
  }
  Ap[5 * 3 + 2] = 1;
}
// New row n + a, column t and new column n + a, row t of an n x n Sigma (t < n), for a = 0..5.
__device__ inline void add_feature_cross(double* Sigma, int ld, int n, int t, const double* A) {
  double col[7], rowv[7];
  for (int c = 0; c < 7; ++c) { col[c] = Sigma[(size_t)c * ld + t]; rowv[c] = Sigma[(size_t)t * ld + c]; }
  for (int a = 0; a < 6; ++a) {
    double s = 0, u = 0;
    for (int c = 0; c < 7; ++c) { s += A[a * 7 + c] * col[c]; u += rowv[c] * A[a * 7 + c]; }
    Sigma[(size_t)(n + a) * ld + t] = s;
    Sigma[(size_t)t * ld + n + a] = u;
  }
}
// Entry e = 7 a + c of T = A Sigma[0:7, 0:7] (6 x 7), the left factor of the 6 x 6 corner.
__device__ inline double add_feature_corner_T(const double* Sigma, int ld, const double* A, int e) {
  const int a = e / 7, c = e % 7;
  double s = 0;
  for (int k = 0; k < 7; ++k) s += A[a * 7 + k] * Sigma[(size_t)k * ld + c];
  return s;
}
// Entry e = 6 a + b of the 6 x 6 corner Sigma'[n + a, n + b].
__device__ inline double add_feature_corner(const double* T, const double* A, const double* Ap, int e, double sigma_pixel_2,
                                            double sigma_rho_0) {
  const int a = e / 6, b = e % 6;
  double s = 0;
  for (int c = 0; c < 7; ++c) s += T[a * 7 + c] * A[b * 7 + c];
  for (int k = 0; k < 3; ++k) {
    const double sd = (k < 2) ? sigma_pixel_2 : sigma_rho_0;  // V:362,365
    s += (Ap[a * 3 + k] * sd) * Ap[b * 3 + k];
  }
  return s;
}
// Template byte e of the Patch constructor (Patch.cpp:78-103): the frame ROI at (int)(pf - w/2).
__device__ __forceinline__ uint8_t add_feature_template_px(const FrameView& fr, int w, float pfx, float pfy, int e) {
  const int x0 = (int)(pfx - w / 2), y0 = (int)(pfy - w / 2);
  return fr.px[(size_t)(y0 + e / w) * fr.stride + x0 + (e % w)];
}
// Feature-table record fidx of a new inverse-depth feature at state position n.
__device__ inline void add_feature_record(const FeatTab& ft, int fidx, int n, float pfx, float pfy, int real_index) {
  ft.pos[fidx] = n; ft.coding[fidx] = 0; ft.innov[fidx] = 0; ft.li[fidx] = 0; ft.hi[fidx] = 0;
  ft.removef[fidx] = 0; ft.n_tot[fidx] = 1; ft.n_find[fidx] = 1; ft.real_index[fidx] = real_index;
  ft.pos_in_z[fidx] = 0; ft.center[2 * fidx] = pfx; ft.center[2 * fidx + 1] = pfy;
  ft.quality[fidx] = 0.0f; ft.last_ncc[fidx] = -1.0f;
  ft.z[2 * fidx] = 0; ft.z[2 * fidx + 1] = 0; ft.h[2 * fidx] = 0; ft.h[2 * fidx + 1] = 0;
  for (int c = 0; c < 26; ++c) ft.Hc[26 * fidx + c] = 0;
  for (int c = 0; c < 4; ++c) ft.S2[4 * fidx + c] = 0;
}

// ---- convert2XYZ_ifLinear (V:741-772) -----------------------------------------------------------------------------------
// Shared by the single filter (k_xyz_decide / k_xyz_apply), the batched filters (ekf_batch.cu) and a host test harness.
//
// Linearity test of inverseDepth2XyzWorld (V:690-738) for the inverse-depth feature f[6] seen from the camera position r[3];
// sigma_rho is Sigma(pos + 5, pos + 5).  Returns 1 if the feature converts and then writes its XYZ point y[3] and the 3 x 6
// Jacobian J (row-major); otherwise writes nothing.  QUIRKS kept: the rho VARIANCE is used as a sigma (V:717); bare
// abs(float) (V:719) is fabs unless abs_int_quirk.
__host__ __device__ inline int xyz_linear_decide(const double* f, const double* r, double sigma_rho, double threshold,
                                                 int abs_int_quirk, double* y, double* J) {
  const double theta = f[3], phi = f[4], ro = f[5];
  double m[3], yy[3], d[3];
  m[0] = sin(theta) * cos(phi);
  m[1] = -sin(phi);
  m[2] = cos(theta) * cos(phi);
  for (int c = 0; c < 3; ++c) yy[c] = f[c] + m[c] / ro;
  for (int c = 0; c < 3; ++c) d[c] = yy[c] - r[c];
  double t = 0;
  for (int c = 0; c < 3; ++c) t += d[c] * m[c];
  const double at = abs_int_quirk ? (double)abs((int)t) : fabs(t);
  const double L_d = 4 * sigma_rho * at / (ro * ro * (d[0] * d[0] + d[1] * d[1] + d[2] * d[2]));
  if (!(L_d < threshold)) return 0;
  for (int c = 0; c < 18; ++c) J[c] = 0;
  for (int c = 0; c < 3; ++c) J[c * 6 + c] = 1;
  J[0 * 6 + 3] = cos(theta) * cos(phi) / ro;
  J[1 * 6 + 3] = 0;
  J[2 * 6 + 3] = -sin(theta) * cos(phi) / ro;
  J[0 * 6 + 4] = -sin(theta) * sin(phi) / ro;
  J[1 * 6 + 4] = -cos(phi) / ro;
  J[2 * 6 + 4] = -cos(theta) * sin(phi) / ro;
  for (int c = 0; c < 3; ++c) J[c * 6 + 5] = -m[c] / (ro * ro);
  for (int c = 0; c < 3; ++c) y[c] = yy[c];
  return 1;
}

// Entry (i, j) of Sigma' = J Sigma J^T for any number of conversions at once, in the reference's association (one
// conversion after the other): the sum over the EARLIER-converted feature's six entries is the inner one.  ri / rj are the
// row-map entries of i and j, (src, code): code < 0 is the plain state entry src; code = 4 f + x is row x of converted
// feature f, whose old 6-entry block starts at src and whose Jacobian is Jall[18 f .. 18 f + 17].  Features keep their
// relative order in the map, so "earlier" is the smaller f.
__host__ __device__ inline double xyz_apply_entry(const double* src, int ld, int2 ri, int2 rj, const double* Jall) {
  if (ri.y < 0 && rj.y < 0) return src[(size_t)ri.x * ld + rj.x];
  double v = 0;
  if (ri.y >= 0 && rj.y < 0) {                // (J Sigma)[i, j]
    const double* Jr = Jall + 18 * (ri.y >> 2) + 6 * (ri.y & 3);
    for (int a = 0; a < 6; ++a) v += Jr[a] * src[(size_t)(ri.x + a) * ld + rj.x];
  } else if (ri.y < 0) {                      // (Sigma J^T)[i, j]
    const double* Jc = Jall + 18 * (rj.y >> 2) + 6 * (rj.y & 3);
    for (int b = 0; b < 6; ++b) v += src[(size_t)ri.x * ld + rj.x + b] * Jc[b];
  } else {
    const double* Jr = Jall + 18 * (ri.y >> 2) + 6 * (ri.y & 3);
    const double* Jc = Jall + 18 * (rj.y >> 2) + 6 * (rj.y & 3);
    if ((ri.y >> 2) <= (rj.y >> 2)) {         // row feature converted first (or diagonal block): (J_r Sigma) J_c^T
      for (int b = 0; b < 6; ++b) {
        double t = 0;
        for (int a = 0; a < 6; ++a) t += Jr[a] * src[(size_t)(ri.x + a) * ld + rj.x + b];
        v += t * Jc[b];
      }
    } else {                                  // column feature converted first: J_r (Sigma J_c^T)
      for (int a = 0; a < 6; ++a) {
        double t = 0;
        for (int b = 0; b < 6; ++b) t += src[(size_t)(ri.x + a) * ld + rj.x + b] * Jc[b];
        v += Jr[a] * t;
      }
    }
  }
  return v;
}
