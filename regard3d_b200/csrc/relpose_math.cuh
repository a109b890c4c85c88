// relpose_math.cuh -- the per-pair and per-inlier arithmetic of robustRelativePose after AC-RANSAC (SURVEY.md A.9):
// E from the scored F, MotionFromEssential (SVD of E, the four (R, t) candidates), TriangulateDLT (4x4 homogeneous
// nullspace), the cheirality depths and the triangulation angle of AutomaticInitialPairChoice.  Host and device; every translation
// unit that includes it is compiled without FMA contraction (relpose.cu is in NO_FMAD), so each value is a pure
// function of its inputs and equals the oracle's restatement (oracle/oracle_relpose.cpp) bit for bit.
//
// Eigen's JacobiSVD is replaced by one-sided (Hestenes) Jacobi with a fixed cyclic pair order and a fixed
// orthogonality test: deterministic, built from + - * / sqrt only, and accurate to rounding level on the column space
// (no normal-equation squaring).  E is defined up to sign and scale, and the nullspace of the DLT system up to sign and
// scale, so neither convention changes the candidate set, the triangulated points or the chosen pose (DESIGN.md sec. 2).
#pragma once
#include "detmath.cuh"

namespace r3d {
namespace rp {

constexpr int kMaxSweeps = 12;

// One Jacobi rotation of columns p < q of a (ROWS x COLS, row-major) and of the accumulated v (COLS x COLS): makes the
// two columns orthogonal.  Returns false (and leaves both untouched) when they already are, to |cos| <= 1e-15.
template <int ROWS, int COLS>
R3D_HD bool hestenes_rotate(double* a, double* v, int p, int q) {
  double alpha = 0.0, beta = 0.0, gamma = 0.0;
  for (int r = 0; r < ROWS; ++r) {
    const double ap = a[r * COLS + p], aq = a[r * COLS + q];
    alpha = alpha + ap * ap;
    beta = beta + aq * aq;
    gamma = gamma + ap * aq;
  }
  if (!(gamma * gamma > 1e-30 * (alpha * beta))) return false;  // also stops on NaN
  const double zeta = (beta - alpha) / (2.0 * gamma);
  const double az = zeta < 0.0 ? -zeta : zeta;
  double t = 1.0 / (az + sqrt(1.0 + zeta * zeta));
  if (zeta < 0.0) t = -t;
  const double c = 1.0 / sqrt(1.0 + t * t);
  const double s = c * t;
  for (int r = 0; r < ROWS; ++r) {
    const double ap = a[r * COLS + p], aq = a[r * COLS + q];
    a[r * COLS + p] = c * ap - s * aq;
    a[r * COLS + q] = s * ap + c * aq;
  }
  for (int r = 0; r < COLS; ++r) {
    const double vp = v[r * COLS + p], vq = v[r * COLS + q];
    v[r * COLS + p] = c * vp - s * vq;
    v[r * COLS + q] = s * vp + c * vq;
  }
  return true;
}

// cyclic sweeps (0,1), (0,2), ..., (N-2,N-1) until a sweep rotates nothing; v starts as the identity
template <int ROWS, int COLS>
R3D_HD void hestenes(double* a, double* v) {
  for (int i = 0; i < COLS * COLS; ++i) v[i] = (i % (COLS + 1) == 0) ? 1.0 : 0.0;
  for (int sweep = 0; sweep < kMaxSweeps; ++sweep) {
    bool rotated = false;
    for (int p = 0; p < COLS - 1; ++p)
      for (int q = p + 1; q < COLS; ++q) rotated = hestenes_rotate<ROWS, COLS>(a, v, p, q) || rotated;
    if (!rotated) break;
  }
}

R3D_HD double col_norm2_3(const double* a, int c) {
  return (a[c] * a[c] + a[3 + c] * a[3 + c]) + a[6 + c] * a[6 + c];
}

// E = K2^T F K1 of the F that AC-RANSAC scored (F = K2^-T E K1^-1 of the winning 5-point model): that E up to rounding
R3D_HD void essential_from_fundamental(const double* F, const double* K1, const double* K2, double* E) {
  const double k1[9] = {K1[0], 0.0, K1[1], 0.0, K1[0], K1[2], 0.0, 0.0, 1.0};
  const double k2[9] = {K2[0], 0.0, K2[1], 0.0, K2[0], K2[2], 0.0, 0.0, 1.0};
  double T[9];
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c) T[3 * r + c] = (k2[r] * F[c] + k2[3 + r] * F[3 + c]) + k2[6 + r] * F[6 + c];  // K2^T F
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c) E[3 * r + c] = (T[3 * r] * k1[c] + T[3 * r + 1] * k1[3 + c]) + T[3 * r + 2] * k1[6 + c];
}

// MotionFromEssential: SVD E = U S V^T (singular values descending; U.col(2) = u1 x u2, so det U = +1; Vt.row(2)
// negated when det Vt < 0), W = [0 -1 0; 1 0 0; 0 0 1].  Candidates in upstream order:
//   0: (U W Vt, +u3)   1: (U W Vt, -u3)   2: (U W^T Vt, +u3)   3: (U W^T Vt, -u3)
// Ra = U W Vt, Rb = U W^T Vt, u3 = U.col(2), all row-major.
R3D_HD void motion_from_essential(const double* E, double* Ra, double* Rb, double* u3) {
  double a[9], v[9];
  for (int i = 0; i < 9; ++i) a[i] = E[i];
  hestenes<3, 3>(a, v);
  const double n0 = col_norm2_3(a, 0), n1 = col_norm2_3(a, 1), n2 = col_norm2_3(a, 2);
  int o0 = 0, o1 = 1, o2 = 2;  // column order by descending singular value (stable)
  if (n1 > n0) { o0 = 1; o1 = 0; }
  const double nn[3] = {n0, n1, n2};
  if (n2 > nn[o1]) {
    o2 = o1;
    o1 = 2;
    if (n2 > nn[o0]) { o1 = o0; o0 = 2; }
  }
  const double s0 = sqrt(nn[o0]), s1 = sqrt(nn[o1]);
  double U[9], Vt[9];
  for (int r = 0; r < 3; ++r) {
    U[3 * r + 0] = a[3 * r + o0] / s0;
    U[3 * r + 1] = a[3 * r + o1] / s1;
  }
  U[2] = U[3] * U[7] - U[6] * U[4];  // u3 = u1 x u2
  U[5] = U[6] * U[1] - U[0] * U[7];
  U[8] = U[0] * U[4] - U[3] * U[1];
  const int ord[3] = {o0, o1, o2};
  for (int k = 0; k < 3; ++k)
    for (int c = 0; c < 3; ++c) Vt[3 * k + c] = v[3 * c + ord[k]];
  const double detVt = (Vt[0] * (Vt[4] * Vt[8] - Vt[5] * Vt[7]) - Vt[1] * (Vt[3] * Vt[8] - Vt[5] * Vt[6])) +
                       Vt[2] * (Vt[3] * Vt[7] - Vt[4] * Vt[6]);
  if (detVt < 0.0)
    for (int c = 0; c < 3; ++c) Vt[6 + c] = -Vt[6 + c];
  // U W = [u2 | -u1 | u3], U W^T = [-u2 | u1 | u3]
  double UW[9], UWt[9];
  for (int r = 0; r < 3; ++r) {
    UW[3 * r + 0] = U[3 * r + 1];
    UW[3 * r + 1] = -U[3 * r + 0];
    UW[3 * r + 2] = U[3 * r + 2];
    UWt[3 * r + 0] = -U[3 * r + 1];
    UWt[3 * r + 1] = U[3 * r + 0];
    UWt[3 * r + 2] = U[3 * r + 2];
  }
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c) {
      Ra[3 * r + c] = (UW[3 * r] * Vt[c] + UW[3 * r + 1] * Vt[3 + c]) + UW[3 * r + 2] * Vt[6 + c];
      Rb[3 * r + c] = (UWt[3 * r] * Vt[c] + UWt[3 * r + 1] * Vt[3 + c]) + UWt[3 * r + 2] * Vt[6 + c];
    }
  for (int r = 0; r < 3; ++r) u3[r] = U[3 * r + 2];
}

// TriangulateDLT(P1 = [I|0], x1, P2 = [R|t], x2): design rows x[0] P.row(2) - x[2] P.row(0) and
// x[1] P.row(2) - x[2] P.row(1), homogeneous nullspace (right singular vector of the smallest singular value; the first
// of equal ones), hnormalized
R3D_HD void triangulate_dlt(const double* R, const double* t, const double* x1, const double* x2, double* X) {
  double D[16], V[16];
  D[0] = -x1[2]; D[1] = 0.0;    D[2] = x1[0];  D[3] = 0.0;
  D[4] = 0.0;    D[5] = -x1[2]; D[6] = x1[1];  D[7] = 0.0;
  for (int i = 0; i < 3; ++i) {
    D[8 + i] = x2[0] * R[6 + i] - x2[2] * R[i];
    D[12 + i] = x2[1] * R[6 + i] - x2[2] * R[3 + i];
  }
  D[11] = x2[0] * t[2] - x2[2] * t[0];
  D[15] = x2[1] * t[2] - x2[2] * t[1];
  hestenes<4, 4>(D, V);
  int m = 0;
  double best = 0.0;
  for (int c = 0; c < 4; ++c) {
    const double n = ((D[c] * D[c] + D[4 + c] * D[4 + c]) + D[8 + c] * D[8 + c]) + D[12 + c] * D[12 + c];
    if (c == 0 || n < best) { best = n; m = c; }
  }
  X[0] = V[m] / V[12 + m];
  X[1] = V[4 + m] / V[12 + m];
  X[2] = V[8 + m] / V[12 + m];
}

// Depth(R, t, X) = (R X + t)[2]
R3D_HD double depth(const double* R, const double* t, const double* X) {
  return ((R[6] * X[0] + R[7] * X[1]) + R[8] * X[2]) + t[2];
}

// the triangulation angle of AutomaticInitialPairChoice, degrees: ray1 = b1.normalized(), ray2 = (R^T b2).normalized(),
// R2D(acos(clamp(ray1 . ray2 / (|ray1| |ray2|), -1 + 1e-8, 1 - 1e-8)))
R3D_HD double ray_angle_deg(const double* R, const double* b1, const double* b2) {
  double r2[3];
  for (int i = 0; i < 3; ++i) r2[i] = (R[i] * b2[0] + R[3 + i] * b2[1]) + R[6 + i] * b2[2];
  const double n1 = sqrt((b1[0] * b1[0] + b1[1] * b1[1]) + b1[2] * b1[2]);
  const double n2 = sqrt((r2[0] * r2[0] + r2[1] * r2[1]) + r2[2] * r2[2]);
  double u1[3], u2[3];
  for (int i = 0; i < 3; ++i) {
    u1[i] = b1[i] / n1;
    u2[i] = r2[i] / n2;
  }
  const double dot = (u1[0] * u2[0] + u1[1] * u2[1]) + u1[2] * u2[2];
  const double m1 = sqrt((u1[0] * u1[0] + u1[1] * u1[1]) + u1[2] * u1[2]);
  const double m2 = sqrt((u2[0] * u2[0] + u2[1] * u2[1]) + u2[2] * u2[2]);
  double c = dot / (m1 * m2);
  const double lo = -1.0 + 1e-8, hi = 1.0 - 1e-8;
  c = c < lo ? lo : (c > hi ? hi : c);
  return dm::acos_det(c) / R3D_PI * 180.0;
}

}  // namespace rp
}  // namespace r3d
