// oracle_relpose.cpp -- CPU ORACLE (test infrastructure; see oracle.h).
//
// Restates openMVG::sfm::robustRelativePose (sfm/pipelines/sfm_robust_model_estimation.cpp) as the SfM engines
// Regard3D drives call it once per pair (src/threads/R3DTriangulationThread.cpp:222-250, :416-441, :492-512;
// SURVEY.md A.9):
//   ACRANSAC(ACKernelAdaptorEssential<FivePointSolver, EpipolarDistanceError>)  -> acransac_E (oracle_acransac.cpp)
//   RelativePoseFromEssential / estimate_Rt_fromE (multiview/solver_essential_kernel.cpp, triangulation.cpp)
//     MotionFromEssential, TriangulateDLT, Depth, std::max_element                -> relative_pose
//   SequentialSfMReconstructionEngine::AutomaticInitialPairChoice's ray angle and median -> the same
// Deliberate, documented deviations (DESIGN.md sec. 2):
//   * Eigen's JacobiSVD (3x3 for E, 4x4 for the DLT nullspace) is one-sided Jacobi with a fixed cyclic order and a
//     fixed orthogonality test; E and the nullspace are defined up to sign and scale, which changes neither the
//     candidate set nor the triangulated points;
//   * acos is oracle_detmath.hpp's;
//   * the essential matrix is K2^T F K1 of the F that AC-RANSAC scored, i.e. the winning 5-point model up to rounding
//     (the AC-RANSAC restatement hands out that F).
// Built as its own library (oracle/relpose.mk -> _build/liboracle_relpose.so, with the AC-RANSAC and 5-point sources).
// The product restates the same arithmetic in regard3d_b200/csrc/relpose_math.cuh; the two are compared bit for bit.
#include "oracle_relpose.h"
#include "oracle_detmath.hpp"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <limits>
#include <vector>
#include <omp.h>

namespace orc {

// oracle_acransac.cpp: the essential AC-RANSAC; F_out = K2^-T E K1^-1 of the winning 5-point model, info[0] = minNFA,
// info[1] = sqrt(errorMax) when inliers were kept
int64_t acransac_E(const double* xI, const double* xJ, uint32_t M, uint32_t wI, uint32_t hI, uint32_t wJ, uint32_t hJ,
                   const double* Kpair, double precision_px, uint32_t max_iter, std::vector<uint32_t>& vec_inliers,
                   double* F_out, double* info);

namespace {

const int kMaxSweeps = 12;

// Pinhole_Intrinsic::operator(): (K^-1 [x y 1]^T).normalized()
void bearing(const double* K, double x, double y, double* b) {
  const double kinv00 = 1.0 / K[0], kinv02 = -K[1] / K[0], kinv12 = -K[2] / K[0];
  const double bx = kinv00 * x + kinv02, by = kinv00 * y + kinv12, bz = 1.0;
  const double n = std::sqrt((bx * bx + by * by) + bz * bz);
  b[0] = bx / n; b[1] = by / n; b[2] = bz / n;
}

// one-sided Jacobi rotation of columns p < q of a (ROWS x COLS row-major), accumulated into v (COLS x COLS);
// false when the columns are already orthogonal to |cos| <= 1e-15
template <int ROWS, int COLS>
bool hestenes_rotate(double* a, double* v, int p, int q) {
  double alpha = 0.0, beta = 0.0, gamma = 0.0;
  for (int r = 0; r < ROWS; ++r) {
    const double ap = a[r * COLS + p], aq = a[r * COLS + q];
    alpha = alpha + ap * ap;
    beta = beta + aq * aq;
    gamma = gamma + ap * aq;
  }
  if (!(gamma * gamma > 1e-30 * (alpha * beta))) return false;
  const double zeta = (beta - alpha) / (2.0 * gamma);
  const double az = zeta < 0.0 ? -zeta : zeta;
  double t = 1.0 / (az + std::sqrt(1.0 + zeta * zeta));
  if (zeta < 0.0) t = -t;
  const double c = 1.0 / std::sqrt(1.0 + t * t);
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

template <int ROWS, int COLS>
void hestenes(double* a, double* v) {
  for (int i = 0; i < COLS * COLS; ++i) v[i] = (i % (COLS + 1) == 0) ? 1.0 : 0.0;
  for (int sweep = 0; sweep < kMaxSweeps; ++sweep) {
    bool rotated = false;
    for (int p = 0; p < COLS - 1; ++p)
      for (int q = p + 1; q < COLS; ++q) rotated = hestenes_rotate<ROWS, COLS>(a, v, p, q) || rotated;
    if (!rotated) break;
  }
}

double col_norm2_3(const double* a, int c) { return (a[c] * a[c] + a[3 + c] * a[3 + c]) + a[6 + c] * a[6 + c]; }

}  // namespace

// E = K2^T F K1 of the F that AC-RANSAC scored (F = K2^-T E K1^-1 of the winning 5-point model): that E up to rounding
void essential_from_fundamental(const double* F, const double* K1, const double* K2, double* E) {
  const double k1[9] = {K1[0], 0.0, K1[1], 0.0, K1[0], K1[2], 0.0, 0.0, 1.0};
  const double k2[9] = {K2[0], 0.0, K2[1], 0.0, K2[0], K2[2], 0.0, 0.0, 1.0};
  double T[9];
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c) T[3 * r + c] = (k2[r] * F[c] + k2[3 + r] * F[3 + c]) + k2[6 + r] * F[6 + c];  // K2^T F
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c) E[3 * r + c] = (T[3 * r] * k1[c] + T[3 * r + 1] * k1[3 + c]) + T[3 * r + 2] * k1[6 + c];
}

// MotionFromEssential: E = U S V^T, singular values descending, U.col(2) = u1 x u2 (det U = +1), Vt.row(2) negated when
// det Vt < 0; candidates (Ra, +u3), (Ra, -u3), (Rb, +u3), (Rb, -u3) with Ra = U W Vt, Rb = U W^T Vt
void motion_from_essential(const double* E, double* Ra, double* Rb, double* u3) {
  double a[9], v[9];
  for (int i = 0; i < 9; ++i) a[i] = E[i];
  hestenes<3, 3>(a, v);
  const double nn[3] = {col_norm2_3(a, 0), col_norm2_3(a, 1), col_norm2_3(a, 2)};
  int o0 = 0, o1 = 1, o2 = 2;
  if (nn[1] > nn[0]) { o0 = 1; o1 = 0; }
  if (nn[2] > nn[o1]) {
    o2 = o1;
    o1 = 2;
    if (nn[2] > nn[o0]) { o1 = o0; o0 = 2; }
  }
  const double s0 = std::sqrt(nn[o0]), s1 = std::sqrt(nn[o1]);
  double U[9], Vt[9];
  for (int r = 0; r < 3; ++r) {
    U[3 * r + 0] = a[3 * r + o0] / s0;
    U[3 * r + 1] = a[3 * r + o1] / s1;
  }
  U[2] = U[3] * U[7] - U[6] * U[4];
  U[5] = U[6] * U[1] - U[0] * U[7];
  U[8] = U[0] * U[4] - U[3] * U[1];
  const int ord[3] = {o0, o1, o2};
  for (int k = 0; k < 3; ++k)
    for (int c = 0; c < 3; ++c) Vt[3 * k + c] = v[3 * c + ord[k]];
  const double detVt = (Vt[0] * (Vt[4] * Vt[8] - Vt[5] * Vt[7]) - Vt[1] * (Vt[3] * Vt[8] - Vt[5] * Vt[6])) +
                       Vt[2] * (Vt[3] * Vt[7] - Vt[4] * Vt[6]);
  if (detVt < 0.0)
    for (int c = 0; c < 3; ++c) Vt[6 + c] = -Vt[6 + c];
  double UW[9], UWt[9];  // U W = [u2 | -u1 | u3], U W^T = [-u2 | u1 | u3]
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

// TriangulateDLT(P1 = [I|0], x1, P2 = [R|t], x2) -> hnormalized nullspace of the 4x4 design matrix
void triangulate_dlt(const double* R, const double* t, const double* x1, const double* x2, double* X) {
  double D[16], V[16];
  D[0] = -x1[2]; D[1] = 0.0;    D[2] = x1[0]; D[3] = 0.0;
  D[4] = 0.0;    D[5] = -x1[2]; D[6] = x1[1]; D[7] = 0.0;
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
static double depth(const double* R, const double* t, const double* X) {
  return ((R[6] * X[0] + R[7] * X[1]) + R[8] * X[2]) + t[2];
}

// AutomaticInitialPairChoice's ray angle in degrees (ray2 = R^T b2)
double ray_angle_deg(const double* R, const double* b1, const double* b2) {
  double r2[3];
  for (int i = 0; i < 3; ++i) r2[i] = (R[i] * b2[0] + R[3 + i] * b2[1]) + R[6 + i] * b2[2];
  const double n1 = std::sqrt((b1[0] * b1[0] + b1[1] * b1[1]) + b1[2] * b1[2]);
  const double n2 = std::sqrt((r2[0] * r2[0] + r2[1] * r2[1]) + r2[2] * r2[2]);
  double u1[3], u2[3];
  for (int i = 0; i < 3; ++i) {
    u1[i] = b1[i] / n1;
    u2[i] = r2[i] / n2;
  }
  const double dot = (u1[0] * u2[0] + u1[1] * u2[1]) + u1[2] * u2[2];
  const double m1 = std::sqrt((u1[0] * u1[0] + u1[1] * u1[1]) + u1[2] * u1[2]);
  const double m2 = std::sqrt((u2[0] * u2[0] + u2[1] * u2[1]) + u2[2] * u2[2]);
  double c = dot / (m1 * m2);
  const double lo = -1.0 + 1e-8, hi = 1.0 - 1e-8;
  c = c < lo ? lo : (c > hi ? hi : c);
  return det::acos(c) / det::kPi * 180.0;
}

// robustRelativePose of one pair (positions in pixels, Kpair = f, ppx, ppy of I then J); r.I / r.J are left alone
void relative_pose(const double* xI, const double* xJ, uint32_t M, uint32_t wI, uint32_t hI, uint32_t wJ, uint32_t hJ,
                   const double* Kpair, double precision_px, uint32_t max_iter, orc_relpose& r,
                   std::vector<uint32_t>& inl) {
  r.valid = 0;
  r.n_inliers = r.n_front = 0;
  r.min_nfa = r.found_residual_precision = std::numeric_limits<double>::infinity();
  std::memset(r.essential, 0, sizeof(r.essential));
  std::memset(r.rotation, 0, sizeof(r.rotation));
  std::memset(r.translation, 0, sizeof(r.translation));
  std::memset(r.center, 0, sizeof(r.center));
  r.median_angle_deg = 0.0;
  inl.clear();
  if (!(Kpair[0] > 0.0) || !(Kpair[3] > 0.0)) return;  // no valid pinhole intrinsic
  double info[3], F[9], E[9];
  acransac_E(xI, xJ, M, wI, hI, wJ, hJ, Kpair, precision_px, max_iter, inl, F, info);
  r.min_nfa = info[0];  // +inf when ACRANSAC returned at once (M <= 5)
  if (!(inl.size() > 5 * 2.5)) {  // minNFA >= 0 clears the inliers; fewer than MINIMUM_SAMPLES * 2.5: false
    inl.clear();
    return;
  }
  r.found_residual_precision = info[1];  // sqrt(errorMax), pixels
  r.n_inliers = (uint32_t)inl.size();
  essential_from_fundamental(F, Kpair, Kpair + 3, E);
  std::memcpy(r.essential, E, sizeof(E));
  // estimate_Rt_fromE
  double Rs[2][9], u3[3];
  motion_from_essential(E, Rs[0], Rs[1], u3);
  const size_t n = inl.size();
  std::vector<double> b1(3 * n), b2(3 * n);
  for (size_t k = 0; k < n; ++k) {
    bearing(Kpair, xI[2 * inl[k]], xI[2 * inl[k] + 1], &b1[3 * k]);
    bearing(Kpair + 3, xJ[2 * inl[k]], xJ[2 * inl[k] + 1], &b2[3 * k]);
  }
  uint32_t f[4] = {0, 0, 0, 0};
  std::vector<uint8_t> front(n);
  for (int i = 0; i < 4; ++i) {
    const double sg = (i & 1) ? -1.0 : 1.0;
    const double t[3] = {sg * u3[0], sg * u3[1], sg * u3[2]};
    for (size_t k = 0; k < n; ++k) {
      double X[3];
      triangulate_dlt(Rs[i >> 1], t, &b1[3 * k], &b2[3 * k], X);
      if (X[2] > 0.0 && depth(Rs[i >> 1], t, X) > 0.0) {
        ++f[i];
        front[k] |= (uint8_t)(1u << i);
      }
    }
  }
  const int best = (int)(std::max_element(f, f + 4) - f);
  if (f[best] == 0) return;
  const double* R = Rs[best >> 1];
  const double sg = (best & 1) ? -1.0 : 1.0;
  const double t[3] = {sg * u3[0], sg * u3[1], sg * u3[2]};
  r.valid = 1;
  r.n_front = f[best];
  std::memcpy(r.rotation, R, sizeof(r.rotation));
  std::memcpy(r.translation, t, sizeof(t));
  for (int i = 0; i < 3; ++i) r.center[i] = -((R[i] * t[0] + R[3 + i] * t[1]) + R[6 + i] * t[2]);
  std::vector<double> ang;
  ang.reserve(f[best]);
  for (size_t k = 0; k < n; ++k)
    if (front[k] & (1u << best)) ang.push_back(ray_angle_deg(R, &b1[3 * k], &b2[3 * k]));
  std::nth_element(ang.begin(), ang.begin() + ang.size() / 2, ang.end());
  r.median_angle_deg = ang[ang.size() / 2];
}

}  // namespace orc

extern "C" {

int orc_relative_pose(const double* xI, const double* xJ, uint32_t M, uint32_t wI, uint32_t hI, uint32_t wJ, uint32_t hJ,
                      const double* Kpair, double precision_px, uint32_t max_iter, orc_relpose* out, uint32_t* inliers) {
  std::vector<uint32_t> inl;
  orc::relative_pose(xI, xJ, M, wI, hI, wJ, hJ, Kpair, precision_px, max_iter, *out, inl);
  if (inliers) std::memcpy(inliers, inl.data(), inl.size() * sizeof(uint32_t));
  return out->valid;
}

int64_t orc_relative_poses(const float* const* xys, const uint32_t* widths, const uint32_t* heights, const double* Ks,
                           uint32_t n_views, const uint32_t* pairs, uint64_t P, const uint64_t* put_ofs,
                           const orc_indmatch* put, double precision_px, uint32_t max_iter, orc_relpose* out,
                           uint64_t* out_ofs, orc_indmatch* out_inl, int n_threads) {
  (void)n_views;
  if (n_threads <= 0) n_threads = omp_get_max_threads();
  std::vector<std::vector<orc_indmatch>> res(P);
#pragma omp parallel for schedule(dynamic) num_threads(n_threads)
  for (int64_t p = 0; p < (int64_t)P; ++p) {
    const uint32_t I = pairs[2 * p], J = pairs[2 * p + 1];
    const uint64_t b = put_ofs[p], e = put_ofs[p + 1];
    const uint32_t M = (uint32_t)(e - b);
    std::vector<double> xI(2 * (size_t)M + 2), xJ(2 * (size_t)M + 2);
    for (uint32_t k = 0; k < M; ++k) {
      xI[2 * k] = (double)xys[I][2 * (size_t)put[b + k].i];
      xI[2 * k + 1] = (double)xys[I][2 * (size_t)put[b + k].i + 1];
      xJ[2 * k] = (double)xys[J][2 * (size_t)put[b + k].j];
      xJ[2 * k + 1] = (double)xys[J][2 * (size_t)put[b + k].j + 1];
    }
    const double Kpair[6] = {Ks[3 * I], Ks[3 * I + 1], Ks[3 * I + 2], Ks[3 * J], Ks[3 * J + 1], Ks[3 * J + 2]};
    std::vector<uint32_t> inl;
    out[p].I = I;
    out[p].J = J;
    orc::relative_pose(xI.data(), xJ.data(), M, widths[I], heights[I], widths[J], heights[J], Kpair, precision_px, max_iter,
                       out[p], inl);
    for (uint32_t idx : inl) res[p].push_back(put[b + idx]);
  }
  uint64_t ofs = 0;
  for (uint64_t p = 0; p < P; ++p) {
    out_ofs[p] = ofs;
    std::memcpy(out_inl + ofs, res[p].data(), res[p].size() * sizeof(orc_indmatch));
    ofs += res[p].size();
  }
  out_ofs[P] = ofs;
  return (int64_t)ofs;
}

void orc_motion_from_essential(const double* E, double* R /* 4 x 9 */, double* t /* 4 x 3 */) {
  double Ra[9], Rb[9], u3[3];
  orc::motion_from_essential(E, Ra, Rb, u3);
  for (int i = 0; i < 4; ++i) {
    std::memcpy(R + 9 * i, (i >> 1) ? Rb : Ra, sizeof(Ra));
    const double sg = (i & 1) ? -1.0 : 1.0;
    for (int k = 0; k < 3; ++k) t[3 * i + k] = sg * u3[k];
  }
}

void orc_triangulate_dlt(const double* R, const double* t, const double* x1, const double* x2, double* X) {
  orc::triangulate_dlt(R, t, x1, x2, X);
}

}  // extern "C"
