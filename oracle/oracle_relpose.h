/*
 * oracle_relpose.h -- C ABI of the CPU ORACLE's relative poses (test infrastructure; see oracle.h).
 * robustRelativePose = essential ACRANSAC + estimate_Rt_fromE, plus AutomaticInitialPairChoice's angle (SURVEY.md A.9).
 * Built as oracle/_build/liboracle_relpose.so by oracle/relpose.mk (with the AC-RANSAC and 5-point restatements).
 */
#ifndef R3D_ORACLE_RELPOSE_H
#define R3D_ORACLE_RELPOSE_H
#include "oracle.h"
#ifdef __cplusplus
extern "C" {
#endif

/* the layout of r3d_relative_pose (include/r3dgpu.h) */
typedef struct {
  uint32_t I, J; int valid;
  uint32_t n_inliers, n_front;
  double min_nfa, found_residual_precision;
  double essential[9], rotation[9], translation[3], center[3];
  double median_angle_deg;
} orc_relpose;
/* one pair; inliers (capacity M, may be null): the AC-RANSAC inliers (indices into the putatives, residual order).
 * returns valid.  out->I / out->J are not touched. */
int orc_relative_pose(const double* xI, const double* xJ, uint32_t M, uint32_t wI, uint32_t hI, uint32_t wJ, uint32_t hJ,
                      const double* Kpair, double precision_px, uint32_t max_iter, orc_relpose* out, uint32_t* inliers);
/* every pair of a CSR map (omp over pairs): out[P], the AC-RANSAC inlier CSR like orc_filter_pairs_E */
int64_t orc_relative_poses(const float* const* xys, const uint32_t* widths, const uint32_t* heights, const double* Ks,
                           uint32_t n_views, const uint32_t* pairs, uint64_t P, const uint64_t* put_ofs,
                           const orc_indmatch* put, double precision_px, uint32_t max_iter, orc_relpose* out,
                           uint64_t* out_ofs, orc_indmatch* out_inl, int n_threads);
/* MotionFromEssential: the 4 candidates (R row-major, t) in upstream order */
void orc_motion_from_essential(const double* E, double* R /* 4 x 9 */, double* t /* 4 x 3 */);
/* TriangulateDLT([I|0], x1, [R|t], x2) -> X (hnormalized) */
void orc_triangulate_dlt(const double* R, const double* t, const double* x1, const double* x2, double* X);

#ifdef __cplusplus
}
#endif
#endif
