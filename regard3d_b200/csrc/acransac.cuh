// acransac.cuh -- shared declarations of the AC-RANSAC fundamental filter (host + device).
#pragma once
#include "r3d_internal.cuh"

namespace r3d {

struct AcPair {          // per image pair (device)
  uint32_t pt_ofs;       // first point of this pair in x1/x2
  uint32_t M;            // number of putative matches
  uint32_t tbl_ofs;      // first entry of this pair's logc_n table
  uint32_t pad_;
  double max_thr;        // precision^2 * N2(0,0)^2
  double logalpha0;      // F: log10(2 D / A / N2(0,0)) ; H: log10(pi / (w h) / N2(0,0)^2), image J
  double loge0;          // log10(MAX_MODELS * (M - MINIMUM_SAMPLES))
  double K[6];           // essential model only: f, ppx, ppy of image I, then of image J (pinhole K)
};

// internal model ids: 0 = F (7-point), 1 = H (4-point), 2 = E (5-point); Kernel::MINIMUM_SAMPLES / MAX_MODELS
__host__ __device__ constexpr uint32_t ac_min_samples(int model) { return model == 0 ? 7u : (model == 1 ? 4u : 5u); }
__host__ __device__ constexpr uint32_t ac_max_models(int model) { return model == 0 ? 3u : (model == 1 ? 1u : 10u); }

struct AcPointSrc {      // per pair: where its matched positions come from and how they are normalised
  const float2* xyI;     // positions of view I / J on the device (uploaded with the regions)
  const float2* xyJ;
  double s1, c1x, c1y;   // x1 = s1 * x + c1  (ACKernelAdaptor normalisation; identity for the essential model)
  double s2, c2x, c2y;
  uint32_t nI, nJ, identity, pad_;
};

struct AcHyp {           // one RANSAC iteration of one pair
  uint32_t pair;
  uint32_t sample[7];
};

struct AcScore {         // per (hypothesis, model)
  double nfa;            // best NFA over k (inf if none)
  double err;            // residual at the best k (errorMax)
  uint32_t k;            // best k (number of inliers)
  uint32_t count;        // residuals <= max_thr (classic-RANSAC phase of ACRANSAC)
};

struct AcInlierReq {
  uint32_t pair;
  uint32_t k;            // number of inliers wanted (prefix of the sorted residuals)
  uint32_t out_ofs;
  uint32_t hyp_model;    // hypothesis * MAX_MODELS + model: where this round's model matrix lives on the device
};

struct AcFusedOut {      // per pair, written by the persistent kernel (acransac_fused.cu)
  double minNFA, errorMax;
  uint32_t n_inliers;    // 0 when minNFA >= 0; else the best model's inliers, listed in residual order
  uint32_t iterations;   // RANSAC iterations the state machine consumed
  uint32_t exact_scores; // models that needed the sort + exact NFA scan (tier 2)
  uint32_t models;       // models scored
  uint32_t events;       // pool replacements
  uint32_t pad_;
};

// persistent one-CTA-per-pair ACRANSAC (acransac_fused.cu); `order`: pair ids of one size class, largest first;
// huge: sort buffers / pool in global scratch (cap entries per CTA of the grid); out_F (essential model only, may be
// nullptr): 9 doubles per pair, the winning model as scored (F = K2^-T E K1^-1), zeros when no model was ever kept
size_t acransac_fused_smem_bytes(int model, uint32_t cap, bool huge);
int acransac_fused_ctas_per_sm(int model, uint32_t cap, bool huge);
int launch_acransac_fused(r3d_ctx* ctx, DeviceWorker& w, int model, bool huge, const AcPair* pairs, const uint32_t* order,
                          uint32_t n_order, uint32_t* work_counter, const double2* x1, const double2* x2, const float* logc_n,
                          const float* logc_k, uint32_t cap, uint32_t max_iter, double* g_se, uint32_t* g_si, uint32_t* g_pool,
                          const uint2* matches, uint2* out_matches, AcFusedOut* out, double* out_F, uint32_t grid);

struct RelposeDev {      // per pair, written by k_relpose (relpose.cu)
  double E[9];           // K2^T F K1 of the winning F (zeros when AC-RANSAC failed)
  double R[9], t[3], C[3];  // chosen candidate of MotionFromEssential: X_J = R X_I + t, C = -R^T t
  double median_angle_deg;
  uint32_t n_front;      // inliers in front of both cameras under the chosen candidate (0: the pair fails)
  uint32_t pad_;
};

// relative pose of every pair from its AC-RANSAC result (relpose.cu, k_relpose: one CTA per pair), on the filter's
// stream: pairs / ac / F (9 doubles per pair) / inlier (i, j) lists as the fused kernel left them; keys / mask:
// pt_total entries of scratch
int launch_relpose(r3d_ctx* ctx, DeviceWorker& w, const AcPair* pairs, const AcPointSrc* src, uint32_t n_pairs,
                   const AcFusedOut* ac, const double* F, const uint2* inl, unsigned long long* keys, uint8_t* mask,
                   RelposeDev* out);

// x1/x2[pt_ofs + k] = normalised positions of putative match k of every pair (double, like MatchesPairToMat)
int launch_ac_points(r3d_ctx* ctx, DeviceWorker& w, const AcPair* pairs, const AcPointSrc* src, uint32_t n_pairs,
                     const uint2* matches, double2* x1, double2* x2, uint32_t* bad_flag);
int launch_ac_tables(r3d_ctx* ctx, DeviceWorker& w, const AcPair* pairs, uint32_t n_pairs, const float* vlog10, float* logc_n);
int launch_f7_solve(r3d_ctx* ctx, DeviceWorker& w, int model, const AcPair* pairs, const double2* x1, const double2* x2,
                    const AcHyp* hyps, uint32_t n_hyp, double* F, uint32_t* nmodels);
int launch_f7_score(r3d_ctx* ctx, DeviceWorker& w, int model, const AcPair* pairs, const double2* x1, const double2* x2,
                    const AcHyp* hyps, uint32_t n_hyp, const double* F, const uint32_t* nmodels, const float* logc_n,
                    const float* logc_k, uint32_t cap, AcScore* scores);
int launch_f7_inliers(r3d_ctx* ctx, DeviceWorker& w, int model, const AcPair* pairs, const double2* x1, const double2* x2,
                      const AcInlierReq* reqs, uint32_t n_req, const double* F, uint32_t cap, uint32_t* out);

}  // namespace r3d
