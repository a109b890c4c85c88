/*
 * r3dgpu.h -- C ABI of libr3dgpu.so: the B200 (sm_100a) replacement of Regard3D's compute-matches
 * hot path and the downstream bundle-adjustment solve.
 *
 * Every entry point names the reference interface it replaces (paths relative to the Regard3D
 * tree, rhiestan/Regard3D @ 2822275).  The reference has no FFI of its own: the binding a
 * maintainer adds is the C++ shim in regard3d_b200/csrc/R3DComputeMatches_b200.{h,cpp} (same
 * class name / method set as src/R3DComputeMatches.h:30-74); see INTEGRATION.md.
 *
 * Conventions: plain pointers + sizes, host memory in and out, no C++/CUDA/torch types.
 * Return value: 0 = R3D_OK, negative = error (r3d_last_error() gives the text).  There is NO CPU
 * fallback: without a usable sm_100 device r3d_create() fails with R3D_ERR_NO_DEVICE.
 * Threading: a context may be used from any one thread at a time (the reference calls
 * computeMatches() on one dedicated wxThread: src/threads/R3DComputeMatchesThread.cpp:91-103).
 */
#ifndef R3DGPU_H
#define R3DGPU_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define R3D_ABI_VERSION 3

typedef enum {
  R3D_OK = 0,
  R3D_ERR_INVALID = -1,      /* bad argument */
  R3D_ERR_CUDA = -2,         /* a CUDA runtime / driver call failed */
  R3D_ERR_NOMEM = -3,
  R3D_ERR_IO = -4,           /* file could not be read / written */
  R3D_ERR_UNSUPPORTED = -5,  /* e.g. descriptor range outside what the fp16 operand can hold */
  R3D_ERR_NO_DEVICE = -6     /* no sm_100 GPU: the library never falls back to the CPU */
} r3d_status;

typedef enum { R3D_F32 = 0, R3D_U8 = 1 } r3d_dtype;

/* openMVG::matching::IndMatch{i_,j_}: i_ indexes the FIRST image of the pair, j_ the second
 * (consumer: src/threads/PreviewGeneratorThread.cpp:373-390). */
typedef struct { uint32_t i, j; } r3d_indmatch;

typedef struct r3d_ctx r3d_ctx;
/* openMVG::matching::PairWiseMatches = std::map<Pair, IndMatches> (opaque, host memory). */
typedef struct r3d_matches r3d_matches;

/* ---- context ------------------------------------------------------------------------------- */
/* One context drives the listed CUDA devices (one worker + stream set per device; pairs shard
 * across them without any collective).  bench.py uses one process per GPU, i.e. n_devices = 1.
 * Replaces: construction of R3DComputeMatches (src/threads/R3DComputeMatchesThread.cpp:91). */
int r3d_create(const int* device_ids, int n_devices, r3d_ctx** out);
void r3d_destroy(r3d_ctx* ctx);
const char* r3d_last_error(const r3d_ctx* ctx); /* ctx may be NULL: last global error */
int r3d_abi_version(void);

/* ---- regions ------------------------------------------------------------------------------- */
/* Replaces Regions_Provider::load (src/R3DComputeMatches.cpp:2040) for one view:
 * desc = Regions::DescriptorRawData() (n x dim row-major, float32 or uint8; Regard3D's native
 * type is Scalar_Regions<SIOPointFeature,float,144>, src/Regard3DFeatures.h:42-48),
 * xy = feature positions (n x 2 float32, from the .feat file; may be NULL if no coordinate
 * de-duplication / geometric filtering will be requested).  Data is copied. */
int r3d_upload_regions(r3d_ctx* ctx, uint32_t view_id, const void* desc, uint32_t n, uint32_t dim,
                       int dtype, const float* xy);
int r3d_clear_regions(r3d_ctx* ctx);

/* ---- descriptors (SURVEY.md 8f-1: the stage that feeds the .desc files) ------------------------------ */
/* cv::KeyPoint as Regard3D uses it: position, size = diameter, angle in degrees. */
typedef struct { float x, y, size, angle; } r3d_keypoint;
/* Replaces Regard3DFeatures::extractLIOPFeatures (src/Regard3DFeatures.cpp:719-861) for one image: per keypoint a
 * 41x41 patch (cv::warpAffine with the inverse map of :766-800, cv::GaussianBlur sigma 1.2) and its LIOP descriptor
 * r3d_vl_liopdesc_process [src/thirdparty/liop/vl_liop.c:434-575] (4 neighbours, 6 spatial bins, radius 6 -> 144
 * floats, unit L2 norm).  image: height x width float32 row-major (openMVG::image::Image<float>, cv::eigen2cv);
 * kp_size_factor: Regard3DFeatures::getKpSizeFactor (:691-716; 8 for AKAZE / Fast-AKAZE); desc_out: n x 144, in
 * keypoint order (the reference appends in thread-completion order, :838-851). */
int r3d_liop_describe(r3d_ctx* ctx, const float* image, uint32_t width, uint32_t height,
                      const r3d_keypoint* keypoints, uint32_t n, float kp_size_factor, float* desc_out);
/* Diagnostics: the descriptor function alone (vl_liop.c:434-575) on n ready 41x41 float32 patches. */
int r3d_debug_liop_process(r3d_ctx* ctx, const float* patches, uint32_t n, float* desc_out);

/* ---- putative matching --------------------------------------------------------------------- */
#define R3D_MATCH_DEFAULT 0u
#define R3D_MATCH_EXACT_SCAN 1u   /* skip the tensor-core candidate pass: CUDA-core exact scan only */
#define R3D_MATCH_NO_COORD_DEDUP 2u /* skip IndMatchDecorator (for callers without positions) */
#define R3D_MATCH_CASCADE_HASHING 8u /* OpenMVG CASCADE_HASHING_L2 (BASELINE config 4) instead of the exhaustive 2-NN:
                                   * approximate by construction, bit-identical to the CPU restatement of the algorithm */
#define R3D_MATCH_MUTUAL_NN 4u    /* OFF by default and NOT reference behaviour (MatchDistanceRatio has no cross-check):
                                   * keep (i, j) only if j is also i's nearest neighbour among J's descriptors */

/* Replaces Matcher_Regions(fDistRatio, BRUTE_FORCE_L2)::Match(regions_provider, pairs, out)
 * (src/R3DComputeMatches.cpp:2039, :2048; loop shape :437-488): for every pair (I,J): 2-NN of each
 * J descriptor in I under squared L2, keep iff d1 < ratio^2 * d2, IndMatch(i in I, j in J),
 * (i,j) de-duplication, coordinate de-duplication.  pairs = P x 2 view ids.  Pairs without
 * matches are absent from the result, like in the reference's map. */
int r3d_match_pairs(r3d_ctx* ctx, const uint32_t* pairs, uint64_t n_pairs, float dist_ratio,
                    uint32_t flags, r3d_matches** out);

/* R3D_MATCH_CASCADE_HASHING replaces Cascade_Hashing_Matcher_Regions::Match (OpenMVG matching_image_collection, the
 * matcher BASELINE config 4 names; Regard3D's own GUI never selects it, src/R3DComputeMatches.cpp:2035-2062).  Its hash
 * codes depend on the zero-mean descriptor of ALL views of the matching job, so a job that is split over several
 * r3d_match_pairs calls (ranks, shards) declares its views once: r3d_cascade_prepare hashes the given views (already
 * uploaded) under their common zero-mean descriptor; later R3D_MATCH_CASCADE_HASHING calls whose pairs stay inside
 * that set reuse the tables.  Without it every call hashes the views of its own pair list (= one call is one job, the
 * reference's behaviour).  Views of more than 65536 features or dimension > 256: R3D_ERR_UNSUPPORTED. */
int r3d_cascade_prepare(r3d_ctx* ctx, const uint32_t* view_ids, uint32_t n_views);

/* Replaces openMVG::matching::ArrayMatcher<float,L2>::SearchNeighbours(query, nbQuery, &idx, &dist,
 * NN=2) -- the plug-in API Regard3D implements in src/utils/matcher_hnsw.h:133-191 -- with the
 * database = regions of view_db (ArrayMatcher::Build, :53-68) and queries = regions of view_query.
 * idx / dist: n_query x 2, ascending exact squared distance (float accumulate, upstream order). */
int r3d_search_neighbours(r3d_ctx* ctx, uint32_t view_db, uint32_t view_query, int32_t* idx,
                          float* dist);

/* ---- PairWiseMatches accessors ------------------------------------------------------------- */
uint64_t r3d_matches_num_pairs(const r3d_matches* m);
uint64_t r3d_matches_total(const r3d_matches* m);
/* k-th pair in std::map order (sorted by I, then J). */
int r3d_matches_get_pair(const r3d_matches* m, uint64_t k, uint32_t* I, uint32_t* J,
                         const r3d_indmatch** matches, uint64_t* count);
/* Build a PairWiseMatches from CSR arrays (pair_ofs has n_pairs+1 entries). */
int r3d_matches_from_csr(const uint32_t* pairs, uint64_t n_pairs, const uint64_t* pair_ofs,
                         const r3d_indmatch* matches, r3d_matches** out);
/* Flat copy of the map in std::map order: pairs_out 2 x num_pairs view ids, ofs_out num_pairs + 1 prefix offsets,
 * matches_out r3d_matches_total() entries; any output may be NULL.  This is what a per-GPU process ships when the
 * pair list is sharded over ranks and the PairWiseMatches map is re-assembled on one of them (SURVEY.md 8e:
 * "results concatenated on host in pair order"; the reference's map insert is src/R3DComputeMatches.cpp:483-486). */
int r3d_matches_export_csr(const r3d_matches* m, uint32_t* pairs_out, uint64_t* ofs_out,
                           r3d_indmatch* matches_out);
void r3d_free_matches(r3d_matches* m);
/* matching::Save / matching::Load, text format (src/R3DComputeMatches.cpp:2064, :2120;
 * SURVEY.md Appendix B.3). */
int r3d_save_matches_txt(const r3d_matches* m, const char* path);
int r3d_load_matches_txt(const char* path, r3d_matches** out);

/* matching::Save / matching::Load as the reference calls them: the extension picks the format -- ".txt" (above) or
 * ".bin" = cereal PortableBinary of std::map<Pair, std::vector<IndMatch>> (SURVEY.md App. B.3; layout restated in
 * regard3d_b200/csrc/sfm_data_io.cpp). */
int r3d_save_matches_bin(const r3d_matches* m, const char* path);
int r3d_load_matches_bin(const char* path, r3d_matches** out);
int r3d_save_matches(const r3d_matches* m, const char* path);
int r3d_load_matches(const char* path, r3d_matches** out);

/* ---- sfm_data.bin (SURVEY.md App. B.4) ------------------------------------------------------------------------
 * openMVG::sfm::SfM_Data as the reference stores it: cereal PortableBinary "sfm_data.bin", written by
 * R3DProject::writeSfmData (src/R3DProject.cpp:1118-1306: views / view priors + intrinsics), read by
 * R3DComputeMatches::computeMatches (src/R3DComputeMatches.cpp:1755) and R3DTriangulationThread
 * (src/threads/R3DTriangulationThread.cpp:403), written back with poses + structure (:453-455).  Opaque handle +
 * plain-struct accessors; maps are walked in key order (k-th element). */
typedef struct r3d_sfm_data r3d_sfm_data;
/* openMVG::sfm::ESfM_Data */
#define R3D_SFM_VIEWS 1u
#define R3D_SFM_EXTRINSICS 2u
#define R3D_SFM_INTRINSICS 4u
#define R3D_SFM_STRUCTURE 8u
#define R3D_SFM_CONTROL_POINTS 16u
#define R3D_SFM_ALL 31u
/* openMVG::cameras::EINTRINSIC (the `cameraModel` argument of computeMatches, src/R3DProject.cpp:1167-1191) */
#define R3D_CAM_PINHOLE 1
#define R3D_CAM_PINHOLE_RADIAL1 2
#define R3D_CAM_PINHOLE_RADIAL3 3
#define R3D_CAM_PINHOLE_BROWN 4
#define R3D_CAM_PINHOLE_FISHEYE 5
typedef struct {
  uint32_t id_view, id_intrinsic, id_pose, width, height;
  const char* local_path;  /* folder part of View::s_Img_path */
  const char* filename;    /* file part */
  int has_prior;           /* openMVG::sfm::ViewPriors with b_use_pose_center_ (GPS; src/R3DProject.cpp:1194-1220) */
  double center_weight[3], pose_center[3];
} r3d_sfm_view;
typedef struct {
  uint32_t id;
  int model;               /* R3D_CAM_* */
  uint32_t width, height;
  double focal, ppx, ppy;
  double disto[5];         /* K1: k1 | K3: k1 k2 k3 | Brown T2: k1 k2 k3 t1 t2 | fisheye: k1 k2 k3 k4 */
} r3d_sfm_intrinsic;
typedef struct { uint32_t id; double rotation[9]; double center[3]; } r3d_sfm_pose;  /* geometry::Pose3: R row-major, C */
typedef struct { uint32_t id_view, id_feat; double x[2]; } r3d_sfm_observation;
int r3d_sfm_data_create(r3d_sfm_data** out);
void r3d_sfm_data_free(r3d_sfm_data* sd);
int r3d_sfm_data_load(const char* path, r3d_sfm_data** out);                       /* Load(sfm_data, path, ALL) */
int r3d_sfm_data_save(const r3d_sfm_data* sd, const char* path, uint32_t parts);   /* Save(sfm_data, path, parts) */
const char* r3d_sfm_root_path(const r3d_sfm_data* sd);
int r3d_sfm_set_root_path(r3d_sfm_data* sd, const char* root_path);
uint32_t r3d_sfm_num_views(const r3d_sfm_data* sd);
uint32_t r3d_sfm_num_intrinsics(const r3d_sfm_data* sd);
uint32_t r3d_sfm_num_poses(const r3d_sfm_data* sd);
uint32_t r3d_sfm_num_landmarks(const r3d_sfm_data* sd, int control_points);
int r3d_sfm_add_view(r3d_sfm_data* sd, const r3d_sfm_view* v);                     /* strings are copied */
int r3d_sfm_get_view(const r3d_sfm_data* sd, uint32_t k, r3d_sfm_view* out);       /* strings owned by sd */
int r3d_sfm_add_intrinsic(r3d_sfm_data* sd, const r3d_sfm_intrinsic* in);
int r3d_sfm_get_intrinsic(const r3d_sfm_data* sd, uint32_t k, r3d_sfm_intrinsic* out);
int r3d_sfm_add_pose(r3d_sfm_data* sd, const r3d_sfm_pose* p);
int r3d_sfm_get_pose(const r3d_sfm_data* sd, uint32_t k, r3d_sfm_pose* out);
int r3d_sfm_add_landmark(r3d_sfm_data* sd, int control_point, uint32_t id, const double X[3],
                         const r3d_sfm_observation* obs, uint32_t n_obs);
int r3d_sfm_get_landmark(const r3d_sfm_data* sd, int control_point, uint32_t k, uint32_t* id, double X[3],
                         r3d_sfm_observation* obs, uint32_t obs_cap, uint32_t* n_obs);

/* ---- geometric filtering ------------------------------------------------------------------- */
typedef enum { R3D_MODEL_F = 0, R3D_MODEL_E = 1, R3D_MODEL_H = 2 } r3d_model;
/* One entry per view id (sfm_data views + their intrinsics).  focal / ppx / ppy: pinhole K of the view as
 * R3DProject builds it (src/R3DProject.cpp:1149-1159: focal = max(w,h) * focal_mm / sensor_width, else
 * 1.1 * max(w,h); pp = (w/2, h/2)); only the essential filter reads them, focal <= 0 = "no valid pinhole
 * intrinsic" (the pair is dropped, as GeometricFilter_EMatrix_AC does). */
typedef struct { uint32_t width, height; double focal, ppx, ppy; } r3d_view_info;

/* Replaces ImageCollectionGeometricFilter::Robust_model_estimation(
 *   GeometricFilter_FMatrix_AC(precision_px = 4.0, max_iter = 2048), putative, false)
 * + Get_geometric_matches() (src/R3DComputeMatches.cpp:2099-2115).  Uses the positions uploaded
 * with r3d_upload_regions.  views[v] = image size of view v (sfm_data views).
 * R3D_MODEL_H: GeometricFilter_HMatrix_AC(4.0, 2048) (src/R3DComputeMatches.cpp:2215-2219; 4-point DLT,
 * asymmetric transfer error, point-to-point a-contrario model).
 * R3D_MODEL_E: GeometricFilter_EMatrix_AC(4.0, 2048) (:2169-2171; Nister/Stewenius 5-point solver on bearing
 * vectors, <= 10 models per sample, one-sided epipolar distance of F = K2^-T E K1^-1 in pixels). The
 * poor-overlap post-filter of :2173-2191 belongs to computeMatches() and is applied by r3d_compute_matches. */
int r3d_filter_pairs(r3d_ctx* ctx, int model, double precision_px, uint32_t max_iter,
                     const r3d_matches* putative, const r3d_view_info* views, uint32_t n_views,
                     r3d_matches** out);

/* ---- relative poses (SURVEY.md App. A.9) ----------------------------------------------------------------------- */
/* openMVG::sfm::RelativePose_Info of one pair, plus what AutomaticInitialPairChoice scores it by. */
typedef struct {
  uint32_t I, J; int valid;            /* valid = robustRelativePose returned true */
  uint32_t n_inliers, n_front;         /* AC-RANSAC inliers; those in front of both cameras (chosen candidate) */
  double min_nfa, found_residual_precision;  /* ACRANSAC's minNFA (+inf when it never ran); sqrt(errorMax) in pixels (+inf unless it succeeded) */
  double essential[9], rotation[9], translation[3], center[3];  /* row-major; X_J = R X_I + t, C = -R^T t, |t| = 1 */
  double median_angle_deg;             /* the (n_front / 2)-th smallest triangulation angle of the front inliers */
} r3d_relative_pose;
/* Replaces openMVG::sfm::robustRelativePose(intrinsics_I, intrinsics_J, x_I, x_J, relativePose_info, size_I, size_J,
 * max_iter) run on every pair of a matches map -- the per-pair step of GlobalSfMReconstructionEngine_RelativeMotions
 * (Compute_Relative_Rotations), of SfMSceneInitializerStellar and of SequentialSfMReconstructionEngine's
 * AutomaticInitialPairChoice (src/threads/R3DTriangulationThread.cpp:222-250, :416-441, :492-512):
 *   ACRANSAC(ACKernelAdaptorEssential<FivePointSolver, EpipolarDistanceError>) with initial_residual_tolerance =
 *   Square(precision_px) (+inf: the unbounded a-contrario mode, robustRelativePose's default) and max_iter iterations
 *   (4096 by default) -- exactly r3d_filter_pairs(R3D_MODEL_E, precision_px, max_iter); the pair fails on minNFA >= 0
 *   or fewer than 2.5 * 5 inliers;
 *   then estimate_Rt_fromE: the four (R, t) of MotionFromEssential, TriangulateDLT of every inlier's bearing vectors
 *   under each, the candidate with the most points in front of both cameras (the first maximum; none: the pair fails).
 * median_angle_deg: the ray angle of AutomaticInitialPairChoice over the n_front inliers, the n_front/2-th smallest
 * (0-based); the thresholds that decide an initial pair are the caller's.  Bearings come from views[] (pinhole K, no
 * undistortion, as the E filter); focal <= 0 on either view or <= 5 matches: invalid.  out: num_pairs entries in map
 * order; essential (K2^T F K1 of the scored F = K2^-T E K1^-1, i.e. the winning 5-point E up to rounding),
 * n_inliers and found_residual_precision are set whenever AC-RANSAC succeeded.  inliers (may be NULL): the AC-RANSAC inlier map,
 * identical to r3d_filter_pairs(R3D_MODEL_E) with the same parameters.  The pairs shard over the context's devices
 * like r3d_filter_pairs; r3d_get_filter_timing then reports the AC-RANSAC kernels as ms_score and the pose kernel
 * inside ms_device_total.  The host-round AC-RANSAC (R3D_FILTER_HOST_ROUNDS set, or the device sample stream failing
 * its self-test, r3d_debug_rng_selftest() == 0) does not support this entry: R3D_ERR_UNSUPPORTED. */
int r3d_relative_poses(r3d_ctx* ctx, const r3d_matches* matches, const r3d_view_info* views, uint32_t n_views,
                       double precision_px, uint32_t max_iter, r3d_relative_pose* out /* num_pairs entries, map order */,
                       r3d_matches** inliers /* or NULL */);

/* ---- bundle adjustment --------------------------------------------------------------------- */
/* Replaces openMVG::sfm::Bundle_Adjustment_Ceres::Adjust as driven by the SfM engines' Process()
 * (src/threads/R3DTriangulationThread.cpp:441, :512, :250).  Default camera model: pinhole radial-K3 (chosen at :398,
 * built at src/R3DProject.cpp:1177-1180); the four other models the reference can store are selected per intrinsic
 * group with intr_model.  Tracks may have any length. */
typedef struct {
  uint32_t n_cams, n_pts, n_intr;
  uint64_t n_obs;
  double* poses;       /* n_cams x 6: angle-axis, t ; X_cam = R X + t          (in/out) */
  double* intrinsics;  /* n_intr x 6: f, ppx, ppy, k1, k2, k3                  (in/out) */
  double* points;      /* n_pts x 3                                            (in/out) */
  const uint32_t* obs_cam;   /* n_obs */
  const uint32_t* obs_pt;    /* n_obs */
  const uint32_t* cam_intr;  /* n_cams: intrinsic group of each camera */
  const double* obs_xy;      /* n_obs x 2 */
  /* --- ABI 3 (all optional: NULL / 0 = round-1 behaviour) --- */
  const uint8_t* intr_model; /* n_intr: camera model of each group, R3D_CAM_* (src/R3DProject.cpp:1167-1191); NULL = radial K3.
                              * intrinsics[g] = f, ppx, ppy, then the model's first three distortion coefficients
                              * (pinhole: none, K1: k1, K3 / Brown: k1 k2 k3, fisheye: k1 k2 k3); slots a model does not
                              * own are ignored and never change */
  const double* intrinsics_ext; /* n_intr x 2 or NULL: Brown T2: t1 t2, fisheye: k4 -- read, HELD FIXED by the solve
                              * (intrinsic blocks of the reduced camera system are 6 wide) */
  uint32_t n_priors;         /* pose-centre priors = openMVG ViewPriors with b_use_pose_center_ (GPS) */
  const uint32_t* prior_cam; /* n_priors: camera (pose) index */
  const double* prior_center;/* n_priors x 3 */
  const double* prior_weight;/* n_priors x 3 (ViewPriors::center_weight_) */
} r3d_ba_problem;

typedef struct {
  uint32_t max_iterations;   /* 500 */
  double huber_a;            /* HuberLoss(Square(4.0)) -> 16 ; <= 0: trivial loss */
  int refine_intrinsics;     /* Intrinsic_Parameter_Type ADJUST_ALL (1) / NONE (0), R3DTriangulationThread.cpp:429-432 */
  double function_tolerance; /* 1e-6 */
  double gradient_tolerance; /* 1e-10 */
  double parameter_tolerance;/* 1e-8 */
  double initial_radius;     /* 1e4 */
  double prior_huber_a;      /* ABI 3: HuberLoss(a) of the pose-centre prior blocks (OpenMVG: Square(pose_center_robust_
                              * fitting_error)); <= 0: trivial loss */
} r3d_ba_options;

typedef struct {
  uint32_t iterations, successful_steps;
  double initial_cost, final_cost;
  int termination;           /* 0 max iters, 1 function tol, 2 gradient tol, 3 parameter tol, 4 failure */
  double seconds_total, seconds_linear;
  double seconds_setup;      /* validation, CSR build, uploads (inside seconds_total) */
} r3d_ba_summary;

void r3d_ba_default_options(r3d_ba_options* o);
int r3d_bundle_adjust(r3d_ctx* ctx, r3d_ba_problem* io, const r3d_ba_options* opt,
                      r3d_ba_summary* summary, double* cost_trace /* max_iterations+1 or NULL */);

/* openMVG::sfm::Bundle_Adjustment_Ceres::Adjust(SfM_Data&, Optimize_Options) on the SfM_Data container itself: poses
 * (R, C) <-> angle-axis | t, one parameter block per intrinsic id in its own camera model, landmarks; refined values are
 * written back into sd.  solver.refine_intrinsics = Intrinsic_Parameter_Type ADJUST_ALL / NONE; use_motion_priors adds
 * one pose-centre block per ViewPriors view (sfmEngine.Set_Use_Motion_Prior, R3DTriangulationThread.cpp:433).  The C++
 * adaptor with the reference's class shape is regard3d_b200/csrc/Bundle_Adjustment_b200.h. */
typedef struct {
  r3d_ba_options solver;
  int use_motion_priors;
} r3d_sfm_ba_options;
void r3d_sfm_ba_default_options(r3d_sfm_ba_options* o);
int r3d_sfm_bundle_adjust(r3d_ctx* ctx, r3d_sfm_data* sd, const r3d_sfm_ba_options* opt, r3d_ba_summary* summary);

/* ---- the steps either side of bundle adjustment (SURVEY.md 8f-3) -------------------------------------------------
 * openMVG::tracks::TracksBuilder Build + Filter(min_length) + ExportToSTL, as Regard3D calls them itself
 * (src/threads/PreviewGeneratorThread.cpp:345-352) and as every SfM engine it drives starts: union-find over the
 * pairwise matches; tracks with two features of one image or fewer than min_length images are dropped.  Tracks come
 * in track-id order (upstream: the union-find root), each as its (view, feature) pairs in view order. */
typedef struct r3d_tracks r3d_tracks;
int r3d_tracks_build(const r3d_matches* m, uint32_t min_length /* 2 */, r3d_tracks** out);
uint64_t r3d_tracks_count(const r3d_tracks* t);
int r3d_tracks_get(const r3d_tracks* t, uint64_t k, uint32_t* track_id, const uint32_t** views, const uint32_t** feats,
                   uint32_t* n);
/* TracksUtilsMap::GetTracksInImages (PreviewGeneratorThread.cpp:354-358): tracks seen in ALL listed views, cut to them */
int r3d_tracks_in_images(const r3d_tracks* t, const uint32_t* view_ids, uint32_t n, r3d_tracks** out);
void r3d_tracks_free(r3d_tracks* t);
/* Tracks -> sd.structure (observation = position of the feature, from r3d_upload_regions of that view id), then
 * SfM_Data_Structure_Computation_Blind::triangulate: every landmark from all its views with a pose and an intrinsic
 * (iteratively re-weighted DLT); landmarks with fewer than two such views or a non-positive depth are erased. */
int r3d_sfm_structure_from_tracks(r3d_ctx* ctx, r3d_sfm_data* sd, const r3d_tracks* tracks, uint32_t* n_rejected);
/* RemoveOutliers_PixelResidualError(sd, max_pixel_residual, min_track_length) then RemoveOutliers_AngleError(sd,
 * min_angle_deg) -- the rejection step the engines run after each bundle adjustment (4.0 px / 2.0 degrees upstream).
 * min_angle_deg <= 0 skips the angle test. */
int r3d_sfm_remove_outliers(r3d_ctx* ctx, r3d_sfm_data* sd, double max_pixel_residual, uint32_t min_track_length,
                            double min_angle_deg, uint32_t* removed_observations, uint32_t* removed_landmarks);

/* ---- multi-GPU bundle adjustment (SURVEY.md 8e: the one path with a real exchange step) -------
 * One process per GPU.  The 3-D points (with all their observations) are partitioned over the
 * ranks, cameras and intrinsics are replicated: every rank passes r3d_bundle_adjust ALL cameras /
 * intrinsics and ITS points + observations.  Per LM iteration the partial reduced camera system
 * S = U - sum W V^-1 W^T and its right-hand side are summed over the ranks with ONE ncclAllReduce
 * (double) over NVLink, the dense Cholesky is replicated, back-substitution is local; cost, camera
 * gradient / Jacobi scaling and the step norms are small all-reduces.  On return poses/intrinsics
 * are identical on every rank, points hold the rank's own slice.  There is no reference counterpart
 * (Ceres is single-process); parity is against the single-GPU path / the oracle.
 * libnccl.so.2 is resolved at run time (the copy already loaded in the process, e.g. torch's, else
 * $R3D_NCCL_LIB, else the system one).  The id is created on rank 0 and distributed by the host
 * (torch.distributed / MPI / a file). */
#define R3D_COMM_ID_BYTES 128
int r3d_comm_unique_id(r3d_ctx* ctx, uint8_t id[R3D_COMM_ID_BYTES]);
int r3d_comm_init(r3d_ctx* ctx, int world, int rank, const uint8_t id[R3D_COMM_ID_BYTES]);
int r3d_comm_destroy(r3d_ctx* ctx);
int r3d_comm_world(const r3d_ctx* ctx);   /* 1 when no communicator is attached */
/* OpenMVGHelper::calculateResiduals (src/utils/OpenMVGHelper.cpp:2572-2590): |residual| per
 * coordinate, 2 per observation -- the BA quality metric the GUI reports. */
int r3d_ba_residuals(r3d_ctx* ctx, const r3d_ba_problem* p, double* res /* n_obs x 2 */);

/* ---- file-level twin of R3DComputeMatches::computeMatches() --------------------------------- */
#define R3D_MATCHING_CASCADE_HASHING 100 /* not a value of the reference's matchingAlgorithm switch */
typedef void (*r3d_progress_cb)(float fraction, const char* message, void* user);

typedef struct {
  float dist_ratio;               /* R3DFParams::distRatio_ (src/Regard3DFeatures.h:52-69) */
  int compute_fundamental;        /* R3DFParams::computeFundalmentalMatrix_ */
  int compute_essential;          /* R3DFParams::computeEssentialMatrix_ -> matches.e.txt (+ the poor-overlap filter) */
  int compute_homography;         /* R3DFParams::computeHomographyMatrix_ -> matches.h.txt */
  int matching_algorithm;         /* 0..8 as src/R3DComputeMatches.cpp:2036-2062; all map to the exact GPU matcher.
                                   * Extension: R3D_MATCHING_CASCADE_HASHING selects R3D_MATCH_CASCADE_HASHING */
  uint32_t descriptor_dim;        /* 144 for R3D_AKAZE_LIOP_Regions */
  int svg_output;                 /* computeMatches(..., bool svgOutput, ...): PutativeAdjacencyMatrix.svg and
                                   * GeometricAdjacencyMatrix.svg in the matches dir (:2074-2076, :2238-2240) */
} r3d_cm_params;

typedef struct {
  const char* matches_dir;        /* R3DProjectPaths::relativeMatchesPath_ : holds <img>.feat/.desc, outputs */
  const char* const* image_basenames; /* n_views names without extension (image%06d, src/R3DProject.cpp:1042) */
  const r3d_view_info* views;     /* image sizes (sfm_data views) */
  uint32_t n_views;
  const char* matches_f_filename; /* R3DProjectPaths::matchesFFilename_ ; NULL -> <matches_dir>/matches.f.txt */
  const char* matches_h_filename; /* R3DProjectPaths::matchesHFilename_ ; NULL -> <matches_dir>/matches.h.txt */
  const char* matches_e_filename; /* R3DProjectPaths::matchesEFilename_ ; NULL -> <matches_dir>/matches.e.txt */
} r3d_cm_paths;

typedef struct {
  uint32_t n_views;
  uint32_t* number_of_keypoints;  /* caller array of n_views (R3DComputeMatchesStatistics::numberOfKeypoints_) */
  uint64_t putative_pairs, putative_matches, f_pairs, f_matches, h_pairs, h_matches, e_pairs, e_matches;
  double seconds_load, seconds_match, seconds_filter;
} r3d_cm_stats;

/* Steps of R3DComputeMatches::computeMatches() after feature extraction
 * (src/R3DComputeMatches.cpp:2035-2126): load regions, exhaustive pairs, putative matching,
 * Save(matches.putative.txt), F filter, Save(matches.f.txt), E filter + poor-overlap removal (< 50 inliers or
 * < 30 % of the putatives, :2173-2191), Save(matches.e.txt), H filter, Save(matches.h.txt); progress fractions
 * as the reference emits them (0.7 putative, 0.8 F, 0.9 E, 0.95 H; SURVEY.md sec. 5). */
int r3d_compute_matches(r3d_ctx* ctx, const r3d_cm_params* params, const r3d_cm_paths* paths,
                        r3d_progress_cb cb, void* user, r3d_cm_stats* stats);

/* ---- instrumentation ----------------------------------------------------------------------- */
typedef struct {
  double ms_prep;        /* upload-time operand preparation kernels */
  double ms_candidates;  /* tcgen05 candidate kernel(s), CUDA-event time on their stream */
  double ms_rerank;      /* exact re-rank + ratio kernel(s) */
  double ms_fallback;    /* exact-scan kernel for uncertified queries + the per-pair pack / (i,j) sort kernel */
  double ms_device_total;/* first launch -> last kernel of the last r3d_match_pairs */
  double ms_host_post;   /* host de-duplication */
  uint64_t kernel_launches;
  uint64_t queries, fallback_queries, third_chunk_queries, fifth_chunk_queries;  /* R3D_MATCH_CASCADE_HASHING: the last two count
                                                                                 * raw / distinct bucket candidates instead */
  uint64_t h2d_bytes, d2h_bytes;
  uint64_t rejected_queries; /* dropped before any exact distance: the ratio test provably cannot pass */
} r3d_match_timing;
int r3d_get_match_timing(const r3d_ctx* ctx, r3d_match_timing* out);

typedef struct {
  double ms_solve, ms_score, ms_device_total, ms_host;
  uint64_t kernel_launches, hypotheses, rounds;
} r3d_filter_timing;
int r3d_get_filter_timing(const r3d_ctx* ctx, r3d_filter_timing* out);

/* Diagnostics (host only, no GPU needed): IndMatch::getDeduplicated + IndMatchDecorator::getDeduplicated of one
 * pair, in place; returns the new count.  The CPU test pins it against std::set. */
int64_t r3d_debug_post_process(r3d_indmatch* m, int64_t n, const float* xyI, const float* xyJ, int coord_dedup);
/* the same for up to 4 pairs advanced in lockstep by one thread (what the batch tails call) */
int r3d_debug_post_process_many(int lanes, r3d_indmatch* const* ms, uint64_t* counts, const float* const* xyIs,
                                const float* const* xyJs, int coord_dedup);
/* the descent-free replay the batch tails use (per-view y-rank / shared-x tables, built here from the n_keypoints
 * positions of view I) */
int64_t r3d_debug_post_process_ranked(r3d_indmatch* m, int64_t n, const float* xyI, uint32_t n_keypoints, const float* xyJ);

/* Diagnostics (host only): 1 when the library's device-side restatement of std::mt19937 +
 * std::uniform_int_distribution<uint32_t> (the ACRANSAC sample stream) reproduces this process's <random>; the
 * filters then run entirely on the device, otherwise samples are drawn on the host, round by round. */
int r3d_debug_rng_selftest(void);
/* test hook: hash tables of a prepared view (code n x ceil(dim/32), bucket n x 6, bk_ofs 6 x 1025, bk_ids 6 x n) */
int r3d_debug_cascade_view(r3d_ctx* ctx, uint32_t view_id, uint32_t* code, uint16_t* bucket, uint32_t* bk_ofs, uint32_t* bk_ids);

/* Diagnostics: the packed candidate keys per query row (n_query padded to 256 rows x 8 uint32:
 * 6 keys ascending + 2 unused)
 * the tensor-core pass produced for (view_db, view_query), and the pair's error bound. */
int r3d_debug_candidate_keys(r3d_ctx* ctx, uint32_t view_db, uint32_t view_query, uint32_t* keys,
                             float* eps_abs);

/* Diagnostics (runs on the host, no GPU needed): residual and analytic Jacobian (2 x 15: intrinsics
 * 0..5, pose 6..11, point 12..14) of one observation, as the BA kernels evaluate them. */
int r3d_debug_ba_jacobian(const double* intr, const double* pose, const double* X, const double* obs,
                          double* r, double* J);
/* the same for any of the five camera models (ext: the model's coefficients 4, 5 or NULL) */
int r3d_debug_ba_jacobian_model(int model, const double* intr, const double* ext, const double* pose, const double* X,
                                const double* obs, double* r, double* J);
/* pose-centre prior block: r[3] = weight .* (C(pose) - center), J[3 x 6] = d r / d (angle-axis, t) */
int r3d_debug_ba_prior(const double* pose, const double* center, const double* weight, double* r, double* J);

#ifdef __cplusplus
}
#endif
#endif /* R3DGPU_H */
