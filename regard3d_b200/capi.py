"""ctypes binding of libr3dgpu.so (include/r3dgpu.h).

Fails loudly: importing works anywhere (the CPU-only tests check the exported symbols), but
`Context()` raises R3DError when no sm_100 device is present -- there is no CPU fallback.
"""
import ctypes as C
import math
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("R3D_LIB") or os.path.join(_HERE, "libr3dgpu.so")  # R3D_LIB: an A/B build of the same ABI

R3D_F32, R3D_U8 = 0, 1
MATCH_DEFAULT, MATCH_EXACT_SCAN, MATCH_NO_COORD_DEDUP, MATCH_MUTUAL_NN, MATCH_CASCADE_HASHING = 0, 1, 2, 4, 8
MATCHING_CASCADE_HASHING = 100  # r3d_cm_params.matching_algorithm extension
MODEL_F, MODEL_E, MODEL_H = 0, 1, 2

indmatch_dtype = np.dtype([("i", np.uint32), ("j", np.uint32)])

EXPORTS = [
    "r3d_create", "r3d_destroy", "r3d_last_error", "r3d_abi_version", "r3d_upload_regions",
    "r3d_clear_regions", "r3d_match_pairs", "r3d_search_neighbours", "r3d_matches_num_pairs",
    "r3d_matches_total", "r3d_matches_get_pair", "r3d_matches_from_csr", "r3d_free_matches",
    "r3d_save_matches_txt", "r3d_load_matches_txt", "r3d_filter_pairs", "r3d_ba_default_options",
    "r3d_bundle_adjust", "r3d_ba_residuals", "r3d_compute_matches", "r3d_get_match_timing",
    "r3d_get_filter_timing", "r3d_debug_candidate_keys", "r3d_debug_ba_jacobian",
    "r3d_comm_unique_id", "r3d_comm_init", "r3d_comm_destroy", "r3d_comm_world", "r3d_debug_post_process",
    "r3d_debug_post_process_many", "r3d_debug_post_process_ranked", "r3d_matches_export_csr", "r3d_debug_rng_selftest", "r3d_liop_describe", "r3d_debug_liop_process",
    "r3d_save_matches_bin", "r3d_load_matches_bin", "r3d_save_matches", "r3d_load_matches", "r3d_sfm_data_create",
    "r3d_sfm_data_free", "r3d_sfm_data_load", "r3d_sfm_data_save", "r3d_sfm_root_path", "r3d_sfm_set_root_path",
    "r3d_sfm_num_views", "r3d_sfm_num_intrinsics", "r3d_sfm_num_poses", "r3d_sfm_num_landmarks", "r3d_sfm_add_view",
    "r3d_sfm_get_view", "r3d_sfm_add_intrinsic", "r3d_sfm_get_intrinsic", "r3d_sfm_add_pose", "r3d_sfm_get_pose",
    "r3d_sfm_add_landmark", "r3d_sfm_get_landmark", "r3d_debug_ba_jacobian_model", "r3d_debug_ba_prior", "r3d_sfm_ba_default_options", "r3d_sfm_bundle_adjust",
    "r3d_tracks_build", "r3d_tracks_count", "r3d_tracks_get", "r3d_tracks_in_images", "r3d_tracks_free",
    "r3d_sfm_structure_from_tracks", "r3d_sfm_remove_outliers", "r3d_cascade_prepare", "r3d_debug_cascade_view",
    "r3d_relative_poses",
]


class R3DError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libr3dgpu error %d: %s" % (code, msg))
        self.code = code


class MatchTiming(C.Structure):
    _fields_ = [("ms_prep", C.c_double), ("ms_candidates", C.c_double), ("ms_rerank", C.c_double),
                ("ms_fallback", C.c_double), ("ms_device_total", C.c_double), ("ms_host_post", C.c_double),
                ("kernel_launches", C.c_uint64), ("queries", C.c_uint64), ("fallback_queries", C.c_uint64),
                ("third_chunk_queries", C.c_uint64), ("fifth_chunk_queries", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
                ("rejected_queries", C.c_uint64)]


class FilterTiming(C.Structure):
    _fields_ = [("ms_solve", C.c_double), ("ms_score", C.c_double), ("ms_device_total", C.c_double),
                ("ms_host", C.c_double), ("kernel_launches", C.c_uint64), ("hypotheses", C.c_uint64),
                ("rounds", C.c_uint64)]


class ViewInfo(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("focal", C.c_double), ("ppx", C.c_double),
                ("ppy", C.c_double)]


def make_views(widths, heights, Ks=None):
    """r3d_view_info array.  Ks: n x 3 (focal, ppx, ppy); default = R3DProject's approximation
    (src/R3DProject.cpp:1149-1159): focal = 1.1 * max(w, h), principal point at the image centre."""
    n = len(widths)
    views = (ViewInfo * n)()
    for k in range(n):
        w, h = int(widths[k]), int(heights[k])
        views[k].width, views[k].height = w, h
        if Ks is None:
            views[k].focal, views[k].ppx, views[k].ppy = 1.1 * max(w, h), w / 2.0, h / 2.0
        else:
            views[k].focal, views[k].ppx, views[k].ppy = float(Ks[k][0]), float(Ks[k][1]), float(Ks[k][2])
    return views


class RelativePose(C.Structure):
    """r3d_relative_pose (openMVG RelativePose_Info + the initial-pair score)."""
    _fields_ = [("I", C.c_uint32), ("J", C.c_uint32), ("valid", C.c_int), ("n_inliers", C.c_uint32), ("n_front", C.c_uint32),
                ("min_nfa", C.c_double), ("found_residual_precision", C.c_double), ("essential", C.c_double * 9),
                ("rotation", C.c_double * 9), ("translation", C.c_double * 3), ("center", C.c_double * 3),
                ("median_angle_deg", C.c_double)]


# the same layout as a numpy record (what Context.relative_poses returns)
relative_pose_dtype = np.dtype({
    "names": [f for f, _ in RelativePose._fields_],
    "formats": [np.uint32, np.uint32, np.int32, np.uint32, np.uint32, np.float64, np.float64, (np.float64, (3, 3)),
                (np.float64, (3, 3)), (np.float64, 3), (np.float64, 3), np.float64],
    "offsets": [getattr(RelativePose, f).offset for f, _ in RelativePose._fields_],
    "itemsize": C.sizeof(RelativePose),
})


class BAProblem(C.Structure):
    _fields_ = [("n_cams", C.c_uint32), ("n_pts", C.c_uint32), ("n_intr", C.c_uint32), ("n_obs", C.c_uint64),
                ("poses", C.c_void_p), ("intrinsics", C.c_void_p), ("points", C.c_void_p),
                ("obs_cam", C.c_void_p), ("obs_pt", C.c_void_p), ("cam_intr", C.c_void_p),
                ("obs_xy", C.c_void_p),
                ("intr_model", C.c_void_p), ("intrinsics_ext", C.c_void_p), ("n_priors", C.c_uint32),
                ("prior_cam", C.c_void_p), ("prior_center", C.c_void_p), ("prior_weight", C.c_void_p)]


class BAOptions(C.Structure):
    _fields_ = [("max_iterations", C.c_uint32), ("huber_a", C.c_double), ("refine_intrinsics", C.c_int),
                ("function_tolerance", C.c_double), ("gradient_tolerance", C.c_double),
                ("parameter_tolerance", C.c_double), ("initial_radius", C.c_double), ("prior_huber_a", C.c_double)]


class BASummary(C.Structure):
    _fields_ = [("iterations", C.c_uint32), ("successful_steps", C.c_uint32), ("initial_cost", C.c_double),
                ("final_cost", C.c_double), ("termination", C.c_int), ("seconds_total", C.c_double),
                ("seconds_linear", C.c_double), ("seconds_setup", C.c_double)]


class CMParams(C.Structure):
    _fields_ = [("dist_ratio", C.c_float), ("compute_fundamental", C.c_int), ("compute_essential", C.c_int),
                ("compute_homography", C.c_int), ("matching_algorithm", C.c_int), ("descriptor_dim", C.c_uint32),
                ("svg_output", C.c_int)]


class CMPaths(C.Structure):
    _fields_ = [("matches_dir", C.c_char_p), ("image_basenames", C.POINTER(C.c_char_p)),
                ("views", C.POINTER(ViewInfo)), ("n_views", C.c_uint32), ("matches_f_filename", C.c_char_p),
                ("matches_h_filename", C.c_char_p), ("matches_e_filename", C.c_char_p)]


class CMStats(C.Structure):
    _fields_ = [("n_views", C.c_uint32), ("number_of_keypoints", C.POINTER(C.c_uint32)),
                ("putative_pairs", C.c_uint64), ("putative_matches", C.c_uint64), ("f_pairs", C.c_uint64),
                ("f_matches", C.c_uint64), ("h_pairs", C.c_uint64), ("h_matches", C.c_uint64), ("e_pairs", C.c_uint64),
                ("e_matches", C.c_uint64), ("seconds_load", C.c_double), ("seconds_match", C.c_double),
                ("seconds_filter", C.c_double)]


PROGRESS_CB = C.CFUNCTYPE(None, C.c_float, C.c_char_p, C.c_void_p)

_lib = None


def lib():
    """Load libr3dgpu.so (raises if it has not been built: `python -m regard3d_b200.build`)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("libr3dgpu.so is not built; run `python -m regard3d_b200.build` "
                              "(there is no fallback implementation)")
        L = C.CDLL(LIB_PATH)
        L.r3d_last_error.restype = C.c_char_p
        L.r3d_last_error.argtypes = [C.c_void_p]
        L.r3d_matches_num_pairs.restype = C.c_uint64
        L.r3d_matches_num_pairs.argtypes = [C.c_void_p]
        L.r3d_matches_total.restype = C.c_uint64
        L.r3d_matches_total.argtypes = [C.c_void_p]
        L.r3d_free_matches.argtypes = [C.c_void_p]
        L.r3d_destroy.argtypes = [C.c_void_p]
        L.r3d_sfm_data_free.argtypes = [C.c_void_p]
        L.r3d_sfm_root_path.restype = C.c_char_p
        L.r3d_sfm_root_path.argtypes = [C.c_void_p]
        for fn in (L.r3d_sfm_num_views, L.r3d_sfm_num_intrinsics, L.r3d_sfm_num_poses):
            fn.restype = C.c_uint32
            fn.argtypes = [C.c_void_p]
        L.r3d_sfm_num_landmarks.restype = C.c_uint32
        L.r3d_sfm_num_landmarks.argtypes = [C.c_void_p, C.c_int]
        L.r3d_sfm_data_save.argtypes = [C.c_void_p, C.c_char_p, C.c_uint32]
        L.r3d_sfm_set_root_path.argtypes = [C.c_void_p, C.c_char_p]
        L.r3d_sfm_add_view.argtypes = [C.c_void_p, C.c_void_p]
        L.r3d_sfm_get_view.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]
        L.r3d_sfm_add_intrinsic.argtypes = [C.c_void_p, C.c_void_p]
        L.r3d_sfm_get_intrinsic.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]
        L.r3d_sfm_add_pose.argtypes = [C.c_void_p, C.c_void_p]
        L.r3d_sfm_get_pose.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]
        L.r3d_sfm_add_landmark.argtypes = [C.c_void_p, C.c_int, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32]
        L.r3d_sfm_get_landmark.argtypes = [C.c_void_p, C.c_int, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
        L.r3d_tracks_count.restype = C.c_uint64
        L.r3d_tracks_count.argtypes = [C.c_void_p]
        L.r3d_tracks_free.argtypes = [C.c_void_p]
        L.r3d_tracks_build.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]
        L.r3d_tracks_get.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.r3d_tracks_in_images.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
        L.r3d_sfm_structure_from_tracks.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.r3d_sfm_remove_outliers.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_uint32, C.c_double, C.c_void_p, C.c_void_p]
        L.r3d_sfm_bundle_adjust.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.r3d_save_matches.argtypes = [C.c_void_p, C.c_char_p]
        L.r3d_save_matches_bin.argtypes = [C.c_void_p, C.c_char_p]
        L.r3d_comm_world.argtypes = [C.c_void_p]
        L.r3d_debug_post_process.restype = C.c_int64
        L.r3d_debug_post_process_ranked.restype = C.c_int64
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class Matches:
    """PairWiseMatches handle (openMVG::matching::PairWiseMatches)."""

    def __init__(self, handle):
        self.handle = C.c_void_p(handle) if not isinstance(handle, C.c_void_p) else handle

    def __del__(self):
        try:
            if self.handle:
                lib().r3d_free_matches(self.handle)
                self.handle = None
        except Exception:
            pass

    @property
    def num_pairs(self):
        return int(lib().r3d_matches_num_pairs(self.handle))

    @property
    def total(self):
        return int(lib().r3d_matches_total(self.handle))

    def pair(self, k):
        I, J = C.c_uint32(), C.c_uint32()
        ptr = C.c_void_p()
        cnt = C.c_uint64()
        rc = lib().r3d_matches_get_pair(self.handle, C.c_uint64(k), C.byref(I), C.byref(J), C.byref(ptr), C.byref(cnt))
        if rc:
            raise R3DError(rc, "r3d_matches_get_pair")
        n = cnt.value
        if n == 0:
            return I.value, J.value, np.zeros(0, indmatch_dtype)
        buf = (C.c_uint8 * (8 * n)).from_address(ptr.value)
        return I.value, J.value, np.frombuffer(buf, dtype=indmatch_dtype).copy()

    def to_dict(self):
        out = {}
        for k in range(self.num_pairs):
            I, J, m = self.pair(k)
            out[(I, J)] = m
        return out

    def to_csr(self, pairs):
        """CSR over the caller's pair list (empty range for pairs absent from the map)."""
        d = self.to_dict()
        pairs = np.asarray(pairs, np.uint32).reshape(-1, 2)
        ofs = np.zeros(len(pairs) + 1, np.uint64)
        chunks = []
        for k, (I, J) in enumerate(pairs):
            m = d.get((int(I), int(J)))
            n = 0 if m is None else len(m)
            ofs[k + 1] = ofs[k] + n
            if n:
                chunks.append(m)
        allm = np.concatenate(chunks) if chunks else np.zeros(0, indmatch_dtype)
        return ofs, allm

    def export_csr(self, pairs_out=None, ofs_out=None, matches_out=None):
        """(pairs[P,2] u32, ofs[P+1] u64, matches[total]) in map order -- one memcpy per pair inside the library.
        Caller buffers (e.g. pinned torch tensors viewed as numpy) may be passed to avoid allocations."""
        P, T = self.num_pairs, self.total
        if pairs_out is None:
            pairs_out = np.empty((P, 2), np.uint32)
        if ofs_out is None:
            ofs_out = np.empty(P + 1, np.uint64)
        if matches_out is None:
            matches_out = np.empty(T, indmatch_dtype)
        assert pairs_out.size >= 2 * P and ofs_out.size >= P + 1 and matches_out.size >= T
        rc = lib().r3d_matches_export_csr(self.handle, _p(pairs_out), _p(ofs_out), _p(matches_out))
        if rc:
            raise R3DError(rc, "r3d_matches_export_csr")
        return pairs_out, ofs_out, matches_out

    def save(self, path):
        """matching::Save: '.txt' or '.bin' (cereal portable binary) by extension."""
        rc = lib().r3d_save_matches(self.handle, path.encode())
        if rc:
            raise R3DError(rc, "r3d_save_matches(%s)" % path)

    @staticmethod
    def load(path):
        h = C.c_void_p()
        rc = lib().r3d_load_matches(path.encode(), C.byref(h))
        if rc:
            raise R3DError(rc, "r3d_load_matches(%s)" % path)
        return Matches(h)

    def save_txt(self, path):
        rc = lib().r3d_save_matches_txt(self.handle, path.encode())
        if rc:
            raise R3DError(rc, "r3d_save_matches_txt(%s)" % path)

    @staticmethod
    def load_txt(path):
        h = C.c_void_p()
        rc = lib().r3d_load_matches_txt(path.encode(), C.byref(h))
        if rc:
            raise R3DError(rc, "r3d_load_matches_txt(%s)" % path)
        return Matches(h)

    @staticmethod
    def from_csr(pairs, ofs, m):
        pairs = np.ascontiguousarray(pairs, np.uint32).reshape(-1, 2)
        ofs = np.ascontiguousarray(ofs, np.uint64)
        m = np.ascontiguousarray(m, indmatch_dtype)
        h = C.c_void_p()
        rc = lib().r3d_matches_from_csr(_p(pairs), C.c_uint64(len(pairs)), _p(ofs), _p(m), C.byref(h))
        if rc:
            raise R3DError(rc, "r3d_matches_from_csr")
        return Matches(h)


class SfmView(C.Structure):
    _fields_ = [("id_view", C.c_uint32), ("id_intrinsic", C.c_uint32), ("id_pose", C.c_uint32), ("width", C.c_uint32),
                ("height", C.c_uint32), ("local_path", C.c_char_p), ("filename", C.c_char_p), ("has_prior", C.c_int),
                ("center_weight", C.c_double * 3), ("pose_center", C.c_double * 3)]


class SfmIntrinsic(C.Structure):
    _fields_ = [("id", C.c_uint32), ("model", C.c_int), ("width", C.c_uint32), ("height", C.c_uint32),
                ("focal", C.c_double), ("ppx", C.c_double), ("ppy", C.c_double), ("disto", C.c_double * 5)]


class SfmPose(C.Structure):
    _fields_ = [("id", C.c_uint32), ("rotation", C.c_double * 9), ("center", C.c_double * 3)]


class SfmObservation(C.Structure):
    _fields_ = [("id_view", C.c_uint32), ("id_feat", C.c_uint32), ("x", C.c_double * 2)]


SFM_VIEWS, SFM_EXTRINSICS, SFM_INTRINSICS, SFM_STRUCTURE, SFM_CONTROL_POINTS, SFM_ALL = 1, 2, 4, 8, 16, 31
CAM_PINHOLE, CAM_RADIAL1, CAM_RADIAL3, CAM_BROWN, CAM_FISHEYE = 1, 2, 3, 4, 5


class SfmData:
    """openMVG::sfm::SfM_Data handle (sfm_data.bin: cereal portable binary, no OpenMVG needed)."""

    def __init__(self, handle=None):
        if handle is None:
            handle = C.c_void_p()
            rc = lib().r3d_sfm_data_create(C.byref(handle))
            if rc:
                raise R3DError(rc, "r3d_sfm_data_create")
        self.h = handle

    def __del__(self):
        try:
            if self.h:
                lib().r3d_sfm_data_free(self.h)
                self.h = None
        except Exception:
            pass

    @staticmethod
    def load(path):
        h = C.c_void_p()
        rc = lib().r3d_sfm_data_load(path.encode(), C.byref(h))
        if rc:
            raise R3DError(rc, "r3d_sfm_data_load(%s)" % path)
        return SfmData(h)

    def save(self, path, parts=SFM_ALL):
        rc = lib().r3d_sfm_data_save(self.h, path.encode(), C.c_uint32(parts))
        if rc:
            raise R3DError(rc, "r3d_sfm_data_save(%s)" % path)

    @property
    def root_path(self):
        return lib().r3d_sfm_root_path(self.h).decode()

    @root_path.setter
    def root_path(self, p):
        lib().r3d_sfm_set_root_path(self.h, p.encode())

    def add_view(self, id_view, filename, width, height, id_intrinsic=None, id_pose=None, local_path="", prior_center=None,
                 prior_weight=(1.0, 1.0, 1.0)):
        v = SfmView(id_view, id_view if id_intrinsic is None else id_intrinsic, id_view if id_pose is None else id_pose,
                    width, height, local_path.encode(), filename.encode(), 0 if prior_center is None else 1,
                    (C.c_double * 3)(*prior_weight), (C.c_double * 3)(*(prior_center or (0.0, 0.0, 0.0))))
        rc = lib().r3d_sfm_add_view(self.h, C.byref(v))
        if rc:
            raise R3DError(rc, "r3d_sfm_add_view")

    def add_intrinsic(self, id, model, width, height, focal, ppx, ppy, disto=()):
        d = list(disto) + [0.0] * (5 - len(disto))
        s = SfmIntrinsic(id, model, width, height, focal, ppx, ppy, (C.c_double * 5)(*d))
        rc = lib().r3d_sfm_add_intrinsic(self.h, C.byref(s))
        if rc:
            raise R3DError(rc, "r3d_sfm_add_intrinsic")

    def add_pose(self, id, R, center):
        s = SfmPose(id, (C.c_double * 9)(*np.asarray(R, float).reshape(9)), (C.c_double * 3)(*np.asarray(center, float)))
        rc = lib().r3d_sfm_add_pose(self.h, C.byref(s))
        if rc:
            raise R3DError(rc, "r3d_sfm_add_pose")

    def add_landmark(self, id, X, obs, control_point=False):
        """obs: list of (id_view, id_feat, x, y)."""
        arr = (SfmObservation * max(len(obs), 1))()
        for k, (v, f, x, y) in enumerate(obs):
            arr[k] = SfmObservation(v, f, (C.c_double * 2)(x, y))
        rc = lib().r3d_sfm_add_landmark(self.h, C.c_int(int(control_point)), C.c_uint32(id), (C.c_double * 3)(*X), arr,
                                        C.c_uint32(len(obs)))
        if rc:
            raise R3DError(rc, "r3d_sfm_add_landmark")

    def views(self):
        out = []
        for k in range(lib().r3d_sfm_num_views(self.h)):
            v = SfmView()
            lib().r3d_sfm_get_view(self.h, C.c_uint32(k), C.byref(v))
            out.append(dict(id_view=v.id_view, id_intrinsic=v.id_intrinsic, id_pose=v.id_pose, width=v.width, height=v.height,
                            local_path=v.local_path.decode(), filename=v.filename.decode(), has_prior=bool(v.has_prior),
                            center_weight=list(v.center_weight), pose_center=list(v.pose_center)))
        return out

    def intrinsics(self):
        out = []
        for k in range(lib().r3d_sfm_num_intrinsics(self.h)):
            s = SfmIntrinsic()
            lib().r3d_sfm_get_intrinsic(self.h, C.c_uint32(k), C.byref(s))
            out.append(dict(id=s.id, model=s.model, width=s.width, height=s.height, focal=s.focal, ppx=s.ppx, ppy=s.ppy,
                            disto=list(s.disto)))
        return out

    def poses(self):
        out = []
        for k in range(lib().r3d_sfm_num_poses(self.h)):
            s = SfmPose()
            lib().r3d_sfm_get_pose(self.h, C.c_uint32(k), C.byref(s))
            out.append(dict(id=s.id, R=np.array(list(s.rotation)).reshape(3, 3), center=np.array(list(s.center))))
        return out

    def landmarks(self, control_points=False):
        out = []
        cp = C.c_int(int(control_points))
        for k in range(lib().r3d_sfm_num_landmarks(self.h, cp)):
            n = C.c_uint32()
            lid = C.c_uint32()
            X = (C.c_double * 3)()
            lib().r3d_sfm_get_landmark(self.h, cp, C.c_uint32(k), C.byref(lid), X, None, C.c_uint32(0), C.byref(n))
            arr = (SfmObservation * max(n.value, 1))()
            lib().r3d_sfm_get_landmark(self.h, cp, C.c_uint32(k), None, None, arr, n, None)
            out.append(dict(id=lid.value, X=list(X), obs=[(arr[q].id_view, arr[q].id_feat, arr[q].x[0], arr[q].x[1])
                                                          for q in range(n.value)]))
        return out


class Tracks:
    """openMVG::tracks::STLMAPTracks handle (TracksBuilder Build + Filter + ExportToSTL)."""

    def __init__(self, handle):
        self.h = handle

    def __del__(self):
        try:
            if self.h:
                lib().r3d_tracks_free(self.h)
                self.h = None
        except Exception:
            pass

    @staticmethod
    def build(matches, min_length=2):
        h = C.c_void_p()
        rc = lib().r3d_tracks_build(matches.handle, C.c_uint32(min_length), C.byref(h))
        if rc:
            raise R3DError(rc, "r3d_tracks_build")
        return Tracks(h)

    def __len__(self):
        return int(lib().r3d_tracks_count(self.h))

    def get(self, k):
        tid, n = C.c_uint32(), C.c_uint32()
        pv, pf = C.c_void_p(), C.c_void_p()
        rc = lib().r3d_tracks_get(self.h, C.c_uint64(k), C.byref(tid), C.byref(pv), C.byref(pf), C.byref(n))
        if rc:
            raise R3DError(rc, "r3d_tracks_get")
        v = np.frombuffer((C.c_uint32 * n.value).from_address(pv.value), np.uint32).copy() if n.value else np.zeros(0, np.uint32)
        f = np.frombuffer((C.c_uint32 * n.value).from_address(pf.value), np.uint32).copy() if n.value else np.zeros(0, np.uint32)
        return tid.value, v, f

    def to_dict(self):
        """{track id: {view: feature}} like STLMAPTracks."""
        out = {}
        for k in range(len(self)):
            tid, v, f = self.get(k)
            out[tid] = dict(zip(v.tolist(), f.tolist()))
        return out

    def in_images(self, view_ids):
        ids = np.ascontiguousarray(view_ids, np.uint32)
        h = C.c_void_p()
        rc = lib().r3d_tracks_in_images(self.h, _p(ids), C.c_uint32(len(ids)), C.byref(h))
        if rc:
            raise R3DError(rc, "r3d_tracks_in_images")
        return Tracks(h)


def debug_ba_jacobian_model(model, intr, ext, pose, X, obs):
    """Host evaluation of the analytic model of any of the five camera types (no GPU needed)."""
    intr, pose, X, obs = [np.ascontiguousarray(a, np.float64) for a in (intr, pose, X, obs)]
    ext = None if ext is None else np.ascontiguousarray(ext, np.float64)
    r = np.zeros(2)
    J = np.zeros((2, 15))
    rc = lib().r3d_debug_ba_jacobian_model(C.c_int(model), _p(intr), None if ext is None else _p(ext), _p(pose), _p(X), _p(obs),
                                           _p(r), _p(J))
    if rc:
        raise R3DError(rc, "r3d_debug_ba_jacobian_model")
    return r, J


def debug_ba_prior(pose, center, weight):
    pose, center, weight = [np.ascontiguousarray(a, np.float64) for a in (pose, center, weight)]
    r = np.zeros(3)
    J = np.zeros((3, 6))
    lib().r3d_debug_ba_prior(_p(pose), _p(center), _p(weight), _p(r), _p(J))
    return r, J


def debug_ba_jacobian(intr, pose, X, obs):
    """Host evaluation of the analytic BA model (no GPU needed)."""
    intr, pose, X, obs = [np.ascontiguousarray(a, np.float64) for a in (intr, pose, X, obs)]
    r = np.zeros(2)
    J = np.zeros((2, 15))
    lib().r3d_debug_ba_jacobian(_p(intr), _p(pose), _p(X), _p(obs), _p(r), _p(J))
    return r, J


class Context:
    """r3d_ctx: one per process / GPU in bench.py; device_ids selects the CUDA devices."""

    def __init__(self, device_ids=(0,)):
        self._h = C.c_void_p()
        ids = (C.c_int * len(device_ids))(*device_ids)
        rc = lib().r3d_create(ids, len(device_ids), C.byref(self._h))
        if rc:
            raise R3DError(rc, lib().r3d_last_error(None).decode())

    def close(self):
        if self._h:
            lib().r3d_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc:
            raise R3DError(rc, lib().r3d_last_error(self._h).decode())

    def upload_regions(self, view_id, desc, xy=None):
        desc = np.ascontiguousarray(desc)
        if desc.dtype == np.float32:
            dt = R3D_F32
        elif desc.dtype == np.uint8:
            dt = R3D_U8
        else:
            raise TypeError("descriptors must be float32 or uint8")
        n, dim = (desc.shape[0], desc.shape[1]) if desc.ndim == 2 else (0, 0)
        xyp = None
        if xy is not None:
            xy = np.ascontiguousarray(xy, np.float32)
            xyp = _p(xy)
        self._check(lib().r3d_upload_regions(self._h, C.c_uint32(view_id), _p(desc), C.c_uint32(n), C.c_uint32(dim),
                                             C.c_int(dt), xyp))

    def liop_describe(self, image, keypoints, kp_size_factor=8.0):
        """image (h, w) float32; keypoints (n, 4) = x, y, size (diameter), angle (degrees) -> (n, 144) float32."""
        image = np.ascontiguousarray(image, np.float32)
        kps = np.ascontiguousarray(keypoints, np.float32).reshape(-1, 4)
        desc = np.zeros((len(kps), 144), np.float32)
        self._check(lib().r3d_liop_describe(self._h, _p(image), C.c_uint32(image.shape[1]), C.c_uint32(image.shape[0]),
                                            _p(kps), C.c_uint32(len(kps)), C.c_float(kp_size_factor), _p(desc)))
        return desc

    def debug_liop_process(self, patches):
        patches = np.ascontiguousarray(patches, np.float32).reshape(-1, 41 * 41)
        desc = np.zeros((len(patches), 144), np.float32)
        self._check(lib().r3d_debug_liop_process(self._h, _p(patches), C.c_uint32(len(patches)), _p(desc)))
        return desc

    def clear_regions(self):
        self._check(lib().r3d_clear_regions(self._h))

    def match_pairs(self, pairs, dist_ratio, flags=MATCH_DEFAULT):
        pairs = np.ascontiguousarray(pairs, np.uint32).reshape(-1, 2)
        h = C.c_void_p()
        self._check(lib().r3d_match_pairs(self._h, _p(pairs), C.c_uint64(len(pairs)), C.c_float(dist_ratio),
                                          C.c_uint32(flags), C.byref(h)))
        return Matches(h)

    def cascade_prepare(self, view_ids):
        """Hash the given (uploaded) views under their common zero-mean descriptor (R3D_MATCH_CASCADE_HASHING jobs that
        span several match_pairs calls)."""
        v = np.ascontiguousarray(view_ids, np.uint32).ravel()
        self._check(lib().r3d_cascade_prepare(self._h, _p(v), C.c_uint32(len(v))))

    def debug_cascade_view(self, view_id, n, dim):
        words = (dim + 31) // 32
        code = np.zeros((n, words), np.uint32)
        bucket = np.zeros((n, 6), np.uint16)
        ofs = np.zeros((6, 1025), np.uint32)
        ids = np.zeros((6, max(n, 1)), np.uint32)
        self._check(lib().r3d_debug_cascade_view(self._h, C.c_uint32(view_id), _p(code), _p(bucket), _p(ofs), _p(ids)))
        return code, bucket, ofs, ids[:, :n]

    def search_neighbours(self, view_db, view_query, n_query):
        idx = np.zeros((n_query, 2), np.int32)
        dist = np.zeros((n_query, 2), np.float32)
        self._check(lib().r3d_search_neighbours(self._h, C.c_uint32(view_db), C.c_uint32(view_query), _p(idx), _p(dist)))
        return idx, dist

    def debug_candidate_keys(self, view_db, view_query, n_query):
        npad = (max(n_query, 1) + 255) // 256 * 256
        keys = np.zeros((npad, 8), np.uint32)
        eps = C.c_float()
        self._check(lib().r3d_debug_candidate_keys(self._h, C.c_uint32(view_db), C.c_uint32(view_query), _p(keys), C.byref(eps)))
        return keys, eps.value

    def filter_pairs(self, putative, widths, heights, model=MODEL_F, precision_px=4.0, max_iter=2048, Ks=None):
        n = len(widths)
        views = make_views(widths, heights, Ks)
        h = C.c_void_p()
        self._check(lib().r3d_filter_pairs(self._h, C.c_int(model), C.c_double(precision_px), C.c_uint32(max_iter),
                                           putative.handle, views, C.c_uint32(n), C.byref(h)))
        return Matches(h)

    def relative_poses(self, matches, widths, heights, Ks, precision_px=math.inf, max_iter=4096, want_inliers=True):
        """robustRelativePose on every pair of `matches` (Ks: n_views x 3 = focal, ppx, ppy; focal <= 0 = no pinhole
        intrinsic).  Returns (structured array of relative_pose_dtype in map order, the AC-RANSAC inlier Matches or
        None)."""
        views = make_views(widths, heights, Ks)
        out = np.zeros(matches.num_pairs, relative_pose_dtype)
        h = C.c_void_p()
        self._check(lib().r3d_relative_poses(self._h, matches.handle, views, C.c_uint32(len(widths)), C.c_double(precision_px),
                                             C.c_uint32(max_iter), _p(out), C.byref(h) if want_inliers else None))
        return out, (Matches(h) if want_inliers else None)

    def match_timing(self):
        t = MatchTiming()
        self._check(lib().r3d_get_match_timing(self._h, C.byref(t)))
        return {k: getattr(t, k) for k, _ in MatchTiming._fields_}

    def filter_timing(self):
        t = FilterTiming()
        self._check(lib().r3d_get_filter_timing(self._h, C.byref(t)))
        return {k: getattr(t, k) for k, _ in FilterTiming._fields_}

    # ---- bundle adjustment ------------------------------------------------------------------
    @staticmethod
    def _ba_struct(p):
        s = BAProblem()
        s.n_cams = p["poses"].shape[0]
        s.n_pts = p["points"].shape[0]
        s.n_intr = p["intrinsics"].shape[0]
        s.n_obs = p["obs_xy"].shape[0]
        for k in ("poses", "intrinsics", "points", "obs_cam", "obs_pt", "cam_intr", "obs_xy"):
            setattr(s, k, p[k].ctypes.data)
        if p.get("intr_model") is not None:
            p["intr_model"] = np.ascontiguousarray(p["intr_model"], np.uint8)
            s.intr_model = p["intr_model"].ctypes.data
        if p.get("intrinsics_ext") is not None:
            p["intrinsics_ext"] = np.ascontiguousarray(p["intrinsics_ext"], np.float64)
            s.intrinsics_ext = p["intrinsics_ext"].ctypes.data
        if p.get("prior_cam") is not None and len(p["prior_cam"]):
            p["prior_cam"] = np.ascontiguousarray(p["prior_cam"], np.uint32)
            p["prior_center"] = np.ascontiguousarray(p["prior_center"], np.float64)
            p["prior_weight"] = np.ascontiguousarray(p["prior_weight"], np.float64)
            s.n_priors = len(p["prior_cam"])
            s.prior_cam = p["prior_cam"].ctypes.data
            s.prior_center = p["prior_center"].ctypes.data
            s.prior_weight = p["prior_weight"].ctypes.data
        return s

    def bundle_adjust(self, p, max_iterations=500, huber_a=16.0, refine_intrinsics=1, **tol):
        """In place on a dict of contiguous arrays (see synth.make_ba_problem / ba_prepare)."""
        o = BAOptions()
        lib().r3d_ba_default_options(C.byref(o))
        o.max_iterations = max_iterations
        o.huber_a = huber_a
        o.refine_intrinsics = refine_intrinsics
        for k, v in tol.items():
            setattr(o, k, v)
        s = self._ba_struct(p)
        summ = BASummary()
        trace = np.full(max_iterations + 1, np.nan, np.float64)
        self._check(lib().r3d_bundle_adjust(self._h, C.byref(s), C.byref(o), C.byref(summ), _p(trace)))
        d = {k: getattr(summ, k) for k, _ in BASummary._fields_}
        return d, trace[: summ.iterations + 1].copy()

    # ---- multi-GPU bundle adjustment: one process per GPU, points partitioned (sharding.partition_ba) ----
    def comm_unique_id(self):
        """Rank 0 creates the id; the host distributes it (torch.distributed.broadcast_object_list, MPI, a file)."""
        buf = (C.c_uint8 * 128)()
        self._check(lib().r3d_comm_unique_id(self._h, buf))
        return bytes(buf)

    def comm_init(self, world, rank, comm_id):
        buf = (C.c_uint8 * 128).from_buffer_copy(comm_id)
        self._check(lib().r3d_comm_init(self._h, int(world), int(rank), buf))

    def comm_destroy(self):
        self._check(lib().r3d_comm_destroy(self._h))

    @property
    def comm_world(self):
        return int(lib().r3d_comm_world(self._h))

    def ba_residuals(self, p):
        s = self._ba_struct(p)
        res = np.zeros((p["obs_xy"].shape[0], 2), np.float64)
        self._check(lib().r3d_ba_residuals(self._h, C.byref(s), _p(res)))
        return res

    # ---- the steps either side of BA on an SfmData container (SURVEY.md 8f-3) --------------------------------
    def structure_from_tracks(self, sd, tracks):
        """Tracks -> landmarks of sd, triangulated from all posed views; returns the number of rejected tracks."""
        n = C.c_uint32()
        self._check(lib().r3d_sfm_structure_from_tracks(self._h, sd.h, tracks.h, C.byref(n)))
        return n.value

    def remove_outliers(self, sd, max_pixel_residual=4.0, min_track_length=2, min_angle_deg=2.0):
        a, b = C.c_uint32(), C.c_uint32()
        self._check(lib().r3d_sfm_remove_outliers(self._h, sd.h, C.c_double(max_pixel_residual), C.c_uint32(min_track_length),
                                                  C.c_double(min_angle_deg), C.byref(a), C.byref(b)))
        return a.value, b.value

    def sfm_bundle_adjust(self, sd, max_iterations=500, refine_intrinsics=1, use_motion_priors=0, huber_a=16.0):
        class SfmBAOptions(C.Structure):
            _fields_ = [("solver", BAOptions), ("use_motion_priors", C.c_int)]
        o = SfmBAOptions()
        lib().r3d_sfm_ba_default_options(C.byref(o))
        o.solver.max_iterations = max_iterations
        o.solver.refine_intrinsics = refine_intrinsics
        o.solver.huber_a = huber_a
        o.use_motion_priors = use_motion_priors
        summ = BASummary()
        self._check(lib().r3d_sfm_bundle_adjust(self._h, sd.h, C.byref(o), C.byref(summ)))
        return {k: getattr(summ, k) for k, _ in BASummary._fields_}

    def compute_matches(self, matches_dir, basenames, widths, heights, dist_ratio=0.6, dim=144,
                        compute_fundamental=True, matching_algorithm=4, progress=None, f_filename=None,
                        compute_homography=False, compute_essential=False, Ks=None, svg_output=False):
        n = len(basenames)
        names = (C.c_char_p * n)(*[b.encode() for b in basenames])
        views = make_views(widths, heights, Ks)
        params = CMParams(dist_ratio, int(compute_fundamental), int(compute_essential), int(compute_homography),
                          matching_algorithm, dim, int(svg_output))
        paths = CMPaths(matches_dir.encode(), names, views, n, f_filename.encode() if f_filename else None, None, None)
        kp = (C.c_uint32 * n)()
        stats = CMStats()
        stats.n_views = n
        stats.number_of_keypoints = kp
        cb = PROGRESS_CB(progress) if progress else C.cast(None, PROGRESS_CB)
        self._check(lib().r3d_compute_matches(self._h, C.byref(params), C.byref(paths), cb, None, C.byref(stats)))
        d = {k: getattr(stats, k) for k, _ in CMStats._fields_ if k != "number_of_keypoints"}
        d["number_of_keypoints"] = [int(kp[k]) for k in range(n)]
        return d
