"""ctypes wrapper of the CPU ORACLE's relative poses (oracle/_build/liboracle_relpose.so, built by oracle/relpose.mk).

TEST INFRASTRUCTURE ONLY -- importable from tests/, __graft_entry__.smoke() and scripts/bench_relpose.py's CPU leg.
The product package (regard3d_b200) never imports this.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from oracle.pyoracle import _p, _ptr_array, indmatch_dtype

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "_build", "liboracle_relpose.so")

# the layout of orc_relpose / r3d_relative_pose
relative_pose_dtype = np.dtype({
    "names": ["I", "J", "valid", "n_inliers", "n_front", "min_nfa", "found_residual_precision", "essential", "rotation",
              "translation", "center", "median_angle_deg"],
    "formats": [np.uint32, np.uint32, np.int32, np.uint32, np.uint32, np.float64, np.float64, (np.float64, (3, 3)),
                (np.float64, (3, 3)), (np.float64, 3), (np.float64, 3), np.float64],
    "offsets": [0, 4, 8, 12, 16, 24, 32, 40, 112, 184, 208, 232],
    "itemsize": 240,
})

_lib = None


def build():
    """Compile the relative-pose oracle with its committed makefile (make tracks the sources)."""
    subprocess.check_call(["make", "-C", _HERE, "-s", "-f", "relpose.mk"])
    return _LIB_PATH


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_LIB_PATH)
        _lib.orc_relative_poses.restype = C.c_int64
    return _lib


def relative_pose(xI, xJ, wI, hI, wJ, hJ, Kpair, precision_px=np.inf, max_iter=4096):
    """robustRelativePose of one pair -> (record of relative_pose_dtype, AC-RANSAC inlier indices)."""
    xI = np.ascontiguousarray(xI, np.float64)
    xJ = np.ascontiguousarray(xJ, np.float64)
    Kpair = np.ascontiguousarray(Kpair, np.float64)
    M = xI.shape[0]
    out = np.zeros(1, relative_pose_dtype)
    inl = np.zeros(max(M, 1), np.uint32)
    lib().orc_relative_pose(_p(xI), _p(xJ), C.c_uint32(M), C.c_uint32(wI), C.c_uint32(hI), C.c_uint32(wJ), C.c_uint32(hJ),
                            _p(Kpair), C.c_double(precision_px), C.c_uint32(max_iter), _p(out), _p(inl))
    return out[0], inl[:int(out[0]["n_inliers"])].copy()


def relative_poses(xys, widths, heights, Ks, pairs, put_ofs, put, precision_px=np.inf, max_iter=4096, n_threads=0):
    """robustRelativePose on every pair of a CSR map -> (relative_pose_dtype[P], inlier ofs[P+1], inlier matches)."""
    xys = [np.ascontiguousarray(x, np.float32) for x in xys]
    pairs = np.ascontiguousarray(pairs, np.uint32).reshape(-1, 2)
    P = pairs.shape[0]
    widths = np.ascontiguousarray(widths, np.uint32)
    heights = np.ascontiguousarray(heights, np.uint32)
    Ks = np.ascontiguousarray(Ks, np.float64)
    put_ofs = np.ascontiguousarray(put_ofs, np.uint64)
    put = np.ascontiguousarray(put, indmatch_dtype)
    out = np.zeros(P, relative_pose_dtype)
    inl = np.zeros(max(1, put.shape[0]), indmatch_dtype)
    inl_ofs = np.zeros(P + 1, np.uint64)
    n = lib().orc_relative_poses(_ptr_array(xys), _p(widths), _p(heights), _p(Ks), C.c_uint32(len(xys)), _p(pairs),
                                 C.c_uint64(P), _p(put_ofs), _p(put), C.c_double(precision_px), C.c_uint32(max_iter), _p(out),
                                 _p(inl_ofs), _p(inl), C.c_int(n_threads))
    return out, inl_ofs, inl[:n].copy()


def motion_from_essential(E):
    """MotionFromEssential -> (R[4, 3, 3], t[4, 3]) in upstream candidate order."""
    E = np.ascontiguousarray(E, np.float64)
    R = np.zeros((4, 3, 3))
    t = np.zeros((4, 3))
    lib().orc_motion_from_essential(_p(E), _p(R), _p(t))
    return R, t


def triangulate_dlt(R, t, x1, x2):
    R, t, x1, x2 = [np.ascontiguousarray(a, np.float64) for a in (R, t, x1, x2)]
    X = np.zeros(3)
    lib().orc_triangulate_dlt(_p(R), _p(t), _p(x1), _p(x2), _p(X))
    return X
