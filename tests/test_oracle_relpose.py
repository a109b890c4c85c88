"""CPU: the oracle's robustRelativePose (oracle/oracle_relpose.cpp) against independent implementations -- OpenCV's
decomposeEssentialMat / recoverPose, numpy's SVD, the scene's ground truth -- and against its own essential AC-RANSAC."""
import numpy as np
import pytest

from regard3d_b200 import synth

cv2 = pytest.importorskip("cv2")

@pytest.fixture(scope="module")
def orp():
    """the relative-pose oracle (oracle/pyoracle_relpose.py)"""
    from oracle import pyoracle_relpose
    pyoracle_relpose.build()
    return pyoracle_relpose


def _skew(t):
    return np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]])


def _Ks(sc):
    return np.array([[1.1 * max(int(w), int(h)), w / 2.0, h / 2.0] for w, h in zip(sc["widths"], sc["heights"])])


def _camera_pose(sc, c):
    """world -> camera c from the scene's own 3-D points and their (0.5 px noisy) projections (cv2.solvePnP)"""
    tid = sc["truth"][c]
    v = tid >= 0
    K = np.array([[sc["f"], 0, sc["w"] / 2.0], [0, sc["f"], sc["h"] / 2.0], [0, 0, 1]])
    ok, rv, tv = cv2.solvePnP(sc["points"][tid[v]], sc["xys"][c][v].astype(np.float64), K, None, flags=cv2.SOLVEPNP_ITERATIVE)
    assert ok
    return cv2.Rodrigues(rv)[0], tv.ravel()


def _truth_motion(sc, I, J):
    """X_J = R X_I + t of the ground truth, |t| = 1"""
    RI, tI = _camera_pose(sc, I)
    RJ, tJ = _camera_pose(sc, J)
    R = RJ @ RI.T
    t = tJ - R @ tI
    return R, t / np.linalg.norm(t)


def _bearings(xy, K):
    b = np.c_[(xy[:, 0] - K[1]) / K[0], (xy[:, 1] - K[2]) / K[0], np.ones(len(xy))]
    return b / np.linalg.norm(b, axis=1, keepdims=True)


def _angle_deg(a, b):
    c = np.clip(np.dot(a, b) / (np.linalg.norm(a) * np.linalg.norm(b)), -1.0, 1.0)
    return np.degrees(np.arccos(c))


@pytest.fixture(scope="module")
def scene(oracle):
    sc = synth.make_scene(4, 1500, 64, "msurf", seed=41)
    pairs = synth.exhaustive_pairs(4)
    ofs, m = oracle.match_pairs(sc["descs"], sc["xys"], pairs, 0.8)
    return sc, pairs, ofs, m


def _pair_xy(sc, ofs, m, k, I, J):
    mm = m[int(ofs[k]):int(ofs[k + 1])]
    return sc["xys"][I][mm["i"]].astype(np.float64), sc["xys"][J][mm["j"]].astype(np.float64), mm


def test_candidates_equal_opencv_decomposition(orp, oracle):
    rng = np.random.default_rng(3)
    for _ in range(20):
        R = synth._rodrigues(rng.normal(size=3))
        t = rng.normal(size=3)
        t /= np.linalg.norm(t)
        E = _skew(t) @ R * rng.uniform(0.1, 10.0) * rng.choice([-1.0, 1.0])
        Rs, ts = orp.motion_from_essential(E)
        R1, R2, tc = cv2.decomposeEssentialMat(E)
        want = [(R1, tc.ravel()), (R1, -tc.ravel()), (R2, tc.ravel()), (R2, -tc.ravel())]
        for Rg, tg in zip(Rs, ts):
            assert abs(np.linalg.det(Rg) - 1.0) < 1e-12 and abs(np.linalg.norm(tg) - 1.0) < 1e-12
            assert sum(np.allclose(Rg, Rw, atol=1e-9) and np.allclose(tg, tw, atol=1e-9) for Rw, tw in want) == 1
        # both rotations of the twisted pair, both signs of t, in upstream order
        assert np.allclose(Rs[0], Rs[1], atol=0) and np.allclose(Rs[2], Rs[3], atol=0)
        assert np.array_equal(ts[0], -ts[1]) and np.array_equal(ts[2], -ts[3]) and np.array_equal(ts[0], ts[2])


def test_dlt_equals_numpy_svd_nullspace(orp, oracle):
    rng = np.random.default_rng(5)
    for _ in range(50):
        R = synth._rodrigues(0.3 * rng.normal(size=3))
        t = rng.normal(size=3)
        X = rng.normal(size=3) + np.array([0, 0, 6.0])
        x1 = X / np.linalg.norm(X)
        x2 = R @ X + t
        x2 = x2 / np.linalg.norm(x2) + 1e-4 * rng.normal(size=3)      # slightly inconsistent rays: a true least squares
        P1 = np.c_[np.eye(3), np.zeros(3)]
        P2 = np.c_[R, t]
        D = np.stack([x1[0] * P1[2] - x1[2] * P1[0], x1[1] * P1[2] - x1[2] * P1[1],
                      x2[0] * P2[2] - x2[2] * P2[0], x2[1] * P2[2] - x2[2] * P2[1]])
        h = np.linalg.svd(D)[2][-1]
        want = h[:3] / h[3]
        got = orp.triangulate_dlt(R, t, x1, x2)
        assert np.linalg.norm(got - want) <= 1e-9 * np.linalg.norm(want)


def test_pose_agrees_with_truth_and_opencv(orp, oracle, scene):
    sc, pairs, ofs, m = scene
    Ks = _Ks(sc)
    n_checked = 0
    for k, (I, J) in enumerate(pairs):
        xI, xJ, _ = _pair_xy(sc, ofs, m, k, I, J)
        r, inl = orp.relative_pose(xI, xJ, sc["w"], sc["h"], sc["w"], sc["h"], np.r_[Ks[I], Ks[J]], np.inf, 4096)
        if not r["valid"]:
            continue
        n_checked += 1
        Rt, tt = _truth_motion(sc, I, J)
        R, t = r["rotation"], r["translation"]
        assert abs(np.linalg.norm(t) - 1.0) < 1e-12
        assert np.allclose(r["center"], -R.T @ t, rtol=0, atol=1e-15)
        dR = np.degrees(np.arccos(np.clip((np.trace(R @ Rt.T) - 1) / 2, -1, 1)))
        assert dR < 0.5, (I, J, dR)                                     # 0.5 px noise, ~1000 inliers
        assert _angle_deg(t, tt) < 2.0, (I, J, _angle_deg(t, tt))
        assert r["n_front"] > 0.9 * r["n_inliers"]
        # OpenCV's cheirality on the oracle's E picks the same candidate
        b1, b2 = _bearings(xI[inl], Ks[I]), _bearings(xJ[inl], Ks[J])
        p1, p2 = b1[:, :2] / b1[:, 2:], b2[:, :2] / b2[:, 2:]
        _, Rc, tc, _ = cv2.recoverPose(r["essential"], p1, p2, np.eye(3))
        assert np.allclose(R, Rc, atol=1e-6) and np.allclose(t, tc.ravel(), atol=1e-6)
    assert n_checked >= 4


def test_inliers_equal_essential_acransac(orp, oracle, scene):
    sc, pairs, ofs, m = scene
    Ks = _Ks(sc)
    for prec, iters in ((np.inf, 4096), (2.5, 256), (4.0, 2048)):
        for k, (I, J) in enumerate(pairs):
            xI, xJ, _ = _pair_xy(sc, ofs, m, k, I, J)
            Kp = np.r_[Ks[I], Ks[J]]
            r, inl = orp.relative_pose(xI, xJ, sc["w"], sc["h"], sc["w"], sc["h"], Kp, prec, iters)
            want, _, info = oracle.acransac_E(xI, xJ, sc["w"], sc["h"], sc["w"], sc["h"], Kp, prec, iters)
            assert np.array_equal(inl, want)
            assert r["n_inliers"] == len(want) and r["min_nfa"] == info[0]
            if len(want):
                assert r["found_residual_precision"] == info[1]


def test_median_angle_equals_numpy(orp, oracle, scene):
    sc, pairs, ofs, m = scene
    Ks = _Ks(sc)
    for k, (I, J) in enumerate(pairs):
        xI, xJ, _ = _pair_xy(sc, ofs, m, k, I, J)
        r, inl = orp.relative_pose(xI, xJ, sc["w"], sc["h"], sc["w"], sc["h"], np.r_[Ks[I], Ks[J]])
        if not r["valid"]:
            continue
        R, t = r["rotation"], r["translation"]
        b1, b2 = _bearings(xI[inl], Ks[I]), _bearings(xJ[inl], Ks[J])
        ang = []
        for a, b in zip(b1, b2):
            X = orp.triangulate_dlt(R, t, a, b)
            if X[2] > 0 and (R @ X + t)[2] > 0:
                ang.append(_angle_deg(a, R.T @ b))
        assert len(ang) == r["n_front"]
        med = np.partition(np.array(ang), len(ang) // 2)[len(ang) // 2]
        assert abs(med - r["median_angle_deg"]) <= 1e-12 * max(1.0, med)


def test_invalid_pairs(orp, oracle, scene):
    sc, pairs, ofs, m = scene
    Ks = _Ks(sc)
    xI, xJ, _ = _pair_xy(sc, ofs, m, 0, 0, 1)
    Kp = np.r_[Ks[0], Ks[1]]
    good, _ = orp.relative_pose(xI, xJ, sc["w"], sc["h"], sc["w"], sc["h"], Kp)
    assert good["valid"]
    bad_K = Kp.copy()
    bad_K[3] = 0.0                                                     # view J without a pinhole intrinsic
    r, inl = orp.relative_pose(xI, xJ, sc["w"], sc["h"], sc["w"], sc["h"], bad_K)
    assert not r["valid"] and len(inl) == 0 and np.isinf(r["min_nfa"])
    r, inl = orp.relative_pose(xI[:5], xJ[:5], sc["w"], sc["h"], sc["w"], sc["h"], Kp)   # <= 5 matches
    assert not r["valid"] and len(inl) == 0 and np.isinf(r["min_nfa"])
    rng = np.random.default_rng(9)
    # shuffled matches, under the E filter's bound (the unbounded mode may fit a few random matches)
    r, inl = orp.relative_pose(xI, xJ[rng.permutation(len(xJ))], sc["w"], sc["h"], sc["w"], sc["h"], Kp, 4.0, 2048)
    assert not r["valid"] and r["n_inliers"] == 0 and len(inl) == 0 and not r["min_nfa"] < 0


def test_relative_poses_over_a_map_equals_per_pair(orp, oracle, scene):
    sc, pairs, ofs, m = scene
    Ks = _Ks(sc)
    out, iofs, im = orp.relative_poses(sc["xys"], sc["widths"], sc["heights"], Ks, pairs, ofs, m, 2.5, 256)
    for k, (I, J) in enumerate(pairs):
        xI, xJ, mm = _pair_xy(sc, ofs, m, k, I, J)
        r, inl = orp.relative_pose(xI, xJ, sc["w"], sc["h"], sc["w"], sc["h"], np.r_[Ks[I], Ks[J]], 2.5, 256)
        assert out[k]["I"] == I and out[k]["J"] == J
        for f in ("valid", "n_inliers", "n_front"):
            assert out[k][f] == r[f]
        for f in ("essential", "rotation", "translation", "center", "min_nfa", "found_residual_precision", "median_angle_deg"):
            assert np.array_equal(np.asarray(out[k][f]).view(np.uint64), np.asarray(r[f]).view(np.uint64)), f
        assert np.array_equal(im[int(iofs[k]):int(iofs[k + 1])], mm[inl])
