"""-m gpu: r3d_relative_poses (essential AC-RANSAC + pose from E + initial-pair score) through the C ABI against the CPU
oracle: identical inlier sequences, equal counts, bit-identical E / R / t / C / minNFA / precision / median angle."""
import os

import numpy as np
import pytest

from regard3d_b200 import synth

pytestmark = pytest.mark.gpu

INT_FIELDS = ("valid", "n_inliers", "n_front")
BIT_FIELDS = ("essential", "rotation", "translation", "center", "min_nfa", "found_residual_precision", "median_angle_deg")



def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def _Ks(sc):
    return np.array([[1.1 * max(int(w), int(h)), w / 2.0, h / 2.0] for w, h in zip(sc["widths"], sc["heights"])])


def _upload(ctx, sc):
    ctx.clear_regions()
    for v, (d, x) in enumerate(zip(sc["descs"], sc["xys"])):
        ctx.upload_regions(v, d, x)


def _compare(ctx, oracle, r3dlib, sc, pairs, ofs, m, Ks, precision_px, max_iter):
    from oracle import pyoracle_relpose as orp     # the relative-pose oracle (its own library)
    put = r3dlib.Matches.from_csr(pairs, ofs, m)
    got, inl = ctx.relative_poses(put, sc["widths"], sc["heights"], Ks, precision_px, max_iter)
    exp, eofs, em = orp.relative_poses(sc["xys"], sc["widths"], sc["heights"], Ks, pairs, ofs, m, precision_px, max_iter)
    by_pair = {(int(r["I"]), int(r["J"])): r for r in got}
    inl = inl.to_dict()
    for k, (I, J) in enumerate(pairs):
        e = exp[k]
        g = by_pair.get((int(I), int(J)))
        seq = em[int(eofs[k]):int(eofs[k + 1])]
        if g is None:              # a pair without putatives is not in the map
            assert int(ofs[k + 1] - ofs[k]) == 0
            continue
        for f in INT_FIELDS:
            assert g[f] == e[f], ((I, J), f, g[f], e[f])
        for f in BIT_FIELDS:
            assert np.array_equal(np.asarray(g[f]).view(np.uint64), np.asarray(e[f]).view(np.uint64)), ((I, J), f, g[f], e[f])
        gi = inl.get((int(I), int(J)))
        if len(seq) == 0:
            assert gi is None
        else:
            assert gi is not None and np.array_equal(gi, seq), (I, J)
    assert len(inl) == sum(1 for k in range(len(pairs)) if eofs[k + 1] > eofs[k])
    return got, inl


def _outlier_map(sc, oracle, ratio, seed):
    """putatives of an exhaustive scene: pair 0 with 40 % gross outliers, pair 1 hopeless (shuffled), pair 2 tiny (12)"""
    pairs = synth.exhaustive_pairs(len(sc["xys"]))
    ofs, m = oracle.match_pairs(sc["descs"], sc["xys"], pairs, ratio)
    rng = np.random.default_rng(seed)
    m2 = m.copy()
    s0 = slice(int(ofs[0]), int(ofs[1]))
    bad = rng.random(int(ofs[1] - ofs[0])) < 0.4
    j0 = m2["j"][s0].copy()
    j0[bad] = rng.integers(0, len(sc["xys"][1]), bad.sum())
    m2["j"][s0] = j0
    s1 = slice(int(ofs[1]), int(ofs[2]))
    m2["j"][s1] = rng.permutation(m2["j"][s1])
    keep = np.ones(len(m2), bool)
    keep[int(ofs[2]) + 12:int(ofs[3])] = False
    new_ofs = np.zeros_like(ofs)
    for k in range(len(pairs)):
        new_ofs[k + 1] = new_ofs[k] + keep[int(ofs[k]):int(ofs[k + 1])].sum()
    return pairs, new_ofs, m2[keep]


def test_relative_poses_clean_scene(gpu_ctx, oracle, r3dlib):
    sc = synth.make_scene(4, 2000, 64, "msurf", seed=31)
    pairs = synth.exhaustive_pairs(4)
    _upload(gpu_ctx, sc)
    ofs, m = oracle.match_pairs(sc["descs"], sc["xys"], pairs, 0.6)
    got, _ = _compare(gpu_ctx, oracle, r3dlib, sc, pairs, ofs, m, _Ks(sc), np.inf, 4096)
    assert got["valid"].sum() >= 4
    t = gpu_ctx.filter_timing()
    assert t["kernel_launches"] >= 3 and t["ms_device_total"] >= t["ms_score"] > 0


@pytest.mark.parametrize("precision_px,max_iter", [(np.inf, 4096), (np.inf, 256), (2.5, 256), (2.5, 4096), (4.0, 4096), (4.0, 256)])
def test_relative_poses_outliers_hopeless_tiny(gpu_ctx, oracle, r3dlib, precision_px, max_iter):
    sc = synth.make_scene(4, 1500, 64, "msurf", seed=32)
    _upload(gpu_ctx, sc)
    pairs, ofs, m = _outlier_map(sc, oracle, 0.8, 1)
    Ks = _Ks(sc)
    Ks[3, 0] = 0.0                                      # view 3 has no pinhole intrinsic: its pairs are invalid
    got, _ = _compare(gpu_ctx, oracle, r3dlib, sc, pairs, ofs, m, Ks, precision_px, max_iter)
    assert not any(r["valid"] for r in got if 3 in (r["I"], r["J"]))
    assert not got[2]["valid"]                          # 12 matches: too few for 2.5 x 5 inliers after any fit


def _big_pair_scene(n_feat, seed):
    """two views; putatives = every shared point (true) plus 25 % random ones, in a random order"""
    sc = synth.make_scene(2, n_feat, 8, "msurf", seed=seed, n_points=int(n_feat * 1.2))
    t0, t1 = sc["truth"]
    pos1 = {int(p): k for k, p in enumerate(t1) if p >= 0}
    i = np.array([k for k, p in enumerate(t0) if p >= 0 and int(p) in pos1], np.uint32)
    j = np.array([pos1[int(t0[k])] for k in i], np.uint32)
    rng = np.random.default_rng(seed)
    n_bad = len(i) // 4
    i = np.r_[i, rng.integers(0, n_feat, n_bad).astype(np.uint32)]
    j = np.r_[j, rng.integers(0, n_feat, n_bad).astype(np.uint32)]
    order = rng.permutation(len(i))
    m = np.zeros(len(i), [("i", np.uint32), ("j", np.uint32)])
    m["i"], m["j"] = i[order], j[order]
    return sc, m


@pytest.mark.parametrize("n_feat,lo,hi", [(14000, 8193, 16384), (30000, 16385, 10 ** 6)])
def test_relative_poses_large_size_classes(gpu_ctx, oracle, r3dlib, n_feat, lo, hi):
    sc, m = _big_pair_scene(n_feat, 60 + n_feat % 7)
    assert lo <= len(m) <= hi, len(m)                   # the 16384 shared-memory class / the huge (global scratch) class
    _upload(gpu_ctx, sc)
    pairs = np.array([[0, 1]], np.uint32)
    ofs = np.array([0, len(m)], np.uint64)
    for precision_px in (np.inf, 4.0):
        got, _ = _compare(gpu_ctx, oracle, r3dlib, sc, pairs, ofs, m, _Ks(sc), precision_px, 256)
        assert got[0]["valid"]


def test_inliers_equal_the_essential_filter(gpu_ctx, oracle, r3dlib):
    sc = synth.make_scene(4, 1500, 64, "msurf", seed=33)
    _upload(gpu_ctx, sc)
    pairs, ofs, m = _outlier_map(sc, oracle, 0.8, 4)
    put = r3dlib.Matches.from_csr(pairs, ofs, m)
    Ks = _Ks(sc)
    for precision_px, max_iter in ((4.0, 2048), (2.5, 256)):
        _, inl = gpu_ctx.relative_poses(put, sc["widths"], sc["heights"], Ks, precision_px, max_iter)
        f = gpu_ctx.filter_pairs(put, sc["widths"], sc["heights"], model=r3dlib.MODEL_E, precision_px=precision_px,
                                 max_iter=max_iter, Ks=Ks).to_dict()
        inl = inl.to_dict()
        assert sorted(inl) == sorted(f)
        for k in f:
            assert np.array_equal(inl[k], f[k]), k


def test_host_round_path_is_unsupported(gpu_ctx, oracle, r3dlib):
    sc = synth.make_scene(3, 800, 32, "msurf", seed=34)
    pairs = synth.exhaustive_pairs(3)
    _upload(gpu_ctx, sc)
    ofs, m = oracle.match_pairs(sc["descs"], sc["xys"], pairs, 0.8)
    put = r3dlib.Matches.from_csr(pairs, ofs, m)
    os.environ["R3D_FILTER_HOST_ROUNDS"] = "1"
    try:
        with pytest.raises(r3dlib.R3DError) as ei:
            gpu_ctx.relative_poses(put, sc["widths"], sc["heights"], _Ks(sc))
        assert ei.value.code == -5
    finally:
        del os.environ["R3D_FILTER_HOST_ROUNDS"]
    gpu_ctx.relative_poses(put, sc["widths"], sc["heights"], _Ks(sc))   # and the device path works again


@pytest.mark.skipif(_n_gpus() < 2, reason="needs two GPUs in one box")
def test_two_devices_equal_one_device(r3dlib, oracle):
    sc = synth.make_scene(5, 1500, 64, "msurf", seed=35)
    pairs = synth.exhaustive_pairs(5)
    ofs, m = oracle.match_pairs(sc["descs"], sc["xys"], pairs, 0.8)
    res = {}
    for devs in ((0,), (0, 1)):
        ctx = r3dlib.Context(devs)
        _upload(ctx, sc)
        res[devs] = _compare(ctx, oracle, r3dlib, sc, pairs, ofs, m, _Ks(sc), np.inf, 4096)[0]
        ctx.close()
    assert res[(0,)].tobytes() == res[(0, 1)].tobytes()
