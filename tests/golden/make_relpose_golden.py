#!/usr/bin/env python
"""Generates tests/golden/relpose_v1.json from the CPU oracle's relative poses (robustRelativePose on every pair).

    python tests/golden/make_relpose_golden.py      # rewrites relpose_v1.json

Content: for one seeded synthetic scene (regard3d_b200/synth.py) and a few (precision, iterations) settings, per pair:
valid, n_inliers, n_front, the SHA-1 of the AC-RANSAC inlier (i, j) sequence and the SHA-1 of the bytes of
(E, R, t, C, minNFA, found residual precision, median angle)."""
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), "..", ".."))
sys.path.insert(0, ROOT)

SCENE = dict(n_img=4, n_feat=1500, dim=64, kind="msurf", seed=111, ratio=0.8)
SETTINGS = [(float("inf"), 4096), (2.5, 256), (4.0, 2048)]
POSE_FIELDS = ("essential", "rotation", "translation", "center", "min_nfa", "found_residual_precision", "median_angle_deg")


def seq_hash(m):
    a = np.stack([np.asarray(m["i"], np.uint32), np.asarray(m["j"], np.uint32)], 1) if len(m) else np.zeros((0, 2), np.uint32)
    return hashlib.sha1(np.ascontiguousarray(a).tobytes()).hexdigest()


def pose_hash(r):
    return hashlib.sha1(b"".join(np.ascontiguousarray(r[f], np.float64).tobytes() for f in POSE_FIELDS)).hexdigest()


def row(r, inl):
    return [int(r["I"]), int(r["J"]), int(r["valid"]), int(r["n_inliers"]), int(r["n_front"]), seq_hash(inl), pose_hash(r)]


def scene_inputs():
    from oracle import pyoracle as po
    from regard3d_b200 import synth
    d = SCENE
    sc = synth.make_scene(d["n_img"], d["n_feat"], d["dim"], d["kind"], seed=d["seed"])
    pairs = synth.exhaustive_pairs(d["n_img"])
    ofs, m = po.match_pairs(sc["descs"], sc["xys"], pairs, d["ratio"])
    Ks = np.array([[1.1 * max(int(w), int(h)), w / 2.0, h / 2.0] for w, h in zip(sc["widths"], sc["heights"])])
    return sc, pairs, ofs, m, Ks


def build_all():
    from oracle import pyoracle_relpose as por
    sc, pairs, ofs, m, Ks = scene_inputs()
    out = []
    for prec, iters in SETTINGS:
        rp, iofs, im = por.relative_poses(sc["xys"], sc["widths"], sc["heights"], Ks, pairs, ofs, m, prec, iters)
        out.append({"precision_px": "inf" if np.isinf(prec) else prec, "max_iter": iters,
                    "pairs": [row(rp[k], im[int(iofs[k]):int(iofs[k + 1])]) for k in range(len(pairs))]})
    return {"scene": SCENE, "settings": out}


if __name__ == "__main__":
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "relpose_v1.json")
    with open(path, "w") as f:
        json.dump(build_all(), f, indent=1)
    print(path)
