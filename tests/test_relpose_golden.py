"""Committed relative-pose fixtures (tests/golden/relpose_v1.json, made by tests/golden/make_relpose_golden.py): the
CPU test pins the oracle against drift, the GPU test holds r3d_relative_poses to the same committed hashes."""
import importlib.util
import json
import os

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = json.load(open(os.path.join(HERE, "golden", "relpose_v1.json")))
_spec = importlib.util.spec_from_file_location("make_relpose_golden", os.path.join(HERE, "golden", "make_relpose_golden.py"))
mk = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(mk)


def test_oracle_reproduces_the_relpose_fixtures(oracle):
    assert mk.build_all() == GOLD


@pytest.mark.gpu
def test_gpu_relative_poses_reproduce_the_fixtures(gpu_ctx, r3dlib, oracle):
    sc, pairs, ofs, m, Ks = mk.scene_inputs()
    gpu_ctx.clear_regions()
    for v in range(len(sc["xys"])):
        gpu_ctx.upload_regions(v, sc["descs"][v], sc["xys"][v])
    put = r3dlib.Matches.from_csr(pairs, ofs, m)
    for s in GOLD["settings"]:
        prec = np.inf if s["precision_px"] == "inf" else float(s["precision_px"])
        rp, inl = gpu_ctx.relative_poses(put, sc["widths"], sc["heights"], Ks, prec, s["max_iter"])
        inl = inl.to_dict()
        empty = np.zeros(0, r3dlib.indmatch_dtype)
        rows = [mk.row(r, inl.get((int(r["I"]), int(r["J"])), empty)) for r in rp]
        assert rows == s["pairs"], s["precision_px"]
