"""LIOP-144 descriptor stage (SURVEY.md 8f-1): the oracle's restatement against THE REFERENCE ITSELF.

`r3d_vl_liopdesc_process` is the one piece of reference arithmetic on the path that compiles standalone
(the reference's src/thirdparty/liop/vl_liop.c -> oracle/_ref/libvlliop_ref.so, recipe: oracle/Makefile `ref`),
so this row of the scope table is PINNED: bit-exact against the golden vectors the compiled reference produced
(tests/golden/liop_ref_v1.npz, liop_ref_random_v1.npz), and against the compiled reference itself where it is built."""
import importlib.util
import os

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
_spec = importlib.util.spec_from_file_location("make_liop_golden", os.path.join(GOLD, "make_liop_golden.py"))
make_liop_golden = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(make_liop_golden)


def test_liop_process_equals_reference_golden(oracle):
    g = np.load(os.path.join(GOLD, "liop_ref_v1.npz"))
    assert oracle.lib().orc_liop_patch_size() == 673          # pixels within sqrt(213) of the centre of a 41x41 patch
    for k in range(len(g["patches"])):
        d = oracle.liop_process(g["patches"][k])
        assert np.array_equal(d.view(np.uint32), g["desc"][k].view(np.uint32)), "patch %d" % k


def test_liop_process_equals_compiled_reference(oracle):
    """Seeded random patches (exact ties among them: the order is the quick sort's own) against the descriptors the
    compiled reference computed for them, stored in liop_ref_random_v1.npz; where oracle/_ref is built, the reference
    is run again and must still give the stored descriptors."""
    g = np.load(os.path.join(GOLD, "liop_ref_random_v1.npz"))
    patches = make_liop_golden.random_patches()
    assert make_liop_golden.patches_sha256(patches) == str(g["patches_sha256"]), "the seeded patches changed"
    ref = g["desc"]
    if oracle.liop_ref_available():
        assert np.array_equal(oracle.liop_ref_process(patches).view(np.uint32), ref.view(np.uint32))
    for k in range(len(patches)):
        assert np.array_equal(oracle.liop_process(patches[k]).view(np.uint32), ref[k].view(np.uint32)), "patch %d" % k
    assert np.allclose(np.linalg.norm(ref, axis=1), 1.0, atol=1e-6)


def test_liop_patch_extraction_against_cv2_golden(oracle):
    """warpAffine restated: bit-exact against cv2's output; + GaussianBlur: within float round-off (OpenCV's row filter
    fuses multiply-adds on AVX2 hosts, the restatement is the plain evaluation order)."""
    g = np.load(os.path.join(GOLD, "liop_patch_cv2_v1.npz"))
    img, kps, factor = g["img"], g["kps"], float(g["factor"])
    worst = 0.0
    for k, (x, y, size, angle) in enumerate(kps):
        M = oracle.liop_affine(x, y, size, angle, factor)
        w = oracle.liop_warp(img, M)
        assert np.array_equal(w.view(np.uint32), g["warped"][k].view(np.uint32)), "warp of keypoint %d" % k
        b = oracle.liop_blur(w)
        worst = max(worst, float(np.max(np.abs(b - g["blurred"][k]))))
    assert worst <= 4e-7 * float(np.max(np.abs(g["blurred"]))) + 1e-12, worst


def test_liop_describe_pipeline(oracle):
    g = np.load(os.path.join(GOLD, "liop_patch_cv2_v1.npz"))
    desc, patches = oracle.liop_describe(g["img"], g["kps"], float(g["factor"]), want_patches=True)
    assert desc.shape == (len(g["kps"]), 144)
    for k in (0, 5, 17):
        assert np.array_equal(desc[k], oracle.liop_process(patches[k]))
    # descriptors from cv2's own patches: LIOP is order based, round-off in the blur rarely moves a rank
    same = sum(np.array_equal(oracle.liop_process(g["blurred"][k]), desc[k]) for k in range(len(desc)))
    assert same >= 0.9 * len(desc), same
