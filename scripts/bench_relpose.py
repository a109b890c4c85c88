#!/usr/bin/env python
"""Relative poses of every pair on one GPU: the input of the global SfM engine (matches.e.txt) through
r3d_relative_poses, with a CPU oracle baseline and an A/B of the F / E filter kernels against another build.

    python scripts/bench_relpose.py --out DIR [--configs c2,c3] [--ab-lib OTHER/libr3dgpu.so] [--profile]

Per config (C2: 50 x 10k LIOP-144, 1225 pairs; C3: 200 x 20k SIFT-u8, 19900 pairs): putative matching, the E filter
(4 px, 2048 iterations) -> the E map, then r3d_relative_poses(+inf, 4096) on it, timed with the device synchronised.
One JSON line per config goes to stdout and DIR/relpose.jsonl:
  * GPU name and power limit (read in the same process), pairs/s of the call;
  * the AC-RANSAC kernel time (filter timing ms_score) and the pose kernels' time (ms_device_total - ms_score);
  * FP64 operations per inlier of the pose kernel, counted from its shapes (Jacobi sweeps counted at a nominal 4),
    and the resulting FP64 rate;
  * the CPU oracle on a fixed sample of pairs (OpenMP, core count stated) and bit parity of the GPU on that sample.
--ab-lib: the F and E filter legs of this build and of the other one, alternated in fresh processes (C2).
--profile: a separate run of the C2 call under torch.profiler; the kernel times it attributes go to DIR/profile.json.
Writes nothing outside DIR (and a temporary directory)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)

CONFIGS = {
    "c2": dict(images=50, feats=10000, dim=144, kind="liop", u8=False, seed=2, name="C2 (LIOP-144)"),
    "c3": dict(images=200, feats=20000, dim=128, kind="sift", u8=True, seed=3, name="C3 (SIFT-u8)"),
}
RATIO = 0.8
SAMPLE_PAIRS = 24
SWEEPS = 4   # nominal one-sided Jacobi sweeps of a 4x4 DLT system (the kernel stops at orthogonality, <= 12)


def fp64_ops_per_inlier():
    """FP64 operations of k_relpose per inlier, from its shapes (relpose_math.cuh)."""
    bearing = 2 * 12
    rotation = 3 * 4 * 2 + 12 + 2 * 4 * 6 + 2 * 4 * 6      # 3 dot products of 4, rotation parameters, 2 columns of D and V
    dlt = 16 + 6 * SWEEPS * rotation + 4 * 7 + 3 + 6 + 2   # design rows, sweeps, column norms, hnormalize, 2 depths
    angle = 15 + 2 * 6 + 6 + 5 + 2 * 6 + 3 + 60            # R^T b2, norms, division, acos_det (series)
    return bearing + 4 * dlt + angle


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, pl = [s.strip() for s in q.split(",")]
        return {"gpu": name, "power_limit": pl}
    except Exception as e:  # the number is still the card's; say that its name could not be read
        return {"gpu": "unknown (%s)" % e, "power_limit": "unknown"}


def make_scene(cfg):
    from regard3d_b200 import synth
    sc = synth.make_scene(cfg["images"], cfg["feats"], cfg["dim"], cfg["kind"], seed=20260924 + cfg["seed"], as_u8=cfg["u8"])
    Ks = np.array([[1.1 * max(int(w), int(h)), w / 2.0, h / 2.0] for w, h in zip(sc["widths"], sc["heights"])])
    return sc, synth.exhaustive_pairs(cfg["images"]), Ks


def e_map(ctx, capi, sc, pairs, Ks):
    for v in range(len(sc["xys"])):
        ctx.upload_regions(v, sc["descs"][v], sc["xys"][v])
    put = ctx.match_pairs(pairs, RATIO)
    return put, ctx.filter_pairs(put, sc["widths"], sc["heights"], model=capi.MODEL_E, precision_px=4.0, max_iter=2048, Ks=Ks)


def run_config(key, out_dir, n_threads):
    import torch
    from regard3d_b200 import capi
    from oracle import pyoracle_relpose as por
    cfg = CONFIGS[key]
    info = gpu_info()
    sc, pairs, Ks = make_scene(cfg)
    ctx = capi.Context((0,))
    _, em = e_map(ctx, capi, sc, pairs, Ks)
    ctx.relative_poses(em, sc["widths"], sc["heights"], Ks)          # warm-up of every shape
    times, tms = [], []
    for _ in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rp, _ = ctx.relative_poses(em, sc["widths"], sc["heights"], Ks, want_inliers=False)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
        tms.append(ctx.filter_timing())
    best = int(np.argmin(times))
    T = tms[best]
    inliers = int(rp["n_inliers"].sum())
    ms_pose = T["ms_device_total"] - T["ms_score"]
    ops = fp64_ops_per_inlier()
    # CPU oracle on a fixed sample of the E map's pairs, and the GPU on the same sample
    pairs_e, ofs_e, m_e = em.export_csr()
    rng = np.random.default_rng(7)
    pick = np.sort(rng.choice(len(pairs_e), min(SAMPLE_PAIRS, len(pairs_e)), replace=False))
    sp = pairs_e[pick]
    chunks = [m_e[int(ofs_e[k]):int(ofs_e[k + 1])] for k in pick]
    sofs = np.zeros(len(pick) + 1, np.uint64)
    sofs[1:] = np.cumsum([len(c) for c in chunks])
    sm = np.concatenate(chunks)
    t0 = time.perf_counter()
    orp, _, _ = por.relative_poses(sc["xys"], sc["widths"], sc["heights"], Ks, sp, sofs, sm, np.inf, 4096, n_threads=n_threads)
    t_cpu = time.perf_counter() - t0
    grp, _ = ctx.relative_poses(capi.Matches.from_csr(sp, sofs, sm), sc["widths"], sc["heights"], Ks, want_inliers=False)
    parity = bool(grp.tobytes() == orp.tobytes())
    ctx.close()
    line = dict(info, config=cfg["name"], images=cfg["images"], feats=cfg["feats"], putative_pairs=len(pairs),
                e_pairs=int(em.num_pairs), e_matches=int(em.total), call_s=times[best], pairs_per_s=em.num_pairs / times[best],
                valid_pairs=int(rp["valid"].sum()), inliers=inliers, ms_acransac=T["ms_score"], ms_pose_kernels=ms_pose,
                fp64_ops_per_inlier=ops, pose_fp64_gflops=(ops * inliers / (ms_pose * 1e-3) / 1e9) if ms_pose > 0 else None,
                cpu_oracle=dict(pairs=len(pick), threads=n_threads or os.cpu_count(), cores=os.cpu_count(), s=t_cpu,
                                pairs_per_s=len(pick) / t_cpu, bit_parity_with_gpu=parity))
    return line


def filter_leg(key):
    """one A/B leg (fresh process, R3D_LIB picks the build): F and E filter kernel times on the config's putatives"""
    from regard3d_b200 import capi
    sc, pairs, Ks = make_scene(CONFIGS[key])
    ctx = capi.Context((0,))
    for v in range(len(sc["xys"])):
        ctx.upload_regions(v, sc["descs"][v], sc["xys"][v])
    put = ctx.match_pairs(pairs, RATIO)
    res = {}
    for name, model in (("F", capi.MODEL_F), ("E", capi.MODEL_E)):
        ctx.filter_pairs(put, sc["widths"], sc["heights"], model=model, Ks=Ks)      # warm-up
        f = ctx.filter_pairs(put, sc["widths"], sc["heights"], model=model, Ks=Ks)
        res[name] = dict(ms_kernel=ctx.filter_timing()["ms_score"], pairs=f.num_pairs, matches=f.total)
    ctx.close()
    print(json.dumps(res))


def profile_c2(out_dir):
    import torch
    from torch.profiler import ProfilerActivity, profile
    from regard3d_b200 import capi
    sc, pairs, Ks = make_scene(CONFIGS["c2"])
    ctx = capi.Context((0,))
    _, em = e_map(ctx, capi, sc, pairs, Ks)
    ctx.relative_poses(em, sc["widths"], sc["heights"], Ks)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ctx.relative_poses(em, sc["widths"], sc["heights"], Ks, want_inliers=False)
        torch.cuda.synchronize()
    k = {}
    for e in prof.events():
        if str(e.device_type).endswith("CUDA") and ("relpose" in e.name or "acransac_fused" in e.name):
            nm = "k_relpose" if "relpose" in e.name else "k_acransac_fused"
            us = getattr(e, "device_time", None)
            k[nm] = k.get(nm, 0.0) + (us if us is not None else e.cuda_time) / 1e3
    line = dict(gpu_info(), config="C2 (LIOP-144)", profiler_kernel_ms=k, filter_timing=ctx.filter_timing())
    ctx.close()
    with open(os.path.join(out_dir, "profile.json"), "w") as f:
        json.dump(line, f, indent=1)
    return line


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True)
    ap.add_argument("--configs", default="c2,c3")
    ap.add_argument("--ab-lib", default=None, help="another build of libr3dgpu.so for the F / E filter A/B (C2)")
    ap.add_argument("--ab-rounds", type=int, default=3)
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--cpu-threads", type=int, default=0)
    ap.add_argument("--filter-leg", default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.filter_leg:
        filter_leg(a.filter_leg)
        return
    os.makedirs(a.out, exist_ok=True)
    lines = []

    def emit(line):
        lines.append(line)
        print(json.dumps(line), flush=True)
        with open(os.path.join(a.out, "relpose.jsonl"), "a") as f:
            f.write(json.dumps(line) + "\n")

    for key in a.configs.split(","):
        if key:
            emit(run_config(key.strip(), a.out, a.cpu_threads))
    if a.ab_lib:
        legs = {"this": [], "other": []}
        for r in range(a.ab_rounds):
            for who in (("this", "other") if r % 2 == 0 else ("other", "this")):
                env = dict(os.environ)
                env.pop("R3D_LIB", None)
                if who == "other":
                    env["R3D_LIB"] = os.path.abspath(a.ab_lib)
                p = subprocess.run([sys.executable, os.path.abspath(__file__), "--out", a.out, "--filter-leg", "c2"], env=env,
                                   capture_output=True, text=True, check=True)
                legs[who].append(json.loads(p.stdout.strip().splitlines()[-1]))
        ab = dict(gpu_info(), ab="F / E filter kernel ms on C2, alternated legs", this=legs["this"], other=legs["other"])
        emit(ab)
    if a.profile:
        emit(profile_c2(a.out))


if __name__ == "__main__":
    main()
