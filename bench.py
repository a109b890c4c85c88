#!/usr/bin/env python
"""bench.py -- matched image-pairs / second on the compute-matches hot path (BASELINE.json metric).

    python bench.py [--gpus N --steps K --warmup W] [--impl reference] [--workload c3|c2|c2-msurf64|c4|c4-exact] [--matcher exact|cascade]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (default): BASELINE.json configs[2] = **C3**, the configuration the north_star target is quoted on:
200 synthetic images x 20 000 SIFT-128 uint8 descriptors, exhaustive pairs (19 900), brute-force L2 2-NN +
ratio 0.6 + (i,j) and coordinate de-duplication.  It fits one B200 (0.5 GB of descriptors + 1.4 GB of fp16
operands), so N = 1 runs the whole set.  One step = one pass over ALL 19 900 pairs.

N > 1 = STRONG scaling of that one set: every rank holds the regions its shard touches, the I-sorted pair list
is cut into cost-balanced contiguous ranges (regard3d_b200/sharding.py, SURVEY.md 8e), no data-path collective;
the per-rank PairWiseMatches are gathered to rank 0 IN PAIR ORDER INSIDE THE TIMED REGION (sharding.Gather: CSR export
straight into a shared-memory segment rank 0 owns, or -- R3D_GATHER=p2p -- pinned -> NCCL send/recv over NVLink ->
rank 0's pinned host buffer), so the clock stops when rank 0 holds every match list in host memory -- the
reference's `map_PutativesMatches` (src/R3DComputeMatches.cpp:437-488).
--workload c4 = BASELINE configs[3] as named: 500 images, OpenMVG's cascade-hashing matcher (hashing of all views inside
the step) + the F filter; c4-exact = the same images through the exact tensor-core matcher.

value : pairs/s, descriptors already resident in HBM (r3d_match_pairs on the shard + gather).
e2e   : pairs/s through the C ABI from pinned HOST buffers: r3d_clear_regions + r3d_upload_regions of every view
        the shard touches + r3d_match_pairs + gather, every step.
roofline : the tcgen05 candidate kernel, algorithmic 2*N_I*N_J*D flop per pair (SURVEY.md 8d) over its
        CUDA-event time on its own stream, against MEASURED_PEAKS.json bf16 TFLOP/s.
cpu_baseline : the oracle port on a bounded sample of the same pairs with all usable host threads (N = 1 only).
f_filter / ba : the F AC-RANSAC leg over the step's putatives and the C5 bundle adjustment, reported alongside.
--impl reference : the reference's CPU path (oracle port; the reference itself cannot be built here) on a
        bounded sample of the same workload per step, explicit OMP team = the usable CPUs (torchrun exports
        OMP_NUM_THREADS=1, which is ignored on purpose).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

RATIO = 0.6
WORKLOADS = {
    "c2": dict(images=50, feats=10000, dim=144, kind="liop", u8=False, name="C2 (LIOP-144)", seed=2),
    "c2-msurf64": dict(images=50, feats=10000, dim=64, kind="msurf", u8=False, name="C2 (MSURF-64 = AKAZE-float)", seed=2),
    "c3": dict(images=200, feats=20000, dim=128, kind="sift", u8=True, name="C3", seed=3),
    "c4": dict(images=500, feats=10000, dim=128, kind="sift", u8=True, name="C4 (cascade hashing + F filter)", seed=4,
               matcher="cascade"),
    "c4-exact": dict(images=500, feats=10000, dim=128, kind="sift", u8=True, name="C4 images, exact matcher + F filter", seed=4),
}
METRIC = "matched_image_pairs_per_sec_exhaustive"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); smax.append(float(f[1])); power.append(float(f[2]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[3 + k].lower().startswith("active"):
                    reasons.add(nm)
        if not sm:  # the region was shorter than one sampling period: one synchronous reading
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=clocks.sm,clocks.max.sm,power.draw",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=10).stdout
                f = [x.strip() for x in out.strip().split(",")]
                sm.append(float(f[0])); smax.append(float(f[1])); power.append(float(f[2]))
            except Exception:
                pass
        med = float(np.median([x for x in sm if x >= 0.5 * max(sm)])) if sm else None  # "under load" samples
        return {"sm_mhz": med, "sm_max_mhz": max(smax) if smax else None, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power) if power else None}


def effective_cpus():
    """Host CPUs this process may actually use: the affinity mask, cut by the cgroup CPU-time quota (the GPU boxes
    give a container ~16 CPUs of quota per GPU although 128 hardware threads are visible)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            n = min(n, max(1, int(round(int(q) / int(per)))))
    except Exception:
        pass
    return n


def measured_traffic_per_pair(wl_key):
    """DRAM bytes per image pair of the candidate kernel, from the committed `ncu --set full` capture of one
    batch launch of THIS workload (profiles/*_keymetrics.csv: dram__bytes_read/write + the pairs the launch held);
    None when no capture of this workload is committed."""
    name = {"c3": "r02_k_l2_candidates_2sm_c3_keymetrics.csv", "c2": "r01_k_l2_candidates_2sm_keymetrics.csv"}.get(wl_key)
    if not name:
        return None, None
    p = os.path.join(ROOT, "profiles", name)
    if not os.path.exists(p):
        return None, None
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    tot, pairs = 0.0, 128.0
    import csv
    for f in csv.reader(open(p)):
        if len(f) >= 4 and f[1] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            tot += float(f[2]) * unit.get(f[3], 1.0)
        if len(f) >= 3 and f[1] == "pairs_in_launch":
            pairs = float(f[2])
    return (tot / pairs if tot else None), "profiles/" + name


def make_workload(wl):
    from regard3d_b200 import synth
    sc = synth.make_scene(wl["images"], wl["feats"], wl["dim"], wl["kind"], seed=20260924 + wl["seed"], as_u8=wl["u8"])
    return sc, synth.exhaustive_pairs(wl["images"])


def workload_config(wl, world):
    P = wl["images"] * (wl["images"] - 1) // 2
    esz = 1 if wl["u8"] else 4
    return {"workload": "%s: %d images x %d feats, D=%d %s (%s-like), exhaustive %d pairs, ratio %.1f"
                        % (wl["name"], wl["images"], wl["feats"], wl["dim"], "uint8" if wl["u8"] else "float32",
                           wl["kind"], P, RATIO),
            "images": wl["images"], "feats_per_image": wl["feats"], "dim": wl["dim"], "pairs": P,
            "parallelism": ("one GPU, all pairs" if world == 1 else
                            "ONE pair list cut into %d cost-balanced contiguous shards (sharding.my_shard), no data-path "
                            "collective, per-rank results gathered to rank 0 in pair order inside the timed region" % world),
            "l2_policy": "inputs (descriptors + fp16 operands, %.1f GB) exceed the 126 MB L2"
                         % (wl["images"] * wl["feats"] * (wl["dim"] * esz + 2 * 2 * (wl["dim"] + 48)) / 1e9)}


def first_pairs(m, n):
    """The first n entries of a PairWiseMatches map as {(I, J): matches}."""
    out = {}
    for k in range(min(m.num_pairs, n)):
        I, J, mm = m.pair(k)
        out[(I, J)] = mm
    return out


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, pairs, parts, max_matches_per_pair):
    """--dump-outputs: the PairWiseMatches of the last timed step, as float64 .npy files (indices are exact in float64).
        pairs.npy          [P, 2]  the step's pair list (I, J)
        match_counts.npy   [P]     matches of each pair (0 for a pair absent from the map)
        sample_pairs.npy   [S]     rows of pairs.npy: a fixed, seeded sample of the pairs
        sample_offsets.npy [S + 1] CSR offsets of the sampled pairs into sample_matches.npy
        sample_matches.npy [M, 2]  (i, j) of every match of the sampled pairs, in the order the map holds them
    parts: [(pairs, ofs, matches)] per rank in pair order (Matches.export_csr / sharding.Gather.result).  S depends on
    the workload's shape alone (S pairs of max_matches_per_pair matches fit DUMP_BYTES), so two builds run on the same
    arguments dump the same sample."""
    os.makedirs(out_dir, exist_ok=True)
    pairs = np.asarray(pairs, np.int64).reshape(-1, 2)
    mp = np.concatenate([p[0].reshape(-1, 2) for p in parts]).astype(np.int64)
    cnt = np.concatenate([np.diff(p[1].astype(np.int64)) for p in parts])
    mm = np.concatenate([p[2] for p in parts])
    ofs = np.concatenate([[0], np.cumsum(cnt)])
    row_of = {(I, J): r for r, (I, J) in enumerate(mp.tolist())}
    row = np.array([row_of.get((I, J), -1) for I, J in pairs.tolist()], np.int64)    # -1: pair absent from the map
    counts = np.append(cnt, 0)[row]
    P = len(pairs)
    fixed = 8 * (3 * P + 1)
    S = int(min(P, max(0, DUMP_BYTES - fixed) // (16 * max_matches_per_pair + 16)))
    sel = np.sort(np.random.default_rng(20260924).choice(P, S, replace=False))
    chunks = [mm[ofs[row[k]]:ofs[row[k] + 1]] for k in sel if row[k] >= 0]
    sm = np.concatenate(chunks) if chunks else np.zeros(0, mm.dtype)
    out = {"pairs": pairs, "match_counts": counts, "sample_pairs": sel,
           "sample_offsets": np.concatenate([[0], np.cumsum(counts[sel])]),
           "sample_matches": np.stack([sm["i"], sm["j"]], 1)}
    assert sum(a.size * 8 for a in out.values()) <= DUMP_BYTES
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, np.float64))


def cpu_match_sample(po, sc, sample, n_threads):
    """The oracle port on `sample` pairs, one pair after another, upstream's own `#pragma omp parallel for` over the
    queries of SearchNeighbours using all n_threads (the outer omp-over-J team of src/R3DComputeMatches.cpp:465 would
    leave threads idle on a sample smaller than the team; this is the CPU's best case)."""
    out = []
    t0 = time.perf_counter()
    for I, J in sample:
        out.append(po.match_distance_ratio(sc["descs"][int(I)], sc["xys"][int(I)], sc["descs"][int(J)],
                                           sc["xys"][int(J)], RATIO, n_threads=n_threads))
    return time.perf_counter() - t0, out


def run_reference(args, wl, rank, emit):
    """--impl reference: the reference's CPU path = the oracle port (the reference's own code cannot be built
    here: OpenMVG/Ceres/Eigen/wx are neither vendored nor installed; DESIGN.md)."""
    if rank != 0:
        return
    from oracle import pyoracle as po
    sc, pairs = make_workload(wl)
    nthreads = effective_cpus()          # explicit team: torchrun's OMP_NUM_THREADS=1 must not shrink the CPU arm
    pair_cost = wl["feats"] * wl["feats"] * wl["dim"] / (20000.0 * 20000.0 * 128.0)     # relative to a C3 pair
    n_sample = int(os.environ.get("R3D_REF_SAMPLE_PAIRS", "0")) or int(np.clip(round(nthreads / 4.0 / pair_cost), 2, 64))
    sample = pairs[:n_sample]
    cascade = wl.get("matcher") == "cascade"
    times = []
    for it in range(args.warmup + args.steps):
        if cascade:   # the sample is its own job: hashing of its views + the bucket search, omp over views / over J
            tc0 = time.perf_counter()
            po.cascade_match_pairs(sc["descs"], sc["xys"], sample, RATIO, n_threads=nthreads)
            dt = time.perf_counter() - tc0
        else:
            dt, _ = cpu_match_sample(po, sc, sample, nthreads)
        if it >= args.warmup:
            times.append(dt)
    total = sum(times)
    value = len(sample) * len(times) / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(wl, max(args.gpus, 1)),
        "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": nthreads, "kind": "port",
                         "sample": "%d pairs (I=0, J=1..%d) of the set per step, pairs in sequence, omp over the queries "
                                   "of SearchNeighbours with %d threads = usable CPUs (cgroup quota; OMP_NUM_THREADS "
                                   "ignored)" % (len(sample), len(sample), nthreads)},
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ba", action="store_true", help="skip the bundle-adjustment leg")
    ap.add_argument("--no-filter", action="store_true", help="skip the F-filter leg")
    ap.add_argument("--no-extras", action="store_true", help="skip the C2 D=64 / D=144 side lines (N = 1)")
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS), help="BASELINE config (default c3 = the north-star set)")
    ap.add_argument("--matcher", default=None, choices=["exact", "cascade"],
                    help="exact = tensor-core brute force (default); cascade = OpenMVG CASCADE_HASHING_L2 (default of c4)")
    ap.add_argument("--feats", type=int, default=0, help="experiment only")
    ap.add_argument("--images", type=int, default=0, help="experiment only")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the matches of the last timed step to DIR/<name>.npy (float64, <= 64 MB; see dump_outputs)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the GPU path's outputs; it does not apply to --impl reference")
    # stdout carries exactly ONE line (the JSON): anything a library prints there (NCCL's version banner
    # at communicator creation, ...) is sent to stderr instead
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(real_stdout, (json.dumps(obj) + "\n").encode())
    wl = dict(WORKLOADS[args.workload])
    if args.matcher:
        wl["matcher"] = args.matcher
    if args.feats:
        wl["feats"] = args.feats
    if args.images:
        wl["images"] = args.images
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, wl, rank, emit)
        return 0

    import torch
    import torch.distributed as dist
    from regard3d_b200 import capi, sharding

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")     # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=device)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(*vals):
        if world == 1:
            return list(vals)
        t = torch.tensor(vals, dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t]

    def sum_over_ranks(*vals):
        if world == 1:
            return list(vals)
        t = torch.tensor(vals, dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [float(x) for x in t]

    warmup = max(args.warmup, 3)
    ctx = capi.Context((local_rank,))
    sc, pairs = make_workload(wl)
    n_img, n_feats, dim = wl["images"], wl["feats"], wl["dim"]
    counts = np.array([len(d) for d in sc["descs"]], np.int64)
    my_pairs, my_ofs = sharding.my_shard(pairs, counts, rank, world)
    my_pairs = np.ascontiguousarray(my_pairs, np.uint32)
    cascade = wl.get("matcher") == "cascade"
    mflags = capi.MATCH_CASCADE_HASHING if cascade else capi.MATCH_DEFAULT
    all_views = list(range(n_img))
    # cascade hashing: the hash tables depend on the zero-mean descriptor of ALL views of the job, so every rank holds
    # (and, in the end-to-end leg, uploads) all of them and hashes them itself -- replicated work, no exchange
    my_views = all_views if cascade else sorted(set(np.unique(my_pairs).tolist()))
    n_pairs = len(pairs)
    # pinned host staging (the e2e leg copies from here every step)
    pinned_desc = {v: torch.from_numpy(sc["descs"][v]).pin_memory() for v in my_views}
    pinned_xy = {v: torch.from_numpy(sc["xys"][v]).pin_memory() for v in my_views}
    gather = sharding.Gather(rank, world, device) if world > 1 else None

    def upload_all():
        for v in my_views:
            ctx.upload_regions(v, pinned_desc[v].numpy(), pinned_xy[v].numpy())

    def step_resident():
        if cascade:
            ctx.cascade_prepare(all_views)   # part of the matcher (Cascade_Hashing_Matcher_Regions::Match hashes first)
        m = ctx.match_pairs(my_pairs, RATIO, mflags)
        if gather is not None:
            gather(m)
        return m

    # ---------------- resident leg: `value` ----------------
    upload_all()
    for _ in range(warmup):
        m = step_resident()
    sampler = ClockSampler(local_rank)
    cand_ms, rerank_ms, fb_ms, dev_ms, host_ms, launches = [], [], [], [], [], 0
    fbq = q = rejq = stbq = stcq = 0
    d2h_lib = 0
    barrier()
    sampler.start()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        m = step_resident()
        t = ctx.match_timing()
        cand_ms.append(t["ms_candidates"]); rerank_ms.append(t["ms_rerank"]); fb_ms.append(t["ms_fallback"])
        dev_ms.append(t["ms_device_total"]); host_ms.append(t["ms_host_post"])
        launches += t["kernel_launches"]
        fbq += t["fallback_queries"]; q += t["queries"]; rejq += t["rejected_queries"]
        stbq += t.get("third_chunk_queries", 0); stcq += t.get("fifth_chunk_queries", 0)
    barrier()
    t_res = time.perf_counter() - t0
    n_matches, n_match_pairs = sum_over_ranks(m.total, m.num_pairs)
    if args.dump_outputs and rank == 0:     # what rank 0 holds after the last step: the gathered map when N > 1
        dump_outputs(args.dump_outputs, pairs, gather.result() if gather is not None else [m.export_csr()],
                     int(counts.max()))

    # ---------------- end-to-end leg: `e2e` ----------------
    for _ in range(2):
        ctx.clear_regions(); upload_all(); step_resident()
    barrier()
    t0 = time.perf_counter()
    h2d_step = d2h_step = 0
    for _ in range(args.steps):
        ctx.clear_regions()
        upload_all()
        m2 = step_resident()
        t = ctx.match_timing()
        h2d_step = t["h2d_bytes"] + (gather.h2d if gather else 0)
        d2h_step = t["d2h_bytes"] + (gather.d2h if gather else 0)
    barrier()
    t_e2e = time.perf_counter() - t0
    clocks = sampler.stop()   # sampled over both timed regions (resident + end-to-end), all of it under load
    t_res, t_e2e = max_over_ranks(t_res, t_e2e)
    h2d_step, d2h_step, launches_all = sum_over_ranks(h2d_step, d2h_step, launches)

    # gathered result == what the ranks hold (rank 0, outside the timed region): pair order and totals
    gather_ok = None
    if gather is not None and rank == 0:
        parts = gather.result()
        allp = np.concatenate([p[0] for p in parts], 0).astype(np.int64)
        key = allp[:, 0] * (1 << 32) + allp[:, 1]
        gather_ok = bool(np.all(np.diff(key) > 0)) and sum(int(p[1][-1]) for p in parts) == int(n_matches) \
            and all(int(p[1][-1]) == len(p[2]) for p in parts)

    # ---------------- geometric filter leg (sharded like the matching; reported alongside) ----------------
    filt = None
    if not args.no_filter:
        ctx.filter_pairs(m2, sc["widths"], sc["heights"])            # warm-up
        barrier()
        tf0 = time.perf_counter()
        fm = ctx.filter_pairs(m2, sc["widths"], sc["heights"])
        torch.cuda.synchronize()
        tf = time.perf_counter() - tf0
        ft = ctx.filter_timing()
        (tf,) = max_over_ranks(tf)
        pin, pkept, inl, hyp = sum_over_ranks(m2.num_pairs, fm.num_pairs, fm.total, ft["hypotheses"])
        filt = {"pairs_per_s": pin / tf, "ms": 1e3 * tf, "pairs_in": int(pin), "pairs_kept": int(pkept),
                "inliers": int(inl), "hypotheses": int(hyp), "rounds": int(ft["rounds"]),
                "ms_solve": ft["ms_solve"], "ms_score": ft["ms_score"], "ms_host": ft["ms_host"],
                "ms_device_total": ft["ms_device_total"], "kernel_launches": int(ft["kernel_launches"]), "n_gpus": world,
                "what": "AC-RANSAC fundamental filter (4 px, 2048 it.) over all putative pairs of the step, each rank "
                        "filtering its own shard; max over ranks"}
        if world == 1 and not args.no_cpu_baseline:
            from oracle import pyoracle as po
            nthreads = effective_cpus()
            ns = int(np.clip(4 * nthreads, 32, 256))
            put_d = first_pairs(m2, 2 * ns)
            sp = np.array(sorted(put_d)[:ns], np.uint32).reshape(-1, 2)
            ns = len(sp)
            sofs = np.zeros(ns + 1, np.uint64)
            sofs[1:] = np.cumsum([len(put_d[(int(I), int(J))]) for I, J in sp])
            sm = np.concatenate([put_d[(int(I), int(J))] for I, J in sp]) if ns else np.zeros(0, capi.indmatch_dtype)
            tc0 = time.perf_counter()
            o_ofs, o_m = po.filter_pairs_F(sc["xys"], sc["widths"], sc["heights"], sp, sofs, sm, n_threads=nthreads)
            tc = time.perf_counter() - tc0
            fd = first_pairs(fm, 2 * ns)
            same = True
            for k, (I, J) in enumerate(sp):
                e = o_m[int(o_ofs[k]):int(o_ofs[k + 1])]
                g = fd.get((int(I), int(J)))
                same &= (len(e) == 0 and g is None) or (g is not None and len(g) == len(e) and
                                                         np.array_equal(g["i"], e["i"]) and np.array_equal(g["j"], e["j"]))
            filt["cpu_baseline"] = {"value": ns / tc, "unit": "pairs/s", "cores": nthreads, "kind": "port",
                                    "sample": "first %d pairs of the step's putatives, omp over pairs, %.1f s" % (ns, tc),
                                    "parity_on_sample": bool(same)}

    # ---------------- bundle-adjustment leg (BASELINE C5, reported alongside) ----------------
    # N > 1: STRONG scaling of the one C5 problem -- points (+ their observations) partitioned over the
    # ranks, cameras replicated, in-library ncclAllReduce of the reduced camera system per LM iteration.
    ba = None
    if not args.no_ba:
        ba = ba_leg(args, ctx, torch, dist, rank, world, barrier, max_over_ranks)

    # ---------------- side lines: C2 at D = 64 (AKAZE-float / MSURF) and D = 144 (LIOP), N = 1 ----------------
    extras = None
    if world == 1 and not args.no_extras and args.workload == "c3":
        extras = {}
        for key in ("c2-msurf64", "c2"):
            w2 = WORKLOADS[key]
            sc2, pairs2 = make_workload(w2)
            ctx.clear_regions()
            for v in range(w2["images"]):
                ctx.upload_regions(v, sc2["descs"][v], sc2["xys"][v])
            for _ in range(3):
                ctx.match_pairs(pairs2, RATIO)
            torch.cuda.synchronize()
            c_ms = []
            te0 = time.perf_counter()
            for _ in range(5):
                mm = ctx.match_pairs(pairs2, RATIO)
                c_ms.append(ctx.match_timing()["ms_candidates"])
            torch.cuda.synchronize()
            te = time.perf_counter() - te0
            fl = 2.0 * w2["feats"] * w2["feats"] * w2["dim"] * len(pairs2)
            peak = float(load_peaks()[0].get("bf16_tflops", 1590.0))
            extras[key] = {"workload": workload_config(w2, 1)["workload"], "pairs_per_s": 5 * len(pairs2) / te,
                           "ms_candidates": float(np.mean(c_ms)),
                           "roofline_frac": fl / (np.mean(c_ms) * 1e-3) / 1e12 / peak, "matches": mm.total}
            del sc2

    # ---- side line: the LIOP-144 descriptor stage (SURVEY.md 8f-1), N = 1 ----
    liop = None
    if world == 1 and not args.no_extras:
        liop = liop_leg(ctx, torch, args)

    if rank == 0:
        peaks, peak_src = load_peaks()
        value = n_pairs * args.steps / t_res
        e2e = n_pairs * args.steps / t_e2e
        my_flop = 2.0 * float(np.sum(counts[my_pairs[:, 0].astype(np.int64)] * counts[my_pairs[:, 1].astype(np.int64)])) * dim
        ms_c = float(np.mean(cand_ms))
        achieved = my_flop / (ms_c * 1e-3) / 1e12
        peak = float(peaks.get("bf16_tflops", 1590.0))
        tpp, tsrc = measured_traffic_per_pair(args.workload)
        line = {
            "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
            "warmup": warmup, "ms_per_step": 1e3 * t_res / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u8" if wl["u8"] else "f32",
            "data": "synthetic", "config": workload_config(wl, world), "clocks": clocks,
            "e2e": {"value": e2e, "unit": "pairs/s", "h2d_bytes_per_step": int(h2d_step),
                    "d2h_bytes_per_step": int(d2h_step), "ms_per_step": 1e3 * t_e2e / args.steps,
                    "bytes": "whole job (sum over ranks): r3d_upload_regions of the views each shard touches + packed "
                             "matches back" + (" + the gather's H2D on the senders / D2H on rank 0" if world > 1 else "")},
            "gpu_launches": int(launches_all),
            "roofline": {"bound": "tensor", "kernel": "k_l2_candidates_2sm (tcgen05 kind::f16 cta_group::2, f16 candidates; "
                                                      "every reported distance is re-computed exactly)",
                         "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                         "peak_source": "%s bf16_tflops (burst; kernel timed alone with CUDA events)" % peak_src,
                         "ms_per_launch": ms_c, "flop_per_launch": my_flop,
                         "launch": "rank 0's shard of the step = %d pairs (batch launches of <= 128 pairs, summed)" % len(my_pairs),
                         "traffic": (tpp * len(my_pairs) if tpp else None),
                         "traffic_unit": "DRAM bytes per step of rank 0 (ncu dram__bytes_read+write of one batch launch, "
                                         "scaled to the shard's pairs; %s)" % tsrc},
            "breakdown_ms": {"candidates": ms_c, "rerank": float(np.mean(rerank_ms)),
                             "exact_scan_and_pack": float(np.mean(fb_ms)), "device_total": float(np.mean(dev_ms)),
                             "host_dedup": float(np.mean(host_ms)), "of": "rank 0's shard"},
            "result": {"pairs_with_matches": int(n_match_pairs), "matches": int(n_matches),
                       "fallback_query_frac": fbq / max(q, 1), "early_rejected_query_frac": rejq / max(q, 1),
                       "stage_b_query_frac": stbq / max(q, 1), "stage_b_key5_query_frac": stcq / max(q, 1),
                       "gathered_in_pair_order": gather_ok,
                       "gather_ms": (gather.ms if gather is not None else None)},
        }
        if cascade:
            # k_cascade_match: L2/HBM-bound integer work.  Algorithmic bytes per query: the candidate ids of its six
            # buckets (4 B each), the hash code of every distinct candidate, 10 descriptors + its own descriptor, code
            # and bucket ids; counted from the kernel's own candidate counters (raw / distinct, summed over the steps).
            words = (dim + 31) // 32
            rowb = dim * (1 if wl["u8"] else 4)
            per_step = (4.0 * stbq + 4.0 * words * stcq + q * (11.0 * rowb + 4.0 * words + 12 + 48)) / max(args.steps, 1)
            ms_k = float(np.mean(fb_ms))
            hbm = float(peaks.get("hbm_gbs", 6650.0))
            line["roofline"] = {"bound": "hbm", "kernel": "k_cascade_match (bucket gather + Hamming + 10 exact distances per query; "
                                                          "timed with the pack kernel that follows it)",
                                "achieved": per_step / (ms_k * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                                "frac": per_step / (ms_k * 1e-3) / 1e9 / hbm,
                                "peak_source": "%s hbm_gbs (the tables of a pair fit the L2: the fraction can exceed what DRAM alone allows)" % peak_src,
                                "ms_per_launch": ms_k, "bytes_per_launch": per_step,
                                "launch": "rank 0's shard of the step = %d pairs" % len(my_pairs), "traffic": None}
            line["result"]["candidates_per_query"] = stbq / max(q, 1)
            line["result"]["distinct_candidates_per_query"] = stcq / max(q, 1)
            line["config"]["matcher"] = "cascade hashing (OpenMVG CASCADE_HASHING_L2 restated: SURVEY.md A.8), hashing of all views inside the step"
        if filt is not None:
            line["f_filter"] = filt
        if ba is not None:
            line["ba"] = ba
        if extras:
            line["extras"] = extras
        if liop:
            line["liop"] = liop
        if world == 1 and not args.no_cpu_baseline:
            from oracle import pyoracle as po
            nthreads = effective_cpus()
            n_sample = int(os.environ.get("R3D_CPU_SAMPLE_PAIRS", "0")) or int(np.clip(nthreads, 8, 32))
            sample = pairs[:n_sample]
            if cascade:   # the sample as a job of its own on both sides (its views' zero-mean descriptor)
                n_sample = max(n_sample, 4 * nthreads)
                sample = pairs[:n_sample]
                tc0 = time.perf_counter()
                o_ofs, o_m = po.cascade_match_pairs(sc["descs"], sc["xys"], sample, RATIO, n_threads=nthreads)
                tc = time.perf_counter() - tc0
                outs = [o_m[int(o_ofs[k]):int(o_ofs[k + 1])] for k in range(len(sample))]
                ctx.cascade_prepare(sorted(set(np.unique(sample).tolist())))
                got = first_pairs(ctx.match_pairs(sample, RATIO, mflags), 4 * n_sample)
            else:
                tc, outs = cpu_match_sample(po, sc, sample, nthreads)
                got = first_pairs(m, 4 * n_sample)
            same = True
            for (I, J), e in zip(sample, outs):
                g = got.get((int(I), int(J)))
                same &= (g is None and len(e) == 0) or (g is not None and len(g) == len(e) and
                                                         np.array_equal(g["i"], e["i"]) and np.array_equal(g["j"], e["j"]))
            line["cpu_baseline"] = {"value": len(sample) / tc, "unit": "pairs/s", "cores": nthreads, "kind": "port",
                                    "sample": "%d pairs (I=0) of the same set, one pass, pairs in sequence, omp over the "
                                              "queries with %d threads = usable CPUs (cgroup quota), %.1f s"
                                              % (len(sample), nthreads, tc),
                                    "parity_on_sample": bool(same)}
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


def liop_leg(ctx, torch, args):
    """LIOP-144 descriptors of one 1080p image with 10 000 keypoints through r3d_liop_describe (host image and keypoints
    in, host descriptors out).  CPU side: the oracle port with OpenMP over keypoints, and THE REFERENCE's own
    r3d_vl_liopdesc_process (oracle/_ref, compiled from the reference source) on the same patches, one thread."""
    rng = np.random.default_rng(20260924)
    h, w, n = 1080, 1920, 10000
    img = rng.random((h, w)).astype(np.float32)
    kps = np.stack([rng.uniform(0, w, n), rng.uniform(0, h, n), rng.uniform(3, 40, n), rng.uniform(0, 360, n)], 1).astype(np.float32)
    for _ in range(2):
        d = ctx.liop_describe(img, kps, 8.0)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    reps = 5
    for _ in range(reps):
        d = ctx.liop_describe(img, kps, 8.0)
    torch.cuda.synchronize()
    tg = (time.perf_counter() - t0) / reps
    out = {"descriptors_per_s": n / tg, "ms_per_image": 1e3 * tg, "keypoints": n, "image": "%dx%d float32" % (w, h),
           "what": "r3d_liop_describe end to end (image H2D, warp + blur + exact quick-sort replay + order patterns, D2H)"}
    if not args.no_cpu_baseline:
        from oracle import pyoracle as po
        ns = 2000
        tc0 = time.perf_counter()
        dc, patches = po.liop_describe(img, kps[:ns], 8.0, want_patches=True)
        tc = time.perf_counter() - tc0
        out["cpu_baseline"] = {"value": ns / tc, "unit": "descriptors/s", "cores": effective_cpus(), "kind": "port",
                               "sample": "%d keypoints of the same image, omp over keypoints" % ns,
                               "parity_on_sample": bool(np.array_equal(dc.view(np.uint32), d[:ns].view(np.uint32)))}
        if po.liop_ref_available():
            tr0 = time.perf_counter()
            dr = po.liop_ref_process(patches[:500])
            tr = time.perf_counter() - tr0
            out["cpu_reference"] = {"value": 500 / tr, "unit": "descriptors/s", "cores": 1, "kind": "reference",
                                    "sample": "r3d_vl_liopdesc_process of oracle/_ref (the reference's vl_liop.c) on 500 of those "
                                              "patches; descriptor step only (warp + blur excluded)",
                                    "parity_on_sample": bool(np.array_equal(dr.view(np.uint32), d[:500].view(np.uint32)))}
    return out


def ba_leg(args, ctx, torch, dist, rank, world, barrier, max_over_ranks):
    from regard3d_b200 import sharding, synth
    prob = synth.make_ba_problem(n_cams=200, n_pts=200000, obs_per_pt=5, seed=20260924 + 5)
    arrs = {k: np.ascontiguousarray(v) for k, v in prob.items() if k != "truth"}
    for k in ("poses", "intrinsics", "points", "obs_xy"):
        arrs[k] = np.ascontiguousarray(arrs[k], np.float64)
    for k in ("obs_cam", "obs_pt", "cam_intr"):
        arrs[k] = np.ascontiguousarray(arrs[k], np.uint32)
    if world > 1:
        ids = [ctx.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        ctx.comm_init(world, rank, ids[0])
    local, _ = sharding.partition_ba(arrs, rank, world)
    ctx.bundle_adjust({k: v.copy() for k, v in local.items()}, max_iterations=2)     # warm-up
    n_it = 10
    g = {k: v.copy() for k, v in local.items()}
    barrier()
    tb0 = time.perf_counter()
    sg, tg = ctx.bundle_adjust(g, max_iterations=n_it, function_tolerance=0.0)
    tb = time.perf_counter() - tb0
    t_loop = max(sg["seconds_total"] - sg["seconds_setup"], 1e-9)
    t_loop, tb = max_over_ranks(t_loop, tb)
    if world > 1:
        ctx.comm_destroy()
    n_obs = int(len(arrs["obs_xy"]))
    nB = 6 * 200 + 6
    bytes_iter = 3 * (n_obs * 24 + len(arrs["points"]) * 24) + 2 * nB * nB * 8          # SURVEY.md 8d
    peak_hbm = float(load_peaks()[0].get("hbm_gbs", 6650.0))
    ba = {"iters_per_s": sg["iterations"] / t_loop, "e2e_iters_per_s": sg["iterations"] / tb,
          "iterations": int(sg["iterations"]), "seconds_lm_loop": t_loop, "seconds_call": tb,
          "seconds_setup": sg["seconds_setup"], "seconds_linear": sg["seconds_linear"],
          "initial_cost": sg["initial_cost"], "final_cost": sg["final_cost"], "n_gpus": world,
          "scaling": "strong", "exchange": "none" if world == 1 else
          "in-library ncclAllReduce(f64) of the reduced camera system per LM iteration",
          "config": "C5: 200 cams / %d pts / %d obs, 1 shared radial-K3 intrinsic, Huber(16)" % (len(arrs["points"]), n_obs),
          "roofline": {"bound": "hbm", "achieved": sg["iterations"] / t_loop * bytes_iter / 1e9,
                       "peak": peak_hbm, "unit": "GB/s",
                       "frac": sg["iterations"] / t_loop * bytes_iter / 1e9 / peak_hbm, "bytes_per_iter": bytes_iter}}
    if world == 1 and rank == 0 and not args.no_cpu_baseline:
        from oracle import pyoracle as po
        c = po.ba_prepare(arrs["poses"], arrs["intrinsics"], arrs["points"], arrs["obs_cam"], arrs["obs_pt"],
                          arrs["cam_intr"], arrs["obs_xy"])
        o = po.default_ba_options(max_iterations=3, n_threads=effective_cpus())
        o.function_tolerance = 0.0
        tc0 = time.perf_counter()
        so, to = po.bundle_adjust(c, o)
        tcb = time.perf_counter() - tc0
        ba["cpu_baseline"] = {"iters_per_s": so["iterations"] / tcb, "iterations": int(so["iterations"]),
                              "cores": effective_cpus(), "kind": "port",
                              "cost_trace_rel_diff": float(np.max(np.abs(tg[:len(to)] - to) / to))}
    return ba


if __name__ == "__main__":
    sys.exit(main())
