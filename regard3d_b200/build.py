"""Build libr3dgpu.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m regard3d_b200.build [--force]

The shared library is a plain C-ABI library (include/r3dgpu.h): no torch, no pybind.
"""
import glob
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libr3dgpu.so")
NVCC = os.environ.get("R3D_NVCC", "/usr/local/cuda/bin/nvcc")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-ccbin", "g++",
    "-Xcompiler", "-fPIC,-O3,-pthread,-ffp-contract=off",
    "--fmad=true",
    "-diag-suppress", "177",
]
# translation units whose floating-point decisions must match the CPU restatement bit for bit are
# compiled without FMA contraction
NO_FMAD = {"acransac_kernels.cu", "acransac_fused.cu", "liop.cu", "relpose.cu"}


def sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")) + glob.glob(os.path.join(CSRC, "*.cpp")))


def needs_build():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = sources() + glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(os.path.join(CSRC, "*.h")) + [
        os.path.join(HERE, "..", "include", "r3dgpu.h"), os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, defines=(), out_path=None, objdir_name="build"):
    """defines / out_path / objdir_name: an A/B variant of the library (e.g. -DR3D_CHUNK=16) next to the default one."""
    if out_path is None and not force and not needs_build():
        return OUT
    objdir = os.path.join(HERE, objdir_name)
    os.makedirs(objdir, exist_ok=True)
    objs = []
    procs = []
    for src in sources():
        obj = os.path.join(objdir, os.path.basename(src) + ".o")
        flags = list(NVCC_FLAGS) + ["-D" + d for d in defines]
        if os.path.basename(src) in NO_FMAD:
            flags[flags.index("--fmad=true")] = "--fmad=false"
        cmd = [NVCC] + flags + (["-Xptxas", "-v"] if verbose else []) + ["-x", "cu", "-c", src, "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            failed = True
            sys.stderr.write("nvcc failed for %s:\n%s\n" % (src, out))
        elif verbose:
            sys.stderr.write(out)
    if failed:
        raise RuntimeError("libr3dgpu build failed")
    cmd = [NVCC, "-shared", "-o", out_path or OUT] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-ccbin", "g++",
                                               "-Xcompiler", "-pthread", "-lpthread", "-ldl"]
    subprocess.check_call(cmd)
    return out_path or OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
