"""Build libbdlm.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m bayesian_dlms_b200.build [--force] [--verbose]

-fmad=false is part of the numerical contract, not a tuning flag: the reference's JVM
arithmetic never fuses multiply-add and the kernels are bit-compared against the oracle.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libbdlm.so")
SOURCES = ["api.cu", "kf_small.cu", "kf_warp.cu", "kf_group.cu", "transpose.cu", "peak.cu", "scan.cu",
           "scalar_filters.cu", "gibbs_draw.cu", "ffbs_small.cu", "comm.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC,-fvisibility=hidden", "--expt-relaxed-constexpr",
]
# Bit-exact kernels never contract a*b+c.  The parallel-in-time scan (scan.cu) has no bit-exact
# counterpart in the reference -- its contract is 1e-9 relative against the sequential kernel --
# and is FP64-issue bound on B200, so it alone is built with contraction enabled.
FMAD = {"scan.cu": "-fmad=true"}


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build_lib(force: bool = False, verbose: bool = False) -> str:
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    headers = [os.path.join(CSRC, h) for h in os.listdir(CSRC) if h.endswith((".cuh", ".h"))]
    headers.append(os.path.join(HERE, "..", "include", "bdlm.h"))
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    nvcc = _nvcc()

    def compile_one(src):
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        path = os.path.join(CSRC, src)
        if force or _stale(obj, [path] + headers):
            cmd = ([nvcc] + NVCC_FLAGS + [FMAD.get(src, "-fmad=false")] +
                   (["-Xptxas", "-v"] if verbose else []) + ["-c", path, "-o", obj])
            r = subprocess.run(cmd, capture_output=True, text=True)
            if verbose or r.returncode:
                sys.stderr.write(r.stdout + r.stderr)
            if r.returncode:
                raise RuntimeError(f"nvcc failed on {src}")
        return obj

    with ThreadPoolExecutor(max_workers=len(srcs)) as ex:
        objs = list(ex.map(compile_one, srcs))
    if force or _stale(LIB, objs):
        cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-ldl"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("link failed")
    return LIB


if __name__ == "__main__":
    print(build_lib(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
