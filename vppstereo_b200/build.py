"""Build the C-ABI library (include/vppstereo_b200.h) for sm_100a, in tree.

    python -m vppstereo_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU.  Output: vppstereo_b200/libvppstereo_b200.so (git-ignored, travels with gpurun).
Flags: -gencode arch=compute_100a,code=sm_100a (B200 only), -lineinfo (ncu source view), -fmad=false (the VPP blends
and the float tails must not be FMA-contracted: a contraction changes uint8 truncations, SURVEY.md A.1.3).
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libvppstereo_b200.so")
SOURCES = ["capi.cu", "rsgm_ops.cu", "sgm.cu", "sgm_sweep.cu", "vpp.cu", "filter.cu"]
HEADERS = [os.path.join(CSRC, "common.cuh"), os.path.join(HERE, "..", "include", "vppstereo_b200.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo", "-fmad=false",
         "-Xcompiler", "-fPIC,-O2,-fvisibility=default", "-cudart", "static"]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    objs = []
    bdir = os.path.join(HERE, "build")
    os.makedirs(bdir, exist_ok=True)
    procs = []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        obj = os.path.join(bdir, s.replace(".cu", ".o"))
        objs.append(obj)
        if force or _stale(obj, [src] + HEADERS):
            cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
            procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for cmd, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            print(" ".join(cmd))
            print(out)
        if p.returncode != 0:
            raise RuntimeError("nvcc failed for " + cmd[-3])
    if force or procs or _stale(LIB, objs):
        cmd = [NVCC, "-shared", "-cudart", "static", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs
        subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
