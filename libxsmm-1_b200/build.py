"""Builds libxsmm_b200.so (the C-ABI library with all sm_100a kernels) in-tree with nvcc.

    python libxsmm-1_b200/build.py [--verbose] [--force]

nvcc cross-compiles for sm_100a without a GPU.  The built library stays next to the sources
(libxsmm-1_b200/lib/) so that it travels with the tree; it is git-ignored.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libxsmm_b200.so")
SOURCES = ["capi.cu", "spmdm_kernels.cu", "spmdm_compute_tma.cu", "spmdm_compute_sp.cu", "spmdm_compute_tc.cu", "spmdm_compute_tcq.cu", "spmdm_compute_tc16p.cu", "spmdm_compute_tc16s.cu", "fsspmdm.cu", "fsspmdm_tc.cu", "fsspmdm_jit.cpp", "rm_soa.cu", "sp24.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC,-fvisibility=hidden", "-I", os.path.join(ROOT, "include")]


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(ROOT, "include", f) for f in os.listdir(os.path.join(ROOT, "include"))]
    return any(os.path.getmtime(d) > t for d in deps)


def build(verbose=False, force=False):
    if not force and not _stale():
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(LIBDIR, os.path.splitext(src)[0] + ".o")
        cmd = [NVCC] + ARCH + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-x", "cu", "-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for cmd, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(out)
        if p.returncode != 0:
            raise RuntimeError("nvcc failed: " + " ".join(cmd))
    link = [NVCC] + ARCH + ["-shared", "-o", LIB] + objs + ["-ldl"]
    subprocess.check_call(link)
    return LIB


if __name__ == "__main__":
    print(build(verbose="--verbose" in sys.argv, force="--force" in sys.argv))
