"""Builds libmt_b200.so (hand-written CUDA for sm_100a) in-tree with nvcc.

    python -m master_thesis_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU.  The library is built next to this file so
that it travels with the repo snapshot to the GPU box; it is never installed
into site-packages.  -fmad=false is part of the arithmetic contract (see
csrc/mt_common.cuh): only explicit __fmaf_rn() calls fuse.
"""
import glob
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libmt_b200.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo", "-fmad=false",
    "--expt-relaxed-constexpr", "--extended-lambda",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
    "-shared",
]


def find_nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (needed to build libmt_b200.so)")


def sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = sources() + glob.glob(os.path.join(CSRC, "*.cuh")) + \
        glob.glob(os.path.join(ROOT, "include", "*.h")) + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force=False, verbose=False, defines=(), out=None):
    """defines / out: developer builds (e.g. -DMT_DEV_PROBES into another file name,
    selected at run time with MT_B200_LIB); the product build uses neither."""
    if not force and not needs_build() and not defines and out is None:
        return LIB
    cmd = [find_nvcc()] + NVCC_FLAGS + ["-I", os.path.join(ROOT, "include"), "-I", CSRC]
    cmd += ["-D" + d for d in defines]
    if verbose:
        cmd += ["-Xptxas", "-v"]
    cmd += ["-o", out or LIB] + sources()
    # the image exports CC=/opt/gcc/bin/gcc (a bare wrapper); let nvcc use the system g++
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    res = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or res.returncode != 0:
        sys.stderr.write(res.stdout)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed (%d): %s" % (res.returncode, " ".join(cmd)))
    return out or LIB


if __name__ == "__main__":
    defs = [a[2:] for a in sys.argv[1:] if a.startswith("-D")]
    outs = [a[len("--out="):] for a in sys.argv[1:] if a.startswith("--out=")]
    print(build_library(force="--force" in sys.argv, verbose="--verbose" in sys.argv,
                        defines=defs, out=outs[0] if outs else None))
