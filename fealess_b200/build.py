"""Build libfealess_b200.so (hand-written CUDA for sm_100a + the C ABI) in-tree with nvcc.

The .so is git-ignored but travels to the GPU box with the gpurun snapshot.  ``-fmad=false`` is deliberate: the
fp32 expressions of the depth-normal quantiser and of ICP must round like the reference's uncontracted x86 build."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libfealess_b200.so")
SOURCES = ["frontend.cu", "similarity.cu", "similarity_staged.cu", "icp.cu", "resize.cu", "api.cu", "group.cu", "pipe.cu", "train.cu", "reco.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-fmad=false", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-O2", "--expt-relaxed-constexpr"]


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found")


def needs_build() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "fealess_b200.h"), __file__]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return OUT
    nvcc = _nvcc()
    objdir = os.path.join(HERE, "_build")
    os.makedirs(objdir, exist_ok=True)
    objs = []
    env = dict(os.environ)
    # the image exports CC=/opt/gcc/bin/gcc which lacks some spec files; nvcc's host compiler is the system g++
    ccbin = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else None
    procs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + (["-ccbin", ccbin] if ccbin else []) + (["-Xptxas", "-v"] if verbose else []) + \
              ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, env=env, text=True)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write("== %s ==\n%s\n" % (src, out))
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    cmd = [nvcc, "-shared", "-o", OUT] + objs + (["-ccbin", ccbin] if ccbin else []) + ["-gencode", "arch=compute_100a,code=sm_100a"]
    subprocess.check_call(cmd, env=env)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
