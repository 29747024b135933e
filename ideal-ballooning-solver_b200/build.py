"""Build recipe of the CUDA library: plain ``nvcc`` for sm_100a, in-tree output.

``python -m ideal_ballooning_solver_b200.build`` (or ``__graft_entry__.build()``) compiles
``csrc/*.cu`` into ``lib/libibs_b200.so``.  nvcc cross-compiles without a GPU.  The ``.so`` is
git-ignored but travels to the GPU box with the ``gpurun`` snapshot.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libibs_b200.so")
SOURCES = ["ibs_api.cu", "ibs_solver.cu", "ibs_scan_solver.cu", "ibs_geometry.cu", "ibs_geometry_full.cu", "ibs_geometry_adjoint.cu", "ibs_adjoint.cu", "ibs_marginal.cu"]
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "-DIBS_BUILD", "-fmad=true"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isfile(cand) or cand == "nvcc"):
            return cand
    raise RuntimeError("nvcc not found")


def _stamp():
    h = hashlib.sha256()
    names = [n for n in sorted(os.listdir(CSRC)) if n.endswith((".cu", ".cuh", ".h"))]
    for name in names + ["../../include/ibs_b200.h"]:
        with open(os.path.join(CSRC, name), "rb") as f:
            h.update(name.encode() + f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile the library if sources changed; returns the path of the ``.so``."""
    os.makedirs(LIBDIR, exist_ok=True)
    stamp_file = os.path.join(LIBDIR, "build.stamp")
    stamp = _stamp()
    if not force and os.path.isfile(LIB) and os.path.isfile(stamp_file) and open(stamp_file).read() == stamp:
        return LIB
    nvcc = _nvcc()
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(LIBDIR, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
            print(" ".join(cmd), flush=True)
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, pr in procs:
        out, _ = pr.communicate()
        if verbose or pr.returncode != 0:
            sys.stdout.write(out)
        failed |= pr.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    link = [nvcc, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static"]
    subprocess.check_call(link)
    with open(stamp_file, "w") as f:
        f.write(stamp)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
