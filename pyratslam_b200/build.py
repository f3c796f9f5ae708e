"""Build libpyratslam_b200.so in-tree with nvcc for sm_100a (no torch headers involved).

``python -m pyratslam_b200.build`` or ``__graft_entry__.build()``.  The shared library lands in
``pyratslam_b200/_lib/`` so that it travels with the source tree to the GPU box.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
LIBDIR = os.path.join(PKG, "_lib")
LIB = os.path.join(LIBDIR, "libpyratslam_b200.so")
SOURCES = ["capi.cu", "posecell_generic.cu", "posecell_resident.cu", "posecell_tiled.cu", "posecell_cluster.cu", "posecell_pair.cu", "posecell_active.cu",
           "view_templates.cu", "sharded.cu", "experience_map.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr"]


def _nvcc():
    nv = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nv):
        raise RuntimeError("nvcc not found; cannot build libpyratslam_b200.so")
    return nv


def _digest():
    h = hashlib.sha256()
    for root in (CSRC, os.path.join(os.path.dirname(PKG), "include")):
        for f in sorted(os.listdir(root)):
            if f.endswith((".cu", ".cuh", ".h")):
                h.update(f.encode())
                h.update(open(os.path.join(root, f), "rb").read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    os.makedirs(LIBDIR, exist_ok=True)
    stamp = os.path.join(LIBDIR, "build.sha256")
    dig = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read().strip() == dig:
        return LIB
    nv = _nvcc()
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(LIBDIR, src.replace(".cu", ".o"))
        cmd = [nv] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, pr in procs:
        out, _ = pr.communicate()
        if verbose or pr.returncode != 0:
            sys.stderr.write(out)
        if pr.returncode != 0:
            raise RuntimeError("nvcc failed on %s" % src)
    cmd = [nv, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static"]
    subprocess.check_call(cmd)
    open(stamp, "w").write(dig + "\n")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
