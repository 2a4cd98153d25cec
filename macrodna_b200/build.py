"""Build the sm_100a shared library ``libmacrodna_b200.so`` in-tree with nvcc.

``python -m macrodna_b200.build`` (or ``__graft_entry__.build()``).  The library is
the whole numeric product: there is no CPU fallback and no other backend.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libmacrodna_b200.so")
SOURCES = ["api.cu", "standardize.cu", "corr_fp64.cu", "corr_tc.cu", "corr_ozaki.cu", "lap.cu", "null_test.cu", "loo.cu", "stage.cu"]
HEADERS = ["mcd_internal.cuh", os.path.join("..", "..", "include", "macrodna_b200.h")]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    nvcc = _nvcc()
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    common = ARCH + ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-diag-suppress", "177"]
    common += os.environ.get("MCD_NVCC_FLAGS", "").split()
    if verbose:
        common += ["-Xptxas", "-v"]
    procs = []
    objs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [nvcc] + common + ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if out.strip() and (verbose or p.returncode != 0):
            print("== %s\n%s" % (src, out), file=sys.stderr)
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    link = [nvcc] + ARCH + ["-shared", "-o", LIB] + objs + ["-cudart", "static"]
    subprocess.run(link, check=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
