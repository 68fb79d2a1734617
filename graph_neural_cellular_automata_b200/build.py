"""Build libgnca.so (sm_100a) in-tree with nvcc.  No JIT, no torch cpp_extension: the product is a plain
C-ABI shared library (include/gnca.h) that the Python host layer loads with ctypes."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
LIBDIR = os.path.join(PKG, "lib")
LIB = os.path.join(LIBDIR, "libgnca.so")
SOURCES = ["gnca_fwd.cu", "gnca_bwd.cu", "gnca_aux.cu", "gnca_rollout.cu", "gnca_resident.cu", "gnca_rep.cu", "gnca_rep_bwd.cu", "gnca_graph.cu", "gnca_update_tc.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "-Xptxas", "-v"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; libgnca.so cannot be built")


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(PKG, "..", "include", "gnca.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = True) -> str:
    # GNCA_PHASE_COUNTERS=1 in the environment compiles the per-phase cycle counters into the resident kernels
    # (read back with GNCA_PHASE_TIMING=<cta> at run time); off by default: they cost registers in the step loops.
    """Compile every CUDA source for sm_100a into lib/libgnca.so (objects in parallel, then one link)."""
    if not force and not _stale():
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    nvcc = _nvcc()
    objs, procs = [], []
    for src in SOURCES:
        path = os.path.join(CSRC, src)
        if not os.path.exists(path):
            continue
        obj = os.path.join(LIBDIR, src.replace(".cu", ".o"))
        objs.append(obj)
        extra = ["-DGNCA_PHASE_COUNTERS"] if os.environ.get("GNCA_PHASE_COUNTERS") else []
        extra += [f"-D{d}" for d in os.environ.get("GNCA_EXTRA_DEFINES", "").split()]      # development experiments
        cmd = [nvcc, *NVCC_FLAGS, *extra, "-c", path, "-o", obj]
        if verbose:
            print("[gnca build]", " ".join(cmd), flush=True)
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
        if verbose and out.strip():
            print(out)
    cmd = [nvcc, "-shared", "-o", LIB, *objs, "-lcudart"]
    if verbose:
        print("[gnca build]", " ".join(cmd), flush=True)
    subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv)
    print(LIB)
