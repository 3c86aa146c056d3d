"""In-tree build of libhmpc_b200.so with nvcc for sm_100a (no JIT cache: the .so travels with the repo).

The solver kernel is a ~30 k-instruction template; each instantiation is its own translation unit
(csrc/inst_*.cu) and the units are compiled in parallel, then linked into one shared library."""
from __future__ import annotations

import concurrent.futures as cf
import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "csrc")
UNITS = ["hmpc_api.cu", "inst_warp.cu", "inst_n10_f64.cu", "inst_n10_f64_admm.cu", "inst_n10_f32.cu", "inst_wide_gmem2.cu", "inst_wide_gmem4.cu"]
HEADERS = ["hmpc_qp.cuh", "hmpc_mpc.cuh", "hmpc_sim.cuh", "hmpc_kernel.cuh", "hmpc_warp.cuh", "hmpc_tile.cuh", "hmpc_plan.cuh", "hmpc_geometry.cuh"]
DEPS = [os.path.join(_CSRC, f) for f in UNITS + HEADERS] + [os.path.join(_HERE, "..", "include", "hmpc.h")]
OUT = os.path.join(_HERE, "libhmpc_b200.so")
OBJ_DIR = os.path.join(_HERE, "build")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC"]


def _nvcc():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def build_lib(force=False, verbose=False):
    if not force and os.path.exists(OUT) and all(os.path.getmtime(OUT) >= os.path.getmtime(d) for d in DEPS):
        return OUT
    os.makedirs(OBJ_DIR, exist_ok=True)
    nvcc = _nvcc()
    extra = ["-Xptxas", "-v"] if verbose else []
    extra += os.environ.get("HMPC_EXTRA_NVCC_FLAGS", "").split()     # experiments: -DHMPC_PHASE_TIMING ...

    def compile_unit(u):
        obj = os.path.join(OBJ_DIR, u.replace(".cu", ".o"))
        subprocess.run([nvcc] + NVCC_FLAGS + extra + ["-c", os.path.join(_CSRC, u), "-o", obj], check=True)
        return obj

    with cf.ThreadPoolExecutor(max_workers=len(UNITS)) as ex:
        objs = list(ex.map(compile_unit, UNITS))
    subprocess.run([nvcc, "-shared", "-Wno-deprecated-gpu-targets", "-o", OUT] + objs, check=True)
    return OUT


if __name__ == "__main__":
    print(build_lib(force=True, verbose=True))
