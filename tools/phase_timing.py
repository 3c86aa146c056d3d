"""Per-phase cycle breakdown of mpc_kernel (needs a library built with -DHMPC_PHASE_TIMING, see
tools/build_variant.py):  HMPC_LIB_PATH=.../libhmpc_b200_X.so python tools/phase_timing.py [batch] [ticks]
Cycles are thread 0's clock64() deltas summed over all CTAs; shares are relative to phase 0 (whole hopper)."""
import ctypes as C
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from hopper_mpc_inertial_b200 import scenarios, _lib   # noqa: E402
from hopper_mpc_inertial_b200.batch import BatchMpc   # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 131072
K = int(sys.argv[2]) if len(sys.argv) > 2 else 10
W = 5
N = int(sys.argv[3]) if len(sys.argv) > 3 else 10
HOT = sys.argv[4] if len(sys.argv) > 4 else "cta"      # the phase counters live in the CTA kernels
sc = scenarios.make_batch(B, N=N, n_ticks=W + K + 1)
dev = torch.device("cuda:0")
T = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=dev)
bm = BatchMpc(B, dyn="3f", N=N, device=0, on_infeasible="respawn", hot_path=HOT)
bm.set_gains(T(sc["Qdiag"]), T(sc["Rdiag"]))
X = T(sc["X0"]).clone()
args = (T(sc["xref_tab"]), T(sc["pf_tab"]), T(np.ascontiguousarray(sc["C_tab"]).view(np.int64)), T(sc["pf_switch"]))
bm.rollout(X, *args, 0, W, True)
torch.cuda.synchronize()
lib = _lib.load() if hasattr(_lib, "load") else C.CDLL(_lib.LIB_PATH)
# one hook per CTA-kernel unit that has one; every read resets, so the sum is the handle's build
hooks = [getattr(lib, f) for f in ("hmpc_debug_phases", "hmpc_debug_phases_wide_gmem4", "hmpc_debug_phases_wide_gmem2") if hasattr(lib, f)]
has = bool(hooks)


def read_phases():
    tot = np.zeros(16, np.uint64)
    for f in hooks:
        b = (C.c_ulonglong * 16)()
        f(b)
        tot += np.array(b[:], np.uint64)
    return tot


read_phases()
t0 = time.perf_counter()
bm.rollout(X, *args, W, K, False)
torch.cuda.synchronize()
dt = time.perf_counter() - t0
print(f"{B * K / dt / 1e6:.3f} M steps/s ({dt / K * 1e3:.2f} ms per tick)")
nf, path, ninf = bm.solve_stats()
print("factorisations per tick", float(nf.double().mean()) / K)
if has:
    buf = read_phases()
    names = ["whole hopper", "load + lin. point", "condense", "solve_exact (all)", "factor", "solve (1 rhs)", "refinement loop (incl. its solves)",
             "verify_active_set", "interior point (incl. its factor/solve)", "rollout", "tiled factor: entry gather (warp 0)", "tiled factor: tile products (warp 0)", "tiled factor: diagonal tiles"]
    tot = buf[0] or 1
    for i, nme in enumerate(names):
        print(f"  {i:2d} {nme:45s} {100.0 * buf[i] / tot:6.2f} %   {buf[i] / (B * K):10.0f} cycles per hopper-tick")
