"""Cost of per-hopper bodies (include/hmpc.h: hmpc_set_body_params) on the closed loop hmpc_rollout runs.

131072 hoppers, 3f, N = 10 and N = 20, four cases:  none (no call), uniform (the config's scalars set explicitly as
arrays: the per-hopper kernels on the reference body), random (make_bodies, model = plant), mismatch (make_bodies,
plant 5 % off the model).  Per case: steps/s from CUDA events around hmpc_rollout, deferred fraction (hot_path_info),
mean factorisations per hopper-tick, infeasible hopper-ticks, simulator-kernel time per tick (hmpc_kernel_times).
Prints the card name and power limit first.  Usage: python tools/body_params_bench.py [--B 131072] [--ticks 20]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hopper_mpc_inertial_b200 import scenarios  # noqa: E402
from hopper_mpc_inertial_b200.batch import BatchMpc  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:           # noqa: BLE001
        q = f"nvidia-smi unavailable ({e})"
    return dict(device=torch.cuda.get_device_name(0), nvidia_smi=q)


def run(B, N, case, ticks, warm):
    sc = scenarios.make_batch(B, N=N, n_ticks=ticks + warm, seed=2024, body=(case in ("random", "mismatch")) or None)
    T = lambda a: torch.as_tensor(np.ascontiguousarray(a), device="cuda:0")
    bm = BatchMpc(B, dyn="3f", N=N)
    bm.set_gains(T(sc["Qdiag"]), T(sc["Rdiag"]))
    if case == "uniform":
        c = bm.cfg
        rep = lambda v, shape: T(np.repeat(np.asarray(list(v) if hasattr(v, "__len__") else [v], float).reshape(shape + (1,)), B, -1))
        bm.set_body_params("both", m=rep(c.m, ()), J=rep(c.J, (3, 3)), Jinv=rep(c.Jinv, (3, 3)), rh=rep(c.rh, (3,)))
        bm.set_body_params("model", m=rep(c.m, ()), Jinv=rep(c.Jinv, (3, 3)), rh=rep(c.rh, (3,)), mu=rep(c.mu, ()))
    elif case in ("random", "mismatch"):
        model, plant = sc["body_model"], sc["body_plant"]
        if case == "random":
            plant = dict(m=model["m"], J=np.ascontiguousarray(np.moveaxis(np.linalg.inv(np.moveaxis(model["Jinv"], -1, 0)), 0, -1)),
                         Jinv=model["Jinv"], rh=model["rh"])
        bm.set_body_params("model", **{k: T(v) for k, v in model.items()})
        bm.set_body_params("plant", **{k: T(v) for k, v in plant.items()})
    X = T(sc["X0"]).clone()
    tabs = (T(sc["xref_tab"]), T(sc["pf_tab"]), T(sc["C_tab"].view(np.int64)), T(sc["pf_switch"]))
    bm.rollout(X, *tabs, 0, warm, True)                     # first tick + warm-up ticks, not timed
    bm.set_timing(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = bm.rollout(X, *tabs, warm, ticks, False)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    info = bm.hot_path_info()
    nf, _, ninf = (a.cpu().numpy() for a in bm.solve_stats())
    _, sim_ms, kt_ticks = bm.kernel_times()
    res = dict(case=case, B=B, N=N, ticks=ticks, steps_per_s=B * ticks / (ms * 1e-3),
               deferred_fraction=info["deferred"] / (B * ticks), mean_factorisations=float(nf.mean()) / ticks,
               infeasible=int(ninf.sum()), sim_ms_per_tick=sim_ms / max(kt_ticks, 1),
               status_nonzero=int((out["status"].cpu().numpy() != 0).sum()))
    bm.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=131072)
    ap.add_argument("--ticks", type=int, default=20)
    ap.add_argument("--warm", type=int, default=3)
    ap.add_argument("--N", type=int, nargs="+", default=[10, 20])
    a = ap.parse_args()
    print(json.dumps(card()), flush=True)
    for N in a.N:
        for case in ("none", "uniform", "random", "mismatch"):
            print(json.dumps(run(a.B, N, case, a.ticks, a.warm)), flush=True)


if __name__ == "__main__":
    main()
