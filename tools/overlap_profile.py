#!/usr/bin/env python
"""Where the deferred hoppers' CTA kernel runs in the overlapped rollout schedule (DESIGN.md section 5).

Runs bench.py's flagship configuration (3f, N = 10, FP64, exact solver, respawn; tables from the device planner) under
torch.profiler with CUDA activities, once with the overlapped schedule and once with HMPC_DEFER_SERIAL=1, and reports
per timed tick:
  defer_ms    the CTA kernel over the deferral list (mpc_kernel in list mode)
  prep_ms     the prep kernel on the main stream (every hopper but the previous tick's deferred ones)
  prep_d_ms   the prep kernel over the previous tick's deferral list (side stream; overlapped schedule only)
  overlap_ms  how much of the tick's deferred kernel runs while the next tick's main-stream prep kernel runs
  tick_ms     start of the tick's lock-step kernel to the start of the next one
Usage:  python tools/overlap_profile.py [--batch 131072] [--warmup 5] [--steps 20] [--out FILE.json]
Profile runs are slower than bench.py's (tracing); take throughput from bench.py."""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def trace_one(batch, warmup, steps):
    import numpy as np
    import torch
    from torch.profiler import ProfilerActivity, profile

    import bench
    from hopper_mpc_inertial_b200 import scenarios
    from hopper_mpc_inertial_b200.batch import BatchMpc

    dev = torch.device("cuda", 0)
    sc = scenarios.make_batch(batch, N=10, n_ticks=warmup + steps + 1, dyn="3f", tables=False)
    bm = BatchMpc(batch, dyn="3f", N=10, device=0, on_infeasible="respawn")
    T = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=dev)
    bm.set_gains(T(sc["Qdiag"]), T(sc["Rdiag"]))
    bench.plan_on_device(bm, sc, dev)
    tabs = bm.plan_tables(0, warmup + steps + 1)
    args = (tabs["xref_tab"], tabs["pf_tab"], tabs["C_tab"], tabs["pf_switch"])
    X = T(sc["X0"]).clone()
    bm.rollout(X, *args, 0, warmup, True)
    torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as tmp:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            bm.rollout(X, *args, warmup, steps, False)
            torch.cuda.synchronize()
        path = os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    deferred = bm.hot_path_info()["deferred"]
    bm.close()
    kern = [e for e in events if e.get("cat") == "kernel"]
    return kern, deferred


def analyse(kern):
    def of(sub):
        return sorted((e for e in kern if sub in e["name"]), key=lambda e: e["ts"])
    warp = of("mpc_warp_rounds_kernel")
    main = warp[0]["args"]["stream"]
    prep = of("mpc_prep_kernel")
    prep_main = [e for e in prep if e["args"]["stream"] == main]
    prep_side = [e for e in prep if e["args"]["stream"] != main]
    defer = [e for e in of("mpc_kernel<") if "prep" not in e["name"] and "warp" not in e["name"]]
    iv = lambda e: (e["ts"], e["ts"] + e["dur"])
    ovl = lambda a, b: max(0.0, min(a[1], b[1]) - max(a[0], b[0]))
    ticks = []
    for t, w in enumerate(warp):
        nxt = warp[t + 1]["ts"] if t + 1 < len(warp) else None
        d = [e for e in defer if e["ts"] >= w["ts"] and (nxt is None or e["ts"] < nxt)]
        p = [e for e in prep_main if e["ts"] <= w["ts"]][-1:]          # this tick's main-stream prep
        pn = [e for e in prep_main if e["ts"] > w["ts"]][:1]            # the next tick's
        pd = [e for e in prep_side if e["ts"] > w["ts"] and (nxt is None or e["ts"] < nxt)]
        rec = {"tick": t, "defer_ms": sum(e["dur"] for e in d) / 1e3, "prep_ms": (p[0]["dur"] / 1e3) if p else None,
               "prep_d_ms": sum(e["dur"] for e in pd) / 1e3,
               "overlap_ms": (sum(ovl(iv(e), iv(pn[0])) for e in d) / 1e3) if pn else 0.0,
               "tick_ms": ((nxt - w["ts"]) / 1e3) if nxt is not None else None}
        ticks.append(rec)
    full = [r for r in ticks if r["tick_ms"] is not None]
    mean = lambda k: float(sum(r[k] for r in full) / max(len(full), 1))
    return {"ticks": ticks, "mean_over_complete_ticks": {k: mean(k) for k in ("defer_ms", "prep_ms", "prep_d_ms", "overlap_ms", "tick_ms")}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=131072)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    ap.add_argument("--one", choices=["overlapped", "serial"], help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.one:
        kern, deferred = trace_one(a.batch, a.warmup, a.steps)
        print(json.dumps(dict(analyse(kern), deferred=deferred)))
        return
    import torch
    gpu = torch.cuda.get_device_name(0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    res = {"gpu": gpu, "nvidia_smi": smi, "batch": a.batch, "warmup": a.warmup, "steps": a.steps}
    # one process per schedule: HMPC_DEFER_SERIAL is read when a handle is created, the profiler is per process
    for mode in ("overlapped", "serial"):
        env = dict(os.environ)
        env.pop("HMPC_DEFER_SERIAL", None)
        if mode == "serial":
            env["HMPC_DEFER_SERIAL"] = "1"
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--one", mode, "--batch", str(a.batch),
                              "--warmup", str(a.warmup), "--steps", str(a.steps)], env=env, capture_output=True, text=True)
        if out.returncode != 0:
            raise SystemExit(out.stderr[-2000:])
        res[mode] = json.loads(out.stdout.strip().splitlines()[-1])
    text = json.dumps(res, indent=1)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")
    for mode in ("overlapped", "serial"):
        print(mode, json.dumps(res[mode]["mean_over_complete_ticks"]))


if __name__ == "__main__":
    main()
