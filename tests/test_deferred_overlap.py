"""The overlapped rollout schedule (DESIGN.md section 5) against the serial one.

In a multi-tick hmpc_rollout the hoppers the warp kernel defers are solved, simulated and condensed for the next tick
on a second stream while the main stream simulates and condenses every other hopper.  Every hopper runs the same
kernels on the same data in the same order, so the two schedules must agree bit for bit: states, controls, statuses,
iteration and factorisation counts, the other solve statistics and the deferral count.  HMPC_DEFER_SERIAL=1 (read
when the handle is created) selects the serial schedule."""
import numpy as np
import pytest
import torch

from hopper_mpc_inertial_b200 import scenarios
from hopper_mpc_inertial_b200.batch import BatchMpc

pytestmark = pytest.mark.gpu


def T(a):
    return torch.as_tensor(np.ascontiguousarray(a), device="cuda:0")


def run(monkeypatch, sc, calls, serial, kcap=None, body=False, timing=False, **kw):
    """Closed loop of scenario sc over the rollout calls [(tick0, n_ticks, init)], on a handle created with or without
    HMPC_DEFER_SERIAL.  Returns (per-call results, final X, launch count)."""
    if serial:
        monkeypatch.setenv("HMPC_DEFER_SERIAL", "1")
    else:
        monkeypatch.delenv("HMPC_DEFER_SERIAL", raising=False)
    if kcap:
        monkeypatch.setenv("HMPC_WARP_KCAP", str(kcap))
    B = sc["X0"].shape[1]
    bm = BatchMpc(B, dyn="3f", N=10, device=0, **kw)
    bm.set_gains(T(sc["Qdiag"]), T(sc["Rdiag"]))
    if body:
        bm.set_body_params("model", **{k: T(v) for k, v in sc["body_model"].items()})
        bm.set_body_params("plant", **{k: T(v) for k, v in sc["body_plant"].items()})
    if timing:
        bm.set_timing(True)
    tabs = (T(sc["xref_tab"]), T(sc["pf_tab"]), T(np.ascontiguousarray(sc["C_tab"]).view(np.int64)), T(sc["pf_switch"]))
    X = T(sc["X0"]).clone()
    res = []
    for tick0, n, init in calls:
        out = bm.rollout(X, *tabs, tick0, n, init, log=True)
        torch.cuda.synchronize()
        r = {k: v.cpu().numpy() for k, v in out.items()}
        r.update(zip(("nfac", "path", "ninf"), (a.cpu().numpy() for a in bm.solve_stats())))
        r["flops"] = bm.solve_flops().cpu().numpy()
        r["deferred"] = bm.hot_path_info()["deferred"]
        if timing:
            r["times"] = bm.tick_times()
        res.append(r)
    launches = bm.launch_count()
    bm.close()
    return res, X.cpu().numpy(), launches


def check_identical(monkeypatch, sc, calls, min_deferred=1, **kw):
    ser, Xs, ls = run(monkeypatch, sc, calls, serial=True, **kw)
    ovl, Xo, lo = run(monkeypatch, sc, calls, serial=False, **kw)
    assert np.array_equal(Xs, Xo)
    for rs, ro in zip(ser, ovl):
        for k in rs:
            if k != "times":
                assert np.array_equal(rs[k], ro[k]), k
    assert sum(r["deferred"] for r in ser) >= min_deferred       # the scenario does defer hoppers
    if any(n > 1 for _, n, _ in calls):
        assert lo > ls                                           # and the overlapped handle did take the side stream
    else:
        assert lo == ls
    return ser, ovl


def test_default_batch_32_ticks_is_bit_identical(monkeypatch):
    sc = scenarios.make_batch(4096, N=10, n_ticks=33, seed=21)
    ser, ovl = check_identical(monkeypatch, sc, [(0, 32, True)], timing=True)
    for r in ser + ovl:
        mpc, sim = r["times"]
        assert len(mpc) == 32 and (mpc > 0).all() and (sim > 0).all()


def test_hard_workload_with_respawn_is_bit_identical(monkeypatch):
    sc = scenarios.make_batch(2048, N=10, n_ticks=21, seed=4, gain_spread=2.0, perturb=1.0)
    ser, _ = check_identical(monkeypatch, sc, [(0, 20, True)], min_deferred=20, on_infeasible="respawn")
    assert (ser[0]["status"] != 0).any()


def test_mostly_deferred_batch_is_bit_identical(monkeypatch):
    """HMPC_WARP_KCAP=40 sends most hoppers to the CTA kernel: more list entries than CTAs, long side-stream work
    against both parities of the tick buffers."""
    sc = scenarios.make_batch(1024, N=10, n_ticks=13, seed=9)
    check_identical(monkeypatch, sc, [(0, 12, True)], min_deferred=5000, kcap=40)


def test_split_rollout_and_single_ticks_are_bit_identical(monkeypatch):
    sc = scenarios.make_batch(2048, N=10, n_ticks=15, seed=3, gain_spread=2.0, perturb=1.0)
    check_identical(monkeypatch, sc, [(0, 1, True), (1, 5, False), (6, 1, False), (7, 3, False), (10, 4, False)],
                    on_infeasible="respawn")
    check_identical(monkeypatch, sc, [(0, 1, True), (1, 1, False), (2, 1, False)], min_deferred=0)   # one tick per call: serial


def test_per_hopper_bodies_are_bit_identical(monkeypatch):
    sc = scenarios.make_batch(2048, N=10, n_ticks=13, seed=31, body=True)
    check_identical(monkeypatch, sc, [(0, 12, True)], body=True)


def test_admm_solver_is_bit_identical(monkeypatch):
    sc = scenarios.make_batch(2048, N=10, n_ticks=11, seed=5, gain_spread=2.0, perturb=1.0)
    check_identical(monkeypatch, sc, [(0, 10, True)], min_deferred=0, solver="admm", on_infeasible="respawn")
    # systems over a smaller factor cap go to the CTA kernel: the ADMM warp kernel's deferral path
    check_identical(monkeypatch, sc, [(0, 10, True)], kcap=40, solver="admm", on_infeasible="respawn")
