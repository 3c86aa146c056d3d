"""Parity tests proper: the CUDA path through the C ABI (libhmpc_b200.so) against the oracle, the golden
fixtures frozen from the reference, and size-independent properties at BASELINE.json's batch sizes.
Run on the B200 box:  python -m pytest tests -m gpu -x -q"""
import numpy as np
import pytest
import torch

from hopper_mpc_inertial_b200 import _lib, scenarios
from oracle import device_port as dp
from oracle import hopper_oracle as ho
from oracle import qp_solvers as qs
from oracle.closed_loop import OracleMpc, QPFailed, closed_loop
from tests.conftest import golden, normalised_oracle_qp, u_tol

pytestmark = pytest.mark.gpu


def T(a, dev="cuda:0"):
    return torch.as_tensor(np.ascontiguousarray(a), device=dev)


def mk(B, dyn="3f", N=10, **kw):
    from hopper_mpc_inertial_b200.batch import BatchMpc
    return BatchMpc(B, dyn=dyn, N=N, device=0, **kw)


def cb64(c):
    return T(np.ascontiguousarray(c).view(np.int64))


# ---- stages -----------------------------------------------------------------------------------
def test_library_is_loaded_and_has_no_fallback():
    assert torch.cuda.is_available()
    lib = _lib.load()
    assert lib.hmpc_abi_version() == 2
    bm = mk(4)
    assert bm.launch_count() == 0
    bm.convert(T(np.tile(np.array([0, 0, .3, 1, 0, 0, 0, 0, 0, 0, 0, 0, 0.0])[:, None], (1, 4))))
    assert bm.launch_count() == 1


def test_sim_kernel_against_reference_golden():
    g = golden("sim.npz")
    K = g["X"].shape[0]
    bm = mk(K)
    x = bm.convert(T(g["X"].T)).cpu().numpy()
    np.testing.assert_allclose(x.T, g["x"], rtol=1e-13, atol=1e-13)
    X = T(g["X"].T).clone()
    Xs = bm.rk4(X, T(g["U"].T), T(g["pf"].T), 20, log_steps=True).cpu().numpy()
    np.testing.assert_allclose(Xs[0].T, g["Xn"], rtol=1e-13, atol=1e-13)
    np.testing.assert_allclose(Xs[19].T, g["X20"], rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(X.cpu().numpy().T, g["X20"], rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("dyn", ["3f", "2f"])
def test_linearise_and_condense_against_reference_golden(dyn):
    N = 10
    gl, gq = golden(f"lin_{dyn}.npz"), golden(f"qp_{dyn}.npz")
    prm = ho.Params(dyn=dyn, N=N)
    bm = mk(1, dyn, N)
    for ci in range(3):
        Ad, Bd = bm.linearize(T(gl[f"x_guess{ci}"][:, :, None]), T(gl[f"pf{ci}"][:, :, None]))
        np.testing.assert_allclose(Ad[..., 0].cpu().numpy(), gl[f"Ad{ci}"], rtol=0, atol=1e-15)
        np.testing.assert_allclose(Bd[..., 0].cpu().numpy(), gl[f"Bd{ci}"], rtol=0, atol=1e-13)
        C = gq[f"C{ci}"]
        cbits = np.array([sum(1 << k for k in range(N) if C[k] != 0)], np.uint64)
        H, g, lo, hi, inf = bm.condense(T(gq[f"x_in{ci}"][:, None]), T(gq[f"x_guess{ci}"][:, :, None]),
                                        T(gq[f"x_ref{ci}"][:, :, None]), T(gq[f"pf{ci}"][:, :, None]), cb64(cbits))
        Ao, Bo, Gd = ho.gen_dt_dynamics(gq[f"x_guess{ci}"], gq[f"pf{ci}"], prm)
        qc = ho.build_qp_condensed(gq[f"x_in{ci}"], gq[f"x_ref{ci}"], Ao, Bo, Gd, C, prm)
        A, l, u = normalised_oracle_qp(qc, prm)
        np.testing.assert_allclose(H[..., 0].cpu().numpy(), qc["H"], rtol=0, atol=1e-12 * np.abs(qc["H"]).max())
        np.testing.assert_allclose(g[:, 0].cpu().numpy(), qc["g"], rtol=0, atol=1e-12 * np.abs(qc["g"]).max())
        np.testing.assert_allclose(lo[:, 0].cpu().numpy(), l, rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(hi[:, 0].cpu().numpy(), u, rtol=1e-12, atol=1e-12)
        assert int(inf[0]) == 0


# ---- QP solutions -----------------------------------------------------------------------------
@pytest.mark.parametrize("dyn,N,B", [("3f", 10, 24), ("2f", 10, 24), ("3f", 20, 4), ("2f", 20, 4), ("3f", 60, 2),
                                     ("3f", 3, 5), ("2f", 5, 7), ("3f", 12, 3), ("3f", 40, 1)])
def test_mpcontrol_matches_oracle_optimum(dyn, N, B):
    """Per-step QP solutions within 1e-5 abs + 1e-4 rel of the exact optimum (FP64), first call (two solves)
    and a warm-started second call.  Horizons cover every kernel instantiation: 128-thread shared-memory
    (N <= 10, incl. the short horizons 3 and 5 and odd batch sizes) and the L2-workspace builds with four (12, 20)
    and two (40, 60) CTAs per SM."""
    sc = scenarios.make_batch(B, N=N, n_ticks=3, seed=13, dyn=dyn)
    bm = mk(B, dyn, N)
    bm.set_gains(T(sc["Qdiag"]), T(sc["Rdiag"]))
    x_in = bm.convert(T(sc["X0"])).cpu().numpy()
    mpcs = [OracleMpc(ho.Params(dyn=dyn, N=N, Qdiag=sc["Qdiag"][:, b].copy(), Rdiag=sc["Rdiag"][:, b].copy()))
            for b in range(B)]
    for t in range(2):
        U, Xs, st, it = bm.solve(T(x_in), T(sc["xref_tab"][t:t + N]), T(sc["pf_tab"][t:t + N]), cb64(sc["C_tab"][t]), t == 0)
        U, Xs, st = U.cpu().numpy(), Xs.cpu().numpy(), st.cpu().numpy()
        assert np.all(st == 0), st
        for b in range(B):
            Uo = mpcs[b].mpcontrol(x_in[:, b], sc["xref_tab"][t:t + N, :, b], sc["pf_tab"][t:t + N, :, b], sc["C"][t, b], t == 0)
            assert np.all(np.abs(U[:, :, b] - Uo) <= u_tol(Uo)), (t, b, np.abs(U[:, :, b] - Uo).max())
            np.testing.assert_allclose(Xs[:, :, b], mpcs[b].xval, rtol=1e-6, atol=1e-7)
        nf, pa, ni = [a.cpu().numpy() for a in bm.solve_stats()]
        if t == 1:
            assert np.sum(pa == _lib.PATH_WARM) > 0


@pytest.mark.parametrize("dyn,precision", [("3f", "fp64"), ("2f", "fp64"), ("3f", "fp32"), ("2f", "fp32")])
def test_closed_loop_rollout_matches_oracle(dyn, precision):
    """fp32 = FP32 factorisation / substitution, FP64 data and refinement (mixed precision): the accepted
    points pass the same KKT test of the original QP, so the FP64 parity bound is kept."""
    B, N, n_ticks = 8, 10, 30
    sc = scenarios.make_batch(B, N=N, n_ticks=n_ticks, seed=7, dyn=dyn)
    bm = mk(B, dyn, N, precision=precision)
    bm.set_gains(T(sc["Qdiag"]), T(sc["Rdiag"]))
    X = T(sc["X0"]).clone()
    out = bm.rollout(X, T(sc["xref_tab"]), T(sc["pf_tab"]), cb64(sc["C_tab"]), T(sc["pf_switch"]), 0, n_ticks, True, log=True)
    st = out["status"].cpu().numpy()
    if precision == "fp64":
        assert np.all(st == 0)
    else:
        # the FP32 interior point can stall on near-infeasible QPs (status MAX_ITER / INEXACT, never a wrong
        # SOLVED); parity is asserted on the hoppers whose every tick was verified
        assert np.sum(st == 0) >= B - 1, st
    Xg, Ug = out["X_log"].cpu().numpy(), out["U_log"].cpu().numpy()
    for b in range(B):
        if st[b] != 0:
            continue
        p = ho.Params(dyn=dyn, N=N, Qdiag=sc["Qdiag"][:, b].copy(), Rdiag=sc["Rdiag"][:, b].copy())
        Xo, Uo = closed_loop(p, sc["X0"][:, b], sc["xref_tab"][:, :, b], sc["pf_tab"][:, :, b], sc["C"][:, b],
                             sc["pf_switch"][:, b], n_ticks)
        assert np.all(np.abs(Ug[:, :, b] - Uo) <= 10 * u_tol(Uo)), np.abs(Ug[:, :, b] - Uo).max()
        # closed-loop state tolerance: 1e-6 abs (errors of the per-tick optimum feed back through the loop)
        np.testing.assert_allclose(Xg[:, :, b], Xo, rtol=0, atol=1e-6)


@pytest.mark.parametrize("dyn", ["3f", "2f"])
def test_warp_kernel_equals_cta_kernel_and_oracle(dyn):
    """hot_path auto (warp-per-hopper kernel + CTA fallback for the hoppers it defers) against hot_path cta (round-1
    CTA-per-hopper kernel only) and against the oracle loop: same closed loop, every tick KKT-verified, and the warp
    kernel really carried the warm ticks (deferred fraction small)."""
    B, N, n_ticks = 256, 10, 40
    sc = scenarios.make_batch(B, N=N, n_ticks=n_ticks, seed=11, dyn=dyn)
    logs = {}
    for mode in ("auto", "cta"):
        bm = mk(B, dyn, N, hot_path=mode)
        bm.set_gains(T(sc["Qdiag"]), T(sc["Rdiag"]))
        X = T(sc["X0"]).clone()
        out = bm.rollout(X, T(sc["xref_tab"]), T(sc["pf_tab"]), cb64(sc["C_tab"]), T(sc["pf_switch"]), 0, n_ticks, True, log=True)
        info = bm.hot_path_info()
        logs[mode] = (out["X_log"].cpu().numpy(), out["U_log"].cpu().numpy(), out["status"].cpu().numpy(), info)
    Xa, Ua, sa, ia = logs["auto"]
    Xc, Uc, sc_, ic = logs["cta"]
    assert ia["warps_per_sm"] >= 8 and ic["warps_per_sm"] == 0
    assert ia["deferred"] < 0.1 * B * (n_ticks - 1), ia
    ok = (sa == 0) & (sc_ == 0)
    assert ok.sum() >= B - 4, (sa, sc_)
    # both paths return the KKT-verified optimum of every tick: the closed loops agree far below the parity bound
    assert np.abs(Ua[:, :, ok] - Uc[:, :, ok]).max() < 1e-5
    np.testing.assert_allclose(Xa[:, :, ok], Xc[:, :, ok], rtol=0, atol=1e-6)
    for b in np.where(ok)[0][:6]:
        p = ho.Params(dyn=dyn, N=N, Qdiag=sc["Qdiag"][:, b].copy(), Rdiag=sc["Rdiag"][:, b].copy())
        Xo, Uo = closed_loop(p, sc["X0"][:, b], sc["xref_tab"][:, :, b], sc["pf_tab"][:, :, b], sc["C"][:, b],
                             sc["pf_switch"][:, b], n_ticks)
        assert np.all(np.abs(Ua[:, :, b] - Uo) <= 10 * u_tol(Uo)), np.abs(Ua[:, :, b] - Uo).max()
        np.testing.assert_allclose(Xa[:, :, b], Xo, rtol=0, atol=1e-6)


def test_sqp_sweeps_match_oracle():
    """hmpc_config.sqp_sweeps = 2 (SURVEY 8 f4): every tick relinearises about its own solution once and solves
    again; same parity bound against the oracle driver doing the same."""
    B, N, n_ticks = 4, 10, 20
    sc = scenarios.make_batch(B, N=N, n_ticks=n_ticks, seed=11)
    bm = mk(B, "3f", N, sqp_sweeps=2)
    bm.set_gains(T(sc["Qdiag"]), T(sc["Rdiag"]))
    out = bm.rollout(T(sc["X0"]).clone(), T(sc["xref_tab"]), T(sc["pf_tab"]), cb64(sc["C_tab"]), T(sc["pf_switch"]),
                     0, n_ticks, True, log=True)
    assert np.all(out["status"].cpu().numpy() == 0)
    Xg, Ug = out["X_log"].cpu().numpy(), out["U_log"].cpu().numpy()
    for b in range(B):
        p = ho.Params(dyn="3f", N=N, Qdiag=sc["Qdiag"][:, b].copy(), Rdiag=sc["Rdiag"][:, b].copy())
        Xo, Uo = closed_loop(p, sc["X0"][:, b], sc["xref_tab"][:, :, b], sc["pf_tab"][:, :, b], sc["C"][:, b],
                             sc["pf_switch"][:, b], n_ticks, sqp_sweeps=2)
        assert np.all(np.abs(Ug[:, :, b] - Uo) <= 10 * u_tol(Uo)), np.abs(Ug[:, :, b] - Uo).max()
        np.testing.assert_allclose(Xg[:, :, b], Xo, rtol=0, atol=1e-6)
        Xo1, _ = closed_loop(p, sc["X0"][:, b], sc["xref_tab"][:, :, b], sc["pf_tab"][:, :, b], sc["C"][:, b],
                             sc["pf_switch"][:, b], n_ticks)
        assert np.abs(Xo1 - Xo).max() > 1e-5           # the option does change the loop


@pytest.mark.parametrize("tag,dyn", [("loop_2f", "2f"), ("loop_3f_curve", "3f"), ("loop_3f_curve_5s", "3f")])
def test_reference_runs_2000ms_N60(tag, dyn):
    """BASELINE configs[0] and [1]: run.py 2f --N_run 2000, run.py 3f --curve --N_run 2000 and run.py 3f --curve
    (default 5 s) at the reference's horizon N = 60 and constants: closed-loop trajectory against the oracle
    loop frozen in tests/golden.  State tolerance 1e-5 abs over 100 / 250 ticks."""
    g = golden(f"{tag}.npz")
    N, n_ticks = int(g["N"]), int(g["n_ticks"])
    bm = mk(1, dyn, N)
    X = T(g["X0"][:, None]).clone()
    out = bm.rollout(X, T(g["xref_tab"][:, :, None]), T(g["pf_tab"][:, :, None]),
                     cb64(_cbits(g["C"]).reshape(n_ticks, 1)), T(g["pf_switch"].reshape(n_ticks, 1).astype(np.uint8)),
                     0, n_ticks, True, log=True)
    assert int(out["status"][0]) == 0
    Xg, Ug = out["X_log"][:, :, 0].cpu().numpy(), out["U_log"][:, :, 0].cpu().numpy()
    np.testing.assert_allclose(Xg, g["X_log"], rtol=0, atol=1e-5)
    assert np.all(np.abs(Ug - g["U_log"]) <= 1e-3 + 1e-4 * np.abs(g["U_log"]))


def _cbits(C):
    from hopper_mpc_inertial_b200.batch import cbits_from_C
    return cbits_from_C(C)


# ---- properties at full batch size ------------------------------------------------------------
def test_fp32_mode_batch_matches_fp64_mode():
    """BASELINE configs[3] asks for FP32 and FP64 modes: over a 2048-hopper closed loop the mixed-precision
    mode solves (almost) every QP to the verified optimum and its trajectories stay within 1e-6 of FP64's."""
    B, N, n_ticks = 2048, 10, 10
    sc = scenarios.make_batch(B, N=N, n_ticks=n_ticks, seed=17)
    res = {}
    for prec in ("fp64", "fp32"):
        bm = mk(B, "3f", N, precision=prec)
        bm.set_gains(T(sc["Qdiag"]), T(sc["Rdiag"]))
        X = T(sc["X0"]).clone()
        out = bm.rollout(X, T(sc["xref_tab"]), T(sc["pf_tab"]), cb64(sc["C_tab"]), T(sc["pf_switch"]), 0, n_ticks, True, log=True)
        res[prec] = (X.cpu().numpy(), out["U_log"].cpu().numpy(), out["status"].cpu().numpy())
    st64, st32 = res["fp64"][2], res["fp32"][2]
    assert np.mean(st32 == 0) > 0.995, np.bincount(st32, minlength=5)
    ok = (st64 == 0) & (st32 == 0)
    assert np.abs(res["fp64"][0][:, ok] - res["fp32"][0][:, ok]).max() < 1e-6
    U64, U32 = res["fp64"][1][:, :, ok], res["fp32"][1][:, :, ok]
    assert np.all(np.abs(U64 - U32) <= 10 * u_tol(U64))


def test_batch_4096_properties():
    """BASELINE config 3 (3f, 4096 hoppers, horizon 10): every hopper is either solved exactly or flagged
    infeasible; results are bit-identical between two runs, between a hopper inside the batch and the same
    hopper in a smaller batch, and a random sample passes the solver-independent KKT certificate."""
    B, N, n_ticks = 4096, 10, 12
    sc = scenarios.make_batch(B, N=N, n_ticks=n_ticks)

    def run(lo, hi, log=True):
        bm = mk(hi - lo, "3f", N)
        sl = slice(lo, hi)
        bm.set_gains(T(sc["Qdiag"][:, sl]), T(sc["Rdiag"][:, sl]))
        X = T(sc["X0"][:, sl]).clone()
        out = bm.rollout(X, T(sc["xref_tab"][..., sl]), T(sc["pf_tab"][..., sl]), cb64(sc["C_tab"][:, sl]),
                         T(sc["pf_switch"][:, sl]), 0, n_ticks, True, log=log)
        return bm, X.cpu().numpy(), out

    bm, X1, o1 = run(0, B)
    st = o1["status"].cpu().numpy()
    assert np.all((st == 0) | (st == 2)), np.bincount(st, minlength=5)
    assert np.mean(st == 0) > 0.99
    assert np.all(np.isfinite(X1))
    _, X2, o2 = run(0, B)
    assert np.array_equal(X1, X2) and torch.equal(o1["U_log"], o2["U_log"])
    _, X3, o3 = run(1000, 1064)
    assert np.array_equal(X3, X1[:, 1000:1064])
    # Full optimality check at this batch size: two more mpcontrol calls on the final states.  The first returns its
    # x.value, so the linearisation point of the second (the time shift, mpc_cvx_euler_3f.py:59-62) is known here and
    # the oracle can rebuild exactly the QP the device solved; a sample of hoppers is compared with the oracle's
    # exact optimum and run through the solver-independent KKT certificate.
    t = n_ticks
    x_in = bm.convert(T(X1)).cpu().numpy()
    win = lambda a: T(np.ascontiguousarray(a[t - 1:t - 1 + N]))
    _, XsA, stA, _ = bm.solve(T(x_in), win(sc["xref_tab"]), win(sc["pf_tab"]), cb64(sc["C_tab"][t - 1]), False)
    XsA = XsA.cpu().numpy()
    U, Xs, st2, it = bm.solve(T(x_in), win(sc["xref_tab"]), win(sc["pf_tab"]), cb64(sc["C_tab"][t - 1]), False)
    U, Xs, st2, stA = U.cpu().numpy(), Xs.cpu().numpy(), st2.cpu().numpy(), stA.cpu().numpy()
    rng = np.random.default_rng(0)
    checked = 0
    for b in rng.choice(B, 48, replace=False):
        if st2[b] != 0 or stA[b] != 0:
            continue
        p = ho.Params(dyn="3f", N=N, Qdiag=sc["Qdiag"][:, b].copy(), Rdiag=sc["Rdiag"][:, b].copy())
        x_guess = np.vstack((x_in[None, :, b], XsA[2:, :, b], XsA[-1:, :, b]))
        Ad, Bd, Gd = ho.gen_dt_dynamics(x_guess, sc["pf_tab"][t - 1:t - 1 + N, :, b], p)
        qp = ho.build_qp_condensed(x_in[:, b], sc["xref_tab"][t - 1:t - 1 + N, :, b], Ad, Bd, Gd, sc["C"][t - 1, b], p)
        ref = qs.exact_qp(qp["H"], qp["g"], qp["A"], qp["l"], qp["u"])
        assert ref["ok"]
        u = U[:, :, b].reshape(-1)
        assert np.all(np.abs(u - ref["x"]) <= u_tol(ref["x"])), (b, np.abs(u - ref["x"]).max())
        cert = qs.kkt_certificate(qp["H"], qp["g"], qp["A"], qp["l"], qp["u"], u, ref["y"])
        gs = max(1.0, np.abs(qp["g"]).max())
        assert cert["prim"] < 1e-8 and cert["stat"] < 1e-6 * gs and cert["sign"] < 1e-6 * gs, cert
        checked += 1
    assert checked >= 40


def test_kkt_certificate_on_device_solutions():
    """Solver-independent certificate: stationarity, feasibility, complementarity and multiplier signs of
    the device's (U, active set) on QPs rebuilt by the oracle for the same linearisation point."""
    B, N = 64, 10
    sc = scenarios.make_batch(B, N=N, n_ticks=2, seed=99)
    bm = mk(B, "3f", N)
    bm.set_gains(T(sc["Qdiag"]), T(sc["Rdiag"]))
    x_in = bm.convert(T(sc["X0"])).cpu().numpy()
    U, Xs, st, it = bm.solve(T(x_in), T(sc["xref_tab"][:N]), T(sc["pf_tab"][:N]), cb64(sc["C_tab"][0]), True)
    U, st = U.cpu().numpy(), st.cpu().numpy()
    assert np.all(st == 0)
    for b in range(B):
        p = ho.Params(dyn="3f", N=N, Qdiag=sc["Qdiag"][:, b].copy(), Rdiag=sc["Rdiag"][:, b].copy())
        om = OracleMpc(p)
        om.mpcontrol(x_in[:, b], sc["xref_tab"][:N, :, b], sc["pf_tab"][:N, :, b], sc["C"][0, b], True)
        qp = om.last["qp"]                               # QP of the second (final) solve
        u = U[:, :, b].reshape(-1)
        # multipliers from the oracle's active set; the certificate is evaluated at the DEVICE's point
        cert = qs.kkt_certificate(qp["H"], qp["g"], qp["A"], qp["l"], qp["u"], u, om.last["res"]["y"])
        gs = max(1.0, np.abs(qp["g"]).max())
        assert cert["prim"] < 1e-8 and cert["stat"] < 1e-6 * gs, cert


def test_admm_mode_matches_numpy_port():
    """OSQP-style ADMM kernel: fixed-iteration iterate equals the numpy statement; early-exit stops at the
    same iteration with OSQP's residual test met at eps = 1e-5 (cvxpy's setting)."""
    N, B, dyn = 10, 8, "3f"
    sc = scenarios.make_batch(B, N=N, n_ticks=2, seed=5, dyn=dyn)
    qps = None
    for kw, fixed in ((dict(mode="fixed_iter", max_iter=40, polish=0), True), (dict(mode="early_exit", max_iter=4000, polish=0), False)):
        bm = mk(B, dyn, N, solver="admm", warm_start=0, **kw)
        bm.set_gains(T(sc["Qdiag"]), T(sc["Rdiag"]))
        x_in = bm.convert(T(sc["X0"])).cpu().numpy()
        xref, pfw = sc["xref_tab"][:N], sc["pf_tab"][:N]
        x_guess = np.concatenate((x_in[None], xref), 0)
        # prime the handle's previous trajectory so that the time shift reproduces x_guess: run an init solve
        # on a copy of the problem is not needed -- compare through hmpc_condense'd data instead
        H, g, lo, hi, inf = [a.cpu().numpy() for a in bm.condense(T(x_in), T(x_guess), T(xref), T(pfw), cb64(sc["C_tab"][0]))]
        U, Xs, st, it = bm.solve(T(x_in), T(xref), T(pfw), cb64(sc["C_tab"][0]), True)
        U, st, it = U.cpu().numpy(), st.cpu().numpy(), it.cpu().numpy()
        for b in range(B):
            p = ho.Params(dyn=dyn, N=N, Qdiag=sc["Qdiag"][:, b].copy(), Rdiag=sc["Rdiag"][:, b].copy())
            # replay the init call's two solves with the numpy port
            Ad, Bd, Gd = ho.gen_dt_dynamics(x_guess[:, :, b], pfw[:, :, b], p)
            qc = ho.build_qp_condensed(x_in[:, b], xref[:, :, b], Ad, Bd, Gd, sc["C"][0, b], p)
            A, l, u = normalised_oracle_qp(qc, p)
            np.testing.assert_allclose(H[..., b], qc["H"], rtol=0, atol=1e-12 * np.abs(qc["H"]).max())
            x1, y1, c1, i1 = dp.admm_solve(qc["H"], qc["g"], A, l, u, max_iter=kw["max_iter"], fixed_iter=fixed)
            xg2 = ho.rollout_linear(x_in[:, b], x1.reshape(N, 6), Ad, Bd, Gd, p)
            Ad2, Bd2, Gd2 = ho.gen_dt_dynamics(xg2, pfw[:, :, b], p)
            qc2 = ho.build_qp_condensed(x_in[:, b], xref[:, :, b], Ad2, Bd2, Gd2, sc["C"][0, b], p)
            A2, l2, u2 = normalised_oracle_qp(qc2, p)
            x2, y2, c2, i2 = dp.admm_solve(qc2["H"], qc2["g"], A2, l2, u2, max_iter=kw["max_iter"], fixed_iter=fixed)
            assert it[b] == i1["iters"] + i2["iters"]
            np.testing.assert_allclose(U[:, :, b].reshape(-1), x2, rtol=1e-6, atol=1e-6)
            if not fixed:
                assert st[b] == 4 and i2["status"] == dp.ST_INEXACT


@pytest.mark.parametrize("dyn", ["3f", "2f"])
def test_admm_with_polish_reaches_the_oracle_optimum(dyn):
    """solver = admm (OSQP iteration at cvxpy's eps 1e-5) followed by the verified polish (OSQP polish=True): the
    returned point is the certified optimum of the QP, within the north_star bound of the oracle's exact solver."""
    N, B = 10, 16
    sc = scenarios.make_batch(B, N=N, n_ticks=2, seed=23, dyn=dyn)
    bm = mk(B, dyn, N, solver="admm", warm_start=0, mode="early_exit", max_iter=4000, polish=1)
    bm.set_gains(T(sc["Qdiag"]), T(sc["Rdiag"]))
    x_in = bm.convert(T(sc["X0"])).cpu().numpy()
    U, Xs, st, it = bm.solve(T(x_in), T(sc["xref_tab"][:N]), T(sc["pf_tab"][:N]), cb64(sc["C_tab"][0]), True)
    U, st = U.cpu().numpy(), st.cpu().numpy()
    assert np.mean(st == 0) >= 0.9, st            # polished and KKT-verified (the rest stays SOLVED_INEXACT)
    for b in np.where(st == 0)[0]:
        p = ho.Params(dyn=dyn, N=N, Qdiag=sc["Qdiag"][:, b].copy(), Rdiag=sc["Rdiag"][:, b].copy())
        Uo = OracleMpc(p).mpcontrol(x_in[:, b], sc["xref_tab"][:N, :, b], sc["pf_tab"][:N, :, b], sc["C"][0, b], True)
        assert np.all(np.abs(U[:, :, b] - Uo) <= u_tol(Uo)), (b, np.abs(U[:, :, b] - Uo).max())


def test_admm_early_exit_matches_independent_osqp_restatement():
    """The ADMM kernel against oracle/qp_solvers.osqp_solve -- the independent restatement of OSQP, not the numpy port
    of the device code: same condensed QP (variables the contact schedule fixes eliminated, as the kernel does), no
    Ruiz scaling, cold start, rho adaptation at every check.  Both stop at the same iteration, i.e. the first check at
    which OSQP's residual test passes at eps = 1e-5, and the iterates agree to 1e-6."""
    N, B, dyn = 10, 8, "3f"
    sc = scenarios.make_batch(B, N=N, n_ticks=3, seed=5, dyn=dyn)
    bm = mk(B, dyn, N, solver="admm", warm_start=0, mode="early_exit", max_iter=4000, polish=0)
    bm.set_gains(T(sc["Qdiag"]), T(sc["Rdiag"]))
    x_in = bm.convert(T(sc["X0"])).cpu().numpy()
    xref, pfw, cb = sc["xref_tab"][:N], sc["pf_tab"][:N], cb64(sc["C_tab"][0])
    _, Xs1, _, _ = bm.solve(T(x_in), T(xref), T(pfw), cb, True)          # primes the handle's x.value
    Xs1 = Xs1.cpu().numpy()
    U, Xs, st, it = bm.solve(T(x_in), T(xref), T(pfw), cb, False)        # ONE cold ADMM solve about the time shift
    U, st, it = U.cpu().numpy(), st.cpu().numpy(), it.cpu().numpy()
    for b in range(B):
        p = ho.Params(dyn=dyn, N=N, Qdiag=sc["Qdiag"][:, b].copy(), Rdiag=sc["Rdiag"][:, b].copy())
        x_guess = np.vstack((x_in[None, :, b], Xs1[2:, :, b], Xs1[-1:, :, b]))   # mpc_cvx_euler_3f.py:59-62
        Ad, Bd, Gd = ho.gen_dt_dynamics(x_guess, pfw[:, :, b], p)
        qc = ho.build_qp_condensed(x_in[:, b], xref[:, :, b], Ad, Bd, Gd, sc["C"][0, b], p)
        A, lo, hi = normalised_oracle_qp(qc, p)
        n = 6 * N
        F = np.where((hi[:n] - lo[:n]) >= 1e-12)[0]
        r = qs.osqp_solve(qc["H"][np.ix_(F, F)], qc["g"][F], A[:, F], lo, hi, scaling=0, polish=False, check_termination=25,
                          adaptive_rho_interval=25, max_iter=4000)
        assert r["status"] == "solved" and st[b] == 4          # SOLVED_INEXACT: residual test met, not polished
        assert it[b] == r["iters"], (b, it[b], r["iters"])
        u = U[:, :, b].reshape(-1)
        np.testing.assert_allclose(u[F], r["x"], rtol=0, atol=1e-6)
        assert np.all(u[np.setdiff1d(np.arange(n), F)] == 0.0)


@pytest.mark.parametrize("tag,dyn", [("loop_ref_2f", "2f"), ("loop_ref_3f_curve", "3f")])
def test_closed_loop_matches_the_references_own_runner(tag, dyn):
    """tests/golden/loop_ref_*.npz hold the first 12 ticks of the REFERENCE'S OWN Runner.run (robotrunner.py:81-124,
    executed unmodified through oracle/refshim.py at its real horizon N = 60; OSQP restated at cvxpy's settings
    eps 1e-5 + polish, oracle/make_loop_ref.py).  The GPU closed loop lands on it within 1e-3 N / 1e-3 Nm in every
    applied control and 1e-5 in the state (measured: 2.6e-4 and 2.3e-6: what is left is OSQP's own eps)."""
    g = golden(f"{tag}.npz")
    N, n_ticks = int(g["N"]), int(g["n_ticks"])
    bm = mk(1, dyn, N)
    X = T(g["X0"][:, None]).clone()
    out = bm.rollout(X, T(g["xref_tab"][:, :, None]), T(g["pf_tab"][:, :, None]),
                     cb64(_cbits(g["C"]).reshape(n_ticks, 1)), T(g["pf_switch"].reshape(n_ticks, 1).astype(np.uint8)),
                     0, n_ticks, True, log=True)
    assert int(out["status"][0]) == 0
    Xg, Ug = out["X_log"][:, :, 0].cpu().numpy(), out["U_log"][:, :, 0].cpu().numpy()
    assert np.abs(Ug - g["U_log"]).max() < 1e-3, np.abs(Ug - g["U_log"]).max()
    np.testing.assert_allclose(Xg, g["X_log"], rtol=0, atol=1e-5)


def test_respawn_keeps_every_hopper_running():
    B, N, n_ticks = 512, 10, 40
    sc = scenarios.make_batch(B, N=N, n_ticks=n_ticks, seed=4, gain_spread=2.0, perturb=1.0)   # harsher -> some fail
    for mode in ("hold", "respawn"):
        bm = mk(B, "3f", N, on_infeasible=mode)
        bm.set_gains(T(sc["Qdiag"]), T(sc["Rdiag"]))
        X = T(sc["X0"]).clone()
        out = bm.rollout(X, T(sc["xref_tab"]), T(sc["pf_tab"]), cb64(sc["C_tab"]), T(sc["pf_switch"]), 0, n_ticks, True)
        nf, pa, ni = [a.cpu().numpy() for a in bm.solve_stats()]
        assert np.all(np.isfinite(X.cpu().numpy()))
        st = out["status"].cpu().numpy()
        assert np.all((st == 0) | (st == 2))
        if mode == "hold":
            n_hold = int((ni > 0).sum())
        else:
            # a respawned hopper is back on its reference and solvable again: few infeasible ticks each
            assert ni.max() <= 0.25 * n_ticks
            assert X.cpu().numpy()[2].min() > 0.05
    assert n_hold > 0


# ---- drop-in classes ----------------------------------------------------------------------------
@pytest.mark.parametrize("dyn", ["3f", "2f"])
def test_dropin_mpc_class(dyn):
    from hopper_mpc_inertial_b200 import mpc_cvx_euler_2f, mpc_cvx_euler_3f
    mod = mpc_cvx_euler_3f if dyn == "3f" else mpc_cvx_euler_2f
    N = 10
    prm = ho.Params(dyn=dyn, N=N)
    mpc = mod.Mpc(t=0.02, N=N, m=7.5, g=9.807, mu=1, Jinv=prm.Jinv, rh=prm.rh)
    g = golden(f"qp_{dyn}.npz")
    om = OracleMpc(prm)
    for ci, init in ((1, True), (1, False)):
        U = mpc.mpcontrol(x_in=g[f"x_in{ci}"], x_ref_in=g[f"x_ref{ci}"], pf=g[f"pf{ci}"], C=g[f"C{ci}"], init=init)
        Uo = om.mpcontrol(g[f"x_in{ci}"], g[f"x_ref{ci}"], g[f"pf{ci}"], g[f"C{ci}"], init)
        assert U.shape == (N, 6) and U.dtype == np.float64
        assert np.all(np.abs(U - Uo) <= u_tol(Uo))
        np.testing.assert_allclose(mpc.x.value, om.xval, rtol=1e-6, atol=1e-7)
    # gains are public attributes (mpc_cvx_euler_3f.py:34-37): changing them changes the solution
    mpc.Q[2, 2] = 20.0
    prm2 = ho.Params(dyn=dyn, N=N); prm2.Qdiag[2] = 20.0
    U2 = mpc.mpcontrol(x_in=g["x_in0"], x_ref_in=g["x_ref0"], pf=g["pf0"], C=g["C0"], init=True)
    Uo2 = OracleMpc(prm2).mpcontrol(g["x_in0"], g["x_ref0"], g["pf0"], g["C0"], True)
    assert np.all(np.abs(U2 - Uo2) <= u_tol(Uo2))
    # infeasible -> the reference's exception text (mpc_cvx_euler_3f.py:158-159)
    x_bad = g["x_in0"].copy(); x_bad[2] = 0.05
    with pytest.raises(Exception, match="QP FAILED"):
        mpc.mpcontrol(x_in=x_bad, x_ref_in=g["x_ref0"], pf=g["pf0"], C=g["C0"], init=True)
    assert mpc.u.value is None


def test_runner_and_cli_dropin():
    """Runner(dt, dyn, curve, N_run).run() tick by tick through Mpc.mpcontrol equals the fused rollout."""
    from hopper_mpc_inertial_b200 import run as cli
    from hopper_mpc_inertial_b200.robotrunner import Runner
    r = cli.main(["3f", "--curve", "--N_run", "200", "--horizon", "10"])
    assert r.X_traj.shape == (201, 13) and r.f_hist.shape == (201, 6)
    r2 = Runner(dt=1e-3, dyn="3f", curve=True, N_run=200, N=10)
    X_log, U_log = r2.run_fused()
    np.testing.assert_allclose(r.X_traj[::20], X_log, rtol=0, atol=1e-9)
    np.testing.assert_allclose(r.f_hist[0:200:20], U_log, rtol=0, atol=1e-7)
    r3 = cli.main(["2f", "--runtime", "100", "--horizon", "10"])       # README spelling (SURVEY App. D10)
    assert r3.X_traj.shape == (101, 13)


def _plan_set(bm, sc, dev="cuda:0"):
    from hopper_mpc_inertial_b200 import planner
    p = sc["plan"]
    gt = planner.global_tables(**p["global_args"])
    bm.plan_set(T(p["x0"], dev), T(p["xf"], dev), T(p["curve"], dev), T(p["tick_offset"], dev), gt)


@pytest.mark.parametrize("dyn,N", [("3f", 10), ("2f", 10), ("3f", 20)])
def test_device_planner_tables_are_bit_identical(dyn, N):
    """SURVEY 8 row f1: path_plan_init / path_plan_grab / gait_map generated on the device (hmpc_plan_tables) against
    the numpy planner (planner.batch_tables, itself pinned to the reference's path_plan_init by planner.npz)."""
    B, n_ticks = 777, 37
    sc = scenarios.make_batch(B, N=N, n_ticks=n_ticks, seed=11, dyn=dyn)
    bm = mk(B, dyn, N)
    _plan_set(bm, sc)
    tabs = bm.plan_tables(0, n_ticks)
    assert np.array_equal(tabs["xref_tab"].cpu().numpy(), sc["xref_tab"])
    assert np.array_equal(tabs["pf_tab"].cpu().numpy(), sc["pf_tab"])
    assert np.array_equal(tabs["C_tab"].cpu().numpy().view(np.uint64), sc["C_tab"])
    assert np.array_equal(tabs["pf_switch"].cpu().numpy(), sc["pf_switch"])
    late = bm.plan_tables(9, 3)
    assert np.array_equal(late["xref_tab"].cpu().numpy(), sc["xref_tab"][9:9 + 3 + N])
    assert np.array_equal(late["pf_tab"].cpu().numpy(), sc["pf_tab"][9:9 + 3 + N + 1])


def test_planned_rollout_equals_table_rollout():
    """hmpc_rollout_planned (reference window generated per tick on the device, nothing uploaded) reproduces
    hmpc_rollout on the host-built tables bit for bit, respawns included."""
    B, N, n_ticks = 512, 10, 24
    sc = scenarios.make_batch(B, N=N, n_ticks=n_ticks, seed=3, gain_spread=2.0, perturb=1.0)
    res = []
    for planned in (False, True):
        bm = mk(B, "3f", N, on_infeasible="respawn")
        bm.set_gains(T(sc["Qdiag"]), T(sc["Rdiag"]))
        X = T(sc["X0"]).clone()
        if planned:
            _plan_set(bm, sc)
            out = bm.rollout_planned(X, 0, 10, True, log=True)
            out2 = bm.rollout_planned(X, 10, n_ticks - 10, False, log=True)     # resumed mid-run
        else:
            args = (T(sc["xref_tab"]), T(sc["pf_tab"]), cb64(sc["C_tab"]), T(sc["pf_switch"]))
            out = bm.rollout(X, *args, 0, 10, True, log=True)
            out2 = bm.rollout(X, *args, 10, n_ticks - 10, False, log=True)
        torch.cuda.synchronize()
        res.append((X.cpu().numpy(), out["U_log"].cpu().numpy(), out2["U_log"].cpu().numpy(), bm.solve_stats()[2].cpu().numpy()))
    for a, b in zip(res[0], res[1]):
        assert np.array_equal(a, b)
    assert res[0][3].sum() > 0        # the scenario does exercise the respawn path


def test_work_order_stress_is_bit_identical(monkeypatch):
    """Race / stale-state stress (compute-sanitizer is closed on this pool): the same closed loop is repeated with the
    hoppers handed to the persistent warps / CTAs in 24 different orders (HMPC_WORK_PERM: ticket i -> hopper
    (i mul + add) mod B, so every hopper meets other neighbours, other shared-memory slices and another position in
    its lock-step group); states, controls, statuses and factorisation counts must be bit-identical every time."""
    B, N, n_ticks = 1531, 10, 7                     # a prime batch: every multiplier is a permutation
    sc = scenarios.make_batch(B, N=N, n_ticks=n_ticks, seed=17, gain_spread=2.0, perturb=1.0)
    args = None
    ref = None
    rng = np.random.default_rng(0)
    perms = [(1, 0)] + [(int(m), int(a)) for m, a in zip(rng.integers(2, B, 23), rng.integers(0, B, 23))]
    for mul, add in perms:
        monkeypatch.setenv("HMPC_WORK_PERM", f"{mul},{add}")
        bm = mk(B, "3f", N, on_infeasible="respawn")
        bm.set_gains(T(sc["Qdiag"]), T(sc["Rdiag"]))
        if args is None:
            args = (T(sc["xref_tab"]), T(sc["pf_tab"]), cb64(sc["C_tab"]), T(sc["pf_switch"]))
        X = T(sc["X0"]).clone()
        out = bm.rollout(X, *args, 0, n_ticks, True, log=True)
        torch.cuda.synchronize()
        got = (X.cpu().numpy(), out["U_log"].cpu().numpy(), out["status"].cpu().numpy(), bm.solve_stats()[0].cpu().numpy())
        bm.close()
        if ref is None:
            ref = got
        else:
            for a, b in zip(ref, got):
                assert np.array_equal(a, b), (mul, add)


def test_runner_forwards_a_non_default_dt():
    """Runner(dt=2e-3): the device integrates with h = dt and runs mpc_dt / dt = 10 steps per tick
    (robotrunner.py:48,154-164); both loops agree with the oracle loop run with the same constants."""
    from hopper_mpc_inertial_b200 import planner
    from hopper_mpc_inertial_b200.robotrunner import Runner
    dt, N, N_run = 2e-3, 10, 120
    r = Runner(dt=dt, dyn="3f", curve=True, N_run=N_run, N=N, progress=False)
    assert r.mpc_factor == 10
    X_log, U_log = r.run_fused()
    n_ticks = N_run // r.mpc_factor
    xt, pt, C, sw = planner.mpc_tables(r.x_ref, r.pf_ref, n_ticks, N, r.mpc_factor, dt, r.mpc_dt, r.t_start)
    prm = ho.Params(dyn="3f", N=N, sim_dt=dt, mpc_factor=r.mpc_factor)
    Xo, Uo = closed_loop(prm, r.X_0, xt, pt, C, sw, n_ticks)
    assert np.all(np.abs(U_log - Uo) <= 10 * u_tol(Uo))
    np.testing.assert_allclose(X_log, Xo, rtol=0, atol=1e-6)
    r2 = Runner(dt=dt, dyn="3f", curve=True, N_run=N_run, N=N, progress=False)
    r2.run()
    np.testing.assert_allclose(r2.X_traj[::r2.mpc_factor], X_log, rtol=0, atol=1e-9)
    # and the default step really differs (the test would not notice a dropped override otherwise)
    r3 = Runner(dt=1e-3, dyn="3f", curve=True, N_run=N_run, N=N, progress=False)
    assert np.abs(r3.run_fused()[0][1] - X_log[1]).max() > 1e-4


def test_sharded_run_equals_unsharded():
    """Sharding by hopper (SURVEY 8e): two shards -- on two GPUs when the box has them, else two handles on one
    GPU -- reproduce the unsharded batch bit for bit (scenarios are keyed by the global hopper index)."""
    from hopper_mpc_inertial_b200 import sharding
    from hopper_mpc_inertial_b200.batch import BatchMpc
    B, N, n_ticks = 301, 10, 6
    full = scenarios.make_batch(B, N=N, n_ticks=n_ticks, seed=31)

    def run(sc, device):
        dev = f"cuda:{device}"
        bm = BatchMpc(sc["X0"].shape[1], dyn="3f", N=N, device=device)
        bm.set_gains(T(sc["Qdiag"], dev), T(sc["Rdiag"], dev))
        X = T(sc["X0"], dev).clone()
        with torch.cuda.device(device):
            bm.use_current_stream()
            out = bm.rollout(X, T(sc["xref_tab"], dev), T(sc["pf_tab"], dev), T(sc["C_tab"].view(np.int64), dev),
                             T(sc["pf_switch"], dev), 0, n_ticks, True, log=True)
            torch.cuda.synchronize(device)
        return X.cpu().numpy(), out["U_log"].cpu().numpy()

    X_full, U_full = run(full, 0)
    ndev = torch.cuda.device_count()
    parts = []
    for r in range(2):
        lo, hi = sharding.shard_range(B, r, 2)
        sc = scenarios.make_batch(hi - lo, idx0=lo, N=N, n_ticks=n_ticks, seed=31)
        parts.append(run(sc, r if ndev >= 2 else 0))
    assert np.array_equal(np.concatenate([p[0] for p in parts], axis=-1), X_full)
    assert np.array_equal(np.concatenate([p[1] for p in parts], axis=-1), U_full)


def test_contact_gate_matches_oracle_and_both_rollout_flavours_agree():
    """SURVEY 8 row f4 (second half): the contact gate of the applied control.  HMPC_GATE_SCHEDULE is the reference's
    commented-out `f_hist[k, :] = U[0, :] * s` (robotrunner.py:99,111) at 1 kHz; HMPC_GATE_DETECT gates on the leg reach.
    Both against the oracle loop with the same gate; the planned flavour (common-clock masks + tick offsets) is
    bit-identical to the table flavour; the default stays ungated."""
    from hopper_mpc_inertial_b200 import planner
    B, N, n_ticks = 6, 10, 16
    sc = scenarios.make_batch(B, N=N, n_ticks=n_ticks, seed=12)
    tabs = (T(sc["xref_tab"]), T(sc["pf_tab"]), cb64(sc["C_tab"]), T(sc["pf_switch"]))
    gate_bits = (sc["gate_tab"][:n_ticks, :, None].astype(np.int64) >> np.arange(20)) & 1        # (T,B,20)
    assert (gate_bits == 0).any() and (gate_bits == 1).any()

    def run(mode, planned=False, **kw):
        bm = mk(B, "3f", N)
        bm.set_gains(T(sc["Qdiag"]), T(sc["Rdiag"]))
        X = T(sc["X0"]).clone()
        if planned:
            _plan_set(bm, sc)
            bm.set_contact_gate(mode, gate_glob=planner.global_tables(**sc["plan"]["global_args"])["gate_glob"], **kw)
            out = bm.rollout_planned(X, 0, n_ticks, True, log=True)
        else:
            bm.set_contact_gate(mode, gate_tab=T(sc["gate_tab"].view(np.int32)) if mode == "schedule" else None, **kw)
            out = bm.rollout(X, *tabs, 0, n_ticks, True, log=True)
        torch.cuda.synchronize()
        return out["X_log"].cpu().numpy(), out["U_log"].cpu().numpy(), out["status"].cpu().numpy(), bm

    Xoff, Uoff, Soff, _ = run("off")
    Xs, Us, Ss, bm = run("schedule")
    Xp, Up, Sp, _ = run("schedule", planned=True)
    Xd, Ud, Sd, _ = run("detect", leg_max=0.45)
    assert np.array_equal(Xs, Xp) and np.array_equal(Us, Up) and np.array_equal(Ss, Sp)
    assert np.abs(Xs - Xoff).max() > 1e-3 and np.abs(Xd - Xoff).max() > 1e-3          # the gates do change the run
    checked = 0
    for b in range(B):
        p = ho.Params(N=N, Qdiag=sc["Qdiag"][:, b].copy(), Rdiag=sc["Rdiag"][:, b].copy())
        args = (p, sc["X0"][:, b], sc["xref_tab"][:, :, b], sc["pf_tab"][:, :, b], sc["C"][:, b], sc["pf_switch"][:, b], n_ticks)
        for Xg, Ug, Sg, kw in ((Xoff, Uoff, Soff, {}), (Xs, Us, Ss, dict(gate=gate_bits[:, b])), (Xd, Ud, Sd, dict(leg_max=0.45))):
            try:
                Xo, Uo = closed_loop(*args, **kw)
            except QPFailed:                       # a gated hopper may fall: the reference would raise, the device flags it
                assert Sg[b] == _lib.STATUS_INFEASIBLE
                continue
            assert Sg[b] == 0
            assert np.all(np.abs(Ug[:, :, b] - Uo) <= 10 * u_tol(Uo)), (b, kw.keys())
            np.testing.assert_allclose(Xg[:, :, b], Xo, rtol=0, atol=1e-6)
            checked += 1
    assert checked >= 3 * B - 2
    # error behaviour: a scheduled gate needs the masks of the rollout flavour that is used
    with pytest.raises(_lib.HmpcError):
        bm.set_contact_gate("schedule")
    bm.set_contact_gate("schedule", gate_glob=np.ones(4, np.uint32))
    with pytest.raises(_lib.HmpcError):
        bm.rollout(T(sc["X0"]).clone(), *tabs, 0, 2, True)
    with pytest.raises(_lib.HmpcError):
        bm.set_contact_gate("detect", leg_max=0.0)


@pytest.mark.parametrize("dyn", ["3f", "2f"])
def test_warp_admm_closed_loop(dyn):
    """north_star K2 on warm ticks = one warp per hopper (mpc_warp_admm_kernel).  Against the CTA statement of the same
    iteration (hot_path = cta): equal iteration counts, factorisations, status; with polish (OSQP's polish=True) every
    tick lands on the certified oracle optimum, so the closed loop follows the oracle loop."""
    B, N, n_ticks = 8, 10, 12
    sc = scenarios.make_batch(B, N=N, n_ticks=n_ticks, seed=7, dyn=dyn)
    tabs = (T(sc["xref_tab"]), T(sc["pf_tab"]), cb64(sc["C_tab"]), T(sc["pf_switch"]))
    res = {}
    for hp in ("auto", "cta"):
        bm = mk(B, dyn, N, solver="admm", polish=1, hot_path=hp, max_iter=4000)
        bm.set_gains(T(sc["Qdiag"]), T(sc["Rdiag"]))
        X = T(sc["X0"]).clone()
        out = bm.rollout(X, *tabs, 0, n_ticks, True, log=True)
        torch.cuda.synchronize()
        nf, pa, ni = [a.cpu().numpy() for a in bm.solve_stats()]
        res[hp] = (out["X_log"].cpu().numpy(), out["U_log"].cpu().numpy(), out["status"].cpu().numpy(), out["iters"].cpu().numpy(), nf, pa,
                   bm.hot_path_info())
    Xa, Ua, sa, ia, nfa, paa, ha = res["auto"]
    Xc, Uc, sc_, ic, nfc, pac, hc = res["cta"]
    assert ha["warps_per_sm"] >= 6 and hc["warps_per_sm"] == 0
    assert ha["deferred"] <= B                         # warm ticks stayed in the warp kernel
    assert np.all(sa == 0) and np.all(sc_ == 0) and np.all(paa == _lib.PATH_ADMM)
    assert np.array_equal(ia, ic) and np.array_equal(nfa, nfc)
    np.testing.assert_allclose(Ua, Uc, rtol=1e-6, atol=1e-6)
    for b in range(B):
        p = ho.Params(dyn=dyn, N=N, Qdiag=sc["Qdiag"][:, b].copy(), Rdiag=sc["Rdiag"][:, b].copy())
        Xo, Uo = closed_loop(p, sc["X0"][:, b], sc["xref_tab"][:, :, b], sc["pf_tab"][:, :, b], sc["C"][:, b], sc["pf_switch"][:, b], n_ticks)
        assert np.all(np.abs(Ua[:, :, b] - Uo) <= 10 * u_tol(Uo)), np.abs(Ua[:, :, b] - Uo).max()
        np.testing.assert_allclose(Xa[:, :, b], Xo, rtol=0, atol=1e-6)


def test_warp_admm_early_exit_iterate_without_polish():
    """polish = 0: the warp kernel returns OSQP's eps-terminated iterate (status INEXACT) -- equal to the CTA statement
    at the same iteration count."""
    B, N = 16, 10
    sc = scenarios.make_batch(B, N=N, n_ticks=3, seed=5)
    outs = []
    for hp in ("auto", "cta"):
        bm = mk(B, "3f", N, solver="admm", polish=0, hot_path=hp, max_iter=4000)
        bm.set_gains(T(sc["Qdiag"]), T(sc["Rdiag"]))
        X = T(sc["X0"]).clone()
        tabs = (T(sc["xref_tab"]), T(sc["pf_tab"]), cb64(sc["C_tab"]), T(sc["pf_switch"]))
        bm.rollout(X, *tabs, 0, 1, True)
        out = bm.rollout(X, *tabs, 1, 1, False, log=True)           # one warm tick from identical state
        torch.cuda.synchronize()
        outs.append((out["U_log"].cpu().numpy(), out["status"].cpu().numpy(), out["iters"].cpu().numpy(), bm.hot_path_info()["deferred"]))
    (Ua, sa, ia, da), (Uc, sc_, ic, dc) = outs
    assert da == 0
    assert np.all(sa == _lib.STATUS_INEXACT) and np.array_equal(sa, sc_) and np.array_equal(ia, ic)
    np.testing.assert_allclose(Ua, Uc, rtol=1e-7, atol=1e-7)


def test_contact_mask_work_order_does_not_change_results(monkeypatch):
    """The lock-step solve kernel takes the hoppers grouped by contact schedule (hmpc_api.cu: order_* kernels, a
    counting sort on the contact masks every tick).  Scheduling only: with the grouping switched off
    (HMPC_WORK_ORDER=0) the closed loop is bit-identical, respawns and deferrals included."""
    B, N, n_ticks = 3000, 10, 14
    sc = scenarios.make_batch(B, N=N, n_ticks=n_ticks, seed=8, gain_spread=2.0, perturb=1.0)
    tabs = (T(sc["xref_tab"]), T(sc["pf_tab"]), cb64(sc["C_tab"]), T(sc["pf_switch"]))
    res = []
    for on in ("1", "0"):
        monkeypatch.setenv("HMPC_WORK_ORDER", on)
        bm = mk(B, "3f", N, on_infeasible="respawn")
        bm.set_gains(T(sc["Qdiag"]), T(sc["Rdiag"]))
        X = T(sc["X0"]).clone()
        out = bm.rollout(X, *tabs, 0, n_ticks, True, log=True)
        torch.cuda.synchronize()
        nf, pa, ni = [a.cpu().numpy() for a in bm.solve_stats()]
        res.append((X.cpu().numpy(), out["U_log"].cpu().numpy(), out["status"].cpu().numpy(), out["iters"].cpu().numpy(), nf, ni,
                    bm.hot_path_info()["deferred"]))
        bm.close()
    for a, b in zip(res[0][:6], res[1][:6]):
        assert np.array_equal(a, b)
    assert res[0][6] == res[1][6] and res[0][6] > 0
