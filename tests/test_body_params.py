"""Per-hopper body parameters (include/hmpc.h: hmpc_set_body_params): the MPC model (m, mu, Jinv, rh) and the simulated
plant (m, J, Jinv, rh) per hopper, for domain randomisation and model mismatch.  CPU tests run the device source
through the emulation (tests/emul_body) against the oracle with each hopper's own Params; the -m gpu tests run the
kernels through the C ABI."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from hopper_mpc_inertial_b200 import scenarios
from oracle import hopper_oracle as ho
from oracle.closed_loop import OracleMpc, QPFailed, leg_reaches
from tests.conftest import normalised_oracle_qp, u_tol
from tests.emul import EmulMpc, _p, load as emul_load

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "emul_body", "emul_body.cpp")
_SO = os.path.join(tempfile.gettempdir(), f"hmpc_emul_body_{os.getuid()}.so")     # built here: the tree may be read-only
_lib = None


def _emul():
    global _lib
    if _lib is None:
        emul_load()                 # builds tests/emul (same dependencies)
        deps = [_SRC, os.path.join(_HERE, "emul", "libhmpc_emul.so")]
        if not os.path.exists(_SO) or any(os.path.getmtime(d) > os.path.getmtime(_SO) for d in deps):
            subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-I", os.path.join(_HERE, "emul", "fake_cuda"),
                            "-I", os.path.join(os.path.dirname(_HERE), "include"), _SRC, "-o", _SO], check=True)
        _lib = C.CDLL(_SO)
        _lib.emul_set_body.argtypes = [C.c_void_p, C.c_void_p]
        _lib.emul_body_sim_tick.argtypes = [C.c_void_p] * 6 + [C.c_int, C.c_double]
    return _lib


def model_rows(bm):
    """body_model dict -> [14][B] rows in QpConst::body order (m, mu, rh, Jinv)."""
    B = bm["m"].shape[0]
    return np.ascontiguousarray(np.concatenate([bm["m"][None], bm["mu"][None], bm["rh"], bm["Jinv"].reshape(9, B)]))


def plant_rows(bp):
    """body_plant dict -> [22][B] rows in SimConst::body order (m, rh, J, Jinv)."""
    B = bp["m"].shape[0]
    return np.ascontiguousarray(np.concatenate([bp["m"][None], bp["rh"], bp["J"].reshape(9, B), bp["Jinv"].reshape(9, B)]))


class EmulBodyMpc(EmulMpc):
    """EmulMpc with per-hopper bodies: set_body_params mirrors BatchMpc.set_body_params (numpy, SoA)."""

    def __init__(self, batch, **kw):
        super().__init__(batch, **kw)
        self.model = None
        self.plant = None

    def set_body_params(self, which="both", m=None, J=None, Jinv=None, rh=None, mu=None):
        cfg, B = self.cfg, self.B
        pick = lambda a, s, shape: np.broadcast_to(np.asarray(s, float).reshape(shape + (1,)), shape + (B,)) if a is None else a
        if J is not None and Jinv is None:
            Jinv = np.ascontiguousarray(np.moveaxis(np.linalg.inv(np.moveaxis(J, -1, 0)), 0, -1))
        if which in ("model", "both"):
            self.model = model_rows(dict(m=pick(m, cfg.m, ()), mu=pick(mu, cfg.mu, ()), rh=pick(rh, list(cfg.rh), (3,)),
                                         Jinv=pick(Jinv, list(cfg.Jinv), (3, 3))))
        if which in ("plant", "both"):
            self.plant = plant_rows(dict(m=pick(m, cfg.m, ()), rh=pick(rh, list(cfg.rh), (3,)), J=pick(J, list(cfg.J), (3, 3)),
                                         Jinv=pick(Jinv, list(cfg.Jinv), (3, 3))))

    def _register(self):
        _emul().emul_set_body(_p(self.model), _p(self.plant))

    def solve(self, x_in, x_ref, pf, Cbits, init):
        B, N = self.B, self.N
        args = [np.ascontiguousarray(a, float) for a in (x_in, x_ref, pf)]
        Cbits = np.ascontiguousarray(Cbits, np.uint64)
        U, Xs = np.zeros((N, 6, B)), np.zeros((N + 1, 12, B))
        st, it, nf, pa = (np.zeros(B, np.int32) for _ in range(4))
        emul_load().emul_set_warm(_p(self.warm), _p(self.warm_ok))
        self._register()
        rc = _emul().emul_body_solve(C.byref(self.cfg), _p(self.Qd), _p(self.Rd), *[_p(a) for a in args], _p(Cbits),
                                     int(bool(init)), _p(self.Xsol), _p(self.Usol), _p(self.code), _p(self.valid),
                                     _p(U), _p(Xs), _p(st), _p(it), _p(nf), _p(pa))
        assert rc == 0
        return U, Xs, st, it, nf, pa

    def condense(self, x_in, x_guess, x_ref, pf, Cbits):
        B, N = self.B, self.N
        n, m = 6 * N, 11 * N
        H, g, lo, hi, inf = np.zeros((n, n, B)), np.zeros((n, B)), np.zeros((m, B)), np.zeros((m, B)), np.zeros(B, np.int32)
        args = [np.ascontiguousarray(a, float) for a in (x_in, x_guess, x_ref, pf)]
        self._register()
        rc = _emul().emul_body_condense(C.byref(self.cfg), _p(self.Qd), _p(self.Rd), *[_p(a) for a in args],
                                        _p(np.ascontiguousarray(Cbits, np.uint64)), _p(H), _p(g), _p(lo), _p(hi), _p(inf))
        assert rc == 0
        return H, g, lo, hi, inf

    def sim_tick(self, X, U, pfa, pfb, sw=None, gate_mode=0, leg_max=0.0):
        X = np.ascontiguousarray(X, float).copy()
        sw = None if sw is None else np.ascontiguousarray(sw, np.uint8)
        self._register()
        rc = _emul().emul_body_sim_tick(C.byref(self.cfg), _p(X), _p(np.ascontiguousarray(U, float)),
                                        _p(np.ascontiguousarray(pfa, float)), _p(np.ascontiguousarray(pfb, float)), _p(sw),
                                        int(gate_mode), float(leg_max))
        assert rc == 0
        return X


def params(sc, b, dyn="3f", N=10, which="model"):
    """Oracle Params of hopper b: its gains and its model (or plant) body."""
    p = ho.Params(dyn=dyn, N=N, Qdiag=sc["Qdiag"][:, b].copy(), Rdiag=sc["Rdiag"][:, b].copy())
    if which == "model":
        bm = sc["body_model"]
        p.m, p.mu, p.rh, p.J = float(bm["m"][b]), float(bm["mu"][b]), bm["rh"][:, b].copy(), np.linalg.inv(bm["Jinv"][:, :, b])
    else:
        bp = sc["body_plant"]
        p.m, p.rh, p.J = float(bp["m"][b]), bp["rh"][:, b].copy(), bp["J"][:, :, b].copy()
    return p


def oracle_loop(prm, plant, X0, xref_tab, pf_tab, C, pf_switch, n_ticks, leg_max=None, gate_prm=None):
    """oracle.closed_loop.closed_loop with the MPC on prm and RK4 / the leg reach on plant (model mismatch);
    gate_prm: the leg reach on another body instead (to show which one the device used)."""
    mpc = OracleMpc(prm)
    X = np.array(X0, float)
    N = prm.N
    X_log, U_log = [X.copy()], []
    for t in range(n_ticks):
        U = mpc.mpcontrol(ho.convert(X), xref_tab[t:t + N], pf_tab[t:t + N], C[t], init=(t == 0))
        u0 = U[0].copy()
        for i in range(prm.mpc_factor):
            pf = pf_tab[t] if i < pf_switch[t] else pf_tab[t + 1]
            s = 1.0 if leg_max is None or leg_reaches(X, pf, gate_prm or plant, leg_max) else 0.0
            X = ho.rk4_normalized(X, u0 * s, pf, plant)
        X_log.append(X.copy())
        U_log.append(u0)
    return np.stack(X_log), np.stack(U_log)


# ---- scenarios ----------------------------------------------------------------------------------------------------------
def test_make_batch_body_is_shard_invariant_and_leaves_other_outputs_alone():
    a = scenarios.make_batch(12, seed=5, n_ticks=4, body=True)
    b = scenarios.make_batch(12, seed=5, n_ticks=4)
    c = scenarios.make_batch(5, idx0=7, seed=5, n_ticks=4, body=dict(mass=(6.0, 9.0), mismatch=0.05))
    assert "body_model" not in b and "body_plant" not in b
    for k, v in b.items():
        if isinstance(v, np.ndarray):
            assert np.array_equal(a[k], v), k
    for part in ("body_model", "body_plant"):
        for k, v in a[part].items():
            assert np.array_equal(v[..., 7:], c[part][k]), (part, k)
    m, p = a["body_model"], a["body_plant"]
    assert np.all((m["m"] >= 6) & (m["m"] <= 9)) and np.all((m["mu"] >= 0.7) & (m["mu"] <= 1.0))
    assert np.all(np.abs(p["m"] / m["m"] - 1) <= 0.05) and not np.array_equal(p["m"], m["m"])
    np.testing.assert_allclose(np.einsum("ijb,jkb->ikb", p["J"], p["Jinv"]), np.eye(3)[..., None].repeat(12, 2), atol=1e-12)
    with pytest.raises(ValueError):
        scenarios.make_bodies(3, mass_kg=(1, 2))


# ---- CPU: emulated device source against the oracle ---------------------------------------------------------------------
def test_condensed_qp_follows_each_hoppers_model():
    B, N = 16, 10
    sc = scenarios.make_batch(B, N=N, n_ticks=2, seed=31, body=True)
    em = EmulBodyMpc(B, N=N)
    em.set_gains(sc["Qdiag"], sc["Rdiag"])
    em.set_body_params("model", **sc["body_model"])
    rng = np.random.default_rng(1)
    x_in = np.stack([ho.convert(sc["X0"][:, b]) for b in range(B)], 1)
    x_ref = sc["xref_tab"][:N]
    x_guess = np.concatenate([x_in[None], x_ref], 0) + 0.01 * rng.normal(size=(N + 1, 12, B))
    pf = sc["pf_tab"][:N]
    H, g, lo, hi, inf = em.condense(x_in, x_guess, x_ref, pf, sc["C_tab"][0])
    for b in range(B):
        prm = params(sc, b, N=N)
        Ad, Bd, Gd = ho.gen_dt_dynamics(x_guess[:, :, b], pf[:, :, b], prm)
        qc = ho.build_qp_condensed(x_in[:, b], x_ref[:, :, b], Ad, Bd, Gd, sc["C"][0, b], prm)
        A, l, u = normalised_oracle_qp(qc, prm)
        np.testing.assert_allclose(H[..., b], qc["H"], rtol=0, atol=1e-12 * np.abs(qc["H"]).max())
        np.testing.assert_allclose(g[:, b], qc["g"], rtol=0, atol=1e-12 * np.abs(qc["g"]).max())
        np.testing.assert_allclose(lo[:, b], l, rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(hi[:, b], u, rtol=1e-12, atol=1e-12)
        assert inf[b] == 0


def test_sim_tick_follows_each_hoppers_plant():
    B = 16
    sc = scenarios.make_batch(B, n_ticks=2, seed=32, body=True)
    em = EmulBodyMpc(B)
    em.set_body_params("plant", **{k: sc["body_plant"][k] for k in ("m", "J", "Jinv", "rh")})
    rng = np.random.default_rng(2)
    U = rng.normal(size=(6, B)) * 5
    U[2] += 75
    X1 = em.sim_tick(sc["X0"], U, sc["pf_tab"][0], sc["pf_tab"][1], np.full(B, 20, np.uint8))
    for b in range(B):
        p = params(sc, b, which="plant")
        Xo = sc["X0"][:, b].copy()
        for _ in range(20):
            Xo = ho.rk4_normalized(Xo, U[:, b], sc["pf_tab"][0][:, b], p)
        np.testing.assert_allclose(X1[:, b], Xo, rtol=1e-12, atol=1e-12)


def _emul_loop(em, sc, n_ticks, N=10):
    B = em.B
    X = sc["X0"].copy()
    Xl, Ul, stl = [X.copy()], [], []
    for t in range(n_ticks):
        x_in = np.stack([ho.convert(X[:, b]) for b in range(B)], 1)
        U, Xs, st, it, nf, pa = em.solve(x_in, sc["xref_tab"][t:t + N], sc["pf_tab"][t:t + N], sc["C_tab"][t], t == 0)
        X = em.sim_tick(X, U[0], sc["pf_tab"][t], sc["pf_tab"][t + 1], sc["pf_switch"][t])
        Xl.append(X.copy()); Ul.append(U[0].copy()); stl.append(st)
    return np.stack(Xl), np.stack(Ul), np.stack(stl)


def test_closed_loop_with_mismatch_matches_oracle():
    """MPC on each hopper's model, simulator on its (5 % different) plant: the emulated warp + CTA path against the
    oracle loop with the same two bodies; the mismatch really changes the run."""
    B, N, n_ticks = 6, 10, 20
    sc = scenarios.make_batch(B, N=N, n_ticks=n_ticks, seed=33, body=True)
    em = EmulBodyMpc(B, N=N)
    em.set_gains(sc["Qdiag"], sc["Rdiag"])
    em.set_body_params("model", **sc["body_model"])
    em.set_body_params("plant", **sc["body_plant"])
    Xl, Ul, st = _emul_loop(em, sc, n_ticks, N)
    assert np.all(st == 0)
    for b in range(B):
        Xo, Uo = oracle_loop(params(sc, b, N=N), params(sc, b, N=N, which="plant"), sc["X0"][:, b], sc["xref_tab"][:, :, b],
                             sc["pf_tab"][:, :, b], sc["C"][:, b], sc["pf_switch"][:, b], n_ticks)
        assert np.all(np.abs(Ul[:, :, b] - Uo) <= 10 * u_tol(Uo)), np.abs(Ul[:, :, b] - Uo).max()
        np.testing.assert_allclose(Xl[:, :, b], Xo, rtol=0, atol=2e-9)
    Xm, _, _ = _emul_loop(EmulBodyMpc(B, N=N), sc, 3, N)
    assert np.abs(Xm[-1] - Xl[3]).max() > 1e-4


def test_explicit_uniform_bodies_are_bit_identical_to_no_call():
    B, N, n_ticks = 4, 10, 6
    sc = scenarios.make_batch(B, N=N, n_ticks=n_ticks, seed=34)
    em0 = EmulBodyMpc(B, N=N)
    em0.set_gains(sc["Qdiag"], sc["Rdiag"])
    em1 = EmulBodyMpc(B, N=N)
    em1.set_gains(sc["Qdiag"], sc["Rdiag"])
    cfg = em1.cfg
    em1.set_body_params("both", m=np.full(B, cfg.m), J=np.repeat(np.array(list(cfg.J)).reshape(3, 3, 1), B, 2),
                        Jinv=np.repeat(np.array(list(cfg.Jinv)).reshape(3, 3, 1), B, 2),
                        rh=np.repeat(np.array(list(cfg.rh))[:, None], B, 1), mu=np.full(B, cfg.mu))
    a, b = _emul_loop(em0, sc, n_ticks, N), _emul_loop(em1, sc, n_ticks, N)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


def _friction_binds(U, mu, tol=1e-6):
    """Some stance stage of some tick has |f_x| or |f_y| on its friction cone mu f_z (U (T,6) or (N,6))."""
    f = np.asarray(U).reshape(-1, 6)
    on = f[:, 2] > 1.0
    return bool(np.any(on & (np.maximum(np.abs(f[:, 0]), np.abs(f[:, 1])) >= mu * f[:, 2] - tol)))


def _mu_only_scenario(B, N, n_ticks, seed):
    """Low, different friction per hopper and nothing else: the friction cones bind."""
    sc = scenarios.make_batch(B, N=N, n_ticks=n_ticks, seed=seed, speed_range=(0.8, 1.0), perturb=1.0)
    sc["mu"] = 0.15 + 0.1 * np.arange(B) / B
    return sc


def test_per_hopper_mu_alone_moves_the_optimum_onto_each_friction_cone():
    B, N, n_ticks = 4, 10, 8
    sc = _mu_only_scenario(B, N, n_ticks, 35)
    em = EmulBodyMpc(B, N=N)
    em.set_gains(sc["Qdiag"], sc["Rdiag"])
    em.set_body_params("model", mu=sc["mu"])
    Xl, Ul, st = _emul_loop(em, sc, n_ticks, N)
    assert np.all(st == 0)
    binds = 0
    for b in range(B):
        p = ho.Params(N=N, Qdiag=sc["Qdiag"][:, b].copy(), Rdiag=sc["Rdiag"][:, b].copy(), mu=float(sc["mu"][b]))
        Xo, Uo = oracle_loop(p, ho.Params(N=N), sc["X0"][:, b], sc["xref_tab"][:, :, b], sc["pf_tab"][:, :, b], sc["C"][:, b],
                             sc["pf_switch"][:, b], n_ticks)
        assert np.all(np.abs(Ul[:, :, b] - Uo) <= 10 * u_tol(Uo)), np.abs(Ul[:, :, b] - Uo).max()
        binds += _friction_binds(Uo, sc["mu"][b])
    assert binds >= B - 1
    em1 = EmulBodyMpc(B, N=N)                 # the scalar mu = 1 gives another optimum
    em1.set_gains(sc["Qdiag"], sc["Rdiag"])
    _, U1, _ = _emul_loop(em1, sc, n_ticks, N)
    assert np.abs(U1 - Ul).max() > 1e-2


# ---- GPU ------------------------------------------------------------------------------------------------------------------
def _T(a, dev="cuda:0"):
    import torch
    return torch.as_tensor(np.ascontiguousarray(a), device=dev)


def _mk(B, dyn="3f", N=10, **kw):
    from hopper_mpc_inertial_b200.batch import BatchMpc
    return BatchMpc(B, dyn=dyn, N=N, device=0, **kw)


def _set(bm, sc, which=("model", "plant")):
    if "model" in which:
        bm.set_body_params("model", **{k: _T(v) for k, v in sc["body_model"].items()})
    if "plant" in which:
        bm.set_body_params("plant", **{k: _T(v) for k, v in sc["body_plant"].items()})


def _rollout(bm, sc, n_ticks, planned=False):
    import torch
    X = _T(sc["X0"]).clone()
    if planned:
        from hopper_mpc_inertial_b200 import planner
        p = sc["plan"]
        bm.plan_set(_T(p["x0"]), _T(p["xf"]), _T(p["curve"]), _T(p["tick_offset"]), planner.global_tables(**p["global_args"]))
        out = bm.rollout_planned(X, 0, n_ticks, True, log=True)
    else:
        out = bm.rollout(X, _T(sc["xref_tab"]), _T(sc["pf_tab"]), _T(sc["C_tab"].view(np.int64)), _T(sc["pf_switch"]), 0,
                         n_ticks, True, log=True)
    torch.cuda.synchronize()
    return out["X_log"].cpu().numpy(), out["U_log"].cpu().numpy(), out["status"].cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("N,kw", [(10, {}), (10, dict(hot_path="cta")), (20, {}), (10, dict(solver="admm", polish=1, max_iter=4000)),
                                  (10, dict(precision="fp32"))])
def test_gpu_per_hopper_model_reaches_each_oracle_optimum(N, kw):
    B, n_ticks = 16, 8
    sc = scenarios.make_batch(B, N=N, n_ticks=n_ticks, seed=41, body=True)
    bm = _mk(B, "3f", N, **kw)
    bm.set_gains(_T(sc["Qdiag"]), _T(sc["Rdiag"]))
    _set(bm, sc, ("model",))
    Xg, Ug, st = _rollout(bm, sc, n_ticks)
    assert np.sum(st == 0) >= B - (1 if kw.get("precision") == "fp32" else 0), st
    for b in np.where(st == 0)[0]:
        p = params(sc, b, N=N)
        Xo, Uo = oracle_loop(p, ho.Params(N=N), sc["X0"][:, b], sc["xref_tab"][:, :, b], sc["pf_tab"][:, :, b], sc["C"][:, b],
                             sc["pf_switch"][:, b], n_ticks)
        assert np.all(np.abs(Ug[:, :, b] - Uo) <= 10 * u_tol(Uo)), (b, np.abs(Ug[:, :, b] - Uo).max())


@pytest.mark.gpu
def test_gpu_warp_and_cta_kernels_agree_and_mismatch_loop_matches_oracle():
    B, N, n_ticks = 64, 10, 30
    sc = scenarios.make_batch(B, N=N, n_ticks=n_ticks, seed=42, body=True)
    logs = {}
    for mode in ("auto", "cta"):
        bm = _mk(B, "3f", N, hot_path=mode)
        bm.set_gains(_T(sc["Qdiag"]), _T(sc["Rdiag"]))
        _set(bm, sc)
        logs[mode] = _rollout(bm, sc, n_ticks)
        if mode == "auto":
            assert bm.hot_path_info()["deferred"] < 0.2 * B * (n_ticks - 1)
    (Xa, Ua, sa), (Xc, Uc, sc_) = logs["auto"], logs["cta"]
    # a heavy hopper may meet a height row no input can satisfy: the device flags it infeasible exactly where the
    # oracle loop (the reference) raises QPFailed, and matches the oracle everywhere else
    assert np.array_equal(sa, sc_) and set(np.unique(sa)) <= {0, 2}, (sa, sc_)
    ok = sa == 0
    assert ok.sum() >= B - 8
    assert np.abs(Ua[:, :, ok] - Uc[:, :, ok]).max() < 1e-5
    for b in range(B):
        try:
            Xo, Uo = oracle_loop(params(sc, b, N=N), params(sc, b, N=N, which="plant"), sc["X0"][:, b], sc["xref_tab"][:, :, b],
                                 sc["pf_tab"][:, :, b], sc["C"][:, b], sc["pf_switch"][:, b], n_ticks)
        except QPFailed:
            assert not ok[b], b
            continue
        assert ok[b], b
        np.testing.assert_allclose(Xa[:, :, b], Xo, rtol=0, atol=1e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("planned", [False, True])
def test_gpu_explicit_uniform_bodies_equal_no_call(planned):
    import torch
    B, N, n_ticks = 256, 10, 10
    sc = scenarios.make_batch(B, N=N, n_ticks=n_ticks, seed=43)
    runs = []
    for explicit in (False, True):
        bm = _mk(B, "3f", N)
        bm.set_gains(_T(sc["Qdiag"]), _T(sc["Rdiag"]))
        if explicit:
            c = bm.cfg
            f = lambda v, shape: _T(np.repeat(np.array(list(v) if hasattr(v, "__len__") else [v]).reshape(shape + (1,)), B, -1)
                                   .reshape(shape + (B,)))
            bm.set_body_params("both", m=f(c.m, ()), J=f(c.J, (3, 3)), Jinv=f(c.Jinv, (3, 3)), rh=f(c.rh, (3,)))
            bm.set_body_params("model", m=f(c.m, ()), Jinv=f(c.Jinv, (3, 3)), rh=f(c.rh, (3,)), mu=f(c.mu, ()))
        runs.append(_rollout(bm, sc, n_ticks, planned) + (bm.solve_stats()[0].cpu().numpy(),))
        torch.cuda.synchronize()
    for a, b in zip(*runs):
        assert np.array_equal(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("order", ["1", "0"])
def test_gpu_permuting_hoppers_permutes_outputs(monkeypatch, order):
    monkeypatch.setenv("HMPC_WORK_ORDER", order)
    B, N, n_ticks = 509, 10, 6
    sc = scenarios.make_batch(B, N=N, n_ticks=n_ticks, seed=44, body=True)
    perm = np.random.default_rng(3).permutation(B)
    ps = {}
    for k, v in sc.items():
        if k in ("body_model", "body_plant"):
            ps[k] = {q: np.ascontiguousarray(a[..., perm]) for q, a in v.items()}
        elif isinstance(v, np.ndarray) and v.shape and v.shape[-1] == B and k not in ("curve", "tick_offset"):
            ps[k] = np.ascontiguousarray(v[..., perm])
        else:
            ps[k] = v
    outs = []
    for s in (sc, ps):
        bm = _mk(B, "3f", N)
        bm.set_gains(_T(s["Qdiag"]), _T(s["Rdiag"]))
        _set(bm, s)
        outs.append(_rollout(bm, s, n_ticks))
    for a, b in zip(*outs):
        assert np.array_equal(a[..., perm], b)


@pytest.mark.gpu
def test_gpu_gate_detect_follows_the_plant_hip_offset():
    B, N, n_ticks, leg = 6, 10, 12, 0.45
    sc = scenarios.make_batch(B, N=N, n_ticks=n_ticks, seed=45, body=dict(rh=0.02))
    bm = _mk(B, "3f", N)
    bm.set_gains(_T(sc["Qdiag"]), _T(sc["Rdiag"]))
    model = {k: v for k, v in sc["body_model"].items() if k != "rh"}          # the model keeps the config's rh
    bm.set_body_params("model", **{k: _T(v) for k, v in model.items()})
    bm.set_body_params("plant", **{k: _T(v) for k, v in sc["body_plant"].items()})
    bm.set_contact_gate("detect", leg_max=leg)
    Xg, Ug, st = _rollout(bm, sc, n_ticks)
    checked = differs = 0
    for b in range(B):
        if st[b] != 0:
            continue
        pm, pp = params(sc, b, N=N), params(sc, b, N=N, which="plant")
        pm.rh = scenarios.RH_REF.copy()
        args = (sc["X0"][:, b], sc["xref_tab"][:, :, b], sc["pf_tab"][:, :, b], sc["C"][:, b], sc["pf_switch"][:, b], n_ticks)
        Xo, Uo = oracle_loop(pm, pp, *args, leg_max=leg)
        np.testing.assert_allclose(Xg[:, :, b], Xo, rtol=0, atol=1e-6)
        try:                                   # the gate on the model's rh instead gives another run
            Xw, _ = oracle_loop(pm, pp, *args, leg_max=leg, gate_prm=pm)
            differs += np.abs(Xw - Xo).max() > 1e-4
        except QPFailed:
            differs += 1
        checked += 1
    assert checked >= B - 1 and differs >= 1


@pytest.mark.gpu
def test_gpu_linearize_and_condense_follow_the_model():
    import torch
    B, N = 8, 10
    sc = scenarios.make_batch(B, N=N, n_ticks=2, seed=46, body=True)
    bm = _mk(B, "3f", N)
    bm.set_gains(_T(sc["Qdiag"]), _T(sc["Rdiag"]))
    _set(bm, sc, ("model",))
    x_in = np.stack([ho.convert(sc["X0"][:, b]) for b in range(B)], 1)
    x_guess = np.concatenate([x_in[None], sc["xref_tab"][:N]], 0)
    pf = sc["pf_tab"][:N]
    Ad, Bd = (a.cpu().numpy() for a in bm.linearize(_T(x_guess), _T(pf)))
    H, g, lo, hi, inf = (a.cpu().numpy() for a in bm.condense(_T(x_in), _T(x_guess), _T(sc["xref_tab"][:N]), _T(pf),
                                                               _T(sc["C_tab"][0].view(np.int64))))
    torch.cuda.synchronize()
    for b in range(B):
        prm = params(sc, b, N=N)
        Ao, Bo, Go = ho.gen_dt_dynamics(x_guess[:, :, b], pf[:, :, b], prm)
        np.testing.assert_allclose(Ad[..., b], Ao, rtol=0, atol=1e-12)
        np.testing.assert_allclose(Bd[..., b], Bo, rtol=0, atol=1e-12 * np.abs(Bo).max())
        qc = ho.build_qp_condensed(x_in[:, b], sc["xref_tab"][:N, :, b], Ao, Bo, Go, sc["C"][0, b], prm)
        A, l, u = normalised_oracle_qp(qc, prm)
        np.testing.assert_allclose(H[..., b], qc["H"], rtol=0, atol=1e-12 * np.abs(qc["H"]).max())
        np.testing.assert_allclose(lo[:, b], l, rtol=1e-12, atol=1e-12)


@pytest.mark.gpu
def test_gpu_invalid_values_are_rejected_and_leave_the_handle_alone():
    import torch
    from hopper_mpc_inertial_b200._lib import HmpcError
    B = 8
    bm = _mk(B, "3f", 10)
    m = torch.full((B,), 7.0, dtype=torch.float64, device="cuda:0")
    J = _T(np.repeat(scenarios.J_REF[..., None], B, 2))
    bad = m.clone(); bad[5] = -1.0
    with pytest.raises(HmpcError, match="hopper 5"):
        bm.set_body_params("both", m=bad)
    nan = m.clone(); nan[3] = float("nan")
    with pytest.raises(HmpcError, match="hopper 3"):
        bm.set_body_params("plant", m=nan)
    with pytest.raises(HmpcError, match="hopper 2"):
        mu = torch.ones(B, dtype=torch.float64, device="cuda:0"); mu[2] = -0.1
        bm.set_body_params("model", mu=mu)
    # J with which = MODEL, mu with which = PLANT, unknown which: no effect, rejected
    assert bm.lib.hmpc_set_body_params(bm._h, 1, None, C.c_void_p(J.data_ptr()), None, None, None) == -1
    assert bm.lib.hmpc_set_body_params(bm._h, 2, None, None, None, None, C.c_void_p(m.data_ptr())) == -1
    assert bm.lib.hmpc_set_body_params(bm._h, 4, C.c_void_p(m.data_ptr()), None, None, None, None) == -1
    bm.set_body_params("both", m=m)
    bm.set_body_params("both")            # all None: back to the scalars


@pytest.mark.gpu
def test_gpu_rejected_call_leaves_the_bodies_in_place():
    B, N, n_ticks = 32, 10, 5
    sc = scenarios.make_batch(B, N=N, n_ticks=n_ticks, seed=47, body=True)
    runs = []
    for reject in (False, True):
        bm = _mk(B, "3f", N)
        bm.set_gains(_T(sc["Qdiag"]), _T(sc["Rdiag"]))
        _set(bm, sc)
        if reject:
            bad = _T(sc["body_plant"]["m"]).clone(); bad[9] = 0.0
            with pytest.raises(Exception, match="hopper 9"):
                bm.set_body_params("both", m=bad, rh=_T(np.zeros((3, B))))
        runs.append(_rollout(bm, sc, n_ticks))
    for a, b in zip(*runs):
        assert np.array_equal(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("hot_path", ["auto", "cta"])
def test_gpu_per_hopper_mu_alone_matches_oracle_on_the_friction_cone(hot_path):
    B, N, n_ticks = 8, 10, 8
    sc = _mu_only_scenario(B, N, n_ticks, 35)
    outs = []
    for mu in (sc["mu"], None):
        bm = _mk(B, "3f", N, hot_path=hot_path)
        bm.set_gains(_T(sc["Qdiag"]), _T(sc["Rdiag"]))
        if mu is not None:
            bm.set_body_params("model", mu=_T(mu))
        outs.append(_rollout(bm, sc, n_ticks))
    (Xg, Ug, st), (_, U1, _) = outs
    assert np.all(st == 0) and np.abs(Ug - U1).max() > 1e-2
    binds = 0
    for b in range(B):
        p = ho.Params(N=N, Qdiag=sc["Qdiag"][:, b].copy(), Rdiag=sc["Rdiag"][:, b].copy(), mu=float(sc["mu"][b]))
        Xo, Uo = oracle_loop(p, ho.Params(N=N), sc["X0"][:, b], sc["xref_tab"][:, :, b], sc["pf_tab"][:, :, b], sc["C"][:, b],
                             sc["pf_switch"][:, b], n_ticks)
        assert np.all(np.abs(Ug[:, :, b] - Uo) <= 10 * u_tol(Uo)), np.abs(Ug[:, :, b] - Uo).max()
        binds += _friction_binds(Uo, sc["mu"][b])
    assert binds >= B - 2
