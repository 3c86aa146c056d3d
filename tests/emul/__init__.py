"""ctypes binding of tests/emul/libhmpc_emul.so: the product's DEVICE source compiled by g++ and run as
one serial thread per hopper (see emul.cpp).  Test infrastructure only."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(os.path.dirname(_HERE))
_SO = os.path.join(_HERE, "libhmpc_emul.so")
_DEPS = [os.path.join(_HERE, "emul.cpp"), os.path.join(_HERE, "fake_cuda", "cuda_runtime.h"),
         os.path.join(_ROOT, "include", "hmpc.h")] + \
        [os.path.join(_ROOT, "hopper_mpc_inertial_b200", "csrc", f) for f in ("hmpc_sim.cuh", "hmpc_qp.cuh", "hmpc_mpc.cuh", "hmpc_warp.cuh", "hmpc_plan.cuh",
                                                                             "hmpc_geometry.cuh")]
_lib = None


def build(force=False):
    if force or not os.path.exists(_SO) or any(os.path.getmtime(d) > os.path.getmtime(_SO) for d in _DEPS):
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-I", os.path.join(_HERE, "fake_cuda"),
                        "-I", os.path.join(_ROOT, "include"), os.path.join(_HERE, "emul.cpp"), "-o", _SO], check=True)
    return _SO


def load():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def default_config(**over):
    """hmpc_config filled with the library defaults WITHOUT loading the CUDA library (values restated from
    hmpc_default_config; tests/test_abi.py checks the two agree)."""
    from hopper_mpc_inertial_b200._lib import HmpcConfig
    cfg = HmpcConfig()
    cfg.abi_version, cfg.device, cfg.batch, cfg.dyn, cfg.N, cfg.mpc_factor = 2, 0, 1, 3, 60, 20
    cfg.precision = cfg.uref_mode = cfg.solver = cfg.mode = 0
    cfg.max_iter, cfg.check_interval, cfg.first_check, cfg.polish = 10000, 25, 25, 1
    cfg.adaptive_rho, cfg.warm_start, cfg.polish_retries, cfg.ipm_max_iter, cfg.on_infeasible = 1, 1, 8, 40, 0
    cfg.sqp_sweeps = 1
    cfg.hot_path = 0
    cfg.mpc_dt, cfg.sim_dt, cfg.m, cfg.g, cfg.mu = 0.02, 1e-3, 7.5, 9.807, 1.0
    J = np.array([[76148072.89e-9, 70089.52e-9, 2067970.36e-9], [70089.52e-9, 45477183.53e-9, -87045.58e-9],
                  [2067970.36e-9, -87045.58e-9, 76287220.47e-9]])
    Ji = np.linalg.inv(J)
    for i in range(9):
        cfg.J[i] = J.reshape(-1)[i]
        cfg.Jinv[i] = Ji.reshape(-1)[i]
    rh = -np.array([0.02663114, 0.04435752, 6.61082088]) / 1000
    tm = [7.78, 7.78, 4.0]
    for i in range(3):
        cfg.rh[i] = rh[i]
        cfg.tau_max[i] = tm[i]
    cfg.fz_max, cfg.z_min, cfg.kf = 206.0, 0.1, 100.0
    cfg.eps_abs = cfg.eps_rel = 1e-5
    cfg.rho0, cfg.sigma, cfg.alpha = 0.1, 1e-6, 1.6
    cfg.kkt_eps = cfg.polish_tol = 1e-9
    cfg.ipm_tol = 1e-6
    for k, v in over.items():
        setattr(cfg, k, v)
    return cfg


class EmulMpc:
    """Host-side state + calls mirroring BatchMpc.solve for the emulated device code (SoA numpy arrays)."""

    def __init__(self, batch, dyn="3f", N=10, **over):
        self.cfg = default_config(batch=int(batch), N=int(N), dyn={"2f": 2, "3f": 3}[dyn], **over)
        self.B, self.N = int(batch), int(N)
        m = 11 * N
        self.Qd = np.tile(np.array([50., 50., 2., 1., 1., 50., 1., 1., 1., 10., 10., 10.])[:, None], (1, batch)).copy()
        self.Rd = np.full((6, batch), 0.001)
        self.Xsol = np.zeros((N + 1, 12, batch))
        self.Usol = np.zeros((N, 6, batch))
        self.code = np.zeros((m, batch), np.int8)
        self.valid = np.zeros(batch, np.int8)
        # warm blocks of the warp kernels (MpcIo::warm), as the library keeps them per handle
        self.warm = np.zeros((batch, load().emul_warm_stride(int(N))))
        self.warm_ok = np.zeros(batch, np.int8)

    def set_gains(self, Qd, Rd):
        self.Qd = np.ascontiguousarray(Qd, float)
        self.Rd = np.ascontiguousarray(Rd, float)

    def solve(self, x_in, x_ref, pf, Cbits, init):
        B, N = self.B, self.N
        x_in = np.ascontiguousarray(x_in, float)
        x_ref = np.ascontiguousarray(x_ref, float)
        pf = np.ascontiguousarray(pf, float)
        Cbits = np.ascontiguousarray(Cbits, np.uint64)
        U = np.zeros((N, 6, B))
        Xs = np.zeros((N + 1, 12, B))
        st = np.zeros(B, np.int32)
        it = np.zeros(B, np.int32)
        nf = np.zeros(B, np.int32)
        pa = np.zeros(B, np.int32)
        load().emul_set_warm.argtypes = [C.c_void_p, C.c_void_p]
        load().emul_set_warm(_p(self.warm), _p(self.warm_ok))
        rc = load().emul_solve(C.byref(self.cfg), _p(self.Qd), _p(self.Rd), _p(x_in), _p(x_ref), _p(pf), _p(Cbits),
                               int(bool(init)), _p(self.Xsol), _p(self.Usol), _p(self.code), _p(self.valid),
                               _p(U), _p(Xs), _p(st), _p(it), _p(nf), _p(pa))
        assert rc == 0
        self.warp_done = load().emul_warp_done()      # hoppers finished by the warp-per-hopper path
        return U, Xs, st, it, nf, pa

    def condense(self, x_in, x_guess, x_ref, pf, Cbits):
        B, N = self.B, self.N
        n, m = 6 * N, 11 * N
        H = np.zeros((n, n, B))
        g = np.zeros((n, B))
        lo = np.zeros((m, B))
        hi = np.zeros((m, B))
        inf = np.zeros(B, np.int32)
        args = [np.ascontiguousarray(a, float) for a in (x_in, x_guess, x_ref, pf)]
        cb = np.ascontiguousarray(Cbits, np.uint64)
        rc = load().emul_condense(C.byref(self.cfg), _p(self.Qd), _p(self.Rd), *[_p(a) for a in args], _p(cb),
                                  _p(H), _p(g), _p(lo), _p(hi), _p(inf))
        assert rc == 0
        return H, g, lo, hi, inf

    def rk4(self, X, U, pf, nsteps, convert=False):
        X = np.ascontiguousarray(X, float).copy()
        x = np.zeros((12, self.B)) if convert else None
        rc = load().emul_rk4(C.byref(self.cfg), _p(X), _p(np.ascontiguousarray(U, float)),
                             _p(np.ascontiguousarray(pf, float)), int(nsteps), _p(x))
        assert rc == 0
        return (X, x) if convert else X


    def sim_tick(self, X, U, pfa, pfb, sw=None, gate_mode=0, bits=None, leg_max=0.0):
        """One MPC tick of the simulator (hmpc_sim.cuh: sim_tick) with the contact gate; returns the new X (13,B)."""
        X = np.ascontiguousarray(X, float).copy()
        sw = None if sw is None else np.ascontiguousarray(sw, np.uint8)
        bits = None if bits is None else np.ascontiguousarray(bits, np.uint32)
        lib = load()
        lib.emul_sim_tick.argtypes = [C.c_void_p] * 6 + [C.c_int, C.c_void_p, C.c_double]
        rc = lib.emul_sim_tick(C.byref(self.cfg), _p(X), _p(np.ascontiguousarray(U, float)), _p(np.ascontiguousarray(pfa, float)),
                               _p(np.ascontiguousarray(pfb, float)), _p(sw), int(gate_mode), _p(bits), float(leg_max))
        assert rc == 0
        return X


GEOMETRY_FIELDS = ("unsupported", "cta", "threads", "grid", "smem", "ws_bytes", "warp", "admm", "wpc", "kcap", "wdoubles",
                   "warp_grid", "warp_per_sm", "regs", "group", "warp_smem")
CTA_BUILDS = ("n10_f64", "n10_f64_admm", "n10_f32", "wide_gmem4", "wide_gmem2")     # enum CtaBuild (hmpc_geometry.cuh)


def launch_geometry(cfg, kcap, sm_count, smem_block, smem_sm, l2, warp_regs, admm_regs):
    """hmpc_create's launch geometry (csrc/hmpc_geometry.cuh) as a dict; cta is the name of the CTA build."""
    lib = load()
    lib.emul_launch_geometry.argtypes = [C.c_void_p, C.c_int, C.c_int] + [C.c_longlong] * 3 + [C.c_void_p] * 3
    wr = np.ascontiguousarray(warp_regs, np.int32)
    ar = np.ascontiguousarray(admm_regs, np.int32)
    out = np.zeros(16, np.int64)
    lib.emul_launch_geometry(C.byref(cfg), int(kcap), int(sm_count), int(smem_block), int(smem_sm), int(l2), _p(wr), _p(ar), _p(out))
    g = dict(zip(GEOMETRY_FIELDS, (int(v) for v in out)))
    g["cta"] = CTA_BUILDS[g["cta"]]
    return g


def kernel_builds():
    """The kernel build lists of csrc/hmpc_geometry.cuh: warp wpc, ADMM warp wpc, CTA build -> threads."""
    n = np.zeros(3, np.int32)
    w, a, t = (np.zeros(16, np.int32) for _ in range(3))
    load().emul_kernel_builds(_p(n), _p(w), _p(a), _p(t))
    return dict(warp=w[:n[0]].tolist(), admm=a[:n[1]].tolist(), cta=dict(zip(CTA_BUILDS, t[:n[2]].tolist())))


def plan_tables(x0, xf, curve, off, gt, N, n_ticks, tick0=0, mpc_factor=20, dt=1e-3):
    """The device planner (csrc/hmpc_plan.cuh) run on the host: same outputs as BatchMpc.plan_tables (numpy)."""
    x0 = np.ascontiguousarray(x0, float); xf = np.ascontiguousarray(xf, float)
    B = x0.shape[1]
    curve = np.ascontiguousarray(curve, np.int32); off = np.ascontiguousarray(off, np.int32)
    sin_tab = np.ascontiguousarray(gt["sin_tab"], float); pf_idx = np.ascontiguousarray(gt["pf_idx"], np.int32)
    cmask = np.ascontiguousarray(gt["cmask"], np.uint64); sw = np.ascontiguousarray(gt["sw_glob"], np.uint8)
    xr = np.zeros((n_ticks + N, 12, B)); pf = np.zeros((n_ticks + N + 1, 3, B))
    Ct = np.zeros((max(n_ticks, 1), B), np.uint64); ps = np.zeros((max(n_ticks, 1), B), np.uint8)
    lib = load()
    lib.emul_plan_tables.argtypes = [C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double,
                                     C.c_double] + [C.c_void_p] * 8 + [C.c_int, C.c_int] + [C.c_void_p] * 4
    rc = lib.emul_plan_tables(B, int(N), int(mpc_factor), float(dt), int(gt["N_run"]), int(gt["n_sim"]), int(gt["max_tick"]),
                              float(gt["t_p"]), float(gt["curve_psi1"]), float(gt["curve_psi2"]), _p(x0), _p(xf), _p(curve), _p(off),
                              _p(sin_tab), _p(pf_idx), _p(cmask), _p(sw), int(tick0), int(n_ticks), _p(xr), _p(pf), _p(Ct), _p(ps))
    assert rc == 0
    return dict(xref_tab=xr, pf_tab=pf, C_tab=Ct, pf_switch=ps)
