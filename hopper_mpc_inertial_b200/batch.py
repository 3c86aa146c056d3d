"""Batched hopper MPC on one B200: torch CUDA tensors as the batch container over the C ABI.

All tensors are float64, structure-of-arrays with the hopper index LAST (contiguous), exactly the
layout include/hmpc.h documents: x_in (12, B), x_ref (N, 12, B), pf (N, 3, B), U (N, 6, B) ...
``soa()`` / ``aos()`` convert from / to the batch-first layout.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib


def soa(t: torch.Tensor) -> torch.Tensor:
    """(B, ...) -> (..., B) contiguous."""
    return t.movedim(0, -1).contiguous()


def aos(t: torch.Tensor) -> torch.Tensor:
    """(..., B) -> (B, ...) contiguous."""
    return t.movedim(-1, 0).contiguous()


def cbits_from_C(Cmat) -> np.ndarray:
    """Contact schedule matrix (B, N) of 0/1 floats (gait_map, robotrunner.py:172-180) -> uint64 masks."""
    Cm = np.asarray(Cmat) != 0
    N = Cm.shape[-1]
    w = (np.uint64(1) << np.arange(N, dtype=np.uint64))
    return (Cm.astype(np.uint64) * w).sum(axis=-1).astype(np.uint64)


def _ptr(t):
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


class BatchMpc:
    """B independent hoppers' MPC state + solver workspace on one GPU (one hmpc handle)."""

    def __init__(self, batch, dyn="3f", N=10, device=0, **overrides):
        if not torch.cuda.is_available():
            raise RuntimeError("hopper_mpc_inertial_b200 needs a CUDA device (no CPU fallback)")
        self.lib = _lib.load()
        cfg = _lib.default_config()
        cfg.batch, cfg.N, cfg.dyn, cfg.device = int(batch), int(N), _lib.DYN[dyn], int(device)
        for k, v in overrides.items():
            if k == "solver" and isinstance(v, str):
                v = _lib.SOLVER[v]
            if k == "mode" and isinstance(v, str):
                v = _lib.MODE[v]
            if k == "on_infeasible" and isinstance(v, str):
                v = _lib.ON_INFEASIBLE[v]
            if k == "precision" and isinstance(v, str):
                v = _lib.PRECISION[v]
            if k == "hot_path" and isinstance(v, str):
                v = _lib.HOT_PATH[v]
            cur = getattr(cfg, k)
            if hasattr(cur, "__len__"):
                arr = np.asarray(v, dtype=float).reshape(-1)
                for i in range(len(cur)):
                    cur[i] = float(arr[i])
            else:
                setattr(cfg, k, v)
        if "J" in overrides and "Jinv" not in overrides:
            Ji = np.linalg.inv(np.asarray(overrides["J"], float).reshape(3, 3)).reshape(-1)
            for i in range(9):
                cfg.Jinv[i] = float(Ji[i])
        self.cfg = cfg
        self.B, self.N, self.dyn = int(batch), int(N), dyn
        self.device = torch.device("cuda", int(device))
        h = C.c_void_p()
        _lib.check(self.lib.hmpc_create(C.byref(cfg), C.byref(h)))
        self._h = h
        with torch.cuda.device(self.device):
            _lib.check(self.lib.hmpc_set_stream(self._h, C.c_void_p(torch.cuda.current_stream().cuda_stream)))

    def close(self):
        if getattr(self, "_h", None):
            self.lib.hmpc_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- helpers -------------------------------------------------------------------------------
    def _chk(self, t, shape, dtype=torch.float64):
        if t.device != self.device or t.dtype != dtype or not t.is_contiguous() or tuple(t.shape) != tuple(shape):
            raise ValueError(f"expected contiguous {dtype} tensor of shape {tuple(shape)} on {self.device}, "
                             f"got {t.dtype} {tuple(t.shape)} on {t.device}")
        return t

    def empty(self, *shape, dtype=torch.float64):
        return torch.empty(*shape, dtype=dtype, device=self.device)

    def use_current_stream(self):
        _lib.check(self.lib.hmpc_set_stream(self._h, C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)))

    # -- ABI calls -----------------------------------------------------------------------------
    def set_gains(self, Qdiag=None, Rdiag=None):
        if Qdiag is not None:
            self._chk(Qdiag, (12, self.B))
        if Rdiag is not None:
            self._chk(Rdiag, (6, self.B))
        _lib.check(self.lib.hmpc_set_gains(self._h, _ptr(Qdiag), _ptr(Rdiag)))

    def set_body_params(self, which="both", m=None, J=None, Jinv=None, rh=None, mu=None):
        """Per-hopper body (include/hmpc.h: hmpc_set_body_params).  which: "model" (what the MPC plans with: m, Jinv,
        rh, mu), "plant" (what rk4 / the rollouts integrate: m, J, Jinv, rh) or "both".  Tensors: m (B,), J and Jinv
        (3, 3, B), rh (3, B), mu (B,); None keeps the config's scalar for every hopper, all None resets the target.
        Jinv is computed from J when only J is given."""
        B = self.B
        if which not in _lib.BODY:
            raise ValueError(f"which must be one of {sorted(_lib.BODY)}, got {which!r}")
        for t, shape in ((m, (B,)), (J, (3, 3, B)), (Jinv, (3, 3, B)), (rh, (3, B)), (mu, (B,))):
            if t is not None:
                self._chk(t, shape)
        if J is not None and Jinv is None and which != "model":
            Jinv = soa(torch.linalg.inv(aos(J)))
        _lib.check(self.lib.hmpc_set_body_params(self._h, _lib.BODY[which], _ptr(m), _ptr(J), _ptr(Jinv), _ptr(rh),
                                                 _ptr(mu)))

    def convert(self, X):
        self._chk(X, (13, self.B))
        x = self.empty(12, self.B)
        _lib.check(self.lib.hmpc_convert(self._h, _ptr(X), _ptr(x)))
        return x

    def rk4(self, X, U, pf, nsteps=1, log_steps=False):
        """In-place on X.  Returns the per-step states (nsteps, 13, B) when log_steps."""
        self._chk(X, (13, self.B)); self._chk(U, (6, self.B)); self._chk(pf, (3, self.B))
        Xs = self.empty(nsteps, 13, self.B) if log_steps else None
        _lib.check(self.lib.hmpc_rk4(self._h, _ptr(X), _ptr(U), _ptr(pf), int(nsteps), _ptr(Xs)))
        return Xs

    def linearize(self, x_guess, pf):
        N, B = self.N, self.B
        self._chk(x_guess, (N + 1, 12, B)); self._chk(pf, (N, 3, B))
        Ad, Bd = self.empty(N, 12, 12, B), self.empty(N, 12, 6, B)
        _lib.check(self.lib.hmpc_linearize(self._h, _ptr(x_guess), _ptr(pf), _ptr(Ad), _ptr(Bd)))
        return Ad, Bd

    def condense(self, x_in, x_guess, x_ref, pf, Cbits):
        N, B = self.N, self.B
        n, m = 6 * N, 11 * N
        self._chk(x_in, (12, B)); self._chk(x_guess, (N + 1, 12, B)); self._chk(x_ref, (N, 12, B))
        self._chk(pf, (N, 3, B)); self._chk(Cbits, (B,), torch.int64)
        H, g = self.empty(n, n, B), self.empty(n, B)
        lo, hi = self.empty(m, B), self.empty(m, B)
        inf = self.empty(B, dtype=torch.int32)
        _lib.check(self.lib.hmpc_condense(self._h, _ptr(x_in), _ptr(x_guess), _ptr(x_ref), _ptr(pf),
                                          _ptr(Cbits), _ptr(H), _ptr(g), _ptr(lo), _ptr(hi), _ptr(inf)))
        return H, g, lo, hi, inf

    def solve(self, x_in, x_ref, pf, Cbits, init, out=None):
        """mpcontrol for the batch.  Returns (U (N,6,B), Xsol (N+1,12,B), status (B,), iters (B,))."""
        N, B = self.N, self.B
        self._chk(x_in, (12, B)); self._chk(x_ref, (N, 12, B)); self._chk(pf, (N, 3, B))
        self._chk(Cbits, (B,), torch.int64)
        if out is None:
            out = (self.empty(N, 6, B), self.empty(N + 1, 12, B),
                   self.empty(B, dtype=torch.int32), self.empty(B, dtype=torch.int32))
        U, Xs, st, it = out
        _lib.check(self.lib.hmpc_solve(self._h, _ptr(x_in), _ptr(x_ref), _ptr(pf), _ptr(Cbits),
                                       1 if init else 0, _ptr(U), _ptr(Xs), _ptr(st), _ptr(it)))
        return U, Xs, st, it

    def rollout(self, X, xref_tab, pf_tab, C_tab, pf_switch=None, tick0=0, n_ticks=1, init=True,
                log=False, out=None):
        """Closed loop for n_ticks ticks, in place on X.  Returns dict(status, iters[, X_log, U_log])."""
        B, N = self.B, self.N
        self._chk(X, (13, B))
        T = C_tab.shape[0]
        self._chk(C_tab, (T, B), torch.int64)
        if xref_tab.shape[0] < tick0 + n_ticks - 1 + N or pf_tab.shape[0] < tick0 + n_ticks + max(N - 1, 1):
            raise ValueError("reference tables too short for the requested ticks")
        self._chk(xref_tab, (xref_tab.shape[0], 12, B)); self._chk(pf_tab, (pf_tab.shape[0], 3, B))
        if tick0 + n_ticks > T:
            raise ValueError("contact table too short")
        if pf_switch is not None:
            self._chk(pf_switch, (T, B), torch.uint8)
        if out is None:
            out = dict(status=self.empty(B, dtype=torch.int32), iters=self.empty(B, dtype=torch.int32))
            if log:
                out["X_log"] = self.empty(n_ticks + 1, 13, B)
                out["U_log"] = self.empty(n_ticks, 6, B)
        _lib.check(self.lib.hmpc_rollout(self._h, _ptr(X), _ptr(xref_tab), _ptr(pf_tab), _ptr(C_tab),
                                         _ptr(pf_switch), int(tick0), int(n_ticks), 1 if init else 0,
                                         _ptr(out.get("X_log")), _ptr(out.get("U_log")),
                                         _ptr(out["status"]), _ptr(out["iters"])))
        return out

    # -- device-side planner (robotrunner.py:166-230 for a batch; include/hmpc.h: hmpc_plan_*) -----------------
    def plan_set(self, x0, xf, curve, tick_offset, gt):
        """x0, xf (12,B) float64, curve, tick_offset (B,) int32 device tensors (kept referenced by the handle);
        ``gt`` = planner.global_tables(...) (host numpy: what depends on the common clock only)."""
        B = self.B
        self._chk(x0, (12, B)); self._chk(xf, (12, B))
        self._chk(curve, (B,), torch.int32); self._chk(tick_offset, (B,), torch.int32)
        pc = _lib.HmpcPlanConfig()
        pc.N_run, pc.n_sim, pc.max_tick = int(gt["N_run"]), int(gt["n_sim"]), int(gt["max_tick"])
        pc.t_p, pc.curve_psi1, pc.curve_psi2 = float(gt["t_p"]), float(gt["curve_psi1"]), float(gt["curve_psi2"])
        tabs = [np.ascontiguousarray(gt["sin_tab"], dtype=np.float64), np.ascontiguousarray(gt["pf_idx"], dtype=np.int32),
                np.ascontiguousarray(gt["cmask"], dtype=np.uint64), np.ascontiguousarray(gt["sw_glob"], dtype=np.uint8)]
        if tabs[0].shape[0] < pc.n_sim or tabs[1].shape[0] < pc.n_sim or tabs[2].shape[0] < pc.max_tick or tabs[3].shape[0] < pc.max_tick:
            raise ValueError("global tables shorter than n_sim / max_tick")
        _lib.check(self.lib.hmpc_plan_set(self._h, C.byref(pc), _ptr(x0), _ptr(xf), _ptr(curve), _ptr(tick_offset),
                                          *[t.ctypes.data_as(C.c_void_p) for t in tabs]))
        self._plan_keep = (x0, xf, curve, tick_offset)
        self._plan_max_tick = pc.max_tick

    def plan_tables(self, tick0, n_ticks):
        """The tables ``rollout`` takes, generated on the device: dict(xref_tab, pf_tab, C_tab, pf_switch)."""
        N, B = self.N, self.B
        out = dict(xref_tab=self.empty(n_ticks + N, 12, B), pf_tab=self.empty(n_ticks + N + 1, 3, B),
                   C_tab=self.empty(max(n_ticks, 1), B, dtype=torch.int64), pf_switch=self.empty(max(n_ticks, 1), B, dtype=torch.uint8))
        _lib.check(self.lib.hmpc_plan_tables(self._h, int(tick0), int(n_ticks), _ptr(out["xref_tab"]), _ptr(out["pf_tab"]),
                                             _ptr(out["C_tab"]), _ptr(out["pf_switch"])))
        return out

    def rollout_planned(self, X, tick0=0, n_ticks=1, init=True, log=False, out=None):
        """``rollout`` with every tick's reference window generated on the device (no tables)."""
        B = self.B
        self._chk(X, (13, B))
        if out is None:
            out = dict(status=self.empty(B, dtype=torch.int32), iters=self.empty(B, dtype=torch.int32))
            if log:
                out["X_log"] = self.empty(n_ticks + 1, 13, B)
                out["U_log"] = self.empty(n_ticks, 6, B)
        _lib.check(self.lib.hmpc_rollout_planned(self._h, _ptr(X), int(tick0), int(n_ticks), 1 if init else 0,
                                                 _ptr(out.get("X_log")), _ptr(out.get("U_log")),
                                                 _ptr(out["status"]), _ptr(out["iters"])))
        return out

    def set_contact_gate(self, mode="off", gate_tab=None, gate_glob=None, leg_max=0.0):
        """Contact gate of the applied control (include/hmpc.h: hmpc_set_contact_gate; robotrunner.py:99,111).
        ``mode``: "off" (the reference as shipped), "schedule" (U[0] * s at every simulator step; ``gate_tab`` (T,B)
        int32 device tensor of per-tick step masks for ``rollout`` and / or ``gate_glob`` (max_tick,) host uint32 array
        for ``rollout_planned``, see planner.gate_masks / global_tables), "detect" (leg reach <= ``leg_max``)."""
        m = _lib.GATE[mode]
        if gate_tab is not None:
            self._chk(gate_tab, (gate_tab.shape[0], self.B), torch.int32)
        gg = None if gate_glob is None else np.ascontiguousarray(gate_glob, dtype=np.uint32)
        _lib.check(self.lib.hmpc_set_contact_gate(self._h, m, _ptr(gate_tab), None if gg is None else gg.ctypes.data_as(C.c_void_p),
                                                  0 if gg is None else int(gg.shape[0]), float(leg_max)))
        self._gate_keep = gate_tab

    def solve_stats(self):
        """Per-hopper (nfac, path, n_infeasible) of the last solve / accumulated over the last rollout."""
        nf = self.empty(self.B, dtype=torch.int32)
        pa = self.empty(self.B, dtype=torch.int32)
        ni = self.empty(self.B, dtype=torch.int32)
        _lib.check(self.lib.hmpc_solve_stats(self._h, _ptr(nf), _ptr(pa), _ptr(ni), None))
        return nf, pa, ni

    def solve_flops(self):
        """Per-hopper algorithmic FLOPs of the solver kernel (last solve / accumulated over the last rollout)."""
        fl = self.empty(self.B)
        _lib.check(self.lib.hmpc_solve_stats(self._h, None, None, None, _ptr(fl)))
        return fl

    def set_timing(self, enable=True):
        _lib.check(self.lib.hmpc_set_timing(self._h, 1 if enable else 0))

    def kernel_times(self):
        """(mpc_ms, sim_ms, n_ticks) summed over the most recent rollout (needs set_timing(True))."""
        a, b, n = C.c_double(), C.c_double(), C.c_int()
        _lib.check(self.lib.hmpc_kernel_times(self._h, C.byref(a), C.byref(b), C.byref(n)))
        return a.value, b.value, n.value

    def tick_times(self, cap=4096):
        """Per-tick (mpc_ms, sim_ms) numpy arrays of the most recent timed rollout (needs set_timing(True))."""
        a, b, n = np.zeros(cap), np.zeros(cap), C.c_int()
        _lib.check(self.lib.hmpc_tick_times(self._h, a.ctypes.data_as(C.c_void_p), b.ctypes.data_as(C.c_void_p), int(cap), C.byref(n)))
        k = min(n.value, cap)
        return a[:k], b[:k]

    def launch_count(self):
        n = C.c_int64()
        _lib.check(self.lib.hmpc_launch_count(self._h, C.byref(n)))
        return n.value

    def hot_path_info(self):
        """dict(warps_per_sm, kcap, regs, deferred): the warp-per-hopper kernel's geometry and how many hopper-ticks
        of the last solve / rollout it handed to the CTA kernel (warps_per_sm = 0: warp kernel not in use)."""
        a, b, r, d = C.c_int(), C.c_int(), C.c_int(), C.c_int64()
        _lib.check(self.lib.hmpc_hot_path_info(self._h, C.byref(a), C.byref(b), C.byref(r), C.byref(d)))
        return dict(warps_per_sm=a.value, kcap=b.value, regs=r.value, deferred=d.value)

    def measure_fp64_peak(self):
        v = C.c_double()
        _lib.check(self.lib.hmpc_measure_fp64_peak(self._h, C.byref(v)))
        return v.value

    def synchronize(self):
        _lib.check(self.lib.hmpc_synchronize(self._h))
