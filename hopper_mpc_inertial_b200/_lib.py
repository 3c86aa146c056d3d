"""ctypes binding of libhmpc_b200.so (C ABI declared in include/hmpc.h).

The shared library is built in-tree by ``hopper_mpc_inertial_b200.build.build_lib()`` (nvcc, sm_100a).
There is no CPU fallback: a missing library or a missing CUDA device raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("HMPC_LIB_PATH") or os.path.join(_HERE, "libhmpc_b200.so")   # override: experiment builds (tools/)

HMPC_ABI_VERSION = 2
HMPC_INF = 1e30
DYN = {"2f": 2, "3f": 3}
STATUS_SOLVED, STATUS_MAX_ITER, STATUS_INFEASIBLE, STATUS_NON_FINITE, STATUS_INEXACT = 0, 1, 2, 3, 4
PATH_NONE, PATH_WARM, PATH_IPM_POLISH, PATH_IPM, PATH_ADMM = 0, 1, 2, 3, 4
SOLVER = {"exact": 0, "admm": 1}
MODE = {"early_exit": 0, "fixed_iter": 1}
ON_INFEASIBLE = {"hold": 0, "respawn": 1}
PRECISION = {"fp64": 0, "fp32": 1}
HOT_PATH = {"auto": 0, "cta": 1}
GATE = {"off": 0, "schedule": 1, "detect": 2}
BODY = {"model": 1, "plant": 2, "both": 3}

# every symbol include/hmpc.h declares (tests/test_abi.py checks the .so exports all of them)
SYMBOLS = [
    "hmpc_default_config", "hmpc_create", "hmpc_destroy", "hmpc_set_stream", "hmpc_synchronize",
    "hmpc_set_gains", "hmpc_set_body_params", "hmpc_convert", "hmpc_rk4", "hmpc_linearize", "hmpc_condense", "hmpc_solve",
    "hmpc_rollout", "hmpc_plan_set", "hmpc_plan_tables", "hmpc_rollout_planned", "hmpc_set_contact_gate", "hmpc_solve_stats", "hmpc_set_timing", "hmpc_kernel_times", "hmpc_tick_times", "hmpc_launch_count", "hmpc_hot_path_info", "hmpc_measure_fp64_peak", "hmpc_last_error",
    "hmpc_abi_version",
]


class HmpcConfig(C.Structure):
    """Mirror of ``hmpc_config`` (include/hmpc.h) -- field order and types must match exactly."""
    _fields_ = [
        ("abi_version", C.c_int32), ("device", C.c_int32), ("batch", C.c_int32), ("dyn", C.c_int32),
        ("N", C.c_int32), ("mpc_factor", C.c_int32), ("precision", C.c_int32), ("uref_mode", C.c_int32),
        ("solver", C.c_int32), ("mode", C.c_int32), ("max_iter", C.c_int32), ("check_interval", C.c_int32),
        ("first_check", C.c_int32), ("polish", C.c_int32), ("adaptive_rho", C.c_int32),
        ("warm_start", C.c_int32), ("polish_retries", C.c_int32), ("ipm_max_iter", C.c_int32),
        ("on_infeasible", C.c_int32), ("sqp_sweeps", C.c_int32), ("hot_path", C.c_int32),
        ("mpc_dt", C.c_double), ("sim_dt", C.c_double), ("m", C.c_double), ("g", C.c_double),
        ("mu", C.c_double), ("J", C.c_double * 9), ("Jinv", C.c_double * 9), ("rh", C.c_double * 3),
        ("tau_max", C.c_double * 3), ("fz_max", C.c_double), ("z_min", C.c_double), ("kf", C.c_double),
        ("eps_abs", C.c_double), ("eps_rel", C.c_double), ("rho0", C.c_double), ("sigma", C.c_double),
        ("alpha", C.c_double), ("kkt_eps", C.c_double), ("polish_tol", C.c_double), ("ipm_tol", C.c_double),
    ]


class HmpcPlanConfig(C.Structure):
    """Mirror of ``hmpc_plan_config`` (include/hmpc.h)."""
    _fields_ = [("N_run", C.c_int32), ("n_sim", C.c_int32), ("max_tick", C.c_int32), ("reserved", C.c_int32),
                ("t_p", C.c_double), ("curve_psi1", C.c_double), ("curve_psi2", C.c_double)]


class HmpcError(RuntimeError):
    pass


_lib = None


def load():
    """Load the shared library (once) and declare prototypes.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  hopper_mpc_inertial_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64p = C.c_void_p, C.c_int, C.POINTER(C.c_int64)
    lib.hmpc_abi_version.restype = C.c_int
    lib.hmpc_last_error.restype = C.c_char_p
    lib.hmpc_default_config.argtypes = [C.POINTER(HmpcConfig)]
    lib.hmpc_create.argtypes = [C.POINTER(HmpcConfig), C.POINTER(vp)]
    lib.hmpc_destroy.argtypes = [vp]
    lib.hmpc_set_stream.argtypes = [vp, vp]
    lib.hmpc_synchronize.argtypes = [vp]
    lib.hmpc_set_gains.argtypes = [vp, vp, vp]
    lib.hmpc_set_body_params.argtypes = [vp, i32, vp, vp, vp, vp, vp]
    lib.hmpc_convert.argtypes = [vp, vp, vp]
    lib.hmpc_rk4.argtypes = [vp, vp, vp, vp, i32, vp]
    lib.hmpc_linearize.argtypes = [vp, vp, vp, vp, vp]
    lib.hmpc_condense.argtypes = [vp] + [vp] * 10
    lib.hmpc_solve.argtypes = [vp, vp, vp, vp, vp, i32, vp, vp, vp, vp]
    lib.hmpc_rollout.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, i32, vp, vp, vp, vp]
    lib.hmpc_plan_set.argtypes = [vp, C.POINTER(HmpcPlanConfig), vp, vp, vp, vp, vp, vp, vp, vp]
    lib.hmpc_plan_tables.argtypes = [vp, i32, i32, vp, vp, vp, vp]
    lib.hmpc_rollout_planned.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, vp]
    lib.hmpc_set_contact_gate.argtypes = [vp, i32, vp, vp, i32, C.c_double]
    lib.hmpc_solve_stats.argtypes = [vp, vp, vp, vp, vp]
    lib.hmpc_set_timing.argtypes = [vp, i32]
    lib.hmpc_kernel_times.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int)]
    lib.hmpc_tick_times.argtypes = [vp, vp, vp, i32, C.POINTER(C.c_int)]
    lib.hmpc_launch_count.argtypes = [vp, i64p]
    lib.hmpc_hot_path_info.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), i64p]
    lib.hmpc_measure_fp64_peak.argtypes = [vp, C.POINTER(C.c_double)]
    for name in SYMBOLS:
        fn = getattr(lib, name)
        if name not in ("hmpc_last_error",):
            fn.restype = C.c_int
    if lib.hmpc_abi_version() != HMPC_ABI_VERSION:
        raise ImportError("libhmpc_b200.so ABI version mismatch; rebuild")
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().hmpc_last_error()
        raise HmpcError(f"hmpc error {rc}: {msg.decode() if msg else ''}")


def default_config():
    cfg = HmpcConfig()
    check(load().hmpc_default_config(C.byref(cfg)))
    return cfg
