"""Synthetic batches of independent hoppers (SURVEY 8d "Configs -> synthetic inputs").

Every per-hopper quantity is drawn from a counter-based generator keyed by the GLOBAL hopper index
(numpy Philox, key = seed, counter = hopper index), so a hopper's scenario does not depend on how the
batch is sharded across GPUs.
"""
from __future__ import annotations

import numpy as np

from . import planner

Q_REF = np.array([50., 50., 2., 1., 1., 50., 1., 1., 1., 10., 10., 10.])
R_REF = np.full(6, 0.001)


def default_gait_period(N, mpc_dt=0.02):
    """Gait period used for synthetic batches: one MPC horizon (N * mpc_dt), capped at the reference's
    0.8 s (robotrunner.py:43).  The reference runs N=60 (1.2 s horizon) over a 0.8 s gait, so its
    horizon always sees the next stance; a 10-stage horizon over the 0.8 s gait cannot see across the
    0.4 s swing and its height rows (z >= 0.1) become infeasible -- the reference raises 'QP FAILED'
    there too."""
    return min(planner.T_P, N * mpc_dt)


def _uniforms(seed, idx0, count, k):
    """(count, k) uniforms in [0,1): row i depends only on (seed, idx0 + i)."""
    out = np.empty((count, k))
    # Philox is counter based: advance() jumps straight to a hopper's private stream segment
    chunk = 4 * ((k + 3) // 4)
    bg = np.random.Philox(key=seed)
    bg.advance(int(idx0) * (chunk // 4))   # one Philox counter step yields 4 x 64 bits
    gen = np.random.Generator(bg)
    out[:] = gen.random((count, chunk))[:, :k]
    return out


# the reference body (robotrunner.py:37-42, hmpc_default_config)
J_REF = np.array([[76148072.89e-9, 70089.52e-9, 2067970.36e-9], [70089.52e-9, 45477183.53e-9, -87045.58e-9],
                  [2067970.36e-9, -87045.58e-9, 76287220.47e-9]])
RH_REF = -np.array([0.02663114, 0.04435752, 6.61082088]) / 1000
# ranges of make_batch(body=...): mass (kg), inertia scale, friction coefficient, hip offset (m, +- per axis), and the
# relative plant/model spread of mass and inertia
BODY_DEFAULTS = dict(mass=(6.0, 9.0), inertia=(0.8, 1.25), mu=(0.7, 1.0), rh=0.002, mismatch=0.05)
_BODY_KEY = 0xB0D7 << 64          # Philox key offset of the body draws: every other draw keeps its stream


def make_bodies(B, idx0=0, seed=1234, **ranges):
    """Per-hopper bodies of hoppers idx0 .. idx0+B-1 for BatchMpc.set_body_params.  The model (what the MPC plans
    with) gets mass U(mass), the reference inertia times U(inertia), friction U(mu) and the reference hip offset plus
    U(-rh, rh) per axis; the plant (what the simulator integrates) gets the model's mass and inertia each times
    1 + U(-mismatch, mismatch), and the model's hip offset.  Ranges default to BODY_DEFAULTS.  Drawn from their own
    Philox stream keyed by the global hopper index.  Returns (body_model, body_plant), dicts of SoA arrays:
    model m (B,), Jinv (3,3,B), rh (3,B), mu (B,);  plant m, J, Jinv, rh."""
    bad = set(ranges) - set(BODY_DEFAULTS)
    if bad:
        raise ValueError(f"unknown body ranges {sorted(bad)}; known: {sorted(BODY_DEFAULTS)}")
    r = dict(BODY_DEFAULTS, **ranges)
    u = _uniforms(int(seed) + _BODY_KEY, idx0, B, 8)
    m = r["mass"][0] + (r["mass"][1] - r["mass"][0]) * u[:, 0]
    js = r["inertia"][0] + (r["inertia"][1] - r["inertia"][0]) * u[:, 1]
    mu = r["mu"][0] + (r["mu"][1] - r["mu"][0]) * u[:, 2]
    rh = RH_REF[None] + r["rh"] * (2.0 * u[:, 3:6] - 1.0)
    mp = m * (1.0 + r["mismatch"] * (2.0 * u[:, 6] - 1.0))
    jp = js * (1.0 + r["mismatch"] * (2.0 * u[:, 7] - 1.0))
    Jm, Jp = J_REF[None] * js[:, None, None], J_REF[None] * jp[:, None, None]
    soa = lambda a: np.ascontiguousarray(np.moveaxis(a, 0, -1))
    model = dict(m=m.copy(), Jinv=soa(np.linalg.inv(Jm)), rh=soa(rh), mu=mu.copy())
    plant = dict(m=mp, J=soa(Jp), Jinv=soa(np.linalg.inv(Jp)), rh=soa(rh))
    return model, plant


def make_batch(B, idx0=0, seed=1234, N=10, n_ticks=100, N_run=None, mpc_factor=20, dt=1e-3, mpc_dt=0.02,
               randomize_gains=True, phase_ticks=None, t_p=None, z_base=(0.30, 0.45), gain_spread=1.25,
               dyn="3f", perturb=0.5, speed_range=(0.2, 1.0), curve_prob=0.5, tables=True, body=None):
    """Scenario for hoppers idx0 .. idx0+B-1.

    Each hopper gets its own straight or curved reference (goal speed 0.2..1.0 x the reference's
    0.4 m/s, random heading), its own gains (reference x logU(1/gain_spread, gain_spread); default spread 1.25, the
    "hard" bench row and test_respawn use 2.0 = SURVEY 8(d)'s logU(0.5, 2)), its own entry point into the gait
    cycle (tick offset 0..phase_ticks-1, i.e. a uniformly random gait phase) and starts near its
    reference state at that instant (perturb = 1: position +-3 cm, height -2..+3 cm, roll/pitch +-0.05 rad, yaw
    +-0.2 rad, velocity +-0.2 m/s, body rates +-0.3 rad/s; the default perturb = 0.5 halves these) -- close enough
    that the height rows stay feasible through the swing phases, as in the reference's own runs.
    body: None (every hopper has the reference body), True (make_bodies' default ranges) or a dict of make_bodies
    ranges: adds body_model / body_plant (make_bodies) and leaves every other output as it is.
    Returns numpy arrays in the SoA layout of include/hmpc.h:
    X0 (13,B), Qdiag (12,B), Rdiag (6,B), xref_tab, pf_tab, C_tab (uint64), pf_switch (uint8), C."""
    if t_p is None:
        t_p = default_gait_period(N, mpc_dt)
    if phase_ticks is None:
        phase_ticks = max(1, int(round(t_p / mpc_dt)))
    if N_run is None:
        N_run = (n_ticks + phase_ticks + 20) * mpc_factor
    u = _uniforms(seed, idx0, B, 41)
    c = 0

    def take(n):
        nonlocal c
        v = u[:, c:c + n]
        c += n
        return v

    def rng(lo, hi, n):
        return lo + (hi - lo) * take(n)

    p_xy0 = rng(-0.5, 0.5, 2)
    dp = rng(-0.03, 0.03, 2) * perturb
    dz = rng(-0.02, 0.03, 1) * perturb
    rp = rng(-0.05, 0.05, 2) * perturb
    dyaw = rng(-0.2, 0.2, 1) * perturb
    dv = rng(-0.2, 0.2, 3) * perturb
    w_b = rng(-0.3, 0.3, 3) * perturb
    gq = np.exp(rng(-np.log(gain_spread), np.log(gain_spread), 12))
    gr = np.exp(rng(-np.log(gain_spread), np.log(gain_spread), 6))
    if not randomize_gains:
        gq[:] = 1.0; gr[:] = 1.0
    speed = rng(speed_range[0], speed_range[1], 1)[:, 0]
    heading = rng(-np.pi, np.pi, 1)[:, 0]
    curve = take(1)[:, 0] < curve_prob
    if dyn == "2f":
        # 2f has no body-y force (mpc_cvx_euler_2f.py:129): the hopper can only be pushed in its own
        # x-z plane, so -- as in the reference's 2f run -- the goal lies straight ahead along +x
        heading[:] = 0.0
        dp[:, 1] = 0.0
        dv[:, 1] = 0.0
    off = np.minimum((take(1)[:, 0] * phase_ticks).astype(np.int64), phase_ticks - 1)
    zb = rng(z_base[0], z_base[1], 1)[:, 0]

    # --curve writes the y-spline into the x column (SURVEY App. D4); start those hoppers on the
    # diagonal so that the quirk does not put a jump between the initial state and the reference
    p_xy0 = np.where(curve[:, None], p_xy0[:, 0:1], p_xy0)
    T = N_run * dt
    x0p = np.zeros((B, 12)); xfp = np.zeros((B, 12))
    x0p[:, 0:2] = p_xy0; x0p[:, 2] = zb
    dist = 0.4 * speed * T
    xfp[:, 0] = p_xy0[:, 0] + dist * np.cos(heading)
    xfp[:, 1] = p_xy0[:, 1] + dist * np.sin(heading)
    xfp[:, 2] = zb
    # tables=False: only the entry row is built here (for the initial states); the device planner generates the
    # rest (BatchMpc.plan_set / plan_tables / rollout_planned with out["plan"])
    t_start = 0.5 * t_p * planner.PHI_SWITCH
    step_adj = int(round(planner.STEP_ADJUSTMENT * t_p / planner.T_P))
    tabs = planner.batch_tables(x0p, xfp, curve, off, N_run, n_ticks if tables else 0, N, mpc_factor, dt, mpc_dt,
                                t_start=t_start, t_p=t_p, step_adjustment=step_adj)
    if not tables:
        tabs = dict(xref_tab=tabs["xref_tab"][:1])
    plan = dict(x0=np.ascontiguousarray(x0p.T), xf=np.ascontiguousarray(xfp.T), curve=curve.astype(np.int32),
                tick_offset=off.astype(np.int32),
                global_args=dict(N_run=N_run, N=N, max_tick=int(phase_ticks) + n_ticks, mpc_factor=mpc_factor, dt=dt,
                                 mpc_dt=mpc_dt, t_start=t_start, t_p=t_p, phi_switch=planner.PHI_SWITCH,
                                 step_adjustment=step_adj))

    # initial simulator state: the reference state at the hopper's entry tick plus a perturbation
    r = tabs["xref_tab"][0]                       # (12,B) reference row at the entry tick
    pos = r[0:3].T + np.concatenate([dp, dz], axis=1)
    roll, pitch, yaw = rp[:, 0], rp[:, 1], r[5] + dyaw[:, 0]
    cr, sr = np.cos(roll / 2), np.sin(roll / 2)
    cp, sp = np.cos(pitch / 2), np.sin(pitch / 2)
    cy, sy = np.cos(yaw / 2), np.sin(yaw / 2)
    q = np.stack([cr * cp * cy + sr * sp * sy, sr * cp * cy - cr * sp * sy,
                  cr * sp * cy + sr * cp * sy, cr * cp * sy - sr * sp * cy], axis=1)
    v_w = r[6:9].T + dv
    # world -> body: v_b = R(q)^T v_w
    qw, qx, qy, qz = q.T
    R = np.stack([np.stack([1 - 2 * (qy * qy + qz * qz), 2 * (qx * qy - qw * qz), 2 * (qx * qz + qw * qy)], -1),
                  np.stack([2 * (qx * qy + qw * qz), 1 - 2 * (qx * qx + qz * qz), 2 * (qy * qz - qw * qx)], -1),
                  np.stack([2 * (qx * qz - qw * qy), 2 * (qy * qz + qw * qx), 1 - 2 * (qx * qx + qy * qy)], -1)], -2)
    v_b = np.einsum("bji,bj->bi", R, v_w)
    X0 = np.concatenate([pos, q, v_b, w_b], axis=1)
    out = dict(X0=np.ascontiguousarray(X0.T), Qdiag=np.ascontiguousarray((Q_REF[None] * gq).T),
               Rdiag=np.ascontiguousarray((R_REF[None] * gr).T), curve=curve, tick_offset=off, t_p=t_p, _x0p=x0p, _xfp=xfp,
               plan=plan)
    out.update(tabs)
    if body is not None and body is not False:
        out["body_model"], out["body_plant"] = make_bodies(B, idx0, seed, **({} if body is True else body))
    return out
