// hmpc_sim.cuh -- simulator-side device functions: quaternion algebra, SE(3)->Euler conversion,
// single-rigid-body dynamics and RK4.  One thread integrates one hopper entirely in registers.
//
// Reference behaviour (file:line into the reference's src/):
//   quat_rotm   = H^T L(q) R(q)^T H                      utils.py:28-43, robotrunner.py:25-27,140
//   quat2euler  = transforms3d quat2euler(axes='rzyx')   utils.py:54-62 (SURVEY App. C3)
//   convert                                              robotrunner.py:19-28
//   dynamics_ct                                          robotrunner.py:126-152
//   rk4_normalized                                       robotrunner.py:154-164
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

namespace hmpc {

struct SimConst {
    double m, g, h;          // mass, gravity, sim_dt
    double J[9], Jinv[9];    // row-major
    double rh[3];
    // per-hopper plant body (hmpc_set_body_params), [kBodyPlant][B]: m, rh[3], J[9], Jinv[9]; or null: the scalars above
    const double* body = nullptr;
};
constexpr int kBodyPlant = 22;        // doubles per hopper of SimConst::body

// The hoppers a one-hopper-per-thread / per-warp kernel of the rollout covers (hmpc_rollout's deferral overlap,
// DESIGN.md section 5):
//   list set:   the entries list[0 .. *list_cnt) of a deferral list (bit 30 of an entry is a flag for the CTA kernel);
//   mark set:   every hopper b with mark[b] != skip, i.e. all but the hoppers deferred in the tick numbered skip;
//   neither:    every hopper.
struct HopperSet {
    const int* list = nullptr;
    const int* list_cnt = nullptr;
    const int32_t* mark = nullptr;
    int skip = 0;
};
constexpr int kListHopperMask = ~(1 << 30);

// c with hopper b's plant body in place of the scalars (the simulator's m, J, Jinv, rh, robotrunner.py:37-42)
__device__ __forceinline__ SimConst plant_body(const SimConst& c, int b, int B) {
    SimConst s = c;
    const double* p = c.body + b;
    const size_t Bs = (size_t)B;
    s.m = p[0];
#pragma unroll
    for (int i = 0; i < 3; ++i) s.rh[i] = p[(1 + i) * Bs];
#pragma unroll
    for (int i = 0; i < 9; ++i) { s.J[i] = p[(4 + i) * Bs]; s.Jinv[i] = p[(13 + i) * Bs]; }
    return s;
}

// (w^2 - v.v) I + 2 v v^T + 2 w hat(v): no division by |q|^2, exactly what L(q) R(q)^T gives for the
// un-normalised quaternions that appear inside RK4 stages.
__device__ __forceinline__ void quat_rotm(const double q[4], double R[9]) {
    const double w = q[0], x = q[1], y = q[2], z = q[3];
    const double ww = w * w, xx = x * x, yy = y * y, zz = z * z;
    R[0] = ww + xx - yy - zz; R[1] = 2.0 * (x * y - w * z); R[2] = 2.0 * (x * z + w * y);
    R[3] = 2.0 * (x * y + w * z); R[4] = ww - xx + yy - zz; R[5] = 2.0 * (y * z - w * x);
    R[6] = 2.0 * (x * z - w * y); R[7] = 2.0 * (y * z + w * x); R[8] = ww - xx - yy + zz;
}

__device__ __forceinline__ void mat3_vec(const double R[9], const double v[3], double o[3]) {
    o[0] = R[0] * v[0] + R[1] * v[1] + R[2] * v[2];
    o[1] = R[3] * v[0] + R[4] * v[1] + R[5] * v[2];
    o[2] = R[6] * v[0] + R[7] * v[1] + R[8] * v[2];
}
__device__ __forceinline__ void mat3T_vec(const double R[9], const double v[3], double o[3]) {
    o[0] = R[0] * v[0] + R[3] * v[1] + R[6] * v[2];
    o[1] = R[1] * v[0] + R[4] * v[1] + R[7] * v[2];
    o[2] = R[2] * v[0] + R[5] * v[1] + R[8] * v[2];
}
__device__ __forceinline__ void cross3(const double a[3], const double b[3], double o[3]) {
    o[0] = a[1] * b[2] - a[2] * b[1];
    o[1] = a[2] * b[0] - a[0] * b[2];
    o[2] = a[0] * b[1] - a[1] * b[0];
}

// [roll, pitch, yaw]; normalising rotation matrix as transforms3d.quat2mat does.
__device__ __forceinline__ void quat2euler(const double q[4], double rpy[3]) {
    const double w = q[0], x = q[1], y = q[2], z = q[3];
    const double nq = w * w + x * x + y * y + z * z;
    if (nq < 2.220446049250313e-16) { rpy[0] = rpy[1] = rpy[2] = 0.0; return; }
    const double s = 2.0 / nq;
    const double X = x * s, Y = y * s, Z = z * s;
    const double wX = w * X, wY = w * Y, wZ = w * Z;
    const double xX = x * X, xY = x * Y, xZ = x * Z;
    const double yY = y * Y, yZ = y * Z, zZ = z * Z;
    const double m00 = 1.0 - (yY + zZ), m10 = xY + wZ, m20 = xZ - wY;
    const double m21 = yZ + wX, m22 = 1.0 - (xX + yY), m11 = 1.0 - (xX + zZ), m12 = yZ - wX;
    const double cy = sqrt(m00 * m00 + m10 * m10);
    if (cy > 4.0 * 2.220446049250313e-16) {
        rpy[0] = atan2(m21, m22);
        rpy[1] = atan2(-m20, cy);
        rpy[2] = atan2(m10, m00);
    } else {
        rpy[0] = atan2(-m12, m11);
        rpy[1] = atan2(-m20, cy);
        rpy[2] = 0.0;
    }
}

__device__ __forceinline__ void convert_state(const double X[13], double x[12]) {
    double R[9];
    quat_rotm(&X[3], R);
    x[0] = X[0]; x[1] = X[1]; x[2] = X[2];
    quat2euler(&X[3], &x[3]);
    mat3_vec(R, &X[7], &x[6]);
    mat3_vec(R, &X[10], &x[9]);
}

__device__ __forceinline__ void dynamics_ct(const SimConst& c, const double X[13], const double U[6],
                                            const double pf[3], double dX[13]) {
    double R[9];
    quat_rotm(&X[3], R);
    const double* v = &X[7];
    const double* w = &X[10];
    double Fsum[3] = {U[0], U[1], U[2] - c.g * c.m};
    double Ftb[3], Fb[3], r[3], d[3] = {pf[0] - X[0], pf[1] - X[1], pf[2] - X[2]};
    mat3T_vec(R, Fsum, Ftb);
    mat3T_vec(R, d, r);
    r[0] += c.rh[0]; r[1] += c.rh[1]; r[2] += c.rh[2];
    mat3T_vec(R, U, Fb);
    double rxF[3];
    cross3(r, Fb, rxF);
    mat3_vec(R, v, &dX[0]);
    const double qw = X[3], qx = X[4], qy = X[5], qz = X[6];
    dX[3] = 0.5 * (-(qx * w[0] + qy * w[1] + qz * w[2]));
    dX[4] = 0.5 * (qw * w[0] + (qy * w[2] - qz * w[1]));
    dX[5] = 0.5 * (qw * w[1] + (qz * w[0] - qx * w[2]));
    dX[6] = 0.5 * (qw * w[2] + (qx * w[1] - qy * w[0]));
    double wxv[3];
    cross3(w, v, wxv);
    const double im = 1.0 / c.m;
    dX[7] = Ftb[0] * im - wxv[0];
    dX[8] = Ftb[1] * im - wxv[1];
    dX[9] = Ftb[2] * im - wxv[2];
    double Jw[3], wxJw[3], t[3];
    mat3_vec(c.J, w, Jw);
    cross3(w, Jw, wxJw);
    t[0] = U[3] + rxF[0] - wxJw[0];
    t[1] = U[4] + rxF[1] - wxJw[1];
    t[2] = U[5] + rxF[2] - wxJw[2];
    mat3_vec(c.Jinv, t, &dX[10]);
}

__device__ __forceinline__ double sim_rsqrt(double a) {
#ifdef HMPC_HOST_EMUL
    return 1.0 / sqrt(a);
#else
    double r;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(a));
    const double h = 0.5 * a;
    r = fma(r, fma(-h * r, r, 0.5), r);
    r = fma(r, fma(-h * r, r, 0.5), r);
    return r;
#endif
}

__device__ __forceinline__ void rk4_step(const SimConst& c, double X[13], const double U[6],
                                         const double pf[3]) {
    double f1[13], f2[13], f3[13], f4[13], Xt[13];
    const double h = c.h;
    dynamics_ct(c, X, U, pf, f1);
#pragma unroll
    for (int i = 0; i < 13; ++i) Xt[i] = X[i] + 0.5 * h * f1[i];
    dynamics_ct(c, Xt, U, pf, f2);
#pragma unroll
    for (int i = 0; i < 13; ++i) Xt[i] = X[i] + 0.5 * h * f2[i];
    dynamics_ct(c, Xt, U, pf, f3);
#pragma unroll
    for (int i = 0; i < 13; ++i) Xt[i] = X[i] + h * f3[i];
    dynamics_ct(c, Xt, U, pf, f4);
#pragma unroll
    for (int i = 0; i < 13; ++i) X[i] = X[i] + (h / 6.0) * (f1[i] + 2.0 * f2[i] + 2.0 * f3[i] + f4[i]);
    // q / |q| (robotrunner.py:163) as q * rsqrt(q.q): one MUFU seed + two Newton steps instead of a square root and
    // four divisions (ncu: that line held 23 % of the kernel's stall samples); within 1-2 ulp of the divided form
    const double iq = sim_rsqrt(X[3] * X[3] + X[4] * X[4] + X[5] * X[5] + X[6] * X[6]);
    X[3] *= iq; X[4] *= iq; X[5] *= iq; X[6] *= iq;
}

// ------------------------------------------------------------------------------------------------
// Contact gate of the applied control (include/hmpc.h: hmpc_set_contact_gate).  The reference computes the scheduled
// contact s = gait_scheduler(t, t0) at every simulator step and logs it, but applies U[0] ungated --
// `f_hist[k, :] = U[0, :]  # * s` (robotrunner.py:99,111-112).  mode 0 is that behaviour; mode 1 switches the
// commented-out factor on (bit k of `bits` = s at simulator step k of the tick); mode 2 detects contact from the state:
// the leg vector of dynamics_ct (robotrunner.py:143), r = rh + R(q)'(pf - p), is no longer than leg_max.
// ------------------------------------------------------------------------------------------------
struct SimGate {
    int mode;                    // HMPC_GATE_*
    const uint32_t* bits;        // [B] masks of this tick (table flavour), or null
    const uint32_t* glob;        // [max_tick] masks on the common clock (planned flavour), or null
    const int32_t* off;          // [B] tick offsets of the hoppers (planned flavour)
    int tick, max_tick;
    double leg_max2;             // leg_max squared
};
__device__ __forceinline__ uint32_t gate_bits_of(const SimGate& gt, int b) {
    if (gt.mode != 1) return 0xffffffffu;
    if (gt.bits) return gt.bits[b];
    const int j = gt.off[b] + gt.tick;
    return gt.glob[j < gt.max_tick ? j : gt.max_tick - 1];
}
__device__ __forceinline__ bool leg_reaches(const SimConst& c, const double X[13], const double pf[3], double leg_max2) {
    double R[9], r[3];
    const double d[3] = {pf[0] - X[0], pf[1] - X[1], pf[2] - X[2]};
    quat_rotm(&X[3], R);
    mat3T_vec(R, d, r);
    r[0] += c.rh[0]; r[1] += c.rh[1]; r[2] += c.rh[2];
    return r[0] * r[0] + r[1] * r[1] + r[2] * r[2] <= leg_max2;
}
// One MPC tick of the simulator for one hopper (robotrunner.py:110-113): nsteps x rk4_normalized with the tick's
// control held (times the contact gate), footstep pa before simulator step sw and pb from it on.  Xsteps (may be
// null): state after every step, [nsteps][13][B].
__device__ __forceinline__ void sim_tick(const SimConst& c, int gate_mode, uint32_t bits, double leg_max2, double X[13],
                                         const double U[6], const double pa[3], const double pb[3], int sw, int nsteps,
                                         double* Xsteps, size_t B, int b) {
    const double Z[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    for (int k = 0; k < nsteps; ++k) {
        const double* pf = (k < sw) ? pa : pb;
        bool on = true;
        if (gate_mode == 1) on = (bits >> k) & 1u;
        else if (gate_mode == 2) on = leg_reaches(c, X, pf, leg_max2);
        rk4_step(c, X, on ? U : Z, pf);
        if (Xsteps) {
#pragma unroll
            for (int i = 0; i < 13; ++i) Xsteps[((size_t)k * 13 + i) * B + b] = X[i];
        }
    }
}

}  // namespace hmpc
