// hmpc_warp.cuh -- the hot path of mpcontrol: ONE WARP per hopper, no CTA barrier anywhere.
//
// Round 1's kernel gave every hopper a 128-thread CTA; its profile (profiles/r1j_full_batch_mpc_kernel_ncu.txt)
// showed 97 k warp-instructions per hopper-tick for ~2.2 k warp-DFMAs of arithmetic, 35 % of the stall samples on
// CTA barriers and four barrier-coupled hoppers per SM.  This file re-states the warm path -- time shift,
// linearise, condense, verified primal-dual active-set refinement (hmpc_qp.cuh: polish_verified), solution
// roll-out -- for a single warp:
//   * every synchronisation is a __syncwarp(); reductions, broadcasts and compactions are shuffles / ballots;
//   * the factor of the compact KKT system (order <= kcap) is the only matrix in shared memory; the condensed
//     Hessian lives in a per-warp slice of a global workspace that stays L2-resident (compact over the non-fixed
//     variables, full square so that every access is one contiguous row segment);
//   * the factorisation is a left-looking, 4-column-blocked SIGNED CHOLESKY  K = V S V'  (S = +1 on the variable
//     columns, -1 on the active-row columns of the quasi-definite polish system): accumulators in registers, one
//     own-row load + four broadcast loads per four FMAs, no store inside the update loop, the summation index split
//     over idle lanes once fewer than 17 rows remain; K's entries are gathered on the fly (no assembly pass);
//   * substitutions keep the right-hand side in registers (rows lane, lane+32, ...) and broadcast the pivot entry
//     with one shuffle per column.
// A hopper the warm path cannot finish (no valid previous tick, infeasible height row, active set not verified
// within the retry budget, system larger than kcap) is appended to a deferral list and handled by the CTA kernel
// (hmpc_kernel.cuh: interior point + polish) in a second launch; results do not depend on which kernel ran first
// because every accepted point passes the same KKT test of the original QP.
//
// Reference behaviour implemented (file:line into the reference's src/): mpc_cvx_euler_3f.py:59-68 (time shift,
// linearise, build, solve), :71-94 (gen_dt_dynamics), :96-153 (build_qp), 2f: the same lines of mpc_cvx_euler_2f.py.
#pragma once
#include <stdlib.h>

#include "hmpc_qp.cuh"
#include "hmpc_mpc.cuh"

#ifndef HMPC_EMUL_COUNT
#define HMPC_EMUL_COUNT(k) ((void)0)     // tests/emul counts events (factorisations, solves, Hessian products)
#endif

namespace hmpc {


// ------------------------------------------------------------------------------------------------
// per-warp shared memory
// ------------------------------------------------------------------------------------------------
struct WWork {
    // linearisation / condensing
    double *cz, *sz, *PC, *PS;   // [N] [N] [N+1] [N+1]
    double *Bw;                  // [N][18]  dt * B[9:12, 0:6]
    double *xin, *Qd, *Rd;       // [12] [12] [6]
    double *hinv, *hlo;          // [N] height-row normalisation 1/(k-1), height-row lower bounds
    double *blo, *bhi;           // [2][6] box bounds by (stance, component)
    double *err;                 // [N+1][12] cfree[i] - xref[i-1]; later the solution trajectory
    // QP + solver vectors
    double *g, *xp, *hx;         // [n]
    double *mul;                 // [m]
    double *rhs;                 // [kcap]  right-hand side / solution of the compact system (padded ordering)
    double *xc;                  // [n + 4] compact copy of xp for the Hessian product
    double *L;                   // factor: lower block triangle of 8x8 tiles, order <= kcap = 56, + one scratch tile
    double *Hc;                  // GLOBAL: Hessian over the non-fixed variables, [nf][ld], ld = nf rounded up to 8
    uint8_t *fr;                 // [n]  compact -> variable, the non-fixed variables in order
    uint8_t *cpos;               // [n]  variable -> compact (undefined for fixed variables)
    uint8_t *idx;                // [n]  variables of the current KKT system (compact Hessian index)
    uint8_t *grow;               // [kcap] active general rows of the current system (row index - n)
    int8_t *code, *pin, *fixed, *side, *stance;   // [m] [n] [n] [m] [N]
    int nf, ld;
    int nt_max;                  // tiles per side of the factor storage (kcap / 8)
    // ADMM mode only: K = H + dadd I + A' diag(wts) A over the system variables (null: K = the KKT system of the
    // active-set refinement)
    const double* wts;
    double dadd;
};

constexpr int kWarpKcap = 56;                       // 7 tiles of 8: largest order of the compact KKT system
// factor storage for systems of order <= kcap: lower block triangle of 8x8 tiles + one scratch tile
__host__ __device__ inline size_t warp_factor_doubles(int kcap) { const size_t nt = ((size_t)kcap + 7) / 8; return (nt * (nt + 1) / 2 + 1) * 64; }
// condense-only arrays (cz sz PC PS Bw err) live on top of the factor, which is dead while they are in use
__host__ __device__ inline size_t warp_alias_doubles(int N) { return (size_t)(4 * N + 2 + 18 * N + 12 * (N + 1)); }
// doubles of one warp's shared-memory slice
__host__ __device__ inline size_t warp_work_doubles(int N, int kcap) {
    const size_t n = 6 * (size_t)N, m = 11 * (size_t)N;
    size_t d = 0;
    const size_t f = warp_factor_doubles(kcap), al = (warp_alias_doubles(N) + 1) & ~(size_t)1;
    d += f > al ? f : al;           // L | cz sz PC PS Bw err
    d += ((n + 7) & ~(size_t)7);    // xc | rhs
    d += 2 * N + 24;                // hinv hlo blo bhi
    d += 12 + 6;                    // Qd Rd
    d += 12;                        // xin
    d += 3 * n;                     // g xp hx
    d += m;                         // mul
    d += (5 * n + (size_t)kcap + 2 * m + N + 7) / 8;   // bytes: fr cpos idx fixed pin | grow | code side | stance
    return (d + 1) & ~(size_t)1;
}
// ------------------------------------------------------------------------------------------------
// The per-hopper QP record the prep kernel leaves in HBM for the solve kernel (phase split: the condensing runs at
// high occupancy in its own launch, the solve kernel's lock-step rounds then all do the same thing -- one trial):
//   [0, hs)   compact Hessian over the non-fixed variables, [nf][ld] row-major, ld = nf rounded up to 8 (hs = ld_max^2)
//   then      g [n -> 8],  hlo [N -> 8],  x_in [12 -> 16]
// and one flag per hopper (PREP_*).
// ------------------------------------------------------------------------------------------------
enum { PREP_OK = 0, PREP_INVALID = 1, PREP_INFEASIBLE = 2 };
__host__ __device__ inline size_t prep_hstride(int N) { const size_t l = (6 * (size_t)N + 7) & ~(size_t)7; return l * l; }
__host__ __device__ inline size_t prep_stride(int N) {
    return prep_hstride(N) + ((6 * (size_t)N + 7) & ~(size_t)7) + (((size_t)N + 7) & ~(size_t)7) + 16;
}
// ADMM mode: three more m-vectors per warp (z, y, rho) behind the slice of warp_work_doubles
__host__ __device__ inline size_t warp_admm_doubles(int N) { return (3 * 11 * (size_t)N + 1) & ~(size_t)1; }
// warm block of a hopper (MpcIo::warm): shifted inputs [n -> 8] | shifted active set [m bytes -> 8 doubles]
__host__ __device__ inline int warm_stride_doubles(int N) { return ((6 * N + 7) & ~7) + ((((11 * N + 7) / 8) + 7) & ~7); }
constexpr int kPrepKcap = 8;      // the prep kernel's per-warp slice: same carve, smallest factor (unused there)

__device__ inline void wcarve(WWork& w, double* base, int N, int kcap) {
    const int n = 6 * N, m = 11 * N;
    double* p = base;
    auto take = [&](size_t k) { double* r = p; p += k; return r; };
    const size_t f = warp_factor_doubles(kcap), al = (warp_alias_doubles(N) + 1) & ~(size_t)1;
    w.L = take(f > al ? f : al);                // 16-byte aligned pieces first (the slice itself is)
    {
        double* q = w.L;                         // aliases of the factor: condense / roll-out only
        w.cz = q; q += N; w.sz = q; q += N; w.PC = q; q += N + 1; w.PS = q; q += N + 1;
        w.Bw = q; q += 18 * N; w.err = q;
    }
    w.xc = take((n + 7) & ~7);
    w.rhs = w.xc;                                // the compact right-hand side is formed after the Hessian product
    w.hinv = take(N); w.hlo = take(N); w.blo = take(12); w.bhi = take(12);
    w.Qd = take(12); w.Rd = take(6); w.xin = take(12);
    w.g = take(n); w.xp = take(n); w.hx = take(n);
    w.mul = take(m);
    uint8_t* q = reinterpret_cast<uint8_t*>(p);
    w.fr = q; q += n; w.cpos = q; q += n; w.idx = q; q += n; w.grow = q; q += kcap;
    w.code = reinterpret_cast<int8_t*>(q); q += m;
    w.side = reinterpret_cast<int8_t*>(q); q += m;
    w.fixed = reinterpret_cast<int8_t*>(q); q += n;
    w.pin = reinterpret_cast<int8_t*>(q); q += n;
    w.stance = reinterpret_cast<int8_t*>(q); q += N;
    w.nf = 0; w.ld = 0; w.nt_max = (kcap + 7) / 8;
    w.wts = nullptr; w.dadd = 0.0;
}

// ------------------------------------------------------------------------------------------------
// warp primitives
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double wmax(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(kFullMask, v, o));
    return v;
}
// ordered compaction by one warp: list[0..count) = { first + i : pred(first + i) }, at most cap stored, all counted
template <class Pred>
__device__ inline int wcompact(int first, int len, int cap, uint8_t* list, int sub, int lane, Pred pred) {
    int c = 0;
    for (int base = 0; base < len; base += 32) {
        const int i = base + lane;
        const bool p = (i < len) && pred(first + i);
        const unsigned mask = __ballot_sync(kFullMask, p);
        const int pos = c + __popc(mask & ((1u << lane) - 1u));
        if (p && pos < cap) list[pos] = (uint8_t)(first + i - sub);
        c += __popc(mask);
    }
    return c;
}


// box bounds of variable v (mpc_cvx_euler_3f.py:123-128,134-136,146; 2f: fy == 0)
__device__ __forceinline__ double wbox_lo(const WWork& w, int v) { const int k = v / 6; return w.blo[6 * w.stance[k] + (v - 6 * k)]; }
__device__ __forceinline__ double wbox_hi(const WWork& w, int v) { const int k = v / 6; return w.bhi[6 * w.stance[k] + (v - 6 * k)]; }
// bounds of row r in the slot layout [6N box | 4N friction | N height]
__device__ __forceinline__ double wrow_lo(const QpConst& c, const WWork& w, int r) {
    const int N = c.N, n = 6 * N;
    if (r < n) return wbox_lo(w, r);
    if (r < n + 4 * N) return -kInf;
    const int k = r - n - 4 * N;
    return k >= 2 ? w.hlo[k] : -kInf;
}
__device__ __forceinline__ double wrow_hi(const QpConst& c, const WWork& w, int r) {
    const int N = c.N, n = 6 * N;
    if (r < n) return wbox_hi(w, r);
    if (r < n + 4 * N) {
        const int k = (r - n) >> 2, s = (r - n) & 3;
        return (w.stance[k] && (s < 2 || c.dyn == 3)) ? 0.0 : kInf;
    }
    return kInf;
}

// Does general row g (row index - n) touch any unpinned variable?  (A decoupled row gets a unit pivot of its own.)
__device__ __forceinline__ bool wrow_coupled(const QpConst& c, const WWork& w, int g) {
    const int N = c.N;
    if (g < 4 * N) {
        const int k = g >> 2, s = g & 3;
        if (!(w.stance[k] && (s < 2 || c.dyn == 3))) return false;
        return !w.pin[6 * k + (s >> 1)] || !w.pin[6 * k + 2];
    }
    const int k = g - 4 * N;
    for (int j = 0; j + 2 <= k; ++j) if (!w.pin[6 * j + 2]) return true;
    return false;
}

// ------------------------------------------------------------------------------------------------
// linearisation of one stage (gen_dt_dynamics, mpc_cvx_euler_3f.py:82-92 / 2f:82-92); one lane per stage.
// Same arithmetic as linearize_stage (hmpc_qp.cuh); Bv is not stored: 3f  dt/m I,  2f  dt/m Rz^T (wbv).
// ------------------------------------------------------------------------------------------------
__device__ inline void wlinearize_stage(const QpConst& c, const Body& bd, const double gp[4], const double pf[3], double* czk,
                                        double* szk, double* Bw) {
    double sn, cs;
    sincos(gp[3], &sn, &cs);
    *czk = cs; *szk = sn;
    const double Rz[9] = {cs, sn, 0, -sn, cs, 0, 0, 0, 1};
    const double d[3] = {pf[0] - gp[0], pf[1] - gp[1], pf[2] - gp[2]};
    double rf[3];
    mat3_vec(Rz, d, rf);
    rf[0] += bd.rh[0]; rf[1] += bd.rh[1]; rf[2] += bd.rh[2];
    double T1[9], Jw[9], JwRzT[9], Bf[9];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            double a = 0;
            for (int l = 0; l < 3; ++l) a += Rz[3 * i + l] * bd.Jinv[3 * l + j];
            T1[3 * i + j] = a;
        }
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            double a = 0;
            for (int l = 0; l < 3; ++l) a += T1[3 * i + l] * Rz[3 * j + l];
            Jw[3 * i + j] = a;
        }
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            double a = 0;
            for (int l = 0; l < 3; ++l) a += Jw[3 * i + l] * Rz[3 * j + l];
            JwRzT[3 * i + j] = a;
        }
    if (c.dyn == 3) {
        double rw[3];
        mat3T_vec(Rz, rf, rw);
        const double hatm[9] = {0, -rw[2], rw[1], rw[2], 0, -rw[0], -rw[1], rw[0], 0};
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) {
                double a = 0;
                for (int l = 0; l < 3; ++l) a += Jw[3 * i + l] * hatm[3 * l + j];
                Bf[3 * i + j] = a;
            }
    } else {
        const double hatm[9] = {0, -rf[2], rf[1], rf[2], 0, -rf[0], -rf[1], rf[0], 0};
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) {
                double a = 0;
                for (int l = 0; l < 3; ++l) a += JwRzT[3 * i + l] * hatm[3 * l + j];
                Bf[3 * i + j] = a;
            }
    }
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            Bw[6 * i + j] = Bf[3 * i + j] * c.dt;
            Bw[6 * i + 3 + j] = JwRzT[3 * i + j] * c.dt;
        }
}
// dt * B[6:9, 0:3] of stage k, row-major (linearize_stage's Bv); m = the hopper's model mass
__device__ __forceinline__ void wbv(const QpConst& c, double m, const WWork& w, int k, double Bv[9]) {
    const double s = (1.0 / m) * c.dt;
    if (c.dyn == 3) {
        Bv[0] = s; Bv[1] = 0; Bv[2] = 0; Bv[3] = 0; Bv[4] = s; Bv[5] = 0; Bv[6] = 0; Bv[7] = 0; Bv[8] = s;
    } else {
        const double cs = w.cz[k], sn = w.sz[k];
        // (Rz^T / m) dt with Rz = [[c, s, 0], [-s, c, 0], [0, 0, 1]]
        Bv[0] = (cs / m) * c.dt; Bv[1] = (-sn / m) * c.dt; Bv[2] = 0;
        Bv[3] = (sn / m) * c.dt; Bv[4] = (cs / m) * c.dt; Bv[5] = 0;
        Bv[6] = 0; Bv[7] = 0; Bv[8] = (1.0 / m) * c.dt;
    }
}

// Linearisation of all stages about the time-shifted previous solution: x_guess[0] = x_in, x_guess[k] = x.value[k+1]
// (mpc_cvx_euler_3f.py:59-62; only p and yaw matter).  Needs w.xin; fills w.cz, w.sz, w.Bw (they alias the factor:
// wcondense fills them before the first factorisation, wfinish again after the last solve).
__device__ inline void wlinearize_all(const QpConst& c, const Body& bd, WWork& w, int b, int B, const MpcIo& io, int lane) {
    const int N = c.N;
    const size_t Bs = (size_t)B;
    for (int k = lane; k < N; k += 32) {
        double gp[4], pf[3];
        if (k == 0) { gp[0] = w.xin[0]; gp[1] = w.xin[1]; gp[2] = w.xin[2]; gp[3] = w.xin[5]; }
        else {
            const size_t o = (size_t)(k + 1) * 12;
            gp[0] = io.Xsol[(o + 0) * Bs + b]; gp[1] = io.Xsol[(o + 1) * Bs + b];
            gp[2] = io.Xsol[(o + 2) * Bs + b]; gp[3] = io.Xsol[(o + 5) * Bs + b];
        }
        for (int i = 0; i < 3; ++i) pf[i] = io.pf[(size_t)(3 * k + i) * Bs + b];
        wlinearize_stage(c, bd, gp, pf, w.cz + k, w.sz + k, w.Bw + 18 * k);
    }
}

// stance flags, box bounds, height-row scaling, fixed variables and the compact ordering of the non-fixed ones: all
// functions of the contact schedule only.  Ends with a __syncwarp().
__device__ inline void wload_sets(const QpConst& c, WWork& w, uint64_t bits, int lane) {
    const int N = c.N, n = 6 * N;
    for (int k = lane; k < N; k += 32) w.stance[k] = (int8_t)((bits >> k) & 1ull);
    if (lane < 12) {   // box bounds by (stance, component)
        const int st = lane / 6, cc = lane - 6 * st;
        double lo = -kInf, hi = kInf;
        if (cc >= 3) { lo = -c.tau_max[cc - 3]; hi = c.tau_max[cc - 3]; }
        else if (!st) { lo = 0.0; hi = 0.0; }
        else if (cc == 2) { lo = 0.0; hi = c.fz_max; }
        if (cc == 1 && c.dyn == 2) { lo = 0.0; hi = 0.0; }
        w.blo[lane] = lo; w.bhi[lane] = hi;
    }
    for (int k = lane; k < N; k += 32) w.hinv[k] = (k >= 2) ? 1.0 / (double)(k - 1) : 0.0;
    __syncwarp();
    for (int v = lane; v < n; v += 32) w.fixed[v] = (wbox_hi(w, v) - wbox_lo(w, v)) < 1e-12 ? 1 : 0;
    __syncwarp();
    // non-fixed variables, in order
    w.nf = wcompact(0, n, n, w.fr, 0, lane, [&](int v) { return w.fixed[v] == 0; });
    w.ld = (w.nf + 7) & ~7;
    __syncwarp();
    for (int i = lane; i < w.nf; i += 32) w.cpos[w.fr[i]] = (uint8_t)i;
    __syncwarp();
}

// ------------------------------------------------------------------------------------------------
// load + time shift + linearise + condense for hopper b (warm tick).  Returns 1 (all lanes) when a height row
// cannot be met (SURVEY App. D2).  Leaves Hc (global, compact), g, bounds, fixed / fr / cpos in place.
// ------------------------------------------------------------------------------------------------
__device__ inline int wcondense(const QpConst& c, WWork& w, int b, int B, const MpcIo& io, int lane) {
    const int N = c.N, n = 6 * N;
    const size_t Bs = (size_t)B;
    // Every global load of the condensing is issued here, back to back, into registers -- state, gains, model body,
    // contact mask, the linearisation point and footstep of this lane's stage, this lane's reference row: ONE HBM round
    // trip instead of four dependent ones (N <= kWarpMaxN < 32: one stage / one row per lane).
    const int k = lane;                                   // stage of wlinearize_all, row i = lane of the error loop
    double xq = 0.0, qq = 0.0, rq = 0.0, gp[4] = {0.0, 0.0, 0.0, 0.0}, pfq[3] = {0.0, 0.0, 0.0}, xr[12];
    const Body bd = model_body(c, b, B);
    if (lane < 12) { xq = io.x_in[lane * Bs + b]; qq = io.Qd[lane * Bs + b]; }
    if (lane < 6) rq = io.Rd[lane * Bs + b];
    const uint64_t bits = io.Cbits[b];
    if (k < N) {
        if (k == 0) {
            gp[0] = io.x_in[0 * Bs + b]; gp[1] = io.x_in[1 * Bs + b]; gp[2] = io.x_in[2 * Bs + b]; gp[3] = io.x_in[5 * Bs + b];
        } else {
            const size_t o = (size_t)(k + 1) * 12;
            gp[0] = io.Xsol[(o + 0) * Bs + b]; gp[1] = io.Xsol[(o + 1) * Bs + b];
            gp[2] = io.Xsol[(o + 2) * Bs + b]; gp[3] = io.Xsol[(o + 5) * Bs + b];
        }
#pragma unroll
        for (int i = 0; i < 3; ++i) pfq[i] = io.pf[(size_t)(3 * k + i) * Bs + b];
    }
#pragma unroll
    for (int q = 0; q < 12; ++q) xr[q] = (lane >= 1 && lane <= N) ? io.x_ref[((size_t)(lane - 1) * 12 + q) * Bs + b] : 0.0;
    if (lane < 12) { w.xin[lane] = xq; w.Qd[lane] = qq; }
    if (lane < 6) w.Rd[lane] = rq;
    wload_sets(c, w, bits, lane);
    if (k < N) wlinearize_stage(c, bd, gp, pfq, w.cz + k, w.sz + k, w.Bw + 18 * k);      // wlinearize_all on the loaded point
    __syncwarp();
    // prefix sums of cos / sin (same summation order as condense())
    for (int i = lane; i <= N; i += 32) {
        double pc = 0, ps = 0;
        for (int k = 0; k < i; ++k) { pc += w.cz[k]; ps += w.sz[k]; }
        w.PC[i] = pc; w.PS[i] = ps;
    }
    __syncwarp();
    const double dt = c.dt, gdt = -c.g * dt;
    const double zc = dt * dt / bd.m;
    int infeasible = 0;
    // free response + tracking error; height rows
    for (int i = lane; i <= N; i += 32) {
        double cf[12];
        const double* x0 = w.xin;
        const double di = (double)i;
        cf[6] = x0[6]; cf[7] = x0[7]; cf[8] = x0[8] + di * gdt;
        cf[9] = x0[9]; cf[10] = x0[10]; cf[11] = x0[11];
        cf[0] = x0[0] + dt * (di * x0[6]);
        cf[1] = x0[1] + dt * (di * x0[7]);
        cf[2] = x0[2] + dt * (di * x0[8] + gdt * (0.5 * di * (di - 1.0)));
        const double pc = w.PC[i], ps = w.PS[i];
        cf[3] = x0[3] + dt * (pc * x0[9] + ps * x0[10]);
        cf[4] = x0[4] + dt * (-ps * x0[9] + pc * x0[10]);
        cf[5] = x0[5] + dt * (di * x0[11]);
        if (i >= 1)
            for (int q = 0; q < 12; ++q) w.err[12 * i + q] = cf[q] - xr[q];           // i == lane (N < 32)
        if (i < N) {
            double up = 0.0;
            for (int j = 0; j + 2 <= i; ++j) if (w.stance[j]) up += (double)(i - j - 1);
            if (cf[2] + zc * c.fz_max * up < c.z_min) infeasible = 1;
            w.hlo[i] = (i >= 2) ? (c.z_min - cf[2]) / (zc * (double)(i - 1)) : -kInf;
        }
    }
    infeasible = __any_sync(kFullMask, infeasible);
    __syncwarp();
    // ---- Hessian blocks (a >= b), non-fixed entries only, written to both triangles of the compact square ----
    const int nf = w.ld;                 // leading dimension of the compact square
    double* Hc = w.Hc;
    for (int i = lane; i < w.nf; i += 32)   // zero pad columns: the tiled Hessian product reads whole 8-column tiles
        for (int j = w.nf; j < nf; ++j) Hc[i * nf + j] = 0.0;
    const int nblk = N * (N + 1) / 2;
    const double q3 = w.Qd[3], q4 = w.Qd[4], q5 = w.Qd[5];
    const double dt2 = dt * dt;
    for (int p = lane; p < nblk; p += 32) {
        int a = (int)((sqrt(8.0 * (double)p + 1.0) - 1.0) * 0.5);
        while ((a + 1) * (a + 2) / 2 <= p) ++a;
        while (a * (a + 1) / 2 > p) --a;
        const int bb = p - a * (a + 1) / 2;
        const double pca = w.PC[a + 1], psa = w.PS[a + 1], pcb = w.PC[bb + 1], psb = w.PS[bb + 1];
        double s0 = 0, NN = 0, CC = 0, SS = 0, CS = 0, SC = 0;
        for (int i = a + 1; i <= N; ++i) {
            const double kap = (i == N) ? c.kf : 1.0;
            const double wca = w.PC[i] - pca, wsa = w.PS[i] - psa, wcb = w.PC[i] - pcb, wsb = w.PS[i] - psb;
            const double na = (double)(i - a - 1), nb = (double)(i - bb - 1);
            s0 += kap; NN += kap * na * nb;
            CC += kap * wca * wcb; SS += kap * wsa * wsb; CS += kap * wca * wsb; SC += kap * wsa * wcb;
        }
        const double M3[9] = {s0 * w.Qd[9] + dt2 * (q3 * CC + q4 * SS), dt2 * (q3 * CS - q4 * SC), 0,
                              dt2 * (q3 * SC - q4 * CS), s0 * w.Qd[10] + dt2 * (q3 * SS + q4 * CC), 0,
                              0, 0, s0 * w.Qd[11] + dt2 * q5 * NN};
        const double dv[3] = {dt2 * NN * w.Qd[0] + s0 * w.Qd[6], dt2 * NN * w.Qd[1] + s0 * w.Qd[7],
                              dt2 * NN * w.Qd[2] + s0 * w.Qd[8]};
        const double* Bwa = w.Bw + 18 * a; const double* Bwb = w.Bw + 18 * bb;
        double Bva[9], Bvb[9];
        wbv(c, bd.m, w, a, Bva); wbv(c, bd.m, w, bb, Bvb);
        double MB[18];   // M3 * Bw_b (3x6)
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 6; ++j)
                MB[6 * i + j] = M3[3 * i] * Bwb[j] + M3[3 * i + 1] * Bwb[6 + j] + M3[3 * i + 2] * Bwb[12 + j];
        // compact positions of the two stages' variables (-1: fixed), read once per block
        int pa[6], pb[6];
#pragma unroll
        for (int r = 0; r < 6; ++r) {
            pa[r] = w.fixed[6 * a + r] ? -1 : (int)w.cpos[6 * a + r];
            pb[r] = w.fixed[6 * bb + r] ? -1 : (int)w.cpos[6 * bb + r];
        }
        // fully unrolled so that MB / Bva / Bvb stay in registers; fixed rows and columns are skipped by predicate
#pragma unroll
        for (int r = 0; r < 6; ++r) {
            const int ci = pa[r];
            if (ci < 0) continue;
#pragma unroll
            for (int cc = 0; cc < 6; ++cc) {
                const int cj = pb[cc];
                if (cj < 0 || (a == bb && r < cc)) continue;          // a == b: the lower half only, mirrored below
                double v = Bwa[r] * MB[cc] + Bwa[6 + r] * MB[6 + cc] + Bwa[12 + r] * MB[12 + cc];
                if (r < 3 && cc < 3)
                    v += Bva[r] * dv[0] * Bvb[cc] + Bva[3 + r] * dv[1] * Bvb[3 + cc] + Bva[6 + r] * dv[2] * Bvb[6 + cc];
                v *= 2.0;
                if (a == bb && r == cc && a != N - 1) v += 2.0 * w.Rd[r];
                Hc[ci * nf + cj] = v;
                Hc[cj * nf + ci] = v;
            }
        }
    }
    // ---- gradient ----
    const double ubar_alias = (c.uref_mode == 0) ? (w.stance[N - 1] ? 2.0 * bd.m * c.g : 0.0) : 0.0;
    for (int a = lane; a < N; a += 32) {
        double ap[3] = {0, 0, 0}, av[3] = {0, 0, 0}, aw[3] = {0, 0, 0}, at[3] = {0, 0, 0};
        const double pca = w.PC[a + 1], psa = w.PS[a + 1];
        for (int i = a + 1; i <= N; ++i) {
            const double kap = (i == N) ? c.kf : 1.0;
            const double* e = w.err + 12 * i;
            const double na = (double)(i - a - 1);
            const double wca = w.PC[i] - pca, wsa = w.PS[i] - psa;
            for (int q = 0; q < 3; ++q) { ap[q] += kap * na * e[q]; av[q] += kap * e[6 + q]; aw[q] += kap * e[9 + q]; }
            at[0] += kap * (wca * q3 * e[3] - wsa * q4 * e[4]);
            at[1] += kap * (wsa * q3 * e[3] + wca * q4 * e[4]);
            at[2] += kap * (na * q5 * e[5]);
        }
        double tv[3], tw[3];
        for (int q = 0; q < 3; ++q) {
            tv[q] = dt * w.Qd[q] * ap[q] + w.Qd[6 + q] * av[q];
            tw[q] = dt * at[q] + w.Qd[9 + q] * aw[q];
        }
        const double* Bwa = w.Bw + 18 * a;
        double Bva[9];
        wbv(c, bd.m, w, a, Bva);
        for (int r = 0; r < 6; ++r) {
            double v = Bwa[r] * tw[0] + Bwa[6 + r] * tw[1] + Bwa[12 + r] * tw[2];
            if (r < 3) v += Bva[r] * tv[0] + Bva[3 + r] * tv[1] + Bva[6 + r] * tv[2];
            v *= 2.0;
            if (r == 2 && a != N - 1) {
                const double ub = (c.uref_mode == 0) ? ubar_alias : (w.stance[a] ? 2.0 * bd.m * c.g : 0.0);
                v -= 2.0 * w.Rd[2] * ub;
            }
            w.g[6 * a + r] = v;
        }
    }
    __syncwarp();
#ifndef HMPC_HOST_EMUL
    __threadfence_block();   // Hc is written and read by lanes of this warp only
#endif
    return infeasible;
}

// ------------------------------------------------------------------------------------------------
// Code-size rule for everything below: the kernel is bound by instruction FETCH (profiles/README.md: with the tile
// loops unrolled the trial code was 140 KB and `no_instruction` the top stall even with every warp of the SM in
// lock-step), so the tile loops are real loops (#pragma unroll 1), vectors travel through shared memory instead of
// statically indexed register arrays, and the hot code of a trial stays within the instruction cache.
// ------------------------------------------------------------------------------------------------


// ------------------------------------------------------------------------------------------------
// hx = H xp over the non-fixed variables.  H: compact square in global memory, row-major, leading dimension
// w.ld = nf rounded up to 8 with zero pad columns.  8x8 tiles through the tensor core, the vector as an 8x1 operand.
// Ends with a __syncwarp().
// ------------------------------------------------------------------------------------------------
__device__ inline void wmatvec(WWork& w, int lane) {
    const int nf = w.nf, ld = w.ld, ntf = ld >> 3, g = lane >> 2, t = lane & 3;
    HMPC_EMUL_COUNT(1);
    for (int j = lane; j < ld; j += 32) w.xc[j] = j < nf ? w.xp[w.fr[j]] : 0.0;
    __syncwarp();
    const double* hp = w.Hc + g * ld + 2 * t;
#pragma unroll 1
    for (int I = 0; I < ntf; I += 2) {
        // all tiles of TWO block rows are requested from L2 before the first product (ntf <= 8): one L2 round trip per
        // pair of block rows (ncu: the products of this loop held 10 % of the kernel's long-scoreboard stalls)
        const bool two = I + 1 < ntf;
        const double* hq = hp + (two ? 8 * ld : 0);
        d2 h[8], q[8];
#pragma unroll
        for (int K = 0; K < 8; ++K) h[K] = (K < ntf) ? ld2(hp + 8 * K) : d2{0.0, 0.0};
#pragma unroll
        for (int K = 0; K < 8; ++K) q[K] = (K < ntf) ? ld2(hq + 8 * K) : d2{0.0, 0.0};
        double a0 = 0.0, a1 = 0.0, b0 = 0.0, b1 = 0.0;            // two chains per block row: even / odd column tiles
        double c0 = 0.0, c1 = 0.0, e0 = 0.0, e1 = 0.0;
#pragma unroll
        for (int K = 0; K < 8; K += 2) {
            if (K < ntf) {
                const d2 v = vec_b(w.xc + 8 * K, lane);
                tile_mac(a0, a1, h[K], v);
                tile_mac(c0, c1, q[K], v);
            }
            if (K + 1 < ntf) {
                const d2 v = vec_b(w.xc + 8 * K + 8, lane);
                tile_mac(b0, b1, h[K + 1], v);
                tile_mac(e0, e1, q[K + 1], v);
            }
        }
        const int i = 8 * I + g;
        if (t == 0 && i < nf) w.hx[w.fr[i]] = a0 + b0;
        if (two && t == 0 && i + 8 < nf) w.hx[w.fr[i + 8]] = c0 + e0;
        hp += 16 * ld;
    }
    __syncwarp();
}

// entry (i, j), i >= j, of the compact KKT system in the ordering [nF variables | ng rows]
// ADMM operator: what A' diag(wts) A + dadd I adds to entry (ci, cj) of the compact Hessian (hmpc_qp.cuh: LinSys::entry)
__device__ __forceinline__ double wweights(const WWork& w, const AOp& A, int ci, int cj) {
    const int vi = (int)w.fr[ci], vj = (int)w.fr[cj];
    double s = A.gram(vi, vj, w.wts);
    if (ci == cj) s += w.wts[vi] + w.dadd;
    return s;
}
template <bool ADMM = false>
static __device__ __noinline__ double wentry(const QpConst& c, const WWork& w, const AOp& A, int nF, int nk, int i, int j) {
    const int n = 6 * c.N;
    if (i < j || i >= nk) return 0.0;
    if (i < nF) {
        const double h = w.Hc[(int)w.idx[j] * w.ld + (int)w.idx[i]];
        return ADMM ? h + wweights(w, A, (int)w.idx[i], (int)w.idx[j]) : h;
    }
    if (j < nF) return A.coef(n + (int)w.grow[i - nF], (int)w.fr[w.idx[j]]);
    if (i == j) return wrow_coupled(c, w, (int)w.grow[i - nF]) ? 0.0 : -1.0;
    return 0.0;
}

// ------------------------------------------------------------------------------------------------
// Signed Cholesky  K = V S V'  of the compact KKT system of order nk = nF + ng (LinSys in hmpc_qp.cuh describes K:
// variables idx[0..nF), active general rows grow[0..ng), K_vv = H, K_rv = A.coef, K_rr = 0 with the Schur
// complement's diagonal scaled by (1 + eps) once the variables are eliminated, -1 for a decoupled row).
// Left-looking, tile by tile (block column J, row tile I >= J):
//   C(I,J) = K(I,J) - sum_{K<J} V(I,K) S_K V(J,K)'      tile products on the tensor core
//   C(J,J) = V(J,J) S_J V(J,J)',  W_J = V(J,J)^-1        wdiag8
//   V(I,J) = C(I,J) W_J' S_J                             the accumulator fragment is the A operand as it stands
// The tile that holds pivot nF mixes both signs: its columns are applied in two masked passes, the regularisation of
// the diagonal in between.  Storage w.L: lower block triangle of row-major 8x8 tiles, the diagonal tiles hold W_J.
// Returns nonzero (all lanes) when a pivot has the wrong sign or is not finite.
// ------------------------------------------------------------------------------------------------
// ADMM = true: K's variable block carries the weights of the ADMM operator (w.wts, w.dadd); a template parameter so
// that the exact path's kernel is not touched by it (154 registers; 168 with a run-time switch, -1.4 % throughput).
template <bool ADMM = false>
__device__ inline int wfactor(const QpConst& c, WWork& w, const AOp& A, int nF, int ng, double eps, int lane) {
    HMPC_EMUL_COUNT(2);
    const int nk = nF + ng, nt = (nk + 7) >> 3;
    const int Jb = nF >> 3;                                          // tile of the first active-row pivot
    const bool mixed = (nF & 7) != 0;                                // ... which also holds variables
    const int g = lane >> 2, t = lane & 3, fo = 8 * g + 2 * t;      // fragment offset inside a tile
    double* L = w.L;
    double* scratch = w.L + tile_off(w.nt_max, 0);                   // one spare tile behind the factor
    // masks of the mixed tile for the two columns of this lane's B fragment: 1 variable column, 0 row column
    const double mv0 = (8 * Jb + 2 * t < nF) ? 1.0 : 0.0, mv1 = (8 * Jb + 2 * t + 1 < nF) ? 1.0 : 0.0;
    const bool ondiag0 = (2 * t == g), ondiag1 = (2 * t + 1 == g);
    int bad = 0;
#pragma unroll 1
    for (int J = 0; J < nt; ++J) {
        const int j0 = 8 * J + 2 * t;
        const double s0 = (j0 < nF) ? 1.0 : -1.0, s1 = (j0 + 1 < nF) ? 1.0 : -1.0;
        const double* Lj = L + tile_off(J, 0) + fo;                  // tiles (J, K), K = 0 .. J
        const bool scaled = (J > Jb) || (J == Jb && !mixed);        // diagonal regularised here (else inside wdiag8)
        // Hessian rows of this lane's two columns (block column J made of variables only: plain gather)
        const bool jvars = 8 * J + 8 <= nF;
        const double* hc0 = w.Hc + (jvars ? (int)w.idx[j0] * w.ld : 0);
        const double* hc1 = w.Hc + (jvars ? (int)w.idx[j0 + 1] * w.ld : 0);
        d2 bw = d2{0.0, 0.0};
#pragma unroll 1
        for (int I = J; I < nt; ++I) {
            const double* Li = L + tile_off(I, 0) + fo;              // tiles (I, K)
            // K(I, J) first: the gather from the L2-resident Hessian is in flight while the tile products run
            const int i = 8 * I + g;
            double k0, k1;
            if (8 * I + 8 <= nF) {                                   // variables x variables (H is stored symmetric)
                const int ri = (int)w.idx[i];
                k0 = hc0[ri]; k1 = hc1[ri];
                if (ADMM) {                                          // ADMM operator (i >= j0, j0 + 1 may exceed i: unused)
                    k0 += wweights(w, A, ri, (int)w.idx[j0]);
                    k1 += wweights(w, A, ri, (int)w.idx[j0 + 1]);
                }
            } else if (i < nF) {
                // a variable row inside the tile row that also holds active rows: its two Hessian entries are gathered
                // like above -- both loads in flight together and ahead of the tile products -- instead of through two
                // dependent wentry() calls (ncu: 20 % of the kernel's long-scoreboard stalls sat in wentry).  A column
                // >= nF lies above the diagonal for this row: never used.
                const int ri = (int)w.idx[i];
                const bool v0 = j0 < nF, v1 = j0 + 1 < nF;
                const int cj0 = v0 ? (int)w.idx[j0] : 0, cj1 = v1 ? (int)w.idx[j0 + 1] : 0;
                const double h0 = w.Hc[cj0 * w.ld + ri], h1 = w.Hc[cj1 * w.ld + ri];
                k0 = v0 ? h0 : 0.0; k1 = v1 ? h1 : 0.0;
                if (ADMM) {
                    if (v0) k0 += wweights(w, A, ri, cj0);
                    if (v1) k1 += wweights(w, A, ri, cj1);
                }
            } else {
                k0 = wentry<ADMM>(c, w, A, nF, nk, i, j0); k1 = wentry<ADMM>(c, w, A, nF, nk, i, j0 + 1);
            }
            double a0 = 0.0, a1 = 0.0;
            const int kplain = J < Jb ? J : Jb;
#pragma unroll 1
            for (int K = 0; K < kplain; ++K) tile_mac(a0, a1, ld2(Li + 64 * K), ld2(Lj + 64 * K));   // variables: +
            if (J > Jb) {
                if (mixed) {                                         // variable columns of the mixed tile
                    const d2 b = ld2(Lj + 64 * Jb);
                    tile_mac(a0, a1, ld2(Li + 64 * Jb), d2{b.x * mv0, b.y * mv1});
                }
            }
            if (scaled && I == J) {                                  // the Schur complement's diagonal
                if (ondiag0) a0 *= 1.0 + eps;
                if (ondiag1) a1 *= 1.0 + eps;
            }
            if (J > Jb) {
                if (mixed) {                                         // row columns of the mixed tile: -
                    const d2 b = ld2(Lj + 64 * Jb);
                    tile_mac(a0, a1, ld2(Li + 64 * Jb), d2{b.x * (mv0 - 1.0), b.y * (mv1 - 1.0)});
                }
#pragma unroll 1
                for (int K = Jb + (mixed ? 1 : 0); K < J; ++K) {     // active-row columns: -
                    const d2 b = ld2(Lj + 64 * K);
                    tile_mac(a0, a1, ld2(Li + 64 * K), d2{-b.x, -b.y});
                }
            }
            // C = K - acc
            if (I == J) {
                if (i >= nk) { if (ondiag0) k0 = -1.0; if (ondiag1) k1 = -1.0; }          // past the end: unit pivots
                else if (scaled && i >= nF) { if (ondiag0) k0 *= 1.0 + eps; if (ondiag1) k1 *= 1.0 + eps; }
            }
            const double c0 = k0 - a0, c1 = k1 - a1;
            if (I == J) {                                            // diagonal tile -> W_J
                st2(scratch + fo, c0, c1);
                __syncwarp();
                double* Wt = L + tile_off(J, J);
                const int jrel = nF - 8 * J;                         // first active-row pivot inside this tile
                if (jrel > 0 && jrel < 8) bad |= wdiag8<true>(scratch, Wt, jrel, 1.0, eps, lane);
                else bad |= wdiag8<false>(scratch, Wt, 0, jrel >= 8 ? 1.0 : -1.0, eps, lane);
                bw = ld2(Wt + fo);
            } else {                                                 // panel: V(I,J) = C(I,J) W_J' S_J
                double d0 = 0.0, d1 = 0.0;
                tile_mac(d0, d1, d2{c0, c1}, bw);
                st2(L + tile_off(I, J) + fo, s0 * d0, s1 * d1);
            }
        }
        __syncwarp();
    }
    return bad;
}

// ------------------------------------------------------------------------------------------------
// Solves K x = b in place on w.rhs (length nk, padded with zeros to 8 nt) with K = V S V':
//   forward   z_I = W_I (b_I - sum_{J<I} V(I,J) z_J)        backward   x_J = W_J' (S z_J - sum_{I>J} V(I,J)' x_I)
// Tile-times-vector products on the tensor core; the vector pieces travel through w.rhs.  Ends with a __syncwarp().
// ------------------------------------------------------------------------------------------------
__device__ inline void wsolve(WWork& w, int nF, int ng, int lane) {
    HMPC_EMUL_COUNT(3);
    const int nk = nF + ng, nt = (nk + 7) >> 3;
    const int g = lane >> 2, t = lane & 3, fo = 8 * g + 2 * t;
    const double* L = w.L;
    double* v = w.rhs;
    if (lane < 8 * nt - nk) v[nk + lane] = 0.0;
    __syncwarp();
#pragma unroll 1
    for (int I = 0; I < nt; ++I) {
        const double* Li = L + tile_off(I, 0) + fo;
        double a0 = 0.0, a1 = 0.0;
#pragma unroll 1
        for (int J = 0; J < I; ++J) tile_mac(a0, a1, ld2(Li + 64 * J), vec_b(v + 8 * J, lane));
        const double r = v[8 * I + g] - a0;
        __syncwarp();
        if (t == 0) v[8 * I + g] = r;
        __syncwarp();
        double z0 = 0.0, z1 = 0.0;
        tile_mac(z0, z1, ld2(Li + 64 * I), vec_b(v + 8 * I, lane));
        __syncwarp();
        if (t == 0) v[8 * I + g] = z0;
        __syncwarp();
    }
#pragma unroll 1
    for (int J = nt - 1; J >= 0; --J) {
        double a0 = 0.0, a1 = 0.0;
#pragma unroll 1
        for (int I = nt - 1; I > J; --I) {
            const double* T = L + tile_off(I, J);                     // A = V(I,J)': A[g][2t + h] = T[2t + h][g]
            tile_mac(a0, a1, d2{T[8 * (2 * t) + g], T[8 * (2 * t + 1) + g]}, vec_b(v + 8 * I, lane));
        }
        const int i = 8 * J + g;
        const double zi = v[i];
        const double r = (i < nF ? zi : -zi) - a0;
        __syncwarp();
        if (t == 0) v[i] = r;
        __syncwarp();
        const double* Wt = L + tile_off(J, J);
        double x0 = 0.0, x1 = 0.0;
        tile_mac(x0, x1, d2{Wt[8 * (2 * t) + g], Wt[8 * (2 * t + 1) + g]}, vec_b(v + i - g, lane));
        __syncwarp();
        if (t == 0) v[i] = x0;
        __syncwarp();
    }
}

struct WInfo { int nfac; double flops; };

// ------------------------------------------------------------------------------------------------
// Verified primal-dual active-set refinement for one warp: the same algorithm, tolerances and update rules
// as polish_verified (hmpc_qp.cuh; numpy statement oracle/device_port.py polish_verified).
// On entry w.xp = starting point, w.code = active-set guess.  Returns 1 (all lanes) with w.xp = solution,
// w.mul = multipliers, w.code = active set; 0 when the warm path gives up.
// ------------------------------------------------------------------------------------------------
__device__ inline void wpolish_init(const QpConst& c, WWork& w, int lane) {
    const int N = c.N, n = 6 * N, m = 11 * N;
    for (int r = lane; r < m; r += 32) {
        int cd = w.code[r];
        if (cd > 0 && wrow_hi(c, w, r) > kInfThresh) cd = 0;
        if (cd < 0 && wrow_lo(c, w, r) < -kInfThresh) cd = 0;
        if (r < n && w.fixed[r]) cd = 0;
        w.code[r] = (int8_t)cd;
    }
    __syncwarp();
}
// One trial: 1 = verified optimum (w.xp, w.mul, w.code), 0 = active set updated, try again, -1 = give up,
// -2 = the system does not fit this kernel's factor storage.
struct NoSync { __device__ __forceinline__ void operator()(int) const {} };
// mid(p): re-alignment points of the lock-step kernel (a group barrier that brings the warps of the SM back in step so
// that they share instruction fetches; NoSync elsewhere).  Every lane calls mid(0) -- after the factorisation -- and
// mid(1) -- after the refinement loop -- exactly once per trial, whatever path it takes.
template <int SLOTS, class Sync = NoSync>
__device__ inline int wtrial(const QpConst& c, WWork& w, const AOp& A, int kcap, WInfo& info, int lane, Sync mid = Sync()) {
    const int N = c.N, n = 6 * N, m = 11 * N;
    const double tol = c.polish_tol;
    double* mul = w.mul;
    {
        for (int r = lane; r < m; r += 32) {
            const int cd = w.code[r];
            mul[r] = 0.0;
            if (r < n) {
                const int pin = (w.fixed[r] || cd != 0) ? 1 : 0;
                w.pin[r] = (int8_t)pin;
                if (pin) w.xp[r] = w.fixed[r] ? 0.0 : (cd < 0 ? wbox_lo(w, r) : wbox_hi(w, r));
            }
        }
        __syncwarp();
        // system variables as compact Hessian indices (the non-fixed, unpinned variables in order)
        const int nF = wcompact(0, w.nf, n, w.idx, 0, lane, [&](int i) { return w.pin[w.fr[i]] == 0; });
        const int ng = wcompact(n, m - n, kcap, w.grow, n, lane, [&](int r) { return w.code[r] != 0; });
        __syncwarp();
        const int nk = nF + ng;
        if (nk > kcap) { HMPC_EMUL_COUNT(6); mid(0); mid(1); return -2; }     // too large for this kernel, not a failed attempt
        ++info.nfac;
        info.flops += flops_factor(nk);
        const int fbad = wfactor(c, w, A, nF, ng, c.kkt_eps, lane);
        mid(0);
        if (fbad) { mid(1); return -1; }
        double prev = 1e300;
        bool hx_current = false;
        for (int k = 0; k < c.max_refine; ++k) {
            wmatvec(w, lane);
            info.flops += flops_matvec(n);
            double v0 = 0.0, v1 = 0.0;   // residual; largest residual relative to the terms it is the difference of
            for (int i = lane; i < nk; i += 32) {
                double r_, mag;
                if (i < nF) {
                    const int vi = w.fr[w.idx[i]];
                    const double aty = A.colT(vi, mul);
                    r_ = -(w.hx[vi] + w.g[vi] + aty);
                    mag = fabs(w.hx[vi]) + fabs(w.g[vi]) + fabs(aty);
                } else {
                    const int rr = n + (int)w.grow[i - nF];
                    const double ax = A.row(rr, w.xp);
                    const double bnd = w.code[rr] < 0 ? wrow_lo(c, w, rr) : wrow_hi(c, w, rr);
                    r_ = bnd - ax;
                    mag = fabs(bnd) + fabs(ax);
                }
                w.rhs[i] = r_;
                v0 = fmax(v0, fabs(r_));
                v1 = fmax(v1, fabs(r_) / (mag + 1e-300));
            }
            v0 = wmax(v0); v1 = wmax(v1);
            __syncwarp();
            if (!(v0 == v0)) { mid(1); return -1; }
            if (k == 1 && ng == 0 && v0 <= 1e-7 * prev) { hx_current = true; break; }
            if (k >= 1 && (v1 <= 1e-12 || (k >= 2 && v0 > c.stagnation * prev))) { hx_current = true; break; }
            prev = v0;
            wsolve(w, nF, ng, lane);
            info.flops += flops_solve(nk);
            for (int i = lane; i < nk; i += 32) {
                if (i < nF) w.xp[w.fr[w.idx[i]]] += w.rhs[i];
                else mul[n + (int)w.grow[i - nF]] += w.rhs[i];
            }
            __syncwarp();
        }
        mid(1);
        // ---- pass 1: multipliers of pinned variables, scales ----
        if (!hx_current) { wmatvec(w, lane); info.flops += flops_matvec(n); }
        double s_stat = 0.0, s_scale = 0.0, s_mult = 0.0;
        int notfinite = 0;                                // fmax() drops NaNs: test the gradient entries themselves
        for (int i = lane; i < n; i += 32) {
            if (w.fixed[i]) continue;                     // eliminated a priori: no Hessian row, multiplier unused
            const double aty = A.colT(i, mul);            // mul[i] == 0 on box rows at this point
            const double G = w.hx[i] + w.g[i] + aty;
            if (!(fabs(G) < 1e300)) notfinite = 1;
            s_scale = fmax(s_scale, fmax(fabs(w.hx[i]), fmax(fabs(w.g[i]), fabs(aty))));
            if (!w.pin[i]) s_stat = fmax(s_stat, fabs(G));
            else { mul[i] = -G; s_mult = fmax(s_mult, fabs(G)); }
        }
        for (int r = n + lane; r < m; r += 32) if (w.code[r]) s_mult = fmax(s_mult, fabs(mul[r]));
        s_stat = wmax(s_stat); s_scale = wmax(s_scale); s_mult = wmax(s_mult);
        __syncwarp();
        const double scale = fmax(1.0, s_scale);
        const double stol = tol * fmax(scale, s_mult);
        // ---- pass 2: per-row verdicts and the refined active set ----
        int bad = (s_stat <= 1e-10 * scale) ? 0 : 1, anywrong = 0;
        const int nonfinite = __any_sync(kFullMask, notfinite) || !(s_stat == s_stat) || !(s_mult == s_mult);
        for (int r = lane; r < m; r += 32) {
            const bool apriori = (r < n) && w.fixed[r];
            const int cd = w.code[r];
            int change = 0;
            if (!apriori) {
                const double ax = A.row(r, w.xp), lo = wrow_lo(c, w, r), hi = wrow_hi(c, w, r);
                if (cd != 0) {
                    const double lam = mul[r];
                    const double bnd = cd < 0 ? lo : hi;
                    if ((cd > 0 && lam < -stol) || (cd < 0 && lam > stol)) { change = 1; bad |= 1; anywrong = 1; }
                    if (r >= n && fabs(ax - bnd) > tol * (1.0 + fabs(bnd))) bad |= 1;   // singular / inconsistent set
                } else {
                    if (lo - ax > tol * (1.0 + fabs(lo))) { change = 2; bad |= 1; }
                    else if (ax - hi > tol * (1.0 + fabs(hi))) { change = 3; bad |= 1; }
                }
            }
            w.side[r] = (int8_t)change;
        }
        bad = __any_sync(kFullMask, bad);
        anywrong = __any_sync(kFullMask, anywrong);
        __syncwarp();
        if (nonfinite) return -1;
        if (!bad) {
            for (int r = n + lane; r < m; r += 32) if (!w.code[r]) mul[r] = 0.0;
            __syncwarp();
            return 1;
        }
        int changed = 0;
        for (int r = lane; r < m; r += 32) {
            const int change = w.side[r];
            if (change == 1) { w.code[r] = 0; changed = 1; }
            else if (change >= 2 && !anywrong) { w.code[r] = (int8_t)(change == 2 ? -1 : 1); changed = 1; }
        }
        changed = __any_sync(kFullMask, changed);
        __syncwarp();
        if (!changed) HMPC_EMUL_COUNT(7);
        return changed ? 0 : -1;
    }
}
// Verified primal-dual active-set refinement, all trials (free-running form).
template <int SLOTS>
__device__ inline int wpolish(const QpConst& c, WWork& w, const AOp& A, int kcap, WInfo& info, int lane) {
    wpolish_init(c, w, lane);
    for (int trial = 0; trial <= c.retries; ++trial) {
        const int r = wtrial<SLOTS>(c, w, A, kcap, info, lane);
        if (r != 0) return r > 0;
    }
    return 0;
}

// ------------------------------------------------------------------------------------------------
// One warm tick of hopper b by one warp.  Returns 1 when the hopper is done (outputs and handle state written),
// 0 when it has to take the CTA kernel (nothing written).
// ------------------------------------------------------------------------------------------------
// wprep (prep kernel): load, time shift, linearise, condense hopper b and leave its QP record in HBM.
__device__ inline void wprep(const QpConst& c, WWork& w, double* rec, int32_t* flag, int b, int B, const MpcIo& io, int lane) {
    const int N = c.N, n = 6 * N;
    if (!io.valid[b]) { if (lane == 0) *flag = PREP_INVALID; return; }
    w.Hc = rec;
    const int infeasible = wcondense(c, w, b, B, io, lane);
    double* rg = rec + prep_hstride(N);
    double* rh = rg + ((n + 7) & ~7);
    double* rx = rh + ((N + 7) & ~7);
    for (int i = lane; i < n; i += 32) rg[i] = w.g[i];
    for (int k = lane; k < N; k += 32) rh[k] = w.hlo[k];
    if (lane < 12) rx[lane] = w.xin[lane];
    if (lane == 0) *flag = infeasible ? PREP_INFEASIBLE : PREP_OK;
}
// wfetch (solve kernel): take hopper b's record, rebuild the index sets, warm start; mu = the hopper's friction
// coefficient.  Returns 0 when the hopper must take the CTA kernel (no valid previous tick / infeasible height row).
__device__ inline int wfetch(const QpConst& c, WWork& w, double& mu, double* rec, const int32_t* flag, int b, int B, const MpcIo& io,
                             int lane) {
    const int N = c.N, n = 6 * N, m = 11 * N;
    const size_t Bs = (size_t)B;
    // Every global load of the fetch is issued here, back to back, into registers (n <= 64: two entries per lane,
    // m <= 128: four): ONE HBM round trip instead of five dependent ones.  In the lock-step kernel the fetch of one
    // warp is on the critical path of its whole group's round.
    const double* rg = rec + prep_hstride(N);
    const double* rh = rg + ((n + 7) & ~7);
    const double* rx = rh + ((N + 7) & ~7);
    const int f = *flag;
    const uint64_t bits = io.Cbits[b];
    const double mub = c.body ? c.body[Bs + b] : c.mu;     // model_body's mu, without the rest of the body
    double gq[2] = {0.0, 0.0}, uq[2] = {0.0, 0.0}, uw[2] = {0.0, 0.0};
    int8_t cq[4] = {0, 0, 0, 0}, cw[4] = {0, 0, 0, 0};
    // Warm start: stage k starts from the previous tick's stage k+1, the last two stages keep their own previous
    // pattern (mpc_hopper in hmpc_mpc.cuh).  A hopper this kernel finished last tick left exactly that, contiguous, in
    // its warm block (wfinish); otherwise it is gathered from the strided state the CTA kernel wrote.  The hoppers come
    // in contact-schedule order, so a strided read costs a 32-byte sector per element: the block is the common case.
    const bool blk = io.warm_ok != nullptr;
    const int fresh = blk ? (int)io.warm_ok[b] : 0;
    const double* wb = blk ? io.warm + (size_t)b * io.warm_stride : nullptr;
    const int8_t* wc = blk ? reinterpret_cast<const int8_t*>(wb + ((n + 7) & ~7)) : nullptr;
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        const int i = lane + 32 * q;
        if (i < n) {
            gq[q] = rg[i];
            if (blk) uw[q] = wb[i];
        }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int r = lane + 32 * q;
        if (r < m && blk) cw[q] = wc[r];
    }
    if (!fresh) {
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int i = lane + 32 * q;
            if (i < n) uq[q] = io.Usol[(size_t)((i / 6 < N - 2) ? i + 6 : i) * Bs + b];
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int r = lane + 32 * q;
            if (r < m) {
                int src;
                if (r < n) src = (r / 6 < N - 2) ? r + 6 : r;
                else if (r < n + 4 * N) src = ((r - n) / 4 < N - 2) ? r + 4 : r;
                else src = (r - n - 4 * N < N - 2) ? r + 1 : r;
                cq[q] = io.code[(size_t)src * Bs + b];
            }
        }
    } else {
#pragma unroll
        for (int q = 0; q < 2; ++q) uq[q] = uw[q];
#pragma unroll
        for (int q = 0; q < 4; ++q) cq[q] = cw[q];
    }
    const double hl = lane < N ? rh[lane] : 0.0;            // N <= kWarpMaxN < 32
    const double xi = lane < 12 ? rx[lane] : 0.0;
    if (f == PREP_INVALID) { HMPC_EMUL_COUNT(4); return 0; }
    if (f == PREP_INFEASIBLE) { HMPC_EMUL_COUNT(5); return 0; }
    mu = mub;
    w.Hc = rec;
    wload_sets(c, w, bits, lane);
#ifndef HMPC_HOST_EMUL
    // the record was written by another kernel long ago: pull the Hessian into L2 while the rest is set up
    for (int o = 16 * lane; o < w.nf * w.ld; o += 16 * 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(rec + o));
#endif
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        const int i = lane + 32 * q;
        if (i < n) { w.g[i] = gq[q]; w.xp[i] = uq[q]; }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int r = lane + 32 * q;
        if (r < m) w.code[r] = cq[q];
    }
    if (lane < N) w.hlo[lane] = hl;
    if (lane < 12) w.xin[lane] = xi;
    __syncwarp();
    wpolish_init(c, w, lane);
    return 1;
}
// wfinish: roll the verified solution out, store outputs and the handle state of hopper b.
__device__ inline void wfinish(const QpConst& c, WWork& w, int b, int B, const MpcIo& io, const WInfo& info, int lane,
                            int st = ST_SOLVED, int path = PATH_WARM, int iters = 0) {
    const int N = c.N, n = 6 * N, m = 11 * N;
    const size_t Bs = (size_t)B;
    // ---- roll the solution out (mpc_cvx_euler_3f.py:133,140 dynamics rows) and store ----
    double* xs = w.err;
    const double* u = w.xp;
    const double dt = c.dt, gdt = -c.g * dt;
    const Body bd = model_body(c, b, B);
    wlinearize_all(c, bd, w, b, B, io, lane);   // the factor overwrote cz / sz / Bw
    __syncwarp();
    if (lane < 12) xs[lane] = w.xin[lane];
    if (lane < 6) {          // velocities
        const int q = lane;
        double acc = w.xin[6 + q];
        for (int k = 0; k < N; ++k) {
            const double* uk = u + 6 * k;
            if (q < 3) {
                // row q of dt B[6:9, 0:3]: 3f  dt/m e_q,  2f  dt/m Rz^T (same products as rollout_solution)
                const double sm = (1.0 / bd.m) * c.dt;
                if (c.dyn == 3) acc += sm * uk[q];
                else {
                    const double cs = w.cz[k], sn = w.sz[k];
                    if (q == 0) acc += ((cs / bd.m) * c.dt) * uk[0] + ((-sn / bd.m) * c.dt) * uk[1];
                    else if (q == 1) acc += ((sn / bd.m) * c.dt) * uk[0] + ((cs / bd.m) * c.dt) * uk[1];
                    else acc += sm * uk[2];
                }
                if (q == 2) acc += gdt;
            } else {
                const double* Bw = w.Bw + 18 * k + 6 * (q - 3);
                acc += Bw[0] * uk[0] + Bw[1] * uk[1] + Bw[2] * uk[2] + Bw[3] * uk[3] + Bw[4] * uk[4] + Bw[5] * uk[5];
            }
            xs[12 * (k + 1) + 6 + q] = acc;
        }
    }
    __syncwarp();
    if (lane < 6) {          // positions / Euler angles integrate the stage-k velocities
        const int q = lane;
        double acc = w.xin[q];
        for (int k = 0; k < N; ++k) {
            const double* xk = xs + 12 * k;
            if (q < 3) acc += dt * xk[6 + q];
            else {
                const double cs = w.cz[k], sn = w.sz[k];
                const double wx = xk[9], wy = xk[10], wz = xk[11];
                const double r = (q == 3) ? (cs * wx + sn * wy) : (q == 4) ? (-sn * wx + cs * wy) : wz;
                acc += dt * r;
            }
            xs[12 * (k + 1) + q] = acc;
        }
    }
    __syncwarp();
    for (int i = lane; i < (N + 1) * 12; i += 32) {
        io.Xsol[(size_t)i * Bs + b] = xs[i];
        if (io.X_out) io.X_out[(size_t)i * Bs + b] = xs[i];
    }
    for (int i = lane; i < n; i += 32) {
        io.Usol[(size_t)i * Bs + b] = u[i];
        if (io.U_out) io.U_out[(size_t)i * Bs + b] = u[i];
    }
    for (int r = lane; r < m; r += 32) io.code[(size_t)r * Bs + b] = w.code[r];
    if (io.warm_ok) {        // the next tick's warm start, shifted (see wfetch), contiguous: full-sector writes and reads
        double* wb = io.warm + (size_t)b * io.warm_stride;
        int8_t* wc = reinterpret_cast<int8_t*>(wb + ((n + 7) & ~7));
        for (int i = lane; i < n; i += 32) wb[i] = u[(i / 6 < N - 2) ? i + 6 : i];
        for (int r = lane; r < m; r += 32) {
            int src;
            if (r < n) src = (r / 6 < N - 2) ? r + 6 : r;
            else if (r < n + 4 * N) src = ((r - n) / 4 < N - 2) ? r + 4 : r;
            else src = (r - n - 4 * N < N - 2) ? r + 1 : r;
            wc[r] = w.code[src];
        }
    }
    if (io.U0_out && lane < 6) io.U0_out[(size_t)lane * Bs + b] = u[lane];
    if (lane == 0) {
        io.valid[b] = (st == ST_SOLVED || st == ST_INEXACT) ? 1 : 0;
        if (io.warm_ok) io.warm_ok[b] = 1;
        if (io.flops) io.flops[b] = (io.accumulate ? io.flops[b] : 0.0) + info.flops;
        io.st_tick[b] = st;
        io.path[b] = path;
        if (io.accumulate) {
            if (st != ST_SOLVED && io.status[b] == 0) io.status[b] = st;
            io.iters[b] += iters;
            io.nfac[b] += info.nfac;
        } else {
            io.status[b] = st;
            io.iters[b] = iters;
            io.nfac[b] = info.nfac;
            io.ninf[b] = 0;
        }
    }
}
// Returns 1: done;  0: not attempted (no valid previous tick / infeasible height row / system larger than kcap): the
// CTA kernel runs its whole solver;  -1: the active-set refinement itself gave up: the CTA kernel goes straight to
// its interior point (same QP, same verified polish afterwards).  No kernel calls it: it is the serial statement of
// the lock-step kernel's per-hopper loop, which the test emulation (tests/emul, tests/emul_body) runs.
constexpr int kDeferWarmFailed = 1 << 30;     // flag bit in a deferral-list entry
template <int SLOTS>
__device__ inline int mpc_hopper_warp(const QpConst& c, WWork& w, double* rec, const int32_t* flag, int kcap, int b, int B, const MpcIo& io, int lane) {
    double mu;
    if (!wfetch(c, w, mu, rec, flag, b, B, io, lane)) return 0;
    AOp A{c.N, 6 * c.N, c.dyn == 3 ? 1 : 0, mu, w.stance, w.hinv};
    WInfo info{0, c.condense_flops};
    for (int trial = 0; trial <= c.retries; ++trial) {
        const int r = wtrial<SLOTS>(c, w, A, kcap, info, lane);
        if (r == -2) return 0;
        if (r < 0) return -1;
        if (r > 0) { wfinish(c, w, b, B, io, info, lane); return 1; }
    }
    return -1;
}

// ------------------------------------------------------------------------------------------------
// OSQP-style ADMM for one warp (north_star K2; the CTA statement is admm_solve in hmpc_qp.cuh, the numpy statement
// oracle/device_port.py admm_solve -- same iteration, same check cadence, same rho rule):
//     x~ = K^-1 (sigma x - g + A'(rho z - y)),  K = H + sigma I + A' diag(rho) A   over the non-fixed variables
//     x+ = alpha x~ + (1-alpha) x ;  z+ = clip(alpha A x~ + (1-alpha) z + y/rho) ;  y+ = y + rho (.. - z+)
// K is factorised once (and again when rho moves by more than 5x) as tensor-core tiles in the warp's shared-memory
// slice (wfactor with the weights of the ADMM operator), every iteration is one tiled substitution (wsolve) plus
// vector work over the m rows; the residuals of OSQP's termination test and the rho update are warp-shuffle
// reductions.  On entry w.xp = warm start (or zeros); on exit w.xp = x, y = multipliers, w.code = OSQP's polish guess
// of the active set.  Returns ST_INEXACT (residual test met), ST_MAX_ITER, ST_NON_FINITE, or -2 when the system
// does not fit the factor storage.  wv and xt live on w.mul and w.hx (both dead while the iteration runs).
// ------------------------------------------------------------------------------------------------
__device__ inline int wadmm(const QpConst& c, WWork& w, const AOp& A, int kcap, WInfo& info, int& iters, double* z, double* y,
                            double* rv, int lane) {
    const int N = c.N, n = 6 * N, m = 11 * N;
    const int nF = w.nf;
    iters = 0;
    if (nF > kcap) return -2;
    double *x = w.xp, *xt = w.hx, *wv = w.mul;
    double rho = c.rho0;
    const double sigma = c.sigma, alpha = c.alpha;
    auto set_rho = [&](double r) {
        for (int i = lane; i < m; i += 32) {
            const double lo = wrow_lo(c, w, i), hi = wrow_hi(c, w, i);
            double v = r;
            if (lo < -kInfThresh && hi > kInfThresh) v = kRhoMin;
            else if (hi - lo < 1e-4) v = fmin(1e3 * r, kRhoMax);
            rv[i] = v;
        }
        __syncwarp();
    };
    set_rho(rho);
    for (int i = lane; i < nF; i += 32) w.idx[i] = (uint8_t)i;       // the system holds every non-fixed variable
    for (int i = lane; i < n; i += 32) {
        const double v = w.fixed[i] ? 0.0 : x[i];
        x[i] = fmin(fmax(v, wbox_lo(w, i)), wbox_hi(w, i));
        xt[i] = 0.0;
    }
    __syncwarp();
    for (int r = lane; r < m; r += 32) { z[r] = A.row(r, x); y[r] = 0.0; }   // OSQP: z = A x at the start, y = 0
    __syncwarp();
    w.wts = rv; w.dadd = sigma;
    ++info.nfac;
    info.flops += flops_factor(nF);
    int st = ST_MAX_ITER;
    if (wfactor<true>(c, w, A, nF, 0, 0.0, lane)) { w.wts = nullptr; return ST_NON_FINITE; }
    const int last_it = c.max_iter;
    int next_check = (c.mode == 1) ? last_it : min(c.first_check, last_it);
    for (int it = 1; it <= last_it; ++it) {
        for (int r = lane; r < m; r += 32) wv[r] = rv[r] * z[r] - y[r];
        __syncwarp();
        for (int i = lane; i < nF; i += 32) { const int vi = w.fr[i]; w.rhs[i] = sigma * x[vi] - w.g[vi] + A.colT(vi, wv); }
        __syncwarp();
        wsolve(w, nF, 0, lane);
        info.flops += flops_solve(nF);
        for (int i = lane; i < nF; i += 32) xt[w.fr[i]] = w.rhs[i];        // fixed entries of xt stay 0
        __syncwarp();
        for (int r = lane; r < m; r += 32) {
            const double zt = A.row(r, xt);
            const double zr = alpha * zt + (1.0 - alpha) * z[r];
            const double rr = rv[r];
            const double zn = fmin(fmax(zr + y[r] / rr, wrow_lo(c, w, r)), wrow_hi(c, w, r));
            y[r] += rr * (zr - zn);
            z[r] = zn;
        }
        for (int i = lane; i < n; i += 32) x[i] = alpha * xt[i] + (1.0 - alpha) * x[i];
        __syncwarp();
        iters = it;
        if (it != next_check && it != last_it) continue;
        next_check = it + c.check;
        // ---- residuals of the unscaled problem (OSQP termination test, SURVEY App. C2) ----
        wmatvec(w, lane);                                  // hx = H x (overwrites xt, recomputed next iteration)
        info.flops += flops_matvec(n);
        double v0 = 0, v1 = 0, v2 = 0, v3 = 0, v4 = 0, v5 = 0;   // pri, npri, dua, |Hx|, |A'y|, |g|
        for (int r = lane; r < m; r += 32) {
            const double ax = A.row(r, x);
            v0 = fmax(v0, fabs(ax - z[r]));
            v1 = fmax(v1, fmax(fabs(ax), fabs(z[r])));
        }
        int notfinite = 0;
        for (int i = lane; i < n; i += 32) {
            if (w.fixed[i]) continue;                      // eliminated variables carry an implicit multiplier
            const double aty = A.colT(i, y);
            const double G = w.hx[i] + w.g[i] + aty;
            if (!(fabs(G) < 1e300)) notfinite = 1;
            v2 = fmax(v2, fabs(G));
            v3 = fmax(v3, fabs(w.hx[i]));
            v4 = fmax(v4, fabs(aty));
            v5 = fmax(v5, fabs(w.g[i]));
        }
        v0 = wmax(v0); v1 = wmax(v1); v2 = wmax(v2); v3 = wmax(v3); v4 = wmax(v4); v5 = wmax(v5);
        notfinite = __any_sync(kFullMask, notfinite);
        __syncwarp();
        for (int i = lane; i < n; i += 32) xt[i] = 0.0;    // hx held H x: fixed entries of xt must read 0 again
        __syncwarp();
        const double pri = v0, npri = v1, dua = v2, ndua = fmax(v3, fmax(v4, v5));
        if (notfinite || !(pri == pri) || !(dua == dua)) { st = ST_NON_FINITE; break; }
        if (c.mode == 1) break;
        if (pri <= c.eps_abs + c.eps_rel * npri && dua <= c.eps_abs + c.eps_rel * ndua) { st = ST_INEXACT; break; }
        if (it == last_it) break;
        if (c.adaptive_rho) {
            double rn = rho * sqrt((pri / fmax(npri, 1e-10)) / fmax(dua / fmax(ndua, 1e-10), 1e-10));
            rn = fmin(fmax(rn, kRhoMin), kRhoMax);
            if (rn > 5.0 * rho || rn < 0.2 * rho) {
                rho = rn;
                set_rho(rho);
                ++info.nfac;
                info.flops += flops_factor(nF);
                if (wfactor<true>(c, w, A, nF, 0, 0.0, lane)) { st = ST_NON_FINITE; break; }
            }
        }
    }
    w.wts = nullptr; w.dadd = 0.0;
    for (int r = lane; r < m; r += 32) {
        const double zz = z[r], yy = y[r];
        w.code[r] = (int8_t)(((zz - wrow_lo(c, w, r)) < -yy) ? -1 : (((wrow_hi(c, w, r) - zz) < yy) ? 1 : 0));
    }
    __syncwarp();
    return st;
}

// One warm ADMM tick of hopper b by one warp: record -> ADMM -> (polish) -> roll-out.  Returns 1 when the hopper is
// done, 0 when it has to take the CTA kernel (no valid previous tick, infeasible height row, system too large,
// non-finite iterate).  extra: the warp's z / y / rho vectors (warp_admm_doubles).
template <int SLOTS>
__device__ inline int mpc_hopper_warp_admm(const QpConst& c, WWork& w, double* extra, double* rec, const int32_t* flag, int kcap,
                                           int b, int B, const MpcIo& io, int lane) {
    const int N = c.N, n = 6 * N, m = 11 * N;
    double mu;
    if (!wfetch(c, w, mu, rec, flag, b, B, io, lane)) return 0;
    AOp A{N, n, c.dyn == 3 ? 1 : 0, mu, w.stance, w.hinv};
    WInfo info{0, c.condense_flops};
    double *z = extra, *y = extra + m, *rv = extra + 2 * m;
    int iters = 0;
    int st = wadmm(c, w, A, kcap, info, iters, z, y, rv, lane);
    if (st < 0 || st == ST_NON_FINITE) return 0;
    if (c.polish) {
        // OSQP's polish=True: the verified active-set refinement from ADMM's guess; the iterate is kept in z (dead now)
        for (int i = lane; i < n; i += 32) z[i] = w.xp[i];
        __syncwarp();
        wpolish_init(c, w, lane);
        int ok = 0;
        for (int trial = 0; trial <= c.retries; ++trial) {
            const int r = wtrial<SLOTS>(c, w, A, kcap, info, lane);
            if (r > 0) ok = 1;
            if (r != 0) break;
        }
        if (ok) st = ST_SOLVED;
        else {
            for (int i = lane; i < n; i += 32) w.xp[i] = z[i];
            __syncwarp();
        }
    }
    wfinish(c, w, b, B, io, info, lane, st, PATH_ADMM, iters);
    return 1;
}

// ------------------------------------------------------------------------------------------------
// Host-side dispatch rules, shared by the library (hmpc_api.cu) and the test emulation (tests/emul).
// ------------------------------------------------------------------------------------------------
constexpr int kWarpMaxN = 10;     // horizons the warp kernel is instantiated for (n = 6N <= 64: two rows per lane)
// cap on the order of the compact KKT system (unpinned variables + active friction / height rows): it sizes the
// factor in shared memory; a trial that needs more goes to the CTA kernel
inline int warp_kcap(const hmpc_config& cfg) {
    int k = kWarpKcap;                 // 7 tiles of 8 (variables padded to a multiple of 8, then the active rows)
    if (const char* e = getenv("HMPC_WARP_KCAP")) { const int v = atoi(e); if (v >= 8 && v <= kWarpKcap) k = v; }
    (void)cfg;
    return k;
}
inline bool warp_path_applies(const hmpc_config& cfg, int init) {
    return cfg.hot_path == HMPC_HOT_AUTO && !init && cfg.warm_start &&
           (cfg.solver == HMPC_SOLVER_EXACT || cfg.solver == HMPC_SOLVER_ADMM) &&
           cfg.precision == HMPC_FP64 && cfg.sqp_sweeps <= 1 && cfg.N >= 3 && cfg.N <= kWarpMaxN;
}

#ifndef HMPC_HOST_EMUL
// ------------------------------------------------------------------------------------------------
// Prep kernel: one warp per hopper, plain grid.  Small per-warp slice and no factor: many warps per SM hide the HBM
// latency of the loads and the dependent arithmetic of the condensing.  hs: the hoppers to condense (the overlapped
// rollout condenses the previous tick's deferred hoppers from their list on the side stream, the rest here).
// ------------------------------------------------------------------------------------------------
template <int WPC>
__global__ void __launch_bounds__(32 * WPC, 4)
mpc_prep_kernel(QpConst c, int B, int wdoubles, double* __restrict__ prep, size_t pstride, int32_t* __restrict__ flags, HopperSet hs,
                MpcIo io) {
    extern __shared__ double smem[];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int ticket = blockIdx.x * WPC + wid;
    int b;
    if (hs.list) {
        if (ticket >= *hs.list_cnt) return;
        b = hs.list[ticket] & kListHopperMask;
    } else {
        if (ticket >= B) return;
        b = work_item(c, ticket, B);
        if (hs.mark && hs.mark[b] == hs.skip) return;
    }
    WWork w;
    wcarve(w, smem + (size_t)wid * wdoubles, c.N, kPrepKcap);
    wprep(c, w, prep + (size_t)b * pstride, flags + b, b, B, io, lane);
}

// ADMM mode (hmpc_config.solver = HMPC_SOLVER_ADMM): WPC free-running warps per CTA, one hopper each, hoppers handed
// out one at a time from a ticket counter, the ones it cannot finish appended to a deferral list.  The iteration
// count differs from hopper to hopper by design (early exit), so there is nothing to run in lock-step.
template <int WPC>
__global__ void __launch_bounds__(32 * WPC, 1)
mpc_warp_admm_kernel(QpConst c, int B, int kcap, int wdoubles, double* __restrict__ prep, size_t pstride,
                     const int32_t* __restrict__ flags, int* __restrict__ work_ctr, int* __restrict__ defer_list,
                     int* __restrict__ defer_cnt, MpcIo io) {
    extern __shared__ double smem[];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    WWork w;
    double* slice = smem + (size_t)wid * wdoubles;
    wcarve(w, slice, c.N, kcap);
    double* extra = slice + warp_work_doubles(c.N, kcap);
    for (;;) {
        int b = 0;
        if (lane == 0) b = atomicAdd(work_ctr, 1);
        b = __shfl_sync(kFullMask, b, 0);
        if (b >= B) break;
        b = work_item(c, b, B);
        const int done = mpc_hopper_warp_admm<2>(c, w, extra, prep + (size_t)b * pstride, flags + b, kcap, b, B, io, lane);
        __syncwarp();
        if (!done && lane == 0) defer_list[atomicAdd(defer_cnt, 1)] = b;
    }
}

// Exact solver, lock-step form: the WPC warps of a CTA still own one hopper each, but start every active-set trial
// together (one CTA barrier per round), so that the warps sharing an SM execute the same code at the same time and
// share its instruction fetches.  A warp whose hopper is finished stores it and fetches the next record; since the
// condensing moved to the prep kernel a round is one trial for every warp.
// AND-reduction of pred over the `nthreads` threads that use named barrier `id` (a lock-step group of warps)
__device__ __forceinline__ bool group_all(int id, int nthreads, bool pred) {
    int r;
    asm volatile("{\n\t.reg .pred p, q;\n\tsetp.ne.s32 q, %3, 0;\n\tbar.red.and.pred p, %1, %2, q;\n\tselp.s32 %0, 1, 0, p;\n\t}"
                 : "=r"(r) : "r"(id), "r"(nthreads), "r"((int)pred) : "memory");
    return r != 0;
}
template <int SLOTS, int WPC, int MIN_CTAS>
__global__ void __launch_bounds__(32 * WPC, MIN_CTAS)
mpc_warp_rounds_kernel(QpConst c, int B, int kcap, int wdoubles, double* __restrict__ prep, size_t pstride,
                       const int32_t* __restrict__ flags, int* __restrict__ work_ctr, int* __restrict__ defer_list,
                       int* __restrict__ defer_cnt, int gw, MpcIo io) {
    extern __shared__ double smem[];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    // lock-step groups of gw warps, each on its own named barrier (the last group takes what is left of the CTA)
    const int nsync = gw >> 8;         // re-alignment barriers inside a trial (0, 1: after the factorisation, 2: + after the refinement)
    gw &= 255;
    const int grp = wid / gw, bar_id = 1 + grp;
    const int bar_threads = 32 * ((grp + 1) * gw <= WPC ? gw : WPC - grp * gw);
    WWork w;
    wcarve(w, smem + (size_t)wid * wdoubles, c.N, kcap);
    AOp A{c.N, 6 * c.N, c.dyn == 3 ? 1 : 0, c.mu, w.stance, w.hinv};
    bool have = false, exhausted = false;
    int b = 0, trial = 0;
    WInfo info{0, 0.0};
    for (;;) {
        while (!have && !exhausted) {
            if (lane == 0) b = atomicAdd(work_ctr, 1);
            b = __shfl_sync(kFullMask, b, 0);
            if (b >= B) { exhausted = true; break; }
            b = work_item(c, b, B);
            double mu;
            if (wfetch(c, w, mu, prep + (size_t)b * pstride, flags + b, b, B, io, lane)) { have = true; trial = 0; info.nfac = 0; info.flops = c.condense_flops; A.mu = mu; }
            else if (lane == 0) defer_list[atomicAdd(defer_cnt, 1)] = b;
        }
        if (group_all(bar_id, bar_threads, !have)) break;
        auto mid = [&](int p) { if (p < nsync) group_all(bar_id, bar_threads, true); };
        if (!have) { mid(0); mid(1); }
        if (have) {
            const int r = wtrial<SLOTS>(c, w, A, kcap, info, lane, mid);
            if (r > 0) { wfinish(c, w, b, B, io, info, lane); have = false; }
            else if (r < 0 || ++trial > c.retries) {
                if (lane == 0) defer_list[atomicAdd(defer_cnt, 1)] = b | (r == -2 ? 0 : kDeferWarmFailed);
                have = false;
            }
            __syncwarp();
        }
    }
}
#endif  // HMPC_HOST_EMUL

}  // namespace hmpc
