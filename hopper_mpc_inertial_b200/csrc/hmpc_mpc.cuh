// hmpc_mpc.cuh -- one hopper's mpcontrol (mpc_cvx_euler_3f.py:41-69) as a device function: load, time
// shift / initial guess, linearise + condense, solve, roll the solution out, store.  Called by the
// persistent mpc_kernel (hmpc_api.cu) with the CTA's shared-memory Work.
#pragma once
#include "hmpc_qp.cuh"
#include "../../include/hmpc.h"

namespace hmpc {

// ------------------------------------------------------------------------------------------------
// shared set-up of one hopper's Work: carve shared memory, point the matrices
// ------------------------------------------------------------------------------------------------
// SMEM_MATS is a compile-time switch so that, in the shared-memory configuration, every access to H and to
// the factor is provably a shared-memory access (LDS/STS instead of generic loads).
template <bool SMEM_MATS>
__device__ inline void setup_work(Work& w, const QpConst& c, double* smem, double* ws, int fsize = 8) {
    const size_t n = 6 * (size_t)c.N;
    double* mat;
    if (SMEM_MATS) {
        carve(w, smem, c.N);
        mat = smem + ((work_vec_doubles(c.N) + 1) & ~(size_t)1);
    } else {
        // per-CTA workspace slice: matrices, then (long horizons) the interior point's m-vectors
        const size_t md = mat_doubles(c.N, fsize);
        mat = ws + (size_t)blockIdx.x * (md + ws_mv_doubles(c.N));
        carve(w, smem, c.N, mv_in_workspace(c.N) ? mat + md : nullptr);
    }
    w.H = mat; w.Lm = mat + n * (n + 1) / 2;
}

__device__ inline void load_hopper(const QpConst& c, Work& w, int b, int B, const double* x_in,
                                   const double* pf, const uint64_t* Cbits, const double* Qd,
                                   const double* Rd) {
    const int N = c.N, tid = threadIdx.x, T = blockDim.x;
    for (int i = tid; i < 12; i += T) { w.xin[i] = x_in[(size_t)i * B + b]; w.Qd[i] = Qd[(size_t)i * B + b]; }
    for (int i = tid; i < 6; i += T) w.Rd[i] = Rd[(size_t)i * B + b];
    for (int i = tid; i < 3 * N; i += T) w.pfw[i] = pf[(size_t)i * B + b];
    const uint64_t bits = Cbits[b];
    for (int k = tid; k < N; k += T) w.stance[k] = (int8_t)((bits >> k) & 1ull);
}

// linear rollout of the solution (mpc_cvx_euler_3f.py:133,140 dynamics rows): xs [(N+1)][12] in shared
__device__ inline void rollout_solution(const QpConst& c, Work& w, const double* u, double* xs) {
    const int N = c.N, tid = threadIdx.x, T = blockDim.x;
    const double dt = c.dt, gdt = -c.g * dt;
    for (int q = tid; q < 12; q += T) xs[q] = w.xin[q];
    __syncthreads();
    for (int q = tid; q < 6; q += T) {          // velocities: v_{k+1} = v_k + Bv u_k + g dt, w_{k+1} = w_k + Bw u_k
        double acc = w.xin[6 + q];
        for (int k = 0; k < N; ++k) {
            const double* uk = u + 6 * k;
            if (q < 3) {
                const double* Bv = w.Bv + 9 * k + 3 * q;
                acc += Bv[0] * uk[0] + Bv[1] * uk[1] + Bv[2] * uk[2];
                if (q == 2) acc += gdt;
            } else {
                const double* Bw = w.Bw + 18 * k + 6 * (q - 3);
                acc += Bw[0] * uk[0] + Bw[1] * uk[1] + Bw[2] * uk[2] + Bw[3] * uk[3] + Bw[4] * uk[4] + Bw[5] * uk[5];
            }
            xs[12 * (k + 1) + 6 + q] = acc;
        }
    }
    __syncthreads();
    for (int q = tid; q < 6; q += T) {          // positions / Euler angles integrate the stage-k velocities
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
    __syncthreads();
}

struct MpcIo {
    const double *x_in, *x_ref, *pf;
    const uint64_t* Cbits;
    const double *Qd, *Rd;
    double *Xsol, *Usol;          // handle state, in/out
    int8_t *code, *valid;         // handle state, in/out
    double *U_out, *X_out, *U0_out;
    int32_t *status, *iters, *st_tick, *nfac, *path, *ninf;
    double* flops;                // [B] algorithmic FLOPs (may be null)
    // warp kernels only (may be null): the next tick's warm start of every hopper they finish, shifted already and
    // contiguous per hopper -- [B][warm_stride] doubles: inputs [n -> 8] | active set [m bytes -> 8] -- and whether it
    // is the hopper's newest state (1) or the CTA kernel has written Usol / code since (0)
    double* warm = nullptr;
    int8_t* warm_ok = nullptr;
    int warm_stride = 0;
    int init, accumulate, respawn;
};

// One hopper b of a batch of B.  All threads of the CTA call this together.
// WITH_ADMM = false compiles the OSQP-style ADMM branch out (smaller kernel for the default exact solver)
// A.mu must be hopper b's friction coefficient (model_body).  The caller sets it on its own A: a modified by-value copy
// here made the compiler lose the shared-memory address space of A's arrays (generic loads instead of LDS).
template <bool WITH_ADMM, class Sys>
__device__ inline void mpc_hopper(const QpConst& c, Work& w, Sys& sys, const AOp& A, int b, int B, const MpcIo& io,
                                  int skip_warm = 0) {
    const int N = c.N, n = 6 * N, m = 11 * N, tid = threadIdx.x, T = blockDim.x;
    double* xs = w.err;   // reused after condense: solution trajectory [(N+1)][12]
    __syncthreads();
    PH_T0(ph_all);
    load_hopper(c, w, b, B, io.x_in, io.pf, io.Cbits, io.Qd, io.Rd);
    // a hopper without a solved previous tick (first call, or re-initialised after a respawn) takes
    // the reference's init branch: two solves, x_guess[1:] = x_ref (mpc_cvx_euler_3f.py:50-58)
    const int init = io.init || (io.respawn && !io.valid[b]);
    __syncthreads();
    int st = 0, its = 0, nfac = 0, path = 0;
    sys.flops = 0.0;
    // first call: two solves (reference); later ticks: c.sqp_sweeps relinearisation sweeps (reference: 1)
    const int passes = init ? 2 : c.sqp_sweeps;
    for (int pass = 0; pass < passes; ++pass) {
        // linearisation point (mpc_cvx_euler_3f.py:50-62); only p and yaw of rows 0..N-1 matter
        for (int k = tid; k < N; k += T) {
            double* gp = w.gp + 4 * k;
            if (k == 0) { gp[0] = w.xin[0]; gp[1] = w.xin[1]; gp[2] = w.xin[2]; gp[3] = w.xin[5]; }
            else if (init && pass == 0) {
                const size_t o = (size_t)(k - 1) * 12;
                gp[0] = io.x_ref[(o + 0) * B + b]; gp[1] = io.x_ref[(o + 1) * B + b];
                gp[2] = io.x_ref[(o + 2) * B + b]; gp[3] = io.x_ref[(o + 5) * B + b];
            } else if (init || pass > 0) {   // later passes relinearise about the previous pass: x_guess = x.value
                gp[0] = xs[12 * k]; gp[1] = xs[12 * k + 1]; gp[2] = xs[12 * k + 2]; gp[3] = xs[12 * k + 5];
            } else {             // time shift: x_guess[k] = x.value[k+1]
                const size_t o = (size_t)(k + 1) * 12;
                gp[0] = io.Xsol[(o + 0) * B + b]; gp[1] = io.Xsol[(o + 1) * B + b];
                gp[2] = io.Xsol[(o + 2) * B + b]; gp[3] = io.Xsol[(o + 5) * B + b];
            }
        }
        // the footstep window and the gains share storage with solver scratch (carve()): reload after a solve
        if (pass > 0) load_hopper(c, w, b, B, io.x_in, io.pf, io.Cbits, io.Qd, io.Rd);
        __syncthreads();
        PH_ADD(1, ph_all);
        PH_T0(ph_c);
        const int infeasible = condense_hopper(c, w, b, B, io.x_ref + b, (size_t)B);
        PH_ADD(2, ph_c);
        PH_T0(ph_sv);
        sys.flops += c.condense_flops;
        // warm start: second init pass re-uses pass 0's solution as is; later ticks shift the
        // previous tick's solution and active set by one stage (the last two stages are kept)
        int warm = 0;
        if (c.warm_start && !infeasible) {
            if (pass >= 1 && st == 0) {          // same QP horizon, new linearisation: start from the last pass as is
                warm = 1;
                for (int i = tid; i < n; i += T) w.xp[i] = w.x[i];
            } else if (!init && io.valid[b]) {
                warm = 1;
                // stage k starts from the previous tick's stage k+1, except the last two stages, which keep
                // their own previous pattern: the terminal stages (no input cost, 100x state cost) look alike
                // from tick to tick, while the stage before them does not look like the old terminal stage.
                // Measured on closed-loop QPs: 2.9 -> 2.2 factorisations per warm solve.
                for (int i = tid; i < n; i += T) {
                    const int src = (i / 6 < N - 2) ? i + 6 : i;
                    w.xp[i] = io.Usol[(size_t)src * B + b];
                }
                for (int r = tid; r < m; r += T) {
                    int src;
                    if (r < n) src = (r / 6 < N - 2) ? r + 6 : r;
                    else if (r < n + 4 * N) src = ((r - n) / 4 < N - 2) ? r + 4 : r;
                    else src = (r - n - 4 * N < N - 2) ? r + 1 : r;
                    w.code[r] = io.code[(size_t)src * B + b];
                }
            }
        }
        if (!warm || (WITH_ADMM && c.solver == HMPC_SOLVER_ADMM)) {
            for (int i = tid; i < n; i += T) w.x[i] = warm ? w.xp[i] : 0.0;
            for (int r = tid; r < m; r += T) w.mv[2][r] = 0.0;    // ADMM multipliers start at zero
        }
        __syncthreads();
        if (infeasible) {
            st = ST_INFEASIBLE;
            for (int i = tid; i < n; i += T) w.x[i] = 0.0;
            for (int r = tid; r < m; r += T) w.code[r] = 0;
            __syncthreads();
        } else {
            SolveInfo info;
            if (WITH_ADMM && c.solver == HMPC_SOLVER_ADMM) {
                info = admm_solve(c, w, sys, A);
                if (c.polish) {
                    for (int i = tid; i < n; i += T) w.xp[i] = w.x[i];
                    __syncthreads();
                    if (polish_verified(c, w, sys, A, info)) info.status = ST_SOLVED;
                }
            } else {
                // skip_warm: the warp kernel ran this very refinement from this very start and gave up
                info = solve_exact(c, w, sys, A, warm && !skip_warm);
            }
            its += info.iters; nfac += info.nfac; path = info.path;
            if (info.status != 0 && st == 0) st = info.status;
        }
        PH_ADD(3, ph_sv);
        PH_T0(ph_r);
        rollout_solution(c, w, w.x, xs);
        PH_ADD(9, ph_r);
    }
    // outputs
    for (int i = tid; i < (N + 1) * 12; i += T) {
        io.Xsol[(size_t)i * B + b] = xs[i];
        if (io.X_out) io.X_out[(size_t)i * B + b] = xs[i];
    }
    for (int i = tid; i < n; i += T) {
        io.Usol[(size_t)i * B + b] = w.x[i];
        if (io.U_out) io.U_out[(size_t)i * B + b] = w.x[i];
    }
    for (int r = tid; r < m; r += T) io.code[(size_t)r * B + b] = (int8_t)w.code[r];
    if (io.U0_out) for (int i = tid; i < 6; i += T) io.U0_out[(size_t)i * B + b] = w.x[i];
    if (tid == 0) {
        io.valid[b] = (st == ST_SOLVED || st == ST_INEXACT) ? 1 : 0;
        if (io.warm_ok) io.warm_ok[b] = 0;        // Usol / code above are this hopper's newest state, not its warm block
        if (io.flops) io.flops[b] = (io.accumulate ? io.flops[b] : 0.0) + sys.flops;
        io.st_tick[b] = st;
        io.path[b] = path;
        if (io.accumulate) {
            if (io.status[b] == 0) io.status[b] = st;
            io.iters[b] += its;
            io.nfac[b] += nfac;
            io.ninf[b] += (st == ST_INFEASIBLE);
        } else {
            io.status[b] = st;
            io.iters[b] = its;
            io.nfac[b] = nfac;
            io.ninf[b] = (st == ST_INFEASIBLE);
        }
    }
    PH_ADD(0, ph_all);
}

}  // namespace hmpc
