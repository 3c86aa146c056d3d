// hmpc_qp.cuh -- per-hopper MPC QP on the device: linearise, condense, solve.
//
// One CTA owns one hopper's QP.  Every vector lives in shared memory; the condensed Hessian H and the
// triangular factor of the current KKT operator live in shared memory when they fit (N <= 10 at FP64),
// else in a per-CTA slice of a global workspace that stays L2-resident (persistent grid).
//
// What is computed (reference file:line into the reference's src/):
//   linearise   gen_dt_dynamics          mpc_cvx_euler_3f.py:71-94 / mpc_cvx_euler_2f.py:70-94
//   condense    build_qp                 mpc_cvx_euler_3f.py:96-153 / 2f:96-151  (SURVEY App. A)
//   solve       cp.Problem(...).solve(solver=cp.OSQP)   mpc_cvx_euler_3f.py:155-160
//
// Condensed form (inputs only, n = 6N):  X = c + S U,  H = 2(S'QS + R),  g = 2(S'Q(c - xref) - R ubar).
// Because A_k A_j = 0 (SURVEY App. A) S has closed-form blocks
//     p-rows  dt (i-a-1) Bv_a     theta-rows  dt W_{a+1,i} Bw_a     v-rows  Bv_a     w-rows  Bw_a
// with W_{a+1,i} = sum_{l=a+1}^{i-1} Rz_l, so H is assembled block-by-block without forming S.
// Constraint rows use a fixed slot layout (m = 11N):  [6N identity box | 4N friction | N height].
// Height row k (k >= 2) is stored NORMALISED by its largest coefficient dt^2 (k-1)/m:
//     sum_{j<=k-2} (k-j-1)/(k-1) fz_j  >=  (z_min - c_z[k]) m / (dt^2 (k-1)).
//
// Solvers (oracle/device_port.py is the numpy statement of the same algorithms):
//   solve_exact   warm-started verified primal-dual active-set refinement; Mehrotra interior point as
//                 the cold start / fallback; every accepted point passes the KKT test of the ORIGINAL QP
//   admm_solve    OSQP iteration (SURVEY App. C2) in the dense condensed form, fixed-iteration or
//                 early-exit, residual-balancing rho adaptation
// Linear algebra: one LDL' factorisation  K = L' D L'^T  of the compacted operator -- the positive definite
// H + A'WA  (IPM, ADMM) or the quasi-definite  [[H_FF, G'],[G, -E]]  (polish; negative pivots for the rows),
// in FP64 or, in the mixed-precision mode, in FP32 (struct LinSys).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "hmpc_sim.cuh"   // mat3_vec / mat3T_vec
#include "hmpc_tile.cuh"  // FP64 tensor-core tile primitives

namespace hmpc {


// ---- optional phase timers (debug builds only: -DHMPC_PHASE_TIMING; see tools/phase_timing.py) ----
#ifdef HMPC_PHASE_TIMING
static __device__ unsigned long long g_phase[16];
#define PH_T0(v) const long long v = clock64()
#define PH_ADD(id, v) do { if (threadIdx.x == 0) atomicAdd(&g_phase[id], (unsigned long long)(clock64() - (v))); } while (0)
#else
#define PH_T0(v) do {} while (0)
#define PH_ADD(id, v) do {} while (0)
#endif
constexpr double kInf = 1e30;
constexpr double kInfThresh = 1e26;   // OSQP: OSQP_INFTY * MIN_SCALING
constexpr double kRhoMin = 1e-6, kRhoMax = 1e6;
constexpr int kNumMVec = 11;          // m-sized scratch vectors shared by the solvers

enum { ST_SOLVED = 0, ST_MAX_ITER = 1, ST_INFEASIBLE = 2, ST_NON_FINITE = 3, ST_INEXACT = 4 };
enum { PATH_NONE = 0, PATH_WARM = 1, PATH_IPM_POLISH = 2, PATH_IPM = 3, PATH_ADMM = 4 };

struct QpConst {
    int N, dyn, uref_mode, solver, mode, max_iter, check, first_check, retries, adaptive_rho, warm_start;
    int ipm_max_iter, polish, max_refine, sqp_sweeps;
    double dt, m, g, mu;
    double Jinv[9], rh[3], tau_max[3];
    double fz_max, z_min, kf;
    double eps_abs, eps_rel, rho0, sigma, alpha, kkt_eps, polish_tol, ipm_tol;
    double condense_flops;   // flops_condense(N), precomputed on the host
    double stagnation;       // refinement stops when the residual shrinks by less than this factor
    // order in which the persistent kernels take the hoppers: ticket i -> hopper (i * work_mul + work_add) mod B
    // (1, 0 = in order).  Results never depend on it; the stress test permutes it (HMPC_WORK_PERM, tests/test_gpu.py).
    int work_mul, work_add;
    // optional second stage of that map (lock-step solve kernel only): a permutation of the hoppers that puts equal
    // contact schedules next to each other (hmpc_api.cu: order_* kernels), or null
    const int* work_order;
    // per-hopper model body (hmpc_set_body_params), [kBodyModel][B] in Body's field order, or null: every hopper plans
    // with the scalars m, mu, rh, Jinv above (the default path then does no extra loads)
    const double* body = nullptr;
};
__device__ __forceinline__ int work_item(const QpConst& c, int i, int B) {
    const int t = (int)(((long long)i * c.work_mul + c.work_add) % B);
    return c.work_order ? c.work_order[t] : t;
}

// The body the MPC plans with for hopper b (the arguments of Mpc.__init__ minus g, mpc_cvx_euler_3f.py:12-39).
// Always indexed by hopper, never by work ticket.
struct Body {
    double m, mu, rh[3], Jinv[9];
};
constexpr int kBodyModel = 14;        // doubles per hopper of QpConst::body
__device__ __forceinline__ Body scalar_body(const QpConst& c) {
    Body bd;
    bd.m = c.m; bd.mu = c.mu;
#pragma unroll
    for (int i = 0; i < 3; ++i) bd.rh[i] = c.rh[i];
#pragma unroll
    for (int i = 0; i < 9; ++i) bd.Jinv[i] = c.Jinv[i];
    return bd;
}
__device__ __forceinline__ Body model_body(const QpConst& c, int b, int B) {
    if (!c.body) return scalar_body(c);
    Body bd;
    {
        const double* p = c.body + b;
        const size_t Bs = (size_t)B;
        bd.m = p[0]; bd.mu = p[Bs];
#pragma unroll
        for (int i = 0; i < 3; ++i) bd.rh[i] = p[(2 + i) * Bs];
#pragma unroll
        for (int i = 0; i < 9; ++i) bd.Jinv[i] = p[(5 + i) * Bs];
    }
    return bd;
}
// The CTA kernel's condensing reads the body through one of two sources, chosen per hopper on QpConst::body: the
// QpConst itself (its scalars) or a shared-memory copy of hopper b's body (condense_hopper: the model array's column,
// or the scalars when none is set).  Neither keeps the body in registers across the condensing: the 128-register
// builds of that kernel have no room for it.
struct SmemBody {
    const double* s;   // [kBodyModel] in QpConst::body's row order
};
__device__ __forceinline__ double body_m(const QpConst& c) { return c.m; }
__device__ __forceinline__ double body_rh(const QpConst& c, int i) { return c.rh[i]; }
__device__ __forceinline__ double body_Jinv(const QpConst& c, int i) { return c.Jinv[i]; }
__device__ __forceinline__ double body_m(const SmemBody& h) { return h.s[0]; }
__device__ __forceinline__ double body_rh(const SmemBody& h, int i) { return h.s[2 + i]; }
__device__ __forceinline__ double body_Jinv(const SmemBody& h, int i) { return h.s[5 + i]; }

// ------------------------------------------------------------------------------------------------
// shared-memory carve-up (all doubles unless noted)
// ------------------------------------------------------------------------------------------------
struct Work {
    // linearisation
    double *gp;      // [N][4]  guess position + yaw per stage
    double *cz, *sz; // [N]
    double *PC, *PS; // [N+1]   prefix sums of cos/sin
    double *Bv;      // [N][9]  dt * B[6:9, 0:3]
    double *Bw;      // [N][18] dt * B[9:12, 0:6]
    double *pfw;     // [N][3]
    double *xin;     // [12]
    double *cfree;   // [N+1][12] free response
    double *err;     // [N+1][12] cfree[i] - xref[i-1]  (row 0 unused); later the solution trajectory
    double *Qd, *Rd; // [12], [6]
    double *hinv;    // [N]  1/(k-1) height-row normalisation (k >= 2)
    // QP data
    double *g, *lo, *hi;               // [n] [m] [m]
    // solver vectors
    double *x, *tmp, *xp;                          // [n] each
    double *xt, *rhs, *sc, *dinv;                  // [kkt_max] each (compact systems: variables + active rows)
    double *mv[kNumMVec];                          // [m] each (roles differ per solver)
    double *red;                                   // [48] reduction scratch
    int *idx;                          // [n]  compact list of the variables in the current system
    int *grow;                         // [kkt_max] polish: active general rows in the current system
    int *cnt;                          // [4]  nF, ng, ...
    int8_t *fixed;                     // [n]  1: variable eliminated a priori (lo == hi == 0)
    int8_t *pin;                       // [n]  polish: variable pinned (fixed or at a bound)
    int8_t *code;                      // [m]  +1 upper active, -1 lower active, 0 inactive
    int8_t *side;                      // [m]  IPM: bit0 finite upper side, bit1 finite lower side
    int8_t *stance;                    // [N]
    // matrices (shared or global), packed lower triangles: H of order n, the LDL' factor of order <= 8N
    double* H;
    void* Lm;
};

// The polish system holds the unpinned variables plus the active friction / height rows: up to 7N+2
// unknowns (a larger active set makes the polish give up and the interior point take over).
__host__ __device__ inline int kkt_max(int N) { return 7 * N + 2; }
// Symmetric / triangular matrices are stored packed, column by column (lower triangle): element (i, j),
// i >= j, of an order-k matrix sits at tri_off(j, k) + (i - j).
__host__ __device__ inline int tri_off(int j, int k) { return j * k - (j * (j - 1)) / 2; }
// fsize: bytes per factor entry (8: FP64 factor, 4: FP32 factor)
// Horizons beyond the 128-thread kernels (6N > 64) keep the FP64 factor as a lower block triangle of 8x8 tiles for the
// tensor-core path (LinSys::factor_tiled): room for both layouts.
__host__ __device__ inline bool tiled_factor_applies(int N, int fsize = 8) { return 6 * N > 64 && fsize == 8; }
__host__ __device__ inline size_t tiled_factor_doubles(int N) {
    const size_t nt = ((size_t)kkt_max(N) + 7) / 8;
    return (nt * (nt + 1) / 2) * 64;
}
__host__ __device__ inline size_t mat_doubles(int N, int fsize = 8) {
    const size_t n = 6 * (size_t)N, kk = (size_t)kkt_max(N);
    size_t f = (kk * (kk + 1) / 2 * (size_t)fsize + 7) / 8;
    if (tiled_factor_applies(N, fsize) && tiled_factor_doubles(N) > f) f = tiled_factor_doubles(N);
    return n * (n + 1) / 2 + f;
}
// compact-system vectors: padded to whole tiles for the tiled path
__host__ __device__ inline int kkt_vec(int N) { return kkt_max(N) + (6 * N > 64 ? 8 : 0); }
// Longest horizons (N >= 58, the reference's N = 60 among them): with every vector in shared memory a CTA needs more
// than half of the SM's 228 KB, so the nine m-vectors only the interior point (and, aliased, the condensing) uses move
// to the L2 workspace next to the matrices -- 47 KB at N = 60, which buys the second resident CTA (65536 hoppers:
// 103 k -> 139 k steps/s; at N = 40, where two CTAs fit anyway, the same move costs 5 %).  The two m-vectors of the
// active-set refinement stay in shared memory.
constexpr int kNumMVecShared = 2;
__host__ __device__ inline bool mv_in_workspace(int N) { return N > 57; }
__host__ __device__ inline size_t ws_mv_doubles(int N) { return mv_in_workspace(N) ? (size_t)(kNumMVec - kNumMVecShared) * 11 * N : 0; }
__host__ __device__ inline size_t work_vec_doubles(int N, bool mv_ws = false) {
    const int n = 6 * N, m = 11 * N;
    size_t d = 0;
    // linearisation (cfree, gp, pfw, Qd, Rd, PC, PS alias the last three m-vectors: dead once condense() returns)
    d += 2 * N + 9 * N + 18 * N + 12 + 12 * (N + 1) + N;
    d += n + 2 * m;           // g lo hi
    d += 3 * n + (N > 14 ? N - 14 : 0) + 4 * kkt_vec(N);   // x xp tmp(+pad) | xt rhs sc dinv
    d += (mv_ws ? kNumMVecShared : kNumMVec) * m;
    d += 48;                  // red
    d += (n + kkt_max(N) + 4 + 1) / 2;          // int32: idx grow cnt
    d += (2 * n + 2 * m + N + 7) / 8;           // int8: fixed pin code side stance
    return d;
}

// mvext: null, or where the m-vectors beyond the first kNumMVecShared live (workspace, ws_mv_doubles(N))
__device__ inline void carve(Work& w, double* base, int N, double* mvext = nullptr) {
    const int n = 6 * N, m = 11 * N, kk = kkt_max(N);
    double* p = base;
    auto take = [&](size_t k) { double* r = p; p += k; return r; };
    w.cz = take(N); w.sz = take(N);
    w.Bv = take(9 * N); w.Bw = take(18 * N); w.xin = take(12);
    w.err = take(12 * (N + 1));
    w.hinv = take(N);
    w.g = take(n); w.lo = take(m); w.hi = take(m);
    // tmp | xt | rhs | sc are contiguous: together they are the 4-column panel scratch of LinSys::factor
    w.x = take(n); w.xp = take(n); w.tmp = take(n + (N > 14 ? N - 14 : 0));   // pad: 4 (kkt_max - 4) panel entries
    { const int kv = kkt_vec(N); w.xt = take(kv); w.rhs = take(kv); w.sc = take(kv); w.dinv = take(kv); }
    for (int i = 0; i < kNumMVecShared; ++i) w.mv[i] = take(m);
    {   // the remaining m-vectors hang off ONE base pointer (shared memory or workspace): constant offsets, no pointer table
        double* mvb = mvext ? mvext : take((size_t)(kNumMVec - kNumMVecShared) * m);
        for (int i = kNumMVecShared; i < kNumMVec; ++i) w.mv[i] = mvb + (size_t)(i - kNumMVecShared) * m;
    }
    // condense-only scratch on top of the solvers' last three m-vectors: 12(N+1) + 4N + 3N + 18 + 2(N+1) <= 33N
    w.cfree = w.mv[kNumMVec - 3]; w.gp = w.cfree + 12 * (N + 1); w.pfw = w.gp + 4 * N;
    w.Qd = w.pfw + 3 * N; w.Rd = w.Qd + 12; w.PC = w.Rd + 6; w.PS = w.PC + (N + 1);
    w.red = take(48);
    w.idx = reinterpret_cast<int*>(p);
    w.grow = w.idx + n;
    w.cnt = w.grow + kk;
    w.fixed = reinterpret_cast<int8_t*>(w.cnt + 4);
    w.pin = w.fixed + n;
    w.code = w.pin + n;
    w.side = w.code + m;
    w.stance = w.side + m;
}

// ------------------------------------------------------------------------------------------------
// block reductions -- warp shuffles + one shared round.  OP: 0 max, 1 min, 2 sum.  Result in all threads.
// ------------------------------------------------------------------------------------------------
template <int OP>
__device__ __forceinline__ double red_op(double a, double b) {
    return OP == 0 ? fmax(a, b) : (OP == 1 ? fmin(a, b) : a + b);
}
template <int K, int OP>
__device__ inline void block_reduce(double (&v)[K], double* red) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#ifndef HMPC_HOST_EMUL   // tests/emul runs this source as one serial "thread" on the CPU
#pragma unroll
    for (int k = 0; k < K; ++k) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[k] = red_op<OP>(v[k], __shfl_xor_sync(0xffffffffu, v[k], o));
    }
#endif
    __syncthreads();
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < K; ++k) red[wid * K + k] = v[k];
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < K; ++k) {
        double r = red[k];
        for (int q = 1; q < nw; ++q) r = red_op<OP>(r, red[q * K + k]);
        v[k] = r;
    }
}

// ------------------------------------------------------------------------------------------------
// constraint operator A (implicit)
//   rows 0..n-1        identity
//   rows n+4k+s        friction, stance stages only:  s=0: fx-mu fz, 1: -fx-mu fz, 2: fy-mu fz, 3: -fy-mu fz
//                      (s>=2 disabled for 2f)
//   rows n+4N+k        height z_k (k>=2), normalised:  sum_{j<=k-2} (k-j-1)/(k-1) * fz_j
// ------------------------------------------------------------------------------------------------
struct AOp {
    int N, n, fy_rows;   // fy_rows: 1 for 3f
    double mu;
    const int8_t* stance;
    const double* hinv;  // [N] 1/(k-1)
    __device__ __forceinline__ bool fr_on(int k, int s) const { return stance[k] && (s < 2 || fy_rows); }
    __device__ inline double row(int r, const double* x) const {
        if (r < n) return x[r];
        r -= n;
        if (r < 4 * N) {
            const int k = r >> 2, s = r & 3;
            if (!fr_on(k, s)) return 0.0;
            const double sg = (s & 1) ? -1.0 : 1.0;
            return sg * x[6 * k + (s >> 1)] - mu * x[6 * k + 2];
        }
        const int k = r - 4 * N;
        if (k < 2) return 0.0;
        double acc = 0.0;
        for (int j = 0; j + 2 <= k; ++j) acc += (double)(k - j - 1) * x[6 * j + 2];
        return acc * hinv[k];
    }
    // coefficient of general row r (r >= n) at variable v
    __device__ inline double coef(int r, int v) const {
        r -= n;
        const int kv = v / 6, cv = v - 6 * kv;
        if (r < 4 * N) {
            const int k = r >> 2, s = r & 3;
            if (k != kv || !fr_on(k, s)) return 0.0;
            if (cv == 2) return -mu;
            if (cv == (s >> 1)) return (s & 1) ? -1.0 : 1.0;
            return 0.0;
        }
        const int k = r - 4 * N;
        if (cv != 2 || k < 2 || kv + 2 > k) return 0.0;
        return (double)(k - kv - 1) * hinv[k];
    }
    // (A^T v)_i
    __device__ inline double colT(int i, const double* v) const {
        double acc = v[i];
        const int k = i / 6, c = i - 6 * k;
        if (c > 2) return acc;
        const double* f = v + n + 4 * k;
        if (stance[k]) {
            if (c == 0) acc += f[0] - f[1];
            else if (c == 1) { if (fy_rows) acc += f[2] - f[3]; }
            else acc -= mu * (f[0] + f[1] + (fy_rows ? f[2] + f[3] : 0.0));
        }
        if (c == 2) {
            const double* zr = v + n + 4 * N;
            for (int kk = k + 2; kk < N; ++kk) acc += (double)(kk - k - 1) * hinv[kk] * zr[kk];
        }
        return acc;
    }
    // (A^T diag(w) A)_{ij} without the identity rows
    __device__ inline double gram(int i, int j, const double* w) const {
        const int ki = i / 6, ci = i - 6 * ki, kj = j / 6, cj = j - 6 * kj;
        if (ci > 2 || cj > 2) return 0.0;
        double acc = 0.0;
        if (ki == kj && stance[ki]) {
            const double* f = w + n + 4 * ki;
            const double w0 = f[0], w1 = f[1], w2 = fy_rows ? f[2] : 0.0, w3 = fy_rows ? f[3] : 0.0;
            const int lo_ = ci < cj ? ci : cj, hi_ = ci < cj ? cj : ci;
            if (lo_ == 0 && hi_ == 0) acc += w0 + w1;
            else if (lo_ == 1 && hi_ == 1) acc += w2 + w3;
            else if (lo_ == 2 && hi_ == 2) acc += mu * mu * (w0 + w1 + w2 + w3);
            else if (lo_ == 0 && hi_ == 2) acc += -mu * (w0 - w1);
            else if (lo_ == 1 && hi_ == 2) acc += -mu * (w2 - w3);
        }
        if (ci == 2 && cj == 2) {
            const double* zr = w + n + 4 * N;
            const int k0 = (ki > kj ? ki : kj) + 2;
            for (int kk = k0; kk < N; ++kk) {
                const double h = hinv[kk];
                acc += zr[kk] * h * h * (double)(kk - ki - 1) * (double)(kk - kj - 1);
            }
        }
        return acc;
    }
};

// ------------------------------------------------------------------------------------------------
// linearisation of one stage (gen_dt_dynamics); thread k handles stage k
// ------------------------------------------------------------------------------------------------
template <class Bd>   // QpConst (the scalars) or SmemBody
__device__ inline void linearize_stage(const QpConst& c, const Bd& bd, int k, Work& w) {
    const double psi = w.gp[4 * k + 3];
    double sn, cs;
    sincos(psi, &sn, &cs);
    w.cz[k] = cs; w.sz[k] = sn;
    const double Rz[9] = {cs, sn, 0, -sn, cs, 0, 0, 0, 1};
    const double d[3] = {w.pfw[3 * k] - w.gp[4 * k], w.pfw[3 * k + 1] - w.gp[4 * k + 1],
                         w.pfw[3 * k + 2] - w.gp[4 * k + 2]};
    double rf[3];
    mat3_vec(Rz, d, rf);
    rf[0] += body_rh(bd, 0); rf[1] += body_rh(bd, 1); rf[2] += body_rh(bd, 2);
    // Jw = Rz Jinv Rz^T
    double T1[9], Jw[9];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            double a = 0;
            for (int l = 0; l < 3; ++l) a += Rz[3 * i + l] * body_Jinv(bd, 3 * l + j);
            T1[3 * i + j] = a;
        }
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            double a = 0;
            for (int l = 0; l < 3; ++l) a += T1[3 * i + l] * Rz[3 * j + l];
            Jw[3 * i + j] = a;
        }
    // JwRzT = Jw Rz^T
    double JwRzT[9];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            double a = 0;
            for (int l = 0; l < 3; ++l) a += Jw[3 * i + l] * Rz[3 * j + l];
            JwRzT[3 * i + j] = a;
        }
    double Bf[9];   // B[9:12, 0:3]
    double* Bv = w.Bv + 9 * k;
    if (c.dyn == 3) {
        double rw[3];
        mat3T_vec(Rz, rf, rw);   // Rz^T rf
        const double hatm[9] = {0, -rw[2], rw[1], rw[2], 0, -rw[0], -rw[1], rw[0], 0};
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) {
                double a = 0;
                for (int l = 0; l < 3; ++l) a += Jw[3 * i + l] * hatm[3 * l + j];
                Bf[3 * i + j] = a;
            }
        for (int i = 0; i < 9; ++i) Bv[i] = 0.0;
        Bv[0] = Bv[4] = Bv[8] = (1.0 / body_m(bd)) * c.dt;
    } else {
        const double hatm[9] = {0, -rf[2], rf[1], rf[2], 0, -rf[0], -rf[1], rf[0], 0};
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) {
                double a = 0;
                for (int l = 0; l < 3; ++l) a += JwRzT[3 * i + l] * hatm[3 * l + j];
                Bf[3 * i + j] = a;
            }
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) Bv[3 * i + j] = (Rz[3 * j + i] / body_m(bd)) * c.dt;   // Rz^T / m
    }
    double* Bw = w.Bw + 18 * k;
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            Bw[6 * i + j] = Bf[3 * i + j] * c.dt;
            Bw[6 * i + 3 + j] = JwRzT[3 * i + j] * c.dt;
        }
}

// ------------------------------------------------------------------------------------------------
// Condense.  Requires w.gp, w.pfw, w.xin, w.Qd, w.Rd, w.stance filled and a __syncthreads() before.
// xref points at this hopper's window, element (k, c) at xref[(k*12 + c) * xs].
// bd: the hopper's model body (QpConst for the scalars, or SmemBody; condense_hopper chooses).
// Leaves H (row-major n x n, symmetric, full), g, lo, hi, fixed, cfree in place.  Returns (all threads)
// 1 when the u-independent height rows k=0,1 are violated (SURVEY App. D2).
// ------------------------------------------------------------------------------------------------
template <class Bd>
__device__ inline int condense(const QpConst& c, const Bd& bd, Work& w, const double* xref, size_t xs) {
    const int N = c.N, n = 6 * N, m = 11 * N, tid = threadIdx.x, T = blockDim.x;
    for (int k = tid; k < N; k += T) {
        linearize_stage(c, bd, k, w);
        w.hinv[k] = (k >= 2) ? 1.0 / (double)(k - 1) : 0.0;
    }
    __syncthreads();
    if (tid == 0) {
        double pc = 0, ps = 0;
        w.PC[0] = 0; w.PS[0] = 0;
        for (int k = 0; k < N; ++k) { pc += w.cz[k]; ps += w.sz[k]; w.PC[k + 1] = pc; w.PS[k + 1] = ps; }
    }
    __syncthreads();
    const double dt = c.dt, gdt = -c.g * dt;
    // free response + tracking error
    for (int i = tid; i <= N; i += T) {
        double* cf = w.cfree + 12 * i;
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
            for (int q = 0; q < 12; ++q) w.err[12 * i + q] = cf[q] - xref[((size_t)(i - 1) * 12 + q) * xs];
    }
    // bounds
    for (int r = tid; r < m; r += T) {
        double lo = -kInf, hi = kInf;
        if (r < n) {
            const int k = r / 6, cc = r - 6 * k;
            if (cc >= 3) { lo = -c.tau_max[cc - 3]; hi = c.tau_max[cc - 3]; }
            else if (!w.stance[k]) { lo = 0.0; hi = 0.0; }
            else if (cc == 2) { lo = 0.0; hi = c.fz_max; }
            if (cc == 1 && c.dyn == 2) { lo = 0.0; hi = 0.0; }
            w.fixed[r] = (hi - lo) < 1e-12 ? 1 : 0;
        } else if (r < n + 4 * N) {
            const int k = (r - n) >> 2, s = (r - n) & 3;
            if (w.stance[k] && (s < 2 || c.dyn == 3)) hi = 0.0;
        }
        w.lo[r] = lo; w.hi[r] = hi;
    }
    __syncthreads();
    // height rows need cfree.  Exact feasibility (all-threads result): the height rows are monotone in
    // the stance fz and fz = fz_max, fx = fy = 0 satisfies every other row, so the QP is feasible iff
    // z_k(fz = fz_max on stance stages) >= z_min for k = 0..N-1 (k = 0, 1 are u-independent, App. D2).
    const double zc = dt * dt / body_m(bd);
    int infeasible = 0;
    for (int k = tid; k < N; k += T) {
        double up = 0.0;
        for (int j = 0; j + 2 <= k; ++j) if (w.stance[j]) up += (double)(k - j - 1);
        if (w.cfree[12 * k + 2] + zc * c.fz_max * up < c.z_min) infeasible = 1;
        if (k >= 2) w.lo[n + 4 * N + k] = (c.z_min - w.cfree[12 * k + 2]) / (zc * (double)(k - 1));
    }
    infeasible = __syncthreads_or(infeasible);
    // Hessian blocks, lower block-triangle a >= b
    const int nblk = N * (N + 1) / 2;
    const double q3 = w.Qd[3], q4 = w.Qd[4], q5 = w.Qd[5];
    for (int p = tid; p < nblk; p += T) {
        // decode p -> (a, b), a >= b
        int a = (int)((sqrt(8.0 * (double)p + 1.0) - 1.0) * 0.5);
        while ((a + 1) * (a + 2) / 2 <= p) ++a;
        while (a * (a + 1) / 2 > p) --a;
        const int b = p - a * (a + 1) / 2;
        const double pca = w.PC[a + 1], psa = w.PS[a + 1], pcb = w.PC[b + 1], psb = w.PS[b + 1];
        double s0 = 0, NN = 0, CC = 0, SS = 0, CS = 0, SC = 0;
        for (int i = a + 1; i <= N; ++i) {
            const double kap = (i == N) ? c.kf : 1.0;
            const double wca = w.PC[i] - pca, wsa = w.PS[i] - psa, wcb = w.PC[i] - pcb, wsb = w.PS[i] - psb;
            const double na = (double)(i - a - 1), nb = (double)(i - b - 1);
            s0 += kap; NN += kap * na * nb;
            CC += kap * wca * wcb; SS += kap * wsa * wsb; CS += kap * wca * wsb; SC += kap * wsa * wcb;
        }
        const double dt2 = dt * dt;
        double M3[9] = {s0 * w.Qd[9] + dt2 * (q3 * CC + q4 * SS), dt2 * (q3 * CS - q4 * SC), 0,
                        dt2 * (q3 * SC - q4 * CS), s0 * w.Qd[10] + dt2 * (q3 * SS + q4 * CC), 0,
                        0, 0, s0 * w.Qd[11] + dt2 * q5 * NN};
        const double dv[3] = {dt2 * NN * w.Qd[0] + s0 * w.Qd[6], dt2 * NN * w.Qd[1] + s0 * w.Qd[7],
                              dt2 * NN * w.Qd[2] + s0 * w.Qd[8]};
        const double* Bwa = w.Bw + 18 * a; const double* Bwb = w.Bw + 18 * b;
        const double* Bva = w.Bv + 9 * a;  const double* Bvb = w.Bv + 9 * b;
        double MB[18];   // M3 * Bw_b  (3x6)
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 6; ++j)
                MB[6 * i + j] = M3[3 * i] * Bwb[j] + M3[3 * i + 1] * Bwb[6 + j] + M3[3 * i + 2] * Bwb[12 + j];
        for (int r = 0; r < 6; ++r)
            for (int cc = 0; cc < 6; ++cc) {
                double v = Bwa[r] * MB[cc] + Bwa[6 + r] * MB[6 + cc] + Bwa[12 + r] * MB[12 + cc];
                if (r < 3 && cc < 3)
                    v += Bva[r] * dv[0] * Bvb[cc] + Bva[3 + r] * dv[1] * Bvb[3 + cc] + Bva[6 + r] * dv[2] * Bvb[6 + cc];
                v *= 2.0;
                if (a == b && r == cc && a != N - 1) v += 2.0 * w.Rd[r];
                const int hi_ = 6 * a + r, hj_ = 6 * b + cc;          // a >= b: only the diagonal blocks hold
                if (hi_ >= hj_) w.H[tri_off(hj_, n) + (hi_ - hj_)] = v;   // entries above the diagonal
            }
    }
    // gradient
    const double ubar_alias = (c.uref_mode == 0) ? (w.stance[N - 1] ? 2.0 * body_m(bd) * c.g : 0.0) : 0.0;
    for (int a = tid; a < N; a += T) {
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
        const double* Bwa = w.Bw + 18 * a; const double* Bva = w.Bv + 9 * a;
        for (int r = 0; r < 6; ++r) {
            double v = Bwa[r] * tw[0] + Bwa[6 + r] * tw[1] + Bwa[12 + r] * tw[2];
            if (r < 3) v += Bva[r] * tv[0] + Bva[3 + r] * tv[1] + Bva[6 + r] * tv[2];
            v *= 2.0;
            if (r == 2 && a != N - 1) {
                const double ub = (c.uref_mode == 0) ? ubar_alias : (w.stance[a] ? 2.0 * body_m(bd) * c.g : 0.0);
                v -= 2.0 * w.Rd[2] * ub;
            }
            w.g[6 * a + r] = v;
        }
    }
    __syncthreads();
    return infeasible;
}
// the same with the handle's scalar body, for callers that condense without a hopper index
__device__ inline int condense(const QpConst& c, Work& w, const double* xref, size_t xs) {
    return condense(c, c, w, xref, xs);
}
// condense hopper b with its model body (QpConst::body) or, when none is set, the scalars.  Either is staged in the
// reduction scratch w.red, which only the solvers use: one instantiation of condense, no body in registers.
__device__ inline void stage_body(const QpConst& c, Work& w, int b, int B) {
    for (int r = threadIdx.x; r < kBodyModel; r += blockDim.x) {
        double v;
        if (c.body) v = c.body[(size_t)r * B + b];
        else v = r == 0 ? c.m : r == 1 ? c.mu : r < 5 ? c.rh[r - 2] : c.Jinv[r - 5];
        w.red[r] = v;
    }
}
__device__ inline int condense_hopper(const QpConst& c, Work& w, int b, int B, const double* xref, size_t xs) {
    stage_body(c, w, b, B);
    __syncthreads();
    return condense(c, SmemBody{w.red}, w, xref, xs);
}

// algorithmic FLOP counts (FMA = 2) of the dense kernels, accumulated per hopper for the roofline report
__host__ __device__ inline double flops_factor(int nk) { return (double)nk * ((double)nk * nk - 1.0) / 3.0; }
__host__ __device__ inline double flops_solve(int nk) { return 2.0 * (double)nk * ((double)nk - 1.0); }
__host__ __device__ inline double flops_matvec(int n) { return 2.0 * (double)n * n; }
// linearise (330 per stage, SURVEY 8d) + closed-form Hessian blocks (~430 per 6x6 block plus 14 per term of
// its stage sums) + gradient (30 per term, 70 per stage)
__host__ __device__ inline double flops_condense(int N) {
    double f = 330.0 * N + 70.0 * N;
    for (int a = 0; a < N; ++a) f += (a + 1) * (430.0 + 14.0 * (N - a)) + 30.0 * (N - a);
    return f;
}

// ------------------------------------------------------------------------------------------------
// Ordered compaction: list[0..count) = { first + i : pred(first + i), 0 <= i < len }, count returned in
// *cnt (shared).  Warp 0 walks the range 32 entries at a time with ballots; at most `cap` entries are
// stored but all are counted.  Callers __syncthreads() afterwards.
// ------------------------------------------------------------------------------------------------
template <class Pred>
__device__ inline void compact_indices(int first, int len, int cap, int* list, int* cnt, Pred pred) {
#ifdef HMPC_HOST_EMUL
    int c = 0;
    for (int i = 0; i < len; ++i) if (pred(first + i)) { if (c < cap) list[c] = first + i; ++c; }
    *cnt = c;
#else
    if (threadIdx.x < 32) {
        const int lane = threadIdx.x;
        int c = 0;
        for (int base = 0; base < len; base += 32) {
            const int i = base + lane;
            const bool p = (i < len) && pred(first + i);
            const unsigned mask = __ballot_sync(0xffffffffu, p);
            const int pos = c + __popc(mask & ((1u << lane) - 1u));
            if (p && pos < cap) list[pos] = first + i;
            c += __popc(mask);
        }
        if (lane == 0) *cnt = c;
    }
#endif
}

// ------------------------------------------------------------------------------------------------
// LDL' factorisation  K = L' D L'^T  (L' unit lower triangular, D diagonal) of the compact system,
// nk = nF + ng:
//   variables  idx[0..nF)   full variable indices kept in the system
//   rows       grow[0..ng)  active general rows (polish only); they follow the variables
//   K_vv = H[idx_i][idx_j] + (wts ? (A' diag(wts) A)_ij : 0) + dadd [i==j];  K_rv = A.coef;
//   K_rr = 0; after the variables are eliminated the row block holds the Schur complement -G K_vv^-1 G',
//   whose diagonal is then scaled by (1 + eps): a relative regularisation that keeps exactly dependent rows
//   at a negative pivot well above the factor's rounding level and is removed again by the refinement
// With ng = 0 this is the positive definite IPM / ADMM operator (all pivots > 0); with ng > 0 the matrix
// is quasi-definite: the LDL' exists for every ordering and the last ng pivots are negative.
//
// Right-looking: K is first assembled into shared memory by all threads, then column j's rank-1 update
// of the trailing matrix is spread over the CTA (warp per trailing column, lane per row) with ONE
// barrier per column; the columns stay unscaled (U = L' D) during the elimination and are scaled to the unit
// lower triangular L' at the end, next to dinv = 1/D.
// Substitutions run warp-synchronously in warp 0 (the dependency chain is serial anyway and a
// __syncwarp() is far cheaper than a CTA barrier).
// U is stored packed (lower triangle, column by column): the forward sweep reads contiguous columns, the
// backward sweep reads a row with the slowly varying stride nk - i.
// ------------------------------------------------------------------------------------------------
// Reciprocal of a pivot without the library's division slow path: MUFU seed + two Newton steps (relative error
// ~1e-16, not correctly rounded -- the factor only feeds an iteratively refined, KKT-verified solve).  The
// library division was 4.6 % of all executed instructions of the kernel (every thread divides once per pivot)
// and sits on the critical path of every pivot (tools/micro/tiled.cu: 145 vs ~70 cycles).
__device__ __forceinline__ double fast_rcp(double d) {
#ifdef HMPC_HOST_EMUL
    return 1.0 / d;
#else
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));
    r = fma(fma(-d, r, 1.0), r, r);
    r = fma(fma(-d, r, 1.0), r, r);
    return r;
#endif
}
__device__ __forceinline__ float fast_rcp(float d) { return 1.0f / d; }

template <typename F>
struct LinSys {
    typedef F real;
    int n, nF, ng;
    F *Lm, *dinv;
    const double* H;
    const int *idx, *grow;
    double flops = 0.0;   // algorithmic FLOPs of factor/solve since the last reset (same value in all threads)
    int solver_warp = 0;  // which warp of the CTA runs the substitutions
    int tiled = 0;        // 1: FP64 tensor-core tiles, all warps of the CTA (factor_tiled / solve_tiled; wide kernels)
    int ipm_tiled = 0;    // 1: the interior point of an N <= 10 kernel may switch to the tiled factor (latency-bound launches only)

    __device__ inline double entry(const AOp& A, const double* wts, double dadd, double eps, int i, int j) const {
        if (i < nF) {   // i >= j
            const int vi = idx[i], vj = idx[j];
            double s = vi >= vj ? H[tri_off(vj, n) + (vi - vj)] : H[tri_off(vi, n) + (vj - vi)];
            if (wts) { s += A.gram(vi, vj, wts); if (i == j) s += wts[vi]; }
            if (i == j) s += dadd;
            return s;
        }
        if (j < nF) return A.coef(grow[i - nF], idx[j]);
        if (i != j) return 0.0;
        // the row block starts at zero: its regularisation is applied relative to the Schur complement once
        // the variables have been eliminated (factor()).  A row without any unpinned variable is decoupled.
        const int r = grow[i - nF];
        for (int q = 0; q < nF; ++q) if (A.coef(r, idx[q]) != 0.0) return 0.0;
        return -1.0;
    }

    // Returns nonzero (same value in all threads) when a pivot has the wrong sign or is not finite.
    // P: scratch of at least 4 (nk - 4) doubles (the pre-scaled panel, see below).
    __device__ inline int factor(const AOp& A, const double* wts, double dadd, double eps, double* scratch) {
#ifndef HMPC_HOST_EMUL
        if (sizeof(F) == 8 && tiled) return factor_tiled(A, wts, dadd, eps, scratch);
#endif
        PH_T0(ph_f);
        F* P = reinterpret_cast<F*>(scratch);
        const int tid = threadIdx.x, T = blockDim.x, nk = nF + ng;
        const int LS = T < 32 ? T : 32, lane = tid % LS, wid = tid / LS, nw = T / LS;
        flops += flops_factor(nk);
        // ---- assemble the lower triangle (packed, column by column); entries are formed in FP64 ----
        for (int jj = wid; jj < nk; jj += nw) {          // warp per column, lane per row: no index division
            F* colp = Lm + tri_off(jj, nk) - jj;
            for (int ii = jj + lane; ii < nk; ii += LS) colp[ii] = (F)entry(A, wts, dadd, eps, ii, jj);
        }
        __syncthreads();
        int bad = 0;
        // ---- blocked right-looking elimination, 4 pivot columns per block ----
        for (int j0 = 0; j0 < nk;) {
            // blocks never straddle the variable / row boundary nF
            const int lim = (j0 < nF ? nF : nk) - j0;
            const int bs = lim < 4 ? lim : 4, t0 = j0 + bs;
            if (j0 == nF && ng > 0) {
                for (int r = tid; r < ng; r += T) Lm[tri_off(nF + r, nk)] *= (F)(1.0 + eps);
                __syncthreads();
            }
            // panel: eliminate column j inside the panel only; keep P[i - t0][p] = U(i, j) / d_j for the rows below
            for (int p = 0; p < bs; ++p) {
                const int j = j0 + p;
                const F* colj = Lm + tri_off(j, nk) - j;      // colj[i] = U(i, j), i >= j
                const F piv = colj[j];
                const F ap = (j < nF) ? piv : -piv;
                const bool ok = (ap > (F)0) && (ap < (F)1e30);
                if (!ok) bad = 1;
                const F rinv = fast_rcp(ok ? piv : (F)1);
                if (tid == 0) dinv[j] = rinv;
                for (int i = j + 1 + tid; i < nk; i += T) {
                    const F uij = colj[i];
                    if (i >= t0) {
                        P[4 * (i - t0) + p] = uij * rinv;
                        if (p == bs - 1) for (int pp = bs; pp < 4; ++pp) P[4 * (i - t0) + pp] = (F)0;   // short block
                    }
                    for (int k = j + 1; k < t0 && k <= i; ++k)
                        Lm[tri_off(k, nk) + (i - k)] -= uij * (colj[k] * rinv);
                }
                __syncthreads();
            }
            // trailing matrix: rank-4 update.  Lanes own row pairs (short row t0+q, long row nk-1-q: equal
            // work per lane, consecutive addresses across lanes), warps own the columns k = t0 + wid (mod nw).
            const int t = nk - t0;
            if (t > 0) {
                const F* c0 = Lm + tri_off(j0, nk) - j0;
                const F* c1 = bs > 1 ? Lm + tri_off(j0 + 1, nk) - (j0 + 1) : c0;     // short block: the unused
                const F* c2 = bs > 2 ? Lm + tri_off(j0 + 2, nk) - (j0 + 2) : c0;     // columns alias c0 and meet
                const F* c3 = bs > 3 ? Lm + tri_off(j0 + 3, nk) - (j0 + 3) : c0;     // zeros in P
                const int npairs = (t + 1) >> 1;
                for (int q = lane; q < npairs; q += LS) {
                    for (int side = 0; side < 2; ++side) {
                        const int r = side ? (nk - 1 - q) : (t0 + q);
                        if (side && r == t0 + q) break;
                        const F a0 = c0[r], a1 = c1[r], a2 = c2[r], a3 = c3[r];
                        int k = t0 + wid;
                        int off = tri_off(k, nk) - k;                 // column k starts at Lm + off + k
                        const F* pk = P + 4 * (k - t0);
                        for (; k <= r; k += nw) {
                            Lm[off + r] -= a0 * pk[0] + a1 * pk[1] + a2 * pk[2] + a3 * pk[3];
                            off += nw * (nk - 1 - k) - (nw * (nw - 1)) / 2;
                            pk += 4 * nw;
                        }
                    }
                }
                __syncthreads();
            }
            j0 = t0;
        }
        // scale the columns: L' = U D^-1 (unit lower triangular), so that the substitutions carry no
        // multiplication by 1/d on their dependency chain
        for (int jj = wid; jj < nk; jj += nw) {
            F* colp = Lm + tri_off(jj, nk) - jj;
            const F dj = dinv[jj];
            for (int ii = jj + 1 + lane; ii < nk; ii += LS) colp[ii] *= dj;
        }
        __syncthreads();
        PH_ADD(4, ph_f);
        return bad;
    }

    // Solves K out = b for compact FP64 vectors of length nk with K = L' D L'^T; the substitutions run in the
    // factor's precision.  b is left untouched unless out aliases it.  Ends with a __syncthreads().
    // One warp runs the (serial) substitution; each lane keeps the right-hand-side entries of its rows
    // (lane, lane+32, lane+64) in registers and the pivot entry is broadcast with a shuffle, so the dependency
    // chain per column is one shuffle and one FMA.
    __device__ inline void solve(const double* b, double* out, double* scratch) {
#ifndef HMPC_HOST_EMUL
        if (sizeof(F) == 8 && tiled) { solve_tiled(b, out, scratch); return; }
#endif
        F* sc = reinterpret_cast<F*>(scratch);
        const int tid = threadIdx.x, T = blockDim.x, nk = nF + ng;
        const int LS = T < 32 ? T : 32;
        PH_T0(ph_s);
        flops += flops_solve(nk);
        __syncthreads();
        // co-resident CTAs use different warp slots so that their substitutions land on different SM
        // sub-partitions (warp w lives on scheduler w % 4)
        const int w0 = (T / LS > 1) ? (solver_warp % (T / LS)) * LS : 0;
        if (tid >= w0 && tid < w0 + LS) {
            const int lane = tid - w0;
#ifndef HMPC_HOST_EMUL
            if (nk <= 96) {
                const unsigned FULL = 0xffffffffu;
                const int i0 = lane, i1 = lane + 32, i2 = lane + 64;
                F b0 = i0 < nk ? (F)b[i0] : (F)0, b1 = i1 < nk ? (F)b[i1] : (F)0, b2 = i2 < nk ? (F)b[i2] : (F)0;
                const F* col = Lm;                          // col[i - j] = L'(i, j)
#pragma unroll 1
                for (int j = 0; j < nk; ++j) {              // L' y = b
                    const F src = j < 32 ? b0 : (j < 64 ? b1 : b2);
                    const F t = __shfl_sync(FULL, src, j & 31);
                    if (i0 > j && i0 < nk) b0 -= col[i0 - j] * t;
                    if (i1 > j && i1 < nk) b1 -= col[i1 - j] * t;
                    if (i2 > j && i2 < nk) b2 -= col[i2 - j] * t;
                    col += nk - j;
                }
                if (i0 < nk) b0 *= dinv[i0];                // z = D^-1 y
                if (i1 < nk) b1 *= dinv[i1];
                if (i2 < nk) b2 *= dinv[i2];
                const F* r0 = Lm + (i0 < nk ? tri_off(i0, nk) - i0 : 0);   // r[j] = L'(j, i), j > i
                const F* r1 = Lm + (i1 < nk ? tri_off(i1, nk) - i1 : 0);
                const F* r2 = Lm + (i2 < nk ? tri_off(i2, nk) - i2 : 0);
#pragma unroll 1
                for (int j = nk - 1; j > 0; --j) {          // L'^T x = z
                    const F src = j < 32 ? b0 : (j < 64 ? b1 : b2);
                    const F xj = __shfl_sync(FULL, src, j & 31);
                    if (i0 < j) b0 -= r0[j] * xj;
                    if (i1 < j) b1 -= r1[j] * xj;
                    if (i2 < j) b2 -= r2[j] * xj;
                }
                if (i0 < nk) out[i0] = (double)b0;
                if (i1 < nk) out[i1] = (double)b1;
                if (i2 < nk) out[i2] = (double)b2;
            } else
#endif
            {
                for (int i = lane; i < nk; i += LS) sc[i] = (F)b[i];
                __syncwarp();
                for (int j = 0; j < nk; ++j) {            // L' y = b
                    const F t = sc[j];
                    const F* col = Lm + tri_off(j, nk) - j;
                    for (int i = j + 1 + lane; i < nk; i += LS) sc[i] -= col[i] * t;
                    __syncwarp();
                }
                for (int i = lane; i < nk; i += LS) sc[i] *= dinv[i];     // z = D^-1 y
                __syncwarp();
                for (int j = nk - 1; j > 0; --j) {        // L'^T x = z
                    const F xj = sc[j];
                    for (int i = lane; i < j; i += LS) sc[i] -= Lm[tri_off(i, nk) + (j - i)] * xj;
                    __syncwarp();
                }
                for (int i = lane; i < nk; i += LS) out[i] = (double)sc[i];
            }
        }
        __syncthreads();
        PH_ADD(5, ph_s);
    }

#ifndef HMPC_HOST_EMUL
    // --------------------------------------------------------------------------------------------
    // Tiled path (horizons N >= 11, 256-thread CTA): the same signed Cholesky  K = V S V'  as the warp kernel
    // (hmpc_warp.cuh: wfactor), in 8x8 tiles through the FP64 tensor core (mma.sync.m8n8k4.f64), with the tile rows of
    // a block column dealt to the warps of the CTA.  Storage: lower block triangle of row-major 8x8 tiles
    // (tile_off), diagonal tiles hold W_J = V(J,J)^-1.  Left-looking per block column J:
    //   phase A  every warp accumulates  C(I,J) = K(I,J) - sum_{K<J} V(I,K) S_K V(J,K)'  for its tiles I in
    //            registers; the owner of I == J factorises the diagonal tile and publishes W_J       | barrier
    //   phase B  V(I,J) = C(I,J) W_J' S_J  from the registers                                         | barrier
    // so a factorisation of order nk costs 2 nk/8 CTA barriers instead of one per pivot column, the summation runs
    // on the tensor core, and nothing is read-modify-written in the (L2-resident) factor storage.
    // --------------------------------------------------------------------------------------------
    // K(i, j) of the compact system for the tile position of this lane; i < j (above the diagonal) is never used
    __device__ __forceinline__ double entry_or_pad(const AOp& A, const double* wts, double dadd, double eps, int nk, int i, int j) const {
        if (i >= nk) return i == j ? -1.0 : 0.0;              // past the end: unit pivots (negative block)
        if (j > i) return 0.0;
        return entry(A, wts, dadd, eps, i, j);
    }
    // C(I,J) = K(I,J) - sum_{K<J} V(I,K) S_K V(J,K)'  for one tile, by one warp.  The operand tiles come from the
    // (L2-resident) factor storage: kBatch tile pairs are requested before the first product so that the latency of a
    // whole batch overlaps (measured: one pair at a time left the tensor core waiting 150-190 cycles per product).
    // Variable columns accumulate in (av0, av1), active-row columns in (ar0, ar1); the regularisation of the Schur
    // complement's diagonal sits between the two.
    static constexpr int kBatch = 6;
    __device__ __forceinline__ void tile_column(const AOp& A, const double* wts, double dadd, double eps, const double* L,
                                                int nk, int I, int J, int lane, double& c0, double& c1) const {
        const int g = lane >> 2, t = lane & 3, fo = 8 * g + 2 * t;
        const int Jb = nF >> 3;
        const bool mixed = (nF & 7) != 0;
        const int i = 8 * I + g, j0 = 8 * J + 2 * t;
        // K(I, J) first: its gather is in flight while the products run
        double k0, k1;
        if (!wts && 8 * I + 8 <= nF) {                       // variables x variables, no weights: branch-free gather
            const int vi = idx[i], va = idx[j0], vb = idx[j0 + 1];
            const int lo0 = vi < va ? vi : va, hi0 = vi < va ? va : vi, lo1 = vi < vb ? vi : vb, hi1 = vi < vb ? vb : vi;
            k0 = H[tri_off(lo0, n) + (hi0 - lo0)];
            k1 = H[tri_off(lo1, n) + (hi1 - lo1)];
            if (i == j0) k0 += dadd;
            if (i == j0 + 1) k1 += dadd;
        } else {
            k0 = entry_or_pad(A, wts, dadd, eps, nk, i, j0);
            k1 = entry_or_pad(A, wts, dadd, eps, nk, i, j0 + 1);
        }
        const double* Li = L + tile_off(I, 0) + fo;
        const double* Lj = L + tile_off(J, 0) + fo;
        const double mv0 = (8 * Jb + 2 * t < nF) ? 1.0 : 0.0, mv1 = (8 * Jb + 2 * t + 1 < nF) ? 1.0 : 0.0;
        double av0 = 0.0, av1 = 0.0, ar0 = 0.0, ar1 = 0.0;
#pragma unroll 1
        for (int K0 = 0; K0 < J; K0 += kBatch) {
            d2 a[kBatch], b[kBatch];
#pragma unroll
            for (int u = 0; u < kBatch; ++u) {
                const int K = K0 + u < J ? K0 + u : J - 1;   // clamped: a harmless repeat load past the end
                a[u] = ld2(Li + 64 * K);
                b[u] = ld2(Lj + 64 * K);
            }
#pragma unroll
            for (int u = 0; u < kBatch; ++u) {
                const int K = K0 + u;
                if (K >= J) break;
                if (K < Jb) tile_mac(av0, av1, a[u], b[u]);
                else if (K > Jb || !mixed) tile_mac(ar0, ar1, a[u], b[u]);
                else {                                       // the tile that holds both kinds of columns
                    tile_mac(av0, av1, a[u], d2{b[u].x * mv0, b[u].y * mv1});
                    tile_mac(ar0, ar1, a[u], d2{b[u].x * (1.0 - mv0), b[u].y * (1.0 - mv1)});
                }
            }
        }
        const bool scaled = (J > Jb) || (J == Jb && !mixed);  // diagonal regularised here (else inside wdiag8)
        if (I == J && scaled) {
            const bool ondiag0 = (2 * t == g), ondiag1 = (2 * t + 1 == g);
            if (ondiag0) { av0 *= 1.0 + eps; if (i >= nF && i < nk) k0 *= 1.0 + eps; }
            if (ondiag1) { av1 *= 1.0 + eps; if (i >= nF && i < nk) k1 *= 1.0 + eps; }
        }
        c0 = k0 - (av0 - ar0);
        c1 = k1 - (av1 - ar1);
    }
    __device__ inline int factor_tiled(const AOp& A, const double* wts, double dadd, double eps, double* scratch) {
        PH_T0(ph_f);
        const int tid = threadIdx.x, T = blockDim.x, nk = nF + ng, nt = (nk + 7) >> 3;
        const int lane = tid & 31, wid = tid >> 5, nw = T >> 5;
        const int g = lane >> 2, t = lane & 3, fo = 8 * g + 2 * t;
        double* L = reinterpret_cast<double*>(Lm);
        flops += flops_factor(nk);
        __syncthreads();                                                 // the previous factor is no longer in use
        int bad = 0;
#pragma unroll 1
        for (int J = 0; J < nt; ++J) {
            const int j0 = 8 * J + 2 * t;
            const double s0 = (j0 < nF) ? 1.0 : -1.0, s1 = (j0 + 1 < nF) ? 1.0 : -1.0;
            // ---- phase A: warp 0 owns the diagonal tile (its 8 sequential pivots are the long pole of the block
            // column) and only joins the others when many tile rows are left; warps 1.. share the rows below ----
            if (wid == 0) {
                double c0, c1;
                PH_T0(ph_k);
                tile_column(A, wts, dadd, eps, L, nk, J, J, lane, c0, c1);
                PH_ADD(11, ph_k);
                PH_T0(ph_d);
                st2(scratch + fo, c0, c1);
                __syncwarp();
                double* Wt = L + tile_off(J, J);
                const int jrel = nF - 8 * J;                             // first active-row pivot inside this tile
                if (jrel > 0 && jrel < 8) bad |= wdiag8<true>(scratch, Wt, jrel, 1.0, eps, lane);
                else bad |= wdiag8<false>(scratch, Wt, 0, jrel >= 8 ? 1.0 : -1.0, eps, lane);
                PH_ADD(12, ph_d);
            } else {
                for (int I = J + wid; I < nt; I += nw - 1) {             // rows J+1 .. nt-1 over warps 1 .. nw-1
                    double c0, c1;
                    tile_column(A, wts, dadd, eps, L, nk, I, J, lane, c0, c1);
                    st2(L + tile_off(I, J) + fo, c0, c1);                // C(I,J) parks where V(I,J) will live
                }
            }
            __syncthreads();
            // ---- phase B: V(I,J) = C(I,J) W_J' S_J ----
            const d2 bw = ld2(L + tile_off(J, J) + fo);
            for (int I = J + 1 + wid; I < nt; I += nw) {
                double* Tt = L + tile_off(I, J) + fo;
                double d0 = 0.0, d1 = 0.0;
                tile_mac(d0, d1, ld2(Tt), bw);
                st2(Tt, s0 * d0, s1 * d1);
            }
            __syncthreads();
        }
        bad = __syncthreads_or(bad);
        PH_ADD(4, ph_f);
        return bad;
    }

    // Substitutions with the tiled factor, column-oriented so that every step is a batch of independent
    // tile-times-vector products dealt to the warps:
    //   forward   z_J = W_J b_J,            b_I -= V(I,J) z_J   (I > J)
    //   backward  x_I = W_I' (S z)_I,       z_J -= V(I,J)' x_I  (J < I)
    // scratch: at least 8 ceil(nk / 8) doubles of shared memory.  Ends with a __syncthreads().
    __device__ inline void solve_tiled(const double* b, double* out, double* scratch) {
        PH_T0(ph_s);
        const int tid = threadIdx.x, T = blockDim.x, nk = nF + ng, nt = (nk + 7) >> 3;
        const int lane = tid & 31, wid = tid >> 5, nw = T >> 5;
        const int g = lane >> 2, t = lane & 3, fo = 8 * g + 2 * t;
        const double* L = reinterpret_cast<const double*>(Lm);
        double* v = scratch;
        flops += flops_solve(nk);
        __syncthreads();
        for (int i = tid; i < 8 * nt; i += T) v[i] = i < nk ? b[i] : 0.0;
        __syncthreads();
#pragma unroll 1
        for (int J = 0; J < nt; ++J) {
            if (wid == 0) {
                double z0 = 0.0, z1 = 0.0;
                tile_mac(z0, z1, ld2(L + tile_off(J, J) + fo), vec_b(v + 8 * J, lane));
                __syncwarp();
                if (t == 0) v[8 * J + g] = z0;
            }
            __syncthreads();
            for (int I = J + 1 + wid; I < nt; I += nw) {
                double a0 = 0.0, a1 = 0.0;
                tile_mac(a0, a1, ld2(L + tile_off(I, J) + fo), vec_b(v + 8 * J, lane));
                if (t == 0) v[8 * I + g] -= a0;
            }
            __syncthreads();
        }
        for (int i = nF + tid; i < 8 * nt; i += T) v[i] = -v[i];          // S z
        __syncthreads();
#pragma unroll 1
        for (int I = nt - 1; I >= 0; --I) {
            if (wid == 0) {
                const double* Wt = L + tile_off(I, I);
                double x0 = 0.0, x1 = 0.0;
                tile_mac(x0, x1, d2{Wt[8 * (2 * t) + g], Wt[8 * (2 * t + 1) + g]}, vec_b(v + 8 * I, lane));
                __syncwarp();
                if (t == 0) v[8 * I + g] = x0;
            }
            __syncthreads();
            for (int J = wid; J < I; J += nw) {
                const double* Tt = L + tile_off(I, J);                    // A = V(I,J)': A[g][2t + h] = T[2t + h][g]
                double a0 = 0.0, a1 = 0.0;
                tile_mac(a0, a1, d2{Tt[8 * (2 * t) + g], Tt[8 * (2 * t + 1) + g]}, vec_b(v + 8 * I, lane));
                if (t == 0) v[8 * J + g] -= a0;
            }
            __syncthreads();
        }
        for (int i = tid; i < nk; i += T) out[i] = v[i];
        __syncthreads();
        PH_ADD(5, ph_s);
    }
#endif  // HMPC_HOST_EMUL
};

// out = H x for the symmetric H of order n (packed lower triangle); every row is split into two halves
// handled by two adjacent threads when the CTA is wide enough.  Callers must __syncthreads() before reading out.
__device__ __forceinline__ double sym_at(const double* H, int n, int i, int j) {
    return i >= j ? H[tri_off(j, n) + (i - j)] : H[tri_off(i, n) + (j - i)];
}
// row i of H times x over the column range [j0, j1): the part left of the diagonal walks the packed columns
// (stride n-1-j), the part right of it is contiguous
__device__ __forceinline__ double sym_row_dot(const double* H, int n, int i, int j0, int j1, const double* x) {
    double acc = 0.0;
    const int je = j1 < i + 1 ? j1 : i + 1;
    int off = tri_off(j0, n) - j0;
    for (int j = j0; j < je; ++j) { acc += H[off + i] * x[j]; off += n - 1 - j; }
    const double* row = H + tri_off(i, n) - i;
    for (int j = (j0 > i + 1 ? j0 : i + 1); j < j1; ++j) acc += row[j] * x[j];
    return acc;
}
template <class Sys>
__device__ inline void sym_matvec(const double* H, int n, const double* x, double* out, Sys* acct) {
    if (acct) acct->flops += flops_matvec(n);
    const int tid = threadIdx.x, T = blockDim.x;
    if (T >= 2 * n) {
        const int i = tid >> 1, h = tid & 1;
        double acc = 0.0;
        if (i < n) acc = sym_row_dot(H, n, i, h ? (n >> 1) : 0, h ? n : (n >> 1), x);
#ifndef HMPC_HOST_EMUL
        acc += __shfl_xor_sync(0xffffffffu, acc, 1);
#endif
        if (i < n && h == 0) out[i] = acc;
    } else {
        for (int i = tid; i < n; i += T) out[i] = sym_row_dot(H, n, i, 0, n, x);
    }
}

struct SolveInfo { int status, iters, nfac, path; double rho; };


// ------------------------------------------------------------------------------------------------
// Verified primal-dual active-set refinement (numpy statement: oracle/device_port.py polish_verified).
//
// w.code holds the active-set guess, w.xp the starting point.  Box-active and a-priori fixed variables
// are pinned exactly; the active friction / height rows G enter the quasi-definite KKT system
// [[H_FF, G'],[G, -eps I]], factorised once per trial and applied in correction form (iterative
// refinement removes the eps perturbation) until the residuals stagnate.  The KKT conditions of the
// ORIGINAL QP are then checked: stationarity on free variables, feasibility of every row, equality on
// active rows, sign of every multiplier.  All satisfied -> accept (exact optimum).  Otherwise rows
// whose multiplier has the wrong sign are released, violated rows are activated, and the trial is
// repeated, at most c.retries times.
// On success: w.x <- solution, w.mv[0] <- multipliers, w.code <- active set; returns 1 (all threads).
// ------------------------------------------------------------------------------------------------
template <class Sys>
__device__ inline int polish_verified(const QpConst& c, Work& w, Sys& sys, const AOp& A, SolveInfo& info) {
    const int N = c.N, n = 6 * N, m = 11 * N, tid = threadIdx.x, T = blockDim.x;
    const double tol = c.polish_tol;
    double* mul = w.mv[0];
    double* bnd = w.mv[1];
    for (int r = tid; r < m; r += T) {
        int cd = w.code[r];
        if (cd > 0 && w.hi[r] > kInfThresh) cd = 0;
        if (cd < 0 && w.lo[r] < -kInfThresh) cd = 0;
        if (r < n && w.fixed[r]) cd = 0;
        w.code[r] = (int8_t)cd;
    }
    __syncthreads();
    for (int trial = 0; trial <= c.retries; ++trial) {
        for (int r = tid; r < m; r += T) {
            const int cd = w.code[r];
            bnd[r] = cd < 0 ? w.lo[r] : w.hi[r];
            mul[r] = 0.0;
            if (r < n) {
                const int pin = (w.fixed[r] || cd != 0) ? 1 : 0;
                w.pin[r] = (int8_t)pin;
                if (pin) w.xp[r] = w.fixed[r] ? 0.0 : bnd[r];
            }
        }
        __syncthreads();
        compact_indices(0, n, n, w.idx, w.cnt + 0, [&](int i) { return w.pin[i] == 0; });
        compact_indices(n, m - n, kkt_max(N), w.grow, w.cnt + 1, [&](int r) { return w.code[r] != 0; });
        __syncthreads();
        const int nF = w.cnt[0], ng = w.cnt[1], nk = nF + ng;
        if (nk > kkt_max(N)) return 0;
        sys.nF = nF; sys.ng = ng;
        ++info.nfac;
        if (sys.factor(A, nullptr, 0.0, c.kkt_eps, w.tmp)) return 0;
        PH_T0(ph_rf);
        double prev = 1e300;
        bool hx_current = false;     // w.tmp == H xp for the final xp (the loop left right after a residual)
        for (int k = 0; k < c.max_refine; ++k) {
            sym_matvec(w.H, n, w.xp, w.tmp, &sys);
            __syncthreads();   // tmp is read through the compact index below (another thread's entry)
            double v[2] = {0.0, 0.0};   // residual; largest residual relative to the terms it is the difference of
            for (int i = tid; i < nk; i += T) {
                double r_, mag;
                if (i < nF) {
                    const int vi = w.idx[i];
                    const double aty = A.colT(vi, mul);
                    r_ = -(w.tmp[vi] + w.g[vi] + aty);
                    mag = fabs(w.tmp[vi]) + fabs(w.g[vi]) + fabs(aty);
                } else {
                    const int rr = w.grow[i - nF];
                    const double ax = A.row(rr, w.xp);
                    r_ = bnd[rr] - ax;
                    mag = fabs(bnd[rr]) + fabs(ax);
                }
                w.rhs[i] = r_;
                v[0] = fmax(v[0], fabs(r_));
                v[1] = fmax(v[1], fabs(r_) / (mag + 1e-300));
            }
            block_reduce<2, 0>(v, w.red);
            if (!(v[0] == v[0])) return 0;
            // stop when every row's residual sits at its rounding level or the residual has stopped contracting
            // Without active general rows the system is exactly H_FF (no regularisation): an FP64 solve that
            // took the residual down by 1e7 is already at working accuracy (error ~ cond * eps), stop there.
            if (k == 1 && ng == 0 && sizeof(typename Sys::real) == 8 && v[0] <= 1e-7 * prev) { hx_current = true; break; }
            if (k >= 1 && (v[1] <= 1e-12 || (k >= 2 && v[0] > c.stagnation * prev))) { hx_current = true; break; }
            prev = v[0];
            sys.solve(w.rhs, w.xt, w.sc);
            for (int i = tid; i < nk; i += T) {
                if (i < nF) w.xp[w.idx[i]] += w.xt[i];
                else mul[w.grow[i - nF]] += w.xt[i];
            }
            __syncthreads();
        }
        PH_ADD(6, ph_rf);
        PH_T0(ph_v);
        // ---- pass 1: multipliers of pinned variables, scales ----
        if (!hx_current) {
            sym_matvec(w.H, n, w.xp, w.tmp, &sys);
            __syncthreads();
        }
        double v[3] = {0, 0, 0};   // stat, scale, |mult|
        for (int i = tid; i < n; i += T) {
            const double aty = A.colT(i, mul);   // mul[i] == 0 on box rows at this point
            const double G = w.tmp[i] + w.g[i] + aty;
            v[1] = fmax(v[1], fmax(fabs(w.tmp[i]), fmax(fabs(w.g[i]), fabs(aty))));
            if (!w.pin[i]) v[0] = fmax(v[0], fabs(G));
            else { w.sc[i] = -G; v[2] = fmax(v[2], fabs(G)); }
        }
        for (int r = n + tid; r < m; r += T) if (w.code[r]) v[2] = fmax(v[2], fabs(mul[r]));
        block_reduce<3, 0>(v, w.red);
        for (int i = tid; i < n; i += T) mul[i] = w.pin[i] ? w.sc[i] : 0.0;
        __syncthreads();
        const double scale = fmax(1.0, v[1]);
        const double stol = tol * fmax(scale, v[2]);
        // ---- pass 2: per-row verdicts and the refined active set ----
        // Rows whose multiplier has the wrong sign are released first; violated rows are only activated by
        // a trial that had no wrong-signed row (measured: fewer trials and fewer give-ups than doing both at
        // once).  w.side (interior-point scratch) holds the proposed change: 1 release, 2 / 3 activate lower / upper.
        int bad = (v[0] <= 1e-10 * scale) ? 0 : 1, anywrong = 0;
        // v[] comes out of a block reduction: every thread sees the same value, no second reduction needed
        const bool nonfinite = !(v[0] == v[0]) || !(v[2] == v[2]);
        if (nonfinite) bad = 1;
        for (int r = tid; r < m; r += T) {
            const double ax = A.row(r, w.xp), lo = w.lo[r], hi = w.hi[r];
            const int cd = w.code[r];
            const bool apriori = (r < n) && w.fixed[r];
            int change = 0;
            if (cd != 0) {
                const double lam = mul[r];
                if ((cd > 0 && lam < -stol) || (cd < 0 && lam > stol)) { change = 1; bad |= 1; anywrong = 1; }
                if (r >= n && fabs(ax - bnd[r]) > tol * (1.0 + fabs(bnd[r]))) bad |= 1;   // singular / inconsistent set
            } else if (!apriori) {
                if (lo - ax > tol * (1.0 + fabs(lo))) { change = 2; bad |= 1; }
                else if (ax - hi > tol * (1.0 + fabs(hi))) { change = 3; bad |= 1; }
            }
            w.side[r] = (int8_t)change;
        }
        bad = __syncthreads_or(bad);
        anywrong = __syncthreads_or(anywrong);
        if (!bad) {
            for (int i = tid; i < n; i += T) w.x[i] = w.xp[i];
            for (int r = n + tid; r < m; r += T) if (!w.code[r]) mul[r] = 0.0;
            __syncthreads();
            return 1;
        }
        int changed = 0;
        for (int r = tid; r < m; r += T) {
            const int change = w.side[r];
            if (change == 1) { w.code[r] = 0; changed = 1; }
            else if (change >= 2 && !anywrong) { w.code[r] = (int8_t)(change == 2 ? -1 : 1); changed = 1; }
        }
        changed = __syncthreads_or(changed);
        PH_ADD(7, ph_v);
        if (!changed || nonfinite) return 0;
    }
    return 0;
}

// ------------------------------------------------------------------------------------------------
// Mehrotra predictor-corrector interior point in the fixed row layout (numpy statement:
// oracle/device_port.py ipm_solve).  Every row keeps an upper and a lower slack / multiplier pair;
// sides at +-inf, rows of a-priori fixed variables and height rows without a free variable are masked.
// Start: one Newton step of the quadratic penalty towards the row mid-points.
// On exit w.x = iterate, w.code = active-set estimate (lambda > slack).  Returns 1 when converged.
// ------------------------------------------------------------------------------------------------
template <class Sys>
__device__ inline int ipm_solve_body(const QpConst& c, Work& w, Sys& sys, const AOp& A, SolveInfo& info) {
    const int N = c.N, n = 6 * N, m = 11 * N, tid = threadIdx.x, T = blockDim.x;
    double *su = w.mv[0], *sl = w.mv[1], *lu = w.mv[2], *ll = w.mv[3], *rpu = w.mv[4], *rpl = w.mv[5];
    double *pu = w.mv[6], *pl = w.mv[7], *tv = w.mv[8], *adx = w.mv[9], *wts = w.mv[10];
    const double s0 = 0.1;
    PH_T0(ph_i);
    // ---- sides ----
    double cntv[1] = {0.0};
    for (int r = tid; r < m; r += T) {
        int s = 0;
        bool on = true;
        if (r < n) on = !w.fixed[r];
        else if (r >= n + 4 * N) {
            const int k = r - n - 4 * N;
            on = false;
            for (int j = 0; j + 2 <= k; ++j) on = on || (w.stance[j] != 0);
        }
        if (on) {
            if (w.hi[r] < kInfThresh) s |= 1;
            if (w.lo[r] > -kInfThresh) s |= 2;
        }
        w.side[r] = (int8_t)s;
        cntv[0] += (double)((s & 1) + ((s >> 1) & 1));
    }
    block_reduce<1, 2>(cntv, w.red);
    const double ni = cntv[0];
    compact_indices(0, n, n, w.idx, w.cnt + 0, [&](int i) { return w.fixed[i] == 0; });
    for (int i = tid; i < n; i += T) { w.x[i] = 0.0; w.xt[i] = 0.0; }
    __syncthreads();
    const int nF = w.cnt[0];
    sys.nF = nF; sys.ng = 0;
    // ---- start: minimise  1/2 x'Hx + g'x + 1/2 sum_r (a_r x - mid_r)^2  over the free variables ----
    for (int r = tid; r < m; r += T) {
        const int s = w.side[r];
        const double lo = w.lo[r], hi = w.hi[r];
        const double mid = (s == 3) ? 0.5 * (lo + hi) : (s == 1 ? hi - 1.0 : (s == 2 ? lo + 1.0 : 0.0));
        wts[r] = s ? 1.0 : 0.0;
        tv[r] = s ? -mid : 0.0;     // w0 (a_r x - mid) at x = 0
        w.code[r] = 0;
    }
    __syncthreads();
    ++info.nfac;
    // N <= 10 kernels with the tiled factor switched on by ipm_solve(): one 64-double tile of scratch (w.sc is free here)
    double* fscr = (sys.tiled && n <= 64) ? w.sc : w.tmp;
    if (sys.factor(A, ni > 0.0 ? wts : nullptr, 0.0, 0.0, fscr)) return 0;
    for (int i = tid; i < nF; i += T) { const int vi = w.idx[i]; w.rhs[i] = -w.g[vi] - (ni > 0.0 ? A.colT(vi, tv) : 0.0); }
    sys.solve(w.rhs, w.rhs, w.sc);
    for (int i = tid; i < nF; i += T) w.x[w.idx[i]] = w.rhs[i];
    __syncthreads();
    if (!(ni > 0.0)) return 1;   // no inequality at all: the Newton step is the optimum
    double mn[1] = {1e300};
    for (int r = tid; r < m; r += T) {
        const int s = w.side[r];
        const double ax = A.row(r, w.x);
        const double a = (s & 1) ? w.hi[r] - ax : 1.0, b = (s & 2) ? ax - w.lo[r] : 1.0;
        su[r] = a; sl[r] = b;
        if (s & 1) mn[0] = fmin(mn[0], a);
        if (s & 2) mn[0] = fmin(mn[0], b);
    }
    block_reduce<1, 1>(mn, w.red);
    const double shift = fmax(0.0, -1.5 * mn[0]);
    double gsv[1] = {0.0};
    for (int i = tid; i < n; i += T) gsv[0] = fmax(gsv[0], fabs(w.g[i]));
    for (int r = tid; r < m; r += T) {
        const int s = w.side[r];
        su[r] = fmax(su[r] + shift, s0); sl[r] = fmax(sl[r] + shift, s0);
        lu[r] = (s & 1) ? s0 : 0.0; ll[r] = (s & 2) ? s0 : 0.0;
    }
    block_reduce<1, 0>(gsv, w.red);
    const double gs = fmax(1.0, gsv[0]);
    int conv = 0;
    for (int it = 0; it <= c.ipm_max_iter; ++it) {
        // ---- residuals ----
        sym_matvec(w.H, n, w.x, w.tmp, &sys);
        for (int r = tid; r < m; r += T) tv[r] = lu[r] - ll[r];
        __syncthreads();
        double v[2] = {0.0, 0.0};
        double sm[1] = {0.0};
        for (int i = tid; i < nF; i += T) {
            const int vi = w.idx[i];
            const double rd = w.tmp[vi] + w.g[vi] + A.colT(vi, tv);
            w.xp[vi] = rd;                       // rd kept in xp (full index)
            v[0] = fmax(v[0], fabs(rd));
        }
        for (int r = tid; r < m; r += T) {
            const int s = w.side[r];
            const double ax = A.row(r, w.x);
            const double a = (s & 1) ? ax + su[r] - w.hi[r] : 0.0;
            const double b = (s & 2) ? -ax + sl[r] + w.lo[r] : 0.0;
            rpu[r] = a; rpl[r] = b;
            v[1] = fmax(v[1], fmax(fabs(a), fabs(b)));
            if (s & 1) sm[0] += su[r] * lu[r];
            if (s & 2) sm[0] += sl[r] * ll[r];
        }
        block_reduce<2, 0>(v, w.red);
        block_reduce<1, 2>(sm, w.red);
        const double mu = sm[0] / ni;
        if (!(mu == mu) || !(v[0] == v[0]) || !(v[1] == v[1])) break;
        if (v[0] < c.ipm_tol * gs && v[1] < c.ipm_tol && mu < c.ipm_tol) { conv = 1; break; }
        if (it == c.ipm_max_iter) break;
        info.iters = it + 1;
        // ---- factor  H + A' diag(lambda/s) A ----
        for (int r = tid; r < m; r += T) {
            const int s = w.side[r];
            wts[r] = ((s & 1) ? lu[r] / su[r] : 0.0) + ((s & 2) ? ll[r] / sl[r] : 0.0);
        }
        __syncthreads();
        ++info.nfac;
        if (sys.factor(A, wts, 0.0, 0.0, fscr)) break;
        double alpha = 1.0, sigmu = 0.0;
        for (int phase = 0; phase < 2; ++phase) {
            // complementarity targets: predictor rc = s*lam ; corrector rc = s*lam + ds*dlam - sigma*mu
            for (int r = tid; r < m; r += T) {
                const int s = w.side[r];
                double tu = 0.0, tl = 0.0;
                if (s & 1) { const double rc = su[r] * lu[r] + (phase ? pu[r] - sigmu : 0.0); tu = (lu[r] * rpu[r] - rc) / su[r]; }
                if (s & 2) { const double rc = sl[r] * ll[r] + (phase ? pl[r] - sigmu : 0.0); tl = (ll[r] * rpl[r] - rc) / sl[r]; }
                tv[r] = tu - tl;
            }
            __syncthreads();
            for (int i = tid; i < nF; i += T) { const int vi = w.idx[i]; w.rhs[i] = -w.xp[vi] - A.colT(vi, tv); }
            sys.solve(w.rhs, w.rhs, w.sc);
            for (int i = tid; i < nF; i += T) w.xt[w.idx[i]] = w.rhs[i];
            for (int i = tid; i < n; i += T) if (w.fixed[i]) w.xt[i] = 0.0;   // xt doubles as factor scratch
            __syncthreads();
            double rmin[1] = {1.0};
            for (int r = tid; r < m; r += T) {
                const int s = w.side[r];
                const double ad = A.row(r, w.xt);
                adx[r] = ad;
                if (s & 1) {
                    const double rc = su[r] * lu[r] + (phase ? pu[r] - sigmu : 0.0);
                    const double ds = -rpu[r] - ad, dl = -(rc + lu[r] * ds) / su[r];
                    if (ds < 0.0) rmin[0] = fmin(rmin[0], -su[r] / ds);
                    if (dl < 0.0) rmin[0] = fmin(rmin[0], -lu[r] / dl);
                }
                if (s & 2) {
                    const double rc = sl[r] * ll[r] + (phase ? pl[r] - sigmu : 0.0);
                    const double ds = -rpl[r] + ad, dl = -(rc + ll[r] * ds) / sl[r];
                    if (ds < 0.0) rmin[0] = fmin(rmin[0], -sl[r] / ds);
                    if (dl < 0.0) rmin[0] = fmin(rmin[0], -ll[r] / dl);
                }
            }
            block_reduce<1, 1>(rmin, w.red);
            if (phase == 0) {
                const double a = rmin[0];
                double ma[1] = {0.0};
                for (int r = tid; r < m; r += T) {
                    const int s = w.side[r];
                    const double ad = adx[r];
                    if (s & 1) {
                        const double ds = -rpu[r] - ad, dl = -(su[r] * lu[r] + lu[r] * ds) / su[r];
                        pu[r] = ds * dl;
                        ma[0] += (su[r] + a * ds) * (lu[r] + a * dl);
                    }
                    if (s & 2) {
                        const double ds = -rpl[r] + ad, dl = -(sl[r] * ll[r] + ll[r] * ds) / sl[r];
                        pl[r] = ds * dl;
                        ma[0] += (sl[r] + a * ds) * (ll[r] + a * dl);
                    }
                }
                block_reduce<1, 2>(ma, w.red);
                const double ratio = (ma[0] / ni) / mu;
                sigmu = ratio * ratio * ratio * mu;
            } else {
                alpha = fmin(1.0, 0.99 * rmin[0]);
            }
        }
        // ---- step ----
        for (int r = tid; r < m; r += T) {
            const int s = w.side[r];
            const double ad = adx[r];
            if (s & 1) {
                const double rc = su[r] * lu[r] + pu[r] - sigmu;
                const double ds = -rpu[r] - ad, dl = -(rc + lu[r] * ds) / su[r];
                su[r] += alpha * ds; lu[r] += alpha * dl;
            }
            if (s & 2) {
                const double rc = sl[r] * ll[r] + pl[r] - sigmu;
                const double ds = -rpl[r] + ad, dl = -(rc + ll[r] * ds) / sl[r];
                sl[r] += alpha * ds; ll[r] += alpha * dl;
            }
        }
        for (int i = tid; i < nF; i += T) { const int vi = w.idx[i]; w.x[vi] += alpha * w.xt[vi]; }
        __syncthreads();
    }
    for (int r = tid; r < m; r += T) {
        const int s = w.side[r];
        w.code[r] = ((s & 1) && lu[r] > su[r]) ? 1 : (((s & 2) && ll[r] > sl[r]) ? -1 : 0);
    }
    __syncthreads();
    PH_ADD(8, ph_i);
    return conv;
}

// ------------------------------------------------------------------------------------------------
// Default solver: warm-started verified active-set refinement, interior-point fallback, verified polish.
// On entry (warm != 0): w.xp = time-shifted previous solution, w.code = time-shifted previous active set.
// On exit: w.x = solution, w.code = active set (for the next tick's warm start).
// ------------------------------------------------------------------------------------------------
// Interior point with the factorisation switched to tensor-core tiles where the system allows it.  The Newton system
// H + A'WA over the free variables is positive definite and of order <= 6N: at N <= 10 it fits the packed factor
// storage as 8x8 tiles, so the factorisation and both substitutions of every iteration run through
// LinSys::factor_tiled / solve_tiled with all warps of the CTA instead of the packed right-looking LDL' and its one-warp
// substitution.  That halves the latency of an interior-point solve but costs throughput when every CTA of the SM is
// in its interior point at once (measured: deferred list of <= one hopper per CTA 1.0 -> 0.5 ms, batch 4096 2.77 ->
// 3.07 M steps/s; first tick of 131072 hoppers 184 -> 300 ms), so the kernel allows it (sys.ipm_tiled) only for a
// deferral list no longer than its grid.  The polish that follows (order up to 7N + 2) uses the packed layout again.
template <class Sys>
__device__ inline int ipm_solve(const QpConst& c, Work& w, Sys& sys, const AOp& A, SolveInfo& info) {
    const int keep = sys.tiled;
#ifndef HMPC_HOST_EMUL
    {
        const int N = c.N, nt = (6 * N + 7) >> 3, kk = kkt_max(N);
        if (sizeof(typename Sys::real) == 8 && sys.ipm_tiled && !sys.tiled && blockDim.x >= 64 && kkt_vec(N) >= 64 &&
            nt * (nt + 1) / 2 * 64 <= kk * (kk + 1) / 2)
            sys.tiled = 1;
    }
#endif
    const int conv = ipm_solve_body(c, w, sys, A, info);
    sys.tiled = keep;
    return conv;
}

template <class Sys>
__device__ inline SolveInfo solve_exact(const QpConst& c, Work& w, Sys& sys, const AOp& A, int warm) {
    const int n = 6 * c.N, tid = threadIdx.x, T = blockDim.x;
    SolveInfo info{ST_MAX_ITER, 0, 0, PATH_NONE, 0.0};
    if (warm) {
        if (polish_verified(c, w, sys, A, info)) { info.status = ST_SOLVED; info.path = PATH_WARM; return info; }
        __syncthreads();
    }
    const int conv = ipm_solve(c, w, sys, A, info);
    int nonfinite = 0;
    for (int i = tid; i < n; i += T) {
        const double v = w.x[i];
        if (!(fabs(v) < 1e300)) nonfinite = 1;
        w.xp[i] = v;
    }
    nonfinite = __syncthreads_or(nonfinite);
    if (nonfinite) {
        for (int i = tid; i < n; i += T) w.x[i] = 0.0;
        __syncthreads();
        info.status = ST_NON_FINITE; info.path = PATH_IPM;
        return info;
    }
    if (polish_verified(c, w, sys, A, info)) { info.status = ST_SOLVED; info.path = PATH_IPM_POLISH; return info; }
    info.status = conv ? ST_INEXACT : ST_MAX_ITER;
    info.path = PATH_IPM;
    return info;
}

// ------------------------------------------------------------------------------------------------
// ADMM (OSQP iteration, SURVEY App. C2, dense condensed form, no Ruiz scaling; numpy statement:
// oracle/device_port.py admm_solve):
//     x~ = K^-1 (sigma x - g + A'(rho z - y)),  K = H + sigma I + A' diag(rho) A   (free variables only)
//     x+ = alpha x~ + (1-alpha) x ;  z+ = clip(alpha A x~ + (1-alpha) z + y/rho) ;  y+ = y + rho (.. - z+)
// mode FIXED_ITER: exactly max_iter iterations, no checks.  mode EARLY_EXIT: OSQP's residual test every
// c.check iterations after c.first_check, rho re-balanced (and K re-factorised) when it moves by > 5x.
// On entry w.x / w.mv[2] hold the warm start (x, y) or zeros.  On exit w.x, w.mv[2] = (x, y) and
// w.code = OSQP's polish guess of the active set.
// ------------------------------------------------------------------------------------------------
template <class Sys>
__device__ inline SolveInfo admm_solve(const QpConst& c, Work& w, Sys& sys, const AOp& A) {
    const int N = c.N, n = 6 * N, m = 11 * N, tid = threadIdx.x, T = blockDim.x;
    SolveInfo info{ST_MAX_ITER, 0, 0, PATH_ADMM, c.rho0};
    double *rv = w.mv[0], *z = w.mv[1], *y = w.mv[2], *wv = w.mv[3];
    double rho = c.rho0;
    const double sigma = c.sigma, alpha = c.alpha;
    auto set_rho = [&](double r) {
        for (int i = tid; i < m; i += T) {
            const double lo = w.lo[i], hi = w.hi[i];
            double v = r;
            if (lo < -kInfThresh && hi > kInfThresh) v = kRhoMin;
            else if (hi - lo < 1e-4) v = fmin(1e3 * r, kRhoMax);
            rv[i] = v;
        }
        __syncthreads();
    };
    set_rho(rho);
    compact_indices(0, n, n, w.idx, w.cnt + 0, [&](int i) { return w.fixed[i] == 0; });
    for (int i = tid; i < n; i += T) {
        const double v = w.fixed[i] ? 0.0 : w.x[i];
        w.x[i] = fmin(fmax(v, w.lo[i]), w.hi[i]);
        w.xt[i] = 0.0;
    }
    __syncthreads();
    const int nF = w.cnt[0];
    sys.nF = nF; sys.ng = 0;
    for (int r = tid; r < m; r += T) z[r] = A.row(r, w.x);     // OSQP: z = A x at a (warm or cold) start, no projection
    __syncthreads();
    info.nfac = 1;
    // N <= 10 kernels: the ADMM system (free variables only, order nF <= 6N, positive definite) fits the packed factor
    // storage as 8x8 tiles, so the factorisation and -- every iteration -- the substitutions run on the FP64 tensor
    // core with all warps of the CTA (factor_tiled / solve_tiled) instead of the one-warp substitution chain
    // (profiles/README.md: 18 k cycles per solve).  The polish that follows uses the packed layout again.
    const int tiled_keep = sys.tiled;
    double* fscr = w.tmp;
#ifndef HMPC_HOST_EMUL
    {
        const int nt = (nF + 7) >> 3, kk = kkt_max(N);
        if (sizeof(typename Sys::real) == 8 && !sys.tiled && T >= 64 && kkt_vec(N) >= 64 && nt * (nt + 1) / 2 * 64 <= kk * (kk + 1) / 2) {
            sys.tiled = 1;
            fscr = w.xt;            // one 64-double tile of scratch; xt is dead while a factorisation runs
        }
    }
#endif
    if (sys.factor(A, rv, sigma, 0.0, fscr)) { sys.tiled = tiled_keep; info.status = ST_NON_FINITE; return info; }
    const int last_it = c.max_iter;
    int next_check = (c.mode == 1) ? last_it : min(c.first_check, last_it);
    for (int it = 1; it <= last_it; ++it) {
        for (int r = tid; r < m; r += T) wv[r] = rv[r] * z[r] - y[r];
        __syncthreads();
        for (int i = tid; i < nF; i += T) { const int vi = w.idx[i]; w.rhs[i] = sigma * w.x[vi] - w.g[vi] + A.colT(vi, wv); }
        sys.solve(w.rhs, w.rhs, w.sc);
        for (int i = tid; i < nF; i += T) w.xt[w.idx[i]] = w.rhs[i];
        for (int i = tid; i < n; i += T) if (w.fixed[i]) w.xt[i] = 0.0;       // xt doubles as factor scratch
        __syncthreads();
        for (int r = tid; r < m; r += T) {
            const double zt = A.row(r, w.xt);
            const double zr = alpha * zt + (1.0 - alpha) * z[r];
            const double rr = rv[r];
            const double zn = fmin(fmax(zr + y[r] / rr, w.lo[r]), w.hi[r]);
            y[r] += rr * (zr - zn);
            z[r] = zn;
        }
        for (int i = tid; i < n; i += T) w.x[i] = alpha * w.xt[i] + (1.0 - alpha) * w.x[i];
        __syncthreads();
        info.iters = it;
        if (it != next_check && it != last_it) continue;
        next_check = it + c.check;
        // ---- residuals of the unscaled problem (OSQP termination test, SURVEY App. C2) ----
        sym_matvec(w.H, n, w.x, w.tmp, &sys);
        __syncthreads();
        double v[6] = {0, 0, 0, 0, 0, 0};   // pri, npri, dua, |Hx|, |A'y|, |g|
        for (int r = tid; r < m; r += T) {
            const double ax = A.row(r, w.x);
            v[0] = fmax(v[0], fabs(ax - z[r]));
            v[1] = fmax(v[1], fmax(fabs(ax), fabs(z[r])));
        }
        for (int i = tid; i < n; i += T) {
            if (w.fixed[i]) continue;   // eliminated variables carry an implicit multiplier
            const double aty = A.colT(i, y);
            v[2] = fmax(v[2], fabs(w.tmp[i] + w.g[i] + aty));
            v[3] = fmax(v[3], fabs(w.tmp[i]));
            v[4] = fmax(v[4], fabs(aty));
            v[5] = fmax(v[5], fabs(w.g[i]));
        }
        block_reduce<6, 0>(v, w.red);
        const double pri = v[0], npri = v[1], dua = v[2], ndua = fmax(v[3], fmax(v[4], v[5]));
        if (!(pri == pri) || !(dua == dua)) { info.status = ST_NON_FINITE; break; }
        if (c.mode == 1) break;
        if (pri <= c.eps_abs + c.eps_rel * npri && dua <= c.eps_abs + c.eps_rel * ndua) { info.status = ST_INEXACT; break; }
        if (it == last_it) break;
        if (c.adaptive_rho) {
            double rn = rho * sqrt((pri / fmax(npri, 1e-10)) / fmax(dua / fmax(ndua, 1e-10), 1e-10));
            rn = fmin(fmax(rn, kRhoMin), kRhoMax);
            if (rn > 5.0 * rho || rn < 0.2 * rho) {
                rho = rn;
                set_rho(rho);
                ++info.nfac;
                if (sys.factor(A, rv, sigma, 0.0, fscr)) { info.status = ST_NON_FINITE; break; }
            }
        }
    }
    sys.tiled = tiled_keep;
    for (int r = tid; r < m; r += T) {
        const double zz = z[r], yy = y[r];
        w.code[r] = ((zz - w.lo[r]) < -yy) ? -1 : (((w.hi[r] - zz) < yy) ? 1 : 0);
    }
    __syncthreads();
    info.rho = rho;
    return info;
}

}  // namespace hmpc
