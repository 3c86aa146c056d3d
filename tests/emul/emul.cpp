// tests/emul/emul.cpp -- TEST INFRASTRUCTURE.  Compiles the product's device source
// (hopper_mpc_inertial_b200/csrc/hmpc_{sim,qp,mpc}.cuh) with g++ and runs it as ONE serial thread per
// hopper, so that the CPU test-suite (no GPU in the build container) exercises the very code the CUDA
// kernels execute: arithmetic, control flow, indexing.  It cannot see races or barrier bugs -- those
// are covered by the -m gpu tests and compute-sanitizer runs on the GPU box.  Never shipped, never
// loaded by the product package.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <ucontext.h>
#include <functional>
#include <vector>

#include "cuda_runtime.h"   // tests/emul/fake_cuda
#include "../../hopper_mpc_inertial_b200/csrc/hmpc_sim.cuh"
#include "../../hopper_mpc_inertial_b200/csrc/hmpc_mpc.cuh"
#include "../../hopper_mpc_inertial_b200/csrc/hmpc_warp.cuh"
#include "../../hopper_mpc_inertial_b200/csrc/hmpc_geometry.cuh"
#include "../../hopper_mpc_inertial_b200/csrc/hmpc_plan.cuh"

using namespace hmpc;

// ---- 32-lane warp emulation: cooperative fibers that meet at every warp-synchronous primitive ----
int hmpc_emul_tid = 0, hmpc_emul_bdim = 1;
double hmpc_emul_xd[32], hmpc_emul_ma[32], hmpc_emul_mb[32];
long long hmpc_emul_xi[32];
long long hmpc_emul_count[8];

namespace {
constexpr int NL = 32;
constexpr size_t kStack = 512 * 1024;
ucontext_t g_main, g_ctx[NL];
std::vector<char> g_stack[NL];
bool g_done[NL];
int g_arrived = 0, g_live = 0;
unsigned long g_gen = 0;
std::function<void(int)> g_body;

void fiber_switch_from(int me) {
    int next = me;
    for (int t = 1; t <= NL; ++t) {
        const int cand = (me + t) % NL;
        if (!g_done[cand]) { next = cand; break; }
    }
    if (next == me) return;
    hmpc_emul_tid = next;
    swapcontext(&g_ctx[me], &g_ctx[next]);
    hmpc_emul_tid = me;
}

void fiber_entry(int lane) {
    g_body(lane);
    g_done[lane] = true;
    --g_live;
    if (g_live == 0) { setcontext(&g_main); }
    for (int t = 1; t <= NL; ++t) {
        const int cand = (lane + t) % NL;
        if (!g_done[cand]) { hmpc_emul_tid = cand; setcontext(&g_ctx[cand]); }
    }
    abort();
}

void run_warp(const std::function<void(int)>& body) {
    g_body = body;
    g_arrived = 0; g_live = NL;
    for (int l = 0; l < NL; ++l) {
        if (g_stack[l].empty()) g_stack[l].resize(kStack);
        g_done[l] = false;
        getcontext(&g_ctx[l]);
        g_ctx[l].uc_stack.ss_sp = g_stack[l].data();
        g_ctx[l].uc_stack.ss_size = kStack;
        g_ctx[l].uc_link = nullptr;
        makecontext(&g_ctx[l], (void (*)())fiber_entry, 1, l);
    }
    hmpc_emul_bdim = NL;
    hmpc_emul_tid = 0;
    swapcontext(&g_main, &g_ctx[0]);
    hmpc_emul_bdim = 1;
    hmpc_emul_tid = 0;
}
}  // namespace

void hmpc_emul_rendezvous() {
    const unsigned long gen = g_gen;
    if (++g_arrived == NL) { g_arrived = 0; ++g_gen; return; }
    long spins = 0;
    while (g_gen == gen) {
        if (g_live < NL || ++spins > 100000) {
            fprintf(stderr, "hmpc emul: warp deadlock (a lane skipped a warp-synchronous primitive or returned early)\n");
            abort();
        }
        fiber_switch_from(hmpc_emul_tid);
    }
}

static QpConst qp_const(const hmpc_config& cfg) {
    QpConst c;
    c.N = cfg.N; c.dyn = cfg.dyn; c.uref_mode = cfg.uref_mode; c.solver = cfg.solver; c.mode = cfg.mode;
    c.max_iter = cfg.max_iter; c.check = cfg.check_interval; c.first_check = cfg.first_check;
    c.retries = cfg.polish_retries; c.adaptive_rho = cfg.adaptive_rho; c.warm_start = cfg.warm_start;
    c.polish = cfg.polish; c.ipm_max_iter = cfg.ipm_max_iter; c.sqp_sweeps = cfg.sqp_sweeps > 1 ? cfg.sqp_sweeps : 1;
    c.dt = cfg.mpc_dt; c.m = cfg.m; c.g = cfg.g; c.mu = cfg.mu;
    for (int i = 0; i < 9; ++i) c.Jinv[i] = cfg.Jinv[i];
    for (int i = 0; i < 3; ++i) { c.rh[i] = cfg.rh[i]; c.tau_max[i] = cfg.tau_max[i]; }
    c.fz_max = cfg.fz_max; c.z_min = cfg.z_min; c.kf = cfg.kf;
    c.eps_abs = cfg.eps_abs; c.eps_rel = cfg.eps_rel; c.rho0 = cfg.rho0; c.sigma = cfg.sigma;
    c.alpha = cfg.alpha; c.kkt_eps = cfg.kkt_eps; c.polish_tol = cfg.polish_tol; c.ipm_tol = cfg.ipm_tol;
    c.condense_flops = hmpc::flops_condense(cfg.N);
    c.work_mul = 1; c.work_add = 0; c.work_order = nullptr;
    c.max_refine = 6;
    c.stagnation = 0.25;
    if (cfg.precision == HMPC_FP32) {
        c.max_refine = 14;
        c.stagnation = 0.7;
        c.kkt_eps = cfg.kkt_eps > 1e-3 ? cfg.kkt_eps : 1e-3;
        c.ipm_tol = cfg.ipm_tol > 1e-6 ? cfg.ipm_tol : 1e-6;
    }
    return c;
}

static int g_emul_warp_done = 0;
// warm blocks of the warp kernels (MpcIo::warm): owned by the Python side, one set per EmulMpc, registered before a solve
static double* g_warm = nullptr;
static int8_t* g_warm_ok = nullptr;

extern "C" {

// Same contract as hmpc_solve, all pointers HOST memory, state arrays owned by the caller:
// Xsol_state [N+1][12][B], Usol_state [N][6][B], code_state int8 [11N][B], valid_state int8 [B].
int emul_solve(const hmpc_config* cfg, const double* Qd, const double* Rd, const double* x_in,
               const double* x_ref, const double* pf, const uint64_t* Cbits, int init, double* Xsol_state,
               double* Usol_state, int8_t* code_state, int8_t* valid_state, double* U, double* Xsol,
               int32_t* status, int32_t* iters, int32_t* nfac, int32_t* path) {
    const QpConst c = qp_const(*cfg);
    const int B = cfg->batch, N = cfg->N, n = 6 * N;
    std::vector<double> smem(((work_vec_doubles(N) + 1) & ~(size_t)1) + mat_doubles(N) + 8);
    std::vector<int32_t> st_tick(B), ninf(B);
    Work w;
    setup_work<true>(w, c, smem.data(), nullptr);
    AOp A{N, n, c.dyn == 3 ? 1 : 0, c.mu, w.stance, w.hinv};
    MpcIo io;
    io.x_in = x_in; io.x_ref = x_ref; io.pf = pf; io.Cbits = Cbits; io.Qd = Qd; io.Rd = Rd;
    io.Xsol = Xsol_state; io.Usol = Usol_state; io.code = code_state; io.valid = valid_state;
    io.U_out = U; io.X_out = Xsol; io.U0_out = nullptr;
    io.status = status; io.iters = iters; io.st_tick = st_tick.data(); io.nfac = nfac; io.path = path;
    io.ninf = ninf.data(); io.flops = nullptr; io.init = init; io.accumulate = 0; io.respawn = 0;
    if (g_warm && g_warm_ok) { io.warm = g_warm; io.warm_ok = g_warm_ok; io.warm_stride = warm_stride_doubles(N); }
    // the library's dispatch (hmpc_api.cu: launch_mpc): warm ticks go through the warp-per-hopper kernel first,
    // hoppers it defers (and everything else) through the CTA kernel
    std::vector<char> deferred(B, 1), skipw(B, 0);
    g_emul_warp_done = 0;
    if (warp_path_applies(*cfg, init)) {
        const int kcap = warp_kcap(*cfg);
        std::vector<double> wsm(warp_work_doubles(N, kcap) + warp_admm_doubles(N) + 8), psm(warp_work_doubles(N, kPrepKcap) + 8), rec(prep_stride(N) + 8);
        const bool admm = cfg->solver == HMPC_SOLVER_ADMM;
        for (int b = 0; b < B; ++b) {
            int done = 0;
            int32_t flag = -1;
            // prep kernel (its own per-warp slice), then the solve kernel on the record it left
            run_warp([&](int lane) {
                WWork ww;
                wcarve(ww, psm.data(), N, kPrepKcap);
                wprep(c, ww, rec.data(), &flag, b, B, io, lane);
            });
            run_warp([&](int lane) {
                WWork ww;
                wcarve(ww, wsm.data(), N, kcap);
                const int d = admm ? mpc_hopper_warp_admm<2>(c, ww, wsm.data() + warp_work_doubles(N, kcap), rec.data(), &flag, kcap, b, B, io, lane)
                                   : mpc_hopper_warp<2>(c, ww, rec.data(), &flag, kcap, b, B, io, lane);
                if (lane == 0) done = d;
            });
            deferred[b] = done > 0 ? 0 : 1;
            skipw[b] = done < 0 ? 1 : 0;
            g_emul_warp_done += done > 0;
        }
    }
    if (cfg->precision == HMPC_FP32) {
        LinSys<float> sys{n, 0, 0, reinterpret_cast<float*>(w.Lm), reinterpret_cast<float*>(w.dinv), w.H, w.idx, w.grow};
        for (int b = 0; b < B; ++b) if (deferred[b]) mpc_hopper<true>(c, w, sys, A, b, B, io, skipw[b]);
    } else {
        LinSys<double> sys{n, 0, 0, reinterpret_cast<double*>(w.Lm), reinterpret_cast<double*>(w.dinv), w.H, w.idx, w.grow};
        for (int b = 0; b < B; ++b) if (deferred[b]) mpc_hopper<true>(c, w, sys, A, b, B, io, skipw[b]);
    }
    return 0;
}

// register (or, with nulls, drop) the warm-block state used by the following emul_solve calls: warm [B][warm_stride_doubles(N)]
void emul_set_warm(double* warm, int8_t* warm_ok) { g_warm = warm; g_warm_ok = warm_ok; }
int emul_warm_stride(int N) { return warm_stride_doubles(N); }
// hoppers the warp path finished in the most recent emul_solve
int emul_warp_done(void) { return g_emul_warp_done; }
// event counters of the warp emulation since the last reset ([0] = DMMA lane-calls)
void emul_counters(long long* out, int reset) {
    for (int i = 0; i < 8; ++i) { out[i] = hmpc_emul_count[i]; if (reset) hmpc_emul_count[i] = 0; }
}

// launch geometry of hmpc_create (hmpc_geometry.cuh) for the given device limits and warp-build register counts (in
// the order of kWarpWpc / kAdmmWpc).  out[16]: unsupported (0/1), cta, threads, grid, smem, ws_bytes, warp, admm, wpc,
// kcap, wdoubles, warp_grid, warp_per_sm, regs, group, warp_smem.
void emul_launch_geometry(const hmpc_config* cfg, int kcap, int sm_count, long long smem_block, long long smem_sm, long long l2,
                          const int* warp_regs, const int* admm_regs, long long* out) {
    DeviceLimits d;
    d.sm_count = sm_count; d.smem_block = (size_t)smem_block; d.smem_sm = (size_t)smem_sm; d.l2 = (size_t)l2;
    for (int i = 0; i < kNumWarpBuilds; ++i) d.warp_regs[i] = warp_regs[i];
    for (int i = 0; i < kNumAdmmBuilds; ++i) d.admm_regs[i] = admm_regs[i];
    const Geometry g = launch_geometry(*cfg, kcap, d);
    const long long v[16] = {g.unsupported ? 1 : 0, g.cta, g.threads, g.grid, (long long)g.smem, (long long)g.ws_bytes, g.warp, g.admm,
                             g.wpc, g.kcap, g.wdoubles, g.warp_grid, g.warp_per_sm, g.regs, g.group, (long long)g.warp_smem};
    for (int i = 0; i < 16; ++i) out[i] = v[i];
}
// the kernel build lists: n[3] = sizes; warp_wpc, admm_wpc, cta_threads (at least 16 entries each)
void emul_kernel_builds(int* n, int* warp_wpc, int* admm_wpc, int* cta_threads) {
    n[0] = kNumWarpBuilds; n[1] = kNumAdmmBuilds; n[2] = kNumCtaBuilds;
    for (int i = 0; i < kNumWarpBuilds; ++i) warp_wpc[i] = kWarpWpc[i];
    for (int i = 0; i < kNumAdmmBuilds; ++i) admm_wpc[i] = kAdmmWpc[i];
    for (int i = 0; i < kNumCtaBuilds; ++i) cta_threads[i] = kCtaThreads[i];
}

// condense only: H [n][n][B], g [n][B], lo/hi [m][B], infeasible [B]
int emul_condense(const hmpc_config* cfg, const double* Qd, const double* Rd, const double* x_in,
                  const double* x_guess, const double* x_ref, const double* pf, const uint64_t* Cbits,
                  double* H, double* g, double* lo, double* hi, int32_t* infeasible) {
    const QpConst c = qp_const(*cfg);
    const int B = cfg->batch, N = cfg->N, n = 6 * N, m = 11 * N;
    std::vector<double> smem(((work_vec_doubles(N) + 1) & ~(size_t)1) + mat_doubles(N) + 8);
    Work w;
    setup_work<true>(w, c, smem.data(), nullptr);
    for (int b = 0; b < B; ++b) {
        load_hopper(c, w, b, B, x_in, pf, Cbits, Qd, Rd);
        for (int k = 0; k < N; ++k) {
            const size_t o = (size_t)k * 12;
            w.gp[4 * k] = x_guess[(o + 0) * B + b]; w.gp[4 * k + 1] = x_guess[(o + 1) * B + b];
            w.gp[4 * k + 2] = x_guess[(o + 2) * B + b]; w.gp[4 * k + 3] = x_guess[(o + 5) * B + b];
        }
        infeasible[b] = condense(c, w, x_ref + b, (size_t)B);
        for (int e = 0; e < n * n; ++e) H[(size_t)e * B + b] = sym_at(w.H, n, e / n, e % n);
        for (int i = 0; i < n; ++i) g[(size_t)i * B + b] = w.g[i];
        for (int r = 0; r < m; ++r) { lo[(size_t)r * B + b] = w.lo[r]; hi[(size_t)r * B + b] = w.hi[r]; }
    }
    return 0;
}

// device planner (hmpc_plan.cuh): rows [row0, row0 + nrows) of the MPC-rate tables for every hopper, then the contact
// masks / switch steps of ticks [row0, row0 + n_ticks); same layout as hmpc_plan_tables.  All pointers HOST memory.
int emul_plan_tables(int B, int N, int mpc_factor, double dt, int N_run, int n_sim, int max_tick, double t_p, double psi1,
                     double psi2, const double* x0, const double* xf, const int32_t* curve, const int32_t* off,
                     const double* sin_tab, const int32_t* pf_idx, const uint64_t* cmask, const uint8_t* sw_glob,
                     int row0, int n_ticks, double* xref_tab, double* pf_tab, uint64_t* C_tab, uint8_t* pf_switch) {
    PlanConst P;
    P.N = N; P.mpc_factor = mpc_factor; P.N_run = N_run; P.t_ref = N_run + N * mpc_factor; P.n_sim = n_sim;
    P.max_tick = max_tick; P.dt = dt; P.amp = t_p / 4; P.T = (double)N_run; P.curve_psi1 = psi1; P.curve_psi2 = psi2;
    P.sin_tab = sin_tab; P.pf_idx = pf_idx; P.cmask = cmask; P.sw_glob = sw_glob;
    P.x0 = x0; P.xf = xf; P.curve = curve; P.off = off;
    const int nrows = n_ticks + N + 1;
    for (int b = 0; b < B; ++b) {
        PlanHopper h;
        plan_load(P, b, B, h);
        for (int r = 0; r < nrows; ++r) {
            double xr[12], pf[3];
            plan_table_row(P, h, off[b], row0 + r, xr, pf);
            if (r < nrows - 1) for (int q = 0; q < 12; ++q) xref_tab[((size_t)r * 12 + q) * B + b] = xr[q];
            for (int q = 0; q < 3; ++q) pf_tab[((size_t)r * 3 + q) * B + b] = pf[q];
        }
        for (int t = 0; t < n_ticks; ++t) {       // plan_masks_kernel
            int j = off[b] + row0 + t;
            if (j >= max_tick) j = max_tick - 1;
            C_tab[(size_t)t * B + b] = cmask[j];
            bool same = true;
            for (int q = 0; q < 3; ++q) same = same && (pf_tab[((size_t)t * 3 + q) * B + b] == pf_tab[((size_t)(t + 1) * 3 + q) * B + b]);
            pf_switch[(size_t)t * B + b] = same ? (uint8_t)mpc_factor : sw_glob[j];
        }
    }
    return 0;
}

// rk4_normalized x nsteps (+ optional convert): X [13][B] in/out, U [6][B], pf [3][B], x_out [12][B] or NULL
int emul_rk4(const hmpc_config* cfg, double* X, const double* U, const double* pf, int nsteps, double* x_out) {
    SimConst s;
    s.m = cfg->m; s.g = cfg->g; s.h = cfg->sim_dt;
    for (int i = 0; i < 9; ++i) { s.J[i] = cfg->J[i]; s.Jinv[i] = cfg->Jinv[i]; }
    for (int i = 0; i < 3; ++i) s.rh[i] = cfg->rh[i];
    const int B = cfg->batch;
    for (int b = 0; b < B; ++b) {
        double Xl[13], Ul[6], p[3];
        for (int i = 0; i < 13; ++i) Xl[i] = X[(size_t)i * B + b];
        for (int i = 0; i < 6; ++i) Ul[i] = U[(size_t)i * B + b];
        for (int i = 0; i < 3; ++i) p[i] = pf[(size_t)i * B + b];
        for (int k = 0; k < nsteps; ++k) rk4_step(s, Xl, Ul, p);
        for (int i = 0; i < 13; ++i) X[(size_t)i * B + b] = Xl[i];
        if (x_out) {
            double x[12];
            convert_state(Xl, x);
            for (int i = 0; i < 12; ++i) x_out[(size_t)i * B + b] = x[i];
        }
    }
    return 0;
}

// One MPC tick of the simulator with the contact gate (hmpc_sim.cuh: sim_tick), all pointers HOST memory:
// X [13][B] in/out, U [6][B], pfa / pfb [3][B], sw [B] uint8 (may be null), bits [B] uint32 (may be null).
int emul_sim_tick(const hmpc_config* cfg, double* X, const double* U, const double* pfa, const double* pfb, const uint8_t* sw,
                  int gate_mode, const uint32_t* bits, double leg_max) {
    SimConst s;
    s.m = cfg->m; s.g = cfg->g; s.h = cfg->sim_dt;
    for (int i = 0; i < 9; ++i) { s.J[i] = cfg->J[i]; s.Jinv[i] = cfg->Jinv[i]; }
    for (int i = 0; i < 3; ++i) s.rh[i] = cfg->rh[i];
    const int B = cfg->batch;
    for (int b = 0; b < B; ++b) {
        double Xl[13], Ul[6], pa[3], pb[3];
        for (int i = 0; i < 13; ++i) Xl[i] = X[(size_t)i * B + b];
        for (int i = 0; i < 6; ++i) Ul[i] = U[(size_t)i * B + b];
        for (int i = 0; i < 3; ++i) { pa[i] = pfa[(size_t)i * B + b]; pb[i] = pfb[(size_t)i * B + b]; }
        sim_tick(s, gate_mode, bits ? bits[b] : 0xffffffffu, leg_max * leg_max, Xl, Ul, pa, pb, sw ? (int)sw[b] : cfg->mpc_factor,
                 cfg->mpc_factor, nullptr, (size_t)B, b);
        for (int i = 0; i < 13; ++i) X[(size_t)i * B + b] = Xl[i];
    }
    return 0;
}

}  // extern "C"
