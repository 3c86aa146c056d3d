// tests/emul_body/emul_body.cpp -- TEST INFRASTRUCTURE.  The emulation of tests/emul (device source compiled by g++,
// one serial thread per hopper, 32-lane warp fibers) with per-hopper bodies (include/hmpc.h: hmpc_set_body_params):
// the model array goes into QpConst::body, the plant array into SimConst::body, exactly as the library passes them.
// All pointers HOST memory; a null body array means the config's scalars, as in the library.
#include "../emul/emul.cpp"

static const double* g_body_model = nullptr;   // [kBodyModel][B]: m, mu, rh[3], Jinv[9]
static const double* g_body_plant = nullptr;   // [kBodyPlant][B]: m, rh[3], J[9], Jinv[9]

static SimConst sim_const(const hmpc_config& cfg) {
    SimConst s;
    s.m = cfg.m; s.g = cfg.g; s.h = cfg.sim_dt;
    for (int i = 0; i < 9; ++i) { s.J[i] = cfg.J[i]; s.Jinv[i] = cfg.Jinv[i]; }
    for (int i = 0; i < 3; ++i) s.rh[i] = cfg.rh[i];
    s.body = g_body_plant;
    return s;
}

extern "C" {

// register (or, with nulls, drop) the bodies used by the following emul_body_* calls
void emul_set_body(const double* model, const double* plant) { g_body_model = model; g_body_plant = plant; }
int emul_body_rows(int plant) { return plant ? kBodyPlant : kBodyModel; }

// emul_solve (tests/emul/emul.cpp) with QpConst::body = the registered model array
int emul_body_solve(const hmpc_config* cfg, const double* Qd, const double* Rd, const double* x_in,
                    const double* x_ref, const double* pf, const uint64_t* Cbits, int init, double* Xsol_state,
                    double* Usol_state, int8_t* code_state, int8_t* valid_state, double* U, double* Xsol,
                    int32_t* status, int32_t* iters, int32_t* nfac, int32_t* path) {
    QpConst c = qp_const(*cfg);
    c.body = g_body_model;
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
    std::vector<char> deferred(B, 1), skipw(B, 0);
    g_emul_warp_done = 0;
    if (warp_path_applies(*cfg, init)) {
        const int kcap = warp_kcap(*cfg);
        std::vector<double> wsm(warp_work_doubles(N, kcap) + warp_admm_doubles(N) + 8), psm(warp_work_doubles(N, kPrepKcap) + 8), rec(prep_stride(N) + 8);
        const bool admm = cfg->solver == HMPC_SOLVER_ADMM;
        for (int b = 0; b < B; ++b) {
            int done = 0;
            int32_t flag = -1;
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
        for (int b = 0; b < B; ++b) if (deferred[b]) { A.mu = model_body(c, b, B).mu; mpc_hopper<true>(c, w, sys, A, b, B, io, skipw[b]); }
    } else {
        LinSys<double> sys{n, 0, 0, reinterpret_cast<double*>(w.Lm), reinterpret_cast<double*>(w.dinv), w.H, w.idx, w.grow};
        for (int b = 0; b < B; ++b) if (deferred[b]) { A.mu = model_body(c, b, B).mu; mpc_hopper<true>(c, w, sys, A, b, B, io, skipw[b]); }
    }
    return 0;
}

// emul_condense with the registered model array: H [n][n][B], g [n][B], lo/hi [m][B], infeasible [B]
int emul_body_condense(const hmpc_config* cfg, const double* Qd, const double* Rd, const double* x_in,
                       const double* x_guess, const double* x_ref, const double* pf, const uint64_t* Cbits,
                       double* H, double* g, double* lo, double* hi, int32_t* infeasible) {
    QpConst c = qp_const(*cfg);
    c.body = g_body_model;
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
        infeasible[b] = condense_hopper(c, w, b, B, x_ref + b, (size_t)B);
        for (int e = 0; e < n * n; ++e) H[(size_t)e * B + b] = sym_at(w.H, n, e / n, e % n);
        for (int i = 0; i < n; ++i) g[(size_t)i * B + b] = w.g[i];
        for (int r = 0; r < m; ++r) { lo[(size_t)r * B + b] = w.lo[r]; hi[(size_t)r * B + b] = w.hi[r]; }
    }
    return 0;
}

// emul_sim_tick with the registered plant array (sim_kernel<true> when it is set)
int emul_body_sim_tick(const hmpc_config* cfg, double* X, const double* U, const double* pfa, const double* pfb, const uint8_t* sw,
                       int gate_mode, double leg_max) {
    const SimConst s = sim_const(*cfg);
    const int B = cfg->batch;
    for (int b = 0; b < B; ++b) {
        double Xl[13], Ul[6], pa[3], pb[3];
        for (int i = 0; i < 13; ++i) Xl[i] = X[(size_t)i * B + b];
        for (int i = 0; i < 6; ++i) Ul[i] = U[(size_t)i * B + b];
        for (int i = 0; i < 3; ++i) { pa[i] = pfa[(size_t)i * B + b]; pb[i] = pfb[(size_t)i * B + b]; }
        const int swb = sw ? (int)sw[b] : cfg->mpc_factor;
        if (s.body) sim_tick(plant_body(s, b, B), gate_mode, 0xffffffffu, leg_max * leg_max, Xl, Ul, pa, pb, swb, cfg->mpc_factor, nullptr, (size_t)B, b);
        else sim_tick(s, gate_mode, 0xffffffffu, leg_max * leg_max, Xl, Ul, pa, pb, swb, cfg->mpc_factor, nullptr, (size_t)B, b);
        for (int i = 0; i < 13; ++i) X[(size_t)i * B + b] = Xl[i];
    }
    return 0;
}

}  // extern "C"
