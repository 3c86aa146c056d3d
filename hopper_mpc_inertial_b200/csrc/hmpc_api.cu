// hmpc_api.cu -- kernels and the C ABI of libhmpc_b200.so (declared in include/hmpc.h).
//
// Kernels
//   sim_kernel        K3: mpc_factor x RK4 (ZOH control) + convert, one thread per hopper, SoA I/O
//   mpc_kernel        K1+K2 (hmpc_kernel.cuh, instantiated in inst_*.cu): time shift, linearise, condense,
//                     solve (warm active-set refinement / interior point / ADMM), solution rollout;
//                     one CTA per hopper (persistent grid-stride loop)
//   convert_kernel / linearize_kernel / condense_kernel   parity-test entry points
//   dfma_peak_kernel  FP64 FMA roofline microbenchmark
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <new>
#include <string>
#include <vector>

#include "../../include/hmpc.h"
#include "hmpc_sim.cuh"
#include "hmpc_qp.cuh"
#include "hmpc_mpc.cuh"
#include "hmpc_kernel.cuh"
#include "hmpc_warp.cuh"
#include "hmpc_geometry.cuh"
#include "hmpc_plan.cuh"

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

#define HMPC_CUDA(call)                                                                       \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess)                                                                \
            return fail(HMPC_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));   \
    } while (0)

}  // namespace

constexpr int kOrderBuckets = 4096;     // buckets of the contact-mask counting sort (order_* kernels)
// timing events per rollout tick: main stream 0 | solver | 1 | simulator | 2; side stream (overlapped ticks) 3 | CTA kernel
// over the deferred hoppers | 4 | their simulator step | 5
constexpr int kTickEvents = 6;

struct hmpc_handle {
    hmpc_config cfg;
    cudaStream_t stream = nullptr;
    int sm_count = 0;
    // per-hopper persistent state
    double* Qd = nullptr;     // [12][B]
    double* Rd = nullptr;     // [6][B]
    double* Xsol = nullptr;   // [N+1][12][B] previous QP state trajectory (x.value)
    double* Usol = nullptr;   // [N][6][B]    previous QP inputs (u.value)
    int8_t* code = nullptr;   // [11N][B]     previous active set (+1 / -1 / 0 per constraint row)
    int8_t* valid = nullptr;  // [B]          1: Xsol / Usol / code hold a solved previous tick
    double* xin = nullptr;    // [12][B]
    double* U0 = nullptr;     // [6][B]
    int32_t* st_tmp = nullptr;
    int32_t* it_tmp = nullptr;
    int32_t* st_tick = nullptr;   // [B] status of the current tick (rollout: read by the simulator kernel)
    int32_t* nfac = nullptr;      // [B]
    int32_t* path = nullptr;      // [B]
    int32_t* ninf = nullptr;      // [B]
    double* flops = nullptr;      // [B] algorithmic FLOPs of the solver kernel
    int* work_ctr = nullptr;      // [2][8] per tick parity: ticket counters and deferral count (launch_mpc)
    // optional per-kernel device timing of hmpc_rollout (hmpc_set_timing): kTickEvents per tick
    int timing = 0;
    std::vector<cudaEvent_t> ev;
    std::vector<uint8_t> ev_side;   // [tick] 1: the tick's deferred hoppers ran on the side stream (events 3..5 valid)
    int ev_ticks = 0;
    // overlapped rollout schedule (DESIGN.md section 5): the deferred hoppers' CTA kernel, their simulator step and their
    // next prep run on a second stream while the main stream simulates and condenses every other hopper
    cudaStream_t side = nullptr;      // null: serial schedule only (no warp path, or HMPC_DEFER_SERIAL=1)
    cudaEvent_t ev_fork = nullptr;    // main -> side: the warp kernel of the tick has finished (deferral list complete)
    cudaEvent_t ev_join = nullptr;    // side -> main: the last side-stream work of the rollout so far
    int32_t* defer_mark = nullptr;    // [B] number of the overlapped tick in which the hopper was last deferred
    int seq = 0;                      // number of the next overlapped tick (handle-wide; its parity picks the buffers)
    bool side_prep = false;           // the side stream condenses the deferred hoppers of tick seq - 1 for tick seq
    hmpc::Geometry geo;               // launch geometry of the CTA kernel and the warp-per-hopper kernel (hmpc_geometry.cuh)
    double* ws = nullptr;     // per-CTA matrix workspace of the N > 10 kernels (geo.ws_bytes)
    int64_t launches = 0;
    // warp-per-hopper warm path (hmpc_warp.cuh)
    size_t pstride = 0;
    double* prep = nullptr;       // [B][pstride] QP records the prep kernel hands to the solve kernel
    int32_t* prep_flag = nullptr; // [B]
    // device-side planner (hmpc_plan.cuh): global tables owned by the handle, per-hopper arrays owned by the caller
    bool plan_ok = false;
    hmpc::PlanConst plan;
    double* plan_sin = nullptr; int32_t* plan_pfidx = nullptr; uint64_t* plan_cmask = nullptr; uint8_t* plan_sw = nullptr;
    double* win_xref = nullptr;   // [N+1][12][B] reference window of the current tick (hmpc_rollout_planned)
    double* win_pf = nullptr;     // [N+1][3][B]
    uint64_t* win_C = nullptr;    // [B]
    uint8_t* win_sw = nullptr;    // [B]
    int* defer_list = nullptr;    // [2][B] per tick parity: hoppers the warp kernel handed to the CTA kernel
    // work order of the lock-step solve kernel: hoppers grouped by contact schedule (order_* kernels)
    int* work_order = nullptr;    // [B] permutation, rebuilt every tick
    double* warm = nullptr;       // [B][warm_stride] warm blocks of the warp kernels (MpcIo::warm)
    int8_t* warm_ok = nullptr;    // [B]
    int* order_cnt = nullptr;     // [2][kOrderBuckets] bucket sizes / cursors
    int order_on = 1;             // HMPC_WORK_ORDER=0 switches the grouping off
    // contact gate of the simulator (hmpc_set_contact_gate)
    int gate_mode = HMPC_GATE_OFF;
    const uint32_t* gate_tab = nullptr;   // caller's [T][B] masks (table flavour)
    uint32_t* gate_glob = nullptr;        // device copy of the common-clock masks (planned flavour)
    int gate_max_tick = 0;
    double leg_max = 0.0;
    int32_t* n_defer = nullptr;   // [1] accumulated deferrals of the most recent solve / rollout
    // per-hopper bodies (hmpc_set_body_params), allocated on the first call; used while the flag is set
    double* body_model = nullptr;   // [kBodyModel][B]  QpConst::body
    double* body_plant = nullptr;   // [kBodyPlant][B]  SimConst::body
    bool model_on = false, plant_on = false;
    int* body_bad = nullptr;        // [1] first hopper with invalid values (body_check_kernel)
};

namespace hmpc {

// ------------------------------------------------------------------------------------------------
// K3: simulator.  X [13][B] in/out; U [6][B]; pfa/pfb [3][B] footstep before/after the switch step.
// PLANT: every hopper integrates its own body (c.body set); the uniform build keeps the body in the kernel's constant
// parameters and needs no registers for it.
// ------------------------------------------------------------------------------------------------
template <bool PLANT>
__global__ void __launch_bounds__(128)
sim_kernel(SimConst c, int B, HopperSet hs, double* __restrict__ X, const double* __restrict__ U,
           const double* __restrict__ pfa, const double* __restrict__ pfb,
           const uint8_t* __restrict__ sw, int nsteps, double* __restrict__ xin_out,
           double* __restrict__ Xlog, double* __restrict__ Ulog, double* __restrict__ Xsteps,
           const int32_t* __restrict__ st_tick, const double* __restrict__ xref_next, SimGate gt) {
    int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (hs.list) {
        if (b >= *hs.list_cnt) return;
        b = hs.list[b] & kListHopperMask;
    } else if (b >= B || (hs.mark && hs.mark[b] == hs.skip)) return;
    double Xl[13], Ul[6], pa[3], pb[3];
#pragma unroll
    for (int i = 0; i < 13; ++i) Xl[i] = X[(size_t)i * B + b];
#pragma unroll
    for (int i = 0; i < 6; ++i) Ul[i] = U[(size_t)i * B + b];
#pragma unroll
    for (int i = 0; i < 3; ++i) { pa[i] = pfa[(size_t)i * B + b]; pb[i] = pfb ? pfb[(size_t)i * B + b] : pa[i]; }
    const int s = sw ? (int)sw[b] : nsteps;
    const bool respawn = st_tick && xref_next && st_tick[b] == HMPC_PRIMAL_INFEASIBLE;
    if (respawn) {
        // put the hopper back onto its reference at the next tick: position, yaw and world velocity of
        // the reference row, level attitude, no body rates (HMPC_INFEASIBLE_RESPAWN)
        double xr[12];
#pragma unroll
        for (int i = 0; i < 12; ++i) xr[i] = xref_next[(size_t)i * B + b];
        double sy, cy;
        sincos(0.5 * xr[5], &sy, &cy);
        Xl[0] = xr[0]; Xl[1] = xr[1]; Xl[2] = xr[2];
        Xl[3] = cy; Xl[4] = 0.0; Xl[5] = 0.0; Xl[6] = sy;
        double R[9];
        quat_rotm(Xl + 3, R);
        mat3T_vec(R, xr + 6, Xl + 7);
        Xl[10] = Xl[11] = Xl[12] = 0.0;
    } else {
        if (PLANT) sim_tick(plant_body(c, b, B), gt.mode, gate_bits_of(gt, b), gt.leg_max2, Xl, Ul, pa, pb, s, nsteps, Xsteps, (size_t)B, b);
        else sim_tick(c, gt.mode, gate_bits_of(gt, b), gt.leg_max2, Xl, Ul, pa, pb, s, nsteps, Xsteps, (size_t)B, b);
    }
#pragma unroll
    for (int i = 0; i < 13; ++i) X[(size_t)i * B + b] = Xl[i];
    if (Xlog) {
#pragma unroll
        for (int i = 0; i < 13; ++i) Xlog[(size_t)i * B + b] = Xl[i];
    }
    if (Ulog) {
#pragma unroll
        for (int i = 0; i < 6; ++i) Ulog[(size_t)i * B + b] = Ul[i];
    }
    if (xin_out) {
        double x[12];
        convert_state(Xl, x);
#pragma unroll
        for (int i = 0; i < 12; ++i) xin_out[(size_t)i * B + b] = x[i];
    }
}

__global__ void convert_kernel(int B, const double* __restrict__ X, double* __restrict__ x) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    double Xl[13], xl[12];
#pragma unroll
    for (int i = 0; i < 13; ++i) Xl[i] = X[(size_t)i * B + b];
    convert_state(Xl, xl);
#pragma unroll
    for (int i = 0; i < 12; ++i) x[(size_t)i * B + b] = xl[i];
}

// parity-test kernels ---------------------------------------------------------------------------
__global__ void linearize_kernel(QpConst c, int B, const double* __restrict__ x_guess,
                                 const double* __restrict__ pf, double* __restrict__ Ad,
                                 double* __restrict__ Bd) {
    extern __shared__ double smem[];
    Work w;
    carve(w, smem, c.N);
    const int N = c.N, tid = threadIdx.x, T = blockDim.x, b = blockIdx.x;
    for (int i = tid; i < 3 * N; i += T) w.pfw[i] = pf[(size_t)i * B + b];
    stage_body(c, w, b, B);
    for (int k = tid; k < N; k += T) {
        const size_t o = (size_t)k * 12;
        w.gp[4 * k] = x_guess[(o + 0) * B + b]; w.gp[4 * k + 1] = x_guess[(o + 1) * B + b];
        w.gp[4 * k + 2] = x_guess[(o + 2) * B + b]; w.gp[4 * k + 3] = x_guess[(o + 5) * B + b];
    }
    __syncthreads();
    for (int k = tid; k < N; k += T) linearize_stage(c, SmemBody{w.red}, k, w);
    __syncthreads();
    for (int e = tid; e < N * 144; e += T) {
        const int k = e / 144, r = (e % 144) / 12, cc = e % 12;
        double v = (r == cc) ? 1.0 : 0.0;
        if (r < 3 && cc == r + 6) v += c.dt;
        if (r >= 3 && r < 6 && cc >= 9) {
            const double cs = w.cz[k], sn = w.sz[k];
            const double Rz[9] = {cs, sn, 0, -sn, cs, 0, 0, 0, 1};
            v += Rz[3 * (r - 3) + (cc - 9)] * c.dt;
        }
        Ad[(size_t)e * B + b] = v;
    }
    for (int e = tid; e < N * 72; e += T) {
        const int k = e / 72, r = (e % 72) / 6, cc = e % 6;
        double v = 0.0;
        if (r >= 6 && r < 9 && cc < 3) v = w.Bv[9 * k + 3 * (r - 6) + cc];
        if (r >= 9) v = w.Bw[18 * k + 6 * (r - 9) + cc];
        Bd[(size_t)e * B + b] = v;
    }
}

__global__ void condense_kernel(QpConst c, int B, int mats_in_smem, double* __restrict__ ws,
                                const double* __restrict__ x_in, const double* __restrict__ x_guess,
                                const double* __restrict__ x_ref, const double* __restrict__ pf,
                                const uint64_t* __restrict__ Cbits, const double* __restrict__ Qd,
                                const double* __restrict__ Rd, double* __restrict__ H,
                                double* __restrict__ g, double* __restrict__ lo, double* __restrict__ hi,
                                int32_t* __restrict__ infeasible) {
    extern __shared__ double smem[];
    Work w;
    if (mats_in_smem) setup_work<true>(w, c, smem, ws); else setup_work<false>(w, c, smem, ws);
    const int N = c.N, n = 6 * N, m = 11 * N, tid = threadIdx.x, T = blockDim.x;
    for (int b = blockIdx.x; b < B; b += gridDim.x) {
        __syncthreads();
        load_hopper(c, w, b, B, x_in, pf, Cbits, Qd, Rd);
        for (int k = tid; k < N; k += T) {
            const size_t o = (size_t)k * 12;
            w.gp[4 * k] = x_guess[(o + 0) * B + b]; w.gp[4 * k + 1] = x_guess[(o + 1) * B + b];
            w.gp[4 * k + 2] = x_guess[(o + 2) * B + b]; w.gp[4 * k + 3] = x_guess[(o + 5) * B + b];
        }
        __syncthreads();
        const int inf = condense_hopper(c, w, b, B, x_ref + b, (size_t)B);
        if (infeasible && tid == 0) infeasible[b] = inf;
        for (int e = tid; e < n * n; e += T) H[(size_t)e * B + b] = sym_at(w.H, n, e / n, e % n);
        for (int i = tid; i < n; i += T) g[(size_t)i * B + b] = w.g[i];
        for (int r = tid; r < m; r += T) { lo[(size_t)r * B + b] = w.lo[r]; hi[(size_t)r * B + b] = w.hi[r]; }
    }
}

// hmpc_set_body_params: *bad = min over the hoppers whose given values are not finite, or m <= 0, or mu < 0
__global__ void body_check_kernel(int B, const double* __restrict__ m, const double* __restrict__ J,
                                  const double* __restrict__ Jinv, const double* __restrict__ rh,
                                  const double* __restrict__ mu, int* __restrict__ bad) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const size_t Bs = (size_t)B;
    bool ok = true;
    if (m) ok = ok && isfinite(m[b]) && m[b] > 0.0;
    if (mu) ok = ok && isfinite(mu[b]) && mu[b] >= 0.0;
    for (int i = 0; i < 9; ++i) {
        if (J) ok = ok && isfinite(J[i * Bs + b]);
        if (Jinv) ok = ok && isfinite(Jinv[i * Bs + b]);
        if (i < 3 && rh) ok = ok && isfinite(rh[i * Bs + b]);
    }
    if (!ok) atomicMin(bad, b);
}
// rows of a body array that take the handle's scalar for every hopper (bit r of mask: row r = v[r])
struct BodyFill {
    double v[kBodyPlant];
    uint32_t mask;
};
__global__ void body_fill_kernel(int B, double* __restrict__ dst, BodyFill f) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    for (int r = 0; r < kBodyPlant; ++r)
        if ((f.mask >> r) & 1u) dst[(size_t)r * B + b] = f.v[r];
}

// FP64 FMA peak: 8 independent accumulator chains per thread, no memory traffic in the loop.
__global__ void dfma_peak_kernel(double* out, int iters, double a, double bseed) {
    double acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = bseed + (double)(threadIdx.x + i);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int r = 0; r < 8; ++r) {
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[i] = fma(acc[i], a, bseed);
        }
    }
    double s = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += acc[i];
    if (s == 123.456) out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

}  // namespace hmpc

// =================================================================================================
// C ABI
// =================================================================================================
namespace {

hmpc::QpConst make_qp_const(const hmpc_config& cfg) {
    hmpc::QpConst c;
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
    if (const char* ev = getenv("HMPC_WORK_PERM")) {      // stress test: "mul,add" permutes the order the hoppers are taken in
        int mul = 1, add = 0;
        auto gcd = [](long long a, long long b) { while (b) { const long long r = a % b; a = b; b = r; } return a; };
        if (sscanf(ev, "%d,%d", &mul, &add) >= 1 && mul >= 1 && add >= 0 && gcd(mul, cfg.batch) == 1) { c.work_mul = mul; c.work_add = add; }
    }
    c.max_refine = 6;
    c.stagnation = 0.25;
    if (cfg.precision == HMPC_FP32) {   // FP32 factor: more refinement sweeps, regularisation / IPM tolerance at FP32 scale
        c.max_refine = 14;
        c.stagnation = 0.7;
        c.kkt_eps = std::max(cfg.kkt_eps, 1e-3);
        c.ipm_tol = std::max(cfg.ipm_tol, 1e-6);
    }
    return c;
}

hmpc::SimConst make_sim_const(const hmpc_config& cfg) {
    hmpc::SimConst s;
    s.m = cfg.m; s.g = cfg.g; s.h = cfg.sim_dt;
    for (int i = 0; i < 9; ++i) { s.J[i] = cfg.J[i]; s.Jinv[i] = cfg.Jinv[i]; }
    for (int i = 0; i < 3; ++i) s.rh[i] = cfg.rh[i];
    return s;
}

hmpc::QpConst qp_const(const hmpc_handle* h) {
    hmpc::QpConst c = make_qp_const(h->cfg);
    c.body = h->model_on ? h->body_model : nullptr;
    return c;
}
hmpc::SimConst sim_const(const hmpc_handle* h) {
    hmpc::SimConst s = make_sim_const(h->cfg);
    s.body = h->plant_on ? h->body_plant : nullptr;
    return s;
}
// the simulator kernel, specialised on whether the hoppers carry their own plant body
template <class... Args>
void launch_sim(const hmpc::SimConst& sc, int grid, cudaStream_t st, Args... args) {
    if (sc.body) hmpc::sim_kernel<true><<<grid, 128, 0, st>>>(sc, args...);
    else hmpc::sim_kernel<false><<<grid, 128, 0, st>>>(sc, args...);
}

int check_handle(hmpc_handle* h) {
    if (!h) return fail(HMPC_ERR_BAD_ARG, "null handle");
    cudaError_t e = cudaSetDevice(h->cfg.device);
    if (e != cudaSuccess) return fail(HMPC_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
    return HMPC_OK;
}

void inv3(const double* J, double* Ji) {
    const double a = J[0], b = J[1], c = J[2], d = J[3], e = J[4], f = J[5], g = J[6], h = J[7], i = J[8];
    const double det = a * (e * i - f * h) - b * (d * i - f * g) + c * (d * h - e * g);
    Ji[0] = (e * i - f * h) / det; Ji[1] = (c * h - b * i) / det; Ji[2] = (b * f - c * e) / det;
    Ji[3] = (f * g - d * i) / det; Ji[4] = (a * i - c * g) / det; Ji[5] = (c * d - a * f) / det;
    Ji[6] = (d * h - e * g) / det; Ji[7] = (b * g - a * h) / det; Ji[8] = (a * e - b * d) / det;
}

// the CTA kernel builds (HMPC_CTA_BUILDS); any other id is refused and nothing is launched
cudaError_t cta_set_smem(hmpc::CtaBuild b, int bytes) {
    switch (b) {
#define CALL(name, threads) case hmpc::CTA_##name: return hmpc::mpc_set_smem_##name(bytes);
        HMPC_CTA_BUILDS(CALL)
#undef CALL
        default: return cudaErrorInvalidValue;
    }
}
// the CTA kernel over every hopper (l.list null) or over the deferral list of the warp kernel
cudaError_t launch_cta(hmpc_handle* h, const hmpc::MpcLaunch& l, const hmpc::QpConst& qc, const hmpc::MpcIo& io) {
    switch (h->geo.cta) {
#define CALL(name, threads) case hmpc::CTA_##name: hmpc::mpc_launch_##name(l, qc, io); break;
        HMPC_CTA_BUILDS(CALL)
#undef CALL
        default: return cudaErrorInvalidValue;
    }
    ++h->launches;
    return cudaSuccess;
}

}  // namespace

extern "C" {

int hmpc_abi_version(void) { return HMPC_ABI_VERSION; }

const char* hmpc_last_error(void) { return g_err.c_str(); }

int hmpc_default_config(hmpc_config* cfg) {
    if (!cfg) return fail(HMPC_ERR_BAD_ARG, "null config");
    memset(cfg, 0, sizeof(*cfg));
    cfg->abi_version = HMPC_ABI_VERSION;
    cfg->device = 0; cfg->batch = 1; cfg->dyn = HMPC_DYN_3F; cfg->N = 60; cfg->mpc_factor = 20;
    cfg->precision = HMPC_FP64; cfg->uref_mode = HMPC_UREF_ALIASED;
    cfg->solver = HMPC_SOLVER_EXACT; cfg->mode = HMPC_MODE_EARLY_EXIT;
    cfg->max_iter = 10000; cfg->check_interval = 25; cfg->first_check = 25; cfg->polish = 1;   // cvxpy -> OSQP
    cfg->adaptive_rho = 1; cfg->warm_start = 1; cfg->polish_retries = 8; cfg->ipm_max_iter = 40;
    cfg->on_infeasible = HMPC_INFEASIBLE_HOLD; cfg->sqp_sweeps = 1;
    cfg->mpc_dt = 0.02; cfg->sim_dt = 1e-3; cfg->m = 7.5; cfg->g = 9.807; cfg->mu = 1.0;
    const double J[9] = {76148072.89e-9, 70089.52e-9, 2067970.36e-9, 70089.52e-9, 45477183.53e-9,
                         -87045.58e-9, 2067970.36e-9, -87045.58e-9, 76287220.47e-9};
    memcpy(cfg->J, J, sizeof(J));
    inv3(cfg->J, cfg->Jinv);
    cfg->rh[0] = -0.02663114 / 1000; cfg->rh[1] = -0.04435752 / 1000; cfg->rh[2] = -6.61082088 / 1000;
    cfg->tau_max[0] = 7.78; cfg->tau_max[1] = 7.78; cfg->tau_max[2] = 4.0;
    cfg->fz_max = 206.0; cfg->z_min = 0.1; cfg->kf = 100.0;
    cfg->eps_abs = 1e-5; cfg->eps_rel = 1e-5; cfg->rho0 = 0.1; cfg->sigma = 1e-6; cfg->alpha = 1.6;
    cfg->kkt_eps = 1e-9; cfg->polish_tol = 1e-9; cfg->ipm_tol = 1e-6;
    return HMPC_OK;
}

int hmpc_create(const hmpc_config* cfg, hmpc_handle** out) {
    if (!cfg || !out) return fail(HMPC_ERR_BAD_ARG, "null argument");
    *out = nullptr;
    if (cfg->abi_version != HMPC_ABI_VERSION) return fail(HMPC_ERR_BAD_ARG, "abi_version mismatch");
    if (cfg->batch < 1) return fail(HMPC_ERR_BAD_ARG, "batch must be >= 1");
    if (cfg->N < 3 || cfg->N > HMPC_MAX_N) return fail(HMPC_ERR_BAD_ARG, "N must be in [3, 64]");
    if (cfg->hot_path != HMPC_HOT_AUTO && cfg->hot_path != HMPC_HOT_CTA) return fail(HMPC_ERR_BAD_ARG, "hot_path must be HMPC_HOT_AUTO or HMPC_HOT_CTA");
    if (cfg->dyn != HMPC_DYN_2F && cfg->dyn != HMPC_DYN_3F) return fail(HMPC_ERR_BAD_ARG, "dyn must be 2 or 3");
    if (cfg->precision != HMPC_FP64 && cfg->precision != HMPC_FP32) return fail(HMPC_ERR_BAD_ARG, "precision must be HMPC_FP64 or HMPC_FP32");
    if (cfg->precision == HMPC_FP32 && cfg->N > 10) return fail(HMPC_ERR_UNSUPPORTED, "FP32 mode is built for horizons N <= 10 only");
    if (cfg->mpc_factor < 1 || cfg->mpc_factor > 255) return fail(HMPC_ERR_BAD_ARG, "mpc_factor must be in [1,255]");
    if (cfg->max_iter < 1 || cfg->check_interval < 1 || cfg->first_check < 1 || cfg->polish_retries < 0 ||
        cfg->ipm_max_iter < 1)
        return fail(HMPC_ERR_BAD_ARG, "max_iter/check_interval/first_check/ipm_max_iter must be >= 1, polish_retries >= 0");
    if (cfg->solver != HMPC_SOLVER_EXACT && cfg->solver != HMPC_SOLVER_ADMM)
        return fail(HMPC_ERR_BAD_ARG, "solver must be HMPC_SOLVER_EXACT or HMPC_SOLVER_ADMM");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(HMPC_ERR_NO_DEVICE, "no CUDA device available (there is no CPU fallback)");
    if (cfg->device < 0 || cfg->device >= ndev) return fail(HMPC_ERR_BAD_ARG, "device ordinal out of range");
    HMPC_CUDA(cudaSetDevice(cfg->device));
    hmpc_handle* h = new (std::nothrow) hmpc_handle();
    if (!h) return fail(HMPC_ERR_ALLOC, "host allocation failed");
    h->cfg = *cfg;
    cudaDeviceProp prop;
    {
        cudaError_t ep = cudaGetDeviceProperties(&prop, cfg->device);
        if (ep != cudaSuccess) { hmpc_destroy(h); return fail(HMPC_ERR_CUDA, std::string("cudaGetDeviceProperties: ") + cudaGetErrorString(ep)); }
    }
    h->sm_count = prop.multiProcessorCount;
    // launch geometry, from the device limits and the register counts of the warp kernel builds
    hmpc::DeviceLimits lim;
    lim.sm_count = prop.multiProcessorCount;
    lim.smem_block = prop.sharedMemPerBlockOptin;
    lim.smem_sm = prop.sharedMemPerMultiprocessor;
    lim.l2 = (size_t)prop.l2CacheSize;
    cudaError_t e = cudaSuccess;
    if (hmpc::warp_path_applies(*cfg, 0)) {
        if (cfg->solver == HMPC_SOLVER_ADMM)
            for (int i = 0; i < hmpc::kNumAdmmBuilds && e == cudaSuccess; ++i) e = hmpc::warp_admm_regs(hmpc::kAdmmWpc[i], &lim.admm_regs[i]);
        else
            for (int i = 0; i < hmpc::kNumWarpBuilds && e == cudaSuccess; ++i) e = hmpc::warp_regs(hmpc::kWarpWpc[i], &lim.warp_regs[i]);
        if (e != cudaSuccess) { hmpc_destroy(h); return fail(HMPC_ERR_CUDA, std::string("cudaFuncGetAttributes (warp kernel): ") + cudaGetErrorString(e)); }
    }
    h->geo = hmpc::launch_geometry(*cfg, hmpc::warp_kcap(*cfg), lim);
    const hmpc::Geometry& g = h->geo;
    if (const char* why = g.unsupported) { hmpc_destroy(h); return fail(HMPC_ERR_UNSUPPORTED, why); }
    const size_t B = (size_t)cfg->batch, N = (size_t)cfg->N;
    auto dalloc = [&](void** p, size_t bytes) { return cudaMalloc(p, bytes); };
    if ((e = dalloc((void**)&h->Qd, 12 * B * 8)) != cudaSuccess || (e = dalloc((void**)&h->Rd, 6 * B * 8)) != cudaSuccess ||
        (e = dalloc((void**)&h->Xsol, (N + 1) * 12 * B * 8)) != cudaSuccess ||
        (e = dalloc((void**)&h->Usol, N * 6 * B * 8)) != cudaSuccess ||
        (e = dalloc((void**)&h->xin, 12 * B * 8)) != cudaSuccess || (e = dalloc((void**)&h->U0, 6 * B * 8)) != cudaSuccess ||
        (e = dalloc((void**)&h->st_tmp, B * 4)) != cudaSuccess || (e = dalloc((void**)&h->it_tmp, B * 4)) != cudaSuccess ||
        (e = dalloc((void**)&h->st_tick, B * 4)) != cudaSuccess || (e = dalloc((void**)&h->nfac, B * 4)) != cudaSuccess ||
        (e = dalloc((void**)&h->path, B * 4)) != cudaSuccess || (e = dalloc((void**)&h->ninf, B * 4)) != cudaSuccess ||
        (e = dalloc((void**)&h->code, 11 * N * B)) != cudaSuccess || (e = dalloc((void**)&h->valid, B)) != cudaSuccess ||
        (e = dalloc((void**)&h->flops, B * 8)) != cudaSuccess || (e = dalloc((void**)&h->work_ctr, 64)) != cudaSuccess ||
        (e = dalloc((void**)&h->defer_list, 2 * B * 4)) != cudaSuccess || (e = dalloc((void**)&h->n_defer, 4)) != cudaSuccess ||
        (e = dalloc((void**)&h->work_order, B * 4)) != cudaSuccess || (e = dalloc((void**)&h->order_cnt, 2 * kOrderBuckets * sizeof(int))) != cudaSuccess) {
        hmpc_destroy(h);
        return fail(HMPC_ERR_ALLOC, std::string("cudaMalloc: ") + cudaGetErrorString(e));
    }
    if ((e = cudaMemset(h->Xsol, 0, (N + 1) * 12 * B * 8)) != cudaSuccess || (e = cudaMemset(h->Usol, 0, N * 6 * B * 8)) != cudaSuccess ||
        (e = cudaMemset(h->code, 0, 11 * N * B)) != cudaSuccess || (e = cudaMemset(h->valid, 0, B)) != cudaSuccess ||
        (e = cudaMemset(h->st_tick, 0, B * 4)) != cudaSuccess || (e = cudaMemset(h->nfac, 0, B * 4)) != cudaSuccess ||
        (e = cudaMemset(h->path, 0, B * 4)) != cudaSuccess || (e = cudaMemset(h->ninf, 0, B * 4)) != cudaSuccess ||
        (e = cudaMemset(h->flops, 0, B * 8)) != cudaSuccess || (e = cudaMemset(h->work_ctr, 0, 64)) != cudaSuccess ||
        (e = cudaMemset(h->n_defer, 0, 4)) != cudaSuccess) {
        hmpc_destroy(h);
        return fail(HMPC_ERR_CUDA, std::string("cudaMemset: ") + cudaGetErrorString(e));
    }
    // default gains = the reference's (mpc_cvx_euler_3f.py:35,37)
    {
        const double Qref[12] = {50., 50., 2., 1., 1., 50., 1., 1., 1., 10., 10., 10.};
        double* tmp = new (std::nothrow) double[18 * B];
        if (!tmp) { hmpc_destroy(h); return fail(HMPC_ERR_ALLOC, "host allocation failed"); }
        for (size_t i = 0; i < 12; ++i) for (size_t b = 0; b < B; ++b) tmp[i * B + b] = Qref[i];
        for (size_t i = 0; i < 6; ++i) for (size_t b = 0; b < B; ++b) tmp[(12 + i) * B + b] = 0.001;
        e = cudaMemcpy(h->Qd, tmp, 12 * B * 8, cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaMemcpy(h->Rd, tmp + 12 * B, 6 * B * 8, cudaMemcpyHostToDevice);
        delete[] tmp;
        if (e != cudaSuccess) { hmpc_destroy(h); return fail(HMPC_ERR_CUDA, std::string("cudaMemcpy gains: ") + cudaGetErrorString(e)); }
    }
    if (g.ws_bytes && (e = cudaMalloc((void**)&h->ws, g.ws_bytes)) != cudaSuccess) {
        hmpc_destroy(h);
        return fail(HMPC_ERR_ALLOC, std::string("cudaMalloc workspace: ") + cudaGetErrorString(e));
    }
    // the attribute is process-global per kernel: always the device maximum (minus room for static shared memory),
    // so that a second handle never lowers it for the first
    const int smem_i = (int)prop.sharedMemPerBlockOptin - 512;
    if ((e = cta_set_smem(g.cta, smem_i)) != cudaSuccess ||
        (e = cudaFuncSetAttribute(hmpc::condense_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_i)) != cudaSuccess ||
        (e = cudaFuncSetAttribute(hmpc::linearize_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_i)) != cudaSuccess) {
        hmpc_destroy(h);
        return fail(HMPC_ERR_CUDA, std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(e));
    }
    // warp-per-hopper warm path: QP records of the prep kernel, warm blocks
    if (g.warp) {
        h->pstride = hmpc::prep_stride((int)N);
        if ((e = cudaMalloc((void**)&h->prep, B * h->pstride * 8)) != cudaSuccess ||
            (e = cudaMalloc((void**)&h->warm, B * (size_t)hmpc::warm_stride_doubles((int)N) * 8)) != cudaSuccess ||
            (e = cudaMalloc((void**)&h->warm_ok, B)) != cudaSuccess || (e = cudaMemset(h->warm_ok, 0, B)) != cudaSuccess ||
            (e = cudaMalloc((void**)&h->prep_flag, B * 4)) != cudaSuccess) {
            hmpc_destroy(h);
            return fail(HMPC_ERR_ALLOC, std::string("cudaMalloc QP records: ") + cudaGetErrorString(e));
        }
        if ((e = g.admm ? hmpc::warp_admm_set_smem(g.wpc, smem_i) : hmpc::warp_set_smem(g.wpc, smem_i)) != cudaSuccess ||
            (e = hmpc::prep_set_smem(smem_i)) != cudaSuccess) {
            hmpc_destroy(h);
            return fail(HMPC_ERR_CUDA, std::string("cudaFuncSetAttribute (warp kernel): ") + cudaGetErrorString(e));
        }
    }
    if (const char* ev = getenv("HMPC_WORK_ORDER")) h->order_on = atoi(ev) ? 1 : 0;
    // overlapped rollout schedule: a second stream, of higher priority so that the deferred hoppers' CTAs are placed
    // first as SM slots free up; HMPC_DEFER_SERIAL=1 keeps every tick on the handle's stream (A/B runs, tests)
    const char* serial = getenv("HMPC_DEFER_SERIAL");
    if (g.warp && !(serial && atoi(serial))) {
        int prio_lo = 0, prio_hi = 0;
        if ((e = cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi)) != cudaSuccess ||
            (e = cudaStreamCreateWithPriority(&h->side, cudaStreamNonBlocking, prio_hi)) != cudaSuccess ||
            (e = cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming)) != cudaSuccess ||
            (e = cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming)) != cudaSuccess ||
            (e = cudaMalloc((void**)&h->defer_mark, B * 4)) != cudaSuccess ||
            (e = cudaMemset(h->defer_mark, 0xff, B * 4)) != cudaSuccess) {    // -1: no overlapped tick has that number
            hmpc_destroy(h);
            return fail(HMPC_ERR_CUDA, std::string("create (side stream): ") + cudaGetErrorString(e));
        }
    }
    if ((e = cudaDeviceSynchronize()) != cudaSuccess) {
        hmpc_destroy(h);
        return fail(HMPC_ERR_CUDA, std::string("create: ") + cudaGetErrorString(e));
    }
    *out = h;
    return HMPC_OK;
}

int hmpc_destroy(hmpc_handle* h) {
    if (!h) return HMPC_OK;
    cudaSetDevice(h->cfg.device);
    cudaFree(h->Qd); cudaFree(h->Rd); cudaFree(h->Xsol); cudaFree(h->Usol); cudaFree(h->xin);
    cudaFree(h->U0); cudaFree(h->st_tmp); cudaFree(h->it_tmp); cudaFree(h->ws);
    cudaFree(h->code); cudaFree(h->valid); cudaFree(h->st_tick); cudaFree(h->nfac); cudaFree(h->path); cudaFree(h->ninf); cudaFree(h->flops); cudaFree(h->work_ctr);
    cudaFree(h->plan_sin); cudaFree(h->plan_pfidx); cudaFree(h->plan_cmask); cudaFree(h->plan_sw);
    cudaFree(h->win_xref); cudaFree(h->win_pf); cudaFree(h->win_C); cudaFree(h->win_sw);
    cudaFree(h->gate_glob);
    cudaFree(h->prep); cudaFree(h->prep_flag); cudaFree(h->defer_list); cudaFree(h->n_defer);
    cudaFree(h->work_order); cudaFree(h->order_cnt); cudaFree(h->warm); cudaFree(h->warm_ok);
    cudaFree(h->body_model); cudaFree(h->body_plant); cudaFree(h->body_bad); cudaFree(h->defer_mark);
    for (cudaEvent_t e : h->ev) cudaEventDestroy(e);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    if (h->side) cudaStreamDestroy(h->side);
    delete h;
    return HMPC_OK;
}

int hmpc_set_stream(hmpc_handle* h, void* s) {
    if (int rc = check_handle(h)) return rc;
    h->stream = (cudaStream_t)s;
    return HMPC_OK;
}

int hmpc_synchronize(hmpc_handle* h) {
    if (int rc = check_handle(h)) return rc;
    HMPC_CUDA(cudaStreamSynchronize(h->stream));
    return HMPC_OK;
}

int hmpc_set_gains(hmpc_handle* h, const double* Qdiag, const double* Rdiag) {
    if (int rc = check_handle(h)) return rc;
    const size_t B = (size_t)h->cfg.batch;
    if (Qdiag) HMPC_CUDA(cudaMemcpyAsync(h->Qd, Qdiag, 12 * B * 8, cudaMemcpyDeviceToDevice, h->stream));
    if (Rdiag) HMPC_CUDA(cudaMemcpyAsync(h->Rd, Rdiag, 6 * B * 8, cudaMemcpyDeviceToDevice, h->stream));
    return HMPC_OK;
}

int hmpc_set_body_params(hmpc_handle* h, int which, const double* m, const double* J, const double* Jinv, const double* rh,
                         const double* mu) {
    if (int rc = check_handle(h)) return rc;
    if (which != HMPC_BODY_MODEL && which != HMPC_BODY_PLANT && which != HMPC_BODY_BOTH)
        return fail(HMPC_ERR_BAD_ARG, "which must be HMPC_BODY_MODEL, HMPC_BODY_PLANT or HMPC_BODY_BOTH");
    if (J && which == HMPC_BODY_MODEL) return fail(HMPC_ERR_BAD_ARG, "J is a plant quantity: the MPC model uses Jinv only");
    if (mu && which == HMPC_BODY_PLANT) return fail(HMPC_ERR_BAD_ARG, "mu is a model quantity: the simulator has no friction");
    const bool model = which & HMPC_BODY_MODEL, plant = which & HMPC_BODY_PLANT;
    if (!m && !J && !Jinv && !rh && !mu) {          // back to the config's scalars for every hopper
        if (model) h->model_on = false;
        if (plant) h->plant_on = false;
        return HMPC_OK;
    }
    const int Bi = h->cfg.batch, grid = (Bi + 127) / 128;
    const size_t B = (size_t)Bi;
    if (!h->body_bad) HMPC_CUDA(cudaMalloc((void**)&h->body_bad, sizeof(int)));
    if (model && !h->body_model) HMPC_CUDA(cudaMalloc((void**)&h->body_model, hmpc::kBodyModel * B * 8));
    if (plant && !h->body_plant) HMPC_CUDA(cudaMalloc((void**)&h->body_plant, hmpc::kBodyPlant * B * 8));
    // validate what was given before anything is replaced: a rejected call leaves the handle as it was
    int bad = INT32_MAX;
    HMPC_CUDA(cudaMemcpyAsync(h->body_bad, &bad, sizeof(int), cudaMemcpyHostToDevice, h->stream));
    hmpc::body_check_kernel<<<grid, 128, 0, h->stream>>>(Bi, m, J, Jinv, rh, mu, h->body_bad);
    ++h->launches;
    HMPC_CUDA(cudaGetLastError());
    HMPC_CUDA(cudaMemcpyAsync(&bad, h->body_bad, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    HMPC_CUDA(cudaStreamSynchronize(h->stream));
    if (bad != INT32_MAX)
        return fail(HMPC_ERR_BAD_ARG, "hmpc_set_body_params: hopper " + std::to_string(bad) +
                                          " has a non-finite value, m <= 0 or mu < 0");
    // one target: rows of the given arrays copied, the other rows filled with the config's scalars
    auto set = [&](double* dst, int r_m, int r_rh, int r_J, int r_Jinv, int r_mu) -> int {
        hmpc::BodyFill f;
        f.mask = 0;
        auto row = [&](int r0, int nr, const double* src, const double* scal) -> int {
            if (r0 < 0) return HMPC_OK;
            if (src) {
                HMPC_CUDA(cudaMemcpyAsync(dst + (size_t)r0 * B, src, (size_t)nr * B * 8, cudaMemcpyDeviceToDevice, h->stream));
            } else {
                for (int i = 0; i < nr; ++i) { f.v[r0 + i] = scal[i]; f.mask |= 1u << (r0 + i); }
            }
            return HMPC_OK;
        };
        int rc;
        if ((rc = row(r_m, 1, m, &h->cfg.m)) || (rc = row(r_rh, 3, rh, h->cfg.rh)) || (rc = row(r_J, 9, J, h->cfg.J)) ||
            (rc = row(r_Jinv, 9, Jinv, h->cfg.Jinv)) || (rc = row(r_mu, 1, mu, &h->cfg.mu)))
            return rc;
        if (f.mask) {
            hmpc::body_fill_kernel<<<grid, 128, 0, h->stream>>>(Bi, dst, f);
            ++h->launches;
            HMPC_CUDA(cudaGetLastError());
        }
        return HMPC_OK;
    };
    // row order: QpConst::body = m, mu, rh, Jinv (hmpc::Body); SimConst::body = m, rh, J, Jinv (hmpc::plant_body)
    if (model) {
        if (int rc = set(h->body_model, 0, 2, -1, 5, 1)) return rc;
        h->model_on = true;
    }
    if (plant) {
        if (int rc = set(h->body_plant, 0, 1, 4, 13, -1)) return rc;
        h->plant_on = true;
    }
    return HMPC_OK;
}

int hmpc_convert(hmpc_handle* h, const double* X, double* x) {
    if (int rc = check_handle(h)) return rc;
    if (!X || !x) return fail(HMPC_ERR_BAD_ARG, "null array");
    const int B = h->cfg.batch;
    hmpc::convert_kernel<<<(B + 127) / 128, 128, 0, h->stream>>>(B, X, x);
    ++h->launches;
    HMPC_CUDA(cudaGetLastError());
    return HMPC_OK;
}

int hmpc_rk4(hmpc_handle* h, double* X, const double* U, const double* pf, int nsteps, double* X_steps) {
    if (int rc = check_handle(h)) return rc;
    if (!X || !U || !pf || nsteps < 0) return fail(HMPC_ERR_BAD_ARG, "bad argument");
    const int B = h->cfg.batch;
    launch_sim(sim_const(h), (B + 127) / 128, h->stream, B, hmpc::HopperSet{}, X, U, pf, (const double*)nullptr, (const uint8_t*)nullptr, nsteps,
               (double*)nullptr, (double*)nullptr, (double*)nullptr, X_steps, (const int32_t*)nullptr, (const double*)nullptr,
               hmpc::SimGate{HMPC_GATE_OFF, nullptr, nullptr, nullptr, 0, 0, 0.0});
    ++h->launches;
    HMPC_CUDA(cudaGetLastError());
    return HMPC_OK;
}

int hmpc_linearize(hmpc_handle* h, const double* x_guess, const double* pf, double* Ad, double* Bd) {
    if (int rc = check_handle(h)) return rc;
    if (!x_guess || !pf || !Ad || !Bd) return fail(HMPC_ERR_BAD_ARG, "null array");
    const size_t vec_bytes = ((hmpc::work_vec_doubles(h->cfg.N) + 1) & ~(size_t)1) * 8;
    hmpc::linearize_kernel<<<h->cfg.batch, 128, vec_bytes, h->stream>>>(qp_const(h), h->cfg.batch,
                                                                        x_guess, pf, Ad, Bd);
    ++h->launches;
    HMPC_CUDA(cudaGetLastError());
    return HMPC_OK;
}

int hmpc_condense(hmpc_handle* h, const double* x_in, const double* x_guess, const double* x_ref,
                  const double* pf, const uint64_t* Cbits, double* H, double* g, double* lo, double* hi,
                  int32_t* infeasible) {
    if (int rc = check_handle(h)) return rc;
    if (!x_in || !x_guess || !x_ref || !pf || !Cbits || !H || !g || !lo || !hi)
        return fail(HMPC_ERR_BAD_ARG, "null array");
    hmpc::condense_kernel<<<h->geo.grid, h->geo.threads, h->geo.smem, h->stream>>>(
        qp_const(h), h->cfg.batch, h->geo.ws_bytes ? 0 : 1, h->ws, x_in, x_guess, x_ref, pf, Cbits,
        h->Qd, h->Rd, H, g, lo, hi, infeasible);
    ++h->launches;
    HMPC_CUDA(cudaGetLastError());
    return HMPC_OK;
}

namespace {
// small horizons: 128 threads, registers capped so that four CTAs share an SM; large: 256 threads
// work_ctr: [0] next hopper of the warp kernel, [1] deferred hoppers, [2] next entry of the CTA kernel
// ------------------------------------------------------------------------------------------------
// Work order of the lock-step solve kernel.  The warps of an SM run their active-set trials in step, so a round lasts
// as long as its slowest trial; hoppers with the same contact schedule over the horizon have systems of similar
// size and shape.  Every tick the hoppers are therefore grouped by their contact mask (a counting sort on a 12-bit
// hash of the mask: equal masks share a bucket, a rare collision merges two groups and costs nothing but a little of
// the grouping) and the persistent warps take them in that order.  Measured, 131072 hoppers with ten gait phases mixed
// at random: 8.56 -> 9.07-9.17 M steps/s (15.2 -> 14.2 ms per tick).  The size class of each hopper's previous system as a
// second key was measured as well: no further gain (9.04 M).  The prep kernel keeps the natural order: it has no
// lock-step, and neighbouring warps share memory sectors there (8.89 M with it reordered).  Results do not depend on the order (tests/test_gpu.py: work-order stress test).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int order_bucket(uint64_t mask) { return (int)((mask * 0x9E3779B97F4A7C15ull) >> 52); }
__global__ void order_count_kernel(const uint64_t* __restrict__ Cbits, int B, int* __restrict__ cnt) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < B) atomicAdd(&cnt[order_bucket(Cbits[b])], 1);
}
// exclusive scan of the kOrderBuckets bucket sizes into the cursors (one block of 1024 threads, four buckets each)
__global__ void order_scan_kernel(const int* __restrict__ cnt, int* __restrict__ cur) {
    __shared__ int part[1024];
    const int t = threadIdx.x;
    int v[4], s = 0;
    for (int q = 0; q < 4; ++q) { v[q] = cnt[4 * t + q]; s += v[q]; }
    part[t] = s;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
        const int add = t >= o ? part[t - o] : 0;
        __syncthreads();
        part[t] += add;
        __syncthreads();
    }
    int base = part[t] - s;
    for (int q = 0; q < 4; ++q) { cur[4 * t + q] = base; base += v[q]; }
}
__global__ void order_scatter_kernel(const uint64_t* __restrict__ Cbits, int B, int* __restrict__ cur, int* __restrict__ order) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < B) order[atomicAdd(&cur[order_bucket(Cbits[b])], 1)] = b;
}

// adds the tick's deferral count to n_defer; with mark set, also stamps every deferred hopper with the tick's number
__global__ void defer_stats_kernel(const int* __restrict__ work_ctr, int32_t* __restrict__ n_defer, const int* __restrict__ list,
                                   int32_t* __restrict__ mark, int seq) {
    const int cnt = work_ctr[1];
    if (blockIdx.x == 0 && threadIdx.x == 0) *n_defer += cnt;
    if (mark)
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < cnt; i += gridDim.x * blockDim.x) mark[list[i] & hmpc::kListHopperMask] = seq;
}

// counters / deferral list of a tick: overlapped ticks alternate between two sets by the parity of their number, so
// that the next tick's reset never touches what the CTA kernel of the previous tick still reads on the side stream
int* tick_ctr(hmpc_handle* h, int par) { return h->work_ctr + 8 * par; }
int* tick_list(hmpc_handle* h, int par) { return h->defer_list + (size_t)par * h->cfg.batch; }

hmpc::WarpLaunch warp_launch_of(hmpc_handle* h, int par, cudaStream_t st) {
    int* ctr = tick_ctr(h, par);
    const hmpc::Geometry& g = h->geo;
    return hmpc::WarpLaunch{g.warp_grid, g.wpc, g.group, g.warp_smem, st, h->cfg.batch, g.kcap, g.wdoubles, h->prep, h->pstride,
                            h->prep_flag, ctr, tick_list(h, par), ctr + 1, g.admm ? 1 : 0};
}

// One tick's solve on h->stream.  overlap (warp path only): the tick takes the buffers of parity h->seq & 1, the prep
// kernel leaves out the hoppers the side stream condenses (h->side_prep), the warp kernel waits for those, h->ev_fork
// marks the complete deferral list, and the CTA kernel over that list is left to the caller (rollout_impl).
cudaError_t launch_mpc(hmpc_handle* h, const hmpc::QpConst& qc, const hmpc::MpcIo& io, bool overlap = false) {
    const int par = overlap ? (h->seq & 1) : 0;
    int* ctr = tick_ctr(h, par);
    cudaError_t e = cudaMemsetAsync(ctr, 0, 4 * sizeof(int), h->stream);
    if (e != cudaSuccess) return e;
    const bool warp = h->geo.warp && hmpc::warp_path_applies(h->cfg, io.init);
    if (warp) {
        const hmpc::WarpLaunch wl = warp_launch_of(h, par, h->stream);
        hmpc::HopperSet ps;
        if (overlap && h->side_prep) { ps.mark = h->defer_mark; ps.skip = h->seq - 1; }
        hmpc::prep_launch(wl, qc, io, ps);   // natural order: no lock-step there, and neighbouring warps share sectors (measured)
        hmpc::QpConst qo = qc;
        if (h->order_on && !h->geo.admm) {
            // group the hoppers by contact schedule for the lock-step kernel (see order_count_kernel)
            const int Bi = h->cfg.batch, grid = (Bi + 255) / 256;
            if ((e = cudaMemsetAsync(h->order_cnt, 0, kOrderBuckets * sizeof(int), h->stream)) != cudaSuccess) return e;
            order_count_kernel<<<grid, 256, 0, h->stream>>>(io.Cbits, Bi, h->order_cnt);
            order_scan_kernel<<<1, 1024, 0, h->stream>>>(h->order_cnt, h->order_cnt + kOrderBuckets);
            order_scatter_kernel<<<grid, 256, 0, h->stream>>>(io.Cbits, Bi, h->order_cnt + kOrderBuckets, h->work_order);
            h->launches += 3;
            qo.work_order = h->work_order;
        }
        if (overlap && h->side_prep && (e = cudaStreamWaitEvent(h->stream, h->ev_join, 0)) != cudaSuccess) return e;
        if ((e = hmpc::warp_launch(wl, qo, io)) != cudaSuccess) return e;
        if (overlap) {
            if ((e = cudaEventRecord(h->ev_fork, h->stream)) != cudaSuccess) return e;
            defer_stats_kernel<<<h->sm_count, 256, 0, h->stream>>>(ctr, h->n_defer, tick_list(h, par), h->defer_mark, h->seq);
        } else {
            defer_stats_kernel<<<1, 1, 0, h->stream>>>(ctr, h->n_defer, nullptr, nullptr, 0);
        }
        h->launches += 3;
        if (overlap) return cudaGetLastError();
    }
    const hmpc::MpcLaunch l{h->geo.grid, h->geo.threads, h->geo.smem, h->stream, h->cfg.batch, h->sm_count, h->ws,
                            ctr + 2, warp ? tick_list(h, par) : nullptr, warp ? ctr + 1 : nullptr};
    if ((e = launch_cta(h, l, qc, io)) != cudaSuccess) return e;
    return cudaGetLastError();
}

hmpc::MpcIo make_io(hmpc_handle* h, const double* x_in, const double* x_ref, const double* pf,
                    const uint64_t* Cbits, int init, int accumulate, double* U, double* Xsol, double* U0,
                    int32_t* status, int32_t* iters) {
    hmpc::MpcIo io;
    io.x_in = x_in; io.x_ref = x_ref; io.pf = pf; io.Cbits = Cbits; io.Qd = h->Qd; io.Rd = h->Rd;
    io.Xsol = h->Xsol; io.Usol = h->Usol; io.code = h->code; io.valid = h->valid;
    if (h->warm) {
        io.warm = h->warm; io.warm_ok = h->warm_ok; io.warm_stride = hmpc::warm_stride_doubles(h->cfg.N);
    }
    io.U_out = U; io.X_out = Xsol; io.U0_out = U0;
    io.status = status ? status : h->st_tmp; io.iters = iters ? iters : h->it_tmp;
    io.st_tick = h->st_tick; io.nfac = h->nfac; io.path = h->path; io.ninf = h->ninf; io.flops = h->flops;
    io.init = init; io.accumulate = accumulate;
    io.respawn = (h->cfg.on_infeasible == HMPC_INFEASIBLE_RESPAWN) ? 1 : 0;
    return io;
}
}  // namespace

int hmpc_solve(hmpc_handle* h, const double* x_in, const double* x_ref, const double* pf,
               const uint64_t* Cbits, int init, double* U, double* Xsol, int32_t* status, int32_t* iters) {
    if (int rc = check_handle(h)) return rc;
    if (!x_in || !x_ref || !pf || !Cbits) return fail(HMPC_ERR_BAD_ARG, "null input array");
    hmpc::MpcIo io = make_io(h, x_in, x_ref, pf, Cbits, init ? 1 : 0, 0, U, Xsol, nullptr, status, iters);
    io.respawn = 0;   // per-hopper re-initialisation only exists inside hmpc_rollout
    HMPC_CUDA(cudaMemsetAsync(h->n_defer, 0, 4, h->stream));
    HMPC_CUDA(launch_mpc(h, qp_const(h), io));
    return HMPC_OK;
}

namespace {
// One closed-loop run.  planned = false: rows of the caller's tables; planned = true: every tick writes its own window
// (N+1 reference / footstep rows, contact mask, switch step) with the device planner first.
int rollout_impl(hmpc_handle* h, bool planned, double* X, const double* xref_tab, const double* pf_tab,
                 const uint64_t* C_tab, const uint8_t* pf_switch, int tick0, int n_ticks, int init,
                 double* X_log, double* U_log, int32_t* status, int32_t* iters) {
    const size_t B = (size_t)h->cfg.batch;
    const int Bi = h->cfg.batch, N = h->cfg.N;
    int32_t* st = status ? status : h->st_tmp;
    int32_t* it = iters ? iters : h->it_tmp;
    HMPC_CUDA(cudaMemsetAsync(st, 0, B * 4, h->stream));
    HMPC_CUDA(cudaMemsetAsync(it, 0, B * 4, h->stream));
    HMPC_CUDA(cudaMemsetAsync(h->nfac, 0, B * 4, h->stream));
    HMPC_CUDA(cudaMemsetAsync(h->ninf, 0, B * 4, h->stream));
    HMPC_CUDA(cudaMemsetAsync(h->flops, 0, B * 8, h->stream));
    HMPC_CUDA(cudaMemsetAsync(h->n_defer, 0, 4, h->stream));
    if (h->timing) {
        while ((int)h->ev.size() < kTickEvents * n_ticks) {
            cudaEvent_t e;
            HMPC_CUDA(cudaEventCreate(&e));
            h->ev.push_back(e);
        }
        h->ev_side.assign(n_ticks, 0);
    }
    h->ev_ticks = h->timing ? n_ticks : 0;
    if (h->gate_mode == HMPC_GATE_SCHEDULE && (planned ? !h->gate_glob : !h->gate_tab))
        return fail(HMPC_ERR_BAD_ARG, planned ? "HMPC_GATE_SCHEDULE: hmpc_set_contact_gate was given no gate_glob for hmpc_rollout_planned"
                                              : "HMPC_GATE_SCHEDULE: hmpc_set_contact_gate was given no gate_tab for hmpc_rollout");
    const hmpc::QpConst qc = qp_const(h);
    const hmpc::SimConst sc = sim_const(h);
    const int sim_grid = (Bi + 127) / 128;
    const bool respawn = h->cfg.on_infeasible == HMPC_INFEASIBLE_RESPAWN;
    // x_in for the first tick; afterwards sim_kernel emits it fused with the integration
    hmpc::convert_kernel<<<sim_grid, 128, 0, h->stream>>>(Bi, X, h->xin);
    ++h->launches;
    if (X_log) HMPC_CUDA(cudaMemcpyAsync(X_log, X, 13 * B * 8, cudaMemcpyDeviceToDevice, h->stream));
    // Overlapped schedule (DESIGN.md section 5): with more than one tick from the caller's tables, the CTA kernel over a
    // warm tick's deferred hoppers, their simulator step and their next condensing run on h->side while h->stream
    // simulates and condenses every other hopper.  The planned rollout rewrites one reference window per tick, which
    // the side stream would still read: it keeps the serial schedule.
    const bool overlap = h->side && !planned && n_ticks > 1;
    h->side_prep = false;
    bool joined = true;
    for (int t = 0; t < n_ticks; ++t) {
        const double *xr, *pf;
        const uint64_t* Cm;
        const uint8_t* sw;
        auto table_rows = [&](int tt) {
            const size_t row = (size_t)(tick0 + tt);
            xr = xref_tab + row * 12 * B; pf = pf_tab + row * 3 * B; Cm = C_tab + row * B;
            sw = pf_switch ? pf_switch + row * B : nullptr;
        };
        if (planned) {
            hmpc::plan_rows_kernel<<<dim3(sim_grid, N + 1), 128, 0, h->stream>>>(h->plan, Bi, tick0 + t, N + 1, N + 1, h->win_xref, h->win_pf);
            hmpc::plan_masks_kernel<<<dim3(sim_grid, 1), 128, 0, h->stream>>>(h->plan, Bi, tick0 + t, 1, h->win_pf, h->win_C, h->win_sw);
            h->launches += 2;
            xr = h->win_xref; pf = h->win_pf; Cm = h->win_C; sw = h->win_sw;
        } else {
            table_rows(t);
        }
        hmpc::SimGate gate{h->gate_mode, nullptr, nullptr, nullptr, tick0 + t, h->gate_max_tick, h->leg_max * h->leg_max};
        if (h->gate_mode == HMPC_GATE_SCHEDULE) {
            if (planned) { gate.glob = h->gate_glob; gate.off = h->plan.off; }
            else gate.bits = h->gate_tab + (size_t)(tick0 + t) * B;
        }
        hmpc::MpcIo io = make_io(h, h->xin, xr, pf, Cm, (init && t == 0) ? 1 : 0, 1, nullptr, nullptr, h->U0, st, it);
        const bool ov = overlap && hmpc::warp_path_applies(h->cfg, io.init);
        cudaEvent_t* ev = h->timing ? &h->ev[(size_t)kTickEvents * t] : nullptr;
        if (ev) HMPC_CUDA(cudaEventRecord(ev[0], h->stream));
        HMPC_CUDA(launch_mpc(h, qc, io, ov));
        if (ev) HMPC_CUDA(cudaEventRecord(ev[1], h->stream));
        // sim_main: every hopper but the ones deferred in this tick (their controls are not solved yet)
        hmpc::HopperSet main_set;
        if (ov) { main_set.mark = h->defer_mark; main_set.skip = h->seq; }
        auto sim = [&](cudaStream_t s, const hmpc::HopperSet& hs) {
            launch_sim(sc, sim_grid, s,
                Bi, hs, X, (const double*)h->U0, pf, pf + 3 * B, sw, h->cfg.mpc_factor, h->xin,
                X_log ? X_log + (size_t)(t + 1) * 13 * B : nullptr, U_log ? U_log + (size_t)t * 6 * B : nullptr,
                (double*)nullptr, respawn ? (const int32_t*)h->st_tick : nullptr, respawn ? xr + 12 * B : nullptr, gate);
            ++h->launches;
        };
        sim(h->stream, main_set);
        if (ev) HMPC_CUDA(cudaEventRecord(ev[2], h->stream));
        if (!ov) continue;
        // side stream: the deferred hoppers of this tick -- CTA kernel, simulator step, next tick's condensing.  Every
        // kernel here reads and writes the columns of these hoppers only (per-hopper state, outputs, prep records); the
        // CTA workspace and this parity's counters / list are not used by the main stream until it waits on ev_join.
        const int par = h->seq & 1;
        int* ctr = tick_ctr(h, par);
        hmpc::HopperSet dset;
        dset.list = tick_list(h, par); dset.list_cnt = ctr + 1;
        HMPC_CUDA(cudaStreamWaitEvent(h->side, h->ev_fork, 0));
        if (ev) HMPC_CUDA(cudaEventRecord(ev[3], h->side));
        HMPC_CUDA(launch_cta(h, hmpc::MpcLaunch{h->geo.grid, h->geo.threads, h->geo.smem, h->side, Bi, h->sm_count, h->ws, ctr + 2,
                                                dset.list, dset.list_cnt},
                             qc, io));
        if (ev) HMPC_CUDA(cudaEventRecord(ev[4], h->side));
        sim(h->side, dset);
        if (ev) { HMPC_CUDA(cudaEventRecord(ev[5], h->side)); h->ev_side[t] = 1; }
        h->side_prep = t + 1 < n_ticks;
        if (h->side_prep) {
            table_rows(t + 1);
            const hmpc::MpcIo io_next = make_io(h, h->xin, xr, pf, Cm, 0, 1, nullptr, nullptr, h->U0, st, it);
            hmpc::prep_launch(warp_launch_of(h, par, h->side), qc, io_next, dset);
            ++h->launches;
        }
        HMPC_CUDA(cudaEventRecord(h->ev_join, h->side));
        joined = false;
        ++h->seq;
    }
    // the caller's stream sees the whole rollout
    if (!joined) HMPC_CUDA(cudaStreamWaitEvent(h->stream, h->ev_join, 0));
    h->side_prep = false;
    HMPC_CUDA(cudaGetLastError());
    return HMPC_OK;
}
}  // namespace

int hmpc_rollout(hmpc_handle* h, double* X, const double* xref_tab, const double* pf_tab,
                 const uint64_t* C_tab, const uint8_t* pf_switch, int tick0, int n_ticks, int init,
                 double* X_log, double* U_log, int32_t* status, int32_t* iters) {
    if (int rc = check_handle(h)) return rc;
    if (!X || !xref_tab || !pf_tab || !C_tab || tick0 < 0 || n_ticks < 0)
        return fail(HMPC_ERR_BAD_ARG, "bad argument");
    return rollout_impl(h, false, X, xref_tab, pf_tab, C_tab, pf_switch, tick0, n_ticks, init, X_log, U_log, status, iters);
}

int hmpc_plan_set(hmpc_handle* h, const hmpc_plan_config* pc, const double* x0, const double* xf, const int32_t* curve,
                  const int32_t* tick_offset, const double* sin_tab_host, const int32_t* pf_idx_host,
                  const uint64_t* cmask_host, const uint8_t* sw_glob_host) {
    if (int rc = check_handle(h)) return rc;
    if (!pc || !x0 || !xf || !curve || !tick_offset || !sin_tab_host || !pf_idx_host || !cmask_host || !sw_glob_host)
        return fail(HMPC_ERR_BAD_ARG, "null argument");
    if (pc->N_run < 2 || pc->n_sim < 1 || pc->max_tick < 1 || !(pc->t_p > 0.0)) return fail(HMPC_ERR_BAD_ARG, "bad plan config");
    const size_t B = (size_t)h->cfg.batch, N = (size_t)h->cfg.N;
    h->plan_ok = false;
    cudaFree(h->plan_sin); cudaFree(h->plan_pfidx); cudaFree(h->plan_cmask); cudaFree(h->plan_sw);
    h->plan_sin = nullptr; h->plan_pfidx = nullptr; h->plan_cmask = nullptr; h->plan_sw = nullptr;
    cudaError_t e;
    if ((e = cudaMalloc((void**)&h->plan_sin, (size_t)pc->n_sim * 8)) != cudaSuccess ||
        (e = cudaMalloc((void**)&h->plan_pfidx, (size_t)pc->n_sim * 4)) != cudaSuccess ||
        (e = cudaMalloc((void**)&h->plan_cmask, (size_t)pc->max_tick * 8)) != cudaSuccess ||
        (e = cudaMalloc((void**)&h->plan_sw, (size_t)pc->max_tick)) != cudaSuccess)
        return fail(HMPC_ERR_ALLOC, std::string("cudaMalloc plan tables: ") + cudaGetErrorString(e));
    if (!h->win_xref) {
        if ((e = cudaMalloc((void**)&h->win_xref, (N + 1) * 12 * B * 8)) != cudaSuccess ||
            (e = cudaMalloc((void**)&h->win_pf, (N + 1) * 3 * B * 8)) != cudaSuccess ||
            (e = cudaMalloc((void**)&h->win_C, B * 8)) != cudaSuccess || (e = cudaMalloc((void**)&h->win_sw, B)) != cudaSuccess)
            return fail(HMPC_ERR_ALLOC, std::string("cudaMalloc plan windows: ") + cudaGetErrorString(e));
    }
    // the host tables may be pageable: synchronous copies, ordered before later work on the handle's stream
    HMPC_CUDA(cudaStreamSynchronize(h->stream));
    HMPC_CUDA(cudaMemcpy(h->plan_sin, sin_tab_host, (size_t)pc->n_sim * 8, cudaMemcpyHostToDevice));
    HMPC_CUDA(cudaMemcpy(h->plan_pfidx, pf_idx_host, (size_t)pc->n_sim * 4, cudaMemcpyHostToDevice));
    HMPC_CUDA(cudaMemcpy(h->plan_cmask, cmask_host, (size_t)pc->max_tick * 8, cudaMemcpyHostToDevice));
    HMPC_CUDA(cudaMemcpy(h->plan_sw, sw_glob_host, (size_t)pc->max_tick, cudaMemcpyHostToDevice));
    hmpc::PlanConst& P = h->plan;
    P.N = h->cfg.N; P.mpc_factor = h->cfg.mpc_factor; P.N_run = pc->N_run; P.t_ref = pc->N_run + h->cfg.N * h->cfg.mpc_factor;
    P.n_sim = pc->n_sim; P.max_tick = pc->max_tick; P.dt = h->cfg.sim_dt; P.amp = pc->t_p / 4; P.T = (double)pc->N_run;
    P.curve_psi1 = pc->curve_psi1; P.curve_psi2 = pc->curve_psi2;
    P.sin_tab = h->plan_sin; P.pf_idx = h->plan_pfidx; P.cmask = h->plan_cmask; P.sw_glob = h->plan_sw;
    P.x0 = x0; P.xf = xf; P.curve = curve; P.off = tick_offset;
    h->plan_ok = true;
    return HMPC_OK;
}

int hmpc_plan_tables(hmpc_handle* h, int tick0, int n_ticks, double* xref_tab, double* pf_tab, uint64_t* C_tab,
                     uint8_t* pf_switch) {
    if (int rc = check_handle(h)) return rc;
    if (!h->plan_ok) return fail(HMPC_ERR_BAD_ARG, "hmpc_plan_set has not been called");
    if (!xref_tab || !pf_tab || !C_tab || !pf_switch || tick0 < 0 || n_ticks < 0) return fail(HMPC_ERR_BAD_ARG, "bad argument");
    const int Bi = h->cfg.batch, N = h->cfg.N, grid = (Bi + 127) / 128;
    const int nrows = n_ticks + N + 1;
    hmpc::plan_rows_kernel<<<dim3(grid, std::min(nrows, 64)), 128, 0, h->stream>>>(h->plan, Bi, tick0, nrows, nrows - 1, xref_tab, pf_tab);
    if (n_ticks > 0)
        hmpc::plan_masks_kernel<<<dim3(grid, std::min(n_ticks, 64)), 128, 0, h->stream>>>(h->plan, Bi, tick0, n_ticks, pf_tab, C_tab, pf_switch);
    h->launches += 2;
    HMPC_CUDA(cudaGetLastError());
    return HMPC_OK;
}

int hmpc_rollout_planned(hmpc_handle* h, double* X, int tick0, int n_ticks, int init, double* X_log, double* U_log,
                         int32_t* status, int32_t* iters) {
    if (int rc = check_handle(h)) return rc;
    if (!h->plan_ok) return fail(HMPC_ERR_BAD_ARG, "hmpc_plan_set has not been called");
    if (!X || tick0 < 0 || n_ticks < 0) return fail(HMPC_ERR_BAD_ARG, "bad argument");
    return rollout_impl(h, true, X, nullptr, nullptr, nullptr, nullptr, tick0, n_ticks, init, X_log, U_log, status, iters);
}

int hmpc_set_contact_gate(hmpc_handle* h, int mode, const uint32_t* gate_tab, const uint32_t* gate_glob_host, int max_tick,
                          double leg_max) {
    if (int rc = check_handle(h)) return rc;
    if (mode != HMPC_GATE_OFF && mode != HMPC_GATE_SCHEDULE && mode != HMPC_GATE_DETECT) return fail(HMPC_ERR_BAD_ARG, "unknown gate mode");
    if (mode == HMPC_GATE_SCHEDULE) {
        if (h->cfg.mpc_factor > 32) return fail(HMPC_ERR_UNSUPPORTED, "HMPC_GATE_SCHEDULE needs mpc_factor <= 32 (one mask bit per simulator step)");
        if (!gate_tab && !gate_glob_host) return fail(HMPC_ERR_BAD_ARG, "HMPC_GATE_SCHEDULE needs gate_tab or gate_glob");
        if (gate_glob_host && max_tick < 1) return fail(HMPC_ERR_BAD_ARG, "gate_glob needs max_tick >= 1");
    }
    if (mode == HMPC_GATE_DETECT && !(leg_max > 0.0)) return fail(HMPC_ERR_BAD_ARG, "HMPC_GATE_DETECT needs leg_max > 0");
    HMPC_CUDA(cudaStreamSynchronize(h->stream));          // the previous tables may still be in use
    cudaFree(h->gate_glob);
    h->gate_glob = nullptr; h->gate_tab = nullptr; h->gate_max_tick = 0; h->gate_mode = HMPC_GATE_OFF; h->leg_max = 0.0;
    if (mode == HMPC_GATE_SCHEDULE) {
        if (gate_glob_host) {
            cudaError_t e = cudaMalloc((void**)&h->gate_glob, (size_t)max_tick * 4);
            if (e != cudaSuccess) return fail(HMPC_ERR_ALLOC, std::string("cudaMalloc gate table: ") + cudaGetErrorString(e));
            HMPC_CUDA(cudaMemcpy(h->gate_glob, gate_glob_host, (size_t)max_tick * 4, cudaMemcpyHostToDevice));
            h->gate_max_tick = max_tick;
        }
        h->gate_tab = gate_tab;
    }
    if (mode == HMPC_GATE_DETECT) h->leg_max = leg_max;
    h->gate_mode = mode;
    return HMPC_OK;
}

int hmpc_set_timing(hmpc_handle* h, int enable) {
    if (int rc = check_handle(h)) return rc;
    h->timing = enable ? 1 : 0;
    return HMPC_OK;
}

namespace {
// solver and simulator device time of rollout tick t: the main-stream intervals plus, for an overlapped tick, the
// side-stream intervals of the deferred hoppers (which overlap the next tick's main-stream work)
int tick_time(hmpc_handle* h, int t, float* mpc, float* sim) {
    const cudaEvent_t* ev = &h->ev[(size_t)kTickEvents * t];
    HMPC_CUDA(cudaEventElapsedTime(mpc, ev[0], ev[1]));
    HMPC_CUDA(cudaEventElapsedTime(sim, ev[1], ev[2]));
    if (h->ev_side[t]) {
        float m = 0, s = 0;
        HMPC_CUDA(cudaEventElapsedTime(&m, ev[3], ev[4]));
        HMPC_CUDA(cudaEventElapsedTime(&s, ev[4], ev[5]));
        *mpc += m; *sim += s;
    }
    return HMPC_OK;
}
}  // namespace

int hmpc_kernel_times(hmpc_handle* h, double* mpc_ms, double* sim_ms, int* n_ticks) {
    if (int rc = check_handle(h)) return rc;
    HMPC_CUDA(cudaStreamSynchronize(h->stream));
    double a = 0.0, b = 0.0;
    for (int t = 0; t < h->ev_ticks; ++t) {
        float m1 = 0, m2 = 0;
        if (int rc = tick_time(h, t, &m1, &m2)) return rc;
        a += m1; b += m2;
    }
    if (mpc_ms) *mpc_ms = a;
    if (sim_ms) *sim_ms = b;
    if (n_ticks) *n_ticks = h->ev_ticks;
    return HMPC_OK;
}

int hmpc_tick_times(hmpc_handle* h, double* mpc_ms, double* sim_ms, int cap, int* n_ticks) {
    if (int rc = check_handle(h)) return rc;
    HMPC_CUDA(cudaStreamSynchronize(h->stream));
    const int n = h->ev_ticks < cap ? h->ev_ticks : cap;
    for (int t = 0; t < n; ++t) {
        float m1 = 0, m2 = 0;
        if (int rc = tick_time(h, t, &m1, &m2)) return rc;
        if (mpc_ms) mpc_ms[t] = m1;
        if (sim_ms) sim_ms[t] = m2;
    }
    if (n_ticks) *n_ticks = h->ev_ticks;
    return HMPC_OK;
}

int hmpc_solve_stats(hmpc_handle* h, int32_t* nfac, int32_t* path, int32_t* n_infeasible, double* flops) {
    if (int rc = check_handle(h)) return rc;
    const size_t B = (size_t)h->cfg.batch;
    if (flops) HMPC_CUDA(cudaMemcpyAsync(flops, h->flops, B * 8, cudaMemcpyDeviceToDevice, h->stream));
    if (nfac) HMPC_CUDA(cudaMemcpyAsync(nfac, h->nfac, B * 4, cudaMemcpyDeviceToDevice, h->stream));
    if (path) HMPC_CUDA(cudaMemcpyAsync(path, h->path, B * 4, cudaMemcpyDeviceToDevice, h->stream));
    if (n_infeasible) HMPC_CUDA(cudaMemcpyAsync(n_infeasible, h->ninf, B * 4, cudaMemcpyDeviceToDevice, h->stream));
    return HMPC_OK;
}

int hmpc_hot_path_info(hmpc_handle* h, int* warps_per_sm, int* kcap, int* regs, int64_t* n_deferred) {
    if (int rc = check_handle(h)) return rc;
    if (warps_per_sm) *warps_per_sm = h->geo.warp ? h->geo.warp_per_sm : 0;
    if (kcap) *kcap = h->geo.warp ? h->geo.kcap : 0;
    if (regs) *regs = h->geo.warp ? h->geo.regs : 0;
    if (n_deferred) {
        int32_t v = 0;
        HMPC_CUDA(cudaMemcpyAsync(&v, h->n_defer, 4, cudaMemcpyDeviceToHost, h->stream));
        HMPC_CUDA(cudaStreamSynchronize(h->stream));
        *n_deferred = v;
    }
    return HMPC_OK;
}

int hmpc_launch_count(hmpc_handle* h, int64_t* n) {
    if (!h || !n) return fail(HMPC_ERR_BAD_ARG, "null argument");
    *n = h->launches;
    return HMPC_OK;
}

int hmpc_measure_fp64_peak(hmpc_handle* h, double* tflops) {
    if (int rc = check_handle(h)) return rc;
    if (!tflops) return fail(HMPC_ERR_BAD_ARG, "null argument");
    double* out = nullptr;
    const int blocks = h->sm_count * 8, threads = 256, iters = 4096;
    HMPC_CUDA(cudaMalloc((void**)&out, (size_t)blocks * threads * 8));
    cudaEvent_t e0, e1;
    HMPC_CUDA(cudaEventCreate(&e0));
    HMPC_CUDA(cudaEventCreate(&e1));
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        HMPC_CUDA(cudaEventRecord(e0, h->stream));
        hmpc::dfma_peak_kernel<<<blocks, threads, 0, h->stream>>>(out, iters, 0.999999, 1e-3);
        HMPC_CUDA(cudaEventRecord(e1, h->stream));
        HMPC_CUDA(cudaEventSynchronize(e1));
        float ms = 0;
        HMPC_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        const double flops = 2.0 * 64.0 * (double)iters * (double)blocks * (double)threads;
        if (rep > 0) best = std::max(best, flops / (ms * 1e-3) / 1e12);
        ++h->launches;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(out);
    *tflops = best;
    return HMPC_OK;
}

}  // extern "C"
