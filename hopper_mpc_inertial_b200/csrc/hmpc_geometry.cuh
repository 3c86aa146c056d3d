// hmpc_geometry.cuh -- launch geometry: which build of each solver kernel a handle launches, and with how many
// threads, how much shared memory and how large a grid (which ticks take the warp path: hmpc_warp.cuh,
// warp_path_applies).  Host code without CUDA calls, shared by the library (hmpc_create) and the test emulation
// (tests/emul), which checks the choice for every configuration.
#pragma once
#include <algorithm>

#include "hmpc_qp.cuh"
#include "hmpc_mpc.cuh"
#include "hmpc_warp.cuh"

namespace hmpc {

// ------------------------------------------------------------------------------------------------
// The kernel builds the library ships, one list per family.  Every dispatch (inst_warp.cu: warp_launch, warp_set_smem,
// warp_regs, warp_admm_*; hmpc_api.cu: cta_set_smem, launch_cta) switches over exactly these lists and answers any
// other id with cudaErrorInvalidValue, launching nothing.
// ------------------------------------------------------------------------------------------------
// lock-step warp kernel mpc_warp_rounds_kernel<2, WPC, MIN_CTAS>.  The order is the order in which inst_warp.cu
// instantiates them, which the machine code of the kernels depends on.
#define HMPC_WARP_BUILDS(X) X(4, 3) X(5, 2) X(6, 2) X(7, 2) X(8, 1) X(10, 1) X(11, 1) X(12, 1) X(13, 1) X(14, 1) X(15, 1)
// ADMM warp kernel mpc_warp_admm_kernel<WPC>, one CTA per SM, in order of preference
#define HMPC_WARP_ADMM_BUILDS(X) X(10) X(6)
// CTA kernel mpc_kernel, csrc/inst_NAME.cu (hmpc_kernel.cuh), with its threads per CTA
#define HMPC_CTA_BUILDS(X) X(n10_f64, 128) X(n10_f64_admm, 128) X(n10_f32, 128) X(wide_gmem4, 128) X(wide_gmem2, 256)

#define HMPC_FIRST_OF2(a, b) a,
#define HMPC_FIRST_OF1(a) a,
#define HMPC_SECOND_OF2(a, b) b,
#define HMPC_CTA_ID(name, threads) CTA_##name,
constexpr int kWarpWpc[] = {HMPC_WARP_BUILDS(HMPC_FIRST_OF2)};
constexpr int kAdmmWpc[] = {HMPC_WARP_ADMM_BUILDS(HMPC_FIRST_OF1)};
constexpr int kCtaThreads[] = {HMPC_CTA_BUILDS(HMPC_SECOND_OF2)};
enum CtaBuild { HMPC_CTA_BUILDS(HMPC_CTA_ID) kNumCtaBuilds };
#undef HMPC_FIRST_OF2
#undef HMPC_FIRST_OF1
#undef HMPC_SECOND_OF2
#undef HMPC_CTA_ID
constexpr int kNumWarpBuilds = (int)(sizeof(kWarpWpc) / sizeof(int));
constexpr int kNumAdmmBuilds = (int)(sizeof(kAdmmWpc) / sizeof(int));

// ------------------------------------------------------------------------------------------------
// Launch geometry
// ------------------------------------------------------------------------------------------------
struct DeviceLimits {
    int sm_count = 0;
    size_t smem_block = 0;                // opt-in shared memory per block
    size_t smem_sm = 0;                   // shared memory per SM
    size_t l2 = 0;                        // L2 bytes
    int warp_regs[kNumWarpBuilds] = {};   // registers per thread of each build of HMPC_WARP_BUILDS (read: exact solver)
    int admm_regs[kNumAdmmBuilds] = {};   // ... of HMPC_WARP_ADMM_BUILDS (read: ADMM solver)
};

struct Geometry {
    const char* unsupported = nullptr;    // set: the CTA kernel does not fit the device (the reason)
    // CTA kernel (cold ticks, the warp kernel's deferrals, hot_path = HMPC_HOT_CTA)
    CtaBuild cta = CTA_n10_f64;
    int threads = 0, grid = 0;
    size_t smem = 0;                      // dynamic shared memory per CTA
    size_t ws_bytes = 0;                  // L2 workspace of all CTAs' matrices (0: the matrices are in shared memory)
    // warp-per-hopper kernel (warp = false: not used by this configuration)
    bool warp = false, admm = false;      // admm: mpc_warp_admm_kernel, else mpc_warp_rounds_kernel
    int wpc = 0, kcap = 0, wdoubles = 0;  // warps per CTA, KKT order cap, doubles of one warp's shared-memory slice
    int warp_grid = 0, warp_per_sm = 0, regs = 0;
    int group = 0;                        // lock-step kernel's gw argument: warps per lock-step group + 256 * barriers
    size_t warp_smem = 0;                 // dynamic shared memory per CTA
};

inline Geometry launch_geometry(const hmpc_config& cfg, int kcap, const DeviceLimits& d) {
    Geometry g;
    const int N = cfg.N;
    const size_t B = (size_t)cfg.batch;
    const size_t mat_bytes = mat_doubles(N, cfg.precision == HMPC_FP32 ? 4 : 8) * 8;
    const size_t ws_cta = mat_bytes + ws_mv_doubles(N) * 8;
    int per_sm;
    if (6 * N <= 64) {
        // matrices in shared memory, as many 128-thread CTAs per SM as it holds
        g.smem = ((work_vec_doubles(N) + 1) & ~(size_t)1) * 8 + mat_bytes;
        if (g.smem + 1024 > d.smem_block) { g.unsupported = "shared memory too small for the N <= 10 solver kernel"; return g; }
        g.cta = cfg.precision == HMPC_FP32 ? CTA_n10_f32 : cfg.solver == HMPC_SOLVER_ADMM ? CTA_n10_f64_admm : CTA_n10_f64;
        per_sm = std::max<int>(1, (int)(d.smem_sm / (g.smem + 1024)));
    } else {
        // N > 10: the matrices go to a per-CTA L2 workspace even when they would fit in shared memory, so that several
        // hoppers share an SM (each hopper's pivot chain leaves most of its warps waiting; DESIGN.md section 5.2):
        // four 128-thread CTAs per SM while 4 x SMs workspaces fit the L2 (N <= 24 on the 126 MB L2 of a B200), else two
        // 256-thread CTAs.  Both builds are compiled for 128 registers.
        g.smem = ((work_vec_doubles(N, mv_in_workspace(N)) + 1) & ~(size_t)1) * 8;
        if (g.smem > d.smem_block) { g.unsupported = "horizon too large for shared memory"; return g; }
        const int fit = (int)(d.smem_sm / (g.smem + 1024));
        if (fit < 2) { g.unsupported = "shared memory too small for two CTAs per SM of the N > 10 solver kernel"; return g; }
        const int want = (size_t)d.sm_count * 4 * ws_cta <= d.l2 ? 4 : 2;
        per_sm = std::min(want, fit) >= 4 ? 4 : 2;
        g.cta = per_sm == 4 ? CTA_wide_gmem4 : CTA_wide_gmem2;
    }
    g.threads = kCtaThreads[g.cta];
    g.grid = (int)std::min<size_t>(B, (size_t)d.sm_count * per_sm);
    if (6 * N > 64) g.ws_bytes = (size_t)g.grid * ws_cta;

    if (!warp_path_applies(cfg, 0)) return g;
    g.kcap = kcap;
    if (cfg.solver == HMPC_SOLVER_ADMM) {
        // free-running warps, one CTA per SM: the first build whose slices (z, y, rho behind the exact path's slice) fit
        g.wdoubles = (int)(warp_work_doubles(N, kcap) + warp_admm_doubles(N));
        const size_t wbytes = (size_t)g.wdoubles * 8;
        for (int i = 0; i < kNumAdmmBuilds && !g.warp; ++i) {
            if (wbytes * kAdmmWpc[i] + 1024 > d.smem_block) continue;
            g.warp = g.admm = true;
            g.wpc = g.warp_per_sm = kAdmmWpc[i];
            g.regs = d.admm_regs[i];
        }
        if (!g.warp) return g;
        g.warp_grid = (int)std::min<size_t>((B + g.wpc - 1) / g.wpc, (size_t)d.sm_count);
    } else {
        // lock-step rounds, all warps of the SM in one CTA (one instruction stream per SM: measured 6 % (3f) to 20 %
        // (2f) faster than free-running warps): the build with the most warps per SM, as shared memory and registers
        // allow; on a tie the one with more warps per CTA
        g.wdoubles = (int)warp_work_doubles(N, kcap);
        const size_t wbytes = (size_t)g.wdoubles * 8;
        for (int i = 0; i < kNumWarpBuilds; ++i) {
            const int wpc = kWarpWpc[i], regs = d.warp_regs[i];
            if (wbytes * wpc + 512 > d.smem_block) continue;
            const int by_smem = (int)(d.smem_sm / (wbytes * wpc + 1024));
            const int by_regs = (int)(65536 / ((size_t)((regs + 7) & ~7) * 32 * wpc));
            const int warps = std::min(std::min(by_smem, by_regs), 32) * wpc;
            if (warps > 0 && warps >= g.warp_per_sm) { g.warp_per_sm = warps; g.wpc = wpc; g.regs = regs; }
        }
        if (g.warp_per_sm == 0) return g;
        g.warp = true;
        g.warp_grid = (int)std::min<size_t>((B + g.wpc - 1) / g.wpc, (size_t)d.sm_count * (g.warp_per_sm / g.wpc));
        // lock-step group = all warps of the CTA, one re-alignment barrier after the factorisation (measured, 131072
        // hoppers: groups of 12 / 6 / 4 / 3 / 2 warps 8.38 / 7.83 / 7.48 / 7.30 / 7.12 M steps/s; with the barrier 8.48 M)
        g.group = g.wpc + 256 * 1;
    }
    g.warp_smem = (size_t)g.wdoubles * 8 * g.wpc;
    return g;
}

}  // namespace hmpc
