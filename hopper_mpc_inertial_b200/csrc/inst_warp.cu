// inst_warp.cu -- instantiations of the warp-per-hopper warm-path kernel (hmpc_warp.cuh), its own translation unit.
#include "hmpc_kernel.cuh"
#include "hmpc_warp.cuh"

namespace hmpc {

// SLOTS = 2: systems of order <= 64 (N <= 10).  Warps per CTA only changes how the SM's shared memory is cut up
// (free-running kernel) / how many hoppers run their trials in lock-step (rounds kernel).
#define HMPC_WARP_DISPATCH(rounds, wpc, CALL)                      \
    if (rounds) {                                                  \
        switch (wpc) {                                             \
            case 4: CALL(mpc_warp_rounds_kernel, 4, 3); break;     \
            case 5: CALL(mpc_warp_rounds_kernel, 5, 2); break;     \
            case 6: CALL(mpc_warp_rounds_kernel, 6, 2); break;     \
            case 7: CALL(mpc_warp_rounds_kernel, 7, 2); break;     \
            case 8: CALL(mpc_warp_rounds_kernel, 8, 1); break;     \
            case 10: CALL(mpc_warp_rounds_kernel, 10, 1); break;   \
            case 11: CALL(mpc_warp_rounds_kernel, 11, 1); break;   \
            case 12: CALL(mpc_warp_rounds_kernel, 12, 1); break;   \
            case 13: CALL(mpc_warp_rounds_kernel, 13, 1); break;   \
            case 14: CALL(mpc_warp_rounds_kernel, 14, 1); break;   \
            default: CALL(mpc_warp_rounds_kernel, 15, 1); break;   \
        }                                                          \
    } else {                                                       \
        switch (wpc) {                                             \
            case 1: CALL(mpc_warp_kernel, 1, 12); break;           \
            case 2: CALL(mpc_warp_kernel, 2, 6); break;            \
            default: CALL(mpc_warp_kernel, 4, 3); break;           \
        }                                                          \
    }

bool warp_wpc_supported(int rounds, int wpc) {
    return rounds ? ((wpc >= 4 && wpc <= 8) || (wpc >= 10 && wpc <= 15)) : (wpc == 1 || wpc == 2 || wpc == 4);
}

cudaError_t warp_set_smem(int rounds, int wpc, int bytes) {
    cudaError_t e = cudaSuccess;
#define CALL(K, W, M) e = cudaFuncSetAttribute(K<2, W, M>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes)
    HMPC_WARP_DISPATCH(rounds, wpc, CALL)
#undef CALL
    return e;
}

cudaError_t warp_regs(int rounds, int wpc, int* regs) {
    cudaFuncAttributes a;
    cudaError_t e = cudaSuccess;
#define CALL(K, W, M) e = cudaFuncGetAttributes(&a, K<2, W, M>)
    HMPC_WARP_DISPATCH(rounds, wpc, CALL)
#undef CALL
    if (e == cudaSuccess) *regs = a.numRegs;
    return e;
}

// prep kernel: 4 warps per CTA, one hopper per warp
constexpr int kPrepWpc = 4;
int prep_wdoubles(int N) { return (int)warp_work_doubles(N, kPrepKcap); }
cudaError_t prep_set_smem(int bytes) {
    return cudaFuncSetAttribute(mpc_prep_kernel<kPrepWpc>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
}
void prep_launch(const WarpLaunch& l, const QpConst& qc, const MpcIo& io, const HopperSet& hs) {
    const int wd = prep_wdoubles(qc.N);
    mpc_prep_kernel<kPrepWpc><<<(l.B + kPrepWpc - 1) / kPrepWpc, 32 * kPrepWpc, (size_t)wd * 8 * kPrepWpc, l.stream>>>(
        qc, l.B, wd, l.prep, l.pstride, l.flags, hs, io);
}

// ADMM mode: free-running warps, one CTA per SM
constexpr int kAdmmWpcA = 10, kAdmmWpcB = 6;
bool warp_admm_wpc_supported(int wpc) { return wpc == kAdmmWpcA || wpc == kAdmmWpcB; }
cudaError_t warp_admm_set_smem(int wpc, int bytes) {
    return wpc == kAdmmWpcA ? cudaFuncSetAttribute(mpc_warp_admm_kernel<kAdmmWpcA>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes)
                            : cudaFuncSetAttribute(mpc_warp_admm_kernel<kAdmmWpcB>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
}
cudaError_t warp_admm_regs(int wpc, int* regs) {
    cudaFuncAttributes a;
    const cudaError_t e = wpc == kAdmmWpcA ? cudaFuncGetAttributes(&a, mpc_warp_admm_kernel<kAdmmWpcA>)
                                           : cudaFuncGetAttributes(&a, mpc_warp_admm_kernel<kAdmmWpcB>);
    if (e == cudaSuccess) *regs = a.numRegs;
    return e;
}

void warp_launch(const WarpLaunch& l, const QpConst& qc, const MpcIo& io) {
    if (l.admm) {
        if (l.wpc == kAdmmWpcA)
            mpc_warp_admm_kernel<kAdmmWpcA><<<l.grid, 32 * kAdmmWpcA, l.smem, l.stream>>>(qc, l.B, l.kcap, l.wdoubles, l.prep, l.pstride, l.flags,
                                                                                         l.work_ctr, l.defer_list, l.defer_cnt, io);
        else
            mpc_warp_admm_kernel<kAdmmWpcB><<<l.grid, 32 * kAdmmWpcB, l.smem, l.stream>>>(qc, l.B, l.kcap, l.wdoubles, l.prep, l.pstride, l.flags,
                                                                                         l.work_ctr, l.defer_list, l.defer_cnt, io);
        return;
    }
#define CALL(K, W, M)                                                                                     \
    K<2, W, M><<<l.grid, 32 * W, l.smem, l.stream>>>(qc, l.B, l.kcap, l.wdoubles, l.prep, l.pstride,      \
                                                     l.flags, l.work_ctr, l.defer_list, l.defer_cnt, l.group, io)
    HMPC_WARP_DISPATCH(l.rounds, l.wpc, CALL)
#undef CALL
}

}  // namespace hmpc
