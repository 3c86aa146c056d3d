// inst_warp.cu -- instantiations of the warp-per-hopper warm-path kernel (hmpc_warp.cuh), its own translation unit.
#include "hmpc_kernel.cuh"
#include "hmpc_warp.cuh"
#include "hmpc_geometry.cuh"

namespace hmpc {

// SLOTS = 2: systems of order <= 64 (N <= 10).  Warps per CTA only changes how many hoppers run their trials in
// lock-step.  The builds are the ones of HMPC_WARP_BUILDS / HMPC_WARP_ADMM_BUILDS (hmpc_geometry.cuh); any other wpc
// is refused.
cudaError_t warp_set_smem(int wpc, int bytes) {
    switch (wpc) {
#define CALL(W, M) case W: return cudaFuncSetAttribute(mpc_warp_rounds_kernel<2, W, M>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
        HMPC_WARP_BUILDS(CALL)
#undef CALL
        default: return cudaErrorInvalidValue;
    }
}

cudaError_t warp_regs(int wpc, int* regs) {
    cudaFuncAttributes a;
    cudaError_t e;
    switch (wpc) {
#define CALL(W, M) case W: e = cudaFuncGetAttributes(&a, mpc_warp_rounds_kernel<2, W, M>); break;
        HMPC_WARP_BUILDS(CALL)
#undef CALL
        default: return cudaErrorInvalidValue;
    }
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
cudaError_t warp_admm_set_smem(int wpc, int bytes) {
    switch (wpc) {
#define CALL(W) case W: return cudaFuncSetAttribute(mpc_warp_admm_kernel<W>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
        HMPC_WARP_ADMM_BUILDS(CALL)
#undef CALL
        default: return cudaErrorInvalidValue;
    }
}
cudaError_t warp_admm_regs(int wpc, int* regs) {
    cudaFuncAttributes a;
    cudaError_t e;
    switch (wpc) {
#define CALL(W) case W: e = cudaFuncGetAttributes(&a, mpc_warp_admm_kernel<W>); break;
        HMPC_WARP_ADMM_BUILDS(CALL)
#undef CALL
        default: return cudaErrorInvalidValue;
    }
    if (e == cudaSuccess) *regs = a.numRegs;
    return e;
}

cudaError_t warp_launch(const WarpLaunch& l, const QpConst& qc, const MpcIo& io) {
    if (l.admm) {
        switch (l.wpc) {
#define CALL(W)                                                                                                          \
    case W:                                                                                                              \
        mpc_warp_admm_kernel<W><<<l.grid, 32 * W, l.smem, l.stream>>>(qc, l.B, l.kcap, l.wdoubles, l.prep, l.pstride,   \
                                                                      l.flags, l.work_ctr, l.defer_list, l.defer_cnt, io); \
        return cudaSuccess;
            HMPC_WARP_ADMM_BUILDS(CALL)
#undef CALL
            default: return cudaErrorInvalidValue;
        }
    }
    switch (l.wpc) {
#define CALL(W, M)                                                                                                       \
    case W:                                                                                                              \
        mpc_warp_rounds_kernel<2, W, M><<<l.grid, 32 * W, l.smem, l.stream>>>(qc, l.B, l.kcap, l.wdoubles, l.prep,       \
                                                                              l.pstride, l.flags, l.work_ctr,          \
                                                                              l.defer_list, l.defer_cnt, l.group, io);   \
        return cudaSuccess;
        HMPC_WARP_BUILDS(CALL)
#undef CALL
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace hmpc
