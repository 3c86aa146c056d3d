// hmpc_kernel.cuh -- the persistent solver kernel (K1+K2) as a template, plus the per-instantiation host
// entry points.  Every instantiation lives in its own translation unit (csrc/inst_*.cu) so that the library
// builds in parallel: one instantiation of this kernel is ~30 k SASS instructions.
#pragma once
#include <cuda_runtime.h>

#include "hmpc_sim.cuh"
#include "hmpc_mpc.cuh"

namespace hmpc {

// ------------------------------------------------------------------------------------------------
// K1+K2: mpcontrol for a batch (mpc_cvx_euler_3f.py:41-69).  Persistent CTAs, one hopper at a time.
// ------------------------------------------------------------------------------------------------
// F: precision of the factorisation and of the substitutions (double, or float = mixed precision: QP data,
// iterates and residuals stay FP64 and the refinement loops recover FP64-level accuracy)
template <int THREADS, int MIN_CTAS, bool SMEM_MATS, typename F, bool WITH_ADMM>
__global__ void __launch_bounds__(THREADS, MIN_CTAS)
mpc_kernel(QpConst c, int B, int sm_count, double* __restrict__ ws, int* __restrict__ work_ctr,
           const int* __restrict__ list, const int* __restrict__ list_cnt, MpcIo io) {
    extern __shared__ double smem[];
    __shared__ int s_next;
    Work w;
    setup_work<SMEM_MATS>(w, c, smem, ws, (int)sizeof(F));
    const int N = c.N, n = 6 * N;
    AOp A{N, n, c.dyn == 3 ? 1 : 0, c.mu, w.stance, w.hinv};
    LinSys<F> sys{n, 0, 0, reinterpret_cast<F*>(w.Lm), reinterpret_cast<F*>(w.dinv), w.H, w.idx, w.grow};
    // CTAs are dealt to the SMs round-robin, so the CTAs sharing an SM differ in blockIdx.x / #SMs
    sys.solver_warp = blockIdx.x / sm_count;
    // horizons beyond N = 10 (256-thread CTAs): tensor-core tiles, all warps of the CTA (LinSys::factor_tiled)
    sys.tiled = (sizeof(F) == 8 && tiled_factor_applies(c.N)) ? 1 : 0;
    // dynamic distribution of hoppers over the persistent CTAs (solve times differ: warm active-set path
    // vs interior-point path); results do not depend on the order
    // list mode: only the hoppers the warp kernel deferred (hmpc_warp.cuh), in any order
    const int count = list ? *list_cnt : B;
    // a short deferral list is latency-bound (at most one hopper per CTA): its interior points take the tiled factor
    sys.ipm_tiled = (list && count <= (int)gridDim.x) ? 1 : 0;
    for (;;) {
        __syncthreads();
        if (threadIdx.x == 0) s_next = atomicAdd(work_ctr, 1);
        __syncthreads();
        const int i = s_next;
        if (i >= count) break;
        const int e = list ? list[i] : work_item(c, i, count);     // bit 30: the warp kernel's active-set refinement already gave up
        const int b = e & ~(1 << 30);
        if (c.body) A.mu = c.body[(size_t)B + b];                  // the hopper's friction coefficient (model_body)
        mpc_hopper<WITH_ADMM>(c, w, sys, A, b, B, io, (e >> 30) & 1);
    }
}

// host entry points of one instantiation
struct MpcLaunch {
    int grid, threads;
    size_t smem;
    cudaStream_t stream;
    int B, sm_count;
    double* ws;
    int* work_ctr;
    const int* list;        // null: hoppers 0..B-1; else the deferral list of the warp kernel
    const int* list_cnt;
};

template <int THREADS, int MIN_CTAS, bool SMEM_MATS, typename F, bool WITH_ADMM>
inline cudaError_t mpc_set_smem(int bytes) {
    return cudaFuncSetAttribute(mpc_kernel<THREADS, MIN_CTAS, SMEM_MATS, F, WITH_ADMM>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
}
template <int THREADS, int MIN_CTAS, bool SMEM_MATS, typename F, bool WITH_ADMM>
inline void mpc_launch(const MpcLaunch& l, const QpConst& qc, const MpcIo& io) {
    mpc_kernel<THREADS, MIN_CTAS, SMEM_MATS, F, WITH_ADMM><<<l.grid, THREADS, l.smem, l.stream>>>(qc, l.B, l.sm_count, l.ws, l.work_ctr, l.list, l.list_cnt, io);
}

// the instantiations the library ships (defined in csrc/inst_*.cu)
cudaError_t mpc_set_smem_n10_f64(int bytes);      // 128 threads, 4 CTAs/SM, shared-memory matrices, FP64 factor, exact solver only
void mpc_launch_n10_f64(const MpcLaunch&, const QpConst&, const MpcIo&);
cudaError_t mpc_set_smem_n10_f64_admm(int bytes); // the same with the ADMM branch compiled in
void mpc_launch_n10_f64_admm(const MpcLaunch&, const QpConst&, const MpcIo&);
cudaError_t mpc_set_smem_n10_f32(int bytes);      // 128 threads, 5 CTAs/SM, shared-memory matrices, FP32 factor
void mpc_launch_n10_f32(const MpcLaunch&, const QpConst&, const MpcIo&);
cudaError_t mpc_set_smem_wide_gmem2(int bytes);   // 256 threads, 2 CTAs/SM (<= 128 registers), matrices in the L2-resident workspace
void mpc_launch_wide_gmem2(const MpcLaunch&, const QpConst&, const MpcIo&);
cudaError_t mpc_set_smem_wide_gmem4(int bytes);   // 128 threads, 4 CTAs/SM, matrices in the L2 workspace
void mpc_launch_wide_gmem4(const MpcLaunch&, const QpConst&, const MpcIo&);


// the warp-per-hopper warm-path kernel (hmpc_warp.cuh, instantiated in inst_warp.cu); the functions taking a wpc
// return cudaErrorInvalidValue for a wpc that has no build
struct WarpLaunch {
    int grid, wpc;          // CTAs, warps per CTA
    int group;              // lock-step kernel: warps per lock-step group (named barrier) + 256 * re-alignment barriers
    size_t smem;            // dynamic shared memory per CTA
    cudaStream_t stream;
    int B, kcap, wdoubles;
    double* prep;           // per-hopper QP records (hmpc_warp.cuh: prep_stride), written by the prep kernel
    size_t pstride;
    int32_t* flags;         // per-hopper PREP_* flag
    int *work_ctr, *defer_list, *defer_cnt;
    int admm = 0;           // 1: the ADMM warp kernel (free-running warps, wdoubles includes warp_admm_doubles)
};
int prep_wdoubles(int N);
cudaError_t prep_set_smem(int bytes);
void prep_launch(const WarpLaunch&, const QpConst&, const MpcIo&, const HopperSet& = HopperSet{});
cudaError_t warp_set_smem(int wpc, int bytes);
cudaError_t warp_regs(int wpc, int* regs);
cudaError_t warp_launch(const WarpLaunch&, const QpConst&, const MpcIo&);
cudaError_t warp_admm_set_smem(int wpc, int bytes);
cudaError_t warp_admm_regs(int wpc, int* regs);

}  // namespace hmpc
