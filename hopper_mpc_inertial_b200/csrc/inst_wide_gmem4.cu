// inst_wide_gmem4.cu -- one instantiation of the solver kernel (see hmpc_kernel.cuh), its own translation unit:
// the L2-workspace kernel of the long horizons with 128-thread CTAs, FOUR resident per SM (<= 128 registers per
// thread): more independent hoppers per SM, fewer warps waiting on each hopper's serial pivot chain.
#include "hmpc_kernel.cuh"

namespace hmpc {
cudaError_t mpc_set_smem_wide_gmem4(int bytes) { return mpc_set_smem<128, 4, false, double, true>(bytes); }
void mpc_launch_wide_gmem4(const MpcLaunch& l, const QpConst& qc, const MpcIo& io) { mpc_launch<128, 4, false, double, true>(l, qc, io); }
}  // namespace hmpc

#ifdef HMPC_PHASE_TIMING
// debug builds only (tools/phase_timing.py): read and reset this translation unit's phase counters
extern "C" int hmpc_debug_phases_wide_gmem4(unsigned long long* out) {
    cudaError_t e = cudaMemcpyFromSymbol(out, hmpc::g_phase, sizeof(unsigned long long) * 16);
    if (e != cudaSuccess) return -1;
    unsigned long long z[16] = {0};
    return cudaMemcpyToSymbol(hmpc::g_phase, z, sizeof(z)) == cudaSuccess ? 0 : -1;
}
#endif
