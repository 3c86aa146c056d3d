// inst_wide_gmem2.cu -- one instantiation of the solver kernel (see hmpc_kernel.cuh), its own translation unit:
// the L2-workspace kernel of the long horizons compiled for TWO resident CTAs per SM (<= 128 registers per thread).
#include "hmpc_kernel.cuh"

namespace hmpc {
cudaError_t mpc_set_smem_wide_gmem2(int bytes) { return mpc_set_smem<256, 2, false, double, true>(bytes); }
void mpc_launch_wide_gmem2(const MpcLaunch& l, const QpConst& qc, const MpcIo& io) { mpc_launch<256, 2, false, double, true>(l, qc, io); }
}  // namespace hmpc

#ifdef HMPC_PHASE_TIMING
// debug builds only (tools/phase_timing.py): read and reset this translation unit's phase counters
extern "C" int hmpc_debug_phases_wide_gmem2(unsigned long long* out) {
    cudaError_t e = cudaMemcpyFromSymbol(out, hmpc::g_phase, sizeof(unsigned long long) * 16);
    if (e != cudaSuccess) return -1;
    unsigned long long z[16] = {0};
    return cudaMemcpyToSymbol(hmpc::g_phase, z, sizeof(z)) == cudaSuccess ? 0 : -1;
}
#endif
