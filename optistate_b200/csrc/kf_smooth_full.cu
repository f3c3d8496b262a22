// Backward kernel of the full-covariance smoother (kf_smooth_full.cuh): instantiations and launch.
#include "kf_smooth_full.cuh"

namespace okf {

// kStats: the E-step.  The caller writes the zero statistics of T = 0 itself.
template <typename Real, bool kStats>
int launch_rts_full(const SmoothFullParams<Real> &p, cudaStream_t stream) {
    if (p.N == 0 || p.T == 0) return OPTI_KF_OK;
    const long long blocks = (p.N + RTSF_TRAJ - 1) / RTSF_TRAJ;
    if (blocks > 0x7fffffffLL) return OPTI_KF_E_SHAPE;
    // 111 KB (FP64): two blocks per SM, 55.5 KB (FP32); the E-step adds no rows
    const size_t smem = (size_t)RTSF_SMEM_ROWS * RTSF_TRAJ * sizeof(Real);
    const auto kern = p.cov_model == OPTI_KF_COV_MPC ? kf_rts_full_kernel<Real, true, kStats> : kf_rts_full_kernel<Real, false, kStats>;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return OPTI_KF_E_CUDA;
    kern<<<(unsigned)blocks, RTSF_THREADS, smem, stream>>>(p);
    return OPTI_KF_OK;
}

template int launch_rts_full<double, false>(const SmoothFullParams<double> &, cudaStream_t);
template int launch_rts_full<float, false>(const SmoothFullParams<float> &, cudaStream_t);
template int launch_rts_full<double, true>(const SmoothFullParams<double> &, cudaStream_t);
template int launch_rts_full<float, true>(const SmoothFullParams<float> &, cudaStream_t);

}  // namespace okf
