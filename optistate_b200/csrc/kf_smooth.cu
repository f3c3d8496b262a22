// Backward kernel of the fixed-interval smoother (kf_smooth.cuh): instantiations and launch.
#include "kf_smooth.cuh"

namespace okf {

// kStats: the E-step.  The caller writes the zero statistics of T = 0 itself.
template <typename Real, bool kStats>
int launch_rts(const SmoothParams<Real> &p, cudaStream_t stream) {
    if (p.N == 0 || p.T == 0) return OPTI_KF_OK;
    const long long blocks = (p.N + RTS_THREADS - 1) / RTS_THREADS;
    if (blocks > 0x7fffffffLL) return OPTI_KF_E_SHAPE;
    // the smoother's 33 KB (FP64) needs no opt-in; the E-step's 55.8 KB (FP64) does, its 27.9 KB (FP32) does not
    const size_t smem = (size_t)(kStats ? EM_SMEM_ROWS : RTS_SMEM_ROWS) * RTS_THREADS * sizeof(Real);
    if (smem > 48 * 1024 &&
        cudaFuncSetAttribute(kf_rts_kernel<Real, kStats>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
        return OPTI_KF_E_CUDA;
    kf_rts_kernel<Real, kStats><<<(unsigned)blocks, RTS_THREADS, smem, stream>>>(p);
    return OPTI_KF_OK;
}

template int launch_rts<double, false>(const SmoothParams<double> &, cudaStream_t);
template int launch_rts<float, false>(const SmoothParams<float> &, cudaStream_t);
template int launch_rts<double, true>(const SmoothParams<double> &, cudaStream_t);
template int launch_rts<float, true>(const SmoothParams<float> &, cudaStream_t);

}  // namespace okf
