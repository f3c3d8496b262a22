// Backward kernel of the fixed-interval smoother (kf_smooth.cuh): instantiations and launch.
#include "kf_smooth.cuh"

namespace okf {

template <typename Real>
int launch_rts(const SmoothParams<Real> &p, cudaStream_t stream) {
    if (p.N == 0 || p.T == 0) return OPTI_KF_OK;
    const long long blocks = (p.N + RTS_THREADS - 1) / RTS_THREADS;
    if (blocks > 0x7fffffffLL) return OPTI_KF_E_SHAPE;
    const size_t smem = (size_t)RTS_SMEM_ROWS * RTS_THREADS * sizeof(Real);  // 33 KB (FP64): no opt-in needed
    kf_rts_kernel<Real, false><<<(unsigned)blocks, RTS_THREADS, smem, stream>>>(p);
    return OPTI_KF_OK;
}

// The caller writes the zero statistics of T = 0 itself.
template <typename Real>
int launch_em_stats(const SmoothParams<Real> &p, cudaStream_t stream) {
    if (p.N == 0 || p.T == 0) return OPTI_KF_OK;
    const long long blocks = (p.N + RTS_THREADS - 1) / RTS_THREADS;
    if (blocks > 0x7fffffffLL) return OPTI_KF_E_SHAPE;
    const size_t smem = (size_t)EM_SMEM_ROWS * RTS_THREADS * sizeof(Real);  // 55.8 KB (FP64), 27.9 KB (FP32)
    if (smem > 48 * 1024 &&
        cudaFuncSetAttribute(kf_rts_kernel<Real, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
        return OPTI_KF_E_CUDA;
    kf_rts_kernel<Real, true><<<(unsigned)blocks, RTS_THREADS, smem, stream>>>(p);
    return OPTI_KF_OK;
}

template int launch_rts<double>(const SmoothParams<double> &, cudaStream_t);
template int launch_rts<float>(const SmoothParams<float> &, cudaStream_t);
template int launch_em_stats<double>(const SmoothParams<double> &, cudaStream_t);
template int launch_em_stats<float>(const SmoothParams<float> &, cudaStream_t);

}  // namespace okf
