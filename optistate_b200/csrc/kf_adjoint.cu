// Adjoint kernel of the sequential filter (kf_adjoint.cuh): instantiations and launch.
#include "kf_adjoint.cuh"

namespace okf {

// The caller writes the zero gradient of T = 0 itself.
template <typename Real>
int launch_adjoint(const AdjointParams<Real> &p, cudaStream_t stream) {
    if (p.N == 0 || p.T == 0) return OPTI_KF_OK;
    const long long blocks = (p.N + ADJ_THREADS - 1) / ADJ_THREADS;
    if (blocks > 0x7fffffffLL) return OPTI_KF_E_SHAPE;
    // 59 KB per block in FP64 needs the dynamic shared-memory opt-in, 29.5 KB in FP32 does not
    const size_t smem = (size_t)ADJ_SMEM_ROWS * ADJ_THREADS * sizeof(Real);
    if (smem > 48 * 1024 &&
        cudaFuncSetAttribute(kf_adjoint_kernel<Real>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
        return OPTI_KF_E_CUDA;
    kf_adjoint_kernel<Real><<<(unsigned)blocks, ADJ_THREADS, smem, stream>>>(p);
    return OPTI_KF_OK;
}

template int launch_adjoint<double>(const AdjointParams<double> &, cudaStream_t);
template int launch_adjoint<float>(const AdjointParams<float> &, cudaStream_t);

}  // namespace okf
