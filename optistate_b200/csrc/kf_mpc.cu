// Batched convex force MPC (kf_mpc.cuh): launch.
#include "kf_mpc.cuh"
#include "kf_mpc_gi.cuh"

#include "kf_launch.cuh"

namespace okf {

int launch_mpc(const MpcParams &p, cudaStream_t stream) {
    // dual active set first (kf_mpc_gi.cuh): one warp per problem for a trot or less, two warps when the batch has three or four
    // legs out of swing somewhere; then the shared-memory interior point (kf_mpc.cuh) for what it flags - or for everything when
    // the caller asks for the interior point
    MpcParams q = p;
    if (p.solver == 0) {
        if (p.max_legs <= MPCG_MAX_LEGS) {
            const size_t smem = mpcg_smem_bytes();
            if (cudaFuncSetAttribute(kf_mpc_gi_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return OPTI_KF_E_CUDA;
            kf_mpc_gi_kernel<<<(unsigned)((p.N + MPCG_WARPS - 1) / MPCG_WARPS), 32 * MPCG_WARPS, smem, stream>>>(p);
        } else {
            const size_t smem2 = mpcg2_smem_bytes(p.max_legs);
            if (cudaFuncSetAttribute(kf_mpc_gi2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2) != cudaSuccess) return OPTI_KF_E_CUDA;
            kf_mpc_gi2_kernel<<<(unsigned)p.N, 64, smem2, stream>>>(p);
        }
        q.only_flagged = 1;
    }
    const size_t smem = mpc_smem_bytes(p.max_legs);
    if (cudaFuncSetAttribute(kf_mpc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return OPTI_KF_E_CUDA;
    const unsigned blocks = (unsigned)((p.N + MPC_WARPS - 1) / MPC_WARPS);
    kf_mpc_kernel<<<blocks, 32 * MPC_WARPS, smem, stream>>>(q);
    return OPTI_KF_OK;
}

}  // namespace okf
