// Host side of the streamed SEQUENTIAL kernel: tensor maps of the per-step input arrays and the launch.  Included by the
// kf_seq_tma_*.cu translation units, each of which instantiates launch_seq_tma for one (Real, kSummary) pair.
#pragma once

#include <cuda.h>

#include <cstring>

#include "kf_launch.cuh"
#include "kf_seq_tma.cuh"

namespace okf {

// cuTensorMapEncodeTiled, fetched from the driver through the runtime (no link-time dependency on libcuda)
using EncodeTiledFn = CUresult (*)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                   const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline EncodeTiledFn encode_tiled() {
    static const EncodeTiledFn fn = [] {
        void *sym = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
            sym = nullptr;
        return (EncodeTiledFn)sym;
    }();
    return fn;
}

// [T*C][S] matrix of one per-step input array, fetched in [rows][box_w] boxes (one warp's tile of one step; rows = the
// leading channels of the C that are wanted)
template <typename Real>
bool make_map(CUtensorMap *m, const Real *base, long long T, int C, long long S, int box_w, int rows) {
    EncodeTiledFn enc = encode_tiled();
    if (!enc || !base) return false;
    const cuuint64_t gdim[2] = {(cuuint64_t)S, (cuuint64_t)(T * C)};
    const cuuint64_t gstride[1] = {(cuuint64_t)S * sizeof(Real)};
    const cuuint32_t box[2] = {(cuuint32_t)box_w, (cuuint32_t)rows};
    const cuuint32_t estride[2] = {1u, 1u};
    return enc(m, sizeof(Real) == 8 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT64 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void *)base, gdim, gstride,
               box, estride, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <typename Real, bool kSummary, int kOut, bool kMpc, bool kBlock, int kW = 0>
int launch_seq_tma_k(const Params<typename Lanes<Real>::scalar> &p, cudaStream_t stream) {
    constexpr int L = Lanes<Real>::n;
    const int n_lab = kSummary ? (p.truth ? 1 : 0) + (p.nominal ? 1 : 0) : 0;
    TmaMaps maps;
    std::memset(&maps, 0, sizeof maps);
    const int bw = 32 * L;
    bool ok = make_map(&maps.mom, p.mom, p.T, NM, p.S, bw, NM) && make_map(&maps.z, p.z_in, p.T, 10, p.S, bw, 10);
    if (ok && kOut == 2) ok = make_map(&maps.p, p.p, p.T, 12, p.S, bw, 12);
    if (ok && kMpc) ok = make_map(&maps.body_ref, p.body_ref, p.T, 12, p.S, bw, 3);
    if (ok && n_lab >= 1) ok = make_map(&maps.lab0, p.truth ? p.truth : p.nominal, p.T, 12, p.S, bw, 12);
    if (ok && n_lab >= 2) ok = make_map(&maps.lab1, p.nominal, p.T, 12, p.S, bw, 12);
    if (!ok) return 1;
    constexpr int kWarps = kW ? kW : tma_warps<kBlock>(), kThreads = 32 * kWarps;
    const size_t smem = TmaSmem<Real, kThreads, tma_noise_rows<kOut>(), tma_stages<kW>()>::total(n_lab, tma_g0_rows<kOut, kMpc>(), kW == 1 ? false : tma_acc_in_smem<Real, kSummary, kBlock>());
    auto kern = kf_seq_tma_kernel<Real, kSummary, kOut, kMpc, kBlock, kW>;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return OPTI_KF_E_CUDA;
    // one block per (stream tile, group of kWarps members): see the index mapping at the top of the kernel
    const long long tiles = p.S / (32 * L), n_pass = (p.N + p.S - 1) / p.S;
    const long long blocks = tiles * ((n_pass + kWarps - 1) / kWarps);
    if (blocks > 0x7fffffffLL) return OPTI_KF_E_SHAPE;
    kern<<<(unsigned)blocks, kThreads, smem, stream>>>(p, maps);
    return OPTI_KF_OK;
}

// per-step outputs, the predict_mpc covariance model and the decoupled-group form are compile-time variants of the kernel
// (see kf_seq_tma.cuh); kBlock is chosen by the caller from Params.block and never combines with the predict_mpc model
template <typename Real, bool kSummary, bool kBlock>
int launch_seq_tma(const Params<typename Lanes<Real>::scalar> &p, cudaStream_t stream) {
    const bool rare = p.x_model_steps || p.p_world_steps || p.z_steps || p.P_ckpt || p.P_steps;
    const bool estimates = p.x_steps || p.p_trace_steps || p.k_gain_steps || p.nis_steps;
    const int out = rare ? 2 : (estimates ? 1 : 0);
    const bool mpc = p.cov_model == OPTI_KF_COV_MPC;
    if constexpr (kBlock) {
        if (mpc) return OPTI_KF_E_UNSUPPORTED;
        switch (out) {
            case 0: return launch_seq_tma_k<Real, kSummary, 0, false, true>(p, stream);
            case 1: return launch_seq_tma_k<Real, kSummary, 1, false, true>(p, stream);
            default: return launch_seq_tma_k<Real, kSummary, 2, false, true>(p, stream);
        }
    } else {
        switch (out * 2 + (mpc ? 1 : 0)) {
            case 0: return launch_seq_tma_k<Real, kSummary, 0, false, false>(p, stream);
            case 1: return launch_seq_tma_k<Real, kSummary, 0, true, false>(p, stream);
            case 2: return launch_seq_tma_k<Real, kSummary, 1, false, false>(p, stream);
            case 3: return launch_seq_tma_k<Real, kSummary, 1, true, false>(p, stream);
            case 4: return launch_seq_tma_k<Real, kSummary, 2, false, false>(p, stream);
            default: return launch_seq_tma_k<Real, kSummary, 2, true, false>(p, stream);
        }
    }
}

// Latency variant (one warp per block, see the kernel): decoupled-group form, predict() covariance model; instantiated in
// kf_seq_tma_lone_*.cu for double and float.
template <typename Real, bool kSummary>
int launch_seq_tma_lone(const Params<typename Lanes<Real>::scalar> &p, cudaStream_t stream) {
    const bool rare = p.x_model_steps || p.p_world_steps || p.z_steps || p.P_ckpt || p.P_steps;
    const bool estimates = p.x_steps || p.p_trace_steps || p.k_gain_steps || p.nis_steps;
    if (rare) return launch_seq_tma_k<Real, kSummary, 2, false, true, 1>(p, stream);
    if (estimates) return launch_seq_tma_k<Real, kSummary, 1, false, true, 1>(p, stream);
    return launch_seq_tma_k<Real, kSummary, 0, false, true, 1>(p, stream);
}

}  // namespace okf
