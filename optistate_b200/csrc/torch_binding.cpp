// Thin PyTorch C++ extension over the C ABI of liboptistate_kf.so: unwraps tensors into raw device pointers,
// checks device / dtype / contiguity / element counts (the C ABI cannot), takes torch's current CUDA stream and
// calls the extern "C" entry points.  No arithmetic happens here and there is no CPU path: CPU tensors are an error.
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/extension.h>

#include <map>
#include <optional>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/optistate_kf.h"

namespace {

using TensorMap = std::map<std::string, at::Tensor>;

struct Checker {
    at::ScalarType st;
    c10::Device dev;
    const void *get(const TensorMap &m, const char *name, int64_t numel, bool required) const {
        auto it = m.find(name);
        if (it == m.end()) {
            TORCH_CHECK(!required, "optistate_b200: missing tensor '", name, "'");
            return nullptr;
        }
        const at::Tensor &t = it->second;
        TORCH_CHECK(t.is_cuda(), "optistate_b200: '", name, "' must be a CUDA tensor (there is no CPU path)");
        TORCH_CHECK(t.device() == dev, "optistate_b200: '", name, "' is on ", t.device(), ", expected ", dev);
        TORCH_CHECK(t.scalar_type() == st, "optistate_b200: '", name, "' has dtype ", t.scalar_type(), ", expected ", st);
        TORCH_CHECK(t.is_contiguous(), "optistate_b200: '", name, "' must be contiguous");
        TORCH_CHECK(t.numel() == numel, "optistate_b200: '", name, "' has ", t.numel(), " elements, expected ", numel);
        return t.data_ptr();
    }
};

int64_t geti(const std::map<std::string, int64_t> &c, const char *k, int64_t dflt) {
    auto it = c.find(k);
    return it == c.end() ? dflt : it->second;
}

int64_t mat_numel(int kind, int64_t n, int64_t N) {
    switch (kind) {
        case OPTI_KF_MAT_NONE: return 0;
        case OPTI_KF_MAT_DIAG: return n;
        case OPTI_KF_MAT_DIAG_PER: return n * N;
        case OPTI_KF_MAT_DENSE: return n * n;
        case OPTI_KF_MAT_DENSE_PER: return n * n * N;
        default: TORCH_CHECK(false, "optistate_b200: bad matrix kind ", kind);
    }
}

// The filter descriptor of kf_batch and kf_smooth.  cfg: integer settings; consts: dt, mass, inertia0..2, gravity; tensors: named
// device arrays (see optistate_kf.h).  Returns the device of the tensors (the caller makes it current).
c10::Device filter_desc(const std::map<std::string, int64_t> &cfg, const std::map<std::string, double> &consts, const TensorMap &tensors,
                        OptiKfDesc &d) {
    std::memset(&d, 0, sizeof d);
    d.struct_size = sizeof d;
    d.abi_version = OPTISTATE_KF_ABI_VERSION;
    d.dtype = (int32_t)geti(cfg, "dtype", OPTI_KF_F64);
    d.algo = (int32_t)geti(cfg, "algo", OPTI_KF_ALGO_AUTO);
    d.cov_model = (int32_t)geti(cfg, "cov_model", OPTI_KF_COV_PREDICT);
    d.phases = (int32_t)geti(cfg, "phases", OPTI_KF_PHASE_ALL);
    d.n_traj = geti(cfg, "n_traj", 0);
    d.n_steps = geti(cfg, "n_steps", 0);
    d.n_streams = geti(cfg, "n_streams", 0);
    d.stream_offset = geti(cfg, "stream_offset", 0);
    d.x0_per_traj = (int32_t)geti(cfg, "x0_per_traj", 0);
    d.p0_kind = (int32_t)geti(cfg, "p0_kind", OPTI_KF_MAT_NONE);
    d.q_kind = (int32_t)geti(cfg, "q_kind", OPTI_KF_MAT_DIAG);
    d.r_kind = (int32_t)geti(cfg, "r_kind", OPTI_KF_MAT_DIAG);
    d.ckpt_every = geti(cfg, "ckpt_every", 0);
    d.flags = (int32_t)geti(cfg, "flags", 0);
    d.dt = consts.at("dt");
    d.mass = consts.at("mass");
    d.inertia[0] = consts.at("inertia0");
    d.inertia[1] = consts.at("inertia1");
    d.inertia[2] = consts.at("inertia2");
    d.gravity = consts.at("gravity");
    TORCH_CHECK(d.dtype == OPTI_KF_F64 || d.dtype == OPTI_KF_F32, "optistate_b200: bad dtype");
    TORCH_CHECK(d.n_traj >= 0 && d.n_steps >= 0 && d.n_streams > 0, "optistate_b200: bad sizes");
    auto x0 = tensors.find("x0");
    TORCH_CHECK(x0 != tensors.end() && x0->second.is_cuda(), "optistate_b200: 'x0' must be a CUDA tensor (there is no CPU path)");
    const Checker ck{d.dtype == OPTI_KF_F64 ? at::kDouble : at::kFloat, x0->second.device()};
    const int64_t N = d.n_traj, T = d.n_steps, S = d.n_streams;
    const bool m = d.phases & OPTI_KF_PHASE_MEASURE, p = d.phases & OPTI_KF_PHASE_PREDICT, u = d.phases & OPTI_KF_PHASE_UPDATE;
    d.imu = ck.get(tensors, "imu", T * 6 * S, m);
    d.p = ck.get(tensors, "p", T * 12 * S, m || p);
    d.dp = ck.get(tensors, "dp", T * 12 * S, m);
    d.contact = ck.get(tensors, "contact", T * 4 * S, m);
    d.f = ck.get(tensors, "f", T * 12 * S, p);
    d.z_in = ck.get(tensors, "z_in", T * 10 * S, u && !m);
    d.body_ref = ck.get(tensors, "body_ref", T * 12 * S, p && d.cov_model == OPTI_KF_COV_MPC);
    d.truth = ck.get(tensors, "truth", T * 12 * S, false);
    d.nominal = ck.get(tensors, "nominal", T * 12 * S, false);
    d.x0 = ck.get(tensors, "x0", d.x0_per_traj ? 12 * N : 12, true);
    d.P0 = ck.get(tensors, "P0", mat_numel(d.p0_kind, 12, N), d.p0_kind != OPTI_KF_MAT_NONE);
    d.Q = ck.get(tensors, "Q", mat_numel(d.q_kind, 12, N), true);
    d.R = ck.get(tensors, "R", mat_numel(d.r_kind, 10, N), true);
    {
        auto it = tensors.find("stream_index");
        if (it != tensors.end()) {
            const at::Tensor &t = it->second;
            TORCH_CHECK(t.is_cuda() && t.device() == ck.dev && t.scalar_type() == at::kInt && t.is_contiguous() && t.numel() == N,
                        "optistate_b200: 'stream_index' must be a contiguous int32 CUDA tensor of N elements");
            d.stream_index = t.data_ptr<int32_t>();
        }
        auto is = tensors.find("status");
        if (is != tensors.end()) {
            const at::Tensor &t = is->second;
            TORCH_CHECK(t.is_cuda() && t.device() == ck.dev && t.scalar_type() == at::kInt && t.is_contiguous() && t.numel() == N,
                        "optistate_b200: 'status' must be a contiguous int32 CUDA tensor of N elements");
            d.status = reinterpret_cast<uint32_t *>(t.data_ptr<int32_t>());
        }
    }
    const int64_t n_ckpt = d.ckpt_every > 0 ? T / d.ckpt_every : 0;
    d.x_steps = const_cast<void *>(ck.get(tensors, "x_steps", T * 12 * N, false));
    d.x_model_steps = const_cast<void *>(ck.get(tensors, "x_model_steps", T * 12 * N, false));
    d.p_world_steps = const_cast<void *>(ck.get(tensors, "p_world_steps", T * 12 * N, false));
    d.z_steps = const_cast<void *>(ck.get(tensors, "z_steps", T * 10 * N, false));
    d.p_trace_steps = const_cast<void *>(ck.get(tensors, "p_trace_steps", T * N, false));
    d.k_gain_steps = const_cast<void *>(ck.get(tensors, "k_gain_steps", T * N, false));
    d.nis_steps = const_cast<void *>(ck.get(tensors, "nis_steps", T * N, false));
    d.P_ckpt = const_cast<void *>(ck.get(tensors, "P_ckpt", n_ckpt * 144 * N, false));
    d.x_final = const_cast<void *>(ck.get(tensors, "x_final", 12 * N, false));
    d.P_final = const_cast<void *>(ck.get(tensors, "P_final", 144 * N, false));
    d.K_final = const_cast<void *>(ck.get(tensors, "K_final", 120 * N, false));
    // fused all-gather: 'summary' is then the whole job's [52][summary_ld] array, this rank owning columns
    // [summary_col0, summary_col0 + N), and summary_peer<k> the addresses of the other GPUs' copies (peer_open)
    d.summary_ld = geti(cfg, "summary_ld", 0);
    const int64_t col0 = geti(cfg, "summary_col0", 0);
    TORCH_CHECK(d.summary_ld >= 0 && col0 >= 0 && (d.summary_ld == 0 ? col0 == 0 : col0 + N <= d.summary_ld),
                "optistate_b200: summary columns [", col0, ", ", col0 + N, ") do not fit summary_ld = ", d.summary_ld);
    d.summary = const_cast<void *>(ck.get(tensors, "summary", (int64_t)OPTI_KF_SUMMARY_ROWS * (d.summary_ld ? d.summary_ld : N), false));
    if (d.summary) {
        const size_t esz = d.dtype == OPTI_KF_F64 ? 8 : 4;
        d.summary = static_cast<char *>(d.summary) + (size_t)col0 * esz;
        d.n_summary_peers = (int32_t)geti(cfg, "n_summary_peers", 0);
        TORCH_CHECK(d.n_summary_peers >= 0 && d.n_summary_peers <= OPTI_KF_MAX_PEERS, "optistate_b200: at most ", OPTI_KF_MAX_PEERS, " peers");
        for (int k = 0; k < d.n_summary_peers; ++k) {
            const int64_t addr = geti(cfg, ("summary_peer" + std::to_string(k)).c_str(), 0);
            TORCH_CHECK(addr != 0, "optistate_b200: summary_peer", k, " missing");
            d.summary_peers[k] = reinterpret_cast<char *>((uintptr_t)addr) + (size_t)col0 * esz;
        }
    }
    {
        auto iw = tensors.find("workspace");
        if (iw != tensors.end()) {
            const at::Tensor &t = iw->second;
            TORCH_CHECK(t.is_cuda() && t.device() == ck.dev && t.scalar_type() == at::kByte && t.is_contiguous(),
                        "optistate_b200: 'workspace' must be a contiguous uint8 CUDA tensor");
            d.workspace = t.data_ptr();
            d.workspace_bytes = (size_t)t.numel();
        }
    }
    return ck.dev;
}

int64_t kf_batch(const std::map<std::string, int64_t> &cfg, const std::map<std::string, double> &consts, const TensorMap &tensors) {
    OptiKfDesc d;
    const c10::cuda::CUDAGuard guard(filter_desc(cfg, consts, tensors, d));
    if (geti(cfg, "query_workspace", 0)) {
        size_t bytes = 0;
        const int rc = optistate_kf_workspace_bytes(&d, &bytes);
        return rc < 0 ? rc : (int64_t)bytes;
    }
    return optistate_kf_batch(&d, at::cuda::getCurrentCUDAStream().stream());
}

// The backward passes: the filter's tensors as for kf_batch, plus the smoother's x_smooth [T][12][N] (required) or the E-step's
// noise_stats [23][N] (required; x_smooth optional), optional var_smooth [T][12][N], or the adjoint's x_bar [T][12][N] and grad
// [46][N] (both required), and the uint8 storage of the entry's storage query, smooth_storage, em_storage or adj_storage (cfg
// query_storage = 1 returns that size instead of running).  Desc: OptiKfSmoothDesc, OptiKfNoiseEmDesc or OptiKfAdjointDesc.
template <typename Desc>
int64_t run_backward(int (*storage_bytes)(const OptiKfDesc *, size_t *), int (*entry)(const Desc *, void *),
                     const std::map<std::string, int64_t> &cfg, const std::map<std::string, double> &consts, const TensorMap &tensors) {
    constexpr bool stats = std::is_same<Desc, OptiKfNoiseEmDesc>::value, adj = std::is_same<Desc, OptiKfAdjointDesc>::value;
    OptiKfDesc d;
    const c10::Device dev = filter_desc(cfg, consts, tensors, d);
    const c10::cuda::CUDAGuard guard(dev);
    if (geti(cfg, "query_storage", 0)) {
        size_t bytes = 0;
        const int rc = storage_bytes(&d, &bytes);
        return rc < 0 ? rc : (int64_t)bytes;
    }
    const Checker ck{d.dtype == OPTI_KF_F64 ? at::kDouble : at::kFloat, dev};
    const int64_t N = d.n_traj, T = d.n_steps;
    Desc s;
    std::memset(&s, 0, sizeof s);
    s.struct_size = sizeof s;
    s.abi_version = OPTISTATE_KF_ABI_VERSION;
    s.filter = &d;
    if constexpr (adj) {
        s.x_bar = ck.get(tensors, "x_bar", T * 12 * N, true);
        s.grad = const_cast<void *>(ck.get(tensors, "grad", OPTI_KF_ADJ_ROWS * N, true));
    } else {
        if constexpr (stats) s.stats = const_cast<void *>(ck.get(tensors, "noise_stats", OPTI_KF_EM_STATS_ROWS * N, true));
        s.x_smooth = const_cast<void *>(ck.get(tensors, "x_smooth", T * 12 * N, !stats));
        s.var_smooth = const_cast<void *>(ck.get(tensors, "var_smooth", T * 12 * N, false));
    }
    const std::string key = adj ? "adj_storage" : stats ? "em_storage" : "smooth_storage";
    auto is = tensors.find(key);
    TORCH_CHECK(is != tensors.end(), "optistate_b200: missing tensor '", key, "'");
    const at::Tensor &t = is->second;
    TORCH_CHECK(t.is_cuda() && t.device() == dev && t.scalar_type() == at::kByte && t.is_contiguous(),
                "optistate_b200: '", key, "' must be a contiguous uint8 CUDA tensor");
    s.storage = t.data_ptr();
    s.storage_bytes = (size_t)t.numel();
    return entry(&s, at::cuda::getCurrentCUDAStream().stream());
}

int64_t kf_smooth(const std::map<std::string, int64_t> &cfg, const std::map<std::string, double> &consts, const TensorMap &tensors) {
    return run_backward(optistate_kf_smooth_storage_bytes, optistate_kf_smooth, cfg, consts, tensors);
}
int64_t kf_smooth_full(const std::map<std::string, int64_t> &cfg, const std::map<std::string, double> &consts, const TensorMap &tensors) {
    return run_backward(optistate_kf_smooth_full_storage_bytes, optistate_kf_smooth_full, cfg, consts, tensors);
}
int64_t kf_noise_em_stats(const std::map<std::string, int64_t> &cfg, const std::map<std::string, double> &consts, const TensorMap &tensors) {
    return run_backward(optistate_kf_noise_em_storage_bytes, optistate_kf_noise_em_stats, cfg, consts, tensors);
}
int64_t kf_noise_em_full_stats(const std::map<std::string, int64_t> &cfg, const std::map<std::string, double> &consts,
                               const TensorMap &tensors) {
    return run_backward(optistate_kf_noise_em_full_storage_bytes, optistate_kf_noise_em_full_stats, cfg, consts, tensors);
}

int64_t kf_adjoint(const std::map<std::string, int64_t> &cfg, const std::map<std::string, double> &consts, const TensorMap &tensors) {
    return run_backward(optistate_kf_adjoint_storage_bytes, optistate_kf_adjoint, cfg, consts, tensors);
}

int kf_resolve_algo(const std::map<std::string, int64_t> &cfg) {
    // shape-free query: only kinds / phases / model matter, pointers are faked as non-null
    OptiKfDesc d;
    std::memset(&d, 0, sizeof d);
    static const double dummy = 0.0;
    d.struct_size = sizeof d;
    d.abi_version = OPTISTATE_KF_ABI_VERSION;
    d.dtype = (int32_t)geti(cfg, "dtype", OPTI_KF_F64);
    d.algo = (int32_t)geti(cfg, "algo", OPTI_KF_ALGO_AUTO);
    d.cov_model = (int32_t)geti(cfg, "cov_model", OPTI_KF_COV_PREDICT);
    d.phases = (int32_t)geti(cfg, "phases", OPTI_KF_PHASE_ALL);
    d.n_traj = 1; d.n_steps = 1; d.n_streams = 1;
    d.p0_kind = (int32_t)geti(cfg, "p0_kind", OPTI_KF_MAT_NONE);
    d.q_kind = (int32_t)geti(cfg, "q_kind", OPTI_KF_MAT_DIAG);
    d.r_kind = (int32_t)geti(cfg, "r_kind", OPTI_KF_MAT_DIAG);
    d.dt = 0.01; d.mass = 1; d.inertia[0] = d.inertia[1] = d.inertia[2] = 1;
    d.imu = d.p = d.dp = d.contact = d.f = d.z_in = d.body_ref = d.x0 = d.P0 = d.Q = d.R = &dummy;
    if (geti(cfg, "want_K", 0)) d.K_final = const_cast<double *>(&dummy);
    return optistate_kf_resolve_algo(&d);
}

int kf_measure(int64_t dtype, int64_t n_steps, int64_t n_streams, const TensorMap &tensors) {
    OptiKfMeasureDesc d;
    std::memset(&d, 0, sizeof d);
    d.struct_size = sizeof d;
    d.abi_version = OPTISTATE_KF_ABI_VERSION;
    d.dtype = (int32_t)dtype;
    d.n_steps = n_steps;
    d.n_streams = n_streams;
    auto imu = tensors.find("imu");
    TORCH_CHECK(imu != tensors.end() && imu->second.is_cuda(), "optistate_b200: 'imu' must be a CUDA tensor (there is no CPU path)");
    const Checker ck{dtype == OPTI_KF_F64 ? at::kDouble : at::kFloat, imu->second.device()};
    const c10::cuda::CUDAGuard guard(ck.dev);
    const int64_t T = n_steps, S = n_streams;
    d.imu = ck.get(tensors, "imu", T * 6 * S, true);
    d.p = ck.get(tensors, "p", T * 12 * S, true);
    d.dp = ck.get(tensors, "dp", T * 12 * S, true);
    d.contact = ck.get(tensors, "contact", T * 4 * S, true);
    d.z = const_cast<void *>(ck.get(tensors, "z", T * 10 * S, false));
    d.odom = const_cast<void *>(ck.get(tensors, "odom", T * 4 * S, false));
    auto is = tensors.find("status");
    if (is != tensors.end()) {
        const at::Tensor &t = is->second;
        TORCH_CHECK(t.is_cuda() && t.scalar_type() == at::kInt && t.is_contiguous() && t.numel() == S,
                    "optistate_b200: 'status' must be a contiguous int32 CUDA tensor of S elements");
        d.status = reinterpret_cast<uint32_t *>(t.data_ptr<int32_t>());
    }
    return optistate_kf_measure(&d, at::cuda::getCurrentCUDAStream().stream());
}

// feature rows [N][T][60] from the filter outputs and the base streams
int kf_features(int64_t dtype, int64_t n_traj, int64_t n_steps, int64_t n_streams, int64_t stream_offset, const TensorMap &tensors) {
    OptiKfFeatureDesc d;
    std::memset(&d, 0, sizeof d);
    d.struct_size = sizeof d;
    d.abi_version = OPTISTATE_KF_ABI_VERSION;
    d.dtype = (int32_t)dtype;
    d.n_traj = n_traj; d.n_steps = n_steps; d.n_streams = n_streams; d.stream_offset = stream_offset;
    auto xs = tensors.find("x_steps");
    TORCH_CHECK(xs != tensors.end() && xs->second.is_cuda(), "optistate_b200: 'x_steps' must be a CUDA tensor (there is no CPU path)");
    const Checker ck{dtype == OPTI_KF_F64 ? at::kDouble : at::kFloat, xs->second.device()};
    const c10::cuda::CUDAGuard guard(ck.dev);
    const int64_t N = n_traj, T = n_steps, S = n_streams;
    d.x_steps = ck.get(tensors, "x_steps", T * 12 * N, true);
    d.p_world_steps = ck.get(tensors, "p_world_steps", T * 12 * N, true);
    d.imu = ck.get(tensors, "imu", T * 6 * S, true);
    d.imu_acc = ck.get(tensors, "imu_acc", T * 6 * S, false);
    d.f = ck.get(tensors, "f", T * 12 * S, true);
    d.dp = ck.get(tensors, "dp", T * 12 * S, true);
    d.rows = const_cast<void *>(ck.get(tensors, "rows", N * T * OPTI_KF_FEATURES, true));
    auto it = tensors.find("stream_index");
    if (it != tensors.end()) {
        const at::Tensor &t = it->second;
        TORCH_CHECK(t.is_cuda() && t.scalar_type() == at::kInt && t.is_contiguous() && t.numel() == N, "optistate_b200: bad 'stream_index'");
        d.stream_index = t.data_ptr<int32_t>();
    }
    return optistate_kf_features(&d, at::cuda::getCurrentCUDAStream().stream());
}

int kf_minmax(const at::Tensor &rows, at::Tensor mn, at::Tensor mx) {
    TORCH_CHECK(rows.is_cuda() && rows.dim() == 2 && rows.is_contiguous(), "optistate_b200: rows must be a contiguous 2-D CUDA tensor");
    TORCH_CHECK(rows.scalar_type() == at::kDouble || rows.scalar_type() == at::kFloat, "optistate_b200: rows must be float64 or float32");
    TORCH_CHECK(mn.is_cuda() && mx.is_cuda() && mn.scalar_type() == rows.scalar_type() && mx.scalar_type() == rows.scalar_type() &&
                    mn.numel() == rows.size(1) && mx.numel() == rows.size(1) && mn.is_contiguous() && mx.is_contiguous(),
                "optistate_b200: min/max must be CUDA vectors of n_cols elements");
    const c10::cuda::CUDAGuard guard(rows.device());
    const int dtype = rows.scalar_type() == at::kDouble ? OPTI_KF_F64 : OPTI_KF_F32;
    const size_t nb = optistate_kf_minmax_scratch_bytes(dtype, (int32_t)rows.size(1));
    at::Tensor scratch = at::empty({(int64_t)nb}, rows.options().dtype(at::kByte));
    return optistate_kf_minmax(dtype, rows.data_ptr(), rows.size(0), (int32_t)rows.size(1), mn.data_ptr(), mx.data_ptr(), scratch.data_ptr(), nb,
                               at::cuda::getCurrentCUDAStream().stream());
}

int kf_windows(const at::Tensor &rows, const std::optional<at::Tensor> &latent, const at::Tensor &mn, const at::Tensor &mx, int64_t n_groups,
               int64_t seq_len, at::Tensor out) {
    TORCH_CHECK(rows.is_cuda() && rows.dim() == 2 && rows.is_contiguous(), "optistate_b200: rows must be a contiguous 2-D CUDA tensor");
    TORCH_CHECK(rows.scalar_type() == at::kDouble || rows.scalar_type() == at::kFloat, "optistate_b200: rows must be float64 or float32");
    TORCH_CHECK(n_groups > 0 && rows.size(0) % n_groups == 0, "optistate_b200: n_rows must be a multiple of n_groups");
    const int64_t rpg = rows.size(0) / n_groups, cols = rows.size(1);
    int64_t n_lat = 0;
    const float *lat = nullptr;
    if (latent.has_value()) {
        const at::Tensor &l = *latent;
        TORCH_CHECK(l.is_cuda() && l.scalar_type() == at::kFloat && l.is_contiguous() && l.dim() == 2 && l.size(0) == rows.size(0),
                    "optistate_b200: latent must be a contiguous float32 CUDA tensor [n_rows, n_latent]");
        n_lat = l.size(1);
        lat = l.data_ptr<float>();
    }
    TORCH_CHECK(mn.is_cuda() && mx.is_cuda() && mn.scalar_type() == rows.scalar_type() && mx.scalar_type() == rows.scalar_type() &&
                    mn.numel() == cols && mx.numel() == cols, "optistate_b200: bad min/max");
    TORCH_CHECK(out.is_cuda() && out.scalar_type() == at::kFloat && out.is_contiguous() &&
                    out.numel() == n_groups * (rpg - seq_len + 1) * seq_len * (cols + n_lat), "optistate_b200: bad out");
    const c10::cuda::CUDAGuard guard(rows.device());
    const size_t nb = optistate_kf_windows_scratch_bytes(n_groups, rpg, (int32_t)cols, (int32_t)n_lat);
    at::Tensor scratch = at::empty({(int64_t)nb}, rows.options().dtype(at::kByte));
    return optistate_kf_windows(rows.scalar_type() == at::kDouble ? OPTI_KF_F64 : OPTI_KF_F32, rows.data_ptr(), lat, mn.data_ptr(), mx.data_ptr(),
                                n_groups, rpg, (int32_t)cols, (int32_t)n_lat, (int32_t)seq_len, out.data_ptr<float>(), scratch.data_ptr(), nb,
                                at::cuda::getCurrentCUDAStream().stream());
}

// Q / R identification pass: tensors gt, imu, p, dp, contact, f [T][C][S]; q_diag [12][N], r_diag [10][N]; optional status [N]
int kf_identify_noise(int64_t dtype, int64_t n_traj, int64_t n_steps, int64_t n_streams, int64_t stream_offset, int64_t alias_last,
                      const std::map<std::string, double> &consts, const TensorMap &tensors) {
    OptiKfIdentifyDesc d;
    std::memset(&d, 0, sizeof d);
    d.struct_size = sizeof d;
    d.abi_version = OPTISTATE_KF_ABI_VERSION;
    d.dtype = (int32_t)dtype;
    d.alias_last_measurement = (int32_t)alias_last;
    d.n_traj = n_traj; d.n_steps = n_steps; d.n_streams = n_streams; d.stream_offset = stream_offset;
    d.dt = consts.at("dt"); d.mass = consts.at("mass"); d.gravity = consts.at("gravity");
    d.inertia[0] = consts.at("inertia0"); d.inertia[1] = consts.at("inertia1"); d.inertia[2] = consts.at("inertia2");
    auto gt = tensors.find("gt");
    TORCH_CHECK(gt != tensors.end() && gt->second.is_cuda(), "optistate_b200: 'gt' must be a CUDA tensor (there is no CPU path)");
    const Checker ck{dtype == OPTI_KF_F64 ? at::kDouble : at::kFloat, gt->second.device()};
    const c10::cuda::CUDAGuard guard(ck.dev);
    const int64_t N = n_traj, T = n_steps, S = n_streams;
    d.gt = ck.get(tensors, "gt", T * 12 * S, true);
    d.imu = ck.get(tensors, "imu", T * 6 * S, true);
    d.p = ck.get(tensors, "p", T * 12 * S, true);
    d.dp = ck.get(tensors, "dp", T * 12 * S, true);
    d.contact = ck.get(tensors, "contact", T * 4 * S, true);
    d.f = ck.get(tensors, "f", T * 12 * S, true);
    d.q_diag = const_cast<void *>(ck.get(tensors, "q_diag", 12 * N, true));
    d.r_diag = const_cast<void *>(ck.get(tensors, "r_diag", 10 * N, true));
    auto it = tensors.find("stream_index");
    if (it != tensors.end()) {
        const at::Tensor &t = it->second;
        TORCH_CHECK(t.is_cuda() && t.scalar_type() == at::kInt && t.is_contiguous() && t.numel() == N, "optistate_b200: bad 'stream_index'");
        d.stream_index = t.data_ptr<int32_t>();
    }
    auto is = tensors.find("status");
    if (is != tensors.end()) {
        const at::Tensor &t = is->second;
        TORCH_CHECK(t.is_cuda() && t.scalar_type() == at::kInt && t.is_contiguous() && t.numel() == N, "optistate_b200: bad 'status'");
        d.status = reinterpret_cast<uint32_t *>(t.data_ptr<int32_t>());
    }
    const size_t nb = optistate_kf_identify_scratch_bytes((int)dtype, N, T);
    at::Tensor scratch = at::empty({(int64_t)nb}, gt->second.options().dtype(at::kByte));
    d.scratch = scratch.data_ptr();
    d.scratch_bytes = nb;
    return optistate_kf_identify_noise(&d, at::cuda::getCurrentCUDAStream().stream());
}

// Convex force MPC: x [12][N], body_ref [5][12][N], p [12][N], contact [4][N] -> forces [5][12][N], status [N]
int kf_mpc_forces(int64_t n, int64_t max_free_legs, const std::map<std::string, double> &consts, const std::vector<double> &w_state, const TensorMap &tensors) {
    OptiKfMpcDesc d;
    std::memset(&d, 0, sizeof d);
    d.struct_size = sizeof d;
    d.abi_version = OPTISTATE_KF_ABI_VERSION;
    d.dtype = OPTI_KF_F64;
    d.n_problems = n;
    d.max_free_legs = (int32_t)max_free_legs;
    auto x = tensors.find("x");
    TORCH_CHECK(x != tensors.end() && x->second.is_cuda(), "optistate_b200: 'x' must be a CUDA tensor (there is no CPU path)");
    TORCH_CHECK(w_state.size() == 12, "optistate_b200: w_state needs 12 entries");
    const Checker ck{at::kDouble, x->second.device()};
    const c10::cuda::CUDAGuard guard(ck.dev);
    d.x = ck.get(tensors, "x", 12 * n, true);
    d.body_ref = ck.get(tensors, "body_ref", OPTI_KF_MPC_HORIZON * 12 * n, true);
    d.p = ck.get(tensors, "p", 12 * n, true);
    d.contact = ck.get(tensors, "contact", 4 * n, true);
    d.forces = const_cast<void *>(ck.get(tensors, "forces", OPTI_KF_MPC_HORIZON * 12 * n, true));
    auto is = tensors.find("status");
    TORCH_CHECK(is != tensors.end(), "optistate_b200: missing tensor 'status'");
    const at::Tensor &st = is->second;
    TORCH_CHECK(st.is_cuda() && st.device() == ck.dev && st.scalar_type() == at::kInt && st.is_contiguous() && st.numel() == n, "optistate_b200: bad 'status'");
    d.status = reinterpret_cast<uint32_t *>(st.data_ptr<int32_t>());
    auto iw = tensors.find("warm_set");
    if (iw != tensors.end()) {
        const at::Tensor &t = iw->second;
        TORCH_CHECK(t.is_cuda() && t.device() == ck.dev && t.scalar_type() == at::kInt && t.is_contiguous() && t.numel() == OPTI_KF_MPC_HORIZON * n,
                    "optistate_b200: bad 'warm_set'");
        d.warm_set = reinterpret_cast<uint32_t *>(t.data_ptr<int32_t>());
        d.warm_mult = const_cast<void *>(ck.get(tensors, "warm_mult", OPTI_KF_MPC_HORIZON * 4 * 5 * n, true));
    }
    auto sv = consts.find("solver");
    d.solver = sv == consts.end() ? 0 : (int32_t)sv->second;
    auto mc = consts.find("max_changes");
    d.max_changes = mc == consts.end() ? 0 : (int32_t)mc->second;
    d.dt = consts.at("dt"); d.mass = consts.at("mass"); d.gravity = consts.at("gravity");
    d.inertia[0] = consts.at("inertia0"); d.inertia[1] = consts.at("inertia1"); d.inertia[2] = consts.at("inertia2");
    d.mu = consts.at("mu"); d.fz_max = consts.at("fz_max"); d.w_force = consts.at("w_force");
    for (int k = 0; k < 12; ++k) d.w_state[k] = w_state[k];
    return optistate_kf_mpc_forces(&d, at::cuda::getCurrentCUDAStream().stream());
}

// The closed loop of the reference driver (estimate_state_mpc at every step) for N trajectories x T steps: one call, queued on the
// current stream.  tensors: imu p dp contact body_ref x0 Q R [P0] x_steps workspace [forces p_world_steps mpc_status status]
int kf_closed_loop(const std::map<std::string, int64_t> &cfg, const std::map<std::string, double> &consts, const std::vector<double> &w_state,
                   const TensorMap &tensors) {
    OptiKfClosedLoopDesc d;
    std::memset(&d, 0, sizeof d);
    d.struct_size = sizeof d;
    d.abi_version = OPTISTATE_KF_ABI_VERSION;
    d.dtype = OPTI_KF_F64;
    const int64_t N = cfg.at("n_traj"), T = cfg.at("n_steps");
    d.n_traj = N; d.n_steps = T;
    d.max_free_legs = (int32_t)geti(cfg, "max_free_legs", 0);
    d.x0_per_traj = (int32_t)geti(cfg, "x0_per_traj", 1);
    d.p0_kind = (int32_t)geti(cfg, "p0_kind", OPTI_KF_MAT_NONE);
    d.q_kind = (int32_t)geti(cfg, "q_kind", OPTI_KF_MAT_DIAG);
    d.r_kind = (int32_t)geti(cfg, "r_kind", OPTI_KF_MAT_DIAG);
    d.warm_start = (int32_t)geti(cfg, "warm_start", 1);
    d.solver = (int32_t)geti(cfg, "solver", 0);
    d.max_changes = (int32_t)geti(cfg, "max_changes", 0);
    auto x = tensors.find("imu");
    TORCH_CHECK(x != tensors.end() && x->second.is_cuda(), "optistate_b200: 'imu' must be a CUDA tensor (there is no CPU path)");
    TORCH_CHECK(w_state.size() == 12, "optistate_b200: w_state needs 12 entries");
    const Checker ck{at::kDouble, x->second.device()};
    const c10::cuda::CUDAGuard guard(ck.dev);
    d.imu = ck.get(tensors, "imu", T * 6 * N, true);
    d.p = ck.get(tensors, "p", T * 12 * N, true);
    d.dp = ck.get(tensors, "dp", T * 12 * N, true);
    d.contact = ck.get(tensors, "contact", T * 4 * N, true);
    d.body_ref = ck.get(tensors, "body_ref", T * OPTI_KF_MPC_HORIZON * 12 * N, true);
    d.x0 = ck.get(tensors, "x0", d.x0_per_traj ? 12 * N : 12, true);
    d.Q = ck.get(tensors, "Q", mat_numel(d.q_kind, 12, N), true);
    d.R = ck.get(tensors, "R", mat_numel(d.r_kind, 10, N), true);
    if (d.p0_kind != OPTI_KF_MAT_NONE) d.P0 = ck.get(tensors, "P0", mat_numel(d.p0_kind, 12, N), true);
    d.x_steps = const_cast<void *>(ck.get(tensors, "x_steps", T * 12 * N, true));
    d.forces = const_cast<void *>(ck.get(tensors, "forces", T * 12 * N, false));
    d.p_world_steps = const_cast<void *>(ck.get(tensors, "p_world_steps", T * 12 * N, false));
    for (const char *name : {"mpc_status", "status"}) {
        auto it = tensors.find(name);
        if (it == tensors.end()) continue;
        const at::Tensor &t = it->second;
        const int64_t want = std::string(name) == "status" ? N : T * N;
        TORCH_CHECK(t.is_cuda() && t.device() == ck.dev && t.scalar_type() == at::kInt && t.is_contiguous() && t.numel() == want, "optistate_b200: bad '", name, "'");
        (std::string(name) == "status" ? d.status : d.mpc_status) = reinterpret_cast<uint32_t *>(t.data_ptr<int32_t>());
    }
    auto w = tensors.find("workspace");
    TORCH_CHECK(w != tensors.end() && w->second.is_cuda() && w->second.device() == ck.dev && w->second.is_contiguous(), "optistate_b200: bad 'workspace'");
    d.workspace = w->second.data_ptr();
    d.workspace_bytes = (size_t)w->second.numel() * w->second.element_size();
    d.dt = consts.at("dt"); d.mass = consts.at("mass"); d.gravity = consts.at("gravity");
    d.inertia[0] = consts.at("inertia0"); d.inertia[1] = consts.at("inertia1"); d.inertia[2] = consts.at("inertia2");
    d.mu = consts.at("mu"); d.fz_max = consts.at("fz_max"); d.w_force = consts.at("w_force");
    for (int k = 0; k < 12; ++k) d.w_state[k] = w_state[k];
    return optistate_kf_closed_loop(&d, at::cuda::getCurrentCUDAStream().stream());
}

// ---- peer memory (fused summary all-gather) ----
at::Tensor peer_alloc(int64_t nbytes, int64_t device_index) {
    TORCH_CHECK(nbytes > 0, "optistate_b200: peer_alloc needs a positive size");
    const c10::cuda::CUDAGuard guard((c10::DeviceIndex)device_index);
    void *ptr = nullptr;
    const int rc = optistate_kf_peer_alloc((size_t)nbytes, &ptr);
    TORCH_CHECK(rc == 0, "optistate_kf_peer_alloc: ", optistate_kf_strerror(rc));
    const int dev = (int)device_index;
    return at::from_blob(ptr, {nbytes}, [dev](void *q) { const c10::cuda::CUDAGuard g((c10::DeviceIndex)dev); optistate_kf_peer_free(q); },
                         at::TensorOptions().dtype(at::kByte).device(at::kCUDA, (c10::DeviceIndex)device_index));
}

py::bytes peer_export(const at::Tensor &t) {
    TORCH_CHECK(t.is_cuda() && t.storage_offset() == 0, "optistate_b200: peer_export needs the tensor peer_alloc returned");
    const c10::cuda::CUDAGuard guard(t.device());
    unsigned char h[OPTI_KF_PEER_HANDLE_BYTES];
    const int rc = optistate_kf_peer_export(t.data_ptr(), h);
    TORCH_CHECK(rc == 0, "optistate_kf_peer_export: ", optistate_kf_strerror(rc));
    return py::bytes(reinterpret_cast<const char *>(h), sizeof h);
}

int64_t peer_open(const std::string &handle, int64_t device_index) {
    TORCH_CHECK(handle.size() == OPTI_KF_PEER_HANDLE_BYTES, "optistate_b200: bad peer handle");
    const c10::cuda::CUDAGuard guard((c10::DeviceIndex)device_index);
    void *ptr = nullptr;
    const int rc = optistate_kf_peer_open(reinterpret_cast<const unsigned char *>(handle.data()), &ptr);
    TORCH_CHECK(rc == 0, "optistate_kf_peer_open: ", optistate_kf_strerror(rc), " (peer memory needs all ranks on one box)");
    return (int64_t)(uintptr_t)ptr;
}

void peer_close(int64_t addr, int64_t device_index) {
    const c10::cuda::CUDAGuard guard((c10::DeviceIndex)device_index);
    optistate_kf_peer_close(reinterpret_cast<void *>((uintptr_t)addr));
}

std::pair<double, double> fma_peak(int64_t dtype, int64_t fma_per_thread) {
    double flops = 0, secs = 0;
    const int rc = optistate_fma_peak((int)dtype, fma_per_thread, &flops, &secs, at::cuda::getCurrentCUDAStream().stream());
    TORCH_CHECK(rc == 0, "optistate_fma_peak: ", optistate_kf_strerror(rc));
    return {flops, secs};
}

// ---- the drop-in class's step (optistate_b200/kalman_filter.py) through ONE call of this binding ------------------------------
// The class keeps one pinned host block with a FIXED layout (the offsets below, in doubles; kalman_filter.py mirrors them) and a device
// block of the same size.  `ops` says which of the reference's methods run, in the reference's order: get_odom + the measurement
// scatter (OPTI_KF_PHASE_MEASURE -> optistate_kf_measure), predict / predict_mpc (PHASE_PREDICT -> optistate_kf_batch, JOINT, dense
// Q / R / P like the class holds them) and update (PHASE_UPDATE).  PREDICT | UPDATE runs the update on the prediction's outputs in the
// same call (two launches, no host round trip in between) and returns both results: the class hands out the second one when its
// update() finds state and measurement untouched since.  One stream synchronisation per call.
// `mode`: 0 = inputs uploaded and outputs downloaded with asynchronous copies; 1 = inputs uploaded, the kernels write their outputs and
// status words straight into the pinned host block (zero-copy stores over PCIe, no download); 2 = the kernels also read their inputs
// from the pinned block (no upload either).
enum : int64_t {
    CS_X = 0, CS_P = 12, CS_Q = 156, CS_R = 300, CS_FEET = 400, CS_F = 412, CS_Z = 424, CS_BREF = 434, CS_IMU = 446, CS_DP = 452,
    CS_CONTACT = 464, CS_IN_END = 468,
    CS_PRED_X = 468, CS_PRED_P = 480, CS_PRED_FEET = 624, CS_PRED_TRACE = 636,
    CS_UPD_X = 637, CS_UPD_P = 649, CS_UPD_K = 793, CS_UPD_TRACE = 913, CS_UPD_KGAIN = 914,
    CS_ODOM = 915, CS_END = 919, CS_TOTAL = 920
};

int64_t kf_class_step(int64_t ops, int64_t cov_model, const std::vector<double> &consts, at::Tensor h_block, at::Tensor d_block,
                      at::Tensor h_status, at::Tensor d_status, int64_t mode) {
    TORCH_CHECK(d_block.is_cuda() && d_status.is_cuda(), "optistate_b200: device buffers must be CUDA tensors (there is no CPU path)");
    TORCH_CHECK(h_block.is_pinned() && h_status.is_pinned(), "optistate_b200: host buffers must be pinned");
    TORCH_CHECK(h_block.scalar_type() == at::kDouble && d_block.scalar_type() == at::kDouble && h_block.numel() >= CS_TOTAL &&
                    d_block.numel() >= CS_TOTAL && h_block.is_contiguous() && d_block.is_contiguous(), "optistate_b200: bad state block");
    TORCH_CHECK(h_status.scalar_type() == at::kInt && d_status.scalar_type() == at::kInt && h_status.numel() >= 4 && d_status.numel() >= 4,
                "optistate_b200: bad status block");
    TORCH_CHECK(consts.size() == 6 && mode >= 0 && mode <= 2, "optistate_b200: bad arguments");
    const c10::cuda::CUDAGuard guard(d_block.device());
    cudaStream_t stream = at::cuda::getCurrentCUDAStream().stream();
    double *host = h_block.data_ptr<double>(), *dev = d_block.data_ptr<double>(), *host_alias = nullptr;
    uint32_t *hst = reinterpret_cast<uint32_t *>(h_status.data_ptr<int32_t>()), *dst = reinterpret_cast<uint32_t *>(d_status.data_ptr<int32_t>()),
             *hst_alias = nullptr;
    if (mode >= 1) {
        TORCH_CHECK(cudaHostGetDevicePointer((void **)&host_alias, host, 0) == cudaSuccess && cudaHostGetDevicePointer((void **)&hst_alias, hst, 0) == cudaSuccess,
                    "optistate_b200: the pinned block is not mapped into the device's address space");
    }
    const double *in = mode == 2 ? host_alias : dev;
    double *out = mode >= 1 ? host_alias : dev;
    uint32_t *st = mode >= 1 ? hst_alias : dst;
    hst[0] = hst[1] = hst[2] = 0;  // [0] predict, [1] update, [2] measure
    if (mode < 2) TORCH_CHECK(cudaMemcpyAsync(dev, host, CS_IN_END * sizeof(double), cudaMemcpyHostToDevice, stream) == cudaSuccess, "upload failed");
    if (mode == 0) TORCH_CHECK(cudaMemsetAsync(dst, 0, 4 * sizeof(uint32_t), stream) == cudaSuccess, "memset failed");
    if (ops & OPTI_KF_PHASE_MEASURE) {
        OptiKfMeasureDesc m;
        std::memset(&m, 0, sizeof m);
        m.struct_size = sizeof m;
        m.abi_version = OPTISTATE_KF_ABI_VERSION;
        m.dtype = OPTI_KF_F64;
        m.n_steps = 1;
        m.n_streams = 1;
        m.imu = in + CS_IMU; m.p = in + CS_FEET; m.dp = in + CS_DP; m.contact = in + CS_CONTACT;
        m.odom = out + CS_ODOM;
        m.status = st + 2;
        const int rc = optistate_kf_measure(&m, stream);
        if (rc != 0) return rc;
    }
    OptiKfDesc d;
    std::memset(&d, 0, sizeof d);
    d.struct_size = sizeof d;
    d.abi_version = OPTISTATE_KF_ABI_VERSION;
    d.dtype = OPTI_KF_F64;
    d.algo = OPTI_KF_ALGO_JOINT;
    d.n_traj = d.n_steps = d.n_streams = 1;
    d.dt = consts[0]; d.mass = consts[1]; d.inertia[0] = consts[2]; d.inertia[1] = consts[3]; d.inertia[2] = consts[4]; d.gravity = consts[5];
    d.p0_kind = d.q_kind = d.r_kind = OPTI_KF_MAT_DENSE;
    d.Q = in + CS_Q;
    d.R = in + CS_R;
    if (ops & OPTI_KF_PHASE_PREDICT) {
        OptiKfDesc p = d;
        p.phases = OPTI_KF_PHASE_PREDICT;
        p.cov_model = (int32_t)cov_model;
        p.x0 = in + CS_X; p.P0 = in + CS_P; p.p = in + CS_FEET; p.f = in + CS_F;
        if (cov_model == OPTI_KF_COV_MPC) p.body_ref = in + CS_BREF;
        p.x_final = out + CS_PRED_X; p.P_final = out + CS_PRED_P; p.p_world_steps = out + CS_PRED_FEET; p.p_trace_steps = out + CS_PRED_TRACE;
        p.status = st + 0;
        const int rc = optistate_kf_batch(&p, stream);
        if (rc != 0) return rc;
    }
    if (ops & OPTI_KF_PHASE_UPDATE) {
        OptiKfDesc u = d;
        u.phases = OPTI_KF_PHASE_UPDATE;
        const bool chained = ops & OPTI_KF_PHASE_PREDICT;  // the update of the state the prediction above has just written
        u.x0 = chained ? out + CS_PRED_X : in + CS_X;
        u.P0 = chained ? out + CS_PRED_P : in + CS_P;
        u.z_in = in + CS_Z;
        u.x_final = out + CS_UPD_X; u.P_final = out + CS_UPD_P; u.K_final = out + CS_UPD_K; u.p_trace_steps = out + CS_UPD_TRACE;
        u.k_gain_steps = out + CS_UPD_KGAIN;
        u.status = st + 1;
        const int rc = optistate_kf_batch(&u, stream);
        if (rc != 0) return rc;
    }
    if (mode == 0) {
        TORCH_CHECK(cudaMemcpyAsync(host + CS_IN_END, dev + CS_IN_END, (CS_END - CS_IN_END) * sizeof(double), cudaMemcpyDeviceToHost, stream) == cudaSuccess, "download failed");
        TORCH_CHECK(cudaMemcpyAsync(hst, dst, 4 * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream) == cudaSuccess, "download failed");
    }
    TORCH_CHECK(cudaStreamSynchronize(stream) == cudaSuccess, "optistate_b200: the launch failed");
    return 0;
}

}  // namespace

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
    m.doc() = "PyTorch loader of liboptistate_kf.so (C ABI in include/optistate_kf.h)";
    m.def("kf_batch", &kf_batch);
    m.def("kf_smooth", &kf_smooth);
    m.def("kf_smooth_full", &kf_smooth_full);
    m.def("kf_noise_em_stats", &kf_noise_em_stats);
    m.def("kf_noise_em_full_stats", &kf_noise_em_full_stats);
    m.def("kf_adjoint", &kf_adjoint);
    m.def("kf_measure", &kf_measure);
    m.def("kf_class_step", &kf_class_step);
    m.def("kf_resolve_algo", &kf_resolve_algo);
    m.def("fma_peak", &fma_peak);
    m.def("kf_identify_noise", &kf_identify_noise);
    m.def("kf_features", &kf_features);
    m.def("kf_minmax", &kf_minmax);
    m.def("kf_windows", &kf_windows);
    m.def("kf_mpc_forces", &kf_mpc_forces);
    m.def("kf_closed_loop", &kf_closed_loop);
    m.def("kf_closed_loop_workspace_bytes", [](int64_t n, int64_t t) { return (int64_t)optistate_kf_closed_loop_workspace_bytes(n, t); });
    m.def("peer_alloc", &peer_alloc);
    m.def("peer_export", &peer_export);
    m.def("peer_open", &peer_open);
    m.def("peer_close", &peer_close);
    m.def("strerror", [](int rc) { return std::string(optistate_kf_strerror(rc)); });
    m.def("launch_count", []() { return optistate_kf_launch_count(); });
    m.def("abi_version", []() { return optistate_kf_abi_version(); });
    m.def("desc_size", []() { return (int64_t)optistate_kf_desc_size(); });
    m.attr("SUMMARY_ROWS") = (int)OPTI_KF_SUMMARY_ROWS;
    m.attr("MAX_PEERS") = (int)OPTI_KF_MAX_PEERS;
}
