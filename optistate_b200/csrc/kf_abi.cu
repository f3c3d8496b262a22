// extern "C" boundary of liboptistate_kf.so (see include/optistate_kf.h): descriptor validation, conversion of
// the POD descriptor into typed kernel parameters, kernel selection and launch.  No torch types, no allocation,
// no exceptions; every failure is a negative return code.
#include <atomic>
#include <cstdlib>
#include <cstring>
#include <type_traits>

#include "kf_features.cuh"
#include "kf_identify.cuh"
#include "kf_launch.cuh"
#include "kf_mpc_params.cuh"
#include "kf_seq_core.cuh"
#include "kf_smooth.cuh"
#include "kf_smooth_full.cuh"

namespace {

std::atomic<long long> g_launches{0};

bool is_diag_kind(int k) { return k == OPTI_KF_MAT_DIAG || k == OPTI_KF_MAT_DIAG_PER; }
bool valid_kind(int k, bool allow_none) { return (k >= (allow_none ? 0 : 1)) && k <= OPTI_KF_MAT_DENSE_PER; }

int validate(const OptiKfDesc *d) {
    if (!d) return OPTI_KF_E_NULL;
    if (d->struct_size != sizeof(OptiKfDesc) || d->abi_version != OPTISTATE_KF_ABI_VERSION) return OPTI_KF_E_VERSION;
    if (d->dtype != OPTI_KF_F64 && d->dtype != OPTI_KF_F32) return OPTI_KF_E_DTYPE;
    if (d->n_traj < 0 || d->n_steps < 0 || d->n_streams <= 0 || d->ckpt_every < 0) return OPTI_KF_E_SHAPE;
    if (d->phases <= 0 || d->phases > OPTI_KF_PHASE_ALL) return OPTI_KF_E_SHAPE;
    if (d->algo < OPTI_KF_ALGO_AUTO || d->algo > OPTI_KF_ALGO_SEQUENTIAL) return OPTI_KF_E_SHAPE;
    if (d->cov_model != OPTI_KF_COV_PREDICT && d->cov_model != OPTI_KF_COV_MPC) return OPTI_KF_E_SHAPE;
    if (!valid_kind(d->q_kind, false) || !valid_kind(d->r_kind, false) || !valid_kind(d->p0_kind, true)) return OPTI_KF_E_SHAPE;
    if (!(d->dt > 0) || !(d->mass > 0) || !(d->inertia[0] > 0) || !(d->inertia[1] > 0) || !(d->inertia[2] > 0)) return OPTI_KF_E_SHAPE;
    const bool work = d->n_traj > 0, steps = work && d->n_steps > 0;  // empty batches carry empty (NULL) arrays
    if (work && (!d->x0 || !d->Q || !d->R)) return OPTI_KF_E_NULL;
    if (work && d->p0_kind != OPTI_KF_MAT_NONE && !d->P0) return OPTI_KF_E_NULL;
    if (steps && (d->phases & OPTI_KF_PHASE_MEASURE) && (!d->imu || !d->p || !d->dp || !d->contact)) return OPTI_KF_E_NULL;
    if (steps && (d->phases & OPTI_KF_PHASE_PREDICT) && (!d->p || !d->f)) return OPTI_KF_E_NULL;
    if (steps && (d->phases & OPTI_KF_PHASE_UPDATE) && !(d->phases & OPTI_KF_PHASE_MEASURE) && !d->z_in) return OPTI_KF_E_NULL;
    if (steps && d->cov_model == OPTI_KF_COV_MPC && (d->phases & OPTI_KF_PHASE_PREDICT) && !d->body_ref) return OPTI_KF_E_NULL;
    if (d->P_ckpt && d->ckpt_every == 0) return OPTI_KF_E_SHAPE;
    if (d->stream_index == nullptr && d->stream_offset < 0) return OPTI_KF_E_SHAPE;
    if (d->summary_ld < 0 || (d->summary_ld > 0 && d->summary_ld < d->n_traj)) return OPTI_KF_E_SHAPE;
    if (d->n_summary_peers < 0 || d->n_summary_peers > OPTI_KF_MAX_PEERS) return OPTI_KF_E_SHAPE;
    if (d->flags & ~(OPTI_KF_FLAG_P0_DECOUPLED | OPTI_KF_FLAG_FULL_COVARIANCE | OPTI_KF_FLAG_SCALAR_FP32 | OPTI_KF_FLAG_STATUS_ACCUMULATE)) return OPTI_KF_E_SHAPE;
    for (int k = 0; k < d->n_summary_peers; ++k)
        if (d->summary && !d->summary_peers[k]) return OPTI_KF_E_NULL;
    return OPTI_KF_OK;
}

// SEQUENTIAL covers the full recursion with diagonal noise; everything else is JOINT.
bool sequential_ok(const OptiKfDesc *d) {
    return is_diag_kind(d->q_kind) && is_diag_kind(d->r_kind) && d->K_final == nullptr &&
           (d->phases == OPTI_KF_PHASE_ALL || (d->phases == (OPTI_KF_PHASE_PREDICT | OPTI_KF_PHASE_UPDATE) && d->z_in));
}

int resolve(const OptiKfDesc *d) {
    if (d->algo == OPTI_KF_ALGO_JOINT) return OPTI_KF_ALGO_JOINT;
    if (d->algo == OPTI_KF_ALGO_SEQUENTIAL) return sequential_ok(d) ? (int)OPTI_KF_ALGO_SEQUENTIAL : (int)OPTI_KF_E_UNSUPPORTED;
    // AUTO: a dense P0 may be non-symmetric, which only JOINT reproduces; the host asks for SEQUENTIAL explicitly
    // once it has checked symmetry.
    const bool p0_sym = d->p0_kind == OPTI_KF_MAT_NONE || is_diag_kind(d->p0_kind);
    return (sequential_ok(d) && p0_sym) ? OPTI_KF_ALGO_SEQUENTIAL : OPTI_KF_ALGO_JOINT;
}

template <typename Real>
okf::Params<Real> make_params(const OptiKfDesc *d) {
    okf::Params<Real> p;
    std::memset(&p, 0, sizeof p);
    p.N = d->n_traj; p.T = d->n_steps; p.S = d->n_streams; p.stream_offset = d->stream_offset;
    p.phases = d->phases; p.cov_model = d->cov_model;
    // decoupled groups (kf_seq_core.cuh): predict() model with a P0 that has no cross-group entries
    const bool p0_groups = d->p0_kind == OPTI_KF_MAT_NONE || is_diag_kind(d->p0_kind) || (d->flags & OPTI_KF_FLAG_P0_DECOUPLED);
    p.block = (d->cov_model == OPTI_KF_COV_PREDICT && p0_groups && !(d->flags & OPTI_KF_FLAG_FULL_COVARIANCE)) ? 1 : 0;
    p.dt = (Real)d->dt;
    p.dt_over_m = (Real)((1.0 / d->mass) * d->dt);  // B*dt with B = 1/m (force_controller.py:246-247,289)
    p.dt_g = (Real)(d->dt * d->gravity);
    for (int k = 0; k < 3; ++k) p.inv_inertia[k] = (Real)(1.0 / d->inertia[k]);
    p.imu = (const Real *)d->imu; p.p = (const Real *)d->p; p.dp = (const Real *)d->dp;
    p.contact = (const Real *)d->contact; p.f = (const Real *)d->f;
    p.z_in = (d->phases & OPTI_KF_PHASE_MEASURE) ? nullptr : (const Real *)d->z_in;
    p.body_ref = (const Real *)d->body_ref; p.truth = (const Real *)d->truth; p.nominal = (const Real *)d->nominal;
    p.stream_index = d->stream_index;
    p.x0 = (const Real *)d->x0; p.x0_ld = d->x0_per_traj ? d->n_traj : 1; p.x0_inc = d->x0_per_traj ? 1 : 0;
    p.P0 = (const Real *)d->P0; p.p0_kind = d->p0_kind;
    p.Q = (const Real *)d->Q; p.q_kind = d->q_kind;
    p.R = (const Real *)d->R; p.r_kind = d->r_kind;
    p.x_steps = (Real *)d->x_steps; p.x_model_steps = (Real *)d->x_model_steps; p.p_world_steps = (Real *)d->p_world_steps;
    p.z_steps = (Real *)d->z_steps; p.p_trace_steps = (Real *)d->p_trace_steps; p.k_gain_steps = (Real *)d->k_gain_steps;
    p.nis_steps = (Real *)d->nis_steps; p.ckpt_every = d->ckpt_every; p.P_ckpt = (Real *)d->P_ckpt;
    p.x_final = (Real *)d->x_final; p.P_final = (Real *)d->P_final; p.K_final = (Real *)d->K_final;
    p.summary = (Real *)d->summary; p.status = d->status;
    p.summary_ld = d->summary_ld > 0 ? d->summary_ld : d->n_traj;
    p.n_summary_peers = d->summary ? d->n_summary_peers : 0;
    for (int k = 0; k < p.n_summary_peers; ++k) p.summary_peers[k] = (Real *)d->summary_peers[k];
    return p;
}

template <typename Real>
void launch_measure(long long T, long long S, const Real *imu, const Real *p, const Real *dp, const Real *contact, const Real *f, Real *z,
                    Real *mom, Real *odom, uint32_t *status, cudaStream_t stream);

inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// Scratch of the streamed SEQUENTIAL path, each part padded to 256 bytes: z [T][10][S] (PHASE_ALL only), the leg moments of the
// mean model M [T][12][S], and the per-stream status [S] (PHASE_ALL only).  Byte offsets; z starts at 0.
struct SeqWorkspace {
    size_t mom, status, total;
    explicit SeqWorkspace(const OptiKfDesc *d) {
        const auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
        const size_t esz = d->dtype == OPTI_KF_F64 ? 8 : 4, ts = (size_t)d->n_steps * (size_t)d->n_streams;
        const bool all = d->phases == OPTI_KF_PHASE_ALL;
        mom = all ? up(ts * okf::NZ * esz) : 0;
        status = mom + up(ts * okf::NM * esz);
        total = status + (all ? up((size_t)d->n_streams * sizeof(uint32_t)) : 0);
    }
};

// The streamed kernel needs every warp (32 consecutive trajectories) to read one aligned tile of 32 consecutive
// streams, 16-byte aligned arrays and row counts that fit the 32-bit tensor-map coordinates.
bool tma_layout_ok(const OptiKfDesc *d) {
    if (d->stream_index != nullptr || d->n_steps == 0) return false;
    if (d->n_streams % 32 != 0 || d->stream_offset % 32 != 0) return false;
    if (d->n_steps * 12 >= (1LL << 31)) return false;
    if (!aligned16(d->p) || !aligned16(d->f)) return false;
    if (d->summary && ((d->truth && !aligned16(d->truth)) || (d->nominal && !aligned16(d->nominal)))) return false;
    if (d->cov_model == OPTI_KF_COV_MPC && !aligned16(d->body_ref)) return false;
    return true;
}

inline bool aligned8(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 7u) == 0; }

// FP32 only: two trajectories per thread on the packed FFMA2 path need even counts, 64-stream tiles and 8-byte
// aligned per-trajectory arrays (every [C][N] row then starts on a float2 boundary).  Measured on B200 (1.2 M
// trajectories x 200 steps): packed 1.57e10 vs one-trajectory 1.37e10 steps/s without the summary, 1.31e10 vs 1.07e10
// with it.  OPTI_KF_FLAG_SCALAR_FP32 asks for the one-trajectory kernel (the tests compare the two).
bool packed_pair_ok(const OptiKfDesc *d) {
    if (d->dtype != OPTI_KF_F32) return false;
    if (d->flags & OPTI_KF_FLAG_SCALAR_FP32) return false;
    if (d->n_traj % 2 != 0 || d->n_streams % 64 != 0 || d->stream_offset % 64 != 0) return false;
    const void *ptrs[] = {d->x0, d->P0, d->Q, d->R, d->x_steps, d->x_model_steps, d->p_world_steps, d->z_steps, d->p_trace_steps,
                          d->k_gain_steps, d->nis_steps, d->P_ckpt, d->x_final, d->P_final, d->summary};
    for (const void *q : ptrs)
        if (q && !aligned8(q)) return false;
    if (d->summary && d->summary_ld % 2 != 0) return false;  // pairs of summary values are stored as one float2
    for (int k = 0; k < d->n_summary_peers; ++k)
        if (d->summary && !aligned8(d->summary_peers[k])) return false;
    return true;
}

template <typename Real>
int launch_streamed_t(const OptiKfDesc *d, const okf::Params<typename okf::Lanes<Real>::scalar> &p, cudaStream_t stream) {
    if constexpr (okf::Lanes<Real>::n == 1) {
        // no more trajectories than streams: every block would hold one working warp - the one-warp-per-block latency variant
        if (p.block && p.N <= p.S && p.cov_model == OPTI_KF_COV_PREDICT)
            return d->summary ? okf::launch_seq_tma_lone<Real, true>(p, stream) : okf::launch_seq_tma_lone<Real, false>(p, stream);
    }
    if (p.block) return d->summary ? okf::launch_seq_tma<Real, true, true>(p, stream) : okf::launch_seq_tma<Real, false, true>(p, stream);
    return d->summary ? okf::launch_seq_tma<Real, true, false>(p, stream) : okf::launch_seq_tma<Real, false, false>(p, stream);
}
template <typename Scalar>
int launch_streamed(const OptiKfDesc *d, const okf::Params<Scalar> &p, cudaStream_t stream);
template <>
int launch_streamed<double>(const OptiKfDesc *d, const okf::Params<double> &p, cudaStream_t stream) {
    return launch_streamed_t<double>(d, p, stream);
}
template <>
int launch_streamed<float>(const OptiKfDesc *d, const okf::Params<float> &p, cudaStream_t stream) {
    return packed_pair_ok(d) ? launch_streamed_t<okf::F2>(d, p, stream) : launch_streamed_t<float>(d, p, stream);
}

// P_steps: the smoothers' per-step posterior covariance, [T][30][N] from the decoupled kernels (optistate_kf_smooth) or [T][78][N]
// from the full ones (optistate_kf_smooth_full)
template <typename Real>
int launch(const OptiKfDesc *d, int algo, cudaStream_t stream, void *P_steps = nullptr) {
    if (d->n_traj == 0) return OPTI_KF_OK;
    okf::Params<Real> p = make_params<Real>(d);
    p.P_steps = (Real *)P_steps;
    cudaGetLastError();
    if ((d->flags & OPTI_KF_FLAG_STATUS_ACCUMULATE) && d->status) {
        // the kernels OR stream_status[stream of i] into what they write: with one stream per trajectory that is the old status
        if (d->stream_index != nullptr || d->n_streams != d->n_traj || d->stream_offset != 0 || d->phases == OPTI_KF_PHASE_ALL) return OPTI_KF_E_UNSUPPORTED;
        p.stream_status = d->status;
    }
    if (algo == OPTI_KF_ALGO_SEQUENTIAL) {
        bool streamed = tma_layout_ok(d) && (d->phases == OPTI_KF_PHASE_ALL || aligned16(p.z_in));
        if (streamed) {
            // hoist the state-independent work into a pre-pass over the S base streams: the leg moments of the mean model
            // and, unless the caller supplies z, the measurements
            const SeqWorkspace ws(d);
            if (d->workspace && d->workspace_bytes >= ws.total && aligned16(d->workspace)) {
                unsigned char *base = (unsigned char *)d->workspace;
                Real *z = nullptr;
                uint32_t *sst = nullptr;
                if (d->phases == OPTI_KF_PHASE_ALL) {
                    z = (Real *)base;
                    sst = (uint32_t *)(base + ws.status);
                    if (cudaMemsetAsync(sst, 0, (size_t)d->n_streams * sizeof(uint32_t), stream) != cudaSuccess) return OPTI_KF_E_CUDA;
                    p.z_in = z;
                    p.stream_status = sst;
                }
                p.mom = (Real *)(base + ws.mom);
                launch_measure<Real>(d->n_steps, d->n_streams, p.imu, p.p, p.dp, p.contact, p.f, z, (Real *)p.mom, nullptr, sst, stream);
            } else {
                streamed = false;
            }
        }
        if (streamed) {
            const int rc = launch_streamed<Real>(d, p, stream);
            if (rc < 0) return rc;
            if (rc == OPTI_KF_OK) {
                g_launches.fetch_add(1, std::memory_order_relaxed);
                return cudaGetLastError() == cudaSuccess ? OPTI_KF_OK : OPTI_KF_E_CUDA;
            }
            // tensor maps unavailable: the direct-load kernel below consumes the same (pre-formed) z
        }
        const int rc = okf::launch_seq_direct<Real>(p, stream);
        if (rc < 0) return rc;
    } else {
        const int rc = okf::launch_joint<Real>(p, stream);
        if (rc < 0) return rc;
    }
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError() == cudaSuccess ? OPTI_KF_OK : OPTI_KF_E_CUDA;
}

// ---- batched get_odom + set_measurements, and the leg moments of the mean model (leg_moments, kf_seq_core.cuh) ----------
// z / odom / status: the measurement (imu, dp and contact are read only then); mom: the moments of p and f
template <typename Real>
__global__ void __launch_bounds__(256) kf_measure_kernel(long long T, long long S, const Real *__restrict__ imu,
                                                         const Real *__restrict__ p, const Real *__restrict__ dp,
                                                         const Real *__restrict__ contact, const Real *__restrict__ f,
                                                         Real *__restrict__ z, Real *__restrict__ mom,
                                                         Real *__restrict__ odom, uint32_t *__restrict__ status) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // (t, s) flattened, s fastest
    if (idx >= T * S) return;
    const long long t = idx / S, s = idx % S;
    Real pp[12];
#pragma unroll
    for (int c = 0; c < 12; ++c) pp[c] = p[(t * 12 + c) * S + s];
    if (z || odom || status) {
        Real im[6], dd[12], cc[4], zz[okf::NZ];
#pragma unroll
        for (int c = 0; c < 6; ++c) im[c] = imu[(t * 6 + c) * S + s];
#pragma unroll
        for (int c = 0; c < 12; ++c) dd[c] = dp[(t * 12 + c) * S + s];
#pragma unroll
        for (int c = 0; c < 4; ++c) cc[c] = contact[(t * 4 + c) * S + s];
        const bool all_swing = okf::form_measurement(im, pp, dd, cc, zz);
        if (z) {
#pragma unroll
            for (int c = 0; c < okf::NZ; ++c) z[(t * okf::NZ + c) * S + s] = zz[c];
        }
        if (odom) {
            odom[(t * 4 + 0) * S + s] = zz[3];
            odom[(t * 4 + 1) * S + s] = zz[7];
            odom[(t * 4 + 2) * S + s] = zz[8];
            odom[(t * 4 + 3) * S + s] = zz[9];
        }
        if (status && all_swing) atomicOr(status + s, (uint32_t)OPTI_KF_ST_ALL_SWING);
    }
    if (mom) {
        Real ff[12], M[okf::NM];
#pragma unroll
        for (int c = 0; c < 12; ++c) ff[c] = f[(t * 12 + c) * S + s];
        okf::leg_moments(pp, ff, M);
#pragma unroll
        for (int c = 0; c < okf::NM; ++c) mom[(t * okf::NM + c) * S + s] = M[c];
    }
}

template <typename Real>
void launch_measure(long long T, long long S, const Real *imu, const Real *p, const Real *dp, const Real *contact, const Real *f, Real *z,
                    Real *mom, Real *odom, uint32_t *status, cudaStream_t stream) {
    const long long total = T * S;
    if (total == 0) return;
    kf_measure_kernel<Real><<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(T, S, imu, p, dp, contact, f, z, mom, odom, status);
    g_launches.fetch_add(1, std::memory_order_relaxed);
}

// ---- FMA issue-peak micro-benchmark ----------------------------------------------------------------------------
template <typename Real>
__global__ void __launch_bounds__(256) fma_peak_kernel(long long iters, Real seed, Real *sink) {
    Real a[16];
    const Real m = Real(0.999) + seed * Real(1e-9), c = Real(1e-3) * (Real)(threadIdx.x & 7);
#pragma unroll
    for (int k = 0; k < 16; ++k) a[k] = seed + (Real)k;
    for (long long it = 0; it < iters; ++it) {
#pragma unroll
        for (int k = 0; k < 16; ++k) a[k] = a[k] * m + c;
    }
    Real s = Real(0);
#pragma unroll
    for (int k = 0; k < 16; ++k) s += a[k];
    if (s == Real(-12345.678)) sink[blockIdx.x * blockDim.x + threadIdx.x] = s;  // never true; keeps the chain alive
}

template <typename Real>
int fma_peak(long long fma_per_thread, double *flops_out, double *seconds_out, cudaStream_t stream) {
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return OPTI_KF_E_NO_DEVICE;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int blocks = sms * 8, threads = 256;
    const long long iters = (fma_per_thread + 15) / 16;
    cudaEvent_t e0, e1;
    if (cudaEventCreate(&e0) != cudaSuccess || cudaEventCreate(&e1) != cudaSuccess) return OPTI_KF_E_CUDA;
    fma_peak_kernel<Real><<<blocks, threads, 0, stream>>>(iters / 8 + 1, Real(1), nullptr);  // warm-up
    cudaEventRecord(e0, stream);
    fma_peak_kernel<Real><<<blocks, threads, 0, stream>>>(iters, Real(1), nullptr);
    cudaEventRecord(e1, stream);
    g_launches.fetch_add(2, std::memory_order_relaxed);
    if (cudaEventSynchronize(e1) != cudaSuccess) { cudaEventDestroy(e0); cudaEventDestroy(e1); return OPTI_KF_E_CUDA; }
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    const double fma = (double)iters * 16.0 * (double)blocks * (double)threads;
    if (flops_out) *flops_out = 2.0 * fma / ((double)ms * 1e-3);
    if (seconds_out) *seconds_out = (double)ms * 1e-3;
    return OPTI_KF_OK;
}

// ---- the backward passes over the SEQUENTIAL filter: smoother and EM E-step ------------------------------------------
// full: the full-covariance kernel (all 78 entries of P+, SmoothFullParams, kf_rts_full_kernel) instead of the decoupled one
// (30 packed entries, SmoothParams, kf_rts_kernel); stats: the E-step of EM, which accepts exactly what its smoother accepts.
struct Backward {
    bool full, stats;
};

// What the backward kernels can take.  Decoupled: the decoupled-group form of the SEQUENTIAL filter (kf_smooth.cuh).  Full:
// whatever the SEQUENTIAL filter runs (AUTO means SEQUENTIAL here, as the symmetric P0 this entry requires permits), in either
// covariance model and with any P0 kind.
int backward_check(const OptiKfDesc *d, bool full) {
    const int rc = validate(d);
    if (rc != OPTI_KF_OK) return rc;
    if (full) return d->algo != OPTI_KF_ALGO_JOINT && sequential_ok(d) ? OPTI_KF_OK : OPTI_KF_E_UNSUPPORTED;
    if (d->cov_model != OPTI_KF_COV_PREDICT || (d->flags & OPTI_KF_FLAG_FULL_COVARIANCE)) return OPTI_KF_E_UNSUPPORTED;
    if (!is_diag_kind(d->q_kind) || !is_diag_kind(d->r_kind)) return OPTI_KF_E_UNSUPPORTED;
    const bool p0_groups = d->p0_kind == OPTI_KF_MAT_NONE || is_diag_kind(d->p0_kind) || (d->flags & OPTI_KF_FLAG_P0_DECOUPLED);
    if (!p0_groups) return OPTI_KF_E_UNSUPPORTED;
    const int algo = resolve(d);
    if (algo < 0) return algo;
    return algo == OPTI_KF_ALGO_SEQUENTIAL ? OPTI_KF_OK : OPTI_KF_E_UNSUPPORTED;
}

// Scratch of the backward passes, each part padded to 256 bytes: P+ [T][np][N] at 0 (np = 30 packed decoupled entries, or all
// 78 when full), then x+ and x- [T][12][N] unless the filter descriptor has x_steps / x_model_steps (the backward kernel reads
// those), then for the E-step z [T][10][S] when the filter forms the measurements.  Byte offsets.
struct BackwardStorage {
    size_t x_post, x_prior, z, total;
    BackwardStorage(const OptiKfDesc *d, Backward v) {
        const auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
        const size_t esz = d->dtype == OPTI_KF_F64 ? 8 : 4, tn = (size_t)d->n_steps * (size_t)d->n_traj;
        const size_t ts = (size_t)d->n_steps * (size_t)d->n_streams;
        x_post = up(tn * (size_t)(v.full ? okf::NP : okf::NPB) * esz);
        x_prior = x_post + (d->x_steps ? 0 : up(tn * okf::NX * esz));
        z = x_prior + (d->x_model_steps ? 0 : up(tn * okf::NX * esz));
        total = z + (v.stats && (d->phases & OPTI_KF_PHASE_MEASURE) ? up(ts * okf::NZ * esz) : 0);
    }
};

// The forward pass, with x+ / x- in the storage where the caller did not ask for them, then the backward kernel.  A full pass runs
// the full-covariance filter kernels whatever the caller's flags, so P+ is [T][78][N] (on decoupled inputs they are bit-identical
// to the kBlock ones, kf_seq_core.cuh).
template <typename Real>
int run_backward(Backward v, const OptiKfDesc *f, void *storage, void *x_smooth, void *var_smooth, void *stats, cudaStream_t stream) {
    const BackwardStorage st(f, v);
    unsigned char *base = (unsigned char *)storage;
    OptiKfDesc fw = *f;
    if (v.full) fw.flags |= OPTI_KF_FLAG_FULL_COVARIANCE;
    if (!fw.x_steps && base) fw.x_steps = base + st.x_post;
    if (!fw.x_model_steps && base) fw.x_model_steps = base + st.x_prior;
    int rc = launch<Real>(&fw, OPTI_KF_ALGO_SEQUENTIAL, stream, base);
    if (rc != OPTI_KF_OK) return rc;
    const long long N = f->n_traj, T = f->n_steps;
    if (N == 0 || (T == 0 && !v.stats)) return OPTI_KF_OK;
    if (T == 0)  // no transition and no measurement: every sum is empty
        return cudaMemsetAsync(stats, 0, (size_t)okf::EM_STATS_ROWS * N * sizeof(Real), stream) == cudaSuccess ? OPTI_KF_OK : OPTI_KF_E_CUDA;
    const Real *z = (const Real *)f->z_in;
    if (v.stats && (f->phases & OPTI_KF_PHASE_MEASURE)) {  // the filter formed z in-kernel: form it once more, per stream, with the same function
        z = (const Real *)(base + st.z);
        launch_measure<Real>(T, f->n_streams, (const Real *)f->imu, (const Real *)f->p, (const Real *)f->dp, (const Real *)f->contact,
                             nullptr, (Real *)z, nullptr, nullptr, nullptr, stream);
    }
    const auto fill = [&](auto &p) {  // the fields SmoothParams and SmoothFullParams share; the E-step's stay zero for the smoother
        std::memset(&p, 0, sizeof p);
        p.N = N; p.T = T; p.dt = (Real)f->dt;
        p.Q = (const Real *)f->Q; p.q_kind = f->q_kind;
        p.x_post = (const Real *)fw.x_steps; p.x_prior = (const Real *)fw.x_model_steps; p.P_post = (const Real *)base;
        p.x_smooth = (Real *)x_smooth; p.var_smooth = (Real *)var_smooth; p.status = f->status;
        if (v.full || v.stats) {  // the stream a trajectory reads z (E-step) and body_ref (full) from
            p.S = f->n_streams; p.stream_offset = f->stream_offset; p.stream_index = f->stream_index;
        }
        if (v.stats) {
            p.z = z;
            p.R = (const Real *)f->R; p.r_kind = f->r_kind;
            p.x0 = (const Real *)f->x0; p.x0_ld = f->x0_per_traj ? N : 1; p.x0_inc = f->x0_per_traj ? 1 : 0;
            p.P0 = (const Real *)f->P0; p.p0_kind = f->p0_kind;
            p.stats = (Real *)stats;
        }
    };
    if (v.full) {
        okf::SmoothFullParams<Real> p;
        fill(p);
        p.cov_model = f->cov_model; p.body_ref = (const Real *)f->body_ref;
        rc = v.stats ? okf::launch_rts_full<Real, true>(p, stream) : okf::launch_rts_full<Real, false>(p, stream);
    } else {
        okf::SmoothParams<Real> p;
        fill(p);
        rc = v.stats ? okf::launch_rts<Real, true>(p, stream) : okf::launch_rts<Real, false>(p, stream);
    }
    if (rc < 0) return rc;
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError() == cudaSuccess ? OPTI_KF_OK : OPTI_KF_E_CUDA;
}

int backward_storage_bytes(const OptiKfDesc *filter, Backward v, size_t *bytes_out) {
    const int rc = backward_check(filter, v.full);
    if (rc != OPTI_KF_OK) return rc;
    if (!bytes_out) return OPTI_KF_E_NULL;
    *bytes_out = BackwardStorage(filter, v).total;
    return OPTI_KF_OK;
}

// The entries' envelope, codes in the order the header documents: the descriptor, the filter, the required output (the smoother's
// x_smooth, the E-step's stats), then the storage.
template <typename Desc>
int backward_entry(const Desc *desc, bool full, void *cuda_stream) {
    constexpr bool stats = std::is_same<Desc, OptiKfNoiseEmDesc>::value;
    if (!desc) return OPTI_KF_E_NULL;
    if (desc->struct_size != sizeof(Desc) || desc->abi_version != OPTISTATE_KF_ABI_VERSION) return OPTI_KF_E_VERSION;
    if (!desc->filter) return OPTI_KF_E_NULL;
    const OptiKfDesc *f = desc->filter;
    const int rc = backward_check(f, full);
    if (rc != OPTI_KF_OK) return rc;
    const bool steps = f->n_traj > 0 && f->n_steps > 0;  // empty batches carry empty (NULL) arrays
    void *out_stats = nullptr;
    if constexpr (stats) {
        out_stats = desc->stats;
        if (f->n_traj > 0 && !out_stats) return OPTI_KF_E_NULL;
    } else {
        if (steps && !desc->x_smooth) return OPTI_KF_E_NULL;
    }
    const Backward v{full, stats};
    if (desc->storage_bytes < BackwardStorage(f, v).total) return OPTI_KF_E_SHAPE;
    if (steps && !desc->storage) return OPTI_KF_E_NULL;
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    return f->dtype == OPTI_KF_F64 ? run_backward<double>(v, f, desc->storage, desc->x_smooth, desc->var_smooth, out_stats, stream)
                                   : run_backward<float>(v, f, desc->storage, desc->x_smooth, desc->var_smooth, out_stats, stream);
}

template <typename Real>
int identify_noise(const OptiKfIdentifyDesc *d, cudaStream_t stream) {
    okf::Params<Real> p;
    std::memset(&p, 0, sizeof p);
    p.N = d->n_traj; p.T = d->n_steps; p.S = d->n_streams; p.stream_offset = d->stream_offset; p.stream_index = d->stream_index;
    p.dt = (Real)d->dt;
    p.dt_over_m = (Real)((1.0 / d->mass) * d->dt);
    p.dt_g = (Real)(d->dt * d->gravity);
    for (int k = 0; k < 3; ++k) p.inv_inertia[k] = (Real)(1.0 / d->inertia[k]);
    p.imu = (const Real *)d->imu; p.p = (const Real *)d->p; p.dp = (const Real *)d->dp;
    p.contact = (const Real *)d->contact; p.f = (const Real *)d->f; p.status = d->status;
    const long long pairs = (d->n_steps - 1) * d->n_traj;
    okf::kf_identify_residuals_kernel<Real><<<(unsigned)((pairs + 127) / 128), 128, 0, stream>>>(p, (const Real *)d->gt, d->alias_last_measurement,
                                                                                                  (Real *)d->scratch);
    const long long comps = (long long)okf::IDENT_ROWS * d->n_traj;
    okf::kf_identify_variance_kernel<Real><<<(unsigned)((comps + 127) / 128), 128, 0, stream>>>(d->n_traj, d->n_steps - 1, (const Real *)d->scratch,
                                                                                                 (Real *)d->q_diag, (Real *)d->r_diag);
    g_launches.fetch_add(2, std::memory_order_relaxed);
    return cudaGetLastError() == cudaSuccess ? OPTI_KF_OK : OPTI_KF_E_CUDA;
}

}  // namespace

extern "C" {

int optistate_kf_abi_version(void) { return OPTISTATE_KF_ABI_VERSION; }
size_t optistate_kf_desc_size(void) { return sizeof(OptiKfDesc); }
int64_t optistate_kf_launch_count(void) { return (int64_t)g_launches.load(std::memory_order_relaxed); }

int optistate_kf_resolve_algo(const OptiKfDesc *desc) {
    const int rc = validate(desc);
    return rc != OPTI_KF_OK ? rc : resolve(desc);
}

int optistate_kf_workspace_bytes(const OptiKfDesc *desc, size_t *bytes_out) {
    const int rc = validate(desc);
    if (rc != OPTI_KF_OK) return rc;
    if (!bytes_out) return OPTI_KF_E_NULL;
    const int algo = resolve(desc);
    if (algo < 0) return algo;
    *bytes_out = (algo == OPTI_KF_ALGO_SEQUENTIAL && tma_layout_ok(desc)) ? SeqWorkspace(desc).total : 0;
    return OPTI_KF_OK;
}

int optistate_kf_smooth_storage_bytes(const OptiKfDesc *filter, size_t *bytes_out) {
    return backward_storage_bytes(filter, {false, false}, bytes_out);
}
int optistate_kf_smooth(const OptiKfSmoothDesc *desc, void *cuda_stream) { return backward_entry(desc, false, cuda_stream); }

int optistate_kf_smooth_full_storage_bytes(const OptiKfDesc *filter, size_t *bytes_out) {
    return backward_storage_bytes(filter, {true, false}, bytes_out);
}
int optistate_kf_smooth_full(const OptiKfSmoothDesc *desc, void *cuda_stream) { return backward_entry(desc, true, cuda_stream); }

int optistate_kf_noise_em_storage_bytes(const OptiKfDesc *filter, size_t *bytes_out) {
    return backward_storage_bytes(filter, {false, true}, bytes_out);
}
int optistate_kf_noise_em_stats(const OptiKfNoiseEmDesc *desc, void *cuda_stream) { return backward_entry(desc, false, cuda_stream); }

int optistate_kf_noise_em_full_storage_bytes(const OptiKfDesc *filter, size_t *bytes_out) {
    return backward_storage_bytes(filter, {true, true}, bytes_out);
}
int optistate_kf_noise_em_full_stats(const OptiKfNoiseEmDesc *desc, void *cuda_stream) { return backward_entry(desc, true, cuda_stream); }

int optistate_kf_batch(const OptiKfDesc *desc, void *cuda_stream) {
    const int rc = validate(desc);
    if (rc != OPTI_KF_OK) return rc;
    const int algo = resolve(desc);
    if (algo < 0) return algo;
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    return desc->dtype == OPTI_KF_F64 ? launch<double>(desc, algo, stream) : launch<float>(desc, algo, stream);
}

int optistate_kf_batch_f64(const OptiKfDesc *desc, void *cuda_stream) {
    if (desc && desc->dtype != OPTI_KF_F64) return OPTI_KF_E_DTYPE;
    return optistate_kf_batch(desc, cuda_stream);
}

int optistate_kf_batch_f32(const OptiKfDesc *desc, void *cuda_stream) {
    if (desc && desc->dtype != OPTI_KF_F32) return OPTI_KF_E_DTYPE;
    return optistate_kf_batch(desc, cuda_stream);
}

int optistate_kf_measure(const OptiKfMeasureDesc *d, void *cuda_stream) {
    if (!d) return OPTI_KF_E_NULL;
    if (d->struct_size != sizeof(OptiKfMeasureDesc) || d->abi_version != OPTISTATE_KF_ABI_VERSION) return OPTI_KF_E_VERSION;
    if (d->dtype != OPTI_KF_F64 && d->dtype != OPTI_KF_F32) return OPTI_KF_E_DTYPE;
    if (d->n_steps < 0 || d->n_streams <= 0) return OPTI_KF_E_SHAPE;
    if (!d->imu || !d->p || !d->dp || !d->contact || (!d->z && !d->odom)) return OPTI_KF_E_NULL;
    const long long total = d->n_steps * d->n_streams;
    if (total == 0) return OPTI_KF_OK;
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    cudaGetLastError();
    if (d->dtype == OPTI_KF_F64)
        launch_measure<double>(d->n_steps, d->n_streams, (const double *)d->imu, (const double *)d->p, (const double *)d->dp,
                               (const double *)d->contact, nullptr, (double *)d->z, nullptr, (double *)d->odom, d->status, stream);
    else
        launch_measure<float>(d->n_steps, d->n_streams, (const float *)d->imu, (const float *)d->p, (const float *)d->dp,
                              (const float *)d->contact, nullptr, (float *)d->z, nullptr, (float *)d->odom, d->status, stream);
    return cudaGetLastError() == cudaSuccess ? OPTI_KF_OK : OPTI_KF_E_CUDA;
}

int optistate_fma_peak(int dtype, int64_t fma_per_thread, double *flops_per_s_out, double *seconds_out, void *cuda_stream) {
    if (fma_per_thread <= 0) return OPTI_KF_E_SHAPE;
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    if (dtype == OPTI_KF_F64) return fma_peak<double>(fma_per_thread, flops_per_s_out, seconds_out, stream);
    if (dtype == OPTI_KF_F32) return fma_peak<float>(fma_per_thread, flops_per_s_out, seconds_out, stream);
    return OPTI_KF_E_DTYPE;
}

int optistate_kf_features(const OptiKfFeatureDesc *d, void *cuda_stream) {
    if (!d) return OPTI_KF_E_NULL;
    if (d->struct_size != sizeof(OptiKfFeatureDesc) || d->abi_version != OPTISTATE_KF_ABI_VERSION) return OPTI_KF_E_VERSION;
    if (d->dtype != OPTI_KF_F64 && d->dtype != OPTI_KF_F32) return OPTI_KF_E_DTYPE;
    if (d->n_traj < 0 || d->n_steps < 0 || d->n_streams <= 0) return OPTI_KF_E_SHAPE;
    if ((d->n_steps + okf::FEAT_STEPS - 1) / okf::FEAT_STEPS > 65535) return OPTI_KF_E_SHAPE;  // grid.y
    if (d->stream_index == nullptr && d->stream_offset < 0) return OPTI_KF_E_SHAPE;
    if (!d->x_steps || !d->p_world_steps || !d->imu || !d->f || !d->dp || !d->rows) return OPTI_KF_E_NULL;
    if (d->n_traj == 0 || d->n_steps == 0) return OPTI_KF_OK;
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    const dim3 grid((unsigned)((d->n_traj + okf::FEAT_TRAJ - 1) / okf::FEAT_TRAJ), (unsigned)((d->n_steps + okf::FEAT_STEPS - 1) / okf::FEAT_STEPS));
    cudaGetLastError();
    if (d->dtype == OPTI_KF_F64)
        okf::kf_features_kernel<double><<<grid, 256, 0, stream>>>(d->n_traj, d->n_steps, d->n_streams, d->stream_offset, d->stream_index,
                                                                  (const double *)d->x_steps, (const double *)d->p_world_steps,
                                                                  (const double *)d->imu, (const double *)d->imu_acc, (const double *)d->f,
                                                                  (const double *)d->dp, (double *)d->rows);
    else
        okf::kf_features_kernel<float><<<grid, 256, 0, stream>>>(d->n_traj, d->n_steps, d->n_streams, d->stream_offset, d->stream_index,
                                                                 (const float *)d->x_steps, (const float *)d->p_world_steps,
                                                                 (const float *)d->imu, (const float *)d->imu_acc, (const float *)d->f,
                                                                 (const float *)d->dp, (float *)d->rows);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError() == cudaSuccess ? OPTI_KF_OK : OPTI_KF_E_CUDA;
}

static const int kMinmaxBlocks = 592;  // upper bound (sizes the scratch buffer); the launch takes 4 blocks per SM of the current device
// multiprocessors of the current device (launch geometry is derived from it, not from the B200's 148)
static int sm_count() {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    return n;
}

size_t optistate_kf_minmax_scratch_bytes(int dtype, int32_t n_cols) {
    return (size_t)kMinmaxBlocks * 2 * (size_t)(n_cols > 0 ? n_cols : 0) * (dtype == OPTI_KF_F64 ? 8 : 4);
}

int optistate_kf_minmax(int dtype, const void *rows, int64_t n_rows, int32_t n_cols, void *min_out, void *max_out, void *scratch,
                        size_t scratch_bytes, void *cuda_stream) {
    if (dtype != OPTI_KF_F64 && dtype != OPTI_KF_F32) return OPTI_KF_E_DTYPE;
    if (!rows || !min_out || !max_out || !scratch) return OPTI_KF_E_NULL;
    if (n_rows <= 0 || n_cols <= 0 || n_cols > 256 || scratch_bytes < optistate_kf_minmax_scratch_bytes(dtype, n_cols)) return OPTI_KF_E_SHAPE;
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    cudaGetLastError();
    const int nblk = 4 * sm_count() < kMinmaxBlocks ? 4 * sm_count() : kMinmaxBlocks;
    if (dtype == OPTI_KF_F64) {
        okf::kf_minmax_partial_kernel<double><<<nblk, 256, 2 * 256 * sizeof(double), stream>>>((const double *)rows, n_rows, n_cols, (double *)scratch);
        okf::kf_minmax_final_kernel<double><<<1, 256, 0, stream>>>((const double *)scratch, nblk, n_cols, (double *)min_out, (double *)max_out);
    } else {
        okf::kf_minmax_partial_kernel<float><<<nblk, 256, 2 * 256 * sizeof(float), stream>>>((const float *)rows, n_rows, n_cols, (float *)scratch);
        okf::kf_minmax_final_kernel<float><<<1, 256, 0, stream>>>((const float *)scratch, nblk, n_cols, (float *)min_out, (float *)max_out);
    }
    g_launches.fetch_add(2, std::memory_order_relaxed);
    return cudaGetLastError() == cudaSuccess ? OPTI_KF_OK : OPTI_KF_E_CUDA;
}

size_t optistate_kf_windows_scratch_bytes(int64_t n_groups, int64_t rows_per_group, int32_t n_cols, int32_t n_latent) {
    if (n_groups <= 0 || rows_per_group <= 0 || n_cols <= 0 || n_latent < 0) return 0;
    return (size_t)n_groups * (size_t)rows_per_group * (size_t)(n_cols + n_latent) * sizeof(float);
}

int optistate_kf_windows(int dtype, const void *rows, const float *latent, const void *mn, const void *mx, int64_t n_groups,
                         int64_t rows_per_group, int32_t n_cols, int32_t n_latent, int32_t seq_len, float *out, void *scratch,
                         size_t scratch_bytes, void *cuda_stream) {
    if (dtype != OPTI_KF_F64 && dtype != OPTI_KF_F32) return OPTI_KF_E_DTYPE;
    if (!rows || !mn || !mx || !out || !scratch || (n_latent > 0 && !latent)) return OPTI_KF_E_NULL;
    if (n_groups <= 0 || seq_len <= 0 || rows_per_group < seq_len || n_cols <= 0 || n_latent < 0) return OPTI_KF_E_SHAPE;
    if (scratch_bytes < optistate_kf_windows_scratch_bytes(n_groups, rows_per_group, n_cols, n_latent)) return OPTI_KF_E_SHAPE;
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    const long long n_rows = n_groups * rows_per_group;
    const int width = n_cols + n_latent;
    float *full = (float *)scratch;
    cudaGetLastError();
    const unsigned nb = (unsigned)sm_count() * 16;
    if (dtype == OPTI_KF_F64)
        okf::kf_normalise_rows_kernel<double><<<nb, 256, 0, stream>>>((const double *)rows, latent, (const double *)mn, (const double *)mx,
                                                                      n_rows, n_cols, n_latent, full);
    else
        okf::kf_normalise_rows_kernel<float><<<nb, 256, 0, stream>>>((const float *)rows, latent, (const float *)mn, (const float *)mx, n_rows,
                                                                     n_cols, n_latent, full);
    const bool vec4 = (width % 4 == 0) && ((reinterpret_cast<uintptr_t>(full) | reinterpret_cast<uintptr_t>(out)) & 15u) == 0;
    if (vec4)
        okf::kf_windows_copy_kernel<float4><<<nb, dim3(64, 4), 0, stream>>>((const float4 *)full, rows_per_group, n_groups, width / 4, seq_len, (float4 *)out);
    else
        okf::kf_windows_copy_kernel<float><<<nb, dim3(64, 4), 0, stream>>>(full, rows_per_group, n_groups, width, seq_len, out);
    g_launches.fetch_add(2, std::memory_order_relaxed);
    return cudaGetLastError() == cudaSuccess ? OPTI_KF_OK : OPTI_KF_E_CUDA;
}

size_t optistate_kf_identify_scratch_bytes(int dtype, int64_t n_traj, int64_t n_steps) {
    if (n_traj <= 0 || n_steps < 2) return 0;
    return (size_t)(n_steps - 1) * okf::IDENT_ROWS * (size_t)n_traj * (dtype == OPTI_KF_F64 ? 8 : 4);
}

int optistate_kf_identify_noise(const OptiKfIdentifyDesc *d, void *cuda_stream) {
    if (!d) return OPTI_KF_E_NULL;
    if (d->struct_size != sizeof(OptiKfIdentifyDesc) || d->abi_version != OPTISTATE_KF_ABI_VERSION) return OPTI_KF_E_VERSION;
    if (d->dtype != OPTI_KF_F64 && d->dtype != OPTI_KF_F32) return OPTI_KF_E_DTYPE;
    if (d->n_traj <= 0 || d->n_steps < 2 || d->n_streams <= 0) return OPTI_KF_E_SHAPE;
    if (d->stream_index == nullptr && d->stream_offset < 0) return OPTI_KF_E_SHAPE;
    if (!(d->dt > 0) || !(d->mass > 0) || !(d->inertia[0] > 0) || !(d->inertia[1] > 0) || !(d->inertia[2] > 0)) return OPTI_KF_E_SHAPE;
    if (!d->gt || !d->imu || !d->p || !d->dp || !d->contact || !d->f || !d->q_diag || !d->r_diag || !d->scratch) return OPTI_KF_E_NULL;
    if (d->scratch_bytes < optistate_kf_identify_scratch_bytes(d->dtype, d->n_traj, d->n_steps)) return OPTI_KF_E_SHAPE;
    cudaGetLastError();
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    return d->dtype == OPTI_KF_F64 ? identify_noise<double>(d, stream) : identify_noise<float>(d, stream);
}

int optistate_kf_mpc_forces(const OptiKfMpcDesc *d, void *cuda_stream) {
    if (!d) return OPTI_KF_E_NULL;
    if (d->struct_size != sizeof(OptiKfMpcDesc) || d->abi_version != OPTISTATE_KF_ABI_VERSION) return OPTI_KF_E_VERSION;
    if (d->dtype != OPTI_KF_F64) return OPTI_KF_E_DTYPE;  // cond(H) ~ 1e5: the QP is solved in double only
    if (d->n_problems < 0 || d->max_free_legs < 0 || d->max_free_legs > 4) return OPTI_KF_E_SHAPE;
    if (!(d->dt > 0) || !(d->mass > 0) || !(d->inertia[0] > 0) || !(d->inertia[1] > 0) || !(d->inertia[2] > 0) || !(d->mu > 0) ||
        !(d->fz_max > 0) || !(d->w_force > 0))
        return OPTI_KF_E_SHAPE;
    for (int k = 0; k < 12; ++k)
        if (!(d->w_state[k] >= 0)) return OPTI_KF_E_SHAPE;
    if (d->n_problems == 0) return OPTI_KF_OK;
    if (!d->x || !d->body_ref || !d->p || !d->contact || !d->forces || !d->status) return OPTI_KF_E_NULL;
    if ((d->warm_set == nullptr) != (d->warm_mult == nullptr)) return OPTI_KF_E_NULL;
    okf::MpcParams p;
    std::memset(&p, 0, sizeof p);
    p.N = d->n_problems;
    p.max_legs = d->max_free_legs == 0 ? 4 : d->max_free_legs;
    p.x = (const double *)d->x; p.body_ref = (const double *)d->body_ref; p.p = (const double *)d->p;
    p.contact = (const double *)d->contact; p.forces = (double *)d->forces; p.status = d->status;
    p.warm_set = d->warm_set; p.warm_mult = (double *)d->warm_mult;
    if (d->solver != 0 && d->solver != 1) return OPTI_KF_E_SHAPE;
    p.solver = d->solver;
    p.max_changes = d->max_changes > 0 ? d->max_changes : 0;
    p.dt = d->dt; p.inv_mass = 1.0 / d->mass; p.gravity = d->gravity; p.mu = d->mu; p.fz_max = d->fz_max; p.w_force = d->w_force;
    for (int k = 0; k < 3; ++k) p.inv_inertia[k] = 1.0 / d->inertia[k];
    for (int k = 0; k < 12; ++k) p.w_state[k] = d->w_state[k];
    cudaGetLastError();
    const int rc = okf::launch_mpc(p, (cudaStream_t)cuda_stream);
    if (rc < 0) return rc;
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return cudaGetLastError() == cudaSuccess ? OPTI_KF_OK : OPTI_KF_E_CUDA;
}

// ---- peer memory for the fused summary all-gather (cudaIpc: one process per GPU on one box) ----
int optistate_kf_peer_alloc(size_t bytes, void **dev_ptr_out) {
    if (!dev_ptr_out || bytes == 0) return OPTI_KF_E_NULL;
    *dev_ptr_out = nullptr;
    return cudaMalloc(dev_ptr_out, bytes) == cudaSuccess ? (int)OPTI_KF_OK : (cudaGetLastError(), (int)OPTI_KF_E_CUDA);
}

int optistate_kf_peer_free(void *dev_ptr) {
    if (!dev_ptr) return OPTI_KF_OK;
    return cudaFree(dev_ptr) == cudaSuccess ? (int)OPTI_KF_OK : (cudaGetLastError(), (int)OPTI_KF_E_CUDA);
}

int optistate_kf_peer_export(void *dev_ptr, unsigned char handle_out[OPTI_KF_PEER_HANDLE_BYTES]) {
    static_assert(sizeof(cudaIpcMemHandle_t) <= OPTI_KF_PEER_HANDLE_BYTES, "handle does not fit");
    if (!dev_ptr || !handle_out) return OPTI_KF_E_NULL;
    cudaIpcMemHandle_t h;
    if (cudaIpcGetMemHandle(&h, dev_ptr) != cudaSuccess) { cudaGetLastError(); return OPTI_KF_E_CUDA; }
    std::memset(handle_out, 0, OPTI_KF_PEER_HANDLE_BYTES);
    std::memcpy(handle_out, &h, sizeof h);
    return OPTI_KF_OK;
}

int optistate_kf_peer_open(const unsigned char handle[OPTI_KF_PEER_HANDLE_BYTES], void **peer_ptr_out) {
    if (!handle || !peer_ptr_out) return OPTI_KF_E_NULL;
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, sizeof h);
    *peer_ptr_out = nullptr;
    if (cudaIpcOpenMemHandle(peer_ptr_out, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); return OPTI_KF_E_CUDA; }
    return OPTI_KF_OK;
}

int optistate_kf_peer_close(void *peer_ptr) {
    if (!peer_ptr) return OPTI_KF_OK;
    return cudaIpcCloseMemHandle(peer_ptr) == cudaSuccess ? (int)OPTI_KF_OK : (cudaGetLastError(), (int)OPTI_KF_E_CUDA);
}

const char *optistate_kf_strerror(int code) {
    switch (code) {
        case OPTI_KF_OK: return "ok";
        case OPTI_KF_E_NULL: return "descriptor or a required pointer is NULL";
        case OPTI_KF_E_VERSION: return "descriptor size / ABI version mismatch";
        case OPTI_KF_E_DTYPE: return "unsupported or mismatching dtype";
        case OPTI_KF_E_SHAPE: return "invalid sizes, kinds or constants";
        case OPTI_KF_E_UNSUPPORTED: return "combination not supported by the requested algo";
        case OPTI_KF_E_CUDA: return "CUDA runtime error at launch";
        case OPTI_KF_E_NO_DEVICE: return "no CUDA device";
        default: return "unknown error";
    }
}

}  // extern "C"
