// optistate_kf_closed_loop: the reference driver's per-step call KF.estimate_state_mpc(...) (kalman_filter.py:176-182,
// data_conversion_Kalman_to_Training.py:193-201) for N trajectories over T steps, stepped from a host loop in C++ on top of the
// library's own entry points - optistate_kf_measure once (the measurements do not depend on the state), then per step
// optistate_kf_mpc_forces from the current estimate and optistate_kf_batch for one predict_mpc + update step.  Everything is queued
// on the caller's stream; nothing in the loop synchronises with the host, allocates or goes through an interpreter (the Python
// loop this replaces spent ~200 us per step on bookkeeping - more than the kernels take for a few hundred trajectories).
#include <cuda_runtime.h>

#include <cstring>

#include "../../include/optistate_kf.h"

namespace {

constexpr size_t kAlign = 256;
inline size_t up(size_t b) { return (b + kAlign - 1) & ~(kAlign - 1); }

// workspace layout (bytes): z [T][10][N] | P ping-pong 2 x [144][N] | forces of the horizon [5][12][N] | warm set [5][N] u32 |
// warm multipliers [100][N] | MPC status scratch [N] u32 | the filter step's workspace (leg moments [12][N])
struct Layout {
    size_t z, p0, p1, fh, wset, wmult, mst, fws, total;
    Layout(int64_t N, int64_t T) {
        size_t o = 0;
        z = o; o += up((size_t)T * 10 * N * 8);
        p0 = o; o += up((size_t)144 * N * 8);
        p1 = o; o += up((size_t)144 * N * 8);
        fh = o; o += up((size_t)OPTI_KF_MPC_HORIZON * 12 * N * 8);
        wset = o; o += up((size_t)OPTI_KF_MPC_HORIZON * N * 4);
        wmult = o; o += up((size_t)OPTI_KF_MPC_HORIZON * 4 * 5 * N * 8);
        mst = o; o += up((size_t)N * 4);
        fws = o; o += up((size_t)12 * N * 8);
        total = o;
    }
};

// a shared initial state [12] as the [12][N] array the MPC reads
__global__ void broadcast_state_kernel(const double *x, double *out, long long N) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 12 * N) out[i] = x[i / N];
}

}  // namespace

extern "C" {

size_t optistate_kf_closed_loop_workspace_bytes(int64_t n_traj, int64_t n_steps) {
    if (n_traj <= 0 || n_steps <= 0) return 0;
    return Layout(n_traj, n_steps).total;
}

int optistate_kf_closed_loop(const OptiKfClosedLoopDesc *d, void *cuda_stream) {
    if (!d) return OPTI_KF_E_NULL;
    if (d->struct_size != sizeof(OptiKfClosedLoopDesc) || d->abi_version != OPTISTATE_KF_ABI_VERSION) return OPTI_KF_E_VERSION;
    if (d->dtype != OPTI_KF_F64) return OPTI_KF_E_DTYPE;
    if (d->n_traj < 0 || d->n_steps < 0 || d->max_free_legs < 0 || d->max_free_legs > 4) return OPTI_KF_E_SHAPE;
    if (d->n_traj == 0 || d->n_steps == 0) return OPTI_KF_OK;
    if (!d->imu || !d->p || !d->dp || !d->contact || !d->body_ref || !d->x0 || !d->Q || !d->R || !d->x_steps || !d->workspace) return OPTI_KF_E_NULL;
    const bool diag_q = d->q_kind == OPTI_KF_MAT_DIAG || d->q_kind == OPTI_KF_MAT_DIAG_PER;
    const bool diag_r = d->r_kind == OPTI_KF_MAT_DIAG || d->r_kind == OPTI_KF_MAT_DIAG_PER;
    if (!diag_q || !diag_r) return OPTI_KF_E_UNSUPPORTED;  // dense noise: the joint form, stepped by the caller
    if (d->p0_kind != OPTI_KF_MAT_NONE && !d->P0) return OPTI_KF_E_NULL;
    const int64_t N = d->n_traj, T = d->n_steps;
    const Layout L(N, T);
    if (d->workspace_bytes < L.total || (reinterpret_cast<uintptr_t>(d->workspace) & 15u)) return OPTI_KF_E_SHAPE;
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    unsigned char *ws = (unsigned char *)d->workspace;
    double *z = (double *)(ws + L.z), *Pbuf[2] = {(double *)(ws + L.p0), (double *)(ws + L.p1)}, *fh = (double *)(ws + L.fh);
    uint32_t *wset = (uint32_t *)(ws + L.wset), *mst_scratch = (uint32_t *)(ws + L.mst);
    double *wmult = (double *)(ws + L.wmult);
    if (cudaMemsetAsync(wset, 0, (size_t)OPTI_KF_MPC_HORIZON * N * 4, stream) != cudaSuccess) return OPTI_KF_E_CUDA;
    if (d->status && cudaMemsetAsync(d->status, 0, (size_t)N * 4, stream) != cudaSuccess) return OPTI_KF_E_CUDA;

    // get_odom + set_measurements of every step (kalman_filter.py:79-117); a step without a stance leg flags the trajectory
    OptiKfMeasureDesc m;
    std::memset(&m, 0, sizeof m);
    m.struct_size = sizeof m; m.abi_version = OPTISTATE_KF_ABI_VERSION; m.dtype = OPTI_KF_F64;
    m.n_steps = T; m.n_streams = N;
    m.imu = d->imu; m.p = d->p; m.dp = d->dp; m.contact = d->contact; m.z = z; m.status = d->status;
    int rc = optistate_kf_measure(&m, stream);
    if (rc != OPTI_KF_OK) return rc;

    OptiKfMpcDesc q;
    std::memset(&q, 0, sizeof q);
    q.struct_size = sizeof q; q.abi_version = OPTISTATE_KF_ABI_VERSION; q.dtype = OPTI_KF_F64;
    q.max_free_legs = d->max_free_legs; q.n_problems = N;
    q.forces = fh;
    q.dt = d->dt; q.mass = d->mass; q.gravity = d->gravity; q.mu = d->mu; q.fz_max = d->fz_max; q.w_force = d->w_force;
    for (int k = 0; k < 3; ++k) q.inertia[k] = d->inertia[k];
    for (int k = 0; k < 12; ++k) q.w_state[k] = d->w_state[k];
    q.solver = d->solver; q.max_changes = d->max_changes;
    if (d->warm_start) { q.warm_set = wset; q.warm_mult = wmult; }

    OptiKfDesc f;
    std::memset(&f, 0, sizeof f);
    f.struct_size = sizeof f; f.abi_version = OPTISTATE_KF_ABI_VERSION; f.dtype = OPTI_KF_F64;
    f.algo = OPTI_KF_ALGO_SEQUENTIAL; f.cov_model = OPTI_KF_COV_MPC; f.phases = OPTI_KF_PHASE_PREDICT | OPTI_KF_PHASE_UPDATE;
    f.n_traj = N; f.n_steps = 1; f.n_streams = N; f.stream_offset = 0;
    f.dt = d->dt; f.mass = d->mass; f.gravity = d->gravity;
    for (int k = 0; k < 3; ++k) f.inertia[k] = d->inertia[k];
    f.q_kind = d->q_kind; f.r_kind = d->r_kind; f.Q = d->Q; f.R = d->R;
    f.status = d->status;
    f.flags = d->status ? OPTI_KF_FLAG_STATUS_ACCUMULATE : 0;
    f.workspace = ws + L.fws; f.workspace_bytes = L.total - L.fws;

    const double *x_cur = (const double *)d->x0;
    int x_per = d->x0_per_traj;
    for (int64_t t = 0; t < T; ++t) {
        const double *p_t = (const double *)d->p + t * 12 * N;
        // the QP of every trajectory from its current estimate (kalman_filter.py:141-152).  A shared x0 ([12]) is what every
        // trajectory starts from: the MPC wants [12][N], so step 0 broadcasts it into the covariance buffer that is still free
        const double *x_mpc = x_cur;
        if (!x_per) {  // only possible at t == 0
            double *xb = Pbuf[1];  // free until the end of step 0
            broadcast_state_kernel<<<(unsigned)((12 * N + 255) / 256), 256, 0, stream>>>(x_cur, xb, N);
            x_mpc = xb;
        }
        q.x = x_mpc;
        q.body_ref = (const double *)d->body_ref + t * OPTI_KF_MPC_HORIZON * 12 * N;
        q.p = p_t;
        q.contact = (const double *)d->contact + t * 4 * N;
        q.status = d->mpc_status ? d->mpc_status + t * N : mst_scratch;
        rc = optistate_kf_mpc_forces(&q, stream);
        if (rc != OPTI_KF_OK) return rc;
        if (d->forces && cudaMemcpyAsync((double *)d->forces + t * 12 * N, fh, (size_t)12 * N * 8, cudaMemcpyDeviceToDevice, stream) != cudaSuccess)
            return OPTI_KF_E_CUDA;
        // one filter step with those forces: predict_mpc (covariance by exp(dt F) element-wise with R from body_ref, mean by
        // next_state, kalman_filter.py:153-161) + update (:164-174)
        f.p = p_t;
        f.f = fh;  // stage 0 = the first [12][N] of the horizon
        f.z_in = z + t * 10 * N;
        f.body_ref = q.body_ref;  // column 0 of the horizon reference
        f.x0 = x_cur; f.x0_per_traj = x_per;
        if (t == 0) { f.p0_kind = d->p0_kind; f.P0 = d->P0; }
        else { f.p0_kind = OPTI_KF_MAT_DENSE_PER; f.P0 = Pbuf[(t - 1) & 1]; }
        f.x_final = (double *)d->x_steps + t * 12 * N;
        f.P_final = Pbuf[t & 1];
        f.p_world_steps = d->p_world_steps ? (double *)d->p_world_steps + t * 12 * N : nullptr;
        rc = optistate_kf_batch(&f, stream);
        if (rc != OPTI_KF_OK) return rc;
        x_cur = (const double *)f.x_final;
        x_per = 1;
    }
    return OPTI_KF_OK;
}

}  // extern "C"
