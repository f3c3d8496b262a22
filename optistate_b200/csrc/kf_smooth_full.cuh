// Backward pass of the fixed-interval Rauch-Tung-Striebel smoother on the FULL covariance of the SEQUENTIAL filter
// (DESIGN.md section 0.2): the predict() model with a coupled P0, and the predict_mpc model, whose F_d = 1 1^T + D makes P
// dense.  The recursion of kf_smooth.cuh on dense 12x12 blocks, from the filter's x+_t, all 78 entries of P+_t
// (Params.P_steps of the full kernels, store_full_P) and x-_{t+1}:
//     P-_{t+1} = F_{t+1} P+_t F_{t+1}^T + Q     recomputed with the forward pass's own functions:
//                                               predict: rot_zyx(x+_t) and cov_predict_sym<false>;
//                                               mpc: E = exp_minus_one(dt Rb^T) of step t + 1's reference angles, cov_predict_mpc_sym
//     P- = L D L^T,  G_t^T = (P-)^-1 C  with  C = F_{t+1} P+_t  (mpc: C = 1 (P+ 1)^T + D P+)
//     xs_t = x+_t + G_t (xs_{t+1} - x-_{t+1}),   Ps_t = P+_t + G_t (Ps_{t+1} - P-_{t+1}) G_t^T
//
//   * Four warps share 32 trajectories; warp q is role q of every trajectory of the block, so the role is warp-uniform (no
//     divergence) and every shared-memory access is [row][32 trajectories]: 32 consecutive words, conflict-free.
//   * Every warp recomputes P- and its L D L^T in registers (the same values in all four; ~25 % of the arithmetic); warp q then
//     solves the three columns G^T[:, rtsf_row(q, 0..2)], gives those rows of xs_t and of W = dPs G^T, and - once W is
//     exchanged through shared memory - those rows of the triangle of Ps_t.  The row sets {0 6 11} {1 5 10} {3 4 9} {2 7 8}
//     give each warp 19 or 20 entries of the triangle.
//   * The next (earlier) step's inputs are copied to shared memory with cp.async while the current one computes (two stages),
//     each warp copying a quarter of the rows; three block barriers per step.
//   * Pivots use rcp_.  One that is not positive and finite sets OPTI_KF_ST_SMOOTH_NOT_PD; the recursion carries on.
#pragma once

#include "kf_smooth.cuh"

namespace okf {

template <typename Real>
struct SmoothFullParams {
    long long N, T;
    Real dt;
    int cov_model;              // OPTI_KF_COV_PREDICT | OPTI_KF_COV_MPC
    const Real *Q; int q_kind;  // OPTI_KF_MAT_DIAG [12] or OPTI_KF_MAT_DIAG_PER [12][N]
    const Real *x_post;         // [T][12][N] x+ (the filter's x_steps)
    const Real *x_prior;        // [T][12][N] x- (x_model_steps)
    const Real *P_post;         // [T][78][N] P+ in tri order (Params.P_steps of the full kernels)
    const Real *body_ref;       // [T][12][S] (mpc): trajectory i reads stream stream_index[i] or (i + stream_offset) % S
    long long S, stream_offset;
    const int32_t *stream_index;
    Real *x_smooth;             // [T][12][N]
    Real *var_smooth;           // [T][12][N] or NULL
    uint32_t *status;           // [N] or NULL: OPTI_KF_ST_SMOOTH_NOT_PD is OR-ed in
};

constexpr int RTSF_TRAJ = 32;                      // trajectories per block
constexpr int RTSF_WARPS = 4;                      // roles per trajectory
constexpr int RTSF_THREADS = RTSF_TRAJ * RTSF_WARPS;
constexpr int RTSF_STAGE_ROWS = NX + NP + NX + 3;  // x+_t, P+_t, x-_{t+1}, reference angles of step t + 1 (mpc)
constexpr int RTSF_SMEM_ROWS = 2 * RTSF_STAGE_ROWS + NP + NX + NX * NX;  // two stages, Ps, xs, W: 111 KB per block in FP64

// row c (0..2) of G handled by warp q: nibble 3 q + c of the table {0 6 11} {1 5 10} {3 4 9} {2 7 8}
constexpr unsigned long long RTSF_ROWS = 0x872943a51b60ull;
__host__ __device__ constexpr int rtsf_row(int q, int c) { return (int)((RTSF_ROWS >> (4 * (3 * q + c))) & 15); }
__host__ __device__ constexpr bool rtsf_rows_ok() {
    int seen = 0;
    for (int q = 0; q < RTSF_WARPS; ++q) {
        int entries = 0;
        for (int c = 0; c < 3; ++c) {
            seen |= 1 << rtsf_row(q, c);
            entries += rtsf_row(q, c) + 1;
        }
        if (entries < 19 || entries > 20) return false;
    }
    return seen == (1 << NX) - 1;
}
static_assert(rtsf_rows_ok(), "the row sets partition the 12 rows with 19-20 triangle entries per warp");

template <typename Real, bool kMpc>
__global__ void __launch_bounds__(RTSF_THREADS, 2) kf_rts_full_kernel(const __grid_constant__ SmoothFullParams<Real> prm) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int nt = RTSF_TRAJ;
    const int lane = threadIdx.x & 31, q = threadIdx.x >> 5;
    Real *stage0 = reinterpret_cast<Real *>(smem_raw) + lane;  // [105][32] x2
    Real *stage1 = stage0 + RTSF_STAGE_ROWS * nt;
    Real *ps = stage1 + RTSF_STAGE_ROWS * nt;  // [78]: Ps_{t+1}, then dPs = Ps_{t+1} - P-_{t+1}, then Ps_t
    Real *xsm = ps + NP * nt;                  // [12]: xs_{t+1}, then xs_t
    Real *W = xsm + NX * nt;                   // [12][12]: W = dPs G^T
    const long long N = prm.N, T = prm.T;
    const long long i = (long long)blockIdx.x * nt + lane;
    const bool active = i < N;
    const long long ic = active ? i : N - 1;  // the last block's spare lanes recompute a real trajectory and store nothing
    const long long s = kMpc ? (prm.stream_index ? (long long)prm.stream_index[ic] : (ic + prm.stream_offset) % prm.S) : 0;
    const Real *qg = prm.Q + (prm.q_kind == OPTI_KF_MAT_DIAG ? 0 : ic);
    const int qs = prm.q_kind == OPTI_KF_MAT_DIAG ? 1 : (int)N;
    int rows[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) rows[c] = rtsf_row(q, c);

    // step t's stage: x+_t, P+_t and (t + 1 < T) x-_{t+1} and the reference angles of step t + 1; warp q copies rows q mod 4
    const auto issue = [&](long long t, Real *st) {
#pragma unroll 1
        for (int r = q; r < RTSF_STAGE_ROWS; r += RTSF_WARPS) {
            const Real *src;
            if (r < NX) src = prm.x_post + (t * NX + r) * N + ic;
            else if (r < NX + NP) src = prm.P_post + (t * NP + (r - NX)) * N + ic;
            else if (t + 1 >= T) continue;
            else if (r < 2 * NX + NP) src = prm.x_prior + ((t + 1) * NX + (r - NX - NP)) * N + ic;
            else if (kMpc) src = prm.body_ref + ((t + 1) * 12 + (r - 2 * NX - NP)) * prm.S + s;
            else continue;
            cp_async_elem(st + r * nt, src);
        }
        cp_async_commit();
    };
    const auto store = [&](long long t, int row, Real x, Real var) {
        if (!active) return;
        st_stream(prm.x_smooth + (t * NX + row) * N + i, x);
        if (prm.var_smooth) st_stream(prm.var_smooth + (t * NX + row) * N + i, var);
    };

    {  // step T - 1: the smoother starts from the filter
        Real *st = ((T - 1) & 1) ? stage1 : stage0;
        issue(T - 1, st);
        cp_async_wait_all();
        __syncthreads();
#pragma unroll 1
        for (int r = q; r < NX; r += RTSF_WARPS) xsm[r * nt] = st[r * nt];
#pragma unroll 1
        for (int k = q; k < NP; k += RTSF_WARPS) ps[k * nt] = st[(NX + k) * nt];
#pragma unroll
        for (int c = 0; c < 3; ++c) store(T - 1, rows[c], st[rows[c] * nt], st[(NX + tri(rows[c], rows[c])) * nt]);
        if (T >= 2) issue(T - 2, ((T - 2) & 1) ? stage1 : stage0);
    }

    uint32_t status[1] = {0};
    const Real e1 = kMpc ? exp_minus_one(prm.dt) : Real(0);
    for (long long t = T - 2; t >= 0; --t) {
        cp_async_wait_all();
        __syncthreads();  // stage t has landed; xs_{t+1}, Ps_{t+1} are written and the previous step's W has been read
        const Real *st = (t & 1) ? stage1 : stage0;
        if (t > 0) issue(t - 1, (t & 1) ? stage0 : stage1);  // that stage was step t + 1's, read before the barrier

        // P-_{t+1}, as the forward pass's predict of step t + 1 formed it
        Real Pm[NP];
#pragma unroll
        for (int k = 0; k < NP; ++k) Pm[k] = st[(NX + k) * nt];
        Real B[9];  // the blocks of F - 1 1^T (mpc: E) or F - I (predict: dt R^T) on the attitude rows
        if constexpr (kMpc) {
            const Real *ref = st + (2 * NX + NP) * nt;
            Real Rb[9];
            rot_zyx(ref[0], ref[nt], ref[2 * nt], Rb);
#pragma unroll
            for (int a = 0; a < 3; ++a)
#pragma unroll
                for (int k = 0; k < 3; ++k) B[3 * a + k] = exp_minus_one(prm.dt * Rb[3 * k + a]);
            cov_predict_mpc_sym(Pm, B, e1, qg, qs);
        } else {
            Real R[9];
            rot_zyx(st[0], st[nt], st[2 * nt], R);
#pragma unroll
            for (int a = 0; a < 3; ++a)
#pragma unroll
                for (int k = 0; k < 3; ++k) B[3 * a + k] = prm.dt * R[3 * k + a];
            cov_predict_sym<false>(Pm, R, prm.dt, qg, qs);
        }
        // dPs = Ps_{t+1} - P-_{t+1}: warp q owns the entries k = q mod 4
#pragma unroll
        for (int k = 0; k < NP; ++k)
            if ((k & 3) == q) ps[k * nt] -= Pm[k];

        // P- = L D L^T in place: L[i][j] (i > j) at tri(i, j), D[j] at tri(j, j)
        Real dinv[NX];
#pragma unroll
        for (int j = 0; j < NX; ++j) {
            Real e[NX];  // e[k] = L[j][k] D[k]
#pragma unroll
            for (int k = 0; k < j; ++k) e[k] = Pm[tri(j, k)] * Pm[tri(k, k)];
            Real dj = Pm[tri(j, j)];
#pragma unroll
            for (int k = 0; k < j; ++k) dj = fnma_(e[k], Pm[tri(j, k)], dj);
            note_bad_pivot(dj, status, OPTI_KF_ST_SMOOTH_NOT_PD);
            Pm[tri(j, j)] = dj;
            dinv[j] = rcp_(dj);
#pragma unroll
            for (int r = j + 1; r < NX; ++r) {
                Real v = Pm[tri(r, j)];
#pragma unroll
                for (int k = 0; k < j; ++k) v = fnma_(Pm[tri(r, k)], e[k], v);
                Pm[tri(r, j)] = v * dinv[j];
            }
        }

        // this warp's columns of C = F P+, then G^T = (P-)^-1 C on them
        Real Gt[NX][3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            Real col[NX];  // P+[:, rows[c]]
#pragma unroll
            for (int u = 0; u < NX; ++u) col[u] = st[(NX + tri(u, rows[c])) * nt];
            Real w = Real(0);  // mpc: (1^T P+)[rows[c]]
            if constexpr (kMpc) {
#pragma unroll
                for (int u = 0; u < NX; ++u) w += col[u];
            }
#pragma unroll
            for (int u = 0; u < NX; ++u) {
                Real v = kMpc ? Real(0) : col[u];
                if (u < 3) {
#pragma unroll
                    for (int k = 0; k < 3; ++k) v = fma_(B[3 * u + k], col[6 + k], v);
                } else if (u < 6) {
                    v = fma_(kMpc ? e1 : prm.dt, col[u + 6], v);
                }
                Gt[u][c] = kMpc ? v + w : v;
            }
#pragma unroll
            for (int u = 1; u < NX; ++u)
#pragma unroll
                for (int k = 0; k < u; ++k) Gt[u][c] = fnma_(Pm[tri(u, k)], Gt[k][c], Gt[u][c]);
#pragma unroll
            for (int u = 0; u < NX; ++u) Gt[u][c] *= dinv[u];
#pragma unroll
            for (int u = NX - 2; u >= 0; --u)
#pragma unroll
                for (int k = u + 1; k < NX; ++k) Gt[u][c] = fnma_(Pm[tri(k, u)], Gt[k][c], Gt[u][c]);
        }
        // xs_t = x+_t + G d on this warp's rows
        Real xn[3];
        {
            Real d[NX];
#pragma unroll
            for (int u = 0; u < NX; ++u) d[u] = xsm[u * nt] - st[(NX + NP + u) * nt];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                Real v = st[rows[c] * nt];
#pragma unroll
                for (int u = 0; u < NX; ++u) v = fma_(Gt[u][c], d[u], v);
                xn[c] = v;
            }
        }
        __syncthreads();  // dPs complete
#pragma unroll
        for (int k = 0; k < NX; ++k) {
            Real dk[NX];
#pragma unroll
            for (int l = 0; l < NX; ++l) dk[l] = ps[tri(k, l) * nt];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                Real v = dk[0] * Gt[0][c];
#pragma unroll
                for (int l = 1; l < NX; ++l) v = fma_(dk[l], Gt[l][c], v);
                W[(k * NX + rows[c]) * nt] = v;
            }
        }
        __syncthreads();  // W complete, dPs read
        // Ps_t(r, j) = P+(r, j) + sum_k G^T[k][r] W[k][j] for this warp's rows r, j <= r
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const int r = rows[c];
            Real diag = Real(0);
#pragma unroll 1
            for (int j = 0; j <= r; ++j) {
                Real v = st[(NX + tri(r, j)) * nt];
#pragma unroll
                for (int k = 0; k < NX; ++k) v = fma_(Gt[k][c], W[(k * NX + j) * nt], v);
                ps[tri(r, j) * nt] = v;
                diag = v;
            }
            xsm[r * nt] = xn[c];
            store(t, r, xn[c], diag);
        }
    }
    if (q == 0 && active && status[0] && prm.status) prm.status[i] |= status[0];
}

// Launch of kf_rts_full_kernel<Real, mpc> (instantiated in kf_smooth_full.cu for double and float).
template <typename Real>
int launch_rts_full(const SmoothFullParams<Real> &p, cudaStream_t stream);

}  // namespace okf
