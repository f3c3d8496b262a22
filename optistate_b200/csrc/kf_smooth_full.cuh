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
//
// kStats: the E-step of EM on the same recursion (DESIGN.md section 0.3), as kf_rts_kernel<Real, true> does for the decoupled
// groups: one more step, t = -1, from x+ = x0 and all 78 entries of P+ = P0, and per trajectory the 23 sums of OptiKfNoiseEmDesc.
//   * Sw: warp q owns the rows rtsf_row(q, .).  It solves those columns of M = (P-)^-1 on the factor it holds, parks them in its
//     own slots of W (dead until W is written), and once dPs is complete adds q + q^2 ((M dPs M)_uu + (M d)_u^2).
//   * Sv: row k goes to the warp that owns the diagonal entry of dPs it reads (tri(sel(k), sel(k)) mod 4), before it subtracts P-.
//   * log-likelihood: warp RTSF_LL_WARP, after its rows of Ps_t, recomputes P- and factors S = H P- H^T + R (10x10) on the
//     innovation; determinants are multiplied into a mantissa with the exponent split off (det_renorm).
//   * The accumulators are registers of the warp that owns them; z is read from global memory (shared by a stream's members).
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
    // E-step of EM (kf_rts_full_kernel<Real, kMpc, true> only; last, so that every field above keeps its constant-bank offset)
    const Real *z;              // [T][10][S] measurements of the stream (S, stream_offset, stream_index as for body_ref)
    const Real *R; int r_kind;  // OPTI_KF_MAT_DIAG [10] or OPTI_KF_MAT_DIAG_PER [10][N]
    const Real *x0; long long x0_ld; int x0_inc;
    const Real *P0; int p0_kind;  // any kind of Params: NONE = Q
    Real *stats;                // [23][N]: Sw (0-11), Sv (12-21), log-likelihood (22)
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

// E-step roles.  Sv row k: the warp that owns dPs entry tri(sel(k), sel(k)) (3 3 2 2 rows for warps 0-3), in accumulator slot
// rtsf_sv_slot(k); the log-likelihood: warp 2 (19 triangle entries, 2 Sv rows).
__host__ __device__ constexpr int rtsf_sv_warp(int k) { return tri(sel(k), sel(k)) & 3; }
__host__ __device__ constexpr int rtsf_sv_slot(int k) {
    int n = 0;
    for (int j = 0; j < k; ++j) n += rtsf_sv_warp(j) == rtsf_sv_warp(k);
    return n;
}
__host__ __device__ constexpr int rtsf_sv_of(int k) {  // measurement row whose Sv reads dPs entry k, or -1
    for (int j = 0; j < NZ; ++j)
        if (tri(sel(j), sel(j)) == k) return j;
    return -1;
}
constexpr int RTSF_SV_SLOTS = 3;
constexpr int RTSF_LL_WARP = 2;
__host__ __device__ constexpr bool rtsf_sv_ok() {
    for (int k = 0; k < NZ; ++k)
        if (rtsf_sv_slot(k) >= RTSF_SV_SLOTS) return false;
    return true;
}
static_assert(rtsf_sv_ok(), "no warp owns more than three Sv rows");

template <typename Real, bool kMpc, bool kStats = false>
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
    const long long s = (kMpc || kStats) ? (prm.stream_index ? (long long)prm.stream_index[ic] : (ic + prm.stream_offset) % prm.S) : 0;
    const Real *qg = prm.Q + (prm.q_kind == OPTI_KF_MAT_DIAG ? 0 : ic);
    const int qs = prm.q_kind == OPTI_KF_MAT_DIAG ? 1 : (int)N;
    int rows[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) rows[c] = rtsf_row(q, c);

    // entry k (tri order) of P0 for the step t = -1
    const auto prior_P0 = [&](int k) -> Real {
        int a = 0;
        while (tri(a, a) < k) ++a;
        const int b = k - tri(a, 0);
        switch (prm.p0_kind) {
            case OPTI_KF_MAT_NONE: return a == b ? qg[a * qs] : Real(0);
            case OPTI_KF_MAT_DIAG: return a == b ? prm.P0[a] : Real(0);
            case OPTI_KF_MAT_DIAG_PER: return a == b ? prm.P0[a * N + ic] : Real(0);
            case OPTI_KF_MAT_DENSE: return prm.P0[a * NX + b];
            default: return prm.P0[(long long)(a * NX + b) * N + ic];
        }
    };
    // step t's stage: x+_t, P+_t and (t + 1 < T) x-_{t+1} and the reference angles of step t + 1; warp q copies rows q mod 4
    const auto issue = [&](long long t, Real *st) {
#pragma unroll 1
        for (int r = q; r < RTSF_STAGE_ROWS; r += RTSF_WARPS) {
            const Real *src;
            if constexpr (kStats) {
                if (t < 0 && r < NX + NP) {  // the step t = -1: x+ = x0, P+ = P0 (Q when absent), every entry
                    st[r * nt] = r < NX ? prm.x0[r * prm.x0_ld + ic * prm.x0_inc] : prior_P0(r - NX);
                    continue;
                }
            }
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
        if constexpr (kStats) {
            if (t < 0) return;  // the step t = -1 stores nothing; x_smooth is optional
            if (prm.x_smooth) st_stream(prm.x_smooth + (t * NX + row) * N + i, x);
        } else {
            st_stream(prm.x_smooth + (t * NX + row) * N + i, x);
        }
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
        else if constexpr (kStats) issue(-1, stage1);
    }

    uint32_t status[1] = {0};
    const Real e1 = kMpc ? exp_minus_one(prm.dt) : Real(0);
    // P-_{t+1}, as the forward pass's predict of step t + 1 formed it, from stage t; B: the blocks of F - 1 1^T (mpc: E) or F - I
    // (predict: dt R^T) on the attitude rows
    const auto prior = [&](const Real *st, Real (&Pm)[NP], Real (&B)[9]) {
#pragma unroll
        for (int k = 0; k < NP; ++k) Pm[k] = st[(NX + k) * nt];
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
    };
    const Real *zs = kStats ? prm.z + s : nullptr;  // z of this trajectory's stream
    Real accw[3], accv[RTSF_SV_SLOTS], ll_quad = Real(0), det_m = Real(1);  // E-step accumulators of this warp's rows
    int det_e = 0;
    uint32_t ll_bad[1] = {0};
#pragma unroll
    for (int c = 0; c < 3; ++c) accw[c] = Real(0);
#pragma unroll
    for (int c = 0; c < RTSF_SV_SLOTS; ++c) accv[c] = Real(0);
    for (long long t = T - 2; t >= (kStats ? -1 : 0); --t) {
        cp_async_wait_all();
        __syncthreads();  // stage t has landed; xs_{t+1}, Ps_{t+1} are written and the previous step's W has been read
        const Real *st = (t & 1) ? stage1 : stage0;
        if (t > 0) issue(t - 1, (t & 1) ? stage0 : stage1);  // that stage was step t + 1's, read before the barrier
        else if constexpr (kStats) {
            if (t == 0) issue(-1, stage1);
        }

        Real Pm[NP], B[9];
        prior(st, Pm, B);
        // dPs = Ps_{t+1} - P-_{t+1}: warp q owns the entries k = q mod 4
#pragma unroll
        for (int k = 0; k < NP; ++k)
            if ((k & 3) == q) {
                if constexpr (kStats) {
                    const int j = rtsf_sv_of(k);  // Sv of measurement row j: (z_{t+1,j} - xs_{t+1,sel(j)})^2 + Ps_{t+1,sel(j)sel(j)}
                    if (j >= 0) {
                        const Real e = ld_stream(zs + ((t + 1) * NZ + j) * prm.S) - xsm[sel(j) * nt];
                        accv[rtsf_sv_slot(j)] += fma_(e, e, ps[k * nt]);
                    }
                }
                ps[k * nt] -= Pm[k];
            }

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

        if constexpr (kStats) {
            // columns rows[c] of M = (P-)^-1 = L^-T D^-1 L^-1, parked in this warp's slots of W until dPs is complete
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                Real m[NX];
#pragma unroll
                for (int u = 0; u < NX; ++u) {
                    Real v = u == rows[c] ? Real(1) : Real(0);
#pragma unroll
                    for (int k = 0; k < u; ++k) v = fnma_(Pm[tri(u, k)], m[k], v);
                    m[u] = v;
                }
#pragma unroll
                for (int u = 0; u < NX; ++u) m[u] *= dinv[u];
#pragma unroll
                for (int u = NX - 2; u >= 0; --u)
#pragma unroll
                    for (int k = u + 1; k < NX; ++k) m[u] = fnma_(Pm[tri(k, u)], m[k], m[u]);
#pragma unroll
                for (int u = 0; u < NX; ++u) W[(u * NX + rows[c]) * nt] = m[u];
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
        Real m[kStats ? 3 : 1][NX], quad[3];  // E-step: this warp's columns of M and m^T dPs m
        if constexpr (kStats) {
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                quad[c] = Real(0);
#pragma unroll
                for (int u = 0; u < NX; ++u) m[c][u] = W[(u * NX + rows[c]) * nt];
            }
        }
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
                if constexpr (kStats) {
                    Real h = dk[0] * m[c][0];
#pragma unroll
                    for (int l = 1; l < NX; ++l) h = fma_(dk[l], m[c][l], h);
                    quad[c] = fma_(m[c][k], h, quad[c]);
                }
                W[(k * NX + rows[c]) * nt] = v;
            }
        }
        if constexpr (kStats) {
            // Sw: E[w_u^2 | Z] = q_u + q_u^2 ((M dPs M)_uu + (M d)_u^2), d = xs_{t+1} - x-_{t+1}
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                Real md = Real(0);
#pragma unroll
                for (int u = 0; u < NX; ++u) md = fma_(m[c][u], xsm[u * nt] - st[(NX + NP + u) * nt], md);
                const Real qc = qg[rows[c] * qs];
                accw[c] += fma_(qc * qc, fma_(md, md, quad[c]), qc);
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
        if constexpr (kStats) {
            if (q == RTSF_LL_WARP) {
                // log N(z_{t+1}; H x-_{t+1}, S), S = H P-_{t+1} H^T + R: P- once more, then L D L^T of S solved on the innovation
                Real y[NZ];
#pragma unroll
                for (int j = 0; j < NZ; ++j) y[j] = ld_stream(zs + ((t + 1) * NZ + j) * prm.S) - st[(NX + NP + sel(j)) * nt];
                Real Sm[NP], Bl[9];
                prior(st, Sm, Bl);
                Real yq = Real(0);
#pragma unroll
                for (int j = 0; j < NZ; ++j) {
                    const int sj = sel(j);
                    Real e[NZ];  // e[k] = L[j][k] D[k]
#pragma unroll
                    for (int k = 0; k < j; ++k) e[k] = Sm[tri(sj, sel(k))] * Sm[tri(sel(k), sel(k))];
                    Real dj = Sm[tri(sj, sj)] + __ldg(prm.r_kind == OPTI_KF_MAT_DIAG ? prm.R + j : prm.R + j * N + ic);
#pragma unroll
                    for (int k = 0; k < j; ++k) dj = fnma_(e[k], Sm[tri(sj, sel(k))], dj);
                    note_bad_pivot(dj, ll_bad, EM_BAD_PIVOT);
                    Sm[tri(sj, sj)] = dj;
                    const Real inv = rcp_(dj);
#pragma unroll
                    for (int r = j + 1; r < NZ; ++r) {
                        Real v = Sm[tri(sel(r), sj)];
#pragma unroll
                        for (int k = 0; k < j; ++k) v = fnma_(Sm[tri(sel(r), sel(k))], e[k], v);
                        Sm[tri(sel(r), sj)] = v * inv;
                    }
                    Real yj = y[j];
#pragma unroll
                    for (int k = 0; k < j; ++k) yj = fnma_(Sm[tri(sj, sel(k))], y[k], yj);
                    y[j] = yj;
                    yq = fma_(yj * inv, yj, yq);
                    det_m *= dj;
                    det_renorm(det_m, det_e);
                }
                ll_quad = fma_(Real(-0.5), yq, ll_quad);
            }
        }
    }
    if constexpr (kStats) {
        if (active) {
#pragma unroll
            for (int c = 0; c < 3; ++c) prm.stats[rows[c] * N + i] = accw[c];
#pragma unroll
            for (int k = 0; k < NZ; ++k)
                if (rtsf_sv_warp(k) == q) prm.stats[(NX + k) * N + i] = accv[rtsf_sv_slot(k)];
            if (q == RTSF_LL_WARP) {
                // -0.5 (10 T log 2 pi + log det) + the accumulated -0.5 y^T S^-1 y; a bad pivot of S makes it NaN
                const double log_det = log((double)det_m) + (double)det_e * 0.69314718055994530942;
                const double ll = (double)ll_quad - 0.5 * (log_det + (double)(NZ * T) * 1.83787706640934548356);
                prm.stats[(EM_STATS_ROWS - 1) * N + i] = ll_bad[0] ? Real(NAN) : (Real)ll;
            }
        }
    }
    if (q == 0 && active && status[0] && prm.status) prm.status[i] |= status[0];
}

// Launch of kf_rts_full_kernel<Real, mpc, kStats> (instantiated in kf_smooth_full.cu for double and float).
template <typename Real, bool kStats>
int launch_rts_full(const SmoothFullParams<Real> &p, cudaStream_t stream);

}  // namespace okf
