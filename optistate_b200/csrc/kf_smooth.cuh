// Backward pass of the fixed-interval Rauch-Tung-Striebel smoother over the SEQUENTIAL filter of the predict() model
// (DESIGN.md section 0).  Per trajectory, from the filter's posterior x+_t, packed posterior P+_t (Params.P_steps) and prior
// mean x-_t:
//     P-_{t+1} = F_{t+1} P+_t F_{t+1}^T + Q          recomputed with the forward pass's own rot_zyx + cov_predict_sym<true>
//     G_t      = P+_t F_{t+1}^T (P-_{t+1})^-1         solved as  P-_{t+1} G_t^T = F_{t+1} P+_t
//     xs_t     = x+_t + G_t (xs_{t+1} - x-_{t+1})
//     Ps_t     = P+_t + G_t (Ps_{t+1} - P-_{t+1}) G_t^T
// starting from xs_{T-1} = x+_{T-1}, Ps_{T-1} = P+_{T-1}.  F_{t+1} = I + dt F with F[0:3,6:9] = R(x+_t)^T is the transition the
// filter's predict of step t + 1 used (not the trunc(R^T) of the mean model, SURVEY 0.2).
//
//   * One thread per trajectory, reverse time loop; xs (12) and the 30 coupled entries of Ps live in registers.
//   * G has the decoupled-group structure of P (kf_seq_core.cuh): per step one 6x6 LDL^T solve (attitude + body rate) and three
//     2x2 ones (position + velocity of one axis), and G dPs G^T on the packed lower triangles.  Pivots use rcp_, not division.
//   * The 54 inputs of the next (earlier) step are copied to shared memory with cp.async before the current step's arithmetic
//     starts, so a whole step hides their HBM latency without holding registers; each thread reads only its own rows.
//   * A pivot of P- that is not positive and finite sets OPTI_KF_ST_SMOOTH_NOT_PD; the recursion carries on.
#pragma once

#include "kf_seq_core.cuh"

namespace okf {

template <typename Real>
struct SmoothParams {
    long long N, T;
    Real dt;
    const Real *Q; int q_kind;  // OPTI_KF_MAT_DIAG [12] or OPTI_KF_MAT_DIAG_PER [12][N]
    const Real *x_post;         // [T][12][N] x+ (the filter's x_steps)
    const Real *x_prior;        // [T][12][N] x- (x_model_steps)
    const Real *P_post;         // [T][30][N] packed P+ (Params.P_steps)
    Real *x_smooth;             // [T][12][N]
    Real *var_smooth;           // [T][12][N] or NULL
    uint32_t *status;           // [N] or NULL: OPTI_KF_ST_SMOOTH_NOT_PD is OR-ed in
    // E-step of EM (kf_rts_kernel<Real, true> only; last, so that every field above keeps its constant-bank offset)
    const Real *z;              // [T][10][S] measurements, trajectory i reads stream stream_index[i] or (i + stream_offset) % S
    long long S, stream_offset;
    const int32_t *stream_index;
    const Real *R; int r_kind;  // OPTI_KF_MAT_DIAG [10] or OPTI_KF_MAT_DIAG_PER [10][N]
    const Real *x0; long long x0_ld; int x0_inc;
    const Real *P0; int p0_kind;  // as in Params (decoupled): NONE = Q
    Real *stats;                // [23][N]: Sw (0-11), Sv (12-21), log-likelihood (22)
};

constexpr int RTS_THREADS = 64;
constexpr int RTS_STAGE_ROWS = NX + NPB + NX;  // x+_t, P+_t, x-_{t+1}
constexpr int RTS_SMEM_ROWS = NX + RTS_STAGE_ROWS;  // q, then the staged step
// E-step: the stage gains z_{t+1}; the innovation and the 23 accumulators follow it (55.8 KB per block in FP64: dynamic shared-memory opt-in)
constexpr int EM_STATS_ROWS = OPTI_KF_EM_STATS_ROWS;
constexpr int EM_STAGE_ROWS = RTS_STAGE_ROWS + NZ;
constexpr int EM_SMEM_ROWS = NX + EM_STAGE_ROWS + NZ + EM_STATS_ROWS;

template <typename Real>
__device__ __forceinline__ void cp_async_elem(Real *dst, const Real *src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], %2;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src), "n"(sizeof(Real))
                 : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// global state index of local index u of group G: G0 = {th, w} (0 1 2 6 7 8), G1..3 = {position, velocity} of one axis
template <int G>
__host__ __device__ constexpr int rts_gi(int u) { return G == 0 ? (u < 3 ? u : u + 3) : (u == 0 ? 2 + G : 8 + G); }

// Per-thread state of the E-step (kf_rts_kernel<Real, true>).  q, the innovation y = z_{t+1} - H x-_{t+1} of the step and the
// 23 accumulators are shared-memory columns (stride nt): in registers they would spill.  r is read where it is used.  The
// log-determinants of the innovation covariances are summed as a product det_m * 2^det_e with det_m kept in [1, 2): no
// logarithm in the loop and no underflow in FP32.
template <typename Real>
struct EmState {
    const Real *q;
    Real *y, *acc;
    int nt;
    const Real *R; int r_kind;
    long long N, i;
    Real det_m;
    int det_e;
    __device__ __forceinline__ Real r(int k) const { return __ldg(r_kind == OPTI_KF_MAT_DIAG ? R + k : R + k * N + i); }
};
// A pivot of an innovation covariance that is not positive and finite: the log-likelihood is NaN.  Private to the kernel.
constexpr uint32_t EM_BAD_PIVOT = 0x80000000u;

// measurement row of local index u of group G, or -1 (x and y are not measured): H selects sel(k) (kf_common.cuh)
template <int G>
__host__ __device__ constexpr int em_row(int u) { return G == 0 ? (u < 3 ? u : u + 1) : G == 1 ? (u == 1 ? 7 : -1) : G == 2 ? (u == 1 ? 8 : -1) : (u == 0 ? 3 : 9); }

__device__ __forceinline__ void det_renorm(double &m, int &e) {  // m > 0 normal
    const int hi = __double2hiint(m);
    e += (hi >> 20) - 1023;
    m = __hiloint2double((hi & 0x000fffff) | 0x3ff00000, __double2loint(m));
}
__device__ __forceinline__ void det_renorm(float &m, int &e) {
    const int b = __float_as_int(m);
    e += (b >> 23) - 127;
    m = __int_as_float((b & 0x007fffff) | 0x3f800000);
}

// One decoupled group of the backward step.  In: P+ (Pp, destroyed), the recomputed P- (Pm), dPs = Ps_{t+1} - P- (Dl),
// d = xs_{t+1} - x-_{t+1}.  Out: xs_t into xs, Ps_t into Dl (both for this group's entries only).  A = dt R^T (group 0).
// kStats: also the group's terms of the E-step (EmState).
template <int G, bool kStats = false, typename Real>
__device__ __forceinline__ void rts_group(const Real (&xp)[NX], Real (&Pp)[NP], Real (&Pm)[NP], Real (&Dl)[NP], const Real (&d)[NX],
                                          const Real (&A)[9], Real dt, Real (&xs)[NX], uint32_t (&status)[1],
                                          EmState<Real> *em = nullptr) {
    constexpr int n = G == 0 ? 6 : 2, h = n / 2;
    const auto pp = [&](int u, int v) { return Pp[tri(rts_gi<G>(u), rts_gi<G>(v))]; };
    // C = F P+ on the group: F = [[I, Fo], [0, I]], Fo = dt R^T (attitude rows on body rate) or dt (position on velocity)
    Real Gt[n][n];
    const auto form_C = [&] {
#pragma unroll
        for (int u = 0; u < n; ++u)
#pragma unroll
            for (int v = 0; v < n; ++v) {
                Real s = pp(u, v);
                if (u < h) {
#pragma unroll
                    for (int w = 0; w < h; ++w) s = fma_(G == 0 ? A[3 * u + w] : dt, pp(h + w, v), s);
                }
                Gt[u][v] = s;
            }
    };
    const auto dl = [&](int k, int l) { return Dl[tri(rts_gi<G>(k), rts_gi<G>(l))]; };
    if constexpr (kStats) {
        // log N(y; 0, S) of the measurements of this group, S = H P- H^T + R: L D L^T of S, solved on y as it is factored
        constexpr int nm = G == 0 ? 6 : G == 3 ? 2 : 1;
        constexpr int m0 = G == 1 || G == 2 ? 1 : 0;  // local index of the first measured state
        Real SL[nm][nm], SD[nm], yv[nm], quad = Real(0);
#pragma unroll
        for (int j = 0; j < nm; ++j) {
            const int uj = m0 + j;
            Real e[nm];
#pragma unroll
            for (int k = 0; k < j; ++k) e[k] = SL[j][k] * SD[k];
            Real dj = Pm[tri(rts_gi<G>(uj), rts_gi<G>(uj))] + em->r(em_row<G>(uj));
#pragma unroll
            for (int k = 0; k < j; ++k) dj = fnma_(e[k], SL[j][k], dj);
            note_bad_pivot(dj, status, EM_BAD_PIVOT);
            SD[j] = dj;
            const Real inv = rcp_(dj);
#pragma unroll
            for (int i = j + 1; i < nm; ++i) {
                Real s = Pm[tri(rts_gi<G>(m0 + i), rts_gi<G>(uj))];
#pragma unroll
                for (int k = 0; k < j; ++k) s = fnma_(SL[i][k], e[k], s);
                SL[i][j] = s * inv;
            }
            Real yj = em->y[em_row<G>(uj) * em->nt];
#pragma unroll
            for (int k = 0; k < j; ++k) yj = fnma_(SL[j][k], yv[k], yj);
            yv[j] = yj;
            quad = fma_(yj * inv, yj, quad);
            em->det_m *= dj;
            det_renorm(em->det_m, em->det_e);
        }
        Real *a = em->acc + (EM_STATS_ROWS - 1) * em->nt;
        *a = fma_(Real(-0.5), quad, *a);
    } else {
        form_C();
    }
    // P- = L D L^T (L unit lower triangular)
    Real L[n][n], D[n], dinv[n];
#pragma unroll
    for (int j = 0; j < n; ++j) {
        Real e[n];  // e[k] = L[j][k] D[k]
#pragma unroll
        for (int k = 0; k < j; ++k) e[k] = L[j][k] * D[k];
        Real dj = Pm[tri(rts_gi<G>(j), rts_gi<G>(j))];
#pragma unroll
        for (int k = 0; k < j; ++k) dj = fnma_(e[k], L[j][k], dj);
        note_bad_pivot(dj, status, OPTI_KF_ST_SMOOTH_NOT_PD);
        D[j] = dj;
        dinv[j] = rcp_(dj);
#pragma unroll
        for (int i = j + 1; i < n; ++i) {
            Real s = Pm[tri(rts_gi<G>(i), rts_gi<G>(j))];
#pragma unroll
            for (int k = 0; k < j; ++k) s = fnma_(L[i][k], e[k], s);
            L[i][j] = s * dinv[j];
        }
    }
    if constexpr (kStats) {
        // Sw: E[w_t w_t^T | Z] = Q + Q M (dPs + d d^T) M Q with M = (P-)^-1, so E[w_i^2 | Z] = q_i + q_i^2 ((M dPs M)_ii + (M d)_i^2).
        // (The form I - F G of Q M cancels when q << P-; this one gives exactly 0 for q_i = 0.)  Column u of M from the L D L^T
        // factor: m = L^-T D^-1 L^-1 e_u.
#pragma unroll
        for (int u = 0; u < n; ++u) {
            Real f[n], m[n];
#pragma unroll
            for (int k = u + 1; k < n; ++k) {  // L f = e_u: f_u = 1, f_k = 0 for k < u
                Real s = -L[k][u];
#pragma unroll
                for (int j = u + 1; j < k; ++j) s = fnma_(L[k][j], f[j], s);
                f[k] = s;
            }
#pragma unroll
            for (int k = n - 1; k >= 0; --k) {
                Real s;
                if (k > u) s = f[k] * dinv[k];
                else if (k == u) s = dinv[k];
                else s = -(L[k + 1][k] * m[k + 1]);
#pragma unroll
                for (int j = (k < u ? k + 2 : k + 1); j < n; ++j) s = fnma_(L[j][k], m[j], s);
                m[k] = s;
            }
            Real md = m[0] * d[rts_gi<G>(0)], quad = Real(0);
#pragma unroll
            for (int k = 1; k < n; ++k) md = fma_(m[k], d[rts_gi<G>(k)], md);
#pragma unroll
            for (int k = 0; k < n; ++k) {  // m^T dPs m on the lower triangle
                Real h = dl(k, k) * m[k];
                if (k > 0) {
                    Real o = dl(k, 0) * m[0];
#pragma unroll
                    for (int l = 1; l < k; ++l) o = fma_(dl(k, l), m[l], o);
                    h = fma_(Real(2), o, h);
                }
                quad = fma_(m[k], h, quad);
            }
            const int c = rts_gi<G>(u);
            const Real qc = em->q[c * em->nt];
            Real *a = em->acc + c * em->nt;
            *a += fma_(qc * qc, fma_(md, md, quad), qc);
        }
        form_C();
    }
    // G^T = (P-)^-1 C, column by column
#pragma unroll
    for (int v = 0; v < n; ++v) {
#pragma unroll
        for (int u = 1; u < n; ++u)
#pragma unroll
            for (int k = 0; k < u; ++k) Gt[u][v] = fnma_(L[u][k], Gt[k][v], Gt[u][v]);
#pragma unroll
        for (int u = 0; u < n; ++u) Gt[u][v] *= dinv[u];
#pragma unroll
        for (int u = n - 2; u >= 0; --u)
#pragma unroll
            for (int k = u + 1; k < n; ++k) Gt[u][v] = fnma_(L[k][u], Gt[k][v], Gt[u][v]);
    }
    // xs_t = x+_t + G d
#pragma unroll
    for (int v = 0; v < n; ++v) {
        Real s = xp[rts_gi<G>(v)];
#pragma unroll
        for (int u = 0; u < n; ++u) s = fma_(Gt[u][v], d[rts_gi<G>(u)], s);
        xs[rts_gi<G>(v)] = s;
    }
    // Ps_t = P+_t + G dPs G^T, lower triangle, column j at a time: w = dPs G^T[:, j], then Ps(i, j) = P+(i, j) + G^T[:, i] . w
#pragma unroll
    for (int j = 0; j < n; ++j) {
        Real w[n];
#pragma unroll
        for (int k = 0; k < n; ++k) {
            Real s = dl(k, 0) * Gt[0][j];
#pragma unroll
            for (int l = 1; l < n; ++l) s = fma_(dl(k, l), Gt[l][j], s);
            w[k] = s;
        }
#pragma unroll
        for (int i = j; i < n; ++i) {
            Real s = pp(i, j);
#pragma unroll
            for (int k = 0; k < n; ++k) s = fma_(Gt[k][i], w[k], s);
            Pp[tri(rts_gi<G>(i), rts_gi<G>(j))] = s;  // P+(i, j) is not read again: accumulate in place
        }
    }
#pragma unroll
    for (int j = 0; j < n; ++j)
#pragma unroll
        for (int i = j; i < n; ++i) Dl[tri(rts_gi<G>(i), rts_gi<G>(j))] = Pp[tri(rts_gi<G>(i), rts_gi<G>(j))];
}

// kStats: the E-step of EM besides (or instead of) the smoothed estimates.  The recursion runs one step further, t = -1, with
// x+ = x0 and P+ = P0: x_{-1} ~ N(x0, P0) is the state before the first predict, and w_{-1} the first transition's noise
// (DESIGN.md section 0).  The step at t adds the terms of w_t and of the measurement of step t + 1: Sw and Sv in the 23
// accumulators, log N(z_{t+1}; H x-_{t+1}, H P-_{t+1} H^T + R) in the last one and in the determinant product.
template <typename Real, bool kStats>
__global__ void __launch_bounds__(RTS_THREADS) kf_rts_kernel(const __grid_constant__ SmoothParams<Real> prm) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int nt = RTS_THREADS;
    constexpr int stage_rows = kStats ? EM_STAGE_ROWS : RTS_STAGE_ROWS;
    Real *q = reinterpret_cast<Real *>(smem_raw) + threadIdx.x;  // [12][nt]
    Real *stage = q + NX * nt;                                     // [54][nt]: this thread's next step (+ z_{t+1}: [64][nt])
    const long long i = (long long)blockIdx.x * nt + threadIdx.x;
    if (i >= prm.N) return;  // no block-wide barrier below
    const long long N = prm.N, T = prm.T;
    if (T <= 0) return;
#pragma unroll
    for (int c = 0; c < NX; ++c) q[c * nt] = prm.q_kind == OPTI_KF_MAT_DIAG ? prm.Q[c] : prm.Q[c * N + i];
    const Real *zs = nullptr;  // z of this trajectory's stream
    EmState<Real> em;
    if constexpr (kStats) {
        zs = prm.z + (prm.stream_index ? (long long)prm.stream_index[i] : (i + prm.stream_offset) % prm.S);
        em.q = q;
        em.y = stage + stage_rows * nt;
        em.acc = em.y + NZ * nt;
        em.nt = nt;
        em.R = prm.R; em.r_kind = prm.r_kind; em.N = N; em.i = i;
#pragma unroll
        for (int c = 0; c < EM_STATS_ROWS; ++c) em.acc[c * nt] = Real(0);
        em.det_m = Real(1); em.det_e = 0;
    }

    // x-_{t+1} (and z_{t+1}) behind x+_t and P+_t in the stage
    const auto issue_next = [&](long long t) {
        const Real *src = prm.x_prior + (t + 1) * NX * N + i;
#pragma unroll 1
        for (int c = 0; c < NX; ++c, src += N) cp_async_elem(stage + (NX + NPB + c) * nt, src);
        if constexpr (kStats) {
            src = zs + (t + 1) * NZ * prm.S;
#pragma unroll 1
            for (int c = 0; c < NZ; ++c, src += prm.S) cp_async_elem(stage + (RTS_STAGE_ROWS + c) * nt, src);
        }
    };
    // x+_t, P+_t and (t + 1 < T) x-_{t+1} into the stage; [t][c][N] rows, coalesced across the warp
    // (rolled loops: the copies are asynchronous, and unrolled they would keep 54 row addresses live next to the recursion)
    const auto issue = [&](long long t) {
        const Real *src = prm.x_post + t * NX * N + i;
#pragma unroll 1
        for (int c = 0; c < NX; ++c, src += N) cp_async_elem(stage + c * nt, src);
        src = prm.P_post + t * NPB * N + i;
#pragma unroll 1
        for (int k = 0; k < NPB; ++k, src += N) cp_async_elem(stage + (NX + k) * nt, src);
        if (t + 1 < T) issue_next(t);
        cp_async_commit();
    };
    // the step t = -1 (E-step only): x0 and the decoupled entries of P0 (Q when absent), then x-_0 and z_0
    const auto issue_prior = [&] {
#pragma unroll 1
        for (int c = 0; c < NX; ++c) stage[c * nt] = prm.x0[c * prm.x0_ld + i * prm.x0_inc];
#pragma unroll
        for (int a = 0; a < NX; ++a)
#pragma unroll
            for (int b = 0; b <= a; ++b) {
                if (!cpl<true>(a, b)) continue;
                Real v = Real(0);
                switch (prm.p0_kind) {
                    case OPTI_KF_MAT_NONE: v = (a == b) ? q[a * nt] : Real(0); break;
                    case OPTI_KF_MAT_DIAG: v = (a == b) ? prm.P0[a] : Real(0); break;
                    case OPTI_KF_MAT_DIAG_PER: v = (a == b) ? prm.P0[a * N + i] : Real(0); break;
                    case OPTI_KF_MAT_DENSE: v = prm.P0[a * NX + b]; break;
                    default: v = prm.P0[(long long)(a * NX + b) * N + i]; break;
                }
                stage[(NX + pk_slot(a, b)) * nt] = v;
            }
        issue_next(-1);
        cp_async_commit();
    };
    const auto store = [&](long long t, const Real (&xs)[NX], const Real (&Ps)[NP]) {
        if (!kStats || prm.x_smooth) {  // optional for the E-step
#pragma unroll
            for (int c = 0; c < NX; ++c) st_stream(prm.x_smooth + (t * NX + c) * N + i, xs[c]);
        }
        if (prm.var_smooth) {
#pragma unroll
            for (int c = 0; c < NX; ++c) st_stream(prm.var_smooth + (t * NX + c) * N + i, Ps[tri(c, c)]);
        }
    };
    // the coupled entries of a packed P from the stage (entries across groups are never read)
    const auto load_P = [&](Real (&P)[NP]) {
#pragma unroll
        for (int a = 0; a < NX; ++a)
#pragma unroll
            for (int b = 0; b <= a; ++b) P[tri(a, b)] = cpl<true>(a, b) ? stage[(NX + pk_slot(a, b)) * nt] : Real(0);
    };

    Real xs[NX], Ps[NP];  // smoothed state and covariance of step t + 1
    issue(T - 1);
    cp_async_wait_all();
#pragma unroll
    for (int c = 0; c < NX; ++c) xs[c] = stage[c * nt];
    load_P(Ps);
    if (T >= 2) issue(T - 2);
    else if constexpr (kStats) issue_prior();
    store(T - 1, xs, Ps);

    uint32_t status[1] = {0};
    for (long long t = T - 2; t >= (kStats ? -1 : 0); --t) {
        cp_async_wait_all();
        Real xp[NX], Pp[NP], d[NX];
#pragma unroll
        for (int c = 0; c < NX; ++c) xp[c] = stage[c * nt];
        load_P(Pp);
#pragma unroll
        for (int c = 0; c < NX; ++c) d[c] = xs[c] - stage[(NX + NPB + c) * nt];
        if constexpr (kStats) {  // Sv and the innovation of the measurement of step t + 1
#pragma unroll
            for (int k = 0; k < NZ; ++k) {
                const Real zk = stage[(RTS_STAGE_ROWS + k) * nt];
                const Real e = zk - xs[sel(k)];
                em.acc[(NX + k) * nt] += fma_(e, e, Ps[tri(sel(k), sel(k))]);
                em.y[k * nt] = zk - stage[(NX + NPB + sel(k)) * nt];
            }
        }
        if (t > 0) issue(t - 1);  // the stage has been read: fetch the earlier step under this one's arithmetic
        else if constexpr (kStats) {
            if (t == 0) issue_prior();
        }

        Real R[9], Pm[NP];
        rot_zyx(xp[0], xp[1], xp[2], R);  // the rotation step t + 1's predict used
#pragma unroll
        for (int k = 0; k < NP; ++k) Pm[k] = Pp[k];
        cov_predict_sym<true>(Pm, R, prm.dt, q, nt);
#pragma unroll
        for (int a = 0; a < NX; ++a)
#pragma unroll
            for (int b = 0; b <= a; ++b)
                if (cpl<true>(a, b)) Ps[tri(a, b)] -= Pm[tri(a, b)];
        Real A[9];  // dt R^T, as in cov_predict_sym
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int k = 0; k < 3; ++k) A[3 * r + k] = prm.dt * R[3 * k + r];
        rts_group<1, kStats>(xp, Pp, Pm, Ps, d, A, prm.dt, xs, status, &em);
        rts_group<2, kStats>(xp, Pp, Pm, Ps, d, A, prm.dt, xs, status, &em);
        rts_group<3, kStats>(xp, Pp, Pm, Ps, d, A, prm.dt, xs, status, &em);
        rts_group<0, kStats>(xp, Pp, Pm, Ps, d, A, prm.dt, xs, status, &em);
        if (!kStats || t >= 0) store(t, xs, Ps);
    }
    if constexpr (kStats) {
        const bool bad = status[0] & EM_BAD_PIVOT;
        status[0] &= ~EM_BAD_PIVOT;
#pragma unroll 1
        for (int c = 0; c < EM_STATS_ROWS - 1; ++c) prm.stats[c * N + i] = em.acc[c * nt];
        // log-likelihood: -0.5 (10 T log 2 pi + log det) + the accumulated -0.5 y^T S^-1 y
        const double log_det = log((double)em.det_m) + (double)em.det_e * 0.69314718055994530942;
        const double ll = (double)em.acc[(EM_STATS_ROWS - 1) * nt] - 0.5 * (log_det + (double)(NZ * T) * 1.83787706640934548356);
        prm.stats[(EM_STATS_ROWS - 1) * N + i] = bad ? Real(NAN) : (Real)ll;
    }
    if (status[0] && prm.status) prm.status[i] |= status[0];
}

// Launch of kf_rts_kernel<Real, kStats> (instantiated in kf_smooth.cu for double and float).
template <typename Real, bool kStats>
int launch_rts(const SmoothParams<Real> &p, cudaStream_t stream);

}  // namespace okf
