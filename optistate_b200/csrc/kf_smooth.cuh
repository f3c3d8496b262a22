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
};

constexpr int RTS_THREADS = 64;
constexpr int RTS_STAGE_ROWS = NX + NPB + NX;  // x+_t, P+_t, x-_{t+1}
constexpr int RTS_SMEM_ROWS = NX + RTS_STAGE_ROWS;  // q, then the staged step

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

// One decoupled group of the backward step.  In: P+ (Pp, destroyed), the recomputed P- (Pm), dPs = Ps_{t+1} - P- (Dl),
// d = xs_{t+1} - x-_{t+1}.  Out: xs_t into xs, Ps_t into Dl (both for this group's entries only).  A = dt R^T (group 0).
template <int G, typename Real>
__device__ __forceinline__ void rts_group(const Real (&xp)[NX], Real (&Pp)[NP], Real (&Pm)[NP], Real (&Dl)[NP], const Real (&d)[NX],
                                          const Real (&A)[9], Real dt, Real (&xs)[NX], uint32_t (&status)[1]) {
    constexpr int n = G == 0 ? 6 : 2, h = n / 2;
    const auto pp = [&](int u, int v) { return Pp[tri(rts_gi<G>(u), rts_gi<G>(v))]; };
    // C = F P+ on the group: F = [[I, Fo], [0, I]], Fo = dt R^T (attitude rows on body rate) or dt (position on velocity)
    Real Gt[n][n];
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
    const auto dl = [&](int k, int l) { return Dl[tri(rts_gi<G>(k), rts_gi<G>(l))]; };
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

template <typename Real>
__global__ void __launch_bounds__(RTS_THREADS) kf_rts_kernel(const __grid_constant__ SmoothParams<Real> prm) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int nt = RTS_THREADS;
    Real *q = reinterpret_cast<Real *>(smem_raw) + threadIdx.x;  // [12][nt]
    Real *stage = q + NX * nt;                                     // [54][nt]: this thread's next step
    const long long i = (long long)blockIdx.x * nt + threadIdx.x;
    if (i >= prm.N) return;  // no block-wide barrier below
    const long long N = prm.N, T = prm.T;
    if (T <= 0) return;
#pragma unroll
    for (int c = 0; c < NX; ++c) q[c * nt] = prm.q_kind == OPTI_KF_MAT_DIAG ? prm.Q[c] : prm.Q[c * N + i];

    // x+_t, P+_t and (t + 1 < T) x-_{t+1} into the stage; [t][c][N] rows, coalesced across the warp
    // (rolled loops: the copies are asynchronous, and unrolled they would keep 54 row addresses live next to the recursion)
    const auto issue = [&](long long t) {
        const Real *src = prm.x_post + t * NX * N + i;
#pragma unroll 1
        for (int c = 0; c < NX; ++c, src += N) cp_async_elem(stage + c * nt, src);
        src = prm.P_post + t * NPB * N + i;
#pragma unroll 1
        for (int k = 0; k < NPB; ++k, src += N) cp_async_elem(stage + (NX + k) * nt, src);
        if (t + 1 < T) {
            src = prm.x_prior + (t + 1) * NX * N + i;
#pragma unroll 1
            for (int c = 0; c < NX; ++c, src += N) cp_async_elem(stage + (NX + NPB + c) * nt, src);
        }
        cp_async_commit();
    };
    const auto store = [&](long long t, const Real (&xs)[NX], const Real (&Ps)[NP]) {
#pragma unroll
        for (int c = 0; c < NX; ++c) st_stream(prm.x_smooth + (t * NX + c) * N + i, xs[c]);
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
    store(T - 1, xs, Ps);

    uint32_t status[1] = {0};
    for (long long t = T - 2; t >= 0; --t) {
        cp_async_wait_all();
        Real xp[NX], Pp[NP], d[NX];
#pragma unroll
        for (int c = 0; c < NX; ++c) xp[c] = stage[c * nt];
        load_P(Pp);
#pragma unroll
        for (int c = 0; c < NX; ++c) d[c] = xs[c] - stage[(NX + NPB + c) * nt];
        if (t > 0) issue(t - 1);  // the stage has been read: fetch the earlier step under this one's arithmetic

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
        rts_group<1>(xp, Pp, Pm, Ps, d, A, prm.dt, xs, status);
        rts_group<2>(xp, Pp, Pm, Ps, d, A, prm.dt, xs, status);
        rts_group<3>(xp, Pp, Pm, Ps, d, A, prm.dt, xs, status);
        rts_group<0>(xp, Pp, Pm, Ps, d, A, prm.dt, xs, status);
        store(t, xs, Ps);
    }
    if (status[0] && prm.status) prm.status[i] |= status[0];
}

// Launch of kf_rts_kernel (instantiated in kf_smooth.cu for double and float).
template <typename Real>
int launch_rts(const SmoothParams<Real> &p, cudaStream_t stream);

}  // namespace okf
