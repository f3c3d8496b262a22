// Adjoint (reverse-mode gradient) of the SEQUENTIAL filter of the predict() model with respect to diagonal Q, R, x0 and P0
// (DESIGN.md section 0.4).  The forward step t = 0 .. T-1, from x+_{-1} = x0, P+_{-1} = P0 (Q when absent), in its joint form
//     x-_t = f(x+_{t-1}; C_t, fs_t)      F_t = I + dt N(R(th+_{t-1}))      P-_t = F_t P+_{t-1} F_t^T + Q
//     y_t = z_t - H x-_t   S_t = H P-_t H^T + R   K_t = P-_t H^T S_t^-1   A_t = I - K_t H   v_t = S_t^-1 y_t
//     x+_t = x-_t + K_t y_t                P+_t = A_t P-_t
// which the sequential update computes in exact arithmetic (DESIGN.md section 2).  Given xb_t = dL/dx+_t, from a = 0, Pi = 0,
// for t = T-1 .. 0:
//     a += xb_t;  b = K^T a;  rb_k += (K^T Pi K)_kk - b_k v_k;  Pb = A^T Pi A + sym(A^T a v^T H);  qb_i += Pb_ii
//     Pi = F^T Pb F;  a = J^T (A^T a) + (th-term of F: thb_m += dt sum_jk B_jk dR_kj/dth_m,  B = (2 Pb F P+_{t-1})[0:3, 6:9])
// and at the end xb0 = a, Pb0 = Pi.  J_t = dx-_t/dx+_{t-1} is the derivative of the formula the filter kernels evaluate
// (propagate_mean_from_moments): dth'/dw = dt trunc(R^T) (only where the truncation fires), dr'/dv = dt I and dw'/dth from
// w' = w + R diag(dt / I_b) g(R), g_i = eps_ijk (C R)_jk.  trunc(R^T) is piecewise constant: at exactly axis-aligned attitudes
// the filter is discontinuous in th and this is the almost-everywhere derivative.
//
//   * Perturbing a diagonal Q, R or P0, or x0, never moves P off the decoupled-group structure (F is group-block-diagonal), so
//     the cross-group entries of Pb meet zero perturbations only and are dropped: Pi is the 30 packed entries P+ has, and the
//     whole reverse step splits into the groups {th, w}, {x, vx}, {y, vy}, {z, vz} (kf_seq_core.cuh).  In {th, w} and {z, vz}
//     every state is measured, so A = diag(r) S^-1; in {x, vx} and {y, vy} only the velocity is, and S is a scalar.
//   * One thread per trajectory, reverse time loop; a (12) and Pi (30) live in registers.  P-_t is recomputed with the forward
//     pass's own rot_zyx + cov_predict_sym<true>; per group one L D L^T of S_t with rcp_ pivots.
//   * The inputs of the next (earlier) step - th+_{t-2}, P+_{t-2}, x-_{t-1}, xb_{t-1}, z_{t-1}, C_{t-1} - are copied to shared
//     memory with cp.async before the current step's arithmetic starts, as in kf_rts_kernel.  q, r and the 22 accumulators of
//     qb, rb are shared-memory columns, as in EmState.
//   * A pivot of S_t that is not positive and finite sets OPTI_KF_ST_SMOOTH_NOT_PD; the recursion carries on.
#pragma once

#include "kf_smooth.cuh"

namespace okf {

template <typename Real>
struct AdjointParams {
    long long N, T;
    Real dt, dt_inv_inertia[3];  // dt / I_b, rounded as the filter kernels round it
    const Real *Q; int q_kind;   // OPTI_KF_MAT_DIAG [12] or OPTI_KF_MAT_DIAG_PER [12][N]
    const Real *R; int r_kind;   // OPTI_KF_MAT_DIAG [10] or OPTI_KF_MAT_DIAG_PER [10][N]
    const Real *x0; long long x0_ld; int x0_inc;
    const Real *P0; int p0_kind;  // as in Params (decoupled): NONE = Q
    const Real *x_post;          // [T][12][N] x+
    const Real *x_prior;         // [T][12][N] x-
    const Real *P_post;          // [T][30][N] packed P+
    const Real *x_bar;           // [T][12][N] dL/dx+
    const Real *z;               // [T][10][S] and
    const Real *mom;             // [T][12][S] leg moments (rows 0-8 used): trajectory i reads stream stream_index[i] or (i + stream_offset) % S
    long long S, stream_offset;
    const int32_t *stream_index;
    Real *grad;                  // [OPTI_KF_ADJ_ROWS][N]
    uint32_t *status;            // [N] or NULL: OPTI_KF_ST_SMOOTH_NOT_PD is OR-ed in
};

constexpr int ADJ_THREADS = 64;
// stage of one reverse step t: th+_{t-1} (3), P+_{t-1} (30), x-_t at the measured states (10), xb_t (12), z_t (10), C_t (9)
constexpr int ADJ_TH = 0, ADJ_P = 3, ADJ_XM = ADJ_P + NPB, ADJ_XB = ADJ_XM + NZ, ADJ_Z = ADJ_XB + NX, ADJ_C = ADJ_Z + NZ;
constexpr int ADJ_STAGE_ROWS = ADJ_C + 9;
constexpr int ADJ_ACC_ROWS = NX + NZ;  // qb, rb
constexpr int ADJ_SMEM_ROWS = NX + NZ + ADJ_ACC_ROWS + ADJ_STAGE_ROWS;  // q, r, accumulators, stage

// The reverse step of one decoupled group G.  Pp: P+_{t-1}; Pm: P-_t; Pi: dL/dP+_t in, dL/dP+_{t-1} out; a: dL/dx+_t (with
// xb_t added) in, the group's entries of dL/dx+_{t-1} out; y: the innovation z_t - H x-_t.  Ao = dt R^T, Jw[3i + m] = dw'_i/dth_m,
// dR[9m + 3k + j] = dR_kj/dth_m, Tm = trunc(R^T) when any_trunc (group 0 only).
template <int G, typename Real>
__device__ __forceinline__ void adj_group(const Real (&Pp)[NP], const Real (&Pm)[NP], Real (&Pi)[NP], Real (&a)[NX], const Real (&y)[NZ],
                                          const Real (&Ao)[9], const Real (&Jw)[9], const Real (&dR)[27], const Real (&Tm)[9],
                                          bool any_trunc, Real dt, const Real *r, Real *acc, int nt, uint32_t (&status)[1]) {
    constexpr int n = G == 0 ? 6 : 2, h = n / 2;
    constexpr int m = G == 0 ? 6 : G == 3 ? 2 : 1, m0 = (G == 1 || G == 2) ? 1 : 0;  // measured: local m0 .. m0 + m - 1
    const auto gi = [](int u) { return rts_gi<G>(u); };
    const auto pm = [&](int u, int v) { return Pm[tri(gi(u), gi(v))]; };
    const auto pi = [&](int u, int v) { return Pi[tri(gi(u), gi(v))]; };
    const auto fo = [&](int u, int w) { return G == 0 ? Ao[3 * u + w] : dt; };  // F = [[I, Fo], [0, I]] on the group
    // S = P-[M, M] + R = L D L^T, then S^-1 column by column
    Real L[m][m], D[m], dinv[m];
#pragma unroll
    for (int j = 0; j < m; ++j) {
        Real e[m];  // e[k] = L[j][k] D[k]
#pragma unroll
        for (int k = 0; k < j; ++k) e[k] = L[j][k] * D[k];
        Real dj = pm(m0 + j, m0 + j) + r[em_row<G>(m0 + j) * nt];
#pragma unroll
        for (int k = 0; k < j; ++k) dj = fnma_(e[k], L[j][k], dj);
        note_bad_pivot(dj, status, OPTI_KF_ST_SMOOTH_NOT_PD);
        D[j] = dj;
        dinv[j] = rcp_(dj);
#pragma unroll
        for (int i = j + 1; i < m; ++i) {
            Real s = pm(m0 + i, m0 + j);
#pragma unroll
            for (int k = 0; k < j; ++k) s = fnma_(L[i][k], e[k], s);
            L[i][j] = s * dinv[j];
        }
    }
    Real Si[m][m];
#pragma unroll
    for (int c = 0; c < m; ++c) {
        Real f[m];
#pragma unroll
        for (int k = 0; k < m; ++k) {  // L f = e_c
            Real s = k == c ? Real(1) : Real(0);
#pragma unroll
            for (int j = c; j < k; ++j) s = fnma_(L[k][j], f[j], s);
            f[k] = k < c ? Real(0) : s;
        }
#pragma unroll
        for (int k = m - 1; k >= 0; --k) {  // L^T s = D^-1 f
            Real s = f[k] * dinv[k];
#pragma unroll
            for (int j = k + 1; j < m; ++j) s = fnma_(L[j][k], Si[j][c], s);
            Si[k][c] = s;
        }
    }
    // A = I - K H and K = P-[:, M] S^-1; all measured: A = diag(r) S^-1, K = I - A
    Real A[n][n], Kp[n][m];
    if constexpr (m == n) {
#pragma unroll
        for (int i = 0; i < n; ++i)
#pragma unroll
            for (int j = 0; j < n; ++j) A[i][j] = r[em_row<G>(i) * nt] * Si[i][j];
    } else {
#pragma unroll
        for (int i = 0; i < n; ++i)
#pragma unroll
            for (int j = 0; j < m; ++j) {
                Real s = pm(i, m0) * Si[0][j];
#pragma unroll
                for (int k = 1; k < m; ++k) s = fma_(pm(i, m0 + k), Si[k][j], s);
                Kp[i][j] = s;
            }
#pragma unroll
        for (int i = 0; i < n; ++i)
#pragma unroll
            for (int j = 0; j < n; ++j) A[i][j] = (i == j ? Real(1) : Real(0)) - (j >= m0 && j < m0 + m ? Kp[i][j - m0] : Real(0));
    }
    const auto K = [&](int i, int j) -> Real {
        if constexpr (m == n) return (i == j ? Real(1) : Real(0)) - A[i][j];
        else return Kp[i][j];
    };
    // v = S^-1 y, b = K^T a, at = A^T a
    Real v[m], b[m], at[n];
#pragma unroll
    for (int j = 0; j < m; ++j) {
        Real s = Real(0), u = Real(0);
#pragma unroll
        for (int k = 0; k < m; ++k) s = fma_(Si[j][k], y[em_row<G>(m0 + k)], s);
#pragma unroll
        for (int i = 0; i < n; ++i) u = fma_(K(i, j), a[gi(i)], u);
        v[j] = s;
        b[j] = u;
    }
#pragma unroll
    for (int j = 0; j < n; ++j) {
        Real s = Real(0);
#pragma unroll
        for (int i = 0; i < n; ++i) s = fma_(A[i][j], a[gi(i)], s);
        at[j] = s;
    }
    // rb_k += (K^T Pi K)_kk - b_k v_k
#pragma unroll
    for (int j = 0; j < m; ++j) {
        Real s = -(b[j] * v[j]);
#pragma unroll
        for (int i = 0; i < n; ++i) {
            Real w = Real(0);
#pragma unroll
            for (int k = 0; k < n; ++k) w = fma_(pi(i, k), K(k, j), w);
            s = fma_(K(i, j), w, s);
        }
        acc[(NX + em_row<G>(m0 + j)) * nt] += s;
    }
    // Pb = A^T Pi A + sym(at w^T), w = H^T v (full symmetric n x n), column j at a time
    Real Pb[n][n];
#pragma unroll
    for (int j = 0; j < n; ++j) {
        Real w[n];
#pragma unroll
        for (int k = 0; k < n; ++k) {
            Real s = Real(0);
#pragma unroll
            for (int l = 0; l < n; ++l) s = fma_(pi(k, l), A[l][j], s);
            w[k] = s;
        }
#pragma unroll
        for (int i = j; i < n; ++i) {
            Real s = Real(0);
#pragma unroll
            for (int k = 0; k < n; ++k) s = fma_(A[k][i], w[k], s);
            const Real vi = (i >= m0 && i < m0 + m) ? v[i - m0] : Real(0), vj = (j >= m0 && j < m0 + m) ? v[j - m0] : Real(0);
            s = fma_(Real(0.5), fma_(at[i], vj, vi * at[j]), s);
            Pb[i][j] = s;
            Pb[j][i] = s;
        }
    }
#pragma unroll
    for (int i = 0; i < n; ++i) acc[gi(i) * nt] += Pb[i][i];
    // a = J^T at (+ the th-term of F in group 0)
    if constexpr (G == 0) {
        // B = (2 Pb C)[th, w] with C = F P+_{t-1}: C[k][3 + l] = P+(k, 3 + l) + (k < 3 ? sum_w Ao[3k + w] P+(3 + w, 3 + l) : 0)
        const auto pp = [&](int u, int v) { return Pp[tri(gi(u), gi(v))]; };
        Real C[n][3];
#pragma unroll
        for (int k = 0; k < n; ++k)
#pragma unroll
            for (int l = 0; l < 3; ++l) {
                Real s = pp(k, 3 + l);
                if (k < 3) {
#pragma unroll
                    for (int w = 0; w < 3; ++w) s = fma_(Ao[3 * k + w], pp(3 + w, 3 + l), s);
                }
                C[k][l] = s;
            }
        Real th[3];
#pragma unroll
        for (int mm = 0; mm < 3; ++mm) {
            Real s = at[mm];
#pragma unroll
            for (int i = 0; i < 3; ++i) s = fma_(Jw[3 * i + mm], at[3 + i], s);
            th[mm] = s;
        }
#pragma unroll
        for (int j = 0; j < 3; ++j)
#pragma unroll
            for (int l = 0; l < 3; ++l) {
                Real s = Real(0);
#pragma unroll
                for (int k = 0; k < n; ++k) s = fma_(Pb[j][k], C[k][l], s);
                s *= Real(2) * dt;  // dF[j][3 + l] = dt dR[l][j]
#pragma unroll
                for (int mm = 0; mm < 3; ++mm) th[mm] = fma_(s, dR[9 * mm + 3 * l + j], th[mm]);
            }
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            Real s = at[3 + k];
            if (any_trunc) {
#pragma unroll
                for (int i = 0; i < 3; ++i) s = fma_(dt * Tm[3 * i + k], at[i], s);
            }
            a[gi(3 + k)] = s;
            a[gi(k)] = th[k];
        }
    } else {
        a[gi(0)] = at[0];
        a[gi(1)] = fma_(dt, at[0], at[1]);
    }
    // Pi = F^T Pb F on the lower triangle: (F^T Pb F)_ij = Pb_ij + [j >= h] (Pb Fo)_i,j-h + [i >= h] (Fo^T Pb F)_i-h,j
#pragma unroll
    for (int j = 0; j < n; ++j) {
        Real w[n];  // column j of Pb F
#pragma unroll
        for (int k = 0; k < n; ++k) {
            Real s = Pb[k][j];
            if (j >= h) {
#pragma unroll
                for (int l = 0; l < h; ++l) s = fma_(Pb[k][l], fo(l, j - h), s);
            }
            w[k] = s;
        }
#pragma unroll
        for (int i = j; i < n; ++i) {
            Real s = w[i];
            if (i >= h) {
#pragma unroll
                for (int l = 0; l < h; ++l) s = fma_(fo(l, i - h), w[l], s);
            }
            Pi[tri(gi(i), gi(j))] = s;
        }
    }
}

template <typename Real>
__global__ void __launch_bounds__(ADJ_THREADS) kf_adjoint_kernel(const __grid_constant__ AdjointParams<Real> prm) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int nt = ADJ_THREADS;
    Real *q = reinterpret_cast<Real *>(smem_raw) + threadIdx.x;  // [12][nt]
    Real *r = q + NX * nt;                                         // [10][nt]
    Real *acc = r + NZ * nt;                                       // [22][nt]: qb, rb
    Real *stage = acc + ADJ_ACC_ROWS * nt;                         // [74][nt]
    const long long i = (long long)blockIdx.x * nt + threadIdx.x;
    if (i >= prm.N) return;  // no block-wide barrier below
    const long long N = prm.N, T = prm.T;
    if (T <= 0) return;
#pragma unroll
    for (int c = 0; c < NX; ++c) q[c * nt] = prm.q_kind == OPTI_KF_MAT_DIAG ? prm.Q[c] : prm.Q[c * N + i];
#pragma unroll
    for (int c = 0; c < NZ; ++c) r[c * nt] = prm.r_kind == OPTI_KF_MAT_DIAG ? prm.R[c] : prm.R[c * N + i];
#pragma unroll
    for (int c = 0; c < ADJ_ACC_ROWS; ++c) acc[c * nt] = Real(0);
    const long long s = prm.stream_index ? (long long)prm.stream_index[i] : (i + prm.stream_offset) % prm.S;
    const Real *zs = prm.z + s, *ms = prm.mom + s;

    // the inputs of reverse step t; for t = 0, x0 and the decoupled entries of P0 (Q when absent) are written directly
    const auto issue = [&](long long t) {
        const Real *src;
        if (t > 0) {
            src = prm.x_post + (t - 1) * NX * N + i;
#pragma unroll 1
            for (int c = 0; c < 3; ++c, src += N) cp_async_elem(stage + (ADJ_TH + c) * nt, src);
            src = prm.P_post + (t - 1) * NPB * N + i;
#pragma unroll 1
            for (int k = 0; k < NPB; ++k, src += N) cp_async_elem(stage + (ADJ_P + k) * nt, src);
        } else {
#pragma unroll 1
            for (int c = 0; c < 3; ++c) stage[(ADJ_TH + c) * nt] = prm.x0[c * prm.x0_ld + i * prm.x0_inc];
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
                    stage[(ADJ_P + pk_slot(a, b)) * nt] = v;
                }
        }
        src = prm.x_prior + t * NX * N + i;
#pragma unroll 1
        for (int k = 0; k < NZ; ++k) cp_async_elem(stage + (ADJ_XM + k) * nt, src + sel(k) * N);
        src = prm.x_bar + t * NX * N + i;
#pragma unroll 1
        for (int c = 0; c < NX; ++c, src += N) cp_async_elem(stage + (ADJ_XB + c) * nt, src);
        src = zs + t * NZ * prm.S;
#pragma unroll 1
        for (int k = 0; k < NZ; ++k, src += prm.S) cp_async_elem(stage + (ADJ_Z + k) * nt, src);
        src = ms + t * NM * prm.S;
#pragma unroll 1
        for (int k = 0; k < 9; ++k, src += prm.S) cp_async_elem(stage + (ADJ_C + k) * nt, src);
        cp_async_commit();
    };

    Real a[NX], Pi[NP];
#pragma unroll
    for (int c = 0; c < NX; ++c) a[c] = Real(0);
#pragma unroll
    for (int k = 0; k < NP; ++k) Pi[k] = Real(0);
    uint32_t status[1] = {0};
    issue(T - 1);
    for (long long t = T - 1; t >= 0; --t) {
        cp_async_wait_all();
        Real th[3], Pp[NP], y[NZ], Cm[9];
#pragma unroll
        for (int c = 0; c < 3; ++c) th[c] = stage[(ADJ_TH + c) * nt];
#pragma unroll
        for (int u = 0; u < NX; ++u)
#pragma unroll
            for (int v = 0; v <= u; ++v) Pp[tri(u, v)] = cpl<true>(u, v) ? stage[(ADJ_P + pk_slot(u, v)) * nt] : Real(0);
#pragma unroll
        for (int k = 0; k < NZ; ++k) y[k] = stage[(ADJ_Z + k) * nt] - stage[(ADJ_XM + k) * nt];
#pragma unroll
        for (int c = 0; c < NX; ++c) a[c] += stage[(ADJ_XB + c) * nt];
#pragma unroll
        for (int k = 0; k < 9; ++k) Cm[k] = stage[(ADJ_C + k) * nt];
        if (t > 0) issue(t - 1);  // the stage has been read: fetch the earlier step under this one's arithmetic

        // R of the prior attitude, its derivatives, and dw'/dth of the mean model
        Real R[9], Tm[9], dR[27];
        rot_zyx(th[0], th[1], th[2], R);
        bool any_trunc = false;
        if (may_truncate(R)) trunc_rt(R, th, Tm, any_trunc);
        {
            Real sa, ca, sb, cb, sc, cc;
            sincos_full(th[0], sa, ca);
            sincos_full(th[1], sb, cb);
            sincos_full(th[2], sc, cc);
            // d/da = R X (X the generator of Rx): columns 1, 2 of R turn into (R2, -R1)
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                dR[3 * k] = Real(0);
                dR[3 * k + 1] = R[3 * k + 2];
                dR[3 * k + 2] = -R[3 * k + 1];
            }
            // d/db: rows 0, 1 are cos(c), sin(c) times (-sb, cb sa, cb ca); row 2 is (-cb, -sb sa, -sb ca)
            const Real r2[3] = {-sb, cb * sa, cb * ca};
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                dR[9 + k] = cc * r2[k];
                dR[12 + k] = sc * r2[k];
            }
            dR[15] = -cb; dR[16] = -(sb * sa); dR[17] = -(sb * ca);
            // d/dc = Z R (Z the generator of Rz): rows (-R_1, R_0, 0)
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                dR[18 + k] = -R[3 + k];
                dR[21 + k] = R[k];
                dR[24 + k] = Real(0);
            }
        }
        Real Jw[9];
        {
            // g_i(M) = sum_m C[j][m] M[m][k] - C[k][m] M[m][j], (i, j, k) cyclic; w' = w + R diag(dt / I) g(R)
            const auto g = [&](const Real *M, int ii) {
                const int j = (ii + 1) % 3, k = (ii + 2) % 3;
                Real s = Real(0);
#pragma unroll
                for (int mm = 0; mm < 3; ++mm) s = fma_(Cm[3 * j + mm], M[3 * mm + k], fnma_(Cm[3 * k + mm], M[3 * mm + j], s));
                return s;
            };
            Real u[3];
#pragma unroll
            for (int ii = 0; ii < 3; ++ii) u[ii] = g(R, ii) * prm.dt_inv_inertia[ii];
#pragma unroll
            for (int mm = 0; mm < 3; ++mm) {
                const Real *D = dR + 9 * mm;
                Real du[3];
#pragma unroll
                for (int ii = 0; ii < 3; ++ii) du[ii] = g(D, ii) * prm.dt_inv_inertia[ii];
#pragma unroll
                for (int ii = 0; ii < 3; ++ii) {
                    Real s = Real(0);
#pragma unroll
                    for (int k = 0; k < 3; ++k) s = fma_(D[3 * ii + k], u[k], fma_(R[3 * ii + k], du[k], s));
                    Jw[3 * ii + mm] = s;
                }
            }
        }
        Real Pm[NP];
#pragma unroll
        for (int k = 0; k < NP; ++k) Pm[k] = Pp[k];
        cov_predict_sym<true>(Pm, R, prm.dt, q, nt);
        Real Ao[9];  // dt R^T, as in cov_predict_sym
#pragma unroll
        for (int u = 0; u < 3; ++u)
#pragma unroll
            for (int k = 0; k < 3; ++k) Ao[3 * u + k] = prm.dt * R[3 * k + u];
        adj_group<1>(Pp, Pm, Pi, a, y, Ao, Jw, dR, Tm, any_trunc, prm.dt, r, acc, nt, status);
        adj_group<2>(Pp, Pm, Pi, a, y, Ao, Jw, dR, Tm, any_trunc, prm.dt, r, acc, nt, status);
        adj_group<3>(Pp, Pm, Pi, a, y, Ao, Jw, dR, Tm, any_trunc, prm.dt, r, acc, nt, status);
        adj_group<0>(Pp, Pm, Pi, a, y, Ao, Jw, dR, Tm, any_trunc, prm.dt, r, acc, nt, status);
    }
#pragma unroll 1
    for (int c = 0; c < ADJ_ACC_ROWS; ++c) prm.grad[c * N + i] = acc[c * nt];
#pragma unroll
    for (int c = 0; c < NX; ++c) {
        prm.grad[(ADJ_ACC_ROWS + c) * N + i] = a[c];
        prm.grad[(ADJ_ACC_ROWS + NX + c) * N + i] = Pi[tri(c, c)];
    }
    if (status[0] && prm.status) prm.status[i] |= status[0];
}

// Launch of kf_adjoint_kernel<Real> (instantiated in kf_adjoint.cu for double and float).
template <typename Real>
int launch_adjoint(const AdjointParams<Real> &p, cudaStream_t stream);

}  // namespace okf
