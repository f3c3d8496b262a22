// Arithmetic core of the SEQUENTIAL path, shared by the TMA-fed kernel (kf_seq_tma.cuh) and the direct-load kernel
// (kf_seq.cuh), with their set-up, per-step stores and epilogue; generic over Real = double | float | F2 (kf_arith.cuh).
//
//   * P is a packed symmetric matrix (78 scalars) that lives in registers for the whole time loop; x (12) too.
//   * The covariance transition F_d P F_d^T + Q (kalman_filter.py:125-135) is evaluated block-wise on the packed form in
//     the reference's W = F_d P, P' = W F_d^T order, skipping the structural zeros of F_d (168 FMAs).
//   * The update (kalman_filter.py:164-174) folds the 10 measurements in one at a time.  For diagonal R this is the same
//     Schur complement the reference evaluates jointly as P - (P H^T) S^-1 (H P): eliminating the block [[S, HP],[PH^T, P]]
//     at once or one scalar pivot after the other gives the same result (also for a non-symmetric P, because with a
//     diagonal R the pivot block of the augmented matrix is P[sel,sel] + R at every stage).  No 10x10 factorisation, no
//     square roots, no gain matrix: per measurement 1 reciprocal + 101 FMAs; row / column k of the result is the old
//     column times r/s, so the old column stays in place until the end and is never copied.
//     K_gain = sum_i K[i][i] follows from the identity K = P'[:, sel] R^-1, NIS from sum_k y_k^2 / s_k.
//   * Independent trajectories => no shuffles, no shared-memory traffic in the recursion, no redundant work.
//   * kBlock variants exploit the DECOUPLING of this particular model.  F_d = I + dt F couples only attitude <-> body rate
//     (F[0:3,6:9] = R^T) and position <-> velocity axis by axis (F[3:6,9:12] = I, kalman_filter.py:45-48), H is a selection and
//     Q, R are diagonal, so the state splits into four groups that never mix in the covariance recursion:
//         G0 = {th_x th_y th_z w_x w_y w_z} (6x6),  G1 = {x, v_x},  G2 = {y, v_y},  G3 = {z, v_z}  (2x2 each).
//     If P0 has no entries across groups (P0 = Q as settings.py:31 has it, or any diagonal P0) every cross-group entry of P is
//     an exact floating-point zero at every step of the REFERENCE too (a sum of products with one factor exactly zero; the
//     pivoted LU of a block-structured S never fills a cross entry), so dropping the terms that multiply those zeros changes
//     no bit of any other entry: 30 packed scalars instead of 78, a rank-1 update of 15 (or 1) FMAs instead of 66.  The kBlock
//     kernels are therefore bit-identical to the full ones on such inputs (tests/test_parity_gpu.py) - they skip multiplications
//     by structural zeros, which SURVEY 8(d) says never to count.  predict_mpc's element-wise exp makes F_d dense: no kBlock there.
#pragma once

#include "kf_common.cuh"

namespace okf {

__host__ __device__ constexpr int tri(int i, int j) { return i >= j ? i * (i + 1) / 2 + j : j * (j + 1) / 2 + i; }
constexpr int NP = 78;

// decoupled groups of the predict() model (see the header comment): attitude + body rate, and one (position, velocity) pair per axis
__host__ __device__ constexpr int grp(int i) { return (i < 3 || (i >= 6 && i < 9)) ? 0 : 1 + (i % 3); }
template <bool kBlock>
__host__ __device__ constexpr bool cpl(int i, int j) { return !kBlock || grp(i) == grp(j); }

// Packed per-step posterior covariance of the decoupled form (Params.P_steps, read by the smoother, kf_smooth.cuh): the 30
// entries (a, b) with b <= a and cpl<true>(a, b), in tri(a, b) order.  pk_slot is the one map the store and the load use.
constexpr int NPB = 30;
// Closed form (straight arithmetic, so it folds to a constant in the unrolled loops that use it): rows 0-2 hold 1, 2, 3 entries,
// rows 3-5 one (the diagonal), rows 6-8 4, 5, 6 (the attitude columns and their own), rows 9-11 two (position, diagonal).
__host__ __device__ constexpr int pk_row_start(int a) {
    return a < 3 ? a * (a + 1) / 2 : a < 6 ? 3 + a : a < 9 ? 9 + 4 * (a - 6) + (a - 6) * (a - 7) / 2 : 24 + 2 * (a - 9);
}
__host__ __device__ constexpr int pk_slot(int a, int b) {
    return pk_row_start(a) + (grp(a) == 0 ? (b < 3 ? b : b - 3) : (b == a && a >= 9 ? 1 : 0));
}
// the same map by enumeration, checked against the closed form at compile time
__host__ __device__ constexpr bool pk_slot_ok() {
    int n = 0;
    for (int i = 0; i < 12; ++i)
        for (int j = 0; j <= i; ++j)
            if (cpl<true>(i, j) && pk_slot(i, j) != n++) return false;
    return n == NPB;
}
static_assert(pk_slot_ok(), "pk_slot enumerates the 30 coupled entries in tri order");

// P's coupled entries of step t to dst[t][pk_slot][N] (Scalar = the array type, Real = double | float | F2)
template <typename Real, typename Scalar>
__device__ __forceinline__ void store_packed_P(Scalar *dst, long long t, long long N, long long i, const Real (&P)[NP]) {
#pragma unroll
    for (int a = 0; a < NX; ++a)
#pragma unroll
        for (int b = 0; b <= a; ++b)
            if (cpl<true>(a, b)) st_traj(dst, (t * NPB + pk_slot(a, b)) * N + i, P[tri(a, b)]);
}

// All 78 entries of P of step t to dst[t][tri(a, b)][N]: Params.P_steps of the full-covariance kernels, read by the dense
// smoother (kf_smooth_full.cuh).  Which of the two layouts a kernel writes follows from its kBlock.
template <typename Real, typename Scalar>
__device__ __forceinline__ void store_full_P(Scalar *dst, long long t, long long N, long long i, const Real (&P)[NP]) {
#pragma unroll
    for (int k = 0; k < NP; ++k) st_traj(dst, (t * NP + k) * N + i, P[k]);
}

// P <- F_d P F_d^T + diag(q), F_d = I + dt N, N[a,c] = R^T, N[b,d] = I   (blocks a=0..2 b=3..5 c=6..8 d=9..11)
// Written with explicit fma_ so that double, float and the packed F2 type run the same operation sequence.
template <bool kBlock = false, typename Real, typename Scalar>
__device__ __forceinline__ void cov_predict_sym(Real (&P)[NP], const Real (&R)[9], Scalar dt_s, const Real *q, int qs) {
    constexpr int a = 0, b = 3, c = 6, d = 9;
    const Real dt = Real(dt_s);
    Real A[9];  // A = dt R^T
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int k = 0; k < 3; ++k) A[3 * i + k] = dt * R[3 * k + i];
        // W rows that feed P'[a,a], P'[b,a], P'[b,b] use the OLD c- and d-rows: do them first.
        // (kBlock: an entry P[i][j] with cpl(i, j) false is a structural zero - neither read nor written)
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j <= i; ++j) {
            Real s = P[tri(a + i, a + j)];
#pragma unroll
            for (int k = 0; k < 3; ++k) s = fma_(A[3 * i + k], P[tri(c + k, a + j)], s);
            P[tri(a + i, a + j)] = s;
        }
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j)
            if (cpl<kBlock>(b + i, a + j)) P[tri(b + i, a + j)] = fma_(dt, P[tri(d + i, a + j)], P[tri(b + i, a + j)]);
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j <= i; ++j)
            if (cpl<kBlock>(b + i, b + j)) P[tri(b + i, b + j)] = fma_(dt, P[tri(d + i, b + j)], P[tri(b + i, b + j)]);
        // P'[c,a] = P[c,a] + P[c,c] A^T ; P'[d,a] = P[d,a] + P[d,c] A^T ; P'[c,b] = P[c,b] + dt P[c,d] ; P'[d,b] = P[d,b] + dt P[d,d]
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            Real s = P[tri(c + i, a + j)];
#pragma unroll
            for (int k = 0; k < 3; ++k) s = fma_(P[tri(c + i, c + k)], A[3 * j + k], s);
            P[tri(c + i, a + j)] = s;
            if (cpl<kBlock>(d + i, a + j)) {
                Real u = P[tri(d + i, a + j)];
#pragma unroll
                for (int k = 0; k < 3; ++k) u = fma_(P[tri(d + i, c + k)], A[3 * j + k], u);
                P[tri(d + i, a + j)] = u;
            }
        }
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            if (cpl<kBlock>(c + i, b + j)) P[tri(c + i, b + j)] = fma_(dt, P[tri(d + j, c + i)], P[tri(c + i, b + j)]);
            if (cpl<kBlock>(d + i, b + j)) P[tri(d + i, b + j)] = fma_(dt, P[tri(d + i, d + j)], P[tri(d + i, b + j)]);
        }
        // second factor: + W[a,c] A^T, + W[b,c] A^T, + dt W[b,d], with W[.,c] = P'[c,.]^T and W[b,d] = P'[d,b]^T
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j <= i; ++j) {
            Real s = P[tri(a + i, a + j)];
#pragma unroll
            for (int k = 0; k < 3; ++k) s = fma_(P[tri(c + k, a + i)], A[3 * j + k], s);
            P[tri(a + i, a + j)] = s;
        }
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j)
            if (cpl<kBlock>(b + i, a + j)) {
                Real s = P[tri(b + i, a + j)];
#pragma unroll
                for (int k = 0; k < 3; ++k) s = fma_(P[tri(c + k, b + i)], A[3 * j + k], s);
                P[tri(b + i, a + j)] = s;
            }
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j <= i; ++j)
            if (cpl<kBlock>(b + i, b + j)) P[tri(b + i, b + j)] = fma_(dt, P[tri(d + j, b + i)], P[tri(b + i, b + j)]);
#pragma unroll
    for (int i = 0; i < NX; ++i) P[tri(i, i)] += q[i * qs];
}

// exp(x) - 1 the way the reference gets it: F_d = np.exp(dt F) rounded to double, minus the ones of 1 1^T (exact).  The
// FP32 kernels take it from the double value, which keeps the small entries of D to full FP32 relative accuracy.
__device__ __forceinline__ double exp_minus_one(double x) { return exp(x) - 1.0; }
__device__ __forceinline__ float exp_minus_one(float x) { return (float)(exp((double)x) - 1.0); }
__device__ __forceinline__ F2 exp_minus_one(F2 x) { return F2(exp_minus_one(x.v.x), exp_minus_one(x.v.y)); }

// Covariance prediction of predict_mpc (kalman_filter.py:153-158): F_d = exp(dt F) ELEMENT-wise, so every entry that is
// zero in F becomes one: F_d = 1 1^T + D, with D zero except D[0:3,6:9] = exp(dt Rb^T) - 1 (Rb from the reference body
// angles) and D[3+a][9+a] = exp(dt) - 1.  Then
//     F_d P F_d^T = s 1 1^T + 1 v^T + v 1^T + D P D^T,   s = 1^T P 1,  v = D P 1,
// which is symmetric by construction and costs ~400 flops instead of two dense 12x12 products (SURVEY 8(f) row 1).
// E[3a + k] = D[a][6 + k], e1 = exp(dt) - 1.  Checked against the golden vector of the unmodified reference
// (next_mpc_cov_seed5): states 8e-11, P 1e-11 with the sequential update that follows.
template <typename Real>
__device__ __forceinline__ void cov_predict_mpc_sym(Real (&P)[NP], const Real (&E)[9], Real e1, const Real *q, int qs) {
    Real w[NX];  // row sums P 1
#pragma unroll
    for (int i = 0; i < NX; ++i) {
        Real acc = P[tri(i, 0)];
#pragma unroll
        for (int j = 1; j < NX; ++j) acc += P[tri(i, j)];
        w[i] = acc;
    }
    Real s = w[0];
#pragma unroll
    for (int i = 1; i < NX; ++i) s += w[i];
    Real v[6];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        v[a] = fma_(E[3 * a + 2], w[8], fma_(E[3 * a + 1], w[7], E[3 * a] * w[6]));
        v[3 + a] = e1 * w[9 + a];
    }
    // G = D P D^T, non-zero in the leading 6x6 block only
    Real U[9];  // U[3a + k'] = sum_k E[a][k] P[6+k][6+k']
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int kk = 0; kk < 3; ++kk)
            U[3 * a + kk] = fma_(E[3 * a + 2], P[tri(8, 6 + kk)], fma_(E[3 * a + 1], P[tri(7, 6 + kk)], E[3 * a] * P[tri(6, 6 + kk)]));
    Real G[21];  // lower triangle of the 6x6 block, G[tri(i, j)]
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int b = 0; b <= a; ++b) G[tri(a, b)] = fma_(U[3 * a + 2], E[3 * b + 2], fma_(U[3 * a + 1], E[3 * b + 1], U[3 * a] * E[3 * b]));
#pragma unroll
        for (int b = 0; b < 3; ++b)
            G[tri(3 + a, b)] = e1 * fma_(P[tri(9 + a, 8)], E[3 * b + 2], fma_(P[tri(9 + a, 7)], E[3 * b + 1], P[tri(9 + a, 6)] * E[3 * b]));
#pragma unroll
        for (int b = 0; b <= a; ++b) G[tri(3 + a, 3 + b)] = (e1 * e1) * P[tri(9 + a, 9 + b)];
    }
#pragma unroll
    for (int i = 0; i < NX; ++i)
#pragma unroll
        for (int j = 0; j <= i; ++j) {
            Real val = s;
            if (i < 6) val += v[i];
            if (j < 6) val += v[j];
            if (i < 6) val += G[tri(i, j)];  // j <= i < 6
            if (i == j) val += q[i * qs];
            P[tri(i, j)] = val;
        }
}

// Measurement J folded in with the reciprocal of its pivot already available (`inv` = 1 / (P_kk + r_J)).  The entry
// that becomes the NEXT pivot is updated first and its reciprocal started at once, so that chain (MUFU + its
// refinement) runs underneath the 65 remaining independent FMAs of this rank-1 update.  `mid` runs after the state update.
template <int J, bool kBlock = false, typename Real, int L, typename Mid>
__device__ __forceinline__ void fold_pipelined(Real (&P)[NP], Real (&x)[NX], Real zj, Real rj, Real r_next, Real inv, Real &inv_next,
                                               Real &nis, uint32_t (&status)[L], Mid mid) {
    constexpr int k = sel(J);
    constexpr int kn = (J + 1 < NZ) ? sel(J + 1) : -1;
    if constexpr (kn >= 0) {
        Real pnn = P[tri(kn, kn)];
        if constexpr (cpl<kBlock>(kn, k)) {
            const Real wn = P[tri(kn, k)] * inv;
            pnn = fnma_(wn, P[tri(kn, k)], pnn);
            P[tri(kn, kn)] = pnn;
        }
        const Real s = pnn + r_next;
        note_bad_pivot(s, status, OPTI_KF_ST_NOT_PD);
        inv_next = rcp_(s);
    }
    const Real y = zj - x[k];
    const Real g = inv * y;
    nis = fma_(y, g, nis);
#pragma unroll
    for (int i = 0; i < NX; ++i)
        if (cpl<kBlock>(i, k)) x[i] = fma_(P[tri(i, k)], g, x[i]);
    mid();
#pragma unroll
    for (int i = 0; i < NX; ++i) {
        if (i == k || !cpl<kBlock>(i, k)) continue;
        const Real w = P[tri(i, k)] * inv;
#pragma unroll
        for (int j = 0; j <= i; ++j) {
            if (j == k || !cpl<kBlock>(j, k) || (i == kn && j == kn)) continue;
            P[tri(i, j)] = fnma_(w, P[tri(j, k)], P[tri(i, j)]);
        }
    }
    const Real cfac = rj * inv;
#pragma unroll
    for (int i = 0; i < NX; ++i)
        if (cpl<kBlock>(i, k)) P[tri(i, k)] *= cfac;
}

// K_gain of the reference (np.trace of the 12x10 gain): K = P'[:, sel] R^-1  =>  K[j][j] = P'[j][sel(j)] / r_j.  The ten
// reciprocals are the straight-line rcp_ (kf_arith.cuh), not IEEE divisions: each division carries a branch to a slow path, and
// ten of those in a row cost a lone warp ~4,000 cycles per step (measured on the 1,024 x 10 k case with k_gain_steps on).
template <bool kBlock = false, typename Real>
__device__ __forceinline__ Real gain_trace(const Real (&P)[NP], const Real *r, int stride) {
    Real g = Real(0);
#pragma unroll
    for (int j = 0; j < NZ; ++j)
        if (cpl<kBlock>(j, sel(j))) g = fma_(P[tri(j, sel(j))], rcp_(r[j * stride]), g);
    return g;
}

// The same with the reciprocals of r supplied (taken once per trajectory by the kernels that write K_gain every step), in two
// interleaved sums: half the dependent chain, no reciprocal in the time loop.
template <bool kBlock = false, typename Real>
__device__ __forceinline__ Real gain_trace_rinv(const Real (&P)[NP], const Real *rinv, int stride) {
    Real g0 = Real(0), g1 = Real(0);
#pragma unroll
    for (int j = 0; j < NZ; j += 2) {
        if (cpl<kBlock>(j, sel(j))) g0 = fma_(P[tri(j, sel(j))], rinv[j * stride], g0);
        if (cpl<kBlock>(j + 1, sel(j + 1))) g1 = fma_(P[tri(j + 1, sel(j + 1))], rinv[(j + 1) * stride], g1);
    }
    return g0 + g1;
}

// trace of P, pairwise: a chain of four additions instead of twelve
template <typename Real>
__device__ __forceinline__ Real trace_of(const Real (&P)[NP]) {
    Real h[6];
#pragma unroll
    for (int c = 0; c < 6; ++c) h[c] = P[tri(2 * c, 2 * c)] + P[tri(2 * c + 1, 2 * c + 1)];
    return ((h[0] + h[1]) + (h[2] + h[3])) + (h[4] + h[5]);
}

// Set-up and outputs of the two kernels.  Loads take `idx` (the streamed kernel's clamped index), stores the thread's first
// trajectory `i`.  N is the caller's prm.N: loaded again here, it changes the kernels' index arithmetic.

// q[12] and r[10] to the caller's shared-memory columns q[c * nt], r[c * nt]
template <typename Real, typename Scalar>
__device__ __forceinline__ void load_noise(const Params<Scalar> &prm, long long N, long long idx, Real *q, Real *r, int nt) {
#pragma unroll
    for (int c = 0; c < NX; ++c) q[c * nt] = prm.q_kind == OPTI_KF_MAT_DIAG ? Real(prm.Q[c]) : ld_traj(prm.Q, c * N + idx, Real());
#pragma unroll
    for (int c = 0; c < NZ; ++c) r[c * nt] = prm.r_kind == OPTI_KF_MAT_DIAG ? Real(prm.R[c]) : ld_traj(prm.R, c * N + idx, Real());
}

// P0; NONE is diag(q).  x0 stays in the kernels: F2 needs a select on x0_inc, which costs the FP64 direct kernels spills.
template <bool kBlock, typename Real, typename Scalar>
__device__ __forceinline__ void load_P0(const Params<Scalar> &prm, long long N, long long idx, const Real *q, int nt, Real (&P)[NP]) {
#pragma unroll
    for (int a = 0; a < NX; ++a)
#pragma unroll
        for (int b = 0; b <= a; ++b) {
            Real v = Real(0);
            if (cpl<kBlock>(a, b)) switch (prm.p0_kind) {  // structural zeros are never loaded
                case OPTI_KF_MAT_NONE: v = (a == b) ? q[a * nt] : Real(0); break;
                case OPTI_KF_MAT_DIAG: v = (a == b) ? Real(prm.P0[a]) : Real(0); break;
                case OPTI_KF_MAT_DIAG_PER: v = (a == b) ? ld_traj(prm.P0, a * N + idx, Real()) : Real(0); break;
                case OPTI_KF_MAT_DENSE: v = Real(prm.P0[a * NX + b]); break;
                default: v = ld_traj(prm.P0, (long long)(a * NX + b) * N + idx, Real()); break;
            }
            P[tri(a, b)] = v;
        }
}

// Outputs of step t after the update; kRare adds P_ckpt (dense 144) and P_steps (packed or full, by kBlock)
template <bool kBlock, bool kRare, typename Real, typename Scalar>
__device__ __forceinline__ void store_step(const Params<Scalar> &prm, long long t, long long N, long long i, const Real (&x)[NX],
                                           const Real (&P)[NP], Real ptrace, Real kgain, Real nis) {
    if (prm.x_steps) {
#pragma unroll
        for (int c = 0; c < NX; ++c) st_traj(prm.x_steps, (t * NX + c) * N + i, x[c]);
    }
    if (prm.p_trace_steps) st_traj(prm.p_trace_steps, t * N + i, ptrace);
    if (prm.k_gain_steps) st_traj(prm.k_gain_steps, t * N + i, kgain);
    if (prm.nis_steps) st_traj(prm.nis_steps, t * N + i, nis);
    if constexpr (kRare) {
        if (prm.P_ckpt && prm.ckpt_every > 0 && (t + 1) % prm.ckpt_every == 0) {
            const long long base = ((t + 1) / prm.ckpt_every - 1) * (long long)(NX * NX) * N + i;
#pragma unroll
            for (int a = 0; a < NX; ++a)
#pragma unroll
                for (int b = 0; b < NX; ++b) st_traj(prm.P_ckpt, base + (long long)(a * NX + b) * N, cpl<kBlock>(a, b) ? P[tri(a, b)] : Real(0));
        }
        if (prm.P_steps) {
            if constexpr (kBlock) store_packed_P(prm.P_steps, t, N, i, P);
            else store_full_P(prm.P_steps, t, N, i, P);
        }
    }
}

// x_final and P_final (dense 144, structural zeros written as zeros)
template <bool kBlock, typename Real, typename Scalar>
__device__ __forceinline__ void store_final(const Params<Scalar> &prm, long long N, long long i, const Real (&x)[NX], const Real (&P)[NP]) {
    if (prm.x_final) {
#pragma unroll
        for (int c = 0; c < NX; ++c) st_traj(prm.x_final, c * N + i, x[c]);
    }
    if (prm.P_final) {
#pragma unroll
        for (int a = 0; a < NX; ++a)
#pragma unroll
            for (int b = 0; b < NX; ++b) st_traj(prm.P_final, (long long)(a * NX + b) * N + i, cpl<kBlock>(a, b) ? P[tri(a, b)] : Real(0));
    }
}

// Summary rows 0-51 from x, P, the running sums acc(k), ptrace, kgain and ymax; an absent label stream gives zeros
constexpr int ACC_ROWS = 25;  // running sums of the summary: 0-11 truth, 12-23 nominal, 24 NIS
template <typename Real, typename Scalar, typename AccGet>
__device__ __forceinline__ void store_summary(const Params<Scalar> &prm, long long i, const Real (&x)[NX], const Real (&P)[NP], AccGet acc,
                                              Real ptrace, Real kgain, Real ymax) {
    const double invT = prm.T > 0 ? 1.0 / (double)prm.T : 0.0;
#pragma unroll
    for (int c = 0; c < NX; ++c) {
        st_summary(prm, c, i, x[c]);
        st_summary(prm, 12 + c, i, P[tri(c, c)]);
        st_summary(prm, 24 + c, i, prm.truth ? rms_out(acc(c), invT, Real()) : Real(0));
        st_summary(prm, 36 + c, i, prm.nominal ? rms_out(acc(12 + c), invT, Real()) : Real(0));
    }
    st_summary(prm, 48, i, mean_out(acc(24), invT, Real()));
    st_summary(prm, 49, i, ptrace);
    st_summary(prm, 50, i, kgain);
    st_summary(prm, 51, i, sqrt_(ymax));
}


// cheap test whether trunc(R^T) can have a non-zero entry in any lane (then the exact decision is taken per lane)
template <typename Real>
__device__ __forceinline__ bool may_truncate(const Real (&R)[9]) {
    using S = typename Lanes<Real>::scalar;
    int m = 0;
#pragma unroll
    for (int k = 0; k < 9; ++k) m = max(m, abs_bits(R[k]));
    return m >= (sizeof(S) == 8 ? 0x3ff00000 : 0x3f7ffff0);  // |entry| >= 1 (double) / >= 1 - 2^-20 (float)
}

// Leg moments of the mean model: C[3m + k] = sum_l p_l[m] f_l[k] (rows 0-8) and fs[k] = sum_l f_l[k] (rows 9-11).  They depend
// on the stream and the step only, so the measurement pre-pass forms them once for every member of a stream; the direct-load
// kernel forms them in-thread with this same function, which keeps the two kernels bit-identical.  Explicit mul_rn / fma_: the
// result does not depend on contraction, and double, float and F2 run the same sequence.
constexpr int NM = 12;
template <typename Real>
__device__ __forceinline__ void leg_moments(const Real (&p)[12], const Real (&f)[12], Real (&M)[NM]) {
#pragma unroll
    for (int m = 0; m < 3; ++m)
#pragma unroll
        for (int k = 0; k < 3; ++k)
            M[3 * m + k] = fma_(p[9 + m], f[9 + k], fma_(p[6 + m], f[6 + k], fma_(p[3 + m], f[3 + k], mul_rn(p[m], f[k]))));
#pragma unroll
    for (int k = 0; k < 3; ++k) M[9 + k] = ((f[k] + f[3 + k]) + f[6 + k]) + f[9 + k];
}

// Feet rotated into the world frame (the reference's in-place mutation of p, force_controller.py:274-277), stored to `pw_out`;
// `pin` reads the feet with channel stride STRIDE (32 for a warp's shared-memory tile, 1 for a per-thread array).
template <int STRIDE, typename Real, typename Scalar>
__device__ __forceinline__ void store_world_feet(const Real *pin, const Real (&R)[9], Scalar *pw_out, long long pw_idx, long long pw_stride) {
#pragma unroll
    for (int l = 0; l < 4; ++l) {
        const Real a = pin[(3 * l) * STRIDE], b = pin[(3 * l + 1) * STRIDE], c = pin[(3 * l + 2) * STRIDE];
        st_traj(pw_out, pw_idx + (3 * l) * pw_stride, fma_(R[2], c, fma_(R[1], b, R[0] * a)));
        st_traj(pw_out, pw_idx + (3 * l + 1) * pw_stride, fma_(R[5], c, fma_(R[4], b, R[3] * a)));
        st_traj(pw_out, pw_idx + (3 * l + 2) * pw_stride, fma_(R[8], c, fma_(R[7], b, R[6] * a)));
    }
}

// Mean model with the rotation of the prior attitude supplied by the caller (see propagate_mean in kf_common.cuh), from the
// leg moments (leg_moments; read through `min` with channel stride STRIDE).  The rate rows need the torque
// tau = sum_l (R p_l) x f_l only in the body frame, as R^T tau.  For a rotation (R a) x (R b) = R (a x b), so
// R^T tau = sum_l p_l x (R^T f_l), i.e. (R^T tau)_i = eps_ijk (C R)_jk: 18 FP64 operations per member instead of 84 for the four
// legs, and w' = w + R (dt I^-1 R^T tau) adds 12.  Unlike the regrouping into moments, this step holds only because R is
// orthogonal, which rot_zyx's R is to rounding.  The result rounds differently from propagate_mean's leg-by-leg order (the
// last bits of the state).
template <int STRIDE, typename Real, typename Scalar>
__device__ __forceinline__ void propagate_mean_from_moments(const Params<Scalar> &prm, Real (&x)[NX], const Real *min, const Real (&R)[9],
                                                            bool any_trunc) {
    constexpr int L = Lanes<Real>::n;
    const auto C = [&](int k) { return min[k * STRIDE]; };
    // u_i = dt I_i^-1 (sum_m C[j][m] R[m][k] - C[k][m] R[m][j])  for (i, j, k) a cyclic permutation of (0, 1, 2)
    Real u[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const int j = (i + 1) % 3, k = (i + 2) % 3;
        u[i] = mul_rn(fnma_(C(3 * k + 2), R[6 + j], fnma_(C(3 * k + 1), R[3 + j], fnma_(C(3 * k), R[j],
                      fma_(C(3 * j + 2), R[6 + k], fma_(C(3 * j + 1), R[3 + k], mul_rn(C(3 * j), R[k])))))),
                      Real(prm.dt * prm.inv_inertia[i]));
    }
    const Real dt = Real(prm.dt);
    Real xn[NX];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        xn[i] = x[i];  // the attitude moves only on the trunc path below: the common path adds no zero increment
        xn[3 + i] = fma_(dt, x[9 + i], x[3 + i]);
        xn[6 + i] = fma_(R[3 * i + 2], u[2], fma_(R[3 * i + 1], u[1], fma_(R[3 * i], u[0], x[6 + i])));
        xn[9 + i] = fma_(Real(prm.dt_over_m), min[(9 + i) * STRIDE], x[9 + i]);  // fs
    }
    xn[11] += Real(prm.dt_g);
    if (any_trunc) {  // rare: an entry of R is exactly +-1 (axis-aligned attitude); exact per-lane decision in trunc_rt
        Real dth[3];
#pragma unroll
        for (int ln = 0; ln < L; ++ln) {
            Scalar Rs[9], Ts[9], ang[3];
            bool any;
#pragma unroll
            for (int k = 0; k < 9; ++k) Rs[k] = lane_get(R[k], ln);
#pragma unroll
            for (int k = 0; k < 3; ++k) ang[k] = lane_get(x[k], ln);
            trunc_rt(Rs, ang, Ts, any);
#pragma unroll
            for (int i = 0; i < 3; ++i)
                lane_set(dth[i], ln, prm.dt * (Ts[3 * i] * lane_get(x[6], ln) + Ts[3 * i + 1] * lane_get(x[7], ln) + Ts[3 * i + 2] * lane_get(x[8], ln)));
        }
#pragma unroll
        for (int i = 0; i < 3; ++i) xn[i] = add_rn(x[i], dth[i]);  // dth rounded before the sum, as in propagate_mean
    }
#pragma unroll
    for (int i = 0; i < NX; ++i) x[i] = xn[i];
}

}  // namespace okf
