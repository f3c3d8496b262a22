// Direct-load variant of the SEQUENTIAL path: the arithmetic of kf_seq_core.cuh fed by plain coalesced loads from the
// [T][C][S] layout (stream index fastest).  It serves everything the TMA-fed kernel (kf_seq_tma.cuh) cannot take:
// an arbitrary stream_index gather, stream counts that are not a multiple of 32, unaligned arrays, or no workspace for
// the measurement pre-pass (the measurement is then formed inside the kernel, kalman_filter.py:79-117).
#pragma once

#include "kf_seq_core.cuh"

namespace okf {

constexpr int SEQ_NOISE_ROWS = 22;  // shared memory rows per thread: q[12] r[10]

template <typename Real, bool kSummary, bool kMpc, bool kBlock = false>
__global__ void __launch_bounds__(128) kf_seq_kernel(const __grid_constant__ Params<Real> prm) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Real *noise = reinterpret_cast<Real *>(smem_raw);  // [SEQ_NOISE_ROWS][blockDim.x]
    const int nt = blockDim.x;
    const long long i = (long long)blockIdx.x * nt + threadIdx.x;
    if (i >= prm.N) return;
    const long long N = prm.N, S = prm.S;
    const long long s = stream_of(prm, i);
    Real *q = noise + threadIdx.x, *r = noise + 12 * nt + threadIdx.x;
#pragma unroll
    for (int c = 0; c < NX; ++c) q[c * nt] = prm.q_kind == OPTI_KF_MAT_DIAG ? prm.Q[c] : prm.Q[c * N + i];
#pragma unroll
    for (int c = 0; c < NZ; ++c) r[c * nt] = prm.r_kind == OPTI_KF_MAT_DIAG ? prm.R[c] : prm.R[c * N + i];

    Real x[NX], P[NP];
#pragma unroll
    for (int c = 0; c < NX; ++c) x[c] = prm.x0[c * prm.x0_ld + i * prm.x0_inc];
#pragma unroll
    for (int a = 0; a < NX; ++a)
#pragma unroll
        for (int b = 0; b <= a; ++b) {
            Real v = Real(0);
            if (cpl<kBlock>(a, b)) switch (prm.p0_kind) {  // structural zeros are never loaded
                case OPTI_KF_MAT_NONE: v = (a == b) ? q[a * nt] : Real(0); break;
                case OPTI_KF_MAT_DIAG: v = (a == b) ? prm.P0[a] : Real(0); break;
                case OPTI_KF_MAT_DIAG_PER: v = (a == b) ? prm.P0[a * N + i] : Real(0); break;
                case OPTI_KF_MAT_DENSE: v = prm.P0[a * NX + b]; break;
                default: v = prm.P0[(long long)(a * NX + b) * N + i]; break;
            }
            P[tri(a, b)] = v;
        }

    uint32_t status[1] = {0};
    Real ptrace = Real(0), kgain = Real(0), ymax = Real(0);
    double acc_truth[kSummary ? NX : 1], acc_nom[kSummary ? NX : 1], acc_nis = 0.0;
    if (kSummary) {
#pragma unroll
        for (int c = 0; c < NX; ++c) { acc_truth[c] = 0.0; acc_nom[c] = 0.0; }
    }

    Real Rm[9];
    rot_zyx(x[0], x[1], x[2], Rm);
    bool any_trunc = may_truncate(Rm);

    for (long long t = 0; t < prm.T; ++t) {
        const bool last = t + 1 == prm.T;
        Real z[NZ], pf[12], ff[12];
#pragma unroll
        for (int c = 0; c < 12; ++c) {
            pf[c] = ld_stream(prm.p + (t * 12 + c) * S + s);
            ff[c] = ld_stream(prm.f + (t * 12 + c) * S + s);
        }
        if (prm.z_in) {
#pragma unroll
            for (int c = 0; c < NZ; ++c) z[c] = ld_stream(prm.z_in + (t * NZ + c) * S + s);
        } else {
            Real imu[6], dp[12], contact[4];
#pragma unroll
            for (int c = 0; c < 6; ++c) imu[c] = ld_stream(prm.imu + (t * 6 + c) * S + s);
#pragma unroll
            for (int c = 0; c < 12; ++c) dp[c] = ld_stream(prm.dp + (t * 12 + c) * S + s);
#pragma unroll
            for (int c = 0; c < 4; ++c) contact[c] = ld_stream(prm.contact + (t * 4 + c) * S + s);
            if (form_measurement(imu, pf, dp, contact, z)) status[0] |= OPTI_KF_ST_ALL_SWING;
        }

        if (prm.p_world_steps) store_world_feet<1>(pf, Rm, prm.p_world_steps, (t * 12) * N + i, N);
        {
            Real M[NM];
            leg_moments(pf, ff, M);
            propagate_mean_from_moments<1>(prm, x, M, Rm, any_trunc);
        }
        if (prm.x_model_steps) {
#pragma unroll
            for (int c = 0; c < NX; ++c) st_stream(prm.x_model_steps + (t * NX + c) * N + i, x[c]);
        }
        if (prm.z_steps) {
#pragma unroll
            for (int c = 0; c < NZ; ++c) st_stream(prm.z_steps + (t * NZ + c) * N + i, z[c]);
        }

        if constexpr (kMpc) {  // predict_mpc covariance model: R of the transition from the reference body angles
            Real Rb[9], E[9];
            rot_zyx(ld_stream(prm.body_ref + (t * 12 + 0) * S + s), ld_stream(prm.body_ref + (t * 12 + 1) * S + s),
                    ld_stream(prm.body_ref + (t * 12 + 2) * S + s), Rb);
#pragma unroll
            for (int a = 0; a < 3; ++a)
#pragma unroll
                for (int k = 0; k < 3; ++k) E[3 * a + k] = exp_minus_one(prm.dt * Rb[3 * k + a]);
            cov_predict_mpc_sym(P, E, exp_minus_one(prm.dt), q, nt);
        } else {
            cov_predict_sym<kBlock>(P, Rm, prm.dt, q, nt);
        }

        Real nis = Real(0), inv, inv_n;
        {
            const Real s0 = P[tri(0, 0)] + r[0];
            note_bad_pivot(s0, status, OPTI_KF_ST_NOT_PD);
            inv = rcp_(s0);
        }
        auto nothing = [] {};
        fold_pipelined<0, kBlock>(P, x, z[0], r[0 * nt], r[1 * nt], inv, inv_n, nis, status, nothing); inv = inv_n;
        fold_pipelined<1, kBlock>(P, x, z[1], r[1 * nt], r[2 * nt], inv, inv_n, nis, status, nothing); inv = inv_n;
        fold_pipelined<2, kBlock>(P, x, z[2], r[2 * nt], r[3 * nt], inv, inv_n, nis, status, nothing); inv = inv_n;
        fold_pipelined<3, kBlock>(P, x, z[3], r[3 * nt], r[4 * nt], inv, inv_n, nis, status, nothing); inv = inv_n;
        fold_pipelined<4, kBlock>(P, x, z[4], r[4 * nt], r[5 * nt], inv, inv_n, nis, status, nothing); inv = inv_n;
        fold_pipelined<5, kBlock>(P, x, z[5], r[5 * nt], r[6 * nt], inv, inv_n, nis, status, nothing); inv = inv_n;
        fold_pipelined<6, kBlock>(P, x, z[6], r[6 * nt], r[7 * nt], inv, inv_n, nis, status, nothing); inv = inv_n;
        fold_pipelined<7, kBlock>(P, x, z[7], r[7 * nt], r[8 * nt], inv, inv_n, nis, status, nothing); inv = inv_n;
        fold_pipelined<8, kBlock>(P, x, z[8], r[8 * nt], r[9 * nt], inv, inv_n, nis, status, nothing); inv = inv_n;
        fold_pipelined<9, kBlock>(P, x, z[9], r[9 * nt], r[9 * nt], inv, inv_n, nis, status, [&] {
            rot_zyx(x[0], x[1], x[2], Rm);  // next step's rotation, started underneath the last rank-1 update
            any_trunc = may_truncate(Rm);
        });

        ymax = max_(ymax, nis);
        ptrace = Real(0);
#pragma unroll
        for (int c = 0; c < NX; ++c) ptrace += P[tri(c, c)];
        if (prm.k_gain_steps != nullptr || (last && prm.summary != nullptr)) {
            kgain = gain_trace<kBlock>(P, r, nt);
        }
        if (prm.x_steps) {
#pragma unroll
            for (int c = 0; c < NX; ++c) st_stream(prm.x_steps + (t * NX + c) * N + i, x[c]);
        }
        if (prm.p_trace_steps) st_stream(prm.p_trace_steps + t * N + i, ptrace);
        if (prm.k_gain_steps) st_stream(prm.k_gain_steps + t * N + i, kgain);
        if (prm.nis_steps) st_stream(prm.nis_steps + t * N + i, nis);
        if (kSummary) {
            acc_nis += (double)nis;
            if (prm.truth) {
#pragma unroll
                for (int c = 0; c < NX; ++c) acc_truth[c] = err_acc(acc_truth[c], x[c], ld_stream(prm.truth + (t * NX + c) * S + s));
            }
            if (prm.nominal) {
#pragma unroll
                for (int c = 0; c < NX; ++c) acc_nom[c] = err_acc(acc_nom[c], x[c], ld_stream(prm.nominal + (t * NX + c) * S + s));
            }
        }
        if (prm.P_ckpt && prm.ckpt_every > 0 && (t + 1) % prm.ckpt_every == 0) {
            Real *dst = prm.P_ckpt + ((t + 1) / prm.ckpt_every - 1) * (long long)(NX * NX) * N + i;
#pragma unroll
            for (int a = 0; a < NX; ++a)
#pragma unroll
                for (int b = 0; b < NX; ++b) dst[(long long)(a * NX + b) * N] = cpl<kBlock>(a, b) ? P[tri(a, b)] : Real(0);
        }
        if (prm.P_steps) {
            if constexpr (kBlock) store_packed_P(prm.P_steps, t, N, i, P);
            else store_full_P(prm.P_steps, t, N, i, P);
        }
    }

#pragma unroll
    for (int c = 0; c < NX; ++c) note_nonfinite(x[c], status, OPTI_KF_ST_NONFINITE);  // absorbing: see kf_seq_tma.cuh
    if (prm.x_final) {
#pragma unroll
        for (int c = 0; c < NX; ++c) prm.x_final[c * N + i] = x[c];
    }
    if (prm.P_final) {
#pragma unroll
        for (int a = 0; a < NX; ++a)
#pragma unroll
            for (int b = 0; b < NX; ++b) prm.P_final[(long long)(a * NX + b) * N + i] = cpl<kBlock>(a, b) ? P[tri(a, b)] : Real(0);
    }
    if (kSummary && prm.summary) {
        const double invT = prm.T > 0 ? 1.0 / (double)prm.T : 0.0;
#pragma unroll
        for (int c = 0; c < NX; ++c) {
            st_summary(prm, c, i, x[c]);
            st_summary(prm, 12 + c, i, P[tri(c, c)]);
            st_summary(prm, 24 + c, i, (Real)sqrt(acc_truth[c] * invT));
            st_summary(prm, 36 + c, i, (Real)sqrt(acc_nom[c] * invT));
        }
        st_summary(prm, 48, i, (Real)(acc_nis * invT));
        st_summary(prm, 49, i, ptrace);
        st_summary(prm, 50, i, kgain);
        st_summary(prm, 51, i, (Real)sqrt((double)ymax));
    }
    if (prm.status) prm.status[i] = status[0] | (prm.stream_status ? prm.stream_status[s] : 0u);  // pre-pass flags (ALL_SWING) of this stream
}

}  // namespace okf
