// Device helpers shared by the Kalman-filter kernels: rotation, measurement formation, the rigid-body mean
// model.  Each function cites the reference lines whose arithmetic it reproduces (paths under /root/reference).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/optistate_kf.h"
#include "kf_arith.cuh"

namespace okf {

constexpr int NX = OPTI_KF_NX;
constexpr int NZ = OPTI_KF_NZ;
// rows of H (kalman_filter.py:15-24): measurement j observes state SEL[j]
__host__ __device__ constexpr int sel(int j) { return j < 3 ? j : j + 2; }

// Kernel-side view of OptiKfDesc: pointers typed, scalars pre-converted on the host.
template <typename Real>
struct Params {
    long long N, T, S, stream_offset;
    int phases, cov_model;
    int block;  // 1: P has the decoupled group structure (OPTI_KF_FLAG_*; kBlock kernels, kf_seq_core.cuh)
    Real dt, dt_over_m, dt_g, inv_inertia[3];
    const Real *imu, *p, *dp, *contact, *f, *z_in, *body_ref, *truth, *nominal;
    const Real *mom;  // [T][12][S] leg moments of the mean model from the measurement pre-pass (streamed kernel only)
    const int32_t *stream_index;
    const Real *x0; long long x0_ld; int x0_inc;
    const Real *P0; int p0_kind;
    const Real *Q; int q_kind;
    const Real *R; int r_kind;
    Real *x_steps, *x_model_steps, *p_world_steps, *z_steps, *p_trace_steps, *k_gain_steps, *nis_steps;
    long long ckpt_every;
    Real *P_ckpt, *x_final, *P_final, *K_final, *summary;
    uint32_t *status;
    const uint32_t *stream_status;  // [S] per-stream flags of the measurement pre-pass, OR-ed into status
    // fused all-gather of the summaries: rows are summary_ld apart (the whole job's trajectory count) and every value
    // is stored to the same element of each peer GPU's copy as well (NVLink stores, OptiKfDesc.summary_peers)
    long long summary_ld;
    int n_summary_peers;
    Real *summary_peers[OPTI_KF_MAX_PEERS];
    // posterior covariance of every step: [T][30][N] decoupled-group entries (pk_slot) in the kBlock kernels, [T][78][N] in tri
    // order in the full ones (kf_seq_core.cuh); set by the smoothers' forward passes alone.  Last, so that every other field
    // keeps its constant-bank offset.
    Real *P_steps;
};

// One summary value of trajectory i (or of the pair i, i+1 for the packed FP32 type): local copy plus every peer copy.
template <typename Real, typename V>
__device__ __forceinline__ void st_summary(const Params<Real> &prm, int row, long long i, V v) {
    const long long idx = (long long)row * prm.summary_ld + i;
    st_traj(prm.summary, idx, v);
    for (int k = 0; k < prm.n_summary_peers; ++k) st_traj(prm.summary_peers[k], idx, v);
}

// sin and cos of an attitude angle, straight-line (no slow-path branch, so the trigonometry of the NEXT step can be
// scheduled underneath the rank-1 FMAs of the current one): Cody-Waite reduction by pi/2 with fused steps, then the
// fdlibm (FP64) / Cephes (FP32) kernel polynomials on [-pi/4, pi/4] and a branch-free quadrant fix-up.  Error <= ~1 ulp for
// |angle| < ~1e6 rad (FP64) / ~8e3 rad (FP32); sin(0) = 0, cos(0) = 1 and sin(nearest(pi/2)) = 1 exactly, which is what
// the trunc(R^T) semantics of the mean model depend on.
template <typename Real> __device__ __forceinline__ void sincos_full(Real a, Real &s, Real &c);
template <> __device__ __forceinline__ void sincos_full<double>(double x, double &s, double &c) {
    const double q = rint(x * 6.36619772367581382433e-01);
    double r = fma(-q, 1.57079632673412561417e+00, x);
    r = fma(-q, 6.07710050630396597660e-11, r);
    r = fma(-q, 2.02226624871116645580e-21, r);
    r = fma(-q, 8.47842766036889956997e-32, r);
    const double z = r * r;
    double ps = fma(z, 1.58969099521155010221e-10, -2.50507602534068634195e-08);
    ps = fma(z, ps, 2.75573137070700676789e-06);
    ps = fma(z, ps, -1.98412698298579493134e-04);
    ps = fma(z, ps, 8.33333333332248946124e-03);
    ps = fma(z, ps, -1.66666666666666324348e-01);
    const double sr = fma(z * r, ps, r);
    double pc = fma(z, -1.13596475577881948265e-11, 2.08757232129817482790e-09);
    pc = fma(z, pc, -2.75573143513906633035e-07);
    pc = fma(z, pc, 2.48015872894767294178e-05);
    pc = fma(z, pc, -1.38888888888741095749e-03);
    pc = fma(z, pc, 4.16666666666666019037e-02);
    const double cr = 1.0 - fma(0.5, z, -(z * (z * pc)));
    const int n = __double2int_rn(q);
    const double s0 = (n & 1) ? cr : sr, c0 = (n & 1) ? sr : cr;
    s = (n & 2) ? -s0 : s0;
    c = ((n + 1) & 2) ? -c0 : c0;
}
template <> __device__ __forceinline__ void sincos_full<float>(float x, float &s, float &c) {
    const float q = rintf(x * 0.636619772367581343f);
    float r = fmaf(-q, 1.5703125f, x);
    r = fmaf(-q, 4.837512969970703125e-4f, r);
    r = fmaf(-q, 7.54978995489188216e-8f, r);
    const float z = r * r;
    float ps = fmaf(z, -1.9515295891e-4f, 8.3321608736e-3f);
    ps = fmaf(z, ps, -1.6666654611e-1f);
    const float sr = fmaf(z * r, ps, r);
    float pc = fmaf(z, 2.443315711809948e-5f, -1.388731625493765e-3f);
    pc = fmaf(z, pc, 4.166664568298827e-2f);
    const float cr = 1.0f - fmaf(0.5f, z, -(z * (z * pc)));
    const int n = __float2int_rn(q);
    const float s0 = (n & 1) ? cr : sr, c0 = (n & 1) ? sr : cr;
    s = (n & 2) ? -s0 : s0;
    c = ((n + 1) & 2) ? -c0 : c0;
}
template <> __device__ __forceinline__ void sincos_full<F2>(F2 a, F2 &s, F2 &c) {
    sincos_full<float>(a.v.x, s.v.x, c.v.x);
    sincos_full<float>(a.v.y, s.v.y, c.v.y);
}

// products/sums that must not be contracted into FMAs: the entries of R decide trunc(R^T) below
__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ F2 mul_rn(F2 a, F2 b) { return a * b; }  // FMUL2 / FADD2 are never contracted
__device__ __forceinline__ F2 add_rn(F2 a, F2 b) { return a + b; }

// R = Rz(c) Ry(b) Rx(a), multiplied out in the association np.matmul(Rz, np.matmul(Ry, Rx)) produces
// (kalman_filter.py:184-193, force_controller.py:227-237).  Row-major R[3*i + j].
template <typename Real>
__device__ __forceinline__ void rot_zyx(Real a, Real b, Real c, Real (&R)[9]) {
    Real sa, ca, sb, cb, sc, cc;
    sincos_full(a, sa, ca);
    sincos_full(b, sb, cb);
    sincos_full(c, sc, cc);
    const Real sbsa = mul_rn(sb, sa), sbca = mul_rn(sb, ca);
    R[0] = mul_rn(cc, cb);
    R[1] = add_rn(mul_rn(cc, sbsa), -mul_rn(sc, ca));
    R[2] = add_rn(mul_rn(cc, sbca), mul_rn(sc, sa));
    R[3] = mul_rn(sc, cb);
    R[4] = add_rn(mul_rn(sc, sbsa), mul_rn(cc, ca));
    R[5] = add_rn(mul_rn(sc, sbca), -mul_rn(cc, sa));
    R[6] = -sb;
    R[7] = mul_rn(cb, sa);
    R[8] = mul_rn(cb, ca);
}

// trunc(R^T): the reference stores R^T into an int64 matrix (force_controller.py:248-251,271), so the attitude
// rows of the mean model see the truncated entries (SURVEY 0.2).  FP64: truncate the FP64 entries.
__device__ __forceinline__ void trunc_rt(const double (&R)[9], const double *, double (&Tm)[9], bool &any) {
    any = false;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const double v = trunc(R[3 * j + i]);
            Tm[3 * i + j] = v;
            any |= (v != 0.0);
        }
}
// FP32: cos(th) rounds to exactly 1.0f for |th| < ~2.4e-4 (FP64: < ~1e-8), so truncating FP32 entries would
// fire the +-1 entries far more often than the reference does.  The decision is therefore taken with FP64
// semantics: only when an FP32 entry is within 2^-20 of +-1 (rare: near axis-aligned attitudes, e.g. the
// all-zero start state) is R re-evaluated in FP64 from the same angles and truncated there.
__device__ __forceinline__ void trunc_rt(const float (&R)[9], const float *ang, float (&Tm)[9], bool &any) {
    float m = 0.f;
#pragma unroll
    for (int k = 0; k < 9; ++k) { m = fmaxf(m, fabsf(R[k])); Tm[k] = 0.f; }
    any = false;
    if (m >= 1.0f - 9.5367431640625e-7f) {
        double Rd[9], Td[9];
        rot_zyx<double>((double)ang[0], (double)ang[1], (double)ang[2], Rd);
        trunc_rt(Rd, nullptr, Td, any);
#pragma unroll
        for (int k = 0; k < 9; ++k) Tm[k] = (float)Td[k];
    }
}

// get_odom + set_measurements (kalman_filter.py:79-117).  Stance legs (contact == 1) contribute dp_x, dp_y, p_z;
// swing legs (contact == 0) contribute dp_z; every sum is scaled by -1/sum(contact).  Returns true when no leg
// is in stance (the reference raises there); the odometry entries are then 0.
template <typename Real>
__device__ __forceinline__ bool form_measurement(const Real (&imu)[6], const Real (&p)[12], const Real (&dp)[12],
                                                 const Real (&contact)[4], Real (&z)[NZ]) {
    Real nc = 0, sx = 0, sy = 0, sv = 0, sz = 0;
#pragma unroll
    for (int l = 0; l < 4; ++l) {
        nc += contact[l];
        const bool stance = (contact[l] == Real(1)), swing = (contact[l] == Real(0));
        sx += stance ? dp[3 * l] : Real(0);
        sy += stance ? dp[3 * l + 1] : Real(0);
        sz += stance ? p[3 * l + 2] : Real(0);
        sv += swing ? dp[3 * l + 2] : Real(0);
    }
    const bool all_swing = (nc == Real(0));
    Real vb[3] = {Real(0), Real(0), Real(0)}, zo = Real(0);
    if (!all_swing) {
        vb[0] = -sx / nc; vb[1] = -sy / nc; vb[2] = -sv / nc; zo = -sz / nc;
    }
    Real Ri[9];
    rot_zyx(imu[0], imu[1], imu[2], Ri);
    z[0] = imu[0]; z[1] = imu[1]; z[2] = imu[2]; z[3] = zo;
    z[4] = imu[3]; z[5] = imu[4]; z[6] = imu[5];
#pragma unroll
    for (int i = 0; i < 3; ++i) z[7 + i] = Ri[3 * i] * vb[0] + Ri[3 * i + 1] * vb[1] + Ri[3 * i + 2] * vb[2];
    return all_swing;
}

// next_state (force_controller.py:269-291): x <- (I + A dt) x + (B dt) f + dt g with
//   attitude rows  th' = th + dt trunc(R^T) w          (int64 A)
//   position rows  r'  = r + dt v
//   rate rows      w'  = w + dt (R I_b R^T)^-1 sum_l (R p_l) x f_l   evaluated as R diag(1/I_b) R^T tau
//   velocity rows  v'  = v + dt sum_l f_l / m + dt [0 0 g]
// p is rotated into the world frame in place, as the reference does (force_controller.py:274-277).
// R (from the prior attitude) is returned for the covariance transition (kalman_filter.py:124-125).
template <typename Real>
__device__ __forceinline__ void propagate_mean(const Params<Real> &P, Real (&x)[NX], Real (&p)[12], const Real (&f)[12],
                                               Real (&R)[9]) {
    rot_zyx(x[0], x[1], x[2], R);
    Real Tm[9];
    bool any;
    trunc_rt(R, x, Tm, any);
    Real tau[3] = {Real(0), Real(0), Real(0)}, fs[3] = {Real(0), Real(0), Real(0)};
#pragma unroll
    for (int l = 0; l < 4; ++l) {
        const Real a = p[3 * l], b = p[3 * l + 1], c = p[3 * l + 2];
        const Real pw0 = R[0] * a + R[1] * b + R[2] * c;
        const Real pw1 = R[3] * a + R[4] * b + R[5] * c;
        const Real pw2 = R[6] * a + R[7] * b + R[8] * c;
        p[3 * l] = pw0; p[3 * l + 1] = pw1; p[3 * l + 2] = pw2;
        const Real f0 = f[3 * l], f1 = f[3 * l + 1], f2 = f[3 * l + 2];
        tau[0] += pw1 * f2 - pw2 * f1;
        tau[1] += pw2 * f0 - pw0 * f2;
        tau[2] += pw0 * f1 - pw1 * f0;
        fs[0] += f0; fs[1] += f1; fs[2] += f2;
    }
    Real u[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) u[k] = (R[k] * tau[0] + R[3 + k] * tau[1] + R[6 + k] * tau[2]) * P.inv_inertia[k];
    Real xn[NX];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        Real dth = Real(0);
        if (any) dth = P.dt * (Tm[3 * i] * x[6] + Tm[3 * i + 1] * x[7] + Tm[3 * i + 2] * x[8]);
        xn[i] = x[i] + dth;
        xn[3 + i] = x[3 + i] + P.dt * x[9 + i];
        xn[6 + i] = x[6 + i] + P.dt * (R[3 * i] * u[0] + R[3 * i + 1] * u[1] + R[3 * i + 2] * u[2]);
        xn[9 + i] = x[9 + i] + P.dt_over_m * fs[i];
    }
    xn[11] += P.dt_g;
#pragma unroll
    for (int i = 0; i < NX; ++i) x[i] = xn[i];
}

template <typename Real>
__device__ __forceinline__ long long stream_of(const Params<Real> &P, long long i) {
    return P.stream_index ? (long long)P.stream_index[i] : (i + P.stream_offset) % P.S;
}

template <typename Real> __device__ __forceinline__ Real ld_stream(const Real *p) { return __ldg(p); }
template <typename Real> __device__ __forceinline__ void st_stream(Real *p, Real v) { __stcs(p, v); }

template <typename Real> __device__ __forceinline__ bool finite_all(const Real (&x)[NX]) {
    bool ok = true;
#pragma unroll
    for (int i = 0; i < NX; ++i) ok &= (fabs((double)x[i]) <= 1.79e308) && (x[i] == x[i]);
    return ok;
}

}  // namespace okf
