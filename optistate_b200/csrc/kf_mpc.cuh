// SURVEY 8(f) row 3: the reference's convex force MPC (misc/force_controller.py:15-225 as Kalman_Filter.predict_mpc sets
// it up, kalman_filter/kalman_filter.py:64-77,140-152), batched: one QP per problem, one WARP per problem.
//
//   horizon NH = 5, u = 12 forces per stage (60 unknowns, stage-major), dynamics linearised around body_mpc[:, i]
//   (column 0 = the current state x, columns 1..5 = body_ref), feet p constant over the horizon:
//       state_{i+1} = (I + dt A_i) state_i + dt B_i u_i + dt g                                    force_controller.py:70-93
//       cost = sum_i (state_{i+1} - body_mpc[:, i+1])^T W (.) + u_i^T R u_i                        force_controller.py:95-104
//       contact == 0: f = 0;  contact == 1: fz <= fz_max, |fx| <= mu fz, |fy| <= mu fz (=> fz >= 0);  other: free   :106-156
//
// The reference hands this to CasADi + qpOASES (an active-set solver), neither of which exists offline.  The QP itself is
// pinned to the reference (the test infrastructure evaluates the unmodified set-up code numerically; golden fixture
// tests/golden/mpc_reference_qp.npz); the SOLVER is unpinned, but the QP is strictly convex (R > 0), so its minimiser is
// unique and any exact solver agrees with qpOASES to solver tolerance.
// Here: swing legs are left out of the unknowns (order n = 15 x legs not in swing), the condensed Hessian H (packed lower
// triangle, <= 1,830 doubles) and gradient g are built in shared memory, a Mehrotra predictor-corrector interior-point
// method brings the iterate to complementarity ~1e-9, and a polish phase (method of multipliers on the identified active
// set, with active-set corrections) removes the interior-point bias: <= 3e-10 of max|u| against an independent active-set
// solve (oracle/mpc_numpy.py) over 256 problems covering every contact pattern (tests/test_mpc_gpu.py).  The normal-equations matrix H + A^T D A only ever gains 3x3 diagonal blocks, because
// every constraint row touches one leg of one stage.
#pragma once

#include "kf_common.cuh"
#include "kf_mpc_params.cuh"

namespace okf {

constexpr int MPC_NH = 5;
constexpr int MPC_N = 12 * MPC_NH;                  // unknowns
constexpr int MPC_TRI = MPC_N * (MPC_N + 1) / 2;    // packed lower triangle
constexpr int MPC_WARPS = 2;                        // problems per block
constexpr int MPC_VEC = 6;                          // per-warp vectors of MPC_N doubles: u, g, r, d, u_keep, 1 / pivots
constexpr int MPC_MAX_IPM = 40;
constexpr int MPC_POLISH_ROUNDS = 16;
constexpr int MPC_MOM_ITERS = 8;

// Shared memory is sized for the largest number of legs not in swing that the batch contains (max_legs, 1..4; the host
// passes 4 when it does not know): order nmax = 15 max_legs.  A trot (two stance legs) then needs 9 KB per problem
// instead of 32 KB, which is what decides how many warps an SM can hold for this latency-bound kernel.
__host__ __device__ constexpr int mpc_mat_doubles(int max_legs) {  // H or M: packed triangle; M also hosts the 12 x nmax sensitivities
    return (15 * max_legs) * (15 * max_legs + 1) / 2 > 12 * 15 * max_legs ? (15 * max_legs) * (15 * max_legs + 1) / 2 : 12 * 15 * max_legs;
}
__host__ __device__ constexpr int mpc_warp_doubles(int max_legs) { return 2 * mpc_mat_doubles(max_legs) + MPC_VEC * 15 * max_legs; }
__host__ __device__ constexpr size_t mpc_smem_bytes(int max_legs) { return (size_t)MPC_WARPS * mpc_warp_doubles(max_legs) * sizeof(double); }

__device__ __forceinline__ int tri_idx(int i, int j) { return i * (i + 1) / 2 + j; }  // j <= i
__device__ __forceinline__ double sym_at(const double *P, int i, int j) { return i >= j ? P[tri_idx(i, j)] : P[tri_idx(j, i)]; }
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// constraint rows of one stance block (fx, fy, fz):  r0: fz <= fz_max;  r1: fx - mu fz <= 0;  r2: -fx - mu fz <= 0;
// r3: fy - mu fz <= 0;  r4: -fy - mu fz <= 0   (fz >= 0 follows from r1 + r2)
__device__ __forceinline__ void rows_times(const double *ub, double mu, double (&au)[5]) {
    au[0] = ub[2];
    au[1] = ub[0] - mu * ub[2];
    au[2] = -ub[0] - mu * ub[2];
    au[3] = ub[1] - mu * ub[2];
    au[4] = -ub[1] - mu * ub[2];
}
__device__ __forceinline__ void rows_transpose_times(const double (&t)[5], double mu, double (&out)[3]) {
    out[0] = t[1] - t[2];
    out[1] = t[3] - t[4];
    out[2] = t[0] - mu * (t[1] + t[2] + t[3] + t[4]);
}
// lower triangle of sum_r d_r a_r a_r^T (xx, yx, yy, zx, zy, zz)
__device__ __forceinline__ void rows_gram(const double (&d)[5], double mu, double (&gm)[6]) {
    gm[0] = d[1] + d[2];
    gm[1] = 0.0;
    gm[2] = d[3] + d[4];
    gm[3] = -mu * (d[1] - d[2]);
    gm[4] = -mu * (d[3] - d[4]);
    gm[5] = d[0] + mu * mu * (d[1] + d[2] + d[3] + d[4]);
}

// In-place Cholesky of the packed lower triangle (row-major, order n) by one warp, left-looking: column k is produced
// from the finished columns to its left, lane by row, as a dot product of two rows - two shared-memory loads per FMA and
// one store per ENTRY (the right-looking form re-writes the whole trailing matrix at every step: a store per FMA).  dinv
// receives 1 / L_kk.  Returns false on a non-positive pivot.
__device__ __forceinline__ bool warp_cholesky(double *M, double *dinv, int n, int lane) {
    for (int k = 0; k < n; ++k) {
        const double *rk = M + tri_idx(k, 0);
        for (int i = k + lane; i < n; i += 32) {
            double *ri = M + tri_idx(i, 0);
            double a0 = ri[k], a1 = 0.0;
            int j = 0;
            for (; j + 1 < k; j += 2) {
                a0 = fma(-ri[j], rk[j], a0);
                a1 = fma(-ri[j + 1], rk[j + 1], a1);
            }
            if (j < k) a0 = fma(-ri[j], rk[j], a0);
            ri[k] = a0 + a1;
        }
        __syncwarp();
        const double dkk = rk[k];
        if (!(dkk > 0.0)) return false;  // warp-uniform
        const double inv = 1.0 / sqrt(dkk);
        __syncwarp();
        for (int i = k + 1 + lane; i < n; i += 32) M[tri_idx(i, k)] *= inv;
        if (lane == 0) { M[tri_idx(k, k)] = dkk * inv; dinv[k] = inv; }
        __syncwarp();
    }
    return true;
}

// v <- (L L^T)^-1 v, v in shared memory
__device__ __forceinline__ void warp_chol_solve(const double *L, const double *dinv, double *v, int n, int lane) {
    for (int j = 0; j < n; ++j) {  // forward, column oriented
        __syncwarp();
        const double yj = v[j] * dinv[j];
        __syncwarp();
        if (lane == 0) v[j] = yj;
        for (int i = j + 1 + lane; i < n; i += 32) v[i] = fma(-L[tri_idx(i, j)], yj, v[i]);
    }
    for (int i = n - 1; i >= 0; --i) {  // backward: L^T x = y, row i of L updates the entries above it
        __syncwarp();
        const double xi = v[i] * dinv[i];
        __syncwarp();
        if (lane == 0) v[i] = xi;
        const double *row = L + tri_idx(i, 0);
        for (int j = lane; j < i; j += 32) v[j] = fma(-row[j], xi, v[j]);
    }
    __syncwarp();
}

// out <- H v for the packed symmetric H of order n
__device__ __forceinline__ void warp_symv(const double *H, const double *v, double *out, int n, int lane) {
    for (int i = lane; i < n; i += 32) {
        double acc = 0.0;
        for (int j = 0; j < n; ++j) acc = fma(sym_at(H, i, j), v[j], acc);
        out[i] = acc;
    }
    __syncwarp();
}

__global__ void __launch_bounds__(32 * MPC_WARPS) kf_mpc_kernel(const __grid_constant__ MpcParams prm) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long prob = (long long)blockIdx.x * MPC_WARPS + warp;
    if (prob >= prm.N) return;  // whole warp
    if (prm.only_flagged && prm.status[prob] != MPC_ST_GIVEN_UP) return;  // second launch behind the dual active-set kernel
    const int nmax = 15 * prm.max_legs, ld = nmax;  // ld: row stride of the sensitivities
    double *base = reinterpret_cast<double *>(smem_raw) + (size_t)warp * mpc_warp_doubles(prm.max_legs);
    double *H = base, *M = base + mpc_mat_doubles(prm.max_legs);
    double *u = M + mpc_mat_doubles(prm.max_legs), *g = u + nmax, *rv = g + nmax, *dv = rv + nmax, *ukeep = dv + nmax, *dinv = ukeep + nmax;
    double *Su = M;  // [12][nmax] sensitivity of the stage state to the forces: only needed while H is built, M only after
    const long long N = prm.N;

    // ---- problem data --------------------------------------------------------------------------------------
    // body[:, 0] = x, body[:, i] = body_ref[:, i - 1]; kind of leg: 0 pinned (swing), 1 pyramid (stance), 2 free
    int kind_leg[4];
#pragma unroll
    for (int l = 0; l < 4; ++l) {
        const double c = prm.contact[l * N + prob];
        kind_leg[l] = c == 0.0 ? 0 : (c == 1.0 ? 1 : 2);
    }
    // Swing legs carry no force: their unknowns are left out altogether.  Compact unknown 3 (nfl i + r) + c = component c
    // of the r-th leg that is not in swing at stage i; order n = 15 nfl, nb = 5 nfl blocks, lane b owns block b.
    int free_leg[4] = {0, 0, 0, 0}, nfl = 0;
#pragma unroll
    for (int l = 0; l < 4; ++l)
        if (kind_leg[l] != 0) {
#pragma unroll
            for (int r = 0; r < 4; ++r)
                if (r == nfl) free_leg[r] = l;
            ++nfl;
        }
    if (nfl > prm.max_legs) {  // the caller's bound on the legs not in swing is wrong for this problem: no answer
        for (int e = lane; e < MPC_N; e += 32) prm.forces[(long long)e * N + prob] = __longlong_as_double(0x7ff8000000000000LL);
        if (prm.status && lane == 0) prm.status[prob] = 4u;
        return;
    }
    const int n = 15 * nfl, nb = 5 * nfl, ntri = n * (n + 1) / 2;
    int my_leg = 0;
#pragma unroll
    for (int r = 0; r < 4; ++r)
        if (nfl > 0 && r == lane % (nfl > 0 ? nfl : 1)) my_leg = free_leg[r];
    int my_kind = 0;
#pragma unroll
    for (int l = 0; l < 4; ++l)
        if (l == my_leg) my_kind = kind_leg[l];
    if (lane >= nb) my_kind = 0;
    const bool my_act = my_kind == 1;
    const double mu_f = prm.mu;

    // ---- condensed QP: H = 2 sum_i Su_i^T W Su_i + 2 R,  g = 2 sum_i Su_i^T W (sc_i - ref_i) ----------------------
    for (int e = lane; e < ntri; e += 32) H[e] = 0.0;
    for (int e = lane; e < 12 * ld; e += 32) Su[e] = 0.0;
    __syncwarp();  // the diagonal entries below were zeroed by other lanes
    for (int e = lane; e < n; e += 32) { g[e] = 0.0; H[tri_idx(e, e)] = 2.0 * prm.w_force; }
    double sc[12];  // free response of the state (replicated in every lane)
#pragma unroll
    for (int k = 0; k < 12; ++k) sc[k] = prm.x[k * N + prob];
    double pf[12];
#pragma unroll
    for (int k = 0; k < 12; ++k) pf[k] = prm.p[k * N + prob];
    __syncwarp();
    for (int i = 0; i < MPC_NH; ++i) {
        double th[3];  // linearisation angles: body_mpc[0:3, i] = the current state for stage 0, body_ref[:, i - 1] after
#pragma unroll
        for (int k = 0; k < 3; ++k) th[k] = i == 0 ? prm.x[k * N + prob] : prm.body_ref[((i - 1) * 12 + k) * N + prob];
        double R[9];
        rot_zyx(th[0], th[1], th[2], R);
        // Su <- (I + dt A) Su: rows 0..2 += dt R^T rows 6..8, rows 3..5 += dt rows 9..11 (rows 6..11 unchanged)
        for (int c = lane; c < n; c += 32) {
            const double w0 = Su[6 * ld + c], w1 = Su[7 * ld + c], w2 = Su[8 * ld + c];
#pragma unroll
            for (int a = 0; a < 3; ++a)
                Su[a * ld + c] += prm.dt * (R[0 * 3 + a] * w0 + R[1 * 3 + a] * w1 + R[2 * 3 + a] * w2);  // R^T[a][k] = R[k][a]
#pragma unroll
            for (int a = 0; a < 3; ++a) Su[(3 + a) * ld + c] += prm.dt * Su[(9 + a) * ld + c];
        }
        __syncwarp();
        // Su[:, 12 i + 3 l + c] += dt B: rows 6..8 = Ihat^-1 skew(R p_l), rows 9..11 = I / m;  Ihat^-1 = R diag(1/I) R^T
        if (lane < 3 * nfl) {
            const int c = lane % 3;
            int l = 0;
#pragma unroll
            for (int r = 0; r < 4; ++r)
                if (r == lane / 3) l = free_leg[r];
            double pw[3];
#pragma unroll
            for (int a = 0; a < 3; ++a) pw[a] = R[3 * a] * pf[3 * l] + R[3 * a + 1] * pf[3 * l + 1] + R[3 * a + 2] * pf[3 * l + 2];
            // column c of skew(pw): skew = [[0,-z,y],[z,0,-x],[-y,x,0]]
            double sk[3];
            sk[0] = c == 0 ? 0.0 : (c == 1 ? -pw[2] : pw[1]);
            sk[1] = c == 0 ? pw[2] : (c == 1 ? 0.0 : -pw[0]);
            sk[2] = c == 0 ? -pw[1] : (c == 1 ? pw[0] : 0.0);
            double t3[3];  // diag(1/I) R^T sk
#pragma unroll
            for (int a = 0; a < 3; ++a) t3[a] = prm.inv_inertia[a] * (R[a] * sk[0] + R[3 + a] * sk[1] + R[6 + a] * sk[2]);
            const int col = 3 * nfl * i + lane;
#pragma unroll
            for (int a = 0; a < 3; ++a) Su[(6 + a) * ld + col] += prm.dt * (R[3 * a] * t3[0] + R[3 * a + 1] * t3[1] + R[3 * a + 2] * t3[2]);
            Su[(9 + c) * ld + col] += prm.dt * prm.inv_mass;
        }
        // free response: sc <- (I + dt A) sc + dt g
        {
            const double w0 = sc[6], w1 = sc[7], w2 = sc[8];
#pragma unroll
            for (int a = 0; a < 3; ++a) sc[a] += prm.dt * (R[a] * w0 + R[3 + a] * w1 + R[6 + a] * w2);
#pragma unroll
            for (int a = 0; a < 3; ++a) sc[3 + a] += prm.dt * sc[9 + a];
            sc[11] += prm.dt * prm.gravity;
        }
        double we[12];  // W (sc - ref)
#pragma unroll
        for (int k = 0; k < 12; ++k) we[k] = prm.w_state[k] * (sc[k] - prm.body_ref[(i * 12 + k) * N + prob]);
        __syncwarp();
        const int ncol = 3 * nfl * (i + 1);  // later columns of Su are still zero
        for (int a = 0; a < ncol; ++a) {
            double sa[12];
#pragma unroll
            for (int k = 0; k < 12; ++k) sa[k] = prm.w_state[k] * Su[k * ld + a];
            for (int b = lane; b <= a; b += 32) {
                double acc = 0.0;
#pragma unroll
                for (int k = 0; k < 12; ++k) acc = fma(sa[k], Su[k * ld + b], acc);
                H[tri_idx(a, b)] += 2.0 * acc;
            }
        }
        for (int a = lane; a < ncol; a += 32) {
            double acc = 0.0;
#pragma unroll
            for (int k = 0; k < 12; ++k) acc = fma(Su[k * ld + a], we[k], acc);
            g[a] += 2.0 * acc;
        }
        __syncwarp();
    }
    double hmax = 0.0, gmax = 0.0;
    for (int e = lane; e < n; e += 32) {
        hmax = fmax(hmax, H[tri_idx(e, e)]);
        gmax = fmax(gmax, fabs(g[e]));
    }
    hmax = warp_max(hmax);
    const double gs = fmax(warp_max(gmax), 1e-300);

    // ---- interior point ------------------------------------------------------------------------------------------
    const double bvec[5] = {prm.fz_max, 0.0, 0.0, 0.0, 0.0};
    for (int e = lane; e < n; e += 32) u[e] = 0.0;
    __syncwarp();
    if (my_act) u[3 * lane + 2] = fmin(10.0, 0.5 * prm.fz_max);  // strictly inside the pyramid
    __syncwarp();
    double s[5], lam[5];
    {
        double au[5];
        rows_times(u + 3 * (lane < nb ? lane : 0), mu_f, au);
#pragma unroll
        for (int r = 0; r < 5; ++r) { s[r] = my_act ? bvec[r] - au[r] : 1.0; lam[r] = my_act ? 1.0 / s[r] : 0.0; }
    }
    const double m_act = warp_sum(my_act ? 5.0 : 0.0);
    uint32_t status = 0;
    int it = 0;
    for (; it < MPC_MAX_IPM; ++it) {
        // residuals: rd = H u + g + A^T lam (free entries), rp = A u + s - b
        warp_symv(H, u, rv, n, lane);
        double rp[5] = {0, 0, 0, 0, 0};
        if (lane < nb) {
            double atl[3] = {0, 0, 0};
            if (my_act) {
                double au[5];
                rows_times(u + 3 * lane, mu_f, au);
#pragma unroll
                for (int r = 0; r < 5; ++r) rp[r] = au[r] + s[r] - bvec[r];
                rows_transpose_times(lam, mu_f, atl);
            }
#pragma unroll
            for (int c = 0; c < 3; ++c) rv[3 * lane + c] += g[3 * lane + c] + atl[c];
        }
        __syncwarp();
        double rdmax = 0.0, rpmax = 0.0, comp = 0.0;
        for (int e = lane; e < n; e += 32) rdmax = fmax(rdmax, fabs(rv[e]));
#pragma unroll
        for (int r = 0; r < 5; ++r) { rpmax = fmax(rpmax, fabs(rp[r])); comp += my_act ? s[r] * lam[r] : 0.0; }
        rdmax = warp_max(rdmax) / gs;
        rpmax = warp_max(rpmax) / prm.fz_max;
        const double mu_c = m_act > 0.0 ? warp_sum(comp) / m_act : 0.0;
        if (it > 0 && (m_act == 0.0 || mu_c < 1e-9) && fmax(rdmax, rpmax) < 1e-8) break;
        // M = H + A^T (lam / s) A
        for (int e = lane; e < ntri; e += 32) M[e] = H[e];
        __syncwarp();
        if (my_act) {
            double d[5], gm[6];
#pragma unroll
            for (int r = 0; r < 5; ++r) d[r] = lam[r] / s[r];
            rows_gram(d, mu_f, gm);
            const int o = 3 * lane;
            M[tri_idx(o, o)] += gm[0];
            M[tri_idx(o + 1, o)] += gm[1];
            M[tri_idx(o + 1, o + 1)] += gm[2];
            M[tri_idx(o + 2, o)] += gm[3];
            M[tri_idx(o + 2, o + 1)] += gm[4];
            M[tri_idx(o + 2, o + 2)] += gm[5];
        }
        __syncwarp();
        // a pivot breakdown once the complementarity is at its target is where the barrier ends at FP64 resolution (lam / s of
        // the active rows near 1e16: seen at gravity -15 on a one-leg stance), not a failure - the polish below settles the
        // active set from this iterate and flags what it cannot
        if (!warp_cholesky(M, dinv, n, lane)) { if (!(mu_c < 1e-9)) status |= 1u; break; }
        if (m_act == 0.0) {  // unconstrained: one Newton step is the answer
            for (int e = lane; e < n; e += 32) dv[e] = -rv[e];
            warp_chol_solve(M, dinv, dv, n, lane);
            for (int e = lane; e < n; e += 32) u[e] += dv[e];
            __syncwarp();
            continue;
        }
        double ds[5] = {0, 0, 0, 0, 0}, dl[5] = {0, 0, 0, 0, 0}, rc[5];
        double alpha_aff_p = 1.0, alpha_aff_d = 1.0;
        for (int pass = 0; pass < 2; ++pass) {
            // pass 0: affine direction (rc = s lam); pass 1: corrector (rc = s lam + ds dl - sigma mu)
            double sigma_mu = 0.0;
            if (pass == 1) {
                double comp_aff = 0.0;
#pragma unroll
                for (int r = 0; r < 5; ++r) comp_aff += my_act ? (s[r] + alpha_aff_p * ds[r]) * (lam[r] + alpha_aff_d * dl[r]) : 0.0;
                const double mu_aff = warp_sum(comp_aff) / m_act;
                const double ratio = mu_aff / mu_c;
                sigma_mu = ratio * ratio * ratio * mu_c;
            }
#pragma unroll
            for (int r = 0; r < 5; ++r) rc[r] = s[r] * lam[r] + (pass == 1 ? ds[r] * dl[r] - sigma_mu : 0.0);
            for (int e = lane; e < n; e += 32) dv[e] = -rv[e];
            __syncwarp();
            if (my_act) {
                double t[5], att[3];
#pragma unroll
                for (int r = 0; r < 5; ++r) t[r] = (-rc[r] + lam[r] * rp[r]) / s[r];
                rows_transpose_times(t, mu_f, att);
#pragma unroll
                for (int c = 0; c < 3; ++c) dv[3 * lane + c] -= att[c];
            }
            __syncwarp();
            warp_chol_solve(M, dinv, dv, n, lane);
            if (my_act) {
                double adu[5];
                rows_times(dv + 3 * lane, mu_f, adu);
#pragma unroll
                for (int r = 0; r < 5; ++r) {
                    ds[r] = -rp[r] - adu[r];
                    dl[r] = (-rc[r] - lam[r] * ds[r]) / s[r];
                }
            }
            double ap = 1.0, ad = 1.0;
#pragma unroll
            for (int r = 0; r < 5; ++r) {
                if (my_act && ds[r] < 0.0) ap = fmin(ap, -s[r] / ds[r]);
                if (my_act && dl[r] < 0.0) ad = fmin(ad, -lam[r] / dl[r]);
            }
            ap = warp_min(ap);
            ad = warp_min(ad);
            if (pass == 0) { alpha_aff_p = ap; alpha_aff_d = ad; }
            else {
                const double a = fmin(fmin(1.0, 0.995 * ap), fmin(1.0, 0.995 * ad));
                for (int e = lane; e < n; e += 32) u[e] = fma(a, dv[e], u[e]);
#pragma unroll
                for (int r = 0; r < 5; ++r) { s[r] = fma(a, ds[r], s[r]); lam[r] = fma(a, dl[r], lam[r]); }
            }
            __syncwarp();
        }
    }
    if (it >= MPC_MAX_IPM) status |= 1u;

    // ---- polish: method of multipliers on the identified active set, with active-set corrections -------------
    if (m_act > 0.0) {
        for (int e = lane; e < n; e += 32) ukeep[e] = u[e];
        bool W[5];
        double lw[5];
#pragma unroll
        for (int r = 0; r < 5; ++r) { W[r] = my_act && s[r] * (gs / prm.fz_max) < lam[r]; lw[r] = W[r] ? lam[r] : 0.0; }
        const double rho = 1e2 * hmax;
        bool ok = false;
        for (int rnd = 0; rnd < MPC_POLISH_ROUNDS && !ok; ++rnd) {
            for (int e = lane; e < ntri; e += 32) M[e] = H[e];
            __syncwarp();
            if (my_act) {
                double d[5], gm[6];
#pragma unroll
                for (int r = 0; r < 5; ++r) d[r] = W[r] ? rho : 0.0;
                rows_gram(d, mu_f, gm);
                const int o = 3 * lane;
                M[tri_idx(o, o)] += gm[0];
                M[tri_idx(o + 1, o)] += gm[1];
                M[tri_idx(o + 1, o + 1)] += gm[2];
                M[tri_idx(o + 2, o)] += gm[3];
                M[tri_idx(o + 2, o + 1)] += gm[4];
                M[tri_idx(o + 2, o + 2)] += gm[5];
            }
            __syncwarp();
            if (!warp_cholesky(M, dinv, n, lane)) break;
            double au[5] = {0, 0, 0, 0, 0};
            for (int k = 0; k < MPC_MOM_ITERS; ++k) {
                for (int e = lane; e < n; e += 32) dv[e] = -g[e];
                __syncwarp();
                if (my_act) {
                    double t[5], att[3];
#pragma unroll
                    for (int r = 0; r < 5; ++r) t[r] = W[r] ? -lw[r] + rho * bvec[r] : 0.0;
                    rows_transpose_times(t, mu_f, att);
#pragma unroll
                    for (int c = 0; c < 3; ++c) dv[3 * lane + c] += att[c];
                }
                __syncwarp();
                warp_chol_solve(M, dinv, dv, n, lane);
                if (my_act) {
                    rows_times(dv + 3 * lane, mu_f, au);
#pragma unroll
                    for (int r = 0; r < 5; ++r) lw[r] = W[r] ? lw[r] + rho * (au[r] - bvec[r]) : 0.0;
                }
                __syncwarp();
            }
            // active-set correction.  The first two rounds take every violated constraint in and every negative multiplier
            // out at once (one round is almost always enough); after that ONE change per round - the most violated
            // constraint, or else the most negative multiplier - because simultaneous changes can cycle.
            bool infeas[5], neg[5], any_inf = false, any_neg = false;
            double worst_inf = 0.0, worst_neg = 0.0;
            int r_inf = -1, r_neg = -1;
#pragma unroll
            for (int r = 0; r < 5; ++r) {
                infeas[r] = my_act && !W[r] && au[r] - bvec[r] > 1e-9 * prm.fz_max;
                neg[r] = W[r] && lw[r] < -1e-9 * gs;
                any_inf |= infeas[r];
                any_neg |= neg[r];
                if (infeas[r] && au[r] - bvec[r] > worst_inf) { worst_inf = au[r] - bvec[r]; r_inf = r; }
                if (neg[r] && lw[r] < worst_neg) { worst_neg = lw[r]; r_neg = r; }
            }
            const bool warp_inf = __any_sync(0xffffffffu, any_inf), warp_neg = __any_sync(0xffffffffu, any_neg);
            ok = !warp_inf && !warp_neg;
            if (!ok && rnd < 2) {
#pragma unroll
                for (int r = 0; r < 5; ++r) {
                    if (infeas[r]) { W[r] = true; lw[r] = 0.0; }
                    if (neg[r]) { W[r] = false; lw[r] = 0.0; }
                }
            } else if (!ok) {
                const double mine = warp_inf ? worst_inf : -worst_neg;           // >= 0, larger is worse
                const double worst = warp_max(mine);
                const unsigned cand = __ballot_sync(0xffffffffu, (warp_inf ? r_inf : r_neg) >= 0 && mine == worst);
                if (lane == __ffs(cand) - 1) {
#pragma unroll
                    for (int r = 0; r < 5; ++r) {
                        if (warp_inf && r == r_inf) { W[r] = true; lw[r] = 0.0; }
                        if (!warp_inf && r == r_neg) { W[r] = false; lw[r] = 0.0; }
                    }
                }
            }
        }
        if (ok) {
            for (int e = lane; e < n; e += 32) u[e] = dv[e];
        } else {
            for (int e = lane; e < n; e += 32) u[e] = ukeep[e];
            status |= 2u;
        }
        __syncwarp();
    }
    for (int e = lane; e < MPC_N; e += 32) prm.forces[(long long)e * N + prob] = 0.0;
    __syncwarp();
    for (int e = lane; e < n; e += 32) {  // compact -> (stage, leg, component)
        const int stage = e / (3 * nfl), within = e % (3 * nfl);
        int l = 0;
#pragma unroll
        for (int r = 0; r < 4; ++r)
            if (r == within / 3) l = free_leg[r];
        prm.forces[(long long)(12 * stage + 3 * l + within % 3) * N + prob] = u[e];
    }
    if (prm.status && lane == 0) prm.status[prob] = status | ((uint32_t)it << 8);
}

}  // namespace okf
