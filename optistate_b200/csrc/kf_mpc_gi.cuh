// Batched force MPC, dual active-set solver (Goldfarb & Idnani 1983) - the primary path of optistate_kf_mpc_forces: one warp per
// problem for at most two legs out of swing (a trot, kf_mpc_gi_kernel), two warps for three and four (kf_mpc_gi2_kernel).  Same
// QP and same minimiser as the interior point of kf_mpc.cuh (the QP is strictly convex: the minimiser is unique and the method
// terminates at it); what changes is the work per problem:
//
//   * the interior point refactorises the n x n normal equations every iteration (~13 factorisations + ~30 triangular solves
//     per QP, each a chain of n dependent columns).  But H is FIXED per problem and every constraint row touches one leg of one
//     stage (three unknowns), so here H is inverted ONCE - symmetric sweeps, lane i owns row i in registers, one broadcast
//     through a shared-memory strip per column - and everything after that is small:
//   * the method starts at the unconstrained minimiser -H^-1 g and adds the most violated constraint p at a time.  With N the
//     normals of the working set: y = H^-1 n_p is THREE columns of H^-1 combined; d = N^T y three products per working
//     constraint; r = S^-1 d a q x q product with S^-1 = (N^T H^-1 N)^-1 KEPT EXPLICITLY and updated by the bordering formula
//     when a constraint enters and by a rank-one downdate when one leaves (no factorisation, no dependent chain); the primal
//     direction z = y - H^-1 N r three columns per working constraint.  One iteration is a few hundred instructions on
//     shared memory instead of a factorisation, and the ~14 iterations of a saturated trot problem cost about what ONE
//     interior-point iteration costs.
//   * a partial step (a multiplier reaches zero first) drops that constraint and repeats with the same p; a normal that is
//     linearly dependent on the working set (the apex of the friction pyramid: four faces, three unknowns) takes the dual
//     step alone, exactly as in the paper.
//   * the loop is rolled and compact (it fits the 32 KB instruction cache); only the inversion is straight-line code, run once.
//   * a problem the method gives up on (iteration cap, working set full, a breakdown of S^-1) is flagged and solved by the
//     interior-point kernel (kf_mpc_kernel, kf_mpc.cuh) in a second launch that only touches flagged problems.
// Measured against the independent active-set solve of the test infrastructure: see tests/test_mpc_gpu.py.
#pragma once

#include <type_traits>

#include "kf_mpc.cuh"

namespace okf {

constexpr int MPCG_MAX_LEGS = 2;  // legs out of swing the one-warp kernel is instantiated for

__host__ __device__ constexpr int mpcg_even(int v) { return v + (v & 1); }

// Reciprocal of a positive normal number, straight-line (20-bit seed + two Newton steps: rounding-limited): the IEEE division is a
// call into a ~70-instruction slow-path routine, and the inversion of H takes one per pivot, every constraint change several more.
__device__ __forceinline__ double rcp2_(double a) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(a));
    double e = fma(-a, r, 1.0);
    r = fma(r, e, r);
    e = fma(-a, r, 1.0);
    return fma(r, e, r);
}

// The threads that work on one problem: one warp, or - for the orders 45 and 60 of three and four legs out of swing in
// kf_mpc_gi.cuh - the two warps of a 64-thread block.  Thread t of the group owns row t / slot t / constraint block t.
// `scr`: eight doubles of shared memory per problem (only the two-warp form touches it).
__device__ __forceinline__ void warp_argmin(double &v, int &idx) {  // smallest (value, index); ties to the smaller index; index < 0 = none
    // Three warp-wide integer reductions (REDUX) on an order-preserving 64-bit key instead of five rounds of three shuffles and a
    // compare chain: the high word, the low word among the lanes that hold the smallest high word, then the index among those.
    unsigned long long u = (unsigned long long)__double_as_longlong(v);
    u = (u >> 63) ? ~u : (u | 0x8000000000000000ull);  // ascending as unsigned: negative values below positive ones
    if (idx < 0) u = ~0ull;
    const unsigned hi = (unsigned)(u >> 32), lo = (unsigned)u;
    const unsigned mhi = __reduce_min_sync(0xffffffffu, hi);
    const unsigned mlo = __reduce_min_sync(0xffffffffu, hi == mhi ? lo : 0xffffffffu);
    const bool mine = idx >= 0 && hi == mhi && lo == mlo;
    const unsigned midx = __reduce_min_sync(0xffffffffu, mine ? (unsigned)idx : 0xffffffffu);
    if (midx == 0xffffffffu) { idx = -1; return; }  // no candidate (v is left as it is)
    unsigned long long m = ((unsigned long long)mhi << 32) | mlo;
    m = (m >> 63) ? (m & 0x7fffffffffffffffull) : ~m;
    v = __longlong_as_double((long long)m);
    idx = (int)midx;
}
template <int NW>
struct MpcGroup;
template <>
struct MpcGroup<1> {
    static constexpr int threads = 32;
    static __device__ __forceinline__ int tid() { return threadIdx.x & 31; }
    static __device__ __forceinline__ void sync() { __syncwarp(); }
    static __device__ __forceinline__ double sum(double v, double *) { return warp_sum(v); }
    static __device__ __forceinline__ double max(double v, double *) { return warp_max(v); }
    static __device__ __forceinline__ void argmin(double &v, int &idx, double *) { warp_argmin(v, idx); }
};
template <>
struct MpcGroup<2> {  // one problem per 64-thread block
    static constexpr int threads = 64;
    static __device__ __forceinline__ int tid() { return threadIdx.x; }
    static __device__ __forceinline__ void sync() { __syncthreads(); }
    static __device__ __forceinline__ double sum(double v, double *scr) {
        v = warp_sum(v);
        if ((threadIdx.x & 31) == 0) scr[threadIdx.x >> 5] = v;
        __syncthreads();
        v = scr[0] + scr[1];
        __syncthreads();
        return v;
    }
    static __device__ __forceinline__ double max(double v, double *scr) {
        v = warp_max(v);
        if ((threadIdx.x & 31) == 0) scr[threadIdx.x >> 5] = v;
        __syncthreads();
        v = fmax(scr[0], scr[1]);
        __syncthreads();
        return v;
    }
    static __device__ __forceinline__ void argmin(double &v, int &idx, double *scr) {
        warp_argmin(v, idx);
        if ((threadIdx.x & 31) == 0) {
            scr[2 + 2 * (threadIdx.x >> 5)] = v;
            scr[3 + 2 * (threadIdx.x >> 5)] = (double)idx;
        }
        __syncthreads();
        const double v0 = scr[2], v1 = scr[4];
        const int i0 = (int)scr[3], i1 = (int)scr[5];
        const bool second = i1 >= 0 && (i0 < 0 || v1 < v0 || (v1 == v0 && i1 < i0));
        v = second ? v1 : v0;
        idx = second ? i1 : i0;
        __syncthreads();
    }
};

// Condensed QP, thread by row in registers: hrow <- row `lane` of 2 sum_i Su_i^T W Su_i (WITHOUT the 2 w_force of the diagonal),
// grow <- entry `lane` of g = 2 sum_i Su_i^T W (sc_i - ref_i).  `lane` is the thread's index in its group (MpcGroup<NW>).
// Unknown 3 (NFL i + r) + c = component c of free_leg[r] at stage i; a free_leg entry that is a swing leg is a phantom (no
// dynamics: its row and column are zero).
// scratch: shared memory, mpc_condense_scratch(NFL) doubles: the sensitivities Su [12][ld] of the stage state to the forces, the five
// rotation matrices of the horizon and its 60 reference values.
//   * the rotations (three sin / cos pairs each) are evaluated ONCE, stage i by thread i, instead of by every thread in every
//     stage; the reference states are fetched once, coalesced, instead of one dependent global load per use;
//   * rows 3..5 and 9..11 of Su (position and velocity sensitivities) are known in closed form - a force component c of stage j
//     changes velocity c by dt / m from stage j on and position c by (i - j) dt^2 / m at stage i, nothing else - so their part of
//     the Gram matrix, sum_i over the common stages of w_pos (i - j)(i - j') (dt^2 / m)^2 + w_vel (dt / m)^2 for equal components,
//     is added once at the end, and the per-stage accumulation runs over the six attitude / body-rate rows only (pairs of columns
//     per 16-byte load): half the FMAs and a third of the shared-memory loads of the straightforward form.
__host__ __device__ constexpr int mpc_condense_scratch(int nfl) { return 12 * mpcg_even(15 * nfl) + 48 + 64; }

template <int NFL, int NW = 1>
__device__ __forceinline__ void mpc_condense(const MpcParams &prm, long long prob, int lane, const int (&kind_leg)[4], const int (&free_leg)[4],
                                             double *scratch, double (&hrow)[15 * NFL], double &grow) {
    using G = MpcGroup<NW>;
    constexpr int n = 15 * NFL, ld = mpcg_even(n), GT = G::threads;
    const long long N = prm.N;
    const int row = lane < n ? lane : n - 1;
    double *Su = scratch, *Rs = scratch + 12 * ld, *bref = Rs + 48;  // Rs [5][9] (padded), bref [5][12]
    for (int e = lane; e < 12 * ld; e += GT) Su[e] = 0.0;
    for (int e = lane; e < MPC_NH * 12; e += GT) bref[e] = prm.body_ref[(long long)e * N + prob];
    grow = 0.0;
#pragma unroll
    for (int j = 0; j < n; ++j) hrow[j] = 0.0;
    double sc[12], pf[12];
#pragma unroll
    for (int k = 0; k < 12; ++k) sc[k] = prm.x[k * N + prob];
#pragma unroll
    for (int k = 0; k < 12; ++k) pf[k] = prm.p[k * N + prob];
    bool real[NFL];  // leg r of the unknowns carries a force (not a phantom)
#pragma unroll
    for (int r = 0; r < NFL; ++r) {
        real[r] = false;
#pragma unroll
        for (int q = 0; q < 4; ++q)
            if (q == free_leg[r]) real[r] = kind_leg[q] != 0;
    }
    G::sync();
    if (lane < MPC_NH) {  // linearisation attitude of stage i: the current state for stage 0, body_ref[:, i - 1] after
        double R[9];
        if (lane == 0) rot_zyx(sc[0], sc[1], sc[2], R);
        else rot_zyx(bref[(lane - 1) * 12], bref[(lane - 1) * 12 + 1], bref[(lane - 1) * 12 + 2], R);
#pragma unroll
        for (int k = 0; k < 9; ++k) Rs[9 * lane + k] = R[k];
    }
    G::sync();
#pragma unroll 1
    for (int i = 0; i < MPC_NH; ++i) {
        double R[9];
#pragma unroll
        for (int k = 0; k < 9; ++k) R[k] = Rs[9 * i + k];
        // Su <- (I + dt A) Su: rows 0..2 += dt R^T rows 6..8, rows 3..5 += dt rows 9..11 (rows 6..11 unchanged)
        if (lane < n) {
            const int c = lane;
            const double w0 = Su[6 * ld + c], w1 = Su[7 * ld + c], w2 = Su[8 * ld + c];
#pragma unroll
            for (int a = 0; a < 3; ++a) Su[a * ld + c] += prm.dt * (R[0 * 3 + a] * w0 + R[1 * 3 + a] * w1 + R[2 * 3 + a] * w2);
#pragma unroll
            for (int a = 0; a < 3; ++a) Su[(3 + a) * ld + c] += prm.dt * Su[(9 + a) * ld + c];
        }
        G::sync();
        // Su[:, 3 NFL i + 3 r + c] += dt B: rows 6..8 = Ihat^-1 skew(R p_l), rows 9..11 = I / m;  Ihat^-1 = R diag(1/I) R^T
        if (lane < 3 * NFL) {
            const int c = lane % 3;
            int l = 0;
            bool real_leg = false;
#pragma unroll
            for (int r = 0; r < NFL; ++r)
                if (r == lane / 3) { l = free_leg[r]; real_leg = real[r]; }
            double pl[3] = {0.0, 0.0, 0.0};
#pragma unroll
            for (int q = 0; q < 4; ++q)
                if (q == l) { pl[0] = pf[3 * q]; pl[1] = pf[3 * q + 1]; pl[2] = pf[3 * q + 2]; }
            double pw[3];
#pragma unroll
            for (int a = 0; a < 3; ++a) pw[a] = R[3 * a] * pl[0] + R[3 * a + 1] * pl[1] + R[3 * a + 2] * pl[2];
            double sk[3];  // column c of skew(pw) = [[0,-z,y],[z,0,-x],[-y,x,0]]
            sk[0] = c == 0 ? 0.0 : (c == 1 ? -pw[2] : pw[1]);
            sk[1] = c == 0 ? pw[2] : (c == 1 ? 0.0 : -pw[0]);
            sk[2] = c == 0 ? -pw[1] : (c == 1 ? pw[0] : 0.0);
            double t3[3];
#pragma unroll
            for (int a = 0; a < 3; ++a) t3[a] = prm.inv_inertia[a] * (R[a] * sk[0] + R[3 + a] * sk[1] + R[6 + a] * sk[2]);
            const int col = 3 * NFL * i + lane;
            if (real_leg) {
#pragma unroll
                for (int a = 0; a < 3; ++a) Su[(6 + a) * ld + col] += prm.dt * (R[3 * a] * t3[0] + R[3 * a + 1] * t3[1] + R[3 * a + 2] * t3[2]);
                Su[(9 + c) * ld + col] += prm.dt * prm.inv_mass;
            }
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
        G::sync();
        // gradient: all twelve rows of this thread's column; Gram matrix: the attitude (0..2) and body-rate (6..8) rows, columns in pairs
        double sa[6], gacc = 0.0;
#pragma unroll
        for (int k = 0; k < 12; ++k) {
            const double s_k = Su[k * ld + row];
            if (k < 3) sa[k] = prm.w_state[k] * s_k;
            if (k >= 6 && k < 9) sa[k - 3] = prm.w_state[k] * s_k;
            gacc = fma(s_k, prm.w_state[k] * (sc[k] - bref[i * 12 + k]), gacc);
        }
        grow = fma(2.0, gacc, grow);
        const int ncol = 3 * NFL * (i + 1);  // the later columns of Su are still zero
#pragma unroll
        for (int b = 0; b + 1 < n; b += 2) {
            if (b < ncol) {  // uniform; ncol is even or the odd last column is handled below
                double a0 = 0.0, a1 = 0.0;
#pragma unroll
                for (int k = 0; k < 6; ++k) {
                    const double2 v = *reinterpret_cast<const double2 *>(Su + (k < 3 ? k : k + 3) * ld + b);
                    a0 = fma(sa[k], v.x, a0);
                    a1 = fma(sa[k], v.y, a1);
                }
                hrow[b] = fma(2.0, a0, hrow[b]);
                hrow[b + 1] = fma(2.0, a1, hrow[b + 1]);
            }
        }
        if (n & 1) {
            double a0 = 0.0;
#pragma unroll
            for (int k = 0; k < 6; ++k) a0 = fma(sa[k], Su[(k < 3 ? k : k + 3) * ld + n - 1], a0);
            hrow[n - 1] = fma(2.0, a0, hrow[n - 1]);
        }
        G::sync();
    }
    // closed-form part: position and velocity rows (see the header)
    {
        const int jr = row / (3 * NFL), rr = (row / 3) % NFL, cr = row % 3;
        bool real_row = false;
#pragma unroll
        for (int r = 0; r < NFL; ++r)
            if (r == rr) real_row = real[r];
        const double d2m = prm.dt * prm.dt * prm.inv_mass, d1m = prm.dt * prm.inv_mass;
        double wp = 0.0, wv = 0.0;  // 2 w_pos (dt^2 / m)^2 and 2 w_vel (dt / m)^2 of this row's component
#pragma unroll
        for (int c = 0; c < 3; ++c)
            if (c == cr) { wp = 2.0 * prm.w_state[3 + c] * d2m * d2m; wv = 2.0 * prm.w_state[9 + c] * d1m * d1m; }
#pragma unroll
        for (int b = 0; b < n; ++b) {
            const int jb = b / (3 * NFL), rb = (b / 3) % NFL, cb = b % 3;  // compile-time after unrolling
            int s1 = 0, cnt = 0;  // sum over the common stages i >= max(jr, jb) of (i - jr)(i - jb), and their number
#pragma unroll
            for (int i = 0; i < MPC_NH; ++i)
                if (i >= jb && i >= jr) { s1 += (i - jr) * (i - jb); ++cnt; }
            if (cb == cr && real_row && real[rb]) hrow[b] += wp * (double)s1 + wv * (double)cnt;
        }
    }
}

#ifndef OKF_MPCG_WARPS
#define OKF_MPCG_WARPS 5
#endif
constexpr int MPCG_WARPS = OKF_MPCG_WARPS;  // problems per block of the one-warp kernel: 3 blocks = 15 warps per SM fit the shared memory (14.7 KB per problem)
// (Measured alternatives, same box: one warp per block x 14 blocks - no block-level tail behind a long active-set sequence, but one warp
// less per SM - 2.57e7 against 2.75e7 trot QPs/s and 2.03e7 against 2.55e7 closed-loop steps/s; two warps x 7 blocks 2.70e7 / 2.23e7.)
// resident blocks per SM the kernel is compiled for: what 227 KB of shared memory hold (each block also costs 1 KB of system shared memory)
constexpr int MPCG_MIN_BLOCKS = MPCG_WARPS == 5 ? 3 : (MPCG_WARPS == 1 ? 14 : (MPCG_WARPS == 2 ? 7 : 3));
constexpr int MPCG_MAX_IT = 400;    // constraints added + dropped
// capacity of the working set for 1..4 legs out of swing (linear independence bounds it by the order n = 15 legs; the test
// batches peak at 21 for two legs and 43 for four).  A problem that needs more is handed to the interior point.
__host__ __device__ constexpr int mpcg_slots(int nfl) { return nfl <= 2 ? 24 : (nfl == 3 ? 40 : 48); }
__host__ __device__ constexpr int mpcg_group(int nfl) { return nfl <= 2 ? 32 : 64; }  // threads per problem

// per-problem shared memory (doubles): H^-1 [n][n|1] (Su [12][n] while H is built) | S^-1 [slots][slots+1] | x g | strip 2 x 64, after the
// inversion y d r (three vectors of one entry per thread) | normals [3][threads] | block and id of a slot, list of the slots in use (3 ints per thread) | scratch 8
__host__ __device__ constexpr int mpcg_problem_doubles(int nfl) {
    return mpcg_even((15 * nfl) * ((15 * nfl) | 1)) + mpcg_slots(nfl) * (mpcg_slots(nfl) + 1) + 2 * mpcg_group(nfl) +
           (3 * mpcg_group(nfl) > 128 ? 3 * mpcg_group(nfl) : 128) + 3 * mpcg_group(nfl) + mpcg_group(nfl) + mpcg_group(nfl) / 2 + 8;
}
__host__ __device__ constexpr size_t mpcg_smem_bytes() { return (size_t)MPCG_WARPS * mpcg_problem_doubles(2) * sizeof(double); }
__host__ __device__ constexpr size_t mpcg2_smem_bytes(int max_legs) { return (size_t)mpcg_problem_doubles(max_legs) * sizeof(double); }

// coefficient c of constraint row r of a stance block:  r0: fz <= fz_max;  r1: fx - mu fz <= 0;  r2: -fx - mu fz <= 0;
// r3: fy - mu fz <= 0;  r4: -fy - mu fz <= 0
__device__ __forceinline__ double row_coef(int r, int c, double mu) {
    if (c == 0) return r == 1 ? 1.0 : (r == 2 ? -1.0 : 0.0);
    if (c == 1) return r == 3 ? 1.0 : (r == 4 ? -1.0 : 0.0);
    return r == 0 ? 1.0 : -mu;
}

// In place: m = row `lane` of the symmetric positive definite H  ->  row `lane` of -H^-1 (symmetric sweeps on every pivot).
// strip: 2 x 64 doubles.  Returns false (warp-uniform) on a non-positive pivot.
template <int N, int NW>
__device__ __forceinline__ bool sweep_invert(double (&m)[N], double *strip, int lane) {
    bool ok = true;
#pragma unroll
    for (int k = 0; k < N; ++k) {
        double *cb = strip + (k & 1) * 64;
        if (lane < N) cb[lane] = m[k];  // column k = row k (symmetry is kept by the sweeps)
        MpcGroup<NW>::sync();
        const double d = cb[k];
        ok = ok && (d > 0.0);
        const double inv = rcp2_(d);
        const double l = lane == k ? 1.0 - inv : m[k] * inv;  // the pivot row is scaled by 1 / d, the others eliminated
        const double2 *cp = reinterpret_cast<const double2 *>(cb);
#pragma unroll
        for (int q = 0; q < N / 2; ++q) {
            const double2 v = cp[q];
            m[2 * q] = fma(-l, v.x, m[2 * q]);
            m[2 * q + 1] = fma(-l, v.y, m[2 * q + 1]);
        }
        if (N & 1) m[N - 1] = fma(-l, cb[N - 1], m[N - 1]);
        m[k] = lane == k ? -inv : l;
    }
    return ok;
}

template <int NFL, int NW>
__device__ __forceinline__ void mpc_solve_gi(const MpcParams &prm, long long prob, double *base, const int (&kind_leg)[4], const int (&free_leg)[4]) {
    using G = MpcGroup<NW>;
    constexpr int n = 15 * NFL, nb = 5 * NFL, ldg = n | 1, GT = G::threads, SLOTS = mpcg_slots(NFL), LDP = SLOTS + 1;
    static_assert(n <= GT && SLOTS <= GT && mpc_condense_scratch(NFL) <= n * ldg && GT == mpcg_group(NFL), "layout");
    const long long N = prm.N;
    const int lane = G::tid();  // index in the group: row / slot / constraint block owned by this thread
    double *Ginv = base, *Su = base, *P = Ginv + mpcg_even(n * ldg), *xs = P + SLOTS * LDP, *g = xs + GT, *strip = g + GT;
    double *y = strip, *dslot = y + GT, *rslot = dslot + GT, *ncoef = strip + (3 * GT > 128 ? 3 * GT : 128);  // y, d, r reuse the strip once H is inverted
    int *sblk = reinterpret_cast<int *>(ncoef + 3 * GT), *sid = sblk + GT, *slist = sid + GT;
    double *scr = reinterpret_cast<double *>(slist + GT);

    int my_leg = 0;  // leg of the block this lane owns (blocks: stage-major, NFL legs per stage)
#pragma unroll
    for (int r = 0; r < NFL; ++r)
        if (r == lane % NFL) my_leg = free_leg[r];
    int my_kind = 0;
#pragma unroll
    for (int l = 0; l < 4; ++l)
        if (l == my_leg) my_kind = kind_leg[l];
    const bool my_act = lane < nb && my_kind == 1;
    const double mu_f = prm.mu;
    const int row = lane < n ? lane : n - 1;
    const double bvec[5] = {prm.fz_max, 0.0, 0.0, 0.0, 0.0};

    // ---- H, g; H^-1; the unconstrained minimiser ----------------------------------------------------------------------------
    for (int e = lane; e < 128; e += GT) strip[e] = 0.0;
    double m[n], grow;
    mpc_condense<NFL, NW>(prm, prob, lane, kind_leg, free_leg, Su, m, grow);
#pragma unroll
    for (int j = 0; j < n; ++j)
        if (j == row) m[j] += 2.0 * prm.w_force;
    if (lane < n) g[lane] = grow;
    G::sync();  // Su is dead from here on: its storage becomes H^-1
    bool ok = sweep_invert<n, NW>(m, strip, lane);
    double xi = 0.0;  // entry `lane` of the iterate
    {
        double a0 = 0.0, a1 = 0.0;
#pragma unroll
        for (int j = 0; j + 1 < n; j += 2) {
            a0 = fma(m[j], g[j], a0);  // m = -H^-1
            a1 = fma(m[j + 1], g[j + 1], a1);
        }
        if (n & 1) a0 = fma(m[n - 1], g[n - 1], a0);
        xi = a0 + a1;
    }
    G::sync();  // every lane has read g: from here on g[] holds the unconstrained minimiser x0 (the warm start needs it)
    if (lane < n) {
#pragma unroll
        for (int j = 0; j < n; ++j) Ginv[lane * ldg + j] = -m[j];
        xs[lane] = xi;
        g[lane] = xi;
    }

    // ---- dual active set -------------------------------------------------------------------------------------------------------
    // slot role (lane j < SLOTS): multiplier uj, normal (nj0, nj1, nj2) and block bj of working constraint j, its id (5 block + row)
    // block role (lane b < nb): inA = rows of block b that are in the working set
    using Mask = typename std::conditional<NW == 1, uint32_t, uint64_t>::type;  // one bit per slot
    const auto lowest = [](Mask mk) { return NW == 1 ? __ffs((int)mk) - 1 : __ffsll((long long)mk) - 1; };
    Mask valid = 0;  // slots in use
    int q = 0;       // their number; slist[0 .. q) lists them in ascending order (loops over the working set are counted loops with
                     // a broadcast load per slot - a bit scan per slot puts its latency on the loop-carried path)
    uint32_t inA = 0u;
    double uj = 0.0, nj0 = 0.0, nj1 = 0.0, nj2 = 0.0;
    int bj = 0, myid = -1;
    int it = 0;
    uint32_t status = 0u;
    const int max_it = prm.max_changes > 0 ? prm.max_changes : MPCG_MAX_IT;
    const double feas_tol = 1e-9 * prm.fz_max;
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    const double *gr = Ginv + row * ldg;  // this lane's row of H^-1
    const auto is_slot = [&]() { return ((valid >> lane) & Mask(1)) != 0; };
    const auto relist = [&]() {  // after every change of `valid`; readers are separated from it by the next barrier
        q = NW == 1 ? __popc((unsigned)valid) : __popcll((unsigned long long)valid);
        if (is_slot()) slist[NW == 1 ? __popc((unsigned)(valid & ((Mask(1) << lane) - Mask(1)))) : __popcll((unsigned long long)(valid & ((Mask(1) << lane) - Mask(1))))] = lane;
    };
    // r_j = sum_k S^-1[j][k] v[k] over the working slots (v in shared memory)
    const auto times_sinv = [&](const double *v) {
        double acc = 0.0;
        if (is_slot()) {
            const double *pr = P + lane * LDP;
#pragma unroll 2
            for (int t = 0; t < q; ++t) {
                const int k = slist[t];
                acc = fma(pr[k], v[k], acc);
            }
        }
        return acc;
    };
    // entry `lane` of sum_k c[k] H^-1 n_k over the working slots.  One warp: three columns of H^-1 per constraint, a loop over the
    // (few) slots.  Two warps (orders 45 / 60, up to 48 slots): the slot threads scatter w = N c into an n-vector (shared-memory
    // atomics: up to three working constraints share a block), then every row thread takes one product with its row of H^-1 -
    // work that does not grow with the size of the working set.  (y[] is free for w: its entries are in registers by now.)
    const auto times_hinv_n = [&](const double *c) {
        double acc = 0.0;
        if constexpr (NW == 1) {
#pragma unroll 2
            for (int t = 0; t < q; ++t) {
                const int k = slist[t];
                const int bk = sblk[k];
                const double hk = fma(gr[3 * bk + 2], ncoef[2 * GT + k], fma(gr[3 * bk + 1], ncoef[GT + k], gr[3 * bk] * ncoef[k]));
                acc = fma(c[k], hk, acc);
            }
        } else {
            double *w = y;
            G::sync();
            if (lane < n) w[lane] = 0.0;
            G::sync();
            if (is_slot()) {
                const double ck = c[lane];
                atomicAdd(&w[3 * bj], ck * nj0);
                atomicAdd(&w[3 * bj + 1], ck * nj1);
                atomicAdd(&w[3 * bj + 2], ck * nj2);
            }
            G::sync();
            double a1 = 0.0;
#pragma unroll 4
            for (int j = 0; j + 1 < n; j += 2) {
                acc = fma(gr[j], w[j], acc);
                a1 = fma(gr[j + 1], w[j + 1], a1);
            }
            if (n & 1) acc = fma(gr[n - 1], w[n - 1], acc);
            acc += a1;
        }
        return acc;
    };
    // constraint p = 5 bp + rp with normal np enters slot s:  S^-1 <- [[S^-1 + r r^T / delta, -r / delta], [-r^T / delta, 1 / delta]]
    // (r in rslot and, per lane, rj;  delta = n^T H^-1 n - d^T r)
    const auto enter = [&](int s, double rj, double delta, int p, int bp, int rp, double np0, double np1, double np2, double u_new) {
        const double idel = rcp2_(delta);
        if (is_slot()) {
            double *pr = P + lane * LDP;
            const double f = rj * idel;
#pragma unroll 2
            for (int t = 0; t < q; ++t) {
                const int k = slist[t];
                pr[k] = fma(f, rslot[k], pr[k]);
            }
            pr[s] = -f;
        }
        if (lane == s) {
            double *pr = P + s * LDP;
            for (int t = 0; t < q; ++t) {
                const int k = slist[t];
                pr[k] = -rslot[k] * idel;
            }
            pr[s] = idel;
            uj = u_new; nj0 = np0; nj1 = np1; nj2 = np2; bj = bp; myid = p;
            sblk[s] = bp;
            ncoef[s] = np0; ncoef[GT + s] = np1; ncoef[2 * GT + s] = np2;
            sid[s] = p;
        }
        valid |= Mask(1) << s;
        if (lane == bp) inA |= 1u << rp;
        G::sync();  // every thread is done with the old list
        relist();
    };
    // working constraint k leaves:  S^-1 <- S^-1 - S^-1[:, k] S^-1[k, :] / S^-1[k][k] on the remaining slots
    const auto leave = [&](int k) {
        const double ipkk = rcp2_(P[k * LDP + k]);
        const Mask rest = valid & ~(Mask(1) << k);
        if ((rest >> lane) & Mask(1)) {
            double *pr = P + lane * LDP;
            const double f = pr[k] * ipkk;
            const double *pk = P + k * LDP;
#pragma unroll 2
            for (int t = 0; t < q; ++t) {
                const int kk = slist[t];
                if (kk != k) pr[kk] = fma(-f, pk[kk], pr[kk]);
            }
        }
        const int idk = sid[k];
        if (lane == idk / 5) inA &= ~(1u << (idk % 5));
        if (lane == k) { uj = 0.0; myid = -1; }
        valid = rest;
        G::sync();  // every thread is done with the old list
        relist();
    };

    uint32_t pattern = 0;
#pragma unroll
    for (int l = 0; l < 4; ++l) pattern |= kind_leg[l] != 0 ? (1u << (24 + l)) : 0u;
    // ---- warm start: the working set of the previous solve of this problem (closed loops) -----------------------------------
    // Its constraints enter by bordering alone (no step, no ratio test), the minimiser on that set and its multipliers follow from
    // one product with S^-1, and constraints whose multiplier comes out negative leave one at a time: what remains is a point the
    // dual method may start from (the minimiser on its working set, all multipliers >= 0), usually the answer or one step from it.
    if (ok && prm.warm_set) {
        const uint32_t word = lane < nb ? prm.warm_set[(long long)(lane / NFL) * N + prob] : 0u;
        if (lane == 0) sid[0] = (int)word;  // (no slot is in use yet: sid is free)
        G::sync();
        const uint32_t word0 = (uint32_t)sid[0];
        G::sync();
        if ((word0 >> 31) && (word0 & 0x0f000000u) == pattern) {
            const uint32_t cand = my_act ? ((word >> (5 * my_leg)) & 31u) : 0u;  // rows of this lane's block in the stored working set
            const double gs = fmax(G::max(lane < n ? fabs(grow) : 0.0, scr), 1e-300);
            // The stored constraints enter TOGETHER: slots in ascending (block, row) order, S = N^T H^-1 N formed row by row (a 3 x 3
            // block of H^-1 per entry), then inverted in place by Gauss-Jordan steps on the pivots in that order.  The pivot of step k
            // is the Schur complement of constraint k on the pivots taken so far - the `delta` that entering them one at a time by
            // bordering would meet - so a normal that depends on the earlier ones is skipped by the same test, and the result is the
            // same working set and the same S^-1 for about a sixth of the instructions (one pass over q columns instead of q
            // bordering steps with two products over the working set each).
            sblk[lane] = __popc(cand);  // (no slot is in use yet: sblk, sid, ncoef, dslot, rslot are free)
            G::sync();
            int first = 0, total = 0;
#pragma unroll
            for (int b = 0; b < nb; ++b) {
                const int c = sblk[b];
                total += c;
                first += b < lane ? c : 0;
            }
            G::sync();
            const int qw = total < SLOTS ? total : SLOTS;
            {
                uint32_t c = cand;
                int s = first;
                while (c) {
                    const int r = __ffs(c) - 1;
                    c &= c - 1u;
                    if (s < SLOTS) {
                        sid[s] = 5 * lane + r;
                        sblk[s] = lane;
                        ncoef[s] = -row_coef(r, 0, mu_f); ncoef[GT + s] = -row_coef(r, 1, mu_f); ncoef[2 * GT + s] = -row_coef(r, 2, mu_f);
                    }
                    ++s;
                }
            }
            G::sync();
            const bool mine = lane < qw;
            if (mine) {
                myid = sid[lane]; bj = sblk[lane];
                nj0 = ncoef[lane]; nj1 = ncoef[GT + lane]; nj2 = ncoef[2 * GT + lane];
                const double *h0 = Ginv + (3 * bj) * ldg, *h1 = h0 + ldg, *h2 = h1 + ldg;
                double *pr = P + lane * LDP;
#pragma unroll 2
                for (int k = 0; k < qw; ++k) {
                    const int c = 3 * sblk[k];
                    const double c0 = ncoef[k], c1 = ncoef[GT + k], c2 = ncoef[2 * GT + k];
                    const double v0 = fma(h0[c + 2], c2, fma(h0[c + 1], c1, h0[c] * c0));
                    const double v1 = fma(h1[c + 2], c2, fma(h1[c + 1], c1, h1[c] * c0));
                    const double v2 = fma(h2[c + 2], c2, fma(h2[c + 1], c1, h2[c] * c0));
                    const double e = fma(nj2, v2, fma(nj1, v1, nj0 * v0));
                    pr[k] = e;
                    if (k == lane) dslot[lane] = e;  // n^T H^-1 n of this constraint: the scale of its pivot test
                }
            }
            Mask taken = 0;
#pragma unroll 1
            for (int k = 0; k < qw; ++k) {
                G::sync();  // S / the previous step's rows are visible
                const double d = P[k * LDP + k];
                if (!(d > 1e-10 * dslot[k])) continue;  // dependent on the constraints taken so far (group-uniform)
                const double inv = rcp2_(d);
                if (mine) rslot[lane] = lane == k ? inv : P[k * LDP + lane] * inv;  // the scaled pivot row
                const double f = (mine && lane != k) ? P[lane * LDP + k] : 0.0;
                G::sync();
                if (mine) {
                    double *pr = P + lane * LDP;
                    if (lane == k) {
#pragma unroll 2
                        for (int c = 0; c < qw; ++c) pr[c] = rslot[c];
                    } else {
#pragma unroll 2
                        for (int c = 0; c < qw; ++c) pr[c] = c == k ? -f * inv : fma(-f, rslot[c], pr[c]);
                    }
                }
                taken |= Mask(1) << k;
            }
            valid = taken;
            if (mine && !is_slot()) { myid = -1; bj = 0; nj0 = nj1 = nj2 = 0.0; }
            {
                uint32_t c = cand;
                int s = first;
                while (c) {
                    const int r = __ffs(c) - 1;
                    c &= c - 1u;
                    if (s < SLOTS && ((taken >> s) & Mask(1))) inA |= 1u << r;
                    ++s;
                }
            }
            G::sync();
            relist();
            if (valid) {
                status |= 8u;
#pragma unroll 1
                while (valid) {
                    G::sync();
                    // u = S^-1 (b' - N^T x0), x = x0 + H^-1 N u   (x0 = the unconstrained minimiser, kept in g[])
                    const int rj_row = myid - 5 * bj;
                    double rhs = 0.0;
#pragma unroll
                    for (int r = 0; r < 5; ++r)
                        if (r == rj_row) rhs = -bvec[r];
                    dslot[lane] = is_slot() ? rhs - fma(nj2, g[3 * bj + 2], fma(nj1, g[3 * bj + 1], nj0 * g[3 * bj])) : 0.0;
                    G::sync();
                    uj = times_sinv(dslot);
                    rslot[lane] = uj;
                    G::sync();
                    xi = (lane < n ? g[lane] : 0.0) + times_hinv_n(rslot);
                    double worst = is_slot() ? uj : inf;
                    int kw = is_slot() ? lane : -1;
                    G::argmin(worst, kw, scr);
                    if (!(worst < -1e-12 * gs)) break;
                    leave(kw);
                    ++it;
                }
                G::sync();
                if (lane < n) xs[lane] = valid ? xi : g[lane];
                if (!valid) xi = lane < n ? g[lane] : 0.0;
            }
        }
    }

    bool done = false;
#pragma unroll 1
    while (ok && !done) {
        G::sync();  // xs is current
        // most violated constraint outside the working set
        double best = inf;
        int p = -1;
        if (my_act) {
            const double x0 = xs[3 * lane], x1 = xs[3 * lane + 1], x2 = xs[3 * lane + 2];
#pragma unroll
            for (int r = 0; r < 5; ++r) {
                const double sl = bvec[r] - (row_coef(r, 0, mu_f) * x0 + row_coef(r, 1, mu_f) * x1 + row_coef(r, 2, mu_f) * x2);
                if (!((inA >> r) & 1u) && sl < best) { best = sl; p = 5 * lane + r; }
            }
        }
        G::argmin(best, p, scr);
        if (p < 0 || best >= -feas_tol) { done = true; break; }
        const int bp = p / 5, rp = p - 5 * bp;
        const double np0 = -row_coef(rp, 0, mu_f), np1 = -row_coef(rp, 1, mu_f), np2 = -row_coef(rp, 2, mu_f);  // normal of n^T x >= b'
        double sp = best, up = 0.0;
        // y = H^-1 n_p, d = N^T y: they do not change while constraints are dropped for this p
        const double yi = fma(gr[3 * bp + 2], np2, fma(gr[3 * bp + 1], np1, gr[3 * bp] * np0));
        if (lane < n) y[lane] = yi;
        G::sync();
        const double nGn = fma(np2, y[3 * bp + 2], fma(np1, y[3 * bp + 1], np0 * y[3 * bp]));
        const double dj = is_slot() ? fma(nj2, y[3 * bj + 2], fma(nj1, y[3 * bj + 1], nj0 * y[3 * bj])) : 0.0;
        dslot[lane] = dj;
        bool added = false;
#pragma unroll 1
        while (!added) {
            G::sync();  // dslot (first pass) / the downdated S^-1 (later passes) is visible
            // r = S^-1 d, z = y - H^-1 N r
            const double rj = is_slot() ? times_sinv(dslot) : 0.0;
            rslot[lane] = rj;
            double zn = 0.0;
            if constexpr (NW == 2) zn = nGn - G::sum(dj * rj, scr);
            G::sync();
            const double zi = yi - times_hinv_n(rslot);
            if constexpr (NW == 1) {  // n_p^T z = n^T H^-1 n - d^T r: three entries of z instead of a warp-wide sum
                zn = fma(np2, __shfl_sync(0xffffffffu, zi, 3 * bp + 2), fma(np1, __shfl_sync(0xffffffffu, zi, 3 * bp + 1), np0 * __shfl_sync(0xffffffffu, zi, 3 * bp)));
            }
            const bool dep = !(zn > 1e-12 * nGn);  // n_p is (numerically) a combination of the working normals: dual step only
            // step lengths: t1 keeps the multipliers non-negative, t2 makes constraint p hold
            double t1 = (is_slot() && rj > 1e-300) ? uj * rcp2_(rj) : inf;
            int k1 = (is_slot() && rj > 1e-300) ? lane : -1;
            G::argmin(t1, k1, scr);
            if (k1 < 0) t1 = inf;
            const double t2 = dep ? inf : -sp * rcp2_(zn);
            const double t = fmin(t1, t2);
            if (!(t < inf)) { ok = false; break; }  // neither step exists: cannot happen for a feasible problem in exact arithmetic
            if (!dep) {
                xi = fma(t, zi, xi);
                sp = fma(t, zn, sp);
            }
            uj = is_slot() ? fma(-t, rj, uj) : 0.0;
            up += t;
            ++it;
            if (it > max_it) { ok = false; break; }
            if (!dep && t2 <= t1) {  // full step: p enters
                const Mask freeslots = ~valid & ((Mask(1) << SLOTS) - Mask(1));
                if (!freeslots) { ok = false; break; }
                enter(lowest(freeslots), rj, zn, p, bp, rp, np0, np1, np2, up);
                if (lane < n) xs[lane] = xi;
                added = true;
            } else {
                leave(k1);  // partial (or purely dual) step: the multiplier of working constraint k1 has reached zero
            }
        }
    }

    // ---- results -----------------------------------------------------------------------------------------------------------------
    for (int e = lane; e < MPC_N; e += GT) prm.forces[(long long)e * N + prob] = ok ? 0.0 : __longlong_as_double(0x7ff8000000000000LL);
    G::sync();
    if (ok && lane < n) {  // compact -> (stage, leg, component)
        const int stage = lane / (3 * NFL), within = lane % (3 * NFL);
        int l = 0;
#pragma unroll
        for (int r = 0; r < NFL; ++r)
            if (r == within / 3) l = free_leg[r];
        prm.forces[(long long)(12 * stage + 3 * l + within % 3) * N + prob] = xi;
    }
    if (prm.warm_set) {
        // the working set of this solve, by absolute (stage, leg, row), and its multipliers
        G::sync();
        sblk[lane] = (int)(ok ? (inA << (5 * my_leg)) : 0u);  // (the slots' block numbers are not needed any more)
        G::sync();
        if (lane < nb && lane % NFL == 0) {
            uint32_t bits = 0u;
#pragma unroll
            for (int r = 0; r < NFL; ++r) bits |= (uint32_t)sblk[lane + r];  // the legs of one stage sit in adjacent threads
            prm.warm_set[(long long)(lane / NFL) * N + prob] = ok ? (bits | pattern | 0x80000000u) : 0u;
        }
        if (ok && is_slot()) {
            int l = 0;
#pragma unroll
            for (int r = 0; r < NFL; ++r)
                if (r == bj % NFL) l = free_leg[r];
            prm.warm_mult[(long long)(((bj / NFL) * 4 + l) * 5 + (myid - 5 * bj)) * N + prob] = uj;
        }
    }
    if (lane == 0) prm.status[prob] = ok ? (status | ((uint32_t)it << 8)) : MPC_ST_GIVEN_UP;
}

// One warp per problem (at most two legs out of swing); prm.status is required (the second launch reads the flags).
__global__ void __launch_bounds__(32 * MPCG_WARPS, MPCG_MIN_BLOCKS) kf_mpc_gi_kernel(const __grid_constant__ MpcParams prm) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long prob = (long long)blockIdx.x * MPCG_WARPS + warp;
    if (prob >= prm.N) return;  // whole warp
    double *base = reinterpret_cast<double *>(smem_raw) + (size_t)warp * mpcg_problem_doubles(2);
    const long long N = prm.N;
    int kind_leg[4];  // 0 pinned (swing), 1 pyramid (stance), 2 free
#pragma unroll
    for (int l = 0; l < 4; ++l) {
        const double c = prm.contact[l * N + prob];
        kind_leg[l] = c == 0.0 ? 0 : (c == 1.0 ? 1 : 2);
    }
    int free_leg[4] = {0, 0, 0, 0}, nfl = 0;
#pragma unroll
    for (int l = 0; l < 4; ++l)
        if (kind_leg[l] != 0) {
#pragma unroll
            for (int r = 0; r < 4; ++r)
                if (r == nfl) free_leg[r] = l;
            ++nfl;
        }
    if (nfl > prm.max_legs || nfl > MPCG_MAX_LEGS) {  // the caller's bound on the legs out of swing is wrong for this problem: no answer
        for (int e = lane; e < MPC_N; e += 32) prm.forces[(long long)e * N + prob] = __longlong_as_double(0x7ff8000000000000LL);
        if (lane == 0) prm.status[prob] = 4u;
        if (prm.warm_set && lane < MPC_NH) prm.warm_set[(long long)lane * N + prob] = 0u;
        return;
    }
    if (nfl == 0) {
        for (int e = lane; e < MPC_N; e += 32) prm.forces[(long long)e * N + prob] = 0.0;
        if (lane == 0) prm.status[prob] = 0u;
        if (prm.warm_set && lane < MPC_NH) prm.warm_set[(long long)lane * N + prob] = 0u;
        return;
    }
    if (nfl == 1) {  // the lone leg is paired with a phantom that decouples exactly (mpc_condense)
#pragma unroll
        for (int l = 3; l >= 0; --l)
            if (kind_leg[l] == 0) free_leg[1] = l;
    }
    mpc_solve_gi<2, 1>(prm, prob, base, kind_leg, free_leg);
}

// Batches with three or four legs out of swing somewhere: one 64-thread block per problem.  Orders 45 and 60 take both warps
// (a thread per row of H^-1, broadcasts and reductions across the two warps through shared memory); a problem of the batch
// with at most two legs out of swing is solved by warp 0 alone, exactly as in the one-warp kernel.
__global__ void __launch_bounds__(64) kf_mpc_gi2_kernel(const __grid_constant__ MpcParams prm) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x;
    const long long prob = blockIdx.x, N = prm.N;
    double *base = reinterpret_cast<double *>(smem_raw);
    int kind_leg[4];
#pragma unroll
    for (int l = 0; l < 4; ++l) {
        const double c = prm.contact[l * N + prob];
        kind_leg[l] = c == 0.0 ? 0 : (c == 1.0 ? 1 : 2);
    }
    int free_leg[4] = {0, 0, 0, 0}, nfl = 0;
#pragma unroll
    for (int l = 0; l < 4; ++l)
        if (kind_leg[l] != 0) {
#pragma unroll
            for (int r = 0; r < 4; ++r)
                if (r == nfl) free_leg[r] = l;
            ++nfl;
        }
    if (nfl > prm.max_legs) {
        for (int e = tid; e < MPC_N; e += 64) prm.forces[(long long)e * N + prob] = __longlong_as_double(0x7ff8000000000000LL);
        if (tid == 0) prm.status[prob] = 4u;
        if (prm.warm_set && tid < MPC_NH) prm.warm_set[(long long)tid * N + prob] = 0u;
        return;
    }
    if (nfl == 0) {
        for (int e = tid; e < MPC_N; e += 64) prm.forces[(long long)e * N + prob] = 0.0;
        if (tid == 0) prm.status[prob] = 0u;
        if (prm.warm_set && tid < MPC_NH) prm.warm_set[(long long)tid * N + prob] = 0u;
        return;
    }
    if (nfl <= 2) {
        if (tid >= 32) return;
        if (nfl == 1) {
#pragma unroll
            for (int l = 3; l >= 0; --l)
                if (kind_leg[l] == 0) free_leg[1] = l;
        }
        mpc_solve_gi<2, 1>(prm, prob, base, kind_leg, free_leg);
    } else if (nfl == 3) {
        mpc_solve_gi<3, 2>(prm, prob, base, kind_leg, free_leg);
    } else {
        mpc_solve_gi<4, 2>(prm, prob, base, kind_leg, free_leg);
    }
}

}  // namespace okf
