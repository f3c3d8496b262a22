// Developer probe: accuracy of the FP64 pivot reciprocal okf::rcp_(double) (kf_arith.cuh) and of the hardware seed it refines.
//   (1) seed: max |1 - a r0| of r0 = rcp.approx.ftz.f64(a) (SASS MUFU.RCP64H), over all 2^20 high-word mantissas x a set of low
//       words (fixed patterns + hashed ones) x every binary exponent of [1e-8, 1e4], the range the filter's pivots P_kk + r_k take;
//   (2) rcp_: max distance in ulps from the IEEE quotient 1.0 / a over the same inputs, and how often it differs from it;
//   (3) the same for the three-Newton-step form it replaced (reference), and what rcp_ returns for zero, subnormal and
//       infinite pivots (NaN, so that a bad pivot the caller flags also poisons what follows).
#include <cstdio>
#include <cstring>
#include <cuda_runtime.h>

#include "../../optistate_b200/csrc/kf_arith.cuh"

constexpr int kExpLo = -27, kExpHi = 13;  // 2^-27 = 7.5e-9 .. 2^14 = 1.6e4
__constant__ unsigned kFixedLow[] = {0x00000000u, 0x00000001u, 0x55555555u, 0x80000000u, 0xaaaaaaaau, 0xfffffffeu, 0xffffffffu};
constexpr int kFixed = 7, kHashedLow = 4;

struct Stats {
    unsigned long long seed_err_bits;  // max |1 - a r0| as the bit pattern of a non-negative double (ordered like the value)
    unsigned long long ulp_new, ulp_old;  // max |bits(rcp) - bits(1.0 / a)|
    unsigned long long diff_new, diff_old;  // inputs on which rcp differs from 1.0 / a
    unsigned long long n;
    unsigned long long worst_seed_input, worst_new_input;
};

__device__ __forceinline__ double rcp_newton3(double a) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(a));
    double e = fma(-a, r, 1.0);
    r = fma(r, e, r);
    e = fma(-a, r, 1.0);
    r = fma(r, e, r);
    e = fma(-a, r, 1.0);
    return fma(r, e, r);
}

__device__ __forceinline__ unsigned hash32(unsigned x) {
    x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
    return x;
}

__device__ __forceinline__ unsigned long long ulp_dist(double a, double b) {
    const long long x = __double_as_longlong(a), y = __double_as_longlong(b);
    return (unsigned long long)(x > y ? x - y : y - x);  // both positive: the bit patterns are ordered like the values
}

__global__ void sweep(Stats *st) {
    const unsigned mhi = blockIdx.x * blockDim.x + threadIdx.x;  // 20-bit high-word mantissa
    if (mhi >= (1u << 20)) return;
    unsigned long long seed_err = 0, u_new = 0, u_old = 0, d_new = 0, d_old = 0, n = 0, w_seed = 0, w_new = 0, w_new_u = 0;
    constexpr int kLow = kFixed + kHashedLow;
    for (int ex = kExpLo; ex <= kExpHi; ++ex) {
        for (int l = 0; l < kLow; ++l) {
            const unsigned lo = l < kFixed ? kFixedLow[l] : hash32(mhi * 131u + (unsigned)(ex - kExpLo) * 7919u + (unsigned)l);
            const unsigned hi = ((unsigned)(ex + 1023) << 20) | mhi;
            const double a = __hiloint2double((int)hi, (int)lo);
            double r0;
            asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r0) : "d"(a));
            const unsigned long long se = (unsigned long long)__double_as_longlong(fabs(fma(-a, r0, 1.0)));
            if (se > seed_err) { seed_err = se; w_seed = (unsigned long long)__double_as_longlong(a); }
            const double q = 1.0 / a, rn = okf::rcp_(a), ro = rcp_newton3(a);
            const unsigned long long dn = ulp_dist(rn, q), dd = ulp_dist(ro, q);
            if (dn > w_new_u) { w_new_u = dn; w_new = (unsigned long long)__double_as_longlong(a); }
            u_new = max(u_new, dn); u_old = max(u_old, dd);
            d_new += dn != 0; d_old += dd != 0;
            ++n;
        }
    }
    if (atomicMax(&st->seed_err_bits, seed_err) < seed_err) st->worst_seed_input = w_seed;  // best effort: a diagnostic only
    if (atomicMax(&st->ulp_new, u_new) < u_new && u_new > 0) st->worst_new_input = w_new;
    atomicMax(&st->ulp_old, u_old);
    atomicAdd(&st->diff_new, d_new);
    atomicAdd(&st->diff_old, d_old);
    atomicAdd(&st->n, n);
}

__global__ void specials(const double *in, double *out, int n) {
    const int i = threadIdx.x;
    if (i < n) out[i] = okf::rcp_(in[i]);
}

int main() {
    Stats *st;
    cudaMallocManaged(&st, sizeof(Stats));
    memset(st, 0, sizeof(Stats));
    sweep<<<(1 << 20) / 256, 256>>>(st);
    if (cudaDeviceSynchronize() != cudaSuccess) { printf("sweep failed: %s\n", cudaGetErrorString(cudaGetLastError())); return 1; }
    double seed_err, wa, wn;
    memcpy(&seed_err, &st->seed_err_bits, 8);
    memcpy(&wa, &st->worst_seed_input, 8);
    memcpy(&wn, &st->worst_new_input, 8);
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, 0);
    printf("device: %s\n", prop.name);
    printf("inputs: %llu (2^20 high-word mantissas x %d low words x binary exponents %d..%d)\n", st->n,
           kFixed + kHashedLow, kExpLo, kExpHi);
    printf("seed rcp.approx.ftz.f64: max |1 - a r0| = %.3e = 2^%.2f  (at a = %.17g)\n", seed_err, log2(seed_err), wa);
    printf("rcp_ (kf_arith.cuh):      max %llu ulp from 1.0 / a, differs on %llu inputs (%.2e)%s%.17g\n", st->ulp_new, st->diff_new,
           (double)st->diff_new / (double)st->n, st->ulp_new ? ", worst at a = " : "", st->ulp_new ? wn : 0.0);
    printf("three Newton steps:       max %llu ulp from 1.0 / a, differs on %llu inputs (%.2e)\n", st->ulp_old, st->diff_old,
           (double)st->diff_old / (double)st->n);
    const double sp[] = {0.0, -0.0, 4.9e-324, 2.2e-308, __builtin_inf(), 1.0, 2.0};
    const int ns = sizeof(sp) / sizeof(sp[0]);
    double *din, *dout;
    cudaMallocManaged(&din, sizeof(sp));
    cudaMallocManaged(&dout, sizeof(sp));
    memcpy(din, sp, sizeof(sp));
    specials<<<1, 32>>>(din, dout, ns);
    cudaDeviceSynchronize();
    printf("rcp_ of special pivots:");
    for (int i = 0; i < ns; ++i) printf("  %g -> %g", sp[i], dout[i]);
    printf("\n");
    return 0;
}
