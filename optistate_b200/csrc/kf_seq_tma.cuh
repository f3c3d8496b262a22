// Throughput kernel, streamed variant: the arithmetic of kf_seq_core.cuh (one thread per trajectory, packed symmetric
// P and x in registers, sequential scalar updates) with the per-step inputs delivered by the TMA engine.
//
//   * 32 consecutive trajectories (one warp) read 32 consecutive base streams, so the inputs of one step are
//     [C] x 32 tiles of the [T*C][S] arrays, delivered by 2-D tensor-map copies (cp.async.bulk.tensor, SASS UTMALDG)
//     per array - leg moments, z, label streams - that complete on an mbarrier (complete_tx).  No per-thread address
//     arithmetic, no LDG in the recursion, no registers tied up by loads in flight, no block-wide barrier.
//   * The WARPS OF A BLOCK SHARE ONE TILE: they filter different members (trajectory i, i + S, i + 2 S, ...) of the same 32
//     streams, so one copy feeds all of them and a block of four needs 12 KB of FP64 input tiles instead of 47 KB.
//     That is what decides occupancy: with a tile per warp the decoupled-group kernels (168 registers, three blocks per
//     SM by registers) were held to two blocks by 108 KB of shared memory; with the shared tile three blocks fit
//     (ncu: launch__occupancy_limit_shared_mem).  The warp that is LAST to finish reading a group (a ticket drawn from a
//     shared-memory counter) issues the refill, so nobody waits on a designated producer.
//   * Three channel groups, each single-buffered and refilled for step t+1 the moment the block has consumed
//     step t's copy, so the copy has most of a filter step (several microseconds) to land:
//         G0 = M[12]            read at the top of the step (mean model)        -> refilled after the covariance predict (kBlock), else right away
//              (+ the feet p[12] in the kOut == 2 instantiations, which write p_world_steps, and the 3 reference body
//              angles of the predict_mpc covariance model in the kMpc instantiations)
//         G1 = z[10]            read one by one as the measurements are folded  -> refilled before the last fold
//         G2 = truth / nominal  label streams of the summary, read inside the last fold -> refilled after it
//   * Inputs are consumed straight from shared memory (conflict-free: consecutive threads, consecutive words);
//     nothing but x, P and the next step's rotation matrix stays live across the step.
//   * Latency of the two long dependent chains is hidden behind the independent rank-1 FMAs: the reciprocal of
//     the NEXT pivot is started as soon as that pivot's entry has been updated, and the sin/cos of the NEXT
//     step's attitude - and the summary's running error sums - are started as soon as the last state update is done.
//   * Template variants instead of branches in the time loop (kSummary, kOut, kMpc): a taken branch over an unused block
//     costs an instruction-fetch bubble at its target, ~10 % of a lone warp's time before they were compiled out.
//   * Instantiated for double, float and F2 (kf_arith.cuh): F2 packs TWO FP32 trajectories into one thread and runs
//     the recursion on FFMA2 / FADD2 / FMUL2, halving the issue slots per trajectory-step; its tiles are [C] x 64.
//   * z and the leg moments M of the mean model (leg_moments, kf_seq_core.cuh) come from the measurement pre-pass: they are
//     state-independent and, with shared base streams, identical for every Monte-Carlo member of a stream.
//   * Its own are the tiles, their refill elections and the schedule around them; the rest is kf_seq_core.cuh's.
#pragma once

#include <cuda.h>  // CUtensorMap (types only; the encoder is fetched through cudaGetDriverEntryPoint)

#include "kf_seq_core.cuh"

namespace okf {

// warps of a block = members that share one copy of a stream tile.  Four: the decoupled-group kernels then run 3 blocks = 12 warps
// per SM at 166 registers.  Five warps x 3 blocks (15 warps per SM) fit the shared memory too, but cap the kernel at 128 registers:
// measured 1.58e10 against 1.90e10 steps/s (FP64) and 2.9e10 against 3.6e10 (FP32) - the spills cost more than the warps bring.
#ifndef OKF_BLK_WARPS
#define OKF_BLK_WARPS 4
#endif
template <bool kBlock>
__host__ __device__ constexpr int tma_warps() { return kBlock ? OKF_BLK_WARPS : 4; }
template <bool kBlock>
__host__ __device__ constexpr int tma_threads() { return 32 * tma_warps<kBlock>(); }
constexpr int TMA_CH_G1 = 10;
constexpr int TMA_CH_REF = 3;  // reference body angles of the predict_mpc covariance model (kMpc kernels), part of group G0
// rows of group G0: the leg moments M, the feet (kOut == 2: p_world_steps) and the reference body angles (kMpc)
template <int kOut, bool kMpc>
__host__ __device__ constexpr int tma_g0_rows() { return NM + (kOut == 2 ? 12 : 0) + (kMpc ? TMA_CH_REF : 0); }
constexpr int TMA_NOISE_ROWS = 22;  // q[12] r[10]
constexpr int TMA_NOISE_ROWS_OUT = 32;  // ... and 1 / r[10] in the instantiations with per-step outputs (K_gain every step)
template <int kW>
__host__ __device__ constexpr int tma_stages() { return kW == 1 ? 2 : 1; }
template <int kOut>
__host__ __device__ constexpr int tma_noise_rows() { return kOut != 0 ? TMA_NOISE_ROWS_OUT : TMA_NOISE_ROWS; }

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!done);
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// tensor maps of the per-step input arrays, each viewed as a [T*C][S] matrix with a [C][32] box
struct alignas(64) TmaMaps {
    CUtensorMap mom, p, z, lab0, lab1, body_ref;
};

__device__ __forceinline__ void tma_tile_g2s(void *dst, const CUtensorMap *map, int col, int row, uint64_t *bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                     smem_u32(dst)),
                 "l"(map), "r"(col), "r"(row), "r"(smem_u32(bar))
                 : "memory");
}

template <typename Real, int kThreads, int kNoiseRows = TMA_NOISE_ROWS, int kStages = 1>
struct TmaSmem {
    // dynamic shared memory: [mbarriers 128 B][election line 128 B][G0 [g0_rows][32] | G1 [10][32] | G2 [12*n_lab][32]] (kStages tile
    //                        sets per block)  [noise [22 | 32][128]][acc [25][128] (8-byte sums; double and F2 kernels only)]   (elements: Real)
    static __host__ __device__ constexpr size_t warp_rows(int n_lab, int g0_rows) { return g0_rows + TMA_CH_G1 + 12 * n_lab; }
    static __host__ __device__ constexpr size_t warp_bytes(int n_lab, int g0_rows) { return warp_rows(n_lab, g0_rows) * 32 * sizeof(Real); }
    static __host__ __device__ constexpr size_t off_elect() { return 128; }
    static __host__ __device__ constexpr size_t off_in() { return 256; }
    static __host__ __device__ constexpr size_t off_noise(int n_lab, int g0_rows) { return off_in() + kStages * warp_bytes(n_lab, g0_rows); }
    static __host__ __device__ constexpr size_t off_acc(int n_lab, int g0_rows) { return off_noise(n_lab, g0_rows) + (size_t)kNoiseRows * kThreads * sizeof(Real); }
    static __host__ __device__ constexpr size_t total(int n_lab, int g0_rows, bool acc_in_smem) {
        return off_acc(n_lab, g0_rows) + (acc_in_smem ? (size_t)ACC_ROWS * kThreads * 8 : 0);
    }
};

// One elected thread (`lane` == 0 of the warp that is entitled to refill): arm the group's mbarrier with the byte count, then
// issue the tile copies of step t.  G0 = M [12] | p [12] (kOut == 2) | body_ref [3] (kMpc), rows of the block's tile.
template <int kOut, bool kMpc, typename Real>
__device__ __forceinline__ void issue_g0(const TmaMaps &m, long long t, int s_warp, Real *g0w, uint64_t *bar, int lane) {
    if (lane == 0) {
        mbar_expect_tx(bar, (uint32_t)(tma_g0_rows<kOut, kMpc>() * 32 * sizeof(Real)));
        tma_tile_g2s(g0w, &m.mom, s_warp, (int)(t * NM), bar);
        if constexpr (kOut == 2) tma_tile_g2s(g0w + NM * 32, &m.p, s_warp, (int)(t * 12), bar);
        if constexpr (kMpc) tma_tile_g2s(g0w + (tma_g0_rows<kOut, kMpc>() - TMA_CH_REF) * 32, &m.body_ref, s_warp, (int)(t * 12), bar);  // rows 0..2 of the step's 12
    }
}
template <typename Real>
__device__ __forceinline__ void issue_g1(const TmaMaps &m, long long t, int s_warp, Real *g1w, uint64_t *bar, int lane) {
    if (lane == 0) {
        mbar_expect_tx(bar, (uint32_t)(TMA_CH_G1 * 32 * sizeof(Real)));
        tma_tile_g2s(g1w, &m.z, s_warp, (int)(t * 10), bar);
    }
}
template <typename Real>
__device__ __forceinline__ void issue_g2(const TmaMaps &m, long long t, int s_warp, int n_lab, Real *g2w, uint64_t *bar, int lane) {
    if (lane == 0) {
        mbar_expect_tx(bar, (uint32_t)(12 * n_lab * 32 * sizeof(Real)));
        tma_tile_g2s(g2w, &m.lab0, s_warp, (int)(t * 12), bar);
        if (n_lab > 1) tma_tile_g2s(g2w + 12 * 32, &m.lab1, s_warp, (int)(t * 12), bar);
    }
}

// kOut: which per-step outputs the instantiation can write.  0 = none; 1 = the estimates (x_steps, p_trace_steps,
// k_gain_steps, nis_steps - what the reference driver records every step); 2 = also the rarely wanted ones
// (x_model_steps, p_world_steps, z_steps, P_ckpt, and the smoother's P_steps).  Blocks of outputs that are not wanted are compiled out instead of being
// jumped over every step: the taken branches across them cost the lone warp of a scheduler ~10 % of its time in
// instruction-fetch bubbles (ncu: stall_no_inst / stall_branch_resolving at the branch targets of the 35 KB loop body).
// kBlock: the decoupled-group form of the covariance recursion (kf_seq_core.cuh): 30 live scalars of P instead of 78, which
// leaves room for more resident warps (see tma_min_blocks).
template <typename Real, bool kSummary, bool kBlock>
__host__ __device__ constexpr int tma_min_blocks() {
#ifdef OKF_BLK_MINB
    if (kBlock) return OKF_BLK_MINB;
#endif
    if (kBlock) return (sizeof(Real) == 8 || kSummary) ? 3 : 4;  // the FP32 summary keeps 25 FP64 sums in registers
    return (sizeof(Real) == 4 && !kSummary) ? 3 : 2;
}
template <typename Real, bool kSummary, bool kBlock>
__host__ __device__ constexpr bool tma_acc_in_smem() {
#ifdef OKF_BLK_ACC_SMEM
    if (kBlock) return kSummary && sizeof(Real) == 8 && OKF_BLK_ACC_SMEM;
#endif
    return kSummary && sizeof(Real) == 8;
}

#ifdef OKF_ELECT_STAMPS
// Diagnostic build (tools/probes/elect_stamps.py compiles ONE translation unit with it): lane 0 of every warp of the first
// kStampBlocks blocks of a throughput-geometry launch writes clock64() at the top of each of steps [kStampT0, kStampT0 + kStampSteps),
// before and after each of the three refill elections (election and copy issue) and at the end of the step, and each of those
// blocks its SM, to the arrays below; okf_elect_stamps_read copies them out.  The stores change the schedule of the loop a little,
// so its numbers are for the election, not for the kernel's rate.
constexpr int kStampBlocks = 1024, kStampWarps = 4, kStampT0 = 400, kStampSteps = 16, kStampEvents = 8;
enum StampEvent { kStTop, kStElect0, kStElect0End, kStElect1, kStElect1End, kStElect2, kStElect2End, kStEnd };
__device__ long long okf_elect_stamps[kStampBlocks * kStampWarps * kStampSteps * kStampEvents];
__device__ unsigned okf_elect_smid[kStampBlocks];
extern "C" int okf_elect_stamps_read(long long *stamps, unsigned *smid) {
    if (cudaMemcpyFromSymbol(stamps, okf_elect_stamps, sizeof(okf_elect_stamps)) != cudaSuccess) return 1;
    return cudaMemcpyFromSymbol(smid, okf_elect_smid, sizeof(okf_elect_smid)) != cudaSuccess ? 1 : 0;
}
#define OKF_STAMP(ev)                                                                                                                 \
    do {                                                                                                                              \
        if (stamp_on && t >= kStampT0 && t < kStampT0 + kStampSteps)                                                                  \
            okf_elect_stamps[((blockIdx.x * kStampWarps + warp) * kStampSteps + (t - kStampT0)) * kStampEvents + (ev)] = clock64(); \
    } while (0)
#else
#define OKF_STAMP(ev) \
    do {              \
    } while (0)
#endif

// kW: warps per block; 0 = the throughput geometry above (tma_warps).  kW = 1 is the LATENCY variant, chosen by the host when there are
// no more trajectories than streams (every block of the throughput geometry would hold one working warp - BASELINE configs[1],
// 1,024 trajectories x 10,000 steps, is the case): a block is its one warp, so nobody counts readers (no shared-memory atomic, whose
// warp-aggregated expansion put ~100 dependent cycles three times into every step of a lone warp), the running sums of the summary
// stay in registers, and the kernel may use the whole register file of its scheduler (launch bound of one block).
template <typename Real, bool kSummary, int kOut, bool kMpc, bool kBlock = false, int kW = 0>
__global__ void __launch_bounds__(kW ? 32 * kW : tma_threads<kBlock>(), kW == 1 ? 1 : tma_min_blocks<Real, kSummary, kBlock>()) kf_seq_tma_kernel(const __grid_constant__ Params<typename Lanes<Real>::scalar> prm,
                                                                 const __grid_constant__ TmaMaps maps) {
    using Scalar = typename Lanes<Real>::scalar;
    using AccT = typename Acc<Real>::type;
    constexpr int L = Lanes<Real>::n;                     // trajectories per thread
    static_assert(!(kBlock && kMpc), "the element-wise exponential of predict_mpc couples every state");
    constexpr bool kAccSmem = kW == 1 ? false : tma_acc_in_smem<Real, kSummary, kBlock>();  // double / F2 with the full P: the 25 running sums do not fit next to P in registers
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int TMA_WARPS = kW ? kW : tma_warps<kBlock>(), nt = 32 * TMA_WARPS;
    // tile sets in flight: the throughput geometry refills a group for step t + 1 as soon as step t's copy has been read (one set; a
    // second one does not fit next to three resident blocks); the latency variant has the shared memory for two and refills for
    // step t + 2, so a copy has two whole steps to land (a lone warp waited ~120 cycles per step on the single set)
    constexpr int kStages = tma_stages<kW>();
    using Smem = TmaSmem<Real, nt, tma_noise_rows<kOut>(), kStages>;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long N = prm.N, S = prm.S;
    // Block (tile k, group j) filters members W j .. W j + W - 1 of the 32 L streams of tile k (W = warps of the block): warp w owns
    // trajectories (W j + w) S + 32 L k + L lane (+ 0 .. L-1), which all read stream tile k (shifted by the stream offset).  Blocks of one
    // tile are launched next to each other, so the tile's whole time series (tens of MB) stays L2-resident however far the
    // resident blocks drift apart in time (measured in round 1: 375 GB -> ~1 GB of DRAM reads per launch on the 1 M x 1 k sweep).
    constexpr int TW = 32 * L;                                     // streams of a tile = trajectories of a warp
    const long long n_pass = (N + S - 1) / S;                      // members per stream (the last pass may be ragged)
    const long long groups = (n_pass + TMA_WARPS - 1) / TMA_WARPS;  // blocks per tile
    const long long tile_k = blockIdx.x / groups, grp_j = blockIdx.x % groups;
    const long long m_pass = grp_j * TMA_WARPS + warp;
    const bool warp_active = m_pass < n_pass;
    const int n_active = (int)(n_pass - grp_j * TMA_WARPS < TMA_WARPS ? n_pass - grp_j * TMA_WARPS : TMA_WARPS);  // warps of this block with work
    const long long i = m_pass * S + tile_k * TW + (long long)lane * L;  // first trajectory of this thread
    const bool active = warp_active && i < N;              // N % L == 0 is guaranteed by the host
    const long long ic = active ? i : N - L;               // clamped index for per-trajectory parameter loads
    const int s_warp = (int)((tile_k * TW + prm.stream_offset) % S);  // first stream of the block's tile
    const int n_lab = kSummary ? (prm.truth ? 1 : 0) + (prm.nominal ? 1 : 0) : 0;

    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw);  // full[G0], full[G1], full[G2]
    // election line: words 0-2 count the warps that have finished reading G0, G1, G2 (see last_reader); the rest is padding that
    // the other lanes of an election touch
    uint32_t *tickets = reinterpret_cast<uint32_t *>(smem_raw + Smem::off_elect());
    constexpr int kG0Rows = tma_g0_rows<kOut, kMpc>();
    Real *g0w = reinterpret_cast<Real *>(smem_raw + Smem::off_in());
    Real *g1w = g0w + kG0Rows * 32, *g2w = g1w + TMA_CH_G1 * 32;  // the block's [C][32] tiles (of Real)
    Real *noise = reinterpret_cast<Real *>(smem_raw + Smem::off_noise(n_lab, kG0Rows));
    AccT *acc_s = reinterpret_cast<AccT *>(smem_raw + Smem::off_acc(n_lab, kG0Rows)) + tid;

    if (grp_j * TMA_WARPS * S + tile_k * TW >= N) return;  // the whole block lies beyond the last trajectory (fewer trajectories than streams)
    const int tile_elems = (int)Smem::warp_rows(n_lab, kG0Rows) * 32;  // elements of one tile set
    if (tid == 0) {
#pragma unroll
        for (int b = 0; b < 3 * kStages; ++b) mbar_init(&bars[b], 1);  // full[G0], full[G1], full[G2] of every tile set
        if constexpr (!kBlock) tickets[0] = tickets[1] = tickets[2] = 0;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (kBlock && tid < 32) tickets[tid] = 0;
#ifdef OKF_ELECT_STAMPS
    const bool stamp_on = TMA_WARPS == kStampWarps && lane == 0 && blockIdx.x < kStampBlocks;
    if (stamp_on && warp == 0) asm volatile("mov.u32 %0, %%smid;" : "=r"(okf_elect_smid[blockIdx.x]));
#endif
    __syncthreads();
    if (!warp_active) return;  // fewer members than warps in the last group of a tile
    if (prm.T > 0 && warp == 0) {  // warp 0 of a block always has work
#pragma unroll
        for (int sg = 0; sg < kStages; ++sg) {
            if (sg < prm.T) {
                issue_g0<kOut, kMpc>(maps, sg, s_warp, g0w + sg * tile_elems, &bars[3 * sg], lane);
                issue_g1(maps, sg, s_warp, g1w + sg * tile_elems, &bars[3 * sg + 1], lane);
                if (n_lab) issue_g2(maps, sg, s_warp, n_lab, g2w + sg * tile_elems, &bars[3 * sg + 2], lane);
            }
        }
    }
    // A warp is done with group g of step t; the LAST warp of the block to get here refills the group for the next step.
    //   * Who is last (decoupled-group kernels): lane 0 draws a ticket, word g of the election line incremented by one; the last
    //     ticket of step t is (t + 1) n_active - 1.  The counter is never reset: no warp can draw for step t + 1 before that refill
    //     has landed, so the tickets of a step are the n_active values after those of the step before.  Every lane executes the
    //     atomic, on its own word of the 32-word line (lane 0 on word g, the others adding 0 to the rest of the line, the other
    //     groups' counters included): one conflict-free pass.  An add that only lane 0 executes is expanded by ptxas into a
    //     warp-aggregated sequence (vote, popc, shuffle, a second branch) whose dependent chain stalls the warp.
    //   * Ordering.  The hazard is the reads of the tile (ld.shared, generic proxy) by every warp against the TMA engine's
    //     overwrite with step t + 1 (async proxy).  __syncwarp orders the warp's reads before lane 0's ticket; the ticket is an
    //     acq_rel atomic on one location, so the last ticket acquires every earlier warp's release of its reads (the
    //     read-modify-writes form one release sequence), and the copy is issued after it by the thread that drew it.  No proxy
    //     fence: fence.proxy.async makes generic-proxy WRITES visible to the async proxy, and only the copies write the tiles.  The
    //     release is one MEMBAR.ALL.CTA ahead of the ticket; the form it replaces fenced with __threadfence_block (MEMBAR.SC.CTA)
    //     twice on the last reader's path and reset the counter in between.  Stamped at the bench shape (tools/probes/elect_stamps.py),
    //     election and copy issue take 577 cycles per warp-step against 934; FP64 bench 2.19e10 -> 2.28e10 trajectory-steps/s on one
    //     B200 at 1,000 W (profiles/r7_elect_ab.txt).  The warps of a scheduler are not in lockstep, so their windows do not stack.
    //   * The full-covariance kernels (!kBlock) keep that form: lane 0 adds 1 between two block-scope fences, and the last reader
    //     resets the counter before it issues the copy.  They run at the 255-register cap, where the ticket spills.
    const auto last_reader = [&](int g, long long t) -> int {
        __syncwarp();  // every lane of this warp has read its values
        if constexpr (TMA_WARPS == 1) {  // the block's only warp is always the last reader
            if (lane == 0) __threadfence_block();
            return lane == 0 ? 0 : 1;
        }
        if constexpr (!kBlock) {
            int last = 0;
            if (lane == 0) {
                __threadfence_block();
                int *consumed = reinterpret_cast<int *>(tickets);
                last = atomicAdd(&consumed[g], 1) == n_active - 1;
                if (last) {
                    consumed[g] = 0;
                    __threadfence_block();
                }
            }
            return last ? 0 : 1;
        }
        uint32_t ticket;
        asm volatile("atom.acq_rel.cta.shared::cta.add.u32 %0, [%1], %2;"
                     : "=r"(ticket)
                     : "r"(smem_u32(tickets + ((g + lane) & 31))), "r"(lane == 0 ? 1u : 0u)
                     : "memory");
        return lane == 0 && ticket == (uint32_t)(t + 1) * (uint32_t)n_active - 1u ? 0 : 1;  // 0 = "this lane issues the copy"
    };

    Real *q = noise + tid, *r = noise + 12 * nt + tid;
    load_noise(prm, N, ic, q, r, nt);
    if constexpr (kOut != 0) {  // K_gain = sum_j P[j][sel j] / r[j] is wanted every step: the ten reciprocals are taken once
#pragma unroll
        for (int c = 0; c < NZ; ++c) r[(NZ + c) * nt] = rcp_(r[c * nt]);
    }
    Real x[NX], P[NP];
#pragma unroll
    for (int c = 0; c < NX; ++c) x[c] = prm.x0_inc ? ld_traj(prm.x0, c * prm.x0_ld + ic, Real()) : Real(prm.x0[c]);
    load_P0<kBlock>(prm, N, ic, q, nt, P);

    uint32_t status[L];
#pragma unroll
    for (int ln = 0; ln < L; ++ln) status[ln] = 0;
    Real ptrace = Real(0), kgain = Real(0), ymax = Real(0);
    constexpr int kAccRegs = (kSummary && !kAccSmem) ? ACC_ROWS : 1;
    AccT acc_r[kAccRegs];
#pragma unroll
    for (int c = 0; c < kAccRegs; ++c) acc_r[c] = acc_zero(AccT());
    auto acc_add = [&](int idx, AccT v) {  // running sums: 0-11 truth, 12-23 nominal, 24 NIS
        if constexpr (kAccSmem) acc_s[idx * nt] = acc_s[idx * nt] + v;
        else if constexpr (kSummary) acc_r[idx] = acc_r[idx] + v;
    };
    auto acc_get = [&](int idx) -> AccT {
        if constexpr (kAccSmem) return acc_s[idx * nt];
        else if constexpr (kSummary) return acc_r[idx];
        else return acc_zero(AccT());
    };
    if constexpr (kSummary) {
#pragma unroll
        for (int c = 0; c < ACC_ROWS; ++c) {
            if constexpr (kAccSmem) acc_s[c * nt] = acc_zero(AccT()); else acc_r[c] = acc_zero(AccT());
        }
    }

    // label tiles of this lane; a label stream that was not given reads the (always valid) moments tile and is ignored
    const Real *lab_truth = (kSummary && prm.truth) ? g2w + lane : g0w + lane;
    const Real *lab_nominal = (kSummary && prm.nominal) ? g2w + (prm.truth ? 12 * 32 : 0) + lane : g0w + lane;
    // labels and running sums are fetched six at a time BEFORE they are used, so the shared-memory latency of one batch
    // overlaps the arithmetic around it
    auto accumulate = [&](int acc0, const Real *lab) {
#pragma unroll
        for (int c0 = 0; c0 < NX; c0 += 6) {
            Real lv[6];
#pragma unroll
            for (int c = 0; c < 6; ++c) lv[c] = lab[(c0 + c) * 32];
            if constexpr (kAccSmem) {
                AccT av[6];
#pragma unroll
                for (int c = 0; c < 6; ++c) av[c] = acc_s[(acc0 + c0 + c) * nt];
#pragma unroll
                for (int c = 0; c < 6; ++c) acc_s[(acc0 + c0 + c) * nt] = err_acc(av[c], x[c0 + c], lv[c]);
            } else if constexpr (kSummary) {
#pragma unroll
                for (int c = 0; c < 6; ++c) acc_r[acc0 + c0 + c] = err_acc(acc_r[acc0 + c0 + c], x[c0 + c], lv[c]);
            }
        }
    };

    const Real e1_mpc = kMpc ? exp_minus_one(Real(prm.dt)) : Real(0);
    // rotation of the prior attitude for step 0; inside the loop it is produced one step ahead
    Real Rm[9];
    rot_zyx(x[0], x[1], x[2], Rm);
    bool any_trunc = may_truncate(Rm);

    for (long long t = 0; t < prm.T; ++t) {
        const int stg = kStages == 2 ? (int)(t & 1) * tile_elems : 0;  // offset of this step's tile set
        const uint32_t par = kStages == 2 ? (uint32_t)((t >> 1) & 1) : (uint32_t)(t & 1);
        const bool more = t + kStages < prm.T;
        uint64_t *bar = bars + (kStages == 2 ? 3 * (int)(t & 1) : 0);
        Real *g0 = g0w + stg, *g1 = g1w + stg, *g2 = g2w + stg;

        // ---- G0: leg moments -> mean model ------------------------------------------------------------------
        OKF_STAMP(kStTop);
        mbar_wait(&bar[0], par);
        if constexpr (kOut == 2) {
            if (active && prm.p_world_steps) store_world_feet<32>(g0 + NM * 32 + lane, Rm, prm.p_world_steps, (t * 12) * N + i, N);
        }
        propagate_mean_from_moments<32>(prm, x, g0 + lane, Rm, any_trunc);
        Real E[kMpc ? 9 : 1];  // D[a][6 + k] = exp(dt Rb^T[a][k]) - 1 of the predict_mpc transition (kalman_filter.py:153-157)
        if constexpr (kMpc) {
            Real Rb[9];
            const Real *rf = g0 + (kG0Rows - TMA_CH_REF) * 32 + lane;
            rot_zyx(rf[0], rf[32], rf[64], Rb);
#pragma unroll
            for (int a = 0; a < 3; ++a)
#pragma unroll
                for (int k = 0; k < 3; ++k) E[3 * a + k] = exp_minus_one(Real(prm.dt) * Rb[3 * k + a]);
        }
        Real nis = Real(0), inv, inv_n;
        const auto first_pivot = [&] {
            const Real s = P[tri(0, 0)] + r[0];
            note_bad_pivot(s, status, OPTI_KF_ST_NOT_PD);
            inv = rcp_(s);
        };
        const auto refill_g0 = [&] {  // this warp has consumed the step's moments: the last one refills G0 for step t + 1
            OKF_STAMP(kStElect0);
            const int elect = last_reader(0, t);
            if (more) issue_g0<kOut, kMpc>(maps, t + kStages, s_warp, g0, &bar[0], elect);
            OKF_STAMP(kStElect0End);
        };
        // kBlock: the first pivot's reciprocal and the G0 refill come after the predict, so that the mean model's dependent chain,
        // the predict's independent FMAs and the reciprocal form one basic block the scheduler can interleave (the copy still has
        // the whole update phase to land).  The full-covariance kernels keep the refill here and the reciprocal after the G1 wait:
        // with 78 live covariance entries the longer live ranges spill.
        if constexpr (!kBlock) refill_g0();
        if constexpr (kOut == 2) {
            if (active && prm.x_model_steps) {
#pragma unroll
                for (int c = 0; c < NX; ++c) st_traj(prm.x_model_steps, (t * NX + c) * N + i, x[c]);
            }
        }

        if constexpr (kMpc) cov_predict_mpc_sym(P, E, e1_mpc, q, nt);
        else cov_predict_sym<kBlock>(P, Rm, prm.dt, q, nt);
        if constexpr (kBlock) {
            first_pivot();
            refill_g0();
        }

        // ---- G1: measurements, folded in one at a time ---------------------------------------------------------
        mbar_wait(&bar[1], par);
        if constexpr (kSummary) {
            if (n_lab) mbar_wait(&bar[2], par);  // G2 (labels, fetched a step ahead like G0 / G1): used inside the last fold
        }
        const Real *z = g1 + lane;
        if constexpr (kOut == 2) {
            if (active && prm.z_steps) {
#pragma unroll
                for (int c = 0; c < NZ; ++c) st_traj(prm.z_steps, (t * NZ + c) * N + i, z[c * 32]);
            }
        }
        if constexpr (!kBlock) first_pivot();
        auto nothing = [] {};
        fold_pipelined<0, kBlock>(P, x, z[0 * 32], r[0 * nt], r[1 * nt], inv, inv_n, nis, status, nothing); inv = inv_n;
        fold_pipelined<1, kBlock>(P, x, z[1 * 32], r[1 * nt], r[2 * nt], inv, inv_n, nis, status, nothing); inv = inv_n;
        fold_pipelined<2, kBlock>(P, x, z[2 * 32], r[2 * nt], r[3 * nt], inv, inv_n, nis, status, nothing); inv = inv_n;
        fold_pipelined<3, kBlock>(P, x, z[3 * 32], r[3 * nt], r[4 * nt], inv, inv_n, nis, status, nothing); inv = inv_n;
        fold_pipelined<4, kBlock>(P, x, z[4 * 32], r[4 * nt], r[5 * nt], inv, inv_n, nis, status, nothing); inv = inv_n;
        fold_pipelined<5, kBlock>(P, x, z[5 * 32], r[5 * nt], r[6 * nt], inv, inv_n, nis, status, nothing); inv = inv_n;
        fold_pipelined<6, kBlock>(P, x, z[6 * 32], r[6 * nt], r[7 * nt], inv, inv_n, nis, status, nothing); inv = inv_n;
        fold_pipelined<7, kBlock>(P, x, z[7 * 32], r[7 * nt], r[8 * nt], inv, inv_n, nis, status, nothing); inv = inv_n;
        fold_pipelined<8, kBlock>(P, x, z[8 * 32], r[8 * nt], r[9 * nt], inv, inv_n, nis, status, nothing); inv = inv_n;
        const Real z9 = z[9 * 32], r9 = r[9 * nt];
        {  // this warp has read its last measurement of the step: the last one refills G1 for step t + 1
            OKF_STAMP(kStElect1);
            const int elect = last_reader(1, t);
            if (more) issue_g1(maps, t + kStages, s_warp, g1, &bar[1], elect);
            OKF_STAMP(kStElect1End);
        }
        fold_pipelined<9, kBlock>(P, x, z9, r9, r9, inv, inv_n, nis, status, [&] {
            // the posterior state is final here: start the next step's sin/cos underneath the last rank-1 update
            rot_zyx(x[0], x[1], x[2], Rm);
            any_trunc = may_truncate(Rm);
            // ... and the running error sums of the summary: straight-line code (no branch on which label streams exist, an
            // absent one reads a valid dummy tile and is masked at the end), so that its shared-memory round trips are
            // scheduled underneath the 78 independent FMAs of the rank-1 update instead of stalling the tail of the step
            if constexpr (kSummary) {
                accumulate(0, lab_truth + stg);
                accumulate(12, lab_nominal + stg);
            }
        });

        ymax = max_(ymax, nis);

        if constexpr (kOut != 0) {
            ptrace = trace_of(P);
            if (prm.k_gain_steps != nullptr) kgain = gain_trace_rinv<kBlock>(P, r + NZ * nt, nt);
            if (active) store_step<kBlock, kOut == 2>(prm, t, N, i, x, P, ptrace, kgain, nis);
        }

        if constexpr (kSummary) {
            acc_add(24, to_acc(nis));
            if (n_lab) {
                OKF_STAMP(kStElect2);
                const int elect = last_reader(2, t);  // this warp has consumed the step's labels: the last one refills G2 for step t + 1
                if (more) issue_g2(maps, t + kStages, s_warp, n_lab, g2, &bar[2], elect);
                OKF_STAMP(kStElect2End);
            }
        }
        OKF_STAMP(kStEnd);
    }

    // A non-finite state is absorbing (NaN and Inf - Inf propagate through every later predict and update, nothing divides by
    // the state), so testing the final state flags the same trajectories as testing after every step.
#pragma unroll
    for (int c = 0; c < NX; ++c) note_nonfinite(x[c], status, OPTI_KF_ST_NONFINITE);
    if (!active) return;
    store_final<kBlock>(prm, N, i, x, P);
    if (kSummary && prm.summary) {
        if (prm.T > 0) {  // of the last step: the posterior P is still in registers
            ptrace = trace_of(P);
            kgain = gain_trace<kBlock>(P, r, nt);
        }
        store_summary(prm, i, x, P, acc_get, ptrace, kgain, ymax);
    }
    if (prm.status) {  // with the pre-pass flags (ALL_SWING) of each trajectory's stream
#pragma unroll
        for (int ln = 0; ln < L; ++ln)
            prm.status[i + ln] = status[ln] | (prm.stream_status ? prm.stream_status[s_warp + lane * L + ln] : 0u);
    }
}

}  // namespace okf
