/*
 * optistate_kf.h - C ABI of the B200-native batched Kalman filter for OptiState's estimation hot path.
 *
 * One shared library (liboptistate_kf.so, built for sm_100a) exports exactly these entry points.  They are
 * what a foreign-function binding of the reference would bind in place of its NumPy filter:
 *
 *   optistate_kf_batch      replaces the per-step call chain of the reference driver,
 *                           get_odom -> set_measurements -> predict(p, f) -> update()
 *                           (/root/reference/kalman_filter/kalman_filter.py:79-138,164-174 and
 *                            /root/reference/misc/force_controller.py:269-291), looped over T steps as in
 *                           /root/reference/data_collection/data_conversion_Kalman_to_Training.py:193-201,
 *                           for N independent trajectories at once.  With `phases` it also serves the
 *                           single calls Kalman_Filter.predict / .update / .predict_mpc (covariance part,
 *                           kalman_filter.py:153-161) make.
 *   optistate_kf_measure    replaces get_odom + set_measurements (kalman_filter.py:79-117) for S streams x T steps.
 *   optistate_fma_peak      measures the FP64 / FP32 FMA issue peak of the device (roofline denominator).
 *   optistate_kf_smooth     runs optistate_kf_batch and then the fixed-interval Rauch-Tung-Striebel smoother backwards over
 *                           its per-step estimates (optistate_kf_smooth_storage_bytes sizes its scratch).  The reference
 *                           has no smoother: this entry point has no reference counterpart.
 *   optistate_kf_smooth_full the same on the full covariance (predict_mpc model, coupled P0).
 *   optistate_kf_noise_em_stats / optistate_kf_noise_em_full_stats
 *                           the E-step of expectation-maximisation for diagonal Q and R on either smoother.
 *   optistate_kf_adjoint    the gradient of the filter's x_steps with respect to diagonal Q, R, x0 and P0 (an adjoint kernel
 *                           backwards over the forward pass).
 *
 * Conventions
 *   - plain C, no torch / C++ types; every pointer is a NON-OWNING DEVICE pointer unless stated otherwise;
 *     the library never allocates device memory and keeps no state besides a launch counter (re-entrant,
 *     thread-safe).
 *   - calls are asynchronous on the CUDA stream passed as `void* cuda_stream` (a cudaStream_t; NULL = default).
 *   - return value: 0 on success, a negative OPTI_KF_E_* code otherwise; nothing is thrown across the boundary.
 *     Per-trajectory numerical events (the reference's exceptions) are reported in `status[N]` bit masks.
 *   - layouts are structure-of-arrays with the trajectory / stream index fastest-varying:
 *       per-step inputs    [T][C][S]   element (t, c, s) at ((t*C + c)*S + s)
 *       per-step outputs   [T][C][N]
 *       per-trajectory     [C][N]
 *     Trajectory i reads base stream  stream_index[i]  or, when stream_index is NULL, (i + stream_offset) % S.
 *   - all floating-point arrays of one call share the scalar type `dtype` (double or float).
 */
#ifndef OPTISTATE_KF_H_
#define OPTISTATE_KF_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OPTISTATE_KF_ABI_VERSION 5

#define OPTI_KF_NX 12 /* states  [thx thy thz | x y z | wx wy wz | vx vy vz]   kalman_filter.py:9  */
#define OPTI_KF_NZ 10 /* measurements [th_imu(3) z_odom w_imu(3) v_odom(3)]    kalman_filter.py:11 */
#define OPTI_KF_SUMMARY_ROWS 52
#define OPTI_KF_MAX_PEERS 7        /* other GPUs of one NVSwitch box */
#define OPTI_KF_PEER_HANDLE_BYTES 64

/* dtype */
enum { OPTI_KF_F64 = 0, OPTI_KF_F32 = 1 };

/* algo
 *   JOINT       the reference's operand order on a full (not symmetrised) 12x12 P:  S = H P H^T + R,
 *               K = (P H^T) S^-1 by a Cholesky solve, P <- P - K (H P); dense Q / R / P0 allowed; emits K.
 *   SEQUENTIAL  diagonal R and Q, symmetric P0: the 10 measurements are folded in one at a time on a packed
 *               symmetric P held in registers (algebraically identical for diagonal R; parity to <=1e-12 of the
 *               reference is part of the test-suite).  This is the throughput path.
 *   AUTO        SEQUENTIAL when the descriptor allows it, JOINT otherwise.                                   */
enum { OPTI_KF_ALGO_AUTO = 0, OPTI_KF_ALGO_JOINT = 1, OPTI_KF_ALGO_SEQUENTIAL = 2 };

/* cov_model: 0 = predict():      F_d = I + dt F               (kalman_filter.py:125-135)
 *            1 = predict_mpc():  F_d = exp(dt F) element-wise, R from body_ref angles (kalman_filter.py:153-158);
 *                needs `body_ref`; both algos (SEQUENTIAL uses F_d = 1 1^T + a 12-entry sparse matrix).        */
enum { OPTI_KF_COV_PREDICT = 0, OPTI_KF_COV_MPC = 1 };

/* phases: which parts of a step run (all three for the batched recursion) */
enum { OPTI_KF_PHASE_MEASURE = 1, OPTI_KF_PHASE_PREDICT = 2, OPTI_KF_PHASE_UPDATE = 4, OPTI_KF_PHASE_ALL = 7 };

/* noise / initial-covariance array kinds */
enum {
    OPTI_KF_MAT_NONE = 0,       /* pointer ignored (P0: use Q, as settings.py:31 does)        */
    OPTI_KF_MAT_DIAG = 1,       /* [n]        one diagonal shared by every trajectory          */
    OPTI_KF_MAT_DIAG_PER = 2,   /* [n][N]     one diagonal per trajectory                      */
    OPTI_KF_MAT_DENSE = 3,      /* [n*n]      one dense row-major matrix shared                */
    OPTI_KF_MAT_DENSE_PER = 4   /* [n*n][N]   one dense row-major matrix per trajectory        */
};

/* flags (OptiKfDesc.flags)
 *   The predict() model decouples: F_d = I + dt F mixes attitude only with body rate (F[0:3,6:9] = R^T) and each position
 *   only with the velocity of the same axis (F[3:6,9:12] = I, kalman_filter.py:45-48); H selects, Q and R are diagonal.  With
 *   a P0 that has no entries across the groups {th, w}, {x, vx}, {y, vy}, {z, vz} - P0 = Q as in settings.py:31, or any
 *   diagonal P0 - every cross-group entry of P stays an exact zero in the reference as well, and the SEQUENTIAL kernels drop
 *   the multiplications by those zeros (30 packed scalars instead of 78; bit-identical results).  Diagonal P0 kinds select
 *   this automatically; P0_DECOUPLED lets the caller vouch for a dense P0; FULL_COVARIANCE turns it off (tests, comparison). */
enum { OPTI_KF_FLAG_P0_DECOUPLED = 1, OPTI_KF_FLAG_FULL_COVARIANCE = 2,
       OPTI_KF_FLAG_SCALAR_FP32 = 4, /* FP32: one trajectory per thread even where the packed two-per-thread kernel (FFMA2) applies */
       OPTI_KF_FLAG_STATUS_ACCUMULATE = 8 /* status[i] |= this call's flags instead of = (one stream per trajectory, no pre-pass):
                                             lets a caller that steps the filter call by call keep one status word per trajectory */ };

/* status[i] bits */
enum {
    OPTI_KF_ST_NOT_PD = 1,     /* a pivot of S was <= 0 or not finite: S is not positive definite.  SEQUENTIAL carries on
                                  with that pivot; JOINT switches to the pivoted inverse the reference uses            */
    OPTI_KF_ST_NONFINITE = 2,  /* a state became inf/nan                                                        */
    /* (Angles: sin / cos use a two-term Cody-Waite reduction, <= 1 ulp for |angle| <= 2e5 rad in FP64 and <= 8e3 rad in FP32 -
     *  thousands of turns; attitudes beyond that lose accuracy gradually and may flip the trunc(R^T) decision of
     *  force_controller.py:271 relative to NumPy.  Physical attitudes are within a few radians.)                              */
    OPTI_KF_ST_ALL_SWING = 4,  /* a step had sum(contact) == 0 (reference raises ValueError, kalman_filter.py:97-103);
                                  the odometry part of z is set to 0 for that step                              */
    OPTI_KF_ST_ASYMMETRIC = 8, /* JOINT: S was visibly asymmetric: pivoted inverse instead of the Cholesky solve */
    OPTI_KF_ST_SINGULAR = 16,  /* JOINT: the pivoted inverse of S met a zero pivot - where the reference's np.linalg.inv raises
                                  LinAlgError (kalman_filter.py:168); an indefinite but regular S does not set it       */
    OPTI_KF_ST_SMOOTH_NOT_PD = 32 /* optistate_kf_smooth: a pivot of a prior covariance P-_{t+1} was <= 0 or not finite; the
                                     backward recursion carries on with that pivot                                    */
};

/* error codes */
enum {
    OPTI_KF_OK = 0,
    OPTI_KF_E_NULL = -1,        /* descriptor or a required pointer is NULL                 */
    OPTI_KF_E_VERSION = -2,     /* struct_size / abi_version mismatch                        */
    OPTI_KF_E_DTYPE = -3,
    OPTI_KF_E_SHAPE = -4,       /* negative / zero sizes, bad ckpt_every, bad kinds          */
    OPTI_KF_E_UNSUPPORTED = -5, /* combination not available for the requested algo          */
    OPTI_KF_E_CUDA = -6,        /* the CUDA runtime reported an error at launch              */
    OPTI_KF_E_NO_DEVICE = -7
};

typedef struct OptiKfDesc {
    uint32_t struct_size; /* sizeof(OptiKfDesc) */
    uint32_t abi_version; /* OPTISTATE_KF_ABI_VERSION */
    int32_t dtype, algo, cov_model, phases;
    int64_t n_traj, n_steps, n_streams, stream_offset;
    double dt, mass, inertia[3], gravity; /* settings.py:5,11,20-23; kalman_filter.py:56 */

    /* per-step inputs [T][C][S]; which are required depends on `phases` */
    const void *imu;      /* C=6   MEASURE                                   */
    const void *p;        /* C=12  MEASURE, PREDICT (body-frame feet)        */
    const void *dp;       /* C=12  MEASURE                                   */
    const void *contact;  /* C=4   MEASURE (0/1 flags stored as dtype)       */
    const void *f;        /* C=12  PREDICT (world-frame forces)              */
    const void *z_in;     /* C=10  UPDATE without MEASURE (pre-formed z)     */
    const void *body_ref; /* C=12  cov_model == OPTI_KF_COV_MPC              */
    const void *truth;    /* C=12  optional label stream for the summary     */
    const void *nominal;  /* C=12  optional second label stream (summary)    */
    const int32_t *stream_index; /* [N] or NULL */

    /* initial state and noise */
    const void *x0; int32_t x0_per_traj;  /* [12] or [12][N] */
    int32_t p0_kind, q_kind, r_kind;
    const void *P0, *Q, *R;

    /* outputs, every one optional (NULL = not wanted) */
    void *x_steps;        /* [T][12][N] posterior state after update      */
    void *x_model_steps;  /* [T][12][N] predicted state (KF.x_model)      */
    void *p_world_steps;  /* [T][12][N] feet rotated into the world frame (the in-place mutation of
                             force_controller.py:274-277)                 */
    void *z_steps;        /* [T][10][N]                                   */
    void *p_trace_steps;  /* [T][N]  trace(P) after update                */
    void *k_gain_steps;   /* [T][N]  sum_{i<10} K[i][i]  (np.trace of the 12x10 gain) */
    void *nis_steps;      /* [T][N]  y^T S^-1 y                            */
    int64_t ckpt_every;   /* P checkpoints after steps ckpt_every, 2*ckpt_every, ... (0 = none) */
    void *P_ckpt;         /* [T/ckpt_every][144][N] row-major P           */
    void *x_final;        /* [12][N]                                      */
    void *P_final;        /* [144][N]                                     */
    void *K_final;        /* [120][N] row-major 12x10 gain of the last step (JOINT only) */
    void *summary;        /* [OPTI_KF_SUMMARY_ROWS][N]: 0-11 final x, 12-23 diag P, 24-35 RMSE vs truth,
                             36-47 RMS deviation from nominal, 48 mean NIS, 49 trace P, 50 K gain,
                             51 sqrt(max_t NIS_t)                          */
    uint32_t *status;     /* [N] */

    /* optional scratch (device memory owned by the caller) of at least optistate_kf_workspace_bytes():
       lets the SEQUENTIAL path hoist the state-independent work of every base stream - the measurement formation
       (unless z_in is given) and the leg moments of the mean model - into a pre-pass and stream the per-step inputs
       with TMA; without it the filter kernel forms both per trajectory */
    void *workspace;
    size_t workspace_bytes;

    /* multi-GPU: the all-gather of the summaries fused into the filter kernel.  `summary` points at this rank's first
       column inside a [OPTI_KF_SUMMARY_ROWS][summary_ld] array (summary_ld = trajectories of the whole job; 0 means
       n_traj, the single-GPU layout), and every summary_peers[k] at the same column of the same array in another
       GPU's memory, mapped into this process (optistate_kf_peer_open).  The kernel stores each summary value to all
       of them, so when the kernels of all ranks have finished every GPU holds the gathered array; the stores travel
       over NVLink while other trajectories are still being filtered.  The caller orders "all kernels finished" with
       a barrier of its own (one NCCL barrier in optistate_b200.distributed). */
    int64_t summary_ld;
    int32_t n_summary_peers; /* 0 .. OPTI_KF_MAX_PEERS */
    int32_t flags;           /* OPTI_KF_FLAG_* */
    void *summary_peers[OPTI_KF_MAX_PEERS];
} OptiKfDesc;

typedef struct OptiKfMeasureDesc {
    uint32_t struct_size, abi_version;
    int32_t dtype, reserved;
    int64_t n_steps, n_streams;
    const void *imu, *p, *dp, *contact; /* [T][6|12|12|4][S] */
    void *z;                            /* [T][10][S] */
    void *odom;                         /* [T][4][S] optional: z_odom, vx, vy, vz (get_odom's return value) */
    uint32_t *status;                   /* [S] optional, OPTI_KF_ST_ALL_SWING */
} OptiKfMeasureDesc;

/* ---- next row after the filter: feature rows, min-max normalisation and sliding windows for the GRU consumer ---- */
#define OPTI_KF_FEATURES 60 /* [x(12) imu_acc(6) f(12) p_world(12) dp(12) imu(6)], data_conversion_Kalman_to_Training.py:245-254 */

typedef struct OptiKfFeatureDesc {
    uint32_t struct_size, abi_version;
    int32_t dtype, reserved;
    int64_t n_traj, n_steps, n_streams, stream_offset;
    const int32_t *stream_index;          /* [N] or NULL, same mapping as OptiKfDesc */
    const void *x_steps, *p_world_steps;  /* [T][12][N] outputs of optistate_kf_batch */
    const void *imu, *imu_acc, *f, *dp;   /* [T][6|6|12|12][S]; imu_acc (the driver's imu_list[i][6:12]) may be NULL = zeros */
    void *rows;                           /* [N][T][60] row-major: the driver's state_INPUT rows per trajectory */
} OptiKfFeatureDesc;

/* Assembles the driver's 60-wide feature rows (replaces data_conversion_Kalman_to_Training.py:245-254). */
int optistate_kf_features(const OptiKfFeatureDesc *desc, void *cuda_stream);
/* Per-column minimum / maximum of a row-major [n_rows][n_cols] matrix (gru/gru_train.py:56-63); n_cols <= 256.
 * `scratch` is device memory of at least optistate_kf_minmax_scratch_bytes(dtype, n_cols). */
size_t optistate_kf_minmax_scratch_bytes(int dtype, int32_t n_cols);
int optistate_kf_minmax(int dtype, const void *rows, int64_t n_rows, int32_t n_cols, void *min_out, void *max_out, void *scratch,
                        size_t scratch_bytes, void *cuda_stream);
/* (v - min) / (max - min) in `dtype`, `n_latent` float32 latent columns appended, sliding windows of seq_len rows inside
 * each of the n_groups row groups, cast to float32 (gru/gru_train.py:108-111,180-192):
 * out [n_groups][rows_per_group - seq_len + 1][seq_len][n_cols + n_latent].  latent may be NULL iff n_latent == 0.
 * Every row is normalised once into `scratch` (device memory, optistate_kf_windows_scratch_bytes), then each window is a
 * contiguous copy of seq_len rows. */
size_t optistate_kf_windows_scratch_bytes(int64_t n_groups, int64_t rows_per_group, int32_t n_cols, int32_t n_latent);
int optistate_kf_windows(int dtype, const void *rows, const float *latent, const void *min, const void *max, int64_t n_groups,
                         int64_t rows_per_group, int32_t n_cols, int32_t n_latent, int32_t seq_len, float *out, void *scratch,
                         size_t scratch_bytes, void *cuda_stream);

/* ---- step before the filter: the driver's Q / R identification pass (data_conversion_Kalman_to_Training.py:31-109) ---- */
typedef struct OptiKfIdentifyDesc {
    uint32_t struct_size, abi_version;
    int32_t dtype;
    int32_t alias_last_measurement;       /* 1: reproduce the driver's aliasing of KF.z (:74) - every stored measurement is the last one */
    int64_t n_traj, n_steps, n_streams, stream_offset;
    const int32_t *stream_index;          /* [N] or NULL, same mapping as OptiKfDesc */
    double dt, mass, inertia[3], gravity;
    const void *gt;                       /* [T][12][S] ground-truth (mocap) states */
    const void *imu, *p, *dp, *contact, *f; /* [T][6|12|12|4|12][S]; f = the forces predict_mpc would apply at each step */
    void *q_diag;                         /* [12][N] variance of gt[i+1] - next_state(gt[i], p[i], f[i]) */
    void *r_diag;                         /* [10][N] variance of H gt[i+1] - z[i+1] */
    uint32_t *status;                     /* [N] optional, pre-zeroed by the caller; OPTI_KF_ST_ALL_SWING */
    void *scratch;                        /* device memory of optistate_kf_identify_scratch_bytes() */
    size_t scratch_bytes;
} OptiKfIdentifyDesc;
size_t optistate_kf_identify_scratch_bytes(int dtype, int64_t n_traj, int64_t n_steps);
int optistate_kf_identify_noise(const OptiKfIdentifyDesc *desc, void *cuda_stream);

/* ---- next row after those: the convex force MPC that predict_mpc solves for its forces (misc/force_controller.py:15-225,
 * set up by kalman_filter.py:64-77,140-152), batched.  One strictly convex QP per problem: 5 stages x 4 legs x 3 force
 * components; swing legs (contact == 0) carry no force, stance legs (contact == 1) satisfy fz <= fz_max, |fx| <= mu fz,
 * |fy| <= mu fz.  The reference solves it with CasADi + qpOASES, which are not available offline and no reference test pins
 * a force vector: the QP (objective and constraints) is pinned to the reference's own set-up code, the solver is anchored on
 * the uniqueness of the minimiser (tests check KKT optimality and an independent active-set solve).  FP64 only. ---- */
#define OPTI_KF_MPC_HORIZON 5
enum { OPTI_KF_MPC_ST_IPM_LIMIT = 1,  /* interior-point phase stopped on its iteration cap or a pivot breakdown       */
       OPTI_KF_MPC_ST_UNPOLISHED = 2, /* active-set polish did not settle: the forces are the interior-point iterate
                                         (~1e-6 relative) instead of the exact vertex solution                         */
       OPTI_KF_MPC_ST_TOO_MANY_LEGS = 4, /* more legs out of swing than max_free_legs promised: forces are NaN         */
       OPTI_KF_MPC_ST_WARM = 8         /* informational: the warm-start active set was verified, no interior-point phase */ };
typedef struct OptiKfMpcDesc {
    uint32_t struct_size, abi_version;
    int32_t dtype;                 /* OPTI_KF_F64 */
    int32_t max_free_legs;         /* bound on the legs with contact != 0 in any problem (1..4; 0 = unknown = 4): sizes the
                                      kernel's shared memory, i.e. its occupancy - a trot needs 2                       */
    int64_t n_problems;
    const void *x;                 /* [12][N] current state (column 0 of body_mpc, kalman_filter.py:143)              */
    const void *body_ref;          /* [5][12][N] reference states of the horizon (columns 1..5 of body_mpc)           */
    const void *p;                 /* [12][N] body-frame feet, held over the horizon (kalman_filter.py:141-142)       */
    const void *contact;           /* [4][N] 0 / 1 flags stored as dtype, held over the horizon (kalman_filter.py:145-146) */
    void *forces;                  /* [5][12][N] optimal forces; stage 0 is what predict_mpc applies (kalman_filter.py:161) */
    uint32_t *status;              /* [N] required: OPTI_KF_MPC_ST_* | iterations << 8; the dual active set also marks in it
                                      the problems it hands to the interior point                                       */
    /* Optional warm start for closed loops (estimate_state_mpc solves a near-identical QP every step), in / out, both or
     * neither: the working set (one word per stage: bit 5 leg + row, bits 24..27 legs out of swing, bit 31 valid; zeroed
     * memory = no warm start) and the multipliers of its rows.  The dual active set enters the stored set, drops the rows
     * whose multipliers come out negative and continues from there; a changed contact pattern starts cold.  (The interior
     * point ignores it.)                                                                                              */
    uint32_t *warm_set;            /* [5][N]                                                                           */
    void *warm_mult;               /* [5][4][5][N] doubles                                                              */
    int32_t solver;                /* 0 = dual active set, interior point for what it gives up on (default); 1 = the interior-point
                                      kernel only                                                                      */
    int32_t max_changes;           /* dual active set: constraints entered + dropped before a problem is handed to the interior
                                      point (0 = default 400) - a time budget for real-time callers                     */
    int32_t reserved0;
    double dt, mass, inertia[3], gravity;
    double mu, fz_max;             /* 0.6, 150 (force_controller.py:149-151)                                          */
    double w_state[12], w_force;   /* diag Q = P (kalman_filter.py:64,70) and the R value (:66)                        */
} OptiKfMpcDesc;
int optistate_kf_mpc_forces(const OptiKfMpcDesc *desc, void *cuda_stream);

/* ---- the closed loop the reference's conversion driver runs: KF.estimate_state_mpc(imu, p, dp, body_ref, contact) at every
 * step of every recording (data_conversion_Kalman_to_Training.py:193-201, kalman_filter.py:140-162,176-182).  For N trajectories
 * over T steps, all on the device and queued on the stream without a host synchronisation: the measurements of all steps in one
 * pre-pass (they do not depend on the state), then per step the force MPC of every trajectory from its CURRENT estimate
 * (optistate_kf_mpc_forces, warm-started from the previous step) and one filter step with those forces and the predict_mpc
 * covariance model (optistate_kf_batch, SEQUENTIAL: diagonal Q / R and a symmetric P0 - callers with dense noise step
 * optistate_kf_batch(algo = JOINT) themselves).  FP64. ---- */
typedef struct OptiKfClosedLoopDesc {
    uint32_t struct_size, abi_version;
    int32_t dtype;                 /* OPTI_KF_F64 */
    int32_t max_free_legs;         /* bound on the legs with contact != 0 at any step of any trajectory (1..4; 0 = unknown = 4) */
    int64_t n_traj, n_steps;
    const void *imu, *p, *dp, *contact; /* [T][6|12|12|4][N] */
    const void *body_ref;          /* [T][5][12][N]: horizon reference of every step; the filter's transition uses column 0   */
    const void *x0; int32_t x0_per_traj;   /* [12] or [12][N] */
    int32_t p0_kind, q_kind, r_kind;       /* OPTI_KF_MAT_NONE (P0 = Q) / _DIAG / _DIAG_PER; P0 also _DENSE / _DENSE_PER (symmetric) */
    const void *P0, *Q, *R;
    void *x_steps;                 /* [T][12][N] posterior state after every step (required)                              */
    void *forces;                  /* [T][12][N] optional: the stage-0 forces the MPC found and the filter applied         */
    void *p_world_steps;           /* [T][12][N] optional: feet rotated into the world frame (the driver's feature rows)   */
    uint32_t *mpc_status;          /* [T][N] optional: OPTI_KF_MPC_ST_* | iterations << 8 of every solve                    */
    uint32_t *status;              /* [N] optional: OPTI_KF_ST_* accumulated over the steps                                 */
    void *workspace;               /* device scratch of optistate_kf_closed_loop_workspace_bytes(n_traj, n_steps)          */
    size_t workspace_bytes;
    double dt, mass, inertia[3], gravity;
    double mu, fz_max, w_state[12], w_force;
    int32_t warm_start;            /* 1: carry the MPC's working set from step to step (default use), 0: cold solves       */
    int32_t solver, max_changes, reserved0;   /* as in OptiKfMpcDesc */
} OptiKfClosedLoopDesc;
size_t optistate_kf_closed_loop_workspace_bytes(int64_t n_traj, int64_t n_steps);
int optistate_kf_closed_loop(const OptiKfClosedLoopDesc *desc, void *cuda_stream);

/* ---- fixed-interval Rauch-Tung-Striebel smoother (offline: every measurement of the recording is known).  Runs the forward
 * pass exactly as optistate_kf_batch runs `filter` (its outputs, summary, status and workspace included), keeping the packed
 * posterior covariance of every step in `storage`, then a backward kernel, one thread per trajectory:
 *     G_t = P+_t F_{t+1}^T (P-_{t+1})^-1,  xs_t = x+_t + G_t (xs_{t+1} - x-_{t+1}),  Ps_t = P+_t + G_t (Ps_{t+1} - P-_{t+1}) G_t^T
 * from xs_{T-1} = x+_{T-1}, Ps_{T-1} = P+_{T-1}, with F_{t+1} the covariance transition of the filter's own predict (F[0:3,6:9] =
 * R(x+_t)^T).  SEQUENTIAL algo, predict() covariance model, diagonal Q and R, and a P0 without cross-group entries only (see the
 * flags above): anything else returns OPTI_KF_E_UNSUPPORTED.  status[i] gains OPTI_KF_ST_SMOOTH_NOT_PD. ---- */
typedef struct OptiKfSmoothDesc {
    uint32_t struct_size;       /* sizeof(OptiKfSmoothDesc) */
    uint32_t abi_version;       /* OPTISTATE_KF_ABI_VERSION */
    const OptiKfDesc *filter;   /* the forward pass (host pointer to its descriptor) */
    void *x_smooth;             /* [T][12][N] required: smoothed state */
    void *var_smooth;           /* [T][12][N] optional: diagonal of the smoothed covariance */
    void *storage;              /* device scratch of optistate_kf_smooth_storage_bytes(filter): packed P+ [T][30][N], plus x+ and x-
                                   [T][12][N] each unless filter->x_steps / filter->x_model_steps are given (they are read there) */
    size_t storage_bytes;
} OptiKfSmoothDesc;
int optistate_kf_smooth_storage_bytes(const OptiKfDesc *filter, size_t *bytes_out);
int optistate_kf_smooth(const OptiKfSmoothDesc *desc, void *cuda_stream);

/* ---- the same smoother on the FULL covariance: the predict_mpc covariance model (cov_model = OPTI_KF_COV_MPC, whose
 * F_d = 1 1^T + D makes P dense), OPTI_KF_FLAG_FULL_COVARIANCE and dense (symmetric) P0 kinds are taken besides everything
 * optistate_kf_smooth takes.  The forward pass always runs the full-covariance kernels and keeps all 78 entries of P+_t in
 * tri order, so `storage` (optistate_kf_smooth_full_storage_bytes) holds P+ [T][78][N] plus x+ and x- as above; the outputs of
 * the forward pass equal optistate_kf_batch's.  The backward kernel recomputes P-_{t+1} with the covariance model the filter
 * ran (predict_mpc: from body_ref rows 0-2 of step t + 1).  Whatever the SEQUENTIAL filter cannot run (dense Q or R, algo =
 * JOINT) returns OPTI_KF_E_UNSUPPORTED; AUTO runs SEQUENTIAL, so a dense P0 must be symmetric.  status[i] gains
 * OPTI_KF_ST_SMOOTH_NOT_PD. ---- */
int optistate_kf_smooth_full_storage_bytes(const OptiKfDesc *filter, size_t *bytes_out);
int optistate_kf_smooth_full(const OptiKfSmoothDesc *desc, void *cuda_stream);

/* ---- E-step of expectation-maximisation for diagonal Q and R, from the sensor streams alone.  Runs the forward pass exactly as
 * optistate_kf_smooth does, then the smoother's backward kernel with one more step, t = -1, for the model
 *     x_{-1} ~ N(x0, P0),  x_{t+1} = x-_{t+1} + F_{t+1} (x_t - x+_t) + w_t,  w_t ~ N(0, Q)  (t = -1 .. T-2, x+_{-1} = x0),
 *     z_t = H x_t + v_t,  v_t ~ N(0, R)  (t = 0 .. T-1),
 * whose smoother for t >= 0 is optistate_kf_smooth's.  Per trajectory, stats[row][i] holds
 *     rows 0-11   Sw_c = sum_t E[w_{t,c}^2 | Z]
 *     rows 12-21  Sv_k = sum_t E[v_{t,k}^2 | Z]
 *     row 22      the prediction-error log-likelihood sum_t log N(z_t; H x-_t, H P-_t H^T + R) of the filter that ran
 * so that the M-step is q = Sw / T, r = Sv / T (pooled: the sums over trajectories over N T).  Accepts exactly what
 * optistate_kf_smooth accepts, with the same return codes.  P0 absent means P0 = Q, as for the filter. ---- */
#define OPTI_KF_EM_STATS_ROWS 23  /* 0-11 Sw, 12-21 Sv, 22 log-likelihood */
typedef struct OptiKfNoiseEmDesc {
    uint32_t struct_size;       /* sizeof(OptiKfNoiseEmDesc) */
    uint32_t abi_version;       /* OPTISTATE_KF_ABI_VERSION */
    const OptiKfDesc *filter;   /* forward pass, run exactly as optistate_kf_batch runs it */
    void *stats;                /* [23][N] required */
    void *x_smooth, *var_smooth;  /* [T][12][N] optional here */
    void *storage;              /* device scratch of optistate_kf_noise_em_storage_bytes(filter): the smoother's storage, plus the
                                   measurements z [T][10][S] when the filter forms them (OPTI_KF_PHASE_MEASURE) */
    size_t storage_bytes;
} OptiKfNoiseEmDesc;
int optistate_kf_noise_em_storage_bytes(const OptiKfDesc *filter, size_t *bytes_out);
int optistate_kf_noise_em_stats(const OptiKfNoiseEmDesc *desc, void *cuda_stream);

/* ---- the same E-step on the FULL covariance: the model above with F_{t+1} the transition of either covariance model (predict_mpc:
 * F_d = 1 1^T + D from body_ref rows 0-2 of step t + 1, and of step 0 for the transition out of x_{-1}), and x_{-1} ~ N(x0, P0) with
 * any P0 kind, coupled or dense (symmetric).  Runs the forward pass exactly as optistate_kf_smooth_full does, then its backward
 * kernel with one more step, t = -1; the rows of `stats` mean what they mean above, and the innovation covariance of the
 * log-likelihood is the dense 10x10 H P-_t H^T + R.  Takes OptiKfNoiseEmDesc unchanged; `storage`
 * (optistate_kf_noise_em_full_storage_bytes) is optistate_kf_smooth_full's, plus z [T][10][S] when the filter forms the
 * measurements.  Accepts exactly what optistate_kf_smooth_full accepts, with the same return codes. ---- */
int optistate_kf_noise_em_full_storage_bytes(const OptiKfDesc *filter, size_t *bytes_out);
int optistate_kf_noise_em_full_stats(const OptiKfNoiseEmDesc *desc, void *cuda_stream);

/* ---- gradient of the filter's x_steps: the vector-Jacobian product of x+_t (t = 0 .. T-1) with respect to the diagonal Q, the
 * diagonal R, x0 and P0.  Runs the forward pass exactly as optistate_kf_smooth does, then an adjoint kernel, one thread per
 * trajectory, backwards over the joint form of the update (which the sequential update equals in exact arithmetic):
 *     a = 0, Pi = 0;  for t = T-1 .. 0:  a += x_bar_t;  b = K_t^T a;  r_bar_k += (K_t^T Pi K_t)_kk - b_k v_k;
 *     Pb = A_t^T Pi A_t + sym(A_t^T a v_t^T H);  q_bar_i += Pb_ii;  Pi = F_t^T Pb F_t;  a = J_t^T (A_t^T a) + (theta-term of F_t)
 * with A_t = I - K_t H, v_t = S_t^-1 (z_t - H x-_t) and J_t = dx-_t/dx+_{t-1} the derivative of the mean model (DESIGN.md section
 * 0.4); at the end x0_bar = a, P0_bar = Pi.  Per trajectory, grad[row][i] holds
 *     rows 0-11   q_bar = sum_t dL/dQ_ii through P-_t (never through P0 = Q: add rows 34-45 for that when P0 is absent)
 *     rows 12-21  r_bar = dL/dR_kk
 *     rows 22-33  x0_bar = dL/dx0
 *     rows 34-45  the diagonal of dL/dP+_{-1} (dL/dP0 when P0 is given)
 * for L any loss with dL/dx+_t = x_bar_t.  At an attitude where the mean model's trunc(R^T) changes (exactly axis-aligned, e.g.
 * the all-zero start) the filter is discontinuous in the attitude; the gradient there is the almost-everywhere one.  Accepts
 * exactly what optistate_kf_smooth accepts, with the same return codes; with a dense decoupled P0 rows 0-33 are exact and rows
 * 34-45 the diagonal of dL/dP0.  status[i] gains OPTI_KF_ST_SMOOTH_NOT_PD when a pivot of S_t is not positive and finite. ---- */
#define OPTI_KF_ADJ_ROWS 46  /* 0-11 q_bar, 12-21 r_bar, 22-33 x0_bar, 34-45 diag P0_bar */
typedef struct OptiKfAdjointDesc {
    uint32_t struct_size;       /* sizeof(OptiKfAdjointDesc) */
    uint32_t abi_version;       /* OPTISTATE_KF_ABI_VERSION */
    const OptiKfDesc *filter;   /* forward pass, run exactly as optistate_kf_batch runs it */
    const void *x_bar;          /* [T][12][N] required: dL/dx+_t */
    void *grad;                 /* [46][N] required */
    void *storage;              /* device scratch of optistate_kf_adjoint_storage_bytes(filter): the smoother's storage, plus the
                                   measurements z [T][10][S] when the filter forms them (OPTI_KF_PHASE_MEASURE) and the leg moments
                                   of the mean model [T][12][S] */
    size_t storage_bytes;
} OptiKfAdjointDesc;
int optistate_kf_adjoint_storage_bytes(const OptiKfDesc *filter, size_t *bytes_out);
int optistate_kf_adjoint(const OptiKfAdjointDesc *desc, void *cuda_stream);

/* Runs the filter; dtype taken from the descriptor. */
int optistate_kf_batch(const OptiKfDesc *desc, void *cuda_stream);
/* Same, asserting the scalar type (the two names a binding would import). */
int optistate_kf_batch_f64(const OptiKfDesc *desc, void *cuda_stream);
int optistate_kf_batch_f32(const OptiKfDesc *desc, void *cuda_stream);
/* Batched measurement formation. */
int optistate_kf_measure(const OptiKfMeasureDesc *desc, void *cuda_stream);
/* Which algo optistate_kf_batch would run for this descriptor (OPTI_KF_ALGO_JOINT / _SEQUENTIAL) or an error. */
int optistate_kf_resolve_algo(const OptiKfDesc *desc);
/* Scratch memory the call can use (0 when it would not be used); see OptiKfDesc.workspace. */
int optistate_kf_workspace_bytes(const OptiKfDesc *desc, size_t *bytes_out);
/* FMA-chain micro-benchmark: sustained FLOP/s (2 per FMA) of dependent-free FMA issue on the current device.
 * Synchronises the stream (it has to time the kernel).  seconds_out may be NULL. */
int optistate_fma_peak(int dtype, int64_t fma_per_thread, double *flops_per_s_out, double *seconds_out, void *cuda_stream);
/* Number of kernel launches this library has made in this process (for bench.py's gpu_launches claim). */
int64_t optistate_kf_launch_count(void);

/* Peer memory for the fused summary all-gather (one process per GPU, all GPUs of one box).  optistate_kf_peer_alloc
 * returns a dedicated device allocation on the current device (exportable: offset 0 of its own cudaMalloc);
 * _export fills an opaque handle that another process passes to _open to map the allocation into its address
 * space with peer access over NVLink (cudaIpc*, lazy peer enable); _close unmaps, _free releases. */
int optistate_kf_peer_alloc(size_t bytes, void **dev_ptr_out);
int optistate_kf_peer_free(void *dev_ptr);
int optistate_kf_peer_export(void *dev_ptr, unsigned char handle_out[OPTI_KF_PEER_HANDLE_BYTES]);
int optistate_kf_peer_open(const unsigned char handle[OPTI_KF_PEER_HANDLE_BYTES], void **peer_ptr_out);
int optistate_kf_peer_close(void *peer_ptr);

const char *optistate_kf_strerror(int code);
int optistate_kf_abi_version(void);
size_t optistate_kf_desc_size(void);

#ifdef __cplusplus
}
#endif
#endif /* OPTISTATE_KF_H_ */
