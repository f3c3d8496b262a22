// Kernel parameters of the batched force MPC (kf_mpc_gi.cuh, kf_mpc.cuh); separate so that kf_abi.cu can fill them without seeing
// the kernels.
#pragma once

#include <stdint.h>

namespace okf {

constexpr uint32_t MPC_ST_GIVEN_UP = 16u;  // internal: the dual active-set kernel hands the problem to the interior-point kernel

struct MpcParams {
    long long N;
    int max_legs;                               // 1..4: bound on the legs not in swing of any problem (sizes shared memory)
    const double *x, *body_ref, *p, *contact;  // [12][N], [NH*12][N], [12][N], [4][N]
    double *forces;                             // [NH*12][N]
    uint32_t *status;                           // [N] required: the dual active-set kernels flag the problems they give up on here
    uint32_t *warm_set;                         // [NH][N] optional, in/out: working set of the previous / this solve (kf_mpc_gi.cuh)
    int only_flagged;                           // interior-point kernel: solve only the problems whose status is MPC_ST_GIVEN_UP
    int solver;                                 // 0 auto (dual active set, interior point behind it), 1 interior point only
    int max_changes;                            // dual active set: iteration cap (0 = MPCG_MAX_IT)
    double *warm_mult;                          // [NH*4*5][N] with warm_set: multipliers of the active rows
    double dt, inv_mass, inv_inertia[3], gravity, mu, fz_max, w_state[12], w_force;
};

}  // namespace okf
