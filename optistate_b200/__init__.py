"""optistate_b200 - B200-native (sm_100a) batched Kalman filter for OptiState's estimation hot path.

    from optistate_b200 import Kalman_Filter, kf_batch

`Kalman_Filter` is the drop-in for the reference class (same constructor / predict / update surface);
`kf_batch` filters thousands to millions of independent trajectories in one kernel launch;
`kf_smooth` adds the fixed-interval (Rauch-Tung-Striebel) smoother for offline recordings (`kf_smooth_full`: the same on the
full covariance, for the predict_mpc model and coupled P0), and `kf_noise_em` estimates
diagonal Q and R from the sensor streams alone by expectation-maximisation on it (`kf_noise_stats`: one E-step;
`kf_noise_em_full` / `kf_noise_stats_full`: the same on the full covariance).  `kf_states` is kf_batch's x_steps as a
differentiable function of Q, R, x0 and P0 for torch autograd (`kf_vjp`: one gradient from the adjoint kernel).
They call the CUDA library liboptistate_kf.so (C ABI: include/optistate_kf.h) through a thin PyTorch C++
extension.  There is no CPU fallback: without the built extension and a CUDA device the calls raise.
"""
from .settings import INITIAL_PARAMS  # noqa: F401


def __getattr__(name):
    # torch and the native extension are imported on first use so that `import optistate_b200` stays cheap
    if name in ("kf_batch", "kf_smooth", "kf_smooth_full", "kf_noise_stats", "kf_noise_em", "kf_noise_stats_full",
                "kf_noise_em_full", "kf_vjp", "kf_states", "kf_measure", "fma_peak", "KfBatchResult", "KfNoiseEmResult",
                "SUMMARY_FIELDS", "EM_FIELDS", "ADJ_FIELDS"):
        from . import batch

        return getattr(batch, name)
    if name == "Kalman_Filter":
        from .kalman_filter import Kalman_Filter

        return Kalman_Filter
    if name == "mpc_forces":
        from .mpc import mpc_forces

        return mpc_forces
    if name in ("shard_range", "kf_batch_sharded", "gather_summaries"):
        from . import distributed

        return getattr(distributed, name)
    raise AttributeError(name)
