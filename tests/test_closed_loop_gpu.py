"""GPU tests of the device closed loop (optistate_kf_closed_loop, csrc/kf_closed_loop.cu, behind estimate_state_mpc_batch) against
independent references, with a certificate local to each step so that nothing depends on how errors grow along the loop:
  * states: the C oracle (oracle/kf_oracle.c, predict_mpc covariance model, body_ref = column 0 of each step's horizon) driven by
    the forces the loop applied, from the same x0, P0, Q, R and model constants.  The predict_mpc covariance does not depend on the
    states or the forces, so the loop's states must be the oracle's to the FP64 bound;
  * forces: at every step, the oracle's QP (oracle/mpc_numpy.py) solved from the loop's own estimate of the step before.
The runs cover both filter kernels of the loop (the streamed one when N is a multiple of 32, the direct one otherwise), every MPC
kernel through the contact schedule and the solver options, all-swing steps, saturating demands, warm and cold starts, the noise
and initial-covariance forms, and the shared initial state, which only the C ABI can pass."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import c_oracle, cases
from oracle import mpc_numpy as mpc
from optistate_b200.mpc import W_STATE, estimate_state_mpc_batch
from optistate_b200.settings import INITIAL_PARAMS
from optistate_b200.synth import make_streams, monte_carlo_noise
from tests import mpc_cases, parity
from tests.test_mpc_constants_gpu import DEFAULTS, base_name, kernel_names

pytestmark = pytest.mark.gpu

MODEL = ("dt", "mass", "inertia", "gravity")       # constants of both the MPC and the filter; the others reach the MPC only
TROT_A, TROT_B = np.array([1.0, 0, 0, 1]), np.array([0, 1.0, 1, 0])


def trot_schedule(T, N, all_swing=()):
    """A trot that changes phase every three steps, a single stance leg every fifth step, and one all-swing step on the
    trajectories `all_swing`: at most two legs out of swing, the one-warp kernel throughout."""
    c = np.empty((T, 4, N))
    for t in range(T):
        for n in range(N):
            if t % 5 == 4:
                c[t, :, n] = 0.0
                c[t, (t + n) % 4, n] = 1.0
            else:
                c[t, :, n] = TROT_A if (t // 3 + n) % 2 == 0 else TROT_B
    for n in all_swing:
        c[T // 2, :, n] = 0.0
    return c


def stance_schedule(T, N):
    """Three and four legs in stance on most steps, a trot in between, each held for three steps (so that the warm start has a
    working set of the same legs to start from): the two-warp kernel."""
    pats = np.array([[1.0, 1, 1, 1], [1, 1, 1, 0], [1, 0, 0, 1], [0, 1, 1, 1], [1, 0, 1, 1], [1, 1, 0, 1]])
    c = np.empty((T, 4, N))
    for t in range(T):
        for n in range(N):
            c[t, :, n] = pats[(t // 3 + 2 * n) % len(pats)]
    return c


def horizon_ref(T, N, seed):
    """Horizon references [T, 5, 12, N]: the standing height, small attitudes, and on half of the trajectories a forward or
    sideways velocity demand large enough to saturate friction."""
    rng = np.random.default_rng(seed)
    ref = np.zeros((T, 5, 12, N))
    ref[:, :, 5, :] = 0.28
    ref[:, :, 0:3, :] = 0.02 * rng.standard_normal((T, 5, 3, N))
    ref[:, :, 9, 1::4] = 3.0
    ref[:, :, 10, 3::4] = -2.5
    return ref


def setup(N, T, seed, contact):
    st = make_streams(range(seed, seed + N), T)
    st["contact"] = np.ascontiguousarray(contact)
    x0 = cases.START.reshape(12, 1) + 0.01 * np.random.default_rng(seed).standard_normal((12, N))
    return st, horizon_ref(T, N, seed + 1), x0


def run_loop(st, ref, x0, profile=False, **kw):
    args = (st["imu"], st["p"], st["dp"], st["contact"], ref)
    call = lambda: [a.cpu().numpy() for a in estimate_state_mpc_batch(*args, x0=x0, return_p_world=True, **kw)]  # noqa: E731
    if profile:
        return kernel_names(call)
    return call(), None


def certify(st, ref, out, x0, P0=None, Q=None, R=None, consts=None, all_swing=()):
    """The step-local certificate of one closed-loop run; returns (worst state error, worst force error)."""
    consts = dict(DEFAULTS, **(consts or {}))
    xs, fs, mst, fst, pws = out
    T, _, N = xs.shape
    # every MPC solve succeeded; an all-swing step applies no force and flags exactly its trajectories
    assert not (mst & 7).any(), np.argwhere(mst & 7)
    swing = st["contact"].sum(axis=1) == 0                          # [T, N]
    assert np.all(fs.transpose(0, 2, 1)[swing] == 0.0)
    assert sorted(np.where(swing.any(axis=0))[0]) == sorted(all_swing)
    assert np.array_equal(fst & 4, np.where(swing.any(axis=0), 4, 0))
    # states: the C oracle on the applied forces
    streams = dict(imu=st["imu"], p=st["p"], dp=st["dp"], contact=st["contact"], f=fs, body_ref=np.ascontiguousarray(ref[:, 0]))
    o = c_oracle.run(streams, N, Q=Q, R=R, x0=x0, P0=P0, cov_model=1, want=("x_steps", "p_world_steps"),
                     **{k: consts[k] for k in MODEL})
    assert np.array_equal(fst, o["status"].astype(fst.dtype))
    x_err = max(parity.state_err(xs[:, :, n], o["x_steps"][:, :, n]) for n in range(N))
    p_err = max(parity.state_err(pws[:, :, n], o["p_world_steps"][:, :, n]) for n in range(N))
    assert x_err < parity.FP64_TOL and p_err < parity.FP64_TOL, (x_err, p_err)
    # forces: the oracle's stage 0 from the loop's estimate of the step before
    qp_kw, con_kw = mpc_cases.oracle_kw(consts)
    f_err = 0.0
    for t in range(T):
        for n in range(N):
            x_prev = x0[:, n] if t == 0 else xs[t - 1, :, n]
            H, g, _ = mpc.build_qp(x_prev, ref[t, :, :, n].T, st["p"][t, :, n], **qp_kw)
            A, b, pinned = mpc.constraints(st["contact"][t, :, n], **con_kw)
            want = mpc.solve_ldp(H, g, A, b, pinned)
            err = np.abs(fs[t, :, n] - want[0:12]).max() / max(1.0, np.abs(want).max())
            assert err <= 1e-8, (t, n, err)
            f_err = max(f_err, err)
    return x_err, f_err


def saturates(out, consts=None):
    """Some applied force sits on a friction face with a real normal force."""
    consts = dict(DEFAULTS, **(consts or {}))
    fs = out[1]
    fx, fy, fz = fs[:, 0::3, :], fs[:, 1::3, :], fs[:, 2::3, :]
    tol = 1e-7 * consts["fz_max"]
    face = (np.abs(np.abs(fx) - consts["mu"] * fz) < tol) | (np.abs(np.abs(fy) - consts["mu"] * fz) < tol)
    return bool((face & (fz > 1.0)).any())


def filter_kernels(names):
    """{'streamed' | 'direct': kMpc template argument} of the filter kernels among the profiler's kernel names."""
    out = {}
    for name in names:
        b = base_name(name)
        if b not in ("kf_seq_tma_kernel", "kf_seq_kernel"):
            continue
        args = [a.strip() for a in name[name.index("<") + 1:name.index(">(")].split(",")]
        k_mpc = args[3] if b == "kf_seq_tma_kernel" else args[2]   # <Real, kSummary, kOut, kMpc, ...> / <Real, kSummary, kMpc, kBlock>
        out.setdefault("streamed" if b == "kf_seq_tma_kernel" else "direct", set()).add(k_mpc in ("true", "1", "(bool)1"))
    return out


def test_trot_with_single_leg_and_all_swing_steps_streamed():
    """N = 64: the streamed predict_mpc filter kernel and the one-warp MPC kernel, default constants, P0 = Q, per-member x0; the
    warm start carries the working set from step to step and a cold run reaches the same loop with more constraint changes."""
    N, T = 64, 24
    swing = (5, 38)
    st, ref, x0 = setup(N, T, 100, trot_schedule(T, N, swing))
    out, names = run_loop(st, ref, x0, profile=True)
    assert filter_kernels(names) == {"streamed": {True}}, names
    assert {"kf_mpc_gi_kernel", "kf_mpc_kernel"} <= {base_name(k) for k in names} and "kf_mpc_gi2_kernel" not in {base_name(k) for k in names}
    assert saturates(out)
    x_err, f_err = certify(st, ref, out, x0, all_swing=swing)
    cold, _ = run_loop(st, ref, x0, warm=False)
    for a, b in ((out[0], cold[0]), (out[1], cold[1])):
        assert np.abs(a - b).max() <= 1e-9 * np.abs(b).max()
    changes_warm, changes_cold = int((out[2] >> 8).sum()), int((cold[2] >> 8).sum())
    assert changes_warm < changes_cold, (changes_warm, changes_cold)
    print(f"trot N=64: state {x_err:.2e} force {f_err:.2e}; constraint changes warm {changes_warm} cold {changes_cold}")


def test_three_and_four_leg_stance_direct_at_other_constants():
    """N = 45: the direct predict_mpc filter kernel and the two-warp MPC kernel, at a non-default constant set whose dt, mass,
    inertia and gravity reach the filter too, with per-member diagonal Q and R and a dense symmetric P0 with cross-group entries.
    (Not the light robot: at its constants the estimates tumble at up to 22 rad/s, and the C oracle's own states move by 5e-10 of
    their range when the forces move by 1e-15 relative, so last-bit differences exceed the FP64 bound; at these constants 7e-13.)"""
    N, T = 45, 20
    consts = mpc_cases.LOW_G
    st, ref, x0 = setup(N, T, 200, stance_schedule(T, N))
    q, r = monte_carlo_noise(np.arange(N), np.diag(cases.Q_DEFAULT), np.diag(cases.R_DEFAULT))
    m = 0.02 * np.random.default_rng(3).standard_normal((12, 12))
    P0 = np.diag(np.diag(cases.Q_DEFAULT)) + m @ m.T                    # couples every group
    out, names = run_loop(st, ref, x0, profile=True, P0=P0, Q=q, R=r, **consts)
    assert filter_kernels(names) == {"direct": {True}}, names
    assert {"kf_mpc_gi2_kernel", "kf_mpc_kernel"} <= {base_name(k) for k in names} and "kf_mpc_gi_kernel" not in {base_name(k) for k in names}
    assert saturates(out, consts)
    x_err, f_err = certify(st, ref, out, x0, P0=P0, Q=q, R=r, consts=consts)
    cold, _ = run_loop(st, ref, x0, P0=P0, Q=q, R=r, warm=False, **consts)
    for a, b in ((out[0], cold[0]), (out[1], cold[1])):
        assert np.abs(a - b).max() <= 1e-9 * np.abs(b).max()
    assert int((out[2] >> 8).sum()) < int((cold[2] >> 8).sum())
    print(f"stance N=45 ({consts['dt']} s, {consts['mass']} kg): state {x_err:.2e} force {f_err:.2e}")


def test_interior_point_solver_in_the_loop():
    """solver='interior_point' for every step, mixed leg counts, a shared diagonal P0 and per-member diagonal noise (N = 64)."""
    N, T = 64, 16
    c = stance_schedule(T, N)
    c[:, :, ::3] = trot_schedule(T, N)[:, :, ::3]
    st, ref, x0 = setup(N, T, 300, c)
    q, r = monte_carlo_noise(np.arange(N), np.diag(cases.Q_DEFAULT), np.diag(cases.R_DEFAULT))
    p0 = np.linspace(0.005, 0.05, 12)
    out, names = run_loop(st, ref, x0, profile=True, P0=p0, Q=q, R=r, solver="interior_point")
    bases = {base_name(k) for k in names}
    assert "kf_mpc_kernel" in bases and not ({"kf_mpc_gi_kernel", "kf_mpc_gi2_kernel"} & bases), bases
    assert filter_kernels(names) == {"streamed": {True}}, names
    assert saturates(out)
    x_err, f_err = certify(st, ref, out, x0, P0=np.diag(p0), Q=q, R=r)
    print(f"interior point N=64: state {x_err:.2e} force {f_err:.2e}")


def test_hand_over_to_the_interior_point_in_the_loop():
    """max_changes=3 on cold solves (N = 45, the trot with its all-swing steps): the dual active set hands the problems that need
    more changes to the interior point inside the loop, at another constant set."""
    N, T = 45, 20
    consts = mpc_cases.HEAVY
    swing = (0, 44)
    st, ref, x0 = setup(N, T, 400, trot_schedule(T, N, swing))
    full, _ = run_loop(st, ref, x0, warm=False, **consts)
    assert int(((full[2] >> 8) > 3).sum()) > N                      # this many solves need more than the cap
    out, names = run_loop(st, ref, x0, profile=True, warm=False, max_changes=3, **consts)
    assert {"kf_mpc_gi_kernel", "kf_mpc_kernel"} <= {base_name(k) for k in names}
    assert filter_kernels(names) == {"direct": {True}}, names
    assert not (out[2] & 16).any()
    x_err, f_err = certify(st, ref, out, x0, consts=consts, all_swing=swing)
    print(f"hand-over N=45: state {x_err:.2e} force {f_err:.2e}")


def test_one_trajectory_one_step():
    st, ref, x0 = setup(1, 1, 500, trot_schedule(1, 1))
    ref[:, :, 9] = 3.0
    out, names = run_loop(st, ref, x0, profile=True)
    assert filter_kernels(names) == {"direct": {True}}, names
    certify(st, ref, out, x0)
    assert out[0].shape == (1, 12, 1) and out[1].shape == (1, 12, 1)


P, I32, D = ctypes.c_void_p, ctypes.c_int32, ctypes.c_double


class _ClosedLoopDesc(ctypes.Structure):  # OptiKfClosedLoopDesc (include/optistate_kf.h)
    _fields_ = ([("struct_size", ctypes.c_uint32), ("abi_version", ctypes.c_uint32), ("dtype", I32), ("max_free_legs", I32),
                 ("n_traj", ctypes.c_int64), ("n_steps", ctypes.c_int64)]
                + [(n, P) for n in ("imu", "p", "dp", "contact", "body_ref", "x0")]
                + [("x0_per_traj", I32), ("p0_kind", I32), ("q_kind", I32), ("r_kind", I32)]
                + [(n, P) for n in ("P0", "Q", "R", "x_steps", "forces", "p_world_steps", "mpc_status", "status", "workspace")]
                + [("workspace_bytes", ctypes.c_size_t), ("dt", D), ("mass", D), ("inertia", D * 3), ("gravity", D), ("mu", D),
                   ("fz_max", D), ("w_state", D * 12), ("w_force", D), ("warm_start", I32), ("solver", I32), ("max_changes", I32),
                   ("reserved0", I32)])


def test_shared_initial_state_through_the_c_abi():
    """x0_per_traj = 0 (one [12] state broadcast to every trajectory at step 0) with forces, mpc_status and status left NULL:
    the same states, bit for bit, as the Python call with that state repeated per trajectory."""
    from optistate_b200 import _build

    lib = ctypes.CDLL(_build.build_all()[0])
    lib.optistate_kf_closed_loop_workspace_bytes.restype = ctypes.c_size_t
    lib.optistate_kf_closed_loop_workspace_bytes.argtypes = [ctypes.c_int64, ctypes.c_int64]
    N, T = 64, 12
    swing = (9,)
    st, ref, _ = setup(N, T, 600, trot_schedule(T, N, swing))
    x_shared = cases.START.reshape(12) + 0.01 * np.random.default_rng(6).standard_normal(12)
    want = estimate_state_mpc_batch(st["imu"], st["p"], st["dp"], st["contact"], ref, x0=np.repeat(x_shared[:, None], N, axis=1))[0]
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()  # noqa: E731
    keep = {k: dev(st[k]) for k in ("imu", "p", "dp", "contact")}
    keep.update(body_ref=dev(ref), x0=dev(x_shared), Q=dev(np.diag(INITIAL_PARAMS.Q)), R=dev(np.diag(INITIAL_PARAMS.R)),
                x_steps=torch.full((T, 12, N), np.nan, dtype=torch.float64, device="cuda"))
    nbytes = int(lib.optistate_kf_closed_loop_workspace_bytes(N, T))
    keep["workspace"] = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    d = _ClosedLoopDesc()
    d.struct_size, d.abi_version, d.dtype = ctypes.sizeof(_ClosedLoopDesc), lib.optistate_kf_abi_version(), 0
    d.max_free_legs, d.n_traj, d.n_steps = int(st["contact"].sum(axis=1).max()), N, T
    for k, t in keep.items():
        setattr(d, k, t.data_ptr())
    d.workspace_bytes = nbytes
    d.x0_per_traj, d.p0_kind, d.q_kind, d.r_kind = 0, 0, 1, 1
    d.dt, d.mass, d.gravity, d.mu, d.fz_max, d.w_force = (DEFAULTS[k] for k in ("dt", "mass", "gravity", "mu", "fz_max", "w_force"))
    d.inertia = (ctypes.c_double * 3)(*DEFAULTS["inertia"])
    d.w_state = (ctypes.c_double * 12)(*W_STATE)
    d.warm_start = 1
    rc = lib.optistate_kf_closed_loop(ctypes.byref(d), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, rc
    torch.cuda.synchronize()
    assert torch.equal(keep["x_steps"], want)
