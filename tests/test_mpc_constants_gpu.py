"""GPU tests of the force MPC's constants (dt, mass, inertia, gravity, mu, fz_max, w_state, w_force) on each of its three solver
kernels: the one-warp dual active set (kf_mpc_gi_kernel, at most two legs out of swing), the two-warp dual active set
(kf_mpc_gi2_kernel, three or four), and the interior point (kf_mpc_kernel), alone and behind the other two when they hand a problem
over.  Every kernel reads each constant itself, so each is compared with the oracle's active-set solve (oracle/mpc_numpy.py) at the
same constants, varied one at a time and in combined sets, and each variant must move the minimiser far beyond the tolerance."""
import numpy as np
import pytest
import torch

from optistate_b200.mpc import ST_WARM, W_FORCE, W_STATE, WarmStart, mpc_forces
from optistate_b200.settings import INITIAL_PARAMS
from oracle import mpc_numpy as mpc
from tests import mpc_cases

pytestmark = pytest.mark.gpu

DEFAULTS = dict(dt=INITIAL_PARAMS.DT_mpc, mass=INITIAL_PARAMS.ROBOT_MASS, inertia=tuple(np.diag(INITIAL_PARAMS.INERTIA_ROT)),
                gravity=INITIAL_PARAMS.GRAVITY, mu=0.6, fz_max=150.0, w_state=W_STATE, w_force=W_FORCE)


def _sweep():
    """Each constant alone: two values of the scalars (w_force above its default of 1e-6 up to 1e-2: below 1e-6, H is too
    ill-conditioned for these bounds), each inertia axis, and each state weight x4 and at zero."""
    out = []
    for key, vals in (("dt", (0.005, 0.02)), ("mass", (6.0, 14.0)), ("gravity", (-3.71, -15.0)), ("mu", (0.3, 0.9)),
                      ("fz_max", (90.0, 250.0)), ("w_force", (1e-5, 1e-2))):
        out += [(f"{key}={v:g}", {key: v}) for v in vals]
    for a in range(3):
        inertia = list(DEFAULTS["inertia"])
        inertia[a] *= 3.0
        out.append((f"inertia{a}x3", {"inertia": tuple(inertia)}))
    for k in range(12):
        for f in (4.0, 0.0):
            w = list(W_STATE)
            w[k] *= f
            out.append((f"w_state{k}x{f:g}", {"w_state": tuple(w)}))
    return out


SWEEP = _sweep()
N = 64          # mpc_cases.batch: all 16 contact patterns at four lateral demands (0, 0.5, 3, -2 m/s), with height errors
worst = {}      # path -> worst |u - u_oracle| / max(1, |u_oracle|) over the module


def base_name(name):
    """'void okf::kf_mpc_gi_kernel(okf::MpcParams)' -> 'kf_mpc_gi_kernel'."""
    head = name.split("(")[0].split("<")[0]
    return head.split()[-1].split("::")[-1]


def kernel_names(fn):
    """(result of fn(), demangled names of the CUDA kernels it ran, as torch.profiler reports them)."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    return res, {ev.key for ev in prof.key_averages()}


def kernels_of(fn):
    """(result of fn(), base names of the CUDA kernels it ran)."""
    res, names = kernel_names(fn)
    return res, {base_name(k) for k in names}


def _problems():
    x, ref, p, c = mpc_cases.batch(N, seed=0)
    legs = c.sum(axis=0)
    return x, ref, p, c, np.where(legs <= 2)[0], np.where(legs >= 3)[0]


def solve_paths(consts, profile=False):
    """Forces [5, 12, N] and status [N] of every problem by each solver path; the dual active-set paths see only the problems of
    their leg count, so that the batch bound (max_free_legs from `contact`) selects their kernel."""
    x, ref, p, c, lo, hi = _problems()
    run = kernels_of if profile else (lambda fn: (fn(), None))
    paths, names = {}, {}

    def sub(idx, **kw):
        return mpc_forces(x[:, idx], ref[:, :, idx], p[:, idx], c[:, idx], **consts, **kw)

    for path, parts in (("one_warp", [(lo, {})]), ("two_warp", [(hi, {})]), ("interior_point", [(np.arange(N), {"solver": "interior_point"})]),
                        ("hand_over", [(lo, {"max_changes": 3}), (hi, {"max_changes": 3})])):
        F = np.full((5, 12, N), np.nan)
        st = np.zeros(N, np.int64)
        names[path] = []
        for idx, kw in parts:
            (f, s), ks = run(lambda: sub(idx, **kw))
            F[:, :, idx], st[idx] = f.cpu().numpy(), s.cpu().numpy()
            names[path].append(ks)
        paths[path] = (F, st, np.concatenate([i for i, _ in parts]))
    return paths, names


def oracle_solutions(consts):
    x, ref, p, c, _, _ = _problems()
    qp_kw, con_kw = mpc_cases.oracle_kw(consts)
    out = []
    for k in range(N):
        H, g, _ = mpc.build_qp(x[:, k], ref[:, :, k].T, p[:, k], **qp_kw)
        A, b, pinned = mpc.constraints(c[:, k], **con_kw)
        out.append((mpc.solve_ldp(H, g, A, b, pinned), H, g, A, b, pinned))
    return out


def check_against_oracle(paths, oracle, consts, label):
    """Each path's forces: the oracle's minimiser to 1e-8 of its size, feasible to 1e-7 N at fz_max = 150 (scaled with fz_max),
    stationary to 1e-8 |g|, no failure bit."""
    fz_tol = 1e-7 * consts["fz_max"] / 150.0
    for path, (F, st, idx) in paths.items():
        assert not (st[idx] & 7).any(), (label, path, np.where(st & 7)[0])
        for k in idx:
            want, H, g, A, b, pinned = oracle[k]
            u = F[:, :, k].reshape(-1)
            err = np.abs(u - want).max() / max(1.0, np.abs(want).max())
            worst[path] = max(worst.get(path, 0.0), err)
            assert err <= 1e-8, (label, path, k, err)
            viol, stat = mpc.kkt_certificate(u, H, g, A, b, pinned)
            assert viol <= fz_tol and stat <= 1e-8, (label, path, k, viol, stat)
            assert np.all(u[pinned] == 0.0)


def check_moved(paths, base, label):
    """The variant's minimiser differs from the default-constant one by more than 1e3 x the tolerance on some problem of every
    path: a kernel that ignored the constant could not pass."""
    for path, (F, _, idx) in paths.items():
        B = base[path][0]
        moved = max(np.abs(F[:, :, k] - B[:, :, k]).max() / max(1.0, np.abs(F[:, :, k]).max()) for k in idx)
        assert moved > 1e-5, (label, path, moved)


@pytest.fixture(scope="module")
def default_paths():
    paths, _ = solve_paths(DEFAULTS)
    check_against_oracle(paths, oracle_solutions(DEFAULTS), DEFAULTS, "defaults")
    return paths


@pytest.mark.parametrize("label,change", SWEEP, ids=[s[0] for s in SWEEP])
def test_one_constant_at_a_time_on_every_solver_path(default_paths, label, change):
    consts = dict(DEFAULTS, **change)
    paths, _ = solve_paths(consts)
    check_against_oracle(paths, oracle_solutions(consts), consts, label)
    check_moved(paths, default_paths, label)


@pytest.mark.parametrize("name", sorted(mpc_cases.CONSTANT_SETS))
def test_combined_constant_sets_on_every_solver_path(default_paths, name):
    """A heavier robot, a lighter one with a longer step, and lower gravity with a shorter step; each has distinct per-axis
    weights with one of them zero.  The profiler shows which kernels ran on each path."""
    consts = mpc_cases.CONSTANT_SETS[name]
    paths, names = solve_paths(consts, profile=True)
    check_against_oracle(paths, oracle_solutions(consts), consts, name)
    check_moved(paths, default_paths, name)
    (one,), (two,), (ipm,), (ho_lo, ho_hi) = names["one_warp"], names["two_warp"], names["interior_point"], names["hand_over"]
    assert "kf_mpc_gi_kernel" in one and "kf_mpc_gi2_kernel" not in one, one
    assert "kf_mpc_gi2_kernel" in two and "kf_mpc_gi_kernel" not in two, two
    assert "kf_mpc_kernel" in ipm and not ({"kf_mpc_gi_kernel", "kf_mpc_gi2_kernel"} & ipm), ipm
    assert {"kf_mpc_gi_kernel", "kf_mpc_kernel"} <= ho_lo and {"kf_mpc_gi2_kernel", "kf_mpc_kernel"} <= ho_hi, (ho_lo, ho_hi)
    # the hand-over really happens: these problems need more than three constraint changes without the cap, so the
    # interior-point kernel solved them in the capped run (and check_against_oracle held its forces to the oracle)
    for part, (idx, st_full) in {"one_warp": (paths["one_warp"][2], paths["one_warp"][1]),
                                 "two_warp": (paths["two_warp"][2], paths["two_warp"][1])}.items():
        handed = int(((st_full[idx] >> 8) > 3).sum())
        assert handed >= 4, (name, part, handed)
    # the fz cap and the friction pyramid bind in this batch at these constants
    F = paths["interior_point"][0]
    fz, mu, fz_max = F[:, 2::3, :], consts["mu"], consts["fz_max"]
    assert (np.abs(fz - fz_max) < 1e-6 * fz_max).any()
    assert ((np.abs(np.abs(F[:, 0::3, :]) - mu * fz) < 1e-7 * fz_max) & (fz > 1.0)).any()
    print("worst |u - u_oracle| / max(1, |u_oracle|) by solver path so far:", {k: f"{v:.2e}" for k, v in sorted(worst.items())})


@pytest.mark.parametrize("name", sorted(mpc_cases.CONSTANT_SETS))
def test_warm_start_at_other_constants(name):
    """The checks test_mpc_gpu.py applies to the warm start at the default constants, at a non-default set, for the one-warp kernel
    (a trot with a few single-leg problems) and the two-warp kernel (all four legs in stance): the first warm solve is the cold one,
    a repeat solve starts from the answer and changes no constraint, and nearby problems reach the same minimiser as from scratch."""
    consts = mpc_cases.CONSTANT_SETS[name]
    qp_kw, con_kw = mpc_cases.oracle_kw(consts)
    n = 512
    x, ref, p, c = mpc_cases.batch(n, seed=11)
    trot = np.where((np.arange(n) % 2 == 0)[None, :], np.array([1.0, 0, 0, 1])[:, None], np.array([0, 1.0, 1, 0])[:, None])
    trot[:, ::17] = np.array([0.0, 1.0, 0.0, 0.0])[:, None]
    rng = np.random.default_rng(5)
    x2 = x + 2e-3 * rng.standard_normal(x.shape)
    ref2 = ref + 1e-3 * rng.standard_normal(ref.shape)
    for contact in (trot, np.ones((4, n))):
        cold, _ = mpc_forces(x, ref, p, contact, **consts)
        scale = float(cold.abs().max())
        warm = WarmStart(n)
        # an empty set is a cold solve; the two-warp kernel's warm path may round the last bit differently (5e-17 N, measured)
        first, s0 = mpc_forces(x, ref, p, contact, warm=warm, **consts)
        assert float((first - cold).abs().max()) <= 1e-15 * scale and not (s0 & (7 | ST_WARM)).any()
        again, s1 = mpc_forces(x, ref, p, contact, warm=warm, **consts)
        constrained = (warm.active[0] & 0xFFFFF) != 0
        assert int(constrained.sum()) > n // 4
        assert float((again - cold).abs().max()) < 1e-9 * scale and bool(((s1 & ST_WARM) != 0)[constrained].all())
        assert int((s1 >> 8)[constrained].max()) == 0
        near, s2 = mpc_forces(x2, ref2, p, contact, warm=warm, **consts)
        plain, s2c = mpc_forces(x2, ref2, p, contact, **consts)
        assert not (s2 & 7).any() and float((near - plain).abs().max()) < 1e-8 * scale
        assert float((s2 >> 8).double().mean()) < 0.5 * float((s2c >> 8).double().mean())
        F = near.cpu().numpy()
        for k in range(0, n, 37):
            H, g, _ = mpc.build_qp(x2[:, k], ref2[:, :, k].T, p[:, k], **qp_kw)
            A, b, pinned = mpc.constraints(contact[:, k], **con_kw)
            want = mpc.solve_ldp(H, g, A, b, pinned)
            u = F[:, :, k].reshape(-1)
            assert np.abs(u - want).max() <= 1e-8 * max(1.0, np.abs(want).max()), (name, k)
            viol, stat = mpc.kkt_certificate(u, H, g, A, b, pinned)
            assert viol <= 1e-7 * consts["fz_max"] / 150.0 and stat <= 1e-8, (name, k, viol, stat)

