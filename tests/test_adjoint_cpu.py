"""CPU tests of the filter's adjoint (no GPU): the NumPy reverse recursion of tests/adjoint_oracle.py against torch autograd through
a float64 torch restatement of the joint-form filter with the kernels' mean model, and the storage query of optistate_kf_adjoint
against the smoother's over a descriptor grid."""
import ctypes
import itertools

import numpy as np
import pytest
import torch

from oracle import cases
from oracle import kf_numpy as kn
from optistate_b200.synth import make_stream
from tests import adjoint_oracle as ao
from tests.test_abi_cpu import _valid_desc, lib  # noqa: F401 - the fixture

SEL = torch.tensor(kn.SEL)


def _rot(th):
    a, b, c = th[0], th[1], th[2]
    sa, ca, sb, cb, sc, cc = torch.sin(a), torch.cos(a), torch.sin(b), torch.cos(b), torch.sin(c), torch.cos(c)
    return torch.stack([torch.stack([cc * cb, cc * (sb * sa) - sc * ca, cc * (sb * ca) + sc * sa]),
                        torch.stack([sc * cb, sc * (sb * sa) + cc * ca, sc * (sb * ca) - cc * sa]),
                        torch.stack([-sb, cb * sa, cb * ca])])


def torch_filter(stream, x0, P0, q, r, dt=kn.DT):
    """The joint-form filter in float64 torch, mean model in the kernels' moment form; returns x+, x- [T, 12] and P+ [T, 12, 12]."""
    z = torch.tensor(np.stack([kn.form_measurement(stream["imu"][t], stream["p"][t], stream["dp"][t], stream["contact"][t])
                               for t in range(stream["imu"].shape[0])]))
    C = torch.tensor(ao.moments(stream["p"], stream["f"])).reshape(-1, 3, 3)
    fs = torch.tensor(stream["f"].reshape(-1, 4, 3).sum(axis=1))
    d = torch.tensor(dt / kn.INERTIA)
    H = torch.zeros(10, 12, dtype=torch.float64)
    H[torch.arange(10), SEL] = 1.0
    x, P = x0, P0
    xs, xm, Ps = [], [], []
    for t in range(z.shape[0]):
        R = _rot(x[0:3])
        CR = C[t] @ R
        g = torch.stack([CR[1, 2] - CR[2, 1], CR[2, 0] - CR[0, 2], CR[0, 1] - CR[1, 0]])
        Tm = torch.trunc(R.T.detach())
        xn = torch.cat([x[0:3] + dt * (Tm @ x[6:9]), x[3:6] + dt * x[9:12], x[6:9] + R @ (d * g),
                        x[9:12] + (dt / kn.MASS) * fs[t] + torch.tensor([0.0, 0.0, dt * kn.GRAVITY], dtype=torch.float64)])
        F = torch.eye(12, dtype=torch.float64)
        F = F + torch.zeros(12, 12, dtype=torch.float64).index_put((torch.arange(3)[:, None], torch.arange(6, 9)[None, :]), dt * R.T)
        F[3:6, 9:12] += dt * torch.eye(3, dtype=torch.float64)
        Pm = F @ P @ F.T + torch.diag(q)
        S = H @ Pm @ H.T + torch.diag(r)
        K = Pm @ H.T @ torch.linalg.inv(S)
        x = xn + K @ (z[t] - H @ xn)
        P = (torch.eye(12, dtype=torch.float64) - K @ H) @ Pm
        xs.append(x)
        xm.append(xn)
        Ps.append(P)
    return torch.stack(xs), torch.stack(xm), torch.stack(Ps), z.numpy(), C.reshape(-1, 9).numpy()


def _case(noise, p0, x0_att):
    stream = make_stream(41, 40)
    Q, R = (cases.Q_DEFAULT, cases.R_DEFAULT) if noise == "default" else cases.q_r_pkl()
    q, r = Q.diagonal().copy(), R.diagonal().copy()
    x0 = cases.START.copy()
    if x0_att:
        x0[0:3] = [0.05, -0.03, 0.2]
        x0[6:9] = [0.1, -0.2, 0.05]
    p0 = q.copy() if p0 is None else np.linspace(0.002, 0.03, 12)
    return stream, q, r, x0, p0


@pytest.mark.parametrize("noise,p0,x0_att", [("default", None, False), ("default", "diag", True), ("qrpkl", None, True),
                                             ("qrpkl", "diag", False)])
def test_oracle_equals_autograd(noise, p0, x0_att):
    """T = 40: q_bar, r_bar, x0_bar and diag P0_bar of the oracle equal torch.autograd's to 1e-11 of each one's largest magnitude.
    With P0 None the initial covariance is Q, held here as a leaf of its own so that its gradient is P0_bar."""
    stream, q, r, x0, p0 = _case(noise, p0, x0_att)
    qt, rt, x0t, p0t = (torch.tensor(v, requires_grad=True) for v in (q, r, x0, p0))
    xs, xm, Ps, z, C = torch_filter(stream, x0t, torch.diag(p0t), qt, rt)
    xbar = np.random.default_rng(7).standard_normal(xs.shape)
    (xs * torch.tensor(xbar)).sum().backward()
    g = ao.adjoint(xs.detach().numpy(), xm.detach().numpy(), Ps.detach().numpy(), z, C, xbar, x0, np.diag(p0), q, r)
    for name, sl, ref in (("q", slice(0, 12), qt.grad), ("r", slice(12, 22), rt.grad), ("x0", slice(22, 34), x0t.grad),
                          ("P0", slice(34, 46), p0t.grad)):
        ref = ref.numpy()
        err = np.abs(g[sl] - ref).max() / np.abs(ref).max()
        assert err <= 1e-11, (name, err)


N, S = 1000, 100
FAKE = ctypes.c_void_p(0x1000)  # never dereferenced: the queries only validate


def _up(b):
    return (b + 255) // 256 * 256


def test_storage_query_matches_the_smoothers_over_a_descriptor_grid(lib):  # noqa: F811
    """optistate_kf_adjoint_storage_bytes accepts exactly what optistate_kf_smooth_storage_bytes accepts, with the same codes, and
    asks for the smoother's storage plus z [T][10][S] when the filter forms it and the moments [T][12][S], each padded to 256 B."""
    accepted, refused = 0, set()
    d = _valid_desc(lib)
    d.n_traj, d.n_streams = N, S
    grid = itertools.product((0, 1), (0, 1, 2), (0, 1), (0, 1, 2, 3), (0, 1, 2, 3, 4), (1, 2, 3, 4), (1, 2, 3, 4), (True, False),
                             (False, True), (False, True), (False, True), (0, 37))
    for dtype, algo, cov, flags, p0k, qk, rk, formed, xs, xm, ref, T in grid:
        d.dtype, d.algo, d.cov_model, d.flags, d.n_steps = dtype, algo, cov, flags, T
        d.p0_kind, d.q_kind, d.r_kind = p0k, qk, rk
        d.P0 = FAKE if p0k else None
        d.phases, d.z_in = (7, None) if formed else (6, FAKE)
        d.x_steps = FAKE if xs else None
        d.x_model_steps = FAKE if xm else None
        d.body_ref = FAKE if ref else None
        esz = 8 if dtype == 0 else 4
        a, b = ctypes.c_size_t(123), ctypes.c_size_t(123)
        rc = lib.optistate_kf_smooth_storage_bytes(ctypes.byref(d), ctypes.byref(a))
        rc_adj = lib.optistate_kf_adjoint_storage_bytes(ctypes.byref(d), ctypes.byref(b))
        point = (dtype, algo, cov, flags, p0k, qk, rk, formed, xs, xm, ref, T)
        assert rc_adj == rc, point
        if rc != 0:
            refused.add(rc)
            continue
        accepted += 1
        assert b.value == a.value + (_up(T * 10 * S * esz) if formed else 0) + _up(T * 12 * S * esz), point
    assert accepted > 0 and refused >= {-1, -5}, (accepted, refused)
