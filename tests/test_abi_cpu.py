"""CPU tests of the boundary: the C-ABI library loads and exports every symbol include/optistate_kf.h declares,
descriptor validation / algorithm resolution / error strings work without a GPU, the PyTorch extension loads and
refuses CPU tensors (there is no CPU fallback), and the product package never imports the oracle."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from optistate_b200 import _build

    path, _ = _build.build_all()
    return ctypes.CDLL(path)


def declared_symbols():
    hdr = open(os.path.join(ROOT, "include", "optistate_kf.h")).read()
    return sorted(set(re.findall(r"\b(optistate_[a-z0-9_]+)\s*\(", hdr)))


def test_every_declared_symbol_is_exported(lib):
    syms = declared_symbols()
    assert {"optistate_kf_batch", "optistate_kf_batch_f64", "optistate_kf_batch_f32", "optistate_kf_measure",
            "optistate_kf_resolve_algo", "optistate_kf_workspace_bytes", "optistate_fma_peak", "optistate_kf_launch_count",
            "optistate_kf_strerror", "optistate_kf_abi_version", "optistate_kf_desc_size", "optistate_kf_peer_alloc",
            "optistate_kf_peer_free", "optistate_kf_peer_export", "optistate_kf_peer_open", "optistate_kf_peer_close"} <= set(syms)
    for s in syms:
        assert getattr(lib, s) is not None, s


def test_library_is_built_for_sm_100a():
    import subprocess

    from optistate_b200 import _build

    out = subprocess.run(["cuobjdump", "-lelf", _build.KF_LIB], capture_output=True, text=True).stdout
    assert "sm_100a" in out, out


def _desc_class(lib):
    """ctypes mirror of OptiKfDesc - what the reference-side binding of INTEGRATION.md declares."""
    P, I32, I64, D = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_double

    class Desc(ctypes.Structure):
        _fields_ = ([("struct_size", ctypes.c_uint32), ("abi_version", ctypes.c_uint32), ("dtype", I32), ("algo", I32),
                     ("cov_model", I32), ("phases", I32), ("n_traj", I64), ("n_steps", I64), ("n_streams", I64),
                     ("stream_offset", I64), ("dt", D), ("mass", D), ("inertia", D * 3), ("gravity", D)]
                    + [(n, P) for n in ("imu", "p", "dp", "contact", "f", "z_in", "body_ref", "truth", "nominal", "stream_index")]
                    + [("x0", P), ("x0_per_traj", I32), ("p0_kind", I32), ("q_kind", I32), ("r_kind", I32), ("P0", P), ("Q", P), ("R", P)]
                    + [(n, P) for n in ("x_steps", "x_model_steps", "p_world_steps", "z_steps", "p_trace_steps", "k_gain_steps", "nis_steps")]
                    + [("ckpt_every", I64)]
                    + [(n, P) for n in ("P_ckpt", "x_final", "P_final", "K_final", "summary", "status", "workspace")]
                    + [("workspace_bytes", ctypes.c_size_t), ("summary_ld", I64), ("n_summary_peers", I32), ("flags", I32),
                       ("summary_peers", P * 7)])

    lib.optistate_kf_desc_size.restype = ctypes.c_size_t
    assert ctypes.sizeof(Desc) == lib.optistate_kf_desc_size()
    return Desc


def _valid_desc(lib):
    Desc = _desc_class(lib)
    d = Desc()
    d.struct_size, d.abi_version = ctypes.sizeof(Desc), lib.optistate_kf_abi_version()
    d.dtype, d.algo, d.cov_model, d.phases = 0, 0, 0, 7
    d.n_traj, d.n_steps, d.n_streams = 4, 10, 4
    d.dt, d.mass, d.gravity = 0.01, 8.8, -9.81
    d.inertia = (ctypes.c_double * 3)(0.055, 0.060, 0.105)
    fake = ctypes.c_void_p(0x1000)  # never dereferenced: validation only
    for n in ("imu", "p", "dp", "contact", "f", "x0", "Q", "R"):
        setattr(d, n, fake)
    d.q_kind, d.r_kind, d.p0_kind = 1, 1, 0
    return d


def test_descriptor_validation_and_algo_resolution(lib):
    lib.optistate_kf_strerror.restype = ctypes.c_char_p
    d = _valid_desc(lib)
    assert lib.optistate_kf_resolve_algo(ctypes.byref(d)) == 2  # diagonal noise -> SEQUENTIAL
    d.q_kind = 3
    assert lib.optistate_kf_resolve_algo(ctypes.byref(d)) == 1  # dense Q -> JOINT
    d.algo = 2
    assert lib.optistate_kf_resolve_algo(ctypes.byref(d)) == -5  # SEQUENTIAL cannot take dense noise
    assert b"not supported" in lib.optistate_kf_strerror(-5)
    d = _valid_desc(lib)
    d.cov_model = 1
    d.body_ref = ctypes.c_void_p(0x1000)
    assert lib.optistate_kf_resolve_algo(ctypes.byref(d)) == 2  # predict_mpc covariance with diagonal noise -> SEQUENTIAL too
    d.body_ref = None
    assert lib.optistate_kf_resolve_algo(ctypes.byref(d)) == -1  # ... but it needs the reference body angles
    d = _valid_desc(lib)
    d.K_final = ctypes.c_void_p(0x1000)
    assert lib.optistate_kf_resolve_algo(ctypes.byref(d)) == 1  # the gain matrix only exists in the joint form
    d = _valid_desc(lib)
    d.struct_size -= 8
    assert lib.optistate_kf_batch(ctypes.byref(d), None) == -2
    d = _valid_desc(lib)
    d.dtype = 7
    assert lib.optistate_kf_batch(ctypes.byref(d), None) == -3
    assert lib.optistate_kf_batch_f32(ctypes.byref(_valid_desc(lib)), None) == -3  # f64 descriptor through the f32 entry
    d = _valid_desc(lib)
    d.n_streams = 0
    assert lib.optistate_kf_batch(ctypes.byref(d), None) == -4
    d = _valid_desc(lib)
    d.f = None
    assert lib.optistate_kf_batch(ctypes.byref(d), None) == -1
    assert lib.optistate_kf_batch(None, None) == -1
    d = _valid_desc(lib)
    d.n_traj = 0  # nothing to do: succeeds without touching the device
    assert lib.optistate_kf_batch(ctypes.byref(d), None) == 0
    # fused summary all-gather: the row stride must cover the local block, peers must be given
    d = _valid_desc(lib)
    d.summary = ctypes.c_void_p(0x1000)
    d.summary_ld = 3
    assert lib.optistate_kf_resolve_algo(ctypes.byref(d)) == -4
    d.summary_ld, d.n_summary_peers = 8, 8
    assert lib.optistate_kf_resolve_algo(ctypes.byref(d)) == -4
    d.n_summary_peers = 1
    assert lib.optistate_kf_resolve_algo(ctypes.byref(d)) == -1  # peer pointer missing
    d.summary_peers[0] = 0x2000
    assert lib.optistate_kf_resolve_algo(ctypes.byref(d)) == 2


def test_workspace_query(lib):
    d = _valid_desc(lib)
    n = ctypes.c_size_t(123)
    assert lib.optistate_kf_workspace_bytes(ctypes.byref(d), ctypes.byref(n)) == 0 and n.value == 0  # S % 128 != 0: direct kernel
    d.n_streams, d.n_traj = 256, 1024
    assert lib.optistate_kf_workspace_bytes(ctypes.byref(d), ctypes.byref(n)) == 0
    assert n.value >= 10 * 10 * 256 * 8 + 256 * 4


def test_extension_loads_at_abi_5_and_refuses_cpu_tensors():
    from optistate_b200 import _native as nv

    ext = nv.ext()
    assert ext.abi_version() == nv.ABI_VERSION == 5 and ext.MAX_PEERS == 7 and ext.launch_count() >= 0
    cfg = dict(dtype=nv.F64, n_traj=1, n_steps=1, n_streams=1)
    consts = dict(dt=0.01, mass=8.8, inertia0=0.05, inertia1=0.06, inertia2=0.1, gravity=-9.81)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        ext.kf_batch(cfg, consts, {"x0": torch.zeros(12, dtype=torch.float64)})


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_product_path_fails_loudly_without_a_gpu():
    from optistate_b200 import Kalman_Filter, kf_batch
    from optistate_b200.synth import make_streams

    st = make_streams([0], 4)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        kf_batch(st["imu"], st["p"], st["dp"], st["contact"], st["f"])
    kf = Kalman_Filter()  # construction is host-only, like the reference's
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        kf.update()
    from optistate_b200 import mpc_forces
    from optistate_b200.synth import make_mpc_problems

    with pytest.raises(RuntimeError, match="no CPU fallback"):
        mpc_forces(*make_mpc_problems(4))


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "optistate_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f
                assert "kf_oracle" not in src and "ref_shim" not in src, f


def test_drop_in_class_surface_matches_reference_attributes():
    from optistate_b200 import Kalman_Filter
    from optistate_b200.settings import INITIAL_PARAMS

    kf = Kalman_Filter()
    for name in ("x", "z", "H", "P", "Q", "R", "P_trace", "F", "B", "g", "dt", "m", "inertia_rot", "x_model", "K", "K_gain", "F_d"):
        assert hasattr(kf, name), name
    for name in ("get_odom", "set_measurements", "predict", "predict_mpc", "update", "estimate_state_mpc", "rotation_matrix_body_world", "skew"):
        assert callable(getattr(kf, name)), name
    assert kf.x is INITIAL_PARAMS.STARTING_STATE and kf.P is INITIAL_PARAMS.Q  # the reference's aliasing (SURVEY 8b)
    assert kf.H.shape == (10, 12) and kf.H.sum() == 10 and kf.H[3, 5] == 1
    assert kf.x.shape == (12, 1) and kf.z.shape == (10, 1)
    kf.set_measurements(np.arange(6.0).reshape(6, 1), np.array([10.0, 11, 12, 13]).reshape(4, 1))
    assert kf.z.reshape(-1).tolist() == [0, 1, 2, 10, 3, 4, 5, 11, 12, 13]
    R = kf.rotation_matrix_body_world(0.1, -0.2, 0.3)
    assert np.allclose(R @ R.T, np.eye(3), atol=1e-15)
    if not torch.cuda.is_available():  # without explicit forces predict_mpc solves the MPC on the device: no CPU solver
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            kf.predict_mpc(np.zeros((12, 1)), np.zeros((12, 1)), np.ones((4, 1)))
