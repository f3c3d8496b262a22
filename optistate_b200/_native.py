"""Loads the in-tree native code.  There is no fallback: if the CUDA library or the PyTorch extension is
missing or does not load, importing the product path raises."""
from __future__ import annotations

import importlib.machinery
import importlib.util
import os

from . import _build

# mirrors of the enums in include/optistate_kf.h
F64, F32 = 0, 1
ALGO_AUTO, ALGO_JOINT, ALGO_SEQUENTIAL = 0, 1, 2
COV_PREDICT, COV_MPC = 0, 1
PHASE_MEASURE, PHASE_PREDICT, PHASE_UPDATE, PHASE_ALL = 1, 2, 4, 7
MAT_NONE, MAT_DIAG, MAT_DIAG_PER, MAT_DENSE, MAT_DENSE_PER = 0, 1, 2, 3, 4
ST_NOT_PD, ST_NONFINITE, ST_ALL_SWING, ST_ASYMMETRIC, ST_SINGULAR, ST_SMOOTH_NOT_PD = 1, 2, 4, 8, 16, 32
FLAG_P0_DECOUPLED, FLAG_FULL_COVARIANCE, FLAG_SCALAR_FP32 = 1, 2, 4
ABI_VERSION = 5
SUMMARY_ROWS = 52

_ext = None


def ext():
    """The PyTorch C++ extension module (optistate_b200/_lib/_optistate_torch.so)."""
    global _ext
    if _ext is None:
        import torch  # noqa: F401  (libtorch must be loaded before the extension)

        if not (os.path.exists(_build.KF_LIB) and os.path.exists(_build.EXT_LIB)):
            raise ImportError(
                "optistate_b200: native libraries not built (expected %s and %s); run "
                "`python -m optistate_b200._build` or __graft_entry__.build(). There is no CPU fallback."
                % (_build.KF_LIB, _build.EXT_LIB)
            )
        loader = importlib.machinery.ExtensionFileLoader(_build.EXT_NAME, _build.EXT_LIB)
        spec = importlib.util.spec_from_loader(_build.EXT_NAME, loader)
        mod = importlib.util.module_from_spec(spec)
        loader.exec_module(mod)
        if mod.SUMMARY_ROWS != SUMMARY_ROWS:
            raise ImportError("optistate_b200: stale native build (summary layout mismatch); rebuild")
        _ext = mod
    return _ext


def require_cuda():
    import torch

    if not torch.cuda.is_available():
        raise RuntimeError("optistate_b200 needs a CUDA device (sm_100a); there is no CPU fallback")


def check(rc: int, what: str):
    if rc != 0:
        raise RuntimeError(f"{what} failed: {ext().strerror(rc)} (code {rc})")
