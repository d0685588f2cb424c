"""ctypes binding of tests/host_emul/libacoc_track_mc_emul.so (TEST-ONLY host replay of the dispersion kernels' per-sample and
reduction code).  The library includes the tracking replay, so track_many runs on the same build."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from .track_emul import DEFAULT_PARAMS, _c, _p

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libacoc_track_mc_emul.so")
_lib = None


def build(force=False):
    srcs = [os.path.join(_HERE, f) for f in ("track_mc_emul.cpp", "track_emul.cpp")] + [
        os.path.join(_HERE, "..", "..", "aircraftoptimalcontrol_b200", "csrc", f) for f in ("acoc_math.cuh", "acoc_kernels.cuh")]
    if force or not os.path.exists(_SO) or any(os.path.getmtime(_SO) < os.path.getmtime(s) for s in srcs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-Wno-unknown-pragmas",
                               "-o", _SO, srcs[0]])
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_SO)
    return _lib


def track_mc(xx_opt, uu_opt, delta, Q, R, QT, tol=None, params=DEFAULT_PARAMS, state_f64=False):
    """Host replay of acoc_lqr_tracking_mc on nominals (N,6,TT)/(N,2,TT), delta (M,6) (shared) or (N,M,6), tol (6,) or None.
    Returns dict(err_max, err_final (N,M,6), worst_max, mean_final (N,6), n_within (N; 0 without tol), n_reg (N))."""
    xo = _c(xx_opt)
    N, _, TT = xo.shape
    d = _c(delta)
    shared = d.ndim == 2
    M = d.shape[0] if shared else d.shape[1]
    em, ef = np.zeros((N, M, 6)), np.zeros((N, M, 6))
    wm, mf, nw, nr = np.zeros((N, 6)), np.zeros((N, 6)), np.zeros(N, dtype=np.int32), np.zeros(N, dtype=np.int32)
    lib().emul_track_mc(C.c_int(N), C.c_int(M), C.c_int(TT), _p(_c(params)), C.c_int(int(state_f64)), _p(_c(Q)), _p(_c(R)), _p(_c(QT)),
                        _p(xo), _p(_c(uu_opt)), _p(d), C.c_int(int(shared)), _p(None if tol is None else _c(tol)), _p(em), _p(ef), _p(wm),
                        _p(mf), _p(nw), _p(nr))
    return dict(err_max=em, err_final=ef, worst_max=wm, mean_final=mf, n_within=nw, n_reg=nr)
