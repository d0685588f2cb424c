"""ctypes binding of tests/host_emul/libacoc_track_emul.so (TEST-ONLY host replay of the tracking kernels' per-instance code)."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libacoc_track_emul.so")
_lib = None
DEFAULT_PARAMS = np.array([0.1716, 2.395, 3.256, 12.0, 9.81, 0.61, 1.2, 0.24, 1e-3])


def build(force=False):
    srcs = [os.path.join(_HERE, "track_emul.cpp")] + [os.path.join(_HERE, "..", "..", "aircraftoptimalcontrol_b200", "csrc", f)
                                                     for f in ("acoc_math.cuh", "acoc_kernels.cuh")]
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


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _c(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def track_many(xx_opt, uu_opt, delta, Q, R, QT, params=DEFAULT_PARAMS, state_f64=False):
    """Host replay of acoc_lqr_tracking_many / acoc_track on nominals (N,6,TT)/(N,2,TT), delta (N,6).
    Returns dict(xx_reg, uu_reg, K (N,2,6,TT), err_max (N,6), err_final (N,6), n_reg (N))."""
    xo = _c(xx_opt)
    N, _, TT = xo.shape
    xr, ur, K = np.zeros((N, 6, TT)), np.zeros((N, 2, TT)), np.zeros((N, 2, 6, TT))
    em, ef, nr = np.zeros((N, 6)), np.zeros((N, 6)), np.zeros(N, dtype=np.int32)
    lib().emul_track_many(C.c_int(N), C.c_int(TT), _p(_c(params)), C.c_int(int(state_f64)), _p(_c(Q)), _p(_c(R)), _p(_c(QT)), _p(xo),
                          _p(_c(uu_opt)), _p(_c(delta)), _p(xr), _p(ur), _p(K), _p(em), _p(ef), _p(nr))
    return dict(xx_reg=xr, uu_reg=ur, K=K, err_max=em, err_final=ef, n_reg=nr)
