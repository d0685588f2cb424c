"""ctypes binding of tests/host_emul/libacoc_vjp_emul.so (TEST-ONLY host replay of the kernels of acoc_result_vjp)."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libacoc_vjp_emul.so")
_lib = None
DEFAULT_PARAMS = np.array([0.1716, 2.395, 3.256, 12.0, 9.81, 0.61, 1.2, 0.24, 1e-3])


def build(force=False):
    srcs = [os.path.join(_HERE, "vjp_emul.cpp")] + [os.path.join(_HERE, "..", "..", "aircraftoptimalcontrol_b200", "csrc", f)
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
    return None if a is None else np.ascontiguousarray(a, dtype=np.float64)


def result_vjp(xx, uu, gx, gu, Q, R, QT, xref=None, uref=None, param=None, params=DEFAULT_PARAMS):
    """Host replay of acoc_result_vjp for results xx (N,6,TT) / uu (N,2,TT) (xx[:, :, 0] = the exact x0) and upstream gradients gx / gu.
    References: xref (N,6,TT) / uref (N,2,TT), or param = dict(tt, zs, vs (or None), zf (N), vx (N), xc (6), uc (2)) as handed to
    acoc_set_refs_generated.  Returns dict(xref, uref, x0, zf, vx, n_indef) (zf / vx None without param)."""
    xx, uu, gx, gu = _c(xx), _c(uu), _c(gx), _c(gu)
    N, _, TT = xx.shape
    xb, ub, x0b = np.zeros((N, 6, TT)), np.zeros((N, 2, TT)), np.zeros((N, 6))
    zb, vb, ni = np.zeros(N), np.zeros(N), np.zeros(N, dtype=np.int32)
    pr = param or {}
    lib().emul_vjp(C.c_int(N), C.c_int(TT), _p(_c(params)), _p(_c(Q)), _p(_c(R)), _p(_c(QT)), _p(xx), _p(uu), _p(_c(xref)), _p(_c(uref)),
                   _p(_c(pr.get("tt"))), _p(_c(pr.get("zs"))), _p(_c(pr.get("vs"))), _p(_c(pr.get("zf"))), _p(_c(pr.get("vx"))),
                   _p(_c(pr.get("xc"))), _p(_c(pr.get("uc"))), _p(gx), _p(gu), _p(xb), _p(ub), _p(x0b), _p(zb), _p(vb), _p(ni))
    return dict(xref=xb, uref=ub, x0=x0b, zf=zb if param else None, vx=vb if param else None, n_indef=ni)
