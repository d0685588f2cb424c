"""ctypes binding of oracle/libacoc_oracle.so (the CPU restatement).  TEST INFRASTRUCTURE ONLY.

Importable from tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs; never from the
product package.  All functions take / return numpy arrays in the REFERENCE's layouts
((6,TT)/(2,TT) trajectories, (n,n,TT) matrix stacks) so that tests read like calls into the reference.
"""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libacoc_oracle.so")
_lib = None

DEFAULT_PARAMS = np.array([0.1716, 2.395, 3.256, 12.0, 9.81, 0.61, 1.2, 0.24, 1e-3])  # aircraft_simplified.py:108-118


def build(force: bool = False) -> str:
    """Compile libacoc_oracle.so beside its source when it is missing or older than the source; in a read-only tree it is compiled
    into a temporary directory (removed at exit) and loaded from there."""
    global _SO
    src = os.path.join(_HERE, "acoc_oracle.c")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        if not os.access(_HERE, os.W_OK):
            tmp = tempfile.mkdtemp(prefix="acoc_oracle_")
            atexit.register(shutil.rmtree, tmp, True)
            _SO = os.path.join(tmp, "libacoc_oracle.so")
        subprocess.check_call(["make", "-C", _HERE, "-s", "-B", "OUT=" + _SO], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    return _SO


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            build()
        _lib = C.CDLL(_SO)
        _lib.orc_stagecost.restype = C.c_double
        _lib.orc_termcost.restype = C.c_double
        _lib.orc_traj_cost.restype = C.c_double
        _lib.orc_rollout.restype = C.c_double
        _lib.orc_armijo.restype = C.c_double
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _c(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None:
        assert a.shape == tuple(shape), (a.shape, shape)
    return a


def max_threads() -> int:
    return int(lib().orc_max_threads())


def step(x, u, lmbd=None, params=DEFAULT_PARAMS, quant_f32=True):
    """Dynamics.step (aircraft_simplified.py:263): returns (xxp, fx, fu, fxx, fuu, fux) in the reference's shapes."""
    x, u, prm = _c(x).ravel(), _c(u).ravel(), _c(params)
    xxp, A, B = np.zeros(6), np.zeros((6, 6)), np.zeros((6, 2))
    if lmbd is None:
        fxx, fux, lam = np.zeros((6, 6, 6)), np.zeros((2, 6, 6)), None
        fuu = np.zeros((2, 2, 6))
    else:
        fxx, fux, lam = np.zeros((6, 6)), np.zeros((2, 6)), _c(lmbd).ravel()
        fuu = np.zeros((2, 2))
    lib().orc_step(_p(prm), _p(x), _p(u), _p(lam), C.c_int(int(quant_f32)), _p(xxp), _p(A), _p(B), _p(fxx), _p(fux))
    return xxp, A.T.copy(), B.T.copy(), fxx, fuu, fux


def stagecost(Q, R, x, u, xr, ur):
    Q, R = _c(Q, (6, 6)), _c(R, (2, 2))
    lx, lu = np.zeros(6), np.zeros(2)
    ll = lib().orc_stagecost(_p(Q), _p(R), _p(_c(x).ravel()), _p(_c(u).ravel()), _p(_c(xr).ravel()), _p(_c(ur).ravel()), _p(lx), _p(lu))
    return ll, lx, lu


def termcost(QT, x, xr):
    QT = _c(QT, (6, 6))
    lTx = np.zeros(6)
    ll = lib().orc_termcost(_p(QT), _p(_c(x).ravel()), _p(_c(xr).ravel()), _p(lTx))
    return ll, lTx


def traj_cost(Q, R, QT, xx, uu, xr, ur):
    TT = xx.shape[1]
    return lib().orc_traj_cost(_p(_c(Q)), _p(_c(R)), _p(_c(QT)), C.c_int(TT), _p(_c(xx)), _p(_c(uu)), _p(_c(xr)), _p(_c(ur)))


def _tm(M, TT):
    """(a,b,TT) or (a,b) reference stack -> time-major contiguous (TT,a,b)."""
    M = np.asarray(M, dtype=np.float64)
    if M.ndim == 2:
        M = np.repeat(M[:, :, None], TT, axis=2)
    return np.ascontiguousarray(np.moveaxis(M, 2, 0))


def ltv_lqr(AA, BB, QQ, RR, SS, QQf, TT, x0, qq=None, rr=None, qqf=None, return_nreg=False):
    """ltv_LQR (optcon.py:533) with the reference's argument layout; returns (KK, PP, xxout, uuout)."""
    A, B, Q, R, S = _tm(AA, TT), _tm(BB, TT), _tm(QQ, TT), _tm(RR, TT), _tm(SS, TT)
    aug = (qq is not None) or (rr is not None) or (qqf is not None)
    n = 7 if aug else 6
    q = r = qf = None
    if aug:
        q = np.zeros((TT, 6)) if qq is None else np.ascontiguousarray(np.broadcast_to(np.asarray(qq, float).reshape(6, -1), (6, TT)).T)
        r = np.zeros((TT, 2)) if rr is None else np.ascontiguousarray(np.broadcast_to(np.asarray(rr, float).reshape(2, -1), (2, TT)).T)
        qf = np.zeros(6) if qqf is None else _c(qqf).ravel()
    K, P = np.zeros((TT, 2, n)), np.zeros((TT, n, n))
    xo, uo = np.zeros((TT, 6)), np.zeros((TT, 2))
    nreg = C.c_int(0)
    rc = lib().orc_ltv_lqr(C.c_int(TT), _p(A), _p(B), _p(Q), _p(R), _p(S), _p(_c(QQf, (6, 6))), _p(_c(x0).ravel()),
                           _p(q), _p(r), _p(qf), _p(K), _p(P), _p(xo), _p(uo), C.byref(nreg))
    assert rc == 0
    out = (np.moveaxis(K, 0, 2).copy(), np.moveaxis(P, 0, 2).copy(), xo.T.copy(), uo.T.copy())
    return out + (nreg.value,) if return_nreg else out


def rollout(x0, uu, du, s, params=DEFAULT_PARAMS, quant_f32=True, cost=None, xr=None, ur=None):
    """get_update (optcon.py:176); with cost=(Q,R,QT) also returns the Armijo candidate cost (optcon.py:257-264)."""
    TT = uu.shape[1]
    xo, uo = np.zeros((6, TT)), np.zeros((2, TT))
    if cost is not None:
        Q, R, QT = (_c(m) for m in cost)
        J = lib().orc_rollout(_p(_c(params)), C.c_int(int(quant_f32)), C.c_int(TT), _p(_c(x0).ravel()), _p(_c(uu)), _p(_c(du)),
                              C.c_double(s), _p(Q), _p(R), _p(QT), _p(_c(xr)), _p(_c(ur)), _p(xo), _p(uo))
        return xo, uo, J
    lib().orc_rollout(_p(_c(params)), C.c_int(int(quant_f32)), C.c_int(TT), _p(_c(x0).ravel()), _p(_c(uu)), _p(_c(du)),
                      C.c_double(s), None, None, None, None, None, _p(xo), _p(uo))
    return xo, uo


def armijo(x0, uu, du, Q, R, QT, xr, ur, JP, descent, stepsize_0=1.0, cc=0.5, beta=0.7, maxiters=10,
           params=DEFAULT_PARAMS, quant_f32=True):
    TT = uu.shape[1]
    costs = np.full(maxiters, np.nan)
    ntried, acc = C.c_int(0), C.c_int(0)
    s = lib().orc_armijo(_p(_c(params)), C.c_int(int(quant_f32)), C.c_int(TT), _p(_c(x0).ravel()), _p(_c(uu)), _p(_c(du)),
                         _p(_c(Q)), _p(_c(R)), _p(_c(QT)), _p(_c(xr)), _p(_c(ur)), C.c_double(JP), C.c_double(descent),
                         C.c_double(stepsize_0), C.c_double(cc), C.c_double(beta), C.c_int(maxiters), _p(costs),
                         C.byref(ntried), C.byref(acc))
    return s, costs, ntried.value, bool(acc.value)


def newton(xx_ref, uu_ref, xx_init, uu_init, Q, R, QT, params=DEFAULT_PARAMS, quant_f32=True, max_iters=200,
           stepsize_0=1.0, cc=0.5, beta=0.7, armijo_maxiters=10, exact_after=8, term_cond=-1e-6, n_iters_cap=0):
    """NewtonMethod.optimize (optcon.py:341) for one instance; returns a history dict like oracle.pyref.run_newton."""
    TT = xx_ref.shape[1]
    hJ, hD, hS = np.zeros(max_iters), np.zeros(max_iters), np.zeros(max_iters)
    hN = np.zeros(max_iters, dtype=np.int32)
    iters, nreg = C.c_int(0), C.c_int(0)
    xs, us, xl, ul = np.zeros((6, TT)), np.zeros((2, TT)), np.zeros((6, TT)), np.zeros((2, TT))
    rc = lib().orc_newton(_p(_c(params)), C.c_int(int(quant_f32)), C.c_int(TT), _p(_c(Q)), _p(_c(R)), _p(_c(QT)),
                          _p(_c(xx_ref)), _p(_c(uu_ref)), _p(_c(xx_init)), _p(_c(uu_init)), C.c_int(max_iters),
                          C.c_double(stepsize_0), C.c_double(cc), C.c_double(beta), C.c_int(armijo_maxiters),
                          C.c_int(exact_after), C.c_double(term_cond), C.c_int(n_iters_cap),
                          _p(hJ), _p(hD), _p(hS), _p(hN), C.byref(iters), _p(xs), _p(us), _p(xl), _p(ul), C.byref(nreg))
    assert rc == 0
    k = iters.value
    return dict(JJ=hJ[:k].copy(), descent=hD[:k].copy(), stepsize=hS[:k].copy(), n_armijo=hN[:k].copy(), iters=k,
                xx_star=xs, uu_star=us, xx_last=xl, uu_last=ul, n_regularized=nreg.value)


def newton_batch(xx_ref, uu_ref, xx_init, uu_init, Q, R, QT, params=DEFAULT_PARAMS, quant_f32=True, max_iters=200,
                 stepsize_0=1.0, cc=0.5, beta=0.7, armijo_maxiters=10, exact_after=8, term_cond=-1e-6, n_iters_cap=0,
                 n_threads=0):
    """Batch of independent instances; xx_ref (N,6,TT) or (6,TT) shared, xx_init (N,6,TT)."""
    xx_init, uu_init = _c(xx_init), _c(uu_init)
    N, _, TT = xx_init.shape
    xr, ur = _c(xx_ref), _c(uu_ref)
    sx = 6 * TT if xr.ndim == 3 else 0
    su = 2 * TT if ur.ndim == 3 else 0
    hJ, hD, hS = (np.zeros((N, max_iters)) for _ in range(3))
    hN = np.zeros((N, max_iters), dtype=np.int32)
    iters = np.zeros(N, dtype=np.int32)
    xs, us = np.zeros((N, 6, TT)), np.zeros((N, 2, TT))
    nt = n_threads if n_threads > 0 else max_threads()
    rc = lib().orc_newton_batch(C.c_int(N), C.c_int(nt), _p(_c(params)), C.c_int(int(quant_f32)), C.c_int(TT),
                                _p(_c(Q)), _p(_c(R)), _p(_c(QT)), _p(xr), C.c_long(sx), _p(ur), C.c_long(su),
                                _p(xx_init), _p(uu_init), C.c_int(max_iters), C.c_double(stepsize_0), C.c_double(cc),
                                C.c_double(beta), C.c_int(armijo_maxiters), C.c_int(exact_after), C.c_double(term_cond),
                                C.c_int(n_iters_cap), _p(hJ), _p(hD), _p(hS), _p(hN), _p(iters), _p(xs), _p(us))
    assert rc == 0
    return dict(JJ=hJ, descent=hD, stepsize=hS, n_armijo=hN, iters=iters, xx_star=xs, uu_star=us, threads=nt)


def gradient(xx_ref, uu_ref, xx_init, uu_init, Q, R, QT, params=DEFAULT_PARAMS, quant_f32=True, max_iters=200,
             stepsize_0=1e-2, cc=0.5, beta=0.7, armijo_maxiters=20, term_cond=1e-6):
    """GradientMethod.optimize (optcon.py:27) with the repaired line-search call, one instance; history dict like
    oracle.pyref.run_gradient (descent = sum |deltau|^2, positive, as the reference stores it)."""
    TT = xx_ref.shape[1]
    hJ, hD, hS = np.zeros(max_iters), np.zeros(max_iters), np.zeros(max_iters)
    hN = np.zeros(max_iters, dtype=np.int32)
    iters = C.c_int(0)
    xs, us, xl, ul, du0 = np.zeros((6, TT)), np.zeros((2, TT)), np.zeros((6, TT)), np.zeros((2, TT)), np.zeros((2, TT))
    rc = lib().orc_gradient(_p(_c(params)), C.c_int(int(quant_f32)), C.c_int(TT), _p(_c(Q)), _p(_c(R)), _p(_c(QT)),
                            _p(_c(xx_ref)), _p(_c(uu_ref)), _p(_c(xx_init)), _p(_c(uu_init)), C.c_int(max_iters),
                            C.c_double(stepsize_0), C.c_double(cc), C.c_double(beta), C.c_int(armijo_maxiters), C.c_double(term_cond),
                            _p(hJ), _p(hD), _p(hS), _p(hN), C.byref(iters), _p(xs), _p(us), _p(xl), _p(ul), _p(du0))
    assert rc == 0
    k = iters.value
    return dict(JJ=hJ[:k].copy(), descent=hD[:k].copy(), stepsize=hS[:k].copy(), n_armijo=hN[:k].copy(), iters=k,
                xx_star=xs, uu_star=us, xx_last=xl, uu_last=ul, deltau_first=du0)


def gradient_batch(xx_ref, uu_ref, xx_init, uu_init, Q, R, QT, params=DEFAULT_PARAMS, quant_f32=True, max_iters=200,
                   stepsize_0=1e-2, cc=0.5, beta=0.7, armijo_maxiters=20, term_cond=1e-6, n_threads=0):
    xx_init, uu_init = _c(xx_init), _c(uu_init)
    N, _, TT = xx_init.shape
    xr, ur = _c(xx_ref), _c(uu_ref)
    sx = 6 * TT if xr.ndim == 3 else 0
    su = 2 * TT if ur.ndim == 3 else 0
    hJ, hD, hS = (np.zeros((N, max_iters)) for _ in range(3))
    hN = np.zeros((N, max_iters), dtype=np.int32)
    iters = np.zeros(N, dtype=np.int32)
    xs, us = np.zeros((N, 6, TT)), np.zeros((N, 2, TT))
    nt = n_threads if n_threads > 0 else max_threads()
    rc = lib().orc_gradient_batch(C.c_int(N), C.c_int(nt), _p(_c(params)), C.c_int(int(quant_f32)), C.c_int(TT),
                                  _p(_c(Q)), _p(_c(R)), _p(_c(QT)), _p(xr), C.c_long(sx), _p(ur), C.c_long(su),
                                  _p(xx_init), _p(uu_init), C.c_int(max_iters), C.c_double(stepsize_0), C.c_double(cc),
                                  C.c_double(beta), C.c_int(armijo_maxiters), C.c_double(term_cond),
                                  _p(hJ), _p(hD), _p(hS), _p(hN), _p(iters), _p(xs), _p(us))
    assert rc == 0
    return dict(JJ=hJ, descent=hD, stepsize=hS, n_armijo=hN, iters=iters, xx_star=xs, uu_star=us, threads=nt)


def lqr_tracking(xx_opt, uu_opt, Q, R, QT, delta, params=DEFAULT_PARAMS, quant_f32=True, n_threads=0):
    """lqr_tracking (lqr_tracking.py:245) for N perturbations delta (N,6); returns (xx_reg (N,6,TT), uu_reg (N,2,TT), K (2,6,TT))."""
    TT = xx_opt.shape[1]
    delta = _c(np.atleast_2d(delta))
    N = delta.shape[0]
    xr, ur, K = np.zeros((N, 6, TT)), np.zeros((N, 2, TT)), np.zeros((TT, 2, 6))
    nt = n_threads if n_threads > 0 else max_threads()
    rc = lib().orc_lqr_tracking(_p(_c(params)), C.c_int(int(quant_f32)), C.c_int(TT), _p(_c(Q)), _p(_c(R)), _p(_c(QT)),
                                _p(_c(xx_opt)), _p(_c(uu_opt)), C.c_int(N), _p(delta), C.c_int(nt), _p(xr), _p(ur), _p(K))
    assert rc == 0
    return xr, ur, np.moveaxis(K, 0, 2).copy()


def initial_trajectory(xx_ref, params=DEFAULT_PARAMS, quant_f32=True, kp=5.0, kt=2.5):
    TT = xx_ref.shape[1]
    xx, uu = np.zeros((6, TT)), np.zeros((2, TT))
    lib().orc_initial_trajectory(_p(_c(params)), C.c_int(int(quant_f32)), C.c_int(TT), _p(_c(xx_ref)), C.c_double(kp),
                                 C.c_double(kt), _p(xx), _p(uu))
    return xx, uu
