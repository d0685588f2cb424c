"""Drop-in for the reference's lqr_tracking.py:245-283, with the module globals it reads (dyn, ns, ni, QQt, RRt,
QQT -- lqr_tracking.py:254-255, :269, :276, defined only under __main__ at :322-328) turned into keyword
arguments that default to the __main__ values.  `lqr_tracking_batch` tracks from many perturbed initial states
with ONE shared LQ solve (the gains depend only on the nominal trajectory).
"""
from __future__ import annotations

import numpy as np

from . import _lib as L
from .aircraft_simplified import Dynamics
from .optcon import ltv_LQR  # noqa: F401  (the reference module also exposes ltv_LQR, lqr_tracking.py:6)


def default_weights():
    """Weights of lqr_tracking.py:324-328."""
    QQt = np.eye(6) * 0.01
    QQt[1, 1] = 10
    QQt[0, 0] = 10
    RRt = np.eye(2) * 1e-5
    return QQt, RRt, QQt.copy()


def lqr_tracking_batch(xx_opt, uu_opt, delta, dyn=None, QQt=None, RRt=None, QQT=None, return_gains=False):
    """delta (N,6) perturbations of the initial state -> xx_reg (N,6,TT), uu_reg (N,2,TT) [, KK (2,6,TT)]."""
    dyn = dyn or Dynamics()
    dQ, dR, dQT = default_weights()
    Q = L.f64(dQ if QQt is None else QQt, (6, 6), "QQt")
    R = L.f64(dR if RRt is None else RRt, (2, 2), "RRt")
    QT = L.f64(dQT if QQT is None else QQT, (6, 6), "QQT")
    xo, uo = L.f64(xx_opt), L.f64(uu_opt)
    TT = xo.shape[1]
    if xo.shape != (6, TT) or uo.shape != (2, TT):
        raise ValueError("xx_opt must be (6,TT) and uu_opt (2,TT)")
    d = L.f64(np.atleast_2d(delta))
    N = d.shape[0]
    if d.shape != (N, 6):
        raise ValueError("delta must be (N,6)")
    xr, ur, K = np.empty((N, 6, TT)), np.empty((N, 2, TT)), np.zeros((TT, 2, 6))
    p = dyn.params
    L.check(L.lib().acoc_lqr_tracking(dyn.device, N, TT, L.ptr(p), int(dyn.state == "f64"), L.ptr(Q), L.ptr(R), L.ptr(QT),
                                      L.ptr(xo), L.ptr(uo), L.ptr(d), L.ptr(xr), L.ptr(ur), L.ptr(K)))
    if return_gains:
        return xr, ur, np.moveaxis(K, 0, 2).copy()
    return xr, ur


def lqr_tracking_many(xx_opt, uu_opt, delta, dyn=None, QQt=None, RRt=None, QQT=None, return_gains=False):
    """One call of the reference's lqr_tracking per nominal: xx_opt (N,6,TT), uu_opt (N,2,TT), delta (N,6) (or (6,), broadcast) ->
    xx_reg (N,6,TT), uu_reg (N,2,TT) [, KK (N,2,6,TT)].  Each nominal gets its own gains; the kernels are those of
    BatchedNewton.track (acoc_lqr_tracking_many).  The weights must be symmetric."""
    dyn = dyn or Dynamics()
    dQ, dR, dQT = default_weights()
    Q = L.f64(dQ if QQt is None else QQt, (6, 6), "QQt")
    R = L.f64(dR if RRt is None else RRt, (2, 2), "RRt")
    QT = L.f64(dQT if QQT is None else QQT, (6, 6), "QQT")
    xo, uo = L.f64(xx_opt), L.f64(uu_opt)
    if xo.ndim != 3 or xo.shape[1] != 6 or xo.shape[2] < 3:
        raise ValueError("xx_opt must be (N,6,TT) with TT >= 3, got %s" % (xo.shape,))
    N, _, TT = xo.shape
    if uo.shape != (N, 2, TT):
        raise ValueError("uu_opt has shape %s, expected %s" % (uo.shape, (N, 2, TT)))
    d = np.asarray(delta, dtype=np.float64)
    if d.shape == (6,):
        d = np.broadcast_to(d, (N, 6))
    d = L.f64(d, (N, 6), "delta")
    xr, ur = np.empty((N, 6, TT)), np.empty((N, 2, TT))
    K = np.empty((N, 2, 6, TT)) if return_gains else None
    L.check(L.lib().acoc_lqr_tracking_many(dyn.device, N, TT, L.ptr(dyn.params), int(dyn.state == "f64"), L.ptr(Q), L.ptr(R), L.ptr(QT),
                                           L.ptr(xo), L.ptr(uo), L.ptr(d), L.ptr(xr), L.ptr(ur), L.ptr(K)))
    if return_gains:
        return xr, ur, K
    return xr, ur


def lqr_tracking(xx_opt, uu_opt, tt, dyn=None, QQt=None, RRt=None, QQT=None):
    """(xx_reg (6,TT), uu_reg (2,TT)) for the shipped perturbation 0.1*ones(6) (lqr_tracking.py:259)."""
    TT = np.asarray(tt).shape[0]
    if np.asarray(xx_opt).shape[1] != TT:
        raise ValueError("tt and xx_opt disagree on the horizon")
    xr, ur = lqr_tracking_batch(xx_opt, uu_opt, np.ones((1, 6)) * 0.1, dyn, QQt, RRt, QQT)
    return xr[0], ur[0]
