"""Drop-in for the reference's lqr_tracking.py:245-283, with the module globals it reads (dyn, ns, ni, QQt, RRt,
QQT -- lqr_tracking.py:254-255, :269, :276, defined only under __main__ at :322-328) turned into keyword
arguments that default to the __main__ values.  `lqr_tracking_batch` tracks from many perturbed initial states
with ONE shared LQ solve (the gains depend only on the nominal trajectory).
"""
from __future__ import annotations

import ctypes as C

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


def mc_layout(shape, N):
    """(shared, M) of a dispersion study's perturbations of `shape`: (M,6) shared by all N instances or (N,M,6)."""
    shape = tuple(shape)
    if len(shape) == 2 and shape[1] == 6:
        shared, M = True, shape[0]
    elif len(shape) == 3 and shape[0] == N and shape[2] == 6:
        shared, M = False, shape[1]
    else:
        raise ValueError("delta has shape %s, expected (M,6) or %s" % (shape, (N, "M", 6)))
    if M < 1:
        raise ValueError("delta holds no sample (M = 0)")
    return shared, M


def mc_deltas(delta, N):
    """Perturbations of a dispersion study: (M,6) shared by all N instances or (N,M,6) -> (contiguous float64 array, shared, M)."""
    d = np.asarray(delta, dtype=np.float64)
    shared, M = mc_layout(d.shape, N)
    return np.ascontiguousarray(d), shared, M


def _np_empty(shape, integer):
    return np.empty(shape, dtype=np.int32 if integer else np.float64)


def mc_call(call, N, M, tol, per_sample, empty=_np_empty):
    """Run acoc_track_mc / acoc_lqr_tracking_mc / acoc_track_mc_dev through call(tol_ptr, out_ptr) and collect its outputs as a dict.
    empty(shape, integer) allocates each output: int32 or float64 numpy arrays (default) or CUDA tensors (track_mc_dev)."""
    t = None if tol is None else L.f64(tol, (6,), "tol")
    res = dict(worst_max=empty((N, 6), False), mean_final=empty((N, 6), False), n_reg=empty((N,), True))
    if t is not None:
        res["n_within"] = empty((N,), True)
    if per_sample:
        res["err_max"], res["err_final"] = empty((N, M, 6), False), empty((N, M, 6), False)

    def addr(a):
        return L.ptr(a) if a is None or isinstance(a, np.ndarray) else a.data_ptr()
    out = L.TrackMcOut(*(addr(res.get(k)) for k in ("err_max", "err_final", "worst_max", "mean_final", "n_within", "n_reg")))
    L.check(call(L.ptr(t), C.addressof(out)))
    return res


def lqr_tracking_mc(xx_opt, uu_opt, delta, dyn=None, QQt=None, RRt=None, QQT=None, tol=None, per_sample=False, return_gains=False):
    """Monte Carlo dispersion of the reference's lqr_tracking around each of N nominals: xx_opt (6,TT) or (N,6,TT), uu_opt (2,TT) or
    (N,2,TT); delta (M,6) (the same M perturbations for every nominal) or (N,M,6).  Each nominal gets its own gains; sample (i, m) is the
    closed loop from x*_0 + delta[i, m].  Returns dict(worst_max (N,6) = max over samples of max_t |x_t - x*_t| (NaN if any sample is
    NaN), mean_final (N,6) = mean over samples of |x_{TT-1} - x*_{TT-1}|, n_reg (N)[, n_within (N) = samples whose max error is within
    tol (6,) in every state][, err_max, err_final (N,M,6) per sample with per_sample=True][, K (N,2,6,TT) with return_gains=True]).
    No trajectory is kept: the trajectory of sample m is lqr_tracking_many(xx_opt, uu_opt, delta[:, m]), whose summaries are bit-identical
    to the per-sample ones here.  Same kernels as BatchedNewton.track_mc (acoc_lqr_tracking_mc).  The weights must be symmetric."""
    dyn = dyn or Dynamics()
    dQ, dR, dQT = default_weights()
    Q = L.f64(dQ if QQt is None else QQt, (6, 6), "QQt")
    R = L.f64(dR if RRt is None else RRt, (2, 2), "RRt")
    QT = L.f64(dQT if QQT is None else QQT, (6, 6), "QQT")
    xo, uo = L.f64(xx_opt), L.f64(uu_opt)
    if xo.ndim == 2:
        xo, uo = xo[None], uo[None]
    if xo.ndim != 3 or xo.shape[1] != 6 or xo.shape[2] < 3:
        raise ValueError("xx_opt must be (6,TT) or (N,6,TT) with TT >= 3, got %s" % (np.shape(xx_opt),))
    N, _, TT = xo.shape
    if uo.shape != (N, 2, TT):
        raise ValueError("uu_opt has shape %s, expected %s" % (np.shape(uu_opt), (N, 2, TT)))
    d, shared, M = mc_deltas(delta, N)
    res = mc_call(lambda t, out: L.lib().acoc_lqr_tracking_mc(dyn.device, N, M, TT, L.ptr(dyn.params), int(dyn.state == "f64"), L.ptr(Q),
                                                              L.ptr(R), L.ptr(QT), L.ptr(xo), L.ptr(uo), L.ptr(d), int(shared), t, out),
                  N, M, tol, per_sample)
    if return_gains:
        # the gains depend on the nominals and weights alone: acoc_lqr_tracking_many runs the same gains sweep on them
        res["K"] = lqr_tracking_many(xo, uo, np.zeros((N, 6)), dyn, Q, R, QT, return_gains=True)[2]
    return res


def lqr_tracking(xx_opt, uu_opt, tt, dyn=None, QQt=None, RRt=None, QQT=None):
    """(xx_reg (6,TT), uu_reg (2,TT)) for the shipped perturbation 0.1*ones(6) (lqr_tracking.py:259)."""
    TT = np.asarray(tt).shape[0]
    if np.asarray(xx_opt).shape[1] != TT:
        raise ValueError("tt and xx_opt disagree on the horizon")
    xr, ur = lqr_tracking_batch(xx_opt, uu_opt, np.ones((1, 6)) * 0.1, dyn, QQt, RRt, QQT)
    return xr[0], ur[0]
