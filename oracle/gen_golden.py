#!/usr/bin/env python
"""Generate tests/golden/*.npz from the LIVE, UNMODIFIED reference (run in the build container only).

    python oracle/gen_golden.py [--only NAME ...] [--jobs 4]

The reference is imported from /root/reference through oracle/pyref.py (matplotlib/cvxpy/animate stubbed);
nothing here is needed at test time on the GPU box -- the fixtures are committed.  Every fixture stores
its inputs next to the reference's outputs so the tests can replay the exact call.

Fixtures
  step_kat.npz          Dynamics.step on random (x,u,lambda): float32-quantised and float64 next state,
                        fx, fu, full fxx/fux tensors and their costate contractions
  cost_kat.npz          Cost.stagecost / Cost.termcost, diagonal (config) and dense random weights
  newton_<cfg>_<q>.npz  full NewtonMethod.optimize histories for configs 1 ("step") and 2 ("acro"),
                        state quantisation q in {f32 (as shipped), f64 (line 300 patched)}, with the LQ
                        sub-problem (KK, deltax, deltau) captured at selected iterations
  lq_forced_reg.npz     ltv_LQR on a synthetic indefinite problem that takes the +0.5*I branch
  lqr_tracking.npz      lqr_tracking.py on Data/xx_star.npy with the shipped delta and random deltas
  newton_quirks.npz     optimize()'s return-slot corner cases: max_iters exhausted, and convergence at kk = 0 (zeros)
  gradient_<cfg>_<q>.npz  GradientMethod.optimize histories (line-search call repaired by pyref.run_gradient's call adapter) on the
                        problems of newton_<cfg>_<q>.npz (inputs are read from there): stepsize_0 = 1, 10 candidates, 25 / 12 iterations
"""
from __future__ import annotations

import argparse
import os
import sys
import time
from concurrent.futures import ProcessPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
GOLD = os.path.join(ROOT, "tests", "golden")

from oracle import pyref  # noqa: E402


def _save(name, **arrs):
    os.makedirs(GOLD, exist_ok=True)
    path = os.path.join(GOLD, name)
    np.savez_compressed(path, **arrs)
    print("wrote %s (%.1f KB)" % (path, os.path.getsize(path) / 1024), flush=True)


# ------------------------------------------------------------------------------------------------
def gen_step_kat():
    rng = np.random.default_rng(20240607)
    n = 256
    X = np.stack([rng.uniform(-5, 20, n), rng.uniform(-5, 5, n), rng.uniform(5, 30, n),
                  rng.uniform(-1, 1, n), rng.uniform(-2, 2, n), rng.uniform(-1, 1, n)], axis=1)
    U = np.stack([rng.uniform(-100, 500, n), rng.uniform(-100, 100, n)], axis=1)
    LAM = rng.normal(size=(n, 6)) * np.array([1, 10, 0.1, 1, 0.01, 1])
    # a few hand-picked rows: the shipped x0 of config 1 (Z = 1.93e-217 flushes to 0 in float32), trim point
    X[0] = [0.0, 1.93076021e-217, 16.0, 0.0, 0.0, 0.0]; U[0] = [46.0, 0.0]
    X[1] = [0.0, 0.0, 9.72482686, 0.0, 0.0, -0.162568]; U[1] = [460.0, -60.0]
    out = {k: [] for k in ("xxp32", "xxp64", "fx", "fu", "fxx", "fux", "fxxc", "fuxc", "fuu_zero")}
    d32 = pyref.load(False).aircraft.Dynamics()
    d64 = pyref.load(True).aircraft.Dynamics()
    for x, u, lam in zip(X, U, LAM):
        r32 = d32.step(x, u)
        r64 = d64.step(x, u)
        rl = d64.step(x, u, lam)
        assert r32[0].dtype == np.float32 and r64[0].dtype == np.float64
        out["xxp32"].append(np.asarray(r32[0], dtype=np.float64))
        out["xxp64"].append(r64[0])
        out["fx"].append(r64[1]); out["fu"].append(r64[2]); out["fxx"].append(r64[3]); out["fux"].append(r64[5])
        out["fxxc"].append(rl[3]); out["fuxc"].append(rl[5])
        out["fuu_zero"].append(float(np.all(r64[4] == 0) and np.all(rl[4] == 0)))
        for a, b in zip(r32[1:], r64[1:]):
            assert np.array_equal(a, b)  # derivatives do not depend on the quantisation
    _save("step_kat.npz", x=X, u=U, lam=LAM, **{k: np.array(v) for k, v in out.items()})


def gen_aero_kat():
    """Dynamics.dragForce / liftForce (aircraft_simplified.py:212-261), get_equilibrium (:152-178) and round_theta (:6-14) of the live
    reference on the states of the step KAT."""
    kat = np.load(os.path.join(GOLD, "step_kat.npz"))
    ac = pyref.load(False).aircraft
    d = ac.Dynamics()
    D, dD, Lf, dL = [], [], [], []
    for x in kat["x"][:64]:
        a, b = d.dragForce(x.copy())
        D.append(a); dD.append(b)
        a, b = d.liftForce(x.copy())
        Lf.append(a); dL.append(b)
    th = np.array([0.3, -7.0, 7.0, 13.0, -20.5, 2 * np.pi, -2 * np.pi, 100.0])
    xe, ue = d.get_equilibrium(np.array([0.0, 0.0, 16.0, 0.0, 0.0, 0.0]), np.linspace(0, 1, 1000))
    _save("aero_kat.npz", x=kat["x"][:64], D=np.array(D), dD=np.array(dD), L=np.array(Lf), dL=np.array(dL), th=th,
          th_rounded=np.array([ac.round_theta(t) for t in th]), xe=np.asarray(xe, dtype=np.float64), ue=np.asarray(ue, dtype=np.float64))


def _config_weights(cfg):
    """Weights of main_newton_method.py:52-63 / acrobatic_newton.py:55-65 (restated, checked against the scripts below)."""
    m, g, J = 12, 9.81, 0.24
    Q = np.eye(6) * 1e-6
    Q[1, 1] = m * g * 0.01; Q[2, 2] = 0.5 * m * 0.001; Q[3, 3] = 0.01; Q[4, 4] = 0.5 * J * 0.001
    R = 1e-6 * np.eye(2)
    QT = Q.copy()
    QT[1, 1] = QT[1, 1] * (20 if cfg == "step" else 100)
    QT[3, 3] = QT[1, 1]; QT[0, 0] = QT[1, 1]
    return Q, R, QT


def gen_cost_kat():
    rng = np.random.default_rng(77)
    ac = pyref.load(False).aircraft
    n = 64
    res = dict(x=[], u=[], xr=[], ur=[], ll=[], lx=[], lu=[], llT=[], lTx=[], which=[])
    Qs, Rs, QTs = [], [], []
    for cfg in ("step", "acro"):
        Q, R, QT = _config_weights(cfg)
        Qs.append(Q); Rs.append(R); QTs.append(QT)
    for _ in range(2):  # dense symmetric and dense NON-symmetric weights: the API takes any matrix
        A = rng.normal(size=(6, 6)); B = rng.normal(size=(2, 2)); Cm = rng.normal(size=(6, 6))
        Qs.append(A @ A.T); Rs.append(B @ B.T); QTs.append(Cm @ Cm.T)
    Qs.append(rng.normal(size=(6, 6))); Rs.append(rng.normal(size=(2, 2))); QTs.append(rng.normal(size=(6, 6)))
    for w, (Q, R, QT) in enumerate(zip(Qs, Rs, QTs)):
        cst = ac.Cost(Q, R, QT)
        for _ in range(n):
            x, xr = rng.normal(size=6) * 5, rng.normal(size=6) * 5
            u, ur = rng.normal(size=2) * 100, rng.normal(size=2) * 100
            ll, lx, lu, lxx, lxu, lux, luu = cst.stagecost(x, u, xr, ur)
            llT, lTx, lTxx = cst.termcost(x, xr)
            assert np.array_equal(lxx, Q) and np.array_equal(luu, R) and np.array_equal(lTxx, QT)
            assert not lxu.any() and not lux.any()
            for k, v in (("x", x), ("u", u), ("xr", xr), ("ur", ur), ("ll", ll.item()), ("lx", lx.ravel()), ("lu", lu.ravel()),
                         ("llT", llT.item()), ("lTx", lTx.ravel()), ("which", w)):
                res[k].append(v)
    _save("cost_kat.npz", Q=np.array(Qs), R=np.array(Rs), QT=np.array(QTs), **{k: np.array(v) for k, v in res.items()})


# ------------------------------------------------------------------------------------------------
_SETUP_CACHE = {}


def script_setup(cfg):
    """Problem set-up of the shipped scripts, obtained by RUNNING them (optimize stubbed out)."""
    if cfg not in _SETUP_CACHE:
        name = "main_newton_method.py" if cfg == "step" else "acrobatic_newton.py"
        g = pyref.run_script(name, skip_optimize=True)
        Q, R, QT = _config_weights(cfg)
        assert np.array_equal(Q, g["QQt"]) and np.array_equal(R, g["RRt"]) and np.array_equal(QT, g["QQT"])
        _SETUP_CACHE[cfg] = {k: np.array(g[k], dtype=np.float64) for k in
                             ("xx_ref", "uu_ref", "xx_init", "uu_init", "QQt", "RRt", "QQT", "xxe", "uue", "tt")}
    return _SETUP_CACHE[cfg]


def _newton_job(args):
    cfg, f64, lq_at = args
    s = script_setup(cfg)
    mods = pyref.load(f64)
    keep = tuple(k - 1 for k in lq_at if k > 0)
    t0 = time.time()
    h = pyref.run_newton(mods, s["xx_ref"], s["uu_ref"], s["xx_init"], s["uu_init"], s["QQt"], s["RRt"], s["QQT"],
                         keep_iterates=keep, capture_lq_at=lq_at)
    wall = time.time() - t0
    arrs = dict(xx_ref=s["xx_ref"], uu_ref=s["uu_ref"], xx_init=s["xx_init"], uu_init=s["uu_init"],
                Q=s["QQt"], R=s["RRt"], QT=s["QQT"], xxe=s["xxe"], uue=s["uue"],
                JJ=h["JJ"], descent=h["descent"], stepsize=h["stepsize"], n_armijo=h["n_armijo"], iters=h["iters"],
                xx_star=h["xx_star"], uu_star=h["uu_star"], xx_last=h["xx_last"], uu_last=h["uu_last"],
                lq_at=np.array(lq_at), ref_wall_s=wall)
    for k in lq_at:
        xx_k, uu_k = (s["xx_init"], s["uu_init"]) if k == 0 else h["iterates"][k - 1]
        arrs["it%d_xx" % k], arrs["it%d_uu" % k] = xx_k, uu_k
        arrs["it%d_KK" % k] = h["lq"][k]["KK"]
        arrs["it%d_deltax" % k] = h["lq"][k]["deltax"]
        arrs["it%d_deltau" % k] = h["lq"][k]["deltau"]
    _save("newton_%s_%s.npz" % (cfg, "f64" if f64 else "f32"), **arrs)
    return cfg, f64, h["iters"], wall


def gen_newton(jobs):
    # step/f64 leaves out iteration 0: its LQ sub-problem is that of step/f32 bit for bit (same initial guess), and without it the
    # fixture stays under 1 MB
    work = [("step", False, (0, 9)), ("step", True, (5, 9, 15)), ("acro", False, (0, 5, 9, 15)), ("acro", True, (0, 9))]
    with ProcessPoolExecutor(max_workers=jobs) as ex:
        for cfg, f64, iters, wall in ex.map(_newton_job, work):
            print("newton %s f64=%s: %d iterations, %.1f s" % (cfg, f64, iters, wall), flush=True)


def _batched_instance_job(args):
    """One instance of a BATCHED configuration (BASELINE configs[3] / [4]) through the live reference's NewtonMethod.optimize."""
    cfg, idx = args
    sys.path.insert(0, ROOT)
    from aircraftoptimalcontrol_b200 import refgen   # pinned to the scripts' globals by tests/test_refgen.py
    from oracle import corcl
    if cfg == "config4":
        zf, xf = refgen.config4_params()
        xr, ur = refgen.step_problem(xf[idx:idx + 1], zf[idx:idx + 1])
        Q, R, QT = refgen.weights("step")
        par, dx0 = np.array([zf[idx], xf[idx]]), np.zeros(6)
    else:
        dx0_all, zf = refgen.config5_params()
        xr, ur = refgen.acrobatic_problem(zf[idx:idx + 1])
        Q, R, QT = refgen.weights("acro")
        par, dx0 = np.array([zf[idx]]), dx0_all[idx]
    xr, ur = xr[0], ur[0]
    start = xr.copy()
    start[:, 0] += dx0                                      # x0 = xx_ref[:,0] + dx0 (SURVEY 8(d) config 5); zero for config 4
    xi, ui = corcl.initial_trajectory(start, quant_f32=True)   # the initial guess is an INPUT: the same arrays go to both sides
    t0 = time.time()
    h = pyref.run_newton(pyref.load(False), xr, ur, xi, ui, Q, R, QT)
    return cfg, idx, par, dx0, xi, ui, h, time.time() - t0


def gen_batched_instances(jobs):
    """SURVEY 8(c): the C oracle that the GPU's batched parity tests compare with is itself validated against the Python reference on
    >= 4 instances of the batched configurations: instances 0, 1 of config 4 (65,536 step references, seed 2024) and instances 0, 1 of
    config 5 (1,048,576 acrobatic instances with perturbed x0, seed 7) -- the same instances the GPU tests sample."""
    work = [("config4", 0), ("config4", 1), ("config5", 0), ("config5", 1)]
    arrs = {}
    with ProcessPoolExecutor(max_workers=jobs) as ex:
        for cfg, idx, par, dx0, xi, ui, h, wall in ex.map(_batched_instance_job, work):
            tag = "%s_%d_" % (cfg, idx)
            arrs.update({tag + "par": par, tag + "dx0": dx0, tag + "xx_init": xi, tag + "uu_init": ui, tag + "JJ": h["JJ"],
                         tag + "descent": h["descent"], tag + "stepsize": h["stepsize"], tag + "n_armijo": h["n_armijo"],
                         tag + "iters": h["iters"], tag + "xx_star": h["xx_star"], tag + "uu_star": h["uu_star"], tag + "ref_wall_s": wall})
            print("batched instance %s[%d]: %d iterations, %.1f s" % (cfg, idx, h["iters"], wall), flush=True)
    _save("newton_batched_instances.npz", **arrs)


# ------------------------------------------------------------------------------------------------
def gen_lq_forced_reg():
    """A problem whose R + B'PB is indefinite at some steps, so optcon.py:745-749 adds 0.5*I."""
    oc = pyref.load(False).optcon
    import io
    from contextlib import redirect_stdout
    rng = np.random.default_rng(5)
    TT = 40
    A = np.repeat(np.eye(6)[:, :, None], TT, 2) + 0.05 * rng.normal(size=(6, 6, TT))
    B = 0.3 * rng.normal(size=(6, 2, TT))
    Q = np.repeat(np.diag([1.0, 2.0, 0.5, 0.1, 0.3, 1.5])[:, :, None], TT, 2)
    R = np.repeat(np.diag([-0.05, 0.02])[:, :, None], TT, 2)  # negative weight -> indefinite M at the tail
    R[:, :, ::3] = np.diag([-2.0, 0.01])[:, :, None]
    S = 0.01 * rng.normal(size=(2, 6, TT))
    Qf = np.diag([0.01, 0.02, 0.01, 0.01, 0.01, 0.03])
    q = rng.normal(size=(6, TT)); r = rng.normal(size=(2, TT)); qf = rng.normal(size=6)
    x0 = rng.normal(size=6)
    nreg = {"n": 0}
    orig = np.linalg.eigvals

    def counting(M):
        w = orig(M)
        nreg["n"] += int(not np.all(w > 0))
        return w

    np.linalg.eigvals = counting
    try:
        with redirect_stdout(io.StringIO()):
            Ka, Pa, xa, ua = oc.ltv_LQR(A, B, Q, R, S, Qf, TT, np.zeros(6), q, r, qf)
            n_aug = nreg["n"]; nreg["n"] = 0
            Kn, Pn, xn, un = oc.ltv_LQR(A, B, Q, R, S, Qf, TT, x0, None, None, None)
            n_non = nreg["n"]
    finally:
        np.linalg.eigvals = orig
    assert n_aug > 0 and n_non > 0, (n_aug, n_non)
    _save("lq_forced_reg.npz", A=A, B=B, Q=Q, R=R, S=S, Qf=Qf, q=q, r=r, qf=qf, x0=x0,
          K_aug=Ka, P_aug=Pa, x_aug=xa, u_aug=ua, n_reg_aug=n_aug, K_non=Kn, P_non=Pn, x_non=xn, u_non=un, n_reg_non=n_non)


def gen_lqr_tracking():
    """lqr_tracking.py:245-283 on the shipped optimum; extra perturbations by patching the hard-coded delta (:259)."""
    import importlib.util
    import io
    from contextlib import redirect_stdout
    pyref._install_stubs()
    ac = pyref.load(False).aircraft
    sys.modules["aircraft_simplified"] = ac
    sys.modules["optcon"] = pyref.load(False).optcon
    spec = importlib.util.spec_from_file_location("_acoc_ref_lqrtrack", os.path.join(pyref.REFERENCE_ROOT, "lqr_tracking.py"))
    lt = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(lt)  # __name__ != "__main__": only the function definitions run
    xx_opt = np.load(os.path.join(pyref.REFERENCE_ROOT, "Data", "xx_star.npy"))
    uu_opt = np.load(os.path.join(pyref.REFERENCE_ROOT, "Data", "uu_star.npy"))
    TT = xx_opt.shape[1]
    Q = np.eye(6) * 0.01; Q[1, 1] = 10; Q[0, 0] = 10
    R = np.eye(2) * 1e-5
    QT = Q.copy()
    lt.dyn = ac.Dynamics(); lt.ns, lt.ni = 6, 2; lt.QQt, lt.RRt, lt.QQT = Q, R, QT  # the globals of :322-328
    tt = np.linspace(0, 1, TT)
    rng = np.random.default_rng(1234)
    deltas = [np.ones(6) * 0.1] + [rng.uniform(-0.1, 0.1, 6) for _ in range(3)]
    xs, us = [], []
    class _Delta:  # stands in for np.ones((6,)) at lqr_tracking.py:259 so that "* 0.1" yields our delta exactly
        def __init__(self, d):
            self.d = d

        def __mul__(self, k):
            return self.d.copy()

    class _NpShim:
        def __init__(self, d):
            self._d = d

        def __getattr__(self, k):
            return getattr(np, k)

        def ones(self, shape):
            return _Delta(self._d) if shape == (6,) else np.ones(shape)

    for i, d in enumerate(deltas):
        lt.np = np if i == 0 else _NpShim(d)  # instance 0 is the unmodified reference case
        with redirect_stdout(io.StringIO()):
            xr, ur = lt.lqr_tracking(xx_opt, uu_opt, tt)
        assert np.array_equal(xr[:, 0], xx_opt[:, 0] + d)
        xs.append(xr); us.append(ur)
    # gains as the reference computes them (needs linearisation along the optimum)
    lt.np = np
    AA = np.zeros((6, 6, TT)); BB = np.zeros((6, 2, TT))
    for t in range(TT):
        _, fx, fu = lt.dyn.step(xx_opt[:, t], uu_opt[:, t])[0:3]
        AA[:, :, t] = fx.T; BB[:, :, t] = fu.T
    with redirect_stdout(io.StringIO()):
        KK = lt.ltv_LQR(AA, BB, Q, R, np.zeros((2, 6, TT)), QT, TT, deltas[0], None, None, None)[0]
    _save("lqr_tracking.npz", xx_opt=xx_opt, uu_opt=uu_opt, Q=Q, R=R, QT=QT, delta=np.array(deltas),
          xx_reg=np.array(xs), uu_reg=np.array(us), KK=KK)


def gen_newton_quirks():
    """Return-value corner cases of NewtonMethod.optimize (optcon.py:499-505) from the live reference:
    (a) max_iters = 4 never reaches the tolerance -> the result is the last iterate written (slot max_iters-1);
    (b) starting from an already converged trajectory stops at kk = 0 -> slot -1 of the history array, i.e. all zeros."""
    s = script_setup("step")
    mods = pyref.load(True)
    a = pyref.run_newton(mods, s["xx_ref"], s["uu_ref"], s["xx_init"], s["uu_init"], s["QQt"], s["RRt"], s["QQT"], max_iters=4)
    full = np.load(os.path.join(GOLD, "newton_step_f64.npz"))
    b = pyref.run_newton(mods, s["xx_ref"], s["uu_ref"], full["xx_last"], full["uu_last"], s["QQt"], s["RRt"], s["QQT"])
    assert a["iters"] == 3 and b["iters"] == 1 and not b["xx_star"].any()
    _save("newton_quirks.npz", xx_ref=s["xx_ref"], uu_ref=s["uu_ref"], Q=s["QQt"], R=s["RRt"], QT=s["QQT"],
          a_xx_init=s["xx_init"], a_uu_init=s["uu_init"], a_JJ=a["JJ"], a_descent=a["descent"], a_stepsize=a["stepsize"], a_iters=a["iters"],
          a_xx_star=a["xx_star"], a_uu_star=a["uu_star"],
          b_xx_init=full["xx_last"], b_uu_init=full["uu_last"], b_JJ=b["JJ"], b_descent=b["descent"], b_stepsize=b["stepsize"], b_iters=b["iters"],
          b_xx_star=b["xx_star"], b_uu_star=b["uu_star"])


def _gradient_job(args):
    cfg, f64, max_iters = args
    tag = "%s_%s" % (cfg, "f64" if f64 else "f32")
    d = np.load(os.path.join(GOLD, "newton_%s.npz" % tag))
    t0 = time.time()
    h = pyref.run_gradient(pyref.load(f64), d["xx_ref"], d["uu_ref"], d["xx_init"], d["uu_init"], d["Q"], d["R"], d["QT"],
                           max_iters=max_iters, stepsize_0=1.0, cc=0.5, beta=0.7, armijo_maxiters=10)
    wall = time.time() - t0
    _save("gradient_%s.npz" % tag, base="newton_%s.npz" % tag, max_iters=max_iters, stepsize_0=1.0, cc=0.5, beta=0.7, armijo_maxiters=10,
          JJ=h["JJ"], descent=h["descent"], stepsize=h["stepsize"], n_armijo=h["n_armijo"], iters=h["iters"],
          xx_star=h["xx_star"], uu_star=h["uu_star"], xx_last=h["xx_last"], uu_last=h["uu_last"], deltau_first=h["deltau_first"],
          ref_wall_s=wall)
    return tag, h["iters"], wall


def gen_gradient(jobs):
    work = [("step", False, 26), ("step", True, 26), ("acro", False, 13)]
    with ProcessPoolExecutor(max_workers=jobs) as ex:
        for tag, iters, wall in ex.map(_gradient_job, work):
            print("gradient %s: %d iterations, %.1f s" % (tag, iters, wall), flush=True)


GENERATORS = {
    "step_kat": lambda a: gen_step_kat(),
    "cost_kat": lambda a: gen_cost_kat(),
    "aero_kat": lambda a: gen_aero_kat(),
    "lq_forced_reg": lambda a: gen_lq_forced_reg(),
    "lqr_tracking": lambda a: gen_lqr_tracking(),
    "newton": lambda a: gen_newton(a.jobs),
    "newton_quirks": lambda a: gen_newton_quirks(),
    "batched_instances": lambda a: gen_batched_instances(a.jobs),
    "gradient": lambda a: gen_gradient(a.jobs),
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", nargs="*", default=None)
    ap.add_argument("--jobs", type=int, default=4)
    a = ap.parse_args()
    if not pyref.available():
        sys.exit("reference tree not found at %s" % pyref.REFERENCE_ROOT)
    for name, fn in GENERATORS.items():
        if a.only and name not in a.only:
            continue
        t0 = time.time()
        fn(a)
        print("[%s] done in %.1f s" % (name, time.time() - t0), flush=True)


if __name__ == "__main__":
    main()
