#!/usr/bin/env python
"""Headless drop-in for the reference's lqr_tracking.py __main__ block (:321-342): LQR tracking of a saved optimum
from perturbed initial states (config 3 with --instances 4096).  When --xx holds a batch of optima (N,6,TT) (and --uu (N,2,TT)), every
optimum is tracked along its own gains from its own perturbation (config3_deltas(N)), one lqr_tracking call per optimum.
With --samples M the script runs a dispersion study instead: M config3_deltas(M) perturbations flown around every optimum in --xx (one
(6,TT) optimum, the reference's own case, or a batch), summarised on the device without keeping trajectories; it prints the worst
tracking error per state and the share of flights whose error stays within --tol in every state.
    python scripts/lqr_tracking.py --xx Data/xx_star.npy --uu Data/uu_star.npy [--instances 4096] [--samples M] [--out Data]
"""
import argparse

import numpy as np

import _common  # noqa: F401
from aircraftoptimalcontrol_b200 import refgen
from aircraftoptimalcontrol_b200.aircraft_simplified import Dynamics
from aircraftoptimalcontrol_b200.lqr_tracking import lqr_tracking_batch, lqr_tracking_many, lqr_tracking_mc

ap = argparse.ArgumentParser()
ap.add_argument("--xx", default="Data/xx_star.npy")
ap.add_argument("--uu", default="Data/uu_star.npy")
ap.add_argument("--instances", type=int, default=1)
ap.add_argument("--state", default="f32", choices=["f32", "f64"])
ap.add_argument("--out", default="Data")
ap.add_argument("--samples", type=int, default=None, help="dispersion study: M perturbed flights around every optimum")
ap.add_argument("--tol", type=float, nargs=6, default=[1.0, 1.0, 1.0, 0.2, 0.5, 0.2],
                help="capture tolerance on the max tracking error of each state (x, z, V, theta, q, gamma)")
args = ap.parse_args()

xx_opt, uu_opt = np.load(args.xx), np.load(args.uu)
QQt, RRt, QQT = refgen.weights("track")
if args.samples is not None:
    tol = np.array(args.tol)
    res = lqr_tracking_mc(xx_opt, uu_opt, refgen.config3_deltas(args.samples), Dynamics(state=args.state), QQt, RRt, QQT, tol=tol)
    n = 1 if xx_opt.ndim == 2 else xx_opt.shape[0]
    print("flew %d perturbed starts around each of %d optima" % (args.samples, n))
    print("worst tracking error per state over all flights: %s" % np.nanmax(res["worst_max"], axis=0))
    print("mean final tracking error per state: %s" % res["mean_final"].mean(0))
    print("capture rate within tol %s: %.4f" % (tol, res["n_within"].sum() / (n * args.samples)))
    raise SystemExit(0)
if xx_opt.ndim == 3:
    deltas = refgen.config3_deltas(xx_opt.shape[0])
    xx_lqr, uu_lqr = lqr_tracking_many(xx_opt, uu_opt, deltas, Dynamics(state=args.state), QQt, RRt, QQT)
    _common.save("xx_lqr.npy", xx_lqr, args.out)
    _common.save("uu_lqr.npy", uu_lqr, args.out)
    err = np.abs(xx_lqr[:, :, -1] - xx_opt[:, :, -1])
    print("tracked %d optima along their own gains; largest final tracking error per state: %s" % (xx_opt.shape[0], err.max(0)))
    raise SystemExit(0)
deltas = refgen.config3_deltas(args.instances)  # instance 0 = the shipped 0.1*ones(6) (lqr_tracking.py:259)
xx_lqr, uu_lqr = lqr_tracking_batch(xx_opt, uu_opt, deltas, Dynamics(state=args.state), QQt, RRt, QQT)
_common.save("xx_lqr.npy", xx_lqr[0] if args.instances == 1 else xx_lqr, args.out)
_common.save("uu_lqr.npy", uu_lqr[0] if args.instances == 1 else uu_lqr, args.out)
print("tracked %d perturbed initial states; final tracking error of instance 0: %s" % (args.instances, np.abs(xx_lqr[0, :, -1] - xx_opt[:, -1])))
