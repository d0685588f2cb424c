#!/usr/bin/env python
"""Host-array calls against their device-resident twins (the _dev entry points, CUDA tensors in and out) on one solved configs[3]
batch of 65,536 step maneuvers x TT = 1000.  Each pair runs in the same process, alternated host / device, after one untimed call of
each; times are the host wall of the whole call (every call ends in a device synchronise), median and minimum over --reps.  Host
arrays are page-locked (pinned) except in the dispersion study, which uses what a numpy user has: numpy deltas and track_mc's own
output arrays.  One JSON line per pair:
  - set_refs vs set_refs_dev, set_init vs set_init_dev (4.2 GB each), result / result_f32 vs result_dev in both dtypes, track + tracked
    vs track + tracked_dev, track_gains vs track_gains_dev;
  - a whole dispersion study at 65,536 x 64 per-instance deltas with per-sample outputs, the generation of the deltas included: numpy
    deltas + track_mc vs torch.randn deltas on the device + track_mc_dev;
  - for each device call that is one layout conversion, the bytes it must move (read + write, counted from the shapes and element
    types) over its wall time, next to acoc_measure_copy_bw (read + write bytes / time of a device copy) from the same run;
  - the GPU name, power limit and maximum SM clock, read in the same run, in every record.
    python tools/time_device_io.py [--reps 5] [--n 65536] [--out profiles/r05_device_io.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import aircraftoptimalcontrol_b200 as pkg  # noqa: E402
from aircraftoptimalcontrol_b200 import _lib, refgen  # noqa: E402


def gpu_label():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True, timeout=30).stdout.strip().splitlines()
    return q[0] if q else pkg.device_info(0)["name"]


class Pool:
    """Consecutive views of one preallocated byte buffer (page-locked host or device), so that the largest pair sets the footprint."""

    def __init__(self, nbytes, device=None):
        self.buf = (torch.empty(nbytes, dtype=torch.uint8, pin_memory=True) if device is None
                    else torch.empty(nbytes, dtype=torch.uint8, device=device))

    def carve(self, *specs):
        out, off = [], 0
        for shape, dtype in specs:
            n = int(np.prod(shape)) * torch.tensor([], dtype=dtype).element_size()
            out.append(self.buf[off:off + n].view(dtype).view(shape))
            off += (n + 255) // 256 * 256
        return out


def timed(fn):
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3


def pair(name, host, dev, reps, label, dev_bytes=None, copy_bw=None, **extra):
    """Alternate host() and dev() after one untimed call of each; dev_bytes: bytes the device call's conversions move."""
    host(), dev()
    th, td = [], []
    for _ in range(reps):
        th.append(timed(host))
        td.append(timed(dev))
    rec = dict(pair=name, gpu=label, reps=reps,
               host_ms=dict(median=float(np.median(th)), min=float(np.min(th))),
               dev_ms=dict(median=float(np.median(td)), min=float(np.min(td))),
               speedup_median=float(np.median(th) / np.median(td)), **extra)
    if dev_bytes is not None:
        gbs = dev_bytes / (np.median(td) * 1e-3) / 1e9
        rec.update(dev_bytes_moved=int(dev_bytes), dev_gb_per_s=float(gbs), copy_bw_gb_per_s=copy_bw, dev_share_of_copy_bw=float(gbs / copy_bw))
    print(json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--n", type=int, default=65536)
    ap.add_argument("--samples", type=int, default=64)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    n, TT, M = a.n, 1000, a.samples
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: these are device timings")
    label = gpu_label()
    copy_bw = _lib.measure_copy_bw(0)
    f64, f32, i32 = torch.float64, torch.float32, torch.int32
    sx, su, sk = (n, 6, TT), (n, 2, TT), (n, 2, 6, TT)
    big = 12 * n * TT * 8 + 4096                     # the gains, the largest single output
    hp, dp = Pool(big), Pool(big, "cuda:0")
    recs = []

    zf, xf = refgen.config4_params(n, 2024)
    bn = pkg.BatchedNewton(n, TT=TT, armijo="lazy")
    bn.set_weights(*refgen.weights("step"))
    bn.set_refs_step(zf, xf)
    bn.init_guess()
    bn.solve()

    # outputs: result / result_f32 vs result_dev
    hx, hu = hp.carve((sx, f64), (su, f64))
    dx, du = dp.carve((sx, f64), (su, f64))
    x_read = n * 6 * TT * 4                          # the state slots hold float32 values (float32 state quantisation)
    u_rw = 2 * n * 2 * TT * 8
    recs.append(pair("result vs result_dev(float64)", lambda: bn.result(out=(hx.numpy(), hu.numpy())),
                     lambda: bn.result_dev(out=(dx, du)), a.reps, label, x_read + n * 6 * TT * 8 + u_rw, copy_bw))
    hx, hu = hp.carve((sx, f32), (su, f64))
    dx, du = dp.carve((sx, f32), (su, f64))
    recs.append(pair("result_f32 vs result_dev(float32)", lambda: bn.result_f32(out=(hx.numpy(), hu.numpy())),
                     lambda: bn.result_dev(f32, out=(dx, du)), a.reps, label, 2 * x_read + u_rw, copy_bw))

    # tracking: track + tracked vs track + tracked_dev; track_gains vs track_gains_dev
    delta = np.full(6, 0.01)
    hx, hu = hp.carve((sx, f64), (su, f64))
    dx, du = dp.carve((sx, f64), (su, f64))
    recs.append(pair("track + tracked vs track + tracked_dev", lambda: (bn.track(delta), bn.tracked(out=(hx.numpy(), hu.numpy()))),
                     lambda: (bn.track(delta), bn.tracked_dev(out=(dx, du))), a.reps, label))
    recs.append(pair("tracked vs tracked_dev", lambda: bn.tracked(out=(hx.numpy(), hu.numpy())), lambda: bn.tracked_dev(out=(dx, du)),
                     a.reps, label, x_read + n * 6 * TT * 8 + u_rw, copy_bw))
    (hk,), (dk,) = hp.carve((sk, f64)), dp.carve((sk, f64))
    hk_np = hk.numpy()

    def host_gains():   # track_gains() allocates its output; the pinned copy below is the same call into page-locked memory
        _lib.check(_lib.lib().acoc_get_track_gains(bn._h, hk_np.ctypes.data))
    recs.append(pair("track_gains vs track_gains_dev", host_gains, lambda: bn.track_gains_dev(out=dk), a.reps, label,
                     2 * n * 12 * TT * 8, copy_bw))

    # a whole dispersion study, the generation of the deltas included
    rng = np.random.default_rng(0)
    gen = torch.Generator(device="cuda:0").manual_seed(0)
    tol = np.array([1.0, 1.0, 1.0, 0.2, 0.5, 0.2])
    recs.append(pair("dispersion study: numpy deltas + track_mc vs torch.randn deltas + track_mc_dev",
                     lambda: bn.track_mc(rng.standard_normal((n, M, 6)) * 0.02, tol=tol, per_sample=True),
                     lambda: bn.track_mc_dev(torch.randn((n, M, 6), dtype=f64, device="cuda:0", generator=gen) * 0.02, tol=tol,
                                             per_sample=True),
                     a.reps, label, samples=M, delta_bytes=n * M * 6 * 8, per_sample_output_bytes=2 * n * M * 6 * 8))

    # inputs: set_refs vs set_refs_dev, set_init vs set_init_dev (the context's solve is over; these reset it)
    xr, ur = bn.refs()
    hx, hu = hp.carve((sx, f64), (su, f64))
    dx, du = dp.carve((sx, f64), (su, f64))
    hx.numpy()[...], hu.numpy()[...] = xr, ur
    dx.copy_(hx), du.copy_(hu)
    del xr, ur
    recs.append(pair("set_refs (pinned) vs set_refs_dev", lambda: bn.set_refs(hx.numpy(), hu.numpy()), lambda: bn.set_refs_dev(dx, du),
                     a.reps, label, 2 * n * 8 * TT * 8, copy_bw))
    xs, us = bn.result()
    hx.numpy()[...], hu.numpy()[...] = xs, us
    dx.copy_(hx), du.copy_(hu)
    del xs, us
    # float32-valued states: the probe pass (float slots) is the only pass over xx_init
    recs.append(pair("set_init (pinned) vs set_init_dev", lambda: bn.set_init(hx.numpy(), hu.numpy()), lambda: bn.set_init_dev(dx, du),
                     a.reps, label, n * 6 * TT * (8 + 4) + u_rw, copy_bw))
    bn.close()
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write("".join(json.dumps(r) + "\n" for r in recs))


if __name__ == "__main__":
    main()
