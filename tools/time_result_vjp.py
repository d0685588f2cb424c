#!/usr/bin/env python
"""Device time of the derivative of the optimum (BatchedNewton.result_vjp_dev, acoc_result_vjp_dev) at 65,536 x 1000: configs[3] step
maneuvers with parametric references, solved on the device.  One JSON line per variant (all outputs / only x0, zf, vx, n_indef):
  - whole-call device ms (CUDA events on the caller's stream around the call; median of --reps calls after one warm-up call) next to
    the solve it differentiates;
  - per-kernel device ms from torch.profiler (CUDA activities, one call of its own);
  - for each sweep, the bytes it moves per lane-step and the fraction of the measured copy bandwidth (acoc_measure_copy_bw) that its
    kernel time reaches.
    python tools/time_result_vjp.py [--n 65536] [--reps 5] [--out profiles/r06_result_vjp.jsonl]
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

# bytes per lane-step with float32-valued states and parametric step references (the V table travels, X / Z are formed)
BYTES = {
    "k_vjp_backward_tma": 24 + 16 + 8 + 48 + 16 + 14 * 8,  # x*, u*, V, gbar_x, gbar_u in; K, sigma out
    "k_vjp_forward_tma": 14 * 8 + 16 + 24 + 8 + 64,        # K, sigma, u*, x*, V in; xref_bar, uref_bar out (full variant)
    "k_track_nominal": 24 + 16 + 24 + 16,                  # gather of the result slot
}


def gpu_label():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception:
        return pkg.device_info(0)["name"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=65536)
    ap.add_argument("--TT", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="profiles/r06_result_vjp.jsonl")
    a = ap.parse_args()
    n, TT = a.n, a.TT
    label = gpu_label()
    bw = _lib.measure_copy_bw(0)
    zf, xf = refgen.config4_params(n, 2024)
    rows = []
    with pkg.BatchedNewton(n, TT=TT, armijo="lazy") as bn:
        bn.set_weights(*refgen.weights("step"))
        bn.set_refs_step(zf, xf)
        bn.init_guess()
        t0 = time.perf_counter()
        bn.solve()
        solve_ms = (time.perf_counter() - t0) * 1e3
        g = torch.Generator(device="cuda:0").manual_seed(0)
        gx = torch.randn((n, 6, TT), dtype=torch.float64, device="cuda:0", generator=g)
        gu = torch.randn((n, 2, TT), dtype=torch.float64, device="cuda:0", generator=g)
        for full in (True, False):
            call = (lambda: bn.result_vjp_dev(gx, gu)) if full else (lambda: _small(bn, gx, gu))
            call()
            ms = []
            for _ in range(a.reps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                call()
                e1.record()
                torch.cuda.synchronize()
                ms.append(e0.elapsed_time(e1))
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                call()
                torch.cuda.synchronize()
            kern = {}
            for ev in prof.key_averages():
                if ev.device_type == torch.autograd.DeviceType.CUDA or getattr(ev, "device_time_total", 0) > 0:
                    name = ev.key.split("<")[0].split("(")[0].replace("void ", "").replace("acoc::", "")
                    kern[name] = kern.get(name, 0.0) + getattr(ev, "device_time_total", getattr(ev, "cuda_time_total", 0.0)) / 1e3
            frac = {}
            for k, b in BYTES.items():
                if k in kern and kern[k] > 0:
                    bb = b if (full or k != "k_vjp_forward_tma") else b - 64
                    frac[k] = dict(bytes_per_lane_step=bb, gbs=n * (TT - 1) * bb / (kern[k] * 1e-3) / 1e9,
                                   fraction_of_copy_bw=n * (TT - 1) * bb / (kern[k] * 1e-3) / 1e9 / bw)
            rows.append(dict(tool="time_result_vjp", gpu=label, n=n, TT=TT, outputs="all" if full else "x0, zf, vx, n_indef",
                             call_ms_median=float(np.median(ms)), call_ms=ms, solve_wall_ms=solve_ms, kernels_ms=kern, sweeps=frac,
                             copy_bw_gbs=bw))
            print(json.dumps(rows[-1]))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")


def _small(bn, gx, gu):
    """result_vjp_dev without the (N,C,TT) outputs: x0, zf, vx and n_indef only (16 B + 48 B per instance written)."""
    import ctypes as C
    dev = torch.device("cuda", bn.device)
    o = dict(x0=torch.empty((bn.N, 6), dtype=torch.float64, device=dev), zf=torch.empty(bn.N, dtype=torch.float64, device=dev),
             vx=torch.empty(bn.N, dtype=torch.float64, device=dev), n_indef=torch.empty(bn.N, dtype=torch.int32, device=dev))
    s = _lib.VjpOut(None, None, o["x0"].data_ptr(), o["zf"].data_ptr(), o["vx"].data_ptr(), o["n_indef"].data_ptr())
    _lib.check(_lib.lib().acoc_result_vjp_dev(bn._h, gx.data_ptr(), gu.data_ptr(), C.addressof(s), _lib.dev_stream(bn.device)))
    return o


if __name__ == "__main__":
    main()
