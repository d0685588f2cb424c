#!/usr/bin/env python
"""Device time of closed-loop tracking of every instance (BatchedNewton.track, acoc_track) at TT = 1000 for N in {1, 4096, 65536}
configs[3] step maneuvers solved on the device.  One JSON line per N:
  - per-kernel device ms (acoc_get_track_timing, CUDA events; median of --reps calls after one warm-up call);
  - closed-loop steps/s (N * (TT-1) / rollout time, and over the three kernels);
  - bytes the algorithm moves per instance-step and the fraction of the measured copy bandwidth (acoc_measure_copy_bw) for the
    nominal and rollout kernels;
  - gains sweep ms per lane-step next to k_backward_tma in Gauss-Newton mode on the same batch (acoc_backward on a fully active context,
    host wall around launch + sync; the small-batch warp-role backward variants are disabled so that the TMA sweep is what runs);
  - end-to-end wall of track + tracked (trajectories downloaded) and of track alone (summaries only).
    python tools/time_track_batch.py [--reps 5] [--out track_batch.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys
import time

os.environ.setdefault("ACOC_NO_BWD_COLS", "1")   # k_backward_tma for every N (read once by the library)
os.environ.setdefault("ACOC_NO_BWD_SPLIT", "1")
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402

import aircraftoptimalcontrol_b200 as pkg  # noqa: E402
from aircraftoptimalcontrol_b200 import _lib, refgen  # noqa: E402


def gpu_label():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        return q
    except Exception:
        return pkg.device_info(0)["name"]


def solved(n, TT, seed=2024):
    zf, xf = refgen.config4_params(max(n, 2), seed)
    bn = pkg.BatchedNewton(n, TT=TT, armijo="lazy")
    bn.set_weights(*refgen.weights("step"))
    bn.set_refs_step(zf[:n], xf[:n])
    bn.init_guess()
    bn.solve()
    return bn, zf[:n], xf[:n]


def backward_gn_ms(n, TT, zf, xf, reps):
    with pkg.BatchedNewton(n, TT=TT, armijo="lazy") as bn:
        bn.set_weights(*refgen.weights("step"))
        bn.set_refs_step(zf, xf)
        bn.init_guess()
        bn.backward(exact=False)
        bn.sync()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            bn.backward(exact=False)
            bn.sync()
            ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sizes", default="1,4096,65536")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    TT = 1000
    bw = _lib.measure_copy_bw(0)  # GB/s, read + write
    label = gpu_label()
    lines = []
    for n in (int(s) for s in a.sizes.split(",")):
        bn, zf, xf = solved(n, TT)
        d = refgen.config3_deltas(max(n, 2))[:n]
        bn.track(d)  # warm-up: allocates the tracking buffers, loads the kernels
        ms, wall_all, wall_sum = [], [], []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            bn.track(d)
            bn.tracked()
            wall_all.append(time.perf_counter() - t0)
            t = bn.track_timing()
            ms.append([t["total_ms"], t["nominal_ms"], t["gains_ms"], t["rollout_ms"]])
            t0 = time.perf_counter()
            bn.track(d)
            wall_sum.append(time.perf_counter() - t0)
        ms = np.median(np.array(ms), axis=0)
        es = 4  # the default context keeps its float32-valued states (and so the nominals and the tracked states) as float
        steps = n * (TT - 1)
        b_nom = (6 * es + 16) * 2              # read the result slot, write Xnom / Unom
        b_gain = (6 * es + 16) + 96            # read x*, u*; write K
        b_roll = (96 + 6 * es + 16) + (6 * es + 16)  # read K, x*, u*; write x, u
        gn_ms = backward_gn_ms(n, TT, zf, xf, a.reps)
        np_lanes = (n + 31) // 32 * 32
        rec = dict(N=n, TT=TT, gpu=label, device_bytes=bn.device_bytes, copy_bw_gbs=round(bw, 1),
                   ms=dict(total=ms[0], nominal=ms[1], gains=ms[2], rollout=ms[3]),
                   closed_loop_steps_per_s=dict(rollout=steps / (ms[3] * 1e-3), all_kernels=steps / (ms[0] * 1e-3)),
                   bytes_per_instance_step=dict(nominal=b_nom, gains=b_gain, rollout=b_roll),
                   hbm_fraction=dict(nominal=n * TT * b_nom / (ms[1] * 1e-3) / (bw * 1e9),
                                     rollout=n * (TT - 1) * b_roll / (ms[3] * 1e-3) / (bw * 1e9)),
                   gains_ms_per_lane_step=ms[2] / (np_lanes * (TT - 1)), backward_tma_gn_ms=gn_ms,
                   backward_tma_gn_ms_per_lane_step=gn_ms / (np_lanes * (TT - 1)),
                   wall_ms=dict(track_and_tracked=float(np.median(wall_all)) * 1e3, track_only=float(np.median(wall_sum)) * 1e3))
        bn.close()
        print(json.dumps(rec), flush=True)
        lines.append(json.dumps(rec))
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
