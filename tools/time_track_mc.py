#!/usr/bin/env python
"""Device time of the Monte Carlo dispersion of closed-loop tracking (BatchedNewton.track_mc, acoc_track_mc) at TT = 1000 on solved
configs[3] step maneuvers, for (N, M) in {(65536, 64), (4096, 64), (1, 4096)} with M shared configs[3] perturbations.  One JSON line per
case:
  - per-kernel device ms of track_mc (acoc_get_track_timing, CUDA events; median of --reps calls after one warm-up call): nominal copy,
    gains sweep, dispersion rollout + reduction, total; and the host wall of the whole call (summaries only);
  - closed-loop sample-steps/s of the dispersion rollout, N * M * (TT-1) / its time;
  - FP64-pipe instructions per sample-step of k_track_mc_rollout_tma, counted statically from its SASS (tools/sass_fp64_count.py: the
    largest backward-branch region, i.e. the time loop; the out-of-line slow paths inside that address range are included, so the count
    is an upper bound), and the computed share of the FP64 issue rate measured by acoc_measure_fp64_peak (computed from counted
    instructions, not measured by a profiler);
  - in the same run, for the same N and deltas: the device time of M back-to-back track(delta[:, m]) calls (sum of their CUDA-event
    totals) and of k_track_rollout_tma alone (median over those calls);
  - the GPU name, power limit and maximum SM clock, read in the same run.
    python tools/time_track_mc.py [--reps 5] [--out profiles/r04_track_mc.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402

import aircraftoptimalcontrol_b200 as pkg  # noqa: E402
from aircraftoptimalcontrol_b200 import _lib, refgen  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def gpu_label():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True, timeout=30).stdout.strip().splitlines()
    return q[0] if q else pkg.device_info(0)["name"]


def sass_fp64_per_step(x_float=True):
    """Static FP64-pipe instruction count of the time loop of k_track_mc_rollout_tma<true, XT> (float32 state quantisation)."""
    nvcc_dir = os.path.dirname(os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc"))
    env = dict(os.environ, PATH=os.environ.get("PATH", "") + os.pathsep + nvcc_dir)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "sass_fp64_count.py"), _lib.LIB_PATH], capture_output=True, text=True,
                         check=True, env=env).stdout
    k = json.loads(out)["kernels"]
    name = "k_track_mc_rollout_tma<true, %s>" % ("float" if x_float else "double")
    return k[name]["fp64_pipe"], k["k_track_rollout_tma<true, %s>" % ("float" if x_float else "double")]["fp64_pipe"]


def solved(n, TT, seed=2024):
    zf, xf = refgen.config4_params(max(n, 2), seed)
    bn = pkg.BatchedNewton(n, TT=TT, armijo="lazy")
    bn.set_weights(*refgen.weights("step"))
    bn.set_refs_step(zf[:n], xf[:n])
    bn.init_guess()
    bn.solve()
    return bn


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--cases", default="65536x64,4096x64,1x4096")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    TT = 1000
    label = gpu_label()
    fp64_peak = _lib.measure_fp64_peak(0)          # TFLOP/s of DFMA = 2 flops per FP64 instruction slot
    fp64_mc, fp64_track = sass_fp64_per_step()
    lines = []
    for case in a.cases.split(","):
        n, M = (int(v) for v in case.split("x"))
        bn = solved(n, TT)
        d = refgen.config3_deltas(M)
        tol = np.array([1.0, 1.0, 1.0, 0.2, 0.5, 0.2])
        res = bn.track_mc(d, tol=tol)                 # warm-up: allocates the buffers, loads the kernels
        ms, wall = [], []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            bn.track_mc(d, tol=tol)
            wall.append((time.perf_counter() - t0) * 1e3)
            t = bn.track_timing()
            ms.append([t["total_ms"], t["nominal_ms"], t["gains_ms"], t["rollout_ms"]])
        ms = np.median(np.array(ms), axis=0)
        mem = bn.device_bytes
        # M back-to-back track calls over the same deltas (per-instance (N,6) = delta[m] broadcast)
        bn.track(np.broadcast_to(d[0], (n, 6)))
        tr_total, tr_roll = [], []
        t0 = time.perf_counter()
        for m in range(M):
            bn.track(np.broadcast_to(d[m], (n, 6)))
            t = bn.track_timing()
            tr_total.append(t["total_ms"])
            tr_roll.append(t["rollout_ms"])
        tr_wall = (time.perf_counter() - t0) * 1e3
        bn.close()
        steps = n * M * (TT - 1)
        roll_s = ms[3] * 1e-3
        fp64_rate = fp64_mc * steps / roll_s           # FP64-pipe lane-instructions per second (computed)
        track_roll_s = float(np.median(tr_roll)) * 1e-3
        rec = dict(
            N=n, M=M, TT=TT, gpu=label, device_bytes_after_track=mem,
            track_mc_ms=dict(total=ms[0], nominal=ms[1], gains=ms[2], rollout_and_reduce=ms[3]),
            track_mc_wall_ms=float(np.median(wall)),
            sample_steps_per_s=dict(dispersion_rollout=steps / roll_s, whole_call=steps / (ms[0] * 1e-3)),
            fp64_per_sample_step_static=dict(k_track_mc_rollout_tma=fp64_mc, k_track_rollout_tma=fp64_track),
            fp64_peak_tflops_measured=fp64_peak,
            fp64_issue_share_computed=fp64_rate / (fp64_peak * 1e12 / 2),
            track_calls=dict(calls=M, device_ms_sum=float(np.sum(tr_total)), wall_ms=tr_wall,
                             k_track_rollout_tma_ms_median=float(np.median(tr_roll)),
                             k_track_rollout_tma_steps_per_s=n * (TT - 1) / track_roll_s),
            speedup=dict(rollout_steps_per_s_vs_k_track_rollout_tma=(steps / roll_s) / (n * (TT - 1) / track_roll_s),
                         track_mc_device_time_over_track_calls=ms[0] / float(np.sum(tr_total))),
            capture_rate=float(res["n_within"].sum()) / (n * M),
        )
        print(json.dumps(rec), flush=True)
        lines.append(json.dumps(rec))
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
