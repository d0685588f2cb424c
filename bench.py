#!/usr/bin/env python
"""bench.py -- trajectory-Newton-iterations / second on B200 (BASELINE.json metric) and the other BASELINE configurations.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload step|acro|track|single-step|single-acro]
                    [--instances M] [--precision f64|f32] [--armijo lazy|speculative] [--state f32|f64] [--no-e2e] [--no-cpu]
                    [--dump-outputs DIR]
    torchrun --nproc-per-node N bench.py --gpus N ...          (one rank per GPU, launched by the driver)

Workloads (config.workload):
  step         BASELINE.json configs[3] (default, the configuration the metric is quoted on): 65,536 randomised step references per
               GPU (weak scaling: rank r of world w holds instances r::w of a 65,536*w batch).
  acro         configs[4]: acrobatic batch with perturbed x0 (1,048,576 instances = --instances 131072 on 8 GPUs).
  track        configs[2]: lqr_tracking of Data/xx_star.npy from 4096 perturbed initial states (unit: closed-loop rollout steps / s).
  single-step  configs[0] / single-acro configs[1]: ONE trajectory (latency: ms per Newton iteration, whole solve).
A "step" of the Newton workloads is ONE Newton iteration (loop body of optcon.py:415-501: fused backward Riccati/costate sweep, LQ
forward pass + descent, Armijo candidate rollouts, update) over the whole batch: W warm-up iterations, then K timed ones -- iterations
W..W+K-1 of the real solve from the device-generated initial guess.  Time = CUDA events on the context's stream, max over ranks.

The JSON line carries: value (device-resident inputs), e2e (full solve through the Python API / C ABI from host buffers with the
copies inside the timed wall), whole_solve, roofline (dominant kernel; per-kernel table with bytes / FP64 instructions counted from
the per-iteration ACTIVE instance counts), cpu_baseline (C port of the reference on the host cores + the Python reference, live when
its tree is present, else the recorded measurement), clocks.

--impl reference times the CPU port alone on the same workload (the reference itself is Python and is not present on the GPU box).
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "trajectory_newton_iterations_per_second"
UNIT = "traj-Newton-it/s"
TT = 1000

# SURVEY.md 8(d): algorithmic FP64 flops / HBM bytes per instance per time step (dense ns=6, ni=2 accounting, float64 storage)
FLOPS = dict(backward=2106, forward=126 + 30, cost=107, candidate=159, update=52 + 107)
BYTES = dict(backward=128 + 128, forward=128 + 64 + 16, cost=128, candidate=32 + 64, candidate_write=32 + 64 + 64, update=32 + 64 + 64)


def moved_bytes(args):
    """Bytes per instance per time step the kernels actually move in the selected mode.  The parity path stores the float32-quantised
    states as float (24 instead of 48 B per state read/write, bit-identical results); references built on the device stay parametric
    (8 B of stored speed reference for the step maneuver, nothing for the acrobatic one, instead of 64 B); the FP32 mode halves
    everything (and keeps expanded references)."""
    if args.precision == "f32":
        return {k: v // 2 for k, v in BYTES.items()}
    mb = dict(BYTES)
    if args.state == "f32" and args.x_storage == "auto":
        for k in ("backward", "forward", "cost", "candidate_write", "update"):
            mb[k] -= 24
    if args.refs == "compact":
        saved = 56 if args.workload == "step" else 64
        for k in ("backward", "cost", "candidate", "candidate_write", "update"):
            mb[k] -= saved
    return mb


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback (B200_PROFILING.md)"


def source_sha16():
    h = hashlib.sha256()
    d = os.path.join(ROOT, "aircraftoptimalcontrol_b200", "csrc")
    for f in sorted(os.listdir(d)):
        h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


def kernel_counters():
    """Per-launch DRAM bytes and executed FP64-pipe instructions of the sweep kernels from the committed `ncu --set full` capture of
    THIS build (profiles/r02_kernel_counters.json, written by profiles/summarize_ncu.py --counters); None if the capture belongs
    to another build of the kernels."""
    p = os.path.join(ROOT, "profiles", "r02_kernel_counters.json")
    try:
        kc = json.load(open(p))
    except Exception:
        return None, "no capture committed"
    if kc.get("source_sha16") != source_sha16():
        return None, "profiles/r02_kernel_counters.json was captured from another build of csrc/ (%s != %s)" % (kc.get("source_sha16"), source_sha16())
    return kc, "profiles/r02_kernel_counters.json (ncu --set full of this build, per launch, %d instances)" % kc.get("instances", 0)


class ClockSampler(threading.Thread):
    """Samples SM clocks and throttle reasons of one GPU with nvidia-smi while the timed region runs."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        self.stop_flag = True
        self.join(timeout=6)
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) > 3 + k and r[3 + k].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


def make_problem(workload, n_total, lo_hi_stride, seed=None):
    """Per-rank shard of the batched configuration: instances rank::world of the n_total-instance batch.
    Returns (xx_ref, uu_ref, dx0, weights, gen) with gen = the arguments of PipelinedNewton.solve(refs=...) that generate the same
    references on the device."""
    from aircraftoptimalcontrol_b200 import refgen
    r, w = lo_hi_stride
    if workload == "step":
        zf, xf = refgen.config4_params(n_total, 2024 if seed is None else seed)
        zf, xf = np.ascontiguousarray(zf[r::w]), np.ascontiguousarray(xf[r::w])
        xr, ur = refgen.step_problem(xf, zf, TT=TT)
        return xr, ur, None, refgen.weights("step"), ("step", zf, xf)
    dx0, zf = refgen.config5_params(n_total, 7 if seed is None else seed)
    zf = np.ascontiguousarray(zf[r::w])
    xr, ur = refgen.acrobatic_problem(zf, TT=TT)
    return xr, ur, np.ascontiguousarray(dx0[r::w]), refgen.weights("acro"), ("acrobatic", zf)


def pinned_like(a):
    """Copy a numpy array into pinned host memory (torch is only the allocator here)."""
    import torch
    t = torch.empty(a.shape, dtype=torch.float64, pin_memory=True)
    t.numpy()[...] = a
    return t  # keep the tensor alive; .numpy() is the view


def host_threads():
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def cpu_port_rate(workload, sample, W, K, state):
    """Newton iterations W..W+K-1 of `sample` instances with the C port of the reference on all host threads."""
    from oracle import corcl
    corcl.build()
    xr, ur, dx0, (Q, R, QT), _ = make_problem(workload, sample, (0, 1))
    xi = np.zeros((sample, 6, TT))
    ui = np.zeros((sample, 2, TT))
    for i in range(sample):  # the initial guess is an input of the hot path (float64 P-law rollout, same as the GPU's)
        xref_i = xr[i].copy()
        if dx0 is not None:
            xref_i[:, 0] += dx0[i]
        xi[i], ui[i] = corcl.initial_trajectory(xref_i if dx0 is not None else xr[i], quant_f32=(state == "f32"))
    nt = host_threads()
    kw = dict(quant_f32=(state == "f32"), n_threads=nt)
    m = min(sample, nt)   # untimed: starts the OpenMP thread pool and faults in the library
    corcl.newton_batch(xr[:m], ur[:m], xi[:m], ui[:m], Q, R, QT, n_iters_cap=1, **kw)
    t0 = time.perf_counter()
    a = corcl.newton_batch(xr, ur, xi, ui, Q, R, QT, n_iters_cap=W, **kw) if W > 0 else None
    t1 = time.perf_counter()
    b = corcl.newton_batch(xr, ur, xi, ui, Q, R, QT, n_iters_cap=W + K, **kw)
    t2 = time.perf_counter()
    its = int(b["iters"].sum()) - (int(a["iters"].sum()) if a is not None else 0)
    dt = (t2 - t1) - (t1 - t0 if a is not None else 0.0)
    if dt <= 0 or its <= 0:  # (only with samples so small that timer noise exceeds K iterations: time the W+K run as a whole)
        dt, its = t2 - t1, int(b["iters"].sum())
    return its / dt, nt, dt, its


def python_reference_baseline(workload):
    """SURVEY.md 8(d) lines (i)/(ii): the unmodified Python reference.  Live (3 Newton iterations of instance 0 of the workload, one
    core) when the reference tree is present; otherwise the measurement recorded in the build container."""
    rec = None
    try:
        rec = json.load(open(os.path.join(ROOT, "profiles", "r02_python_reference_cpu.json")))
    except Exception:
        pass
    out = {"unit": UNIT}
    key = "acro" if workload in ("acro", "single-acro") else "step"
    if rec is not None:
        w = rec["workloads"][key]
        out["recorded"] = {"one_core": w["one_core"], "all_cores": w["all_cores"], "machine": rec["machine"], "what": rec["what"],
                           "whole_solves_configs_1_2": rec.get("whole_solves_configs_1_2"),
                           "source": "profiles/r02_python_reference_cpu.json (oracle/time_python_reference.py; the reference tree does not travel to the GPU box)"}
    try:
        from oracle import pyref
        if pyref.available():
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            import time_python_reference as tpr
            done, dt = tpr.time_one((key, 0, 3))
            out["live"] = {"value": done / dt, "cores": 1, "iterations": done, "wall_s": dt,
                           "what": "unmodified reference at %s, NewtonMethod.optimize, 3 iterations of instance 0" % pyref.REFERENCE_ROOT}
    except Exception as e:  # never let the optional baseline break the bench line
        out["live_error"] = repr(e)[:200]
    src = out.get("live") or (out.get("recorded", {}).get("one_core"))
    if src:
        out["value"] = src["value"]
        out["cores"] = 1
        out["kind"] = "reference (live)" if "live" in out else "reference (recorded)"
    return out


def bind_to_gpu_numa_node(local):
    """Multi-GPU runs: keep this rank's threads (and with them the page-locked host buffers it allocates, which follow the allocating
    thread's NUMA policy) on the NUMA node its GPU hangs off, so that eight ranks do not push their results through one socket's
    memory controllers.  Best effort: returns a description of what was done, or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        bdf = pynvml.nvmlDeviceGetPciInfo(h).busId
        bdf = (bdf.decode() if isinstance(bdf, bytes) else bdf).lower()
        if len(bdf.split(":")[0]) == 8:
            bdf = bdf[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read().strip())
        if node < 0:
            return None
        cpus = []
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return {"gpu": local, "pci": bdf, "numa_node": node, "cpus": len(allowed)}
    except Exception:
        return None


def emit(line: dict):
    """Print the ONE JSON line on the process's original stdout."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = os.dup(1)

DUMP_SAMPLE = 512            # instances whose trajectories --dump-outputs writes: 512 x 8 x TT float64 = 33 MB
DUMP_MAX_BYTES = 64 << 20


def dump_sample(n):
    """The instances --dump-outputs writes: all of a small batch, else a fixed, seeded sample (sorted)."""
    if n <= DUMP_SAMPLE:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, DUMP_SAMPLE, replace=False))


def dump_outputs(d, arrays):
    """--dump-outputs: every array as d/<name>.npy, float32 kept, everything else as float64."""
    arrays = {k: np.ascontiguousarray(a, dtype=np.float32 if a.dtype == np.float32 else np.float64) for k, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise ValueError("--dump-outputs: %d bytes exceed the %d-byte budget" % (total, DUMP_MAX_BYTES))
    os.makedirs(d, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(d, k + ".npy"), a)


def dump_newton(d, bn, stats, idx):
    """What a caller of BatchedNewton.iterate receives after it: the newest iterate (xx, uu) and the per-instance statistics."""
    xx, uu = bn.iterate_at(0)
    dump_outputs(d, dict(xx=xx[idx], uu=uu[idx], **{k: v[idx] for k, v in stats.items()}))


def config_dict(args, n_per_gpu, world):
    names = {"step": "BASELINE.json configs[3]: batched step-maneuver Newton, randomised step references (zf~U(1.5,3.5), xf~U(14,18), seed 2024)",
             "acro": "BASELINE.json configs[4]: acrobatic Newton OCP batch (x0 perturbed, bump height zf~U(2.0,3.4), seed 7)"}
    return {"workload": names[args.workload],
            "instances_per_gpu": n_per_gpu, "instances_total": n_per_gpu * world, "TT": TT, "ns": 6, "ni": 2,
            "state_quant": args.state, "precision": args.precision,
            "state_storage": "float32 in HBM (lossless: quantised states are float32 values)" if (args.precision == "f64" and args.state == "f32" and args.x_storage == "auto") else
                             ("float32" if args.precision == "f32" else "float64"),
            "references": {"compact": "built on the device (acoc_set_refs_generated), kept parametric in HBM", "expanded": "built on the device, per-instance arrays",
                           "host": "per-instance arrays uploaded from the host"}[args.refs if args.precision == "f64" else ("expanded" if args.refs == "compact" else args.refs)],
            "armijo": args.armijo, "armijo_maxiters": 10, "max_iters": 200,
            "step": "one Newton iteration over the whole batch (iterations W..W+K-1 of the solve)",
            "l2": "working set per GPU (%.1f GB) >> 126 MB L2, no flush needed" % (n_per_gpu * 400e3 / 1e9),
            "parallelism": "instances sharded round-robin, %d per GPU, no hot-path collective" % n_per_gpu}


# =====================================================================================================================
# batched Newton workloads (configs 4 and 5)
# =====================================================================================================================
def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    sample = args.cpu_sample
    rate, nt, dt, its = cpu_port_rate(args.workload, sample, args.warmup, args.steps, args.state)
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / max(args.steps, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        # the configuration of our arm (the driver compares the two lines' config); what the CPU actually ran is the bounded sample below
        "data": "synthetic", "config": config_dict(args, args.instances, world),
        "sample": {"instances": sample, "newton_iterations": [args.warmup, args.warmup + args.steps - 1], "cpu_seconds": dt,
                   "note": "a throughput metric: the rate of the sample stands for the workload (instances are independent)"},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": nt, "kind": "port",
                         "sample": "%d instances x Newton iterations %d..%d of the workload, C port of the reference (oracle/acoc_oracle.c), "
                                   "OpenMP over instances; time(W+K iterations) - time(W iterations)" % (sample, args.warmup, args.warmup + args.steps - 1),
                         "python_reference": python_reference_baseline(args.workload)},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def roofline_tables(args, n, K, W, hist, phases, peaks, peak_src, fp64_peak, fused_fc):
    """Per-kernel accounting of the K profiled iterations.  Units come from the history of the profiled run: an instance is ACTIVE in
    iteration k iff it executed it (n_armijo[:, k] > 0); the sweeps process every lane of every tile (32 instances) that still holds
    an active instance."""
    steps_per = float(TT - 1)
    ncand = hist["n_armijo"][:, W:W + K]
    act = ncand > 0                                        # (N, K) instance executed iteration W+k
    pad = (-act.shape[0]) % 32
    act_t = np.pad(act, ((0, pad), (0, 0))).reshape(-1, 32, K)
    a_k = act.sum(0).astype(np.float64)                    # active instances per iteration
    lanes_k = act_t.any(1).sum(0).astype(np.float64) * 32  # lanes the tile-granular sweeps process per iteration
    fail = ncand > 1                                       # candidate 0 failed
    fail_k = fail.sum(0).astype(np.float64)
    fail_lanes_k = np.pad(fail, ((0, pad), (0, 0))).reshape(-1, 32, K).any(1).sum(0).astype(np.float64) * 32
    exact = (np.arange(W, W + K) > 8)                      # optcon.py:443
    # candidate rollouts executed after candidate 0 (lazy search: 1..9 at once in the exact-Hessian iterations; 1..3, then 4..9
    # where those failed too, in the Gauss-Newton iterations)
    if args.armijo == "lazy":
        roll_k = np.where(exact, 9.0 * fail_k, 3.0 * fail_k + 6.0 * (ncand > 4).sum(0))
        cand0_units = 0.0 if fused_fc else float(a_k.sum())
        upd_k = fail_k
        upd_lanes_k = fail_lanes_k
    else:
        roll_k = 10.0 * a_k
        cand0_units = 0.0
        upd_k = a_k
        upd_lanes_k = lanes_k
    MB = moved_bytes(args)
    x_float = args.precision == "f64" and args.state == "f32" and args.x_storage == "auto"
    fwd_alg = BYTES["forward"] + (BYTES["candidate_write"] if fused_fc else 0)
    fwd_flops = FLOPS["forward"] + (FLOPS["candidate"] if fused_fc else 0)
    # the fused forward + candidate-0 sweep does not write du and re-read it, reads u once, and fetches only V, theta, gamma of x
    fwd_moved = MB["forward"] + ((MB["candidate_write"] - (16 if args.precision == "f32" else 32) - (12 if x_float else 24)) if fused_fc else 0)
    kc, kc_src = kernel_counters()

    def counters(name):
        if not kc:
            return None
        return kc["kernels"].get(name)

    names = {"backward": "k_backward_tma" if not args.no_tma else "k_backward",
             "forward": ("k_forward_cand0_tma" if fused_fc else ("k_forward_tma" if not args.no_tma else "k_forward")),
             "candidates": "k_candidates", "update": "k_rollout_write_tma<.,1>" if not args.no_tma else "k_update"}
    # kernel names as launched (the counters file keeps the candidate stage under "k_candidates" whichever kernel ran it)
    shown = dict(names, candidates="k_candidates_list" if (args.armijo == "lazy" and not args.no_tma) else "k_candidates")
    units = {  # (useful instance-sweeps, processed lane-sweeps) over the K iterations
        "backward": (a_k.sum(), lanes_k.sum()), "forward": (a_k.sum(), lanes_k.sum()),
        "candidates": (roll_k.sum() + cand0_units, roll_k.sum() + cand0_units), "update": (upd_k.sum(), upd_lanes_k.sum())}
    alg_b = {"backward": BYTES["backward"], "forward": fwd_alg, "candidates": BYTES["candidate"], "update": BYTES["update"]}
    mov_b = {"backward": MB["backward"], "forward": fwd_moved, "candidates": MB["candidate"], "update": MB["update"]}
    alg_f = {"backward": FLOPS["backward"], "forward": fwd_flops, "candidates": FLOPS["candidate"], "update": FLOPS["update"]}
    bound = {"backward": "hbm", "forward": "hbm", "candidates": "fp64", "update": "hbm"}
    tbl = {}
    for k in ("backward", "forward", "candidates", "update"):
        ms = phases[k]
        useful, lanes = units[k]
        if ms <= 0 or useful <= 0:
            continue
        sec = ms * 1e-3
        e = {"kernel": shown[k], "bound": bound[k], "ms_per_iteration": ms / K, "instance_sweeps_useful": useful, "lane_sweeps_processed": lanes}
        c = counters(names[k])
        if c and c.get("fp64_inst_per_lane_step"):   # executed FP64-pipe instructions (ncu: sm__inst_executed_pipe_fp64 of this build)
            ex = c["fp64_inst_per_lane_step"] * lanes * steps_per
            e["fp64_executed_ginst_per_s"] = ex / sec / 1e9
            e["fp64_executed_frac"] = ex / sec / (fp64_peak * 1e12 / 2.0)
        if bound[k] == "hbm":
            gbs = useful * steps_per * alg_b[k] / sec / 1e9
            e.update({"hbm_gbs": gbs, "hbm_frac": gbs / peaks["hbm_gbs"],
                      "hbm_gbs_moved": lanes * steps_per * mov_b[k] / sec / 1e9})
            e["hbm_frac_moved"] = e["hbm_gbs_moved"] / peaks["hbm_gbs"]
        else:  # FP64-bound: the inputs of the 9 candidate rollouts of an instance are shared through L1, HBM is not the limiter
            e["fp64_algorithmic_tflops"] = useful * steps_per * alg_f[k] / sec / 1e12
        if c:
            e["ncu_dram_bytes_per_instance_step"] = c.get("dram_bytes_per_lane_step")
        tbl[k] = e
    tot_ms = sum(phases[k] for k in ("backward", "forward", "candidates", "update"))
    whole_b = sum(units[k][0] * steps_per * alg_b[k] for k in ("backward", "forward", "update"))
    tbl["whole_iteration"] = {"ms_per_iteration": tot_ms / K, "hbm_gbs": whole_b / (tot_ms * 1e-3) / 1e9,
                              "hbm_frac": whole_b / (tot_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                              "note": "bytes of the HBM-bound sweeps over the whole profiled time (candidates included in the time only)"}
    dom = max(("backward", "forward", "candidates", "update"), key=lambda k: phases[k])
    d = tbl[dom]
    c = counters(names[dom])
    n_launch_lanes = units[dom][1] / K
    traffic = c["dram_bytes_per_lane_step"] * n_launch_lanes * steps_per if c and c.get("dram_bytes_per_lane_step") else None
    alg_per_launch = units[dom][0] / K * steps_per * alg_b[dom]
    if bound[dom] == "hbm":
        achieved, peak, unit, frac = d["hbm_gbs"], peaks["hbm_gbs"], "GB/s", d["hbm_frac"]
    else:
        achieved, peak, unit = d.get("fp64_executed_ginst_per_s"), fp64_peak * 1e3 / 2.0, "G FP64-inst/s (thread-level)"
        frac = d.get("fp64_executed_frac")
    # the same fraction for ONE launch over a fully active batch, from the committed ncu capture of this build (duration under ncu:
    # serialised, cold cache); the window above also sweeps the finished lanes of live tiles, which lowers `frac`
    full_launch = None
    if c and c.get("duration_ms") and kc and bound[dom] == "hbm":
        fb = float(kc["instances"]) * (kc["TT"] - 1) * alg_b[dom]
        full_launch = {"instances": kc["instances"], "ms": c["duration_ms"], "algorithmic_bytes": fb, "achieved": fb / (c["duration_ms"] * 1e-3) / 1e9,
                       "frac": fb / (c["duration_ms"] * 1e-3) / 1e9 / peaks["hbm_gbs"], "traffic": c.get("dram_bytes"),
                       "source": "profiles/r02_kernel_counters.json (ncu --set full of this build; recorded, not re-measured in this run)"}
    roofline = {"kernel": shown[dom] + ("<EXACT>" if dom == "backward" and exact.any() else ""), "bound": "hbm" if bound[dom] == "hbm" else "fp64 (tensor cores unused by design)",
                "achieved": achieved, "peak": peak, "unit": unit, "frac": frac, "traffic": traffic, "traffic_source": kc_src,
                "algorithmic_bytes_per_launch": alg_per_launch, "peak_source": peak_src,
                "units": {"active_instances_per_iteration": a_k.tolist(), "lanes_processed_per_iteration": lanes_k.tolist(),
                          "failed_candidate0_per_iteration": fail_k.tolist(),
                          "note": "achieved = SURVEY.md 8(d) bytes x (TT-1) x ACTIVE instances of each profiled iteration / that kernel's summed "
                                  "time; the sweeps also process the finished lanes of live tiles (lanes_processed)"},
                "fp64": {"peak_tflops": fp64_peak, "peak_source": "DFMA microbenchmark run in this process (acoc_measure_fp64_peak)",
                         "executed_frac_dominant_kernel": d.get("fp64_executed_frac"),
                         "note": "executed FP64-pipe instructions per lane and step from the ncu capture of this build x lanes processed, against the "
                                 "measured DFMA issue rate; null when no capture of this build is committed"},
                "fully_active_launch": full_launch,
                "per_kernel": tbl, "share_of_step": phases[dom] / max(tot_ms, 1e-9),
                "algorithmic": {"bytes_per_instance_step": BYTES, "flops_per_instance_step": FLOPS, "note": "SURVEY.md 8(d) per-unit figures"},
                "moved": {"bytes_per_instance_step": dict(MB, forward_fused=fwd_moved),
                          "note": "bytes the kernels move in this mode (float32-valued states stored as float: -24 B per state access)"}}
    return roofline


def run_batched(args, rank, world, local):
    import aircraftoptimalcontrol_b200 as pkg
    from aircraftoptimalcontrol_b200 import _lib, dist as D

    dist = None
    numa = None
    if world > 1:
        numa = None if args.no_numa_bind else bind_to_gpu_numa_node(local)
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n = args.instances
    n_total = n * world
    K, W = args.steps, args.warmup

    xr, ur, dx0, (Q, R, QT), gen = make_problem(args.workload, n_total, (rank, world))
    kw = dict(TT=TT, device=local, state=args.state, armijo=args.armijo, precision=args.precision, x_storage=args.x_storage, tma=not args.no_tma,
              split=not args.no_split, fused=not args.no_fused)
    kw["refs_compact"] = args.refs != "expanded"
    bn = pkg.BatchedNewton(n, **kw)
    bn.set_weights(Q, R, QT)
    if args.refs == "host":
        bn.set_refs(xr, ur)                  # per-instance arrays uploaded from the host
    elif gen[0] == "step":
        bn.set_refs_step(gen[1], gen[2])     # the scripts' generators on the device (bit-identical references)
    else:
        bn.set_refs_acrobatic(gen[1])
    bn.init_guess(dx0=dx0)
    if W:
        bn.iterate(W, count_active=False)
    bn.sync()

    state = {"bn_open": True}

    def barrier():
        if dist is not None:
            dist.barrier()
        if state["bn_open"]:
            bn.sync()

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()  # keeps sampling through the timed region, the per-phase re-run and the end-to-end solves
    its_before = int(bn.stats()["iters"].astype(np.int64).sum())
    barrier()
    bn.iterate(K, count_active=False)  # K Newton iterations, timed by CUDA events inside the library
    bn.sync()
    barrier()
    tm = bn.timing()
    ms = tm["total_ms"]
    launches = tm["launches"]
    st = bn.stats()
    if args.dump_outputs and rank == 0:
        dump_newton(args.dump_outputs, bn, st, dump_sample(n))
    its_done = int(st["iters"].astype(np.int64).sum()) - its_before  # instance-iterations actually executed in the timed region
    if dist is not None:
        import torch
        t = torch.tensor([ms, float(launches), float(its_done)], dtype=torch.float64, device="cuda")
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        ms, launches, its_done = float(tmax[0]), int(t[1]), int(t[2])
    n_active = int((st["status"] == 0).sum())
    value = its_done / (ms * 1e-3)   # = instances x K while every instance is still iterating

    # ---- roofline (rank 0): the same iterations re-run with per-phase events (one stream, no tile ranges) ------------
    roofline = fp64 = phases = None
    peaks, peak_src = load_peaks()
    if rank == 0 and not args.no_roofline:
        bn.set_profiling(True)
        bn.init_guess(dx0=dx0)
        bn.iterate(W, count_active=False)
        bn.iterate(K, count_active=False)
        tp = bn.timing()
        bn.set_profiling(False)
        phases = tp["phases"]
        fp64_peak = _lib.measure_fp64_peak(local)
        fused_fc = args.armijo == "lazy" and not args.no_tma and not args.no_fused
        roofline = roofline_tables(args, n, K, W, bn.history(), phases, peaks, peak_src, fp64_peak, fused_fc)
        fp64 = {"peak_tflops_measured": fp64_peak, "dependent_dfma_latency_cycles": _lib.measure_fp64_latency(local)}

    # ---- whole solve, device-resident (every instance to the reference's criterion; includes the float32-noise phase
    #      with its full Armijo searches and the thinning tail) ------------------------------------------------------
    bn.init_guess(dx0=dx0)
    bn.solve()  # untimed: the first solve allocates the survivor-generation contexts (cudaMalloc inside the timed span otherwise)
    bn.init_guess(dx0=dx0)
    tot_solve = bn.solve()
    tsolve = bn.timing()
    whole = {"value": tot_solve / (tsolve["total_ms"] * 1e-3), "unit": UNIT, "device_ms": tsolve["total_ms"], "total_newton_iterations": int(tot_solve),
             "lockstep_iterations": int(bn.stats()["iters"].max()), "gpu_launches": tsolve["launches"],
             "survivor_generation_moves_ms": tsolve["phases"]["select"], "scope": "this rank"}

    device_bytes = bn.device_bytes
    bn.close()  # the end-to-end legs below build their own contexts: release this one (and its survivor generations) first
    state["bn_open"] = False

    # ---- end to end through the public API, host buffers, full solve -----------------------------------------
    e2e = e2e_host = None
    if not args.no_e2e:
        import torch
        if dist is not None:  # warm the communicator the statistics gather uses (its first collective builds the NCCL channels)
            D.gather_stats({"iters": np.zeros(n, dtype=np.int32), "status": np.zeros(n, dtype=np.int32), "J": np.zeros(n), "descent": np.zeros(n),
                            "n_reg": np.zeros(n, dtype=np.int32)}, n_total)
        pn = pkg.PipelinedNewton(n, n_chunks=args.chunks_generated, stagger=not args.no_stagger, **kw)
        pn.set_weights(Q, R, QT)

        def timed(solve):
            solve()          # untimed warm-up of the whole path
            barrier()
            t0 = time.perf_counter()
            st2 = solve()
            barrier()
            wall = time.perf_counter() - t0
            t1 = time.perf_counter()
            g = D.gather_stats(st2, n_total)   # NCCL all_gather of the per-instance statistics (off the hot path), timed alone
            gather_s = time.perf_counter() - t1
            if dist is not None:
                tw = torch.tensor([wall], dtype=torch.float64, device="cuda")
                dist.all_reduce(tw, op=dist.ReduceOp.MAX)
                wall = float(tw[0])
            return wall, g, gather_s

        def describe(wall, g, gather_s, h2d, d2h, what, chunks):
            tot = int(g["iters"].sum())
            steps_e2e = int(g["iters"].max())
            return {"value": tot / wall, "unit": UNIT, "h2d_bytes_per_step": h2d / max(steps_e2e, 1), "d2h_bytes_per_step": d2h / max(steps_e2e, 1),
                    "h2d_bytes_per_solve": h2d, "d2h_bytes_per_solve": d2h,
                    "wall_s": wall, "total_newton_iterations": tot, "solver_steps": steps_e2e,
                    "converged": int((g["status"] == 1).sum()), "instances": n_total, "mean_iters": float(g["iters"].mean()),
                    "stats_gather_s": gather_s, "chunks": chunks, "staggered_priorities": not args.no_stagger, "what": what}

        # (a) headline: the randomisation parameters are the host inputs (16-56 B per instance); the scripts' reference generators run on
        #     the device (bit-identical arrays, tests/test_gpu_parity_r2.py); states come back as the float32 values they are
        f32_dl = args.precision == "f64" and args.state == "f32" and args.x_storage == "auto"
        par_t = [pinned_like(np.asarray(p, dtype=np.float64)) for p in gen[1:]]
        dx0_t = pinned_like(dx0) if dx0 is not None else None
        xs32_t = torch.empty((n, 6, TT), dtype=torch.float32 if f32_dl else torch.float64, pin_memory=True)
        us_t = torch.empty((n, 2, TT), dtype=torch.float64, pin_memory=True)
        refs = (gen[0],) + tuple(p.numpy() for p in par_t)

        def solve_generated():
            return pn.solve(refs=refs, dx0=None if dx0_t is None else dx0_t.numpy(), out=(xs32_t.numpy(), us_t.numpy()),
                            x_dtype=np.float32 if f32_dl else np.float64)[2]

        wall, g, gs = timed(solve_generated)
        h2d = (sum(p.numel() for p in par_t) * 8 + (dx0_t.numel() * 8 if dx0_t is not None else 0) + 3 * TT * 8 * args.chunks_generated) * world
        d2h = (xs32_t.numel() * xs32_t.element_size() + us_t.numel() * 8 + (n * 48 if f32_dl else 0)) * world + n_total * 28
        e2e = describe(wall, g, gs, h2d, d2h,
                       "PipelinedNewton.solve(refs=(kind, per-instance parameters) in pinned host memory): per sub-batch H2D of the parameters -> "
                       "reference generators + initial guess on the device -> solve() to descent >= -1e-6 -> D2H of xx_star (%s), uu_star "
                       "(float64) straight into the pinned host arrays by the delivery kernel (finished instances while the survivor generations "
                       "still iterate), statistics"
                       % ("float32: lossless, the quantised states are float32 values" if f32_dl else "float64"), args.chunks_generated)
        del xs32_t
        pn.close()
        # (b) the same solve with the reference ARRAYS uploaded from the host and float64 results (the round-1 path, still available)
        if not args.no_e2e_host:
            pn = pkg.PipelinedNewton(n, n_chunks=args.chunks, stagger=not args.no_stagger, **kw)
            pn.set_weights(Q, R, QT)
            xr_p, ur_p = pinned_like(xr), pinned_like(ur)
            xs_t = torch.empty((n, 6, TT), dtype=torch.float64, pin_memory=True)

            def solve_host():
                return pn.solve(xr_p.numpy(), ur_p.numpy(), dx0=dx0, out=(xs_t.numpy(), us_t.numpy()))[2]

            wall, g, gs = timed(solve_host)
            e2e_host = describe(wall, g, gs, (xr.nbytes + ur.nbytes) * world, (xs_t.numel() + us_t.numel()) * 8 * world + n_total * 28,
                                "PipelinedNewton.solve(xx_ref, uu_ref in pinned host memory): per sub-batch set_refs (H2D of 64 KB per instance) -> "
                                "init_guess (device) -> solve() -> result()/stats() (D2H, float64)", args.chunks)
            pn.close()

    clocks = sampler.summary() if sampler else None
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        rate, nt, dt, its = cpu_port_rate(args.workload, args.cpu_sample, W, K, args.state)
        cpu = {"value": rate, "unit": UNIT, "cores": nt, "kind": "port",
               "sample": "%d instances x Newton iterations %d..%d of the same workload, C port of the reference (oracle/acoc_oracle.c), OpenMP over "
                         "instances, %.1f s" % (args.cpu_sample, W, W + K - 1, dt),
               "python_reference": python_reference_baseline(args.workload)}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / max(K, 1),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
                "config": config_dict(args, n, world), "clocks": clocks, "e2e": e2e, "e2e_host_refs": e2e_host, "gpu_launches": launches,
                "active_after_timed_region": n_active, "instance_iterations_timed": its_done, "whole_solve": whole, "roofline": roofline, "fp64": fp64,
                "phase_ms": phases, "cpu_baseline": cpu, "device": pkg.device_info(local)["name"], "device_bytes": device_bytes, "numa_binding_rank0": numa}
        emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


# =====================================================================================================================
# config 3: lqr_tracking of the saved optimum from 4096 perturbed initial states
# =====================================================================================================================
TRACK_UNIT = "rollout-steps/s"


def track_inputs(n):
    from aircraftoptimalcontrol_b200 import refgen
    d = np.load(os.path.join(ROOT, "tests", "golden", "lqr_tracking.npz"))   # Data/xx_star.npy, uu_star.npy of the reference (inputs)
    return d["xx_opt"], d["uu_opt"], refgen.config3_deltas(n), (d["Q"], d["R"], d["QT"])


def track_config(n):
    return {"workload": "BASELINE.json configs[2]: lqr_tracking.py LQR tracking of Data/xx_star.npy with %d perturbed initial states (instance 0: "
                        "delta = 0.1, the rest U(-0.1,0.1)^6, seed 1234)" % n,
            "instances_per_gpu": n, "TT": TT, "step": "one lqr_tracking_batch call: linearise along the nominal (TT points), ONE shared LQ solve, "
            "%d closed-loop rollouts of %d steps" % (n, TT - 1), "l2": "outputs (%.0f MB) exceed the 126 MB L2; the shared gains are L1/L2 resident by design" % (n * 64e3 / 1e6)}


def run_track(args, rank, world, local):
    import aircraftoptimalcontrol_b200 as pkg
    from aircraftoptimalcontrol_b200 import _lib
    from aircraftoptimalcontrol_b200.aircraft_simplified import Dynamics
    from aircraftoptimalcontrol_b200.lqr_tracking import lqr_tracking_batch
    import ctypes as C
    n = args.instances if args.instances_given else 4096
    K, W = args.steps, max(args.warmup, 3)
    xo, uo, deltas, (Q, R, QT) = track_inputs(n * world)
    deltas = np.ascontiguousarray(deltas[rank::world])
    dyn = Dynamics(device=local)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ms3 = (C.c_double * 3)()
    dev, walls = [], []
    for k in range(W + K):
        t0 = time.perf_counter()
        xx_reg, uu_reg = lqr_tracking_batch(xo, uo, deltas, dyn=dyn, QQt=Q, RRt=R, QQT=QT)
        t1 = time.perf_counter()
        _lib.check(_lib.lib().acoc_last_pointwise_timing(C.addressof(ms3)))
        if k >= W:
            dev.append((ms3[0], ms3[1], ms3[2]))
            walls.append(t1 - t0)
    if args.dump_outputs and rank == 0:
        idx = dump_sample(n)
        dump_outputs(args.dump_outputs, dict(xx=xx_reg[idx], uu=uu_reg[idx]))
    dev = np.array(dev)
    units = n * (TT - 1)
    ms = float(dev[:, 0].mean())
    wall = float(np.mean(walls))
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        t = torch.tensor([ms, wall], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, wall = float(t[0]), float(t[1])
    peaks, peak_src = load_peaks()
    trk_ms, lq_ms = float(dev[:, 2].mean()), float(dev[:, 1].mean())
    out_bytes = units * 64.0   # x_t (float64 here) and u_t written once; the shared K_t, x_opt, u_opt stay in L1/L2
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = track_cpu(n, args.state)
    if rank == 0:
        line = {"metric": "closed_loop_rollout_steps_per_second", "value": units * world / (ms * 1e-3), "unit": TRACK_UNIT, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": track_config(n), "clocks": sampler.summary() if sampler else None,
                "e2e": {"value": units * world / wall, "unit": TRACK_UNIT, "h2d_bytes_per_step": float(deltas.nbytes + xo.nbytes + uo.nbytes + 76 * 8),
                        "d2h_bytes_per_step": float(n * 8 * TT * 8), "wall_s": wall,
                        "what": "lqr_tracking_batch(xx_opt, uu_opt, delta) through the C ABI (acoc_lqr_tracking) with host numpy buffers"},
                "gpu_launches": 3 * K,
                "phase_ms": {"linearise_and_shared_lq_solve": lq_ms, "closed_loop_rollouts": trk_ms},
                "roofline": {"kernel": "k_track", "bound": "hbm", "achieved": out_bytes / (trk_ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                             "frac": out_bytes / (trk_ms * 1e-3) / 1e9 / peaks["hbm_gbs"], "traffic": None, "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": out_bytes,
                             "note": "latency-bound by construction: %d instances are %d warps on 148 SMs, each walking 999 dependent steps (about 1 us per "
                                     "step); the shared LQ solve is ONE thread's literal dense recursion (lqr_tracking.py:276).  The roofline "
                                     "fraction says how far such a small batch is from bandwidth, not kernel quality" % (n, (n + 31) // 32),
                             "share_of_step": trk_ms / max(ms, 1e-9)},
                "cpu_baseline": cpu, "device": pkg.device_info(local)["name"]}
        emit(line)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


def track_cpu(n, state):
    from oracle import corcl
    corcl.build()
    xo, uo, deltas, (Q, R, QT) = track_inputs(n)
    nt = host_threads()
    corcl.lqr_tracking(xo, uo, Q, R, QT, deltas[:nt], quant_f32=(state == "f32"), n_threads=nt)
    t0 = time.perf_counter()
    corcl.lqr_tracking(xo, uo, Q, R, QT, deltas, quant_f32=(state == "f32"), n_threads=nt)
    dt = time.perf_counter() - t0
    return {"value": n * (TT - 1) / dt, "unit": TRACK_UNIT, "cores": nt, "kind": "port",
            "sample": "the whole workload (%d instances) with the C port of the reference (oracle/acoc_oracle.c), OpenMP over instances, %.2f s; the Python "
                      "reference needs 1.43 s for ONE instance (SURVEY.md 8(a) a9)" % (n, dt)}


def run_track_reference(args, rank):
    if rank != 0:
        return
    n = args.instances if args.instances_given else 4096
    c = track_cpu(n, args.state)
    emit({"impl": "reference", "metric": "closed_loop_rollout_steps_per_second", "value": c["value"], "unit": TRACK_UNIT, "n_gpus": args.gpus, "steps": args.steps,
          "warmup": args.warmup, "ms_per_step": 1e3 * n * (TT - 1) / c["value"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
          "data": "synthetic", "config": track_config(n), "cpu_baseline": c,
          "e2e": {"value": c["value"], "unit": TRACK_UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0})


# =====================================================================================================================
# configs 1 and 2: one trajectory (latency)
# =====================================================================================================================
def single_inputs(workload):
    d = np.load(os.path.join(ROOT, "tests", "golden", "newton_step_f32.npz" if workload == "single-step" else "newton_acro_f32.npz"))
    return d


def single_steps(args, d):
    """--steps of a single-trajectory workload: the timed iterations have to end before the trajectory converges."""
    k_max = int(d["iters"]) - args.warmup - 1
    if args.steps > k_max:
        sys.exit("--workload %s converges after %d Newton iterations: with --warmup %d at most %d steps can be timed"
                 % (args.workload, int(d["iters"]), args.warmup, k_max))
    return args.steps


def single_config(workload):
    return {"workload": ("BASELINE.json configs[0]: main_newton_method.py step maneuver, single trajectory" if workload == "single-step" else
                         "BASELINE.json configs[1]: acrobatic_newton.py acrobatic maneuver, single trajectory"),
            "instances_per_gpu": 1, "TT": TT, "inputs": "xx_ref, uu_ref, xx_init, uu_init of the live reference run (tests/golden/*.npz)",
            "step": "one Newton iteration of the single trajectory (iterations W..W+K-1)", "l2": "working set 0.4 MB: L2-resident by nature of the configuration"}


def run_single(args, rank, world, local):
    import aircraftoptimalcontrol_b200 as pkg
    if rank != 0:   # a single trajectory does not shard: replicas would only repeat rank 0
        return
    d = single_inputs(args.workload)
    K, W = single_steps(args, d), args.warmup
    iters_ref = int(d["iters"])
    sampler = ClockSampler(local)
    sampler.start()
    with pkg.BatchedNewton(1, TT=TT, device=local, state=args.state, refs_shared=True, armijo=args.armijo, precision=args.precision) as bn:
        bn.set_weights(d["Q"], d["R"], d["QT"])
        bn.set_refs(d["xx_ref"], d["uu_ref"])
        bn.set_init(d["xx_init"][None], d["uu_init"][None])
        bn.iterate(W, count_active=False)
        bn.iterate(K, count_active=False)
        tm = bn.timing()
        ms, launches = tm["total_ms"], tm["launches"]
        if args.dump_outputs:
            dump_newton(args.dump_outputs, bn, bn.stats(), dump_sample(1))
        solves = []
        for _ in range(3):
            bn.set_init(d["xx_init"][None], d["uu_init"][None])
            tot = bn.solve()
            solves.append(bn.timing()["total_ms"])
        # end to end through the drop-in signature: host arrays in, optimize()'s result out
        walls = []
        for _ in range(3):
            t0 = time.perf_counter()
            bn.set_refs(d["xx_ref"], d["uu_ref"])
            bn.set_init(d["xx_init"][None], d["uu_init"][None])
            tot = bn.solve()
            bn.result()
            walls.append(time.perf_counter() - t0)
    cpu = None
    if not args.no_cpu:
        cpu = single_cpu(args.workload, W, K, args.state)
    peaks, peak_src = load_peaks()
    per_it = ms / K
    line = {"metric": METRIC, "value": K / (ms * 1e-3), "unit": UNIT, "n_gpus": 1, "steps": K, "warmup": W, "ms_per_step": per_it, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": args.precision, "data": "synthetic", "config": single_config(args.workload),
            "clocks": sampler.summary(),
            "e2e": {"value": tot / min(walls), "unit": UNIT, "h2d_bytes_per_step": float(2 * 8 * 8 * TT) / tot, "d2h_bytes_per_step": float(8 * 8 * TT) / tot,
                    "wall_s": min(walls), "total_newton_iterations": int(tot),
                    "what": "set_refs + set_init (H2D) -> solve() to descent >= -1e-6 -> result() (D2H), host numpy buffers, best of 3"},
            "gpu_launches": launches,
            "whole_solve": {"device_ms": min(solves), "total_newton_iterations": int(tot), "reference_iterations": iters_ref, "value": tot / (min(solves) * 1e-3), "unit": UNIT},
            "roofline": {"kernel": "k_backward_cols + k_search_fused (12 warp roles / 12 warps per tile)", "bound": "hbm",
                         "achieved": (TT - 1) * (BYTES["backward"] + BYTES["forward"] + 11 * BYTES["candidate"]) / (per_it * 1e-3) / 1e9,
                         "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": (TT - 1) * (BYTES["backward"] + BYTES["forward"] + 11 * BYTES["candidate"]) / (per_it * 1e-3) / 1e9 / peaks["hbm_gbs"],
                         "traffic": None, "peak_source": peak_src,
                         "note": "one trajectory is one lane of every warp role: the iteration is two dependent sweeps of 999 sequential steps, i.e. pure "
                                 "arithmetic latency (%.2f us per backward+search step pair); no roofline is within reach of a single trajectory" % (per_it * 1e3 / (TT - 1))},
            "cpu_baseline": cpu, "device": pkg.device_info(local)["name"]}
    emit(line)


def single_cpu(workload, W, K, state):
    from oracle import corcl
    corcl.build()
    d = single_inputs(workload)
    a = (d["xx_ref"], d["uu_ref"], d["xx_init"], d["uu_init"], d["Q"], d["R"], d["QT"])
    corcl.newton(*a, quant_f32=(state == "f32"), n_iters_cap=1)
    t0 = time.perf_counter()
    if W:
        corcl.newton(*a, quant_f32=(state == "f32"), n_iters_cap=W)
    t1 = time.perf_counter()
    corcl.newton(*a, quant_f32=(state == "f32"), n_iters_cap=W + K)
    t2 = time.perf_counter()
    dt = (t2 - t1) - (t1 - t0 if W else 0.0)
    return {"value": K / dt, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": "Newton iterations %d..%d of the same trajectory, C port of the reference (oracle/acoc_oracle.c), one thread, %.3f s" % (W, W + K - 1, dt),
            "python_reference": python_reference_baseline(workload)}


def run_single_reference(args, rank):
    if rank != 0:
        return
    d = single_inputs(args.workload)
    K = single_steps(args, d)
    c = single_cpu(args.workload, args.warmup, K, args.state)
    emit({"impl": "reference", "metric": METRIC, "value": c["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": K, "warmup": args.warmup,
          "ms_per_step": 1e3 / c["value"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
          "config": single_config(args.workload), "cpu_baseline": c,
          "e2e": {"value": c["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0})


def main():
    os.dup2(2, 1)  # anything native code prints to fd 1 (e.g. the NCCL version banner) lands on stderr
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--instances", type=int, default=None, help="instances per GPU (default 65536; 4096 for --workload track)")
    ap.add_argument("--workload", default="step", choices=["step", "acro", "track", "single-step", "single-acro"])
    ap.add_argument("--armijo", default="lazy", choices=["lazy", "speculative"])
    ap.add_argument("--state", default="f32", choices=["f32", "f64"])
    ap.add_argument("--precision", default="f64", choices=["f64", "f32"], help="f64 = the parity path (default); f32 = the optional FP32 mode")
    ap.add_argument("--x-storage", default="auto", choices=["auto", "f64"], help="f64: keep float32-valued states in float64 buffers (A/B)")
    ap.add_argument("--refs", default="compact", choices=["compact", "expanded", "host"],
                    help="references of the batched workloads: built on the device and kept parametric (default), built on the device and written "
                         "out as per-instance arrays, or per-instance arrays uploaded from the host (A/B; identical results)")
    ap.add_argument("--no-tma", action="store_true", help="plain-load sweeps instead of the TMA rings (A/B)")
    ap.add_argument("--no-split", action="store_true", help="one stream for the whole batch instead of the tile-range sweep (A/B)")
    ap.add_argument("--no-fused", action="store_true", help="separate LQ forward pass / candidate sweeps instead of the fused ones (A/B)")
    ap.add_argument("--cpu-sample", type=int, default=16384, help="instances of the bounded CPU sample (about 10 s of work on 16 host threads)")
    ap.add_argument("--chunks", type=int, default=4, help="sub-batches of the pipelined end-to-end solve with reference arrays uploaded from the host")
    ap.add_argument("--chunks-generated", type=int, default=None, help="sub-batches of the headline end-to-end solve (references generated on the device: "
                    "little to upload, so fewer, larger sub-batches win on one GPU -- 1: 0.322 s, 2: 0.325 s, 4: 0.338 s, 8: 0.345 s; with 8 GPUs "
                    "sharing the host 4 is best -- 2: 0.500 s, 4: 0.490 s, 8: 0.514 s); default 1, or 4 from four GPUs on")
    ap.add_argument("--no-stagger", action="store_true", help="end-to-end leg: same stream priority for every sub-batch (A/B)")
    ap.add_argument("--no-numa-bind", action="store_true", help="multi-GPU: do not bind the rank to its GPU's NUMA node (A/B)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-e2e-host", action="store_true", help="skip the second end-to-end leg (reference arrays uploaded from the host)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (rank 0; trajectories of a fixed, seeded "
                         "sample of %d instances, float64) so that two builds can be compared output for output" % DUMP_SAMPLE)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of our arm; the reference arm has none to write")
    args.warmup = max(args.warmup, 0)
    if args.workload != "track" and args.warmup + args.steps > 199:
        ap.error("--warmup + --steps must not exceed 199, the Newton iterations optimize() runs at most (max_iters - 1, optcon.py:415)")
    args.instances_given = args.instances is not None
    if args.chunks_generated is None:
        args.chunks_generated = 4 if int(os.environ.get("WORLD_SIZE", "1")) >= 4 else 1
    if args.instances is None:
        args.instances = 65536

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.workload == "track":
        return run_track_reference(args, rank) if args.impl == "reference" else run_track(args, rank, world, local)
    if args.workload.startswith("single"):
        return run_single_reference(args, rank) if args.impl == "reference" else run_single(args, rank, world, local)
    if args.impl == "reference":
        return run_reference_arm(args, rank, world)
    run_batched(args, rank, world, local)


if __name__ == "__main__":
    main()
