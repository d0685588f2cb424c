"""ctypes binding of libacoc.so (include/acoc.h).  No fallback: if the library is missing or no CUDA
device is usable every call raises -- the product never computes on the CPU."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ACOC_LIB", os.path.join(_HERE, "libacoc.so"))  # ACOC_LIB: tuning experiments only
_lib = None

DEFAULT_PARAMS = (0.1716, 2.395, 3.256, 12.0, 9.81, 0.61, 1.2, 0.24, 1e-3)  # aircraft_simplified.py:108-118

STATE_F64 = 1
REFS_SHARED = 2
ARMIJO_LAZY = 4
SOLVE_IN_PLACE = 8
FP32 = 16
X_F64 = 32
NO_TMA = 64
NO_SPLIT = 128
NO_FUSED = 256
REFS_EXPANDED = 512
METHOD_NEWTON, METHOD_GRADIENT = 0, 1
PRIORITY_SHIFT = 16

INST_ACTIVE, INST_CONVERGED, INST_MAXITER, INST_NONFINITE = 0, 1, 2, 3


class AcocError(RuntimeError):
    """A libacoc call returned a negative status."""


class NewtonOptions(C.Structure):
    _fields_ = [("max_iters", C.c_int), ("armijo_maxiters", C.c_int), ("exact_after", C.c_int), ("method", C.c_int),
                ("stepsize_0", C.c_double), ("cc", C.c_double), ("beta", C.c_double), ("term_cond", C.c_double)]


class TrackMcOut(C.Structure):
    """acoc_track_mc_out: output addresses (0 = not wanted)."""
    _fields_ = [("err_max", C.c_void_p), ("err_final", C.c_void_p), ("worst_max", C.c_void_p), ("mean_final", C.c_void_p),
                ("n_within", C.c_void_p), ("n_reg", C.c_void_p)]


class VjpOut(C.Structure):
    """acoc_vjp_out: output addresses (0 = not wanted)."""
    _fields_ = [("xref_bar", C.c_void_p), ("uref_bar", C.c_void_p), ("x0_bar", C.c_void_p), ("zf_bar", C.c_void_p),
                ("vx_bar", C.c_void_p), ("n_indef", C.c_void_p)]


_dp = C.c_void_p  # double* / int* passed as raw addresses


def _sig(lib):
    i, d, vp = C.c_int, C.c_double, C.c_void_p
    lib.acoc_version.restype = i
    lib.acoc_last_error.restype = C.c_char_p
    table = {
        "acoc_device_count": [vp],
        "acoc_device_info": [i, vp, i, vp, vp, vp],
        "acoc_step_batch": [i, i, vp, i, vp, vp, vp, vp, vp, vp, vp, vp],
        "acoc_cost_batch": [i, i, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp],
        "acoc_ltv_lqr": [i, i, i] + [vp] * 15,
        "acoc_lqr_tracking": [i, i, i, vp, i] + [vp] * 9,
        "acoc_last_pointwise_timing": [vp],
        "acoc_ctx_create": [i, i, i, C.c_uint, vp],
        "acoc_ctx_destroy": [vp],
        "acoc_ctx_device_bytes": [vp, vp],
        "acoc_set_model": [vp, vp],
        "acoc_set_weights": [vp, vp, vp, vp],
        "acoc_set_options": [vp, vp],
        "acoc_set_refs": [vp, vp, vp],
        "acoc_set_refs_generated": [vp] * 8,
        "acoc_get_refs": [vp, vp, vp],
        "acoc_get_result_f32": [vp, vp, vp, vp],
        "acoc_set_init": [vp, vp, vp],
        "acoc_init_guess": [vp, d, d, vp],
        "acoc_newton_iterate": [vp, i, vp],
        "acoc_newton_solve": [vp, vp],
        "acoc_newton_solve_deliver": [vp, vp, i, vp, vp, vp],
        "acoc_sync": [vp],
        "acoc_get_result": [vp, vp, vp],
        "acoc_get_iterate": [vp, i, vp, vp],
        "acoc_get_deltau": [vp, vp],
        "acoc_get_gains": [vp, vp, vp],
        "acoc_get_history": [vp, vp, vp, vp, vp],
        "acoc_get_stats": [vp, vp, vp, vp, vp, vp],
        "acoc_track": [vp] * 8,
        "acoc_get_tracked": [vp, vp, vp],
        "acoc_get_track_gains": [vp, vp],
        "acoc_get_track_timing": [vp, vp],
        "acoc_lqr_tracking_many": [i, i, i, vp, i] + [vp] * 9,
        "acoc_track_mc": [vp] * 4 + [i, vp, i, vp, vp],
        "acoc_lqr_tracking_mc": [i, i, i, i, vp, i] + [vp] * 6 + [i, vp, vp],
        "acoc_eval_cost": [vp, vp],
        "acoc_set_deltau": [vp, vp],
        "acoc_set_scalars": [vp, vp, vp],
        "acoc_backward": [vp, i],
        "acoc_forward": [vp, vp],
        "acoc_armijo": [vp, vp, vp],
        "acoc_gradient": [vp, vp],
        "acoc_armijo_sweep": [vp, i, vp, vp],
        "acoc_update": [vp, vp],
        "acoc_get_timing": [vp, vp, vp, vp],
        "acoc_set_profiling": [vp, i],
        "acoc_measure_fp64_peak": [i, vp],
        "acoc_measure_copy_bw": [i, vp],
        "acoc_measure_fp64_latency": [i, vp],
        "acoc_set_refs_dev": [vp] * 4,
        "acoc_set_init_dev": [vp] * 4,
        "acoc_get_result_dev": [vp, vp, i, vp, vp, vp],
        "acoc_get_tracked_dev": [vp] * 4,
        "acoc_get_track_gains_dev": [vp] * 3,
        "acoc_track_mc_dev": [vp] * 4 + [i, vp, i, vp, vp, vp],
        "acoc_result_vjp": [vp] * 4,
        "acoc_result_vjp_dev": [vp] * 5,
    }
    for name, args in table.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = i
    return table


EXPORTS = None


def lib():
    """The loaded library.  Raises if libacoc.so has not been built (python __graft_entry__.py / build.py)."""
    global _lib, EXPORTS
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise AcocError("libacoc.so not found at %s -- build it with `python -m aircraftoptimalcontrol_b200.build`; "
                            "there is no CPU fallback" % LIB_PATH)
        _lib = C.CDLL(LIB_PATH)
        EXPORTS = _sig(_lib)
    return _lib


def check(rc: int):
    if rc != 0:
        msg = lib().acoc_last_error()
        raise AcocError("libacoc error %d: %s" % (rc, msg.decode() if msg else "?"))


def ptr(a):
    """Address of a C-contiguous numpy array (or None)."""
    if a is None:
        return None
    if not a.flags["C_CONTIGUOUS"]:
        raise ValueError("array must be C-contiguous")
    return a.ctypes.data


def out_array(a, shape, dtypes, name="out"):
    """Validate a caller-supplied OUTPUT array before its address crosses the C boundary (the library writes prod(shape) elements of
    the dtype it was told, whatever the array really is): numpy array, exact shape, one of `dtypes`, C-contiguous, writeable."""
    dtypes = tuple(np.dtype(d) for d in (dtypes if isinstance(dtypes, (tuple, list)) else (dtypes,)))
    if not isinstance(a, np.ndarray):
        raise ValueError("%s must be a numpy array" % name)
    if tuple(a.shape) != tuple(shape):
        raise ValueError("%s has shape %s, expected %s" % (name, a.shape, tuple(shape)))
    if a.dtype not in dtypes:
        raise ValueError("%s has dtype %s, expected %s" % (name, a.dtype, " or ".join(str(d) for d in dtypes)))
    if not a.flags["C_CONTIGUOUS"] or not a.flags["WRITEABLE"]:
        raise ValueError("%s must be C-contiguous and writeable" % name)
    return a


def dev_tensor(t, device, shape, dtype, name="tensor"):
    """Address of a caller's CUDA tensor before it crosses the C boundary of a _dev entry point (the library reads or writes
    prod(shape) elements of `dtype` there): a torch.Tensor of `dtype` with exactly `shape`, contiguous, on cuda:`device`."""
    import torch
    if not isinstance(t, torch.Tensor):
        raise ValueError("%s must be a torch.Tensor, got %s" % (name, type(t).__name__))
    if t.dtype != dtype:
        raise ValueError("%s has dtype %s, expected %s" % (name, t.dtype, dtype))
    if tuple(t.shape) != tuple(shape):
        raise ValueError("%s has shape %s, expected %s" % (name, tuple(t.shape), tuple(shape)))
    if not t.is_contiguous():
        raise ValueError("%s must be contiguous" % name)
    if not t.is_cuda or t.device.index != device:
        raise ValueError("%s is on %s, expected cuda:%d" % (name, t.device, device))
    return t.data_ptr()


def dev_stream(device):
    """The current torch stream of cuda:`device` as the stream argument of a _dev entry point."""
    import torch
    return torch.cuda.current_stream(device).cuda_stream


def f64(a, shape=None, name="array"):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None and tuple(a.shape) != tuple(shape):
        raise ValueError("%s has shape %s, expected %s" % (name, a.shape, tuple(shape)))
    return a


def device_count() -> int:
    n = C.c_int(0)
    rc = lib().acoc_device_count(C.addressof(n))
    return n.value if rc == 0 else 0


def device_info(device=0):
    name = C.create_string_buffer(128)
    sm, cc = C.c_int(0), C.c_int(0)
    mem = C.c_ulonglong(0)
    check(lib().acoc_device_info(device, C.addressof(name), 128, C.addressof(sm), C.addressof(mem), C.addressof(cc)))
    return dict(name=name.value.decode(), sm_count=sm.value, mem_bytes=mem.value, cc=cc.value)


def measure_fp64_peak(device=0) -> float:
    v = C.c_double(0)
    check(lib().acoc_measure_fp64_peak(device, C.addressof(v)))
    return v.value


def measure_fp64_latency(device=0) -> float:
    v = C.c_double(0)
    check(lib().acoc_measure_fp64_latency(device, C.addressof(v)))
    return v.value


def measure_copy_bw(device=0) -> float:
    v = C.c_double(0)
    check(lib().acoc_measure_copy_bw(device, C.addressof(v)))
    return v.value
