"""Device-resident inputs and outputs (acoc_*_dev): CUDA tensors in and out of the batched solver and the tracker without a host round
trip.  CPU: the tensor validator.  GPU: every _dev call against its host-array twin, bit for bit (inputs: result, history and
statistics of the solve; outputs: the arrays themselves), the order against the caller's stream, the refusals of host, page-locked
and foreign-device addresses, and a 65,536-instance read-back."""
import ctypes as C

import numpy as np
import pytest

from tests.test_track_batch import _assert_same, _solved_batch, _track_weights

torch = pytest.importorskip("torch")

N, TT = 100, 60   # ragged: not a multiple of 32


def _problem(n=N, TT=TT, seed=0):
    from aircraftoptimalcontrol_b200 import refgen
    rng = np.random.default_rng(seed)
    return refgen.step_problem(rng.uniform(14, 18, n), rng.uniform(1.5, 3.5, n), tf=TT / 1000, TT=TT)


def _cuda(a, device=0):
    return torch.from_numpy(np.ascontiguousarray(a)).to(torch.device("cuda", device))


def _np(t):
    return t.cpu().numpy()


def _tree_np(d):
    return {k: _np(v) for k, v in d.items()}


# ---------------------------------------------------------------------------------------------------------------------------- CPU
def test_validator_rejects():
    from aircraftoptimalcontrol_b200 import _lib
    good = torch.zeros((3, 6, 5), dtype=torch.float64)
    for bad, what in ((np.zeros((3, 6, 5)), "torch.Tensor"),
                      (good, "cuda:0"),                                             # a CPU tensor
                      (good.to(torch.float32), "dtype"),
                      (torch.zeros((3, 6, 4), dtype=torch.float64), "shape"),
                      (torch.zeros((3, 5, 6), dtype=torch.float64).transpose(1, 2), "contiguous")):
        with pytest.raises(ValueError, match=what):
            _lib.dev_tensor(bad, 0, (3, 6, 5), torch.float64, "x")
    from aircraftoptimalcontrol_b200.batch import BatchedNewton
    bn = BatchedNewton.__new__(BatchedNewton)   # shape and type checks come before any library call
    bn.N, bn.TT, bn.device, bn._h = 3, 5, 0, None
    for delta in (np.zeros((4, 6)), torch.zeros((0, 6), dtype=torch.float64), torch.zeros((2, 4, 6), dtype=torch.float64)):
        with pytest.raises(ValueError):
            bn.track_mc_dev(delta)


# ---------------------------------------------------------------------------------------------------------------------------- GPU
def _init_guess(gpu, xr, ur, **kw):
    from aircraftoptimalcontrol_b200 import refgen
    with gpu.BatchedNewton(xr.shape[0] if xr.ndim == 3 else N, TT=xr.shape[-1], **kw) as bn:
        bn.set_weights(*refgen.weights("step"))
        bn.set_refs(xr, ur)
        bn.init_guess()
        return bn.iterate_at(0)


INPUT_CASES = {
    "f32": dict(kw=dict()),
    "f64": dict(kw=dict(state="f64")),
    "f64_slots": dict(kw=dict(), perturb=True),   # float32 quantisation, initial states that are not float32 values
    "refs_shared": dict(kw=dict(refs_shared=True)),
    "fp32": dict(kw=dict(precision="f32")),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(INPUT_CASES))
def test_inputs_equal_host(gpu, case):
    """set_refs_dev / set_init_dev solve to the same result(), history() and stats() as set_refs / set_init, bit for bit."""
    from aircraftoptimalcontrol_b200 import _lib, refgen
    kw, perturb = INPUT_CASES[case]["kw"], INPUT_CASES[case].get("perturb", False)
    xr, ur = _problem()
    if kw.get("refs_shared"):
        xr, ur = xr[0], ur[0]
    xi, ui = _init_guess(gpu, xr, ur, **kw)
    if perturb:
        xi = xi.copy()
        xi[:, :, 1:] += 1e-9
    out = []
    for dev in (False, True):
        with gpu.BatchedNewton(N, TT=TT, armijo="lazy", max_iters=30, **kw) as bn:
            bn.set_weights(*refgen.weights("step"))
            if dev:
                bn.set_refs_dev(_cuda(xr), _cuda(ur))
                bn.set_init_dev(_cuda(xi), _cuda(ui))
            else:
                bn.set_refs(xr, ur)
                bn.set_init(xi, ui)
            bn.solve()
            f32 = None
            try:
                f32 = bn.result_f32()
            except _lib.AcocError:
                pass
            out.append((bn.result(), bn.history(), bn.stats(), bn.refs(), f32))
    _assert_same(out[0][:4], out[1][:4])
    assert (out[0][4] is None) == (out[1][4] is None) == (case in ("f64", "f64_slots"))
    if out[0][4] is not None:
        _assert_same(out[0][4], out[1][4])


@pytest.mark.gpu
@pytest.mark.parametrize("state", ["f32", "f64"])
def test_outputs_equal_host(gpu, state):
    """result_dev = result() (and result_f32() with torch.float32, x0 included); tracked_dev = tracked(); track_gains_dev =
    track_gains(); into fresh tensors and into caller-supplied ones."""
    from aircraftoptimalcontrol_b200 import _lib
    with _solved_batch(gpu, N, TT, 3, state=state) as bn:
        xs, us = bn.result()
        xd, ud, x0 = bn.result_dev()
        assert xd.dtype == torch.float64 and xd.device == torch.device("cuda", 0)
        _assert_same((xs, us), (_np(xd), _np(ud)))
        assert np.array_equal(_np(x0), xs[:, :, 0])
        xd2, ud2 = torch.full_like(xd, np.nan), torch.full_like(ud, np.nan)
        r = bn.result_dev(out=(xd2, ud2))
        assert r[0] is xd2 and r[1] is ud2
        _assert_same((xs, us), (_np(xd2), _np(ud2)))
        if state == "f32":
            xf, uf, x0f = bn.result_f32()
            xfd, ufd, x0fd = bn.result_dev(torch.float32)
            assert xfd.dtype == torch.float32
            _assert_same((xf, uf, x0f), (_np(xfd), _np(ufd), _np(x0fd)))
            assert np.array_equal(x0f, _np(x0))
        else:
            with pytest.raises(_lib.AcocError, match="not float32 values"):
                bn.result_dev(torch.float32)
        with pytest.raises(_lib.AcocError, match="call acoc_track first"):
            bn.tracked_dev()
        bn.track(np.random.default_rng(1).uniform(-0.02, 0.02, (N, 6)))
        _assert_same(bn.tracked(), tuple(_np(t) for t in bn.tracked_dev()))
        K = bn.track_gains()
        assert np.array_equal(K, _np(bn.track_gains_dev()), equal_nan=True)
        Kd = torch.empty((N, 2, 6, TT), dtype=torch.float64, device="cuda:0")
        assert bn.track_gains_dev(out=Kd) is Kd and np.array_equal(K, _np(Kd), equal_nan=True)


@pytest.mark.gpu
@pytest.mark.parametrize("shared", [True, False])
def test_track_mc_dev_equals_host(gpu, shared):
    """track_mc_dev = track_mc on the same deltas held on the host, every output, with and without tol and per_sample; afterwards
    tracked() and tracked_dev() are refused and track_gains_dev() returns the gains the call used."""
    from aircraftoptimalcontrol_b200 import _lib
    M = 9
    d = np.random.default_rng(5).uniform(-0.05, 0.05, (M, 6) if shared else (N, M, 6))
    dd = _cuda(d)
    with _solved_batch(gpu, N, TT, 4) as bn:
        for tol in (None, np.full(6, 0.02)):
            for per_sample in (False, True):
                h = bn.track_mc(d, tol=tol, per_sample=per_sample)
                r = bn.track_mc_dev(dd, tol=tol, per_sample=per_sample)
                assert r["n_reg"].dtype == torch.int32 and r["worst_max"].device == torch.device("cuda", 0)
                _assert_same(h, _tree_np(r))
        with pytest.raises(_lib.AcocError):
            bn.tracked()
        with pytest.raises(_lib.AcocError):
            bn.tracked_dev()
        assert np.array_equal(bn.track_gains(), _np(bn.track_gains_dev()), equal_nan=True)


@pytest.mark.gpu
def test_stream_order(gpu):
    """Inputs written on a side stream behind a long device sleep, outputs overwritten there before the read-back: with that stream
    current, every call sees the writes queued before it, and its outputs can be consumed on that stream right after it returns."""
    from aircraftoptimalcontrol_b200 import refgen
    xr, ur = _problem(seed=7)
    xi, ui = _init_guess(gpu, xr, ur)
    d = np.random.default_rng(8).uniform(-0.05, 0.05, (N, 4, 6))
    with gpu.BatchedNewton(N, TT=TT, armijo="lazy", max_iters=30) as bn:
        bn.set_weights(*refgen.weights("step"))
        bn.set_refs(xr, ur)
        bn.set_init(xi, ui)
        bn.solve()
        host = (bn.result(), bn.history(), bn.stats(), bn.track_mc(d, per_sample=True))
    src = [_cuda(a) for a in (xr, ur, xi, ui, d)]
    torch.cuda.synchronize()
    sleep = 200_000_000   # clock cycles, ~0.1 s: the writes behind it land long after the next call has been queued
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        dst = [torch.zeros_like(s) for s in src]
        torch.cuda._sleep(sleep)
        for a, b in zip(dst[:4], src[:4]):
            a.copy_(b)
        with gpu.BatchedNewton(N, TT=TT, armijo="lazy", max_iters=30) as bn:
            bn.set_weights(*refgen.weights("step"))
            bn.set_refs_dev(dst[0], dst[1])
            bn.set_init_dev(dst[2], dst[3])
            bn.solve()
            xs = torch.empty((N, 6, TT), dtype=torch.float64, device="cuda:0")
            us = torch.empty((N, 2, TT), dtype=torch.float64, device="cuda:0")
            torch.cuda._sleep(sleep)
            xs.fill_(np.nan)                  # queued before the read-back: must not overwrite its result
            us.fill_(np.nan)
            bn.result_dev(out=(xs, us))
            xs2, us2 = xs * 1.0, us * 1.0     # consumed on the side stream right away
            torch.cuda._sleep(sleep)
            dst[4].copy_(src[4])
            mc = bn.track_mc_dev(dst[4], per_sample=True)
            mc2 = {k: v.clone() for k, v in mc.items()}
            dev = ((_np(xs2), _np(us2)), bn.history(), bn.stats(), _tree_np(mc2))
    _assert_same(host, dev)


def _host_buffers(n_doubles):
    """A numpy array and a page-locked host tensor of n_doubles float64 each."""
    return np.zeros(n_doubles), torch.zeros(n_doubles, dtype=torch.float64).pin_memory()


@pytest.mark.gpu
def test_refusals(gpu):
    """Numpy and page-locked host addresses handed straight to every _dev entry point are refused with ACOC_ERR_INVALID, naming the
    argument, and change nothing: a host-path solve on the same context afterwards equals one on a fresh context.  A tensor on
    another GPU is refused too (skipped with one GPU); track_mc_dev refuses what track_mc refuses."""
    from aircraftoptimalcontrol_b200 import _lib, refgen
    lib = _lib.lib()
    xr, ur = _problem(seed=11)
    xi, ui = _init_guess(gpu, xr, ur)
    Wt = [np.ascontiguousarray(w, dtype=np.float64) for w in _track_weights()]
    tol = np.ones(6)
    big = N * 12 * TT
    arr, pinned = _host_buffers(big)
    g = torch.zeros(big, dtype=torch.float64, device="cuda:0")
    G = g.data_ptr()
    ref = None
    for refused in (False, True):
        with gpu.BatchedNewton(N, TT=TT, armijo="lazy", max_iters=30) as bn:
            bn.set_weights(*refgen.weights("step"))
            bn.set_refs(xr, ur)
            bn.set_init(xi, ui)
            bn.track(np.full(6, 0.01))
            if refused:
                h = bn._h
                for host in (arr.ctypes.data, pinned.data_ptr()):
                    calls = {
                        "xx_ref_dev": lambda: lib.acoc_set_refs_dev(h, host, G, None),
                        "uu_ref_dev": lambda: lib.acoc_set_refs_dev(h, G, host, None),
                        "xx_init_dev": lambda: lib.acoc_set_init_dev(h, host, G, None),
                        "uu_init_dev": lambda: lib.acoc_set_init_dev(h, G, host, None),
                        "xx_star_dev": lambda: lib.acoc_get_result_dev(h, host, 0, G, None, None),
                        "uu_star_dev": lambda: lib.acoc_get_result_dev(h, G, 1, host, None, None),
                        "x0_dev": lambda: lib.acoc_get_result_dev(h, G, 0, G, host, None),
                        "xx_reg_dev": lambda: lib.acoc_get_tracked_dev(h, host, G, None),
                        "uu_reg_dev": lambda: lib.acoc_get_tracked_dev(h, G, host, None),
                        "K_dev": lambda: lib.acoc_get_track_gains_dev(h, host, None),
                        "delta_dev": lambda: lib.acoc_track_mc_dev(h, *map(_lib.ptr, Wt), 2, host, 1, None, None, None),
                    }
                    for field in ("err_max", "err_final", "worst_max", "mean_final", "n_within", "n_reg"):
                        o = _lib.TrackMcOut(**{field: host})
                        calls["out_dev->" + field] = (lambda o=o: lib.acoc_track_mc_dev(h, *map(_lib.ptr, Wt), 2, G, 1, _lib.ptr(tol),
                                                                                     C.addressof(o), None))
                    for name, call in calls.items():
                        assert call() == -1, name
                        msg = lib.acoc_last_error().decode()
                        assert name in msg and "host memory" in msg, (name, msg)
                assert np.array_equal(pinned.numpy(), np.zeros(big)) and np.array_equal(arr, np.zeros(big))
                if torch.cuda.device_count() > 1:
                    g1 = torch.zeros(big, dtype=torch.float64, device="cuda:1")
                    assert lib.acoc_set_refs_dev(h, g1.data_ptr(), G, None) == -1
                    assert "device 0" in lib.acoc_last_error().decode()
                    with pytest.raises(ValueError, match="cuda:0"):
                        bn.result_dev(out=(g1[:N * 6 * TT].view(N, 6, TT), g1[:N * 2 * TT].view(N, 2, TT)))
            tracked = bn.tracked()
            bn.solve()
            snap = (bn.result(), bn.history(), bn.stats(), tracked)
        if ref is None:
            ref = snap
    _assert_same(ref, snap)
    with _solved_batch(gpu, N, TT, 2) as bn:
        dl = torch.zeros((2, 6), dtype=torch.float64, device="cuda:0")
        D = dl.data_ptr()
        o = _lib.TrackMcOut()
        for m, ptr, tol, out in ((0, D, None, None), (-1, D, None, None), (2, None, None, None),
                                 (2, D, None, _lib.TrackMcOut(n_within=torch.zeros(N, dtype=torch.int32, device="cuda:0").data_ptr()))):
            assert lib.acoc_track_mc_dev(bn._h, *map(_lib.ptr, Wt), m, ptr, 1, tol, None if out is None else C.addressof(out), None) == -1
        Q = np.eye(6)
        Q[0, 1] = 1e-3
        with pytest.raises(_lib.AcocError, match="symmetric"):
            bn.track_mc_dev(dl, QQt=Q)
        with pytest.raises(ValueError):
            bn.track_mc_dev(dl, tol=np.ones(5))
        with pytest.raises(ValueError):
            bn.track_mc_dev(dl.to(torch.float32))
        assert lib.acoc_track_mc_dev(bn._h, *map(_lib.ptr, Wt), 2, D, 1, None, C.addressof(o), None) == 0
    with gpu.BatchedNewton(32, TT=50, precision="f32") as bn:
        bn.set_refs_step(np.full(32, 2.0), np.full(32, 16.0), tf=0.05)
        bn.init_guess()
        with pytest.raises(_lib.AcocError, match="FP32"):
            bn.track_mc_dev(torch.zeros((2, 6), dtype=torch.float64, device="cuda:0"))
    with gpu.BatchedNewton(32, TT=50) as bn:
        with pytest.raises(_lib.AcocError, match="no iterate"):
            bn.track_mc_dev(torch.zeros((2, 6), dtype=torch.float64, device="cuda:0"))


@pytest.mark.gpu
def test_result_dev_65536(gpu):
    """A 65,536 x 1000 solve (step maneuvers, lazy Armijo) read back with result_dev equals result() bit for bit, in both dtypes."""
    from aircraftoptimalcontrol_b200 import refgen
    n, TT_ = 65536, 1000
    zf, xf = refgen.config4_params(n, 2024)
    with gpu.BatchedNewton(n, TT=TT_, armijo="lazy") as bn:
        bn.set_weights(*refgen.weights("step"))
        bn.set_refs_step(zf, xf)
        bn.init_guess()
        bn.solve()
        xs, us = bn.result()
        xd, ud, x0 = bn.result_dev()
        assert np.array_equal(xs, _np(xd)) and np.array_equal(us, _np(ud)) and np.array_equal(xs[:, :, 0], _np(x0))
        del xd, ud
        xf32, _, x0f = bn.result_f32()
        xfd, ufd, x0fd = bn.result_dev(torch.float32)
        assert np.array_equal(xf32, _np(xfd)) and np.array_equal(us, _np(ufd)) and np.array_equal(x0f, _np(x0fd))
