"""Monte Carlo dispersion of closed-loop LQR tracking (acoc_track_mc, acoc_lqr_tracking_mc): M perturbed starts per instance along the
instance's own nominal and gains.  CPU: the host replay of the new per-sample and reduction code against the replay of acoc_track (one
sample = one acoc_track lane, bit for bit) and against the C oracle, the fixed-order aggregates against a plain loop, argument
validation.  GPU: kernels vs host replay, the device path vs the host-array path, per-sample summaries vs track(delta[:, m]), no side
effects on the solve, isolation of invalid lanes, refusals, and a 65,536-instance study."""
import ctypes as C

import numpy as np
import pytest

from tests.test_track_batch import R_INDEFINITE, _assert_same, _dyn, _nominal_sets, _solved_batch, _track_weights
from tests.util import golden


@pytest.fixture(scope="module")
def temul():
    from tests.host_emul import track_emul
    track_emul.build()
    return track_emul


@pytest.fixture(scope="module")
def mcemul():
    from tests.host_emul import track_mc_emul
    track_mc_emul.build()
    return track_mc_emul


def _sets_with_indefinite_r():
    sets = _nominal_sets()
    Qt, _, QTt = _track_weights()
    sets.append(("indefinite R",) + sets[0][1:4] + (Qt, R_INDEFINITE, QTt))
    return sets


def _max_nan(m, v):
    return v if (v > m or v != v) else m


def _aggregates(em, ef, tol):
    """Plain loop over the samples of every instance, in sample order: worst_max, mean_final, n_within."""
    N, M, _ = em.shape
    wm, mf, nw = np.empty((N, 6)), np.empty((N, 6)), np.zeros(N, dtype=np.int32)
    for i in range(N):
        for c in range(6):
            w, s = em[i, 0, c], ef[i, 0, c]
            for m in range(1, M):
                w = _max_nan(w, em[i, m, c])
                s = s + ef[i, m, c]
            wm[i, c], mf[i, c] = w, s / np.float64(M)
        if tol is not None:
            nw[i] = sum(all(em[i, m, c] <= tol[c] for c in range(6)) for m in range(M))
    return wm, mf, nw


# ---------------------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("f64", [False, True])
def test_replay_equals_track_replay_and_oracle(temul, mcemul, oracle, f64):
    """n = 1, M = 516 / 64: every sample equals acoc_track's replay with the deltas laid out one per instance, bit for bit, and the
    summaries of the oracle's trajectories (bit for bit where the replay reproduces the trajectory, within its tolerance elsewhere)."""
    for name, xo, uo, d, Q, R, QT in _sets_with_indefinite_r():
        e = mcemul.track_mc(xo[:1], uo[:1], d, Q, R, QT, state_f64=f64)
        t = temul.track_many(xo, uo, d, Q, R, QT, state_f64=f64)
        assert np.array_equal(e["err_max"][0], t["err_max"], equal_nan=True), name
        assert np.array_equal(e["err_final"][0], t["err_final"], equal_nan=True), name
        assert np.all(t["n_reg"] == e["n_reg"][0]), name
        o = oracle.lqr_tracking(xo[0], uo[0], Q, R, QT, d, quant_f32=not f64)
        err = np.abs(o[0] - xo[0][None])
        om, of = err.max(-1), err[..., -1]
        same = np.array([np.array_equal(t["xx_reg"][k], o[0][k]) for k in range(len(d))])
        if not f64:
            assert same.mean() >= 0.99, (name, same.mean())
        assert np.array_equal(e["err_max"][0][same], om[same]) and np.array_equal(e["err_final"][0][same], of[same]), name
        scale = np.abs(o[0]).max(-1)
        rel = 1e-9 if f64 else 1e-5
        assert np.all(np.abs(e["err_max"][0] - om) <= rel * scale) and np.all(np.abs(e["err_final"][0] - of) <= rel * scale), name


def test_replay_aggregates(mcemul):
    """worst_max, mean_final and n_within equal a plain loop over the per-sample values in sample order, with NaN samples injected,
    with M = 1, and shared deltas equal the per-instance layout with the same deltas broadcast."""
    from aircraftoptimalcontrol_b200 import refgen
    g = golden("lqr_tracking.npz")
    Q, R, QT = _track_weights()
    n, TT = 3, 300
    xo = np.repeat(g["xx_opt"][None, :, :TT], n, 0)
    uo = np.repeat(g["uu_opt"][None, :, :TT], n, 0)
    d = refgen.config3_deltas(3 * 9, seed=8).reshape(3, 9, 6)
    d[1, 3, 2] = np.nan                       # one NaN sample in instance 1
    d[2, :, 0] = np.nan                       # every sample of instance 2
    e0 = mcemul.track_mc(xo, uo, d, Q, R, QT)
    tol = np.median(e0["err_max"][0], axis=0)  # about half of the samples of instance 0 are within in each state
    e = mcemul.track_mc(xo, uo, d, Q, R, QT, tol=tol)
    wm, mf, nw = _aggregates(e["err_max"], e["err_final"], tol)
    assert np.array_equal(e["worst_max"], wm, equal_nan=True) and np.array_equal(e["mean_final"], mf, equal_nan=True)
    assert np.array_equal(e["n_within"], nw)
    assert 0 < nw[0] < 9 and nw[2] == 0 and np.isnan(e["err_max"][1, 3]).all()
    assert np.isnan(e["worst_max"][1]).all() and np.isnan(e["mean_final"][1]).all() and np.isfinite(e["worst_max"][0]).all()
    e1 = mcemul.track_mc(xo, uo, d[:, :1], Q, R, QT, tol=tol)   # M = 1: the aggregates are the one sample
    assert np.array_equal(e1["worst_max"], e1["err_max"][:, 0], equal_nan=True)
    assert np.array_equal(e1["mean_final"], e1["err_final"][:, 0], equal_nan=True)
    ds = refgen.config3_deltas(9, seed=9)
    es = mcemul.track_mc(xo, uo, ds, Q, R, QT, tol=tol)
    eb = mcemul.track_mc(xo, uo, np.broadcast_to(ds, (n, 9, 6)), Q, R, QT, tol=tol)
    _assert_same(es, eb)


def test_track_mc_validation():
    from aircraftoptimalcontrol_b200 import _lib
    from aircraftoptimalcontrol_b200.batch import BatchedNewton
    from aircraftoptimalcontrol_b200.lqr_tracking import lqr_tracking_mc
    x, u, d = np.zeros((3, 6, 20)), np.zeros((3, 2, 20)), np.zeros((4, 6))
    for args in ((x[0, :5], u[0], d), (x, u[:2], d), (x, u[..., :19], d), (x, u, np.zeros((4, 5))), (x, u, np.zeros((2, 4, 6))),
                 (x, u, np.zeros(6)), (x, u, np.zeros((0, 6))), (x, u, np.zeros((3, 0, 6))), (x[..., :2], u[..., :2], d)):
        with pytest.raises(ValueError):
            lqr_tracking_mc(*args)
    with pytest.raises(ValueError):
        lqr_tracking_mc(x, u, d, QQt=np.eye(5))
    with pytest.raises(ValueError):
        lqr_tracking_mc(x, u, d, tol=np.ones(5))
    bn = BatchedNewton.__new__(BatchedNewton)   # shape checks come before any library call
    bn.N, bn._h = 3, None
    for delta in (np.zeros((0, 6)), np.zeros((3, 0, 6)), np.zeros((2, 4, 6)), np.zeros(6), np.zeros((4, 7))):
        with pytest.raises(ValueError):
            bn.track_mc(delta)
    if _lib.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(_lib.AcocError, match="no CPU fallback|no CUDA device"):
        lqr_tracking_mc(x, u, d)


# ---------------------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("f64", [False, True])
def test_gpu_matches_host_replay(gpu, mcemul, f64):
    """lqr_tracking_mc = emul_track_mc bit for bit: one nominal with shared deltas, and two nominals with per-instance deltas."""
    from aircraftoptimalcontrol_b200.lqr_tracking import lqr_tracking_mc
    for name, xo, uo, d, Q, R, QT in _sets_with_indefinite_r():
        tol = np.full(6, 0.05)
        r = lqr_tracking_mc(xo[:1], uo[:1], d, _dyn(f64), Q, R, QT, tol=tol, per_sample=True)
        _assert_same(r, mcemul.track_mc(xo[:1], uo[:1], d, Q, R, QT, tol=tol, state_f64=f64))
        dp = np.stack([d, d[::-1] * 0.5])
        r = lqr_tracking_mc(xo[:2], uo[:2], dp, _dyn(f64), Q, R, QT, tol=tol, per_sample=True)
        _assert_same(r, mcemul.track_mc(xo[:2], uo[:2], dp, Q, R, QT, tol=tol, state_f64=f64))


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(), dict(state="f64"), dict(x_storage="f64"), dict(tma=False), dict(generations=False)])
def test_device_path_equals_host_path(gpu, kw):
    """track_mc on a solved context = lqr_tracking_mc on the downloaded result, bit for bit; its gains are track_gains()."""
    from aircraftoptimalcontrol_b200.lqr_tracking import lqr_tracking_mc
    n = 4200 if kw == dict(generations=False) or not kw else 300
    d = np.random.default_rng(2).uniform(-0.05, 0.05, (9, 6))
    tol = np.full(6, 0.02)
    with _solved_batch(gpu, n, 200, 7, **kw) as bn:
        res = bn.track_mc(d, tol=tol, per_sample=True)
        K = bn.track_gains()
        t = bn.track_timing()
        xs, us = bn.result()
    h = lqr_tracking_mc(xs, us, d, _dyn(kw.get("state") == "f64"), tol=tol, per_sample=True, return_gains=True)
    assert np.array_equal(K, h.pop("K"))
    _assert_same(res, h)
    assert t["total_ms"] > 0 and t["gains_ms"] > 0 and t["rollout_ms"] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 37, 4500])
def test_samples_equal_track(gpu, n):
    """Sample m of track_mc = track(delta[:, m]) bit for bit on ragged shapes; M = 1 reproduces track; two calls agree; TMA = plain
    loads."""
    rng = np.random.default_rng(n)
    out = {}
    for tma in (True, False):
        with _solved_batch(gpu, n, 200, 3, tma=tma) as bn:
            for M in ((1, 7, 33, 64, 4096) if n == 1 else (1, 7, 33, 64)):
                d = np.random.default_rng(M).uniform(-0.05, 0.05, (n, M, 6))
                r = bn.track_mc(d, per_sample=True)
                out[tma, M] = r
                if not tma:
                    continue
                for m in sorted({0, M // 2, M - 1, int(rng.integers(M))}):
                    t = bn.track(d[:, m])
                    assert np.array_equal(r["err_max"][:, m], t["err_max"], equal_nan=True), (M, m)
                    assert np.array_equal(r["err_final"][:, m], t["err_final"], equal_nan=True), (M, m)
                    assert np.array_equal(r["n_reg"], t["n_reg"])
                if M == 1:
                    assert np.array_equal(r["worst_max"], t["err_max"], equal_nan=True)
                    assert np.array_equal(r["mean_final"], t["err_final"], equal_nan=True)
                _assert_same(r, bn.track_mc(d, per_sample=True))
    for M in (1, 7, 33, 64):
        _assert_same(out[True, M], out[False, M])


@pytest.mark.gpu
def test_track_mc_has_no_side_effects(gpu):
    """Everything the solve exposes is unchanged by track_mc, iterating on afterwards equals a run without it; afterwards tracked()
    raises and track_gains() returns the gains it used."""
    from aircraftoptimalcontrol_b200 import _lib
    n, TT = 2000, 200
    d = np.random.default_rng(6).uniform(-0.02, 0.02, (16, 6))
    snaps = []
    for with_mc in (False, True):
        with _solved_batch(gpu, n, TT, 11, iters=3) as bn:
            before = (bn.result(), bn.iterate_at(0), bn.iterate_at(1), bn.gains(), bn.deltau(), bn.history(), bn.stats())
            if with_mc:
                bn.track(np.full(6, 0.01))
                K_track = bn.track_gains()
                bn.track_mc(d, tol=np.full(6, 0.05))
                with pytest.raises(_lib.AcocError):
                    bn.tracked()
                assert np.array_equal(bn.track_gains(), K_track, equal_nan=True)
                after = (bn.result(), bn.iterate_at(0), bn.iterate_at(1), bn.gains(), bn.deltau(), bn.history(), bn.stats())
                _assert_same(before, after)
                bn.track(np.full(6, 0.01))
                bn.tracked()
            bn.iterate(2)
            bn.solve()
            snaps.append((bn.result(), bn.history(), bn.stats()))
    _assert_same(snaps[0], snaps[1])


@pytest.mark.gpu
def test_invalid_lanes_isolated_and_refusals(gpu):
    """The zero-slot and NONFINITE lanes of a 96-instance batch: NaN in every sample, n_within = 0, every other lane bit-identical to
    the batch without them.  Refused: the FP32 mode, non-symmetric weights, M < 1, a NULL delta, buffers that do not fit (the context
    is left as it was)."""
    from aircraftoptimalcontrol_b200 import _lib, refgen
    q = golden("newton_quirks.npz")
    n, TT = 96, q["xx_ref"].shape[1]
    rng = np.random.default_rng(4)
    xr, ur = refgen.step_problem(rng.uniform(14, 18, n), rng.uniform(1.5, 3.5, n), tf=1, TT=TT)
    with gpu.BatchedNewton(n, TT=TT, state="f64") as bn:
        bn.set_weights(q["Q"], q["R"], q["QT"])
        bn.set_refs(xr, ur)
        bn.init_guess()
        xi, ui = bn.iterate_at(0)
    zero, nonfin = 7, 40
    xb, ub, xrb, urb = xi.copy(), ui.copy(), xr.copy(), ur.copy()
    xb[zero], ub[zero], xrb[zero], urb[zero] = q["b_xx_init"], q["b_uu_init"], q["xx_ref"], q["uu_ref"]
    xb[nonfin, 2, 0] = 0.0
    d = rng.uniform(-0.05, 0.05, (n, 5, 6))
    tol = np.full(6, 1.0)
    out = []
    for x_, u_, r_, s_ in ((xi, ui, xr, ur), (xb, ub, xrb, urb)):
        with gpu.BatchedNewton(n, TT=TT, state="f64") as bn:
            bn.set_weights(q["Q"], q["R"], q["QT"])
            bn.set_refs(r_, s_)
            bn.set_init(x_, u_)
            bn.solve()
            out.append((bn.track_mc(d, tol=tol, per_sample=True), bn.stats()))
    st = out[1][1]
    assert st["status"][zero] == 1 and st["status"][nonfin] == 3
    good = np.setdiff1d(np.arange(n), [zero, nonfin])
    ra, rb = out[0][0], out[1][0]
    for k in ra:
        assert np.array_equal(ra[k][good], rb[k][good]), k
    for i in (zero, nonfin):
        assert np.isnan(rb["err_max"][i]).any(-1).all() and rb["n_within"][i] == 0
    assert rb["n_within"][good].sum() > 0
    with gpu.BatchedNewton(32, TT=50, precision="f32") as bn:
        bn.set_refs_step(np.full(32, 2.0), np.full(32, 16.0), tf=0.05)
        bn.init_guess()
        with pytest.raises(_lib.AcocError):
            bn.track_mc(np.zeros((2, 6)))
    with gpu.BatchedNewton(32, TT=50) as bn:
        with pytest.raises(_lib.AcocError):
            bn.track_mc(np.zeros((2, 6)))     # no iterate yet
        bn.set_refs_step(np.full(32, 2.0), np.full(32, 16.0), tf=0.05)
        bn.init_guess()
        Q = np.eye(6)
        Q[0, 1] = 1e-3
        with pytest.raises(_lib.AcocError, match="symmetric"):
            bn.track_mc(np.zeros((2, 6)), QQt=Q)
        bn.track(np.full(6, 0.01))
        x_before, _ = bn.tracked()
        mem = bn.device_bytes
        W = [np.ascontiguousarray(w, dtype=np.float64) for w in _track_weights()]
        dl = np.zeros((2, 6))
        o = _lib.TrackMcOut()
        for m, ptr in ((0, dl), (-1, dl), (2, None)):
            with pytest.raises(_lib.AcocError):
                _lib.check(_lib.lib().acoc_track_mc(bn._h, _lib.ptr(W[0]), _lib.ptr(W[1]), _lib.ptr(W[2]), m, _lib.ptr(ptr), 1, None,
                                                    C.addressof(o)))
        # 2^35 samples (3.3 TB of per-sample buffers) cannot be allocated: refused before the deltas are read
        with pytest.raises(_lib.AcocError, match="cudaMalloc"):
            _lib.check(_lib.lib().acoc_track_mc(bn._h, _lib.ptr(W[0]), _lib.ptr(W[1]), _lib.ptr(W[2]), 1 << 30, _lib.ptr(dl), 1, None,
                                                C.addressof(o)))
        assert bn.device_bytes == mem
        assert np.array_equal(bn.tracked()[0], x_before)


@pytest.mark.gpu
def test_pipelined_65536_track_mc(gpu, mcemul):
    """configs[3] at scale: 65,536 step maneuvers solved by PipelinedNewton, 64 shared perturbations each; 64 sampled instances against
    the host replay on the downloaded results, finite aggregates for every converged instance."""
    from aircraftoptimalcontrol_b200 import refgen
    n, TT, M = 65536, 1000, 64
    zf, xf = refgen.config4_params(n, 2024)
    d = refgen.config3_deltas(M)
    tol = np.array([1.0, 1.0, 1.0, 0.2, 0.5, 0.2])
    with gpu.PipelinedNewton(n, n_chunks=1, TT=TT, armijo="lazy") as pn:
        pn.set_weights(*refgen.weights("step"))
        xs, us, st = pn.solve(refs=("step", zf, xf))
        res = pn.track_mc(d, tol=tol, per_sample=True)
        mem = pn.parts[0].device_bytes
    idx = np.linspace(0, n - 1, 64).astype(int)
    e = mcemul.track_mc(xs[idx], us[idx], d, *_track_weights(), tol=tol)
    for k in e:
        assert np.array_equal(res[k][idx], e[k], equal_nan=True), k
    ok = st["status"] == 1
    assert np.isfinite(res["worst_max"][ok]).all() and np.isfinite(res["mean_final"][ok]).all()
    print("device bytes of the 65,536 x 1000 context after track_mc (64 samples): %.2f GB; capture rate %.3f"
          % (mem / 1e9, res["n_within"].sum() / (n * M)))
