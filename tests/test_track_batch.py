"""Closed-loop LQR tracking of every instance along its own nominal (acoc_track, acoc_lqr_tracking_many; lqr_tracking.py:245-283 per
instance).  CPU: the host replay of the new per-instance kernel code against the C oracle (itself pinned to the live reference by
test_oracle_golden.py::test_lqr_tracking), and argument validation.  GPU: kernels vs host replay (bit for bit), the device path vs the
oracle on solved batches, vs the host-array path, and the promise that tracking leaves the Newton state alone."""
import numpy as np
import pytest

from tests.util import golden

@pytest.fixture(scope="module")
def temul():
    from tests.host_emul import track_emul
    track_emul.build()
    return track_emul


R_INDEFINITE = np.array([[1e-5, 0.0], [0.0, -1.0]])  # symmetric, indefinite: G = R + B'PB takes the +0.5 I gain branch


def _track_weights():
    from aircraftoptimalcontrol_b200.lqr_tracking import default_weights
    return default_weights()


def _nominal_sets():
    """(name, xx_opt (N,6,TT), uu_opt (N,2,TT), delta (N,6), Q, R, QT): the shipped tracking golden with its 4 deltas and 512 of the
    config-3 deltas, and the four live-reference optima of the batched configurations with 64 perturbations each."""
    from aircraftoptimalcontrol_b200 import refgen
    g = golden("lqr_tracking.npz")
    d = np.concatenate([g["delta"], refgen.config3_deltas()[:512]])
    n = len(d)
    sets = [("golden", np.repeat(g["xx_opt"][None], n, 0), np.repeat(g["uu_opt"][None], n, 0), d, g["Q"], g["R"], g["QT"])]
    b = golden("newton_batched_instances.npz")
    Q, R, QT = _track_weights()
    rng = np.random.default_rng(5)
    for k in ("config4_0", "config4_1", "config5_0", "config5_1"):
        sets.append((k, np.repeat(b[k + "_xx_star"][None], 64, 0), np.repeat(b[k + "_uu_star"][None], 64, 0), rng.normal(0, 0.05, (64, 6)),
                     Q, R, QT))
    return sets


def _check_vs_oracle(oracle, xx_opt, uu_opt, delta, Q, R, QT, xr, ur, K, f64):
    """One oracle lqr_tracking call per nominal.  Gains (K None: not checked) within 1e-9 (the sparse Riccati step vs the dense ltv_LQR
    differ by ~1e-13); states within 1e-5 relative and nearly all bit-identical under the float32 quantisation (a 1e-13 difference in K
    may flip a rounding), within 1e-9 in float64; inputs within 1e-6.  Measured on the host replay: test_host_replay_matches_oracle."""
    same = []
    for i in range(len(delta)):
        o = oracle.lqr_tracking(xx_opt[i], uu_opt[i], Q, R, QT, delta[i:i + 1], quant_f32=not f64, n_threads=1)
        if K is not None:
            assert np.max(np.abs(K[i] - o[2])) <= 1e-9 * np.max(np.abs(o[2])), i
        assert np.max(np.abs(xr[i] - o[0][0]) / np.abs(o[0][0]).max(-1, keepdims=True)) <= (1e-9 if f64 else 1e-5), i
        assert np.max(np.abs(ur[i] - o[1][0]) / np.abs(o[1][0]).max(-1, keepdims=True)) <= 1e-6, i
        same.append(np.array_equal(xr[i], o[0][0]))
    if not f64:
        assert np.mean(same) >= 0.95, np.mean(same)


def _check_summaries(res, xr, xx_opt):
    err = np.abs(xr - xx_opt)
    assert np.array_equal(res["err_max"], err.max(-1), equal_nan=True)
    assert np.array_equal(res["err_final"], err[..., -1], equal_nan=True)


# ---------------------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("f64", [False, True])
def test_host_replay_matches_oracle(temul, oracle, f64):
    for name, xo, uo, d, Q, R, QT in _nominal_sets():
        e = temul.track_many(xo, uo, d, Q, R, QT, state_f64=f64)
        o_all = oracle.lqr_tracking(xo[0], uo[0], Q, R, QT, d, quant_f32=not f64)   # one nominal per set: one call covers every delta
        assert np.max(np.abs(e["K"] - o_all[2][None])) <= 1e-9 * np.max(np.abs(o_all[2])), name
        same = np.array([np.array_equal(e["xx_reg"][i], o_all[0][i]) for i in range(len(d))])
        if not f64:
            assert same.mean() >= 0.99, (name, same.mean())
        assert np.max(np.abs(e["xx_reg"] - o_all[0]).max(-1) / np.abs(o_all[0]).max(-1)) <= (1e-5 if not f64 else 1e-9), name
        assert np.max(np.abs(e["uu_reg"] - o_all[1]) / np.abs(o_all[1]).max(-1, keepdims=True)) <= 1e-9, name
        assert not e["uu_reg"][:, :, -1].any() and not e["K"][..., -1].any()
        _check_summaries(e, e["xx_reg"], xo)
        assert not e["n_reg"].any()


def test_host_replay_regularised_branch(temul, oracle):
    g = golden("lqr_tracking.npz")
    Q, _, QT = _track_weights()
    d = np.full((2, 6), 0.01)
    e = temul.track_many(np.repeat(g["xx_opt"][None], 2, 0), np.repeat(g["uu_opt"][None], 2, 0), d, Q, R_INDEFINITE, QT)
    o = oracle.lqr_tracking(g["xx_opt"], g["uu_opt"], Q, R_INDEFINITE, QT, d)
    assert np.all(e["n_reg"] > 900)
    assert np.max(np.abs(e["K"] - o[2][None])) <= 1e-9 * np.max(np.abs(o[2]))
    assert np.array_equal(e["xx_reg"], o[0])


def test_host_replay_zero_nominal_is_nan(temul):
    """The all-zero slot (an instance stopped at kk = 0) divides by V = 0 like the reference: NaN summaries, no exception."""
    Q, R, QT = _track_weights()
    e = temul.track_many(np.zeros((1, 6, 50)), np.zeros((1, 2, 50)), np.full((1, 6), 0.01), Q, R, QT)
    assert np.isnan(e["err_max"]).all() and np.isnan(e["err_final"]).all()


def test_lqr_tracking_many_validation():
    from aircraftoptimalcontrol_b200 import _lib
    from aircraftoptimalcontrol_b200.lqr_tracking import lqr_tracking_many
    x, u, d = np.zeros((3, 6, 20)), np.zeros((3, 2, 20)), np.zeros((3, 6))
    for args in ((x[0], u, d), (x, u[:2], d), (x, u[..., :19], d), (x, u, d[:2]), (x, u, np.zeros(5)), (x[:, :5], u, d),
                 (x[..., :2], u[..., :2], d)):
        with pytest.raises(ValueError):
            lqr_tracking_many(*args)
    with pytest.raises(ValueError):
        lqr_tracking_many(x, u, d, QQt=np.eye(5))
    if _lib.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(_lib.AcocError, match="no CPU fallback|no CUDA device"):
        lqr_tracking_many(x, u, d)


# ---------------------------------------------------------------------------------------------------------------------------- GPU
def _dyn(f64):
    from aircraftoptimalcontrol_b200.aircraft_simplified import Dynamics
    return Dynamics(state="f64" if f64 else "f32")


@pytest.mark.gpu
@pytest.mark.parametrize("f64", [False, True])
def test_gpu_matches_host_replay(gpu, temul, f64):
    from aircraftoptimalcontrol_b200.lqr_tracking import lqr_tracking_many
    sets = _nominal_sets()
    Qt, _, QTt = _track_weights()
    sets.append(("indefinite R",) + sets[0][1:4] + (Qt, R_INDEFINITE, QTt))
    for name, xo, uo, d, Q, R, QT in sets:
        xr, ur, K = lqr_tracking_many(xo, uo, d, _dyn(f64), Q, R, QT, return_gains=True)
        e = temul.track_many(xo, uo, d, Q, R, QT, state_f64=f64)
        assert np.array_equal(K, e["K"]), name
        assert np.array_equal(xr, e["xx_reg"]) and np.array_equal(ur, e["uu_reg"]), name


def _solved_batch(gpu, n, TT, seed, iters=None, **kw):
    from aircraftoptimalcontrol_b200 import refgen
    rng = np.random.default_rng(seed)
    zf, xf = rng.uniform(1.5, 3.5, n), rng.uniform(14, 18, n)
    bn = gpu.BatchedNewton(n, TT=TT, armijo="lazy", **kw)
    bn.set_weights(*refgen.weights("step"))
    bn.set_refs_step(zf, xf, tf=TT / 1000)
    bn.init_guess()
    if iters is None:
        bn.solve()
    else:
        bn.iterate(iters)
    return bn


@pytest.mark.gpu
def test_device_path_matches_oracle(gpu, oracle):
    """A ragged 4,500-instance configs[3] batch (step maneuvers, lazy Armijo), solved and tracked with per-instance deltas: 64 sampled
    instances and every MAXITER instance against one oracle lqr_tracking call on the downloaded result each."""
    from aircraftoptimalcontrol_b200 import refgen
    n = 4500
    with _solved_batch(gpu, n, 1000, 2024) as bn:
        d = refgen.config3_deltas(n, seed=3)
        res = bn.track(d)
        xr, ur = bn.tracked()
        K = bn.track_gains()
        xs, us = bn.result()
        st = bn.stats()
    idx = np.unique(np.concatenate([np.linspace(0, n - 1, 64).astype(int), np.flatnonzero(st["status"] == 2)]))
    _check_vs_oracle(oracle, xs[idx], us[idx], d[idx], *_track_weights(), xr[idx], ur[idx], K[idx], f64=False)
    _check_summaries(res, xr, xs)
    assert np.isfinite(res["err_max"][st["status"] == 1]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(), dict(state="f64"), dict(x_storage="f64"), dict(tma=False), dict(generations=False)])
def test_device_path_equals_host_path(gpu, kw):
    """track + tracked on a solved context is bit-identical to lqr_tracking_many on the downloaded result (same kernels), the summaries
    are numpy's abs(xx_reg - xx_star).max(-1) / [..., -1], and a (6,) delta broadcasts."""
    from aircraftoptimalcontrol_b200.lqr_tracking import lqr_tracking_many
    n = 4200 if kw == dict(generations=False) or not kw else 300
    with _solved_batch(gpu, n, 200, 7, **kw) as bn:
        d = np.random.default_rng(1).uniform(-0.05, 0.05, (n, 6))
        res = bn.track(d)
        xr, ur = bn.tracked()
        K = bn.track_gains()
        xs, us = bn.result()
        t = bn.track_timing()
        res1 = bn.track(d[0])
        xr1, _ = bn.tracked()
    hx, hu, hK = lqr_tracking_many(xs, us, d, _dyn(kw.get("state") == "f64"), return_gains=True)
    assert np.array_equal(xr, hx) and np.array_equal(ur, hu) and np.array_equal(K, hK)
    _check_summaries(res, xr, xs)
    assert t["total_ms"] > 0 and t["gains_ms"] > 0 and t["rollout_ms"] > 0
    hx1, _ = lqr_tracking_many(xs, us, np.broadcast_to(d[0], (n, 6)), _dyn(kw.get("state") == "f64"))
    assert np.array_equal(xr1, hx1)
    _check_summaries(res1, xr1, xs)


@pytest.mark.gpu
def test_track_has_no_side_effects(gpu):
    """Everything the solve exposes is bit-identical before and after track, and iterating on after it gives what a run without it gives."""
    n, TT = 2000, 200
    snaps = []
    for with_track in (False, True):
        with _solved_batch(gpu, n, TT, 11, iters=3) as bn:
            before = (bn.result(), bn.iterate_at(0), bn.iterate_at(1), bn.gains(), bn.deltau(), bn.history(), bn.stats())
            if with_track:
                bn.track(np.full(6, 0.01))
                after = (bn.result(), bn.iterate_at(0), bn.iterate_at(1), bn.gains(), bn.deltau(), bn.history(), bn.stats())
                _assert_same(before, after)
            bn.iterate(2)
            bn.solve()
            snaps.append((bn.result(), bn.history(), bn.stats()))
    _assert_same(snaps[0], snaps[1])


def _assert_same(a, b):
    if isinstance(a, dict):
        assert a.keys() == b.keys()
        for k in a:
            _assert_same(a[k], b[k])
    elif isinstance(a, (tuple, list)):
        for x, y in zip(a, b):
            _assert_same(x, y)
    else:
        assert np.array_equal(a, b, equal_nan=True)


@pytest.mark.gpu
def test_regularised_branch_count(gpu, oracle, temul):
    """n_reg counts the steps whose gain took the +0.5 I branch, forced by a symmetric indefinite R; gains still match the oracle."""
    with _solved_batch(gpu, 64, 300, 5) as bn:
        Q, _, QT = _track_weights()
        res = bn.track(np.full(6, 0.01), Q, R_INDEFINITE, QT)
        K = bn.track_gains()
        xs, us = bn.result()
    e = temul.track_many(xs, us, np.full((64, 6), 0.01), Q, R_INDEFINITE, QT)
    assert np.array_equal(res["n_reg"], e["n_reg"]) and res["n_reg"].min() > 0
    for i in (0, 31, 63):
        o = oracle.lqr_tracking(xs[i], us[i], Q, R_INDEFINITE, QT, np.full((1, 6), 0.01))
        assert np.max(np.abs(K[i] - o[2])) <= 1e-9 * np.max(np.abs(o[2]))


@pytest.mark.gpu
def test_invalid_lanes_are_nan_and_isolated(gpu):
    """newton_quirks.npz case b (converged at kk = 0: the zero slot) and a V = 0 start (NONFINITE) in a 96-instance batch: NaN summaries
    for those two, every other lane bit-identical to the batch without them."""
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
    d = rng.uniform(-0.05, 0.05, (n, 6))
    out = []
    for x_, u_, r_, s_ in ((xi, ui, xr, ur), (xb, ub, xrb, urb)):
        with gpu.BatchedNewton(n, TT=TT, state="f64") as bn:
            bn.set_weights(q["Q"], q["R"], q["QT"])
            bn.set_refs(r_, s_)
            bn.set_init(x_, u_)
            bn.solve()
            out.append((bn.track(d), bn.tracked(), bn.track_gains(), bn.stats()))
    st = out[1][3]
    assert st["iters"][zero] == 1 and st["status"][zero] == 1 and st["status"][nonfin] == 3
    good = np.setdiff1d(np.arange(n), [zero, nonfin])
    (ra, (xa, ua), Ka, _), (rb, (xb_, ub_), Kb, _) = out
    for k in ra:
        assert np.array_equal(ra[k][good], rb[k][good]), k
    assert np.array_equal(xa[good], xb_[good]) and np.array_equal(ua[good], ub_[good]) and np.array_equal(Ka[good], Kb[good])
    for i in (zero, nonfin):
        assert np.isnan(rb["err_max"][i]).any() and np.isnan(rb["err_final"][i]).any()
    # refused: the FP32 mode, non-symmetric weights, tracking before there is an iterate
    with gpu.BatchedNewton(32, TT=50, precision="f32") as bn:
        bn.set_refs_step(np.full(32, 2.0), np.full(32, 16.0), tf=0.05)
        bn.init_guess()
        with pytest.raises(_lib.AcocError):
            bn.track()
    with gpu.BatchedNewton(32, TT=50) as bn:
        with pytest.raises(_lib.AcocError):
            bn.track()
        bn.set_refs_step(np.full(32, 2.0), np.full(32, 16.0), tf=0.05)
        bn.init_guess()
        Q = np.eye(6)
        Q[0, 1] = 1e-3
        with pytest.raises(_lib.AcocError, match="symmetric"):
            bn.track(QQt=Q)
        with pytest.raises(_lib.AcocError):
            bn.tracked()


@pytest.mark.gpu
def test_pipelined_65536_track(gpu, oracle):
    """configs[3] at scale: 65,536 step maneuvers solved by PipelinedNewton, then every one tracked; 64 sampled against the oracle, finite
    summaries for every converged instance."""
    from aircraftoptimalcontrol_b200 import refgen
    n, TT = 65536, 1000
    zf, xf = refgen.config4_params(n, 2024)
    d = refgen.config3_deltas(n)
    with gpu.PipelinedNewton(n, n_chunks=1, TT=TT, armijo="lazy") as pn:
        pn.set_weights(*refgen.weights("step"))
        xs, us, st = pn.solve(refs=("step", zf, xf))
        res = pn.track(d)
        xr, ur = pn.tracked()
        mem = pn.parts[0].device_bytes
    idx = np.linspace(0, n - 1, 64).astype(int)
    _check_vs_oracle(oracle, xs[idx], us[idx], d[idx], *_track_weights(), xr[idx], ur[idx], None, f64=False)
    assert np.isfinite(res["err_max"][st["status"] == 1]).all() and np.isfinite(res["err_final"][st["status"] == 1]).all()
    print("device bytes of the 65,536 x 1000 context after track: %.2f GB" % (mem / 1e9))
