"""acoc_result_vjp on the GPU: the sm_100a sweeps against the host replay of their per-instance code (bit for bit), the device-array twin,
finite differences of whole solves, the autograd Functions, the promise that the call changes nothing of the solve or the tracking, and
the refusals.  The dense-KKT oracle of the definition is on the CPU side (tests/test_result_vjp.py)."""
import ctypes as C

import numpy as np
import pytest


TT = 200


def _problem(gpu, n, TT=TT, state="f32", maneuver="step", refs="param", weights="diag", tma=True, nan_lane=None, max_iters=40, **kw):
    """A solved batch (returned open) with its references as the replay wants them."""
    from aircraftoptimalcontrol_b200 import refgen
    rng = np.random.default_rng(n + TT)
    zf = rng.uniform(1.5, 3.5, n)
    tf = TT / 1000
    Q, R, QT = refgen.weights("step" if maneuver == "step" else "acro")
    if weights == "dense":
        M = rng.normal(size=(6, 6)) * 1e-3
        Q, QT, R = Q + M @ M.T, QT + M @ M.T, R + np.array([[0.0, 2e-7], [2e-7, 0.0]])
    bn = gpu.BatchedNewton(n, TT=TT, state=state, armijo="lazy", max_iters=max_iters, tma=tma, refs_compact=(refs == "param"), **kw)
    bn.set_weights(Q, R, QT)
    if maneuver == "step":
        xf = rng.uniform(14, 18, n) * tf
        tt, zs, vs = refgen.step_bases(tf, TT)
        prm = dict(tt=tt, zs=zs, vs=vs, zf=zf, vx=(xf - 0) / tf, xc=refgen.STEP_CONST[0], uc=refgen.STEP_CONST[1])
        if refs == "host":
            bn.set_refs(*refgen.step_problem(xf, zf, tf=tf, TT=TT))
        else:
            bn.set_refs_step(zf, xf, tf)
    else:
        tt, zs = refgen.acrobatic_bases(tf, TT)
        prm = dict(tt=tt, zs=zs, vs=None, zf=zf, vx=np.full(n, 18.0 * tf / tf), xc=refgen.ACRO_CONST[0], uc=refgen.ACRO_CONST[1])
        if refs == "host":
            bn.set_refs(*refgen.acrobatic_problem(zf, 18.0 * tf, tf=tf, TT=TT))
        else:
            bn.set_refs_acrobatic(zf, 18.0 * tf, tf)
        prm["vx"] = np.full(n, (18.0 * tf - 0) / tf)
    bn.init_guess()
    if nan_lane is not None:
        xi, ui = bn.iterate_at(0)
        xi[nan_lane, 2, 5:] = np.nan
        bn.set_init(xi, ui)
    bn.solve()
    return bn, (Q, R, QT), prm


def _replay(bn, W, prm, gx, gu):
    from tests.host_emul import vjp_emul
    xs, us = bn.result()
    if bn._refs_param:
        return vjp_emul.result_vjp(xs, us, gx, gu, *W, param=prm)
    xr, ur = bn.refs()
    return vjp_emul.result_vjp(xs, us, gx, gu, *W, xref=xr, uref=ur)


def _grads(n, seed=0):
    rng = np.random.default_rng(seed)
    return rng.normal(size=(n, 6, TT)), rng.normal(size=(n, 2, TT))


def _same(a, b):
    for k in ("xref", "uref", "x0", "zf", "vx", "n_indef"):
        if a[k] is None or b[k] is None:
            assert a[k] is None and b[k] is None, k
            continue
        assert np.array_equal(np.asarray(a[k]), np.asarray(b[k]), equal_nan=True), k


CASES = [(37, "f32", "step", "param", "diag", True), (37, "f64", "step", "host", "dense", True), (37, "f32", "acro", "param", "diag", False),
         (37, "f64", "step", "param", "dense", False), (37, "f32", "step", "expanded", "diag", True), (1, "f64", "acro", "host", "diag", True),
         (4500, "f32", "step", "param", "diag", True), (4500, "f64", "acro", "param", "dense", False)]


@pytest.mark.gpu
@pytest.mark.parametrize("n,state,maneuver,refs,weights,tma", CASES)
def test_kernels_match_replay(gpu, n, state, maneuver, refs, weights, tma):
    """Every output bit-identical to the host replay: float32 / float64 state storage, diagonal / dense weights, TMA / plain loads,
    parametric / expanded / host-array references.  4500 instances solve through survivor generations."""
    from tests.host_emul import vjp_emul
    vjp_emul.build()
    bn, W, prm = _problem(gpu, n, state=state, maneuver=maneuver, refs=refs, weights=weights, tma=tma)
    with bn:
        gx, gu = _grads(n, 1)
        r = bn.result_vjp(gx, gu)
        e = _replay(bn, W, prm, gx, gu)
        _same(r, e)
        assert np.all(np.isfinite(r["xref"])) and np.all(np.isfinite(r["x0"]))


@pytest.mark.gpu
def test_big_batch_and_special_lanes(gpu):
    """65,536 instances with a NONFINITE lane: that lane is NaN, the other lanes (sampled across tiles) bit-identical to the replay."""
    from aircraftoptimalcontrol_b200 import _lib
    from tests.host_emul import vjp_emul
    n, T = 65536, 40
    bn, W, prm = _problem(gpu, n, TT=T, nan_lane=3, max_iters=15)
    with bn:
        assert bn.stats()["status"][3] == _lib.INST_NONFINITE
        rng = np.random.default_rng(2)
        gx, gu = rng.normal(size=(n, 6, T)), rng.normal(size=(n, 2, T))
        r = bn.result_vjp(gx, gu)
        assert np.all(np.isnan(r["x0"][3])) and np.all(np.isnan(r["xref"][3][:, 2:]))
        idx = np.r_[0:64, 40000:40032, n - 33:n]
        xs, us = bn.result()
        sub = {k: v[idx] for k, v in prm.items() if isinstance(v, np.ndarray) and v.shape == (n,)}
        e = vjp_emul.result_vjp(xs[idx], us[idx], gx[idx], gu[idx], *W, param=dict(prm, **sub))
        _same({k: (None if v is None else v[idx]) for k, v in r.items()}, e)


@pytest.mark.gpu
def test_dev_twin_and_stream_order(gpu):
    """result_vjp_dev is bit-identical to result_vjp, also when its inputs are written on a side stream behind torch.cuda._sleep and its
    outputs overwritten there right after the call has been queued."""
    import torch
    bn, W, prm = _problem(gpu, 37)
    with bn:
        gx, gu = _grads(37, 4)
        host = bn.result_vjp(gx, gu)
        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            tx = torch.zeros((37, 6, TT), dtype=torch.float64, device="cuda:0")
            tu = torch.zeros((37, 2, TT), dtype=torch.float64, device="cuda:0")
            torch.cuda._sleep(200_000_000)
            tx.copy_(torch.from_numpy(gx))
            tu.copy_(torch.from_numpy(gu))
            dev = bn.result_vjp_dev(tx, tu)
            dev = {k: None if v is None else v.clone() for k, v in dev.items()}
        torch.cuda.synchronize()
        _same(host, {k: None if v is None else v.cpu().numpy() for k, v in dev.items()})


@pytest.mark.gpu
def test_no_side_effects(gpu):
    """A VJP between iterations changes nothing: iterating on, result, history, stats, tracked() and track_gains() equal those of a
    context that never ran it."""
    from aircraftoptimalcontrol_b200 import refgen
    out = []
    for vjp in (False, True):
        with gpu.BatchedNewton(64, TT=TT, armijo="lazy", max_iters=20) as bn:
            bn.set_weights(*refgen.weights("step"))
            bn.set_refs_step(np.linspace(1.5, 3.5, 64), np.full(64, 3.2), TT / 1000)
            bn.init_guess()
            bn.iterate(3)
            bn.track(np.full(6, 0.01))
            before = (bn.tracked(), bn.track_gains(), bn.result(), bn.history(), bn.stats())
            if vjp:
                bn.result_vjp(*_grads(64, 5))
            after = (bn.tracked(), bn.track_gains(), bn.result(), bn.history(), bn.stats())
            for a, b in zip(before, after):
                for x, y in zip(a.values() if isinstance(a, dict) else a, b.values() if isinstance(b, dict) else b):
                    assert np.array_equal(x, y)
            bn.iterate(4)
            out.append((bn.result(), bn.history(), bn.stats()))
    a, b = out
    assert all(np.array_equal(x, y) for x, y in zip(a[0], b[0]))
    for k in a[1]:
        assert np.array_equal(a[1][k], b[1][k])
    for k in a[2]:
        assert np.array_equal(a[2][k], b[2][k])


@pytest.mark.gpu
def test_refusals(gpu):
    """FP32 and before init: ACOC_ERR_STATE; NULL gx / gu, zf_bar with non-parametric references, host or page-locked arrays handed to
    the _dev call: ACOC_ERR_INVALID.  Each leaves the context as it was (a VJP afterwards equals one on a fresh context)."""
    import torch
    from aircraftoptimalcontrol_b200 import _lib, refgen
    lib = _lib.lib()
    gx, gu = _grads(37, 6)
    with gpu.BatchedNewton(37, TT=TT, precision="f32") as bf:
        bf.set_weights(*refgen.weights("step"))
        bf.set_refs_step(np.full(37, 2.0), np.full(37, 3.2), 0.2)
        bf.init_guess()
        assert lib.acoc_result_vjp(bf._h, _lib.ptr(gx), _lib.ptr(gu), None) == -3
    with gpu.BatchedNewton(37, TT=TT) as b0:
        b0.set_weights(*refgen.weights("step"))
        assert lib.acoc_result_vjp(b0._h, _lib.ptr(gx), _lib.ptr(gu), None) == -3
    ref = None
    for refuse in (False, True):
        bn, W, prm = _problem(gpu, 37, refs="host")
        with bn:
            if refuse:
                zb = np.zeros(37)
                o = _lib.VjpOut(None, None, None, _lib.ptr(zb), None, None)
                assert lib.acoc_result_vjp(bn._h, _lib.ptr(gx), _lib.ptr(gu), C.addressof(o)) == -1
                assert lib.acoc_result_vjp(bn._h, None, _lib.ptr(gu), None) == -1
                assert lib.acoc_result_vjp(bn._h, _lib.ptr(gx), None, None) == -1
                pinned = torch.zeros(37 * 6 * TT, dtype=torch.float64).pin_memory()
                tg = torch.from_numpy(gu).cuda()
                assert lib.acoc_result_vjp_dev(bn._h, _lib.ptr(gx), tg.data_ptr(), None, None) == -1
                assert lib.acoc_result_vjp_dev(bn._h, pinned.data_ptr(), tg.data_ptr(), None, None) == -1
                assert b"gx_dev" in lib.acoc_last_error()
            r = bn.result_vjp(gx, gu)
            if ref is None:
                ref = r
            else:
                _same(ref, r)


def _fd_problem(gpu, n):
    return gpu.BatchedNewton(n, TT=TT, state="f64", armijo="lazy", max_iters=100, term_cond=-1e-13)


@pytest.mark.gpu
def test_finite_differences(gpu):
    """32 random directions in (zf, xf, dx0, xref) against central differences of whole float64-state solves (every +h / -h solve is an
    instance of one batch).  The result is an optimum only up to the termination residual (|descent| < 1e-13, a stationarity residual of
    order 3e-7 in the scaled problem) and the central difference has an O(h^2) error: both stay below the stated 2e-4 of the directional
    derivative's scale |gbar| |J v|."""
    import torch
    from aircraftoptimalcontrol_b200 import autograd, refgen
    rng = np.random.default_rng(9)
    tf = TT / 1000
    zf0, xf0 = 2.5, 16.0 * tf
    xr0, ur0 = refgen.step_problem(np.array([xf0]), np.array([zf0]), tf=tf, TT=TT)
    K = 32
    d = rng.normal(size=(K, 3 + 6 + 6 * TT))
    d[:, 3 + 6:] *= 0.02
    d[:, 0:2] *= 0.2
    d[:, 2] = 0
    h = 1e-4
    # base solve with gradients through the autograd Function (expanded references so that xref is differentiable too)
    with _fd_problem(gpu, 1) as bn:
        Q, R, QT = refgen.weights("step")
        bn.set_weights(Q, R, QT)
        xref = torch.tensor(xr0, device="cuda:0", requires_grad=True)
        uref = torch.tensor(ur0, device="cuda:0")
        dx0 = torch.zeros((1, 6), dtype=torch.float64, device="cuda:0", requires_grad=True)
        xs, us = autograd.solve(bn, xref, uref, dx0)
        gbx, gbu = torch.randn_like(xs), torch.randn_like(us)
        g_xref, g_dx0 = torch.autograd.grad((xs * gbx).sum() + (us * gbu).sum(), (xref, dx0))
    g_xref, g_dx0 = g_xref.cpu().numpy()[0], g_dx0.cpu().numpy()[0]
    gbx, gbu = gbx.cpu().numpy(), gbu.cpu().numpy()
    # the perturbed problems: zf and xf move the whole reference family, dx0 the start, the last block xref directly
    tt, zs, vs = refgen.step_bases(tf, TT)
    xr, ur, x0d = [], [], []
    for k in range(K):
        for s in (1, -1):
            zf, xf = zf0 + s * h * d[k, 0], xf0 + s * h * d[k, 1]
            a, b = refgen.step_problem(np.array([xf]), np.array([zf]), tf=tf, TT=TT)
            xr.append(a[0] + s * h * d[k, 9:].reshape(6, TT))
            ur.append(b[0])
            x0d.append(s * h * d[k, 3:9])
    with _fd_problem(gpu, 2 * K) as bp:
        bp.set_weights(Q, R, QT)
        bp.set_refs(np.array(xr), np.array(ur))
        bp.init_guess(dx0=np.array(x0d))
        bp.solve()
        xs2, us2 = bp.result()
    # derivative of the reference family with respect to zf, xf (numpy, same expressions as refgen)
    vx0 = xf0 / tf
    V = np.sqrt((vs * zf0) ** 2 + vx0 ** 2)
    dref_dzf = np.zeros((6, TT)); dref_dzf[1] = zs; dref_dzf[2] = vs * vs * zf0 / V
    dref_dxf = np.zeros((6, TT)); dref_dxf[0] = tt / tf; dref_dxf[2] = vx0 / V / tf
    worst = 0.0
    for k in range(K):
        L = [np.sum(gbx[0] * xs2[2 * k + j]) + np.sum(gbu[0] * us2[2 * k + j]) for j in (0, 1)]
        fd = (L[0] - L[1]) / (2 * h)
        an = (np.sum(g_xref * (d[k, 0] * dref_dzf + d[k, 1] * dref_dxf + d[k, 9:].reshape(6, TT))) + np.sum(g_dx0 * d[k, 3:9]))
        scale = np.linalg.norm(np.r_[gbx.ravel(), gbu.ravel()]) * np.linalg.norm(np.r_[(xs2[2 * k] - xs2[2 * k + 1]).ravel(),
                                                                                        (us2[2 * k] - us2[2 * k + 1]).ravel()]) / (2 * h)
        worst = max(worst, abs(fd - an) / scale)
    print("finite differences: worst |fd - vjp| / scale = %.2e" % worst)
    assert worst < 2e-4


@pytest.mark.gpu
def test_autograd_matches_vjp_and_detects_resolve(gpu):
    """torch.autograd.grad through solve_step equals result_vjp_dev plus the documented chain rule through x0 = xref_0 + dx0; a backward
    pass after the context solved something else raises."""
    import torch
    from aircraftoptimalcontrol_b200 import autograd, refgen
    n, tf = 37, TT / 1000
    rng = np.random.default_rng(8)
    zf = torch.tensor(rng.uniform(1.5, 3.5, n), device="cuda:0", requires_grad=True)
    xf = torch.tensor(rng.uniform(14, 18, n) * tf, device="cuda:0", requires_grad=True)
    dx0 = torch.tensor(rng.normal(size=(n, 6)) * 0.01, device="cuda:0", requires_grad=True)
    with gpu.BatchedNewton(n, TT=TT, armijo="lazy", max_iters=40) as bn:
        bn.set_weights(*refgen.weights("step"))
        xs, us = autograd.solve_step(bn, zf, xf, tf, dx0)
        gx, gu = torch.randn_like(xs), torch.randn_like(us)
        gz, gxf, gd = torch.autograd.grad((xs * gx).sum() + (us * gu).sum(), (zf, xf, dx0), retain_graph=True)
        r = bn.result_vjp_dev(gx, gu)
        tt, zs, vs = refgen.step_bases(tf, TT)
        vx = xf.detach() / tf
        V0 = torch.sqrt((vs[0] * zf.detach()) ** 2 + vx ** 2)
        ez = r["zf"] + zs[0] * r["x0"][:, 1] + (vs[0] * vs[0] * zf.detach() / V0) * r["x0"][:, 2]
        ev = r["vx"] + tt[0] * r["x0"][:, 0] + (vx / V0) * r["x0"][:, 2]
        assert torch.equal(gz, ez) and torch.equal(gxf, ev / tf) and torch.equal(gd, r["x0"])
        xs2, us2 = autograd.solve(bn, torch.tensor(refgen.step_problem(np.full(n, 3.2), np.full(n, 2.0), tf=tf, TT=TT)[0], device="cuda:0"),
                                  torch.tensor(refgen.step_problem(np.full(n, 3.2), np.full(n, 2.0), tf=tf, TT=TT)[1], device="cuda:0"))
        with pytest.raises(RuntimeError):
            torch.autograd.grad((xs * gx).sum(), (zf,))
