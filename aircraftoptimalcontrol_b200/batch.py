"""Batched regularized-Newton solver: thousands to millions of independent aircraft OCP instances on one GPU.

`BatchedNewton` is a thin handle on one libacoc context (include/acoc.h).  It mirrors
`optcon.NewtonMethod` (reference optcon.py:329-529) with a leading instance axis on every array.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib as L


class BatchedNewton:
    """N independent instances of NewtonMethod.optimize (optcon.py:341) solved in lock-step on one GPU.

    Parameters mirror NewtonMethod.__init__ (optcon.py:335-337); `term_cond` defaults to the value the
    reference actually uses (-1e-6, optcon.py:368), `exact_after` to its hard-coded 8 (optcon.py:443).
    state: "f32" reproduces aircraft_simplified.py:300 (next state rounded to float32), "f64" keeps float64.
    armijo: "speculative" evaluates all candidates concurrently, "lazy" evaluates candidate 0 for everyone and
    the rest only where it failed; both return exactly the step the reference's sequential search returns.
    generations: let solve() gather the still-iterating instances into smaller internal batches as the others finish
    (same results, faster tail).
    precision: "f64" (default) is the parity path -- float64 arithmetic like the reference's numpy code.  "f32" is the
    optional FP32 mode: float32 arithmetic and trajectory storage with float64 cost/descent accumulation; it converges
    like the reference does with its float32 state (final cost within 2e-6 relative, states within 2e-3, inputs within
    2e-4 of their range; see DESIGN.md) at roughly half the memory traffic.  `state` is irrelevant in that mode.
    x_storage: "auto" keeps the state iterates as float32 in HBM whenever they are float32 values anyway (state="f32");
    "f64" forces float64 buffers.  Results are bit-identical; "f64" only costs bandwidth (A/B measurements).
    tma: run the time sweeps as warp-private TMA (bulk asynchronous copy) pipelines (default); False uses plain global loads
    (bit-identical results, A/B measurements).
    split: sweep a fully active batch that needs more than one round of resident backward CTAs as two tile ranges on two streams
    (default; identical results, A/B measurements).
    method: "newton" runs NewtonMethod.optimize (optcon.py:341); "gradient" runs GradientMethod.optimize (optcon.py:27, steepest
    descent) with the repaired line-search call described in include/acoc.h (ACOC_METHOD_GRADIENT).  In that mode the `descent`
    entries of history() / stats() are the slope -sum|deltau|^2 handed to the Armijo test (the reference's descent[kk] is its
    negative), `term_cond` keeps its meaning (stop when slope >= term_cond, i.e. descent <= 1e-6, optcon.py:52,157).
    priority: stream priority level 0..15 of this context (ACOC_PRIORITY): of several contexts working on one GPU at the same time the
    one with the higher level gets the SMs first (used by PipelinedNewton to stagger its sub-batches); no effect on results.
    fused: fuse the LQ forward pass with the line-search rollouts that follow it -- with candidate 0 of the lazy search in one sweep
    (any batch size), and, for batches of at most 4096 instances (late survivor generations, single trajectories), with the whole
    Armijo search, get_update then being a copy of the chosen candidate (default; identical results, A/B measurements).
    refs_compact: keep references built by set_refs_step / set_refs_acrobatic in their parametric form in HBM (default; the sweeps then
    move 8 or 0 instead of 64 bytes of references per instance and step); False writes them out as per-instance arrays (ACOC_REFS_EXPANDED;
    identical results, A/B measurements).
    """

    version = 0          # bumped by every call that changes the context's problem or iterates (autograd checks it before backward)
    _refs_param = False  # the context holds parametric references (result_vjp's zf / vx)
    _refs_compact = True

    def __init__(self, n_instances, TT=1000, device=0, state="f32", refs_shared=False, armijo="speculative", params=None, generations=True,
                 max_iters=200, stepsize_0=1.0, cc=0.5, beta=0.7, armijo_maxiters=10, term_cond=-1e-6, exact_after=8, precision="f64",
                 x_storage="auto", tma=True, split=True, fused=True, method="newton", priority=0, refs_compact=True):
        if state not in ("f32", "f64"):
            raise ValueError("state must be 'f32' or 'f64'")
        if armijo not in ("speculative", "lazy"):
            raise ValueError("armijo must be 'speculative' or 'lazy'")
        if precision not in ("f64", "f32"):
            raise ValueError("precision must be 'f64' or 'f32'")
        if x_storage not in ("auto", "f64"):
            raise ValueError("x_storage must be 'auto' or 'f64'")
        if method not in ("newton", "gradient"):
            raise ValueError("method must be 'newton' or 'gradient'")
        self.method = method
        self._refs_compact = bool(refs_compact) and precision == "f64"
        self.N, self.TT, self.device = int(n_instances), int(TT), int(device)
        self.refs_shared = bool(refs_shared)
        self.precision = precision
        flags = ((L.STATE_F64 if state == "f64" else 0) | (L.REFS_SHARED if refs_shared else 0) | (L.ARMIJO_LAZY if armijo == "lazy" else 0)
                 | (0 if generations else L.SOLVE_IN_PLACE) | (L.FP32 if precision == "f32" else 0) | (L.X_F64 if x_storage == "f64" else 0)
                 | (0 if tma else L.NO_TMA) | (0 if split else L.NO_SPLIT) | (0 if fused else L.NO_FUSED) | (0 if refs_compact else L.REFS_EXPANDED)
                 | ((max(0, min(15, int(priority))) & 15) << L.PRIORITY_SHIFT))
        self._h = C.c_void_p(None)
        L.check(L.lib().acoc_ctx_create(self.device, self.N, self.TT, flags, C.addressof(self._h)))
        self.opts = L.NewtonOptions(int(max_iters), int(armijo_maxiters), int(exact_after),
                                    L.METHOD_GRADIENT if method == "gradient" else L.METHOD_NEWTON, float(stepsize_0), float(cc), float(beta),
                                    float(term_cond))
        L.check(L.lib().acoc_set_options(self._h, C.addressof(self.opts)))
        if params is not None:
            self.set_model(params)

    # -- life cycle -----------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            L.lib().acoc_ctx_destroy(self._h)
            self._h = C.c_void_p(None)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def device_bytes(self):
        v = C.c_ulonglong(0)
        L.check(L.lib().acoc_ctx_device_bytes(self._h, C.addressof(v)))
        return v.value

    # -- problem data ---------------------------------------------------------------------------------
    def set_model(self, params):
        self.version += 1
        p = L.f64(params, (9,), "params")
        L.check(L.lib().acoc_set_model(self._h, L.ptr(p)))

    def set_weights(self, QQt, RRt, QQT):
        self.version += 1
        Q, R, QT = L.f64(QQt, (6, 6), "QQt"), L.f64(RRt, (2, 2), "RRt"), L.f64(QQT, (6, 6), "QQT")
        L.check(L.lib().acoc_set_weights(self._h, L.ptr(Q), L.ptr(R), L.ptr(QT)))

    def set_refs(self, xx_ref, uu_ref):
        self.version += 1
        self._refs_param = False
        sx = (6, self.TT) if self.refs_shared else (self.N, 6, self.TT)
        su = (2, self.TT) if self.refs_shared else (self.N, 2, self.TT)
        xr, ur = L.f64(xx_ref, sx, "xx_ref"), L.f64(uu_ref, su, "uu_ref")
        L.check(L.lib().acoc_set_refs(self._h, L.ptr(xr), L.ptr(ur)))

    def set_refs_generated(self, tt, zshape, vshape, zf, vx, xconst, uconst):
        """acoc_set_refs_generated: build the per-instance references on the device from per-instance (zf, vx) and shared time bases."""
        self.version += 1
        self._refs_param = self._refs_compact
        if self.refs_shared:
            raise ValueError("generated references are per instance (refs_shared=False)")
        tt, zs = L.f64(tt, (self.TT,), "tt"), L.f64(zshape, (self.TT,), "zshape")
        vs = None if vshape is None else L.f64(vshape, (self.TT,), "vshape")
        zf = L.f64(np.broadcast_to(np.asarray(zf, dtype=np.float64), (self.N,)), (self.N,), "zf")
        vx = L.f64(np.broadcast_to(np.asarray(vx, dtype=np.float64), (self.N,)), (self.N,), "vx")
        xc, uc = L.f64(xconst, (6,), "xconst"), L.f64(uconst, (2,), "uconst")
        L.check(L.lib().acoc_set_refs_generated(self._h, L.ptr(tt), L.ptr(zs), L.ptr(vs), L.ptr(zf), L.ptr(vx), L.ptr(xc), L.ptr(uc)))

    def set_refs_step(self, zf, xf, tf=1):
        """The step-maneuver references of main_newton_method.py:96-142 for final heights zf (N,) and final positions xf (N,), built on
        the device; bit-identical to set_refs(*refgen.step_problem(xf, zf, tf, TT))."""
        from . import refgen
        tt, s, ds = refgen.step_bases(tf, self.TT)
        vx = (np.asarray(xf, dtype=np.float64) - 0) / tf
        self.set_refs_generated(tt, s, ds, zf, vx, *refgen.STEP_CONST)

    def set_refs_acrobatic(self, zf, xf=18, tf=1):
        """The acrobatic references of acrobatic_newton.py:99-154 for bump heights zf (N,), built on the device; bit-identical to
        set_refs(*refgen.acrobatic_problem(zf, xf, tf, TT))."""
        from . import refgen
        tt, bump = refgen.acrobatic_bases(tf, self.TT)
        self.set_refs_generated(tt, bump, None, zf, (xf - 0) / tf, *refgen.ACRO_CONST)

    def refs(self):
        """(xx_ref, uu_ref) held by the context, in set_refs' layout."""
        sx = (6, self.TT) if self.refs_shared else (self.N, 6, self.TT)
        su = (2, self.TT) if self.refs_shared else (self.N, 2, self.TT)
        xr, ur = np.empty(sx), np.empty(su)
        L.check(L.lib().acoc_get_refs(self._h, L.ptr(xr), L.ptr(ur)))
        return xr, ur

    def set_init(self, xx_init, uu_init):
        self.version += 1
        xi, ui = L.f64(xx_init, (self.N, 6, self.TT), "xx_init"), L.f64(uu_init, (self.N, 2, self.TT), "uu_init")
        L.check(L.lib().acoc_set_init(self._h, L.ptr(xi), L.ptr(ui)))

    def init_guess(self, kp=5.0, kt=2.5, dx0=None):
        """Dynamics.get_initial_trajectory (aircraft_simplified.py:126-148) for every instance, on the device.
        dx0 (N,6): start from xx_ref[:,0] + dx0 (perturbed-initial-state batches)."""
        self.version += 1
        d = None if dx0 is None else L.f64(dx0, (self.N, 6), "dx0")
        L.check(L.lib().acoc_init_guess(self._h, float(kp), float(kt), L.ptr(d)))

    # -- solve ------------------------------------------------------------------------------------------
    def iterate(self, n_iters=1, count_active=True):
        self.version += 1
        na = C.c_int(-1)
        L.check(L.lib().acoc_newton_iterate(self._h, int(n_iters), C.addressof(na) if count_active else None))
        return na.value

    def solve(self):
        self.version += 1
        tot = C.c_longlong(0)
        L.check(L.lib().acoc_newton_solve(self._h, C.addressof(tot)))
        return tot.value

    def solve_deliver(self, out, x0=None):
        """solve() and the read-back of the result in one call: out = (xx_star (N,6,TT) float32 or float64, uu_star (N,2,TT) float64).
        With page-locked arrays (e.g. torch pin_memory) the results are written straight into them and the finished instances are
        delivered while the last ones still iterate (acoc_newton_solve_deliver); pageable arrays get the same values through
        solve() + result().  Returns (total Newton iterations, x0 (N,6))."""
        self.version += 1
        xs, us = out
        L.out_array(xs, (self.N, 6, self.TT), (np.float32, np.float64), "xx_star")
        L.out_array(us, (self.N, 2, self.TT), np.float64, "uu_star")
        x0 = np.empty((self.N, 6)) if x0 is None else L.out_array(x0, (self.N, 6), np.float64, "x0")
        tot = C.c_longlong(0)
        L.check(L.lib().acoc_newton_solve_deliver(self._h, L.ptr(xs), int(xs.dtype == np.float32), L.ptr(us), L.ptr(x0), C.addressof(tot)))
        return tot.value, x0

    def sync(self):
        L.check(L.lib().acoc_sync(self._h))

    # -- pieces (parity tests, drop-in method names) ---------------------------------------------------------
    def eval_cost(self):
        J = np.zeros(self.N)
        L.check(L.lib().acoc_eval_cost(self._h, L.ptr(J)))
        return J

    def backward(self, exact=False):
        L.check(L.lib().acoc_backward(self._h, int(bool(exact))))

    def forward(self):
        d = np.zeros(self.N)
        L.check(L.lib().acoc_forward(self._h, L.ptr(d)))
        return d

    def gradient(self):
        """One costate sweep of GradientMethod.optimize (optcon.py:95-118) on the current iterate: writes deltau, returns the
        reference's descent = sum_t |deltau_t|^2 per instance."""
        d = np.zeros(self.N)
        L.check(L.lib().acoc_gradient(self._h, L.ptr(d)))
        return d

    def armijo_sweep(self, steps):
        """Costs (N, len(steps)) of the rollouts u + steps[k]*deltau: the data behind the reference's visu_armijo plot
        (optcon.py:280-296, which uses np.linspace(0, stepsize_0, 10))."""
        st = L.f64(np.asarray(steps, dtype=np.float64).reshape(-1), None, "steps")
        costs = np.zeros((self.N, st.size))
        L.check(L.lib().acoc_armijo_sweep(self._h, int(st.size), L.ptr(st), L.ptr(costs)))
        return costs

    def set_deltau(self, deltau):
        self.version += 1
        du = L.f64(deltau, (self.N, 2, self.TT), "deltau")
        L.check(L.lib().acoc_set_deltau(self._h, L.ptr(du)))

    def set_scalars(self, J=None, descent=None):
        self.version += 1
        Jc = None if J is None else L.f64(J, (self.N,), "J")
        dc = None if descent is None else L.f64(descent, (self.N,), "descent")
        L.check(L.lib().acoc_set_scalars(self._h, L.ptr(Jc), L.ptr(dc)))

    def armijo(self):
        s, costs = np.zeros(self.N), np.zeros((self.N, self.opts.armijo_maxiters))
        L.check(L.lib().acoc_armijo(self._h, L.ptr(s), L.ptr(costs)))
        return s, costs

    def update(self, stepsize=None):
        self.version += 1
        s = None if stepsize is None else L.f64(np.broadcast_to(np.asarray(stepsize, dtype=np.float64), (self.N,)), (self.N,), "stepsize")
        L.check(L.lib().acoc_update(self._h, L.ptr(s)))

    # -- read-back --------------------------------------------------------------------------------------
    def result(self, out=None):
        """(xx_star (N,6,TT), uu_star (N,2,TT)) with the reference's return semantics (optcon.py:503-505)."""
        if out is None:
            xs, us = np.empty((self.N, 6, self.TT)), np.empty((self.N, 2, self.TT))
        else:
            xs, us = out
            L.out_array(xs, (self.N, 6, self.TT), np.float64, "xx_star")
            L.out_array(us, (self.N, 2, self.TT), np.float64, "uu_star")
        L.check(L.lib().acoc_get_result(self._h, L.ptr(xs), L.ptr(us)))
        return xs, us

    def result_f32(self, out=None):
        """(xx_star float32 (N,6,TT), uu_star float64 (N,2,TT), x0 float64 (N,6)): the result with the states as the float32 values
        they are under the reference's state quantisation (aircraft_simplified.py:300) -- lossless, 40 instead of 64 bytes per time
        step over the bus.  xx_star[:, :, 0] is float32(x0); the exact x0 comes back separately.  Raises for float64-state contexts."""
        if out is None:
            xs, us = np.empty((self.N, 6, self.TT), dtype=np.float32), np.empty((self.N, 2, self.TT))
        else:
            xs, us = out
            L.out_array(xs, (self.N, 6, self.TT), np.float32, "xx_star")
            L.out_array(us, (self.N, 2, self.TT), np.float64, "uu_star")
        x0 = np.empty((self.N, 6))
        L.check(L.lib().acoc_get_result_f32(self._h, L.ptr(xs), L.ptr(us), L.ptr(x0)))
        return xs, us, x0

    def iterate_at(self, which=0):
        xs, us = np.empty((self.N, 6, self.TT)), np.empty((self.N, 2, self.TT))
        L.check(L.lib().acoc_get_iterate(self._h, int(which), L.ptr(xs), L.ptr(us)))
        return xs, us

    def deltau(self):
        du = np.empty((self.N, 2, self.TT))
        L.check(L.lib().acoc_get_deltau(self._h, L.ptr(du)))
        return du

    def gains(self):
        K, s = np.empty((self.N, 2, 6, self.TT)), np.empty((self.N, 2, self.TT))
        L.check(L.lib().acoc_get_gains(self._h, L.ptr(K), L.ptr(s)))
        return K, s

    def history(self):
        mi = self.opts.max_iters
        J, d, s = np.zeros((self.N, mi)), np.zeros((self.N, mi)), np.zeros((self.N, mi))
        nc = np.zeros((self.N, mi), dtype=np.int32)
        L.check(L.lib().acoc_get_history(self._h, L.ptr(J), L.ptr(d), L.ptr(s), L.ptr(nc)))
        return dict(JJ=J, descent=d, stepsize=s, n_armijo=nc)

    def stats(self):
        it, st, nr = (np.zeros(self.N, dtype=np.int32) for _ in range(3))
        J, d = np.zeros(self.N), np.zeros(self.N)
        L.check(L.lib().acoc_get_stats(self._h, L.ptr(it), L.ptr(st), L.ptr(J), L.ptr(d), L.ptr(nr)))
        return dict(iters=it, status=st, J=J, descent=d, n_reg=nr)

    # -- closed-loop tracking of every instance (lqr_tracking.py:245-283 per instance) ---------------------------------------------
    def track(self, delta=None, QQt=None, RRt=None, QQT=None):
        """Fly the closed loop of the reference's lqr_tracking around EVERY instance's own result (what result() returns now), on the
        device: gains of the time-varying LQR along that nominal with the tracking weights (default lqr_tracking.default_weights(),
        independent of the Newton weights), then u = u* + K (x - x*) from x*_0 + delta.  delta (N,6), (6,) broadcast, or None (zero).
        Returns dict(err_max (N,6) = max_t |x_t - x*_t|, err_final (N,6) at t = TT-1, n_reg (N) = steps that took the +0.5 I gain
        branch); NaN summaries mark an instance whose nominal is not finite.  Trajectories: tracked(); gains: track_gains().
        Changes nothing of the solve."""
        from .lqr_tracking import default_weights
        dQ, dR, dQT = default_weights()
        Q = L.f64(dQ if QQt is None else QQt, (6, 6), "QQt")
        R = L.f64(dR if RRt is None else RRt, (2, 2), "RRt")
        QT = L.f64(dQT if QQT is None else QQT, (6, 6), "QQT")
        d = None
        if delta is not None:
            d = np.asarray(delta, dtype=np.float64)
            if d.shape == (6,):
                d = np.broadcast_to(d, (self.N, 6))
            d = L.f64(d, (self.N, 6), "delta")
        em, ef, nr = np.empty((self.N, 6)), np.empty((self.N, 6)), np.empty(self.N, dtype=np.int32)
        L.check(L.lib().acoc_track(self._h, L.ptr(Q), L.ptr(R), L.ptr(QT), L.ptr(d), L.ptr(em), L.ptr(ef), L.ptr(nr)))
        return dict(err_max=em, err_final=ef, n_reg=nr)

    def track_mc(self, delta, QQt=None, RRt=None, QQT=None, tol=None, per_sample=False):
        """Monte Carlo dispersion of track(): M closed loops per instance, on the device, along the same nominal (what result() returns
        now) and gains as track().  delta (M,6) (the same perturbations for every instance) or (N,M,6); tol (6,) or None.  Returns
        dict(worst_max (N,6) = max over samples of max_t |x_t - x*_t| (NaN if any sample is NaN), mean_final (N,6) = mean over samples
        of |x_{TT-1} - x*_{TT-1}|, n_reg (N)[, n_within (N) = samples whose max error is within tol in every state, with tol]
        [, err_max, err_final (N,M,6) per sample, with per_sample=True]).  The per-sample summaries are bit-identical to
        track(delta[:, m]); no trajectory is kept (fly track(delta[:, m]) for the trajectory of sample m).  Afterwards track_gains() and
        track_timing() report this call and tracked() raises until the next track().  Changes nothing of the solve."""
        from .lqr_tracking import default_weights, mc_call, mc_deltas
        dQ, dR, dQT = default_weights()
        Q = L.f64(dQ if QQt is None else QQt, (6, 6), "QQt")
        R = L.f64(dR if RRt is None else RRt, (2, 2), "RRt")
        QT = L.f64(dQT if QQT is None else QQT, (6, 6), "QQT")
        d, shared, M = mc_deltas(delta, self.N)
        return mc_call(lambda t, out: L.lib().acoc_track_mc(self._h, L.ptr(Q), L.ptr(R), L.ptr(QT), M, L.ptr(d), int(shared), t, out),
                       self.N, M, tol, per_sample)

    def tracked(self, out=None):
        """(xx_reg (N,6,TT), uu_reg (N,2,TT)) of the last track()."""
        if out is None:
            xr, ur = np.empty((self.N, 6, self.TT)), np.empty((self.N, 2, self.TT))
        else:
            xr, ur = out
            L.out_array(xr, (self.N, 6, self.TT), np.float64, "xx_reg")
            L.out_array(ur, (self.N, 2, self.TT), np.float64, "uu_reg")
        L.check(L.lib().acoc_get_tracked(self._h, L.ptr(xr), L.ptr(ur)))
        return xr, ur

    def track_gains(self):
        """K (N,2,6,TT) of the last track(): lqr_tracking's KK for every instance."""
        K = np.empty((self.N, 2, 6, self.TT))
        L.check(L.lib().acoc_get_track_gains(self._h, L.ptr(K)))
        return K

    def track_timing(self):
        """Device time (ms) of the last track(): total and per kernel (nominal, gains sweep, rollout)."""
        ms = (C.c_double * 4)()
        L.check(L.lib().acoc_get_track_timing(self._h, C.addressof(ms)))
        return dict(total_ms=ms[0], nominal_ms=ms[1], gains_ms=ms[2], rollout_ms=ms[3])

    # -- device-resident inputs and outputs (include/acoc.h): CUDA tensors of this context's device, no host round trip ------------
    # Each method is the twin of the method without _dev (same shapes, state rules, refusals and bit-identical results).  Tensors
    # must be contiguous and of the exact shape and dtype; the call is ordered after the work queued so far on the current torch
    # stream of the device and returns once its outputs are written, so they may be used on any stream.
    def set_refs_dev(self, xx_ref, uu_ref):
        """set_refs from float64 CUDA tensors xx_ref (N,6,TT) / uu_ref (N,2,TT), or (6,TT) / (2,TT) with refs_shared."""
        self.version += 1
        self._refs_param = False
        import torch
        sx = (6, self.TT) if self.refs_shared else (self.N, 6, self.TT)
        su = (2, self.TT) if self.refs_shared else (self.N, 2, self.TT)
        xr = L.dev_tensor(xx_ref, self.device, sx, torch.float64, "xx_ref")
        ur = L.dev_tensor(uu_ref, self.device, su, torch.float64, "uu_ref")
        L.check(L.lib().acoc_set_refs_dev(self._h, xr, ur, L.dev_stream(self.device)))

    def set_init_dev(self, xx_init, uu_init):
        """set_init from float64 CUDA tensors xx_init (N,6,TT) / uu_init (N,2,TT)."""
        self.version += 1
        import torch
        xi = L.dev_tensor(xx_init, self.device, (self.N, 6, self.TT), torch.float64, "xx_init")
        ui = L.dev_tensor(uu_init, self.device, (self.N, 2, self.TT), torch.float64, "uu_init")
        L.check(L.lib().acoc_set_init_dev(self._h, xi, ui, L.dev_stream(self.device)))

    def result_dev(self, x_dtype=None, out=None):
        """(xx_star (N,6,TT), uu_star (N,2,TT) float64, x0 (N,6) float64) as CUDA tensors: result() with x_dtype=torch.float64 (default),
        result_f32() with torch.float32 (refused for float64-state contexts).  x0 is the exact initial state either way.
        out = (xx_star, uu_star) tensors to write into."""
        import torch
        x_dtype = torch.float64 if x_dtype is None else x_dtype
        if x_dtype not in (torch.float32, torch.float64):
            raise ValueError("x_dtype must be torch.float32 or torch.float64")
        dev = torch.device("cuda", self.device)
        if out is None:
            xs = torch.empty((self.N, 6, self.TT), dtype=x_dtype, device=dev)
            us = torch.empty((self.N, 2, self.TT), dtype=torch.float64, device=dev)
        else:
            xs, us = out
        x0 = torch.empty((self.N, 6), dtype=torch.float64, device=dev)
        px = L.dev_tensor(xs, self.device, (self.N, 6, self.TT), x_dtype, "xx_star")
        pu = L.dev_tensor(us, self.device, (self.N, 2, self.TT), torch.float64, "uu_star")
        L.check(L.lib().acoc_get_result_dev(self._h, px, int(x_dtype == torch.float32), pu, x0.data_ptr(), L.dev_stream(self.device)))
        return xs, us, x0

    def tracked_dev(self, out=None):
        """tracked() as float64 CUDA tensors (xx_reg (N,6,TT), uu_reg (N,2,TT)); out = such tensors to write into."""
        import torch
        if out is None:
            dev = torch.device("cuda", self.device)
            out = (torch.empty((self.N, 6, self.TT), dtype=torch.float64, device=dev),
                   torch.empty((self.N, 2, self.TT), dtype=torch.float64, device=dev))
        xr, ur = out
        px = L.dev_tensor(xr, self.device, (self.N, 6, self.TT), torch.float64, "xx_reg")
        pu = L.dev_tensor(ur, self.device, (self.N, 2, self.TT), torch.float64, "uu_reg")
        L.check(L.lib().acoc_get_tracked_dev(self._h, px, pu, L.dev_stream(self.device)))
        return xr, ur

    def track_gains_dev(self, out=None):
        """track_gains() as a float64 CUDA tensor K (N,2,6,TT); out = such a tensor to write into."""
        import torch
        K = torch.empty((self.N, 2, 6, self.TT), dtype=torch.float64, device=torch.device("cuda", self.device)) if out is None else out
        pk = L.dev_tensor(K, self.device, (self.N, 2, 6, self.TT), torch.float64, "K")
        L.check(L.lib().acoc_get_track_gains_dev(self._h, pk, L.dev_stream(self.device)))
        return K

    def track_mc_dev(self, delta, QQt=None, RRt=None, QQT=None, tol=None, per_sample=False):
        """track_mc() with the perturbations and every output as CUDA tensors: delta a float64 tensor (M,6) (shared by every instance)
        or (N,M,6); returns track_mc's dict with float64 / int32 tensors in place of arrays.  The weights and tol are host arrays."""
        import torch
        from .lqr_tracking import default_weights, mc_call, mc_layout
        dQ, dR, dQT = default_weights()
        Q = L.f64(dQ if QQt is None else QQt, (6, 6), "QQt")
        R = L.f64(dR if RRt is None else RRt, (2, 2), "RRt")
        QT = L.f64(dQT if QQT is None else QQT, (6, 6), "QQT")
        if not isinstance(delta, torch.Tensor):
            raise ValueError("delta must be a torch.Tensor, got %s" % type(delta).__name__)
        shared, M = mc_layout(delta.shape, self.N)
        d = L.dev_tensor(delta, self.device, delta.shape, torch.float64, "delta")
        dev, stream = torch.device("cuda", self.device), L.dev_stream(self.device)

        def empty(shape, integer):
            return torch.empty(shape, dtype=torch.int32 if integer else torch.float64, device=dev)
        return mc_call(lambda t, out: L.lib().acoc_track_mc_dev(self._h, L.ptr(Q), L.ptr(R), L.ptr(QT), M, d, int(shared), t, out, stream),
                       self.N, M, tol, per_sample, empty)

    # -- derivative of the optimum (include/acoc.h "derivative of the optimum") ------------------------------------------------------
    def _vjp_out(self, empty):
        o = dict(xref=empty((self.N, 6, self.TT), False), uref=empty((self.N, 2, self.TT), False), x0=empty((self.N, 6), False),
                 zf=empty((self.N,), False) if self._refs_param else None, vx=empty((self.N,), False) if self._refs_param else None,
                 n_indef=empty((self.N,), True))
        return o

    def result_vjp(self, gx, gu):
        """Reverse-mode derivative of result() (the optimum of the smooth float64 problem, linearised at the returned point) with respect
        to the references and the initial state: upstream gradients gx (N,6,TT), gu (N,2,TT) with respect to result()'s arrays -> dict(
        xref (N,6,TT), uref (N,2,TT), x0 (N,6), zf (N) and vx (N) with parametric references (set_refs_step / set_refs_acrobatic; else None),
        n_indef (N) = steps whose G = R + B'PB is not positive definite).  zf / vx do not include the path through x0; see
        aircraftoptimalcontrol_b200.autograd.  Changes nothing of the solve."""
        g1, g2 = L.f64(gx, (self.N, 6, self.TT), "gx"), L.f64(gu, (self.N, 2, self.TT), "gu")
        o = self._vjp_out(lambda shape, integer: np.empty(shape, dtype=np.int32 if integer else np.float64))
        s = L.VjpOut(*(L.ptr(o[k]) for k in ("xref", "uref", "x0", "zf", "vx", "n_indef")))
        L.check(L.lib().acoc_result_vjp(self._h, L.ptr(g1), L.ptr(g2), C.addressof(s)))
        return o

    def result_vjp_dev(self, gx, gu):
        """result_vjp with float64 CUDA tensors gx (N,6,TT), gu (N,2,TT); returns the same dict with CUDA tensors (n_indef int32)."""
        import torch
        p1 = L.dev_tensor(gx, self.device, (self.N, 6, self.TT), torch.float64, "gx")
        p2 = L.dev_tensor(gu, self.device, (self.N, 2, self.TT), torch.float64, "gu")
        dev = torch.device("cuda", self.device)
        o = self._vjp_out(lambda shape, integer: torch.empty(shape, dtype=torch.int32 if integer else torch.float64, device=dev))
        s = L.VjpOut(*(None if o[k] is None else o[k].data_ptr() for k in ("xref", "uref", "x0", "zf", "vx", "n_indef")))
        L.check(L.lib().acoc_result_vjp_dev(self._h, p1, p2, C.addressof(s), L.dev_stream(self.device)))
        return o

    def set_profiling(self, on=True):
        L.check(L.lib().acoc_set_profiling(self._h, int(bool(on))))

    def timing(self):
        tot = C.c_double(0)
        ph = (C.c_double * 6)()
        nl = C.c_longlong(0)
        L.check(L.lib().acoc_get_timing(self._h, C.addressof(tot), C.addressof(ph), C.addressof(nl)))
        names = ("cost", "backward", "forward", "candidates", "select", "update")
        return dict(total_ms=tot.value, launches=nl.value, phases={k: ph[i] for i, k in enumerate(names)})



class PipelinedNewton:
    """A large batch solved as `n_chunks` independent sub-batches, each with its own context/stream and its own host
    thread, so that the host->device copy of one chunk, the Newton iterations of another and the device->host copy of
    a third overlap.  Instances are independent, so chunking changes no result.  The sub-contexts are created once and
    reused across `solve` calls.
    """

    def __init__(self, n_instances, n_chunks=4, TT=1000, device=0, stagger=True, **solver_kw):
        self.N, self.TT = int(n_instances), int(TT)
        n_chunks = max(1, min(int(n_chunks), self.N))
        self.bounds = [(self.N * k) // n_chunks for k in range(n_chunks + 1)]
        # stagger: earlier sub-batches get a higher stream priority, so that they finish (and download) one after the other while the
        # later ones still iterate, instead of all sub-batches finishing together with every download left for the end
        self.parts = [BatchedNewton(self.bounds[k + 1] - self.bounds[k], TT=TT, device=device,
                                    priority=(min(15, n_chunks - k) if stagger and n_chunks > 1 else 0), **solver_kw) for k in range(n_chunks)]

    def close(self):
        for p in self.parts:
            p.close()
        self.parts = []

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_weights(self, QQt, RRt, QQT):
        for p in self.parts:
            p.set_weights(QQt, RRt, QQT)

    def solve(self, xx_ref=None, uu_ref=None, xx_init=None, uu_init=None, dx0=None, out=None, refs=None, x_dtype=np.float64, direct=True):
        """xx_ref (N,6,TT), uu_ref (N,2,TT) per-instance references (pinned host memory makes the copies fast), or
        refs = ("step", zf (N,), xf (N,)[, tf]) / ("acrobatic", zf (N,)[, xf, tf]): the scripts' reference generators run on the device
        (BatchedNewton.set_refs_step / set_refs_acrobatic; bit-identical arrays, 16 bytes per instance over the bus).  Initial
        guess = (xx_init, uu_init) if given, else the device P-law rollout (optionally started at xx_ref[:,0] + dx0).
        x_dtype = np.float32 downloads the states as the float32 values they are (BatchedNewton.result_f32; column 0 then holds
        float32(x0), the exact x0 is stats["x0"]).  direct: deliver through BatchedNewton.solve_deliver (results written straight into
        page-locked `out` arrays while the last instances still iterate; pageable arrays: same values, staged download).
        Returns (xx_star, uu_star, stats) with stats = dict(iters, status, J, descent, n_reg), each of length N."""
        import threading

        N, TT = self.N, self.TT
        f32 = np.dtype(x_dtype) == np.float32
        if (xx_ref is None) == (refs is None):
            raise ValueError("give either xx_ref/uu_ref or refs=(kind, ...)")
        if np.dtype(x_dtype) not in (np.dtype(np.float32), np.dtype(np.float64)):
            raise ValueError("x_dtype must be float32 or float64")
        xs, us = out if out is not None else (np.empty((N, 6, TT), dtype=x_dtype), np.empty((N, 2, TT)))
        L.out_array(xs, (N, 6, TT), x_dtype, "xx_star")     # (the sub-batches write into slices of these arrays)
        L.out_array(us, (N, 2, TT), np.float64, "uu_star")
        for name, a, cols in (("xx_ref", xx_ref, 6), ("uu_ref", uu_ref, 2), ("xx_init", xx_init, 6), ("uu_init", uu_init, 2)):
            if a is not None and tuple(np.shape(a)) != (N, cols, TT):
                raise ValueError("%s has shape %s, expected %s" % (name, np.shape(a), (N, cols, TT)))
        if (xx_ref is None) != (uu_ref is None) or (xx_init is None) != (uu_init is None):
            raise ValueError("xx_ref/uu_ref and xx_init/uu_init are given in pairs")
        if dx0 is not None and tuple(np.shape(dx0)) != (N, 6):
            raise ValueError("dx0 has shape %s, expected %s" % (np.shape(dx0), (N, 6)))
        stats = dict(iters=np.zeros(N, dtype=np.int32), status=np.zeros(N, dtype=np.int32), J=np.zeros(N), descent=np.zeros(N),
                     n_reg=np.zeros(N, dtype=np.int32))
        x0_out = np.zeros((N, 6)) if f32 else None
        errors = []
        # The host<->device link is the shared resource of the two copy phases, so they are serialised across sub-batches
        # (uploads in sub-batch order, downloads as sub-batches finish): sub-batch 0 starts iterating as soon as ITS references
        # have arrived while the others are still uploading, and the downloads trail the solves the same way.  Without this
        # all sub-batches would copy, then iterate, then copy back in lock-step and nothing would overlap.
        turn = threading.Condition()
        state = {"next_upload": 0}
        download = threading.Lock()

        def work(k):
            lo, hi = self.bounds[k], self.bounds[k + 1]
            bn = self.parts[k]
            try:
                with turn:
                    turn.wait_for(lambda: state["next_upload"] == k or errors)
                if errors:  # another sub-batch failed: do not upload / solve this one
                    return
                try:
                    if refs is None:
                        bn.set_refs(xx_ref[lo:hi], uu_ref[lo:hi])
                    elif refs[0] == "step":
                        bn.set_refs_step(np.asarray(refs[1])[lo:hi], np.asarray(refs[2])[lo:hi], *refs[3:])
                    elif refs[0] == "acrobatic":
                        bn.set_refs_acrobatic(np.asarray(refs[1])[lo:hi], *refs[2:])
                    else:
                        raise ValueError("refs[0] must be 'step' or 'acrobatic'")
                    if xx_init is not None:
                        bn.set_init(xx_init[lo:hi], uu_init[lo:hi])
                except Exception as e:   # recorded BEFORE the turn is handed on, so that the next sub-batch sees it and stays out
                    errors.append(e)
                    raise
                finally:
                    with turn:
                        state["next_upload"] = k + 1
                        turn.notify_all()
                if xx_init is None:
                    bn.init_guess(dx0=None if dx0 is None else dx0[lo:hi])
                if direct:   # results written straight into the (page-locked) output arrays, overlapping the tail of the solve
                    x0c = bn.solve_deliver((xs[lo:hi], us[lo:hi]))[1]
                    if f32:
                        x0_out[lo:hi] = x0c
                    st = bn.stats()
                else:
                    bn.solve()
                    with download:
                        if f32:
                            x0_out[lo:hi] = bn.result_f32(out=(xs[lo:hi], us[lo:hi]))[2]
                        else:
                            bn.result(out=(xs[lo:hi], us[lo:hi]))
                        st = bn.stats()
                for key in stats:
                    stats[key][lo:hi] = st[key]
            except Exception as e:  # surfaced after the join
                if not any(e is x for x in errors):
                    errors.append(e)
                with turn:
                    turn.notify_all()

        threads = [threading.Thread(target=work, args=(k,)) for k in range(len(self.parts))]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        if errors:
            raise errors[0]
        if f32:
            stats["x0"] = x0_out
        return xs, us, stats

    def track(self, delta=None, QQt=None, RRt=None, QQT=None):
        """BatchedNewton.track on every sub-batch (each on its own context): delta (N,6) or (6,); returns the concatenated summaries."""
        d = None
        if delta is not None:
            d = np.asarray(delta, dtype=np.float64)
            if d.shape == (6,):
                d = np.broadcast_to(d, (self.N, 6))
            if d.shape != (self.N, 6):
                raise ValueError("delta has shape %s, expected %s or (6,)" % (d.shape, (self.N, 6)))
        res = [p.track(None if d is None else d[lo:hi], QQt, RRt, QQT) for p, lo, hi in zip(self.parts, self.bounds[:-1], self.bounds[1:])]
        return {k: np.concatenate([r[k] for r in res]) for k in ("err_max", "err_final", "n_reg")}

    def track_mc(self, delta, QQt=None, RRt=None, QQT=None, tol=None, per_sample=False):
        """BatchedNewton.track_mc on every sub-batch: delta (M,6) as it is, (N,M,6) sliced; returns the concatenated results."""
        from .lqr_tracking import mc_deltas
        d, shared, _ = mc_deltas(delta, self.N)
        res = [p.track_mc(d if shared else d[lo:hi], QQt, RRt, QQT, tol, per_sample)
               for p, lo, hi in zip(self.parts, self.bounds[:-1], self.bounds[1:])]
        return {k: np.concatenate([r[k] for r in res]) for k in res[0]}

    def tracked(self, out=None):
        """(xx_reg (N,6,TT), uu_reg (N,2,TT)) of the last track()."""
        xr, ur = out if out is not None else (np.empty((self.N, 6, self.TT)), np.empty((self.N, 2, self.TT)))
        L.out_array(xr, (self.N, 6, self.TT), np.float64, "xx_reg")
        L.out_array(ur, (self.N, 2, self.TT), np.float64, "uu_reg")
        for p, lo, hi in zip(self.parts, self.bounds[:-1], self.bounds[1:]):
            p.tracked(out=(xr[lo:hi], ur[lo:hi]))
        return xr, ur
