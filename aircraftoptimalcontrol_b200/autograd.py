"""Differentiable batched solves: torch.autograd.Functions whose forward pass is a BatchedNewton solve on the device and whose backward
pass is BatchedNewton.result_vjp_dev (acoc_result_vjp, definition in include/acoc.h).  A network that produces references (whole
trajectories, or the parameters of the scripts' maneuvers) can be trained through the optimizer:

    xs, us = autograd.solve_step(bn, zf, xf)          # zf, xf: CUDA tensors (N,) with requires_grad
    loss = ((xs[:, 1, -1] - target) ** 2).mean()
    loss.backward()                                   # zf.grad, xf.grad

What is differentiated: the optimum of the smooth float64 problem (no float32 rounding of the next state), linearised at the point the
solve returned, with respect to the references and the initial state.  The initial GUESS gets no gradient: a local optimum does not
depend on where the iteration started (locally, away from the basin boundaries), so d(result)/d(guess) is zero.  With init_guess the
initial state is xi = xx_ref[:, :, 0] + dx0, so the gradient of xi goes to both dx0 and xx_ref[:, :, 0] (and through them to zf, xf).
The solve's own termination residual sets how exactly the result is an optimum; use state="f64" and a tight term_cond when the
derivative should match finite differences closely.

Not differentiated: the weights, the model parameters, the FP32 mode, PipelinedNewton and the tracking calls.
A backward pass raises if the context was used for anything else (another solve, new references, ...) after the forward pass.
"""
from __future__ import annotations

import torch

from . import refgen


def _dx0_host(bn, dx0):
    return None if dx0 is None else dx0.detach().to("cpu", torch.float64).numpy().reshape(bn.N, 6)


def _solve_and_read(bn, kp, kt, dx0):
    bn.init_guess(kp, kt, _dx0_host(bn, dx0))
    bn.solve()
    xs, us, _ = bn.result_dev(torch.float64)
    return xs, us


def _vjp(ctx, gx, gu):
    bn = ctx.bn
    if bn.version != ctx.version:
        raise RuntimeError("autograd: the BatchedNewton context changed after the forward pass (another solve, new references or iterates); "
                           "its derivative is no longer available")
    return bn.result_vjp_dev(gx.to(torch.float64).contiguous(), gu.to(torch.float64).contiguous())


class _Solve(torch.autograd.Function):
    @staticmethod
    def forward(ctx, bn, kp, kt, xx_ref, uu_ref, dx0):
        bn.set_refs_dev(xx_ref.detach().contiguous(), uu_ref.detach().contiguous())
        xs, us = _solve_and_read(bn, kp, kt, dx0)
        ctx.bn, ctx.version, ctx.has_dx0 = bn, bn.version, dx0 is not None
        return xs, us

    @staticmethod
    def backward(ctx, gx, gu):
        r = _vjp(ctx, gx, gu)
        bn = ctx.bn
        gxr, gur = r["xref"], r["uref"]
        gxr[:, :, 0] += r["x0"]  # xi = xx_ref[:, :, 0] + dx0
        if bn.refs_shared:
            gxr, gur = gxr.sum(0), gur.sum(0)
        gdx0 = r["x0"] if ctx.has_dx0 and ctx.needs_input_grad[5] else None
        return None, None, None, gxr, gur, gdx0


class _SolveParam(torch.autograd.Function):
    @staticmethod
    def forward(ctx, bn, kind, tf, kp, kt, zf, xf, dx0):
        if not bn._refs_compact:
            raise ValueError("solve_step / solve_acrobatic need a context that keeps parametric references (refs_compact=True, precision='f64')")
        z, x = zf.detach().to("cpu", torch.float64).numpy(), xf.detach().to("cpu", torch.float64).numpy()
        if kind == "step":
            bn.set_refs_step(z, x, tf)
            tt, zs, vs = refgen.step_bases(tf, bn.TT)
        else:
            bn.set_refs_acrobatic(z, x, tf)
            (tt, zs), vs = refgen.acrobatic_bases(tf, bn.TT), None
        xs, us = _solve_and_read(bn, kp, kt, dx0)
        ctx.bn, ctx.version, ctx.has_dx0, ctx.tf = bn, bn.version, dx0 is not None, tf
        ctx.t0 = (tt[0], zs[0], None if vs is None else vs[0])
        ctx.save_for_backward(zf.detach().to(torch.float64), xf.detach().to(torch.float64))
        return xs, us

    @staticmethod
    def backward(ctx, gx, gu):
        r = _vjp(ctx, gx, gu)
        zf, xf = ctx.saved_tensors
        vx = (xf - 0) / ctx.tf
        xi_bar = r["x0"]
        tt0, zs0, vs0 = ctx.t0
        # xi = xref_0(zf, vx) + dx0: the chain rule through the references at t = 0 (X_0 = vx tt_0, Z_0 = zs_0 zf, V_0 for the step)
        zf_bar = r["zf"] + zs0 * xi_bar[:, 1]
        vx_bar = r["vx"] + tt0 * xi_bar[:, 0]
        if vs0 is not None:
            V0 = torch.sqrt((vs0 * zf) ** 2 + vx ** 2)
            zf_bar = zf_bar + (vs0 * vs0 * zf / V0) * xi_bar[:, 2]
            vx_bar = vx_bar + (vx / V0) * xi_bar[:, 2]
        gdx0 = xi_bar if ctx.has_dx0 and ctx.needs_input_grad[7] else None
        return None, None, None, None, None, zf_bar, vx_bar / ctx.tf, gdx0


def solve(bn, xx_ref, uu_ref, dx0=None, kp=5.0, kt=2.5):
    """(xx_star (N,6,TT), uu_star (N,2,TT)) float64 CUDA tensors = bn.set_refs_dev(xx_ref, uu_ref); bn.init_guess(kp, kt, dx0); bn.solve();
    bn.result_dev(), differentiable with respect to xx_ref, uu_ref (float64 CUDA tensors, (N,6,TT) / (N,2,TT) or (6,TT) / (2,TT) with
    refs_shared) and dx0 ((N,6) tensor or None)."""
    return _Solve.apply(bn, kp, kt, xx_ref, uu_ref, dx0)


def solve_step(bn, zf, xf, tf=1, dx0=None, kp=5.0, kt=2.5):
    """The step maneuver of main_newton_method.py (bn.set_refs_step) for final heights zf (N,) and final positions xf (N,): only these
    2 x N values cross to the host.  Differentiable with respect to zf, xf and dx0."""
    return _SolveParam.apply(bn, "step", tf, kp, kt, zf, xf, dx0)


def solve_acrobatic(bn, zf, xf=18, tf=1, dx0=None, kp=5.0, kt=2.5):
    """The acrobatic maneuver of acrobatic_newton.py (bn.set_refs_acrobatic) for bump heights zf (N,) and final positions xf (N,) or a
    number.  Differentiable with respect to zf, xf (when a tensor) and dx0."""
    if not isinstance(xf, torch.Tensor):
        xf = torch.full_like(zf, float(xf), dtype=torch.float64)
    return _SolveParam.apply(bn, "acrobatic", tf, kp, kt, zf, xf, dx0)
