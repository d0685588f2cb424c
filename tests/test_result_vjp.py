"""Derivative of the optimum with respect to the references and the initial state (acoc_result_vjp; definition in include/acoc.h).
CPU: the host replay of the new per-instance kernel code against a dense KKT solve assembled in numpy from the C oracle's pointwise step,
the adjoint identity against the sparse forward sensitivity, and the parametric chain rule.  The GPU side is tests/test_result_vjp_gpu.py."""
import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spl

from tests.util import golden

PARAMS = np.array([0.1716, 2.395, 3.256, 12.0, 9.81, 0.61, 1.2, 0.24, 1e-3])
R_INDEFINITE = np.array([[1e-5, 0.0], [0.0, -1.0]])  # symmetric, indefinite: G = R + B'PB is not positive definite at some steps


@pytest.fixture(scope="module")
def vemul():
    from tests.host_emul import vjp_emul
    vjp_emul.build()
    return vjp_emul


def _linearisation(oracle, xx, uu, xr, Q, QT):
    """A_t, B_t, the lam_{t+1}-contracted f_xx and f_ux along (xx, uu) (smooth float64 model), from the C oracle's pointwise step."""
    TT = xx.shape[1]
    A, B, Hxx, Sux = np.zeros((TT - 1, 6, 6)), np.zeros((TT - 1, 6, 2)), np.zeros((TT - 1, 6, 6)), np.zeros((TT - 1, 2, 6))
    lam = QT @ (xx[:, -1] - xr[:, -1])
    for t in range(TT - 2, -1, -1):
        _, fx, fu, fxx, _, fux = oracle.step(xx[:, t], uu[:, t], lam, quant_f32=False)
        A[t], B[t], Hxx[t], Sux[t] = fx.T, fu.T, fxx, fux
        lam = A[t].T @ lam + Q @ (xx[:, t] - xr[:, t])
    return A, B, Hxx, Sux


def _kkt(A, B, Hxx, Sux, Q, R, QT):
    """KKT matrix of the problem in the variables z = (x_1..x_{TT-1}, u_0..u_{TT-2}) and the multipliers of x_{t+1} = f(x_t, u_t)."""
    T1 = A.shape[0]  # TT - 1
    nx, nz = 6 * T1, 8 * T1
    xi = lambda t: 6 * (t - 1)  # noqa: E731
    ui = lambda t: nx + 2 * t  # noqa: E731
    H = sp.lil_matrix((nz, nz))
    Cm = sp.lil_matrix((nx, nz))
    for t in range(T1):
        H[ui(t):ui(t) + 2, ui(t):ui(t) + 2] = R
        if t >= 1:
            H[xi(t):xi(t) + 6, xi(t):xi(t) + 6] = Q + Hxx[t]
            H[ui(t):ui(t) + 2, xi(t):xi(t) + 6] = Sux[t]
            H[xi(t):xi(t) + 6, ui(t):ui(t) + 2] = Sux[t].T
            Cm[6 * t:6 * t + 6, xi(t):xi(t) + 6] = A[t]
        Cm[6 * t:6 * t + 6, ui(t):ui(t) + 2] = B[t]
        Cm[6 * t:6 * t + 6, xi(t + 1):xi(t + 1) + 6] = -np.eye(6)
    H[xi(T1):xi(T1) + 6, xi(T1):xi(T1) + 6] = QT
    K = sp.bmat([[H.tocsr(), Cm.T.tocsr()], [Cm.tocsr(), None]]).tocsc()
    return K, nx, nz, xi, ui


def dense_vjp(oracle, xx, uu, xr, gx, gu, Q, R, QT):
    """Reverse mode by one sparse solve of the KKT system: (xref_bar, uref_bar, x0_bar) of one instance."""
    A, B, Hxx, Sux = _linearisation(oracle, xx, uu, xr, Q, QT)
    K, nx, nz, xi, ui = _kkt(A, B, Hxx, Sux, Q, R, QT)
    T1 = A.shape[0]
    g = gu.copy()
    g[:, T1 - 1] += g[:, T1]
    rhs = np.zeros(nz + nx)
    for t in range(1, T1 + 1):
        rhs[xi(t):xi(t) + 6] = gx[:, t]
    for t in range(T1):
        rhs[ui(t):ui(t) + 2] = g[:, t]
    s = spl.spsolve(K, rhs)
    w, eta = s[:nz], s[nz:]
    xb, ub = np.zeros((6, T1 + 1)), np.zeros((2, T1 + 1))
    for t in range(1, T1 + 1):
        xb[:, t] = (QT if t == T1 else Q) @ w[xi(t):xi(t) + 6]
    for t in range(T1):
        ub[:, t] = R @ w[ui(t):ui(t) + 2]
    x0b = gx[:, 0] - A[0].T @ eta[0:6] - Sux[0].T @ w[ui(0):ui(0) + 2]
    return xb, ub, x0b, (A, B, Hxx, Sux, K, nx, nz, xi, ui)


def forward_sens(lin, v_xref, v_uref, v_x0, Q, R, QT):
    """Forward mode: the derivative of the result (x (6,TT), u (2,TT) with u[:, TT-1] = u[:, TT-2]) in the direction (v_xref, v_uref, v_x0)."""
    A, B, Hxx, Sux, K, nx, nz, xi, ui = lin
    T1 = A.shape[0]
    rhs = np.zeros(nz + nx)
    for t in range(1, T1 + 1):
        rhs[xi(t):xi(t) + 6] = (QT if t == T1 else Q) @ v_xref[:, t]
    for t in range(T1):
        rhs[ui(t):ui(t) + 2] = R @ v_uref[:, t]
    rhs[ui(0):ui(0) + 2] -= Sux[0] @ v_x0
    rhs[nz:nz + 6] = -A[0] @ v_x0
    s = spl.spsolve(K, rhs)
    dx, du = np.zeros((6, T1 + 1)), np.zeros((2, T1 + 1))
    dx[:, 0] = v_x0
    for t in range(1, T1 + 1):
        dx[:, t] = s[xi(t):xi(t) + 6]
    for t in range(T1):
        du[:, t] = s[ui(t):ui(t) + 2]
    du[:, T1] = du[:, T1 - 1]
    return dx, du


def _optima():
    """(name, xx (6,TT), uu (2,TT), xref, uref, Q, R, QT) at which the derivative is checked."""
    from aircraftoptimalcontrol_b200 import refgen
    out = []
    for name in ("newton_step_f64", "newton_acro_f64"):
        g = golden(name + ".npz")
        out.append((name, g["xx_star"], g["uu_star"], g["xx_ref"], g["uu_ref"], g["Q"], g["R"], g["QT"]))
    b = golden("newton_batched_instances.npz")
    zf4, xf4 = refgen.config4_params()
    _, zf5 = refgen.config5_params()
    for i in range(2):
        xr, ur = refgen.step_problem(xf4[i:i + 1], zf4[i:i + 1])
        out.append(("config4_%d" % i, b["config4_%d_xx_star" % i], b["config4_%d_uu_star" % i], xr[0], ur[0]) + refgen.weights("step"))
        xr, ur = refgen.acrobatic_problem(zf5[i:i + 1])
        out.append(("config5_%d" % i, b["config5_%d_xx_star" % i], b["config5_%d_uu_star" % i], xr[0], ur[0]) + refgen.weights("acro"))
    g = golden("newton_step_f64.npz")
    rng = np.random.default_rng(3)
    M = rng.normal(size=(6, 6)) * 1e-3
    Qd = g["Q"] + M @ M.T
    Rd = g["R"] + np.array([[0.0, 2e-7], [2e-7, 0.0]])
    out.append(("dense", g["xx_star"], g["uu_star"], g["xx_ref"], g["uu_ref"], Qd, Rd, g["QT"] + M @ M.T))
    out.append(("indefinite", g["xx_star"], g["uu_star"], g["xx_ref"], g["uu_ref"], g["Q"], R_INDEFINITE, g["QT"]))
    return out


OPTIMA = _optima()


def _grads(TT, seed):
    rng = np.random.default_rng(seed)
    return rng.normal(size=(6, TT)), rng.normal(size=(2, TT))


def _rel(a, b):
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


@pytest.mark.parametrize("case", OPTIMA, ids=[o[0] for o in OPTIMA])
def test_replay_matches_dense_kkt(vemul, oracle, case):
    """Replay of the kernels' code vs the sparse KKT solve: xref_bar, uref_bar, x0_bar within 1e-8 of each output's max-norm (measured:
    at most 1.1e-12 over these optima, the differences of a Riccati sweep and a sparse LU on the same system).  The indefinite case has
    n_indef > 0 (998 of 999 steps) and a nonsingular KKT system."""
    name, xx, uu, xr, ur, Q, R, QT = case
    gx, gu = _grads(xx.shape[1], 11)
    r = vemul.result_vjp(xx[None], uu[None], gx[None], gu[None], Q, R, QT, xref=xr[None], uref=ur[None])
    xb, ub, x0b, _ = dense_vjp(oracle, xx, uu, xr, gx, gu, Q, R, QT)
    assert _rel(r["xref"][0], xb) < 1e-8
    assert _rel(r["uref"][0], ub) < 1e-8
    assert _rel(r["x0"][0], x0b) < 1e-8
    assert np.all(r["xref"][0][:, 0] == 0) and np.all(r["uref"][0][:, -1] == 0)
    if name == "indefinite":
        assert r["n_indef"][0] > 0
    elif name.startswith("newton_"):
        assert r["n_indef"][0] == 0


@pytest.mark.parametrize("case", OPTIMA[:2] + OPTIMA[-2:], ids=[o[0] for o in OPTIMA[:2] + OPTIMA[-2:]])
def test_adjoint_identity(vemul, oracle, case):
    """<gbar, J v> = <J' gbar, v> for random gbar and v, J v from the sparse forward solve: pins x0_bar (the S_0 and A_0 terms) and the
    fold of gbar_u[TT-1] independently of the reverse-mode oracle above."""
    name, xx, uu, xr, ur, Q, R, QT = case
    TT = xx.shape[1]
    gx, gu = _grads(TT, 12)
    r = vemul.result_vjp(xx[None], uu[None], gx[None], gu[None], Q, R, QT, xref=xr[None], uref=ur[None])
    _, _, _, lin = dense_vjp(oracle, xx, uu, xr, gx, gu, Q, R, QT)
    rng = np.random.default_rng(13)
    vx, vu, v0 = rng.normal(size=(6, TT)), rng.normal(size=(2, TT)), rng.normal(size=6)
    dx, du = forward_sens(lin, vx, vu, v0, Q, R, QT)
    lhs = np.sum(gx * dx) + np.sum(gu * du)
    rhs = np.sum(r["xref"][0] * vx) + np.sum(r["uref"][0] * vu) + np.sum(r["x0"][0] * v0)
    assert abs(lhs - rhs) <= 1e-8 * max(abs(lhs), np.sum(np.abs(gx * dx)) + np.sum(np.abs(gu * du)))


@pytest.mark.parametrize("maneuver", ["step", "acrobatic"])
def test_parametric_reductions(vemul, maneuver):
    """zf_bar / vx_bar of parametric references against the chain rule applied in numpy to the replay's xref_bar (1e-13), and the
    expanded-reference replay of the same problem gives the same xref_bar bit for bit."""
    from aircraftoptimalcontrol_b200 import refgen
    b = golden("newton_batched_instances.npz")
    n, TT = 2, 1000
    if maneuver == "step":
        zf, xf = refgen.config4_params()
        zf, vx = zf[:n], xf[:n]
        tt, zs, vs = refgen.step_bases(1, TT)
        xc, uc = refgen.STEP_CONST
        xr, ur = refgen.step_problem(vx, zf)
        Q, R, QT = refgen.weights("step")
        cfg = "config4"
    else:
        _, zf = refgen.config5_params()
        zf, vx = zf[:n], np.full(n, 18.0)
        tt, zs = refgen.acrobatic_bases(1, TT)
        vs = None
        xc, uc = refgen.ACRO_CONST
        xr, ur = refgen.acrobatic_problem(zf)
        Q, R, QT = refgen.weights("acro")
        cfg = "config5"
    xx = np.stack([b["%s_%d_xx_star" % (cfg, i)] for i in range(n)])
    uu = np.stack([b["%s_%d_uu_star" % (cfg, i)] for i in range(n)])
    rng = np.random.default_rng(21)
    gx, gu = rng.normal(size=(n, 6, TT)), rng.normal(size=(n, 2, TT))
    prm = dict(tt=tt, zs=zs, vs=vs, zf=zf, vx=vx, xc=xc, uc=uc)
    r = vemul.result_vjp(xx, uu, gx, gu, Q, R, QT, param=prm)
    e = vemul.result_vjp(xx, uu, gx, gu, Q, R, QT, xref=xr, uref=ur)
    assert np.array_equal(r["xref"], e["xref"]) and np.array_equal(r["uref"], e["uref"]) and np.array_equal(r["x0"], e["x0"])
    xb = r["xref"]
    zf_bar = np.sum(zs * xb[:, 1], axis=1)
    vx_bar = np.sum(tt * xb[:, 0], axis=1)
    if vs is not None:
        V = np.sqrt((vs * zf[:, None]) ** 2 + vx[:, None] ** 2)
        zf_bar = zf_bar + np.sum(vs ** 2 * zf[:, None] / V * xb[:, 2], axis=1)
        vx_bar = vx_bar + np.sum(vx[:, None] / V * xb[:, 2], axis=1)
    assert np.max(np.abs(r["zf"] - zf_bar) / np.abs(zf_bar)) < 1e-13
    assert np.max(np.abs(r["vx"] - vx_bar) / np.abs(vx_bar)) < 1e-13


def test_nonfinite_lane_is_nan_and_isolated(vemul):
    """An all-zero result (the zero slot) gives NaN outputs (except the structural zeros) and leaves the other lane bit-identical."""
    g = golden("newton_step_f64.npz")
    xx, uu = g["xx_star"], g["uu_star"]
    gx, gu = _grads(xx.shape[1], 5)
    one = vemul.result_vjp(xx[None], uu[None], gx[None], gu[None], g["Q"], g["R"], g["QT"], xref=g["xx_ref"][None], uref=g["uu_ref"][None])
    two = vemul.result_vjp(np.stack([np.zeros_like(xx), xx]), np.stack([np.zeros_like(uu), uu]), np.stack([gx, gx]), np.stack([gu, gu]),
                           g["Q"], g["R"], g["QT"], xref=np.stack([g["xx_ref"]] * 2), uref=np.stack([g["uu_ref"]] * 2))
    for k in ("xref", "uref", "x0", "n_indef"):
        assert np.array_equal(two[k][1], one[k][0])
    assert np.all(np.isnan(two["xref"][0][:, 2:])) and np.all(np.isnan(two["uref"][0][:, :-1])) and np.all(np.isnan(two["x0"][0]))
