// acoc_kernels.cuh -- per-trajectory sweeps of the regularized-Newton loop (one thread = one OCP instance).
//
// Each *_instance() function is the complete body of one kernel for one instance: it walks the horizon
// sequentially (the Riccati / costate / rollout recurrences are true recurrences, optcon.py:434-464,
// :719-762, :196-198) with every per-step quantity in registers.  The __global__ wrappers at the bottom map
// threadIdx -> instance.  Trajectories live in HBM as warp-tiled struct-of-arrays (see at()): time-major, then
// tiles of 32 consecutive instances, then the component, then the lane:
//     X[((t*(Np/32) + i/32)*6 + c)*32 + i%32],   U[... *2 ...],   KSG[... *16 ...]
// so a warp reads ONE contiguous block per array per step (X 1.5 KB as double / 768 B as float, KSG 4 KB), every
// access is a full 128/256-byte line, and all components of a step sit at compile-time offsets from one base pointer
// that advances by a constant stride per step (no per-access 64-bit address arithmetic in the time loops).
//
// Reference call stack covered (SURVEY.md 3.1):
//   traj_cost_instance    optcon.py:417-424            cost of the current iterate
//   backward_instance     optcon.py:429-464 + the Riccati / gain loops of ltv_LQR (optcon.py:716-751),
//                         fused: linearisation, costate, lambda-contracted Hessians, P/p recursion, K, sigma
//   forward_lq_instance   optcon.py:756-762 (LQ forward pass) + :474-477 (descent)
//   rollout_instance      optcon.py:247-264 (one Armijo candidate) and :176-200 (get_update)
//   armijo_select_instance optcon.py:266-273, :327 and the bookkeeping of :488-501
//   track_instance        lqr_tracking.py:279-281
//   track_gains_instance, lqr_tracking.py:245-283 along each instance's own nominal (gains, closed loop, summaries)
//   track_rollout_instance
//   track_mc_sample,      the same closed loop from M perturbed starts per instance (summaries only) and their fixed-order
//   track_mc_reduce       per-instance aggregates
//   init_guess_instance   aircraft_simplified.py:142-147
//
// Types: F is the arithmetic type and the storage type of U, DU, KSG, the references and x0 (double = the parity path,
// float = the optional FP32 mode).  XT is the storage type of the state iterates X.  With the reference's float32 state
// quantisation (aircraft_simplified.py:300) every stored state x_t, t >= 1, IS a float32 value, so the parity path keeps
// X as float (XT = float, F = double): 24 instead of 48 bytes per step, bit-identical results.  Row t = 0 of such a slot
// is not exact (x0 is an arbitrary float64); readers take x_0 from P.x0 instead (it never changes, optcon.py:398/:194).
// Costs and the descent are accumulated in float64 in every mode.
#pragma once
#include <type_traits>

#include "acoc_math.cuh"

namespace acoc {

// ------------------------------------------------------------------------------------------------------
// problem description shared by all sweeps
// ------------------------------------------------------------------------------------------------------
template <typename F>
struct ProblemT {
    ModelT<F> M;
    WeightsT<F> W;
    int N;         // instances
    int Np;        // padded instance count (multiple of 32) = stride between components
    int TT;        // horizon samples
    int q32;       // 1: round the next state to float32 like aircraft_simplified.py:300
    int ref_shared;  // 1: xref/uref hold one trajectory shared by all instances (stride 1)
    const F* xref;  // warp-tiled [TT][Np/32][6][32], or [TT][6] when shared
    const F* uref;  // warp-tiled [TT][Np/32][2][32], or [TT][2] when shared
    const F* x0;    // [6][Np]   x0 = xx_init[:,0]  (optcon.py:398)
    // Parametric references (acoc_set_refs_generated): the references of the scripts are a two-parameter family per instance,
    //   X_t = vx_i * tt_t,  Z_t = zs_t * zf_i,  V_t = v_{t,i} (stored, step maneuver) or xc[2],  theta, q, gamma = xc[3..5],  uref = uc
    // (main_newton_method.py:96-142, acrobatic_newton.py:99-154), so the sweeps form X_t and Z_t with one multiplication each from two
    // shared tables instead of streaming 64 bytes per instance and step: 8 bytes (V) or none.  The products are the ones the
    // generator kernel stores in the expanded layout, so both layouts give bit-identical references.
    int ref_param;     // 1: xref / uref are not used
    const F* rp_tt;    // [TT] time grid
    const F* rp_zs;    // [TT] height shape
    const F* rp_zf;    // [Np] final / bump height per instance
    const F* rp_vx;    // [Np] (xf - x0)/tf per instance
    const F* rp_v;     // warp-tiled [TT][Np/32][1][32] speed reference, or nullptr: V_ref = rp_xc[2]
    F rp_xc[NS], rp_uc[NI];
};
using Problem = ProblemT<double>;

constexpr int TILE = 32;  // instances per tile = lanes of a warp; Np is a multiple of it
// element index of component c (of C) of instance i at time t in a warp-tiled trajectory array
ACOC_HD size_t at(int t, int C, int c, int Np, int i)
{
    return (((size_t)t * (size_t)(Np / TILE) + (size_t)(i / TILE)) * C + c) * TILE + (i % TILE);
}

// references: per instance (warp-tiled like the trajectories) or one shared trajectory stored time-major [TT][C]
// parametric references of instance i at time t from its parameters (zf, vx) and, if stored, its speed reference v
template <typename F>
ACOC_HD void param_xref(const ProblemT<F>& P, int t, F zf, F vx, F v, F* xr)
{
    xr[0] = vx * P.rp_tt[t];
    xr[1] = P.rp_zs[t] * zf;
    xr[2] = v;
    xr[3] = P.rp_xc[3]; xr[4] = P.rp_xc[4]; xr[5] = P.rp_xc[5];
}
template <typename F>
ACOC_HD F param_vref(const ProblemT<F>& P, int t, int i) { return P.rp_v ? P.rp_v[at(t, 1, 0, P.Np, i)] : P.rp_xc[2]; }

template <typename F>
ACOC_HD void load_xref(const ProblemT<F>& P, int t, int i, F* xr)
{
    if (P.ref_param) {
        param_xref(P, t, P.rp_zf[i], P.rp_vx[i], param_vref(P, t, i), xr);
        return;
    }
    if (P.ref_shared) {
#pragma unroll
        for (int c = 0; c < NS; ++c) xr[c] = P.xref[(size_t)t * NS + c];
    } else {
#pragma unroll
        for (int c = 0; c < NS; ++c) xr[c] = P.xref[at(t, NS, c, P.Np, i)];
    }
}
template <typename F>
ACOC_HD void load_ref(const ProblemT<F>& P, int t, int i, F* xr, F* ur)
{
    load_xref(P, t, i, xr);
    if (P.ref_param) { ur[0] = P.rp_uc[0]; ur[1] = P.rp_uc[1]; return; }
    if (P.ref_shared) {
#pragma unroll
        for (int c = 0; c < NI; ++c) ur[c] = P.uref[(size_t)t * NI + c];
    } else {
#pragma unroll
        for (int c = 0; c < NI; ++c) ur[c] = P.uref[at(t, NI, c, P.Np, i)];
    }
}

// state iterate slot: x_t of instance i (see "Types" above for the t = 0 rule)
// Split in two so that a sweep can issue the raw loads one step ahead (software prefetch) and convert where the value is
// consumed: a conversion placed right after the load would wait for the data at the prefetch point.
template <typename XT>
ACOC_HD void load_x_raw(const XT* X, int t, int Np, int i, XT* raw)
{
#pragma unroll
    for (int c = 0; c < NS; ++c) raw[c] = X[at(t, NS, c, Np, i)];
}
template <typename F, typename XT>
ACOC_HD void finish_x(const ProblemT<F>& P, int t, int i, const XT* raw, F* x)
{
#pragma unroll
    for (int c = 0; c < NS; ++c) x[c] = (F)raw[c];
    if (!std::is_same<F, XT>::value && t == 0) {  // once per sweep
#pragma unroll
        for (int c = 0; c < NS; ++c) x[c] = P.x0[(size_t)c * P.Np + i];
    }
}
template <typename F, typename XT>
ACOC_HD void load_x(const ProblemT<F>& P, const XT* X, int t, int i, F* x)
{
    XT raw[NS];
    load_x_raw(X, t, P.Np, i, raw);
    finish_x(P, t, i, raw, x);
}
template <typename F, typename XT>
ACOC_HD void store_x(XT* X, int t, int Np, int i, const F* x)
{
#pragma unroll
    for (int c = 0; c < NS; ++c) X[at(t, NS, c, Np, i)] = (XT)x[c];
}

// symmetric 6x6 in 21 registers, (i <= j)
ACOC_HD constexpr int sym(int i, int j) { return i <= j ? i * 6 - (i * (i - 1)) / 2 + (j - i) : j * 6 - (j * (j - 1)) / 2 + (i - j); }

// sum_c v[c] * A[c][J] : the dot product of v with column J of the sparse Jacobian (Appendix A of SURVEY.md)
template <typename F>
ACOC_HD F acol(const Lin<F>& l, F dt, const F* v, int J)
{
    switch (J) {
        case 0: return v[0];
        case 1: return v[1];
        case 2: return fma_(l.a52, v[5], fma_(l.a22, v[2], fma_(l.a12, v[1], l.a02 * v[0])));
        case 3: return fma_(l.a53, v[5], fma_(l.a23, v[2], v[3]));
        case 4: return fma_(dt, v[3], v[4]);
        default: return fma_(l.a55, v[5], fma_(l.a25, v[2], fma_(l.a15, v[1], l.a05 * v[0])));
    }
}

// ------------------------------------------------------------------------------------------------------
// cost of a stored trajectory, optcon.py:417-424
// ------------------------------------------------------------------------------------------------------
template <typename F, typename XT>
ACOC_HD double traj_cost_instance(const ProblemT<F>& P, const XT* X, const F* U, int i)
{
    double J = 0.0;
    F x[NS], dx[NS], du[NI], xr[NS], ur[NI];
    for (int t = 0; t < P.TT - 1; ++t) {
        load_ref(P, t, i, xr, ur);
        load_x(P, X, t, i, x);
#pragma unroll
        for (int c = 0; c < NS; ++c) dx[c] = x[c] - xr[c];
#pragma unroll
        for (int c = 0; c < NI; ++c) du[c] = U[at(t, NI, c, P.Np, i)] - ur[c];
        J += (double)stage_cost(P.W, dx, du);
    }
    load_xref(P, P.TT - 1, i, xr);
    load_x(P, X, P.TT - 1, i, x);
#pragma unroll
    for (int c = 0; c < NS; ++c) dx[c] = x[c] - xr[c];
    J += (double)term_cost(P.W, dx);
    return J;
}

// ------------------------------------------------------------------------------------------------------
// one step of the fused backward recursion
// ------------------------------------------------------------------------------------------------------
// In : Pm (sym 6x6), p, lam  at t+1;  Lin at (x_t,u_t);  q = Q dx, r = R du;  Hess (used iff EXACT)
// Out: Pm, p, lam at t;  K (2x6 row-major), sig (2), g (2) = B'lam_{t+1} + r
// Equations (decomposition of the reference's 7x7 augmented recursion, optcon.py:673-689, :727-728, :743-751,
// with P~ = [[pi, p'],[p, P]], S~ = [r/2, S], Q~ = [[0, q'/2],[q/2, Q]]):
//   Mx = B'PA + S,  m = B'p + r/2,  G = R + B'PB
//   P_t = Q + A'PA - Mx' G^-1 Mx          p_t = q/2 + A'p - Mx' G^-1 m
//   MM  = G, or G + 0.5 I when G has a non-positive eigenvalue;  K = -MM^-1 Mx,  sigma = -MM^-1 m
// The step has two halves that share only the linearisation: the COSTATE half (g, lambda_t: needs lambda_{t+1} only) and the MATRIX
// half (G, m, the column sweep, gains, P_t, p_t: needs P_{t+1}, p_{t+1} only).  riccati_step() is their composition.  (Running the
// halves in two warps of a CTA -- costate warp one step ahead, linearisation handed over through shared memory -- was measured in
// round 2: the matrix half alone needs ~230 registers to stay spill-free, so only 4 tiles per SM are resident instead of 8 and the
// sweep takes 4.0 ms instead of 3.2; bounded to 168 / 128 registers it spills and takes 5.0 / 6.4 ms.  Big batches therefore keep the
// one-thread step below; batches that leave the machine idle run it as warp roles: k_backward_split (two halves) up to two tiles per
// SM, k_backward_cols (the halves cut further: linearisation ahead of time, costate, gain block, outputs, one warp per column of the
// matrix half -- the pieces further down) up to one tile per SM.  acoc_tma.cuh, profiles/README.md.)

// costate half: g = B' lam_{t+1} + r (optcon.py:475), lam_t = A' lam_{t+1} + q (:461)
template <typename F>
ACOC_HD void riccati_costate(const ModelT<F>& M, const Lin<F>& l, const F* q, const F* r, F* lam, F* g)
{
    g[0] = fma_(l.b50, lam[5], fma_(l.b20, lam[2], r[0]));
    g[1] = fma_(M.b41, lam[4], r[1]);
    F Atl[NS];
#pragma unroll
    for (int i = 0; i < NS; ++i) Atl[i] = acol(l, M.dt, lam, i);
#pragma unroll
    for (int i = 0; i < NS; ++i) lam[i] = Atl[i] + q[i];
}

// matrix half: Pm, p at t+1 -> K_t, sigma_t, Pm, p at t.  Returns 1 if the gain took the +0.5 I branch.
template <bool EXACT, int DG = -1, typename F>
ACOC_HD int riccati_matrix(const ModelT<F>& M, const WeightsT<F>& W, const Lin<F>& l, const Hess<F>& h, const F* q, const F* r,
                           F* Pm, F* p, F* K, F* sig)
{
    const F dt = M.dt, b41 = M.b41;
    // G = R + B'PB, m = B'p + r/2  (need P_{t+1}, p_{t+1})
    const F P22 = Pm[sym(2, 2)], P25 = Pm[sym(2, 5)], P55 = Pm[sym(5, 5)], P24 = Pm[sym(2, 4)], P45 = Pm[sym(4, 5)], P44 = Pm[sym(4, 4)];
    const F pb2 = fma_(l.b50, P25, l.b20 * P22), pb5 = fma_(l.b50, P55, l.b20 * P25);
    const F G00 = fma_(l.b50, pb5, fma_(l.b20, pb2, W.R[0]));
    const F G01 = fma_(b41, fma_(l.b50, P45, l.b20 * P24), W.R[1]);
    const F G11 = fma_(b41 * b41, P44, W.R[3]);
    const F m0 = fma_(l.b50, p[5], fma_(l.b20, p[2], F(0.5) * r[0]));
    const F m1 = fma_(b41, p[4], F(0.5) * r[1]);

    // column sweep: W = P A (column j), N = A'W (upper triangle), Mx = B'W (+S)
    F Pn[21], Mx0[NS], Mx1[NS];
#pragma unroll
    for (int j = 0; j < NS; ++j) {
        F Wc[NS];
#pragma unroll
        for (int k = 0; k < NS; ++k) {
            F row[NS];
#pragma unroll
            for (int c = 0; c < NS; ++c) row[c] = Pm[sym(k, c)];
            Wc[k] = acol(l, dt, row, j);
        }
#pragma unroll
        for (int i = 0; i <= j; ++i) Pn[sym(i, j)] = acol(l, dt, Wc, i);
        Mx0[j] = fma_(l.b50, Wc[5], l.b20 * Wc[2]);
        Mx1[j] = b41 * Wc[4];
    }
    if (EXACT) { Mx0[2] += h.s2; Mx0[3] += h.s3; Mx0[5] += h.s5; }  // S = lux + fux (optcon.py:446)

    // A'p
    F Atp[NS];
#pragma unroll
    for (int i = 0; i < NS; ++i) Atp[i] = acol(l, dt, p, i);

    // G^-1 (explicit inverse, optcon.py:728)
    const F det = fma_(G00, G11, -(G01 * G01));
    const F idet = F(1.0) / det;
    const F gi00 = G11 * idet, gi01 = -G01 * idet, gi11 = G00 * idet;
    F Y0[NS], Y1[NS];  // G^-1 Mx
#pragma unroll
    for (int j = 0; j < NS; ++j) {
        Y0[j] = fma_(gi01, Mx1[j], gi00 * Mx0[j]);
        Y1[j] = fma_(gi11, Mx1[j], gi01 * Mx0[j]);
    }
    const F y0 = fma_(gi01, m1, gi00 * m0), y1 = fma_(gi11, m1, gi01 * m0);

    // gains: positive-definiteness test on G (optcon.py:743-749) -- eigenvalues of the symmetric 2x2
    const F hd = F(0.5) * (G00 - G11), mid = F(0.5) * (G00 + G11);
    const F rad = sqrt_(fma_(hd, hd, G01 * G01));
    int reg = 0;
    if (mid - rad > F(0.0)) {
#pragma unroll
        for (int j = 0; j < NS; ++j) { K[j] = -Y0[j]; K[NS + j] = -Y1[j]; }
        sig[0] = -y0; sig[1] = -y1;
    } else {  // regularised gain MM = G + 0.5 I; the Riccati update below still uses the plain G^-1
        reg = 1;
        const F H00 = G00 + F(0.5), H11 = G11 + F(0.5);
        const F id2 = F(1.0) / fma_(H00, H11, -(G01 * G01));
        const F hi00 = H11 * id2, hi01 = -G01 * id2, hi11 = H00 * id2;
#pragma unroll
        for (int j = 0; j < NS; ++j) {
            K[j] = -fma_(hi01, Mx1[j], hi00 * Mx0[j]);
            K[NS + j] = -fma_(hi11, Mx1[j], hi01 * Mx0[j]);
        }
        sig[0] = -fma_(hi01, m1, hi00 * m0);
        sig[1] = -fma_(hi11, m1, hi01 * m0);
    }

    // P_t, p_t
#pragma unroll
    for (int i = 0; i < NS; ++i) {
#pragma unroll
        for (int j = i; j < NS; ++j) {
            const F corr = fma_(Mx1[i], Y1[j], Mx0[i] * Y0[j]);
            if (DG == 1 && i != j) Pm[sym(i, j)] = Pn[sym(i, j)] - corr;  // (the structural zero of a diagonal Q is not added)
            else {
                const F qij = weights_diag<DG>(W) ? (i == j ? W.Q[i * 7] : F(0.0)) : W.Q[i * 6 + j];
                Pm[sym(i, j)] = (Pn[sym(i, j)] + qij) - corr;
            }
        }
        p[i] = fma_(F(0.5), q[i], Atp[i]) - fma_(Mx1[i], y1, Mx0[i] * y0);
    }
    if (EXACT) {  // Q_t = lxx + fxx (optcon.py:444)
        Pm[sym(2, 2)] += h.h22; Pm[sym(2, 3)] += h.h23; Pm[sym(2, 5)] += h.h25;
        Pm[sym(3, 3)] += h.h33; Pm[sym(3, 5)] += h.h35; Pm[sym(5, 5)] += h.h55;
    }
    return reg;
}

// ---- the matrix half BY COLUMNS (k_backward_cols: one warp per column of P, small batches) -----------------------------
// riccati_matrix() cut along the columns j of the sweep.  Everything column j produces -- W = P A e_j, N(i,j) = (A'W)_i for i <= j,
// Mx(:,j), then Y(:,j) and P_t(i,j) for i <= j -- needs, beside the old P and the linearisation, only the inverse of the 2x2 block G
// (riccati_gain, its own warp) and Mx(:,i) of the columns i < j (exchanged once per step); the affine term p and the outputs K, sigma
// are separate pieces as well.
// Every number is formed by the same expression as in riccati_matrix(), so the two are bit-identical (tests/test_kernel_math_host.py
// replays both on the host).
template <typename F>
struct RicGain {
    F G00, G01, G11;     // G = R + B'PB
    F gi00, gi01, gi11;  // G^-1 (the Riccati update always uses the plain inverse, optcon.py:728)
    F k00, k01, k11;     // the inverse the GAIN uses: G^-1, or (G + 0.5 I)^-1 when G has a non-positive eigenvalue (optcon.py:743-749)
    F m0, m1, y0, y1;    // m = B'p + r/2, y = G^-1 m
    int reg;
};

// what the recurrence needs: G, m, G^-1, y
template <typename F>
ACOC_HD void riccati_gain_core(const ModelT<F>& M, const WeightsT<F>& W, const Lin<F>& l, const F* r, const F* Pm, const F* p, RicGain<F>& o)
{
    const F b41 = M.b41;
    const F P22 = Pm[sym(2, 2)], P25 = Pm[sym(2, 5)], P55 = Pm[sym(5, 5)], P24 = Pm[sym(2, 4)], P45 = Pm[sym(4, 5)], P44 = Pm[sym(4, 4)];
    const F pb2 = fma_(l.b50, P25, l.b20 * P22), pb5 = fma_(l.b50, P55, l.b20 * P25);
    o.G00 = fma_(l.b50, pb5, fma_(l.b20, pb2, W.R[0]));
    o.G01 = fma_(b41, fma_(l.b50, P45, l.b20 * P24), W.R[1]);
    o.G11 = fma_(b41 * b41, P44, W.R[3]);
    o.m0 = fma_(l.b50, p[5], fma_(l.b20, p[2], F(0.5) * r[0]));
    o.m1 = fma_(b41, p[4], F(0.5) * r[1]);
    const F det = fma_(o.G00, o.G11, -(o.G01 * o.G01));
    const F idet = F(1.0) / det;
    o.gi00 = o.G11 * idet; o.gi01 = -o.G01 * idet; o.gi11 = o.G00 * idet;
    o.y0 = fma_(o.gi01, o.m1, o.gi00 * o.m0); o.y1 = fma_(o.gi11, o.m1, o.gi01 * o.m0);
}
// what only the outputs K, sigma need: the positive-definiteness test on G (eigenvalues of the symmetric 2x2) and the inverse the gain uses
template <typename F>
ACOC_HD void riccati_gain_test(RicGain<F>& o)
{
    const F hd = F(0.5) * (o.G00 - o.G11), mid = F(0.5) * (o.G00 + o.G11);
    const F rad = sqrt_(fma_(hd, hd, o.G01 * o.G01));
    if (mid - rad > F(0.0)) { o.reg = 0; o.k00 = o.gi00; o.k01 = o.gi01; o.k11 = o.gi11; }
    else {  // regularised gain MM = G + 0.5 I; the Riccati update still uses the plain G^-1
        o.reg = 1;
        const F H00 = o.G00 + F(0.5), H11 = o.G11 + F(0.5);
        const F id2 = F(1.0) / fma_(H00, H11, -(o.G01 * o.G01));
        o.k00 = H11 * id2; o.k01 = -o.G01 * id2; o.k11 = H00 * id2;
    }
}
template <typename F>
ACOC_HD RicGain<F> riccati_gain(const ModelT<F>& M, const WeightsT<F>& W, const Lin<F>& l, const F* r, const F* Pm, const F* p)
{
    RicGain<F> o;
    riccati_gain_core(M, W, l, r, Pm, p, o);
    riccati_gain_test(o);
    return o;
}

// first half of column J: PnJ[i] = N(i,J) for i <= J, Mx(:,J)
template <bool EXACT, int J, typename F>
ACOC_HD void riccati_col_sweep(const ModelT<F>& M, const Lin<F>& l, const Hess<F>& h, const F* Pm, F* PnJ, F& mx0, F& mx1)
{
    F Wc[NS];
#pragma unroll
    for (int k = 0; k < NS; ++k) {
        F row[NS];
#pragma unroll
        for (int c = 0; c < NS; ++c) row[c] = Pm[sym(k, c)];
        Wc[k] = acol(l, M.dt, row, J);
    }
#pragma unroll
    for (int i = 0; i <= J; ++i) PnJ[i] = acol(l, M.dt, Wc, i);
    mx0 = fma_(l.b50, Wc[5], l.b20 * Wc[2]);
    mx1 = M.b41 * Wc[4];
    if (EXACT) {  // S = lux + fux (optcon.py:446)
        if (J == 2) mx0 += h.s2;
        if (J == 3) mx0 += h.s3;
        if (J == 5) mx0 += h.s5;
    }
}

// second half of column J: Mx0[i], Mx1[i] for i <= J (own column included) and G^-1 -> P_t(i,J) for i <= J
template <bool EXACT, int DG, int J, typename F>
ACOC_HD void riccati_col_finish(const WeightsT<F>& W, const Hess<F>& h, F gi00, F gi01, F gi11, const F* PnJ, const F* Mx0, const F* Mx1, F* PJ)
{
    const F Y0 = fma_(gi01, Mx1[J], gi00 * Mx0[J]);
    const F Y1 = fma_(gi11, Mx1[J], gi01 * Mx0[J]);
#pragma unroll
    for (int i = 0; i <= J; ++i) {
        const F corr = fma_(Mx1[i], Y1, Mx0[i] * Y0);
        if (DG == 1 && i != J) PJ[i] = PnJ[i] - corr;
        else {
            const F qij = weights_diag<DG>(W) ? (i == J ? W.Q[i * 7] : F(0.0)) : W.Q[i * 6 + J];
            PJ[i] = (PnJ[i] + qij) - corr;
        }
    }
    if (EXACT) {  // Q_t = lxx + fxx (optcon.py:444)
        if (J == 2) PJ[2] += h.h22;
        if (J == 3) { PJ[2] += h.h23; PJ[3] += h.h33; }
        if (J == 5) { PJ[2] += h.h25; PJ[3] += h.h35; PJ[5] += h.h55; }
    }
}

// the affine term: A'p before the exchange, p_t after it (one of the light column warps carries it)
template <typename F>
ACOC_HD void riccati_p_sweep(const ModelT<F>& M, const Lin<F>& l, const F* p, F* Atp)
{
#pragma unroll
    for (int i = 0; i < NS; ++i) Atp[i] = acol(l, M.dt, p, i);
}
template <typename F>
ACOC_HD void riccati_p_finish(const F* q, const F* Atp, const F* Mx0, const F* Mx1, F y0, F y1, F* p)
{
#pragma unroll
    for (int i = 0; i < NS; ++i) p[i] = fma_(F(0.5), q[i], Atp[i]) - fma_(Mx1[i], y1, Mx0[i] * y0);
}

// the outputs of the step from the gain block and Mx (the GAIN warp forms them after the exchange, beside the columns' second half)
template <typename F>
ACOC_HD void riccati_gain_out(const RicGain<F>& gn, const F* Mx0, const F* Mx1, F* K, F* sig)
{
#pragma unroll
    for (int j = 0; j < NS; ++j) {
        K[j] = -fma_(gn.k01, Mx1[j], gn.k00 * Mx0[j]);
        K[NS + j] = -fma_(gn.k11, Mx1[j], gn.k01 * Mx0[j]);
    }
    sig[0] = -fma_(gn.k01, gn.m1, gn.k00 * gn.m0);
    sig[1] = -fma_(gn.k11, gn.m1, gn.k01 * gn.m0);
}

// riccati_matrix() recomposed from these pieces (host replay of k_backward_cols' arithmetic; the kernel runs them in eight warps and
// exchanges Mx, the gain block and the new P, p through shared memory)
template <bool EXACT, int DG, int J, typename F>
ACOC_HD void riccati_cols_a_(const ModelT<F>& M, const Lin<F>& l, const Hess<F>& h, const F* Pm, F (*Pn)[NS], F* Mx0, F* Mx1)
{
    riccati_col_sweep<EXACT, J, F>(M, l, h, Pm, Pn[J], Mx0[J], Mx1[J]);
    if constexpr (J + 1 < NS) riccati_cols_a_<EXACT, DG, J + 1, F>(M, l, h, Pm, Pn, Mx0, Mx1);
}
template <bool EXACT, int DG, int J, typename F>
ACOC_HD void riccati_cols_b_(const WeightsT<F>& W, const Hess<F>& h, const RicGain<F>& gn, F (*Pn)[NS], const F* Mx0, const F* Mx1, F* Pm)
{
    F PJ[NS];
    riccati_col_finish<EXACT, DG, J, F>(W, h, gn.gi00, gn.gi01, gn.gi11, Pn[J], Mx0, Mx1, PJ);
#pragma unroll
    for (int i = 0; i <= J; ++i) Pm[sym(i, J)] = PJ[i];
    if constexpr (J + 1 < NS) riccati_cols_b_<EXACT, DG, J + 1, F>(W, h, gn, Pn, Mx0, Mx1, Pm);
}
template <bool EXACT, int DG = -1, typename F>
ACOC_HD int riccati_matrix_by_columns(const ModelT<F>& M, const WeightsT<F>& W, const Lin<F>& l, const Hess<F>& h, const F* q, const F* r,
                                      F* Pm, F* p, F* K, F* sig)
{
    const RicGain<F> gn = riccati_gain(M, W, l, r, Pm, p);
    F Pn[NS][NS], Mx0[NS], Mx1[NS], Atp[NS];
    riccati_cols_a_<EXACT, DG, 0, F>(M, l, h, Pm, Pn, Mx0, Mx1);   // every column reads the OLD P
    riccati_p_sweep(M, l, p, Atp);
    riccati_cols_b_<EXACT, DG, 0, F>(W, h, gn, Pn, Mx0, Mx1, Pm);  // ... and only then is it overwritten
    riccati_p_finish(q, Atp, Mx0, Mx1, gn.y0, gn.y1, p);
    riccati_gain_out(gn, Mx0, Mx1, K, sig);
    return gn.reg;
}

template <bool EXACT, int DG = -1, typename F>
ACOC_HD int riccati_step(const ModelT<F>& M, const WeightsT<F>& W, const Lin<F>& l, const Hess<F>& h, const F* q, const F* r,
                         F* Pm, F* p, F* lam, F* K, F* sig, F* g)
{
    const int reg = riccati_matrix<EXACT, DG, F>(M, W, l, h, q, r, Pm, p, K, sig);
    riccati_costate(M, l, q, r, lam, g);   // (after the matrix half only for the order of the statements; the halves share no state)
    return reg;
}

// ------------------------------------------------------------------------------------------------------
// backward sweep of one Newton iteration
// ------------------------------------------------------------------------------------------------------
// KSG[t][0..11] = K_t (row-major 2x6), [12..13] = sigma_t, [14..15] = g_t ; t = 0..TT-2.
// Returns the number of steps whose gain took the +0.5 I branch.
// terminal condition: lam_{T-1} = QT dx (optcon.py:429-432), P_{T-1} = QT, p_{T-1} = lam/2 (:688-690, :716)
template <int DG = -1, typename F>
ACOC_HD void backward_terminal(const WeightsT<F>& W, const F* x, const F* xr, F* Pm, F* p, F* lam)
{
    F dx[NS];
#pragma unroll
    for (int c = 0; c < NS; ++c) dx[c] = x[c] - xr[c];
    wmul6(W.QT, (int)weights_diag<DG>(W), dx, lam);
#pragma unroll
    for (int a = 0; a < NS; ++a) {
        p[a] = F(0.5) * lam[a];
#pragma unroll
        for (int b = a; b < NS; ++b) Pm[sym(a, b)] = weights_diag<DG>(W) ? (a == b ? W.QT[a * 7] : F(0.0)) : W.QT[a * 6 + b];
    }
}

// one time step of the backward sweep: (x_t, u_t, refs) and the carried (P, p, lam) -> K_t, sigma_t, g_t.  Returns 1 if the
// gain took the +0.5 I branch.
template <bool EXACT, int DG = -1, typename F>
ACOC_HD int backward_step(const ModelT<F>& M, const WeightsT<F>& W, const F* x, const F* u, const F* xr, const F* ur, F* Pm, F* p, F* lam,
                          F* K, F* sig, F* g)
{
    F dx[NS], du[NI], q[NS], r[NI];
#pragma unroll
    for (int c = 0; c < NS; ++c) dx[c] = x[c] - xr[c];
#pragma unroll
    for (int c = 0; c < NI; ++c) du[c] = u[c] - ur[c];
    wmul6(W.Q, (int)weights_diag<DG>(W), dx, q);   // lx = Q dx   (aircraft_simplified.py:63)
    wmul2(W.R, (int)weights_diag<DG>(W), du, r);   // lu = R du   (:64)
    const Trig<F> tg = make_trig(x);
    const Lin<F> l = linearize(M, x, u, tg);
    Hess<F> h;
    if (EXACT) h = hess_contract(M, x, u, tg, l, lam);
    return riccati_step<EXACT, DG, F>(M, W, l, h, q, r, Pm, p, lam, K, sig, g);
}

template <bool EXACT, typename F, typename XT>
ACOC_HD int backward_instance(const ProblemT<F>& P, const XT* X, const F* U, F* KSG, int i)
{
    const int TT = P.TT, Np = P.Np;
    F Pm[21], p[NS], lam[NS], x[NS], u[NI], xr[NS], ur[NI];
    load_xref(P, TT - 1, i, xr);
    load_x(P, X, TT - 1, i, x);
    backward_terminal(P.W, x, xr, Pm, p, lam);
    int nreg = 0;
    // software prefetch: the loads of step t-1 are issued before the arithmetic of step t
    XT nx[NS];
    F nu[NI], nxr[NS], nur[NI];
    {
        const int t = TT - 2;
        load_ref(P, t, i, nxr, nur);
        load_x_raw(X, t, Np, i, nx);
#pragma unroll
        for (int c = 0; c < NI; ++c) nu[c] = U[at(t, NI, c, Np, i)];
    }
    for (int t = TT - 2; t >= 0; --t) {
        finish_x(P, t, i, nx, x);
#pragma unroll
        for (int c = 0; c < NS; ++c) xr[c] = nxr[c];
#pragma unroll
        for (int c = 0; c < NI; ++c) { u[c] = nu[c]; ur[c] = nur[c]; }
        if (t > 0) {
            load_ref(P, t - 1, i, nxr, nur);
            load_x_raw(X, t - 1, Np, i, nx);
#pragma unroll
            for (int c = 0; c < NI; ++c) nu[c] = U[at(t - 1, NI, c, Np, i)];
        }
        F K[2 * NS], sig[NI], g[NI];
        nreg += backward_step<EXACT>(P.M, P.W, x, u, xr, ur, Pm, p, lam, K, sig, g);
#pragma unroll
        for (int c = 0; c < 12; ++c) KSG[at(t, 16, c, Np, i)] = K[c];
        KSG[at(t, 16, 12, Np, i)] = sig[0]; KSG[at(t, 16, 13, Np, i)] = sig[1];
        KSG[at(t, 16, 14, Np, i)] = g[0];   KSG[at(t, 16, 15, Np, i)] = g[1];
    }
    return nreg;
}

// ------------------------------------------------------------------------------------------------------
// steepest-descent costate sweep (GradientMethod.optimize, optcon.py:95-118)
// ------------------------------------------------------------------------------------------------------
// one time step: (x_t, u_t, refs) and lam_{t+1} -> deltau_t = -B'lam_{t+1} - lu (:111), lam_t = A'lam_{t+1} + lx (:110),
// sq += deltau_t'deltau_t (:118)
template <typename F>
ACOC_HD void gradient_step(const ModelT<F>& M, const WeightsT<F>& W, const F* x, const F* u, const F* xr, const F* ur, F* lam, F* du, double& sq)
{
    F dx[NS], dv[NI], q[NS], r[NI];
#pragma unroll
    for (int c = 0; c < NS; ++c) dx[c] = x[c] - xr[c];
#pragma unroll
    for (int c = 0; c < NI; ++c) dv[c] = u[c] - ur[c];
    wmul6(W.Q, W.diag, dx, q);   // aa = lx = Q dx   (aircraft_simplified.py:63)
    wmul2(W.R, W.diag, dv, r);   // bb = lu = R du   (:64)
    const Trig<F> tg = make_trig(x);
    const Lin<F> l = linearize(M, x, u, tg);
    du[0] = -fma_(l.b50, lam[5], fma_(l.b20, lam[2], r[0]));
    du[1] = -fma_(M.b41, lam[4], r[1]);
    sq = fma_((double)du[1], (double)du[1], fma_((double)du[0], (double)du[0], sq));
    F Atl[NS];
#pragma unroll
    for (int i = 0; i < NS; ++i) Atl[i] = acol(l, M.dt, lam, i);
#pragma unroll
    for (int i = 0; i < NS; ++i) lam[i] = Atl[i] + q[i];
}

// terminal costate lam_{T-1} = QT (x_{T-1} - xref_{T-1})  (optcon.py:98-99)
template <typename F>
ACOC_HD void gradient_terminal(const WeightsT<F>& W, const F* x, const F* xr, F* lam)
{
    F dx[NS];
#pragma unroll
    for (int c = 0; c < NS; ++c) dx[c] = x[c] - xr[c];
    wmul6(W.QT, W.diag, dx, lam);
}

// whole sweep of one instance: writes deltau (DU[TT-1] = 0: deltau[:,TT-1] is never assigned, optcon.py:74), returns sum_t |deltau_t|^2
template <typename F, typename XT>
ACOC_HD double gradient_instance(const ProblemT<F>& P, const XT* X, const F* U, F* DU, int i)
{
    const int TT = P.TT, Np = P.Np;
    F lam[NS], x[NS], u[NI], xr[NS], ur[NI], du[NI];
    load_xref(P, TT - 1, i, xr);
    load_x(P, X, TT - 1, i, x);
    gradient_terminal(P.W, x, xr, lam);
    DU[at(TT - 1, NI, 0, Np, i)] = F(0.0);
    DU[at(TT - 1, NI, 1, Np, i)] = F(0.0);
    double sq = 0.0;
    for (int t = TT - 2; t >= 0; --t) {
        load_ref(P, t, i, xr, ur);
        load_x(P, X, t, i, x);
#pragma unroll
        for (int c = 0; c < NI; ++c) u[c] = U[at(t, NI, c, Np, i)];
        gradient_step(P.M, P.W, x, u, xr, ur, lam, du, sq);
        DU[at(t, NI, 0, Np, i)] = du[0];
        DU[at(t, NI, 1, Np, i)] = du[1];
    }
    return sq;
}

// ------------------------------------------------------------------------------------------------------
// LQ forward pass + descent
// ------------------------------------------------------------------------------------------------------
// du_t = sigma_t + K_t dx_t ; dx_{t+1} = A_t dx_t + B_t du_t (optcon.py:759-760 with x~ = [1; dx], x0 = 0);
// descent = sum_t g_t' du_t (optcon.py:474-477).  A_t, B_t are recomputed from (x_t,u_t) instead of being
// stored by the backward sweep (12 doubles per step of HBM traffic saved for ~60 flops and two sincos).
// DX (optional, warp-tiled like X) receives the state increments for the drop-in ltv_LQR-style outputs.
// one time step: ksg = (K row-major 2x6, sigma, g) of this step; dx is advanced in place, du returned, descent accumulated
// (two halves so that a caller can drop ksg -- 16 values -- before the trigonometry of the second half)
template <typename F>
ACOC_HD void forward_du(const F* ksg, const F* dx, F* du, double& descent)
{
    du[0] = ksg[12]; du[1] = ksg[13];
#pragma unroll
    for (int c = 0; c < NS; ++c) { du[0] = fma_(ksg[c], dx[c], du[0]); du[1] = fma_(ksg[NS + c], dx[c], du[1]); }
    descent = fma_((double)ksg[15], (double)du[1], fma_((double)ksg[14], (double)du[0], descent));
}

template <typename F>
ACOC_HD void forward_advance(const ModelT<F>& M, const F* x, const F* u, const F* du, F* dx)
{
    const Trig<F> tg = make_trig(x);
    const Lin<F> l = linearize(M, x, u, tg);
    F nx[NS];
    nx[0] = fma_(l.a05, dx[5], fma_(l.a02, dx[2], dx[0]));
    nx[1] = fma_(l.a15, dx[5], fma_(l.a12, dx[2], dx[1]));
    nx[2] = fma_(l.b20, du[0], fma_(l.a25, dx[5], fma_(l.a23, dx[3], l.a22 * dx[2])));
    nx[3] = fma_(M.dt, dx[4], dx[3]);
    nx[4] = fma_(M.b41, du[1], dx[4]);
    nx[5] = fma_(l.b50, du[0], fma_(l.a55, dx[5], fma_(l.a53, dx[3], l.a52 * dx[2])));
#pragma unroll
    for (int c = 0; c < NS; ++c) dx[c] = nx[c];
}

template <typename F>
ACOC_HD void forward_step(const ModelT<F>& M, const F* x, const F* u, const F* ksg, F* dx, F* du, double& descent)
{
    forward_du(ksg, dx, du, descent);
    forward_advance(M, x, u, du, dx);
}

template <typename F, typename XT>
ACOC_HD double forward_lq_instance(const ProblemT<F>& P, const XT* X, const F* U, const F* KSG, F* DU, F* DX, int i)
{
    const int TT = P.TT, Np = P.Np;
    F dx[NS] = {0, 0, 0, 0, 0, 0}, x[NS], u[NI], du[NI];
    double descent = 0.0;
    for (int t = 0; t < TT - 1; ++t) {
        XT xraw[NS];
        load_x_raw(X, t, Np, i, xraw);
#pragma unroll
        for (int c = 0; c < NI; ++c) u[c] = U[at(t, NI, c, Np, i)];
        F ksg[16];
#pragma unroll
        for (int c = 0; c < 16; ++c) ksg[c] = KSG[at(t, 16, c, Np, i)];
        finish_x(P, t, i, xraw, x);
        if (DX) {
#pragma unroll
            for (int c = 0; c < NS; ++c) DX[at(t, NS, c, Np, i)] = dx[c];
        }
        forward_step(P.M, x, u, ksg, dx, du, descent);
        DU[at(t, NI, 0, Np, i)] = du[0];
        DU[at(t, NI, 1, Np, i)] = du[1];
    }
    DU[at(TT - 1, NI, 0, Np, i)] = F(0.0);  // uuout[:, TT-1] stays zero (optcon.py:694)
    DU[at(TT - 1, NI, 1, Np, i)] = F(0.0);
    if (DX) {
#pragma unroll
        for (int c = 0; c < NS; ++c) DX[at(TT - 1, NS, c, Np, i)] = dx[c];
    }
    return descent;
}

// ------------------------------------------------------------------------------------------------------
// open-loop rollout of u' = u + s*du from x0: one Armijo candidate (COST) and/or get_update (WRITE)
// ------------------------------------------------------------------------------------------------------
// one step of a rollout: stage cost of (x_t, u_t) (COST) and x_{t+1} = f(x_t, u_t) in place
template <bool COST, bool Q32, int DG = -1, typename F>
ACOC_HD void rollout_step(const ModelT<F>& M, const WeightsT<F>& W, F* x, const F* u, const F* xr, const F* ur, double& J)
{
    if (COST) {
        F dx[NS], du[NI];
#pragma unroll
        for (int c = 0; c < NS; ++c) dx[c] = x[c] - xr[c];
#pragma unroll
        for (int c = 0; c < NI; ++c) du[c] = u[c] - ur[c];
        J += (double)stage_cost<DG>(W, dx, du);
    }
    const Trig<F> tg = make_trig(x);
    F xn[NS];
    next_state<Q32>(M, x, u, tg, xn);
#pragma unroll
    for (int c = 0; c < NS; ++c) x[c] = xn[c];
}

template <bool WRITE, bool COST, bool Q32, typename F, typename XT>
ACOC_HD double rollout_instance(const ProblemT<F>& P, const F* U, const F* DU, double step, XT* Xn, F* Un, int i)
{
    const int TT = P.TT, Np = P.Np;
    const F s = (F)step;
    F x[NS], u[NI], xr[NS], ur[NI], dx[NS];
    double J = 0.0;
#pragma unroll
    for (int c = 0; c < NS; ++c) x[c] = P.x0[(size_t)c * Np + i];
    for (int t = 0; t < TT - 1; ++t) {
#pragma unroll
        for (int c = 0; c < NI; ++c) u[c] = U[at(t, NI, c, Np, i)] + s * DU[at(t, NI, c, Np, i)];  // optcon.py:197 / :253
        if (WRITE) {
            store_x(Xn, t, Np, i, x);
#pragma unroll
            for (int c = 0; c < NI; ++c) Un[at(t, NI, c, Np, i)] = u[c];
        }
        if (COST) load_ref(P, t, i, xr, ur);
        rollout_step<COST, Q32>(P.M, P.W, x, u, xr, ur, J);
    }
    if (WRITE) {
        store_x(Xn, TT - 1, Np, i, x);
        Un[at(TT - 1, NI, 0, Np, i)] = F(0.0);  // uu_temp[:, TT-1] is never written (optcon.py:193)
        Un[at(TT - 1, NI, 1, Np, i)] = F(0.0);
    }
    if (COST) {
        load_xref(P, TT - 1, i, xr);
#pragma unroll
        for (int c = 0; c < NS; ++c) dx[c] = x[c] - xr[c];
        J += (double)term_cost(P.W, dx);
    }
    return J;
}

// ------------------------------------------------------------------------------------------------------
// Armijo decision + Newton bookkeeping for one instance (optcon.py:266-273, :327, :497-501)
// ------------------------------------------------------------------------------------------------------
struct NewtonOpts {
    int max_iters;         // optcon.py:367 (loop runs max_iters-1 bodies, :415)
    int armijo_maxiters;   // :230
    int exact_after;       // exact Hessian iff kk > exact_after (:443; 8 in the reference)
    double stepsize_0, cc, beta;  // :224-229
    double term_cond;      // :368  (-1e-6, hard-coded in the reference)
    int method;            // 0: NewtonMethod.optimize; 1: GradientMethod.optimize (steepest descent; S.descent holds the slope -|deltau|^2)
};

enum InstStatus : int { ST_ACTIVE = 0, ST_CONVERGED = 1, ST_MAXITER = 2, ST_NONFINITE = 3 };

struct NewtonState {          // all arrays of length Np unless noted
    int* status;              // InstStatus
    int* iters;               // loop bodies executed so far
    int* result_slot;         // slot (0..2) holding what optimize() returns, -1 = the all-zero slot (:503 with kk = 0)
    double* Jcur;             // cost of the current iterate
    double* descent;          // descent of the current iterate
    double* step;             // chosen step
    double* Jcand;            // [armijo_maxiters][Np]
    double* hist_J;           // [max_iters][Np]
    double* hist_descent;     // [max_iters][Np]
    double* hist_step;        // [max_iters][Np]
    int* hist_ncand;          // [max_iters][Np]   candidates the sequential search would have rolled out
    int* n_reg;               // accumulated +0.5 I firings
};

// cand_steps[c] = stepsize_0 * beta^c built by repeated multiplication like :270 (length armijo_maxiters+1)
ACOC_HD void armijo_select_instance(const NewtonOpts& O, const NewtonState& S, const double* cand_steps, int kk, int Np, int i)
{
    const double JP = S.Jcur[i], d = S.descent[i];
    int chosen = -1;
    for (int c = 0; c < O.armijo_maxiters; ++c) {
        const double Jc = S.Jcand[(size_t)c * Np + i];
        const double sc = cand_steps[c];
        if (!(Jc > JP + O.cc * sc * d)) { chosen = c; break; }   // :268, NaN accepts like the reference's else-branch
    }
    const double s = cand_steps[chosen >= 0 ? chosen : O.armijo_maxiters];  // untested step on exhaustion (:327)
    S.step[i] = s;
    S.hist_J[(size_t)kk * Np + i] = JP;
    S.hist_descent[(size_t)kk * Np + i] = d;
    S.hist_step[(size_t)kk * Np + i] = s;
    S.hist_ncand[(size_t)kk * Np + i] = chosen >= 0 ? chosen + 1 : O.armijo_maxiters;
}

// after get_update: termination test (:499-501) and result-slot bookkeeping (:503)
ACOC_HD void newton_finish_instance(const NewtonOpts& O, const NewtonState& S, double Jnext, int kk, int i)
{
    const double d = S.descent[i];
    S.iters[i] = kk + 1;
    S.Jcur[i] = Jnext;
    if (d >= O.term_cond) {
        S.status[i] = ST_CONVERGED;
        S.result_slot[i] = kk == 0 ? -1 : (kk - 1) % 3;
    } else if (!(fabs(d) <= 1.7e308) || !(fabs(Jnext) <= 1.7e308)) {
        // NaN/Inf: the reference would keep iterating on NaNs until max_iters; we freeze the instance instead
        S.status[i] = ST_NONFINITE;
        S.result_slot[i] = (kk + 1) % 3;
    } else if (kk + 1 >= O.max_iters - 1) {
        S.status[i] = ST_MAXITER;
        S.result_slot[i] = (kk + 1) % 3;
    }
}

// ------------------------------------------------------------------------------------------------------
// closed-loop tracking rollout, lqr_tracking.py:279-281: u = u_opt + K (x - x_opt) with shared K, nominal
// ------------------------------------------------------------------------------------------------------
// the input of one closed-loop step: u = u_opt + K@(x - x_opt), K row-major 2x6.  Plain sums in index order (the reference's 2x6
// matvec), then u_opt + (.)
template <typename F>
ACOC_HD void track_input(const F* K, const F* x, const F* xopt, const F* uopt, F* u)
{
#pragma unroll
    for (int a = 0; a < NI; ++a) {
        F s = F(0.0);
#pragma unroll
        for (int c = 0; c < NS; ++c) s += K[a * NS + c] * (x[c] - xopt[c]);
        u[a] = uopt[a] + s;
    }
}

// Kt: [TT][12] (row-major 2x6), xopt [TT][6], uopt [TT][2] shared by all instances; x_start [6][Np].
template <bool Q32, typename F, typename XT>
ACOC_HD void track_instance(const ProblemT<F>& P, const F* Kt, const F* xopt, const F* uopt,
                            const F* xstart, XT* Xn, F* Un, int i)
{
    const int TT = P.TT, Np = P.Np;
    F x[NS], xn[NS], u[NI];
#pragma unroll
    for (int c = 0; c < NS; ++c) x[c] = xstart[(size_t)c * Np + i];
    for (int t = 0; t < TT - 1; ++t) {
        track_input(Kt + (size_t)t * 12, x, xopt + (size_t)t * NS, uopt + (size_t)t * NI, u);
        store_x(Xn, t, Np, i, x);
#pragma unroll
        for (int c = 0; c < NI; ++c) Un[at(t, NI, c, Np, i)] = u[c];
        const Trig<F> tg = make_trig(x);
        next_state<Q32>(P.M, x, u, tg, xn);
#pragma unroll
        for (int c = 0; c < NS; ++c) x[c] = xn[c];
    }
    store_x(Xn, TT - 1, Np, i, x);
    Un[at(TT - 1, NI, 0, Np, i)] = F(0.0);
    Un[at(TT - 1, NI, 1, Np, i)] = F(0.0);
}

// ------------------------------------------------------------------------------------------------------
// closed-loop LQR tracking of every instance along its OWN nominal, lqr_tracking.py:245-283 (acoc_track, acoc_lqr_tracking_many)
// ------------------------------------------------------------------------------------------------------
// Each instance is one call of the reference's lqr_tracking: nominal Xnom/Unom (warp-tiled like the iterates, Ktrk [TT][Np/32][12][32]),
// P.W = the TRACKING weights, P.x0 = the exact row 0 of the nominal (finish_x reads it when Xnom is float).
// Gains (:276, non-augmented ltv_LQR): riccati_matrix<false> with q = r = 0 on the linearisation at (x*_t, u*_t), from P_{TT-1} = QT; the
// affine terms it also carries stay zero (NaN along a non-finite nominal) and do not enter K.  K_{TT-1} = 0 (ltv_LQR never assigns it).
template <int DG = -1, typename F>
ACOC_HD void track_terminal(const WeightsT<F>& W, F* Pm, F* p)
{
#pragma unroll
    for (int a = 0; a < NS; ++a) {
        p[a] = F(0.0);
#pragma unroll
        for (int b = a; b < NS; ++b) Pm[sym(a, b)] = weights_diag<DG>(W) ? (a == b ? W.QT[a * 7] : F(0.0)) : W.QT[a * 6 + b];
    }
}

// one step of the gains sweep: (x*_t, u*_t) and the carried (P, p) -> K_t.  Returns 1 if the gain took the +0.5 I branch.
template <int DG = -1, typename F>
ACOC_HD int track_gains_step(const ModelT<F>& M, const WeightsT<F>& W, const F* x, const F* u, F* Pm, F* p, F* K)
{
    const F q[NS] = {F(0.0), F(0.0), F(0.0), F(0.0), F(0.0), F(0.0)}, r[NI] = {F(0.0), F(0.0)};
    const Trig<F> tg = make_trig(x);
    const Lin<F> l = linearize(M, x, u, tg);
    Hess<F> h;
    F sig[NI];
    return riccati_matrix<false, DG, F>(M, W, l, h, q, r, Pm, p, K, sig);
}

template <int DG, typename F, typename XT>
ACOC_HD int track_gains_instance(const ProblemT<F>& P, const XT* Xnom, const F* Unom, F* Ktrk, int i)
{
    const int TT = P.TT, Np = P.Np;
    F Pm[21], p[NS], x[NS], u[NI], K[2 * NS];
    track_terminal<DG>(P.W, Pm, p);
#pragma unroll
    for (int c = 0; c < 2 * NS; ++c) Ktrk[at(TT - 1, 2 * NS, c, Np, i)] = F(0.0);
    int nreg = 0;
    for (int t = TT - 2; t >= 0; --t) {
        load_x(P, Xnom, t, i, x);
#pragma unroll
        for (int c = 0; c < NI; ++c) u[c] = Unom[at(t, NI, c, Np, i)];
        nreg += track_gains_step<DG>(P.M, P.W, x, u, Pm, p, K);
#pragma unroll
        for (int c = 0; c < 2 * NS; ++c) Ktrk[at(t, 2 * NS, c, Np, i)] = K[c];
    }
    return nreg;
}

// running max that keeps a NaN once it has seen one (fmax would drop it)
template <typename F>
ACOC_HD F max_nan(F m, F v) { return (v > m || v != v) ? v : m; }

// closed loop (:279-281): x_0 = x*_0 + delta; u_t = u*_t + K_t (x_t - x*_t), x_{t+1} = f(x_t, u_t) for t < TT-1; u_{TT-1} = 0.
// Summaries: err_max[c] = max_t |x_t[c] - x*_t[c]|, err_final[c] at t = TT-1 ([6][Np] each).  Row 0 of a float Xtrk is not exact:
// the exact x_0 goes to xtrk0 [6][Np].
template <typename F>
ACOC_HD void track_error(const F* x, const F* xnom, F* emax)
{
#pragma unroll
    for (int c = 0; c < NS; ++c) emax[c] = max_nan(emax[c], F(fabs(x[c] - xnom[c])));
}
template <bool Q32, typename F>
ACOC_HD void track_advance(const ModelT<F>& M, F* x, const F* u)
{
    const Trig<F> tg = make_trig(x);
    F xn[NS];
    next_state<Q32>(M, x, u, tg, xn);
#pragma unroll
    for (int c = 0; c < NS; ++c) x[c] = xn[c];
}
// x_0 = x*_0 + d6 (d6 = this start's perturbation, 6 values): the one start expression of acoc_track and acoc_track_mc
template <typename F>
ACOC_HD void track_start_from(const ProblemT<F>& P, int i, const F* d6, F* x, F* emax)
{
#pragma unroll
    for (int c = 0; c < NS; ++c) { x[c] = P.x0[(size_t)c * P.Np + i] + d6[c]; emax[c] = F(0.0); }
}
template <typename F>
ACOC_HD void track_start(const ProblemT<F>& P, const F* delta, int i, F* x, F* emax)
{
    F d6[NS];
#pragma unroll
    for (int c = 0; c < NS; ++c) d6[c] = delta[(size_t)c * P.Np + i];
    track_start_from(P, i, d6, x, emax);
}
// summaries at t = TT-1: emax takes the last error, efin = |x_{TT-1} - x*_{TT-1}|
template <typename F>
ACOC_HD void track_final_err(const F* x, const F* xnom, F* emax, F* efin)
{
    track_error(x, xnom, emax);
#pragma unroll
    for (int c = 0; c < NS; ++c) efin[c] = F(fabs(x[c] - xnom[c]));
}
template <typename F>
ACOC_HD void track_final(const F* x, const F* xnom, F* emax, F* err_max, F* err_final, int Np, int i)
{
    F efin[NS];
    track_final_err(x, xnom, emax, efin);
#pragma unroll
    for (int c = 0; c < NS; ++c) {
        err_max[(size_t)c * Np + i] = emax[c];
        err_final[(size_t)c * Np + i] = efin[c];
    }
}

template <bool Q32, typename F, typename XT>
ACOC_HD void track_rollout_instance(const ProblemT<F>& P, const XT* Xnom, const F* Unom, const F* Ktrk, const F* delta, XT* Xtrk, F* xtrk0,
                                    F* Utrk, F* err_max, F* err_final, int i)
{
    const int TT = P.TT, Np = P.Np;
    F x[NS], emax[NS], xn[NS], un[NI], u[NI], K[2 * NS];
    track_start(P, delta, i, x, emax);
#pragma unroll
    for (int c = 0; c < NS; ++c) xtrk0[(size_t)c * Np + i] = x[c];
    for (int t = 0; t < TT - 1; ++t) {
        load_x(P, Xnom, t, i, xn);
#pragma unroll
        for (int c = 0; c < NI; ++c) un[c] = Unom[at(t, NI, c, Np, i)];
#pragma unroll
        for (int c = 0; c < 2 * NS; ++c) K[c] = Ktrk[at(t, 2 * NS, c, Np, i)];
        track_error(x, xn, emax);
        track_input(K, x, xn, un, u);
        store_x(Xtrk, t, Np, i, x);
#pragma unroll
        for (int c = 0; c < NI; ++c) Utrk[at(t, NI, c, Np, i)] = u[c];
        track_advance<Q32>(P.M, x, u);
    }
    load_x(P, Xnom, TT - 1, i, xn);
    store_x(Xtrk, TT - 1, Np, i, x);
    Utrk[at(TT - 1, NI, 0, Np, i)] = F(0.0);
    Utrk[at(TT - 1, NI, 1, Np, i)] = F(0.0);
    track_final(x, xn, emax, err_max, err_final, Np, i);
}

// ------------------------------------------------------------------------------------------------------
// Monte Carlo dispersion of the closed loop (acoc_track_mc, acoc_lqr_tracking_mc): M perturbed starts per instance, same nominal and
// gains.  One sample is acoc_track's closed loop without the trajectory stores: its summaries are bit-identical to acoc_track's with
// delta[i] = d6.  Per-sample summaries are stored sample-major, em / ef [N][M][6].
// ------------------------------------------------------------------------------------------------------
template <bool Q32, typename F, typename XT>
ACOC_HD void track_mc_sample(const ProblemT<F>& P, const XT* Xnom, const F* Unom, const F* Ktrk, const F* d6, int i, F* em, F* ef)
{
    const int TT = P.TT, Np = P.Np;
    F x[NS], emax[NS], xn[NS], un[NI], u[NI], K[2 * NS];
    track_start_from(P, i, d6, x, emax);
    for (int t = 0; t < TT - 1; ++t) {
        load_x(P, Xnom, t, i, xn);
#pragma unroll
        for (int c = 0; c < NI; ++c) un[c] = Unom[at(t, NI, c, Np, i)];
#pragma unroll
        for (int c = 0; c < 2 * NS; ++c) K[c] = Ktrk[at(t, 2 * NS, c, Np, i)];
        track_error(x, xn, emax);
        track_input(K, x, xn, un, u);
        track_advance<Q32>(P.M, x, u);
    }
    load_x(P, Xnom, TT - 1, i, xn);
    track_final_err(x, xn, emax, ef);
#pragma unroll
    for (int c = 0; c < NS; ++c) em[c] = emax[c];
}

// Fixed-order aggregates of one instance over its M samples (em, ef: [M][6] of that instance): worst[c] = max_nan over m in sample
// order, mean[c] = (((ef_0 + ef_1) + ef_2) + ...) / M, and (tol != nullptr) the number of samples with em[m][c] <= tol[c] for every c
// (a NaN is never within).
template <typename F>
ACOC_HD int track_mc_reduce(const F* em, const F* ef, int M, const F* tol, F* worst, F* mean)
{
    int within = 0;
#pragma unroll
    for (int c = 0; c < NS; ++c) { worst[c] = em[c]; mean[c] = ef[c]; }
    for (int m = 0; m < M; ++m) {
        const F* e = em + (size_t)m * NS;
        if (m > 0) {
#pragma unroll
            for (int c = 0; c < NS; ++c) { worst[c] = max_nan(worst[c], e[c]); mean[c] += ef[(size_t)m * NS + c]; }
        }
        if (tol) {
            bool in = true;
#pragma unroll
            for (int c = 0; c < NS; ++c) in = in && e[c] <= tol[c];
            within += in ? 1 : 0;
        }
    }
#pragma unroll
    for (int c = 0; c < NS; ++c) mean[c] /= F(M);
    return within;
}

// ------------------------------------------------------------------------------------------------------
// derivative of the optimum with respect to the references and the initial state (acoc_result_vjp; definition in include/acoc.h)
// ------------------------------------------------------------------------------------------------------
// The adjoint LQ problem along the result (x*, u*):  min 1/2 w'Hw - gbar'w  s.t.  w_{x,t+1} = A_t w_{x,t} + B_t w_{u,t},  w_{x,0} = 0,
// H = the Hessian of the Lagrangian (Q + lam_{t+1}-contracted f_xx, S_t, R; Q_T at t = TT-1).  The backward sweep carries the adjoint's
// value function V_t(w) = 1/2 w'P_t w + p_t'w and the costate lam of the original problem (the Newton sweep's recursion, with the
// exact Hessian at every step).  riccati_matrix's affine terms are half the linear terms (q/2, r/2), so the sweep hands it q = -2 gbar_x,
// r = -2 gbar_u (exact scalings).  The gains use the plain G^-1 (never G + 0.5 I): the result is then the exact solution of the KKT
// system wherever it is nonsingular; the steps whose G is not positive definite (riccati_gain_test) are counted.
// The sensitivity of the initial state needs no forward pass: x0 enters the adjoint only through w_{x,0}, so xi_bar = gbar_{x,0} -
// A_0'eta_1 - S_0'w_{u,0} = -grad V_0(0) = -p_0 (with the linear term -gbar_{x,0} of step 0 folded into p_0).
// VKS (warp-tiled, 14 components): K_t row-major 2x6, sigma_t.

// terminal condition: P = QT, p = -gbar_{x,TT-1}, lam = QT (x*_{TT-1} - xref_{TT-1})
template <int DG = -1, typename F>
ACOC_HD void vjp_terminal(const WeightsT<F>& W, const F* x, const F* xr, const F* gx, F* Pm, F* p, F* lam)
{
    F dx[NS];
#pragma unroll
    for (int c = 0; c < NS; ++c) dx[c] = x[c] - xr[c];
    wmul6(W.QT, (int)weights_diag<DG>(W), dx, lam);
    track_terminal<DG>(W, Pm, p);
#pragma unroll
    for (int c = 0; c < NS; ++c) p[c] = -gx[c];
}

// riccati_matrix_by_columns with the plain inverse in the gains.  Returns 1 if G is not positive definite.
template <int DG = -1, typename F>
ACOC_HD int vjp_matrix(const ModelT<F>& M, const WeightsT<F>& W, const Lin<F>& l, const Hess<F>& h, const F* q, const F* r, F* Pm, F* p, F* K,
                       F* sig)
{
    RicGain<F> gn;
    riccati_gain_core(M, W, l, r, Pm, p, gn);
    riccati_gain_test(gn);
    gn.k00 = gn.gi00; gn.k01 = gn.gi01; gn.k11 = gn.gi11;
    F Pn[NS][NS], Mx0[NS], Mx1[NS], Atp[NS];
    riccati_cols_a_<true, DG, 0, F>(M, l, h, Pm, Pn, Mx0, Mx1);
    riccati_p_sweep(M, l, p, Atp);
    riccati_cols_b_<true, DG, 0, F>(W, h, gn, Pn, Mx0, Mx1, Pm);
    riccati_p_finish(q, Atp, Mx0, Mx1, gn.y0, gn.y1, p);
    riccati_gain_out(gn, Mx0, Mx1, K, sig);
    return gn.reg;
}

// one backward step: (x*_t, u*_t, refs, gbar_t) and the carried (P, p, lam_{t+1}) -> K_t, sigma_t; (P, p, lam) at t.  Returns 1 if G_t is
// not positive definite.
template <int DG = -1, typename F>
ACOC_HD int vjp_backward_step(const ModelT<F>& M, const WeightsT<F>& W, const F* x, const F* u, const F* xr, const F* ur, const F* gx,
                              const F* gu, F* Pm, F* p, F* lam, F* K, F* sig)
{
    F dx[NS], du[NI], q[NS], r[NI], qa[NS], ra[NI], g[NI];
#pragma unroll
    for (int c = 0; c < NS; ++c) { dx[c] = x[c] - xr[c]; qa[c] = F(-2.0) * gx[c]; }
#pragma unroll
    for (int c = 0; c < NI; ++c) { du[c] = u[c] - ur[c]; ra[c] = F(-2.0) * gu[c]; }
    wmul6(W.Q, (int)weights_diag<DG>(W), dx, q);
    wmul2(W.R, (int)weights_diag<DG>(W), du, r);
    const Trig<F> tg = make_trig(x);
    const Lin<F> l = linearize(M, x, u, tg);
    const Hess<F> h = hess_contract(M, x, u, tg, l, lam);
    const int indef = vjp_matrix<DG, F>(M, W, l, h, qa, ra, Pm, p, K, sig);
    riccati_costate(M, l, q, r, lam, g);
    return indef;
}

// gbar of instance i at time t (warp-tiled GX [TT][6], GU [TT][2]); gbar_u[TT-1] is folded into t = TT-2 (result() copies u_{TT-2} there)
template <typename F>
ACOC_HD void vjp_load_g(const F* GX, const F* GU, int t, int TT, int Np, int i, F* gx, F* gu)
{
#pragma unroll
    for (int c = 0; c < NS; ++c) gx[c] = GX[at(t, NS, c, Np, i)];
#pragma unroll
    for (int c = 0; c < NI; ++c) gu[c] = GU[at(t, NI, c, Np, i)];
    if (t == TT - 2) {
#pragma unroll
        for (int c = 0; c < NI; ++c) gu[c] = gu[c] + GU[at(TT - 1, NI, c, Np, i)];
    }
}

// whole backward sweep of one instance over the nominal (X, U; P.x0 = its exact row 0): VKS, xi_bar [6][Np]; returns n_indef
template <int DG, typename F, typename XT>
ACOC_HD int vjp_backward_instance(const ProblemT<F>& P, const XT* X, const F* U, const F* GX, const F* GU, F* VKS, F* xi_bar, int i)
{
    const int TT = P.TT, Np = P.Np;
    F Pm[21], p[NS], lam[NS], x[NS], u[NI], xr[NS], ur[NI], gx[NS], gu[NI];
    load_xref(P, TT - 1, i, xr);
    load_x(P, X, TT - 1, i, x);
    vjp_load_g(GX, GU, TT - 1, TT, Np, i, gx, gu);
    vjp_terminal<DG>(P.W, x, xr, gx, Pm, p, lam);
    int n = 0;
    for (int t = TT - 2; t >= 0; --t) {
        load_ref(P, t, i, xr, ur);
        load_x(P, X, t, i, x);
#pragma unroll
        for (int c = 0; c < NI; ++c) u[c] = U[at(t, NI, c, Np, i)];
        vjp_load_g(GX, GU, t, TT, Np, i, gx, gu);
        F K[2 * NS], sig[NI];
        n += vjp_backward_step<DG>(P.M, P.W, x, u, xr, ur, gx, gu, Pm, p, lam, K, sig);
#pragma unroll
        for (int c = 0; c < 12; ++c) VKS[at(t, 14, c, Np, i)] = K[c];
        VKS[at(t, 14, 12, Np, i)] = sig[0]; VKS[at(t, 14, 13, Np, i)] = sig[1];
    }
#pragma unroll
    for (int c = 0; c < NS; ++c) xi_bar[(size_t)c * Np + i] = -p[c];
    return n;
}

// Parametric references (acoc_set_refs_generated): zf_bar, vx_bar from xref_bar by the chain rule, in ascending t.  X_t = vx tt_t,
// Z_t = zs_t zf, and for the step maneuver V_t = sqrt((vs_t zf)^2 + vx^2): dV/dzf = vs_t^2 zf / V_t, dV/dvx = vx / V_t.
struct VjpParamSums {
    double z, zv, x, xv;  // sum zs_t Zbar_t, sum dV/dzf Vbar_t, sum tt_t Xbar_t, sum dV/dvx Vbar_t
};
// vs_t, v_t: the step maneuver's speed table entry and this instance's stored V_t (has_v); xb: xref_bar_t
ACOC_HD void vjp_param_add(VjpParamSums& s, double tt_t, double zs_t, bool has_v, double vs_t, double v_t, double zf, double vx, const double* xb)
{
    s.z += zs_t * xb[1];
    s.x += tt_t * xb[0];
    if (has_v) {
        s.zv += (((vs_t * vs_t) * zf) / v_t) * xb[2];
        s.xv += (vx / v_t) * xb[2];
    }
}

// one forward step: w_{u,t} = sigma_t + K_t w_{x,t} (ks: K_t, sigma_t), outputs xb = Q w_{x,t} (QT at TT-1, 0 at t = 0), ub = R w_{u,t},
// w_{x,t+1} = A_t w_{x,t} + B_t w_{u,t}
template <int DG = -1, typename F>
ACOC_HD void vjp_forward_step(const ModelT<F>& M, const WeightsT<F>& W, int t, const F* x, const F* u, const F* ks, F* wx, F* xb, F* ub)
{
    F ksg[16], wu[NI];
#pragma unroll
    for (int c = 0; c < 14; ++c) ksg[c] = ks[c];
    ksg[14] = F(0.0); ksg[15] = F(0.0);
    double unused = 0.0;
    forward_du(ksg, wx, wu, unused);
    if (t == 0) {
#pragma unroll
        for (int c = 0; c < NS; ++c) xb[c] = F(0.0);
    } else wmul6(W.Q, (int)weights_diag<DG>(W), wx, xb);
    wmul2(W.R, (int)weights_diag<DG>(W), wu, ub);
    forward_advance(M, x, u, wu, wx);
}

// whole forward sweep of one instance: XB (N,6) / UB (N,2) warp-tiled (either may be nullptr), zv [2][Np] (nullptr: no parametric sums)
template <int DG, typename F, typename XT>
ACOC_HD void vjp_forward_instance(const ProblemT<F>& P, const XT* X, const F* U, const F* VKS, const double* vs, F* XB, F* UB, double* zv, int i)
{
    const int TT = P.TT, Np = P.Np;
    const bool has_v = P.ref_param && P.rp_v;
    const double zf = zv ? (double)P.rp_zf[i] : 0.0, vx = zv ? (double)P.rp_vx[i] : 0.0;
    VjpParamSums s = {0.0, 0.0, 0.0, 0.0};
    F wx[NS] = {0, 0, 0, 0, 0, 0}, x[NS], u[NI], ks[14], xb[NS], ub[NI];
    for (int t = 0; t < TT - 1; ++t) {
        load_x(P, X, t, i, x);
#pragma unroll
        for (int c = 0; c < NI; ++c) u[c] = U[at(t, NI, c, Np, i)];
#pragma unroll
        for (int c = 0; c < 14; ++c) ks[c] = VKS[at(t, 14, c, Np, i)];
        vjp_forward_step<DG>(P.M, P.W, t, x, u, ks, wx, xb, ub);
        if (XB) {
#pragma unroll
            for (int c = 0; c < NS; ++c) XB[at(t, NS, c, Np, i)] = xb[c];
        }
        if (UB) {
#pragma unroll
            for (int c = 0; c < NI; ++c) UB[at(t, NI, c, Np, i)] = ub[c];
        }
        if (zv) vjp_param_add(s, P.rp_tt[t], P.rp_zs[t], has_v, has_v ? vs[t] : 0.0, has_v ? (double)param_vref(P, t, i) : 0.0, zf, vx, xb);
    }
    wmul6(P.W.QT, (int)weights_diag<DG>(P.W), wx, xb);
    if (XB) {
#pragma unroll
        for (int c = 0; c < NS; ++c) XB[at(TT - 1, NS, c, Np, i)] = xb[c];
    }
    if (UB) {
#pragma unroll
        for (int c = 0; c < NI; ++c) UB[at(TT - 1, NI, c, Np, i)] = F(0.0);
    }
    if (zv) {
        const int t = TT - 1;
        vjp_param_add(s, P.rp_tt[t], P.rp_zs[t], has_v, has_v ? vs[t] : 0.0, has_v ? (double)param_vref(P, t, i) : 0.0, zf, vx, xb);
        zv[i] = s.z + s.zv;
        zv[(size_t)Np + i] = s.x + s.xv;
    }
}

// ------------------------------------------------------------------------------------------------------
// initial guess, aircraft_simplified.py:126-148 (float64 arithmetic; see DESIGN.md "initial guess")
// ------------------------------------------------------------------------------------------------------
// dx0 (optional, [6][Np]): start from xx_ref[:,0] + dx0 instead (perturbed-initial-state batches, config 5)
// x0_out (optional, [6][Np], may alias dx0): receives the exact start state (row 0 of a float X slot is not exact)
template <bool Q32, typename F, typename XT>
ACOC_HD void init_guess_instance(const ProblemT<F>& P, F kp, F kt, const F* dx0, XT* Xn, F* Un, F* x0_out, int i)
{
    const int TT = P.TT, Np = P.Np;
    F x[NS], xn[NS], u[NI], xr[NS];
    load_xref(P, 0, i, x);  // x_temp = xx_ref[:,0]  (:139)
    if (dx0) {
#pragma unroll
        for (int c = 0; c < NS; ++c) x[c] += dx0[(size_t)c * Np + i];
    }
    if (x0_out) {
#pragma unroll
        for (int c = 0; c < NS; ++c) x0_out[(size_t)c * Np + i] = x[c];
    }
    for (int t = 0; t < TT - 1; ++t) {
        load_xref(P, t + 1, i, xr);
        u[0] = kp * ((x[0] - xr[0]) + (x[1] - xr[1]));   // :143
        u[1] = kt * ((x[3] - xr[3]) + (x[5] - xr[5]));   // :144
        store_x(Xn, t, Np, i, x);
#pragma unroll
        for (int c = 0; c < NI; ++c) Un[at(t, NI, c, Np, i)] = u[c];
        const Trig<F> tg = make_trig(x);
        next_state<Q32>(P.M, x, u, tg, xn);
#pragma unroll
        for (int c = 0; c < NS; ++c) x[c] = xn[c];
    }
    store_x(Xn, TT - 1, Np, i, x);
    Un[at(TT - 1, NI, 0, Np, i)] = F(0.0);
    Un[at(TT - 1, NI, 1, Np, i)] = F(0.0);
}

// ------------------------------------------------------------------------------------------------------
// pointwise entry points: Dynamics.step with all derivative tensors, Cost.stagecost / termcost
// ------------------------------------------------------------------------------------------------------
// Sample-major inputs x[n][6], u[n][2], lam[n][6] (NULL -> full tensors).  Outputs per sample:
//   xxp[6]; A[36] = fx.T row-major; B[12] = fu.T (6x2 row-major);
//   lam == NULL: fxx[216] ([i][j][k] = d2f_k/dx_i dx_j), fux[72] ([a][j][k]);  else fxx[36], fux[12] contracted.
ACOC_HD void step_sample(const Model& M, bool q32, const double* x, const double* u, const double* lam,
                         double* xxp, double* A, double* B, double* fxx, double* fux)
{
    const Trig<double> tg = make_trig(x);
    if (xxp) { if (q32) next_state<true>(M, x, u, tg, xxp); else next_state<false>(M, x, u, tg, xxp); }
    const Lin<double> l = linearize(M, x, u, tg);
    if (A) {
        for (int e = 0; e < 36; ++e) A[e] = 0.0;
        A[0] = 1.0; A[2] = l.a02; A[5] = l.a05;
        A[7] = 1.0; A[8] = l.a12; A[11] = l.a15;
        A[14] = l.a22; A[15] = l.a23; A[17] = l.a25;
        A[21] = 1.0; A[22] = M.dt;
        A[28] = 1.0;
        A[32] = l.a52; A[33] = l.a53; A[35] = l.a55;
    }
    if (B) {
        for (int e = 0; e < 12; ++e) B[e] = 0.0;
        B[4] = l.b20; B[9] = M.b41; B[10] = l.b50;
    }
    if (!fxx && !fux) return;
    if (lam) {
        const Hess<double> h = hess_contract(M, x, u, tg, l, lam);
        if (fxx) {
            for (int e = 0; e < 36; ++e) fxx[e] = 0.0;
            fxx[2 * 6 + 2] = h.h22; fxx[2 * 6 + 3] = h.h23; fxx[3 * 6 + 2] = h.h23; fxx[2 * 6 + 5] = h.h25; fxx[5 * 6 + 2] = h.h25;
            fxx[3 * 6 + 3] = h.h33; fxx[3 * 6 + 5] = h.h35; fxx[5 * 6 + 3] = h.h35; fxx[5 * 6 + 5] = h.h55;
        }
        if (fux) {
            for (int e = 0; e < 12; ++e) fux[e] = 0.0;
            fux[2] = h.s2; fux[3] = h.s3; fux[5] = h.s5;
        }
    } else {
        // full tensors: contract with unit costates, one output slice at a time
        const int ks[4] = {0, 1, 2, 5};
        if (fxx) for (int e = 0; e < 216; ++e) fxx[e] = 0.0;
        if (fux) for (int e = 0; e < 72; ++e) fux[e] = 0.0;
        for (int c = 0; c < 4; ++c) {
            double e6[NS] = {0, 0, 0, 0, 0, 0};
            e6[ks[c]] = 1.0;
            const Hess<double> h = hess_contract(M, x, u, tg, l, e6);
            const int k = ks[c];
            if (fxx) {
                fxx[(2 * 6 + 2) * 6 + k] = h.h22; fxx[(2 * 6 + 3) * 6 + k] = h.h23; fxx[(3 * 6 + 2) * 6 + k] = h.h23;
                fxx[(2 * 6 + 5) * 6 + k] = h.h25; fxx[(5 * 6 + 2) * 6 + k] = h.h25; fxx[(3 * 6 + 3) * 6 + k] = h.h33;
                fxx[(3 * 6 + 5) * 6 + k] = h.h35; fxx[(5 * 6 + 3) * 6 + k] = h.h35; fxx[(5 * 6 + 5) * 6 + k] = h.h55;
            }
            if (fux) { fux[(0 * 6 + 2) * 6 + k] = h.s2; fux[(0 * 6 + 3) * 6 + k] = h.s3; fux[(0 * 6 + 5) * 6 + k] = h.s5; }
        }
    }
}

// stagecost / termcost for one sample: ll, lx[6], lu[2], llT, lTx[6]
ACOC_HD void cost_sample(const Weights& W, const double* x, const double* u, const double* xr, const double* ur,
                         double* ll, double* lx, double* lu, double* llT, double* lTx)
{
    double dx[NS], du[NI];
    for (int c = 0; c < NS; ++c) dx[c] = x[c] - xr[c];
    if (u && ll) {
        for (int c = 0; c < NI; ++c) du[c] = u[c] - ur[c];
        *ll = stage_cost(W, dx, du);
        wmul6(W.Q, W.diag, dx, lx);
        wmul2(W.R, W.diag, du, lu);
    }
    if (llT) { *llT = term_cost(W, dx); wmul6(W.QT, W.diag, dx, lTx); }
}

// ------------------------------------------------------------------------------------------------------
// generic dense LTV-LQ solve: the drop-in for ltv_LQR (optcon.py:533-771) on arbitrary A_t, B_t, Q_t, R_t, S_t
// ------------------------------------------------------------------------------------------------------
// One thread solves one problem, literally: n = 7 (augmented by the affine terms, optcon.py:655-697) or 6.
// Time-major row-major inputs A[t][6][6], B[t][6][2], Q[t][6][6], R[t][2][2], S[t][2][6], Qf[6][6], x0[6],
// q[t][6], r[t][2], qf[6].  Outputs K[t][2][n], P[t][n][n] (optional), xout[t][6], uout[t][2].
// Used by the ltv_LQR drop-in and by lqr_tracking (one shared solve); the Newton loop uses the fused
// structure-exploiting sweeps above instead.
template <int N>
ACOC_HD void lq_dense_problem(int TT, const double* A, const double* B, const double* Q, const double* R, const double* S,
                              const double* Qf, const double* x0, const double* q, const double* r, const double* qf,
                              double* K, double* Pout, double* xout, double* uout, int* n_reg)
{
    constexpr int off = N - NS;  // 1 when augmented
    double Pn[N * N], At[N * N], Bt[N * NI], Qt[N * N], St[NI * N];
    for (int e = 0; e < N * N; ++e) Pn[e] = 0.0;
    for (int i = 0; i < NS; ++i) {
        if (off) { const double hq = 0.5 * qf[i]; Pn[(i + 1) * N] = hq; Pn[i + 1] = hq; }   // optcon.py:688-689
        for (int j = 0; j < NS; ++j) Pn[(i + off) * N + (j + off)] = Qf[i * NS + j];            // :690 / :706
    }
    if (Pout) for (int e = 0; e < N * N; ++e) Pout[(size_t)(TT - 1) * N * N + e] = Pn[e];
    for (int e = 0; e < NI * N; ++e) K[(size_t)(TT - 1) * NI * N + e] = 0.0;
    int nreg = 0;
    for (int t = TT - 2; t >= 0; --t) {
        for (int e = 0; e < N * N; ++e) { At[e] = 0.0; Qt[e] = 0.0; }
        for (int e = 0; e < N * NI; ++e) { Bt[e] = 0.0; St[e] = 0.0; }
        if (off) {
            At[0] = 1.0;  // :684
            for (int i = 0; i < NS; ++i) { const double hq = 0.5 * q[(size_t)t * NS + i]; Qt[(i + 1) * N] = hq; Qt[i + 1] = hq; }  // :673-674
            for (int a = 0; a < NI; ++a) St[a * N] = 0.5 * r[(size_t)t * NI + a];                                                 // :679
        }
        for (int i = 0; i < NS; ++i)
            for (int j = 0; j < NS; ++j) {
                At[(i + off) * N + (j + off)] = A[((size_t)t * NS + i) * NS + j];
                Qt[(i + off) * N + (j + off)] = Q[((size_t)t * NS + i) * NS + j];
            }
        for (int i = 0; i < NS; ++i) for (int a = 0; a < NI; ++a) Bt[(i + off) * NI + a] = B[((size_t)t * NS + i) * NI + a];
        for (int a = 0; a < NI; ++a) for (int j = 0; j < NS; ++j) St[a * N + (j + off)] = S[((size_t)t * NI + a) * NS + j];
        // BtP = B'P (2xN), Mx = BtP A + S, G = R + BtP B
        double BtP[NI * N], Mx[NI * N], G[4];
        for (int a = 0; a < NI; ++a)
            for (int j = 0; j < N; ++j) { double s = 0.0; for (int k = 0; k < N; ++k) s = fma_(Bt[k * NI + a], Pn[k * N + j], s); BtP[a * N + j] = s; }
        for (int a = 0; a < NI; ++a)
            for (int j = 0; j < N; ++j) { double s = 0.0; for (int k = 0; k < N; ++k) s = fma_(BtP[a * N + k], At[k * N + j], s); Mx[a * N + j] = s + St[a * N + j]; }
        for (int a = 0; a < NI; ++a)
            for (int b = 0; b < NI; ++b) { double s = 0.0; for (int k = 0; k < N; ++k) s = fma_(BtP[a * N + k], Bt[k * NI + b], s); G[a * NI + b] = R[(size_t)t * 4 + a * NI + b] + s; }
        // explicit inverse of G (:728)
        const double idet = 1.0 / fma_(G[0], G[3], -(G[1] * G[2]));
        const double Gi[4] = {G[3] * idet, -G[1] * idet, -G[2] * idet, G[0] * idet};
        // gain matrix: eigenvalue test (:745), +0.5 I (:749), K = -inv(MM) Mx (:751)
        double MM[4] = {G[0], G[1], G[2], G[3]};
        {
            const double hd = 0.5 * (MM[0] - MM[3]), disc = fma_(hd, hd, MM[1] * MM[2]), mid = 0.5 * (MM[0] + MM[3]);
            bool pd;
            if (disc >= 0.0) { const double rad = sqrt(disc); pd = (mid - rad > 0.0) && (mid + rad > 0.0); }
            else pd = (disc < 0.0) && (mid > 0.0);
            if (!pd) { MM[0] += 0.5; MM[3] += 0.5; ++nreg; }
        }
        const double id2 = 1.0 / fma_(MM[0], MM[3], -(MM[1] * MM[2]));
        const double Mi[4] = {MM[3] * id2, -MM[1] * id2, -MM[2] * id2, MM[0] * id2};
        for (int a = 0; a < NI; ++a)
            for (int j = 0; j < N; ++j)
                K[((size_t)t * NI + a) * N + j] = -fma_(Mi[a * NI + 1], Mx[N + j], Mi[a * NI] * Mx[j]);
        // P_t = Q + A'PA - Mx' Gi Mx (:727-728)
        double AtP[N * N], Y[NI * N], Pt[N * N];
        for (int i = 0; i < N; ++i)
            for (int j = 0; j < N; ++j) { double s = 0.0; for (int k = 0; k < N; ++k) s = fma_(At[k * N + i], Pn[k * N + j], s); AtP[i * N + j] = s; }
        for (int a = 0; a < NI; ++a)
            for (int j = 0; j < N; ++j) Y[a * N + j] = fma_(Gi[a * NI + 1], Mx[N + j], Gi[a * NI] * Mx[j]);
        for (int i = 0; i < N; ++i)
            for (int j = 0; j < N; ++j) {
                double s = 0.0;
                for (int k = 0; k < N; ++k) s = fma_(AtP[i * N + k], At[k * N + j], s);
                Pt[i * N + j] = (Qt[i * N + j] + s) - fma_(Mx[N + i], Y[N + j], Mx[i] * Y[j]);
            }
        for (int e = 0; e < N * N; ++e) Pn[e] = Pt[e];
        if (Pout) for (int e = 0; e < N * N; ++e) Pout[(size_t)t * N * N + e] = Pt[e];
    }
    if (n_reg) *n_reg = nreg;
    // forward pass (:756-762)
    double xa[N], xb[N], ua[NI];
    if (off) xa[0] = 1.0;
    for (int i = 0; i < NS; ++i) { xa[i + off] = x0[i]; xout[i] = x0[i]; }
    for (int t = 0; t < TT - 1; ++t) {
        for (int a = 0; a < NI; ++a) {
            double s = 0.0;
            for (int j = 0; j < N; ++j) s = fma_(K[((size_t)t * NI + a) * N + j], xa[j], s);
            ua[a] = s; uout[(size_t)t * NI + a] = s;
        }
        if (off) xb[0] = 1.0;
        for (int i = 0; i < NS; ++i) {
            double s1 = 0.0, s2 = 0.0;
            for (int j = 0; j < NS; ++j) s1 = fma_(A[((size_t)t * NS + i) * NS + j], xa[j + off], s1);
            for (int a = 0; a < NI; ++a) s2 = fma_(B[((size_t)t * NS + i) * NI + a], ua[a], s2);
            xb[i + off] = s1 + s2;
        }
        for (int i = 0; i < N; ++i) xa[i] = xb[i];
        for (int i = 0; i < NS; ++i) xout[(size_t)(t + 1) * NS + i] = xa[i + off];
    }
    uout[(size_t)(TT - 1) * NI] = 0.0; uout[(size_t)(TT - 1) * NI + 1] = 0.0;
}

}  // namespace acoc
