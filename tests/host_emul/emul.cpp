// emul.cpp -- TEST-ONLY host replay of the CUDA kernels' per-instance code.
//
// The build container has no GPU.  The per-instance bodies of every kernel (acoc_kernels.cuh) are
// __host__ __device__, so this file compiles them with g++ (-ffp-contract=off, matching nvcc -fmad=false)
// and drives them with plain loops over instances, using the same struct-of-arrays buffers and the same
// iteration sequence as acoc_api.cu.  `-m "not gpu"` tests use it to check the kernel arithmetic against the
// oracle before any GPU time is spent.  It is NOT part of the product: libacoc.so does not contain it and
// the package never loads it.
#include <algorithm>
#include <cstring>
#include <vector>

#include "../../aircraftoptimalcontrol_b200/csrc/acoc_kernels.cuh"

using namespace acoc;

namespace {
// dispatch on the runtime state-quantisation flag like the kernel launches in acoc_api.cu (with_flag)
template <bool WRITE, bool COST, typename F, typename XT>
double rollout_q(const ProblemT<F>& P, const F* U, const F* DU, double s, XT* Xn, F* Un, int i)
{
    return P.q32 ? rollout_instance<WRITE, COST, true>(P, U, DU, s, Xn, Un, i) : rollout_instance<WRITE, COST, false>(P, U, DU, s, Xn, Un, i);
}

// host (n,C,TT) float64 -> SoA of D (k_to_soa); returns whether any value at t >= 1 does not survive the conversion
template <typename D>
bool to_soa(const double* host, D* dst, int n, int C, int TT, int Np)
{
    bool inexact = false;
    for (int i = 0; i < n; ++i)
        for (int c = 0; c < C; ++c)
            for (int t = 0; t < TT; ++t) {
                const double v = host[((size_t)i * C + c) * TT + t];
                const D d = (D)v;
                dst[Np == 1 ? (size_t)t * C + c : at(t, C, c, Np, i)] = d;  // Np == 1: shared reference, plain [TT][C]
                if (t >= 1 && !((double)d == v) && v == v) inexact = true;
            }
    return inexact;
}
// SoA -> host (k_from_soa); row0 (optional): exact t = 0 column
template <typename D, typename R0>
void from_soa(const D* src, double* host, int i, int C, int TT, int Np, const R0* row0 = (const R0*)nullptr)
{
    for (int c = 0; c < C; ++c)
        for (int t = 0; t < TT; ++t)
            host[(size_t)c * TT + t] = (row0 && t == 0) ? (double)row0[(size_t)c * Np + i] : (double)src[Np == 1 ? (size_t)t * C + c : at(t, C, c, Np, i)];
}
template <typename D>
void from_soa(const D* src, double* host, int i, int C, int TT, int Np) { from_soa<D, double>(src, host, i, C, TT, Np, nullptr); }

void fill_weights(Weights* W, const double* Q, const double* R, const double* QT)
{
    memcpy(W->Q, Q, sizeof(W->Q)); memcpy(W->R, R, sizeof(W->R)); memcpy(W->QT, QT, sizeof(W->QT));
    bool d = true;
    for (int i = 0; i < 6; ++i) for (int j = 0; j < 6; ++j) if (i != j && (Q[i * 6 + j] != 0.0 || QT[i * 6 + j] != 0.0)) d = false;
    if (R[1] != 0.0 || R[2] != 0.0) d = false;
    W->diag = d;
}

struct NewtonArgs {
    int N, TT;
    const double* params;
    int state_f64;
    const double *Q, *R, *QT, *xx_ref, *uu_ref;
    int ref_shared;
    const double *xx_init, *uu_init;
    int max_iters;
    double stepsize_0, cc, beta;
    int armijo_maxiters, exact_after;
    double term_cond;
    int n_iters_cap, lazy;
    double *hist_J, *hist_descent, *hist_step;
    int *hist_ncand, *iters, *status;
    double *xx_star, *uu_star, *xx_last, *uu_last, *du_last, *K_last, *sigma_last;
    int* n_reg_out;
    int method;  // 0 NewtonMethod.optimize, 1 GradientMethod.optimize (ACOC_METHOD_GRADIENT)
};

// The lock-step Newton driver of acoc_api.cu (acoc_newton_iterate) replayed on the host for one <F, XT> instantiation.
template <typename F, typename XT>
int newton_impl(const NewtonArgs& a)
{
    const int N = a.N, TT = a.TT, max_iters = a.max_iters, armijo_maxiters = a.armijo_maxiters;
    const int Np = (N + 31) / 32 * 32;
    std::vector<XT> X[3];
    std::vector<F> U[3], DU, KSG, xref, uref, x0;
    for (int s = 0; s < 3; ++s) { X[s].assign((size_t)TT * 6 * Np, XT(0)); U[s].assign((size_t)TT * 2 * Np, F(0)); }
    DU.assign((size_t)TT * 2 * Np, F(0)); KSG.assign((size_t)TT * 16 * Np, F(0));
    const int Nr = a.ref_shared ? 1 : Np;
    xref.assign((size_t)TT * 6 * Nr, F(0)); uref.assign((size_t)TT * 2 * Nr, F(0)); x0.assign((size_t)6 * Np, F(0));
    to_soa(a.xx_ref, xref.data(), a.ref_shared ? 1 : N, 6, TT, Nr);
    to_soa(a.uu_ref, uref.data(), a.ref_shared ? 1 : N, 2, TT, Nr);
    to_soa(a.xx_init, X[0].data(), N, 6, TT, Np);
    to_soa(a.uu_init, U[0].data(), N, 2, TT, Np);
    for (int i = 0; i < N; ++i) for (int c = 0; c < 6; ++c) x0[(size_t)c * Np + i] = (F)a.xx_init[((size_t)i * 6 + c) * TT];  // x0 = xx_init[:,0]

    Weights W64;
    fill_weights(&W64, a.Q, a.R, a.QT);
    ProblemT<F> P;
    P.M = model_as<F>(make_model(a.params));
    P.W = weights_as<F>(W64);
    P.N = N; P.Np = Np; P.TT = TT; P.q32 = a.state_f64 ? 0 : 1; P.ref_shared = a.ref_shared; P.ref_param = 0;
    P.xref = xref.data(); P.uref = uref.data(); P.x0 = x0.data();
    NewtonOpts O;
    O.max_iters = max_iters; O.armijo_maxiters = armijo_maxiters; O.exact_after = a.exact_after;
    O.stepsize_0 = a.stepsize_0; O.cc = a.cc; O.beta = a.beta; O.term_cond = a.term_cond; O.method = a.method;
    std::vector<int> st(Np, ST_ACTIVE), its(Np, 0), slot(Np, 0), ncand((size_t)max_iters * Np, 0), nreg(Np, 0);
    std::vector<double> Jcur(Np, 0.0), desc(Np, 0.0), step(Np, 0.0), Jc((size_t)(armijo_maxiters + 1) * Np, 0.0);
    std::vector<double> hJ((size_t)max_iters * Np, 0.0), hD((size_t)max_iters * Np, 0.0), hS((size_t)max_iters * Np, 0.0);
    NewtonState S;
    S.status = st.data(); S.iters = its.data(); S.result_slot = slot.data(); S.Jcur = Jcur.data(); S.descent = desc.data();
    S.step = step.data(); S.Jcand = Jc.data(); S.hist_J = hJ.data(); S.hist_descent = hD.data(); S.hist_step = hS.data();
    S.hist_ncand = ncand.data(); S.n_reg = nreg.data();
    std::vector<double> cs(armijo_maxiters + 1);
    { double s = a.stepsize_0; for (int k = 0; k <= armijo_maxiters; ++k) { cs[k] = s; s = a.beta * s; } }

    int kk = 0;
    for (;; ++kk) {
        if (kk >= max_iters - 1) break;
        if (a.n_iters_cap > 0 && kk >= a.n_iters_cap) break;
        int active = 0;
        for (int i = 0; i < N; ++i) active += st[i] == ST_ACTIVE;
        if (!active) break;
        const int cur = kk % 3, nxt = (kk + 1) % 3;
        const XT* Xc = X[cur].data();
        const F* Uc = U[cur].data();
        XT* Xn = X[nxt].data();
        F* Un = U[nxt].data();
        for (int i = 0; i < N; ++i) {
            if (st[i] != ST_ACTIVE) continue;
            if (kk == 0) Jcur[i] = traj_cost_instance(P, Xc, Uc, i);
            if (a.method == 1) desc[i] = -gradient_instance(P, Xc, Uc, DU.data(), i);  // k_gradient_tma: slope = -sum |deltau|^2
            else {
                nreg[i] += (kk > a.exact_after) ? backward_instance<true>(P, Xc, Uc, KSG.data(), i) : backward_instance<false>(P, Xc, Uc, KSG.data(), i);
                desc[i] = forward_lq_instance(P, Xc, Uc, KSG.data(), DU.data(), (F*)nullptr, i);
            }
            bool cand0_in_place = false;
            if (a.lazy && armijo_maxiters > 1) {
                Jc[i] = rollout_q<true, true>(P, Uc, DU.data(), cs[0], Xn, Un, i);
                const bool need = Jc[i] > Jcur[i] + a.cc * cs[0] * desc[i];
                if (need) for (int c = 1; c < armijo_maxiters; ++c) Jc[(size_t)c * Np + i] = rollout_q<false, true>(P, Uc, DU.data(), cs[c], (XT*)nullptr, (F*)nullptr, i);
                cand0_in_place = !need;
            } else {
                for (int c = 0; c < armijo_maxiters; ++c) Jc[(size_t)c * Np + i] = rollout_q<false, true>(P, Uc, DU.data(), cs[c], (XT*)nullptr, (F*)nullptr, i);
            }
            armijo_select_instance(O, S, cs.data(), kk, Np, i);
            const double Jn = cand0_in_place ? Jc[i] : rollout_q<true, true>(P, Uc, DU.data(), step[i], Xn, Un, i);
            newton_finish_instance(O, S, Jn, kk, i);
        }
    }
    const F* row0 = std::is_same<F, XT>::value ? (const F*)nullptr : x0.data();
    for (int i = 0; i < N; ++i) {
        for (int k = 0; k < max_iters; ++k) {
            if (a.hist_J) a.hist_J[(size_t)i * max_iters + k] = hJ[(size_t)k * Np + i];
            if (a.hist_descent) a.hist_descent[(size_t)i * max_iters + k] = hD[(size_t)k * Np + i];
            if (a.hist_step) a.hist_step[(size_t)i * max_iters + k] = hS[(size_t)k * Np + i];
            if (a.hist_ncand) a.hist_ncand[(size_t)i * max_iters + k] = ncand[(size_t)k * Np + i];
        }
        if (a.iters) a.iters[i] = its[i];
        if (a.status) a.status[i] = st[i];
        if (a.n_reg_out) a.n_reg_out[i] = nreg[i];
        const int sl = st[i] == ST_ACTIVE ? kk % 3 : slot[i];
        if (a.xx_star) {
            double *xs = a.xx_star + (size_t)i * 6 * TT, *us = a.uu_star + (size_t)i * 2 * TT;
            if (sl < 0) { memset(xs, 0, sizeof(double) * 6 * TT); memset(us, 0, sizeof(double) * 2 * TT); }
            else { from_soa(X[sl].data(), xs, i, 6, TT, Np, row0); from_soa(U[sl].data(), us, i, 2, TT, Np); }
            for (int c = 0; c < 2; ++c) us[(size_t)c * TT + TT - 1] = us[(size_t)c * TT + TT - 2];
        }
        // newest iterate of instance i: the one written in its last executed body
        const int last = its[i] % 3;
        if (a.xx_last) from_soa(X[last].data(), a.xx_last + (size_t)i * 6 * TT, i, 6, TT, Np, row0);
        if (a.uu_last) from_soa(U[last].data(), a.uu_last + (size_t)i * 2 * TT, i, 2, TT, Np);
        if (a.du_last) from_soa(DU.data(), a.du_last + (size_t)i * 2 * TT, i, 2, TT, Np);
        if (a.K_last) {
            std::vector<double> tmp((size_t)16 * TT);
            from_soa(KSG.data(), tmp.data(), i, 16, TT, Np);
            memcpy(a.K_last + (size_t)i * 12 * TT, tmp.data(), sizeof(double) * 12 * TT);
            if (a.sigma_last) memcpy(a.sigma_last + (size_t)i * 2 * TT, tmp.data() + (size_t)12 * TT, sizeof(double) * 2 * TT);
        }
    }
    return kk;
}
}  // namespace

// riccati_matrix() against its decomposition by columns (k_backward_cols), driven along the backward sweep of a real trajectory so that
// P, p, the linearisation and the Hessian terms have their real magnitudes: both variants carry their own (P, p) and every K, sigma,
// P, p is compared bit for bit.  scale_R < 1 shrinks R so that the +0.5 I branch is taken too.  Returns the number of differing
// numbers (0 = identical); *n_reg_out = steps that took the regularised branch.
template <bool EXACT, int DG>
static long cols_check(const Model& M, const Weights& W, int TT, const double* xx, const double* uu, const double* xr_, const double* ur_, int* n_reg_out)
{
    double Pa[21], pa[NS], Pb[21], pb[NS], lam[NS], x[NS], xr[NS], u[NI], ur[NI];
    for (int c = 0; c < NS; ++c) { x[c] = xx[(size_t)c * TT + TT - 1]; xr[c] = xr_[(size_t)c * TT + TT - 1]; }
    backward_terminal<DG>(W, x, xr, Pa, pa, lam);
    memcpy(Pb, Pa, sizeof(Pa)); memcpy(pb, pa, sizeof(pa));
    long bad = 0;
    int nreg = 0;
    for (int t = TT - 2; t >= 0; --t) {
        for (int c = 0; c < NS; ++c) { x[c] = xx[(size_t)c * TT + t]; xr[c] = xr_[(size_t)c * TT + t]; }
        for (int c = 0; c < NI; ++c) { u[c] = uu[(size_t)c * TT + t]; ur[c] = ur_[(size_t)c * TT + t]; }
        double dx[NS], du[NI], q[NS], r[NI], g[NI];
        for (int c = 0; c < NS; ++c) dx[c] = x[c] - xr[c];
        for (int c = 0; c < NI; ++c) du[c] = u[c] - ur[c];
        wmul6(W.Q, (int)weights_diag<DG>(W), dx, q);
        wmul2(W.R, (int)weights_diag<DG>(W), du, r);
        const Trig<double> tg = make_trig(x);
        const Lin<double> l = linearize(M, x, u, tg);
        Hess<double> h = Hess<double>();
        if (EXACT) h = hess_contract(M, x, u, tg, l, lam);
        double Ka[12], sa[2], Kb[12], sb[2];
        const int ra = riccati_matrix<EXACT, DG, double>(M, W, l, h, q, r, Pa, pa, Ka, sa);
        Hess<double> h2 = Hess<double>();
        if (EXACT) {   // the kernel's warps form the Hessian terms in two pieces
            h2 = hess_post(hess_pre(M, x, tg, l), lam);
            bad += memcmp(&h, &h2, sizeof(h)) != 0;
        }
        const int rb = riccati_matrix_by_columns<EXACT, DG, double>(M, W, l, h2, q, r, Pb, pb, Kb, sb);
        riccati_costate(M, l, q, r, lam, g);
        nreg += ra;
        bad += ra != rb;
        bad += memcmp(Ka, Kb, sizeof(Ka)) != 0;
        bad += memcmp(sa, sb, sizeof(sa)) != 0;
        bad += memcmp(Pa, Pb, sizeof(Pa)) != 0;
        bad += memcmp(pa, pb, sizeof(pa)) != 0;
    }
    if (n_reg_out) *n_reg_out = nreg;
    return bad;
}

extern "C" {

void emul_step_batch(int n, const double* params, int state_f64, const double* x, const double* u, const double* lam,
                     double* xxp, double* A, double* B, double* fxx, double* fux)
{
    const Model M = make_model(params);
    const size_t nxx = lam ? 36 : 216, nux = lam ? 12 : 72;
    for (int s = 0; s < n; ++s)
        step_sample(M, !state_f64, x + (size_t)s * 6, u + (size_t)s * 2, lam ? lam + (size_t)s * 6 : nullptr, xxp ? xxp + (size_t)s * 6 : nullptr,
                    A ? A + (size_t)s * 36 : nullptr, B ? B + (size_t)s * 12 : nullptr, fxx ? fxx + s * nxx : nullptr, fux ? fux + s * nux : nullptr);
}

void emul_cost_batch(int n, const double* Q, const double* R, const double* QT, const double* x, const double* u, const double* xr,
                     const double* ur, double* ll, double* lx, double* lu, double* llT, double* lTx)
{
    Weights W;
    fill_weights(&W, Q, R, QT);
    for (int s = 0; s < n; ++s)
        cost_sample(W, x + (size_t)s * 6, u + (size_t)s * 2, xr + (size_t)s * 6, ur + (size_t)s * 2, ll + s, lx + (size_t)s * 6, lu + (size_t)s * 2,
                    llT + s, lTx + (size_t)s * 6);
}

long emul_riccati_cols_check(int TT, const double* params, const double* Q, const double* R, const double* QT, const double* xx, const double* uu,
                             const double* xx_ref, const double* uu_ref, int exact, int* n_reg_out)
{
    const Model M = make_model(params);
    Weights W;
    fill_weights(&W, Q, R, QT);
    if (W.diag) return exact ? cols_check<true, 1>(M, W, TT, xx, uu, xx_ref, uu_ref, n_reg_out) : cols_check<false, 1>(M, W, TT, xx, uu, xx_ref, uu_ref, n_reg_out);
    return exact ? cols_check<true, 0>(M, W, TT, xx, uu, xx_ref, uu_ref, n_reg_out) : cols_check<false, 0>(M, W, TT, xx, uu, xx_ref, uu_ref, n_reg_out);
}

void emul_ltv_lqr(int TT, const double* A, const double* B, const double* Q, const double* R, const double* S, const double* Qf,
                  const double* x0, const double* q, const double* r, const double* qf, double* K, double* P, double* xout, double* uout, int* n_reg)
{
    if (q) lq_dense_problem<7>(TT, A, B, Q, R, S, Qf, x0, q, r, qf, K, P, xout, uout, n_reg);
    else lq_dense_problem<6>(TT, A, B, Q, R, S, Qf, x0, nullptr, nullptr, nullptr, K, P, xout, uout, n_reg);
}

// The lock-step Newton driver replayed on the host.
// hist_* are (N, max_iters) row-major; xx_* (N,6,TT); uu_* (N,2,TT); K_last (N,12,TT); sigma_last (N,2,TT).
// mode 0: like the library -- float64 arithmetic; the state slots are float when the states are float32-quantised and the
//         initial trajectory is exactly representable (acoc_set_init), else float64
// mode 1: float64 state slots always (ACOC_X_F64);  mode 2: the FP32 mode (ACOC_FP32)
int emul_newton_batch(int N, int TT, const double* params, int state_f64, const double* Q, const double* R, const double* QT,
                      const double* xx_ref, const double* uu_ref, int ref_shared, const double* xx_init, const double* uu_init,
                      int max_iters, double stepsize_0, double cc, double beta, int armijo_maxiters, int exact_after, double term_cond,
                      int n_iters_cap, int lazy,
                      double* hist_J, double* hist_descent, double* hist_step, int* hist_ncand, int* iters, int* status,
                      double* xx_star, double* uu_star, double* xx_last, double* uu_last, double* du_last, double* K_last, double* sigma_last,
                      int* n_reg_out, int mode)
{
    const NewtonArgs a{N, TT, params, state_f64, Q, R, QT, xx_ref, uu_ref, ref_shared, xx_init, uu_init, max_iters, stepsize_0, cc, beta,
                       armijo_maxiters, exact_after, term_cond, n_iters_cap, lazy, hist_J, hist_descent, hist_step, hist_ncand, iters, status,
                       xx_star, uu_star, xx_last, uu_last, du_last, K_last, sigma_last, n_reg_out, mode >> 8};
    mode &= 255;  // (bits 8.. of `mode`: the method, so that the signature stays what emul.py binds)
    if (mode == 2) return newton_impl<float, float>(a);
    bool x_float = false;
    if (mode == 0 && !state_f64) {
        x_float = true;
        for (size_t i = 0; i < (size_t)N * 6 && x_float; ++i)
            for (int t = 1; t < TT; ++t) { const double v = xx_init[i * TT + t]; if (!((double)(float)v == v) && v == v) { x_float = false; break; } }
    }
    return x_float ? newton_impl<double, float>(a) : newton_impl<double, double>(a);
}

// rollout of u + s*du for a batch (get_update / one Armijo candidate)
void emul_rollout_batch(int N, int TT, const double* params, int state_f64, const double* Q, const double* R, const double* QT,
                        const double* xx_ref, const double* uu_ref, const double* x0, const double* uu, const double* du, const double* s,
                        double* xx_out, double* uu_out, double* J)
{
    const int Np = (N + 31) / 32 * 32;
    std::vector<double> U((size_t)TT * 2 * Np), DU((size_t)TT * 2 * Np), Xn((size_t)TT * 6 * Np), Un((size_t)TT * 2 * Np);
    std::vector<double> xr((size_t)TT * 6 * Np), ur((size_t)TT * 2 * Np), x0s((size_t)6 * Np, 0.0);
    to_soa(uu, U.data(), N, 2, TT, Np); to_soa(du, DU.data(), N, 2, TT, Np);
    to_soa(xx_ref, xr.data(), N, 6, TT, Np); to_soa(uu_ref, ur.data(), N, 2, TT, Np);
    for (int i = 0; i < N; ++i) for (int c = 0; c < 6; ++c) x0s[(size_t)c * Np + i] = x0[(size_t)i * 6 + c];
    Problem P;
    P.M = make_model(params); fill_weights(&P.W, Q, R, QT);
    P.N = N; P.Np = Np; P.TT = TT; P.q32 = state_f64 ? 0 : 1; P.ref_shared = 0; P.ref_param = 0;
    P.xref = xr.data(); P.uref = ur.data(); P.x0 = x0s.data();
    for (int i = 0; i < N; ++i) {
        J[i] = rollout_q<true, true>(P, (const double*)U.data(), (const double*)DU.data(), s[i], Xn.data(), Un.data(), i);
        from_soa(Xn.data(), xx_out + (size_t)i * 6 * TT, i, 6, TT, Np);
        from_soa(Un.data(), uu_out + (size_t)i * 2 * TT, i, 2, TT, Np);
    }
}

void emul_lqr_tracking(int N, int TT, const double* params, int state_f64, const double* Q, const double* R, const double* QT,
                       const double* xx_opt, const double* uu_opt, const double* delta, double* xx_reg, double* uu_reg, double* K)
{
    const int Np = (N + 31) / 32 * 32;
    const Model M = make_model(params);
    std::vector<double> xo((size_t)TT * 6), uo((size_t)TT * 2), A((size_t)TT * 36), B((size_t)TT * 12), S((size_t)TT * 12, 0.0);
    std::vector<double> Qr((size_t)TT * 36), Rr((size_t)TT * 4), Kt((size_t)TT * 12), xout((size_t)TT * 6), uout((size_t)TT * 2);
    to_soa(xx_opt, xo.data(), 1, 6, TT, 1); to_soa(uu_opt, uo.data(), 1, 2, TT, 1);
    for (int t = 0; t < TT; ++t) {
        step_sample(M, !state_f64, &xo[(size_t)t * 6], &uo[(size_t)t * 2], nullptr, nullptr, &A[(size_t)t * 36], &B[(size_t)t * 12], nullptr, nullptr);
        memcpy(&Qr[(size_t)t * 36], Q, sizeof(double) * 36); memcpy(&Rr[(size_t)t * 4], R, sizeof(double) * 4);
    }
    lq_dense_problem<6>(TT, A.data(), B.data(), Qr.data(), Rr.data(), S.data(), QT, delta, nullptr, nullptr, nullptr, Kt.data(), nullptr, xout.data(), uout.data(), nullptr);
    if (K) memcpy(K, Kt.data(), sizeof(double) * TT * 12);
    std::vector<double> xs((size_t)6 * Np, 0.0), Xn((size_t)TT * 6 * Np), Un((size_t)TT * 2 * Np);
    for (int i = 0; i < N; ++i) for (int c = 0; c < 6; ++c) xs[(size_t)c * Np + i] = xx_opt[(size_t)c * TT] + delta[(size_t)i * 6 + c];
    Problem P;
    P.M = M; P.N = N; P.Np = Np; P.TT = TT; P.q32 = state_f64 ? 0 : 1; P.ref_shared = 1; P.ref_param = 0;
    P.xref = xo.data(); P.uref = uo.data(); P.x0 = xs.data();
    for (int i = 0; i < N; ++i) {
        if (P.q32) track_instance<true>(P, Kt.data(), xo.data(), uo.data(), xs.data(), Xn.data(), Un.data(), i);
        else track_instance<false>(P, Kt.data(), xo.data(), uo.data(), xs.data(), Xn.data(), Un.data(), i);
        from_soa(Xn.data(), xx_reg + (size_t)i * 6 * TT, i, 6, TT, Np);
        from_soa(Un.data(), uu_reg + (size_t)i * 2 * TT, i, 2, TT, Np);
    }
}

void emul_init_guess(int N, int TT, const double* params, int state_f64, const double* xx_ref, double kp, double kt, double* xx, double* uu)
{
    const int Np = (N + 31) / 32 * 32;
    std::vector<double> xr((size_t)TT * 6 * Np), Xn((size_t)TT * 6 * Np), Un((size_t)TT * 2 * Np);
    to_soa(xx_ref, xr.data(), N, 6, TT, Np);
    Problem P;
    P.M = make_model(params); P.N = N; P.Np = Np; P.TT = TT; P.q32 = state_f64 ? 0 : 1; P.ref_shared = 0; P.ref_param = 0;
    P.xref = xr.data(); P.uref = nullptr; P.x0 = nullptr;
    for (int i = 0; i < N; ++i) {
        if (P.q32) init_guess_instance<true>(P, kp, kt, (const double*)nullptr, Xn.data(), Un.data(), (double*)nullptr, i);
        else init_guess_instance<false>(P, kp, kt, (const double*)nullptr, Xn.data(), Un.data(), (double*)nullptr, i);
        from_soa(Xn.data(), xx + (size_t)i * 6 * TT, i, 6, TT, Np);
        from_soa(Un.data(), uu + (size_t)i * 2 * TT, i, 2, TT, Np);
    }
}

}  // extern "C"
