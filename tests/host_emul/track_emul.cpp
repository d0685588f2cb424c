// track_emul.cpp -- TEST-ONLY host replay of the kernels of closed-loop tracking of every instance (acoc_track, acoc_lqr_tracking_many).
//
// Compiled with g++ -ffp-contract=off like emul.cpp (matching nvcc -fmad=false): the per-instance functions of acoc_kernels.cuh
// (track_gains_instance, track_rollout_instance) driven with plain loops over instances, on the same warp-tiled buffers and with the same
// choice of state storage as acoc_lqr_tracking_many.  Not part of the product: libacoc.so does not contain it.
#include <cstring>
#include <vector>

#include "../../aircraftoptimalcontrol_b200/csrc/acoc_kernels.cuh"

using namespace acoc;

namespace {
// host (n,C,TT) float64 -> warp-tiled SoA of D (k_to_soa)
template <typename D>
void to_soa(const double* host, D* dst, int n, int C, int TT, int Np)
{
    for (int i = 0; i < n; ++i)
        for (int c = 0; c < C; ++c)
            for (int t = 0; t < TT; ++t) dst[at(t, C, c, Np, i)] = (D)host[((size_t)i * C + c) * TT + t];
}
// warp-tiled SoA -> host (C,TT) of instance i (k_from_soa); row0 (optional, [C][Np]): exact t = 0 column
template <typename D>
void from_soa(const D* src, double* host, int i, int C, int TT, int Np, const double* row0)
{
    for (int c = 0; c < C; ++c)
        for (int t = 0; t < TT; ++t) host[(size_t)c * TT + t] = (row0 && t == 0) ? row0[(size_t)c * Np + i] : (double)src[at(t, C, c, Np, i)];
}
// fill_weights of acoc_api.cu: diagonal iff every off-diagonal entry of Q, R, QT is zero
void fill_weights(Weights* W, const double* Q, const double* R, const double* QT)
{
    memcpy(W->Q, Q, sizeof(W->Q)); memcpy(W->R, R, sizeof(W->R)); memcpy(W->QT, QT, sizeof(W->QT));
    bool d = true;
    for (int i = 0; i < 6; ++i) for (int j = 0; j < 6; ++j) if (i != j && (Q[i * 6 + j] != 0.0 || QT[i * 6 + j] != 0.0)) d = false;
    if (R[1] != 0.0 || R[2] != 0.0) d = false;
    W->diag = d;
}

template <typename XT>
void track_many_impl(int N, int TT, const double* params, int state_f64, const double* Q, const double* R, const double* QT,
                     const double* xx_opt, const double* uu_opt, const double* delta, double* xx_reg, double* uu_reg, double* K,
                     double* err_max, double* err_final, int* n_reg)
{
    const int Np = (N + 31) / 32 * 32;
    std::vector<XT> Xnom((size_t)TT * 6 * Np, XT(0)), Xtrk((size_t)TT * 6 * Np, XT(0));
    std::vector<double> Unom((size_t)TT * 2 * Np, 0.0), Kt((size_t)TT * 12 * Np, 0.0), Utrk((size_t)TT * 2 * Np, 0.0);
    std::vector<double> x0((size_t)6 * Np, 0.0), xt0((size_t)6 * Np, 0.0), dl((size_t)6 * Np, 0.0), em((size_t)6 * Np), ef((size_t)6 * Np);
    to_soa(xx_opt, Xnom.data(), N, 6, TT, Np);
    to_soa(uu_opt, Unom.data(), N, 2, TT, Np);
    for (int i = 0; i < N; ++i)
        for (int c = 0; c < 6; ++c) { x0[(size_t)c * Np + i] = xx_opt[((size_t)i * 6 + c) * TT]; dl[(size_t)c * Np + i] = delta[(size_t)i * 6 + c]; }
    Problem P;
    P.M = make_model(params);
    fill_weights(&P.W, Q, R, QT);
    P.N = N; P.Np = Np; P.TT = TT; P.q32 = state_f64 ? 0 : 1; P.ref_shared = 0; P.ref_param = 0;
    P.xref = nullptr; P.uref = nullptr; P.x0 = x0.data();
    const XT* Xn = Xnom.data();
    const double *Un = Unom.data(), *Kc = Kt.data(), *D = dl.data();
    for (int i = 0; i < N; ++i) {
        n_reg[i] = P.W.diag ? track_gains_instance<1>(P, Xn, Un, Kt.data(), i) : track_gains_instance<0>(P, Xn, Un, Kt.data(), i);
        if (P.q32) track_rollout_instance<true>(P, Xn, Un, Kc, D, Xtrk.data(), xt0.data(), Utrk.data(), em.data(), ef.data(), i);
        else track_rollout_instance<false>(P, Xn, Un, Kc, D, Xtrk.data(), xt0.data(), Utrk.data(), em.data(), ef.data(), i);
        from_soa(Xtrk.data(), xx_reg + (size_t)i * 6 * TT, i, 6, TT, Np, xt0.data());
        from_soa(Utrk.data(), uu_reg + (size_t)i * 2 * TT, i, 2, TT, Np, nullptr);
        from_soa(Kt.data(), K + (size_t)i * 12 * TT, i, 12, TT, Np, nullptr);
        for (int c = 0; c < 6; ++c) { err_max[(size_t)i * 6 + c] = em[(size_t)c * Np + i]; err_final[(size_t)i * 6 + c] = ef[(size_t)c * Np + i]; }
    }
}
}  // namespace

extern "C" {

// acoc_lqr_tracking_many replayed: float state storage when every state at t >= 1 is a float32 value (float32 quantisation only), exact
// row 0 always.  xx_opt (N,6,TT), uu_opt (N,2,TT), delta (N,6) -> xx_reg (N,6,TT), uu_reg (N,2,TT), K (N,2,6,TT), err_max / err_final
// (N,6), n_reg (N).
void emul_track_many(int N, int TT, const double* params, int state_f64, const double* Q, const double* R, const double* QT, const double* xx_opt,
                     const double* uu_opt, const double* delta, double* xx_reg, double* uu_reg, double* K, double* err_max, double* err_final,
                     int* n_reg)
{
    bool x_float = !state_f64;
    for (size_t i = 0; i < (size_t)N * 6 && x_float; ++i)
        for (int t = 1; t < TT; ++t) { const double v = xx_opt[i * TT + t]; if (!((double)(float)v == v) && v == v) { x_float = false; break; } }
    if (x_float) track_many_impl<float>(N, TT, params, state_f64, Q, R, QT, xx_opt, uu_opt, delta, xx_reg, uu_reg, K, err_max, err_final, n_reg);
    else track_many_impl<double>(N, TT, params, state_f64, Q, R, QT, xx_opt, uu_opt, delta, xx_reg, uu_reg, K, err_max, err_final, n_reg);
}

}  // extern "C"
