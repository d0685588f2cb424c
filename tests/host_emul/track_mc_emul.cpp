// track_mc_emul.cpp -- TEST-ONLY host replay of the Monte Carlo dispersion kernels (acoc_track_mc, acoc_lqr_tracking_mc).
//
// Compiled with g++ -ffp-contract=off like the other replays (matching nvcc -fmad=false): the per-instance gains sweep and the
// per-sample / reduction functions of acoc_kernels.cuh (track_gains_instance, track_mc_sample, track_mc_reduce) driven with plain loops
// over instances and samples, on the same warp-tiled buffers and with the same choice of state storage as acoc_lqr_tracking_mc.  It
// reuses the layout helpers of the tracking replay by including it, so this library also exports emul_track_many.  Not part of the
// product: libacoc.so does not contain it.
#include "track_emul.cpp"

namespace {
template <typename XT>
void track_mc_impl(int N, int M, int TT, const double* params, int state_f64, const double* Q, const double* R, const double* QT,
                   const double* xx_opt, const double* uu_opt, const double* delta, int delta_shared, const double* tol, double* err_max,
                   double* err_final, double* worst_max, double* mean_final, int* n_within, int* n_reg)
{
    const int Np = (N + 31) / 32 * 32;
    std::vector<XT> Xnom((size_t)TT * 6 * Np, XT(0));
    std::vector<double> Unom((size_t)TT * 2 * Np, 0.0), Kt((size_t)TT * 12 * Np, 0.0), x0((size_t)6 * Np, 0.0);
    to_soa(xx_opt, Xnom.data(), N, 6, TT, Np);
    to_soa(uu_opt, Unom.data(), N, 2, TT, Np);
    for (int i = 0; i < N; ++i)
        for (int c = 0; c < 6; ++c) x0[(size_t)c * Np + i] = xx_opt[((size_t)i * 6 + c) * TT];
    Problem P;
    P.M = make_model(params);
    fill_weights(&P.W, Q, R, QT);
    P.N = N; P.Np = Np; P.TT = TT; P.q32 = state_f64 ? 0 : 1; P.ref_shared = 0; P.ref_param = 0;
    P.xref = nullptr; P.uref = nullptr; P.x0 = x0.data();
    const size_t dstride = delta_shared ? 0 : (size_t)M * 6;
    for (int i = 0; i < N; ++i) {
        n_reg[i] = P.W.diag ? track_gains_instance<1>(P, Xnom.data(), Unom.data(), Kt.data(), i)
                            : track_gains_instance<0>(P, Xnom.data(), Unom.data(), Kt.data(), i);
        for (int m = 0; m < M; ++m) {
            const double* d6 = delta + i * dstride + (size_t)m * 6;
            const size_t o = ((size_t)i * M + m) * 6;
            if (P.q32) track_mc_sample<true>(P, Xnom.data(), Unom.data(), Kt.data(), d6, i, err_max + o, err_final + o);
            else track_mc_sample<false>(P, Xnom.data(), Unom.data(), Kt.data(), d6, i, err_max + o, err_final + o);
        }
        const size_t o = (size_t)i * M * 6;
        const int nw = track_mc_reduce(err_max + o, err_final + o, M, tol, worst_max + (size_t)i * 6, mean_final + (size_t)i * 6);
        n_within[i] = tol ? nw : 0;
    }
}
}  // namespace

extern "C" {

// acoc_lqr_tracking_mc replayed: float state storage when every state at t >= 1 is a float32 value (float32 quantisation only), exact
// row 0 always.  delta (M,6) if delta_shared else (N,M,6), tol (6) or NULL -> err_max / err_final (N,M,6), worst_max / mean_final (N,6),
// n_within (N) (0 without tol), n_reg (N).
void emul_track_mc(int N, int M, int TT, const double* params, int state_f64, const double* Q, const double* R, const double* QT,
                   const double* xx_opt, const double* uu_opt, const double* delta, int delta_shared, const double* tol, double* err_max,
                   double* err_final, double* worst_max, double* mean_final, int* n_within, int* n_reg)
{
    bool x_float = !state_f64;
    for (size_t i = 0; i < (size_t)N * 6 && x_float; ++i)
        for (int t = 1; t < TT; ++t) { const double v = xx_opt[i * TT + t]; if (!((double)(float)v == v) && v == v) { x_float = false; break; } }
    if (x_float)
        track_mc_impl<float>(N, M, TT, params, state_f64, Q, R, QT, xx_opt, uu_opt, delta, delta_shared, tol, err_max, err_final, worst_max,
                             mean_final, n_within, n_reg);
    else
        track_mc_impl<double>(N, M, TT, params, state_f64, Q, R, QT, xx_opt, uu_opt, delta, delta_shared, tol, err_max, err_final, worst_max,
                              mean_final, n_within, n_reg);
}

}  // extern "C"
