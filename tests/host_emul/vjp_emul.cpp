// vjp_emul.cpp -- TEST-ONLY host replay of the kernels of acoc_result_vjp (derivative of the optimum).
//
// Compiled with g++ -ffp-contract=off like emul.cpp (matching nvcc -fmad=false): the per-instance functions of acoc_kernels.cuh
// (vjp_backward_instance, vjp_forward_instance) driven with plain loops over instances, on warp-tiled buffers laid out as the library lays
// them out.  Not part of the product: libacoc.so does not contain it.
#include <cmath>
#include <cstring>
#include <vector>

#include "../../aircraftoptimalcontrol_b200/csrc/acoc_kernels.cuh"

using namespace acoc;

namespace {
void to_soa(const double* host, double* dst, int n, int C, int TT, int Np)
{
    for (int i = 0; i < n; ++i)
        for (int c = 0; c < C; ++c)
            for (int t = 0; t < TT; ++t) dst[at(t, C, c, Np, i)] = host[((size_t)i * C + c) * TT + t];
}
void from_soa(const double* src, double* host, int n, int C, int TT, int Np)
{
    for (int i = 0; i < n; ++i)
        for (int c = 0; c < C; ++c)
            for (int t = 0; t < TT; ++t) host[((size_t)i * C + c) * TT + t] = src[at(t, C, c, Np, i)];
}
void fill_weights(Weights* W, const double* Q, const double* R, const double* QT)
{
    memcpy(W->Q, Q, sizeof(W->Q)); memcpy(W->R, R, sizeof(W->R)); memcpy(W->QT, QT, sizeof(W->QT));
    bool d = true;
    for (int i = 0; i < 6; ++i) for (int j = 0; j < 6; ++j) if (i != j && (Q[i * 6 + j] != 0.0 || QT[i * 6 + j] != 0.0)) d = false;
    if (R[1] != 0.0 || R[2] != 0.0) d = false;
    W->diag = d;
}
}  // namespace

extern "C" {

// xx (N,6,TT) / uu (N,2,TT): the result (uu[:, :, TT-1] is not read); references either per instance xref (N,6,TT) / uref (N,2,TT), or
// parametric (xref == NULL): tables tt, zs [TT], vs [TT] or NULL, per instance zf, vx [N], constants xc [6], uc [2] (V_t formed as
// k_gen_vref forms it).  gx (N,6,TT), gu (N,2,TT).  Outputs xref_bar (N,6,TT), uref_bar (N,2,TT), x0_bar (N,6), zf_bar / vx_bar (N, parametric
// only, else untouched), n_indef (N).
void emul_vjp(int N, int TT, const double* params, const double* Q, const double* R, const double* QT, const double* xx, const double* uu,
              const double* xref, const double* uref, const double* tt, const double* zs, const double* vs, const double* zf, const double* vx,
              const double* xc, const double* uc, const double* gx, const double* gu, double* xref_bar, double* uref_bar, double* x0_bar,
              double* zf_bar, double* vx_bar, int* n_indef)
{
    const int Np = (N + 31) / 32 * 32;
    const size_t T = TT;
    std::vector<double> X(T * 6 * Np, 0.0), U(T * 2 * Np, 0.0), x0((size_t)6 * Np, 0.0), GX(T * 6 * Np, 0.0), GU(T * 2 * Np, 0.0);
    std::vector<double> KS(T * 14 * Np, 0.0), XB(T * 6 * Np, 0.0), UB(T * 2 * Np, 0.0), xi((size_t)6 * Np, 0.0), zv((size_t)2 * Np, 0.0);
    std::vector<double> XR, UR, V, ZF((size_t)Np, 0.0), VX((size_t)Np, 0.0);
    to_soa(xx, X.data(), N, 6, TT, Np);
    to_soa(uu, U.data(), N, 2, TT, Np);
    for (int i = 0; i < N; ++i) for (int c = 0; c < 6; ++c) x0[(size_t)c * Np + i] = xx[((size_t)i * 6 + c) * TT];
    to_soa(gx, GX.data(), N, 6, TT, Np);
    to_soa(gu, GU.data(), N, 2, TT, Np);
    Problem P;
    P.M = make_model(params);
    fill_weights(&P.W, Q, R, QT);
    P.N = N; P.Np = Np; P.TT = TT; P.q32 = 0; P.ref_shared = 0; P.x0 = x0.data();
    P.xref = nullptr; P.uref = nullptr; P.ref_param = 0; P.rp_tt = P.rp_zs = P.rp_zf = P.rp_vx = P.rp_v = nullptr;
    const bool param = xref == nullptr;
    if (param) {
        P.ref_param = 1;
        P.rp_tt = tt; P.rp_zs = zs;
        for (int i = 0; i < N; ++i) { ZF[i] = zf[i]; VX[i] = vx[i]; }
        P.rp_zf = ZF.data(); P.rp_vx = VX.data();
        if (vs) {
            V.assign(T * Np, 0.0);
            for (int i = 0; i < N; ++i)
                for (int t = 0; t < TT; ++t) { const double zd = vs[t] * (zf[i] - 0.0); V[at(t, 1, 0, Np, i)] = std::sqrt(zd * zd + vx[i] * vx[i]); }
            P.rp_v = V.data();
        }
        for (int k = 0; k < 6; ++k) P.rp_xc[k] = xc[k];
        P.rp_uc[0] = uc[0]; P.rp_uc[1] = uc[1];
    } else {
        XR.assign(T * 6 * Np, 0.0); UR.assign(T * 2 * Np, 0.0);
        to_soa(xref, XR.data(), N, 6, TT, Np);
        to_soa(uref, UR.data(), N, 2, TT, Np);
        P.xref = XR.data(); P.uref = UR.data();
    }
    for (int i = 0; i < N; ++i) {
        if (P.W.diag) {
            n_indef[i] = vjp_backward_instance<1>(P, X.data(), U.data(), GX.data(), GU.data(), KS.data(), xi.data(), i);
            vjp_forward_instance<1>(P, X.data(), U.data(), KS.data(), vs, XB.data(), UB.data(), param ? zv.data() : nullptr, i);
        } else {
            n_indef[i] = vjp_backward_instance<0>(P, X.data(), U.data(), GX.data(), GU.data(), KS.data(), xi.data(), i);
            vjp_forward_instance<0>(P, X.data(), U.data(), KS.data(), vs, XB.data(), UB.data(), param ? zv.data() : nullptr, i);
        }
        for (int c = 0; c < 6; ++c) x0_bar[(size_t)i * 6 + c] = xi[(size_t)c * Np + i];
        if (param) { zf_bar[i] = zv[i]; vx_bar[i] = zv[(size_t)Np + i]; }
    }
    from_soa(XB.data(), xref_bar, N, 6, TT, Np);
    from_soa(UB.data(), uref_bar, N, 2, TT, Np);
}

}  // extern "C"
