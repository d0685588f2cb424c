// acoc_tma.cuh -- the time sweeps as warp-private TMA pipelines (sm_100a only; device code).
//
// With the warp-tiled layout (acoc_kernels.cuh, at()) everything one warp (= one tile of 32 instances) needs from an
// array at time t is ONE contiguous block: X 6*32 elements, U/DU/uref 2*32, xref 6*32, KSG 16*32.  Each warp therefore
// runs its own producer/consumer ring in shared memory: lane 0 issues one bulk asynchronous copy per array and step
// (cp.async.bulk.shared.global, completion counted in bytes on an mbarrier), S steps ahead of the arithmetic; all lanes
// wait on the step's mbarrier, read their column of the block from shared memory (conflict-free: lane-contiguous) and
// hand the stage back with a __syncwarp().  The copies are in flight while the warp computes, independent of how ptxas
// schedules the loop body, with no staging registers -- the DRAM latency that the plain-load sweeps pay once or twice
// per time step is hidden by the ring depth.  No CTA-wide barrier exists in these kernels; warps never wait on each other.
//
// The arithmetic is the same *_step() code as in the plain sweeps (acoc_kernels.cuh), so results are bit-identical;
// tests/test_gpu_parity.py runs every parity case through these kernels (they are the default) and A/B against the
// plain-load kernels (ACOC_NO_TMA).
#pragma once
#include <stdint.h>

#include "acoc_kernels.cuh"

namespace acoc {

// ---- PTX wrappers ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// one arrival + the number of bytes the bulk copies of this phase will deliver
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// plain arrival (release at CTA scope): hands a shared-memory stage from one warp to another
__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// global -> shared bulk copy (TMA, 1-D): 16-byte aligned addresses, size a multiple of 16
__device__ __forceinline__ void tma_load(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// Hand a ring stage back after every lane has read it, so that lane 0 may issue the bulk copy that refills it.
// The reads are ordinary shared-memory loads (generic proxy); the refill is written by the bulk-copy engine (async proxy).  Program
// order and bar.warp.sync order generic-proxy accesses only: without a proxy fence the refill of a stage is NOT ordered behind the
// loads that read its previous contents, even when the same thread issues both.  Round 1 shipped without the fence and passed; in
// round 2 a re-scheduled backward sweep (nothing consumed the loaded registers before the copy was issued any more) showed the hazard
// whenever several tile ranges ran concurrently on an L2-resident batch: about one tile in a thousand per sweep read the references of
// step t+3 at step t (tools/det_check.py; membar.cta alone did not help, fence.proxy.async does).
__device__ __forceinline__ void stage_release()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
}

// ---- warp-private ring ---------------------------------------------------------------------------------------
// A stage holds up to four blocks (offsets are compile-time); step k uses stage k % S with mbarrier parity (k / S) & 1.
template <int S, int STAGE_BYTES>
struct WarpRing {
    unsigned char* buf;  // S * STAGE_BYTES, 128-byte aligned
    uint64_t* bar;       // S mbarriers
    __device__ __forceinline__ void init(unsigned char* smem_base, int warp, int n_warps, int lane)
    {
        buf = smem_base + (size_t)warp * (S * STAGE_BYTES);
        bar = reinterpret_cast<uint64_t*>(smem_base + (size_t)n_warps * (S * STAGE_BYTES)) + warp * S;
        if (lane == 0) {
            for (int s = 0; s < S; ++s) mbar_init(bar + s, 1);
            mbar_fence_init();
        }
        __syncwarp();
    }
    __device__ __forceinline__ unsigned char* stage(int k) const { return buf + (k % S) * STAGE_BYTES; }
    __device__ __forceinline__ uint64_t* barrier(int k) const { return bar + (k % S); }
    __device__ __forceinline__ void wait(int k) const { mbar_wait(bar + (k % S), (uint32_t)((k / S) & 1)); }
    static constexpr size_t smem_bytes(int n_warps) { return (size_t)n_warps * (S * STAGE_BYTES + S * sizeof(uint64_t)); }
};

// tile of this warp from the (tile-granular) work list, or -1
struct TileList {
    const int* tiles;  // nullptr: identity
    const int* count;
    int off, end;      // this launch covers list entries [off, end) (a batch may be swept as two ranges on two streams)
};
__device__ __forceinline__ int warp_tile(const TileList& L, int w, int Np)
{
    const int e = L.off + w;
    if (e >= L.end) return -1;
    if (!L.tiles) return e < Np / TILE ? e : -1;
    return e < *L.count ? L.tiles[e] : -1;
}

// compacted, ORDERED list of groups of 2^shift consecutive instances that still contain work (shift = 0: a per-instance list)
struct WorkList {
    const int* groups;  // nullptr: identity (thread j -> instance j)
    const int* count;   // number of valid groups (device memory)
    int shift;
};

__device__ __forceinline__ int work_instance(const WorkList& L, int j, int N)
{
    if (!L.groups) return j < N ? j : -1;
    const int g = j >> L.shift;
    if (g >= *L.count) return -1;
    const int i = (L.groups[g] << L.shift) + (j & ((1 << L.shift) - 1));
    return i < N ? i : -1;
}

// first element of the block of tile `tile` at time t in a warp-tiled array with C components
__device__ __forceinline__ size_t tile_base(int t, int C, int Np, int tile) { return ((size_t)t * (size_t)(Np / TILE) + tile) * C * TILE; }

// How a sweep gets the references of a step (ProblemT): per-instance arrays (one block per tile and step through the ring), one shared
// trajectory (plain loads, L1-resident), or the parametric family (two multiplications from shared tables; the stored speed reference,
// if there is one, is the only block that still travels through the ring, in the place of the xref block).
template <typename F>
struct RefMode {
    bool shared, param, tiled, has_v;
    F zf, vx;   // parameters of this lane's instance (parametric mode)
    __device__ __forceinline__ RefMode(const ProblemT<F>& P, int i, bool live)
    {
        shared = P.ref_shared != 0; param = P.ref_param != 0; tiled = !shared && !param; has_v = param && P.rp_v != nullptr;
        zf = (param && live) ? P.rp_zf[i] : F(0.0);
        vx = (param && live) ? P.rp_vx[i] : F(0.0);
    }
    // references of (t, i) for the modes that do not come out of the ring stage; v = this lane's entry of the stage's V block
    __device__ __forceinline__ void fill(const ProblemT<F>& P, int t, int i, F v, F* xr, F* ur) const
    {
        if (shared) load_ref(P, t, i, xr, ur);
        else if (param) {
            param_xref(P, t, zf, vx, has_v ? v : P.rp_xc[2], xr);
            ur[0] = P.rp_uc[0]; ur[1] = P.rp_uc[1];
        }
    }
    // the same with the table entries tt_t, zs_t already in registers (the latency-bound backward sweep fetches them one step ahead)
    __device__ __forceinline__ void fill(const ProblemT<F>& P, int t, int i, F v, F tt_t, F zs_t, F* xr, F* ur) const
    {
        if (shared) load_ref(P, t, i, xr, ur);
        else if (param) {
            xr[0] = vx * tt_t; xr[1] = zs_t * zf; xr[2] = has_v ? v : P.rp_xc[2];
            xr[3] = P.rp_xc[3]; xr[4] = P.rp_xc[4]; xr[5] = P.rp_xc[5];
            ur[0] = P.rp_uc[0]; ur[1] = P.rp_uc[1];
        }
    }
};

// =================================================================================================================
// LQ forward pass + descent (forward_lq_instance): in K/sigma/g, x, u per step; out du
// =================================================================================================================
constexpr int FWD_STAGES = 2;
// Of the state only V, theta, gamma (components 2, 3, 5) enter the linearisation: the stage holds [V theta] and [gamma].
template <typename F, typename XT>
struct FwdStage {
    static constexpr int KSG_B = 16 * TILE * sizeof(F), XC_B = TILE * sizeof(XT), U_B = NI * TILE * sizeof(F);
    static constexpr int KSG_O = 0, X23_O = KSG_B, X5_O = KSG_B + 2 * XC_B, U_O = KSG_B + 3 * XC_B + (sizeof(XT) == 4 ? 128 : 0),
                         BYTES_TX = KSG_B + 3 * XC_B + U_B, BYTES = U_O + U_B;
};

template <typename F, typename XT>
__global__ void __launch_bounds__(64) k_forward_tma(ProblemT<F> P, TileList L, const XT* __restrict__ X, const F* __restrict__ U,
                                                    const F* __restrict__ KSG, F* __restrict__ DU, const int* __restrict__ status,
                                                    double* __restrict__ descent)
{
    using St = FwdStage<F, XT>;
    extern __shared__ __align__(128) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int tile = warp_tile(L, blockIdx.x * nw + warp, P.Np);
    if (tile < 0) return;  // warp-uniform
    WarpRing<FWD_STAGES, St::BYTES> ring;
    ring.init(smem, warp, nw, lane);
    const int TT = P.TT, Np = P.Np, i = tile * TILE + lane, nsteps = TT - 1;
    const bool live = i < P.N;  // padding lanes of the last tile idle (but keep the warp converged for the ring)
    auto issue = [&](int t) {   // lane 0: bulk copies of step t into its stage
        unsigned char* st = ring.stage(t);
        uint64_t* b = ring.barrier(t);
        mbar_arrive_expect_tx(b, St::BYTES_TX);
        tma_load(st + St::KSG_O, KSG + tile_base(t, 16, Np, tile), St::KSG_B, b);
        tma_load(st + St::X23_O, X + tile_base(t, NS, Np, tile) + 2 * TILE, 2 * St::XC_B, b);
        tma_load(st + St::X5_O, X + tile_base(t, NS, Np, tile) + 5 * TILE, St::XC_B, b);
        tma_load(st + St::U_O, U + tile_base(t, NI, Np, tile), St::U_B, b);
    };
    if (lane == 0)
        for (int t = 0; t < FWD_STAGES && t < nsteps; ++t) issue(t);
    F dx[NS] = {0, 0, 0, 0, 0, 0};
    double d = 0.0;
    for (int t = 0; t < nsteps; ++t) {
        ring.wait(t);
        const unsigned char* st = ring.stage(t);
        F ksg[16], x[NS], u[NI], du[NI];
        XT xraw[NS];
#pragma unroll
        for (int c = 0; c < 16; ++c) ksg[c] = reinterpret_cast<const F*>(st + St::KSG_O)[c * TILE + lane];
        xraw[0] = xraw[1] = xraw[4] = XT(0);  // X, Z, q do not enter the linearisation
        xraw[2] = reinterpret_cast<const XT*>(st + St::X23_O)[lane];
        xraw[3] = reinterpret_cast<const XT*>(st + St::X23_O)[TILE + lane];
        xraw[5] = reinterpret_cast<const XT*>(st + St::X5_O)[lane];
#pragma unroll
        for (int c = 0; c < NI; ++c) u[c] = reinterpret_cast<const F*>(st + St::U_O)[c * TILE + lane];
        stage_release();  // every lane has read the stage: it can be refilled
        if (lane == 0 && t + FWD_STAGES < nsteps) issue(t + FWD_STAGES);
        if (live) {
            finish_x(P, t, i, xraw, x);
            forward_step(P.M, x, u, ksg, dx, du, d);
            DU[at(t, NI, 0, Np, i)] = du[0];
            DU[at(t, NI, 1, Np, i)] = du[1];
        }
    }
    if (live) {
        DU[at(TT - 1, NI, 0, Np, i)] = F(0.0);  // uuout[:, TT-1] stays zero (optcon.py:694)
        DU[at(TT - 1, NI, 1, Np, i)] = F(0.0);
        if (status[i] == ST_ACTIVE) descent[i] = d;
    }
}

// =================================================================================================================
// rollouts with cost that write the new iterate (rollout_instance<true, true>): candidate 0 of the lazy Armijo search
// (MODE 0) and get_update with the per-instance step + Newton bookkeeping (MODE 1).  In: u, du, references per step.
// =================================================================================================================
constexpr int ROLL_STAGES = 3;
template <typename F>
struct RollStage {
    static constexpr int U_B = NI * TILE * sizeof(F), XR_B = NS * TILE * sizeof(F);
    static constexpr int U_O = 0, DU_O = U_B, UR_O = 2 * U_B, XR_O = 3 * U_B, BYTES = 3 * U_B + XR_B;
};

template <bool Q32, typename F, typename XT, int MODE, int DG>
__global__ void __launch_bounds__(64, 7) k_rollout_write_tma(ProblemT<F> P, TileList L, NewtonOpts O, NewtonState S, const F* __restrict__ U,
                                                          const F* __restrict__ DU, const double* __restrict__ cand_steps,
                                                          XT* __restrict__ Xn, F* __restrict__ Un, const int* __restrict__ only, int kk,
                                                          int bookkeeping)
{
    using St = RollStage<F>;
    extern __shared__ __align__(128) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int tile = warp_tile(L, blockIdx.x * nw + warp, P.Np);
    if (tile < 0) return;
    const int TT = P.TT, Np = P.Np, i = tile * TILE + lane, nsteps = TT - 1;
    const bool act = i < P.N && S.status[i] == ST_ACTIVE;
    // MODE 1: lanes whose candidate 0 was accepted keep the trajectory already in the next slot (lazy Armijo)
    const bool roll = act && !(MODE == 1 && only && !only[i]);
    double J = 0.0;
    if (__any_sync(0xffffffffu, roll)) {
        WarpRing<ROLL_STAGES, St::BYTES> ring;
        ring.init(smem, warp, nw, lane);
        const RefMode<F> rm(P, i, i < P.N);
        auto issue = [&](int t) {
            unsigned char* st = ring.stage(t);
            uint64_t* b = ring.barrier(t);
            mbar_arrive_expect_tx(b, 2 * St::U_B + (rm.tiled ? St::U_B + St::XR_B : 0) + (rm.has_v ? (uint32_t)(TILE * sizeof(F)) : 0));
            tma_load(st + St::U_O, U + tile_base(t, NI, Np, tile), St::U_B, b);
            tma_load(st + St::DU_O, DU + tile_base(t, NI, Np, tile), St::U_B, b);
            if (rm.tiled) {
                tma_load(st + St::UR_O, P.uref + tile_base(t, NI, Np, tile), St::U_B, b);
                tma_load(st + St::XR_O, P.xref + tile_base(t, NS, Np, tile), St::XR_B, b);
            } else if (rm.has_v)
                tma_load(st + St::XR_O, P.rp_v + tile_base(t, 1, Np, tile), (uint32_t)(TILE * sizeof(F)), b);
        };
        if (lane == 0)
            for (int t = 0; t < ROLL_STAGES && t < nsteps; ++t) issue(t);
        const F s = (F)(MODE == 0 ? cand_steps[0] : (act ? S.step[i] : 0.0));
        F x[NS], u[NI], xr[NS], ur[NI];
#pragma unroll
        for (int c = 0; c < NS; ++c) x[c] = (i < P.N) ? P.x0[(size_t)c * Np + i] : F(0.0);
        for (int t = 0; t < nsteps; ++t) {
            ring.wait(t);
            const unsigned char* st = ring.stage(t);
            F du[NI];
#pragma unroll
            for (int c = 0; c < NI; ++c) {
                u[c] = reinterpret_cast<const F*>(st + St::U_O)[c * TILE + lane];
                du[c] = reinterpret_cast<const F*>(st + St::DU_O)[c * TILE + lane];
            }
            F vv = F(0.0);
            if (rm.tiled) {
#pragma unroll
                for (int c = 0; c < NI; ++c) ur[c] = reinterpret_cast<const F*>(st + St::UR_O)[c * TILE + lane];
#pragma unroll
                for (int c = 0; c < NS; ++c) xr[c] = reinterpret_cast<const F*>(st + St::XR_O)[c * TILE + lane];
            } else if (rm.has_v) vv = reinterpret_cast<const F*>(st + St::XR_O)[lane];
            stage_release();
            if (lane == 0 && t + ROLL_STAGES < nsteps) issue(t + ROLL_STAGES);
            if (roll) {
                rm.fill(P, t, i, vv, xr, ur);
#pragma unroll
                for (int c = 0; c < NI; ++c) u[c] = u[c] + s * du[c];  // optcon.py:197 / :253
                store_x(Xn, t, Np, i, x);
#pragma unroll
                for (int c = 0; c < NI; ++c) Un[at(t, NI, c, Np, i)] = u[c];
                rollout_step<true, Q32, DG>(P.M, P.W, x, u, xr, ur, J);
            }
        }
        if (roll) {
            store_x(Xn, TT - 1, Np, i, x);
            Un[at(TT - 1, NI, 0, Np, i)] = F(0.0);  // uu_temp[:, TT-1] is never written (optcon.py:193)
            Un[at(TT - 1, NI, 1, Np, i)] = F(0.0);
            load_xref(P, TT - 1, i, xr);
            F dx[NS];
#pragma unroll
            for (int c = 0; c < NS; ++c) dx[c] = x[c] - xr[c];
            J += (double)term_cost<DG>(P.W, dx);
        }
    }
    if (!act) return;
    if (MODE == 0) {
        S.Jcand[i] = J;
    } else {
        const double Jn = roll ? J : S.Jcand[i];
        if (bookkeeping) newton_finish_instance(O, S, Jn, kk, i);
        else { S.Jcur[i] = Jn; S.iters[i] = kk + 1; }
    }
}

// =================================================================================================================
// LQ forward pass + candidate 0 of the lazy Armijo search in ONE sweep (k_forward_tma followed by k_rollout_write_tma<.,0>):
// both walk forward in time and the rollout needs du_t only at step t, so du never makes the round trip through HBM before
// its first use and u_t is fetched once.  In: K/sigma/g, (V,theta,gamma), u, references per step; out: du, the tentative next
// iterate, descent and the cost of candidate 0.  Same per-step functions in the same order: bit-identical to the two sweeps.
// =================================================================================================================
constexpr int FC_STAGES = 2;
template <typename F, typename XT>
struct FwdCandStage {
    using Fw = FwdStage<F, XT>;
    static constexpr int U_B = Fw::U_B, XR_B = NS * TILE * sizeof(F);
    static constexpr int KSG_O = Fw::KSG_O, X23_O = Fw::X23_O, X5_O = Fw::X5_O, U_O = Fw::U_O, UR_O = Fw::U_O + U_B, XR_O = UR_O + U_B,
                         BYTES = XR_O + XR_B;
};

template <bool Q32, typename F, typename XT, int DG>
__global__ void __launch_bounds__(64, 7) k_forward_cand0_tma(ProblemT<F> P, TileList L, NewtonState S, const XT* __restrict__ X,
                                                              const F* __restrict__ U, const F* __restrict__ KSG, F* __restrict__ DU,
                                                              const double* __restrict__ cand_steps, XT* __restrict__ Xn, F* __restrict__ Un)
{
    using St = FwdCandStage<F, XT>;
    using Fw = FwdStage<F, XT>;
    extern __shared__ __align__(128) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int tile = warp_tile(L, blockIdx.x * nw + warp, P.Np);
    if (tile < 0) return;  // warp-uniform
    WarpRing<FC_STAGES, St::BYTES> ring;
    ring.init(smem, warp, nw, lane);
    const int TT = P.TT, Np = P.Np, i = tile * TILE + lane, nsteps = TT - 1;
    const bool live = i < P.N;                          // the forward pass runs for finished lanes of a live tile too (whole du lines)
    const bool act = live && S.status[i] == ST_ACTIVE;  // the rollout only for instances that are still iterating
    const RefMode<F> rm(P, i, live);
    auto issue = [&](int t) {
        unsigned char* st = ring.stage(t);
        uint64_t* b = ring.barrier(t);
        mbar_arrive_expect_tx(b, Fw::BYTES_TX + (rm.tiled ? St::U_B + St::XR_B : 0) + (rm.has_v ? (uint32_t)(TILE * sizeof(F)) : 0));
        tma_load(st + St::KSG_O, KSG + tile_base(t, 16, Np, tile), Fw::KSG_B, b);
        tma_load(st + St::X23_O, X + tile_base(t, NS, Np, tile) + 2 * TILE, 2 * Fw::XC_B, b);
        tma_load(st + St::X5_O, X + tile_base(t, NS, Np, tile) + 5 * TILE, Fw::XC_B, b);
        tma_load(st + St::U_O, U + tile_base(t, NI, Np, tile), St::U_B, b);
        if (rm.tiled) {
            tma_load(st + St::UR_O, P.uref + tile_base(t, NI, Np, tile), St::U_B, b);
            tma_load(st + St::XR_O, P.xref + tile_base(t, NS, Np, tile), St::XR_B, b);
        } else if (rm.has_v)
            tma_load(st + St::XR_O, P.rp_v + tile_base(t, 1, Np, tile), (uint32_t)(TILE * sizeof(F)), b);
    };
    if (lane == 0)
        for (int t = 0; t < FC_STAGES && t < nsteps; ++t) issue(t);
    const F s = (F)cand_steps[0];
    F dx[NS] = {0, 0, 0, 0, 0, 0}, xc[NS];  // LQ state increment; state of the candidate rollout
    double d = 0.0, J = 0.0;
#pragma unroll
    for (int c = 0; c < NS; ++c) xc[c] = live ? P.x0[(size_t)c * Np + i] : F(0.0);
    for (int t = 0; t < nsteps; ++t) {
        ring.wait(t);
        const unsigned char* st = ring.stage(t);
        F ksg[16], u[NI], xr[NS], ur[NI];
        XT xraw[NS];
#pragma unroll
        for (int c = 0; c < 16; ++c) ksg[c] = reinterpret_cast<const F*>(st + St::KSG_O)[c * TILE + lane];
        xraw[0] = xraw[1] = xraw[4] = XT(0);  // X, Z, q do not enter the linearisation
        xraw[2] = reinterpret_cast<const XT*>(st + St::X23_O)[lane];
        xraw[3] = reinterpret_cast<const XT*>(st + St::X23_O)[TILE + lane];
        xraw[5] = reinterpret_cast<const XT*>(st + St::X5_O)[lane];
#pragma unroll
        for (int c = 0; c < NI; ++c) u[c] = reinterpret_cast<const F*>(st + St::U_O)[c * TILE + lane];
        F vv = F(0.0);
        if (rm.tiled) {
#pragma unroll
            for (int c = 0; c < NI; ++c) ur[c] = reinterpret_cast<const F*>(st + St::UR_O)[c * TILE + lane];
#pragma unroll
            for (int c = 0; c < NS; ++c) xr[c] = reinterpret_cast<const F*>(st + St::XR_O)[c * TILE + lane];
        } else if (rm.has_v) vv = reinterpret_cast<const F*>(st + St::XR_O)[lane];
        stage_release();  // every lane has read the stage: it can be refilled
        if (lane == 0 && t + FC_STAGES < nsteps) issue(t + FC_STAGES);
        if (live) {
            F du[NI], xnom[NS];
            forward_du(ksg, dx, du, d);
            DU[at(t, NI, 0, Np, i)] = du[0];
            DU[at(t, NI, 1, Np, i)] = du[1];
            finish_x(P, t, i, xraw, xnom);
            forward_advance(P.M, xnom, u, du, dx);
            if (act) {
                rm.fill(P, t, i, vv, xr, ur);
                F uc[NI];
#pragma unroll
                for (int c = 0; c < NI; ++c) uc[c] = u[c] + s * du[c];  // optcon.py:197 / :253
                store_x(Xn, t, Np, i, xc);
#pragma unroll
                for (int c = 0; c < NI; ++c) Un[at(t, NI, c, Np, i)] = uc[c];
                rollout_step<true, Q32, DG>(P.M, P.W, xc, uc, xr, ur, J);
            }
        }
    }
    if (!live) return;
    DU[at(TT - 1, NI, 0, Np, i)] = F(0.0);  // uuout[:, TT-1] stays zero (optcon.py:694)
    DU[at(TT - 1, NI, 1, Np, i)] = F(0.0);
    if (!act) return;
    S.descent[i] = d;
    store_x(Xn, TT - 1, Np, i, xc);
    Un[at(TT - 1, NI, 0, Np, i)] = F(0.0);  // uu_temp[:, TT-1] is never written (optcon.py:193)
    Un[at(TT - 1, NI, 1, Np, i)] = F(0.0);
    F xrT[NS], dxT[NS];
    load_xref(P, TT - 1, i, xrT);
#pragma unroll
    for (int c = 0; c < NS; ++c) dxT[c] = xc[c] - xrT[c];
    J += (double)term_cost<DG>(P.W, dxT);
    S.Jcand[i] = J;
}

// =================================================================================================================
// fused backward sweep (backward_instance): in x, u, references per step (walking t = TT-2 .. 0); out K/sigma/g
// =================================================================================================================
constexpr int BWD_STAGES = 3;
template <typename F, typename XT>
struct BwdStage {
    static constexpr int X_B = NS * TILE * sizeof(XT), U_B = NI * TILE * sizeof(F), XR_B = NS * TILE * sizeof(F);
    static constexpr int U_O = 0, UR_O = U_B, XR_O = 2 * U_B, X_O = 2 * U_B + XR_B, BYTES = 2 * U_B + XR_B + X_B;
};

template <bool EXACT, typename F, typename XT, int DG>
__global__ void __launch_bounds__(64) k_backward_tma(ProblemT<F> P, TileList L, const XT* __restrict__ X, const F* __restrict__ U,
                                                     F* __restrict__ KSG, const int* __restrict__ status, int* __restrict__ n_reg)
{
    using St = BwdStage<F, XT>;
    extern __shared__ __align__(128) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int tile = warp_tile(L, blockIdx.x * nw + warp, P.Np);
    if (tile < 0) return;
    WarpRing<BWD_STAGES, St::BYTES> ring;
    ring.init(smem, warp, nw, lane);
    const int TT = P.TT, Np = P.Np, i = tile * TILE + lane, nsteps = TT - 1;
    const bool live = i < P.N;
    const RefMode<F> rm(P, i, live);
    // ring step k <-> time t = TT-2-k
    auto issue = [&](int k) {
        const int t = TT - 2 - k;
        unsigned char* st = ring.stage(k);
        uint64_t* b = ring.barrier(k);
        mbar_arrive_expect_tx(b, St::U_B + St::X_B + (rm.tiled ? St::U_B + St::XR_B : 0) + (rm.has_v ? (uint32_t)(TILE * sizeof(F)) : 0));
        tma_load(st + St::U_O, U + tile_base(t, NI, Np, tile), St::U_B, b);
        tma_load(st + St::X_O, X + tile_base(t, NS, Np, tile), St::X_B, b);
        if (rm.tiled) {
            tma_load(st + St::UR_O, P.uref + tile_base(t, NI, Np, tile), St::U_B, b);
            tma_load(st + St::XR_O, P.xref + tile_base(t, NS, Np, tile), St::XR_B, b);
        } else if (rm.has_v)
            tma_load(st + St::XR_O, P.rp_v + tile_base(t, 1, Np, tile), (uint32_t)(TILE * sizeof(F)), b);
    };
    if (lane == 0)
        for (int k = 0; k < BWD_STAGES && k < nsteps; ++k) issue(k);
    F Pm[21], p[NS], lam[NS], x[NS], u[NI], xr[NS], ur[NI];
    int nreg = 0;
    if (live) {
        load_xref(P, TT - 1, i, xr);
        load_x(P, X, TT - 1, i, x);
        backward_terminal<DG>(P.W, x, xr, Pm, p, lam);
    }
    F tt_n = F(0.0), zs_n = F(0.0);  // parametric references: table entries of the next step, fetched one step ahead
    if (rm.param) { tt_n = P.rp_tt[TT - 2]; zs_n = P.rp_zs[TT - 2]; }
    for (int k = 0; k < nsteps; ++k) {
        const int t = TT - 2 - k;
        const F tt_c = tt_n, zs_c = zs_n;
        if (rm.param && t > 0) { tt_n = P.rp_tt[t - 1]; zs_n = P.rp_zs[t - 1]; }
        ring.wait(k);
        const unsigned char* st = ring.stage(k);
        XT xraw[NS];
#pragma unroll
        for (int c = 0; c < NS; ++c) xraw[c] = reinterpret_cast<const XT*>(st + St::X_O)[c * TILE + lane];
#pragma unroll
        for (int c = 0; c < NI; ++c) u[c] = reinterpret_cast<const F*>(st + St::U_O)[c * TILE + lane];
        F vv = F(0.0);
        if (rm.tiled) {
#pragma unroll
            for (int c = 0; c < NI; ++c) ur[c] = reinterpret_cast<const F*>(st + St::UR_O)[c * TILE + lane];
#pragma unroll
            for (int c = 0; c < NS; ++c) xr[c] = reinterpret_cast<const F*>(st + St::XR_O)[c * TILE + lane];
        } else if (rm.has_v) vv = reinterpret_cast<const F*>(st + St::XR_O)[lane];
        stage_release();
        if (lane == 0 && k + BWD_STAGES < nsteps) issue(k + BWD_STAGES);
        if (live) {
            rm.fill(P, t, i, vv, tt_c, zs_c, xr, ur);
            finish_x(P, t, i, xraw, x);
            F K[2 * NS], sig[NI], g[NI];
            nreg += backward_step<EXACT, DG>(P.M, P.W, x, u, xr, ur, Pm, p, lam, K, sig, g);
            F* out = KSG + tile_base(t, 16, Np, tile) + lane;
#pragma unroll
            for (int c = 0; c < 12; ++c) out[c * TILE] = K[c];
            out[12 * TILE] = sig[0]; out[13 * TILE] = sig[1];
            out[14 * TILE] = g[0];   out[15 * TILE] = g[1];
        }
    }
    if (live && nreg && status[i] == ST_ACTIVE) n_reg[i] += nreg;
}

// =================================================================================================================
// fused backward sweep of SMALL batches, warp-specialised: one CTA = one tile of 32 instances = two warps with one role each.
//   warp 0 (COSTATE): TMA ring of x, u, references (as in k_backward_tma) -> dx, lx, lu, trigonometry, linearisation, lambda-contracted
//                     Hessians, g_t, lambda_t.  Hands the linearisation (12 numbers), lx (6), lu (2) and the Hessian terms (7) of the
//                     step to warp 1 through a shared-memory message ring, writes g_t.
//   warp 1 (MATRIX):  carries P, p; G, m, the column sweep P A / A'PA / B'PA, gains, P_t, p_t.  Writes K_t, sigma_t.
// The two halves of a step share nothing but that message (riccati_costate / riccati_matrix), so warp 0 runs ahead of warp 1 by the
// depth of the message ring and the chain of dependent instructions per step -- which is all a batch of a few thousand instances
// pays for: a lone warp needs ~1.45 us per step -- is cut to the matrix half.  The matrix half needs ~230 registers, so only four
// tiles fit on an SM: the kernel is used when the whole batch is resident at once (late survivor generations, single trajectories);
// big batches keep k_backward_tma, where eight tiles per SM matter more (4.0 vs 3.2 ms at 65,536 instances).  Arithmetic per entry is
// unchanged: bit-identical results (ACOC_NO_BWD_SPLIT for A/B).
// =================================================================================================================
#ifndef ACOC_BS_XSTAGES
#define ACOC_BS_XSTAGES 2
#endif

constexpr int BS_XSTAGES = ACOC_BS_XSTAGES;
template <bool EXACT>
struct BsMsg { static constexpr int N = 12 + NS + NI + (EXACT ? 7 : 0); };
template <bool EXACT, typename F, typename XT>
constexpr size_t backward_split_smem()
{
    return (size_t)BWD_STAGES * BwdStage<F, XT>::BYTES + (size_t)BS_XSTAGES * BsMsg<EXACT>::N * TILE * sizeof(F) +
           (BWD_STAGES + 2 * BS_XSTAGES) * sizeof(uint64_t);
}

// The COSTATE role of the warp-specialised backward sweeps (one warp per tile): TMA ring of x, u, references -> dx, lx, lu, trigonometry,
// linearisation, lambda-contracted Hessians; hands the step's message (BsMsg) to the consumer warp(s) through the XS-deep message ring
// (xfull: one arrival by this warp; xempty: one arrival per consumer warp), then g_t, lambda_t.
template <bool EXACT, typename F, typename XT, int DG, int XS>
__device__ __forceinline__ void bs_costate_role(const ProblemT<F>& P, int tile, int lane, bool live, F* x, F* xr, unsigned char* ring, F* msg,
                                                uint64_t* bar_in, uint64_t* xfull, uint64_t* xempty, const XT* __restrict__ X,
                                                const F* __restrict__ U, F* __restrict__ KSG)
{
    using St = BwdStage<F, XT>;
    constexpr int NMSG = BsMsg<EXACT>::N;
    const int TT = P.TT, Np = P.Np, i = tile * TILE + lane, nsteps = TT - 1;
    const RefMode<F> rm(P, i, live);
    auto issue = [&](int k) {  // ring step k <-> time t = TT-2-k
        const int t = TT - 2 - k;
        unsigned char* st = ring + (k % BWD_STAGES) * St::BYTES;
        uint64_t* b = bar_in + (k % BWD_STAGES);
        mbar_arrive_expect_tx(b, St::U_B + St::X_B + (rm.tiled ? St::U_B + St::XR_B : 0) + (rm.has_v ? (uint32_t)(TILE * sizeof(F)) : 0));
        tma_load(st + St::U_O, U + tile_base(t, NI, Np, tile), St::U_B, b);
        tma_load(st + St::X_O, X + tile_base(t, NS, Np, tile), St::X_B, b);
        if (rm.tiled) {
            tma_load(st + St::UR_O, P.uref + tile_base(t, NI, Np, tile), St::U_B, b);
            tma_load(st + St::XR_O, P.xref + tile_base(t, NS, Np, tile), St::XR_B, b);
        } else if (rm.has_v)
            tma_load(st + St::XR_O, P.rp_v + tile_base(t, 1, Np, tile), (uint32_t)(TILE * sizeof(F)), b);
    };
    if (lane == 0)
        for (int k = 0; k < BWD_STAGES && k < nsteps; ++k) issue(k);
    F lam[NS], u[NI], ur[NI];
    if (live) {
        F dxT[NS];
#pragma unroll
        for (int c = 0; c < NS; ++c) dxT[c] = x[c] - xr[c];
        wmul6(P.W.QT, (int)weights_diag<DG>(P.W), dxT, lam);  // lam_{T-1} = QT dx (optcon.py:429-432)
    }
    for (int k = 0; k < nsteps; ++k) {
        const int t = TT - 2 - k;
        mbar_wait(bar_in + (k % BWD_STAGES), (uint32_t)((k / BWD_STAGES) & 1));
        const unsigned char* st = ring + (k % BWD_STAGES) * St::BYTES;
        XT xraw[NS];
#pragma unroll
        for (int c = 0; c < NS; ++c) xraw[c] = reinterpret_cast<const XT*>(st + St::X_O)[c * TILE + lane];
#pragma unroll
        for (int c = 0; c < NI; ++c) u[c] = reinterpret_cast<const F*>(st + St::U_O)[c * TILE + lane];
        F vv = F(0.0);
        if (rm.tiled) {
#pragma unroll
            for (int c = 0; c < NI; ++c) ur[c] = reinterpret_cast<const F*>(st + St::UR_O)[c * TILE + lane];
#pragma unroll
            for (int c = 0; c < NS; ++c) xr[c] = reinterpret_cast<const F*>(st + St::XR_O)[c * TILE + lane];
        } else if (rm.has_v) vv = reinterpret_cast<const F*>(st + St::XR_O)[lane];
        stage_release();
        if (lane == 0 && k + BWD_STAGES < nsteps) issue(k + BWD_STAGES);
        const int s = k % XS;
        F* const m = msg + (size_t)s * NMSG * TILE + lane;
        F q[NS], r[NI];
        Lin<F> l;
        if (live) {
            rm.fill(P, t, i, vv, xr, ur);
            finish_x(P, t, i, xraw, x);
            F dx[NS], du[NI];
#pragma unroll
            for (int c = 0; c < NS; ++c) dx[c] = x[c] - xr[c];
#pragma unroll
            for (int c = 0; c < NI; ++c) du[c] = u[c] - ur[c];
            wmul6(P.W.Q, (int)weights_diag<DG>(P.W), dx, q);   // lx = Q dx   (aircraft_simplified.py:63)
            wmul2(P.W.R, (int)weights_diag<DG>(P.W), du, r);   // lu = R du   (:64)
            const Trig<F> tg = make_trig(x);
            l = linearize(P.M, x, u, tg);
            Hess<F> h;
            if (EXACT) h = hess_contract(P.M, x, u, tg, l, lam);
            if (k >= XS) mbar_wait(xempty + s, (uint32_t)((k / XS - 1) & 1));
            m[0 * TILE] = l.a02; m[1 * TILE] = l.a05; m[2 * TILE] = l.a12; m[3 * TILE] = l.a15; m[4 * TILE] = l.a22; m[5 * TILE] = l.a23;
            m[6 * TILE] = l.a25; m[7 * TILE] = l.a52; m[8 * TILE] = l.a53; m[9 * TILE] = l.a55; m[10 * TILE] = l.b20; m[11 * TILE] = l.b50;
#pragma unroll
            for (int c = 0; c < NS; ++c) m[(12 + c) * TILE] = q[c];
            m[18 * TILE] = r[0]; m[19 * TILE] = r[1];
            if (EXACT) {
                m[20 * TILE] = h.h22; m[21 * TILE] = h.h23; m[22 * TILE] = h.h25; m[23 * TILE] = h.h33; m[24 * TILE] = h.h55;
                m[25 * TILE] = h.s2; m[26 * TILE] = h.s3;
            }
        } else if (k >= XS) mbar_wait(xempty + s, (uint32_t)((k / XS - 1) & 1));
        __syncwarp();
        if (lane == 0) mbar_arrive(xfull + s);
        if (live) {
            F g[NI];
            riccati_costate(P.M, l, q, r, lam, g);
            F* out = KSG + tile_base(t, 16, Np, tile) + lane;
            out[14 * TILE] = g[0]; out[15 * TILE] = g[1];
        }
    }
}

template <bool EXACT, typename F, typename XT, int DG>
__global__ void __launch_bounds__(64, 4) k_backward_split(ProblemT<F> P, TileList L, const XT* __restrict__ X, const F* __restrict__ U,
                                                          F* __restrict__ KSG, const int* __restrict__ status, int* __restrict__ n_reg)
{
    using St = BwdStage<F, XT>;
    constexpr int NMSG = BsMsg<EXACT>::N;
    extern __shared__ __align__(128) unsigned char smem[];
    const int lane = threadIdx.x & 31, role = threadIdx.x >> 5;
    const int tile = warp_tile(L, blockIdx.x, P.Np);
    if (tile < 0) return;  // (uniform over the CTA)
    unsigned char* const ring = smem;
    F* const msg = reinterpret_cast<F*>(smem + (size_t)BWD_STAGES * St::BYTES);
    uint64_t* const bar_in = reinterpret_cast<uint64_t*>(smem + (size_t)BWD_STAGES * St::BYTES + (size_t)BS_XSTAGES * NMSG * TILE * sizeof(F));
    uint64_t* const xfull = bar_in + BWD_STAGES;
    uint64_t* const xempty = xfull + BS_XSTAGES;
    if (threadIdx.x == 0) {
        for (int s = 0; s < BWD_STAGES; ++s) mbar_init(bar_in + s, 1);
        for (int s = 0; s < BS_XSTAGES; ++s) { mbar_init(xfull + s, 1); mbar_init(xempty + s, 1); }
        mbar_fence_init();
    }
    __syncthreads();
    const int TT = P.TT, Np = P.Np, i = tile * TILE + lane, nsteps = TT - 1;
    const bool live = i < P.N;
    F x[NS], xr[NS];
    if (live) {  // terminal condition: both roles need x_{T-1} - xref_{T-1}
        load_xref(P, TT - 1, i, xr);
        load_x(P, X, TT - 1, i, x);
    }
    if (role == 0) {
        bs_costate_role<EXACT, F, XT, DG, BS_XSTAGES>(P, tile, lane, live, x, xr, ring, msg, bar_in, xfull, xempty, X, U, KSG);
        return;
    }
    // ---------------------------------------------------------------- matrix warp
    F Pm[21], p[NS];
    int nreg = 0;
    if (live) {
        F lamT[NS];
        backward_terminal<DG>(P.W, x, xr, Pm, p, lamT);  // P_{T-1} = QT, p_{T-1} = lam_{T-1}/2 (optcon.py:688-690, :716)
    }
    for (int k = 0; k < nsteps; ++k) {
        const int t = TT - 2 - k, s = k % BS_XSTAGES;
        mbar_wait(xfull + s, (uint32_t)((k / BS_XSTAGES) & 1));
        const F* const m = msg + (size_t)s * NMSG * TILE + lane;
        Lin<F> l;
        Hess<F> h;
        F q[NS], r[NI];
        if (live) {
            l.a02 = m[0 * TILE]; l.a05 = m[1 * TILE]; l.a12 = m[2 * TILE]; l.a15 = m[3 * TILE]; l.a22 = m[4 * TILE]; l.a23 = m[5 * TILE];
            l.a25 = m[6 * TILE]; l.a52 = m[7 * TILE]; l.a53 = m[8 * TILE]; l.a55 = m[9 * TILE]; l.b20 = m[10 * TILE]; l.b50 = m[11 * TILE];
#pragma unroll
            for (int c = 0; c < NS; ++c) q[c] = m[(12 + c) * TILE];
            r[0] = m[18 * TILE]; r[1] = m[19 * TILE];
            if (EXACT) {
                h.h22 = m[20 * TILE]; h.h23 = m[21 * TILE]; h.h25 = m[22 * TILE]; h.h33 = m[23 * TILE]; h.h55 = m[24 * TILE];
                h.s2 = m[25 * TILE]; h.s3 = m[26 * TILE];
                h.h35 = -h.h33; h.s5 = -h.s3;  // (as hess_contract forms them)
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(xempty + s);
        if (live) {
            F K[2 * NS], sig[NI];
            nreg += riccati_matrix<EXACT, DG, F>(P.M, P.W, l, h, q, r, Pm, p, K, sig);
            F* out = KSG + tile_base(t, 16, Np, tile) + lane;
#pragma unroll
            for (int c = 0; c < 12; ++c) out[c * TILE] = K[c];
            out[12 * TILE] = sig[0]; out[13 * TILE] = sig[1];
        }
    }
    if (live && nreg && status[i] == ST_ACTIVE) n_reg[i] += nreg;
}

// =================================================================================================================
// fused backward sweep of SMALL batches as a pipeline of warp roles: one CTA = one tile of 32 instances = BC_NPRE + 3 + NS = 12 warps.
// A lone warp pays ~4-6 cycles per instruction of a backward step whatever it does (dependent FP64 chains, in-order issue), so what a
// latency-bound batch pays per step is the instruction count of the LONGEST role.  The step is cut along its true recurrences:
//   PRE warps (BC_NPRE of them; warp w takes the steps k = w mod BC_NPRE -- nothing here depends on another step): own TMA ring of
//       x, u, references -> dx, lx, lu, trigonometry, linearisation, and the costate-independent part of the Hessian terms (hess_pre).
//       Message A per step: linearisation (12), lx (6), lu (2), hess_pre (16).
//   LAMBDA warp: the costate recurrence lam_t = A'lam_{t+1} + lx and g_t, and the fused multiply-adds of the Hessian terms with
//       lam_{t+1} (hess_post).  Message B per step: the 7 Hessian terms the matrix half needs.
//   GAIN warp:   G = R + B'PB, m, G^-1, y = G^-1 m (riccati_gain_core) -- what the recurrence needs of the 2x2 block.
//   OUT warp:    the outputs K_t, sigma_t: eigenvalue test on G, regularised inverse (riccati_gain_test), -(MM^-1) Mx (riccati_gain_out).
//       Nothing depends on it, so it works on step k from double-buffered copies of Mx and the gain block while the others run step k+1.
//   COLUMN warps j = 0..5: the matrix half cut along the columns of the sweep (riccati_col_sweep / riccati_col_finish): W = P A e_j,
//       N(i<=j, j), Mx(:,j); after ONE exchange of Mx and G^-1 through shared memory (named barrier of the GAIN, OUT and COLUMN warps)
//       Y(:,j) and P_t(i<=j, j); the new column goes back into the shared P (second barrier).  Column 0, the lightest, also carries
//       the affine term (A'p before the exchange, p_t after it).
// Messages travel through shared-memory rings with full/empty mbarriers (the producer's lane 0 arrives on "full" after a __syncwarp,
// every consumer warp's lane 0 on "empty"), P / p / Mx / the gain block through plain shared arrays ordered by the two named barriers.
// The sweep executes more instructions than k_backward_tma and holds 12 warps per tile, so it is used only while every tile has an SM
// of its own (late survivor generations, single trajectories).  Every number is formed by the same expression as in the one-thread
// sweep: bit-identical results (ACOC_NO_BWD_COLS for A/B; the host replay checks the decomposition,
// tests/test_kernel_math_host.py::test_riccati_by_columns_bit_identical; every small-batch parity test on the GPU runs through it).
// =================================================================================================================
#ifndef ACOC_BC_NPRE
#define ACOC_BC_NPRE 3
#endif
constexpr int BC_NPRE = ACOC_BC_NPRE;
constexpr int BC_XA = 2 * BC_NPRE;  // slots of message ring A (a PRE warp owns the slots w, w + BC_NPRE)
constexpr int BC_XB = 4;            // slots of message ring B
constexpr int BC_WARPS = BC_NPRE + 3 + NS;
constexpr int BC_THREADS = BC_WARPS * TILE;
constexpr int BC_SYNC1_THREADS = (2 + NS) * TILE;  // barrier 1: GAIN, OUT and the COLUMN warps
constexpr int BC_SYNC2_THREADS = (1 + NS) * TILE;  // barrier 2: GAIN and the COLUMN warps
constexpr int BC_PB = 21 + NS;  // shared P (21 entries of the upper triangle) and p (6)
constexpr int BC_GB = 10;       // gain block: gi00 gi01 gi11 y0 y1 | G00 G01 G11 m0 m1 (the second half for the OUT warp)
constexpr int BC_MSGB = 7;      // h22 h23 h25 h33 h55 s2 s3
template <bool EXACT>
struct BcMsgA { static constexpr int N = 12 + NS + NI + (EXACT ? 16 : 0); };
template <bool EXACT, typename F, typename XT>
constexpr size_t backward_cols_smem()
{
    return (size_t)BC_NPRE * BWD_STAGES * BwdStage<F, XT>::BYTES +
           ((size_t)BC_XA * BcMsgA<EXACT>::N + (size_t)BC_XB * BC_MSGB + BC_PB + 2 * (2 * NS + BC_GB)) * TILE * sizeof(F) +
           (BC_NPRE * BWD_STAGES + 2 * BC_XA + 2 * BC_XB) * sizeof(uint64_t);
}
// named barriers of the matrix-half warps (barrier 0 is __syncthreads)
__device__ __forceinline__ void bc_bar1() { asm volatile("bar.sync 1, %0;" ::"n"(BC_SYNC1_THREADS) : "memory"); }
__device__ __forceinline__ void bc_bar2() { asm volatile("bar.sync 2, %0;" ::"n"(BC_SYNC2_THREADS) : "memory"); }

template <typename F>
struct BcShared {
    F *msgA, *msgB, *PB, *MX, *GB;
    uint64_t *afull, *aempty, *bfull, *bempty;
};

// ring position without a division per step: slot and phase parity of message-ring use number k
struct BcSlot {
    int s;
    uint32_t par;
    __device__ __forceinline__ BcSlot() : s(0), par(0) {}
    template <int N>
    __device__ __forceinline__ void next() { if (++s == N) { s = 0; par ^= 1u; } }
};

// ---- PRE warp w: steps k = w, w + BC_NPRE, ...
template <bool EXACT, typename F, typename XT, int DG>
__device__ __forceinline__ void bc_pre_role(const ProblemT<F>& P, int tile, int lane, bool live, int w, unsigned char* ring, uint64_t* bar_in,
                                            const BcShared<F>& sh, const XT* __restrict__ X, const F* __restrict__ U)
{
    using St = BwdStage<F, XT>;
    constexpr int NA = BcMsgA<EXACT>::N;
    const int TT = P.TT, Np = P.Np, i = tile * TILE + lane, nsteps = TT - 1;
    const int nmine = nsteps > w ? (nsteps - w + BC_NPRE - 1) / BC_NPRE : 0;
    const RefMode<F> rm(P, i, live);
    auto issue = [&](int j) {  // own step j <-> ring step k = w + j*BC_NPRE <-> time t = TT-2-k
        const int t = TT - 2 - (w + j * BC_NPRE);
        unsigned char* st = ring + (j % BWD_STAGES) * St::BYTES;
        uint64_t* b = bar_in + (j % BWD_STAGES);
        mbar_arrive_expect_tx(b, St::U_B + St::X_B + (rm.tiled ? St::U_B + St::XR_B : 0) + (rm.has_v ? (uint32_t)(TILE * sizeof(F)) : 0));
        tma_load(st + St::U_O, U + tile_base(t, NI, Np, tile), St::U_B, b);
        tma_load(st + St::X_O, X + tile_base(t, NS, Np, tile), St::X_B, b);
        if (rm.tiled) {
            tma_load(st + St::UR_O, P.uref + tile_base(t, NI, Np, tile), St::U_B, b);
            tma_load(st + St::XR_O, P.xref + tile_base(t, NS, Np, tile), St::XR_B, b);
        } else if (rm.has_v)
            tma_load(st + St::XR_O, P.rp_v + tile_base(t, 1, Np, tile), (uint32_t)(TILE * sizeof(F)), b);
    };
    if (lane == 0)
        for (int j = 0; j < BWD_STAGES && j < nmine; ++j) issue(j);
    F x[NS], xr[NS], u[NI], ur[NI];
    for (int j = 0; j < nmine; ++j) {
        const int k = w + j * BC_NPRE, t = TT - 2 - k;
        mbar_wait(bar_in + (j % BWD_STAGES), (uint32_t)((j / BWD_STAGES) & 1));
        const unsigned char* st = ring + (j % BWD_STAGES) * St::BYTES;
        XT xraw[NS];
#pragma unroll
        for (int c = 0; c < NS; ++c) xraw[c] = reinterpret_cast<const XT*>(st + St::X_O)[c * TILE + lane];
#pragma unroll
        for (int c = 0; c < NI; ++c) u[c] = reinterpret_cast<const F*>(st + St::U_O)[c * TILE + lane];
        F vv = F(0.0);
        if (rm.tiled) {
#pragma unroll
            for (int c = 0; c < NI; ++c) ur[c] = reinterpret_cast<const F*>(st + St::UR_O)[c * TILE + lane];
#pragma unroll
            for (int c = 0; c < NS; ++c) xr[c] = reinterpret_cast<const F*>(st + St::XR_O)[c * TILE + lane];
        } else if (rm.has_v) vv = reinterpret_cast<const F*>(st + St::XR_O)[lane];
        stage_release();
        if (lane == 0 && j + BWD_STAGES < nmine) issue(j + BWD_STAGES);
        const int s = k % BC_XA;   // (= w or w + BC_NPRE, alternating)
        F* const m = sh.msgA + (size_t)s * NA * TILE + lane;
        if (live) {
            rm.fill(P, t, i, vv, xr, ur);
            finish_x(P, t, i, xraw, x);
            F dx[NS], du[NI], q[NS], r[NI];
#pragma unroll
            for (int c = 0; c < NS; ++c) dx[c] = x[c] - xr[c];
#pragma unroll
            for (int c = 0; c < NI; ++c) du[c] = u[c] - ur[c];
            wmul6(P.W.Q, (int)weights_diag<DG>(P.W), dx, q);   // lx = Q dx   (aircraft_simplified.py:63)
            wmul2(P.W.R, (int)weights_diag<DG>(P.W), du, r);   // lu = R du   (:64)
            const Trig<F> tg = make_trig(x);
            const Lin<F> l = linearize(P.M, x, u, tg);
            HessPre<F> a;
            if (EXACT) a = hess_pre(P.M, x, tg, l);
            if (k >= BC_XA) mbar_wait(sh.aempty + s, (uint32_t)((k / BC_XA - 1) & 1));
            m[0 * TILE] = l.a02; m[1 * TILE] = l.a05; m[2 * TILE] = l.a12; m[3 * TILE] = l.a15; m[4 * TILE] = l.a22; m[5 * TILE] = l.a23;
            m[6 * TILE] = l.a25; m[7 * TILE] = l.a52; m[8 * TILE] = l.a53; m[9 * TILE] = l.a55; m[10 * TILE] = l.b20; m[11 * TILE] = l.b50;
#pragma unroll
            for (int c = 0; c < NS; ++c) m[(12 + c) * TILE] = q[c];
            m[18 * TILE] = r[0]; m[19 * TILE] = r[1];
            if (EXACT) {
                m[20 * TILE] = a.v22; m[21 * TILE] = a.v23; m[22 * TILE] = a.v33; m[23 * TILE] = a.v55; m[24 * TILE] = a.g22; m[25 * TILE] = a.g23;
                m[26 * TILE] = a.g25; m[27 * TILE] = a.g33; m[28 * TILE] = a.g55; m[29 * TILE] = a.c0; m[30 * TILE] = a.c1; m[31 * TILE] = a.c2;
                m[32 * TILE] = a.c3; m[33 * TILE] = a.e2; m[34 * TILE] = a.e3a; m[35 * TILE] = a.e3b;
            }
        } else if (k >= BC_XA) mbar_wait(sh.aempty + s, (uint32_t)((k / BC_XA - 1) & 1));
        __syncwarp();
        if (lane == 0) mbar_arrive(sh.afull + s);
    }
}

// the linearisation out of a message-A slot
template <typename F>
__device__ __forceinline__ void bc_read_lin(const F* m, Lin<F>& l)
{
    l.a02 = m[0 * TILE]; l.a05 = m[1 * TILE]; l.a12 = m[2 * TILE]; l.a15 = m[3 * TILE]; l.a22 = m[4 * TILE]; l.a23 = m[5 * TILE];
    l.a25 = m[6 * TILE]; l.a52 = m[7 * TILE]; l.a53 = m[8 * TILE]; l.a55 = m[9 * TILE]; l.b20 = m[10 * TILE]; l.b50 = m[11 * TILE];
}

// ---- LAMBDA warp
template <bool EXACT, typename F, int DG>
__device__ __forceinline__ void bc_lambda_role(const ProblemT<F>& P, int tile, int lane, bool live, const F* x, const F* xr, const BcShared<F>& sh,
                                               F* __restrict__ KSG)
{
    constexpr int NA = BcMsgA<EXACT>::N;
    const int TT = P.TT, Np = P.Np, nsteps = TT - 1;
    F lam[NS];
    if (live) {
        F dxT[NS];
#pragma unroll
        for (int c = 0; c < NS; ++c) dxT[c] = x[c] - xr[c];
        wmul6(P.W.QT, (int)weights_diag<DG>(P.W), dxT, lam);  // lam_{T-1} = QT dx (optcon.py:429-432)
    }
    BcSlot sa, sbs;
    for (int k = 0; k < nsteps; ++k, sa.next<BC_XA>(), sbs.next<BC_XB>()) {
        const int t = TT - 2 - k, s = sa.s, sb = sbs.s;
        mbar_wait(sh.afull + s, sa.par);
        const F* const m = sh.msgA + (size_t)s * NA * TILE + lane;
        Lin<F> l;
        HessPre<F> a;
        F q[NS], r[NI];
        if (live) {
            bc_read_lin(m, l);
#pragma unroll
            for (int c = 0; c < NS; ++c) q[c] = m[(12 + c) * TILE];
            r[0] = m[18 * TILE]; r[1] = m[19 * TILE];
            if (EXACT) {
                a.v22 = m[20 * TILE]; a.v23 = m[21 * TILE]; a.v33 = m[22 * TILE]; a.v55 = m[23 * TILE]; a.g22 = m[24 * TILE]; a.g23 = m[25 * TILE];
                a.g25 = m[26 * TILE]; a.g33 = m[27 * TILE]; a.g55 = m[28 * TILE]; a.c0 = m[29 * TILE]; a.c1 = m[30 * TILE]; a.c2 = m[31 * TILE];
                a.c3 = m[32 * TILE]; a.e2 = m[33 * TILE]; a.e3a = m[34 * TILE]; a.e3b = m[35 * TILE];
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(sh.aempty + s);
        if (EXACT) {
            if (k >= BC_XB) mbar_wait(sh.bempty + sb, sbs.par ^ 1u);
            if (live) {
                const Hess<F> h = hess_post(a, lam);   // with lam_{t+1} (optcon.py:437)
                F* const mb = sh.msgB + (size_t)sb * BC_MSGB * TILE + lane;
                mb[0 * TILE] = h.h22; mb[1 * TILE] = h.h23; mb[2 * TILE] = h.h25; mb[3 * TILE] = h.h33; mb[4 * TILE] = h.h55;
                mb[5 * TILE] = h.s2; mb[6 * TILE] = h.s3;
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(sh.bfull + sb);
        }
        if (live) {
            F g[NI];
            riccati_costate(P.M, l, q, r, lam, g);
            F* out = KSG + tile_base(t, 16, Np, tile) + lane;
            out[14 * TILE] = g[0]; out[15 * TILE] = g[1];
        }
    }
}

// ---- GAIN warp: G, m, G^-1, y (riccati_gain_core) into the gain block of the step
template <bool EXACT, typename F>
__device__ __forceinline__ void bc_gain_role(const ProblemT<F>& P, int lane, bool live, const BcShared<F>& sh)
{
    constexpr int NA = BcMsgA<EXACT>::N;
    const int nsteps = P.TT - 1;
    bc_bar2();  // the COLUMN warps have stored the terminal P, p
    BcSlot sa;
    for (int k = 0; k < nsteps; ++k, sa.next<BC_XA>()) {
        mbar_wait(sh.afull + sa.s, sa.par);
        const F* const m = sh.msgA + (size_t)sa.s * NA * TILE + lane;
        Lin<F> l;
        F r[NI], Pm[21], p[NS];
        if (live) {
            l.b20 = m[10 * TILE]; l.b50 = m[11 * TILE];
            r[0] = m[18 * TILE]; r[1] = m[19 * TILE];
            Pm[sym(2, 2)] = sh.PB[sym(2, 2) * TILE + lane]; Pm[sym(2, 5)] = sh.PB[sym(2, 5) * TILE + lane]; Pm[sym(5, 5)] = sh.PB[sym(5, 5) * TILE + lane];
            Pm[sym(2, 4)] = sh.PB[sym(2, 4) * TILE + lane]; Pm[sym(4, 5)] = sh.PB[sym(4, 5) * TILE + lane]; Pm[sym(4, 4)] = sh.PB[sym(4, 4) * TILE + lane];
            p[2] = sh.PB[(21 + 2) * TILE + lane]; p[4] = sh.PB[(21 + 4) * TILE + lane]; p[5] = sh.PB[(21 + 5) * TILE + lane];
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(sh.aempty + sa.s);
        if (live) {
            RicGain<F> gn;
            riccati_gain_core(P.M, P.W, l, r, Pm, p, gn);
            F* const gb = sh.GB + (size_t)(k & 1) * BC_GB * TILE + lane;
            gb[0 * TILE] = gn.gi00; gb[1 * TILE] = gn.gi01; gb[2 * TILE] = gn.gi11; gb[3 * TILE] = gn.y0; gb[4 * TILE] = gn.y1;
            gb[5 * TILE] = gn.G00; gb[6 * TILE] = gn.G01; gb[7 * TILE] = gn.G11; gb[8 * TILE] = gn.m0; gb[9 * TILE] = gn.m1;
        }
        bc_bar1();  // Mx of every column and the gain block of step k are in shared memory (buffer k & 1); every warp has read the old P, p
        bc_bar2();  // the new P, p are in shared memory
    }
}

// ---- OUT warp: the outputs K_t, sigma_t (eigenvalue test, regularised inverse, riccati_gain_out) from Mx and the gain block of the step.
// Takes part in barrier 1 only: Mx and the gain block are double-buffered, so it works on step k while the other warps are already in
// the first half of step k+1 (buffer k & 1 is rewritten in step k+2, after barrier 1 of step k+1, which this warp reaches after its reads).
template <typename F>
__device__ __forceinline__ void bc_out_role(const ProblemT<F>& P, int tile, int lane, bool live, const BcShared<F>& sh, F* __restrict__ KSG,
                                            const int* __restrict__ status, int* __restrict__ n_reg)
{
    const int TT = P.TT, Np = P.Np, i = tile * TILE + lane, nsteps = TT - 1;
    int nreg = 0;
    F* out = KSG + tile_base(TT - 2, 16, Np, tile) + lane;
    const size_t ostride = (size_t)(Np / TILE) * 16 * TILE;
    for (int k = 0; k < nsteps; ++k, out -= ostride) {
        bc_bar1();
        if (live) {
            const F* const gb = sh.GB + (size_t)(k & 1) * BC_GB * TILE + lane;
            const F* const mx = sh.MX + (size_t)(k & 1) * 2 * NS * TILE + lane;
            RicGain<F> gn;
            gn.gi00 = gb[0 * TILE]; gn.gi01 = gb[1 * TILE]; gn.gi11 = gb[2 * TILE];
            gn.G00 = gb[5 * TILE]; gn.G01 = gb[6 * TILE]; gn.G11 = gb[7 * TILE]; gn.m0 = gb[8 * TILE]; gn.m1 = gb[9 * TILE];
            F Mx0[NS], Mx1[NS], K[2 * NS], sig[NI];
#pragma unroll
            for (int a = 0; a < NS; ++a) { Mx0[a] = mx[a * TILE]; Mx1[a] = mx[(NS + a) * TILE]; }
            riccati_gain_test(gn);
            riccati_gain_out(gn, Mx0, Mx1, K, sig);
#pragma unroll
            for (int c = 0; c < 12; ++c) out[c * TILE] = K[c];
            out[12 * TILE] = sig[0]; out[13 * TILE] = sig[1];
            nreg += gn.reg;
        }
    }
    if (live && nreg && status[i] == ST_ACTIVE) n_reg[i] += nreg;
}

// ---- COLUMN warp J (column 0, the lightest, also carries the affine term p)
template <bool EXACT, int DG, int J, typename F>
__device__ __forceinline__ void bc_column_role(const ProblemT<F>& P, int tile, int lane, bool live, const F* x, const F* xr, const BcShared<F>& sh)
{
    constexpr int NA = BcMsgA<EXACT>::N;
    constexpr bool NEEDS_H = EXACT && (J == 2 || J == 3 || J == 5);
    constexpr bool HAS_P = J == 0;
    const int nsteps = P.TT - 1;
    F* const PB = sh.PB;
    if (live) {  // terminal condition P_{T-1} = QT, p_{T-1} = lam_{T-1}/2 (optcon.py:688-690, :716): every warp forms it, column J stores its part
        F Pm[21], p[NS], lamT[NS];
        backward_terminal<DG>(P.W, x, xr, Pm, p, lamT);
#pragma unroll
        for (int a = 0; a <= J; ++a) PB[sym(a, J) * TILE + lane] = Pm[sym(a, J)];
        if (HAS_P) {
#pragma unroll
            for (int c = 0; c < NS; ++c) PB[(21 + c) * TILE + lane] = p[c];
        }
    }
    bc_bar2();
    BcSlot sa, sb;
    for (int k = 0; k < nsteps; ++k, sa.next<BC_XA>(), sb.next<BC_XB>()) {
        mbar_wait(sh.afull + sa.s, sa.par);
        const F* const m = sh.msgA + (size_t)sa.s * NA * TILE + lane;
        Lin<F> l;
        Hess<F> h;
        F q[NS], Pm[21], p[NS];
        if (live) {
            bc_read_lin(m, l);
#pragma unroll
            for (int e = 0; e < 21; ++e) Pm[e] = PB[e * TILE + lane];   // (entries this column does not touch are dead loads)
            if (HAS_P) {
#pragma unroll
                for (int c = 0; c < NS; ++c) { q[c] = m[(12 + c) * TILE]; p[c] = PB[(21 + c) * TILE + lane]; }
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(sh.aempty + sa.s);
        if (NEEDS_H) {   // ring B is consumed by the columns 2, 3, 5 only
            mbar_wait(sh.bfull + sb.s, sb.par);
            if (live) {
                const F* const mb = sh.msgB + (size_t)sb.s * BC_MSGB * TILE + lane;
                h.h22 = mb[0 * TILE]; h.h23 = mb[1 * TILE]; h.h25 = mb[2 * TILE]; h.h33 = mb[3 * TILE]; h.h55 = mb[4 * TILE];
                h.s2 = mb[5 * TILE]; h.s3 = mb[6 * TILE];
                h.h35 = -h.h33; h.s5 = -h.s3;  // (as hess_contract forms them)
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(sh.bempty + sb.s);
        }
        F PnJ[NS], Atp[NS], mx0 = F(0.0), mx1 = F(0.0);
        if (live) {
            riccati_col_sweep<EXACT, J, F>(P.M, l, h, Pm, PnJ, mx0, mx1);
            F* const mx = sh.MX + (size_t)(k & 1) * 2 * NS * TILE + lane;
            mx[J * TILE] = mx0; mx[(NS + J) * TILE] = mx1;
            if (HAS_P) riccati_p_sweep(P.M, l, p, Atp);
        }
        bc_bar1();  // Mx of every column and the gain block are in shared memory; every warp has read the old P, p
        if (live) {
            const F* const gb = sh.GB + (size_t)(k & 1) * BC_GB * TILE + lane;
            const F* const mx = sh.MX + (size_t)(k & 1) * 2 * NS * TILE + lane;
            const F gi00 = gb[0 * TILE], gi01 = gb[1 * TILE], gi11 = gb[2 * TILE];
            F Mx0[NS], Mx1[NS], PJ[NS];
#pragma unroll
            for (int a = 0; a < (HAS_P ? NS : J); ++a) { Mx0[a] = mx[a * TILE]; Mx1[a] = mx[(NS + a) * TILE]; }
            Mx0[J] = mx0; Mx1[J] = mx1;
            riccati_col_finish<EXACT, DG, J, F>(P.W, h, gi00, gi01, gi11, PnJ, Mx0, Mx1, PJ);
#pragma unroll
            for (int a = 0; a <= J; ++a) PB[sym(a, J) * TILE + lane] = PJ[a];
            if (HAS_P) {
                riccati_p_finish(q, Atp, Mx0, Mx1, gb[3 * TILE], gb[4 * TILE], p);
#pragma unroll
                for (int c = 0; c < NS; ++c) PB[(21 + c) * TILE + lane] = p[c];
            }
        }
        bc_bar2();  // the new P, p are in shared memory
    }
}

template <bool EXACT, typename F, typename XT, int DG>
__global__ void __launch_bounds__(BC_THREADS, 1) k_backward_cols(ProblemT<F> P, TileList L, const XT* __restrict__ X, const F* __restrict__ U,
                                                                 F* __restrict__ KSG, const int* __restrict__ status, int* __restrict__ n_reg)
{
    using St = BwdStage<F, XT>;
    extern __shared__ __align__(128) unsigned char smem[];
    const int lane = threadIdx.x & 31, role = threadIdx.x >> 5;
    const int tile = warp_tile(L, blockIdx.x, P.Np);
    if (tile < 0) return;  // (uniform over the CTA)
    BcShared<F> sh;
    unsigned char* const rings = smem;
    sh.msgA = reinterpret_cast<F*>(smem + (size_t)BC_NPRE * BWD_STAGES * St::BYTES);
    sh.msgB = sh.msgA + (size_t)BC_XA * BcMsgA<EXACT>::N * TILE;
    sh.PB = sh.msgB + (size_t)BC_XB * BC_MSGB * TILE;
    sh.MX = sh.PB + (size_t)BC_PB * TILE;
    sh.GB = sh.MX + (size_t)2 * 2 * NS * TILE;
    uint64_t* const bar_in = reinterpret_cast<uint64_t*>(sh.GB + (size_t)2 * BC_GB * TILE);
    sh.afull = bar_in + BC_NPRE * BWD_STAGES;
    sh.aempty = sh.afull + BC_XA;
    sh.bfull = sh.aempty + BC_XA;
    sh.bempty = sh.bfull + BC_XB;
    if (threadIdx.x == 0) {
        for (int s = 0; s < BC_NPRE * BWD_STAGES; ++s) mbar_init(bar_in + s, 1);
        for (int s = 0; s < BC_XA; ++s) { mbar_init(sh.afull + s, 1); mbar_init(sh.aempty + s, 2 + NS); }  // consumers: LAMBDA, GAIN, 6 COLUMN (OUT reads no message)
        for (int s = 0; s < BC_XB; ++s) { mbar_init(sh.bfull + s, 1); mbar_init(sh.bempty + s, 3); }       // consumers: COLUMN 2, 3, 5
        mbar_fence_init();
    }
    __syncthreads();
    const int i = tile * TILE + lane;
    const bool live = i < P.N;
    F x[NS], xr[NS];
    if (live && (role == BC_NPRE || role >= BC_NPRE + 3)) {  // terminal condition: LAMBDA and the COLUMN warps need x_{T-1} - xref_{T-1}
        load_xref(P, P.TT - 1, i, xr);
        load_x(P, X, P.TT - 1, i, x);
    }
    if (role < BC_NPRE) {
        bc_pre_role<EXACT, F, XT, DG>(P, tile, lane, live, role, rings + (size_t)role * BWD_STAGES * St::BYTES, bar_in + role * BWD_STAGES, sh, X, U);
        return;
    }
    switch (role - BC_NPRE) {
        case 0: bc_lambda_role<EXACT, F, DG>(P, tile, lane, live, x, xr, sh, KSG); break;
        case 1: bc_gain_role<EXACT, F>(P, lane, live, sh); break;
        case 2: bc_out_role<F>(P, tile, lane, live, sh, KSG, status, n_reg); break;
        case 3: bc_column_role<EXACT, DG, 0, F>(P, tile, lane, live, x, xr, sh); break;
        case 4: bc_column_role<EXACT, DG, 1, F>(P, tile, lane, live, x, xr, sh); break;
        case 5: bc_column_role<EXACT, DG, 2, F>(P, tile, lane, live, x, xr, sh); break;
        case 6: bc_column_role<EXACT, DG, 3, F>(P, tile, lane, live, x, xr, sh); break;
        case 7: bc_column_role<EXACT, DG, 4, F>(P, tile, lane, live, x, xr, sh); break;
        default: bc_column_role<EXACT, DG, 5, F>(P, tile, lane, live, x, xr, sh); break;
    }
}

// =================================================================================================================
// steepest-descent costate sweep (gradient_instance): same ring as the backward sweep (x, u, references per step, walking
// t = TT-2 .. 0); out deltau and the slope -sum |deltau|^2 the Armijo test uses
// =================================================================================================================
template <typename F, typename XT>
__global__ void __launch_bounds__(64) k_gradient_tma(ProblemT<F> P, TileList L, const XT* __restrict__ X, const F* __restrict__ U,
                                                     F* __restrict__ DU, const int* __restrict__ status, double* __restrict__ descent)
{
    using St = BwdStage<F, XT>;
    extern __shared__ __align__(128) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int tile = warp_tile(L, blockIdx.x * nw + warp, P.Np);
    if (tile < 0) return;
    WarpRing<BWD_STAGES, St::BYTES> ring;
    ring.init(smem, warp, nw, lane);
    const int TT = P.TT, Np = P.Np, i = tile * TILE + lane, nsteps = TT - 1;
    const bool live = i < P.N;
    const RefMode<F> rm(P, i, live);
    auto issue = [&](int k) {  // ring step k <-> time t = TT-2-k
        const int t = TT - 2 - k;
        unsigned char* st = ring.stage(k);
        uint64_t* b = ring.barrier(k);
        mbar_arrive_expect_tx(b, St::U_B + St::X_B + (rm.tiled ? St::U_B + St::XR_B : 0) + (rm.has_v ? (uint32_t)(TILE * sizeof(F)) : 0));
        tma_load(st + St::U_O, U + tile_base(t, NI, Np, tile), St::U_B, b);
        tma_load(st + St::X_O, X + tile_base(t, NS, Np, tile), St::X_B, b);
        if (rm.tiled) {
            tma_load(st + St::UR_O, P.uref + tile_base(t, NI, Np, tile), St::U_B, b);
            tma_load(st + St::XR_O, P.xref + tile_base(t, NS, Np, tile), St::XR_B, b);
        } else if (rm.has_v)
            tma_load(st + St::XR_O, P.rp_v + tile_base(t, 1, Np, tile), (uint32_t)(TILE * sizeof(F)), b);
    };
    if (lane == 0)
        for (int k = 0; k < BWD_STAGES && k < nsteps; ++k) issue(k);
    F lam[NS], x[NS], u[NI], xr[NS], ur[NI];
    double sq = 0.0;
    if (live) {
        load_xref(P, TT - 1, i, xr);
        load_x(P, X, TT - 1, i, x);
        gradient_terminal(P.W, x, xr, lam);
        DU[at(TT - 1, NI, 0, Np, i)] = F(0.0);
        DU[at(TT - 1, NI, 1, Np, i)] = F(0.0);
    }
    for (int k = 0; k < nsteps; ++k) {
        const int t = TT - 2 - k;
        ring.wait(k);
        const unsigned char* st = ring.stage(k);
        XT xraw[NS];
#pragma unroll
        for (int c = 0; c < NS; ++c) xraw[c] = reinterpret_cast<const XT*>(st + St::X_O)[c * TILE + lane];
#pragma unroll
        for (int c = 0; c < NI; ++c) u[c] = reinterpret_cast<const F*>(st + St::U_O)[c * TILE + lane];
        F vv = F(0.0);
        if (rm.tiled) {
#pragma unroll
            for (int c = 0; c < NI; ++c) ur[c] = reinterpret_cast<const F*>(st + St::UR_O)[c * TILE + lane];
#pragma unroll
            for (int c = 0; c < NS; ++c) xr[c] = reinterpret_cast<const F*>(st + St::XR_O)[c * TILE + lane];
        } else if (rm.has_v) vv = reinterpret_cast<const F*>(st + St::XR_O)[lane];
        stage_release();
        if (lane == 0 && k + BWD_STAGES < nsteps) issue(k + BWD_STAGES);
        if (live) {
            rm.fill(P, t, i, vv, xr, ur);
            finish_x(P, t, i, xraw, x);
            F du[NI];
            gradient_step(P.M, P.W, x, u, xr, ur, lam, du, sq);
            F* out = DU + tile_base(t, NI, Np, tile) + lane;
            out[0] = du[0];
            out[TILE] = du[1];
        }
    }
    if (live && status[i] == ST_ACTIVE) descent[i] = -sq;
}


// =================================================================================================================
// Armijo candidates over a per-instance work list (the instances whose candidate 0 failed): rollout_instance<false, true>, one
// consumer warp per candidate.
//
// The lanes of a CTA are 32 list entries -- arbitrary instances, so their inputs are not one contiguous block and the bulk-TMA rings
// above do not apply.  Instead ONE producer warp gathers u, du and the references of the next steps of its 32 instances into a
// shared-memory ring with 8-byte cp.async copies (completion counted on an mbarrier by cp.async.mbarrier.arrive), CR_SB time steps
// per stage, and every candidate warp of the CTA reads them from there: the nine candidate rollouts of an instance used to issue the
// same twelve global loads each, with their 64-bit address arithmetic, and wait for them every step (4.1 long-scoreboard stall
// cycles per issued instruction in the round-1 profile); now the loads are in flight CR_STAGES stages ahead of the arithmetic and
// are issued once per CTA.  Same per-step function (rollout_step) as every other rollout kernel: bit-identical costs.
// (get_update over the same list was measured too: with one consumer warp per CTA the gathers are not amortised -- 17.8 GB of
// 32-byte sectors for 8-byte elements -- and the tile-granular TMA sweep k_rollout_write_tma<.,1> stays faster: 2.1 vs 2.9 ms.)
// =================================================================================================================
#ifndef ACOC_CR_SB
#define ACOC_CR_SB 4
#endif
#ifndef ACOC_CR_STAGES
#define ACOC_CR_STAGES 3
#endif
#ifndef ACOC_CAND_MINB
#define ACOC_CAND_MINB 3  // resident candidate CTAs per SM the register allocation is bounded for
#endif
constexpr int CR_SB = ACOC_CR_SB, CR_STAGES = ACOC_CR_STAGES;
constexpr int CR_NV = 2 * NI + NI + NS;  // u, du, uref, xref

// the mbarrier receives one arrival when every cp.async issued so far by this thread has landed (the count is part of init)
__device__ __forceinline__ void cp_async_mbar_arrive(uint64_t* bar)
{
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
template <int BYTES>
__device__ __forceinline__ void cp_async_elem(void* dst_smem, const void* src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], %2;" ::"r"(smem_u32(dst_smem)), "l"(src), "n"(BYTES) : "memory");
}

template <typename F>
constexpr size_t candidates_list_smem() { return (size_t)CR_STAGES * CR_SB * CR_NV * TILE * sizeof(F) + 2 * CR_STAGES * sizeof(uint64_t); }

// blockDim = (32, rows + 1): warps 0..rows-1 roll candidate c0 + pass*rows + y (as many passes as it takes to reach c1), warp `rows`
// gathers.  Jcand[c][i] receives the cost.
template <bool Q32, typename F, int MAXROWS, int DG, int REFS>
__global__ void __launch_bounds__(TILE * (MAXROWS + 1), ACOC_CAND_MINB)
k_candidates_list(ProblemT<F> P, WorkList L, const F* __restrict__ U, const F* __restrict__ DU, const double* __restrict__ steps, int c0, int c1,
                  double* __restrict__ Jcand)
{
    extern __shared__ __align__(128) unsigned char smem[];
    F* const data = reinterpret_cast<F*>(smem);
    uint64_t* const full = reinterpret_cast<uint64_t*>(smem + (size_t)CR_STAGES * CR_SB * CR_NV * TILE * sizeof(F));
    uint64_t* const empty = full + CR_STAGES;
    const int lane = threadIdx.x, row = threadIdx.y, rows = blockDim.y - 1;
    if (work_instance(L, blockIdx.x * TILE, P.N) < 0) return;  // no list entry for this CTA (uniform: the list is dense from the front)
    const int i = work_instance(L, blockIdx.x * TILE + lane, P.N);
    if (lane == 0 && row == 0) {
        for (int s = 0; s < CR_STAGES; ++s) { mbar_init(full + s, TILE); mbar_init(empty + s, rows); }
        mbar_fence_init();
    }
    __syncthreads();
    const int TT = P.TT, Np = P.Np, nsteps = TT - 1, nst = (nsteps + CR_SB - 1) / CR_SB;
    constexpr bool shared_ref = REFS == 1, param_ref = REFS == 2;  // 0: per-instance arrays (P.ref_shared / P.ref_param, known at compile time here)
    const bool has_v = param_ref && P.rp_v != nullptr;
    const int passes = (c1 - c0 + rows - 1) / rows;
    if (row == rows) {  // ---- producer warp
        const size_t tstride_u = (size_t)(Np / TILE) * NI * TILE, tstride_x = (size_t)(Np / TILE) * NS * TILE;
        const size_t ou = i >= 0 ? at(0, NI, 0, Np, i) : 0, ox = i >= 0 ? at(0, NS, 0, Np, i) : 0;
        for (int g = 0; g < passes * nst; ++g) {
            const int st = g % CR_STAGES, sidx = g % nst;
            if (g >= CR_STAGES) mbar_wait(empty + st, (uint32_t)((g / CR_STAGES - 1) & 1));
            if (i >= 0) {
                F* d = data + (size_t)st * CR_SB * CR_NV * TILE + lane;
                for (int k = 0; k < CR_SB; ++k, d += CR_NV * TILE) {
                    const int t = sidx * CR_SB + k;
                    if (t >= nsteps) break;
                    const F* pu = U + ou + (size_t)t * tstride_u;
                    const F* pd = DU + ou + (size_t)t * tstride_u;
                    cp_async_elem<sizeof(F)>(d, pu);
                    cp_async_elem<sizeof(F)>(d + TILE, pu + TILE);
                    cp_async_elem<sizeof(F)>(d + 2 * TILE, pd);
                    cp_async_elem<sizeof(F)>(d + 3 * TILE, pd + TILE);
                    if (!shared_ref && !param_ref) {
                        const F* pr = P.uref + ou + (size_t)t * tstride_u;
                        const F* px = P.xref + ox + (size_t)t * tstride_x;
                        cp_async_elem<sizeof(F)>(d + 4 * TILE, pr);
                        cp_async_elem<sizeof(F)>(d + 5 * TILE, pr + TILE);
#pragma unroll
                        for (int c = 0; c < NS; ++c) cp_async_elem<sizeof(F)>(d + (6 + c) * TILE, px + c * TILE);
                    } else if (has_v)
                        cp_async_elem<sizeof(F)>(d + 8 * TILE, P.rp_v + at(t, 1, 0, Np, i));  // (the slot of xref[2])
                }
            }
            cp_async_mbar_arrive(full + st);
        }
        asm volatile("cp.async.wait_all;" ::: "memory");  // no copy may be in flight when the warp exits
        return;
    }
    // ---- candidate warps
    for (int pass = 0; pass < passes; ++pass) {
        const int c = c0 + pass * rows + row;
        const bool work = i >= 0 && c < c1;
        const F s = (F)(c < c1 ? steps[c] : 0.0);
        const F zf_i = (param_ref && work) ? P.rp_zf[i] : F(0.0), vx_i = (param_ref && work) ? P.rp_vx[i] : F(0.0);
        F x[NS], u[NI], xr[NS], ur[NI];
        double J = 0.0;
#pragma unroll
        for (int cc = 0; cc < NS; ++cc) x[cc] = work ? P.x0[(size_t)cc * Np + i] : F(0.0);
        for (int sidx = 0; sidx < nst; ++sidx) {
            const int g = pass * nst + sidx, st = g % CR_STAGES;
            mbar_wait(full + st, (uint32_t)((g / CR_STAGES) & 1));
            if (work) {
                const F* d = data + (size_t)st * CR_SB * CR_NV * TILE + lane;
#pragma unroll 1
                for (int k = 0; k < CR_SB; ++k, d += CR_NV * TILE) {  // (not unrolled: 64 registers hold one step without spills)
                    const int t = sidx * CR_SB + k;
                    if (t >= nsteps) break;
#pragma unroll
                    for (int cc = 0; cc < NI; ++cc) u[cc] = d[cc * TILE] + s * d[(2 + cc) * TILE];  // optcon.py:197 / :253
                    if (shared_ref) load_ref(P, t, i, xr, ur);
                    else if (param_ref) {
                        param_xref(P, t, zf_i, vx_i, has_v ? d[8 * TILE] : P.rp_xc[2], xr);
                        ur[0] = P.rp_uc[0]; ur[1] = P.rp_uc[1];
                    } else {
#pragma unroll
                        for (int cc = 0; cc < NI; ++cc) ur[cc] = d[(4 + cc) * TILE];
#pragma unroll
                        for (int cc = 0; cc < NS; ++cc) xr[cc] = d[(6 + cc) * TILE];
                    }
                    rollout_step<true, Q32, DG>(P.M, P.W, x, u, xr, ur, J);
                }
            }
            stage_release();
            if (lane == 0) mbar_arrive(empty + st);
        }
        if (work) {
            load_xref(P, TT - 1, i, xr);
            F dx[NS];
#pragma unroll
            for (int cc = 0; cc < NS; ++cc) dx[cc] = x[cc] - xr[cc];
            J += (double)term_cost<DG>(P.W, dx);
            Jcand[(size_t)c * Np + i] = J;
        }
    }
}

// =================================================================================================================
// closed-loop LQR tracking of every instance along its own nominal (track_gains_instance / track_rollout_instance)
// =================================================================================================================
// gains sweep: in x*_t, u*_t (walking t = TT-2 .. 0); out K_t.  40 B read + 96 B written per instance and step with float states; the
// Riccati step is a chain of dependent FP64 operations like k_backward_tma's Gauss-Newton sweep, minus the costate and the references.
constexpr int TRK_GAIN_STAGES = 3;
template <typename XT>
struct TrkGainStage {
    static constexpr int X_B = NS * TILE * sizeof(XT), U_B = NI * TILE * sizeof(double);
    static constexpr int X_O = 0, U_O = X_B, BYTES = X_B + U_B;
};

template <int DG, typename XT>
__global__ void __launch_bounds__(64) k_track_gains_tma(Problem P, const XT* __restrict__ Xnom, const double* __restrict__ Unom,
                                                        double* __restrict__ Ktrk, int* __restrict__ n_reg)
{
    using St = TrkGainStage<XT>;
    extern __shared__ __align__(128) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int tile = blockIdx.x * nw + warp;
    if (tile * TILE >= P.N) return;  // warp-uniform
    WarpRing<TRK_GAIN_STAGES, St::BYTES> ring;
    ring.init(smem, warp, nw, lane);
    const int TT = P.TT, Np = P.Np, i = tile * TILE + lane, nsteps = TT - 1;
    const bool live = i < P.N;
    auto issue = [&](int k) {  // ring step k <-> time t = TT-2-k
        const int t = TT - 2 - k;
        unsigned char* st = ring.stage(k);
        uint64_t* b = ring.barrier(k);
        mbar_arrive_expect_tx(b, St::BYTES);
        tma_load(st + St::X_O, Xnom + tile_base(t, NS, Np, tile), St::X_B, b);
        tma_load(st + St::U_O, Unom + tile_base(t, NI, Np, tile), St::U_B, b);
    };
    if (lane == 0)
        for (int k = 0; k < TRK_GAIN_STAGES && k < nsteps; ++k) issue(k);
    double Pm[21], p[NS];
    track_terminal<DG>(P.W, Pm, p);
    {
        double* out = Ktrk + tile_base(TT - 1, 2 * NS, Np, tile) + lane;
#pragma unroll
        for (int c = 0; c < 2 * NS; ++c) out[c * TILE] = 0.0;
    }
    int nreg = 0;
    for (int k = 0; k < nsteps; ++k) {
        const int t = TT - 2 - k;
        ring.wait(k);
        const unsigned char* st = ring.stage(k);
        XT xraw[NS];
        double x[NS], u[NI];
#pragma unroll
        for (int c = 0; c < NS; ++c) xraw[c] = reinterpret_cast<const XT*>(st + St::X_O)[c * TILE + lane];
#pragma unroll
        for (int c = 0; c < NI; ++c) u[c] = reinterpret_cast<const double*>(st + St::U_O)[c * TILE + lane];
        stage_release();
        if (lane == 0 && k + TRK_GAIN_STAGES < nsteps) issue(k + TRK_GAIN_STAGES);
        if (live) {
            finish_x(P, t, i, xraw, x);
            double K[2 * NS];
            nreg += track_gains_step<DG>(P.M, P.W, x, u, Pm, p, K);
            double* out = Ktrk + tile_base(t, 2 * NS, Np, tile) + lane;
#pragma unroll
            for (int c = 0; c < 2 * NS; ++c) out[c * TILE] = K[c];
        }
    }
    if (live) n_reg[i] = nreg;
}

// closed-loop rollout: in K_t, x*_t, u*_t per step; out x_t, u_t and the per-instance summaries.  136 B read + 40 B written per instance
// and step with float states, a few dozen FP64 operations and one sincos per step: bandwidth-bound like k_forward_cand0_tma.
constexpr int TRK_ROLL_STAGES = 3;
template <typename XT>
struct TrkRollStage {
    static constexpr int K_B = 2 * NS * TILE * sizeof(double), X_B = NS * TILE * sizeof(XT), U_B = NI * TILE * sizeof(double);
    static constexpr int K_O = 0, X_O = K_B, U_O = K_B + X_B, BYTES = K_B + X_B + U_B;
};

template <bool Q32, typename XT>
__global__ void __launch_bounds__(64, 7) k_track_rollout_tma(Problem P, const XT* __restrict__ Xnom, const double* __restrict__ Unom,
                                                             const double* __restrict__ Ktrk, const double* __restrict__ delta,
                                                             XT* __restrict__ Xtrk, double* __restrict__ xtrk0, double* __restrict__ Utrk,
                                                             double* __restrict__ err_max, double* __restrict__ err_final)
{
    using St = TrkRollStage<XT>;
    extern __shared__ __align__(128) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int tile = blockIdx.x * nw + warp;
    if (tile * TILE >= P.N) return;  // warp-uniform
    WarpRing<TRK_ROLL_STAGES, St::BYTES> ring;
    ring.init(smem, warp, nw, lane);
    const int TT = P.TT, Np = P.Np, i = tile * TILE + lane, nsteps = TT - 1;
    const bool live = i < P.N;
    auto issue = [&](int t) {
        unsigned char* st = ring.stage(t);
        uint64_t* b = ring.barrier(t);
        mbar_arrive_expect_tx(b, St::BYTES);
        tma_load(st + St::K_O, Ktrk + tile_base(t, 2 * NS, Np, tile), St::K_B, b);
        tma_load(st + St::X_O, Xnom + tile_base(t, NS, Np, tile), St::X_B, b);
        tma_load(st + St::U_O, Unom + tile_base(t, NI, Np, tile), St::U_B, b);
    };
    if (lane == 0)
        for (int t = 0; t < TRK_ROLL_STAGES && t < nsteps; ++t) issue(t);
    double x[NS], emax[NS];
    if (live) {
        track_start(P, delta, i, x, emax);
#pragma unroll
        for (int c = 0; c < NS; ++c) xtrk0[(size_t)c * Np + i] = x[c];
    }
    for (int t = 0; t < nsteps; ++t) {
        ring.wait(t);
        const unsigned char* st = ring.stage(t);
        double K[2 * NS], un[NI];
        XT xraw[NS];
#pragma unroll
        for (int c = 0; c < 2 * NS; ++c) K[c] = reinterpret_cast<const double*>(st + St::K_O)[c * TILE + lane];
#pragma unroll
        for (int c = 0; c < NS; ++c) xraw[c] = reinterpret_cast<const XT*>(st + St::X_O)[c * TILE + lane];
#pragma unroll
        for (int c = 0; c < NI; ++c) un[c] = reinterpret_cast<const double*>(st + St::U_O)[c * TILE + lane];
        stage_release();
        if (lane == 0 && t + TRK_ROLL_STAGES < nsteps) issue(t + TRK_ROLL_STAGES);
        if (live) {
            double xn[NS], u[NI];
            finish_x(P, t, i, xraw, xn);
            track_error(x, xn, emax);
            track_input(K, x, xn, un, u);
            store_x(Xtrk, t, Np, i, x);
#pragma unroll
            for (int c = 0; c < NI; ++c) Utrk[at(t, NI, c, Np, i)] = u[c];
            track_advance<Q32>(P.M, x, u);
        }
    }
    if (!live) return;
    double xn[NS];
    load_x(P, Xnom, TT - 1, i, xn);
    store_x(Xtrk, TT - 1, Np, i, x);
    Utrk[at(TT - 1, NI, 0, Np, i)] = 0.0;
    Utrk[at(TT - 1, NI, 1, Np, i)] = 0.0;
    track_final(x, xn, emax, err_max, err_final, Np, i);
}

// =================================================================================================================
// Monte Carlo dispersion of the closed loop (track_mc_sample): M perturbed starts per instance along the same nominal and gains.
// The gains and the nominal of an instance are the same for all of its samples, so a CTA flies many (instance, sample) pairs of ONE
// tile through one CTA-shared ring: a producer warp issues the bulk copies of the tile's K / x* / u* block of step t (the TrkRollStage
// of k_track_rollout_tma, 4,352 B with float states) and TRK_MC_WARPS consumer warps read it, full / empty mbarriers per stage as in
// k_candidates_list.  The 136 B an instance-step needs are read once per CTA and step instead of once per sample, which turns the
// bandwidth-bound sweep into an FP64-bound one.
// Pairs of a tile: p -> (lane column j = p mod L, sample m = p div L), L = live lanes of the tile; CTA r of the tile covers pairs
// [r, r+1) * TRK_MC_WARPS * 32, consumer warp w the 32 of them at offset 32 w.  With N >= 32 that is lane = instance, warp = sample;
// with N = 1 every lane flies a sample of the one instance and reads the same shared-memory column (a broadcast).  blockIdx.x =
// tile * ctas_per_tile + r: the CTAs of one tile are adjacent and their copies of its blocks mostly hit L2.
// Same per-step functions as k_track_rollout_tma (finish_x, track_error, track_input, track_advance, track_final_err): bit-identical
// summaries.
// =================================================================================================================
#ifndef ACOC_TRK_MC_WARPS
#define ACOC_TRK_MC_WARPS 8
#endif
#ifndef ACOC_TRK_MC_MINB
#define ACOC_TRK_MC_MINB 2
#endif
constexpr int TRK_MC_WARPS = ACOC_TRK_MC_WARPS, TRK_MC_STAGES = 4;
constexpr int TRK_MC_THREADS = TILE * (TRK_MC_WARPS + 1);
template <typename XT>
constexpr size_t track_mc_smem() { return (size_t)TRK_MC_STAGES * TrkRollStage<XT>::BYTES + 2 * TRK_MC_STAGES * sizeof(uint64_t); }

// delta: per-sample perturbations, d6 of (instance i, sample m) at delta + i * dstride + m * 6 (dstride = 0: shared (M,6), M * 6: (N,M,6))
template <bool Q32, typename XT>
__global__ void __launch_bounds__(TRK_MC_THREADS, ACOC_TRK_MC_MINB)
k_track_mc_rollout_tma(Problem P, const XT* __restrict__ Xnom, const double* __restrict__ Unom, const double* __restrict__ Ktrk,
                       const double* __restrict__ delta, long long dstride, int M, int ctas_per_tile, double* __restrict__ em,
                       double* __restrict__ ef)
{
    using St = TrkRollStage<XT>;
    extern __shared__ __align__(128) unsigned char smem[];
    uint64_t* const full = reinterpret_cast<uint64_t*>(smem + (size_t)TRK_MC_STAGES * St::BYTES);
    uint64_t* const empty = full + TRK_MC_STAGES;
    const int tile = blockIdx.x / ctas_per_tile, r = blockIdx.x % ctas_per_tile;
    const int L = min(TILE, P.N - tile * TILE), lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long pairs = (long long)L * M, p0 = (long long)r * TRK_MC_WARPS * TILE;
    if (p0 >= pairs) return;  // CTA-uniform: a partial tile needs fewer CTAs
    if (threadIdx.x == 0) {
        for (int s = 0; s < TRK_MC_STAGES; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, TRK_MC_WARPS); }
        mbar_fence_init();
    }
    __syncthreads();
    const int TT = P.TT, Np = P.Np, nsteps = TT - 1;
    if (warp == TRK_MC_WARPS) {  // ---- producer warp
        if (lane == 0)
            for (int t = 0; t < nsteps; ++t) {
                const int s = t % TRK_MC_STAGES;
                if (t >= TRK_MC_STAGES) mbar_wait(empty + s, (uint32_t)((t / TRK_MC_STAGES - 1) & 1));
                unsigned char* st = smem + (size_t)s * St::BYTES;
                mbar_arrive_expect_tx(full + s, St::BYTES);
                tma_load(st + St::K_O, Ktrk + tile_base(t, 2 * NS, Np, tile), St::K_B, full + s);
                tma_load(st + St::X_O, Xnom + tile_base(t, NS, Np, tile), St::X_B, full + s);
                tma_load(st + St::U_O, Unom + tile_base(t, NI, Np, tile), St::U_B, full + s);
            }
        return;  // the consumers wait for every copy before they exit
    }
    // ---- consumer warps
    const long long p = p0 + (long long)warp * TILE + lane;
    const bool work = p < pairs;
    const int j = work ? (int)(p % L) : 0, m = work ? (int)(p / L) : 0, i = tile * TILE + j;
    double x[NS], emax[NS];
    if (work) {
        double d6[NS];
        const double* d = delta + (size_t)i * (size_t)dstride + (size_t)m * NS;
#pragma unroll
        for (int c = 0; c < NS; ++c) d6[c] = d[c];
        track_start_from(P, i, d6, x, emax);
    }
    for (int t = 0; t < nsteps; ++t) {
        const int s = t % TRK_MC_STAGES;
        mbar_wait(full + s, (uint32_t)((t / TRK_MC_STAGES) & 1));
        const unsigned char* st = smem + (size_t)s * St::BYTES;
        double K[2 * NS], un[NI];
        XT xraw[NS];
#pragma unroll
        for (int c = 0; c < 2 * NS; ++c) K[c] = reinterpret_cast<const double*>(st + St::K_O)[c * TILE + j];
#pragma unroll
        for (int c = 0; c < NS; ++c) xraw[c] = reinterpret_cast<const XT*>(st + St::X_O)[c * TILE + j];
#pragma unroll
        for (int c = 0; c < NI; ++c) un[c] = reinterpret_cast<const double*>(st + St::U_O)[c * TILE + j];
        stage_release();  // proxy fence before the stage goes back to the bulk-copy engine
        if (lane == 0) mbar_arrive(empty + s);
        if (work) {
            double xn[NS], u[NI];
            finish_x(P, t, i, xraw, xn);
            track_error(x, xn, emax);
            track_input(K, x, xn, un, u);
            track_advance<Q32>(P.M, x, u);
        }
    }
    if (!work) return;
    double xn[NS], efin[NS];
    load_x(P, Xnom, TT - 1, i, xn);
    track_final_err(x, xn, emax, efin);
    const size_t o = ((size_t)i * M + m) * NS;
#pragma unroll
    for (int c = 0; c < NS; ++c) { em[o + c] = emax[c]; ef[o + c] = efin[c]; }
}

// =================================================================================================================
// derivative of the optimum (acoc_result_vjp): the adjoint LQ problem along the result (vjp_backward_instance / vjp_forward_instance)
// =================================================================================================================
// backward sweep: in x*_t, u*_t, references, gbar_t (walking t = TT-2 .. 0); out K_t, sigma_t, and per instance xi_bar, n_indef.  The
// step is k_backward_tma's exact-Hessian step (column pieces of the Riccati update, the costate recursion), plus the 64 B of gbar.
constexpr int VJP_BWD_STAGES = 3;
template <typename XT>
struct VjpBwdStage {
    static constexpr int U_B = NI * TILE * sizeof(double), XR_B = NS * TILE * sizeof(double), X_B = NS * TILE * sizeof(XT);
    static constexpr int U_O = 0, UR_O = U_B, GU_O = 2 * U_B, XR_O = 3 * U_B, GX_O = 3 * U_B + XR_B, X_O = 3 * U_B + 2 * XR_B, BYTES = X_O + X_B;
};

template <int DG, typename XT>
__global__ void __launch_bounds__(64) k_vjp_backward_tma(Problem P, const XT* __restrict__ X, const double* __restrict__ U,
                                                         const double* __restrict__ GX, const double* __restrict__ GU, double* __restrict__ VKS,
                                                         double* __restrict__ xi_bar, int* __restrict__ n_indef)
{
    using St = VjpBwdStage<XT>;
    extern __shared__ __align__(128) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int tile = blockIdx.x * nw + warp;
    if (tile * TILE >= P.N) return;  // warp-uniform
    WarpRing<VJP_BWD_STAGES, St::BYTES> ring;
    ring.init(smem, warp, nw, lane);
    const int TT = P.TT, Np = P.Np, i = tile * TILE + lane, nsteps = TT - 1;
    const bool live = i < P.N;
    const RefMode<double> rm(P, i, live);
    auto issue = [&](int k) {  // ring step k <-> time t = TT-2-k
        const int t = TT - 2 - k;
        unsigned char* st = ring.stage(k);
        uint64_t* b = ring.barrier(k);
        mbar_arrive_expect_tx(b, 2 * St::U_B + St::XR_B + St::X_B + (rm.tiled ? St::U_B + St::XR_B : 0) +
                                     (rm.has_v ? (uint32_t)(TILE * sizeof(double)) : 0));
        tma_load(st + St::U_O, U + tile_base(t, NI, Np, tile), St::U_B, b);
        tma_load(st + St::X_O, X + tile_base(t, NS, Np, tile), St::X_B, b);
        tma_load(st + St::GU_O, GU + tile_base(t, NI, Np, tile), St::U_B, b);
        tma_load(st + St::GX_O, GX + tile_base(t, NS, Np, tile), St::XR_B, b);
        if (rm.tiled) {
            tma_load(st + St::UR_O, P.uref + tile_base(t, NI, Np, tile), St::U_B, b);
            tma_load(st + St::XR_O, P.xref + tile_base(t, NS, Np, tile), St::XR_B, b);
        } else if (rm.has_v)
            tma_load(st + St::XR_O, P.rp_v + tile_base(t, 1, Np, tile), (uint32_t)(TILE * sizeof(double)), b);
    };
    if (lane == 0)
        for (int k = 0; k < VJP_BWD_STAGES && k < nsteps; ++k) issue(k);
    double Pm[21], p[NS], lam[NS], x[NS], u[NI], xr[NS], ur[NI], gx[NS], gu[NI], gl[NI];
    int n = 0;
    if (live) {
        load_xref(P, TT - 1, i, xr);
        load_x(P, X, TT - 1, i, x);
        vjp_load_g(GX, GU, TT - 1, TT, Np, i, gx, gu);
        vjp_terminal<DG>(P.W, x, xr, gx, Pm, p, lam);
#pragma unroll
        for (int c = 0; c < NI; ++c) gl[c] = gu[c];  // gbar_u[TT-1], folded into step TT-2
    }
    for (int k = 0; k < nsteps; ++k) {
        const int t = TT - 2 - k;
        ring.wait(k);
        const unsigned char* st = ring.stage(k);
        XT xraw[NS];
#pragma unroll
        for (int c = 0; c < NS; ++c) xraw[c] = reinterpret_cast<const XT*>(st + St::X_O)[c * TILE + lane];
#pragma unroll
        for (int c = 0; c < NS; ++c) gx[c] = reinterpret_cast<const double*>(st + St::GX_O)[c * TILE + lane];
#pragma unroll
        for (int c = 0; c < NI; ++c) {
            u[c] = reinterpret_cast<const double*>(st + St::U_O)[c * TILE + lane];
            gu[c] = reinterpret_cast<const double*>(st + St::GU_O)[c * TILE + lane];
        }
        double vv = 0.0;
        if (rm.tiled) {
#pragma unroll
            for (int c = 0; c < NI; ++c) ur[c] = reinterpret_cast<const double*>(st + St::UR_O)[c * TILE + lane];
#pragma unroll
            for (int c = 0; c < NS; ++c) xr[c] = reinterpret_cast<const double*>(st + St::XR_O)[c * TILE + lane];
        } else if (rm.has_v) vv = reinterpret_cast<const double*>(st + St::XR_O)[lane];
        stage_release();
        if (lane == 0 && k + VJP_BWD_STAGES < nsteps) issue(k + VJP_BWD_STAGES);
        if (live) {
            if (t == TT - 2) {
#pragma unroll
                for (int c = 0; c < NI; ++c) gu[c] = gu[c] + gl[c];  // vjp_load_g's fold
            }
            rm.fill(P, t, i, vv, xr, ur);
            finish_x(P, t, i, xraw, x);
            double K[2 * NS], sig[NI];
            n += vjp_backward_step<DG>(P.M, P.W, x, u, xr, ur, gx, gu, Pm, p, lam, K, sig);
            double* out = VKS + tile_base(t, 14, Np, tile) + lane;
#pragma unroll
            for (int c = 0; c < 12; ++c) out[c * TILE] = K[c];
            out[12 * TILE] = sig[0]; out[13 * TILE] = sig[1];
        }
    }
    if (!live) return;
#pragma unroll
    for (int c = 0; c < NS; ++c) xi_bar[(size_t)c * Np + i] = -p[c];
    n_indef[i] = n;
}

// forward sweep: in K_t / sigma_t, x*_t, u*_t (and the stored speed reference when the parametric sums are wanted); out xref_bar and
// uref_bar (skipped when XB / UB are nullptr) and the sums zf_bar, vx_bar (zv [2][Np], nullptr: not parametric)
constexpr int VJP_FWD_STAGES = 3;
template <typename XT>
struct VjpFwdStage {
    static constexpr int KS_B = 14 * TILE * sizeof(double), U_B = NI * TILE * sizeof(double), V_B = TILE * sizeof(double),
                         X_B = NS * TILE * sizeof(XT);
    static constexpr int KS_O = 0, U_O = KS_B, V_O = KS_B + U_B, X_O = KS_B + U_B + V_B, BYTES = X_O + X_B;
};

template <int DG, typename XT>
__global__ void __launch_bounds__(64) k_vjp_forward_tma(Problem P, const XT* __restrict__ X, const double* __restrict__ U,
                                                        const double* __restrict__ VKS, const double* __restrict__ vs, double* __restrict__ XB,
                                                        double* __restrict__ UB, double* __restrict__ zv)
{
    using St = VjpFwdStage<XT>;
    extern __shared__ __align__(128) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int tile = blockIdx.x * nw + warp;
    if (tile * TILE >= P.N) return;  // warp-uniform
    WarpRing<VJP_FWD_STAGES, St::BYTES> ring;
    ring.init(smem, warp, nw, lane);
    const int TT = P.TT, Np = P.Np, i = tile * TILE + lane, nsteps = TT - 1;
    const bool live = i < P.N;
    const bool has_v = zv && P.ref_param && P.rp_v;
    auto issue = [&](int t) {
        unsigned char* st = ring.stage(t);
        uint64_t* b = ring.barrier(t);
        mbar_arrive_expect_tx(b, St::KS_B + St::U_B + St::X_B + (has_v ? St::V_B : 0));
        tma_load(st + St::KS_O, VKS + tile_base(t, 14, Np, tile), St::KS_B, b);
        tma_load(st + St::U_O, U + tile_base(t, NI, Np, tile), St::U_B, b);
        tma_load(st + St::X_O, X + tile_base(t, NS, Np, tile), St::X_B, b);
        if (has_v) tma_load(st + St::V_O, P.rp_v + tile_base(t, 1, Np, tile), St::V_B, b);
    };
    if (lane == 0)
        for (int t = 0; t < VJP_FWD_STAGES && t < nsteps; ++t) issue(t);
    const double zf = (zv && live) ? P.rp_zf[i] : 0.0, vx = (zv && live) ? P.rp_vx[i] : 0.0;
    VjpParamSums s = {0.0, 0.0, 0.0, 0.0};
    double wx[NS] = {0, 0, 0, 0, 0, 0}, xb[NS], ub[NI];
    for (int t = 0; t < nsteps; ++t) {
        ring.wait(t);
        const unsigned char* st = ring.stage(t);
        double ks[14], u[NI];
        XT xraw[NS];
#pragma unroll
        for (int c = 0; c < 14; ++c) ks[c] = reinterpret_cast<const double*>(st + St::KS_O)[c * TILE + lane];
#pragma unroll
        for (int c = 0; c < NS; ++c) xraw[c] = reinterpret_cast<const XT*>(st + St::X_O)[c * TILE + lane];
#pragma unroll
        for (int c = 0; c < NI; ++c) u[c] = reinterpret_cast<const double*>(st + St::U_O)[c * TILE + lane];
        const double vv = has_v ? reinterpret_cast<const double*>(st + St::V_O)[lane] : 0.0;
        stage_release();
        if (lane == 0 && t + VJP_FWD_STAGES < nsteps) issue(t + VJP_FWD_STAGES);
        if (live) {
            double x[NS];
            finish_x(P, t, i, xraw, x);
            vjp_forward_step<DG>(P.M, P.W, t, x, u, ks, wx, xb, ub);
            if (XB) {
                double* o = XB + tile_base(t, NS, Np, tile) + lane;
#pragma unroll
                for (int c = 0; c < NS; ++c) o[c * TILE] = xb[c];
            }
            if (UB) {
                double* o = UB + tile_base(t, NI, Np, tile) + lane;
#pragma unroll
                for (int c = 0; c < NI; ++c) o[c * TILE] = ub[c];
            }
            if (zv) vjp_param_add(s, P.rp_tt[t], P.rp_zs[t], has_v, has_v ? vs[t] : 0.0, vv, zf, vx, xb);
        }
    }
    if (!live) return;
    wmul6(P.W.QT, (int)weights_diag<DG>(P.W), wx, xb);
    if (XB) {
#pragma unroll
        for (int c = 0; c < NS; ++c) XB[at(TT - 1, NS, c, Np, i)] = xb[c];
    }
    if (UB) {
#pragma unroll
        for (int c = 0; c < NI; ++c) UB[at(TT - 1, NI, c, Np, i)] = 0.0;
    }
    if (zv) {
        const int t = TT - 1;
        vjp_param_add(s, P.rp_tt[t], P.rp_zs[t], has_v, has_v ? vs[t] : 0.0, has_v ? param_vref(P, t, i) : 0.0, zf, vx, xb);
        zv[i] = s.z + s.zv;
        zv[(size_t)Np + i] = s.x + s.xv;
    }
}

}  // namespace acoc
