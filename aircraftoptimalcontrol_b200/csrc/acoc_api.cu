// acoc_api.cu -- libacoc.so: CUDA kernels (sm_100a) + C ABI declared in include/acoc.h.
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -fmad=false -shared -Xcompiler -fPIC
// (-fmad=false: every FMA in this library is written explicitly as fma(); see acoc_math.cuh).
//
// Execution model: one thread = one OCP instance for the sequential-in-time sweeps (backward Riccati /
// costate sweep, LQ forward pass, rollouts); the Armijo candidates add a second thread dimension
// (candidate x instance) so that the 10 candidates of 32 neighbouring instances share one CTA and hit the
// same input/reference lines in L1.  All trajectory buffers are warp-tiled struct-of-arrays (time, tile of 32 instances,
// component, lane; see acoc_kernels.cuh); host buffers use the reference's (N,6,TT) layout and are transposed on
// the device through a staging buffer.  The time sweeps of the Newton loop run as warp-private TMA pipelines
// (acoc_tma.cuh); the plain-load versions of the same sweeps below are kept for A/B runs (ACOC_NO_TMA).
//
// Every sweep kernel is a template on the arithmetic/storage type F (double: the parity path; float: the optional FP32
// mode, ACOC_FP32) and on the storage type XT of the state iterates (float whenever the states are float32 values anyway,
// see acoc_kernels.cuh "Types").  The context keeps untyped device buffers; DISPATCH_FX / DISPATCH_F pick the instantiation of a
// host routine, and with_flag / with_flags / with_mode / with_real that of a kernel whose other template arguments (state
// quantisation, diagonal weights, exact Hessians, reference mode, ...) are runtime facts of the context.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>

#include "../../include/acoc.h"
#include "acoc_kernels.cuh"
#include "acoc_tma.cuh"

using namespace acoc;

// ======================================================================================================
// error plumbing
// ======================================================================================================
static thread_local std::string g_err;
static thread_local double g_pt_ms[3] = {0, 0, 0};  // device time of the kernels of the last acoc_lqr_tracking call (acoc_last_pointwise_timing)

static int fail(int code, const char* fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CK(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e__ = (call);                                                                        \
        if (e__ != cudaSuccess) {                                                                        \
            cudaGetLastError(); /* clear the per-thread error state */                                   \
            return fail(ACOC_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
        }                                                                                                \
    } while (0)

#define REQUIRE(cond, ...)                                   \
    do {                                                     \
        if (!(cond)) return fail(ACOC_ERR_INVALID, __VA_ARGS__); \
    } while (0)

// ======================================================================================================
// kernels
// ======================================================================================================
constexpr int ST_PAD = 4;  // padding lanes beyond N: never active
constexpr unsigned ACOC_CTX_LITE = 0x40000000u;  // internal flag of acoc_ctx_create (not part of the ABI), see there
constexpr unsigned ACOC_CTX_NO_SLOTS = 0x20000000u;  // internal, with ACOC_CTX_LITE: no iterate slot either (acoc_lqr_tracking_many)

// granularity of the active-work list of the sweeps: groups of 2^shift consecutive instances that still contain an active one
#ifndef ACOC_ACT_SHIFT
#define ACOC_ACT_SHIFT 5  // whole tiles of 32 instances (one warp): measured 366 ms vs 374 ms (groups of 4) on the config-4 solve
#endif
constexpr int BWD_THREADS = 64;
constexpr int FWD_THREADS = 64;
constexpr int ROLL_THREADS = 64;
#ifndef ACOC_CAND_TILE
#define ACOC_CAND_TILE 32
#endif
#ifndef ACOC_CAND_MINB
#define ACOC_CAND_MINB 3  // 64 registers (72 B of spills): 27 resident candidate warps per SM instead of 18
#endif
constexpr int CAND_TILE = ACOC_CAND_TILE;  // instances per candidate CTA (one warp per candidate)
constexpr int CAND_MAXY = 10;              // candidates per CTA; more candidates than this loop inside the thread

// pick the instantiation of a host-side launch template for a context: <F, XT> or <F>
#define DISPATCH_FX(c, fn, ...) \
    ((c)->fp32 ? fn<float, float>(__VA_ARGS__) : ((c)->x_float ? fn<double, float>(__VA_ARGS__) : fn<double, double>(__VA_ARGS__)))
#define DISPATCH_F(c, fn, ...) ((c)->fp32 ? fn<float>(__VA_ARGS__) : fn<double>(__VA_ARGS__))

// Pick the instantiation of a single launch: fn is called with the compile-time twin of a runtime value (std::true_type /
// std::false_type, std::integral_constant<int, 0..2>, or type_tag<float> / type_tag<double>), which it uses as a template argument.
// Every arm is instantiated, so a selector may only be used where every combination it produces is a kernel the library needs.
template <typename Fn>
static int with_flag(bool b, Fn&& fn) { return b ? fn(std::true_type{}) : fn(std::false_type{}); }
template <typename Fn>
static int with_flags(bool a, bool b, Fn&& fn)
{
    return with_flag(a, [&](auto A) { return with_flag(b, [&](auto B) { return fn(A, B); }); });
}
template <typename Fn>
static int with_mode(int m, Fn&& fn)  // m = 0, 1 or 2
{
    return m == 2 ? fn(std::integral_constant<int, 2>{}) : m == 1 ? fn(std::integral_constant<int, 1>{}) : fn(std::integral_constant<int, 0>{});
}
template <typename T>
struct type_tag { using type = T; };
template <typename Fn>
static int with_real(bool f32, Fn&& fn) { return f32 ? fn(type_tag<float>{}) : fn(type_tag<double>{}); }

// launch a kernel that stages its inputs in dynamic shared memory (the TMA rings): the largest shared-memory carveout, and the
// opt-in above the default 48 KB of dynamic shared memory where the kernel needs more
template <typename... P, typename... A>
static int launch_ring(void (*kernel)(P...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, A&&... a)
{
    CK(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    if (smem > 48 * 1024) CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kernel<<<grid, block, smem, st>>>(std::forward<A>(a)...);
    CK(cudaGetLastError());
    return 0;
}

template <typename F, typename XT>
__global__ void __launch_bounds__(128) k_traj_cost(ProblemT<F> P, const XT* __restrict__ X, const F* __restrict__ U,
                                                  const int* __restrict__ status, double* __restrict__ J)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P.N || status[i] != ST_ACTIVE) return;
    J[i] = traj_cost_instance(P, X, U, i);
}

// ---- work lists -----------------------------------------------------------------------------------------
// Late in a solve most instances have terminated and, in the float32-noise phase, only some instances need the
// remaining Armijo candidates.  Threads are therefore mapped to instances through a compacted, ORDERED list of
// groups of G = 2^shift consecutive instances that still contain work.  G = 32 (one tile = one warp = one TMA block) for the
// sweeps; G = 1 for the compute-bound candidate rollouts.
// (struct WorkList / work_instance: acoc_tma.cuh)

// One CTA, ordered stream compaction.  mode 0: group alive iff any status[i] == ST_ACTIVE; mode 1: iff any flag[i] != 0.
// Every thread owns a contiguous range of groups: count, one block-wide exclusive scan, write (two passes over the flags, which
// stay in L1/L2; ~10 us for 65,536 entries instead of ~75 us for a tile-by-tile loop with two barriers per 1024 entries).
// base: the list covers instances [base, base + N) and holds absolute group numbers (base must be a multiple of the group size).
__global__ void __launch_bounds__(1024) k_build_list(const int* __restrict__ flag, int mode, int N, int shift, int* __restrict__ groups,
                                                     int* __restrict__ count, int base = 0)
{
    flag += base;
    const int gbase = base >> shift;
    __shared__ int warp_tot[32];
    const int G = 1 << shift, ngroups = (N + G - 1) >> shift;
    const int per = (ngroups + 1023) / 1024, lo = min(ngroups, (int)threadIdx.x * per), hi = min(ngroups, lo + per);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    auto alive = [&](int g) {
        bool a = false;
        if (shift == 5 && (g << 5) + 32 <= N) {  // whole tile: eight independent 16-byte loads instead of 32 dependent ones
            const int4* q = reinterpret_cast<const int4*>(flag + (g << 5));
            int4 v[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) v[k] = q[k];
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                if (mode == 0) a |= v[k].x == ST_ACTIVE || v[k].y == ST_ACTIVE || v[k].z == ST_ACTIVE || v[k].w == ST_ACTIVE;
                else a |= (v[k].x | v[k].y | v[k].z | v[k].w) != 0;
            }
            return a;
        }
        for (int k = 0; k < G; ++k) {
            const int i = (g << shift) + k;
            if (i < N) a |= mode == 0 ? (flag[i] == ST_ACTIVE) : (flag[i] != 0);
        }
        return a;
    };
    int cnt = 0;
    for (int g = lo; g < hi; ++g) cnt += alive(g) ? 1 : 0;
    int incl = cnt;  // inclusive scan inside the warp
    for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int t = warp_tot[lane], it = t;
        for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, it, o); if (lane >= o) it += v; }
        warp_tot[lane] = it - t;  // exclusive offsets of the warps
        if (lane == 31) *count = it;
    }
    __syncthreads();
    int off = warp_tot[warp] + incl - cnt;
    for (int g = lo; g < hi; ++g) if (alive(g)) groups[off++] = gbase + g;
}

template <bool EXACT, typename F, typename XT>
__global__ void __launch_bounds__(BWD_THREADS) k_backward(ProblemT<F> P, WorkList L, const XT* __restrict__ X, const F* __restrict__ U,
                                                          F* __restrict__ KSG, const int* __restrict__ status, int* __restrict__ n_reg)
{
    const int i = work_instance(L, blockIdx.x * blockDim.x + threadIdx.x, P.N);
    if (i < 0) return;
    // Lanes of already finished instances inside a live group run the sweep too: K/sigma/g are per-iteration scratch, and
    // writing all lanes keeps every 32-byte sector fully written (a partially written sector costs a DRAM read-modify-write);
    // the lane would otherwise idle for the same number of warp instructions.
    const int r = backward_instance<EXACT>(P, X, U, KSG, i);
    if (r && status[i] == ST_ACTIVE) n_reg[i] += r;
}

template <typename F, typename XT>
__global__ void __launch_bounds__(FWD_THREADS) k_forward(ProblemT<F> P, WorkList L, const XT* __restrict__ X, const F* __restrict__ U,
                                                         const F* __restrict__ KSG, F* __restrict__ DU, F* DX,
                                                         const int* __restrict__ status, double* __restrict__ descent)
{
    const int i = work_instance(L, blockIdx.x * blockDim.x + threadIdx.x, P.N);
    if (i < 0) return;
    const double d = forward_lq_instance(P, X, U, KSG, DU, DX, i);  // finished lanes of a live group: see k_backward
    if (status[i] == ST_ACTIVE) descent[i] = d;
}

// steepest-descent costate sweep (GradientMethod.optimize): deltau and the slope -sum |deltau|^2 (plain-load version)
template <typename F, typename XT>
__global__ void __launch_bounds__(FWD_THREADS) k_gradient(ProblemT<F> P, WorkList L, const XT* __restrict__ X, const F* __restrict__ U,
                                                          F* __restrict__ DU, const int* __restrict__ status, double* __restrict__ descent)
{
    const int i = work_instance(L, blockIdx.x * blockDim.x + threadIdx.x, P.N);
    if (i < 0) return;
    const double sq = gradient_instance(P, X, U, DU, i);  // finished lanes of a live group: see k_backward
    if (status[i] == ST_ACTIVE) descent[i] = -sq;
}

// thread (x = position in the work list, y = candidate): J of candidate c0 + y for instance i
// MAXY: most candidates (blockDim.y) per CTA.  9 (the lazy search: candidates 1..9) lets three CTAs per SM use 72 registers with
// no spills to speak of; 10 (all candidates at once) gets 64.
template <bool Q32, typename F, int MAXY>
__global__ void __launch_bounds__(CAND_TILE * MAXY, ACOC_CAND_MINB)
k_candidates(ProblemT<F> P, WorkList L, const F* __restrict__ U, const F* __restrict__ DU, const double* __restrict__ cand_steps, int c0,
             int c1, const int* __restrict__ status, double* __restrict__ Jcand)
{
    const int i = work_instance(L, blockIdx.x * CAND_TILE + threadIdx.x, P.N);
    if (i < 0 || status[i] != ST_ACTIVE) return;
    for (int c = c0 + threadIdx.y; c < c1; c += blockDim.y)
        Jcand[(size_t)c * P.Np + i] = rollout_instance<false, true, Q32>(P, U, DU, cand_steps[c], (F*)nullptr, (F*)nullptr, i);
}

// ---- small batches: the whole line search in ONE sweep -------------------------------------------------------------------------
// A batch of a few thousand instances (a late survivor generation, a single trajectory) is latency-bound: every time sweep costs
// about 1 us per step whatever the batch size, so an iteration costs as many milliseconds as it has sequential sweeps.  Both the LQ
// forward pass and the Armijo rollouts run forward in time and candidate c needs du_t only at step t, so they run as ONE sweep:
// CTA = one tile of 32 instances, warp y < n_rows = the rollout of step cand_steps[y] (the armijo_maxiters candidates and, as the last
// row, the untested step the search falls back to on exhaustion, optcon.py:327), warp n_rows = the LQ forward pass one step ahead of
// them, handing du_t over through double-buffered shared-memory blocks of FUSE_BLOCK steps (one barrier per block).  Every row keeps its trajectory
// (Xc / Uc: one trajectory slot per row), so that get_update is a copy of the chosen row (k_pick) instead of one more sweep.
// Inputs of the next step are fetched into registers before the arithmetic of the current one.  Same per-step functions as the
// separate sweeps (forward_step, rollout_step), so the results are bit-identical to them.
constexpr int FUSE_MAXROWS = 11;
#ifndef ACOC_FUSE_BLOCK
#define ACOC_FUSE_BLOCK 8
#endif
constexpr int FUSE_BLOCK = ACOC_FUSE_BLOCK;  // steps between two CTA-wide barriers
template <bool Q32, typename F, typename XT>
__global__ void __launch_bounds__(TILE * (FUSE_MAXROWS + 1))
k_search_fused(ProblemT<F> P, TileList L, const XT* __restrict__ X, const F* __restrict__ U, const F* __restrict__ KSG, F* __restrict__ DU,
               const double* __restrict__ cand_steps, int n_rows, XT* __restrict__ Xc, F* __restrict__ Uc, size_t row_x, size_t row_u,
               const int* __restrict__ status, double* __restrict__ descent, double* __restrict__ Jcand)
{
    __shared__ F sdu[2][FUSE_BLOCK][NI][TILE];
    const int tile = warp_tile(L, blockIdx.x, P.Np);
    if (tile < 0) return;  // (uniform over the CTA)
    const int lane = threadIdx.x, row = threadIdx.y, TT = P.TT, Np = P.Np;
    const int i = tile * TILE + lane;
    const bool valid = i < P.N;
    const bool fwd = row == n_rows;
    // finished lanes of a live tile: the forward pass keeps writing du (scratch, whole lines); the rollouts skip them
    const bool act = valid && (fwd || status[i] == ST_ACTIVE);
    // The two roles overlay their loop-carried state in one register array (a warp has one role for its whole life, but the compiler
    // would otherwise keep both sets live across the loop):
    //   forward pass: st[0..5] = dx, st[6..21] = K, sigma, g of the next step      rollout: st[0..5] = x, st[6..11] / st[12..13] = refs of the next step
    F st[22];
    F* const dx = st;
    F* const ksg_n = st + 6;
    F* const x = st;
    F* const xr_n = st + 6;
    F* const ur_n = st + 12;
    XT xraw_n[NS];
    double acc = 0.0;  // descent (forward warp) / cost (rollout warps)
    F u_n[NI];  // both roles: u_t of the nominal iterate, fetched one step ahead
    F s = F(0.0);
    XT* Xn = nullptr;
    F* Un = nullptr;
#pragma unroll
    for (int c = 0; c < 22; ++c) st[c] = F(0.0);
    if (act) {
#pragma unroll
        for (int c = 0; c < NI; ++c) u_n[c] = U[at(0, NI, c, Np, i)];
        if (fwd) {
            load_x_raw(X, 0, Np, i, xraw_n);
#pragma unroll
            for (int c = 0; c < 16; ++c) ksg_n[c] = KSG[at(0, 16, c, Np, i)];
        } else {
            s = (F)cand_steps[row];
            Xn = Xc + (size_t)row * row_x;
            Un = Uc + (size_t)row * row_u;
#pragma unroll
            for (int c = 0; c < NS; ++c) x[c] = P.x0[(size_t)c * Np + i];
            load_ref(P, 0, i, xr_n, ur_n);
        }
    }
    // blocks of FUSE_BLOCK steps: in block b the forward warp produces du of steps [b*FUSE_BLOCK, ...) into buffer b & 1 while the rollout
    // warps consume the steps of block b - 1 from the other buffer; one barrier per block, warps run freely inside a block
    const int nsteps = TT - 1, nblk = (nsteps + FUSE_BLOCK - 1) / FUSE_BLOCK;
    for (int b = 0; b <= nblk; ++b) {
        if (fwd) {
            if (act && b < nblk) {
                for (int j = 0; j < FUSE_BLOCK; ++j) {
                    const int tau = b * FUSE_BLOCK + j;
                    if (tau >= nsteps) break;
                    F xx[NS], u[NI], du[NI];
                    forward_du(ksg_n, dx, du, acc);  // (K, sigma, g of this step are dead from here on: their registers take the next step's)
                    DU[at(tau, NI, 0, Np, i)] = du[0];
                    DU[at(tau, NI, 1, Np, i)] = du[1];
                    sdu[b & 1][j][0][lane] = du[0];
                    sdu[b & 1][j][1][lane] = du[1];
                    finish_x(P, tau, i, xraw_n, xx);
#pragma unroll
                    for (int c = 0; c < NI; ++c) u[c] = u_n[c];
                    if (tau + 1 < nsteps) {
                        load_x_raw(X, tau + 1, Np, i, xraw_n);
#pragma unroll
                        for (int c = 0; c < NI; ++c) u_n[c] = U[at(tau + 1, NI, c, Np, i)];
#pragma unroll
                        for (int c = 0; c < 16; ++c) ksg_n[c] = KSG[at(tau + 1, 16, c, Np, i)];
                    }
                    forward_advance(P.M, xx, u, du, dx);
                }
            }
        } else if (act && b >= 1) {
            for (int j = 0; j < FUSE_BLOCK; ++j) {
                const int t = (b - 1) * FUSE_BLOCK + j;
                if (t >= nsteps) break;
                F u[NI], xr[NS], ur[NI];
#pragma unroll
                for (int c = 0; c < NI; ++c) u[c] = u_n[c] + s * sdu[(b - 1) & 1][j][c][lane];  // optcon.py:197 / :253
#pragma unroll
                for (int c = 0; c < NS; ++c) xr[c] = xr_n[c];
#pragma unroll
                for (int c = 0; c < NI; ++c) ur[c] = ur_n[c];
                if (t + 1 < nsteps) {
#pragma unroll
                    for (int c = 0; c < NI; ++c) u_n[c] = U[at(t + 1, NI, c, Np, i)];
                    load_ref(P, t + 1, i, xr_n, ur_n);
                }
                store_x(Xn, t, Np, i, x);
#pragma unroll
                for (int c = 0; c < NI; ++c) Un[at(t, NI, c, Np, i)] = u[c];
                rollout_step<true, Q32>(P.M, P.W, x, u, xr, ur, acc);
            }
        }
        __syncthreads();
    }
    if (!act) return;
    if (fwd) {
        DU[at(TT - 1, NI, 0, Np, i)] = F(0.0);  // uuout[:, TT-1] stays zero (optcon.py:694)
        DU[at(TT - 1, NI, 1, Np, i)] = F(0.0);
        if (status[i] == ST_ACTIVE) descent[i] = acc;
    } else {
        store_x(Xn, TT - 1, Np, i, x);
        Un[at(TT - 1, NI, 0, Np, i)] = F(0.0);  // uu_temp[:, TT-1] is never written (optcon.py:193)
        Un[at(TT - 1, NI, 1, Np, i)] = F(0.0);
        F xr[NS], dxT[NS];
        load_xref(P, TT - 1, i, xr);
#pragma unroll
        for (int c = 0; c < NS; ++c) dxT[c] = x[c] - xr[c];
        acc += (double)term_cost(P.W, dxT);
        Jcand[(size_t)row * Np + i] = acc;
    }
}

// get_update as a copy: the row of the step k_select chose (row armijo_maxiters after exhaustion) becomes the next iterate; thread
// (x = lane, y = time lane), blockIdx.x = position in the tile list, blockIdx.y strides over time.  Jpick[i] = cost of that row.
template <typename F, typename XT>
__global__ void k_pick(TileList L, NewtonOpts O, NewtonState S, const double* __restrict__ cand_steps, const XT* __restrict__ Xc,
                       const F* __restrict__ Uc, size_t row_x, size_t row_u, XT* __restrict__ Xn, F* __restrict__ Un, int N, int Np, int TT,
                       double* __restrict__ Jpick)
{
    const int tile = warp_tile(L, blockIdx.x, Np);
    if (tile < 0) return;
    const int i = tile * TILE + threadIdx.x;
    if (i >= N || S.status[i] != ST_ACTIVE) return;
    const double s = S.step[i];
    int r = O.armijo_maxiters;
    for (int c = 0; c < O.armijo_maxiters; ++c) if (cand_steps[c] == s) { r = c; break; }
    const XT* xs = Xc + (size_t)r * row_x;
    const F* us = Uc + (size_t)r * row_u;
    for (int t = blockIdx.y * blockDim.y + threadIdx.y; t < TT; t += gridDim.y * blockDim.y) {
#pragma unroll
        for (int c = 0; c < NS; ++c) Xn[at(t, NS, c, Np, i)] = xs[at(t, NS, c, Np, i)];
#pragma unroll
        for (int c = 0; c < NI; ++c) Un[at(t, NI, c, Np, i)] = us[at(t, NI, c, Np, i)];
    }
    if (blockIdx.y == 0 && threadIdx.y == 0) Jpick[i] = S.Jcand[(size_t)r * Np + i];
}

// termination test and result-slot bookkeeping after k_pick (a separate launch: k_pick's CTAs read the status it changes)
__global__ void k_finish(NewtonOpts O, NewtonState S, const double* __restrict__ Jpick, int kk, int N)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N && S.status[i] == ST_ACTIVE) newton_finish_instance(O, S, Jpick[i], kk, i);
}

// lazy Armijo, first round: candidate 0 for every active instance, writing the trajectory tentatively into
// the next slot (it IS the update whenever the candidate is accepted)
template <bool Q32, typename F, typename XT>
__global__ void __launch_bounds__(ROLL_THREADS) k_candidate0_write(ProblemT<F> P, WorkList L, const F* __restrict__ U, const F* __restrict__ DU,
                                                                   const double* __restrict__ cand_steps, XT* __restrict__ Xn,
                                                                   F* __restrict__ Un, const int* __restrict__ status,
                                                                   double* __restrict__ Jcand)
{
    const int i = work_instance(L, blockIdx.x * blockDim.x + threadIdx.x, P.N);
    if (i < 0 || status[i] != ST_ACTIVE) return;
    Jcand[i] = rollout_instance<true, true, Q32>(P, U, DU, cand_steps[0], Xn, Un, i);
}

// lazy Armijo: flag the instances whose candidates 0 .. n_tested-1 all failed the test of optcon.py:268
__global__ void k_lazy_need(NewtonOpts O, NewtonState S, const double* __restrict__ cand_steps, int i0, int i1, int Np, int n_tested,
                            int* __restrict__ need)
{
    const int i = i0 + blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= i1) return;
    int nd = 0;
    if (S.status[i] == ST_ACTIVE) {
        const double JP = S.Jcur[i], d = S.descent[i];
        nd = 1;
        for (int c = 0; c < n_tested; ++c)
            if (!(S.Jcand[(size_t)c * Np + i] > JP + O.cc * cand_steps[c] * d)) { nd = 0; break; }
    }
    need[i] = nd;
}

__global__ void k_select(NewtonOpts O, NewtonState S, const double* __restrict__ cand_steps, int kk, int i0, int i1, int Np)
{
    const int i = i0 + blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= i1 || S.status[i] != ST_ACTIVE) return;
    armijo_select_instance(O, S, cand_steps, kk, Np, i);
}

// get_update with the per-instance step + termination bookkeeping.
// only (optional): when non-null, instances with only[i] == 0 keep the trajectory already present in the next
// slot (lazy Armijo: candidate 0 was accepted and is already there) and just run the bookkeeping.
template <bool Q32, typename F, typename XT>
__global__ void __launch_bounds__(ROLL_THREADS) k_update(ProblemT<F> P, WorkList L, NewtonOpts O, NewtonState S, const F* __restrict__ U,
                                                         const F* __restrict__ DU, XT* __restrict__ Xn, F* __restrict__ Un,
                                                         const int* __restrict__ only, int kk, int bookkeeping)
{
    const int i = work_instance(L, blockIdx.x * blockDim.x + threadIdx.x, P.N);
    if (i < 0 || S.status[i] != ST_ACTIVE) return;
    double Jn;
    if (only && !only[i]) Jn = S.Jcand[i];
    else Jn = rollout_instance<true, true, Q32>(P, U, DU, S.step[i], Xn, Un, i);
    if (bookkeeping) newton_finish_instance(O, S, Jn, kk, i);
    else { S.Jcur[i] = Jn; S.iters[i] = kk + 1; }
}

__global__ void k_count_active(const int* __restrict__ status, int N, int* __restrict__ count, long long* __restrict__ iters_sum,
                               const int* __restrict__ iters)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    int a = 0;
    long long it = 0;
    if (i < N) { a = status[i] == ST_ACTIVE; it = iters[i]; }
    for (int o = 16; o; o >>= 1) { a += __shfl_down_sync(0xffffffffu, a, o); it += __shfl_down_sync(0xffffffffu, it, o); }
    if ((threadIdx.x & 31) == 0) {
        if (a) atomicAdd(count, a);
        if (it) atomicAdd((unsigned long long*)iters_sum, (unsigned long long)it);
    }
}

template <bool Q32>
__global__ void __launch_bounds__(ROLL_THREADS) k_track(Problem P, const double* __restrict__ Kt, const double* __restrict__ xopt,
                                                        const double* __restrict__ uopt, const double* __restrict__ xstart,
                                                        double* __restrict__ Xn, double* __restrict__ Un)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P.N) return;
    track_instance<Q32>(P, Kt, xopt, uopt, xstart, Xn, Un, i);
}

// ---- closed-loop tracking of every instance (acoc_track) --------------------------------------------------------------------------
// The nominal of each instance = what acoc_get_result returns (slot per instance, -1 = all zeros, u[TT-1] = u[TT-2], exact row 0), copied
// into dedicated warp-tiled buffers: the lanes of one tile may have their results in different slots, and a warp-private TMA ring copies
// the block of ONE array.  Thread = (instance, chunk of tchunk time steps).
template <typename XT>
__global__ void __launch_bounds__(128) k_track_nominal(const XT* __restrict__ X0, const XT* __restrict__ X1, const XT* __restrict__ X2,
                                                       const double* __restrict__ U0, const double* __restrict__ U1,
                                                       const double* __restrict__ U2, const int* __restrict__ slot,
                                                       const double* __restrict__ x0, XT* __restrict__ Xnom, double* __restrict__ Unom,
                                                       double* __restrict__ xnom0, int N, int Np, int TT, int tchunk)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const int sl = slot[i];
    const XT* X = sl == 0 ? X0 : (sl == 1 ? X1 : X2);
    const double* U = sl == 0 ? U0 : (sl == 1 ? U1 : U2);
    const int t0 = blockIdx.y * tchunk, t1 = min(TT, t0 + tchunk);
    for (int t = t0; t < t1; ++t) {
        const int tu = t == TT - 1 ? TT - 2 : t;  // uu_star[:,-1] = uu_star[:,-2], optcon.py:505
#pragma unroll
        for (int c = 0; c < NS; ++c) Xnom[at(t, NS, c, Np, i)] = sl < 0 ? XT(0) : X[at(t, NS, c, Np, i)];
#pragma unroll
        for (int c = 0; c < NI; ++c) Unom[at(t, NI, c, Np, i)] = sl < 0 ? 0.0 : U[at(tu, NI, c, Np, i)];
    }
    if (blockIdx.y == 0) {
#pragma unroll
        for (int c = 0; c < NS; ++c)
            xnom0[(size_t)c * Np + i] = sl < 0 ? 0.0 : (std::is_same<XT, float>::value ? x0[(size_t)c * Np + i] : (double)X[at(0, NS, c, Np, i)]);
    }
}

// the tracking sweeps with plain global loads (ACOC_NO_TMA): same per-instance functions as the TMA rings
template <int DG, typename XT>
__global__ void __launch_bounds__(64) k_track_gains(Problem P, const XT* __restrict__ Xnom, const double* __restrict__ Unom,
                                                    double* __restrict__ Ktrk, int* __restrict__ n_reg)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P.N) return;
    n_reg[i] = track_gains_instance<DG>(P, Xnom, Unom, Ktrk, i);
}
template <bool Q32, typename XT>
__global__ void __launch_bounds__(64) k_track_rollout(Problem P, const XT* __restrict__ Xnom, const double* __restrict__ Unom,
                                                      const double* __restrict__ Ktrk, const double* __restrict__ delta, XT* __restrict__ Xtrk,
                                                      double* __restrict__ xtrk0, double* __restrict__ Utrk, double* __restrict__ err_max,
                                                      double* __restrict__ err_final)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P.N) return;
    track_rollout_instance<Q32>(P, Xnom, Unom, Ktrk, delta, Xtrk, xtrk0, Utrk, err_max, err_final, i);
}
// the dispersion rollout with plain global loads (ACOC_NO_TMA): thread = (instance i, sample m), g = m * N + i
template <bool Q32, typename XT>
__global__ void __launch_bounds__(64) k_track_mc_rollout(Problem P, const XT* __restrict__ Xnom, const double* __restrict__ Unom,
                                                         const double* __restrict__ Ktrk, const double* __restrict__ delta, long long dstride,
                                                         int M, double* __restrict__ em, double* __restrict__ ef)
{
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= (long long)P.N * M) return;
    const int i = (int)(g % P.N), m = (int)(g / P.N);
    const size_t o = ((size_t)i * M + m) * NS;
    track_mc_sample<Q32>(P, Xnom, Unom, Ktrk, delta + (size_t)i * (size_t)dstride + (size_t)m * NS, i, em + o, ef + o);
}
// per-instance aggregates of the dispersion in sample order; worst / mean [6][Np]
struct TrackTol {
    double v[NS];
    int on;  // 0: no tolerance, n_within is not computed
};
__global__ void __launch_bounds__(128) k_track_mc_reduce(const double* __restrict__ em, const double* __restrict__ ef, int N, int Np, int M,
                                                         TrackTol tol, double* __restrict__ worst, double* __restrict__ mean,
                                                         int* __restrict__ n_within)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    double tl[NS], w[NS], mf[NS];
#pragma unroll
    for (int c = 0; c < NS; ++c) tl[c] = tol.v[c];
    const size_t o = (size_t)i * M * NS;
    const int nw = track_mc_reduce(em + o, ef + o, M, tol.on ? tl : (const double*)nullptr, w, mf);
#pragma unroll
    for (int c = 0; c < NS; ++c) { worst[(size_t)c * Np + i] = w[c]; mean[(size_t)c * Np + i] = mf[c]; }
    n_within[i] = nw;
}

// dx0 and x0_out may alias (each thread reads its dx0 before it writes its x0)
template <bool Q32, typename F, typename XT>
__global__ void __launch_bounds__(ROLL_THREADS) k_init_guess(ProblemT<F> P, double kp, double kt, const F* dx0, XT* __restrict__ Xn,
                                                             F* __restrict__ Un, F* x0_out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P.N) return;
    init_guess_instance<Q32>(P, (F)kp, (F)kt, dx0, Xn, Un, x0_out, i);
}

__global__ void k_step_batch(Model M, int q32, int n, const double* __restrict__ x, const double* __restrict__ u,
                             const double* __restrict__ lam, double* xxp, double* A, double* B, double* fxx, double* fux)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    double xs[NS], us[NI], ls[NS];
    for (int c = 0; c < NS; ++c) xs[c] = x[(size_t)s * NS + c];
    for (int c = 0; c < NI; ++c) us[c] = u[(size_t)s * NI + c];
    if (lam) for (int c = 0; c < NS; ++c) ls[c] = lam[(size_t)s * NS + c];
    const size_t nxx = lam ? 36 : 216, nux = lam ? 12 : 72;
    step_sample(M, q32 != 0, xs, us, lam ? ls : nullptr, xxp ? xxp + (size_t)s * NS : nullptr, A ? A + (size_t)s * 36 : nullptr,
                B ? B + (size_t)s * 12 : nullptr, fxx ? fxx + s * nxx : nullptr, fux ? fux + s * nux : nullptr);
}

__global__ void k_cost_batch(Weights W, int n, const double* __restrict__ x, const double* __restrict__ u, const double* __restrict__ xr,
                             const double* __restrict__ ur, double* ll, double* lx, double* lu, double* llT, double* lTx)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    double l1 = 0, l2 = 0, gx[NS], gu[NI], gT[NS];
    cost_sample(W, x + (size_t)s * NS, u ? u + (size_t)s * NI : nullptr, xr + (size_t)s * NS, ur ? ur + (size_t)s * NI : nullptr,
                (u && (ll || lx || lu)) ? &l1 : nullptr, gx, gu, (llT || lTx) ? &l2 : nullptr, gT);
    if (ll) ll[s] = l1;
    if (lx) for (int c = 0; c < NS; ++c) lx[(size_t)s * NS + c] = gx[c];
    if (lu) for (int c = 0; c < NI; ++c) lu[(size_t)s * NI + c] = gu[c];
    if (llT) llT[s] = l2;
    if (lTx) for (int c = 0; c < NS; ++c) lTx[(size_t)s * NS + c] = gT[c];
}

template <int N>
__global__ void k_lq_dense(int nb, int TT, const double* A, const double* B, const double* Q, const double* R, const double* S,
                           const double* Qf, const double* x0, const double* q, const double* r, const double* qf, double* K, double* P,
                           double* xout, double* uout, int* n_reg)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nb) return;
    const size_t t = (size_t)b * TT;
    lq_dense_problem<N>(TT, A + t * 36, B + t * 12, Q + t * 36, R + t * 4, S + t * 12, Qf + (size_t)b * 36, x0 + (size_t)b * NS,
                        q ? q + t * NS : nullptr, r ? r + t * NI : nullptr, qf ? qf + (size_t)b * NS : nullptr, K + t * NI * N,
                        P ? P + t * N * N : nullptr, xout + t * NS, uout + t * NI, n_reg ? n_reg + b : nullptr);
}

// ---- layout conversion: host (n, C, TT) chunk  <->  SoA [TT][C][Np] ------------------------------------
// D: device element type.  row0 (optional, [C][Np] of R0): receives the t = 0 column exactly (x0 = xx_init[:,0], optcon.py:398).
// inexact (optional): set to 1 when a value at t >= 1 does not survive the conversion to D (float state slots).
template <typename D, typename R0>
__global__ void k_to_soa(const double* __restrict__ src, D* __restrict__ dst, int n0, int nchunk, int C, int TT, int Np, R0* __restrict__ row0,
                         int* __restrict__ inexact)
{
    __shared__ double tile[32][33];
    const int c = blockIdx.z, tb = blockIdx.x * 32, nb = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int n = nb + r, t = tb + threadIdx.x;
        if (n < nchunk && t < TT) tile[r][threadIdx.x] = src[((size_t)n * C + c) * TT + t];
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int t = tb + r, n = nb + threadIdx.x;
        if (n < nchunk && t < TT) {
            const double v = tile[threadIdx.x][r];
            const D d = (D)v;
            dst[Np == 1 ? (size_t)t * C + c : at(t, C, c, Np, n0 + n)] = d;  // Np == 1: a shared reference, plain [TT][C]
            if (row0 && t == 0) row0[(size_t)c * Np + n0 + n] = (R0)v;
            if (inexact && t >= 1 && !((double)d == v) && v == v) *inexact = 1;
        }
    }
}

// s0..s2: up to three source slots; slot[i] selects per instance (-1 -> zeros; NULL -> s0); dup_last: t = TT-1 reads TT-2
// row0 (optional, [C][Np]): exact t = 0 column of float state slots (see acoc_kernels.cuh "Types")
// O: element type of the host-side chunk (double: the reference's layout; float: the lossless float32 download of float state slots)
template <typename D, typename O>
__global__ void k_from_soa(const D* __restrict__ s0, const D* __restrict__ s1, const D* __restrict__ s2, const int* __restrict__ slot,
                           const double* __restrict__ row0, O* __restrict__ dst, int n0, int nchunk, int C, int TT, int Np, int dup_last)
{
    __shared__ O tile[32][33];
    const int c = blockIdx.z, tb = blockIdx.x * 32, nb = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        int t = tb + r;
        const int n = nb + threadIdx.x;
        if (n < nchunk && t < TT) {
            if (dup_last && t == TT - 1 && TT > 1) t = TT - 2;
            const int sl = slot ? slot[n0 + n] : 0;
            const D* s = sl == 0 ? s0 : (sl == 1 ? s1 : s2);
            tile[r][threadIdx.x] = sl < 0 ? O(0) : ((row0 && t == 0) ? (O)row0[(size_t)c * Np + n0 + n] : (O)s[Np == 1 ? (size_t)t * C + c : at(t, C, c, Np, n0 + n)]);
        }
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int n = nb + r, t = tb + threadIdx.x;
        if (n < nchunk && t < TT) dst[((size_t)n * C + c) * TT + t] = tile[threadIdx.x][r];
    }
}

// ---- result delivery straight into page-locked host memory ----------------------------------------------------------------------
// What optimize() returns (optcon.py:503-505) for every instance of this context whose status is FINAL, written into the caller's
// (N, C, TT) array at row uidx[n] (the instance's index in the caller's batch; NULL: identity) by the layout-conversion kernel itself:
// dst is the device alias of page-locked host memory, so no staging buffer, no separate copy, and any subset of instances costs only
// its own bytes.  acoc_newton_solve_deliver launches it for a batch's finished instances at the moment the still-iterating ones move
// on to a survivor generation, so that the transfer overlaps the latency-bound tail of the solve.
// row0 (optional, [C][Np]): exact t = 0 column of float state slots; dup_last: t = TT-1 reads TT-2 (uu_star[:,-1] = uu_star[:,-2]).
// rows[n]: destination row of instance n in this delivery, or -1 (k_deliver_select)
template <typename D, typename O>
__global__ void k_deliver(const D* __restrict__ s0, const D* __restrict__ s1, const D* __restrict__ s2, const int* __restrict__ result_slot,
                          const int* __restrict__ rows, const double* __restrict__ row0, O* __restrict__ dst,
                          int N, int C, int TT, int Np, int dup_last)
{
    // A small persistent grid (64 CTAs) walks the (instance tile, time tile, component) blocks.  The stores drain at the speed of the
    // host link and back up in the memory pipe of the SMs that issue them; on every SM they slow the solver's own kernels -- the
    // latency-bound tail this transfer is meant to hide behind -- by 3x, on 64 of the 148 SMs by a quarter, at 35 of the 40 GB/s the
    // machine-filling grid reaches.
    __shared__ O tile[32][33];
    __shared__ int row_of[32];
    const int nt = (TT + 31) / 32, nn = (N + 31) / 32;
    const long long nblk = (long long)nn * nt * C;
    for (long long blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
        const int c = (int)(blk % C), tb = (int)((blk / C) % nt) * 32, nb = (int)(blk / ((long long)C * nt)) * 32;
        int mine = 0;
        __syncthreads();  // (the previous block's tile / row_of have been read)
        if (threadIdx.y == 0) {
            const int n = nb + threadIdx.x;
            const int row = n < N ? rows[n] : -1;
            row_of[threadIdx.x] = row;
            mine = row >= 0;
        }
        if (!__syncthreads_or(mine)) continue;  // no finished instance in this tile
        for (int r = threadIdx.y; r < 32; r += blockDim.y) {
            int t = tb + r;
            const int n = nb + threadIdx.x;
            if (n < N && t < TT && row_of[threadIdx.x] >= 0) {
                if (dup_last && t == TT - 1 && TT > 1) t = TT - 2;
                const int sl = result_slot[n];
                const D* s = sl == 0 ? s0 : (sl == 1 ? s1 : s2);
                tile[r][threadIdx.x] = sl < 0 ? O(0) : ((row0 && t == 0) ? (O)row0[(size_t)c * Np + n] : (O)s[at(t, C, c, Np, n)]);
            }
        }
        __syncthreads();
        for (int r = threadIdx.y; r < 32; r += blockDim.y) {
            const int t = tb + threadIdx.x, row = row_of[r];
            if (row >= 0 && t < TT) dst[((size_t)row * C + c) * TT + t] = tile[threadIdx.x][r];
        }
    }
}

// the instances of a context that are final and have not been delivered yet: rows[n] = their row in the caller's batch (uidx; NULL:
// identity), else -1; marks them delivered.  Runs on the SOLVER's stream between two calls of the lock-step driver, so it sees a
// consistent snapshot; the trajectories of a final instance never change again, so the delivery itself may run beside later iterations.
__global__ void k_deliver_select(const int* __restrict__ status, const int* __restrict__ uidx, int* __restrict__ delivered, int* __restrict__ rows,
                                 int* __restrict__ count, int N)
{
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const int st = status[n];
    int row = -1;
    if ((st == ST_CONVERGED || st == ST_MAXITER || st == ST_NONFINITE) && !delivered[n]) {
        row = uidx ? uidx[n] : n;
        delivered[n] = 1;
        atomicAdd(count, 1);
    }
    rows[n] = row;
}

// index of a child generation's instances in the caller's batch: uidx_child[j] = uidx_parent[origin[j]] (parent NULL: the root, identity)
__global__ void k_compose_uidx(const int* __restrict__ origin, const int* __restrict__ uidx_parent, int* __restrict__ uidx_child, int n)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) { const int o = origin[j]; uidx_child[j] = uidx_parent ? uidx_parent[o] : o; }
}

// ---- reference generators of the scripts, on the device (SURVEY.md 8(f) N2) ---------------------------------------------------
// xref / uref of instance i from per-instance parameters and shared time bases, in the operation order of the scripts' numpy code
// (main_newton_method.py:96-142, acrobatic_newton.py:99-154; restated in refgen.py) so that the result is bit-identical to it:
//   X_t = x0 + vx_i * tt_t            (x0 = 0)                      Z_t = p0 + zshape_t * (zf_i - p0)   (p0 = 0)
//   V_t = ((vshape_t * zf_i)**2 + vx_i**2)**0.5  (numpy: square, square, add, sqrt), or the constant xc[2] when vshape == NULL
//   theta, q, gamma = xc[3..5];  uref = uc[0..1]
struct RefConst { double xc[6], uc[2]; };
template <typename F>
__global__ void __launch_bounds__(128) k_gen_refs(int N, int Np, int TT, const double* __restrict__ tt, const double* __restrict__ zshape,
                                                  const double* __restrict__ vshape, const double* __restrict__ zf, const double* __restrict__ vx,
                                                  RefConst K, F* __restrict__ xref, F* __restrict__ uref)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const double z = zf[i], v = vx[i], v2 = v * v;
    for (int t = blockIdx.y; t < TT; t += gridDim.y) {
        const double X = 0.0 + v * tt[t];
        const double Z = 0.0 + zshape[t] * (z - 0.0);
        double V = K.xc[2];
        if (vshape) { const double zd = vshape[t] * (z - 0.0); V = sqrt(zd * zd + v2); }
        F* xo = xref + at(t, NS, 0, Np, i);
        xo[0] = (F)X; xo[TILE] = (F)Z; xo[2 * TILE] = (F)V; xo[3 * TILE] = (F)K.xc[3]; xo[4 * TILE] = (F)K.xc[4]; xo[5 * TILE] = (F)K.xc[5];
        F* uo = uref + at(t, NI, 0, Np, i);
        uo[0] = (F)K.uc[0]; uo[TILE] = (F)K.uc[1];
    }
}

// compact storage of the same references: only the speed reference is a per-instance array ([TT][Np/32][1][32]); X and Z are formed
// in the sweeps from the tables (ProblemT, "parametric references").  Same expression as k_gen_refs: bit-identical values.
__global__ void __launch_bounds__(128) k_gen_vref(int N, int Np, int TT, const double* __restrict__ vshape, const double* __restrict__ zf,
                                                  const double* __restrict__ vx, double* __restrict__ vref)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const double z = zf[i], v = vx[i], v2 = v * v;
    for (int t = blockIdx.y; t < TT; t += gridDim.y) {
        const double zd = vshape[t] * (z - 0.0);
        vref[at(t, 1, 0, Np, i)] = sqrt(zd * zd + v2);
    }
}

// parametric references written out in the expanded layout (acoc_get_refs)
__global__ void __launch_bounds__(128) k_expand_refs(Problem P, double* __restrict__ xref, double* __restrict__ uref)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P.N) return;
    for (int t = blockIdx.y; t < P.TT; t += gridDim.y) {
        double xr[NS], ur[NI];
        load_ref(P, t, i, xr, ur);
#pragma unroll
        for (int c = 0; c < NS; ++c) xref[at(t, NS, c, P.Np, i)] = xr[c];
#pragma unroll
        for (int c = 0; c < NI; ++c) uref[at(t, NI, c, P.Np, i)] = ur[c];
    }
}

__global__ void k_fill_int(int* p, int n, int v_lo, int n_lo, int v_hi)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = i < n_lo ? v_lo : v_hi;
}

// slot of the (which = 0: newest, 1: previous) iterate of every instance: iterate k lives in slot k % 3 and a finished
// instance stopped at its own iteration count
__global__ void k_iterate_slot(const int* __restrict__ iters, int which, int* __restrict__ slot_out, int N)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) { const int k = iters[i] - which; slot_out[i] = k < 0 ? -1 : k % 3; }
}

__global__ void k_result_slot_default(const int* __restrict__ status, int* __restrict__ slot_out, const int* __restrict__ result_slot,
                                      int newest, int N)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) slot_out[i] = status[i] == ST_ACTIVE ? newest : result_slot[i];
}

// ---- survivor generations (acoc_newton_solve) ----------------------------------------------------------
// When at most half of a batch is still iterating, the survivors are gathered into a smaller child context so that
// every lane of every warp does useful work again (the instances are independent; the parent keeps the finished
// ones untouched).  origin[j] = index in the parent of child instance j.
constexpr int ST_MOVED = 5;  // the instance continues in a child generation

// element (row r, instance i) of a per-instance array: C == 0 -> plain [rows][Np]; C > 0 -> warp-tiled trajectory with C components,
// row r = t*C + c
__device__ __forceinline__ size_t row_elem(int r, int C, int Np, int i)
{
    return C == 0 ? (size_t)r * Np + i : at(r / C, C, r % C, Np, i);
}

// dst[row][j] = src[row][origin[j]]   (coalesced writes, scattered reads)
template <typename T>
__global__ void k_gather_rows(const T* __restrict__ src, int src_stride, T* __restrict__ dst, int dst_stride, const int* __restrict__ origin,
                              int n, int rows, int C)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const int o = origin[j];
    for (int r = blockIdx.y; r < rows; r += gridDim.y) dst[row_elem(r, C, dst_stride, j)] = src[row_elem(r, C, src_stride, o)];
}

// dst[row][origin[j]] = src[row][j]   (fold a finished child generation back into its parent)
template <typename T>
__global__ void k_scatter_rows(const T* __restrict__ src, int src_stride, T* __restrict__ dst, int dst_stride, const int* __restrict__ origin,
                               int n, int rows, int C)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const int o = origin[j];
    for (int r = blockIdx.y; r < rows; r += gridDim.y) dst[row_elem(r, C, dst_stride, o)] = src[row_elem(r, C, src_stride, j)];
}

__global__ void k_mark_moved(int* __restrict__ status, const int* __restrict__ origin, int n)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) status[origin[j]] = ST_MOVED;
}

// ---- microbenchmarks for the roofline denominators ----------------------------------------------------
__global__ void k_fp64_peak(double* out, int iters, double seed)
{
    double a0 = seed + threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double b = 1.0000001, c = 1e-9;
    for (int i = 0; i < iters; ++i) {
        a0 = fma(a0, b, c); a1 = fma(a1, b, c); a2 = fma(a2, b, c); a3 = fma(a3, b, c);
        a4 = fma(a4, b, c); a5 = fma(a5, b, c); a6 = fma(a6, b, c); a7 = fma(a7, b, c);
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}

// one warp, one chain of dependent DFMAs: cycles per dependent FP64 operation (the sweeps are bound by this, DESIGN.md 4)
__global__ void k_fp64_latency(double* out, long long* cycles, int iters, double seed)
{
    double a = seed + threadIdx.x;
    const double b = 1.0000001, c = 1e-9;
    const long long t0 = clock64();
#pragma unroll 16
    for (int i = 0; i < iters; ++i) a = fma(a, b, c);
    const long long t1 = clock64();
    out[threadIdx.x] = a;
    if (threadIdx.x == 0) *cycles = t1 - t0;
}

__global__ void k_copy(const double2* __restrict__ a, double2* __restrict__ b, size_t n)
{
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) b[i] = a[i];
}

// ======================================================================================================
// context
// ======================================================================================================
constexpr int MAX_RANGES = 8;  // independent tile ranges of a fully active batch (acoc_newton_iterate)

struct acoc_ctx {
    int device = 0, N = 0, Np = 0, TT = 0;
    unsigned flags = 0;
    cudaStream_t stream = nullptr;
    Problem P;   // float64 master copy of model, weights and sizes; the typed view handed to kernels is built by prob<F>()
    NewtonOpts O;
    NewtonState S;
    bool have_model = false, have_weights = false, have_refs = false, have_init = false;
    int kk = 0;  // Newton iterations (loop bodies) executed by the lock-step driver
    // element types of the device buffers: F = float iff fp32 (else double) for U, DU, KSG, references, x0;
    // the state slots X hold float iff x_float (FP32 mode, or float32-quantised states that are exactly representable)
    bool fp32 = false, x_float = false;
    void *X[3] = {nullptr, nullptr, nullptr}, *U[3] = {nullptr, nullptr, nullptr};
    void *DU = nullptr, *KSG = nullptr, *xref = nullptr, *uref = nullptr, *x0 = nullptr;
    // parametric references (acoc_set_refs_generated): shared tables [TT], per-instance parameters [Np], stored speed reference
    void *rp_tt = nullptr, *rp_zs = nullptr, *rp_zf = nullptr, *rp_vx = nullptr, *rp_v = nullptr;
    bool rp_has_v = false;
    double* cand_steps = nullptr;
    double* stage = nullptr;  // device staging for layout conversion (always float64: the host side of the ABI)
    size_t stage_doubles = 0;
    int *need = nullptr, *need2 = nullptr, *counters = nullptr, *slot_tmp = nullptr;
    int *act_groups = nullptr, *need_groups = nullptr, *need_groups2 = nullptr;  // work lists (see WorkList); counts live in counters[1], counters[2]
    long long* iters_sum = nullptr;
    std::vector<std::pair<void*, size_t>> allocs;
    unsigned long long bytes = 0;
    int hist_iters = 0, hist_cand = 0;  // sizes the history / candidate-cost buffers were allocated for
    // timing
    bool profiling = false;
    cudaEvent_t ev[8];
    bool ev_ok = false;
    double total_ms = 0, phase_ms[6] = {0, 0, 0, 0, 0, 0};
    long long launches = 0;
    bool weights_sym = true;
    // survivor generations (see acoc_newton_solve)
    acoc_ctx* child = nullptr;  // reusable smaller context (capacity N/2) for the instances that are still iterating
    int* origin = nullptr;      // [capacity] index in the PARENT of each instance of this context (child contexts only)
    int* uidx = nullptr;        // [capacity] index in the caller's batch (child contexts during acoc_newton_solve_deliver)
    int *delivered = nullptr, *deliver_rows = nullptr;  // [capacity] delivery bookkeeping of acoc_newton_solve_deliver
    cudaEvent_t ev_deliver = nullptr;
    int n_delivered = 0;        // instances of this context handed to the delivery stream so far (host-side count)
    cudaStream_t dstream = nullptr;  // result delivery (root context)
    int cap = 0;                // instance capacity (N may be smaller in a child)
    int spawn_kk = 0;           // iteration at which this child took over its instances
    double gen_ms = 0;          // device time spent moving instances between generations in the last solve
    // launch scope of the sweep kernels: stream and range of the tile list (see acoc_newton_iterate, "two ranges")
    cudaStream_t ls_stream = nullptr;
    int ls_off = 0, ls_end = 0x7fffffff;
    bool ls_identity = false;
    int ls_range = 0;           // index of the current range (its need-list counter)
    cudaStream_t rstream[MAX_RANGES] = {};  // streams of ranges 1.. (range 0 uses `stream`)
    cudaEvent_t ev_fork = nullptr, ev_join[MAX_RANGES] = {};
    int stream_priority = 0;    // CUDA priority of the context's streams (ACOC_PRIORITY)
    int last_need = -1;         // instances whose candidate 0 failed in the last iteration of the previous call (lazy search); -1: unknown
    int sm_count = 0;
    bool all_active = false;    // more than half of the instances were active at the last host-side count (reset: all of them)
    int bwd_wave_ctas = 0;      // CTAs of the backward sweep that are resident at once on this device (occupancy x SMs)
    // small batches: one trajectory slot per Armijo candidate (+ the exhausted step), see k_search_fused
    void *candX = nullptr, *candU = nullptr;
    double* candJ = nullptr;    // [Np] cost of the row k_pick copied
    size_t cand_bytes_x = 0, cand_bytes_u = 0;
    bool cand_failed = false;   // the buffers could not be allocated: separate sweeps
    // closed-loop tracking (acoc_track, acoc_lqr_tracking_many), allocated on the first call: nominal Xnom / Unom + exact row 0, gains
    // Ktrk, tracked Xtrk / Utrk + exact row 0 (warp-tiled), delta and summaries [6][Np], n_reg [Np].  State buffers hold tk_es-byte elements.
    void *tk_xnom = nullptr, *tk_unom = nullptr, *tk_xnom0 = nullptr, *tk_K = nullptr, *tk_x = nullptr, *tk_x0 = nullptr, *tk_u = nullptr;
    void *tk_delta = nullptr, *tk_emax = nullptr, *tk_efin = nullptr;
    int* tk_nreg = nullptr;
    size_t tk_es = 0;           // 0: not allocated
    bool tk_done = false, tk_xfloat = false;  // Xtrk holds the result of acoc_track; its element type
    bool tk_swept = false;      // Ktrk and tk_ms hold the result of acoc_track or acoc_track_mc
    // dispersion (acoc_track_mc), allocated on the first call and grown with N*M: per-sample summaries em | ef [2][N][M][6], the
    // deltas as given ((M,6) or (N,M,6)), n_within [Np]; capacities in bytes
    void *mc_sum = nullptr, *mc_delta = nullptr;
    int* mc_nw = nullptr;
    size_t mc_sum_cap = 0, mc_delta_cap = 0;
    cudaEvent_t tk_ev[4] = {};
    double tk_ms[4] = {0, 0, 0, 0};
};

static int dalloc_bytes(acoc_ctx* c, void** p, size_t bytes)
{
    void* q = nullptr;
    cudaError_t e = cudaMalloc(&q, bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();  // clear the per-thread error state: the caller decides what an allocation failure means
        return fail(ACOC_ERR_NOMEM, "cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
    }
    e = cudaMemsetAsync(q, 0, bytes, c->stream);
    if (e != cudaSuccess) return fail(ACOC_ERR_CUDA, "cudaMemset failed: %s", cudaGetErrorString(e));
    c->allocs.push_back({q, bytes});
    c->bytes += bytes;
    *p = q;
    return 0;
}
// release one buffer of the context before the context itself goes away (option changes resize the histories)
template <typename T>
static void dfree(acoc_ctx* c, T** p)
{
    if (!*p) return;
    for (size_t k = 0; k < c->allocs.size(); ++k)
        if (c->allocs[k].first == (void*)*p) {
            c->bytes -= c->allocs[k].second;
            c->allocs.erase(c->allocs.begin() + k);
            break;
        }
    cudaFree(*p);
    *p = nullptr;
}
template <typename T>
static int dalloc(acoc_ctx* c, T** p, size_t n)
{
    void* q = nullptr;
    const int rc = dalloc_bytes(c, &q, n * sizeof(T));
    *p = (T*)q;
    return rc;
}
// typed view of the problem for the kernels
template <typename F>
static ProblemT<F> prob(const acoc_ctx* c)
{
    ProblemT<F> P;
    P.M = model_as<F>(c->P.M);
    P.W = weights_as<F>(c->P.W);
    P.N = c->P.N; P.Np = c->P.Np; P.TT = c->P.TT; P.q32 = c->P.q32; P.ref_shared = c->P.ref_shared;
    P.xref = (const F*)c->xref; P.uref = (const F*)c->uref; P.x0 = (const F*)c->x0;
    P.ref_param = c->P.ref_param;
    P.rp_tt = (const F*)c->rp_tt; P.rp_zs = (const F*)c->rp_zs; P.rp_zf = (const F*)c->rp_zf; P.rp_vx = (const F*)c->rp_vx;
    P.rp_v = c->rp_has_v ? (const F*)c->rp_v : nullptr;
    for (int k = 0; k < NS; ++k) P.rp_xc[k] = (F)c->P.rp_xc[k];
    for (int k = 0; k < NI; ++k) P.rp_uc[k] = (F)c->P.rp_uc[k];
    return P;
}
#define TRY(x) do { int rc__ = (x); if (rc__) return rc__; } while (0)

static int use_device(int device)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) return fail(ACOC_ERR_CUDA, "no CUDA device available (%s): libacoc has no CPU fallback", e == cudaSuccess ? "count = 0" : cudaGetErrorString(e));
    if (device < 0 || device >= n) return fail(ACOC_ERR_INVALID, "device %d out of range (0..%d)", device, n - 1);
    CK(cudaSetDevice(device));
    return 0;
}

static void default_opts(NewtonOpts* o)
{
    o->max_iters = 200; o->armijo_maxiters = 10; o->exact_after = 8;
    o->stepsize_0 = 1.0; o->cc = 0.5; o->beta = 0.7; o->term_cond = -1e-6; o->method = 0;
}

// the Armijo step table cand_steps[c] = stepsize_0 * beta^c (length armijo_maxiters + 1), on the context's stream
static int write_cand_steps(acoc_ctx* c)
{
    std::vector<double> cs(c->O.armijo_maxiters + 1);
    double s = c->O.stepsize_0;
    for (int k = 0; k <= c->O.armijo_maxiters; ++k) { cs[k] = s; s = c->O.beta * s; }  // stepsize = beta*stepsize, optcon.py:270
    CK(cudaMemcpyAsync(c->cand_steps, cs.data(), cs.size() * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

// histories [max_iters][Np] and candidate costs [armijo_maxiters + 1][Np]: (re)allocated when the option that sizes them changes
static int alloc_history(acoc_ctx* c)
{
    const size_t Np = c->Np;
    if (c->hist_iters != c->O.max_iters) {
        CK(cudaStreamSynchronize(c->stream));
        dfree(c, &c->S.hist_J); dfree(c, &c->S.hist_descent); dfree(c, &c->S.hist_step); dfree(c, &c->S.hist_ncand);
        c->hist_iters = 0;
        TRY(dalloc(c, &c->S.hist_J, (size_t)c->O.max_iters * Np));
        TRY(dalloc(c, &c->S.hist_descent, (size_t)c->O.max_iters * Np));
        TRY(dalloc(c, &c->S.hist_step, (size_t)c->O.max_iters * Np));
        TRY(dalloc(c, &c->S.hist_ncand, (size_t)c->O.max_iters * Np));
        c->hist_iters = c->O.max_iters;
    }
    if (c->hist_cand != c->O.armijo_maxiters) {
        CK(cudaStreamSynchronize(c->stream));
        dfree(c, &c->S.Jcand); dfree(c, &c->cand_steps);
        c->hist_cand = 0;
        TRY(dalloc(c, &c->S.Jcand, (size_t)(c->O.armijo_maxiters + 1) * Np));
        TRY(dalloc(c, &c->cand_steps, (size_t)c->O.armijo_maxiters + 2));
        c->hist_cand = c->O.armijo_maxiters;
    }
    return write_cand_steps(c);
}

static int reset_state(acoc_ctx* c)
{
    const int Np = c->Np, N = c->N;
    k_fill_int<<<(Np + 255) / 256, 256, 0, c->stream>>>(c->S.status, Np, ST_ACTIVE, N, ST_PAD);
    CK(cudaMemsetAsync(c->S.iters, 0, Np * sizeof(int), c->stream));
    CK(cudaMemsetAsync(c->S.n_reg, 0, Np * sizeof(int), c->stream));
    CK(cudaMemsetAsync(c->S.result_slot, 0, Np * sizeof(int), c->stream));
    CK(cudaMemsetAsync(c->S.Jcur, 0, Np * sizeof(double), c->stream));
    CK(cudaMemsetAsync(c->S.descent, 0, Np * sizeof(double), c->stream));
    CK(cudaMemsetAsync(c->S.step, 0, Np * sizeof(double), c->stream));
    // histories start from zero so that rows beyond an instance's own iteration count never show an earlier solve
    const size_t hrows = (size_t)c->O.max_iters * Np;
    CK(cudaMemsetAsync(c->S.hist_J, 0, hrows * sizeof(double), c->stream));
    CK(cudaMemsetAsync(c->S.hist_descent, 0, hrows * sizeof(double), c->stream));
    CK(cudaMemsetAsync(c->S.hist_step, 0, hrows * sizeof(double), c->stream));
    CK(cudaMemsetAsync(c->S.hist_ncand, 0, hrows * sizeof(int), c->stream));
    CK(cudaGetLastError());
    c->kk = 0;
    c->all_active = true;
    c->last_need = -1;
    return 0;
}

// host (n,C,TT) float64 -> SoA of D, chunked through the staging buffer.  row0 / inexact: see k_to_soa.
template <typename D, typename R0>
static int upload_soa_t(acoc_ctx* c, const double* host, void* dst, int n, int C, int Np, R0* row0, int* inexact)
{
    const int TT = c->TT;
    const size_t per = (size_t)C * TT;
    int chunk = (int)std::min<size_t>((size_t)n, std::max<size_t>(1, c->stage_doubles / per));
    for (int n0 = 0; n0 < n; n0 += chunk) {
        const int nc = std::min(chunk, n - n0);
        CK(cudaMemcpyAsync(c->stage, host + (size_t)n0 * per, (size_t)nc * per * sizeof(double), cudaMemcpyHostToDevice, c->stream));
        dim3 grid((TT + 31) / 32, (nc + 31) / 32, C), block(32, 8);
        k_to_soa<D, R0><<<grid, block, 0, c->stream>>>(c->stage, (D*)dst, n0, nc, C, TT, Np, row0, inexact);
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(c->stream));  // the staging buffer is reused by the next chunk
    }
    return 0;
}
// buffers of the context's arithmetic type F (inputs, references, gains)
static int upload_soa(acoc_ctx* c, const double* host, void* dst, int n, int C, int Np)
{
    return c->fp32 ? upload_soa_t<float, float>(c, host, dst, n, C, Np, nullptr, nullptr)
                   : upload_soa_t<double, double>(c, host, dst, n, C, Np, nullptr, nullptr);
}

template <typename D, typename O = double>
static int download_soa_t(acoc_ctx* c, const void* s0, const void* s1, const void* s2, const int* slot, const double* row0, O* host, int n,
                          int C, int Np, int dup_last)
{
    const int TT = c->TT;
    const size_t per = (size_t)C * TT;
    int chunk = (int)std::min<size_t>((size_t)n, std::max<size_t>(1, c->stage_doubles * (sizeof(double) / sizeof(O)) / per));
    for (int n0 = 0; n0 < n; n0 += chunk) {
        const int nc = std::min(chunk, n - n0);
        dim3 grid((TT + 31) / 32, (nc + 31) / 32, C), block(32, 8);
        k_from_soa<D, O><<<grid, block, 0, c->stream>>>((const D*)s0, (const D*)s1, (const D*)s2, slot, row0, (O*)c->stage, n0, nc, C, TT, Np, dup_last);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(host + (size_t)n0 * per, c->stage, (size_t)nc * per * sizeof(O), cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
    }
    return 0;
}
// buffers of type F
static int download_soa(acoc_ctx* c, const void* s0, const void* s1, const void* s2, const int* slot, double* host, int n, int C, int Np,
                        int dup_last)
{
    return c->fp32 ? download_soa_t<float>(c, s0, s1, s2, slot, nullptr, host, n, C, Np, dup_last)
                   : download_soa_t<double>(c, s0, s1, s2, slot, nullptr, host, n, C, Np, dup_last);
}
// state slots (element type by x_float; exact t = 0 column from x0 when the slots are float but the arithmetic is float64)
static int download_x(acoc_ctx* c, const int* slot, double* host)
{
    if (!c->x_float) return download_soa_t<double>(c, c->X[0], c->X[1], c->X[2], slot, nullptr, host, c->N, 6, c->Np, 0);
    return download_soa_t<float>(c, c->X[0], c->X[1], c->X[2], slot, c->fp32 ? nullptr : (const double*)c->x0, host, c->N, 6, c->Np, 0);
}

static bool is_diag(const double* M, int n)
{
    for (int i = 0; i < n; ++i) for (int j = 0; j < n; ++j) if (i != j && M[i * n + j] != 0.0) return false;
    return true;
}
static bool is_sym(const double* M, int n)
{
    for (int i = 0; i < n; ++i) for (int j = 0; j < i; ++j) if (M[i * n + j] != M[j * n + i]) return false;
    return true;
}
static void fill_weights(Weights* W, const double* Q, const double* R, const double* QT)
{
    memcpy(W->Q, Q, sizeof(W->Q)); memcpy(W->R, R, sizeof(W->R)); memcpy(W->QT, QT, sizeof(W->QT));
    W->diag = is_diag(Q, 6) && is_diag(R, 2) && is_diag(QT, 6);
}

// ======================================================================================================
// C ABI -- library
// ======================================================================================================
// (the functions below are declared extern "C" in acoc.h, which gives these definitions C linkage)

int acoc_version(void) { return ACOC_VERSION; }

const char* acoc_last_error(void) { return g_err.c_str(); }

int acoc_device_count(int* count)
{
    REQUIRE(count, "count is NULL");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) { *count = 0; return fail(ACOC_ERR_CUDA, "cudaGetDeviceCount: %s", cudaGetErrorString(e)); }
    *count = n;
    return 0;
}

int acoc_device_info(int device, char* name, int len, int* sm_count, unsigned long long* mem_bytes, int* cc)
{
    TRY(use_device(device));
    cudaDeviceProp p;
    CK(cudaGetDeviceProperties(&p, device));
    if (name && len > 0) { strncpy(name, p.name, len - 1); name[len - 1] = 0; }
    if (sm_count) *sm_count = p.multiProcessorCount;
    if (mem_bytes) *mem_bytes = p.totalGlobalMem;
    if (cc) *cc = p.major * 10 + p.minor;
    return 0;
}

// ======================================================================================================
// pointwise entry points
// ======================================================================================================
// Device scratch of the pointwise entry points (acoc_step_batch, acoc_cost_batch, acoc_ltv_lqr, acoc_lqr_tracking): one cached
// arena per device, carved up by bump allocation, so that a call costs no cudaMalloc / cudaFree once the arena has grown to the
// call's size (a Dynamics.step of one sample was ~10 allocations + frees before).  Calls that do not fit take individual
// allocations for the overflow and the arena is regrown for the next call.  The arena lock makes these entry points serialise
// per process; the batched contexts do not use it.
struct Arena { char* base = nullptr; size_t cap = 0; };
static std::mutex g_arena_mu;
static Arena g_arena[64];

struct TmpBuf {
    std::unique_lock<std::mutex> lk;
    Arena* a;
    size_t used = 0, want = 0;
    std::vector<void*> extra;
    explicit TmpBuf(int device) : lk(g_arena_mu), a(&g_arena[device & 63]) {}
    ~TmpBuf()
    {
        for (void* q : extra) cudaFree(q);
        if (want > a->cap) {  // regrow for the next call of this size (the work of this call has been synchronised by DOWN / sync)
            cudaDeviceSynchronize();
            if (a->base) cudaFree(a->base);
            a->base = nullptr; a->cap = 0;
            void* q = nullptr;
            const size_t cap = want + want / 4 + 4096;
            if (cudaMalloc(&q, cap) == cudaSuccess) { a->base = (char*)q; a->cap = cap; }
            else cudaGetLastError();
        }
    }
    int take(void** d, size_t bytes)
    {
        const size_t b = (std::max<size_t>(bytes, 8) + 255) & ~(size_t)255;
        want += b;
        if (used + b <= a->cap) { *d = a->base + used; used += b; return 0; }
        void* q;
        CK(cudaMalloc(&q, b));
        extra.push_back(q);
        *d = q;
        return 0;
    }
    template <typename T> int up(T** d, const T* h, size_t n)
    {
        *d = nullptr;
        if (!h) return 0;
        void* q;
        TRY(take(&q, n * sizeof(T)));
        CK(cudaMemcpy(q, h, n * sizeof(T), cudaMemcpyHostToDevice));
        *d = (T*)q;
        return 0;
    }
    template <typename T> int out(T** d, const T* h, size_t n)
    {
        *d = nullptr;
        if (!h) return 0;
        void* q;
        TRY(take(&q, n * sizeof(T)));
        CK(cudaMemset(q, 0, n * sizeof(T)));
        *d = (T*)q;
        return 0;
    }
};
#define DOWN(h, d, n) do { if (h) CK(cudaMemcpy(h, d, (size_t)(n) * sizeof(*(h)), cudaMemcpyDeviceToHost)); } while (0)

int acoc_step_batch(int device, int n, const double* params, int state_f64, const double* x, const double* u, const double* lmbd,
                    double* xxp, double* A, double* B, double* fxx, double* fux)
{
    REQUIRE(n > 0 && params && x && u, "acoc_step_batch: n > 0 and params, x, u must be given");
    TRY(use_device(device));
    const Model M = make_model(params);
    TmpBuf t(device);
    double *dx, *du, *dl, *oxp, *oA, *oB, *oxx, *oux;
    const size_t nxx = lmbd ? 36 : 216, nux = lmbd ? 12 : 72;
    TRY(t.up(&dx, x, (size_t)n * 6)); TRY(t.up(&du, u, (size_t)n * 2)); TRY(t.up(&dl, lmbd, (size_t)n * 6));
    TRY(t.out(&oxp, xxp, (size_t)n * 6)); TRY(t.out(&oA, A, (size_t)n * 36)); TRY(t.out(&oB, B, (size_t)n * 12));
    TRY(t.out(&oxx, fxx, n * nxx)); TRY(t.out(&oux, fux, n * nux));
    k_step_batch<<<(n + 127) / 128, 128>>>(M, state_f64 ? 0 : 1, n, dx, du, dl, oxp, oA, oB, oxx, oux);
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    DOWN(xxp, oxp, (size_t)n * 6); DOWN(A, oA, (size_t)n * 36); DOWN(B, oB, (size_t)n * 12);
    DOWN(fxx, oxx, n * nxx); DOWN(fux, oux, n * nux);
    return 0;
}

int acoc_cost_batch(int device, int n, const double* Q, const double* R, const double* QT, const double* x, const double* u,
                    const double* xr, const double* ur, double* ll, double* lx, double* lu, double* llT, double* lTx)
{
    REQUIRE(n > 0 && Q && R && QT && x && xr, "acoc_cost_batch: n > 0 and Q, R, QT, x, xr must be given");
    REQUIRE((u == nullptr) == (ur == nullptr), "acoc_cost_batch: u and ur must be given together");
    REQUIRE(u || !(ll || lx || lu), "acoc_cost_batch: stage outputs need u, ur");
    TRY(use_device(device));
    Weights W;
    fill_weights(&W, Q, R, QT);
    TmpBuf t(device);
    double *dx, *du, *dxr, *dur, *oll, *olx, *olu, *ollT, *olTx;
    TRY(t.up(&dx, x, (size_t)n * 6)); TRY(t.up(&du, u, (size_t)n * 2)); TRY(t.up(&dxr, xr, (size_t)n * 6)); TRY(t.up(&dur, ur, (size_t)n * 2));
    TRY(t.out(&oll, ll, n)); TRY(t.out(&olx, lx, (size_t)n * 6)); TRY(t.out(&olu, lu, (size_t)n * 2));
    TRY(t.out(&ollT, llT, n)); TRY(t.out(&olTx, lTx, (size_t)n * 6));
    k_cost_batch<<<(n + 127) / 128, 128>>>(W, n, dx, du, dxr, dur, oll, olx, olu, ollT, olTx);
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    DOWN(ll, oll, n); DOWN(lx, olx, (size_t)n * 6); DOWN(lu, olu, (size_t)n * 2); DOWN(llT, ollT, n); DOWN(lTx, olTx, (size_t)n * 6);
    return 0;
}

static int lq_dense_dev(int nb, int TT, bool aug, const double* A, const double* B, const double* Q, const double* R, const double* S,
                        const double* Qf, const double* x0, const double* q, const double* r, const double* qf, double* K, double* P,
                        double* xo, double* uo, int* nreg, cudaStream_t st)
{
    if (aug) k_lq_dense<7><<<(nb + 31) / 32, 32, 0, st>>>(nb, TT, A, B, Q, R, S, Qf, x0, q, r, qf, K, P, xo, uo, nreg);
    else k_lq_dense<6><<<(nb + 31) / 32, 32, 0, st>>>(nb, TT, A, B, Q, R, S, Qf, x0, nullptr, nullptr, nullptr, K, P, xo, uo, nreg);
    CK(cudaGetLastError());
    return 0;
}

int acoc_ltv_lqr(int device, int nb, int TT, const double* A, const double* B, const double* Q, const double* R, const double* S,
                 const double* Qf, const double* x0, const double* q, const double* r, const double* qf, double* K, double* P,
                 double* xout, double* uout, int* n_reg)
{
    REQUIRE(nb > 0 && TT >= 2, "acoc_ltv_lqr: nb > 0 and TT >= 2 required");
    REQUIRE(A && B && Q && R && S && Qf && x0 && K && xout && uout, "acoc_ltv_lqr: NULL matrix argument");
    const bool aug = q || r || qf;
    REQUIRE(!aug || (q && r && qf), "acoc_ltv_lqr: give all of q, r, qf (zero-filled if absent) or none");
    TRY(use_device(device));
    const int n = aug ? 7 : 6;
    const size_t T = (size_t)nb * TT;
    TmpBuf t(device);
    double *dA, *dB, *dQ, *dR, *dS, *dQf, *dx0, *dq, *dr, *dqf, *oK, *oP, *ox, *ou;
    int* onr;
    TRY(t.up(&dA, A, T * 36)); TRY(t.up(&dB, B, T * 12)); TRY(t.up(&dQ, Q, T * 36)); TRY(t.up(&dR, R, T * 4)); TRY(t.up(&dS, S, T * 12));
    TRY(t.up(&dQf, Qf, (size_t)nb * 36)); TRY(t.up(&dx0, x0, (size_t)nb * 6));
    TRY(t.up(&dq, q, T * 6)); TRY(t.up(&dr, r, T * 2)); TRY(t.up(&dqf, qf, (size_t)nb * 6));
    TRY(t.out(&oK, K, T * 2 * n)); TRY(t.out(&oP, P, T * n * n)); TRY(t.out(&ox, xout, T * 6)); TRY(t.out(&ou, uout, T * 2));
    TRY(t.out(&onr, n_reg, nb));
    TRY(lq_dense_dev(nb, TT, aug, dA, dB, dQ, dR, dS, dQf, dx0, dq, dr, dqf, oK, oP, ox, ou, onr, 0));
    CK(cudaDeviceSynchronize());
    DOWN(K, oK, T * 2 * n); DOWN(P, oP, T * n * n); DOWN(xout, ox, T * 6); DOWN(uout, ou, T * 2); DOWN(n_reg, onr, nb);
    return 0;
}

// ======================================================================================================
// context life cycle
// ======================================================================================================
int acoc_ctx_create(int device, int n_instances, int TT, unsigned flags, acoc_ctx** out)
{
    REQUIRE(out, "out is NULL");
    *out = nullptr;
    REQUIRE(n_instances > 0 && TT >= 3, "need n_instances > 0 and TT >= 3 (got %d, %d)", n_instances, TT);
    TRY(use_device(device));
    acoc_ctx* c = new acoc_ctx();
    c->device = device; c->N = n_instances; c->Np = (n_instances + 31) / 32 * 32; c->TT = TT; c->flags = flags;
    c->cap = n_instances;
    memset(&c->P, 0, sizeof(c->P)); memset(&c->S, 0, sizeof(c->S));
    default_opts(&c->O);
    auto bail = [&](int rc) { acoc_ctx_destroy(c); return rc; };
    // ACOC_PRIORITY(level): the context's streams are scheduled before those of contexts with a lower level (see acoc.h)
    int prio_least = 0, prio_greatest = 0;
    cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest);  // numerically smaller = higher priority
    const int level = (int)((flags >> ACOC_PRIORITY_SHIFT) & 15u);
    const int prio = std::max(prio_greatest, prio_least - level);
    c->stream_priority = prio;
    if (cudaStreamCreateWithPriority(&c->stream, cudaStreamNonBlocking, prio) != cudaSuccess)
        return bail(fail(ACOC_ERR_CUDA, "cudaStreamCreate failed"));
    const size_t Np = c->Np, T = TT;
    c->fp32 = (flags & ACOC_FP32) != 0;
    c->x_float = c->fp32;
    const size_t es = c->fp32 ? sizeof(float) : sizeof(double);  // the state slots are sized for es too: they may have to hold float64
    int rc = 0;
    // (internal) a context that only hosts one trajectory slot: acoc_lqr_tracking rolls out into X[0]/U[0] and needs no Newton state
    const bool lite = (flags & ACOC_CTX_LITE) != 0;
    const int n_slots = lite ? ((flags & ACOC_CTX_NO_SLOTS) ? 0 : 1) : 3;
    for (int s = 0; s < n_slots && !rc; ++s) { rc = dalloc_bytes(c, &c->X[s], T * 6 * Np * es); if (!rc) rc = dalloc_bytes(c, &c->U[s], T * 2 * Np * es); }
    if (!rc) rc = dalloc_bytes(c, &c->DU, lite ? 64 : T * 2 * Np * es);
    if (!rc) rc = dalloc_bytes(c, &c->KSG, lite ? 64 : T * 16 * Np * es);
    const bool shared = flags & ACOC_REFS_SHARED;
    if (!rc) rc = dalloc_bytes(c, &c->xref, (shared ? T * 6 : T * 6 * Np) * es);
    if (!rc) rc = dalloc_bytes(c, &c->uref, (shared ? T * 2 : T * 2 * Np) * es);
    if (!rc) rc = dalloc_bytes(c, &c->x0, 6 * Np * es);
    if (!rc) rc = dalloc(c, &c->S.status, Np);
    if (!rc) rc = dalloc(c, &c->S.iters, Np);
    if (!rc) rc = dalloc(c, &c->S.result_slot, Np);
    if (!rc) rc = dalloc(c, &c->S.n_reg, Np);
    if (!rc) rc = dalloc(c, &c->S.Jcur, Np);
    if (!rc) rc = dalloc(c, &c->S.descent, Np);
    if (!rc) rc = dalloc(c, &c->S.step, Np);
    if (!rc) rc = dalloc(c, &c->need, Np);
    if (!rc) rc = dalloc(c, &c->need2, Np);
    if (!rc) rc = dalloc(c, &c->slot_tmp, Np);
    if (!rc) rc = dalloc(c, &c->origin, Np);
    if (!rc) rc = dalloc(c, &c->counters, 4 + 2 * MAX_RANGES);  // [0] active count, [1] tile list, [2] need list of range 0, [3 + r] of range r >= 1,
                                                               // [4 + MAX_RANGES + r] second-stage need list of range r
    if (!rc) rc = dalloc(c, &c->act_groups, Np);
    if (!rc) rc = dalloc(c, &c->need_groups, Np);
    if (!rc) rc = dalloc(c, &c->need_groups2, Np);
    if (!rc) rc = dalloc(c, &c->iters_sum, 2);
    // staging: up to 256 MiB or the whole batch, whichever is smaller (at least one instance of 6*TT doubles)
    c->stage_doubles = std::max<size_t>(16 * T, std::min<size_t>((size_t)n_instances * 16 * T, (size_t)32 << 20));
    if (!rc) rc = dalloc(c, &c->stage, c->stage_doubles);
    if (!rc) rc = alloc_history(c);
    if (rc) return bail(rc);
    c->P.N = c->N; c->P.Np = c->Np; c->P.TT = TT;
    c->P.q32 = (flags & ACOC_STATE_F64) ? 0 : 1;
    c->P.ref_shared = shared ? 1 : 0;
    c->P.xref = nullptr; c->P.uref = nullptr; c->P.x0 = nullptr;  // typed pointers are filled in by prob<F>()
    const double defp[9] = {0.1716, 2.395, 3.256, 12.0, 9.81, 0.61, 1.2, 0.24, 1e-3};
    c->P.M = make_model(defp);
    c->have_model = true;
    for (int e = 0; e < 8; ++e) if (cudaEventCreate(&c->ev[e]) != cudaSuccess) return bail(fail(ACOC_ERR_CUDA, "cudaEventCreate failed"));
    c->ev_ok = true;
    if (cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming) != cudaSuccess) return bail(fail(ACOC_ERR_CUDA, "event creation failed"));
    for (int r = 1; r < MAX_RANGES; ++r)
        if (cudaStreamCreateWithPriority(&c->rstream[r], cudaStreamNonBlocking, c->stream_priority) != cudaSuccess ||
            cudaEventCreateWithFlags(&c->ev_join[r], cudaEventDisableTiming) != cudaSuccess)
            return bail(fail(ACOC_ERR_CUDA, "stream/event creation failed"));
    rc = reset_state(c);
    if (rc) return bail(rc);
    if (cudaStreamSynchronize(c->stream) != cudaSuccess) return bail(fail(ACOC_ERR_CUDA, "stream sync failed"));
    *out = c;
    return 0;
}

int acoc_ctx_destroy(acoc_ctx* c)
{
    if (!c) return 0;
    if (c->child) acoc_ctx_destroy(c->child);
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    for (auto& p : c->allocs) cudaFree(p.first);
    if (c->ev_ok) for (int e = 0; e < 8; ++e) cudaEventDestroy(c->ev[e]);
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    for (int r = 1; r < MAX_RANGES; ++r) {
        if (c->ev_join[r]) cudaEventDestroy(c->ev_join[r]);
        if (c->rstream[r]) { cudaStreamSynchronize(c->rstream[r]); cudaStreamDestroy(c->rstream[r]); }
    }
    if (c->dstream) { cudaStreamSynchronize(c->dstream); cudaStreamDestroy(c->dstream); }
    if (c->ev_deliver) cudaEventDestroy(c->ev_deliver);
    for (auto& e : c->tk_ev) if (e) cudaEventDestroy(e);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return 0;
}

int acoc_ctx_device_bytes(const acoc_ctx* c, unsigned long long* bytes)
{
    REQUIRE(c && bytes, "NULL argument");
    *bytes = c->bytes;
    return 0;
}

int acoc_set_model(acoc_ctx* c, const double* params)
{
    REQUIRE(c && params, "NULL argument");
    REQUIRE(params[3] != 0.0 && params[7] != 0.0, "mass and inertia must be non-zero");
    c->P.M = make_model(params);
    return 0;
}

int acoc_set_weights(acoc_ctx* c, const double* Q, const double* R, const double* QT)
{
    REQUIRE(c && Q && R && QT, "NULL argument");
    // the fused backward sweep keeps P symmetric (21 registers); that needs symmetric cost Hessians
    REQUIRE(is_sym(Q, 6) && is_sym(R, 2) && is_sym(QT, 6), "Q, R and QT must be symmetric for the batched Newton path");
    fill_weights(&c->P.W, Q, R, QT);
    c->have_weights = true;
    return 0;
}

int acoc_set_options(acoc_ctx* c, const acoc_newton_options* o)
{
    REQUIRE(c && o, "NULL argument");
    REQUIRE(o->max_iters >= 2 && o->max_iters <= 100000, "max_iters out of range");
    REQUIRE(o->armijo_maxiters >= 1 && o->armijo_maxiters <= 30, "armijo_maxiters must be in 1..30");
    REQUIRE(o->method == ACOC_METHOD_NEWTON || o->method == ACOC_METHOD_GRADIENT, "method must be ACOC_METHOD_NEWTON or ACOC_METHOD_GRADIENT");
    TRY(use_device(c->device));
    c->O.max_iters = o->max_iters; c->O.armijo_maxiters = o->armijo_maxiters; c->O.exact_after = o->exact_after;
    c->O.stepsize_0 = o->stepsize_0; c->O.cc = o->cc; c->O.beta = o->beta; c->O.term_cond = o->term_cond; c->O.method = o->method;
    TRY(alloc_history(c));  // resizes the history buffers if needed, rewrites the Armijo step table
    return reset_state(c);
}

int acoc_set_refs(acoc_ctx* c, const double* xx_ref, const double* uu_ref)
{
    REQUIRE(c && xx_ref && uu_ref, "NULL argument");
    TRY(use_device(c->device));
    if (c->P.ref_shared) {
        TRY(upload_soa(c, xx_ref, c->xref, 1, 6, 1));
        TRY(upload_soa(c, uu_ref, c->uref, 1, 2, 1));
    } else {
        TRY(upload_soa(c, xx_ref, c->xref, c->N, 6, c->Np));
        TRY(upload_soa(c, uu_ref, c->uref, c->N, 2, c->Np));
    }
    c->P.ref_param = 0;
    c->have_refs = true;
    return 0;
}

// device buffers of the parametric references (allocated on first use: tables, per-instance parameters, speed reference)
static int ensure_param_buffers(acoc_ctx* c)
{
    if (c->rp_tt) return 0;
    const size_t T = c->TT, Np = c->Np;
    TRY(dalloc_bytes(c, &c->rp_tt, T * sizeof(double)));
    TRY(dalloc_bytes(c, &c->rp_zs, T * sizeof(double)));
    TRY(dalloc_bytes(c, &c->rp_zf, Np * sizeof(double)));
    TRY(dalloc_bytes(c, &c->rp_vx, Np * sizeof(double)));
    TRY(dalloc_bytes(c, &c->rp_v, T * Np * sizeof(double)));
    return 0;
}

int acoc_set_refs_generated(acoc_ctx* c, const double* tt, const double* zshape, const double* vshape, const double* zf, const double* vx,
                            const double* xconst, const double* uconst)
{
    REQUIRE(c && tt && zshape && zf && vx && xconst && uconst, "NULL argument");
    REQUIRE(!c->P.ref_shared, "acoc_set_refs_generated needs per-instance reference storage (no ACOC_REFS_SHARED)");
    TRY(use_device(c->device));
    const size_t T = c->TT, N = c->N;
    REQUIRE(3 * T + 2 * N <= c->stage_doubles, "staging buffer too small for the generator inputs");
    double* d = c->stage;  // [tt | zshape | vshape | zf | vx]
    CK(cudaMemcpyAsync(d, tt, T * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(d + T, zshape, T * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    if (vshape) CK(cudaMemcpyAsync(d + 2 * T, vshape, T * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(d + 3 * T, zf, N * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(d + 3 * T + N, vx, N * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    RefConst K;
    for (int k = 0; k < 6; ++k) K.xc[k] = xconst[k];
    K.uc[0] = uconst[0]; K.uc[1] = uconst[1];
    const dim3 grid((unsigned)((N + 127) / 128), (unsigned)std::min<size_t>(T, 64));
    if (!c->fp32 && !(c->flags & ACOC_REFS_EXPANDED)) {
        // compact (parametric) storage: tables + parameters + the speed reference; the sweeps form X and Z themselves
        TRY(ensure_param_buffers(c));
        CK(cudaMemcpyAsync(c->rp_tt, d, T * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
        CK(cudaMemcpyAsync(c->rp_zs, d + T, T * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
        CK(cudaMemcpyAsync(c->rp_zf, d + 3 * T, N * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
        CK(cudaMemcpyAsync(c->rp_vx, d + 3 * T + N, N * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
        if (vshape) k_gen_vref<<<grid, 128, 0, c->stream>>>(c->N, c->Np, c->TT, d + 2 * T, d + 3 * T, d + 3 * T + N, (double*)c->rp_v);
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(c->stream));
        c->rp_has_v = vshape != nullptr;
        c->P.ref_param = 1;
        for (int k = 0; k < 6; ++k) c->P.rp_xc[k] = xconst[k];
        c->P.rp_uc[0] = uconst[0]; c->P.rp_uc[1] = uconst[1];
        c->have_refs = true;
        return 0;
    }
    c->P.ref_param = 0;
    with_real(c->fp32, [&](auto R) {
        using F = typename decltype(R)::type;
        k_gen_refs<F><<<grid, 128, 0, c->stream>>>(c->N, c->Np, c->TT, d, d + T, vshape ? d + 2 * T : nullptr, d + 3 * T, d + 3 * T + N, K,
                                                   (F*)c->xref, (F*)c->uref);
        return 0;
    });
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(c->stream));  // the staging buffer is free again; the host arrays may be reused
    c->have_refs = true;
    return 0;
}

int acoc_set_init(acoc_ctx* c, const double* xx_init, const double* uu_init)
{
    REQUIRE(c && xx_init && uu_init, "NULL argument");
    TRY(use_device(c->device));
    TRY(reset_state(c));
    // x0 = xx[:,0,0] (optcon.py:398) is taken from the t = 0 column during the upload
    if (c->fp32) {
        TRY((upload_soa_t<float, float>(c, xx_init, c->X[0], c->N, 6, c->Np, (float*)c->x0, nullptr)));
    } else {
        c->x_float = false;
        if (c->P.q32) {
            // float32-quantised states: a trajectory produced by the reference's get_initial_trajectory (or by any rollout of
            // Dynamics.step) consists of float32 values for t >= 1 and is stored as float; anything else keeps float64 slots
            CK(cudaMemsetAsync(c->counters + 3, 0, sizeof(int), c->stream));
            TRY((upload_soa_t<float, double>(c, xx_init, c->X[0], c->N, 6, c->Np, (double*)c->x0, c->counters + 3)));
            int inexact = 0;
            CK(cudaMemcpyAsync(&inexact, c->counters + 3, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
            CK(cudaStreamSynchronize(c->stream));
            c->x_float = !inexact && !(c->flags & ACOC_X_F64);
        }
        if (!c->x_float) TRY((upload_soa_t<double, double>(c, xx_init, c->X[0], c->N, 6, c->Np, (double*)c->x0, nullptr)));
    }
    TRY(upload_soa(c, uu_init, c->U[0], c->N, 2, c->Np));
    CK(cudaStreamSynchronize(c->stream));
    c->have_init = true;
    return 0;
}

template <typename F, typename XT>
static int init_guess_t(acoc_ctx* c, double kp, double kt, const double* dx0)
{
    F* d_dx0 = nullptr;
    if (dx0) {  // host (N,6) -> device [6][Np]; x0 doubles as the scratch for it (the kernel writes x0 after reading dx0)
        std::vector<F> tmp((size_t)6 * c->Np, F(0));
        for (int i = 0; i < c->N; ++i) for (int k = 0; k < 6; ++k) tmp[(size_t)k * c->Np + i] = (F)dx0[(size_t)i * 6 + k];
        CK(cudaMemcpyAsync(c->x0, tmp.data(), tmp.size() * sizeof(F), cudaMemcpyHostToDevice, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        d_dx0 = (F*)c->x0;
    }
    with_flag(c->P.q32, [&](auto Q) {
        k_init_guess<Q, F, XT><<<(c->N + ROLL_THREADS - 1) / ROLL_THREADS, ROLL_THREADS, 0, c->stream>>>(prob<F>(c), kp, kt, d_dx0, (XT*)c->X[0],
                                                                                                        (F*)c->U[0], (F*)c->x0);
        return 0;
    });
    CK(cudaGetLastError());
    return 0;
}

int acoc_init_guess(acoc_ctx* c, double kp, double kt, const double* dx0)
{
    REQUIRE(c, "NULL argument");
    if (!c->have_refs) return fail(ACOC_ERR_STATE, "acoc_init_guess: set the references first");
    TRY(use_device(c->device));
    TRY(reset_state(c));
    c->x_float = c->fp32 || (c->P.q32 && !(c->flags & ACOC_X_F64));  // a float32-quantised rollout produces float32 states
    TRY(DISPATCH_FX(c, init_guess_t, c, kp, kt, dx0));
    CK(cudaStreamSynchronize(c->stream));
    c->have_init = true;
    return 0;
}

// ======================================================================================================
// Newton pieces
// ======================================================================================================
static int ready(acoc_ctx* c)
{
    if (!c) return fail(ACOC_ERR_INVALID, "ctx is NULL");
    if (!c->have_weights || !c->have_refs || !c->have_init)
        return fail(ACOC_ERR_STATE, "context not ready: set weights (%d), references (%d) and the initial trajectory (%d) first",
                    (int)c->have_weights, (int)c->have_refs, (int)c->have_init);
    return use_device(c->device);
}

template <typename F, typename XT>
static int launch_cost_t(acoc_ctx* c)
{
    const int cur = c->kk % 3;
    k_traj_cost<F, XT><<<(c->N + 127) / 128, 128, 0, c->stream>>>(prob<F>(c), (const XT*)c->X[cur], (const F*)c->U[cur], c->S.status, c->S.Jcur);
    CK(cudaGetLastError());
    ++c->launches;
    return 0;
}
static int launch_cost(acoc_ctx* c) { return DISPATCH_FX(c, launch_cost_t, c); }
// the sweeps run as warp-private TMA pipelines (acoc_tma.cuh) unless the context was created with ACOC_NO_TMA
static bool use_tma(const acoc_ctx* c) { return ACOC_ACT_SHIFT == 5 && !(c->flags & ACOC_NO_TMA); }
static TileList tile_list(acoc_ctx* c, bool use_list = true)
{
    TileList L;
    L.tiles = (use_list && !c->ls_identity) ? c->act_groups : nullptr;
    L.count = c->counters + 1;
    L.off = c->ls_off; L.end = c->ls_end;
    return L;
}
// instance range and need-list counter of the current launch scope
static int scope_i0(const acoc_ctx* c) { return c->ls_off * 32; }
static int n_tiles(const acoc_ctx* c) { return (c->N + 31) / 32; }  // tiles that hold instances (a child context may use less than its capacity Np)
static int scope_i1(const acoc_ctx* c) { return (int)std::min<long long>(c->N, (long long)std::min(n_tiles(c), c->ls_end) * 32); }
static int* scope_need_count(acoc_ctx* c) { return c->counters + (c->ls_range == 0 ? 2 : 3 + c->ls_range); }
static int* scope_need2_count(acoc_ctx* c) { return c->counters + 4 + MAX_RANGES + c->ls_range; }  // second-stage list of the Gauss-Newton split
// stream and grid of a sweep launch in the current launch scope (the whole padded batch, or a range of its tiles)
static cudaStream_t sweep_stream(const acoc_ctx* c) { return c->ls_stream ? c->ls_stream : c->stream; }
static int sweep_grid(const acoc_ctx* c, int threads)
{
    const int tiles = std::max(1, std::min(n_tiles(c), c->ls_end) - c->ls_off);
    return (tiles * 32 + threads - 1) / threads;
}

static WorkList act_list(acoc_ctx* c)
{
    WorkList L;
    L.groups = c->act_groups;
    L.count = c->counters + 1;
    L.shift = ACOC_ACT_SHIFT;
    return L;
}
// rebuild the list of instance groups that still have an active member (start of every iteration)
static int launch_build_active(acoc_ctx* c)
{
    k_build_list<<<1, 1024, 0, c->stream>>>(c->S.status, 0, c->N, ACOC_ACT_SHIFT, c->act_groups, c->counters + 1);
    CK(cudaGetLastError());
    ++c->launches;
    return 0;
}
// the warp-specialised backward sweep: batches of at most two tiles per SM (9,472 instances on a B200) -- all resident at once with room
// to spare for the kernels of other contexts (the sub-batches of a pipelined solve); its register budget allows four per SM
#ifndef ACOC_BWD_SPLIT_TILES_PER_SM
#define ACOC_BWD_SPLIT_TILES_PER_SM 2
#endif
static bool bwd_split(const acoc_ctx* c)
{
    static const bool off = getenv("ACOC_NO_BWD_SPLIT") != nullptr;  // A/B: the single-warp sweep k_backward_tma
    static const int per_sm = getenv("ACOC_BWD_SPLIT_TILES_PER_SM") ? atoi(getenv("ACOC_BWD_SPLIT_TILES_PER_SM")) : ACOC_BWD_SPLIT_TILES_PER_SM;
    int sms = c->sm_count;
    if (sms <= 0) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device);
    return !off && n_tiles(c) <= per_sm * sms;
}
// the backward sweep as a pipeline of warp roles (k_backward_cols, 11 warps per tile: linearisation ahead of time in three warps, costate
// warp, gain warp, one warp per column of the Riccati matrix): the shortest chain of instructions per step, for batches in which every
// tile has an SM of its own (4,736 instances on a B200)
#ifndef ACOC_BWD_COLS_TILES_PER_SM
#define ACOC_BWD_COLS_TILES_PER_SM 1
#endif
static bool bwd_cols(const acoc_ctx* c)
{
    static const bool off = getenv("ACOC_NO_BWD_COLS") != nullptr;  // A/B: k_backward_split / k_backward_tma
    static const int per_sm = getenv("ACOC_BWD_COLS_TILES_PER_SM") ? atoi(getenv("ACOC_BWD_COLS_TILES_PER_SM")) : ACOC_BWD_COLS_TILES_PER_SM;
    int sms = c->sm_count;
    if (sms <= 0) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device);
    return !off && n_tiles(c) <= per_sm * sms;
}
template <typename F, typename XT>
static int launch_backward_t(acoc_ctx* c, bool exact)
{
    const int cur = c->kk % 3, g = (c->Np + BWD_THREADS - 1) / BWD_THREADS;
    const ProblemT<F> P = prob<F>(c);
    const XT* X = (const XT*)c->X[cur];
    const F* U = (const F*)c->U[cur];
    F* KSG = (F*)c->KSG;
    const bool dg = c->P.W.diag != 0;
    if (use_tma(c) && bwd_cols(c)) {  // small batch: warp-role pipeline per tile (k_backward_cols)
        TRY(with_flags(exact, dg, [&](auto EX, auto DG) {
            return launch_ring(k_backward_cols<EX, F, XT, DG>, sweep_grid(c, TILE), BC_THREADS, backward_cols_smem<EX, F, XT>(), sweep_stream(c), P,
                               tile_list(c), X, U, KSG, c->S.status, c->S.n_reg);
        }));
    } else if (use_tma(c) && bwd_split(c)) {  // small batch: costate warp + matrix warp per tile (k_backward_split)
        TRY(with_flags(exact, dg, [&](auto EX, auto DG) {
            return launch_ring(k_backward_split<EX, F, XT, DG>, sweep_grid(c, TILE), 64, backward_split_smem<EX, F, XT>(), sweep_stream(c), P,
                               tile_list(c), X, U, KSG, c->S.status, c->S.n_reg);
        }));
    } else if (use_tma(c)) {
        const size_t sm = WarpRing<BWD_STAGES, BwdStage<F, XT>::BYTES>::smem_bytes(BWD_THREADS / 32);
        TRY(with_flags(exact, dg, [&](auto EX, auto DG) {
            return launch_ring(k_backward_tma<EX, F, XT, DG>, sweep_grid(c, BWD_THREADS), BWD_THREADS, sm, sweep_stream(c), P, tile_list(c), X, U,
                               KSG, c->S.status, c->S.n_reg);
        }));
        if (!c->bwd_wave_ctas) {  // resident CTAs of this sweep on the whole device (for the two-range split of acoc_newton_iterate)
            int nb = 0, sms = 0;
            CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_backward_tma<true, F, XT, 1>, BWD_THREADS, sm));
            CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device));
            c->bwd_wave_ctas = std::max(1, nb * sms);
            c->sm_count = sms;
        }
    } else
        with_flag(exact, [&](auto EX) {
            k_backward<EX, F, XT><<<g, BWD_THREADS, 0, c->stream>>>(P, act_list(c), X, U, KSG, c->S.status, c->S.n_reg);
            return 0;
        });
    CK(cudaGetLastError());
    ++c->launches;
    return 0;
}
static int launch_backward(acoc_ctx* c, bool exact) { return DISPATCH_FX(c, launch_backward_t, c, exact); }

// GradientMethod.optimize: costate sweep -> deltau, slope (replaces backward + forward of the Newton iteration)
template <typename F, typename XT>
static int launch_gradient_t(acoc_ctx* c)
{
    const int cur = c->kk % 3;
    const ProblemT<F> P = prob<F>(c);
    const XT* X = (const XT*)c->X[cur];
    const F* U = (const F*)c->U[cur];
    if (use_tma(c)) {
        const size_t sm = WarpRing<BWD_STAGES, BwdStage<F, XT>::BYTES>::smem_bytes(BWD_THREADS / 32);
        TRY(launch_ring(k_gradient_tma<F, XT>, sweep_grid(c, BWD_THREADS), BWD_THREADS, sm, sweep_stream(c), P, tile_list(c), X, U, (F*)c->DU,
                        c->S.status, c->S.descent));
    } else
        k_gradient<F, XT><<<(c->Np + FWD_THREADS - 1) / FWD_THREADS, FWD_THREADS, 0, c->stream>>>(P, act_list(c), X, U, (F*)c->DU, c->S.status,
                                                                                               c->S.descent);
    CK(cudaGetLastError());
    ++c->launches;
    return 0;
}
static int launch_gradient(acoc_ctx* c) { return DISPATCH_FX(c, launch_gradient_t, c); }

template <typename F, typename XT>
static int launch_forward_t(acoc_ctx* c)
{
    const int cur = c->kk % 3, g = (c->Np + FWD_THREADS - 1) / FWD_THREADS;
    if (use_tma(c)) {
        TRY(launch_ring(k_forward_tma<F, XT>, sweep_grid(c, FWD_THREADS), FWD_THREADS,
                        WarpRing<FWD_STAGES, FwdStage<F, XT>::BYTES>::smem_bytes(FWD_THREADS / 32), sweep_stream(c), prob<F>(c), tile_list(c),
                        (const XT*)c->X[cur], (const F*)c->U[cur], (const F*)c->KSG, (F*)c->DU, c->S.status, c->S.descent));
    } else
        k_forward<F, XT><<<g, FWD_THREADS, 0, c->stream>>>(prob<F>(c), act_list(c), (const XT*)c->X[cur], (const F*)c->U[cur], (const F*)c->KSG,
                                                           (F*)c->DU, (F*)nullptr, c->S.status, c->S.descent);
    CK(cudaGetLastError());
    ++c->launches;
    return 0;
}
static int launch_forward(acoc_ctx* c) { return DISPATCH_FX(c, launch_forward_t, c); }
// Armijo: fills S.step and the history row kk.  Returns through *lazy_only whether the update may skip
// instances whose candidate 0 is already in the next slot.
// The lazy search saves work, the speculative one a sequential sweep: a small batch (a late survivor generation, a handful of
// trajectories) is latency-bound -- about 1 ms per sweep whatever its size -- and some instance fails candidate 0 in nearly every
// iteration of the float32-noise phase, so lazy costs five sweeps in a row there (backward, forward, candidate 0, candidates 1..9,
// update) against four for speculative (backward, forward, all candidates, update).  Same results either way.
#ifndef ACOC_SPECULATIVE_MAX_N
#define ACOC_SPECULATIVE_MAX_N 4096
#endif
static bool is_lazy(const acoc_ctx* c)
{
    static const int spec_max = getenv("ACOC_SPECULATIVE_MAX_N") ? atoi(getenv("ACOC_SPECULATIVE_MAX_N")) : ACOC_SPECULATIVE_MAX_N;
    // (in the Gauss-Newton iterations candidate 0 is accepted almost everywhere and lazy is three sweeps: keep it there)
    return (c->flags & ACOC_ARMIJO_LAZY) && c->O.armijo_maxiters > 1 && (c->N > spec_max || c->kk <= c->O.exact_after);
}

// lazy Armijo, first round: candidate 0 for every active instance, written tentatively into the next slot
template <typename F, typename XT>
static int launch_cand0_t(acoc_ctx* c)
{
    const int cur = c->kk % 3, nxt = (c->kk + 1) % 3, Np = c->Np;
    const ProblemT<F> P = prob<F>(c);
    const F *U = (const F*)c->U[cur], *DU = (const F*)c->DU;
    if (use_tma(c)) {
        const size_t sm = WarpRing<ROLL_STAGES, RollStage<F>::BYTES>::smem_bytes(ROLL_THREADS / 32);
        TRY(with_flags(c->P.q32, c->P.W.diag != 0, [&](auto Q, auto DG) {
            return launch_ring(k_rollout_write_tma<Q, F, XT, 0, DG>, sweep_grid(c, ROLL_THREADS), ROLL_THREADS, sm, sweep_stream(c), P,
                               tile_list(c), c->O, c->S, U, DU, c->cand_steps, (XT*)c->X[nxt], (F*)c->U[nxt], nullptr, c->kk, 0);
        }));
    } else
        with_flag(c->P.q32, [&](auto Q) {
            k_candidate0_write<Q, F, XT><<<(Np + ROLL_THREADS - 1) / ROLL_THREADS, ROLL_THREADS, 0, c->stream>>>(
                P, act_list(c), U, DU, c->cand_steps, (XT*)c->X[nxt], (F*)c->U[nxt], c->S.status, c->S.Jcand);
            return 0;
        });
    CK(cudaGetLastError());
    ++c->launches;
    return 0;
}
static int launch_cand0(acoc_ctx* c) { return DISPATCH_FX(c, launch_cand0_t, c); }

// lazy Armijo on the TMA path: the LQ forward pass and candidate 0 as one sweep (k_forward_cand0_tma)
static bool fwd_cand0_fused(const acoc_ctx* c)
{
    static const bool off = getenv("ACOC_NO_FWD_CAND0") != nullptr;  // tuning experiments
    return use_tma(c) && is_lazy(c) && !(c->flags & ACOC_NO_FUSED) && c->O.method == ACOC_METHOD_NEWTON && !off;
}
template <typename F, typename XT>
static int launch_forward_cand0_t(acoc_ctx* c)
{
    const int cur = c->kk % 3, nxt = (c->kk + 1) % 3;
    const ProblemT<F> P = prob<F>(c);
    const size_t sm = WarpRing<FC_STAGES, FwdCandStage<F, XT>::BYTES>::smem_bytes(FWD_THREADS / 32);
    TRY(with_flags(c->P.q32, c->P.W.diag != 0, [&](auto Q, auto DG) {
        return launch_ring(k_forward_cand0_tma<Q, F, XT, DG>, sweep_grid(c, FWD_THREADS), FWD_THREADS, sm, sweep_stream(c), P, tile_list(c), c->S,
                           (const XT*)c->X[cur], (const F*)c->U[cur], (const F*)c->KSG, (F*)c->DU, c->cand_steps, (XT*)c->X[nxt], (F*)c->U[nxt]);
    }));
    ++c->launches;
    return 0;
}
static int launch_forward_cand0(acoc_ctx* c) { return DISPATCH_FX(c, launch_forward_cand0_t, c); }

// candidates c0..c1-1 of the instances on a per-instance work list (n list slots at most): the ring kernel of acoc_tma.cuh (one
// producer warp gathers the inputs for all candidate warps of a CTA) or, with ACOC_NO_TMA, the plain-load kernel
constexpr int LIST_ROWS = 9;  // candidate warps per CTA of k_candidates_list (more candidates: several passes)
static bool list_ring(const acoc_ctx* c)
{
    static const bool off = getenv("ACOC_NO_LIST_RING") != nullptr;  // tuning experiments
    return use_tma(c) && !off;
}
// the plain-load kernel k_candidates<Q32, F, MAXY> for candidates c0..c1-1 with step table `steps`: at most CAND_MAXY candidates
// per CTA (blockDim.y), the 9-wide instantiation when it fits
template <typename F>
static void launch_candidates(acoc_ctx* c, const WorkList& L, int n, const F* U, const F* DU, const double* steps, int c0, int c1,
                              cudaStream_t st)
{
    const int ny = std::min(c1 - c0, CAND_MAXY);
    with_flags(c->P.q32, ny <= 9, [&](auto Q, auto Y9) {
        k_candidates<Q, F, Y9 ? 9 : CAND_MAXY><<<(n + CAND_TILE - 1) / CAND_TILE, dim3(CAND_TILE, ny), 0, st>>>(prob<F>(c), L, U, DU, steps, c0, c1,
                                                                                                               c->S.status, c->S.Jcand);
        return 0;
    });
}
template <typename F>
static int launch_list_candidates(acoc_ctx* c, const WorkList& L, int n, int c0, int c1, cudaStream_t st)
{
    const int cur = c->kk % 3;
    const ProblemT<F> P = prob<F>(c);
    const F *U = (const F*)c->U[cur], *DU = (const F*)c->DU;
    if (list_ring(c)) {
        const dim3 blk(TILE, std::min(c1 - c0, LIST_ROWS) + 1);
        const int rf = c->P.ref_param ? 2 : (c->P.ref_shared ? 1 : 0);
        TRY(with_flags(c->P.q32, c->P.W.diag != 0, [&](auto Q, auto DG) {
            return with_mode(rf, [&](auto REFS) {
                return launch_ring(k_candidates_list<Q, F, LIST_ROWS, DG, REFS>, (n + TILE - 1) / TILE, blk, candidates_list_smem<F>(), st, P, L, U,
                                   DU, c->cand_steps, c0, c1, c->S.Jcand);
            });
        }));
    } else
        launch_candidates<F>(c, L, n, U, DU, c->cand_steps, c0, c1, st);
    CK(cudaGetLastError());
    return 0;
}

// Armijo after candidate 0 (lazy) or all candidates at once (speculative): fills S.step and the history row kk.  Returns through
// *lazy_only whether the update may skip instances whose candidate 0 is already in the next slot.
template <typename F, typename XT>
static int launch_armijo_t(acoc_ctx* c, bool* lazy_only)
{
    const int cur = c->kk % 3, Np = c->Np, nc = c->O.armijo_maxiters;
    const F *U = (const F*)c->U[cur], *DU = (const F*)c->DU;
    *lazy_only = false;
    cudaStream_t st = sweep_stream(c);
    const int i0 = scope_i0(c), i1 = scope_i1(c), n = i1 - i0;
    if (is_lazy(c)) {
        int* cnt = scope_need_count(c);
        k_lazy_need<<<(n + 255) / 256, 256, 0, st>>>(c->O, c->S, c->cand_steps, i0, i1, Np, 1, c->need);
        CK(cudaGetLastError());
        WorkList L;  // per-instance list of the instances whose candidate 0 failed: the rollouts are compute-bound
        L.groups = c->need_groups + i0; L.count = cnt; L.shift = 0;
        k_build_list<<<1, 1024, 0, st>>>(c->need, 1, n, 0, c->need_groups + i0, cnt, i0);
        CK(cudaGetLastError());
        c->launches += 2;
        // In the Gauss-Newton iterations (kk <= exact_after) an instance that fails the full step is accepted within the next
        // few candidates (mean 2.6 / 1.9 candidates in iterations 0 / 1 of config 4): candidates 1..3 first, the rest only where
        // those failed too.  Later (float32-noise phase) the search usually runs to the end and one round of 1..9 is cheaper.
        const int split = (c->kk <= c->O.exact_after && nc > 5) ? 4 : nc;
        TRY(launch_list_candidates<F>(c, L, n, 1, split, st));
        if (split < nc) {
            k_lazy_need<<<(n + 255) / 256, 256, 0, st>>>(c->O, c->S, c->cand_steps, i0, i1, Np, split, c->need2);
            CK(cudaGetLastError());
            int* cnt2 = scope_need2_count(c);  // (a counter of its own: the first-stage count tells the host how many searches failed candidate 0)
            L.count = cnt2;
            L.groups = c->need_groups2 + i0;  // (the first-stage list stays: the update rolls exactly those instances)
            k_build_list<<<1, 1024, 0, st>>>(c->need2, 1, n, 0, c->need_groups2 + i0, cnt2, i0);
            CK(cudaGetLastError());
            TRY(launch_list_candidates<F>(c, L, n, split, nc, st));
            c->launches += 3;
        }
        *lazy_only = true;
    } else {
        launch_candidates<F>(c, act_list(c), Np, U, DU, c->cand_steps, 0, nc, c->stream);
        CK(cudaGetLastError());
        ++c->launches;
    }
    k_select<<<(n + 255) / 256, 256, 0, st>>>(c->O, c->S, c->cand_steps, c->kk, i0, i1, c->Np);
    CK(cudaGetLastError());
    ++c->launches;
    return 0;
}
static int launch_armijo(acoc_ctx* c, bool* lazy_only) { return DISPATCH_FX(c, launch_armijo_t, c, lazy_only); }

template <typename F, typename XT>
static int launch_update_t(acoc_ctx* c, bool lazy_only, bool bookkeeping, bool use_list)
{
    const int cur = c->kk % 3, nxt = (c->kk + 1) % 3;
    WorkList L = act_list(c);
    if (!use_list) L.groups = nullptr;
    const int* only = lazy_only ? c->need : nullptr;
    if (use_tma(c)) {
        const size_t sm = WarpRing<ROLL_STAGES, RollStage<F>::BYTES>::smem_bytes(ROLL_THREADS / 32);
        TRY(with_flags(c->P.q32, c->P.W.diag != 0, [&](auto Q, auto DG) {
            return launch_ring(k_rollout_write_tma<Q, F, XT, 1, DG>, sweep_grid(c, ROLL_THREADS), ROLL_THREADS, sm, sweep_stream(c), prob<F>(c),
                               tile_list(c, use_list), c->O, c->S, (const F*)c->U[cur], (const F*)c->DU, c->cand_steps, (XT*)c->X[nxt],
                               (F*)c->U[nxt], only, c->kk, bookkeeping ? 1 : 0);
        }));
    } else
        with_flag(c->P.q32, [&](auto Q) {
            k_update<Q, F, XT><<<(c->Np + ROLL_THREADS - 1) / ROLL_THREADS, ROLL_THREADS, 0, c->stream>>>(
                prob<F>(c), L, c->O, c->S, (const F*)c->U[cur], (const F*)c->DU, (XT*)c->X[nxt], (F*)c->U[nxt], only, c->kk, bookkeeping ? 1 : 0);
            return 0;
        });
    CK(cudaGetLastError());
    ++c->launches;
    return 0;
}
static int launch_update(acoc_ctx* c, bool lazy_only, bool bookkeeping, bool use_list)
{
    return DISPATCH_FX(c, launch_update_t, c, lazy_only, bookkeeping, use_list);
}

// ---- small batches: fused line search (k_search_fused, k_pick, k_finish) -----------------------------------------------------
#ifndef ACOC_FUSED_MAX_N
#define ACOC_FUSED_MAX_N 4096
#endif
// Whether this context runs its iterations with the fused line search; allocates the per-row trajectory slots on first use
// (rows x ~40 KB per instance: 1.8 GB for 4096 instances) and falls back to the separate sweeps if that fails.
template <typename F, typename XT>
static bool fused_search_t(acoc_ctx* c)
{
    static const int fuse_max = getenv("ACOC_FUSED_MAX_N") ? atoi(getenv("ACOC_FUSED_MAX_N")) : ACOC_FUSED_MAX_N;
    const size_t rows = (size_t)c->O.armijo_maxiters + 1;
    if (ACOC_ACT_SHIFT != 5 || c->N > fuse_max || rows > (size_t)FUSE_MAXROWS || c->cand_failed || c->ls_identity || (c->flags & ACOC_NO_FUSED) ||
        c->O.method != ACOC_METHOD_NEWTON)
        return false;
    const size_t bx = rows * c->TT * NS * c->Np * sizeof(XT), bu = rows * c->TT * NI * c->Np * sizeof(F);
    if (c->cand_bytes_x < bx) {
        dfree(c, &c->candX);
        if (dalloc_bytes(c, &c->candX, bx)) { c->cand_failed = true; return false; }
        c->cand_bytes_x = bx;
    }
    if (c->cand_bytes_u < bu) {
        dfree(c, &c->candU);
        if (dalloc_bytes(c, &c->candU, bu)) { c->cand_failed = true; return false; }
        c->cand_bytes_u = bu;
    }
    if (!c->candJ && dalloc(c, &c->candJ, (size_t)c->Np)) { c->cand_failed = true; return false; }
    return true;
}
static bool fused_search(acoc_ctx* c) { return DISPATCH_FX(c, fused_search_t, c); }

// LQ forward pass + every Armijo candidate (+ the exhausted step) in one sweep, trajectories kept per row
template <typename F, typename XT>
static int launch_fused_sweep_t(acoc_ctx* c)
{
    const int cur = c->kk % 3, rows = c->O.armijo_maxiters + 1;
    const size_t rx = (size_t)c->TT * NS * c->Np, ru = (size_t)c->TT * NI * c->Np;
    const dim3 blk(TILE, rows + 1);
    with_flag(c->P.q32, [&](auto Q) {
        k_search_fused<Q, F, XT><<<n_tiles(c), blk, 0, c->stream>>>(prob<F>(c), tile_list(c), (const XT*)c->X[cur], (const F*)c->U[cur],
                                                                   (const F*)c->KSG, (F*)c->DU, c->cand_steps, rows, (XT*)c->candX, (F*)c->candU,
                                                                   rx, ru, c->S.status, c->S.descent, c->S.Jcand);
        return 0;
    });
    CK(cudaGetLastError());
    ++c->launches;
    return 0;
}
static int launch_fused_sweep(acoc_ctx* c) { return DISPATCH_FX(c, launch_fused_sweep_t, c); }

static int launch_fused_select(acoc_ctx* c)
{
    k_select<<<(c->N + 255) / 256, 256, 0, c->stream>>>(c->O, c->S, c->cand_steps, c->kk, 0, c->N, c->Np);
    CK(cudaGetLastError());
    ++c->launches;
    return 0;
}

// get_update (copy of the chosen row into the next slot) + termination bookkeeping
template <typename F, typename XT>
static int launch_fused_pick_t(acoc_ctx* c)
{
    const int nxt = (c->kk + 1) % 3, tiles = n_tiles(c);
    const size_t rx = (size_t)c->TT * NS * c->Np, ru = (size_t)c->TT * NI * c->Np;
    const int gy = std::max(1, std::min((c->TT + 7) / 8, 1184 / tiles));
    k_pick<F, XT><<<dim3(tiles, gy), dim3(TILE, 8), 0, c->stream>>>(tile_list(c), c->O, c->S, c->cand_steps, (const XT*)c->candX,
                                                                    (const F*)c->candU, rx, ru, (XT*)c->X[nxt], (F*)c->U[nxt], c->N, c->Np,
                                                                    c->TT, c->candJ);
    CK(cudaGetLastError());
    k_finish<<<(c->N + 255) / 256, 256, 0, c->stream>>>(c->O, c->S, c->candJ, c->kk, c->N);
    CK(cudaGetLastError());
    c->launches += 2;
    return 0;
}
static int launch_fused_pick(acoc_ctx* c) { return DISPATCH_FX(c, launch_fused_pick_t, c); }

static int count_active(acoc_ctx* c, int* n_active, long long* iters_sum)
{
    CK(cudaMemsetAsync(c->counters, 0, sizeof(int), c->stream));
    CK(cudaMemsetAsync(c->iters_sum, 0, sizeof(long long), c->stream));
    k_count_active<<<(c->Np + 255) / 256, 256, 0, c->stream>>>(c->S.status, c->N, c->counters, c->iters_sum, c->S.iters);
    CK(cudaGetLastError());
    int h = 0;
    long long s = 0;
    CK(cudaMemcpyAsync(&h, c->counters, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(&s, c->iters_sum, sizeof(long long), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    if (n_active) *n_active = h;
    if (iters_sum) *iters_sum = s;
    // ranged iterations sweep every tile; the tile-granular work lists of the single-scope path only start to drop tiles when a few
    // percent of the instances are left (a tile of 32 is finished with probability (1-p)^32), so the ranges stay until then
    static const int active_div = getenv("ACOC_ACTIVE_DIV") ? atoi(getenv("ACOC_ACTIVE_DIV")) : 16;  // tuning experiments
    c->all_active = (long long)active_div * h > c->N;
    return 0;
}

static void scope_reset(acoc_ctx* c) { c->ls_stream = nullptr; c->ls_off = 0; c->ls_end = 0x7fffffff; c->ls_identity = false; c->ls_range = 0; }

// one Newton iteration (loop body of optcon.py:415-501) of the instances in the current launch scope, without the list rebuild
static int launch_iteration_body(acoc_ctx* c)
{
    bool lazy_only = false;
    TRY(launch_backward(c, c->kk > c->O.exact_after));  // optcon.py:443
    if (fused_search(c)) {
        TRY(launch_fused_sweep(c));
        TRY(launch_fused_select(c));
        return launch_fused_pick(c);
    }
    if (fwd_cand0_fused(c)) TRY(launch_forward_cand0(c));
    else {
        TRY(launch_forward(c));
        if (is_lazy(c)) TRY(launch_cand0(c));
    }
    TRY(launch_armijo(c, &lazy_only));
    TRY(launch_update(c, lazy_only, true, true));
    return 0;
}

// Whether the next iteration(s) of this context run as independent tile ranges (see acoc_newton_iterate)
static bool ranged_mode(const acoc_ctx* c)
{
    const int ctas = (n_tiles(c) + 1) / 2, wave = c->bwd_wave_ctas;
    return use_tma(c) && is_lazy(c) && !c->profiling && c->all_active && !(c->flags & ACOC_NO_SPLIT) && c->kk > 0 && wave > 0 && ctas > wave &&
           ctas % wave != 0 && c->O.method != ACOC_METHOD_GRADIENT;
}

// one iteration on the context's stream over the work lists (any batch, any mode; per-phase events when profiling)
static int single_scope_iteration(acoc_ctx* c)
{
    const bool prof = c->profiling, grad = c->O.method == ACOC_METHOD_GRADIENT;
    bool lazy_only = false;
    if (prof) CK(cudaEventRecord(c->ev[0], c->stream));
    TRY(launch_build_active(c));
    if (c->kk == 0) TRY(launch_cost(c));  // later iterations inherit the cost from the update rollout
    if (prof) CK(cudaEventRecord(c->ev[1], c->stream));
    if (grad) TRY(launch_gradient(c));                       // optcon.py:95-118
    else TRY(launch_backward(c, c->kk > c->O.exact_after));  // optcon.py:443
    if (prof) CK(cudaEventRecord(c->ev[2], c->stream));
    if (grad) {  // the costate sweep already produced deltau and the slope: straight to the line search
        if (prof) CK(cudaEventRecord(c->ev[3], c->stream));
        if (is_lazy(c)) TRY(launch_cand0(c));
        TRY(launch_armijo(c, &lazy_only));
        if (prof) CK(cudaEventRecord(c->ev[4], c->stream));
        TRY(launch_update(c, lazy_only, true, true));
    } else if (fused_search(c)) {  // small batch: forward pass and line search in one sweep, get_update as a copy
        TRY(launch_fused_sweep(c));
        if (prof) CK(cudaEventRecord(c->ev[3], c->stream));
        TRY(launch_fused_select(c));
        if (prof) CK(cudaEventRecord(c->ev[4], c->stream));
        TRY(launch_fused_pick(c));
    } else {
        if (fwd_cand0_fused(c)) {  // (the "forward" phase of the profile then contains candidate 0)
            TRY(launch_forward_cand0(c));
            if (prof) CK(cudaEventRecord(c->ev[3], c->stream));
        } else {
            TRY(launch_forward(c));
            if (prof) CK(cudaEventRecord(c->ev[3], c->stream));
            if (is_lazy(c)) TRY(launch_cand0(c));
        }
        TRY(launch_armijo(c, &lazy_only));
        if (prof) CK(cudaEventRecord(c->ev[4], c->stream));
        TRY(launch_update(c, lazy_only, true, true));
    }
    if (prof) {
        CK(cudaEventRecord(c->ev[5], c->stream));
        CK(cudaEventSynchronize(c->ev[5]));
        // phases: cost, backward, forward, candidates+select, (select folded), update
        for (int p = 0; p < 5; ++p) {
            float ms = 0;
            CK(cudaEventElapsedTime(&ms, c->ev[p], c->ev[p + 1]));
            c->phase_ms[p == 4 ? 5 : p] += ms;
        }
    }
    ++c->kk;
    return 0;
}

// `todo` iterations as independent tile ranges on their own streams, joined on the context's stream.  Returns the number of ranges.
// Why ranges: the backward sweep keeps only bwd_wave_ctas CTAs resident (216 registers per thread), so a batch with more CTAs than that
// runs in rounds, and the last, partial round leaves most of the machine idle while every warp of it still needs its full
// latency-bound sweep time.  While most of the batch is active, tile ranges therefore run their iterations independently of each
// other (every kernel of an iteration takes a tile / instance range): one range's bandwidth-bound forward and rollout sweeps fill the
// machine while another's backward sweep is latency-bound, across iteration boundaries too.  Instances are independent, so the split
// changes no result.
static int ranged_iterations(acoc_ctx* c, int todo, int* nr_out)
{
    const int tiles = n_tiles(c), ctas = (tiles + 1) / 2, wave = c->bwd_wave_ctas;
    int bound[MAX_RANGES + 1] = {0, (ctas / wave) * wave * 2}, nr = 2;  // default: the full rounds of resident backward CTAs | the partial round
    // Clean phase (candidate 0 was accepted by practically every instance in the last iteration the host knows of): every iteration
    // is backward -> forward + candidate 0, one latency-bound and one bandwidth-bound sweep, and they overlap the better the more
    // ranges there are -- ranges of about one backward CTA per SM (2 x SMs tiles).  With failing searches the compute-bound
    // candidate kernels of many small ranges cost more than the overlap gains, so fewer ranges are used there.
    static const bool many = getenv("ACOC_NO_MANY_RANGES") == nullptr;
    // (with failing searches: up to four ranges -- 9.06 vs 9.26 ms per iteration over iterations 5..24 with two, gpurun_out r2_ab4)
    static const int noisy_nr = getenv("ACOC_NOISY_RANGES") ? atoi(getenv("ACOC_NOISY_RANGES")) : 4;
    const bool clean = c->last_need >= 0 && (long long)c->last_need * 2048 < c->N;
    if (many && (clean || noisy_nr > 1) && c->sm_count > 0) {
        nr = std::max(2, std::min(MAX_RANGES, (tiles + 2 * c->sm_count - 1) / (2 * c->sm_count)));
        if (!clean) nr = std::min(nr, noisy_nr);
        const int size = ((tiles + nr - 1) / nr + 1) / 2 * 2;  // whole CTAs (two tiles)
        for (int r = 1; r < nr; ++r) bound[r] = std::min(tiles, r * size);
    }
    if (const char* e = getenv("ACOC_RANGES")) {  // tuning experiments: ascending tile boundaries "a,b,c,..."
        nr = 1;
        for (const char* q = e; *q && nr < MAX_RANGES; ++nr) {
            bound[nr] = std::max(bound[nr - 1] + 2, std::min(tiles - 2, atoi(q)));
            while (*q && *q != ',') ++q;
            if (*q == ',') ++q;
        }
    }
    for (int r = nr; r <= MAX_RANGES; ++r) bound[r] = tiles;
    const int kk0 = c->kk;
    CK(cudaEventRecord(c->ev_fork, c->stream));
    for (int r = 1; r < nr; ++r) CK(cudaStreamWaitEvent(c->rstream[r], c->ev_fork, 0));
    int rc = 0;
    for (int r = 0; r < nr && !rc; ++r) {
        c->ls_identity = true;
        c->ls_range = r;
        c->ls_stream = r == 0 ? c->stream : c->rstream[r];
        c->ls_off = bound[r];
        c->ls_end = bound[r + 1];
        c->kk = kk0;
        for (int j = 0; j < todo && !rc; ++j, ++c->kk) rc = launch_iteration_body(c);
    }
    scope_reset(c);
    c->kk = kk0 + todo;
    if (rc) return rc;
    for (int r = 1; r < nr; ++r) {
        CK(cudaEventRecord(c->ev_join[r], c->rstream[r]));
        CK(cudaStreamWaitEvent(c->stream, c->ev_join[r], 0));
    }
    *nr_out = nr;
    return 0;
}

// lengths of the need lists of the lazy search in the last iteration (instances whose candidate 0 failed), summed over the ranges:
// decides between the clean-phase and the two-range split of the following iterations
static int read_last_need(acoc_ctx* c, int nr_last)
{
    int hc[4 + MAX_RANGES] = {};
    CK(cudaMemcpyAsync(hc, c->counters, sizeof(hc), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    c->last_need = hc[2];
    for (int r = 1; r < nr_last; ++r) c->last_need += hc[3 + r];
    return 0;
}

int acoc_newton_iterate(acoc_ctx* c, int n_iters, int* n_active_out)
{
    TRY(ready(c));
    REQUIRE(n_iters >= 0, "n_iters must be >= 0");
    c->total_ms = 0; for (int p = 0; p < 6; ++p) c->phase_ms[p] = 0;
    c->launches = 0;
    CK(cudaEventRecord(c->ev[6], c->stream));
    int it = 0, nr_last = 1;
    const int kk_in = c->kk;
    const bool fused_small = fused_search(c);  // (no need lists in that mode)
    while (it < n_iters && c->kk < c->O.max_iters - 1) {  // for kk in range(max_iters-1), optcon.py:415
        if (!ranged_mode(c)) {
            TRY(single_scope_iteration(c));
            nr_last = 1;
            ++it;
            continue;
        }
        // Ranged iterations come in chunks, and the host looks at the device state between chunks: how many searches failed candidate 0
        // (picks the number of ranges) and how many instances are still active (the ranges sweep every tile; once half of the batch
        // has finished the work lists of the single-scope path are cheaper).  8 iterations per chunk while the phase is clean -- nothing
        // converges there and the many-range split needs longer runs to amortise its fill and drain -- else 4.
        const bool clean = c->last_need >= 0 && (long long)c->last_need * 2048 < c->N;
        static const int noisy_chunk = getenv("ACOC_NOISY_CHUNK") ? atoi(getenv("ACOC_NOISY_CHUNK")) : 4;  // tuning experiments
        const int todo = std::min(std::min(n_iters - it, c->O.max_iters - 1 - c->kk), clean ? 8 : noisy_chunk);
        TRY(ranged_iterations(c, todo, &nr_last));
        it += todo;
        if (it < n_iters && c->kk < c->O.max_iters - 1) {
            TRY(read_last_need(c, nr_last));
            TRY(count_active(c, nullptr, nullptr));
        }
    }
    const bool lazy_counts = (c->flags & ACOC_ARMIJO_LAZY) && c->O.armijo_maxiters > 1 && c->kk > kk_in && !fused_small && is_lazy(c) &&
                             c->O.method == ACOC_METHOD_NEWTON;
    if (lazy_counts) TRY(read_last_need(c, nr_last));
    CK(cudaEventRecord(c->ev[7], c->stream));
    CK(cudaEventSynchronize(c->ev[7]));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, c->ev[6], c->ev[7]));
    c->total_ms = ms;
    if (n_active_out) TRY(count_active(c, n_active_out, nullptr));
    return 0;
}

// gather/scatter every per-instance row set between a parent and its child; to_child = true: parent -> child
// C: 0 for plain [rows][Np] arrays (scalars, histories, x0), else the component count of a warp-tiled trajectory (rows = TT*C)
template <typename T>
static int move_rows(acoc_ctx* par, acoc_ctx* ch, T* pbuf, T* cbuf, int rows, bool to_child, int C = 0)
{
    const int n = ch->N;
    dim3 grid((n + 127) / 128, std::min(rows, 2048));
    if (to_child) k_gather_rows<T><<<grid, 128, 0, par->stream>>>(pbuf, par->Np, cbuf, ch->Np, ch->origin, n, rows, C);
    else k_scatter_rows<T><<<grid, 128, 0, par->stream>>>(cbuf, ch->Np, pbuf, par->Np, ch->origin, n, rows, C);
    CK(cudaGetLastError());
    return 0;
}

// untyped trajectory buffers: rows of float or double
static int move_rows_e(acoc_ctx* par, acoc_ctx* ch, void* pbuf, void* cbuf, int rows, bool to_child, bool is_float, int C)
{
    return is_float ? move_rows<float>(par, ch, (float*)pbuf, (float*)cbuf, rows, to_child, C)
                    : move_rows<double>(par, ch, (double*)pbuf, (double*)cbuf, rows, to_child, C);
}

// Move the n_active still-iterating instances of `par` into its child generation.  Returns 1 if no child could be made.
static int spawn_child(acoc_ctx* par, int n_active, acoc_ctx** out)
{
    *out = nullptr;
    const int cap = par->N / 2;
    if (n_active > cap) return 1;
    if (!par->child) {
        acoc_ctx* ch = nullptr;
        if (acoc_ctx_create(par->device, cap, par->TT, par->flags, &ch) != 0) {
            cudaGetLastError();  // a failed cudaMalloc leaves its error behind; the parent simply keeps iterating in place
            return 1;
        }
        par->child = ch;
    }
    acoc_ctx* ch = par->child;
    if (ch->O.max_iters != par->O.max_iters || ch->O.armijo_maxiters != par->O.armijo_maxiters) {
        acoc_newton_options o;
        o.max_iters = par->O.max_iters; o.armijo_maxiters = par->O.armijo_maxiters; o.exact_after = par->O.exact_after;
        o.stepsize_0 = par->O.stepsize_0; o.cc = par->O.cc; o.beta = par->O.beta; o.term_cond = par->O.term_cond; o.method = par->O.method;
        TRY(acoc_set_options(ch, &o));
    }
    ch->O = par->O;
    TRY(write_cand_steps(ch));  // stepsize_0 / beta may differ from what the child last ran with (its table is per context)
    ch->N = n_active;
    ch->P.M = par->P.M; ch->P.W = par->P.W; ch->P.q32 = par->P.q32; ch->P.N = n_active;
    ch->have_model = ch->have_weights = ch->have_refs = ch->have_init = true;
    ch->profiling = par->profiling;
    ch->x_float = par->x_float;  // (fp32 follows from the creation flags)
    const bool ff = par->fp32, xf = par->x_float;
    TRY(use_device(par->device));
    TRY(reset_state(ch));
    CK(cudaStreamSynchronize(ch->stream));
    // everything below is ordered on the PARENT's stream; the child's stream waits for it through the final sync
    const int TT = par->TT;
    k_build_list<<<1, 1024, 0, par->stream>>>(par->S.status, 0, par->N, 0, ch->origin, par->counters + 3);
    CK(cudaGetLastError());
    k_fill_int<<<(ch->Np + 255) / 256, 256, 0, par->stream>>>(ch->S.status, ch->Np, ST_ACTIVE, n_active, ST_PAD);
    CK(cudaGetLastError());
    for (int sl = 0; sl < 3; ++sl) {
        if (sl == (par->kk + 1) % 3) continue;  // the "next" slot is overwritten by the child's first update anyway
        TRY(move_rows_e(par, ch, par->X[sl], ch->X[sl], 6 * TT, true, xf, 6));
        TRY(move_rows_e(par, ch, par->U[sl], ch->U[sl], 2 * TT, true, ff, 2));
    }
    ch->P.ref_param = par->P.ref_param;
    if (par->P.ref_param) {  // parametric references: tables, per-instance parameters and the stored speed reference of the survivors
        TRY(ensure_param_buffers(ch));
        CK(cudaMemcpyAsync(ch->rp_tt, par->rp_tt, (size_t)TT * sizeof(double), cudaMemcpyDeviceToDevice, par->stream));
        CK(cudaMemcpyAsync(ch->rp_zs, par->rp_zs, (size_t)TT * sizeof(double), cudaMemcpyDeviceToDevice, par->stream));
        TRY(move_rows(par, ch, (double*)par->rp_zf, (double*)ch->rp_zf, 1, true));
        TRY(move_rows(par, ch, (double*)par->rp_vx, (double*)ch->rp_vx, 1, true));
        if (par->rp_has_v) TRY(move_rows(par, ch, (double*)par->rp_v, (double*)ch->rp_v, TT, true, 1));
        ch->rp_has_v = par->rp_has_v;
        for (int k = 0; k < NS; ++k) ch->P.rp_xc[k] = par->P.rp_xc[k];
        for (int k = 0; k < NI; ++k) ch->P.rp_uc[k] = par->P.rp_uc[k];
    } else if (par->flags & ACOC_REFS_SHARED) {
        const size_t es = ff ? sizeof(float) : sizeof(double);
        CK(cudaMemcpyAsync(ch->xref, par->xref, (size_t)TT * 6 * es, cudaMemcpyDeviceToDevice, par->stream));
        CK(cudaMemcpyAsync(ch->uref, par->uref, (size_t)TT * 2 * es, cudaMemcpyDeviceToDevice, par->stream));
    } else {
        TRY(move_rows_e(par, ch, par->xref, ch->xref, 6 * TT, true, ff, 6));
        TRY(move_rows_e(par, ch, par->uref, ch->uref, 2 * TT, true, ff, 2));
    }
    TRY(move_rows_e(par, ch, par->x0, ch->x0, 6, true, ff, 0));
    TRY(move_rows(par, ch, par->S.Jcur, ch->S.Jcur, 1, true));
    TRY(move_rows(par, ch, par->S.descent, ch->S.descent, 1, true));
    TRY(move_rows(par, ch, par->S.step, ch->S.step, 1, true));
    TRY(move_rows(par, ch, par->S.iters, ch->S.iters, 1, true));
    TRY(move_rows(par, ch, par->S.n_reg, ch->S.n_reg, 1, true));
    TRY(move_rows(par, ch, par->S.result_slot, ch->S.result_slot, 1, true));
    k_mark_moved<<<(n_active + 255) / 256, 256, 0, par->stream>>>(par->S.status, ch->origin, n_active);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(par->stream));
    ch->kk = par->kk;
    ch->spawn_kk = par->kk;
    *out = ch;
    return 0;
}

// Fold a finished child generation back into its parent: afterwards the parent looks as if it had iterated everything itself.
static int fold_child(acoc_ctx* par, acoc_ctx* ch)
{
    TRY(use_device(par->device));
    CK(cudaStreamSynchronize(ch->stream));
    const int TT = par->TT, mi = par->O.max_iters;
    for (int sl = 0; sl < 3; ++sl) {
        TRY(move_rows_e(par, ch, par->X[sl], ch->X[sl], 6 * TT, false, par->x_float, 6));
        TRY(move_rows_e(par, ch, par->U[sl], ch->U[sl], 2 * TT, false, par->fp32, 2));
    }
    TRY(move_rows(par, ch, par->S.Jcur, ch->S.Jcur, 1, false));
    TRY(move_rows(par, ch, par->S.descent, ch->S.descent, 1, false));
    TRY(move_rows(par, ch, par->S.step, ch->S.step, 1, false));
    TRY(move_rows(par, ch, par->S.iters, ch->S.iters, 1, false));
    TRY(move_rows(par, ch, par->S.n_reg, ch->S.n_reg, 1, false));
    TRY(move_rows(par, ch, par->S.result_slot, ch->S.result_slot, 1, false));
    TRY(move_rows(par, ch, par->S.status, ch->S.status, 1, false));
    const int r0 = ch->spawn_kk, nr = ch->kk - ch->spawn_kk;  // history rows written by the child
    if (nr > 0) {
        TRY(move_rows(par, ch, par->S.hist_J + (size_t)r0 * par->Np, ch->S.hist_J + (size_t)r0 * ch->Np, nr, false));
        TRY(move_rows(par, ch, par->S.hist_descent + (size_t)r0 * par->Np, ch->S.hist_descent + (size_t)r0 * ch->Np, nr, false));
        TRY(move_rows(par, ch, par->S.hist_step + (size_t)r0 * par->Np, ch->S.hist_step + (size_t)r0 * ch->Np, nr, false));
        TRY(move_rows(par, ch, par->S.hist_ncand + (size_t)r0 * par->Np, ch->S.hist_ncand + (size_t)r0 * ch->Np, nr, false));
    }
    (void)mi;
    CK(cudaStreamSynchronize(par->stream));
    par->kk = ch->kk;
    return 0;
}

#ifndef ACOC_GEN_MIN
#define ACOC_GEN_MIN 4096  // smallest batch that still spawns a survivor generation
#endif

// where acoc_newton_solve_deliver puts the results: device-accessible aliases of the caller's page-locked arrays
struct Delivery {
    void* xx = nullptr;      // (N,6,TT) float or double
    bool x_f32 = false;
    double* uu = nullptr;    // (N,2,TT)
    cudaStream_t stream = nullptr;
};

// optimize()'s result of every instance of `ctx` that is final and not delivered yet, straight into the caller's arrays: selection on
// the context's own stream (which must be idle: call between two driver calls), copies on the delivery stream behind it.
// Returns through *n_new how many instances this delivery carries (0: nothing launched).
static int deliver_finished(acoc_ctx* ctx, const Delivery& dv, int* n_new)
{
    const int N = ctx->N, TT = ctx->TT, Np = ctx->Np;
    if (!ctx->delivered) {
        TRY(dalloc(ctx, &ctx->delivered, (size_t)Np));
        TRY(dalloc(ctx, &ctx->deliver_rows, (size_t)Np));
        CK(cudaEventCreateWithFlags(&ctx->ev_deliver, cudaEventDisableTiming));
    }
    int* cnt = ctx->counters + 3;
    CK(cudaMemsetAsync(cnt, 0, sizeof(int), ctx->stream));
    // (the rows table of the previous delivery of this context may still be in use: wait for it on the solver's stream)
    CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_deliver, 0));
    k_deliver_select<<<(N + 255) / 256, 256, 0, ctx->stream>>>(ctx->S.status, ctx->uidx, ctx->delivered, ctx->deliver_rows, cnt, N);
    CK(cudaGetLastError());
    int h = 0;
    CK(cudaMemcpyAsync(&h, cnt, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaEventRecord(ctx->ev_deliver, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (n_new) *n_new = h;
    ctx->n_delivered += h;
    if (h == 0) return 0;
    CK(cudaStreamWaitEvent(dv.stream, ctx->ev_deliver, 0));
    const dim3 block(32, 8);
    static const int ctas = getenv("ACOC_DELIVER_CTAS") ? atoi(getenv("ACOC_DELIVER_CTAS")) : 64;  // (8: 536 ms, 16: 373, 32: 293, 64: 281 ms end to end; a machine-filling grid: 320)
    const int gx = std::max(1, ctas), gu = gx;
    const int *rs = ctx->S.result_slot, *rows = ctx->deliver_rows;
    // k_deliver<D, O>: the three slots s (elements of type D) into dst (elements of type O)
    const auto deliver = [&](auto d, auto o, int grid, void* const* s, const double* row0, void* dst, int C, int dup_last) {
        using D = typename decltype(d)::type;
        using O = typename decltype(o)::type;
        k_deliver<D, O><<<grid, block, 0, dv.stream>>>((const D*)s[0], (const D*)s[1], (const D*)s[2], rs, rows, row0, (O*)dst, N, C, TT, Np, dup_last);
        return 0;
    };
    if (ctx->x_float)  // float32 values: delivered as float, or as double with the exact row 0
        with_real(dv.x_f32, [&](auto O) {
            return deliver(type_tag<float>{}, O, gx, ctx->X, dv.x_f32 || ctx->fp32 ? nullptr : (const double*)ctx->x0, dv.xx, 6, 0);
        });
    else
        deliver(type_tag<double>{}, type_tag<double>{}, gx, ctx->X, nullptr, dv.xx, 6, 0);
    CK(cudaGetLastError());
    with_real(ctx->fp32, [&](auto D) {
        return deliver(D, type_tag<double>{}, gu, ctx->U, nullptr, dv.uu, 2, 1);  // uu_star[:,-1] = uu_star[:,-2], optcon.py:505
    });
    CK(cudaGetLastError());
    CK(cudaEventRecord(ctx->ev_deliver, dv.stream));  // the rows table is free again once these copies are done
    return 0;
}

static int reset_delivery(acoc_ctx* ctx)
{
    ctx->n_delivered = 0;
    if (ctx->delivered) CK(cudaMemsetAsync(ctx->delivered, 0, (size_t)ctx->Np * sizeof(int), ctx->stream));
    return 0;
}

static int solve_impl(acoc_ctx* c, long long* total_iters, const Delivery* dv)
{
    TRY(ready(c));
    if (dv) TRY(reset_delivery(c));
    int active = 1;
    double total_ms = 0, phase[6] = {0, 0, 0, 0, 0, 0}, gen_ms = 0;
    long long launches = 0;
    std::vector<acoc_ctx*> chain{c};
    acoc_ctx* cur = c;
    while (active > 0 && cur->kk < cur->O.max_iters - 1) {
        // check for completion every 4 iterations: one tiny D2H per check keeps the stream busy in between.  In the clean phase (no
        // failing search in the last iteration seen) nothing converges yet and the many-range split of acoc_newton_iterate needs
        // longer calls to amortise its fill and drain: 8 iterations per call there.
        const bool clean = cur->last_need >= 0 && (long long)cur->last_need * 2048 < cur->N;
        const int kk_before = cur->kk;
        TRY(acoc_newton_iterate(cur, clean ? 8 : 4, &active));
        total_ms += cur->total_ms; launches += cur->launches;
        static const bool trace = getenv("ACOC_TRACE") != nullptr;  // diagnostics: one line per call of the lock-step driver
        if (trace)
            fprintf(stderr, "acoc_trace gen=%zu n=%d kk=%d..%d active_after=%d need_last=%d ms=%.3f launches=%lld\n", chain.size() - 1, cur->N, kk_before,
                    cur->kk - 1, active, cur->last_need, cur->total_ms, cur->launches);
        for (int p = 0; p < 6; ++p) phase[p] += cur->phase_ms[p];
        // (Deliveries between spawns -- whenever another 1/deliver_div of the batch has finished -- were measured too: the copies then run
        // beside the throughput-bound iterations of the noise phase and slow them by more than they hide: 0.317 s end to end against
        // 0.295 s with deliveries at the spawns only.  Off by default.)
        static const int deliver_div = getenv("ACOC_DELIVER_DIV") ? atoi(getenv("ACOC_DELIVER_DIV")) : 0;
        if (dv && deliver_div > 0 && active > 0 && (long long)(cur->N - active - cur->n_delivered) * deliver_div >= cur->N) TRY(deliver_finished(cur, *dv, nullptr));
        if (active > 0 && !(c->flags & ACOC_SOLVE_IN_PLACE) && cur->N >= ACOC_GEN_MIN && 2 * active <= cur->N && cur->kk < cur->O.max_iters - 1) {
            acoc_ctx* ch = nullptr;
            CK(cudaEventRecord(cur->ev[6], cur->stream));
            int rc = spawn_child(cur, active, &ch);
            if (rc < 0) return rc;
            if (rc == 0 && ch) {
                if (dv) {
                    // the finished instances of `cur` are final: deliver them now, while the survivors iterate in the child
                    TRY(reset_delivery(ch));
                    if (!ch->uidx) TRY(dalloc(ch, &ch->uidx, (size_t)ch->Np));
                    k_compose_uidx<<<(active + 255) / 256, 256, 0, cur->stream>>>(ch->origin, cur->uidx, ch->uidx, active);
                    CK(cudaGetLastError());
                }
                CK(cudaEventRecord(cur->ev[7], cur->stream));
                CK(cudaEventSynchronize(cur->ev[7]));
                float ms = 0;
                CK(cudaEventElapsedTime(&ms, cur->ev[6], cur->ev[7]));
                gen_ms += ms;
                if (dv) TRY(deliver_finished(cur, *dv, nullptr));
                chain.push_back(ch);
                cur = ch;
            }
        }
    }
    if (dv) {
        // whatever `cur` (the last generation, or the batch itself) still holds: instances that ran out of iterations while active get
        // their status from the driver, so everything is final here
        TRY(deliver_finished(cur, *dv, nullptr));
        CK(cudaStreamSynchronize(dv->stream));  // (the folds below rewrite rows of the parents; keep them behind the deliveries)
    }
    for (size_t k = chain.size() - 1; k >= 1; --k) {
        acoc_ctx* par = chain[k - 1];
        CK(cudaEventRecord(par->ev[6], par->stream));
        TRY(fold_child(par, chain[k]));
        CK(cudaEventRecord(par->ev[7], par->stream));
        CK(cudaEventSynchronize(par->ev[7]));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, par->ev[6], par->ev[7]));
        gen_ms += ms;
    }
    c->total_ms = total_ms + gen_ms; c->launches = launches; c->gen_ms = gen_ms;
    for (int p = 0; p < 6; ++p) c->phase_ms[p] = phase[p];
    c->phase_ms[4] = gen_ms;  // reported as the "select" slot of acoc_get_timing: time spent moving instances between generations
    if (total_iters) TRY(count_active(c, nullptr, total_iters));
    return 0;
}

int acoc_newton_solve(acoc_ctx* c, long long* total_iters) { return solve_impl(c, total_iters, nullptr); }

// device alias of a page-locked host pointer, or NULL for pageable memory
static void* pinned_alias(const void* host)
{
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, host) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    if (at.type != cudaMemoryTypeHost || !at.devicePointer) return nullptr;
    return at.devicePointer;
}

int acoc_newton_solve_deliver(acoc_ctx* c, void* xx_star, int x_is_f32, double* uu_star, double* x0, long long* total_iters)
{
    TRY(ready(c));
    REQUIRE(xx_star && uu_star, "NULL output");
    if (x_is_f32 && !(c->x_float))
        return fail(ACOC_ERR_STATE, "acoc_newton_solve_deliver: float32 states requested but the state iterates of this context are not float32 values");
    void* dx = pinned_alias(xx_star);
    void* du = pinned_alias(uu_star);
    if (!dx || !du) {  // pageable buffers: solve, then the staged download
        TRY(solve_impl(c, total_iters, nullptr));
        if (x_is_f32) return acoc_get_result_f32(c, (float*)xx_star, uu_star, x0);
        TRY(acoc_get_result(c, (double*)xx_star, uu_star));
    } else {
        if (!c->dstream) CK(cudaStreamCreateWithFlags(&c->dstream, cudaStreamNonBlocking));
        Delivery dv;
        dv.xx = dx; dv.x_f32 = x_is_f32 != 0; dv.uu = (double*)du; dv.stream = c->dstream;
        TRY(solve_impl(c, total_iters, &dv));
    }
    if (x0) {  // exact x0 = xx_init[:,0] (optcon.py:398): device [6][Np] -> host (N,6)
        const size_t Np = c->Np;
        std::vector<double> tmp(6 * Np);
        if (c->fp32) {
            std::vector<float> t32(6 * Np);
            CK(cudaMemcpyAsync(t32.data(), c->x0, t32.size() * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
            CK(cudaStreamSynchronize(c->stream));
            for (size_t k = 0; k < t32.size(); ++k) tmp[k] = t32[k];
        } else {
            CK(cudaMemcpyAsync(tmp.data(), c->x0, tmp.size() * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
            CK(cudaStreamSynchronize(c->stream));
        }
        for (int i = 0; i < c->N; ++i) for (int k = 0; k < 6; ++k) x0[(size_t)i * 6 + k] = tmp[k * Np + i];
    }
    return 0;
}

int acoc_sync(acoc_ctx* c)
{
    REQUIRE(c, "ctx is NULL");
    TRY(use_device(c->device));
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

int acoc_eval_cost(acoc_ctx* c, double* J)
{
    TRY(ready(c));
    TRY(launch_cost(c));
    if (J) { CK(cudaMemcpyAsync(J, c->S.Jcur, c->N * sizeof(double), cudaMemcpyDeviceToHost, c->stream)); }
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

int acoc_backward(acoc_ctx* c, int exact)
{
    TRY(ready(c));
    TRY(launch_build_active(c));
    TRY(launch_backward(c, exact != 0));
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

int acoc_forward(acoc_ctx* c, double* descent)
{
    TRY(ready(c));
    TRY(launch_build_active(c));
    TRY(launch_forward(c));
    if (descent) { CK(cudaMemcpyAsync(descent, c->S.descent, c->N * sizeof(double), cudaMemcpyDeviceToHost, c->stream)); }
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

int acoc_gradient(acoc_ctx* c, double* descent)
{
    TRY(ready(c));
    TRY(launch_build_active(c));
    TRY(launch_gradient(c));
    if (descent) {  // the reference's descent[kk] = sum |deltau|^2 (optcon.py:118); the context keeps the slope -descent
        std::vector<double> tmp(c->N);
        CK(cudaMemcpyAsync(tmp.data(), c->S.descent, c->N * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        for (int i = 0; i < c->N; ++i) descent[i] = -tmp[i];
    }
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

template <typename F>
static int launch_all_candidates_t(acoc_ctx* c)
{
    const int cur = c->kk % 3, N = c->N, nc = c->O.armijo_maxiters;
    WorkList L;
    L.groups = nullptr; L.count = c->counters + 1; L.shift = 0;
    launch_candidates<F>(c, L, N, (const F*)c->U[cur], (const F*)c->DU, c->cand_steps, 0, nc, c->stream);
    CK(cudaGetLastError());
    return 0;
}

int acoc_armijo(acoc_ctx* c, double* stepsize, double* costs)
{
    TRY(ready(c));
    REQUIRE(c->kk < c->O.max_iters, "iteration counter exhausted");
    // always the speculative evaluation here: this entry point reports the cost of every candidate
    const int N = c->N, nc = c->O.armijo_maxiters;
    TRY(DISPATCH_F(c, launch_all_candidates_t, c));
    k_select<<<(N + 255) / 256, 256, 0, c->stream>>>(c->O, c->S, c->cand_steps, c->kk, 0, N, c->Np);
    CK(cudaGetLastError());
    if (stepsize) CK(cudaMemcpyAsync(stepsize, c->S.step, N * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    if (costs) {  // device [nc][Np] -> host [N][nc]
        std::vector<double> tmp((size_t)nc * c->Np);
        CK(cudaMemcpy(tmp.data(), c->S.Jcand, tmp.size() * sizeof(double), cudaMemcpyDeviceToHost));
        for (int i = 0; i < N; ++i) for (int k = 0; k < nc; ++k) costs[(size_t)i * nc + k] = tmp[(size_t)k * c->Np + i];
    }
    return 0;
}

// cost of u + steps[k]*deltau for arbitrary step sizes, every instance (the visu_armijo sweep, optcon.py:282-296): the candidate
// kernel with a caller-supplied step table, armijo_maxiters steps per launch
template <typename F>
static int launch_sweep_candidates_t(acoc_ctx* c, const double* dsteps, int n)
{
    const int cur = c->kk % 3, N = c->N;
    WorkList L;
    L.groups = nullptr; L.count = c->counters + 1; L.shift = 0;
    launch_candidates<F>(c, L, N, (const F*)c->U[cur], (const F*)c->DU, dsteps, 0, n, c->stream);
    CK(cudaGetLastError());
    return 0;
}

int acoc_armijo_sweep(acoc_ctx* c, int n_steps, const double* steps, double* costs)
{
    TRY(ready(c));
    REQUIRE(n_steps >= 1 && steps && costs, "need n_steps >= 1, steps and costs");
    const int N = c->N, chunk = c->O.armijo_maxiters;
    double* dsteps = nullptr;
    CK(cudaMalloc(&dsteps, sizeof(double) * chunk));
    std::vector<double> tmp((size_t)chunk * c->Np);
    int rc = 0;
    for (int k0 = 0; k0 < n_steps && !rc; k0 += chunk) {
        const int n = std::min(chunk, n_steps - k0);
        if (cudaMemcpyAsync(dsteps, steps + k0, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream) != cudaSuccess) { rc = fail(ACOC_ERR_CUDA, "H2D of the step table failed"); break; }
        rc = DISPATCH_F(c, launch_sweep_candidates_t, c, dsteps, n);
        if (rc) break;
        if (cudaMemcpyAsync(tmp.data(), c->S.Jcand, (size_t)n * c->Np * sizeof(double), cudaMemcpyDeviceToHost, c->stream) != cudaSuccess ||
            cudaStreamSynchronize(c->stream) != cudaSuccess) { rc = fail(ACOC_ERR_CUDA, "D2H of the sweep costs failed: %s", cudaGetErrorString(cudaGetLastError())); break; }
        for (int i = 0; i < N; ++i) for (int k = 0; k < n; ++k) costs[(size_t)i * n_steps + k0 + k] = tmp[(size_t)k * c->Np + i];
    }
    cudaFree(dsteps);
    return rc;
}

int acoc_update(acoc_ctx* c, const double* stepsize)
{
    TRY(ready(c));
    REQUIRE(c->kk < c->O.max_iters - 1, "iteration counter exhausted");
    if (stepsize) CK(cudaMemcpyAsync(c->S.step, stepsize, c->N * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    TRY(launch_update(c, false, false, false));
    ++c->kk;
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

int acoc_set_deltau(acoc_ctx* c, const double* deltau)
{
    REQUIRE(c && deltau, "NULL argument");
    TRY(use_device(c->device));
    return upload_soa(c, deltau, c->DU, c->N, 2, c->Np);
}

int acoc_set_scalars(acoc_ctx* c, const double* J, const double* descent)
{
    REQUIRE(c, "ctx is NULL");
    TRY(use_device(c->device));
    if (J) CK(cudaMemcpyAsync(c->S.Jcur, J, c->N * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    if (descent) CK(cudaMemcpyAsync(c->S.descent, descent, c->N * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

// ======================================================================================================
// read-back
// ======================================================================================================
int acoc_get_result(acoc_ctx* c, double* xx_star, double* uu_star)
{
    TRY(ready(c));
    REQUIRE(xx_star && uu_star, "NULL output");
    k_result_slot_default<<<(c->N + 255) / 256, 256, 0, c->stream>>>(c->S.status, c->slot_tmp, c->S.result_slot, c->kk % 3, c->N);
    CK(cudaGetLastError());
    TRY(download_x(c, c->slot_tmp, xx_star));
    TRY(download_soa(c, c->U[0], c->U[1], c->U[2], c->slot_tmp, uu_star, c->N, 2, c->Np, 1));  // uu_star[:,-1] = uu_star[:,-2], optcon.py:505
    return 0;
}

int acoc_get_refs(acoc_ctx* c, double* xx_ref, double* uu_ref)
{
    REQUIRE(c && (xx_ref || uu_ref), "NULL argument");
    if (!c->have_refs) return fail(ACOC_ERR_STATE, "acoc_get_refs: no references set");
    TRY(use_device(c->device));
    const int n = c->P.ref_shared ? 1 : c->N, Np = c->P.ref_shared ? 1 : c->Np;
    if (c->P.ref_param) {  // write the parametric references out in the expanded layout (the arrays are otherwise unused in this mode)
        const dim3 grid((unsigned)((c->N + 127) / 128), (unsigned)std::min(c->TT, 64));
        k_expand_refs<<<grid, 128, 0, c->stream>>>(prob<double>(c), (double*)c->xref, (double*)c->uref);
        CK(cudaGetLastError());
    }
    if (xx_ref) TRY(download_soa(c, c->xref, nullptr, nullptr, nullptr, xx_ref, n, 6, Np, 0));
    if (uu_ref) TRY(download_soa(c, c->uref, nullptr, nullptr, nullptr, uu_ref, n, 2, Np, 0));
    return 0;
}

int acoc_get_result_f32(acoc_ctx* c, float* xx_star, double* uu_star, double* x0)
{
    TRY(ready(c));
    REQUIRE(xx_star && uu_star, "NULL output");
    if (!c->x_float)
        return fail(ACOC_ERR_STATE, "acoc_get_result_f32: the state iterates of this context are not float32 values (ACOC_STATE_F64, "
                                    "ACOC_X_F64 or an initial trajectory with float64 states); use acoc_get_result");
    k_result_slot_default<<<(c->N + 255) / 256, 256, 0, c->stream>>>(c->S.status, c->slot_tmp, c->S.result_slot, c->kk % 3, c->N);
    CK(cudaGetLastError());
    TRY((download_soa_t<float, float>(c, c->X[0], c->X[1], c->X[2], c->slot_tmp, nullptr, xx_star, c->N, 6, c->Np, 0)));
    TRY(download_soa(c, c->U[0], c->U[1], c->U[2], c->slot_tmp, uu_star, c->N, 2, c->Np, 1));  // uu_star[:,-1] = uu_star[:,-2], optcon.py:505
    if (x0) {  // device [6][Np] -> host (N,6); float64 unless the context computes in FP32
        const size_t Np = c->Np;
        if (c->fp32) {
            std::vector<float> tmp(6 * Np);
            CK(cudaMemcpyAsync(tmp.data(), c->x0, tmp.size() * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
            CK(cudaStreamSynchronize(c->stream));
            for (int i = 0; i < c->N; ++i) for (int k = 0; k < 6; ++k) x0[(size_t)i * 6 + k] = tmp[k * Np + i];
        } else {
            std::vector<double> tmp(6 * Np);
            CK(cudaMemcpyAsync(tmp.data(), c->x0, tmp.size() * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
            CK(cudaStreamSynchronize(c->stream));
            for (int i = 0; i < c->N; ++i) for (int k = 0; k < 6; ++k) x0[(size_t)i * 6 + k] = tmp[k * Np + i];
        }
    }
    return 0;
}

int acoc_get_iterate(acoc_ctx* c, int which, double* xx, double* uu)
{
    TRY(ready(c));
    REQUIRE(which == 0 || which == 1, "which must be 0 (newest) or 1 (previous)");
    k_iterate_slot<<<(c->N + 255) / 256, 256, 0, c->stream>>>(c->S.iters, which, c->slot_tmp, c->N);
    CK(cudaGetLastError());
    if (xx) TRY(download_x(c, c->slot_tmp, xx));
    if (uu) TRY(download_soa(c, c->U[0], c->U[1], c->U[2], c->slot_tmp, uu, c->N, 2, c->Np, 0));
    return 0;
}

int acoc_get_deltau(acoc_ctx* c, double* deltau)
{
    TRY(ready(c));
    REQUIRE(deltau, "NULL output");
    return download_soa(c, c->DU, nullptr, nullptr, nullptr, deltau, c->N, 2, c->Np, 0);
}

int acoc_get_gains(acoc_ctx* c, double* K, double* sigma)
{
    TRY(ready(c));
    // KSG is a warp-tiled trajectory with 16 components; as a "C = 16" trajectory it downloads to (N,16,TT): rows 0..11 = K (2x6 row-major), 12..13 = sigma
    std::vector<double> tmp((size_t)c->N * 16 * c->TT);
    TRY(download_soa(c, c->KSG, nullptr, nullptr, nullptr, tmp.data(), c->N, 16, c->Np, 0));
    const size_t TT = c->TT;
    for (int i = 0; i < c->N; ++i) {
        const double* src = tmp.data() + (size_t)i * 16 * TT;
        if (K) memcpy(K + (size_t)i * 12 * TT, src, 12 * TT * sizeof(double));
        if (sigma) memcpy(sigma + (size_t)i * 2 * TT, src + 12 * TT, 2 * TT * sizeof(double));
    }
    return 0;
}

template <typename T>
static int get_hist(acoc_ctx* c, const T* dev, T* host)
{
    if (!host) return 0;
    const int mi = c->O.max_iters;
    std::vector<T> tmp((size_t)mi * c->Np);
    CK(cudaMemcpyAsync(tmp.data(), dev, tmp.size() * sizeof(T), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    for (int i = 0; i < c->N; ++i) for (int k = 0; k < mi; ++k) host[(size_t)i * mi + k] = tmp[(size_t)k * c->Np + i];
    return 0;
}

int acoc_get_history(acoc_ctx* c, double* JJ, double* descent, double* stepsize, int* n_cand)
{
    REQUIRE(c, "ctx is NULL");
    TRY(use_device(c->device));
    TRY(get_hist(c, c->S.hist_J, JJ)); TRY(get_hist(c, c->S.hist_descent, descent));
    TRY(get_hist(c, c->S.hist_step, stepsize)); TRY(get_hist(c, c->S.hist_ncand, n_cand));
    return 0;
}

int acoc_get_stats(acoc_ctx* c, int* iters, int* status, double* J, double* descent, int* n_reg)
{
    REQUIRE(c, "ctx is NULL");
    TRY(use_device(c->device));
    const size_t N = c->N;
    if (iters) CK(cudaMemcpyAsync(iters, c->S.iters, N * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    if (status) CK(cudaMemcpyAsync(status, c->S.status, N * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    if (J) CK(cudaMemcpyAsync(J, c->S.Jcur, N * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    if (descent) CK(cudaMemcpyAsync(descent, c->S.descent, N * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    if (n_reg) CK(cudaMemcpyAsync(n_reg, c->S.n_reg, N * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

int acoc_get_timing(acoc_ctx* c, double* total_ms, double phase_ms[6], long long* kernel_launches)
{
    REQUIRE(c, "ctx is NULL");
    if (total_ms) *total_ms = c->total_ms;
    if (phase_ms) for (int p = 0; p < 6; ++p) phase_ms[p] = c->phase_ms[p];
    if (kernel_launches) *kernel_launches = c->launches;
    return 0;
}

int acoc_set_profiling(acoc_ctx* c, int on)
{
    REQUIRE(c, "ctx is NULL");
    c->profiling = on != 0;
    return 0;
}

// ======================================================================================================
// lqr_tracking
// ======================================================================================================
int acoc_lqr_tracking(int device, int n, int TT, const double* params, int state_f64, const double* Q, const double* R, const double* QT,
                      const double* xx_opt, const double* uu_opt, const double* delta, double* xx_reg, double* uu_reg, double* K)
{
    REQUIRE(n > 0 && TT >= 3 && params && Q && R && QT && xx_opt && uu_opt && delta && xx_reg && uu_reg, "acoc_lqr_tracking: bad argument");
    // the rollout context (one trajectory slot for n instances + staging) is kept between calls of the same size: creating it costs
    // more than the tracking itself (~0.5 GB of cudaMalloc + memset for 4096 instances)
    static std::mutex mu;
    static acoc_ctx* cached = nullptr;
    std::lock_guard<std::mutex> lock(mu);
    const unsigned flags = (state_f64 ? ACOC_STATE_F64 : 0) | ACOC_REFS_SHARED | ACOC_CTX_LITE;
    if (cached && (cached->device != device || cached->N != n || cached->TT != TT || cached->flags != flags)) { acoc_ctx_destroy(cached); cached = nullptr; }
    if (!cached) TRY(acoc_ctx_create(device, n, TT, flags, &cached));
    acoc_ctx* c = cached;
    TRY(use_device(device));
    TRY(acoc_set_model(c, params));
    const Model M = c->P.M;
    // nominal trajectory, time-major [TT][6] / [TT][2] (this is exactly the "shared reference" SoA layout)
    TRY(upload_soa(c, xx_opt, c->xref, 1, 6, 1));
    TRY(upload_soa(c, uu_opt, c->uref, 1, 2, 1));
    // linearise along the nominal at all TT points (lqr_tracking.py:268-273): one thread per time step
    TmpBuf t(device);
    double *dA, *dB, *dQ, *dR, *dS, *dQf, *dx0, *dK, *dxo, *duo, *dstart;
    TRY(t.out(&dA, xx_reg, (size_t)TT * 36)); TRY(t.out(&dB, xx_reg, (size_t)TT * 12)); TRY(t.out(&dS, xx_reg, (size_t)TT * 12));
    TRY(t.out(&dK, xx_reg, (size_t)TT * 12)); TRY(t.out(&dxo, xx_reg, (size_t)TT * 6)); TRY(t.out(&duo, xx_reg, (size_t)TT * 2));
    std::vector<double> Qrep((size_t)TT * 36), Rrep((size_t)TT * 4);
    for (int k = 0; k < TT; ++k) { memcpy(&Qrep[(size_t)k * 36], Q, 36 * sizeof(double)); memcpy(&Rrep[(size_t)k * 4], R, 4 * sizeof(double)); }  // .repeat(TT), optcon.py:603-606
    TRY(t.up(&dQ, Qrep.data(), Qrep.size())); TRY(t.up(&dR, Rrep.data(), Rrep.size())); TRY(t.up(&dQf, QT, 36)); TRY(t.up(&dx0, delta, 6));
    // perturbed initial states: x_start[c][i] = xx_opt[c][0] + delta[i][c]   (lqr_tracking.py:265)
    std::vector<double> xs((size_t)6 * c->Np, 0.0);
    for (int i = 0; i < n; ++i) for (int k = 0; k < 6; ++k) xs[(size_t)k * c->Np + i] = xx_opt[(size_t)k * TT] + delta[(size_t)i * 6 + k];
    TRY(t.up(&dstart, xs.data(), xs.size()));
    // the uploads and memsets above ran on the legacy default stream; the context's stream is non-blocking, so order them explicitly
    CK(cudaDeviceSynchronize());
    const double *d_xopt = (const double*)c->xref, *d_uopt = (const double*)c->uref;
    CK(cudaEventRecord(c->ev[0], c->stream));
    k_step_batch<<<(TT + 127) / 128, 128, 0, c->stream>>>(M, c->P.q32, TT, d_xopt, d_uopt, nullptr, nullptr, dA, dB, nullptr, nullptr);
    CK(cudaGetLastError());
    TRY(lq_dense_dev(1, TT, false, dA, dB, dQ, dR, dS, dQf, dx0, nullptr, nullptr, nullptr, dK, nullptr, dxo, duo, nullptr, c->stream));
    CK(cudaEventRecord(c->ev[1], c->stream));
    const Problem P = prob<double>(c);
    with_flag(c->P.q32, [&](auto Q) {
        k_track<Q><<<(n + ROLL_THREADS - 1) / ROLL_THREADS, ROLL_THREADS, 0, c->stream>>>(P, dK, d_xopt, d_uopt, dstart, (double*)c->X[0],
                                                                                          (double*)c->U[0]);
        return 0;
    });
    CK(cudaGetLastError());
    CK(cudaEventRecord(c->ev[2], c->stream));
    TRY(download_soa(c, c->X[0], nullptr, nullptr, nullptr, xx_reg, n, 6, c->Np, 0));
    TRY(download_soa(c, c->U[0], nullptr, nullptr, nullptr, uu_reg, n, 2, c->Np, 0));
    {
        float a = 0, b = 0;
        CK(cudaEventElapsedTime(&a, c->ev[0], c->ev[1]));
        CK(cudaEventElapsedTime(&b, c->ev[1], c->ev[2]));
        g_pt_ms[0] = (double)a + b; g_pt_ms[1] = a; g_pt_ms[2] = b;
    }
    if (K) CK(cudaMemcpy(K, dK, (size_t)TT * 12 * sizeof(double), cudaMemcpyDeviceToHost));
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

int acoc_last_pointwise_timing(double* ms)
{
    REQUIRE(ms, "NULL output");
    for (int k = 0; k < 3; ++k) ms[k] = g_pt_ms[k];
    return 0;
}

// ======================================================================================================
// closed-loop LQR tracking of every instance along its own nominal (lqr_tracking.py:245-283 per instance)
// ======================================================================================================
static void free_track_buffers(acoc_ctx* c)
{
    dfree(c, &c->tk_xnom); dfree(c, &c->tk_unom); dfree(c, &c->tk_xnom0); dfree(c, &c->tk_K); dfree(c, &c->tk_x); dfree(c, &c->tk_x0);
    dfree(c, &c->tk_u); dfree(c, &c->tk_delta); dfree(c, &c->tk_emax); dfree(c, &c->tk_efin); dfree(c, &c->tk_nreg);
    c->tk_es = 0;
    c->tk_done = false;
    c->tk_swept = false;
}

// the buffers of the nominal, the gains and the per-instance summaries, for state elements of es bytes (reallocated when the storage
// type changes); ACOC_ERR_NOMEM leaves none behind
static int ensure_track_buffers(acoc_ctx* c, size_t es)
{
    if (c->tk_es == es) return 0;
    CK(cudaStreamSynchronize(c->stream));
    free_track_buffers(c);
    const size_t T = c->TT, Np = c->Np, d = sizeof(double);
    int rc = dalloc_bytes(c, &c->tk_xnom, T * NS * Np * es);
    if (!rc) rc = dalloc_bytes(c, &c->tk_unom, T * NI * Np * d);
    if (!rc) rc = dalloc_bytes(c, &c->tk_K, T * 2 * NS * Np * d);
    if (!rc) rc = dalloc_bytes(c, &c->tk_xnom0, NS * Np * d);
    if (!rc) rc = dalloc_bytes(c, &c->tk_delta, NS * Np * d);
    if (!rc) rc = dalloc_bytes(c, &c->tk_emax, NS * Np * d);
    if (!rc) rc = dalloc_bytes(c, &c->tk_efin, NS * Np * d);
    if (!rc) rc = dalloc(c, &c->tk_nreg, Np);
    for (auto& e : c->tk_ev)
        if (!rc && !e && cudaEventCreate(&e) != cudaSuccess) rc = fail(ACOC_ERR_CUDA, "cudaEventCreate failed");
    if (rc) { free_track_buffers(c); return rc; }
    c->tk_es = es;
    return 0;
}

// the tracked trajectories Xtrk / Utrk and their exact row 0, which only acoc_track and acoc_lqr_tracking_many write (after
// ensure_track_buffers); ACOC_ERR_NOMEM leaves no tracking buffer behind
static int ensure_tracked_buffers(acoc_ctx* c)
{
    if (c->tk_x) return 0;
    const size_t T = c->TT, Np = c->Np, d = sizeof(double);
    int rc = dalloc_bytes(c, &c->tk_x, T * NS * Np * c->tk_es);
    if (!rc) rc = dalloc_bytes(c, &c->tk_u, T * NI * Np * d);
    if (!rc) rc = dalloc_bytes(c, &c->tk_x0, NS * Np * d);
    if (rc) free_track_buffers(c);
    return rc;
}

// the dispersion buffers for n * m samples (96 B each) and `delta_bytes` of deltas, grown when too small.  The new buffers are allocated
// before the old ones are released, so ACOC_ERR_NOMEM leaves the context as it was.
static int ensure_mc_buffers(acoc_ctx* c, size_t samples, size_t delta_bytes)
{
    const size_t sum_bytes = samples * 2 * NS * sizeof(double);
    void *ns = nullptr, *nd = nullptr;
    int* nw = nullptr;
    int rc = 0;
    if (c->mc_sum_cap < sum_bytes) rc = dalloc_bytes(c, &ns, sum_bytes);
    if (!rc && c->mc_delta_cap < delta_bytes) rc = dalloc_bytes(c, &nd, delta_bytes);
    if (!rc && !c->mc_nw) rc = dalloc(c, &nw, c->Np);
    if (rc) { dfree(c, &ns); dfree(c, &nd); dfree(c, &nw); return rc; }
    if (ns || nd) CK(cudaStreamSynchronize(c->stream));
    if (ns) { dfree(c, &c->mc_sum); c->mc_sum = ns; c->mc_sum_cap = sum_bytes; }
    if (nd) { dfree(c, &c->mc_delta); c->mc_delta = nd; c->mc_delta_cap = delta_bytes; }
    if (nw) c->mc_nw = nw;
    return 0;
}

// Q, R, QT of the tracking cost: symmetric like acoc_set_weights (the gains sweep carries P as its upper triangle)
static int track_weights(const double* Q, const double* R, const double* QT, Weights* W)
{
    REQUIRE(Q && R && QT, "tracking weights: NULL argument");
    REQUIRE(is_sym(Q, 6) && is_sym(R, 2) && is_sym(QT, 6), "tracking weights: Q, R and QT must be symmetric");
    fill_weights(W, Q, R, QT);
    return 0;
}

// host delta (N,6) or NULL (zeros) -> device [6][Np]
static int upload_delta(acoc_ctx* c, const double* delta)
{
    if (!delta) { CK(cudaMemsetAsync(c->tk_delta, 0, (size_t)NS * c->Np * sizeof(double), c->stream)); return 0; }
    std::vector<double> tmp((size_t)NS * c->Np, 0.0);
    for (int i = 0; i < c->N; ++i) for (int k = 0; k < NS; ++k) tmp[(size_t)k * c->Np + i] = delta[(size_t)i * NS + k];
    CK(cudaMemcpyAsync(c->tk_delta, tmp.data(), tmp.size() * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    CK(cudaStreamSynchronize(c->stream));  // tmp goes out of scope
    return 0;
}

// the problem the tracking sweeps see: tracking weights, x0 = the exact row 0 of the nominal (finish_x)
static Problem track_problem(acoc_ctx* c, const Weights& W)
{
    Problem P = prob<double>(c);
    P.W = W;
    P.x0 = (const double*)c->tk_xnom0;
    return P;
}

// gains sweep over the nominal in tk_xnom / tk_unom / tk_xnom0 (events tk_ev[1..2])
template <typename XT>
static int launch_track_gains(acoc_ctx* c, const Problem& P)
{
    const XT* Xn = (const XT*)c->tk_xnom;
    const double* Un = (const double*)c->tk_unom;
    double* K = (double*)c->tk_K;
    cudaStream_t st = c->stream;
    const int g = (c->N + 63) / 64;  // 64 threads = two tiles per CTA
    CK(cudaEventRecord(c->tk_ev[1], st));
    TRY(with_flag(P.W.diag != 0, [&](auto DG) {
        if (use_tma(c))
            return launch_ring(k_track_gains_tma<DG, XT>, g, 64, WarpRing<TRK_GAIN_STAGES, TrkGainStage<XT>::BYTES>::smem_bytes(2), st, P, Xn, Un, K,
                               c->tk_nreg);
        k_track_gains<DG, XT><<<g, 64, 0, st>>>(P, Xn, Un, K, c->tk_nreg);
        return 0;
    }));
    CK(cudaGetLastError());
    CK(cudaEventRecord(c->tk_ev[2], st));
    return 0;
}

// gains sweep + closed-loop rollout over the nominal (events tk_ev[1..3])
template <typename XT>
static int launch_track_sweeps(acoc_ctx* c, const Weights& W)
{
    const Problem P = track_problem(c, W);
    TRY(launch_track_gains<XT>(c, P));
    const XT* Xn = (const XT*)c->tk_xnom;
    const double *Un = (const double*)c->tk_unom, *dl = (const double*)c->tk_delta;
    double *K = (double*)c->tk_K, *x0 = (double*)c->tk_x0, *U = (double*)c->tk_u, *em = (double*)c->tk_emax, *ef = (double*)c->tk_efin;
    XT* X = (XT*)c->tk_x;
    cudaStream_t st = c->stream;
    const int g = (c->N + 63) / 64;
    TRY(with_flag(c->P.q32, [&](auto Q) {
        if (use_tma(c))
            return launch_ring(k_track_rollout_tma<Q, XT>, g, 64, WarpRing<TRK_ROLL_STAGES, TrkRollStage<XT>::BYTES>::smem_bytes(2), st, P, Xn, Un, K,
                               dl, X, x0, U, em, ef);
        k_track_rollout<Q, XT><<<g, 64, 0, st>>>(P, Xn, Un, K, dl, X, x0, U, em, ef);
        return 0;
    }));
    CK(cudaGetLastError());
    CK(cudaEventRecord(c->tk_ev[3], st));
    return 0;
}

// gains sweep + dispersion rollout of m samples per instance + per-instance reduction (events tk_ev[1..3]); deltas in mc_delta with
// instance stride dstride (doubles)
template <typename XT>
static int launch_track_mc(acoc_ctx* c, const Weights& W, int m, long long dstride, const double* tol)
{
    const Problem P = track_problem(c, W);
    TRY(launch_track_gains<XT>(c, P));
    const XT* Xn = (const XT*)c->tk_xnom;
    const double *Un = (const double*)c->tk_unom, *K = (const double*)c->tk_K, *dl = (const double*)c->mc_delta;
    double* em = (double*)c->mc_sum;
    double* ef = em + (size_t)c->N * m * NS;
    cudaStream_t st = c->stream;
    if (use_tma(c)) {
        const long long lanes = std::min(c->N, TILE);  // live lanes of the fullest tile
        const int cpt = (int)((lanes * m + TRK_MC_WARPS * TILE - 1) / (TRK_MC_WARPS * TILE));
        const long long grid = (long long)n_tiles(c) * cpt;
        REQUIRE(grid <= 0x7fffffffLL, "acoc_track_mc: %d instances x %d samples is too many for one launch", c->N, m);
        TRY(with_flag(c->P.q32, [&](auto Q) {
            return launch_ring(k_track_mc_rollout_tma<Q, XT>, (unsigned)grid, TRK_MC_THREADS, track_mc_smem<XT>(), st, P, Xn, Un, K, dl, dstride, m,
                               cpt, em, ef);
        }));
    } else {
        const long long grid = ((long long)c->N * m + 63) / 64;
        REQUIRE(grid <= 0x7fffffffLL, "acoc_track_mc: %d instances x %d samples is too many for one launch", c->N, m);
        with_flag(c->P.q32, [&](auto Q) {
            k_track_mc_rollout<Q, XT><<<(unsigned)grid, 64, 0, st>>>(P, Xn, Un, K, dl, dstride, m, em, ef);
            return 0;
        });
    }
    CK(cudaGetLastError());
    TrackTol tl{};
    tl.on = tol != nullptr;
    for (int k = 0; k < NS && tol; ++k) tl.v[k] = tol[k];
    k_track_mc_reduce<<<(c->N + 127) / 128, 128, 0, st>>>(em, ef, c->N, c->Np, m, tl, (double*)c->tk_emax, (double*)c->tk_efin, c->mc_nw);
    CK(cudaGetLastError());
    CK(cudaEventRecord(c->tk_ev[3], st));
    return 0;
}

// after the sweeps: wait, read the event times, mark the gains valid and the tracked trajectories valid (acoc_track) or not
static int track_finish(acoc_ctx* c, bool xfloat, bool trajectories)
{
    CK(cudaStreamSynchronize(c->stream));
    float a = 0, b = 0, r = 0;
    CK(cudaEventElapsedTime(&a, c->tk_ev[0], c->tk_ev[1]));
    CK(cudaEventElapsedTime(&b, c->tk_ev[1], c->tk_ev[2]));
    CK(cudaEventElapsedTime(&r, c->tk_ev[2], c->tk_ev[3]));
    c->tk_ms[0] = (double)a + b + r; c->tk_ms[1] = a; c->tk_ms[2] = b; c->tk_ms[3] = r;
    c->tk_swept = true;
    c->tk_done = trajectories;
    c->tk_xfloat = xfloat;
    return 0;
}

static int download_tracked(acoc_ctx* c, double* xx_reg, double* uu_reg)
{
    const double* row0 = (const double*)c->tk_x0;
    if (xx_reg) {
        if (c->tk_xfloat) TRY((download_soa_t<float>(c, c->tk_x, nullptr, nullptr, nullptr, row0, xx_reg, c->N, NS, c->Np, 0)));
        else TRY((download_soa_t<double>(c, c->tk_x, nullptr, nullptr, nullptr, row0, xx_reg, c->N, NS, c->Np, 0)));
    }
    if (uu_reg) TRY((download_soa_t<double>(c, c->tk_u, nullptr, nullptr, nullptr, nullptr, uu_reg, c->N, NI, c->Np, 0)));
    return 0;
}

// device [6][Np] -> host (N,6)
template <typename T>
static int download_rows(acoc_ctx* c, const void* dev, T* host, int rows)
{
    if (!host) return 0;
    std::vector<T> tmp((size_t)rows * c->Np);
    CK(cudaMemcpyAsync(tmp.data(), dev, tmp.size() * sizeof(T), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    for (int i = 0; i < c->N; ++i) for (int k = 0; k < rows; ++k) host[(size_t)i * rows + k] = tmp[(size_t)k * c->Np + i];
    return 0;
}

// the nominal of every lane = its current result (k_result_slot_default + k_track_nominal; event tk_ev[0])
static int copy_track_nominal(acoc_ctx* c, bool xf)
{
    CK(cudaEventRecord(c->tk_ev[0], c->stream));
    k_result_slot_default<<<(c->N + 255) / 256, 256, 0, c->stream>>>(c->S.status, c->slot_tmp, c->S.result_slot, c->kk % 3, c->N);
    const int tchunk = 8;
    const dim3 grid((unsigned)((c->N + 127) / 128), (unsigned)((c->TT + tchunk - 1) / tchunk));
    with_real(xf, [&](auto T) {
        using XT = typename decltype(T)::type;
        k_track_nominal<XT><<<grid, 128, 0, c->stream>>>((const XT*)c->X[0], (const XT*)c->X[1], (const XT*)c->X[2], (const double*)c->U[0],
                                                         (const double*)c->U[1], (const double*)c->U[2], c->slot_tmp, (const double*)c->x0,
                                                         (XT*)c->tk_xnom, (double*)c->tk_unom, (double*)c->tk_xnom0, c->N, c->Np, c->TT, tchunk);
        return 0;
    });
    CK(cudaGetLastError());
    return 0;
}

static int track_ctx_check(acoc_ctx* c, const char* fn)
{
    REQUIRE(c, "ctx is NULL");
    if (c->fp32) return fail(ACOC_ERR_STATE, "%s: not available in the FP32 mode (ACOC_FP32)", fn);
    if (!c->have_init) return fail(ACOC_ERR_STATE, "%s: no iterate to track yet: call acoc_set_init or acoc_init_guess first", fn);
    return 0;
}

int acoc_track(acoc_ctx* c, const double* Q, const double* R, const double* QT, const double* delta, double* err_max, double* err_final,
               int* n_reg)
{
    TRY(track_ctx_check(c, "acoc_track"));
    Weights W;
    TRY(track_weights(Q, R, QT, &W));
    TRY(use_device(c->device));
    const bool xf = c->x_float;
    TRY(ensure_track_buffers(c, xf ? sizeof(float) : sizeof(double)));
    TRY(ensure_tracked_buffers(c));
    TRY(upload_delta(c, delta));
    TRY(copy_track_nominal(c, xf));
    TRY(xf ? launch_track_sweeps<float>(c, W) : launch_track_sweeps<double>(c, W));
    TRY(track_finish(c, xf, true));
    TRY(download_rows(c, c->tk_emax, err_max, NS));
    TRY(download_rows(c, c->tk_efin, err_final, NS));
    TRY(download_rows(c, c->tk_nreg, n_reg, 1));
    return 0;
}

// the common part of acoc_track_mc and acoc_lqr_tracking_mc once the nominal is in place: deltas (one copy, as given), the sweeps, the
// outputs
static int track_mc_run(acoc_ctx* c, bool xf, const Weights& W, int m, const double* delta, int delta_shared, const double* tol,
                        acoc_track_mc_out* out)
{
    const size_t per = (size_t)m * NS;
    CK(cudaMemcpyAsync(c->mc_delta, delta, (delta_shared ? 1 : (size_t)c->N) * per * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    const long long dstride = delta_shared ? 0 : (long long)per;
    TRY(xf ? launch_track_mc<float>(c, W, m, dstride, tol) : launch_track_mc<double>(c, W, m, dstride, tol));
    TRY(track_finish(c, xf, false));
    if (!out) return 0;
    const size_t bytes = (size_t)c->N * per * sizeof(double);
    if (out->err_max) CK(cudaMemcpyAsync(out->err_max, c->mc_sum, bytes, cudaMemcpyDeviceToHost, c->stream));
    if (out->err_final) CK(cudaMemcpyAsync(out->err_final, (const char*)c->mc_sum + bytes, bytes, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    TRY(download_rows(c, c->tk_emax, out->worst_max, NS));
    TRY(download_rows(c, c->tk_efin, out->mean_final, NS));
    if (tol) TRY(download_rows(c, c->mc_nw, out->n_within, 1));
    TRY(download_rows(c, c->tk_nreg, out->n_reg, 1));
    return 0;
}

static int track_mc_args(int m, const double* delta, const double* tol, acoc_track_mc_out* out, const char* fn)
{
    REQUIRE(m >= 1, "%s: m = %d, need at least one sample", fn, m);
    REQUIRE(delta, "%s: delta is NULL", fn);
    REQUIRE(!(out && out->n_within && !tol), "%s: n_within needs a tolerance", fn);
    return 0;
}

int acoc_track_mc(acoc_ctx* c, const double* Q, const double* R, const double* QT, int m, const double* delta, int delta_shared,
                  const double* tol, acoc_track_mc_out* out)
{
    TRY(track_ctx_check(c, "acoc_track_mc"));
    TRY(track_mc_args(m, delta, tol, out, "acoc_track_mc"));
    Weights W;
    TRY(track_weights(Q, R, QT, &W));
    TRY(use_device(c->device));
    const size_t per = (size_t)m * NS * sizeof(double);
    TRY(ensure_mc_buffers(c, (size_t)c->N * m, delta_shared ? per : (size_t)c->N * per));
    const bool xf = c->x_float;
    TRY(ensure_track_buffers(c, xf ? sizeof(float) : sizeof(double)));
    c->tk_done = false;  // the nominal and gains buffers are about to change
    TRY(copy_track_nominal(c, xf));
    return track_mc_run(c, xf, W, m, delta, delta_shared, tol, out);
}

int acoc_get_tracked(acoc_ctx* c, double* xx_reg, double* uu_reg)
{
    REQUIRE(c, "ctx is NULL");
    if (!c->tk_done) return fail(ACOC_ERR_STATE, "acoc_get_tracked: call acoc_track first");
    TRY(use_device(c->device));
    return download_tracked(c, xx_reg, uu_reg);
}

int acoc_get_track_gains(acoc_ctx* c, double* K)
{
    REQUIRE(c && K, "NULL argument");
    if (!c->tk_swept) return fail(ACOC_ERR_STATE, "acoc_get_track_gains: call acoc_track or acoc_track_mc first");
    TRY(use_device(c->device));
    // Ktrk as a trajectory with 12 components downloads to (N,12,TT) = (N,2,6,TT)
    return download_soa_t<double>(c, c->tk_K, nullptr, nullptr, nullptr, nullptr, K, c->N, 2 * NS, c->Np, 0);
}

int acoc_get_track_timing(acoc_ctx* c, double* ms)
{
    REQUIRE(c && ms, "NULL argument");
    if (!c->tk_swept) return fail(ACOC_ERR_STATE, "acoc_get_track_timing: call acoc_track or acoc_track_mc first");
    for (int k = 0; k < 4; ++k) ms[k] = c->tk_ms[k];
    return 0;
}

// One context without iterate slots per (device, n, TT, quantisation) for the host-array tracking calls, kept between calls: no
// allocation once it exists.  The caller holds g_host_track_mu while it uses the context.
static std::mutex g_host_track_mu;
static acoc_ctx* g_host_track_ctx = nullptr;

// that context with the nominals xx_opt (n,6,TT) / uu_opt (n,2,TT) in Xnom / Unom: float storage when every state at t >= 1 is a
// float32 value (as acoc_set_init decides), the exact row 0 always
static int host_track_ctx(int device, int n, int TT, const double* params, int state_f64, const double* xx_opt, const double* uu_opt,
                          acoc_ctx** out, bool* xf_out)
{
    const unsigned flags = (state_f64 ? ACOC_STATE_F64 : 0) | ACOC_REFS_SHARED | ACOC_CTX_LITE | ACOC_CTX_NO_SLOTS;
    acoc_ctx*& cached = g_host_track_ctx;
    if (cached && (cached->device != device || cached->N != n || cached->TT != TT || cached->flags != flags)) { acoc_ctx_destroy(cached); cached = nullptr; }
    if (!cached) TRY(acoc_ctx_create(device, n, TT, flags, &cached));
    acoc_ctx* c = cached;
    TRY(use_device(device));
    TRY(acoc_set_model(c, params));
    bool xf = false;
    if (c->P.q32) {
        TRY(ensure_track_buffers(c, sizeof(float)));
        CK(cudaMemsetAsync(c->counters + 3, 0, sizeof(int), c->stream));
        TRY((upload_soa_t<float, double>(c, xx_opt, c->tk_xnom, n, NS, c->Np, (double*)c->tk_xnom0, c->counters + 3)));
        int inexact = 0;
        CK(cudaMemcpyAsync(&inexact, c->counters + 3, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        xf = !inexact;
    }
    if (!xf) {
        TRY(ensure_track_buffers(c, sizeof(double)));
        TRY((upload_soa_t<double, double>(c, xx_opt, c->tk_xnom, n, NS, c->Np, (double*)c->tk_xnom0, (int*)nullptr)));
    }
    TRY((upload_soa_t<double, double>(c, uu_opt, c->tk_unom, n, NI, c->Np, (double*)nullptr, (int*)nullptr)));
    *out = c;
    *xf_out = xf;
    return 0;
}

int acoc_lqr_tracking_many(int device, int n, int TT, const double* params, int state_f64, const double* Q, const double* R, const double* QT,
                           const double* xx_opt, const double* uu_opt, const double* delta, double* xx_reg, double* uu_reg, double* K)
{
    REQUIRE(n > 0 && TT >= 3 && params && xx_opt && uu_opt && delta && xx_reg && uu_reg, "acoc_lqr_tracking_many: bad argument");
    REQUIRE(params[3] != 0.0 && params[7] != 0.0, "acoc_lqr_tracking_many: mass and inertia must be non-zero");
    Weights W;
    TRY(track_weights(Q, R, QT, &W));
    std::lock_guard<std::mutex> lock(g_host_track_mu);
    acoc_ctx* c = nullptr;
    bool xf = false;
    TRY(host_track_ctx(device, n, TT, params, state_f64, xx_opt, uu_opt, &c, &xf));
    TRY(ensure_tracked_buffers(c));
    TRY(upload_delta(c, delta));
    CK(cudaEventRecord(c->tk_ev[0], c->stream));
    TRY(xf ? launch_track_sweeps<float>(c, W) : launch_track_sweeps<double>(c, W));
    TRY(track_finish(c, xf, true));
    TRY(download_tracked(c, xx_reg, uu_reg));
    if (K) TRY(download_soa_t<double>(c, c->tk_K, nullptr, nullptr, nullptr, nullptr, K, n, 2 * NS, c->Np, 0));
    return 0;
}

int acoc_lqr_tracking_mc(int device, int n, int m, int TT, const double* params, int state_f64, const double* Q, const double* R,
                         const double* QT, const double* xx_opt, const double* uu_opt, const double* delta, int delta_shared, const double* tol,
                         acoc_track_mc_out* out)
{
    REQUIRE(n > 0 && TT >= 3 && params && xx_opt && uu_opt, "acoc_lqr_tracking_mc: bad argument");
    REQUIRE(params[3] != 0.0 && params[7] != 0.0, "acoc_lqr_tracking_mc: mass and inertia must be non-zero");
    TRY(track_mc_args(m, delta, tol, out, "acoc_lqr_tracking_mc"));
    Weights W;
    TRY(track_weights(Q, R, QT, &W));
    std::lock_guard<std::mutex> lock(g_host_track_mu);
    acoc_ctx* c = nullptr;
    bool xf = false;
    TRY(host_track_ctx(device, n, TT, params, state_f64, xx_opt, uu_opt, &c, &xf));
    const size_t per = (size_t)m * NS * sizeof(double);
    TRY(ensure_mc_buffers(c, (size_t)n * m, delta_shared ? per : (size_t)n * per));
    CK(cudaEventRecord(c->tk_ev[0], c->stream));
    return track_mc_run(c, xf, W, m, delta, delta_shared, tol, out);
}

// ======================================================================================================
// roofline denominators
// ======================================================================================================
int acoc_measure_fp64_peak(int device, double* tflops)
{
    REQUIRE(tflops, "NULL output");
    TRY(use_device(device));
    cudaDeviceProp p;
    CK(cudaGetDeviceProperties(&p, device));
    const int blocks = p.multiProcessorCount * 8, threads = 256, iters = 1 << 14;
    double* out;
    CK(cudaMalloc(&out, (size_t)blocks * threads * sizeof(double)));
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    double best = 0;
    for (int rep = 0; rep < 6; ++rep) {
        CK(cudaEventRecord(e0));
        k_fp64_peak<<<blocks, threads>>>(out, iters, 1.0 + rep);
        CK(cudaEventRecord(e1));
        CK(cudaEventSynchronize(e1));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        const double tf = 2.0 * 8.0 * iters * (double)blocks * threads / (ms * 1e-3) * 1e-12;
        if (rep > 0) best = std::max(best, tf);
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(out);
    *tflops = best;
    return 0;
}

int acoc_measure_fp64_latency(int device, double* cycles_per_op)
{
    REQUIRE(cycles_per_op, "NULL output");
    TRY(use_device(device));
    const int iters = 1 << 16;
    double* out;
    long long* cyc;
    CK(cudaMalloc(&out, 32 * sizeof(double)));
    CK(cudaMalloc(&cyc, sizeof(long long)));
    long long h = 0, best = 0;
    for (int rep = 0; rep < 3; ++rep) {
        k_fp64_latency<<<1, 32>>>(out, cyc, iters, 1.0 + rep);
        CK(cudaGetLastError());
        CK(cudaMemcpy(&h, cyc, sizeof(h), cudaMemcpyDeviceToHost));
        if (rep == 0 || h < best) best = h;
    }
    cudaFree(out); cudaFree(cyc);
    *cycles_per_op = (double)best / iters;
    return 0;
}

int acoc_measure_copy_bw(int device, double* gbs)
{
    REQUIRE(gbs, "NULL output");
    TRY(use_device(device));
    const size_t n = (size_t)1 << 27;  // 2 GiB per buffer of double2
    double2 *a, *b;
    CK(cudaMalloc(&a, n * sizeof(double2)));
    if (cudaMalloc(&b, n * sizeof(double2)) != cudaSuccess) { cudaFree(a); return fail(ACOC_ERR_NOMEM, "copy benchmark allocation failed"); }
    CK(cudaMemset(a, 1, n * sizeof(double2)));
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    cudaDeviceProp p;
    CK(cudaGetDeviceProperties(&p, device));
    double best = 0;
    for (int rep = 0; rep < 6; ++rep) {
        CK(cudaEventRecord(e0));
        k_copy<<<p.multiProcessorCount * 16, 512>>>(a, b, n);
        CK(cudaEventRecord(e1));
        CK(cudaEventSynchronize(e1));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        if (rep > 0) best = std::max(best, 2.0 * n * sizeof(double2) / (ms * 1e-3) * 1e-9);
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(a); cudaFree(b);
    *gbs = best;
    return 0;
}

