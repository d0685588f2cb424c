/*
 * acoc.h -- C ABI of libacoc.so: batched regularized-Newton trajectory optimisation for the 2-D
 * longitudinal aircraft model on NVIDIA B200 (sm_100a).
 *
 * This is the drop-in boundary for the hot path of MohamedAtwan/AirCraftOptimalControl.  The reference
 * is pure Python with no FFI of its own, so each entry point below cites the Python interface it
 * replaces (file:line into the reference); INTEGRATION.md shows the ctypes stub a maintainer of the
 * reference would add to route those functions here.
 *
 * Conventions
 *   - every function returns 0 on success and a negative acoc_status on failure; nothing throws or
 *     calls exit() across the boundary (the reference print()+exit()s on shape errors, optcon.py:585-596);
 *     acoc_last_error() returns a human-readable message for the calling thread.
 *   - all floating-point buffers are C-contiguous IEEE float64 HOST memory unless the name ends in _dev (CUDA memory of the
 *     context's device, see "device-resident inputs and outputs").
 *   - host trajectory layout is the reference's: one instance is (6,TT) / (2,TT) component-major
 *     (xx[i*TT + t]); a batch adds a leading instance axis (N,6,TT) / (N,2,TT).
 *   - matrices are row-major; "A" means fx.T (A[i][j] = d f_i / d x_j), "B" means fu.T.
 *   - params[9] = {cd0, cda, cla, m, g, S, rho, J, dt}          (aircraft_simplified.py:108-118)
 *   - there is no CPU fallback: every entry point runs CUDA kernels on the selected device and fails with
 *     ACOC_ERR_CUDA when no B200-class device is usable.
 */
#ifndef ACOC_H
#define ACOC_H

#ifdef __cplusplus
extern "C" {
#endif

#define ACOC_VERSION 100 /* 0.1.0 */

typedef enum acoc_status {
    ACOC_OK = 0,
    ACOC_ERR_INVALID = -1, /* bad argument (shape, NULL, option out of range) */
    ACOC_ERR_CUDA = -2,    /* CUDA runtime error, message in acoc_last_error() */
    ACOC_ERR_STATE = -3,   /* call sequence error (e.g. iterate before set_init) */
    ACOC_ERR_NOMEM = -4
} acoc_status;

/* flags for acoc_ctx_create */
#define ACOC_STATE_F32 0u        /* round the next state to float32 like aircraft_simplified.py:300 (default) */
#define ACOC_STATE_F64 1u        /* keep the next state in float64 (the reference with line 300 patched) */
#define ACOC_REFS_SHARED 2u      /* one reference trajectory shared by all instances */
#define ACOC_ARMIJO_SPECULATIVE 0u /* evaluate all armijo_maxiters candidates concurrently (default) */
#define ACOC_ARMIJO_LAZY 4u      /* candidate 0 for everyone, the remaining candidates only for instances that failed it */
#define ACOC_SOLVE_IN_PLACE 8u   /* acoc_newton_solve: never gather the still-iterating instances into a smaller survivor generation */
#define ACOC_FP32 16u            /* optional FP32 mode: float32 arithmetic and trajectory storage (costs/descent still accumulated in
                                    float64); NOT the parity path -- results agree with the float64 path to a tolerance only (DESIGN.md) */
#define ACOC_NO_TMA 64u          /* run the sweeps with plain global loads instead of the warp-private TMA (bulk async copy) rings;
                                    results are bit-identical, this is for A/B measurements */
#define ACOC_NO_SPLIT 128u        /* never sweep a fully active batch as two tile ranges on two streams (A/B measurements; identical results) */
#define ACOC_NO_FUSED 256u       /* never fuse the LQ forward pass with line-search rollouts: neither with candidate 0 of the lazy search
                                    (k_forward_cand0_tma, any batch size) nor with the whole search of small batches (k_search_fused, <= 4096
                                    instances); the separate sweeps run instead (A/B tests; identical results) */
#define ACOC_PRIORITY_SHIFT 16
#define ACOC_PRIORITY(level) (((unsigned)(level) & 15u) << ACOC_PRIORITY_SHIFT)
                                 /* stream priority level of the context, 0 (default) .. 15: the device schedules the thread blocks of a
                                    context with a higher level first (clamped to the device's priority range).  Contexts that solve
                                    concurrently on one GPU (the sub-batches of a pipelined solve) then finish one after the other instead of
                                    all at the end, so that the device->host copy of one overlaps the iterations of the next.  No effect
                                    on results. */
#define ACOC_REFS_EXPANDED 512u  /* acoc_set_refs_generated: write the generated references out as per-instance arrays (64 B per
                                    instance and step, as acoc_set_refs would hold them) instead of keeping them in their parametric
                                    form (8 B or none); bit-identical results, A/B tests */
#define ACOC_X_F64 32u           /* keep the state iterates in float64 device buffers even when every stored state is a float32 value
                                    (ACOC_STATE_F32); results are bit-identical either way, this only costs bandwidth (A/B tests) */

/* per-instance status written by the Newton driver */
#define ACOC_INST_ACTIVE 0
#define ACOC_INST_CONVERGED 1   /* descent >= term_cond (optcon.py:499) */
#define ACOC_INST_MAXITER 2     /* ran max_iters-1 loop bodies (optcon.py:415) */
#define ACOC_INST_NONFINITE 3   /* NaN/Inf cost or descent: frozen */

/* acoc_newton_options.method: which optimize() loop acoc_newton_iterate / acoc_newton_solve run.
 *   ACOC_METHOD_NEWTON    NewtonMethod.optimize (optcon.py:341-529).
 *   ACOC_METHOD_GRADIENT  GradientMethod.optimize (optcon.py:27-174), steepest descent: deltau_t = -B_t' lam_{t+1} - lu_t (:111),
 *       descent = sum_t |deltau_t|^2 (:118), stop when descent <= -term_cond (1e-6 hard-coded at :52).  The reference's call of its own
 *       line search (optcon.py:125) passes 8 of armijo_stepsize's 9 arguments and raises TypeError; the repair used here (and by the
 *       oracle: oracle/pyref.py::run_gradient) supplies the missing JP = JJ[kk] and hands the search the directional derivative
 *       -descent, so that the test of optcon.py:268 is the sufficient-decrease condition.  Histories report the slope -descent. */
#define ACOC_METHOD_NEWTON 0
#define ACOC_METHOD_GRADIENT 1

typedef struct acoc_ctx acoc_ctx;

/* NewtonMethod.__init__ keyword arguments (optcon.py:335-337) */
typedef struct acoc_newton_options {
    int max_iters;        /* 200 in the shipped scripts (main_newton_method.py:32) */
    int armijo_maxiters;  /* 10   (main_newton_method.py:38) */
    int exact_after;      /* exact Hessian iff kk > exact_after; the reference hard-codes 8 (optcon.py:443) */
    int method;           /* ACOC_METHOD_NEWTON (0, default) or ACOC_METHOD_GRADIENT: which optimize() the driver runs (see below) */
    double stepsize_0;    /* 1    (main_newton_method.py:33) */
    double cc;            /* 0.5 */
    double beta;          /* 0.7 */
    double term_cond;     /* the reference hard-codes -1e-6 and ignores the constructor's value (optcon.py:368) */
} acoc_newton_options;

/* ---------------------------------------------------------------- library ---------------------------- */
int acoc_version(void);
const char* acoc_last_error(void);
int acoc_device_count(int* count);
/* name[len], SM count, memory bytes, compute capability major*10+minor of `device` */
int acoc_device_info(int device, char* name, int len, int* sm_count, unsigned long long* mem_bytes, int* cc);

/* ------------------------------------------------- pointwise entry points ---------------------------- */
/* Dynamics.step(xx, uu[, lmbd])  -- aircraft_simplified.py:263-393 (+ tensorCont :397-404)
 * n independent samples: x[n][6], u[n][2], lmbd[n][6] or NULL.
 * Outputs (any may be NULL): xxp[n][6]; A[n][36]; B[n][12] (6x2);
 *   lmbd == NULL: fxx[n][216] ([i][j][k] = d2 f_k/dx_i dx_j), fux[n][72] ([a][j][k]);
 *   lmbd != NULL: fxx[n][36], fux[n][12] contracted with the costate.   fuu is identically zero (:382). */
int acoc_step_batch(int device, int n, const double* params, int state_f64, const double* x, const double* u,
                    const double* lmbd, double* xxp, double* A, double* B, double* fxx, double* fux);

/* Cost.stagecost / Cost.termcost -- aircraft_simplified.py:25-69, :71-97.  n samples x[n][6], u[n][2],
 * xr[n][6], ur[n][2]; dense Q[36], R[4], QT[36].  Outputs (NULL to skip): ll[n], lx[n][6], lu[n][2],
 * llT[n], lTx[n][6].  The constant Hessians lxx=Q, luu=R, lxu=lux=0, lTxx=QT are the caller's inputs. */
int acoc_cost_batch(int device, int n, const double* Q, const double* R, const double* QT, const double* x,
                    const double* u, const double* xr, const double* ur, double* ll, double* lx, double* lu,
                    double* llT, double* lTx);

/* ltv_LQR(AAin,BBin,QQin,RRin,SSin,QQfin,TT,x0,qq,rr,qqf) -- optcon.py:533-771 (= lqr_tracking.py:6-242)
 * nb independent problems, time-major: A[nb][TT][6][6], B[nb][TT][6][2], Q[nb][TT][6][6], R[nb][TT][2][2],
 * S[nb][TT][2][6], Qf[nb][6][6], x0[nb][6]; affine terms q[nb][TT][6], r[nb][TT][2], qf[nb][6] or all three
 * NULL (non-augmented branch).  n = 7 when augmented else 6.
 * Outputs: K[nb][TT][2][n], P[nb][TT][n][n] (may be NULL), xout[nb][TT][6], uout[nb][TT][2],
 * n_reg[nb] (may be NULL) = number of steps that took the +0.5*I branch (optcon.py:745-749). */
int acoc_ltv_lqr(int device, int nb, int TT, const double* A, const double* B, const double* Q, const double* R,
                 const double* S, const double* Qf, const double* x0, const double* q, const double* r,
                 const double* qf, double* K, double* P, double* xout, double* uout, int* n_reg);

/* lqr_tracking(xx_opt, uu_opt, tt) -- lqr_tracking.py:245-283, batched over n perturbations delta[n][6]
 * of the initial state.  xx_opt (6,TT), uu_opt (2,TT).  Outputs xx_reg[n] (6,TT), uu_reg[n] (2,TT) and
 * (optional) the shared gains K[TT][2][6]. */
int acoc_lqr_tracking(int device, int n, int TT, const double* params, int state_f64, const double* Q,
                      const double* R, const double* QT, const double* xx_opt, const double* uu_opt,
                      const double* delta, double* xx_reg, double* uu_reg, double* K);

/* Device time (CUDA events, ms) of the kernels of this thread's last acoc_lqr_tracking call: ms[0] total, ms[1] linearisation along
 * the nominal + the shared LQ solve (k_step_batch + k_lq_dense<6>), ms[2] the closed-loop rollouts (k_track). */
int acoc_last_pointwise_timing(double* ms);

/* ------------------------------------------------- batched Newton context ---------------------------- */
/* One context = one GPU, one CUDA stream, N OCP instances with horizon TT held struct-of-arrays in HBM.
 * A context is not thread-safe; different contexts are independent. */
int acoc_ctx_create(int device, int n_instances, int TT, unsigned flags, acoc_ctx** out);
int acoc_ctx_destroy(acoc_ctx* ctx);
/* bytes of device memory owned by the context */
int acoc_ctx_device_bytes(const acoc_ctx* ctx, unsigned long long* bytes);

int acoc_set_model(acoc_ctx* ctx, const double* params);                                  /* Dynamics() attrs */
/* Cost(QQt,RRt,QQT), aircraft_simplified.py:20-23.  Q, R and QT must be SYMMETRIC here (ACOC_ERR_INVALID otherwise): the fused
 * backward sweep carries the Riccati matrix as its upper triangle.  This is a documented deviation: the reference accepts any matrix
 * (aircraft_simplified.py:61-68) -- a non-symmetric Q there makes the gradient Q dx inconsistent with the cost dx'Q dx, which no
 * shipped configuration does.  The pointwise acoc_cost_batch and the literal acoc_ltv_lqr accept arbitrary matrices like the
 * reference (tests: test_weight_symmetry_contract). */
int acoc_set_weights(acoc_ctx* ctx, const double* Q, const double* R, const double* QT);
int acoc_set_options(acoc_ctx* ctx, const acoc_newton_options* opt);                      /* NewtonMethod(...) */
/* xx_ref (N,6,TT) / uu_ref (N,2,TT), or (6,TT) / (2,TT) when the context was created with ACOC_REFS_SHARED */
int acoc_set_refs(acoc_ctx* ctx, const double* xx_ref, const double* uu_ref);
/* The reference generators of the scripts, on the device (main_newton_method.py:96-142, acrobatic_newton.py:99-154): per-instance
 * xx_ref / uu_ref are built in HBM from per-instance parameters zf[N] (final / bump height), vx[N] (= (xf - x0)/tf) and shared time
 * bases tt[TT], zshape[TT], vshape[TT] (NULL: V_ref = xconst[2]) that the caller computed with the scripts' own numpy code:
 *   X = 0 + vx*tt,  Z = 0 + zshape*(zf - 0),  V = ((vshape*zf)**2 + vx**2)**0.5,  theta, q, gamma = xconst[3..5],  uu_ref = uconst[0..1]
 * in the scripts' operation order, so the references are bit-identical to what the scripts build on the host and acoc_set_refs
 * would upload (16 B per instance cross the bus instead of 64 KB).  The context keeps them in this parametric form -- the sweeps form
 * X and Z from the tables with one multiplication each, only V (step maneuver) is a stored per-instance array -- which removes 56-64 of
 * the ~230-280 bytes a sweep moves per instance and step (ACOC_REFS_EXPANDED keeps per-instance arrays instead; same results up to the
 * sign of a zero reference).  Not for ACOC_REFS_SHARED contexts. */
int acoc_set_refs_generated(acoc_ctx* ctx, const double* tt, const double* zshape, const double* vshape, const double* zf,
                            const double* vx, const double* xconst, const double* uconst);
/* the references held by the context, in acoc_set_refs' layout (either pointer may be NULL) */
int acoc_get_refs(acoc_ctx* ctx, double* xx_ref, double* uu_ref);
/* xx_init (N,6,TT), uu_init (N,2,TT): NewtonMethod.optimize(xx_init, uu_init, tf, dt), optcon.py:341, :395-398.
 * Resets the Newton state (iteration counter, histories). */
int acoc_set_init(acoc_ctx* ctx, const double* xx_init, const double* uu_init);
/* Dynamics.get_initial_trajectory(xx_ref, tt) -- aircraft_simplified.py:126-148 -- computed on the device for
 * every instance from the references already set (float64 arithmetic), then used as the initial guess.
 * dx0 (N,6) or NULL: start instance i from xx_ref[:,0] + dx0[i] (perturbed-initial-state batches). */
int acoc_init_guess(acoc_ctx* ctx, double kp, double kt, const double* dx0);

/* Run up to n_iters more Newton iterations (loop bodies of optcon.py:415-501) on every instance that is
 * still active; returns after the device has finished them (the call is timed with CUDA events, see
 * acoc_get_timing).  *n_active_out (may be NULL) = instances still active afterwards. */
int acoc_newton_iterate(acoc_ctx* ctx, int n_iters, int* n_active_out);
/* Iterate until no instance is active.  *total_iters = sum over instances of loop bodies executed.
 * Whenever at most half of a batch (of >= 4096 instances) is still iterating, the survivors are gathered into a smaller
 * internal context so that every warp lane does useful work again; they are folded back before the call returns, so
 * results, histories and statistics are exactly those of iterating in place (ACOC_SOLVE_IN_PLACE disables this). */
int acoc_newton_solve(acoc_ctx* ctx, long long* total_iters);
/* Block until all work queued on the context's stream has finished. */
/* acoc_newton_solve and the read-back of what optimize() returns in ONE call.  xx_star: (N,6,TT) float32 if x_is_f32 (lossless under the
 * float32 state quantisation, see acoc_get_result_f32; column 0 then holds float32(x0)) else float64; uu_star (N,2,TT) float64; x0 (N,6)
 * or NULL receives the exact initial states.  When xx_star and uu_star are PAGE-LOCKED host memory (cudaHostAlloc / cudaHostRegister,
 * e.g. torch pin_memory) the layout-conversion kernels write straight into them, and the instances that have finished are delivered at
 * the moment the still-iterating ones move on to a survivor generation, so the transfer overlaps the latency-bound tail of the solve.
 * Pageable buffers: same results through acoc_newton_solve + acoc_get_result[_f32]. */
int acoc_newton_solve_deliver(acoc_ctx* ctx, void* xx_star, int x_is_f32, double* uu_star, double* x0, long long* total_iters);
int acoc_sync(acoc_ctx* ctx);

/* What NewtonMethod.optimize returns (optcon.py:503-505): iterate kk-1 with uu[:, -1] = uu[:, -2]. */
int acoc_get_result(acoc_ctx* ctx, double* xx_star, double* uu_star);
/* The same result with the states as float32 (N,6,TT): LOSSLESS whenever the context keeps its state iterates as float (float32
 * state quantisation of aircraft_simplified.py:300, the default): every x_t, t >= 1, is a float32 value.  Column t = 0 holds
 * float32(x0); the exact float64 x0 = xx_init[:,0] (optcon.py:398) is returned in x0 (N,6) when non-NULL.  uu_star stays float64.
 * ACOC_ERR_STATE if the context holds float64 states (ACOC_STATE_F64, ACOC_X_F64, or acoc_set_init with non-float32 states). */
int acoc_get_result_f32(acoc_ctx* ctx, float* xx_star, double* uu_star, double* x0);
/* which: 0 = the newest iterate (last get_update), 1 = the one before it. */
int acoc_get_iterate(acoc_ctx* ctx, int which, double* xx, double* uu);
/* Descent direction of the last iteration: deltau (N,2,TT) (optcon.py:468).  deltau and the gains are per-iteration
 * scratch: they are meaningful for instances that were still active in that iteration. */
int acoc_get_deltau(acoc_ctx* ctx, double* deltau);
/* Gains of the last backward sweep: K (N,2,6,TT), sigma (N,2,TT) -- KK[:,1:,:] and KK[:,0,:] of optcon.py:468.
 * Stages N*16*TT doubles on the host: meant for inspection / parity tests on small batches. */
int acoc_get_gains(acoc_ctx* ctx, double* K, double* sigma);
/* Per-instance, per-iteration history, each (N, max_iters): JJ[k], descent[k] (optcon.py:497), the Armijo step
 * (optcon.py:327) and the number of candidates the sequential search rolls out.  Any pointer may be NULL. */
int acoc_get_history(acoc_ctx* ctx, double* JJ, double* descent, double* stepsize, int* n_cand);
/* Per-instance summary (length N each, any may be NULL): loop bodies executed, ACOC_INST_* status, cost of
 * the newest iterate, last descent, number of +0.5*I regularisations. */
int acoc_get_stats(acoc_ctx* ctx, int* iters, int* status, double* J, double* descent, int* n_reg);

/* ------------------------------------------ closed-loop tracking of every instance ----------------------- */
/* lqr_tracking(xx_opt, uu_opt, tt) -- lqr_tracking.py:245-283 -- for EVERY instance of the context along its own result: the nominal of
 * instance i is what acoc_get_result returns now (iterate kk-1 with uu[:,-1] = uu[:,-2]; all zeros for an instance stopped at kk = 0;
 * the newest iterate while still active; column 0 the exact x0).  Gains of the non-augmented ltv_LQR (:276) linearised along the nominal
 * (:268-273) with the tracking weights Q, R, QT (P_{TT-1} = QT); closed loop (:279-281) from x*_0 + delta[i] under the context's model and
 * state quantisation: u_t = u*_t + K_t (x_t - x*_t), u_{TT-1} = 0.
 * Q, R, QT symmetric (ACOC_ERR_INVALID otherwise, same contract as acoc_set_weights; the pointwise acoc_lqr_tracking accepts any); they
 * are independent of the context's Newton weights.  delta (N,6) or NULL (= 0).  Per-instance summaries computed on the device (any may
 * be NULL): err_max (N,6) = max_t |x_t - x*_t|, err_final (N,6) = |x_{TT-1} - x*_{TT-1}| (a NaN anywhere gives NaN), n_reg (N) = steps
 * whose gain took the +0.5*I branch (optcon.py:745-749).  An instance whose nominal is the zero slot or not finite is computed as the
 * reference would (its outputs are NaN) and disturbs no other.
 * The tracking buffers (~176 B per instance and time step with float32-valued states) are allocated on the first call and freed with
 * the context (ACOC_ERR_NOMEM if they do not fit; the Newton state is untouched).  Tracking writes no iterate, gain, deltau, history or
 * statistic of the Newton solve: solving or reading back afterwards behaves as if it had not been called.
 * ACOC_ERR_STATE for ACOC_FP32 contexts and before acoc_set_init / acoc_init_guess. */
int acoc_track(acoc_ctx* ctx, const double* Q, const double* R, const double* QT, const double* delta, double* err_max, double* err_final,
               int* n_reg);
/* trajectories of the last acoc_track: xx_reg (N,6,TT), uu_reg (N,2,TT); either may be NULL */
int acoc_get_tracked(acoc_ctx* ctx, double* xx_reg, double* uu_reg);
/* gains of the last acoc_track or acoc_track_mc: K (N,2,6,TT), lqr_tracking's KK per instance (K[:,:,:,TT-1] = 0) */
int acoc_get_track_gains(acoc_ctx* ctx, double* K);
/* device time (CUDA events, ms) of the last acoc_track (or acoc_track_mc): ms[0] total, ms[1] nominal (k_track_nominal), ms[2] gains
 * sweep, ms[3] rollout (acoc_track_mc: dispersion rollout + reduction) */
int acoc_get_track_timing(acoc_ctx* ctx, double* ms);
/* lqr_tracking (lqr_tracking.py:245-283) for n independent nominals from host arrays: xx_opt (n,6,TT), uu_opt (n,2,TT), delta (n,6);
 * outputs xx_reg (n,6,TT), uu_reg (n,2,TT), K (n,2,6,TT) or NULL.  The same kernels as acoc_track (bit-identical results for the same
 * nominals); states are stored as float32 only when that is lossless.  Q, R, QT symmetric as above. */
int acoc_lqr_tracking_many(int device, int n, int TT, const double* params, int state_f64, const double* Q, const double* R,
                           const double* QT, const double* xx_opt, const double* uu_opt, const double* delta, double* xx_reg,
                           double* uu_reg, double* K);

/* ------------------------------------------ Monte Carlo dispersion of the closed loop -------------------- */
/* Outputs of acoc_track_mc / acoc_lqr_tracking_mc; any pointer may be NULL.  M = samples per instance. */
typedef struct acoc_track_mc_out {
    double* err_max;    /* (N,M,6) per sample: max_t |x_t - x*_t| */
    double* err_final;  /* (N,M,6) per sample: |x_{TT-1} - x*_{TT-1}| */
    double* worst_max;  /* (N,6)  max over m of err_max[i,m,c], folded in sample order; one NaN sample gives NaN */
    double* mean_final; /* (N,6)  (((e_0 + e_1) + e_2) + ...) / M of e_m = err_final[i,m,c] */
    int* n_within;      /* (N)    samples with err_max[i,m,c] <= tol[c] for all six c (a NaN is never within); needs tol */
    int* n_reg;         /* (N)    as acoc_track */
} acoc_track_mc_out;
/* acoc_track's closed loop from M perturbed starts per instance: nominal and gains exactly those of acoc_track (the instance's current
 * result, tracking weights Q, R, QT symmetric), sample (i, m) flown from x*_0 + delta[i, m].  The per-sample summaries are bit-identical
 * to acoc_track(delta = delta[:, m]) for instance i; the aggregates are computed on the device in a fixed order (no atomics).
 * delta (M,6) when delta_shared (the same perturbations for every instance: common random numbers), else (N,M,6); copied as given.
 * tol (6) or NULL: the tolerance of n_within.  No trajectory is kept: the trajectory of sample m is what acoc_track(delta[:, m]) returns.
 * Reuses acoc_track's nominal and gains buffers: acoc_get_track_gains returns the gains it used, acoc_get_track_timing reports its
 * kernels (ms[3] = dispersion rollout + reduction), and acoc_get_tracked returns ACOC_ERR_STATE until the next acoc_track.  It does
 * not allocate the tracked-trajectory buffers; the per-sample buffers (96 B per sample, plus the deltas) are allocated on the first
 * call, grow with N*M and are freed with the context (ACOC_ERR_NOMEM if they do not fit; the context is left as it was).  Writes
 * nothing of the Newton solve.  ACOC_ERR_STATE for ACOC_FP32 contexts and before acoc_set_init / acoc_init_guess; ACOC_ERR_INVALID
 * for m < 1, a NULL delta, non-symmetric weights, or n_within without tol. */
int acoc_track_mc(acoc_ctx* ctx, const double* Q, const double* R, const double* QT, int m, const double* delta, int delta_shared,
                  const double* tol, acoc_track_mc_out* out);
/* acoc_track_mc for n nominals from host arrays xx_opt (n,6,TT), uu_opt (n,2,TT) (the twin of acoc_lqr_tracking_many, same cached
 * context and float-storage decision; n = 1 with many deltas is the reference's single-optimum study, as summaries). */
int acoc_lqr_tracking_mc(int device, int n, int m, int TT, const double* params, int state_f64, const double* Q, const double* R,
                         const double* QT, const double* xx_opt, const double* uu_opt, const double* delta, int delta_shared,
                         const double* tol, acoc_track_mc_out* out);

/* ------------------------------------------ device-resident inputs and outputs --------------------------- */
/* Twins of the calls of the same name without _dev for arrays that live in CUDA memory of the context's device (e.g. torch tensors):
 * same shapes and layouts (float64 unless stated, C-contiguous), same state rules, same refusals, same effect on the context and
 * bit-identical results.  Only the arrays whose size grows with TT or with the number of samples have such a twin; small inputs
 * (weights, tol, dx0, acoc_track's delta) stay in host memory.  The context's sm_100a layout-conversion kernels read and write the
 * caller's arrays directly: no staging buffer, no host copy.
 *   - Every _dev pointer must be device (or managed) memory of the context's device; anything else (pageable or page-locked host
 *     memory, another GPU) is refused with ACOC_ERR_INVALID before any work is queued, naming the argument.
 *   - stream: the caller's CUDA stream (cudaStream_t; NULL = the legacy default stream).  The context's streams are non-blocking, so
 *     a call first makes its stream wait for the work queued on `stream` so far (the writes of the inputs, earlier reads of the
 *     outputs).  It returns once its outputs are written and its inputs read, like the host-array calls: the arrays may then be used
 *     on any stream. */
int acoc_set_refs_dev(acoc_ctx* ctx, const double* xx_ref_dev, const double* uu_ref_dev, void* stream);
int acoc_set_init_dev(acoc_ctx* ctx, const double* xx_init_dev, const double* uu_init_dev, void* stream);
/* x_is_f32 = 0: what acoc_get_result writes; x_is_f32 = 1: xx_star_dev is float32 and receives what acoc_get_result_f32 writes
 * (refused in the same cases).  x0_dev (N,6) float64 or NULL: the exact x0, as acoc_get_result_f32 returns it. */
int acoc_get_result_dev(acoc_ctx* ctx, void* xx_star_dev, int x_is_f32, double* uu_star_dev, double* x0_dev, void* stream);
int acoc_get_tracked_dev(acoc_ctx* ctx, double* xx_reg_dev, double* uu_reg_dev, void* stream);
int acoc_get_track_gains_dev(acoc_ctx* ctx, double* K_dev, void* stream);
/* delta_dev (M,6) or (N,M,6) and every pointer of *out_dev in device memory: per-sample values (N,M,6), aggregates (N,6), counts (N)
 * int32.  Q, R, QT and tol stay host arrays. */
int acoc_track_mc_dev(acoc_ctx* ctx, const double* Q, const double* R, const double* QT, int m, const double* delta_dev, int delta_shared,
                      const double* tol, acoc_track_mc_out* out_dev, void* stream);

/* ------------------------------------------ derivative of the optimum (vector-Jacobian product) ------------ */
/* The derivative of what acoc_get_result returns with respect to the references and the initial state, applied to upstream gradients
 * (reverse mode): the backward pass of a differentiable solve (aircraftoptimalcontrol_b200/autograd.py).
 * Definition.  For instance i, the optimum is that of the problem the Newton driver solves, with the smooth float64 model (the next
 * state is NOT rounded to float32: the derivative of a float32-rounded map is zero almost everywhere):
 *     J = sum_{t=0}^{TT-2} 1/2 (x_t - xref_t)'Q(x_t - xref_t) + 1/2 (u_t - uref_t)'R(u_t - uref_t) + 1/2 (x_{TT-1} - xref_{TT-1})'QT(...)
 *     s.t. x_{t+1} = f(x_t, u_t),  x_0 = xi.
 * It is linearised at the returned point (x*, u*) (what acoc_get_result returns now) with the costates lam_{TT-1} = QT (x*_{TT-1} -
 * xref_{TT-1}), lam_t = A_t' lam_{t+1} + Q (x*_t - xref_t) and H = the Hessian of the Lagrangian there (Q + sum_k lam_{t+1,k} d2f_k,
 * S_t = the lam-contracted d2f/dudx, R; QT at TT-1) -- the Newton sweep's exact-Hessian terms.  Given gx (N,6,TT) and gu (N,2,TT), the
 * upstream gradients with respect to the arrays acoc_get_result writes:
 *   1. gu[:,:,TT-1] is added to gu[:,:,TT-2] (the result repeats u_{TT-2} there); gx[:,:,0] is a gradient of xi itself.
 *   2. w = argmin 1/2 w'Hw - g'w  s.t.  w_{x,t+1} = A_t w_{x,t} + B_t w_{u,t},  w_{x,0} = 0  (a Riccati sweep with the plain G^-1 in
 *      the recursion and the gains -- never G + 0.5 I -- and a forward pass): the exact solution of the KKT system wherever that
 *      system is nonsingular.
 *   3. xref_bar_t = Q w_{x,t} (1 <= t <= TT-2), QT w_{x,TT-1} at TT-1, 0 at t = 0;  uref_bar_t = R w_{u,t} (t <= TT-2), 0 at TT-1;
 *      x0_bar = gx_0 - A_0' eta_1 - S_0' w_{u,0} (eta_1: multiplier of the first dynamics constraint of the adjoint problem) = -p_0 of
 *      the adjoint's Riccati sweep;  n_indef = steps whose G = R + B'PB is not positive definite (there the second-order sufficient
 *      condition fails: the point is not a strict local optimum and the derivative is that of a KKT point).
 *   With parametric references (acoc_set_refs_generated) the per-instance chain rule, summed on the device in ascending t:
 *      zf_bar = sum_t zs_t Xbar_{t,Z} + sum_t (vs_t^2 zf / V_t) Xbar_{t,V},   vx_bar = sum_t tt_t Xbar_{t,X} + sum_t (vx / V_t) Xbar_{t,V}
 *   (Xbar = xref_bar; the V terms for a stored speed reference only, the step maneuver; V_t the stored table).  They do not include
 *   the dependence of xi on the references: a caller whose x0 is xref_0 + dx0 (acoc_init_guess) adds x0_bar to that chain itself.
 * Not built: gradients with respect to the weights or the model parameters, forward mode, the FP32 mode, the tracking calls.
 * Outputs (any pointer may be NULL): */
typedef struct acoc_vjp_out {
    double* xref_bar; /* (N,6,TT); per instance also for ACOC_REFS_SHARED contexts (the caller sums them) */
    double* uref_bar; /* (N,2,TT) */
    double* x0_bar;   /* (N,6) */
    double* zf_bar;   /* (N)  parametric references only (ACOC_ERR_INVALID otherwise) */
    double* vx_bar;   /* (N)  parametric references only */
    int* n_indef;     /* (N) */
} acoc_vjp_out;
/* Writes nothing of the Newton state (iterates, gains, deltau, histories, statistics) and changes no answer of the tracking getters.  Its
 * buffers (~(72 + 6 s) * TT + 100 bytes per instance, s = 4 or 8 bytes per stored state) are allocated on the first call and freed with
 * the context (ACOC_ERR_NOMEM leaves the context unchanged).  An instance whose result is the zero slot or not finite gets NaN and disturbs
 * no other.  ACOC_ERR_STATE for ACOC_FP32 contexts and before the weights, the references and acoc_set_init / acoc_init_guess;
 * ACOC_ERR_INVALID for a NULL gx or gu. */
int acoc_result_vjp(acoc_ctx* ctx, const double* gx, const double* gu, acoc_vjp_out* out);
/* the twin for device memory (see "device-resident inputs and outputs"): gx_dev, gu_dev and every pointer of *out_dev (n_indef int32) */
int acoc_result_vjp_dev(acoc_ctx* ctx, const double* gx_dev, const double* gu_dev, acoc_vjp_out* out_dev, void* stream);

/* Single pieces of the loop on the context's current iterate, exposed for parity tests and for the
 * reference's own method names:
 *   acoc_eval_cost        optcon.py:417-424   -> J[N]
 *   acoc_backward         optcon.py:429-464 + Riccati/gains of ltv_LQR; exact != 0 uses the exact Hessian (:443)
 *   acoc_forward          optcon.py:756-762 + :474-477 -> descent[N]
 *   acoc_armijo           GradientMethod.armijo_stepsize (optcon.py:204-327) -> stepsize[N], costs[N][armijo_maxiters]
 *   acoc_update           GradientMethod.get_update (optcon.py:176-200) with per-instance steps -> becomes the newest iterate */
int acoc_eval_cost(acoc_ctx* ctx, double* J);
/* Overwrite the descent direction deltau (N,2,TT) and/or the scalars the Armijo test uses (JP = J[N],
 * descent[N]); lets GradientMethod.armijo_stepsize / get_update be called with caller-supplied arguments. */
int acoc_set_deltau(acoc_ctx* ctx, const double* deltau);
int acoc_set_scalars(acoc_ctx* ctx, const double* J, const double* descent);
int acoc_backward(acoc_ctx* ctx, int exact);
int acoc_forward(acoc_ctx* ctx, double* descent);
int acoc_armijo(acoc_ctx* ctx, double* stepsize, double* costs);
/* One costate sweep of GradientMethod.optimize (optcon.py:95-118) on the current iterate: deltau (readable with acoc_get_deltau)
 * and descent[N] = sum_t |deltau_t|^2 (may be NULL).  The context keeps -descent as the slope of the following acoc_armijo. */
int acoc_gradient(acoc_ctx* ctx, double* descent);
/* The visu_armijo sweep (optcon.py:280-296): costs[N][n_steps] of the rollouts u + steps[k]*deltau for caller-chosen step sizes
 * (the reference plots np.linspace(0, stepsize_0, 10)) along the current deltau. */
int acoc_armijo_sweep(acoc_ctx* ctx, int n_steps, const double* steps, double* costs);
int acoc_update(acoc_ctx* ctx, const double* stepsize);

/* Device-side timing of the last acoc_newton_iterate call, in milliseconds (CUDA events on the context's
 * stream): total and per phase {cost, backward, forward, candidates, select, update}; plus launch count. */
int acoc_get_timing(acoc_ctx* ctx, double* total_ms, double phase_ms[6], long long* kernel_launches);
/* Enable (1) / disable (0) per-phase event timing; off by default because it adds events to the stream. */
int acoc_set_profiling(acoc_ctx* ctx, int on);

/* FP64 FMA throughput microbenchmark (register-resident DFMA chains on every SM): the measured denominator
 * for the FP64 side of the roofline.  Returns TFLOP/s (2 flops per DFMA). */
int acoc_measure_fp64_peak(int device, double* tflops);
/* Cycles per operation of one warp's chain of dependent DFMAs (8.7 on B200): the in-order latency a lone warp of the
 * sequential sweeps pays per dependent instruction. */
int acoc_measure_fp64_latency(int device, double* cycles_per_op);
/* Device copy bandwidth microbenchmark (read + write bytes / time), GB/s. */
int acoc_measure_copy_bw(int device, double* gbs);

#ifdef __cplusplus
}
#endif
#endif /* ACOC_H */
