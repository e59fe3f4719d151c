/*
 * pnode_b200 -- C ABI of the B200-native neural-ODE integrator / discrete-adjoint engine.
 *
 * This is the drop-in boundary: the host side (pnode_b200/petsc_adjoint.py, a mirror of the reference's
 * pnode/petsc_adjoint.py) binds exactly these entry points through ctypes.  Plain pointers and sizes only; every
 * pointer named `d_*` is a DEVICE pointer owned by the caller (torch allocations), `stream` is a cudaStream_t passed as
 * void* (torch.cuda.current_stream().cuda_stream).  No entry point synchronises the stream or allocates memory unless
 * stated.  Every function returns 0 on success; on failure it returns a non-zero code and pnode_last_error() describes
 * it (the reference surfaces PETSc error codes as petsc4py.PETSc.Error -- SURVEY.md section 8b "Errors").
 *
 * Each entry point cites the reference interface it replaces.  "[PETSc]" marks arithmetic that lives inside the PETSc
 * library the reference calls (not vendored under the reference tree; see DESIGN.md "Oracle").
 */
#ifndef PNODE_B200_H
#define PNODE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PNODE_ABI_VERSION 1

/* scalar type of state vectors: the reference requires tensor dtype == PETSc's compiled scalar type
 * (tests/test_pnode.py:127-130, README.md:27) */
#define PNODE_F32 0
#define PNODE_F64 1

#define PNODE_MAX_TERMS 16  /* terms of one stage combination (ARK5: 7 implicit + 7 explicit slopes) */
#define PNODE_MAX_STAGES 7  /* dopri5 */
#define PNODE_MAX_SRCS 32   /* parameter tensors per multi-axpy launch */

int pnode_abi_version(void);
const char *pnode_last_error(void);

/* Number of SMs / device name of the current device (used to size persistent grids; 148 on B200). */
int pnode_device_sm_count(int *sm_count);

/* ----------------------------------------------------------------------------------------------------------------
 * Generic path: the vector arithmetic PETSc performs between callbacks, one launch per stage instead of one per
 * AXPY term.
 * -------------------------------------------------------------------------------------------------------------- */

/* out[i] = base_coef * base[i] + sum_j coefs[j] * vecs[j][i],  i < n.   (base may be NULL; out may alias base.)
 * Replaces [PETSc] VecCopy + VecMAXPY in TSStep_RK / TSStep_ARKIMEX (stage value Y_i = u + h sum a_ij k_j, called
 * between the reference's evalRHSFunction callbacks, pnode/petsc_adjoint.py:393-412) and VecMAXPY / VecAXPY in
 * TSAdjointStep_RK (w = lambda + sum_j (a_ji/b_i) lambda_s,j, called before RHSJacShell.multTranspose,
 * petsc_adjoint.py:52-82).  `vecs` and `coefs` are HOST arrays of nterms device pointers / doubles. */
int pnode_lincomb(void *d_out, const void *d_base, double base_coef, const void *const *vecs, const double *coefs,
                  int nterms, int64_t n, int dtype, void *stream);

/* Step completion fused with the embedded error estimate and the weighted RMS norm:
 *   u_new[i] = u[i] + sum_j bw[j] * k[j][i]                 ([PETSc] TSEvaluateStep_RK, order p)
 *   x[i]     = u_new[i] + sum_j ew[j] * k[j][i]             ([PETSc] TSEvaluateStep_RK, order p-1; ew = h (bhat - b))
 *   *d_sumsq = sum_i ((u_new[i]-x[i]) / (atol + rtol*max(|u_new[i]|,|x[i]|)))^2      ([PETSc] TSErrorWeightedNorm2)
 * d_sumsq is ONE double on the device; the sum is formed in a fixed order (per-block partials in d_work, combined by the
 * last block) so accept/reject decisions are reproducible.  d_work must hold pnode_wrms_work_bytes() bytes and be
 * zero-initialised once by the caller (the kernel restores it).  ew == NULL skips the error part (plain completion).
 * Replaces the launches between the last evalRHSFunction of a step and TSAdaptChoose. */
int64_t pnode_wrms_work_bytes(void);
int pnode_rk_complete_wrms(void *d_unew, const void *d_u, const void *const *k, const double *bw, const double *ew,
                           int nterms, int64_t n, double atol, double rtol, double *d_sumsq, void *d_work, int dtype,
                           void *stream);

/* mu[off_k + i] += coef * src_k[i] for each of nsrc parameter-gradient tensors laid end to end (off_k = sum of sizes
 * before k).  Replaces RHSJacPShell.multTranspose / IJacPShell.multTranspose (petsc_adjoint.py:303-363: flatten the cached
 * per-parameter VJPs) + [PETSc] VecAXPY on mu in TSAdjointStep_*.  srcs may contain NULL (parameter unused => zeros,
 * pnode/misc.py:9-14).  `srcs`/`sizes` are HOST arrays. */
int pnode_multi_axpy(void *d_mu, const void *const *srcs, const int64_t *sizes, int nsrc, double coef, int dtype,
                     void *stream);

/* d_out[j] = <vecs[j], w> for j < nvec (<= 16 per call) and d_out[nvec] = <w, w>, accumulated in double, fixed
 * reduction order.  Replaces [PETSc] VecMDot + VecNorm inside KSPGMRES's classical Gram-Schmidt, which the reference
 * reaches through SNES/KSP on IJacShell.mult / multTranspose (petsc_adjoint.py:98-177) when linear_solver="petsc".
 * d_work: pnode_mdot_work_bytes() bytes, zero-initialised once.  `vecs` is a HOST array of device pointers. */
int64_t pnode_mdot_work_bytes(void);
int pnode_mdot(double *d_out, const void *const *vecs, int nvec, const void *d_w, int64_t n, void *d_work, int dtype,
               void *stream);

/* Column-wise variants for the block Krylov solver behind linear_solver="hpddm" (pnode/hpddm_linearsolve.py:13-49: KSPHPDDM
 * BGMRES on the state seen as a dense [n/batch x batch] matrix, one right-hand side per sample).  Vectors are
 * [nseg][seglen], sample-major like the flattened batch.
 *   pnode_mdot_seg:    d_out[j*nseg + s] = <vecs[j][s,:], w[s,:]> for j < nvec (<= 16), d_out[nvec*nseg + s] = <w[s,:], w[s,:]>
 *                      (double accumulation, fixed order; the coefficients stay on the device)
 *   pnode_lincomb_seg: out[s,:] = base_coef * base[s,:] + sum_j c_j[s] * vecs[j][s,:] with c_j[s] derived from the DEVICE array
 *                      d_coef[j*nseg + s]: as is (COEF), negated (NEG: Gram-Schmidt with the dots just computed), or
 *                      1/sqrt (RSQRT, 0 where the entry is 0: normalisation by a squared norm; a segment that broke down
 *                      gets a zero basis vector and drops out).  base may be NULL; out may alias base. */
#define PNODE_SEG_COEF 0
#define PNODE_SEG_NEG 1
#define PNODE_SEG_RSQRT 2
int pnode_mdot_seg(double *d_out, const void *const *vecs, int nvec, const void *d_w, int64_t nseg, int64_t seglen, int dtype,
                   void *stream);
int pnode_lincomb_seg(void *d_out, const void *d_base, double base_coef, const void *const *vecs, const double *d_coef,
                      int nvec, int mode, int64_t nseg, int64_t seglen, int dtype, void *stream);

/* ----------------------------------------------------------------------------------------------------------------
 * Fused path for tiny-state MLP right-hand sides  f(t,y) = W2 * tanh(W1 * phi(y) + b1) + b2,  phi = cube | identity
 * (the spiral model of examples-pnode/ode_demo_petsc.py:207-230: Linear(2,50)-Tanh-Linear(50,2) applied to y**3).
 * One launch advances every trajectory through ALL steps and stages of a fixed-step explicit RK scheme; weights stay
 * in shared memory; stage values are checkpointed in HBM for the adjoint (replaces -ts_trajectory_type memory).
 * -------------------------------------------------------------------------------------------------------------- */

typedef struct pnode_rk_tableau {
    int32_t s;                                        /* stages */
    int32_t fsal;                                     /* 1: last stage has b = 0 and nothing depends on it */
    double a[PNODE_MAX_STAGES][PNODE_MAX_STAGES];     /* strictly lower triangular */
    double b[PNODE_MAX_STAGES];
    double c[PNODE_MAX_STAGES];
    double be[PNODE_MAX_STAGES];                      /* embedded (order p-1) weights, used when has_be != 0 */
    int32_t has_be;
    int32_t order;                                    /* order p of the scheme ([PETSc] TSAdapt candidate order) */
} pnode_rk_tableau;

typedef struct pnode_mlp_desc {
    int32_t dim;        /* state dimension per trajectory (2) */
    int32_t hidden;     /* hidden width (50) */
    int32_t phi;        /* 0 identity, 1 cube (y**3) */
    int32_t dtype;      /* PNODE_F32 | PNODE_F64 */
    const void *d_w1;   /* [hidden, dim]  row-major (torch nn.Linear.weight) */
    const void *d_b1;   /* [hidden] */
    const void *d_w2;   /* [dim, hidden] */
    const void *d_b2;   /* [dim] */
} pnode_mlp_desc;

/* 1 if a fused kernel is compiled for (dim, hidden, phi, dtype, stages), else 0 (caller uses the generic path).
 * Compiled (dim, hidden): (2,50) -- the spiral model, with tuned occupancy and small-batch kernels -- and (2,100), (3,50),
 * (4,50), (1,50); stages 1, 2, 3, 4, 7 (PETSc TSRK 1fe, 2a/2b, 3, 3bs/4, 5dp).  A layer with fewer hidden units than a
 * compiled width runs on that width with zero weights for the missing units (the caller pads W1 / b1 / W2 and cuts the
 * padded entries out of mu; pnode_b200/fused.py does): a padded unit changes no result bit. */
int pnode_mlp_rk_supported(int dim, int hidden, int phi, int dtype, int stages);

/* One entry of the step schedule the host controller hands to a fused sweep.  In fixed-step runs (-ts_adapt_type none,
 * or a tableau without an embedded method) every step size is known before the launch: the host applies the reference's
 * step_size / per-step list semantics (petsc_adjoint.py:518-532, 812-817) and [PETSc] MATCHSTEP clamping. */
typedef struct pnode_step {
    double t;          /* step start time t_n */
    double h;          /* step size */
    int32_t out_slot;  /* forward: slot of d_sol that receives u_{n+1}, or -1 ([PETSc] TSSetTimeSpan slots) */
    int32_t in_slot;   /* adjoint: slot of d_gout added to lambda AFTER this step's adjoint (forcing), or -1 */
} pnode_step;

/* Forward sweep.  Replaces ODEPetsc.odeint's ts.solve(U) (petsc_adjoint.py:777-869) with all of [PETSc] TSStep_RK /
 * TSEvaluateStep_RK / TSTrajectorySet and the reference's evalRHSFunction callbacks inside one kernel.
 *   d_u0     [ntraj, dim]                 initial states (C-order flatten of the caller's tensor, petsc_adjoint.py:596)
 *   d_sched  DEVICE [nsteps] pnode_step   schedule
 *   d_sol    [nout, ntraj, dim]           span solutions (slots named by out_slot; others untouched)
 *   d_ckpt   [nsteps, s, rows, ntraj]     stage checkpoints, rows = pnode_mlp_rk_ckpt_rows(): the stage value Y_i in rows
 *                                         0..dim-1, for some shapes followed by the stage Jacobian df/dy(Y_i) (dim x dim,
 *                                         row-major) that the adjoint sweep uses; NULL when no adjoint will follow
 */
int pnode_mlp_rk_ckpt_rows(const pnode_mlp_desc *mlp, const pnode_rk_tableau *tab);
int pnode_mlp_rk_forward(const pnode_mlp_desc *mlp, const pnode_rk_tableau *tab, const void *d_u0, int64_t ntraj,
                         const pnode_step *d_sched, int nsteps, void *d_sol, void *d_ckpt, void *stream);

/* Discrete-adjoint sweep over the same schedule, last step first.  Replaces OdeintAdjointMethod.backward
 * (petsc_adjoint.py:916-947): lambda <- grad_out[last_slot]; per step [PETSc] TSAdjointStep_RK with the reference's
 * RHSJacShell.multTranspose / RHSJacPShell.multTranspose callbacks fused in; lambda += grad_out[in_slot] after the
 * adjoint of a step that starts at an output point (the reference's forcing, petsc_adjoint.py:938).
 *   d_gout   [nout, ntraj, dim]   dL/d(solution slots)
 *   d_ckpt   the stage checkpoints pnode_mlp_rk_forward wrote ([nsteps, s, pnode_mlp_rk_ckpt_rows(), ntraj])
 *   d_lambda [ntraj, dim]         out: dL/du0
 *   d_mu     [np]                 out: dL/dparams, order W1,b1,W2,b2 (func.parameters() order, petsc_adjoint.py:618-620)
 *   d_work   scratch of pnode_mlp_rk_adjoint_work_bytes() bytes, zero-initialised once by the caller (per-block partial
 *            mu, combined in a fixed order by the last block so that mu is bit-reproducible)
 */
int64_t pnode_mlp_rk_adjoint_work_bytes(const pnode_mlp_desc *mlp);
int pnode_mlp_rk_adjoint(const pnode_mlp_desc *mlp, const pnode_rk_tableau *tab, int64_t ntraj,
                         const pnode_step *d_sched, int nsteps, int last_slot, const void *d_gout, const void *d_ckpt,
                         void *d_lambda, void *d_mu, void *d_work, void *stream);

/* Bounded checkpoint storage for the fused sweeps: [PETSc] -ts_trajectory_solution_only 1 (TSTrajectory "memory" keeping
 * the step solutions only, SURVEY.md A.7; the reference reaches it through ts.setFromOptions(), petsc_adjoint.py:775).
 * The forward sweep keeps u_n per step -- d_usteps [nsteps, dim, ntraj], at most 1/s of the stage checkpoints -- and the adjoint
 * sweep recomputes the s stage values (and stage Jacobians) of a step from u_n with the forward sweep's own arithmetic before it runs the
 * step's adjoint stages (same results as the stage-checkpoint sweeps, bit for bit).  d_peer_bufs NULL / world 1: single
 * GPU; otherwise as pnode_mlp_rk_adjoint_dp. */
int pnode_mlp_rk_forward_so(const pnode_mlp_desc *mlp, const pnode_rk_tableau *tab, const void *d_u0, int64_t ntraj,
                            const pnode_step *d_sched, int nsteps, void *d_sol, void *d_usteps, void *stream);
int pnode_mlp_rk_adjoint_so(const pnode_mlp_desc *mlp, const pnode_rk_tableau *tab, int64_t ntraj,
                            const pnode_step *d_sched, int nsteps, int last_slot, const void *d_gout,
                            const void *d_usteps, void *d_lambda, void *d_mu, void *d_work, const uint64_t *d_peer_bufs,
                            int rank, int world, uint64_t epoch, void *stream);

/* ----------------------------------------------------------------------------------------------------------------
 * Fused path for FFJORD continuous-normalising-flow right-hand sides (ffjord-pnode/lib/layers/odefunc.py:322-385 with
 * an ODEnet of two ConcatSquashLinear layers + softplus, diffeq_layers/basic.py:76-86):
 *     a    = (W1 z + b1) * sigmoid(hgw1 t + hgb1) + hb1 t            hidden pre-activation   [H]
 *     dz   = (W2 softplus(a) + b2) * sigmoid(hgw2 t + hgb2) + hb2 t                          [D]
 *     dlogp = - e^T (d dz / d z) e           Hutchinson estimator, e fixed per solve (odefunc.py:53-57, 359-364)
 * evaluated ANALYTICALLY per trajectory (no autograd graph, no second-order autograd in the adjoint).  State layout is the
 * reference's flattened cat(z.view(-1), logp.view(-1)) (cnf.py:74, 140-142): z block [ntraj, D] then logp block [ntraj].
 * Parameter / mu order = func.parameters(): per layer _layer.weight, _layer.bias, _hyper_bias.weight,
 * _hyper_gate.weight, _hyper_gate.bias.
 * -------------------------------------------------------------------------------------------------------------- */

typedef struct pnode_cnf_desc {
    int32_t dim;     /* D (6 for POWER) */
    int32_t hidden;  /* H (60) */
    int32_t dtype;
    int32_t t_via_f32; /* 1: the module rounds t through float32 (odefunc.py:356 `torch.tensor(t).type_as(y)`) */
    const void *d_w1, *d_b1, *d_hb1, *d_hgw1, *d_hgb1; /* [H,D], [H], [H], [H], [H] */
    const void *d_w2, *d_b2, *d_hb2, *d_hgw2, *d_hgb2; /* [D,H], [D], [D], [D], [D] */
    const void *d_e;                                   /* [ntraj, D] Hutchinson probe */
} pnode_cnf_desc;

int pnode_cnf_rk_supported(int dim, int hidden, int dtype, int stages);

/* ONE step attempt of an explicit RK scheme from (t, u) with size h: all stages, completion, and -- when d_sumsq is not
 * NULL and the tableau has embedded weights -- the weighted squared error sum of [PETSc] TSErrorWeightedNorm2 over the
 * local shard (deterministic reduction, see pnode_rk_complete_wrms).  Accept/reject stays with the caller, who first
 * all-reduces *d_sumsq across ranks.  Replaces one pass of [PETSc] TSStep_RK + TSEvaluateStep_RK + the reference's
 * evalRHSFunction callbacks (petsc_adjoint.py:393-412).
 *   d_u, d_unew   [ntraj*(D+1)]      current state / candidate u_{n+1}
 *   d_kfsal_in    [ntraj*(D+1)] or NULL: slope f(t,u) carried over from the previous ACCEPTED step (FSAL tableaux)
 *   d_kfsal_out   [ntraj*(D+1)] or NULL: receives the last stage slope
 *   d_ckpt        [s_eff, D, ntraj] or NULL: z-part of the stage values Y_i (s_eff = s-1 for FSAL tableaux)
 */
int pnode_cnf_rk_attempt(const pnode_cnf_desc *cnf, const pnode_rk_tableau *tab, const void *d_u,
                         const void *d_kfsal_in, int64_t ntraj, double t, double h, void *d_unew, void *d_kfsal_out,
                         void *d_ckpt, double atol, double rtol, double *d_sumsq, void *d_work, void *stream);

/* The same attempt with the STEP CONTROLLER ON THE DEVICE: [PETSc] TSAdaptChoose_Basic (accept iff the weighted error norm
 * <= 1, h_next = h clip(safety enorm^(-1/order), 0.1, 10), halved safety after a rejected attempt), the MATCHSTEP clamp onto the
 * next output time and pnode's tspanPostStep bookkeeping (petsc_adjoint.py:518-532) are evaluated by the last block of the
 * attempt kernel, which then publishes (t, h, buffers to use) for the next attempt in *d_ctl.  The host launches `nlaunch`
 * attempts back to back with NO read in between (attempts launched after the end time has been reached return at once) and
 * reads d_ctl once per batch.  State lives in ping-pong buffers: d_ubuf [2][ntraj*(D+1)] (ctl->cur selects the current state),
 * d_kbuf [2][ntraj*(D+1)] (FSAL slope); stage checkpoints of accepted step n go to d_ckpt_base + n * ckpt_step_elems (the host
 * guarantees room for ctl->steps + nlaunch steps; NULL: no checkpoints); states at the output times go to d_sol [nspan][ntraj*(D+1)]
 * (NULL when nspan == 0).  Every attempt is logged (t, h, error norm, accepted) for the host's
 * bookkeeping.  Single rank only (a batch-sharded run needs the cross-rank sum of the error norm before the decision). */
#define PNODE_CTL_MAX_SPAN 16
#define PNODE_CTL_MAX_LOG 1024
typedef struct pnode_cnf_ctl {
    double t, h, t_end;              /* next attempt starts at t with size h */
    double dt_span_cached;           /* [PETSc] tspan: un-shortened step remembered across an output-time hit */
    double span[PNODE_CTL_MAX_SPAN]; /* output times (nspan == 0: single end time, integrate [t, t_end]) */
    double n_global;                 /* length of the state vector in the WRMS norm */
    double delta;                    /* tspanPostStep hit tolerance: 1e-5 (fp64) / 1e-3 (fp32) */
    int32_t nspan, order, max_reject;
    int32_t done;                    /* 0 running, 1 end time reached, 2 too many rejections, 3 log full, 4 max_steps reached */
    int32_t cur, kcur, have_k;       /* ping-pong indices of d_ubuf / d_kbuf; have_k: a carried-over FSAL slope exists */
    int32_t steps, attempts, rejections, prev_ok;
    int32_t ctr, cur_sol_index;      /* [PETSc] tspan->spanctr; pnode's cur_sol_index */
    int32_t pending_slot;            /* output slot the state reached by the last accepted step belongs to (-1: none); the
                                        NEXT attempt copies its input state there (the final state is read from d_ubuf) */
    int32_t max_steps;               /* room in the checkpoint buffer: the loop stops (done = 4) when ctl->steps reaches it and
                                        the end time has not been reached (0: no limit) */
    int32_t single;                  /* 1: one-element t (no forcing at interior output times: in_slot = -1 everywhere) */
    int32_t prev_out_slot;           /* output slot of the previous accepted step (forcing slot of the next one) */
    double sumsq;                    /* the last attempt's weighted error sum of squares (the global one in sharded runs) */
    uint64_t epoch_next;             /* sharded runs (pnode_cnf_rk_solve_ctl_dp): number of the next in-kernel collective; the
                                        host sets it before the solve and reads back how far the loop got */
    double log_t[PNODE_CTL_MAX_LOG], log_h[PNODE_CTL_MAX_LOG], log_enorm[PNODE_CTL_MAX_LOG];
    int32_t log_accepted[PNODE_CTL_MAX_LOG];
    pnode_step sched[PNODE_CTL_MAX_LOG]; /* the accepted steps, in the form the adjoint sweep consumes (first ctl->steps entries) */
} pnode_cnf_ctl;
int pnode_cnf_rk_attempts_ctl(const pnode_cnf_desc *cnf, const pnode_rk_tableau *tab, void *d_ubuf, void *d_kbuf,
                              int64_t ntraj, void *d_ckpt_base, int64_t ckpt_step_elems, void *d_sol, double atol,
                              double rtol, pnode_cnf_ctl *d_ctl, void *d_work, int nlaunch, void *stream);

/* The whole adaptive time loop in ONE launch: a CUDA graph whose WHILE node repeats the attempt kernel for as long as the
 * last block of the previous attempt left ctl->done == 0 (it calls cudaGraphSetConditional on the node's handle).  Same
 * arguments and state as pnode_cnf_rk_attempts_ctl; no host involvement until the loop ends -- with done = 1 (finished),
 * 2 (more than max_reject rejections in a row), 3 (attempt log full: reset ctl->attempts and call again) or 4 (ctl->steps
 * reached ctl->max_steps: provide more checkpoint room and call again).  Graphs are cached by their full argument list
 * (the arguments are baked into the kernel node), so callers should reuse their buffers.  Must not be called on a stream
 * that is itself being captured. */
int pnode_cnf_rk_solve_ctl(const pnode_cnf_desc *cnf, const pnode_rk_tableau *tab, void *d_ubuf, void *d_kbuf,
                           int64_t ntraj, void *d_ckpt_base, int64_t ckpt_step_elems, void *d_sol, double atol, double rtol,
                           pnode_cnf_ctl *d_ctl, void *d_work, void *stream);
/* Batch-sharded variant: every rank runs the loop on its shard; the last block of each attempt all-reduces the weighted error
 * sum of squares over NVLink peer memory (same symmetric inbox and flag protocol as the *_adjoint_dp kernels, collective number
 * ctl->epoch_next++), so all ranks take the same verdict and the same next step -- no NCCL call, no host in the loop.
 * ctl->n_global is the state length of the WHOLE batch. */
int pnode_cnf_rk_solve_ctl_dp(const pnode_cnf_desc *cnf, const pnode_rk_tableau *tab, void *d_ubuf, void *d_kbuf,
                              int64_t ntraj, void *d_ckpt_base, int64_t ckpt_step_elems, void *d_sol, double atol, double rtol,
                              pnode_cnf_ctl *d_ctl, void *d_work, const uint64_t *d_peer_bufs, int rank, int world,
                              void *stream);

/* An adaptive solve with NO host in it at all (so that the caller's whole training step can be captured in a CUDA graph):
 *   pnode_cnf_rk_attempts_ctl(..., nlaunch)   a fixed budget of attempts (the ones after the end time return at once);
 *   pnode_cnf_rk_gather_ctl                   d_out[k] (k = 1 .. nout-1; [nout][ntraj*(D+1)]) <- the states at the output times
 *                                             (the last one from d_ubuf); NaN everywhere if the budget did not reach the end
 *                                             time (ctl->done != 1), so that an unfinished solve cannot pass unnoticed;
 *   pnode_cnf_rk_adjoint_ctl                  the adjoint sweep over ctl->sched[0 .. ctl->steps), read on the device. */
int pnode_cnf_rk_gather_ctl(const pnode_cnf_ctl *d_ctl, const void *d_ubuf, const void *d_sol, void *d_out, int nout,
                            int64_t n, int dtype, void *stream);
int pnode_cnf_rk_adjoint_ctl(const pnode_cnf_desc *cnf, const pnode_rk_tableau *tab, int64_t ntraj, const pnode_cnf_ctl *d_ctl,
                             int last_slot, const void *d_gout, const void *d_ckpt, void *d_lambda, void *d_mu, void *d_work,
                             void *stream);

/* Test hook: feeds `n` weighted error sums of squares to the device step controller one after the other (one thread, the
 * code path the attempt kernel's last block runs) -- so that its decisions can be compared with the host controller on
 * sequences no real solve produces.  Stops early when ctl->done becomes non-zero. */
int pnode_cnf_ctl_probe(pnode_cnf_ctl *d_ctl, const double *d_sumsq, int n, void *stream);

/* Whole discrete-adjoint sweep over the accepted steps (same conventions as pnode_mlp_rk_adjoint); the per-stage VJP
 * (RHSJacShell.multTranspose, petsc_adjoint.py:52-82, which needs second-order autograd in the reference) is evaluated
 * analytically.  d_ckpt is [nsteps, s_eff, D, ntraj]; d_gout / d_lambda use the flattened state layout. */
int64_t pnode_cnf_rk_adjoint_work_bytes(const pnode_cnf_desc *cnf);
int pnode_cnf_rk_adjoint(const pnode_cnf_desc *cnf, const pnode_rk_tableau *tab, int64_t ntraj,
                         const pnode_step *d_sched, int nsteps, int last_slot, const void *d_gout, const void *d_ckpt,
                         void *d_lambda, void *d_mu, void *d_work, void *stream);

/* ----------------------------------------------------------------------------------------------------------------
 * Convolutional ODE block (BASELINE config 4: the SqueezeNext block of examples-pnode/models/sqnxt_PETSc.py:70-121, five
 * times relu(bn(conv(x))) with nn.BatchNorm2d in TRAIN mode).  On the reference's path evalRHSFunction
 * (petsc_adjoint.py:393-412) and RHSJacShell.multTranspose (52-82) spend most of their GPU time in cuDNN's one-CTA-per-
 * channel batch-norm kernels; these entry points are the train-mode BatchNorm2d + ReLU forward / backward as
 * many-CTA-per-channel HBM-streaming reductions (NCHW, contiguous, H*W a multiple of 16 bytes).
 *   forward : y = relu(gamma (x - mean_c) / sqrt(var_c + eps) + beta); saves mean_c / inv-std_c; updates
 *             running_mean / running_var like nn.BatchNorm2d (momentum, unbiased variance) when they are not NULL.
 *   backward: dx, dgamma, dbeta from dy (gradient w.r.t. the ReLU output), the saved x, y, mean, inv-std.
 * d_work: pnode_bn_work_bytes(C) bytes of scratch (per-CTA partial sums; reductions are formed in a fixed order).
 * -------------------------------------------------------------------------------------------------------------- */
int64_t pnode_bn_work_bytes(int channels);
int pnode_bn_relu_forward(const void *d_x, void *d_y, const void *d_gamma, const void *d_beta, void *d_running_mean,
                          void *d_running_var, void *d_save_mean, void *d_save_invstd, int N, int C, int HW, double eps,
                          double momentum, void *d_work, int dtype, void *stream);
int pnode_bn_relu_backward(const void *d_dy, const void *d_x, const void *d_y, const void *d_gamma,
                           const void *d_save_mean, const void *d_save_invstd, void *d_dx, void *d_dgamma,
                           void *d_dbeta, int N, int C, int HW, void *d_work, int dtype, void *stream);

/* ----------------------------------------------------------------------------------------------------------------
 * Whole right-hand side of a convolutional ODE block and its vector-Jacobian products (csrc/conv_block.cu): a chain of
 * relu(bn_k(conv_k(.))) with stride-1 "same" convolutions of kernel 1x1, (1,3) or (3,1) and train-mode BatchNorm2d
 * (sqnxt_PETSc.py:70-121).  One kernel per layer: BatchNorm+ReLU of the previous layer applied on load, convolution,
 * bias, batch statistics of the next BatchNorm in the epilogue; relu(bn(z)) is never written between layers.
 *   pnode_convblock_forward  replaces evalRHSFunction for this module family (petsc_adjoint.py:393-412) and, with d_base,
 *                            the [PETSc] VecMAXPY that follows it in TSStep_RK:   k = f(x);  out = base_coef*base + k_coef*k
 *   pnode_convblock_vjp      replaces RHSJacShell.multTranspose (petsc_adjoint.py:52-82: forward re-evaluation + backward)
 *                            and RHSJacPShell.multTranspose + [PETSc] VecAXPY on mu (341-363):
 *                            vu = (df/dx)^T w;   grads = (df/dp)^T w   or   grads += coef * (df/dp)^T w  (accumulate != 0)
 * Both advance running_mean / running_var / num_batches_tracked of every layer once, like the module's forward.
 * Parameter order of d_grads = func.parameters(): per layer conv.weight [cout,cin,kh,kw], conv.bias, bn.weight, bn.bias.
 * Tensors are NCHW contiguous, 16-byte aligned; W a power of two in 4..128; channel counts multiples of 4.
 * Memory: d_act (pnode_convblock_act_bytes) receives the raw layer outputs z_1..z_L and the exact batch statistics of ONE
 * evaluation -- the forward's by-product; kept by the caller, it lets the adjoint skip the forward re-evaluation of that stage
 * (act_valid != 0: same x, same parameters; the BatchNorm buffers still advance once, as the module's re-evaluation would).
 * d_work (pnode_convblock_work_bytes) is scratch shared by all calls.  Neither needs initialising.
 * Batch statistics are accumulated exactly (128-bit fixed point, integer atomics): results are bit-reproducible.
 * -------------------------------------------------------------------------------------------------------------- */
#define PNODE_CONV_MAX_LAYERS 8
typedef struct pnode_conv_layer {
    int32_t cin, cout, kh, kw, ph, pw;
    const void *d_weight, *d_bias;          /* conv */
    const void *d_gamma, *d_beta;           /* BatchNorm affine */
    void *d_running_mean, *d_running_var;   /* may be NULL */
    void *d_num_batches_tracked;            /* int64 on the device, may be NULL */
    double eps, momentum;
} pnode_conv_layer;

typedef struct pnode_convblock_desc {
    int32_t nlayers, dtype;
    int32_t N, H, W, reserved;
    pnode_conv_layer layer[PNODE_CONV_MAX_LAYERS];
    /* Batch-sharded runs (one process per GPU; all zero / NULL otherwise).  BatchNorm statistics must be those of the GLOBAL
     * batch: the last CTA of every statistics-producing kernel exchanges this rank's exact totals with the other ranks through
     * the symmetric-memory inbox of pnode_peer_buffer_bytes() (same buffer, flags and epoch counter as *_adjoint_dp below:
     * peer stores over NVLink + system-scope release/acquire flags, no NCCL call, no extra launch) and the integer sums make
     * every rank's statistics bit-identical to a single-GPU run of the whole batch.  A forward call consumes nlayers
     * consecutive epochs starting at `epoch`; a vjp call nlayers (+ nlayers more when it re-evaluates the forward).
     * The BatchNorm affine gradients written by pnode_convblock_vjp are global: rank 0 alone contributes them to d_grads, so
     * that the caller's all-reduce(sum) of mu over ranks counts them once. */
    const uint64_t *d_peer_bufs;   /* DEVICE array [world] of peer-mapped inbox base addresses */
    int32_t rank, world;
    uint64_t epoch;                /* first collective number of this call (>= 1, strictly increasing, equal on all ranks) */
    int64_t global_pixels;         /* N*H*W summed over ranks */
} pnode_convblock_desc;

int64_t pnode_convblock_act_bytes(const pnode_convblock_desc *desc);   /* -1: unsupported shape (pnode_last_error) */
int64_t pnode_convblock_work_bytes(const pnode_convblock_desc *desc);
int64_t pnode_convblock_param_count(const pnode_convblock_desc *desc);
/* d_out (may be NULL) = base_coef * d_base + k_coef * f(x)  (d_base NULL: d_out = f(x));  d_k (may be NULL) = f(x) */
int pnode_convblock_forward(const pnode_convblock_desc *desc, const void *d_x, void *d_out, const void *d_base,
                            double base_coef, double k_coef, void *d_k, void *d_act, void *stream);
/* d_vu (may be NULL: parameter gradients only); d_grads (may be NULL: state VJP only) [param_count] */
int pnode_convblock_vjp(const pnode_convblock_desc *desc, const void *d_x, const void *d_w, void *d_vu, void *d_grads,
                        double coef, int accumulate, void *d_act, int act_valid, void *d_work, void *stream);

/* The same right-hand side on the TENSOR CORES (csrc/conv_mma.cu) for GEMM-sized shapes (few pixels, many channels: the
 * CIFAR blocks [256,128,8,8] and [256,256,4,4]; fp32): every convolution, data gradient and weight gradient is an
 * implicit GEMM through the sliced products above (3xTF32), BatchNorm + ReLU folded into the operand gathers, batch
 * statistics and ReLU masks in the products' epilogues.  Same descriptor, same contract and reference lines as
 * pnode_convblock_forward / _vjp; additionally d_wbuf (pnode_convmma_weight_bytes) holds the weight operands written by
 * pnode_convmma_prepare once per solve, and d_work is needed by the forward as well.  N*H*W <= 65536, channel counts
 * multiples of 4 and >= 8, kernels 1x1 / (1,3) / (3,1) with "same" padding. */
int64_t pnode_convmma_act_bytes(const pnode_convblock_desc *desc);     /* -1: unsupported shape (pnode_last_error) */
int64_t pnode_convmma_work_bytes(const pnode_convblock_desc *desc);
int64_t pnode_convmma_weight_bytes(const pnode_convblock_desc *desc);
int64_t pnode_convmma_param_count(const pnode_convblock_desc *desc);
int pnode_convmma_prepare(const pnode_convblock_desc *desc, void *d_wbuf, void *stream);
int pnode_convmma_forward(const pnode_convblock_desc *desc, const void *d_wbuf, const void *d_x, void *d_out,
                          const void *d_base, double base_coef, double k_coef, void *d_k, void *d_act, void *d_work,
                          void *stream);
int pnode_convmma_vjp(const pnode_convblock_desc *desc, const void *d_wbuf, const void *d_x, const void *d_w, void *d_vu,
                      void *d_grads, double coef, int accumulate, void *d_act, int act_valid, void *d_work, void *stream);

/* ----------------------------------------------------------------------------------------------------------------
 * Data-parallel variants of the adjoint sweeps: the all-reduce of mu over the GPUs of one NVLink/NVSwitch domain is fused
 * into the tail of the sweep kernel (one-shot all-reduce over peer-mapped symmetric memory: peer stores + system-scope
 * release/acquire flags; no NCCL call, no extra launch).  The reference has no counterpart (single process,
 * petsc_adjoint.py:367); it replaces the `all_reduce(mu)` a data-parallel training loop would issue after
 * OdeintAdjointMethod.backward (petsc_adjoint.py:916-947).
 * d_peer_bufs: DEVICE array [world] with the peer-mapped base address of every rank's symmetric buffer of
 * pnode_peer_buffer_bytes(world) bytes (zero-initialised once); epoch: strictly increasing (>= 1) across calls and equal on
 * all ranks.  world == 1 or d_peer_bufs == NULL: identical to the non-DP entry points.
 * -------------------------------------------------------------------------------------------------------------- */
#define PNODE_PEER_NP_MAX 1024
int64_t pnode_peer_buffer_bytes(int world);
int pnode_mlp_rk_adjoint_dp(const pnode_mlp_desc *mlp, const pnode_rk_tableau *tab, int64_t ntraj,
                            const pnode_step *d_sched, int nsteps, int last_slot, const void *d_gout, const void *d_ckpt,
                            void *d_lambda, void *d_mu, void *d_work, const uint64_t *d_peer_bufs, int rank, int world,
                            uint64_t epoch, void *stream);
int pnode_cnf_rk_adjoint_dp(const pnode_cnf_desc *cnf, const pnode_rk_tableau *tab, int64_t ntraj,
                            const pnode_step *d_sched, int nsteps, int last_slot, const void *d_gout, const void *d_ckpt,
                            void *d_lambda, void *d_mu, void *d_work, const uint64_t *d_peer_bufs, int rank, int world,
                            uint64_t epoch, void *stream);

/* ----------------------------------------------------------------------------------------------------------------
 * Tensor-core matrix products on SLICED operands (csrc/umma_gemm.cu): TMA-fed tcgen05.mma, accumulators in tensor
 * memory.  They replace the library GEMMs the reference reaches through ATen for wide right-hand sides: the Linear
 * layers of examples-sinode/KS/models/imex.py:40-70 (forward in evalRHSFunction, pnode/petsc_adjoint.py:393-412; the
 * two backward products per layer inside RHSJacShell.multTranspose's autograd.grad, 52-82) and the batched solve
 * X = R A^-1 of pnode/torch_linearsolve.py:25-35 (inverse-apply as one product).
 *
 * A sliced operand holds a row-major matrix [rows][k] as S slice matrices [S][rows][pitch] (pitch = k elements rounded
 * up to 128 bytes) such that products of slices are exact on the tensor cores:
 *   PNODE_SLICED_I8   fp64 source: x[r][c] = 2^exp[r] * sum_s q_s[r][c] 2^-(6+8s), q_s signed bytes (balanced base-256
 *                     digits), S = PNODE_I8_SLICES = 6 (Ozaki splitting: int8 x int8 -> int32 products are exact on the
 *                     tensor cores; 46 bits of every entry relative to its row maximum, rounded to nearest, are kept for
 *                     row maxima in [2^-961, 2^960); the row exponent is clamped to [-960, 960], so smaller rows keep 46
 *                     bits relative to 2^-960 and rows of 2^960 and above are outside the range; a product needs the 21
 *                     slice pairs i + j < 6).  Reduction length <= PNODE_I8_MAX_K (int32 accumulators).
 *   PNODE_SLICED_I8X  signed digits in [-64, 64], base 128, S = PNODE_I8X_SLICES = 8 (55 bits, same exponent range, 36 slice
 *                     pairs, reduction length <= PNODE_I8X_MAX_K = 65535: diagonal 7 sums 8 digit pairs of up to 64 x 64 per
 *                     reduction index in int32): the truncation error of a sliced product is relative to (row maximum)(column
 *                     maximum), so products whose terms cancel by many orders of magnitude -- applying (shift I - J)^-1 of a
 *                     stiff operator to a rough vector -- need the extra digits to stay at fp64 level
 *   PNODE_SLICED_TF32 fp32 source: x = hi + lo with hi = tf32(x), S = 2 (3xTF32: hi.hi + hi.lo + lo.hi)
 * pnode_slice_rows slices x itself (operand row = row of x); pnode_slice_cols slices x^T (operand row = column of x,
 * reduction over the rows of x) and can add coef * (column sums of x) into d_colsum (bias gradients).
 * pnode_sliced_gemm:  C[m][n] (op)= mask( relu( alpha * ( sum_k A[m][k] B[n][k] + bias[n] ) ) ),  C row-major with leading
 * dimension ldc, fp64 for I8 operands / fp32 for TF32; `accumulate` adds into C; mask (same type and layout as C,
 * leading dimension ldmask) keeps the result where mask > 0 (ReLU backward).  d_a_exp / d_b_exp: the row exponents
 * written by the slicing kernels (ignored for TF32).
 * -------------------------------------------------------------------------------------------------------------- */
#define PNODE_SLICED_I8 0
#define PNODE_SLICED_TF32 1
#define PNODE_SLICED_I8X 2   /* int8 slices with one more digit (55 bits): for products with heavy cancellation */
#define PNODE_I8_SLICES 6
#define PNODE_I8X_SLICES 8
#define PNODE_I8_MAX_K 16384
#define PNODE_I8X_MAX_K 65535
int64_t pnode_sliced_bytes(int kind, int rows, int k);
int pnode_slice_rows(int kind, const void *d_x, int64_t ldx, int rows, int k, void *d_slices, int32_t *d_exp, void *stream);
int pnode_slice_cols(int kind, const void *d_x, int64_t ldx, int rows, int cols, void *d_slices, int32_t *d_exp,
                     void *d_colsum, double coef, void *stream);
int pnode_sliced_gemm(int kind, const void *d_a, const int32_t *d_a_exp, const void *d_b, const int32_t *d_b_exp, int M,
                      int N, int K, void *d_c, int64_t ldc, double alpha, const void *d_bias, int relu, const void *d_mask,
                      int64_t ldmask, int accumulate, void *stream);

/* ----------------------------------------------------------------------------------------------------------------
 * Wide ReLU-MLP right-hand side f(t, u) = out_scale * net(u), net = Linear -> ReLU -> ... -> Linear (csrc/dense_mlp.cu):
 * the explicit half of the SINODE pair (ODEFuncEX, examples-sinode/KS/models/imex.py:46-70: returns -F(y);
 * examples-sinode/Burgers/Burgers.py:134-160: returns net(y)).  One call per right-hand-side evaluation
 * (replaces evalRHSFunction -> func(t, u), pnode/petsc_adjoint.py:393-412) and one per adjoint stage (replaces
 * RHSJacShell.multTranspose's forward re-evaluation + autograd.grad, 52-82, AND RHSJacPShell.multTranspose + the VecAXPY on
 * mu, 341-363: the weight gradients are accumulated straight into mu by the product's epilogue).  Every product runs
 * on the tensor cores through the sliced operands above (fp64: int8 slices; fp32: 3xTF32).
 *   prepare : slice every weight matrix in both orientations (once per solve: parameters are borrowed, never cached
 *             across optimiser steps)
 *   forward : d_out[batch][dims[L]] = f(d_u[batch][dims[0]]); with d_act != NULL the evaluation keeps what the adjoint
 *             stage at the same point needs (column-sliced layer inputs, post-ReLU activations) -- the stage checkpoint
 *             of this right-hand side
 *   vjp     : d_vu = J^T w (skipped if NULL);  if d_mu != NULL:  mu[mu_w_off[l] ...] += coef * dW_l,
 *             mu[mu_b_off[l] ...] += coef * db_l  (offsets in elements, -1: that parameter takes no gradient)
 * -------------------------------------------------------------------------------------------------------------- */
#define PNODE_DMLP_MAX_LAYERS 8
typedef struct pnode_dmlp_desc {
    int32_t nlayers, dtype, batch, reserved;
    int32_t dims[PNODE_DMLP_MAX_LAYERS + 1];        /* dims[0] = input width ... dims[nlayers] = output width */
    const void *d_weight[PNODE_DMLP_MAX_LAYERS];    /* [dims[l+1]][dims[l]] row-major (torch nn.Linear.weight) */
    const void *d_bias[PNODE_DMLP_MAX_LAYERS];      /* [dims[l+1]] or NULL */
    int64_t mu_w_off[PNODE_DMLP_MAX_LAYERS];
    int64_t mu_b_off[PNODE_DMLP_MAX_LAYERS];
    double out_scale;
} pnode_dmlp_desc;
int64_t pnode_dmlp_weight_bytes(const pnode_dmlp_desc *desc);   /* -1: unsupported (pnode_last_error) */
int64_t pnode_dmlp_act_bytes(const pnode_dmlp_desc *desc);
int64_t pnode_dmlp_work_bytes(const pnode_dmlp_desc *desc);
int pnode_dmlp_prepare(const pnode_dmlp_desc *desc, void *d_wslices, void *stream);
int pnode_dmlp_forward(const pnode_dmlp_desc *desc, const void *d_wslices, const void *d_u, void *d_out, void *d_act,
                       void *d_work, void *stream);
int pnode_dmlp_vjp(const pnode_dmlp_desc *desc, const void *d_wslices, const void *d_act, const void *d_w, void *d_vu,
                   void *d_mu, double coef, void *d_work, void *stream);
/* Same, recording layer_events[l] (HOST array of nlayers cudaEvent_t, entries may be NULL) on the stream right after the last
 * kernel that adds to layer l's slice of mu (weight and bias gradient).  Layers are processed last to first, so a
 * batch-sharded caller can start the all-reduce of a layer's gradient while the earlier layers are still being
 * differentiated (pnode_b200/petsc_adjoint.py, the 298 MB mu of BASELINE config 5). */
int pnode_dmlp_vjp_ev(const pnode_dmlp_desc *desc, const void *d_wslices, const void *d_act, const void *d_w, void *d_vu,
                      void *d_mu, double coef, void *d_work, void *const *layer_events, void *stream);

/* ----------------------------------------------------------------------------------------------------------------
 * FFJORD right-hand side with an ODEnet of any depth (csrc/cnf_net.cu): L ConcatSquashLinear layers with Softplus(beta=1,
 * threshold=20) between them, state cat(z.view(-1), logp.view(-1)) of B samples.  The trace is the Hutchinson estimate
 * e^T J e with the probe d_e (trace = 0, divergence_approx) or the exact trace tr J (trace = 1, divergence_bf; d_e is not
 * read), formed as the forward tangents of one chain (e) or of D chains (the unit vectors).
 * Replaces ODEfunc.forward (ffjord-pnode/lib/layers/odefunc.py:53-57, 345-385; ConcatSquashLinear, diffeq_layers/basic.py:
 * 76-86) in evalRHSFunction, and the second-order autograd of RHSJacShell.multTranspose + RHSJacPShell.multTranspose
 * (pnode/petsc_adjoint.py:52-82, 341-363) in every adjoint stage.  Every product runs on the tensor cores through the
 * sliced operands above (fp64: int8 slices, I8X when (1 + chains) B or a width exceeds PNODE_I8_MAX_K; fp32: 3xTF32), with
 * the value and tangent chains stacked as (1 + chains) B rows (2B for the Hutchinson trace, (D + 1) B for the exact one),
 * which must be within one product's reduction length (PNODE_I8X_MAX_K in fp64, 65536 in fp32).
 *   prepare : slice every weight matrix in both orientations (once per solve: parameters are borrowed)
 *   forward : d_out[B*(D+1)] = F(t, d_u); with d_act != NULL the evaluation keeps what the adjoint stage at the same point
 *             needs (column-sliced layer inputs, pre-activations, gates)
 *   vjp     : from the activation set of a forward at the same t: d_vu = J^T w (skipped if NULL); if d_mu != NULL,
 *             mu[<param>_off[l] ...] += coef * d<param>_l (offsets in elements, -1: that parameter takes no gradient).
 *             Bit-reproducible: the column sums are combined in a fixed order.
 * -------------------------------------------------------------------------------------------------------------- */
typedef struct pnode_cnfnet_desc {
    int32_t nlayers, dtype, batch, t_f32;         /* t_f32 = 1: the module rounds t through float32 (odefunc.py:356) */
    int32_t dims[PNODE_DMLP_MAX_LAYERS + 1];      /* dims[0] = D ... dims[nlayers] = D */
    const void *d_weight[PNODE_DMLP_MAX_LAYERS];  /* _layer.weight [dims[l+1]][dims[l]] */
    const void *d_bias[PNODE_DMLP_MAX_LAYERS];    /* _layer.bias [dims[l+1]] */
    const void *d_hyper_bias[PNODE_DMLP_MAX_LAYERS];  /* _hyper_bias.weight [dims[l+1]][1] */
    const void *d_gate_weight[PNODE_DMLP_MAX_LAYERS]; /* _hyper_gate.weight [dims[l+1]][1] */
    const void *d_gate_bias[PNODE_DMLP_MAX_LAYERS];   /* _hyper_gate.bias [dims[l+1]] */
    int64_t mu_w_off[PNODE_DMLP_MAX_LAYERS], mu_b_off[PNODE_DMLP_MAX_LAYERS], mu_hbw_off[PNODE_DMLP_MAX_LAYERS],
        mu_hgw_off[PNODE_DMLP_MAX_LAYERS], mu_hgb_off[PNODE_DMLP_MAX_LAYERS];
    const void *d_e;                              /* [B][D] Hutchinson probe (read when trace = 0) */
    int32_t trace;                                /* 0: Hutchinson e^T J e, 1: exact tr J */
} pnode_cnfnet_desc;
int64_t pnode_cnfnet_weight_bytes(const pnode_cnfnet_desc *desc);   /* -1: unsupported (pnode_last_error) */
int64_t pnode_cnfnet_act_bytes(const pnode_cnfnet_desc *desc);
int64_t pnode_cnfnet_work_bytes(const pnode_cnfnet_desc *desc);
int pnode_cnfnet_prepare(const pnode_cnfnet_desc *desc, void *d_wslices, void *stream);
int pnode_cnfnet_forward(const pnode_cnfnet_desc *desc, const void *d_wslices, double t, const void *d_u, void *d_out,
                         void *d_act, void *d_work, void *stream);
int pnode_cnfnet_vjp(const pnode_cnfnet_desc *desc, const void *d_wslices, double t, const void *d_act, const void *d_w,
                     void *d_vu, void *d_mu, double coef, void *d_work, void *stream);

/* Circulant linear operator J[i][j] = c[(i - j) mod n] applied to every row of d_x[rows][n] (the implicit half of the
 * SINODE pair: a circular-padding Conv1d stencil, imex.py:6-44; replaces evalIFunction's func(t, u), petsc_adjoint.py:
 * 414-431, and IJacShell's J^T x, 179-196).  `offsets` / `coefs` (HOST arrays, ntaps <= PNODE_CIRC_MAX_TAPS) list the
 * non-zero entries c[offsets[d]] = coefs[d].  transpose != 0 applies J^T. */
#define PNODE_CIRC_MAX_TAPS 16
int pnode_circulant_apply(const void *d_x, void *d_out, int rows, int n, const int32_t *offsets, const double *coefs,
                          int ntaps, int transpose, int dtype, void *stream);
/* d_inverse[n][n] = (shift * I - J)^-1 for the circulant J with first column d_col (fp64, on the device), from its
 * spectrum: lam_k = sum_j a_j exp(-2 pi i jk/n), inverse first column = (1/n) sum_k exp(2 pi i mk/n) / lam_k (compensated
 * O(n^2) sums, exact argument reduction).  Replaces torch_linearsolve.PCShell.get_factor's LU (pnode/torch_linearsolve.py:
 * 15-19); the solves of 25-35 become one sliced product with this matrix.  d_work: pnode_circulant_work_bytes(n). */
int64_t pnode_circulant_work_bytes(int n);
int pnode_circulant_inverse(const double *d_col, int n, double shift, void *d_inverse, int dtype, void *d_work, void *stream);

/* ----------------------------------------------------------------------------------------------------------------
 * Measurement helpers (bench.py): peak FMA issue rate of the CUDA-core pipe in the given dtype, used as the
 * compute-roofline denominator for the MLP kernels (MEASURED_PEAKS.json only has HBM and bf16 tensor peaks).
 * Launches a register-resident FMA chain on every SM; *flops = 2 * FMAs executed.  Synchronous.
 * -------------------------------------------------------------------------------------------------------------- */
int pnode_peak_fma(int dtype, int iters, double *flops, float *ms);

/* *d_out = sum of d_values[0..n) formed with the conv block's exact 128-bit fixed-point accumulator (integer atomics, one add per
 * thread, arbitrary order): unit-test hook for its exactness and order independence.  NaN if any value is not finite.
 * d_work: 256 bytes of scratch. */
int pnode_acc128_probe(const double *d_values, int64_t n, double *d_out, void *d_work, void *stream);

/* out[i] = tanh(in[i]) evaluated with the kernels' own tanh (unit-test hook for its accuracy). */
int pnode_tanh_probe(const void *d_in, void *d_out, int64_t n, int dtype, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* PNODE_B200_H */
