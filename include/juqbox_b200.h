/*
 * juqbox_b200.h — C ABI of the B200-native objective + adjoint-gradient path of Juqbox.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  The reference has no FFI: its boundary is the Julia
 * method  traceobjgrad(pcof0, params::objparams, wa::Working_Arrays, verbose, evaladjoint)
 * (/root/reference/src/evalobjgrad.jl:504) and its only production caller, the risk-neutral sample loop
 * eval_f_g_grad! (/root/reference/src/ipopt_interface.jl:24-70).  A Julia maintainer binds the entry points
 * below with `ccall` (see INTEGRATION.md and julia/JuqboxB200.jl); this repo's own host mirror binds them
 * with ctypes (juqbox_b200/_lib.py).
 *
 * Conventions: plain C, FP64 only, column-major matrices (Julia layout), 0-based CSC, host pointers unless the
 * name says `_device`.  Every function returns 0 on success or a negative jq_status; jq_last_error() gives the
 * text.  A handle is bound to one GPU and is not thread-safe (the reference is single-threaded, synchronous).
 * There is no CPU fallback: without a CUDA device jq_create fails with JQ_ERR_CUDA.
 */
#ifndef JUQBOX_B200_H
#define JUQBOX_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct jq_handle jq_handle;

typedef enum jq_status {
    JQ_OK = 0,
    JQ_ERR_ARG = -1,         /* bad argument / unsupported option (message says which) */
    JQ_ERR_PCOF_LENGTH = -2, /* mirrors error() at src/evalobjgrad.jl:604-606 and DimensionMismatch at src/bsplines.jl:178-181 */
    JQ_ERR_CUDA = -3,        /* CUDA runtime error, or no device */
    JQ_ERR_ALLOC = -4
} jq_status;

enum { JQ_DENSE = 0, JQ_CSC = 1 };

/* One real n x n operator: Hconst, Hsym_ops[q] or Hanti_ops[q] of objparams (src/evalobjgrad.jl:85-90).
 * JQ_DENSE: nzval = n*n values, column-major (Array{Float64,2}); colptr/rowval ignored.
 * JQ_CSC:   SparseMatrixCSC{Float64,Int64} converted to 0-based indices. */
typedef struct jq_operator {
    int32_t format;
    int64_t nnz;
    const int64_t *colptr; /* n+1 */
    const int64_t *rowval; /* nnz */
    const double *nzval;
} jq_operator;

/* The fields of `objparams` that the Stormer-Verlet path reads (SURVEY.md 8a row a10). */
typedef struct jq_problem {
    int32_t n;             /* Ntot = N + Nguard                         (evalobjgrad.jl:522) */
    int32_t m;             /* N, number of propagated columns           (:508)               */
    int32_t ncoupled;      /* length(Hsym_ops) == length(Hanti_ops)     (:170,:243)          */
    int32_t nfreq;         /* size(Cfreq, 2)                            (:169)               */
    int32_t neumann_terms; /* linear_solver.max_iter: Neumann terms, or the Jacobi sweep limit (linear_solvers.jl:41,46) */
    int32_t obj_func_type; /* objFuncType: 1 = infidelity+leak, 2/3 = also return infidelity-only gradient (:848-855) */
    int32_t pfid_type;     /* pFidType 1, 2, 3 or 4 (:755-763, :2026-2059); 2 is the reference constructor's value (:164).  With 3 every
                              pcof vector carries the global phase as an extra last entry and every gradient has one more entry
                              (:589-596, :923-945): npar below is then 2*(ncoupled+nuncoupled)*nfreq*D1 + 1 */
    int32_t linear_solver; /* linear_solver.solver_id: 0 or 1 = NEUMANN_SOLVER, 2 = JACOBI_SOLVER (linear_solvers.jl:4-5) */
    int64_t nsteps;
    double T;
    const double *uinit;     /* n*m, params.Uinit */
    const double *vtarget_r; /* n*m, params.Utarget_r */
    const double *vtarget_i; /* n*m, params.Utarget_i */
    const double *wdiag;     /* n, diagonal of params.wmat_real (Diagonal weights only) */
    const double *cfreq;     /* (ncoupled+nuncoupled)*nfreq, params.Cfreq[1:Nctrl,:] column-major: (c,f) at c + Nctrl*f */
    jq_operator h0;          /* params.Hconst */
    const jq_operator *hsym; /* ncoupled */
    const jq_operator *hanti;/* ncoupled */
    double solver_tol;       /* linear_solver.tol (Jacobi only; already multiplied by sqrt(nrhs), linear_solvers.jl:40) */
    /* --- SURVEY.md 8f rank 3; all zero / NULL = the core path --- */
    double global_phase;     /* params.globalPhase (pFidType 1 and 4) */
    const double *wmat_real; /* n*n column-major dense params.wmat_real when use_custom_forbidden (:214-232), else NULL: Diagonal(wdiag) */
    const double *wmat_imag; /* n*n column-major params.wmat_imag, or NULL (zero) */
    int32_t nuncoupled;      /* length(Hunc_ops): uncoupled (lab-frame) controls, two splines each as KS! reads them (:2372-2387) */
    int32_t reserved0;
    const jq_operator *hunc;      /* nuncoupled, each symmetric or antisymmetric */
    const int32_t *unc_is_symm;   /* nuncoupled: params.isSymm (:186-199) */
    const double *unc_rfreq;      /* nuncoupled: params.Rfreq[q] in GHz: f_q(t) = 2 (p cos(2 pi Rfreq t) - q sin(2 pi Rfreq t)) */
} jq_problem;

/* Replaces Working_Arrays(params, nCoeff) (src/evalobjgrad.jl:405): copies the problem to the GPU `device`,
 * builds the row-wise operator tables and picks the kernel.  Create once, reuse for every evaluation. */
int jq_create(const jq_problem *problem, int device, jq_handle **out);
int jq_destroy(jq_handle *h);

/* change_target! (src/evalobjgrad.jl:1492-1505): new n*m target, real and imaginary parts. */
int jq_update_target(jq_handle *h, const double *vtarget_r, const double *vtarget_i);

/* Batched traceobjgrad(pcof, params, wa, false, evaladjoint) — replaces the body of the `for i = 1:nquad` loop of
 * eval_f_g_grad! (src/ipopt_interface.jl:38-65) and the epsilon sweep of examples/Risk_Neutral/run_all.jl:9-28.
 *
 * Trajectory (b, s) evaluates candidate pcof[b*npar .. ] with Hconst + Diagonal(h0_diag_shift[s*n .. ]);
 * h0_diag_shift == NULL means nsamples must be 1 and no shift.  (The reference's noise model is
 * shift[j] = 0.01*ep*10^(j-2) for j = 2..n, 1-based, src/ipopt_interface.jl:41-44; any diagonal is accepted.)
 *
 * weights == NULL: per-trajectory outputs, index t = b*nsamples + s:  infid[t] (primaryobjf), leak[t]
 *   (secondaryobjf), trace_infid[t], grad[t*npar ..] (totalgrad) and, if obj_func_type != 1, infidgrad / leakgrad.
 * weights != NULL ([nsamples]): outputs are the weighted sums over s that eval_f_g_grad! accumulates
 *   (src/ipopt_interface.jl:48-59), one per candidate b.
 * Any output pointer may be NULL.  evaladjoint == 0 skips the backward sweep (gradients are not written).
 * For obj_func_type == 1 infidgrad receives a copy of grad (reference :951) and leakgrad is left untouched.
 * Blocking: returns after the results are in the host buffers. */
int jq_traceobjgrad_batch(jq_handle *h, int32_t nbatch, const double *pcof, int32_t npar, int32_t nsamples,
                          const double *h0_diag_shift, const double *weights, int32_t evaladjoint,
                          double *infid, double *leak, double *trace_infid, double *grad, double *infidgrad,
                          double *leakgrad);

/* Same, with every array already in device memory of the handle's GPU and the work enqueued on `cuda_stream`
 * (a cudaStream_t, used as given: NULL is CUDA's legacy default stream).  Asynchronous: no host synchronisation. */
int jq_traceobjgrad_batch_device(jq_handle *h, int32_t nbatch, const double *pcof, int32_t npar, int32_t nsamples,
                                 const double *h0_diag_shift, const double *weights, int32_t evaladjoint,
                                 double *infid, double *leak, double *trace_infid, double *grad,
                                 double *infidgrad, double *leakgrad, void *cuda_stream);

/* Fused Ipopt-callback entry: one call serves eval_f_par AND eval_grad_f_par (src/ipopt_interface.jl:77-148), plus eval_g_par /
 * eval_jac_g_par for objFuncType 3 (:104-179).  Everything those callbacks do per evaluation happens behind this call:
 *   - the last-evaluation cache: trajectories run only if ||pcof - last_pcof||_2 > 1e-15 (the reference's own test, :84,:131),
 *     otherwise the stored results are returned without touching the GPU;
 *   - eval_f_g_grad! (:24-70): the nsamples noise samples of ONE pcof in one launch, weighted sums on the device (and the
 *     all-reduce over sample shards if a communicator is attached); weights == NULL with nsamples == 1 means weight 1;
 *   - Tikhonov on the device (tikhonov_pen / tikhonov_grad!, src/evalobjgrad.jl:2291-2351):
 *       f      = last_infidelity (+ last_leak if objFuncType == 1) + tik0 * ||pcof - prior||^2 / npar          (:89-98)
 *       grad_f = last_infidelity_grad + 2 tik0 (pcof - prior) / npar   (the total gradient when objFuncType == 1, :136-141)
 *     prior == NULL means usingPriorCoeffs == false;
 *   - infid / leak: last_infidelity and last_leak (eval_g_par's g[1]); leakgrad: last_leak_grad (eval_jac_g_par), written
 *     only for objFuncType != 1.  Any output pointer may be NULL.  *evaluated = 1 if trajectories ran, 0 on a cache hit.
 * The cache is keyed on pcof like the reference's (nodes/weights are fixed per optimisation); jq_update_target,
 * jq_cache_invalidate and a changed nsamples or tik0-independent input (shift/weights pointers' contents are compared) reset it.
 * Host pointers, blocking. */
int jq_eval_f_grad(jq_handle *h, const double *pcof, int32_t npar, int32_t nsamples, const double *h0_diag_shift,
                   const double *weights, double tik0, const double *prior, double *f, double *grad_f, double *infid,
                   double *leak, double *leakgrad, int32_t *evaluated);
int jq_cache_invalidate(jq_handle *h);

/* Layout self-description for bindings that mirror the structs by hand (julia/JuqboxB200.jl, ctypes): what = 0 ABI version,
 * 1 sizeof(jq_problem), 2 sizeof(jq_operator), 3 offsetof(jq_problem, nsteps), 4 offsetof(T), 5 offsetof(uinit), 6 offsetof(h0),
 * 7 offsetof(hsym), 8 offsetof(solver_tol), 9 offsetof(jq_operator, nnz), 10 offsetof(jq_operator, nzval); -1 otherwise. */
int64_t jq_abi_info(int32_t what);

/* Forward propagation with state history: eval_forward(U0 = Uinit, pcof, params; saveEndOnly=false, saveEvery)
 * (src/evalobjgrad.jl:2727-2873) and the history that traceobjgrad(verbose=true, evaladjoint=false) returns
 * (:676-680,:748-752,:1029-1031).  hist_r / hist_i receive Re / Im of the state (vr and -vi) at t = 0 and after every
 * save_every-th step: [ntraj][nsteps/save_every + 1][n*m] doubles each, column-major n x m blocks (the Julia array
 * Ntot x N x nsave of each trajectory).  nsteps must be divisible by save_every (reference :2797-2799).  infid / leak as in
 * jq_traceobjgrad_batch (may be NULL).  Host pointers, blocking; same kernel selection as jq_traceobjgrad_batch. */
int jq_eval_forward(jq_handle *h, int32_t nbatch, const double *pcof, int32_t npar, int32_t nsamples,
                    const double *h0_diag_shift, int32_t save_every, double *hist_r, double *hist_i, double *infid, double *leak);

/* Forward sensitivities (the reference's traceobjgrad(verbose=true, evaladjoint=true) check, src/evalobjgrad.jl:724-745,768-784, for
 * ndir directions at once).  Trajectory (b, s, k) evaluates candidate b with sample shift s and differentiates along
 * dirs[(b*ndir + k)*npar ..].  One launch of the forward-sensitivity kernel (jq_query(h, 0) = 8) runs the forward sweep and its tangent
 * (step_fwdGrad!, src/StormerVerlet.jl:151-251; fgradforce!, src/evalobjgrad.jl:2467-2563) side by side for every trajectory, so
 * dirs = the unit vectors give the whole forward-mode gradient in one call, and dstate the sensitivity of the final state.
 * pcof, dirs, h0_diag_shift and weights as in jq_traceobjgrad_batch; with pFidType 3 every pcof and direction vector carries the
 * global phase as its last entry.
 * weights == NULL: infid[t], leak[t] with t = b*nsamples + s (the objective-only outputs of the generic kernel, bit for bit);
 *   dinfid[t*ndir + k], dleak[t*ndir + k], their directional derivatives; dstate_r / dstate_i [(t*ndir + k)][n*m] the tangents of
 *   Re and Im of the final state (vr' and -vi', the convention of jq_eval_forward), column-major n x m blocks.
 * weights != NULL ([nsamples]): infid[b], leak[b], dinfid[b*ndir + k], dleak[b*ndir + k], the weighted sums over s that
 *   eval_f_g_grad! forms (fixed summation order); dstate must then be NULL.
 * Any output may be NULL.  JQ_ERR_ARG (no launch) for ndir < 1, dirs == NULL, nbatch*nsamples*ndir > 2^31 - 1, the Jacobi solver,
 * weights with a dstate output, weights while a communicator of more than one rank is attached (this entry never communicates:
 * shard directions, not samples), or a problem whose trajectory does not fit in 227 KB of shared memory.
 * Host pointers, blocking. */
int jq_forward_sensitivity(jq_handle *h, int32_t nbatch, const double *pcof, int32_t npar, int32_t nsamples,
                           const double *h0_diag_shift, const double *weights, int32_t ndir, const double *dirs,
                           double *infid, double *leak, double *dinfid, double *dleak,
                           double *dstate_r, double *dstate_i);

/* Final-state vector-Jacobian products: the gradient of any real objective of the final state U(T), one backward sweep per cotangent
 * whatever npar is (the dual of dstate in jq_forward_sensitivity).  Trajectory (b, s, k) evaluates candidate b with sample shift s and
 * pulls back cotangent k.  One launch of the final-state VJP kernel (jq_query(h, 0) = 9) runs, per trajectory, the forward sweep and
 * then the backward sweep of the reference's unforced adjoint (the objFuncType 2/3 set, src/StormerVerlet.jl:365-406, gradient
 * src/evalobjgrad.jl:2567-2619) from the terminal condition lambda_r(T) = -cot_r / 2, lambda_i(T) = cot_i / 2.
 * Conventions: U(T) = vr - i vi as in jq_eval_forward, so Re U = vr and Im U = -vi.  With c = cot_r + i cot_i,
 *   vjp[p] = sum_e cot_r[e] dRe U[e]/dpcof[p] + cot_i[e] dIm U[e]/dpcof[p]  (= Re vdot(c, dU . e_p), vdot conjugating c),
 * which for a real loss L and c = dL/dRe U + i dL/dIm U is dL/dpcof.  With c = dinfid/d(Re U, Im U) the result is the infidelity
 * gradient of jq_traceobjgrad_batch for every pFidType.  The guard penalty, its weights and obj_func_type play no part; the solver and
 * uncoupled controls do.  pcof, h0_diag_shift as in jq_traceobjgrad_batch; with pFidType 3 every pcof and vjp vector carries the global
 * phase as its last entry, and U(T) does not depend on it: that entry of vjp is 0.
 * cot_r, cot_i: [(t*ncot + k)][n*m] with t = b*nsamples + s, column-major n x m blocks (the layout of dstate); NULL means zero, not both.
 * vjp: [(t*ncot + k)][npar].  state_r, state_i: [t][n*m], Re and Im of U(T), or NULL.
 * JQ_ERR_ARG (no launch) for ncot < 1, both cotangent parts NULL, vjp == NULL, nbatch*nsamples*ncot > 2^31 - 1, or a problem whose
 * trajectory does not fit in 227 KB of shared memory.  Never communicates; jq_set_kernel and jq_comm_set_cooperative do not affect it.
 * Host pointers, blocking. */
int jq_final_state_vjp(jq_handle *h, int32_t nbatch, const double *pcof, int32_t npar, int32_t nsamples,
                       const double *h0_diag_shift, int32_t ncot, const double *cot_r, const double *cot_i,
                       double *vjp, double *state_r, double *state_i);

/* The same vector-Jacobian products on the time-parallel path (kernel 7, DESIGN.md 4.9): the time axis is cut into segments swept
 * concurrently and joined through their propagators, so one cotangent at batch 1 takes about one time-parallel evaluation instead of two
 * serial sweeps.  Kernel 7's stages for its unforced adjoint set, started from lambda_r(T) = -cot_r / 2, lambda_i(T) = cot_i / 2 instead
 * of the objective's terminal adjoint; trajectory (b, s, k) is one kernel-7 trajectory, its propagators computed per cotangent (few
 * trajectories: the call pattern of one optimizer step).  Arguments, layouts and conventions as jq_final_state_vjp; the results agree
 * with it to rounding.
 * ncot = 0: U(T) only (cotangents and vjp ignored; state_r or state_i required), from the state propagators and their join alone.
 * Host pointers, blocking; never communicates (jq_comm_set_cooperative does not apply) and ignores jq_set_kernel; honours
 * jq_set_time_segments (0 = automatic, as for kernel 7).  Afterwards jq_query reports kernel 7, the segments (item 7), the launches
 * (item 2) and the CUDA-event time (item 1).
 * JQ_ERR_ARG (no launch) for ncot < 0, a NULL required array, nbatch*nsamples*max(ncot, 1) > 2^31 - 1, a problem without kernel 7
 * (Jacobi solver, dense weights, uncoupled controls, no tile or fibre layout; the message of jq_set_kernel(h, 7)), or, for ncot >= 1,
 * one whose fibre layout has no segment gradient sweep with the second adjoint set.  JQ_ERR_ALLOC with the size when the segment
 * workspace does not fit on the device. */
int jq_final_state_vjp_time_parallel(jq_handle *h, int32_t nbatch, const double *pcof, int32_t npar, int32_t nsamples,
                                     const double *h0_diag_shift, int32_t ncot, const double *cot_r, const double *cot_i,
                                     double *vjp, double *state_r, double *state_i);

/* Derivatives of the state history of jq_eval_forward, U_j = U(t_j) with t_j after step j*save_every, j = 0 ... nsave - 1,
 * nsave = nsteps/save_every + 1 (U_0 = Uinit does not depend on pcof).  A block is a column-major n x m matrix; Re U_j = vr,
 * Im U_j = -vi as in jq_eval_forward.  Both entries use host pointers, block until done, never communicate, and are not affected by
 * jq_set_kernel or jq_comm_set_cooperative.  pcof, h0_diag_shift as in jq_traceobjgrad_batch, with t = b*nsamples + s.
 * JQ_ERR_ARG (no launch) for save_every < 1 or nsteps % save_every != 0 (the message of jq_eval_forward), ncot / ndir < 1, a NULL
 * required array, more than 2^31 - 1 trajectories, or a problem whose trajectory does not fit in 227 KB of shared memory.
 * Histories are large: one history of nsave blocks is 16 * nsave * n * m bytes (the cnot3 example, 64 x 4 with 31325 steps, at
 * save_every = 1: 128 MB per trajectory and cotangent or direction), and every cotangent and tangent history of a call sits on the
 * device at once; a request the device cannot hold returns JQ_ERR_ALLOC.
 *
 * jq_history_vjp: reverse mode, vjp[p] = sum_j sum_e cot_r[j,e] dRe U_j[e]/dpcof[p] + cot_i[j,e] dIm U_j[e]/dpcof[p], i.e. dL/dpcof of
 * L = sum_j Re vdot(c_j, U_j), one forward and one backward sweep per cotangent whatever npar and nsave are.  One launch of the VJP
 * kernel of jq_final_state_vjp (jq_query(h, 0) = 9): its adjoint sweep starts from the last block as in jq_final_state_vjp, and the
 * cotangent of every earlier saved state jumps into the adjoint when the backward sweep reaches that state (block 0 has no effect).
 * cot_r, cot_i: [(t*ncot + k)][nsave][n*m]; NULL means zero, not both.  vjp: [(t*ncot + k)][npar] (pFidType 3: the phase entry is 0).
 * hist_r, hist_i: [t][nsave][n*m], the states the forward sweep saved (bit-identical to jq_eval_forward on kernel 1), or NULL.
 * With nsave blocks of which only the last is nonzero the result is jq_final_state_vjp's, bit for bit. */
int jq_history_vjp(jq_handle *h, int32_t nbatch, const double *pcof, int32_t npar, int32_t nsamples,
                   const double *h0_diag_shift, int32_t save_every, int32_t ncot, const double *cot_r, const double *cot_i,
                   double *vjp, double *hist_r, double *hist_i);

/* jq_history_vjp_time_parallel: jq_history_vjp on the time-parallel path (kernel 7), the latency route for one or a few trajectories
 * (a path-dependent loss inside an optimizer loop).  Arguments, layouts and conventions as jq_history_vjp; the results agree with it to
 * rounding, and a cotangent history that is nonzero only in its last block gives jq_final_state_vjp_time_parallel's vjp bit for bit at
 * the same segments.  The cotangent of a save jumps into the segment that recomputes it (DESIGN.md §4.10), so the call costs about one
 * final-state VJP on kernel 7 whatever nsave is.  ncot = 0: the history only (cotangents and vjp ignored; hist_r or hist_i required).
 * Semantics and restrictions as jq_final_state_vjp_time_parallel: host pointers, blocking, never communicates, ignores jq_set_kernel,
 * honours jq_set_time_segments; afterwards jq_query reports kernel 7, the segments, the launches and the event time.  JQ_ERR_ARG (no
 * launch) for the rejections of both entries (save_every, ncot < 0, NULL required arrays, trajectories, no kernel 7, for ncot >= 1 no
 * segment gradient sweep with the second adjoint set) and for a layout without segment sweeps carrying the history paths; JQ_ERR_ALLOC
 * with the size when the workspace and histories do not fit. */
int jq_history_vjp_time_parallel(jq_handle *h, int32_t nbatch, const double *pcof, int32_t npar, int32_t nsamples,
                                 const double *h0_diag_shift, int32_t save_every, int32_t ncot, const double *cot_r,
                                 const double *cot_i, double *vjp, double *hist_r, double *hist_i);

/* jq_history_jvp: forward mode, the tangent dU_j . d of every saved state along ndir directions per candidate.  One launch of the
 * forward-sensitivity kernel (jq_query(h, 0) = 8); dirs as in jq_forward_sensitivity.  dhist_r, dhist_i: [(t*ndir + k)][nsave][n*m],
 * the tangents of Re and Im of U_j (block 0 is zero; block nsave - 1 is jq_forward_sensitivity's dstate, bit for bit).  The Jacobi
 * solver has no tangent sweep: JQ_ERR_ARG. */
int jq_history_jvp(jq_handle *h, int32_t nbatch, const double *pcof, int32_t npar, int32_t nsamples,
                   const double *h0_diag_shift, int32_t save_every, int32_t ndir, const double *dirs,
                   double *dhist_r, double *dhist_i);

/* evalctrl(params, pcof, td, func) (src/plotstatectrl.jl:246-276): the control functions p_q(t), q_q(t) (rad/ns) of EVERY
 * coupled control q on the time grid `times`, evaluated by the device function the time loop uses (bcarrier2,
 * src/bsplines.jl:211-304).  p, q: [ncoupled][ntimes] doubles, host pointers, blocking. */
int jq_eval_controls(jq_handle *h, const double *pcof, int32_t npar, int32_t ntimes, const double *times, double *p, double *q);

/* Multi-GPU (one process and one handle per GPU).  The path's only exchange step is the weighted sum over noise
 * samples of eval_f_g_grad! (src/ipopt_interface.jl:48-59) when the samples are sharded across GPUs.
 * jq_comm_unique_id fills a 128-byte NCCL unique id on one rank (distribute it with whatever the host has);
 * jq_comm_init joins the communicator.  Afterwards every jq_traceobjgrad_batch[_device] call WITH weights ends with one
 * grouped ncclAllReduce(sum, double) of the weighted outputs, so each rank passes its own shard of
 * (h0_diag_shift, weights) and every rank receives the full risk-neutral objective and gradients.  Calls without
 * weights (independent candidates / per-sample outputs) never communicate.  NCCL is loaded with dlopen("libnccl.so.2")
 * at jq_comm_unique_id / jq_comm_init time; the library has no link-time NCCL dependency. */
int jq_comm_unique_id(void *id128);
int jq_comm_init(jq_handle *h, int32_t rank, int32_t nranks, const void *id128);
int jq_comm_destroy(jq_handle *h);
/* Cooperative evaluation (on = 1; needs a communicator): every rank passes IDENTICAL arguments and the ranks share out ONE evaluation --
 * the time segments of the time-parallel path (kernel 7): rank r sweeps the propagators of its nseg / nranks segments, one in-place
 * ncclAllGather per propagator array completes them everywhere, the rest is replicated, and every rank returns the same bits as a
 * single GPU would.  Pays when the propagator launch dominates (cnot3: 4.1 of 5.9 ms on one GPU); launches that do not take kernel 7
 * are simply evaluated by every rank.  Sample-sharded calls (weights given) are not affected. */
int jq_comm_set_cooperative(jq_handle *h, int32_t on);

/* Kernel selection, for tests and profiling: 0 = automatic, 1 = generic (any operators, dense weights, uncoupled controls),
 * 2 = register-resident kernel, slot layout (sparse rows with <= 2 entries per row and control), 3 = fibre layout (Kronecker
 * ladder structure), 4 = tile layout (all subsystems with 4 levels: mirrored half-tiles, shuffle-only exchange), 5 = the tile
 * layout with the fewest elements per lane and pipelined state / adjoint / gradient roles (latency layout; also the single-qudit
 * shapes).  Automatic: launches of very few trajectories of at least 256 steps take 7 (below); launches that fit one latency CTA per SM
 * take 5 (then 3 for three subsystems); otherwise 4, 3, 2, 1 in that order, each handing over when it has no instantiation for the problem.
 * 6 = dense-operator kernel on the FP64 tensor-core path (mma.sync f64; unstructured operators, the noise samples of a candidate
 * batched as columns of one contraction); automatic mode takes it when no register-resident layout applies, n >= 8 and the
 * operators are at least 20% filled.
 * 7 = time-parallel evaluation for launches of very few trajectories (the reference's own call pattern: one pcof per Ipopt
 * callback): the time axis is cut into segments that are swept concurrently by the layout-3/4 steppers and joined through the
 * segments' discrete propagators (every step of the scheme is linear in the state and affine in the adjoint); same results to
 * rounding (~1e-14 relative), critical path ~ 4 nsteps / nseg steps.  Neumann solver, diagonal weights, tile / fibre layouts.
 * 2 ... 7 fail with JQ_ERR_ARG if the problem has no instantiation. */
int jq_set_kernel(jq_handle *h, int32_t kernel);
/* Number of time segments of kernel 7; 0 = automatic (about sqrt(1.6 nsteps), whole waves of the propagator launch). */
int jq_set_time_segments(jq_handle *h, int32_t nseg);
/* Host-only helper (no device needed): the times at which kernel 7 starts the sweeps of its nseg segments.  Segment p covers the steps
 * [p nsteps / nseg, (p + 1) nsteps / nseg); t_first[p] is the value the reference's forward recurrence t = t + dt from 0
 * (src/evalobjgrad.jl:745) has at the segment's first step, t_last[p] the value its backward recurrence t = t - dt from T (:810, :919)
 * has at the segment's last step -- bit-identical to what a single sweep sees, not k dt.  Returns the steps of the longest segment. */
int64_t jq_time_segments(double T, int64_t nsteps, int32_t nseg, double *t_first, double *t_last);
/* what: 0 = kernel actually used by the last evaluation (1 ... 7, 8 = the forward-sensitivity kernel of jq_forward_sensitivity and
 * jq_history_jvp, or 9 = the VJP kernel of jq_final_state_vjp and jq_history_vjp; 7 after jq_final_state_vjp_time_parallel and
 * jq_history_vjp_time_parallel),
 * 1 = CUDA-event time of the last evaluation's trajectory kernel(s) in ms (synchronises), 2 = number of kernels launched by the last
 * evaluation,
 * 3 = trajectories resident per CTA, 4 = CTAs launched, 5 = registers per thread, 6 = dynamic smem bytes per CTA,
 * 7 = time segments of the last evaluation (kernel 7; else 0). */
int jq_query(jq_handle *h, int32_t what, double *value);

/* Measured FP64 FMA throughput of `device` in TFLOP/s (8 independent DFMA chains per thread on every SM, best of
 * 5 CUDA-event timed launches) — the roofline denominator for this path; MEASURED_PEAKS.json has no FP64 entry. */
int jq_fp64_peak(int device, double *tflops);
/* Same with three distinct, changing register operands per DFMA (no operand-reuse hits): on B200 the register file then
 * sustains one warp-DFMA per 3 cycles per scheduler instead of 2, i.e. 2/3 of the figure above — the realistic ceiling for
 * FMAs that are not coefficient-broadcast shaped.  Reported next to the roofline, not used as its denominator. */
int jq_fp64_peak_3op(int device, double *tflops);
/* FP64 tensor-core (DMMA, mma.sync m16n8k16) peak of `device` in TFLOP/s; reported next to the roofline, the path
 * itself does not use the tensor pipe (see DESIGN.md). */
int jq_fp64_peak_dmma(int device, double *tflops);

const char *jq_last_error(void);
const char *jq_version(void);

#ifdef __cplusplus
}
#endif
#endif /* JUQBOX_B200_H */
