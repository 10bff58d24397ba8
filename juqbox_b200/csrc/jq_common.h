// Internal declarations shared by the C-ABI layer (jq_api.cu) and the kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include <stdio.h>

#define JQ_MAX_CTRL 8

// Problem data as the kernels see it (device pointers).  Operators are row-wise CSR, one per
// o in {0: Hconst (diagonal included even if zero), 1..Nc: Hsym_q, Nc+1..2Nc: Hanti_q}.
struct DevProblem {
    int n, m, Nc, Nfreq, J, objFuncType;
    int solver;            // 1 Neumann (J terms), 2 Jacobi (at most J sweeps, stop at ||dX||_F < tol)
    double tol;
    long long nsteps;
    double T;
    const double *uinit, *vtr, *vti, *wdiag, *cfreq;  // n*m, n*m, n*m, n, Nc*Nfreq
    const int *rowptr;     // (1+2Nc)*(n+1), positions absolute into col/val
    const int *col;
    const double *val;
    const int *h0diag;     // n: position of H0[i,i] inside col/val (always present)
    // the same table as ONE 16-byte aligned blob [rowptr | col | pad | val] (byte offsets below), the source of the generic
    // kernel's TMA bulk copy into shared memory; csr_bytes is a multiple of 16
    const void *csr_blob;
    int csr_bytes, csr_off_col, csr_off_val;
    const double *dense_ops;   // the same operators as dense row-major matrices [H0, Hsym.., Hanti..], zero padded to n8 x ldk each
                               // (jq_dense_padding; n <= 64, else nullptr): the dense kernel's MMA A operands
    // --- SURVEY 8f rank 3 ---
    int pFidType;          // 1, 2, 3 or 4 (src/evalobjgrad.jl:755-763); 3: the global phase is the last entry of every pcof vector
    double globalPhase;    // params.globalPhase (pFidType 1 and 4)
    const double *wreal, *wimag;   // dense n x n column-major weights (custom forbidden states) or nullptr -> Diagonal(wdiag)
    // Controls 0..Nc-1 are uniform for the kernels: (Hsym_q, Hanti_q, p_q(t), q_q(t)).  An UNCOUPLED control (KS!, :2372-2387) is
    // entered as kind 1 (symmetric Hunc: Hsym = Hunc, Hanti = 0, p = f, q = 0) or kind 2 (antisymmetric: Hanti = Hunc, q = f),
    // with f(t) = 2 (p_spline cos(2 pi rfreq t) - q_spline sin(2 pi rfreq t)); kind 0 = coupled.
    int ctrl_kind[JQ_MAX_CTRL];
    double ctrl_rfreq[JQ_MAX_CTRL];
    int any_unc;
};

// Time-parallel evaluation (jq_seg.cu): the time axis is cut into nseg segments, every segment is swept by its own sub-trajectories
// and the segments are joined through the discrete propagators (the one-step maps are linear in the state / the adjoint).
// What the CTAs of one trajectory-kernel launch do: CTAs [0, ctas0) run mode[0], the others mode[1] (0 = none)
//   1 forward sweep of a block of m unit vectors of R^2n           -> Phi   (state propagator of the segment, column by column)
//   2 forward sweep of the true state from X[seg]                  -> penpart (the segment's share of the guard-level penalty)
//   3 adjoint sweep without forcing from a block of unit vectors   -> Adj   (homogeneous adjoint propagator)
//   4 backward sweep (state from Xb[seg+1], zero terminal adjoint) -> cpart (particular adjoint solution at the segment start)
//   5 backward sweep (state from Xb[seg+1], adjoint from Lam[seg+1]) -> gpart (the segment's share of the gradient)
//   6 backward state sweep of the true state from X[seg+1]         -> dpart = J (state reached - X[seg]), J (u; v) = (v; -u): the
//     defect of the backward recomputation, from which the join builds Xb = X + J' Eta, the states the reference's backward sweep
//     sees (its time recurrence from T is shifted against the forward one by the rounding of nsteps additions, ~1e-10)
// Layouts: Phi, Adj [seg][traj][ld (unit vector j)][ld (u rows, then v rows)]; X, Lam, Eta, cpart, dpart [seg][traj][m (column)][2n
// (u rows, then v rows)] (X, Lam, Eta have nseg + 1 boundary entries); gpart [seg][traj][Npar]; penpart [seg][traj].
struct SegArgs {
    int nseg;              // 0: whole trajectories (the plain evaluation)
    int mode[2], ctas0;
    int seg_lo, seg_cnt;   // this launch sweeps the segments [seg_lo, seg_lo + seg_cnt) only (seg_cnt = 0: all) -- segments sharded over GPUs
    int ld;                // leading dimension of Phi / Adj: [seg][traj][ld][ld], zero padded past 2n (jq_seg_ld)
    double *Phi, *Adj, *X, *Lam, *Eta, *cpart, *dpart, *gpart, *penpart;
    double *Lam2, *gpart2; // objFuncType 2/3: boundary values of the second adjoint set (no forcing: Lam2_p = Adj_p Lam2_{p+1}), its gradient shares
    int pass;              // mode 6: 0 = defect against the forward boundary states; r > 0 = refinement against X + J' Eta (runs only if flags[r - 1])
    int *flags;            // [4]: flags[r] = 1 when pass r left a defect entry above refine_tol
    double refine_tol;
    const double *times;   // [2][nseg]: time at the first step of segment p in the reference's forward recurrence t = t + dt from 0, and at
                           // its last step in the backward recurrence t = t - dt from T (jq_seg_times): the sweeps see bit-identical times
};

// Per-launch arguments common to both kernels.
struct LaunchArgs {
    int ntraj, nsamples, Npar, D1, evaladjoint;
    int pstride, gstride;  // row stride of pcof and of grad / infidgrad: Npar, or Npar + 1 when the global phase rides along (pFidType 3)
    const double *pcof;    // [nbatch][pstride]
    const double *shift;   // [nsamples][n] or nullptr
    double *scal;          // [ntraj][4]: infid, leak, trace_infid, spare
    double *grad;          // [ntraj][gstride] total gradient
    double *infidgrad;     // [ntraj][gstride] (objFuncType != 1) or nullptr
    // forward-history output (generic kernel only): state after every save_every-th step, [ntraj][nsave][n*m]
    double *hist_r, *hist_i;   // Re(psi) = vr, Im(psi) = -vi  (src/evalobjgrad.jl:679-680,750-751)
    int save_every;
    long long nsave;
    SegArgs seg;           // register-resident kernels only
};

// ---- generic kernel (jq_generic.cu): one CTA per trajectory, blocks in shared memory ----
size_t jq_generic_smem_bytes(const DevProblem &P, int Npar);
cudaError_t jq_generic_launch(const DevProblem &P, const LaunchArgs &A, cudaStream_t st, int *nctas, int *regs, size_t *smem);
cudaError_t jq_controls_launch(const DevProblem &P, int D1, const double *pcof, int ntimes, const double *times, double *p, double *q,
                               cudaStream_t st);

// ---- forward-sensitivity kernel (jq_generic.cu): the forward sweep and its tangent along one direction per trajectory, generic layout ----
struct SensArgs {
    int ntraj, nsamples, ndir, Npar, D1;   // ntraj = nbatch * nsamples * ndir; Npar: spline coefficients (without the pFidType 3 phase)
    int pstride;           // length of every pcof and direction vector: Npar, or Npar + 1 with the global phase (pFidType 3)
    const double *pcof;    // [nbatch][pstride]
    const double *dirs;    // [nbatch][ndir][pstride]
    const double *shift;   // [nsamples][n] or nullptr
    double *scal;          // [nbatch * nsamples][4]: infid, leak, trace_infid, spare (written by direction 0)
    double *dinfid, *dleak;            // [ntraj]: traj = (b * nsamples + s) * ndir + k
    double *dstate_r, *dstate_i;       // [ntraj][n*m] tangents of Re and Im of the final state (vr', -vi'), or nullptr
};
size_t jq_fwdsens_smem_bytes(const DevProblem &P, int Npar);     // one group
cudaError_t jq_fwdsens_launch(const DevProblem &P, const SensArgs &S, cudaStream_t st, int *nctas, int *regs, size_t *smem, int *gpc);

// ---- dense-operator kernel on the FP64 tensor-core path (jq_dense.cu): one CTA per (candidate, tile of samples) ----
bool jq_dense_supported(const DevProblem &P, char *why, size_t len);
void jq_dense_padding(int n, int *n8, int *ldk);      // layout of DevProblem::dense_ops: [1 + 2 Nc][n8][ldk], zero padded
cudaError_t jq_dense_launch(const DevProblem &P, const LaunchArgs &A, cudaStream_t st, int *nctas, int *regs, size_t *smem, int *traj_per_cta);

// Host copy of the operators in row-wise form, used by the planners.
struct HostOps {
    int n, m, Nc, Nfreq;
    const int *rowptr;
    const int *col;
    const double *val;
};

// ---- register-resident trajectory kernels (jq_traj.cu): slot layout (kind 2) and fibre layout (kind 3) ----
struct TrajPlan;   // opaque, built at jq_create; nullptr + reason when the problem shape has no instantiation
TrajPlan *jq_slot_plan_create(const DevProblem &Pdev, const HostOps &H, const double *wdiag_host, char *err, size_t errlen);
TrajPlan *jq_fiber_plan_create(const DevProblem &Pdev, const HostOps &H, const double *wdiag_host, char *err, size_t errlen, int pipe = 0);
TrajPlan *jq_tile_plan_create(const DevProblem &Pdev, const HostOps &H, const double *wdiag_host, int NT, char *err, size_t errlen, int pipe = 0);
void jq_traj_plan_destroy(TrajPlan *);
int jq_traj_plan_kind(const TrajPlan *);
int jq_traj_plan_tpc(const TrajPlan *);      // trajectories per CTA
int jq_traj_plan_lanes(const TrajPlan *);    // lanes per trajectory
cudaError_t jq_traj_launch(TrajPlan *plan, const DevProblem &P, const LaunchArgs &A, cudaStream_t st, int *nctas, int *regs,
                           size_t *smem, int *traj_per_cta);

// ---- time-parallel evaluation (jq_seg.cu): segment sweeps on a trajectory plan, joined through the segment propagators ----
bool jq_seg_supported(const TrajPlan *plan, const DevProblem &P, bool second_adjoint = false);      // the plan has segment-sweep instantiations
int jq_seg_ld(const DevProblem &P);
int jq_seg_auto_segments(const DevProblem &P, int ntraj, int evaladjoint, int tpc, int sms);
size_t jq_seg_workspace_doubles(const DevProblem &P, int ntraj, int Npar, int nseg, int evaladjoint);
void jq_seg_times(const DevProblem &P, int nseg, double *times /* [2][nseg], host */);
// plan_prop: plan of the propagator launch (many independent sweeps: a throughput layout pays), plan: the boundary-to-boundary sweeps
// plan_obj: plan of the gradient sweep when objFuncType != 1 (second adjoint set; nullptr otherwise)
// coop: several GPUs evaluate the SAME trajectories together (nullptr: one GPU).  The propagator launch is independent per segment and
// dominates large problems: rank r sweeps its nseg / nranks segments, then `allgather` (in place, count doubles per rank, on the stream)
// completes Phi and Adj on every rank; everything after that is replicated, so all ranks return bit-identical results.
struct SegCoop {
    int rank, nranks;
    int (*allgather)(void *ctx, double *buf, size_t count_per_rank, cudaStream_t st);
    void *ctx;
};
cudaError_t jq_seg_launch(TrajPlan *plan_prop, TrajPlan *plan, TrajPlan *plan_obj, const DevProblem &P, const LaunchArgs &A, int nseg, const double *times, int *flags /* 4 ints, device */, double *work, cudaStream_t st, const SegCoop *coop,
                          int *nctas, int *regs, size_t *smem, int *traj_per_cta, int *nlaunch);
