// Generic trajectory kernel: one CTA per trajectory, all n x m blocks in shared memory, operators as CSR rows
// read through L1/L2.  Handles any operator sparsity (dense input is just CSR with full rows), any n*m that fits in
// shared memory, and objFuncType 1/2/3.  It is the fallback for shapes the register-resident kernels (jq_traj.cu) have
// no instantiation for, their independent cross-check in the tests, and the kernel behind jq_eval_forward (state history).  The whole forward + backward time loop runs
// inside the kernel; HBM is touched only for the launch inputs and the final outputs.
//
// Algorithm (reference lines): forward loop src/evalobjgrad.jl:698-753, infidelity :755-766, adjoint terminal
// condition :810-844 / :2026-2042, backward loop :859-921, steppers src/StormerVerlet.jl:255-303,:365-406,:461-504,
// Neumann src/linear_solvers.jl:94-106, controls src/bsplines.jl:211-304,:321-381, gradient :2567-2619.
// K(t) and S(t) are never assembled: K(t)x = H0 x + sum_q p_q(t) Hsym_q x,  S(t)x = sum_q q_q(t) Hanti_q x.
//
// Work decomposition: a GROUP of TPT threads (32, 64, 128 or 256: the smallest that covers n*m, one element per thread where
// possible) owns one trajectory; a CTA of GEN_THREADS threads runs GEN_THREADS / TPT groups side by side, each looping over its
// own trajectories and synchronising only with itself (__syncwarp for one-warp groups, a named barrier per group otherwise).
// Operators: the whole row-wise CSR table (row pointers, columns, values of Hconst, Hsym_q, Hanti_q) is staged into shared
// memory ONCE per CTA with a 1-D TMA bulk copy (cp.async.bulk.shared::cluster.global + mbarrier complete_tx) when it fits next to
// the state blocks; otherwise the products read it through L1.
#include "jq_common.h"

#define GEN_THREADS 256

// Geometry of one launch (host-computed): threads per group, groups per CTA, doubles of shared memory per group, and whether
// the operator table is staged into shared memory.
struct GenGeom { int tpt, gpc, per_group, stage; };

namespace {

__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }

struct Ctx {
    const DevProblem *P;
    int gtid, tpt, bar, gwarps;          // thread in group, threads per group, named-barrier id of the group, warps per group
    const int *rp, *cl;                  // row pointers / columns / values of the operator table: shared memory or global
    const double *vl;
    int n, m, len, Nc, Nfreq, D1, Npar, J;
    double *vr, *vi, *vi05, *vr0;
    double *lr, *li, *lr05, *li0;
    double *lrn, *lin, *lr05n, *li0n;
    double *rhs, *scr, *k1, *k2, *l1, *l2;
    double *pcof, *grad, *igrad, *ctrl, *shift, *red;
    double dtknot, tinv;
};

// Dense forbidden-state weights (src/evalobjgrad.jl:214-232): (W x)[i, j] for a column-major n x n W read through L1.
__device__ __forceinline__ double wapply(const Ctx &c, const double *W, const double *x, int i, int j) {
    const double *xc = x + j * c.n;
    double s = 0.0;
    for (int k = 0; k < c.n; ++k) s += W[i + (size_t)k * c.n] * xc[k];
    return s;
}
// (wmat_real x)[i, j] for either form of the weights
__device__ __forceinline__ double wreal_apply(const Ctx &c, const double *x, int e, int i, int j) {
    return c.P->wreal ? wapply(c, c.P->wreal, x, i, j) : c.P->wdiag[i] * x[e];
}

// all threads of the group (the trajectory's n x m blocks live in the group's shared memory)
__device__ __forceinline__ void gsync(const Ctx &c) {
    if (c.tpt == 32) __syncwarp();
    else asm volatile("bar.sync %0, %1;" ::"r"(c.bar), "r"(c.tpt) : "memory");
}
__device__ __forceinline__ double op_apply(const Ctx &c, int o, const double *x, int i, int j) {
    const int *rp = c.rp + o * (c.n + 1);
    const double *xc = x + j * c.n;
    double s = 0.0;
    for (int p = rp[i]; p < rp[i + 1]; ++p) s += c.vl[p] * xc[c.cl[p]];
    return s;
}
// Tangents of the forward sweep along one direction d (forward-sensitivity kernel): the tangent of every state block the step
// touches, and the control tables differentiated along d (ctrl_dot = the same table with d in place of pcof: p, q and the
// uncoupled f are linear in pcof).
struct Tan {
    double *vr, *vi, *vi05, *vr0, *rhs, *scr, *k1, *k2, *l1, *l2;
    double *ctrl;
};
// a tangent block when the tangent is carried, nullptr otherwise (td is only dereferenced with TAN)
#define TD(f) (TAN ? td->f : nullptr)

// K(t) x.  TAN: also *yd = (K x)' = K xd + sum_q p_q' Hsym_q x, one product of Hsym_q x feeding both sums.
template <bool TAN = false>
__device__ __forceinline__ double applyK(const Ctx &c, int level, const double *x, int i, int j, const Tan *td = nullptr,
                                         const double *xd = nullptr, double *yd = nullptr) {
    double s = op_apply(c, 0, x, i, j) + c.shift[i] * x[i + j * c.n];
    const double *ct = c.ctrl + level * 2 * c.Nc;
    double sd = 0.0;
    if constexpr (TAN) sd = op_apply(c, 0, xd, i, j) + c.shift[i] * xd[i + j * c.n];
    for (int q = 0; q < c.Nc; ++q) {
        const double hx = op_apply(c, 1 + q, x, i, j);
        s += ct[2 * q] * hx;
        if constexpr (TAN) sd += ct[2 * q] * op_apply(c, 1 + q, xd, i, j) + td->ctrl[level * 2 * c.Nc + 2 * q] * hx;
    }
    if constexpr (TAN) *yd = sd;
    return s;
}
// S(t) x.  TAN: also *yd = (S x)' = S xd + sum_q q_q' Hanti_q x.
template <bool TAN = false>
__device__ __forceinline__ double applyS(const Ctx &c, int level, const double *x, int i, int j, const Tan *td = nullptr,
                                         const double *xd = nullptr, double *yd = nullptr) {
    const double *ct = c.ctrl + level * 2 * c.Nc;
    double s = 0.0, sd = 0.0;
    for (int q = 0; q < c.Nc; ++q) {
        const double hx = op_apply(c, 1 + c.Nc + q, x, i, j);
        s += ct[2 * q + 1] * hx;
        if constexpr (TAN) sd += ct[2 * q + 1] * op_apply(c, 1 + c.Nc + q, xd, i, j) + td->ctrl[level * 2 * c.Nc + 2 * q + 1] * hx;
    }
    if constexpr (TAN) *yd = sd;
    return s;
}

// src/bsplines.jl:211-304 (0-based indices)
__device__ double bcarrier2(const Ctx &c, double t, int func) {
    const int osc = func >> 1, qf = func & 1;
    const double width = 3.0 * c.dtknot;
    long long k = (long long)ceil(t / c.dtknot + 2.0);
    k = k < 3 ? 3 : (k > c.D1 ? c.D1 : k);
    double f = 0.0;
    for (int fr = 0; fr < c.Nfreq; ++fr) {
        const int off1 = 2 * osc * c.Nfreq * c.D1 + fr * 2 * c.D1 - 1, off2 = off1 + c.D1;
        double fbs1 = 0.0, fbs2 = 0.0;
        double tau = (t - c.dtknot * ((double)k - 1.5)) / width;
        double b = 9.0 / 8 + 4.5 * tau + 4.5 * tau * tau;
        fbs1 += c.pcof[off1 + k] * b;
        fbs2 += c.pcof[off2 + k] * b;
        tau = (t - c.dtknot * ((double)(k - 1) - 1.5)) / width;
        b = 0.75 - 9.0 * tau * tau;
        fbs1 += c.pcof[off1 + k - 1] * b;
        fbs2 += c.pcof[off2 + k - 1] * b;
        tau = (t - c.dtknot * ((double)(k - 2) - 1.5)) / width;
        b = 9.0 / 8 - 4.5 * tau + 4.5 * tau * tau;
        fbs1 += c.pcof[off1 + k - 2] * b;
        fbs2 += c.pcof[off2 + k - 2] * b;
        double sn, cs;
        sincos(c.P->cfreq[osc + c.Nc * fr] * t, &sn, &cs);
        f += qf ? fbs1 * sn + fbs2 * cs : fbs1 * cs - fbs2 * sn;
    }
    return f;
}

__device__ void eval_controls(const Ctx &c, double t, double dt) {
    const int nf = 2 * c.Nc;
    for (int idx = c.gtid; idx < 3 * nf; idx += c.tpt) {
        const int level = idx / nf, func = idx % nf;
        const double tt = level == 0 ? t : (level == 1 ? t + 0.5 * dt : t + dt);
        const int kind = c.P->ctrl_kind[func >> 1];
        if (kind == 0) {
            c.ctrl[idx] = bcarrier2(c, tt, func);
        } else {                               // uncoupled control (KS!, src/evalobjgrad.jl:2372-2387): f = 2 (p cos - q sin) goes to K or to S
            double v = 0.0;
            if ((func & 1) == (kind == 2)) {
                double sr, cr;
                sincos(2.0 * M_PI * c.P->ctrl_rfreq[func >> 1] * tt, &sr, &cr);
                v = 2.0 * (bcarrier2(c, tt, func & ~1) * cr - bcarrier2(c, tt, func | 1) * sr);
            }
            c.ctrl[idx] = v;
        }
    }
    gsync(c);
}

// element loop of the group: e = gtid, gtid + tpt, ...; (i, j) = (row, column) advanced without divisions
#define FOR_E for (int e = c.gtid, i = c.gtid % c.n, j = c.gtid / c.n, di_ = c.tpt % c.n, dj_ = c.tpt / c.n; e < c.len; \
                   e += c.tpt, i += di_, j += dj_ + (i >= c.n ? 1 : 0), i -= (i >= c.n ? c.n : 0))

// X = sum_{j<=J} (h/2)^j S^j B ; B destroyed, T scratch (src/linear_solvers.jl:94-106)
// TAN: the tangent alongside, Td_j = S Td_{j-1} + S' T_{j-1}, Xd += (h/2)^j Td_j; Bd destroyed, Td scratch.
template <bool TAN = false>
__device__ void neumann(const Ctx &c, int level, double h, double *B, double *T, double *X, const Tan *td = nullptr,
                        double *Bd = nullptr, double *Td = nullptr, double *Xd = nullptr) {
    FOR_E { X[e] = B[e]; if constexpr (TAN) Xd[e] = Bd[e]; }
    double coeff = 1.0;
    for (int it = 0; it < c.J; ++it) {
        coeff *= 0.5 * h;
        FOR_E {
            double yd;
            double tv = applyS<TAN>(c, level, B, i, j, td, Bd, &yd); T[e] = tv; X[e] += coeff * tv;
            if constexpr (TAN) { Td[e] = yd; Xd[e] += coeff * yd; }
        }
        gsync(c);
        double *sw = B; B = T; T = sw;
        if constexpr (TAN) { sw = Bd; Bd = Td; Td = sw; }
    }
}

// Jacobi sweeps (src/linear_solvers.jl:110-152): X = B; T = B + (h/2) S X; err = ||T - X||_F; X = T; stop when
// err < tol or after J sweeps.  B is preserved, the result is left in X.  The reference multiplies S by -h/2 in place
// and computes B - (scaled S) X; the sign and factor are folded here (differences are rounding-level only).
__device__ void block_sum(const Ctx &c, double *v, int cnt);
__device__ void jacobi(const Ctx &c, int level, double h, const double *B, double *T, double *X) {
    FOR_E X[e] = B[e];
    gsync(c);
    for (int it = 0; it < c.J; ++it) {
        double err[1] = {0.0};
        FOR_E { double tv = B[e] + 0.5 * h * applyS(c, level, X, i, j); double d = tv - X[e]; err[0] += d * d; T[e] = tv; }
        block_sum(c, err, 1);                 // also orders the T writes before the copy below
        FOR_E X[e] = T[e];
        gsync(c);
        if (sqrt(err[0]) < c.P->tol) break;   // uniform across the CTA: block_sum broadcasts
    }
}

// TAN: Neumann only (the Jacobi solver has no tangent; the host rejects it for the forward-sensitivity kernel)
template <bool TAN = false>
__device__ __forceinline__ void solve(const Ctx &c, int level, double h, double *B, double *T, double *X, const Tan *td = nullptr,
                                      double *Bd = nullptr, double *Td = nullptr, double *Xd = nullptr) {
    if constexpr (TAN) neumann<true>(c, level, h, B, T, X, td, Bd, Td, Xd);
    else if (c.P->solver == 2) jacobi(c, level, h, B, T, X);
    else neumann(c, level, h, B, T, X);
}

// src/StormerVerlet.jl:461-504.  TAN: every statement differentiated along d as well (step_fwdGrad!, src/StormerVerlet.jl:151-251).
template <bool TAN = false>
__device__ void state_step(const Ctx &c, double h, const Tan *td = nullptr) {
    double *u = c.vr, *v = c.vi, *v05 = c.vi05;
    FOR_E {
        double kd, sd;
        c.rhs[e] = applyK<TAN>(c, 1, u, i, j, td, TD(vr), &kd) + applyS<TAN>(c, 1, v, i, j, td, TD(vi), &sd);
        if constexpr (TAN) td->rhs[e] = kd + sd;
    }
    gsync(c);
    solve<TAN>(c, 1, h, c.rhs, c.scr, c.l1, td, TD(rhs), TD(scr), TD(l1));
    FOR_E { v05[e] = v[e] + 0.5 * h * c.l1[e]; if constexpr (TAN) td->vi05[e] = td->vi[e] + 0.5 * h * td->l1[e]; }
    gsync(c);
    FOR_E {
        double sd, kd;
        c.k1[e] = applyS<TAN>(c, 0, u, i, j, td, TD(vr), &sd) - applyK<TAN>(c, 0, v05, i, j, td, TD(vi05), &kd);
        if constexpr (TAN) td->k1[e] = sd - kd;
    }
    gsync(c);
    FOR_E {
        double ad, bd, kd;
        c.rhs[e] = applyS<TAN>(c, 2, u, i, j, td, TD(vr), &ad) + 0.5 * h * applyS<TAN>(c, 2, c.k1, i, j, td, TD(k1), &bd) -
                   applyK<TAN>(c, 2, v05, i, j, td, TD(vi05), &kd);
        if constexpr (TAN) td->rhs[e] = ad + 0.5 * h * bd - kd;
    }
    gsync(c);
    FOR_E { u[e] += 0.5 * h * c.k1[e]; if constexpr (TAN) td->vr[e] += 0.5 * h * td->k1[e]; }
    solve<TAN>(c, 2, h, c.rhs, c.scr, c.k2, td, TD(rhs), TD(scr), TD(k2));
    FOR_E { u[e] += 0.5 * h * c.k2[e]; if constexpr (TAN) td->vr[e] += 0.5 * h * td->k2[e]; }
    gsync(c);
    FOR_E {
        double kd, sd;
        c.l2[e] = applyK<TAN>(c, 1, u, i, j, td, TD(vr), &kd) + applyS<TAN>(c, 1, v05, i, j, td, TD(vi05), &sd);
        v[e] += 0.5 * h * (c.l1[e] + c.l2[e]);
        if constexpr (TAN) { td->l2[e] = kd + sd; td->vi[e] += 0.5 * h * (td->l1[e] + td->l2[e]); }
    }
    gsync(c);
}

// Forbidden-state penalty of one forward step, accumulated per thread into *pen (summed over the group by the caller).
// Before the step: penalf2aTrap(vr) (diagonal W), its dense form (src/evalobjgrad.jl:2210-2223) and the vr0 copy for penalf2imag.
// TAN: the tangent along d into *pd: 2 sum W vr vr' (diagonal), vr'^T W vr + vr^T W vr' (dense).  The tangent runs in its own element
// loop behind a group barrier: sharing products such as W vr with the primal loop lets the compiler contract the primal sum
// differently, and the primal penalty must stay the generic kernel's to the bit.
template <bool TAN = false>
__device__ __forceinline__ void penalty_pre(const Ctx &c, double *pen, const Tan *td = nullptr, double *pd = nullptr) {
    const DevProblem &P = *c.P;
    if (!P.wreal) {
        FOR_E *pen += P.wdiag[i] * c.vr[e] * c.vr[e];
    } else {
        FOR_E { *pen += c.vr[e] * wapply(c, P.wreal, c.vr, i, j); c.vr0[e] = c.vr[e]; }
    }
    if constexpr (TAN) {
        gsync(c);
        if (!P.wreal) {
            FOR_E *pd += 2.0 * P.wdiag[i] * c.vr[e] * td->vr[e];
        } else {
            FOR_E {
                *pd += td->vr[e] * wapply(c, P.wreal, c.vr, i, j) + c.vr[e] * wapply(c, P.wreal, td->vr, i, j);
                td->vr0[e] = td->vr[e];
            }
        }
    }
}
// After the step: penalf2a(vr, vi05) (diagonal W); dense penalf2a (:2183-2197) and -2 penalf2imag(vr0, vi05, wmat_imag) =
// -2 tr(vi05' Wi vr0) (:716-718,:2226-2228).  The caller's next barrier orders the reads of vr0 before its rewrite.
template <bool TAN = false>
__device__ __forceinline__ void penalty_post(const Ctx &c, double *pen, const Tan *td = nullptr, double *pd = nullptr) {
    const DevProblem &P = *c.P;
    if (!P.wreal) {
        FOR_E *pen += P.wdiag[i] * (c.vr[e] * c.vr[e] + 2.0 * c.vi05[e] * c.vi05[e]);
    } else {
        FOR_E {
            *pen += c.vr[e] * wapply(c, P.wreal, c.vr, i, j) + 2.0 * c.vi05[e] * wapply(c, P.wreal, c.vi05, i, j);
            if (P.wimag) *pen -= 2.0 * c.vi05[e] * wapply(c, P.wimag, c.vr0, i, j);
        }
    }
    if constexpr (TAN) {
        gsync(c);
        if (!P.wreal) {
            FOR_E *pd += 2.0 * P.wdiag[i] * (c.vr[e] * td->vr[e] + 2.0 * c.vi05[e] * td->vi05[e]);
        } else {
            FOR_E {
                *pd += td->vr[e] * wapply(c, P.wreal, c.vr, i, j) + c.vr[e] * wapply(c, P.wreal, td->vr, i, j) +
                       2.0 * (td->vi05[e] * wapply(c, P.wreal, c.vi05, i, j) + c.vi05[e] * wapply(c, P.wreal, td->vi05, i, j));
                if (P.wimag)
                    *pd -= 2.0 * (td->vi05[e] * wapply(c, P.wimag, c.vr0, i, j) + c.vi05[e] * wapply(c, P.wimag, td->vr0, i, j));
            }
        }
    }
}

// src/StormerVerlet.jl:255-303 (forcing) / :365-406 (no forcing).  Forcing with diagonal W:
// hr0 = W vr0 / T, hi0 = hi1 = W vi05 / T, hr1 = W vr / T  (src/evalobjgrad.jl:862,882-888).
// General weights (:882-888): hr0 = Wr vr0 / T, hi0 = Wr vi05 / T, hr1 = (Wr vr + Wi vi05) / T, hi1 = hi0 - Wi vr / T.
__device__ void adjoint_step(const Ctx &c, double *mu, double *nu, double *X, double h, bool forcing, double tinv) {
    const double *Wi = c.P->wimag;
    FOR_E {
        double f = forcing ? tinv * wreal_apply(c, c.vr0, e, i, j) : 0.0;
        c.rhs[e] = applyS(c, 0, mu, i, j) - applyK(c, 1, nu, i, j) + f;
    }
    gsync(c);
    solve(c, 0, h, c.rhs, c.scr, c.k2);
    FOR_E { mu[e] += 0.5 * h * c.k2[e]; X[e] = mu[e]; }
    gsync(c);
    FOR_E {
        double f = forcing ? tinv * wreal_apply(c, c.vi05, e, i, j) : 0.0;
        c.l2[e] = applyK(c, 0, X, i, j) + applyS(c, 1, nu, i, j) + f;
    }
    gsync(c);
    FOR_E {
        double f = forcing ? tinv * wreal_apply(c, c.vi05, e, i, j) : 0.0;
        if (forcing && Wi) f -= tinv * wapply(c, Wi, c.vr, i, j);
        c.rhs[e] = applyS(c, 1, nu, i, j) + 0.5 * h * applyS(c, 1, c.l2, i, j) + applyK(c, 2, X, i, j) + f;
    }
    gsync(c);
    solve(c, 1, h, c.rhs, c.scr, c.l1);
    FOR_E nu[e] += 0.5 * h * (c.l2[e] + c.l1[e]);
    gsync(c);
    FOR_E {
        double f = forcing ? tinv * wreal_apply(c, c.vr, e, i, j) : 0.0;
        if (forcing && Wi) f += tinv * wapply(c, Wi, c.vi05, i, j);
        c.k1[e] = applyS(c, 2, X, i, j) - applyK(c, 1, nu, i, j) + f;
    }
    gsync(c);
    FOR_E mu[e] += 0.5 * h * c.k1[e];
    gsync(c);
}

// Sum `cnt` (<= 8) per-thread values over the group; result broadcast to every thread of the group.
__device__ void block_sum(const Ctx &c, double *v, int cnt) {
    const int lane = threadIdx.x & 31, w = c.gtid >> 5;
    for (int k = 0; k < cnt; ++k) {
        double x = v[k];
        for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
        if (c.gwarps == 1) v[k] = x;
        else if (lane == 0) c.red[w * 8 + k] = x;
    }
    if (c.gwarps == 1) return;
    gsync(c);
    for (int k = 0; k < cnt; ++k) {
        double x = 0.0;
        for (int ww = 0; ww < c.gwarps; ++ww) x += c.red[ww * 8 + k];
        v[k] = x;
    }
    gsync(c);
}

// One step's contribution to the gradient (src/evalobjgrad.jl:2567-2619), scaled by dt at the end of the sweep.
// tr(A,H,C) := sum_ij A_ij (H C)_ij.
__device__ void grad_step(const Ctx &c, const double *lr05, const double *li, const double *li0, double t0, double dt,
                          double *g) {
    for (int q = 0; q < c.Nc; ++q) {
        double T[5] = {0, 0, 0, 0, 0};
        const int os = 1 + q, oa = 1 + c.Nc + q;
        FOR_E {
            const double aX = op_apply(c, oa, lr05, i, j), sX = op_apply(c, os, lr05, i, j);
            T[0] += c.vr0[e] * aX;                                                              // tr(vr0, Ha, lr05)
            T[1] += c.vi05[e] * sX;                                                             // tr(vi05, Hs, lr05)
            T[2] += c.vr[e] * aX;                                                               // tr(vr, Ha, lr05)
            T[3] += c.vr[e] * op_apply(c, os, li, i, j) + c.vr0[e] * op_apply(c, os, li0, i, j); // tr(vr,Hs,li)+tr(vr0,Hs,li0)
            T[4] += c.vi05[e] * (op_apply(c, oa, li, i, j) + op_apply(c, oa, li0, i, j));        // tr(vi05,Ha,li)+tr(vi05,Ha,li0)
        }
        block_sum(c, T, 5);
        // threads (f, alpha) scatter into the 3 knots of each of the 3 time points; deterministic order
        const int kind = c.P->ctrl_kind[q];
        for (int idx = c.gtid; idx < 2 * c.Nfreq; idx += c.tpt) {
            const int fr = idx >> 1, alpha = idx & 1;
            const int base = 2 * q * c.Nfreq * c.D1 + fr * 2 * c.D1 + alpha * c.D1 - 1;
            const double om = c.P->cfreq[q + c.Nc * fr];
            for (int tp = 0; tp < 3; ++tp) {
                const double tt = tp == 0 ? t0 : (tp == 1 ? t0 + dt : t0 + 0.5 * dt);
                double Pc = tp == 2 ? T[3] : -T[1];                       // multiplies grad p
                double Qc = tp == 0 ? -T[0] : (tp == 1 ? -T[2] : -T[4]);  // multiplies grad q
                if (kind != 0) {
                    // uncoupled control: the K-type (kind 1) or S-type (kind 2) trace combination multiplies grad f,
                    // f = 2 (p cos(w t) - q sin(w t))  ->  d/dp: 2 cos, d/dq: -2 sin  (exact gradient of KS!'s model; the
                    // reference's adjoint_grad_calc! :2621-2654 omits these factors, see oracle header)
                    const double C0 = kind == 1 ? Pc : Qc;
                    double sr, cr;
                    sincos(2.0 * M_PI * c.P->ctrl_rfreq[q] * tt, &sr, &cr);
                    Pc = 2.0 * cr * C0;
                    Qc = -2.0 * sr * C0;
                }
                double sn, cs;
                sincos(om * tt, &sn, &cs);
                const double X = alpha == 0 ? Pc * cs + Qc * sn : Qc * cs - Pc * sn;
                long long k = (long long)ceil(tt / c.dtknot + 2.0);
                k = k < 3 ? 3 : (k > c.D1 ? c.D1 : k);
                const double width = 3.0 * c.dtknot;
                double tau = (tt - c.dtknot * ((double)k - 1.5)) / width;
                g[base + k] += X * (9.0 / 8 + 4.5 * tau + 4.5 * tau * tau);
                tau = (tt - c.dtknot * ((double)(k - 1) - 1.5)) / width;
                g[base + k - 1] += X * (0.75 - 9.0 * tau * tau);
                tau = (tt - c.dtknot * ((double)(k - 2) - 1.5)) / width;
                g[base + k - 2] += X * (9.0 / 8 - 4.5 * tau + 4.5 * tau * tau);
            }
        }
    }
    gsync(c);
}

__device__ void trace_fid(const Ctx &c, double *re, double *im) {
    double v[2] = {0.0, 0.0};
    FOR_E {
        v[0] += c.vr[e] * c.P->vtr[e] - c.vi[e] * c.P->vti[e];  // tr(ur'vtr + ui'vti), ui = -vi
        v[1] += c.vr[e] * c.P->vti[e] + c.vi[e] * c.P->vtr[e];  // tr(ur'vti - ui'vtr)
    }
    block_sum(c, v, 2);
    *re = v[0] / c.m;
    *im = v[1] / c.m;
}

// Context of this thread's group and the operator table (staged into shared memory when G.stage); returns the start of the
// group's own shared-memory region.  Every thread of the CTA calls it (the staging waits on a CTA-wide barrier).
__device__ __forceinline__ double *group_setup(Ctx &c, const DevProblem &P, int Npar, int D1, const GenGeom &G, double *sm) {
    c.P = &P;
    c.n = P.n; c.m = P.m; c.len = P.n * P.m; c.Nc = P.Nc; c.Nfreq = P.Nfreq; c.J = P.J;
    c.Npar = Npar; c.D1 = D1;
    c.dtknot = P.T / (D1 - 2);
    c.tinv = 1.0 / P.T;
    c.tpt = G.tpt; c.gwarps = G.tpt / 32;
    const int grp = threadIdx.x / G.tpt;
    c.gtid = threadIdx.x % G.tpt;
    c.bar = 1 + grp;                                   // named barrier of this group (0 is __syncthreads)
    // ---- operator table: one TMA bulk copy into shared memory per CTA (cp.async.bulk + mbarrier), or global memory through L1
    c.rp = P.rowptr; c.cl = P.col; c.vl = P.val;
    size_t off = 0;                                    // doubles
    if (G.stage) {
        unsigned char *blob = reinterpret_cast<unsigned char *>(sm);
        unsigned long long *mbar = reinterpret_cast<unsigned long long *>(blob + P.csr_bytes);
        if (threadIdx.x == 0) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(mbar)));
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(mbar)), "r"(P.csr_bytes) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(smem_u32(blob)), "l"(P.csr_blob), "r"(P.csr_bytes), "r"(smem_u32(mbar)) : "memory");
        }
        unsigned done = 0;
        while (!done)
            asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0; selp.u32 %0, 1, 0, p; }"
                         : "=r"(done) : "r"(smem_u32(mbar)) : "memory");
        c.rp = reinterpret_cast<const int *>(blob);
        c.cl = reinterpret_cast<const int *>(blob + P.csr_off_col);
        c.vl = reinterpret_cast<const double *>(blob + P.csr_off_val);
        off = (P.csr_bytes + 16) / sizeof(double);
    }
    return sm + off + (size_t)grp * G.per_group;
}

__global__ void __launch_bounds__(GEN_THREADS) jq_generic_kernel(DevProblem P, LaunchArgs A, GenGeom G) {
    extern __shared__ __align__(16) double sm[];
    Ctx c;
    double *p = group_setup(c, P, A.Npar, A.D1, G, sm);
    const int grp = threadIdx.x / G.tpt;
    double **blk[] = {&c.vr, &c.vi, &c.vi05, &c.vr0, &c.lr, &c.li, &c.lr05, &c.li0, &c.lrn, &c.lin, &c.lr05n, &c.li0n,
                      &c.rhs, &c.scr, &c.k1, &c.k2, &c.l1, &c.l2};
    for (int b = 0; b < 18; ++b) {
        if (b >= 8 && b < 12 && P.objFuncType == 1) { *blk[b] = nullptr; continue; }
        *blk[b] = p; p += c.len;
    }
    c.pcof = p; p += c.Npar;
    c.grad = p; p += c.Npar;
    c.igrad = p; p += (P.objFuncType != 1 ? c.Npar : 0);
    c.ctrl = p; p += 6 * c.Nc;
    c.shift = p; p += c.n;
    c.red = p;
    if (grp >= G.gpc) return;                          // threads beyond the last whole group (none with the host's geometry)

    const double tinv = 1.0 / P.T;
    for (int traj = blockIdx.x * G.gpc + grp; traj < A.ntraj; traj += gridDim.x * G.gpc) {      // persistent: groups loop over trajectories
        const int b = traj / A.nsamples, s = traj % A.nsamples;
        for (int k = c.gtid; k < c.Npar; k += c.tpt) { c.pcof[k] = A.pcof[(size_t)b * A.pstride + k]; c.grad[k] = 0.0; if (P.objFuncType != 1) c.igrad[k] = 0.0; }
        const double phase = P.pFidType == 3 ? A.pcof[(size_t)b * A.pstride + c.Npar] : P.globalPhase;   // src/evalobjgrad.jl:591-596
        for (int k = c.gtid; k < c.n; k += c.tpt) c.shift[k] = A.shift ? A.shift[(size_t)s * c.n + k] : 0.0;
        FOR_E { c.vr[e] = P.uinit[e]; c.vi[e] = 0.0; c.vi05[e] = 0.0; }
        gsync(c);

        // ---------------- forward sweep ----------------
        double dt = P.T / (double)P.nsteps, t = 0.0, pen = 0.0;
        double *hr = A.hist_r ? A.hist_r + (size_t)traj * A.nsave * c.len : nullptr;
        double *hi = A.hist_i ? A.hist_i + (size_t)traj * A.nsave * c.len : nullptr;
        if (hr) FOR_E { hr[e] = c.vr[e]; hi[e] = -c.vi[e]; }
        const bool densew = P.wreal != nullptr;
        for (long long step = 0; step < P.nsteps; ++step) {
            penalty_pre(c, &pen);
            eval_controls(c, t, dt);                                               // (its barrier also orders the vr0 copy)
            state_step(c, dt);
            t = t + dt;
            penalty_post(c, &pen);
            if (densew) gsync(c);                                                  // vr0 is rewritten at the top of the next step
            if (hr && (step + 1) % A.save_every == 0) {                                      // src/evalobjgrad.jl:2847-2849
                const size_t o = (size_t)((step + 1) / A.save_every) * c.len;
                FOR_E { hr[o + e] = c.vr[e]; hi[o + e] = -c.vi[e]; }
            }
        }
        double re, im, pv[1] = {pen};
        block_sum(c, pv, 1);
        trace_fid(c, &re, &im);
        double sph, cph;
        sincos(phase, &sph, &cph);
        const int pfid = P.pFidType;
        const double abs2 = re * re + im * im;
        // src/evalobjgrad.jl:755-763: type 1: 1 + |s|^2 - 2 Re(s e^{-i phase}); type 2: 1 - |s|^2; types 3, 4: 1 - tracefidreal(v, e^{i phase} Vtg) = 1 - (Re s cos(phase) - Im s sin(phase))
        const double infid = pfid == 1 ? 1.0 + abs2 - 2.0 * (re * cph + im * sph) : pfid == 2 ? 1.0 - abs2 : 1.0 - (re * cph - im * sph);
        const double leak = 0.5 * dt * tinv * pv[0];
        if (c.gtid == 0) {
            double *o = A.scal + (size_t)traj * 4;
            o[0] = infid; o[1] = leak; o[2] = 1.0 - abs2; o[3] = 0.0;      // traceInfidelity is always 1 - |s|^2 (:792)
        }
        if (!A.evaladjoint) { gsync(c); continue; }

        // ---------------- backward sweep ----------------
        // terminal condition (init_adjoint!, :2026-2059).  Types 1 and 2 share the formula, type 1 on scomplex0 = e^{i phase} - s
        // (:825-826; the reference's init_adjoint! has no branch for type 1 and leaves lambda(T) stale — see the oracle header);
        // types 3, 4: lambda_r = Re(rot) / 2N, lambda_i = -Im(rot) / 2N with rot = e^{i phase} (Vtr + i Vti).
        const double rs_ = pfid == 1 ? cph - re : re, is_ = pfid == 1 ? sph - im : im;
        FOR_E {
            double lr, li;
            if (pfid <= 2) { lr = (rs_ * P.vtr[e] + is_ * P.vti[e]) / c.m; li = (is_ * P.vtr[e] - rs_ * P.vti[e]) / c.m; }
            else { lr = 0.5 * (cph * P.vtr[e] - sph * P.vti[e]) / c.m; li = -0.5 * (sph * P.vtr[e] + cph * P.vti[e]) / c.m; }
            c.lr[e] = lr; c.lr05[e] = lr; c.li[e] = li; c.li0[e] = li;
            if (P.objFuncType != 1) { c.lrn[e] = lr; c.lr05n[e] = lr; c.lin[e] = li; c.li0n[e] = li; }
        }
        t = P.T;
        dt = -dt;
        gsync(c);
        for (long long step = P.nsteps - 1; step >= 0; --step) {
            const double t0 = t;
            FOR_E c.vr0[e] = c.vr[e];
            eval_controls(c, t, dt);
            state_step(c, dt);
            t = t + dt;
            adjoint_step(c, c.lr, c.li, c.lr05, dt, true, tinv);
            grad_step(c, c.lr05, c.li, c.li0, t0, dt, c.grad);
            FOR_E c.li0[e] = c.li[e];
            if (P.objFuncType != 1) {
                adjoint_step(c, c.lrn, c.lin, c.lr05n, dt, false, tinv);
                grad_step(c, c.lr05n, c.lin, c.li0n, t0, dt, c.igrad);
                FOR_E c.li0n[e] = c.lin[e];
            }
            gsync(c);
        }
        for (int k = c.gtid; k < c.Npar; k += c.tpt) {
            A.grad[(size_t)traj * A.gstride + k] = dt * c.grad[k];
            if (P.objFuncType != 1 && A.infidgrad) A.infidgrad[(size_t)traj * A.gstride + k] = dt * c.igrad[k];
        }
        if (pfid == 3 && c.gtid == 0) {
            // primObjGradPhase = -tracefidreal(vfinal, Re(i rot), Im(i rot)) = Re(s) sin(phase) + Im(s) cos(phase) (:923-945),
            // appended to the total and to the infidelity gradient (leakgrad's last entry is their difference, 0)
            const double pg = re * sph + im * cph;
            A.grad[(size_t)traj * A.gstride + c.Npar] = pg;
            if (P.objFuncType != 1 && A.infidgrad) A.infidgrad[(size_t)traj * A.gstride + c.Npar] = pg;
        }
        gsync(c);
    }
}

}  // namespace

// Forward sensitivities (the reference's traceobjgrad(verbose = true, evaladjoint = true) check, src/evalobjgrad.jl:724-745,768-784,
// with step_fwdGrad! src/StormerVerlet.jl:151-251 and fgradforce! src/evalobjgrad.jl:2467-2563): the forward sweep and its tangent
// along a direction d side by side, in the generic kernel's layout.  Trajectory traj = t * ndir + k, t = b * nsamples + s.  The primal
// statements are the generic kernel's own helpers (TAN = true adds the tangent next to each), so infid / leak are its objective-only
// outputs bit for bit.
__global__ void __launch_bounds__(GEN_THREADS) jq_forward_sensitivity_kernel(DevProblem P, SensArgs S, GenGeom G) {
    extern __shared__ __align__(16) double sm[];
    Ctx c{};
    double *p = group_setup(c, P, S.Npar, S.D1, G, sm);
    const int grp = threadIdx.x / G.tpt;
    Tan td;
    double **blk[] = {&c.vr, &c.vi, &c.vi05, &c.vr0, &c.rhs, &c.scr, &c.k1, &c.k2, &c.l1, &c.l2,
                      &td.vr, &td.vi, &td.vi05, &td.vr0, &td.rhs, &td.scr, &td.k1, &td.k2, &td.l1, &td.l2};
    for (int b = 0; b < 20; ++b) { *blk[b] = p; p += c.len; }
    c.pcof = p; p += c.Npar;
    double *dv = p; p += c.Npar;
    c.ctrl = p; p += 6 * c.Nc;
    td.ctrl = p; p += 6 * c.Nc;
    c.shift = p; p += c.n;
    c.red = p;
    // the tangent seen through the primal helpers: the controls of d are the control tables' tangents, trace_fid is linear in the state
    Ctx cd = c;
    cd.pcof = dv; cd.ctrl = td.ctrl; cd.vr = td.vr; cd.vi = td.vi;
    if (grp >= G.gpc) return;

    const double tinv = 1.0 / P.T;
    for (int traj = blockIdx.x * G.gpc + grp; traj < S.ntraj; traj += gridDim.x * G.gpc) {
        const int t_ = traj / S.ndir, k_ = traj % S.ndir, b = t_ / S.nsamples, s = t_ % S.nsamples;
        const double *pc = S.pcof + (size_t)b * S.pstride, *dd = S.dirs + ((size_t)b * S.ndir + k_) * S.pstride;
        for (int k = c.gtid; k < c.Npar; k += c.tpt) { c.pcof[k] = pc[k]; dv[k] = dd[k]; }
        const double phase = P.pFidType == 3 ? pc[c.Npar] : P.globalPhase, dphase = P.pFidType == 3 ? dd[c.Npar] : 0.0;
        for (int k = c.gtid; k < c.n; k += c.tpt) c.shift[k] = S.shift ? S.shift[(size_t)s * c.n + k] : 0.0;
        FOR_E { c.vr[e] = P.uinit[e]; c.vi[e] = 0.0; c.vi05[e] = 0.0; td.vr[e] = 0.0; td.vi[e] = 0.0; td.vi05[e] = 0.0; }
        gsync(c);

        double dt = P.T / (double)P.nsteps, t = 0.0, pen = 0.0, pend = 0.0;
        const bool densew = P.wreal != nullptr;
        for (long long step = 0; step < P.nsteps; ++step) {
            penalty_pre<true>(c, &pen, &td, &pend);
            eval_controls(c, t, dt);
            eval_controls(cd, t, dt);                                              // ctrl_dot: bcarrier2 of d
            state_step<true>(c, dt, &td);
            t = t + dt;
            penalty_post<true>(c, &pen, &td, &pend);
            if (densew) gsync(c);
        }
        double re, im, red, imd, pv[2] = {pen, pend};
        block_sum(c, pv, 2);
        trace_fid(c, &re, &im);
        trace_fid(cd, &red, &imd);
        double sph, cph;
        sincos(phase, &sph, &cph);
        const int pfid = P.pFidType;
        const double abs2 = re * re + im * im;
        const double infid = pfid == 1 ? 1.0 + abs2 - 2.0 * (re * cph + im * sph) : pfid == 2 ? 1.0 - abs2 : 1.0 - (re * cph - im * sph);
        const double leak = 0.5 * dt * tinv * pv[0];
        // tangents of the four pFidType formulas (the phase of type 3 is the last entry of pcof, and of d)
        const double dabs2 = 2.0 * (re * red + im * imd);
        const double dinfid = pfid == 1 ? dabs2 - 2.0 * (red * cph + imd * sph)
                            : pfid == 2 ? -dabs2
                                        : -(red * cph - imd * sph) + dphase * (re * sph + im * cph);
        const double dleak = 0.5 * dt * tinv * pv[1];
        if (c.gtid == 0) {
            if (k_ == 0) {
                double *o = S.scal + (size_t)t_ * 4;
                o[0] = infid; o[1] = leak; o[2] = 1.0 - abs2; o[3] = 0.0;
            }
            S.dinfid[traj] = dinfid;
            S.dleak[traj] = dleak;
        }
        if (S.dstate_r) {
            double *dr = S.dstate_r + (size_t)traj * c.len, *di = S.dstate_i + (size_t)traj * c.len;
            FOR_E { dr[e] = td.vr[e]; di[e] = -td.vi[e]; }
        }
        gsync(c);
    }
}

// doubles of shared memory per trajectory group
static size_t per_group_doubles(const DevProblem &P, int Npar) {
    const size_t len = (size_t)P.n * P.m;
    const size_t nblk = P.objFuncType == 1 ? 14 : 18;
    size_t d = nblk * len + (size_t)Npar * (P.objFuncType == 1 ? 2 : 3) + 6 * P.Nc + P.n + (GEN_THREADS / 32) * 8;
    return (d + 1) & ~(size_t)1;                       // keep every group's region 16-byte aligned
}

// forward-sensitivity kernel: the 10 forward-sweep blocks and their tangents, pcof, d, the control table and its tangent
static size_t fwdsens_group_doubles(const DevProblem &P, int Npar) {
    const size_t len = (size_t)P.n * P.m;
    size_t d = 20 * len + 2 * (size_t)Npar + 12 * P.Nc + P.n + (GEN_THREADS / 32) * 8;
    return (d + 1) & ~(size_t)1;
}

static GenGeom generic_geometry(const DevProblem &P, size_t per_group, size_t *bytes) {
    const size_t len = (size_t)P.n * P.m, limit = 227 * 1024;
    GenGeom G{};
    G.tpt = len <= 32 ? 32 : len <= 64 ? 64 : len <= 128 ? 128 : 256;
    G.gpc = GEN_THREADS / G.tpt;
    G.per_group = (int)per_group;
    const size_t blob = P.csr_blob ? (size_t)P.csr_bytes + 16 : 0;      // + mbarrier
    while (G.gpc > 1 && (size_t)G.gpc * G.per_group * sizeof(double) > limit) G.gpc >>= 1;
    size_t need = (size_t)G.gpc * G.per_group * sizeof(double);
    G.stage = blob != 0 && need + blob <= limit;
    // staging beats more groups per CTA only if the groups still fit: give up groups down to half before giving up staging
    if (!G.stage && blob != 0 && G.gpc > 1 && (size_t)(G.gpc / 2) * G.per_group * sizeof(double) + blob <= limit) {
        G.gpc /= 2;
        need = (size_t)G.gpc * G.per_group * sizeof(double);
        G.stage = 1;
    }
    *bytes = need + (G.stage ? blob : 0);
    return G;
}

size_t jq_generic_smem_bytes(const DevProblem &P, int Npar) {          // minimum: one group, operators through L1
    return per_group_doubles(P, Npar) * sizeof(double);
}

size_t jq_fwdsens_smem_bytes(const DevProblem &P, int Npar) {
    return fwdsens_group_doubles(P, Npar) * sizeof(double);
}

// evalctrl (src/plotstatectrl.jl:246-276): the control functions of every coupled control on an arbitrary time grid,
// with the same device function the time loop uses.  p, q: [Nc][ntimes].
__global__ void jq_controls_kernel(DevProblem P, int D1, const double *pcof, int ntimes, const double *times, double *p, double *q) {
    Ctx c{};
    c.P = &P; c.Nc = P.Nc; c.Nfreq = P.Nfreq; c.D1 = D1; c.pcof = const_cast<double *>(pcof); c.dtknot = P.T / (D1 - 2);
    const long long total = (long long)P.Nc * ntimes;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int q_ = (int)(idx / ntimes);
        const double t = times[idx % ntimes];
        p[idx] = bcarrier2(c, t, 2 * q_);
        q[idx] = bcarrier2(c, t, 2 * q_ + 1);
    }
}

cudaError_t jq_controls_launch(const DevProblem &P, int D1, const double *pcof, int ntimes, const double *times, double *p, double *q,
                               cudaStream_t st) {
    const long long total = (long long)P.Nc * ntimes;
    const int grid = (int)((total + 127) / 128 < 148 * 8 ? (total + 127) / 128 : 148 * 8);
    jq_controls_kernel<<<grid > 0 ? grid : 1, 128, 0, st>>>(P, D1, pcof, ntimes, times, p, q);
    return cudaGetLastError();
}

cudaError_t jq_generic_launch(const DevProblem &P, const LaunchArgs &A, cudaStream_t st, int *nctas, int *regs, size_t *smem) {
    size_t bytes = 0;
    const GenGeom G = generic_geometry(P, per_group_doubles(P, A.Npar), &bytes);
    cudaError_t e = cudaFuncSetAttribute(jq_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return e;
    cudaFuncAttributes fa;
    e = cudaFuncGetAttributes(&fa, jq_generic_kernel);
    if (e != cudaSuccess) return e;
    int dev = 0, sms = 148, occ = 1;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, jq_generic_kernel, G.tpt * G.gpc, bytes);
    if (occ < 1) occ = 1;
    const int want = (A.ntraj + G.gpc - 1) / G.gpc;
    int grid = want < sms * occ ? want : sms * occ;   // persistent: groups loop over trajectories
    jq_generic_kernel<<<grid, G.tpt * G.gpc, bytes, st>>>(P, A, G);
    if (nctas) *nctas = grid;
    if (regs) *regs = fa.numRegs;
    if (smem) *smem = bytes;
    return cudaGetLastError();
}

cudaError_t jq_fwdsens_launch(const DevProblem &P, const SensArgs &S, cudaStream_t st, int *nctas, int *regs, size_t *smem, int *gpc) {
    size_t bytes = 0;
    const GenGeom G = generic_geometry(P, fwdsens_group_doubles(P, S.Npar), &bytes);
    cudaError_t e = cudaFuncSetAttribute(jq_forward_sensitivity_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return e;
    cudaFuncAttributes fa;
    e = cudaFuncGetAttributes(&fa, jq_forward_sensitivity_kernel);
    if (e != cudaSuccess) return e;
    int dev = 0, sms = 148, occ = 1;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, jq_forward_sensitivity_kernel, G.tpt * G.gpc, bytes);
    if (occ < 1) occ = 1;
    const int want = (S.ntraj + G.gpc - 1) / G.gpc;
    const int grid = want < sms * occ ? want : sms * occ;   // persistent: groups loop over trajectories
    jq_forward_sensitivity_kernel<<<grid, G.tpt * G.gpc, bytes, st>>>(P, S, G);
    if (nctas) *nctas = grid;
    if (regs) *regs = fa.numRegs;
    if (smem) *smem = bytes;
    if (gpc) *gpc = G.gpc;
    return cudaGetLastError();
}
