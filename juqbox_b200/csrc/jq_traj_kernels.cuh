// Register-resident trajectory kernels: the state of a trajectory lives in REGISTERS for the whole forward and
// backward time loops; shared memory is only the exchange medium of the sparse operator products.
//
// One kernel template, two lane layouts ("how the n x m block is cut into per-lane register elements"):
//
//  SlotLane<R,C,NC,WQ>  (kernel id 2) generic sparse rows.  A group = NL lanes; lane l owns rows l, l+NL, .. (R rows)
//      and C columns.  Every row keeps per control <= WQ entries (neighbour position, Hsym value, Hanti value); one
//      product pass stores the lane's elements to the group's exchange buffer and loads every neighbour.
//  FiberLane<R,NC,LMASK,AS,XM> (kernel id 3) Kronecker ladder structure.  A lane owns a whole fibre of R consecutive rows
//      (the levels of the fastest subsystem) of ONE column.  Controls in LMASK couple only rows inside a fibre
//      (tridiagonal, coefficients in registers, no memory traffic at all); the other controls couple whole fibres
//      with a fibre-uniform coefficient, so a pass exchanges one R-vector per neighbour fibre instead of one load
//      per nonzero.  Single-subsystem problems (n = R) never touch shared memory inside the time loops.
//
// Common structure.  Up to 4 warps per CTA (fewer only when very long pcof vectors would overflow shared memory); a
// group of GL lanes (a power of two, or m lanes for single-fibre columns) covers (part of) one trajectory, GPT groups
// per trajectory, TPC trajectories per CTA.  Columns never couple inside the time loops, so products only need
// __syncwarp; groups meet through shared memory + __syncthreads once per CH-step chunk (control table), at the
// infidelity between the sweeps and at the final gradient sum.
//   pass(x):  A_q = Hsym_q x and/or D_q = Hanti_q x ;  K(t)x = h0.*x + sum_q p_q(t) A_q ;  S(t)x = sum_q q_q(t) D_q
// The A_q, D_q of the adjoint passes are exactly what the gradient traces need (tr(A'HC) = sum A.*(HC)), so the
// gradient costs no extra products.  Control table: every CH steps all threads fill knot index, the three B-spline
// values and cos/sin of every carrier at the 2CH+1 time points, then p_q, q_q for every resident trajectory.
// Template switches: UPL gradient-scatter roles per lane, MINB register cap, JT compile-time number of Neumann terms,
// OBJ second adjoint set (objFuncType 2/3), GLT compile-time group size.
//
// Reference lines: forward loop src/evalobjgrad.jl:698-753, infidelity :755-766, adjoint init :810-844/:2026-2042,
// backward loop :859-921, steppers src/StormerVerlet.jl:255-303,:461-504, Neumann src/linear_solvers.jl:94-106,
// controls src/bsplines.jl:211-304,:321-381, gradient src/evalobjgrad.jl:2567-2619.  Algebraic regroupings (rounding-level
// effect only, goldens still met at 1e-14..1e-13): S1*u + (h/2) S1*k1 = S1*(u + (h/2) k1)  (src/StormerVerlet.jl:483-484), and
// the truncated Neumann sum evaluated in Horner form with (h/2) folded into the coefficients (see neumann()).
#pragma once
#include "jq_common.h"
#include <type_traits>

#include <cstdio>
#include <cstdlib>
#include <vector>

#define TRAJ_WARPS 4
#define TRAJ_THREADS (TRAJ_WARPS * 32)
#define TRAJ_CH 16   // steps per control-table chunk
#define TRAJ_RING 4  // pipelined instantiations: hand-over slots between the state role and the adjoint role
#define TRAJ_TABS 4  // pipelined instantiations: control-table buffers the table warp runs ahead with

struct TrajParams {
    DevProblem P;
    LaunchArgs A;
    int NL;                                  // lanes per column block (slot: lanes per slot; fibre: fibres per column)
    int GL, GPT, TPC, ngroups;               // lanes per group, groups per trajectory, trajectories / groups per CTA
    int CPG;                                 // fibre layout: columns per group
    int NLR;                                 // slot layout: NL * R (rows incl. padding)
    const int *plan_i;                       // layout-specific integer table
    const double *plan_d;                    // layout-specific coefficient table
    const double *plan_d0, *plan_w;          // per (padded) row: H0 diagonal, guard weight
    int o_exch, o_pcof, o_gsm, o_times, o_tabb, o_tabph, o_tabpq, o_red, o_tabk, o_tred, o_gsm2;   // shared-memory offsets in doubles
    int exch_per_unit;                       // doubles of exchange buffer per group (slot) / per warp (fibre)
    int NparS;                               // shared-memory row stride of the staged pcof vectors (odd: no bank conflicts)
    int GPW;                                 // groups per warp (32 / GL, rounded down: GL need not be a power of two)
    // pipelined (PIPE) instantiations: state-role and adjoint-role warps of one CTA
    int o_ring, o_cnt, tab_role_stride;      // rings of (vr0, vi05, vr) and of lane-partial traces, the int step / chunk counters, size of one control-table buffer
    SegHist H;                               // HIST instantiations: the history VJP's launch arguments (zero otherwise)
};

typedef void (*traj_kernel_t)(const TrajParams);

// What an instantiation of jq_traj_kernel computes and for which layout.  In a table entry every field follows from the template
// arguments (traj_inst); a plan holds the key of its layout, and a query adds what the problem asks for (find_inst in jq_traj.cu).
//   kind 2 slot, 3 fibre, 4 tile; R rows per lane (tile: tiled directions NT), C columns per lane, NC controls, WQ entries per row
//   and control, LMASK controls coupling inside a fibre, UPL gradient-scatter roles per lane, NF tile: in-lane directions;
//   obj2 second adjoint set (objFuncType 2/3), jacobi Jacobi solver, hx exchange-coupled drift, general_hanti Hanti not of the
//   ladder form (AS = 0);
//   glt group size (entry: compile-time, 0 = any); jt Neumann terms compiled in (0 = run-time J; a query passes J instead);
//   nw warps per CTA and role (query: 0 = the entry's own); pipe pipelined roles (matched as zero / non-zero); seg segment sweep
//   of the time-parallel evaluation; hist segment sweep with the history VJP's paths (SegHist).
struct InstKey {
    int kind, R, C, NC, WQ, LMASK, UPL;
    bool obj2 = false, jacobi = false, hx = false, general_hanti = false;
    int glt = 0, jt = 0, nw = TRAJ_WARPS, pipe = 0, seg = 0;
    int NF = 0;
    bool hist = false;
};
struct Inst { InstKey key; traj_kernel_t fn; };
// The instantiation table is split over jq_traj.cu and the jq_traj_inst_*.cu files so that they compile in parallel.
struct InstPart { const Inst *inst; int count; };
template <int N> constexpr InstPart inst_part(const Inst (&t)[N]) { return {t, N}; }
extern const InstPart kInstB, kInstC, kInstD, kInstE, kInstF, kInstG;

struct TrajPlan {
    InstKey key;                             // glt: the group size GL; nw: warps per CTA (per role), 0 for the instantiation's own
    int NL, GPT, TPC, ngroups, CPG, NLR, exch_per_unit;
    int *d_i = nullptr;
    double *d_d = nullptr, *d_d0 = nullptr, *d_w = nullptr;
};

namespace {

#define UNROLL _Pragma("unroll")

// ------------------------------------------------------------------------------------------------ exchange access
// V doubles per position, laid out in planes of `stride` positions so that consecutive lanes hit consecutive banks.
template <int V> struct Xch {          // general V: V/2 planes of double2 followed by one plane of double when V is odd
    static __device__ __forceinline__ void st(double *b, int pos, int s, const double *x) {
        UNROLL for (int p = 0; p < V / 2; ++p) reinterpret_cast<double2 *>(b)[p * s + pos] = make_double2(x[2 * p], x[2 * p + 1]);
        if (V & 1) b[2 * (V / 2) * s + pos] = x[V - 1];
    }
    static __device__ __forceinline__ void ld(const double *b, int pos, int s, double *x) {
        UNROLL for (int p = 0; p < V / 2; ++p) { double2 v = reinterpret_cast<const double2 *>(b)[p * s + pos]; x[2 * p] = v.x; x[2 * p + 1] = v.y; }
        if (V & 1) x[V - 1] = b[2 * (V / 2) * s + pos];
    }
};
template <> struct Xch<1> {
    static __device__ __forceinline__ void st(double *b, int pos, int, const double *x) { b[pos] = x[0]; }
    static __device__ __forceinline__ void ld(const double *b, int pos, int, double *x) { x[0] = b[pos]; }
};
template <> struct Xch<2> {
    static __device__ __forceinline__ void st(double *b, int pos, int, const double *x) { reinterpret_cast<double2 *>(b)[pos] = make_double2(x[0], x[1]); }
    static __device__ __forceinline__ void ld(const double *b, int pos, int, double *x) { double2 v = reinterpret_cast<const double2 *>(b)[pos]; x[0] = v.x; x[1] = v.y; }
};
template <> struct Xch<3> {
    static __device__ __forceinline__ void st(double *b, int pos, int s, const double *x) { b[pos] = x[0]; b[s + pos] = x[1]; b[2 * s + pos] = x[2]; }
    static __device__ __forceinline__ void ld(const double *b, int pos, int s, double *x) { x[0] = b[pos]; x[1] = b[s + pos]; x[2] = b[2 * s + pos]; }
};
template <> struct Xch<4> {
    static __device__ __forceinline__ void st(double *b, int pos, int s, const double *x) {
        reinterpret_cast<double2 *>(b)[pos] = make_double2(x[0], x[1]);
        reinterpret_cast<double2 *>(b)[s + pos] = make_double2(x[2], x[3]);
    }
    static __device__ __forceinline__ void ld(const double *b, int pos, int s, double *x) {
        double2 v = reinterpret_cast<const double2 *>(b)[pos], w = reinterpret_cast<const double2 *>(b)[s + pos];
        x[0] = v.x; x[1] = v.y; x[2] = w.x; x[3] = w.y;
    }
};
template <> struct Xch<6> {
    static __device__ __forceinline__ void st(double *b, int pos, int s, const double *x) {
        UNROLL for (int p = 0; p < 3; ++p) reinterpret_cast<double2 *>(b)[p * s + pos] = make_double2(x[2 * p], x[2 * p + 1]);
    }
    static __device__ __forceinline__ void ld(const double *b, int pos, int s, double *x) {
        UNROLL for (int p = 0; p < 3; ++p) { double2 v = reinterpret_cast<const double2 *>(b)[p * s + pos]; x[2 * p] = v.x; x[2 * p + 1] = v.y; }
    }
};

// ------------------------------------------------------------------------------------------------ lane layouts
// Geometry of this thread inside the CTA, common to both layouts.
struct Geo {
    int lane, warp, lg, group, tloc, gi;     // lane in warp, warp, lane in group, group in CTA, trajectory in CTA, group in trajectory
};

template <int R_, int C_, int NC_, int WQ_>
struct SlotLane {
    static constexpr int KIND = 2, R = R_, C = C_, NC = NC_, WQ = WQ_, LMASK = 0, AS = 1, E = R_ * C_, HX = 0, NF = 0;
    int pos[R][NC][WQ], own[R];
    double hs[R][NC][WQ], ha[R][NC][WQ];
    double d0[E], w[E];
    double p[3][NC], q[3][NC];
    double *buf;
    int nlr, parity, c0;
    int sGL, sbase; double stol;             // Jacobi instantiations: group geometry and tolerance for the residual norm

    __device__ __forceinline__ void setup(const TrajParams &S, double *sm, const Geo &g) {
        nlr = S.NLR; parity = 0; c0 = g.gi * C;
        buf = sm + S.o_exch + g.group * S.exch_per_unit;
        UNROLL for (int k = 0; k < R; ++k) {
            const int r = k * S.NL + g.lg;
            own[k] = r;
            UNROLL for (int qq = 0; qq < NC; ++qq)
                UNROLL for (int e = 0; e < WQ; ++e) {
                    const int ix = (r * NC + qq) * WQ + e;
                    pos[k][qq][e] = S.plan_i[ix];
                    hs[k][qq][e] = S.plan_d[2 * ix];
                    ha[k][qq][e] = S.plan_d[2 * ix + 1];
                }
        }
    }
    // (padded) row and column of element e
    __device__ __forceinline__ int row(int e) const { return own[e / C]; }
    __device__ __forceinline__ int col(int e) const { return c0 + e % C; }

    __device__ __forceinline__ void sync_reset() { __syncwarp(); parity = 0; }
    // Neighbour handle: for this layout the exchange buffer itself (neighbours are loaded entry by entry).
    struct Nbr { const double *b; };
    __device__ __forceinline__ void exchange(const double (&x)[E], Nbr &nb) {
        double *b = buf + parity * (2 * nlr * C);
        parity ^= 1;
        UNROLL for (int k = 0; k < R; ++k) Xch<C>::st(b, own[k], nlr, &x[k * C]);
        __syncwarp();
        nb.b = b;
    }

    // S(level) with the control values folded into the coefficients: one solve uses it for J+1 products
    struct SC { double c[R][NC][WQ]; };
    __device__ __forceinline__ void s_prescale(int level, SC &sc) const {
        UNROLL for (int k = 0; k < R; ++k) UNROLL for (int qq = 0; qq < NC; ++qq) UNROLL for (int e = 0; e < WQ; ++e)
            sc.c[k][qq][e] = q[level][qq] * ha[k][qq][e];
    }
    __device__ __forceinline__ void s_scale(SC &sc, double f) const {
        UNROLL for (int k = 0; k < R; ++k) UNROLL for (int qq = 0; qq < NC; ++qq) UNROLL for (int e = 0; e < WQ; ++e) sc.c[k][qq][e] *= f;
    }
    // t = S x  (ADD: t = add + S x)
    template <bool ADD>
    __device__ __forceinline__ void s_from(const SC &sc, const double (&)[E], const Nbr &nb, const double (&add)[E], double (&t)[E]) const {
        UNROLL for (int k = 0; k < R; ++k) {
            UNROLL for (int c = 0; c < C; ++c) t[k * C + c] = ADD ? add[k * C + c] : 0.0;
            UNROLL for (int qq = 0; qq < NC; ++qq)
                UNROLL for (int e = 0; e < WQ; ++e) {
                    double xv[C];
                    Xch<C>::ld(nb.b, pos[k][qq][e], nlr, xv);
                    UNROLL for (int c = 0; c < C; ++c) t[k * C + c] = fma(sc.c[k][qq][e], xv[c], t[k * C + c]);
                }
        }
    }
    __device__ __forceinline__ void s_pass(const SC &sc, const double (&x)[E], double (&t)[E]) {
        Nbr nb;
        exchange(x, nb);
        s_from<false>(sc, x, nb, x, t);
    }
    __device__ __forceinline__ void s_pass_add(const SC &sc, const double (&x)[E], const double (&add)[E], double (&t)[E]) {
        Nbr nb;
        exchange(x, nb);
        s_from<true>(sc, x, nb, add, t);
    }

    // f(e, Ae, De) is called once per element with Ae[q] = (Hsym_q x)_e, De[q] = (Hanti_q x)_e: the per-control
    // partial products only live for one row at a time.
    template <bool WA, bool WD, class F>
    __device__ __forceinline__ void each_from(const double (&)[E], const Nbr &nb, F f) const {
        UNROLL for (int k = 0; k < R; ++k) {
            double Ar[C][NC + 1], Dr[C][NC];          // Ar[.][NC]: off-diagonal drift product (fibre layout only)
            UNROLL for (int c = 0; c < C; ++c) Ar[c][NC] = 0.0;
            UNROLL for (int qq = 0; qq < NC; ++qq) {
                UNROLL for (int c = 0; c < C; ++c) { Ar[c][qq] = 0.0; Dr[c][qq] = 0.0; }
                UNROLL for (int e = 0; e < WQ; ++e) {
                    double xv[C];
                    Xch<C>::ld(nb.b, pos[k][qq][e], nlr, xv);
                    UNROLL for (int c = 0; c < C; ++c) {
                        if (WA) Ar[c][qq] = fma(hs[k][qq][e], xv[c], Ar[c][qq]);
                        if (WD) Dr[c][qq] = fma(ha[k][qq][e], xv[c], Dr[c][qq]);
                    }
                }
            }
            UNROLL for (int c = 0; c < C; ++c) f(k * C + c, Ar[c], Dr[c]);
        }
    }
    template <bool WA, bool WD, class F>
    __device__ __forceinline__ void pass_each(const double (&x)[E], F f) {
        Nbr nb;
        exchange(x, nb);
        each_from<WA, WD>(x, nb, f);
    }
};

// AS = 1: the control Hamiltonians have the ladder form Hanti = (upper part of Hsym) - (lower part of Hsym), i.e.
// (a - a') next to (a + a'): only the Hsym coefficients are kept and D = upper - lower, A = upper + lower.
// HX != 0: the drift Hamiltonian has exchange-type couplings a_0' a_q + a_0 a_q' between the fastest subsystem and the remote
// subsystems (bit q of HX): row k of this fibre takes element k+1 of the lower and element k-1 of the upper neighbour fibre of
// control q -- fibres every K-product fetches anyway.
template <int R_, int NC_, int LMASK_, int AS_ = 1, int XM_ = 0, int HX_ = 0>
struct FiberLane {
    static constexpr int KIND = 3, R = R_, C = 1, NC = NC_, WQ = 2, LMASK = LMASK_, E = R_, AS = AS_, XM = XM_, HX = HX_, NF = 0;   // XM: 0 = shared-memory exchange, 1 = warp shuffles (16 instead of 24 data-pipe wavefronts per round for R = 4, NC = 2, but 16 instead of 7 instructions)
    static constexpr bool REMOTE = (LMASK_ != (1 << NC_) - 1);
    static constexpr int RM1 = R_ > 1 ? R_ - 1 : 1;
    // local (inside the fibre) tridiagonal coefficients: x_{k+1} -> row k ("u"), x_k -> row k+1 ("l")
    double lsu[NC][RM1], lsl[NC][RM1], lau[NC][RM1], lal[NC][RM1];
    // remote: lower (entry 0) and upper (entry 1) neighbour fibre per control, fibre-uniform coefficients
    int rpos[NC][2];
    double rhs[NC][2], rha[NC][2];
    double xlo[HX_ ? NC : 1][RM1], xhi[HX_ ? NC : 1][RM1];   // drift exchange coefficients (HX only)
    double d0[E], w[E];
    double p[3][NC], q[3][NC];
    double *buf;
    int parity, lane, row0, colj;
    int sGL, sbase; double stol;             // Jacobi instantiations: group geometry and tolerance for the residual norm

    __device__ __forceinline__ void setup(const TrajParams &S, double *sm, const Geo &g) {
        parity = 0; lane = g.lane;
        const int rho = g.lg % S.NL, cj = g.lg / S.NL;
        row0 = rho * R;
        colj = g.gi * S.CPG + cj;
        buf = sm + S.o_exch + g.warp * S.exch_per_unit;
        const int *pi = S.plan_i + rho * (NC * 2);
        constexpr int PERQ = 4 * (R - 1) + 4 + (HX ? 2 * (R - 1) : 0);
        const double *pd = S.plan_d + rho * (NC * PERQ);
        UNROLL for (int qq = 0; qq < NC; ++qq) {
            const double *c = pd + qq * PERQ;
            if constexpr (HX != 0) {
                UNROLL for (int k = 0; k < R - 1; ++k) { xlo[qq][k] = c[4 * (R - 1) + 4 + 2 * k]; xhi[qq][k] = c[4 * (R - 1) + 4 + 2 * k + 1]; }
            }
            UNROLL for (int k = 0; k < R - 1; ++k) {
                lsu[qq][k] = c[4 * k]; lsl[qq][k] = c[4 * k + 1];
                if (!AS) { lau[qq][k] = c[4 * k + 2]; lal[qq][k] = c[4 * k + 3]; }
            }
            UNROLL for (int e = 0; e < 2; ++e) {
                rpos[qq][e] = g.lane + pi[qq * 2 + e];          // plan stores the fibre offset (0 = padding -> own lane)
                rhs[qq][e] = c[4 * (R - 1) + 2 * e];
                if (!AS) rha[qq][e] = c[4 * (R - 1) + 2 * e + 1];
            }
        }
    }
    __device__ __forceinline__ int row(int e) const { return row0 + e; }
    __device__ __forceinline__ int col(int) const { return colj; }

    __device__ __forceinline__ void sync_reset() { if (REMOTE && XM == 0) { __syncwarp(); parity = 0; } }
    // Neighbour handle: the two neighbour fibres of every remote control, in registers.
    struct Nbr { double v[NC][2][R]; };
    __device__ __forceinline__ void fetch(const double *b, const double (&x)[E], Nbr &nb) const {
        UNROLL for (int qq = 0; qq < NC; ++qq)
            if (!((LMASK >> qq) & 1)) {
                if (XM == 0) {
                    Xch<R>::ld(b, rpos[qq][0], 32, nb.v[qq][0]);
                    Xch<R>::ld(b, rpos[qq][1], 32, nb.v[qq][1]);
                } else {
                    UNROLL for (int k = 0; k < R; ++k) {
                        nb.v[qq][0][k] = __shfl_sync(0xffffffffu, x[k], rpos[qq][0]);
                        nb.v[qq][1][k] = __shfl_sync(0xffffffffu, x[k], rpos[qq][1]);
                    }
                }
            }
    }
    // Publish the fibre and fetch the neighbour fibres of every remote control.
    __device__ __forceinline__ void exchange(const double (&x)[E], Nbr &nb) {
        if (!REMOTE) return;
        const double *b = buf;
        if (XM == 0) {
            double *bw = buf + parity * (2 * R * 32);
            parity ^= 1;
            Xch<R>::st(bw, lane, 32, x);
            __syncwarp();
            b = bw;
        }
        fetch(b, x, nb);
    }

    // S(level) with the control values folded into the coefficients: one solve uses it for J+1 products
    struct SC { double lu[RM1], ll[RM1], r[NC][2]; };
    __device__ __forceinline__ void s_prescale(int level, SC &sc) const {
        UNROLL for (int k = 0; k < R - 1; ++k) {
            double u = 0.0, l = 0.0;
            UNROLL for (int qq = 0; qq < NC; ++qq)
                if ((LMASK >> qq) & 1) {
                    u = fma(q[level][qq], AS ? lsu[qq][k] : lau[qq][k], u);
                    l = AS ? fma(-q[level][qq], lsl[qq][k], l) : fma(q[level][qq], lal[qq][k], l);
                }
            sc.lu[k] = u; sc.ll[k] = l;
        }
        UNROLL for (int qq = 0; qq < NC; ++qq)
            if (!((LMASK >> qq) & 1)) {
                sc.r[qq][0] = AS ? -q[level][qq] * rhs[qq][0] : q[level][qq] * rha[qq][0];
                sc.r[qq][1] = q[level][qq] * (AS ? rhs[qq][1] : rha[qq][1]);
            }
    }
    __device__ __forceinline__ void s_scale(SC &sc, double f) const {
        UNROLL for (int k = 0; k < R - 1; ++k) { sc.lu[k] *= f; sc.ll[k] *= f; }
        UNROLL for (int qq = 0; qq < NC; ++qq)
            if (!((LMASK >> qq) & 1)) { sc.r[qq][0] *= f; sc.r[qq][1] *= f; }
    }
    // t = S x  (ADD: t = add + S x)
    template <bool ADD>
    __device__ __forceinline__ void s_from(const SC &sc, const double (&x)[E], const Nbr &nb, const double (&add)[E], double (&t)[E]) const {
        UNROLL for (int k = 0; k < R; ++k) {       // local part first: independent of the exchange
            double a = ADD ? add[k] : 0.0;
            if (k + 1 < R) a = ADD ? fma(sc.lu[k], x[k + 1], a) : sc.lu[k] * x[k + 1];
            if (k > 0) a = fma(sc.ll[k - 1], x[k - 1], a);
            t[k] = a;
        }
        UNROLL for (int qq = 0; qq < NC; ++qq)
            if (!((LMASK >> qq) & 1))
                UNROLL for (int k = 0; k < R; ++k) t[k] = fma(sc.r[qq][1], nb.v[qq][1][k], fma(sc.r[qq][0], nb.v[qq][0][k], t[k]));
    }
    __device__ __forceinline__ void s_pass(const SC &sc, const double (&x)[E], double (&t)[E]) {
        Nbr nb;
        exchange(x, nb);
        s_from<false>(sc, x, nb, x, t);
    }
    __device__ __forceinline__ void s_pass_add(const SC &sc, const double (&x)[E], const double (&add)[E], double (&t)[E]) {
        Nbr nb;
        exchange(x, nb);
        s_from<true>(sc, x, nb, add, t);
    }

    template <bool WA, bool WD, class F>
    __device__ __forceinline__ void each_from(const double (&x)[E], const Nbr &nb, F f) const {
        UNROLL for (int k = 0; k < R; ++k) {
            double Ae[NC + 1], De[NC];                 // Ae[NC]: off-diagonal drift product of row k
            Ae[NC] = 0.0;
            if constexpr (HX != 0 && WA) {
                UNROLL for (int qq = 0; qq < NC; ++qq)
                    if ((HX >> qq) & 1) {
                        if (k + 1 < R) Ae[NC] = fma(xlo[qq][k], nb.v[qq][0][k + 1], Ae[NC]);
                        if (k > 0) Ae[NC] = fma(xhi[qq][k - 1], nb.v[qq][1][k - 1], Ae[NC]);
                    }
            }
            UNROLL for (int qq = 0; qq < NC; ++qq) {
                double up = 0.0, lo = 0.0, a = 0.0, d = 0.0;
                if ((LMASK >> qq) & 1) {
                    if (AS) {
                        if (k + 1 < R) up = lsu[qq][k] * x[k + 1];
                        if (k > 0) lo = lsl[qq][k - 1] * x[k - 1];
                    } else {
                        if (k + 1 < R) { if (WA) a = lsu[qq][k] * x[k + 1]; if (WD) d = lau[qq][k] * x[k + 1]; }
                        if (k > 0) { if (WA) a = fma(lsl[qq][k - 1], x[k - 1], a); if (WD) d = fma(lal[qq][k - 1], x[k - 1], d); }
                    }
                } else {
                    if (AS) {
                        lo = rhs[qq][0] * nb.v[qq][0][k];
                        up = rhs[qq][1] * nb.v[qq][1][k];
                    } else {
                        if (WA) a = fma(rhs[qq][1], nb.v[qq][1][k], rhs[qq][0] * nb.v[qq][0][k]);
                        if (WD) d = fma(rha[qq][1], nb.v[qq][1][k], rha[qq][0] * nb.v[qq][0][k]);
                    }
                }
                if (AS) { a = up + lo; d = up - lo; }
                Ae[qq] = a; De[qq] = d;
            }
            f(k, Ae, De);
        }
    }
    template <bool WA, bool WD, class F>
    __device__ __forceinline__ void pass_each(const double (&x)[E], F f) {
        Nbr nb;
        exchange(x, nb);
        each_from<WA, WD>(x, nb, f);
    }
};


// Tile layout (kernel id 4): Kronecker ladder Hamiltonians whose subsystems all have 4 levels (the cnot2 and cnot3 examples).
// Control q <-> direction q (row stride 4^q).  The first NF directions lie WHOLE in the lane ("in-lane directions": all 4
// levels, a tridiagonal product with no traffic, coefficients the same in every lane).  The next NT ("tiled directions") are
// cut in HALVES: a lane owns 2 of the 4 levels.  E = 4^NF 2^NT elements, element e = sum_{d<NF} l_d 4^d + 4^NF sum_d i_d 2^d
// with l_d the level of in-lane direction d and i_d the position inside the half of tiled direction NF + d.  The upper half
// keeps its levels in MIRRORED order (i = 0 -> level 3, i = 1 -> level 2; lower half i = 0 -> level 0, i = 1 -> level 1), so in
// every lane i = 1 is the level at the interface and i = 0 the outer level: the code is uniform, each lane has exactly ONE
// neighbour lane per tiled direction (lane ^ 2^d) and needs only the interface face of its tile (E/2 values) from it -- for
// cnot2, 4 doubles per product for 4 elements (NF = 0, NT = 2) where the fibre layout moves 8, or 4 doubles for 8 elements
// (NF = 1, NT = 1) -- and the in-lane pair coupling needs no traffic at all.  Mirroring swaps "upper" and "lower" neighbour,
// i.e. flips the sign of the antisymmetric product D = Hanti x of that direction; the sign sg[d] is folded into the lane's copy
// of q_d(t) (LOAD_LEVELS) and applied to the lane's partial traces that contain D (dsign); in-lane directions have none.
// Controls NF+NT..NC-1 are remote as in the fibre layout (a lane per level, lower and upper neighbour lane, lane-uniform
// coefficients).  Exchange is by warp shuffle only.  Requires Hanti = upper(Hsym) - lower(Hsym) and a diagonal Hconst (the
// planner checks).
template <int NC_, int NT_, int NF_ = 0>
struct TileLane {
    static constexpr int KIND = 4, NC = NC_, NT = NT_, NF = NF_, E = (1 << (2 * NF_)) << NT_, HX = 0, R = NT_, C = 1, WQ = 0, LMASK = 0, AS = 1;
    static constexpr bool SIGNED = true;
    static constexpr int HB = 2 * NF_;                  // bit of the element index where the tiled directions start
    static constexpr int NT1 = NT_ > 0 ? NT_ : 1, EH = NT_ > 0 ? E / 2 : 1;      // array extents (NT = 0: no faces)
    static constexpr int NF1 = NF_ > 0 ? NF_ : 1;
    double cf[NF1][3];                       // in-lane ladder coefficients between levels l and l+1
    double cin[NT1], cx[NT1], sg[NT1];       // in-lane pair coupling, cross-lane (interface) coupling, mirror sign
    static constexpr int NRC = NC_ - NT_ - NF_, NREM = NRC > 0 ? NRC : 1;
    int rpos[NREM][2];
    double rhs[NREM][2];
    double d0[E], w[E];
    double p[3][NC], q[3][NC];
    int lane, rho, colj, gdim;
    int sGL, sbase; double stol;

    __device__ __forceinline__ void setup(const TrajParams &S, double *, const Geo &g) {
        lane = g.lane;
        rho = g.lg % S.NL;
        colj = g.gi * S.CPG + g.lg / S.NL;
        gdim = rho >> NT;                                  // level index of the remote directions (row offset 4^(NF+NT) * gdim)
        const double *pd = S.plan_d + rho * (3 * NF + 3 * NT + 2 * NRC);
        UNROLL for (int d = 0; d < NF; ++d) UNROLL for (int l = 0; l < 3; ++l) cf[d][l] = pd[3 * d + l];
        pd += 3 * NF;
        UNROLL for (int d = 0; d < NT; ++d) { cin[d] = pd[3 * d]; cx[d] = pd[3 * d + 1]; sg[d] = pd[3 * d + 2]; }
        UNROLL for (int r = 0; r < NRC; ++r) {
            UNROLL for (int e = 0; e < 2; ++e) {
                rpos[r][e] = g.lane + S.plan_i[(rho * NRC + r) * 2 + e];
                rhs[r][e] = pd[3 * NT + 2 * r + e];
            }
        }
    }
    __device__ __forceinline__ int row(int e) const {
        int r = 0, st = 1;
        UNROLL for (int d = 0; d < NF; ++d) { r += st * ((e >> (2 * d)) & 3); st *= 4; }
        UNROLL for (int d = 0; d < NT; ++d) {
            const int i = (e >> (HB + d)) & 1, hb = (rho >> d) & 1;
            r += st * (hb ? 3 - i : i);
            st *= 4;
        }
        return r + st * gdim;
    }
    __device__ __forceinline__ int col(int) const { return colj; }
    __device__ __forceinline__ double dsign(int qq) const { return qq >= NF && qq < NF + NT ? sg[qq - NF] : 1.0; }
    __device__ __forceinline__ void sync_reset() {}

    // index of element e inside the interface face of tiled direction d (its bit removed)
    static __device__ __forceinline__ constexpr int face(int e, int d) { return (e & ((1 << (HB + d)) - 1)) | ((e >> (HB + d + 1)) << (HB + d)); }
    struct Nbr { double t[NT1][EH]; double r[NREM][2][E]; };
    __device__ __forceinline__ void exchange(const double (&x)[E], Nbr &nb) const {
        UNROLL for (int d = 0; d < NT; ++d)
            UNROLL for (int e = 0; e < E; ++e)
                if ((e >> (HB + d)) & 1) nb.t[d][face(e, d)] = __shfl_xor_sync(0xffffffffu, x[e], 1 << d);
        UNROLL for (int r = 0; r < NRC; ++r)
            UNROLL for (int e = 0; e < E; ++e) {
                nb.r[r][0][e] = __shfl_sync(0xffffffffu, x[e], rpos[r][0]);
                nb.r[r][1][e] = __shfl_sync(0xffffffffu, x[e], rpos[r][1]);
            }
    }

    // Control-weighted neighbour coefficients of W x = sum_q wt_q (Hsym_q x) (symmetric form) or sum_q wt_q (Hanti_q x) (antisymmetric
    // form, wt = q[level], which already carries sg).  The remote lower coefficients carry the sign of their form; the in-lane and pair
    // terms get it in w_from.
    struct SC { double f[NF1][3], a[NT1], b[NT1], r[NREM][2]; };
    template <bool ANTI>
    __device__ __forceinline__ void w_prescale(const double (&wt)[NC], SC &sc) const {
        UNROLL for (int d = 0; d < NF; ++d) UNROLL for (int l = 0; l < 3; ++l) sc.f[d][l] = wt[d] * cf[d][l];
        UNROLL for (int d = 0; d < NT; ++d) { sc.a[d] = wt[NF + d] * cin[d]; sc.b[d] = wt[NF + d] * cx[d]; }
        UNROLL for (int r = 0; r < NRC; ++r) { sc.r[r][0] = (ANTI ? -wt[NF + NT + r] : wt[NF + NT + r]) * rhs[r][0]; sc.r[r][1] = wt[NF + NT + r] * rhs[r][1]; }
    }
    __device__ __forceinline__ void s_prescale(int level, SC &sc) const { w_prescale<true>(q[level], sc); }
    __device__ __forceinline__ void s_scale(SC &sc, double f) const {
        UNROLL for (int d = 0; d < NF; ++d) UNROLL for (int l = 0; l < 3; ++l) sc.f[d][l] *= f;
        UNROLL for (int d = 0; d < NT; ++d) { sc.a[d] *= f; sc.b[d] *= f; }
        UNROLL for (int r = 0; r < NRC; ++r) { sc.r[r][0] *= f; sc.r[r][1] *= f; }
    }
    // t[o] = (bit o of ADDM: add) +- ((bit o of DIAG: d0.*x) + W_o x) for the N coefficient sets sc[o], all from one exchange; bit o
    // of ANTI: W_o has the antisymmetric form, of NEG: the minus sign (it rides on the FMAs).  In-lane products first (independent of
    // the exchange), direction outer / element inner: neighbouring FMAs share the coefficient register.  In-lane directions:
    // (W x)_l = c_l x_{l+1} +- c_{l-1} x_{l-1}; without a diagonal or an addend the first term met starts the sum.
    template <int N, unsigned ANTI, unsigned DIAG, unsigned ADDM, unsigned NEG = 0u>
    __device__ __forceinline__ void w_from(const SC *sc, const double (&x)[E], const Nbr &nb, const double (&add)[E], double (*t)[E]) const {
        UNROLL for (int o = 0; o < N; ++o) {
            const bool an = (ANTI >> o) & 1, dg = (DIAG >> o) & 1, ad = (ADDM >> o) & 1, ng = (NEG >> o) & 1;
            const bool open = !dg && !ad && (NF > 0 || NT > 0);      // the first neighbour term starts the sum
            auto sgn = [ng](double c) { return ng ? -c : c; };
            if (!open) { UNROLL for (int e = 0; e < E; ++e) t[o][e] = dg ? (ad ? fma(sgn(d0[e]), x[e], add[e]) : sgn(d0[e]) * x[e]) : (ad ? add[e] : 0.0); }
            UNROLL for (int d = 0; d < NF; ++d)
                UNROLL for (int e = 0; e < E; ++e) {
                    const int l = (e >> (2 * d)) & 3, st = 1 << (2 * d);
                    if (l < 3) { const double c = sgn(sc[o].f[d][l]); t[o][e] = open && d == 0 ? c * x[e + st] : fma(c, x[e + st], t[o][e]); }
                    if (l > 0) {
                        const double c = sgn(an ? -sc[o].f[d][l - 1] : sc[o].f[d][l - 1]);
                        t[o][e] = open && d == 0 && l == 3 ? c * x[e - st] : fma(c, x[e - st], t[o][e]);
                    }
                }
            UNROLL for (int d = 0; d < NT; ++d)
                UNROLL for (int e = 0; e < E; ++e) {
                    const double c = sgn(an && ((e >> (HB + d)) & 1) ? -sc[o].a[d] : sc[o].a[d]);
                    const int en = e ^ (1 << (HB + d));
                    t[o][e] = open && NF == 0 && d == 0 ? c * x[en] : fma(c, x[en], t[o][e]);
                }
            UNROLL for (int d = 0; d < NT; ++d)
                UNROLL for (int e = 0; e < E; ++e)
                    if ((e >> (HB + d)) & 1) t[o][e] = fma(sgn(sc[o].b[d]), nb.t[d][face(e, d)], t[o][e]);
            UNROLL for (int r = 0; r < NRC; ++r)
                UNROLL for (int e = 0; e < E; ++e)
                    t[o][e] = fma(sgn(sc[o].r[r][1]), nb.r[r][1][e], fma(sgn(sc[o].r[r][0]), nb.r[r][0][e], t[o][e]));
        }
    }
    // t = S x  (ADD: t = add + S x)
    template <bool ADD>
    __device__ __forceinline__ void s_from(const SC &sc, const double (&x)[E], const Nbr &nb, const double (&add)[E], double (&t)[E]) const {
        w_from<1, 1u, 0u, ADD ? 1u : 0u>(&sc, x, nb, add, &t);
    }
    __device__ __forceinline__ void s_pass(const SC &sc, const double (&x)[E], double (&t)[E]) {
        Nbr nb;
        exchange(x, nb);
        s_from<false>(sc, x, nb, x, t);
    }
    __device__ __forceinline__ void s_pass_add(const SC &sc, const double (&x)[E], const double (&add)[E], double (&t)[E]) {
        Nbr nb;
        exchange(x, nb);
        s_from<true>(sc, x, nb, add, t);
    }
    // Ae[q] = (Hsym_q x)_e, De[q] = sg[q] * (Hanti_q x)_e  (the sign rides on q[.][q] and dsign)
    template <bool WA, bool WD, class F>
    __device__ __forceinline__ void each_from(const double (&x)[E], const Nbr &nb, F f) const {
        UNROLL for (int e = 0; e < E; ++e) {
            double Ae[NC + 1], De[NC];
            Ae[NC] = 0.0;
            UNROLL for (int d = 0; d < NF; ++d) {          // up = c_l x_{l+1}, lo = c_{l-1} x_{l-1}: A = up + lo, D = up - lo
                const int l = (e >> (2 * d)) & 3, st = 1 << (2 * d);
                if (l == 0) { const double up = cf[d][0] * x[e + st]; Ae[d] = up; De[d] = up; }
                else if (l == 3) { const double lo = cf[d][2] * x[e - st]; Ae[d] = lo; De[d] = -lo; }
                else { const double up = cf[d][l] * x[e + st], lo = cf[d][l - 1] * x[e - st]; Ae[d] = up + lo; De[d] = up - lo; }
            }
            UNROLL for (int d = 0; d < NT; ++d) {
                const double pin = cin[d] * x[e ^ (1 << (HB + d))];
                if ((e >> (HB + d)) & 1) {
                    const double xc = cx[d] * nb.t[d][face(e, d)];
                    Ae[NF + d] = xc + pin; De[NF + d] = xc - pin;
                } else {
                    Ae[NF + d] = pin; De[NF + d] = pin;
                }
            }
            UNROLL for (int r = 0; r < NRC; ++r) {
                const double lo = rhs[r][0] * nb.r[r][0][e], up = rhs[r][1] * nb.r[r][1][e];
                Ae[NF + NT + r] = up + lo; De[NF + NT + r] = up - lo;
            }
            f(e, Ae, De);
        }
    }
    template <bool WA, bool WD, class F>
    __device__ __forceinline__ void pass_each(const double (&x)[E], F f) {
        Nbr nb;
        exchange(x, nb);
        each_from<WA, WD>(x, nb, f);
    }
};

// Sign of the lane's antisymmetric products of control qq relative to Hanti_qq x (tile layout: mirrored halves); 1 elsewhere.
template <class LaneT, class = void> struct LaneSigned : std::false_type {};
template <class LaneT> struct LaneSigned<LaneT, std::enable_if_t<LaneT::SIGNED>> : std::true_type {};
// Layouts with control-weighted neighbour products (w_prescale / w_from): the state steps weight the coefficients instead of forming
// the per-control products A_q x, D_q x, which no trace of a state step reads.
template <class LaneT, class = void> struct LaneWeighted : std::false_type {};
// With fewer than 4 elements per lane (the latency layouts) the coefficient prescales would cost more than the weighting saves.
template <class LaneT> struct LaneWeighted<LaneT, std::void_t<decltype(&LaneT::template w_from<1, 0u, 0u, 0u>)>> : std::bool_constant<(LaneT::E >= 4)> {};

// ------------------------------------------------------------------------------------------------ steppers
// Sum over the GL lanes of a group, result on every lane.  Power-of-two groups use the xor butterfly; other sizes
// (single-fibre columns with m = 3) gather the GL values in lane order.
__device__ __forceinline__ double group_sum(double x, int GL, int base) {
    if ((GL & (GL - 1)) == 0) {
        for (int o = 1; o < GL; o <<= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
        return x;
    }
    double s = 0.0;
    for (int j = 0; j < GL; ++j) s += __shfl_sync(0xffffffffu, x, base + j);
    return s;
}

// The same for N values at once, ROUNDS OUTER / VALUES INNER: the N shuffles of a round are independent and pipeline,
// so the dependent chain is log2(GL) shuffle latencies in total instead of N * log2(GL) (measured: the value-by-value
// form was 22% of all stall samples of the kernel).
template <int N>
__device__ __forceinline__ void group_sum_n(double (&v)[N], int GL, int base) {
    if ((GL & (GL - 1)) == 0) {
#pragma unroll
        for (int o = 1; o < GL; o <<= 1) {       // unrolled when GL is a compile-time constant (GLT instantiations)
            double r[N];
            UNROLL for (int i = 0; i < N; ++i) r[i] = __shfl_xor_sync(0xffffffffu, v[i], o);
            UNROLL for (int i = 0; i < N; ++i) v[i] += r[i];
        }
        return;
    }
    double s[N];
    UNROLL for (int i = 0; i < N; ++i) s[i] = 0.0;
#pragma unroll
    for (int j = 0; j < GL; ++j) {           // unrolled for GLT instantiations
        UNROLL for (int i = 0; i < N; ++i) s[i] += __shfl_sync(0xffffffffu, v[i], base + j);
    }
    UNROLL for (int i = 0; i < N; ++i) v[i] = s[i];
}

// Reduce-scatter of N values over the GL lanes of a group (GL a compile-time power of two) by recursive halving: the values,
// padded with zeros to M = a power of two, are halved over the low lane bits -- a lane sends the half it gives up to its partner
// and adds the half it keeps -- and when fewer than GL lanes share them, the last K = max(M / GL, 1) are summed by xor butterfly over
// the remaining bits.  Lane lg ends with the full sums of values first .. first + K - 1 in s (returned: first); the lanes whose
// butterfly bits are zero own them.  The pair sums are the same on both partners (addition commutes), so the summation tree, and
// every result bit, depends only on the group's lanes, not on where the group sits.  A lane sends M - K values over the halving
// rounds and K per butterfly round, where the butterfly of group_sum_n sends N per round.
constexpr int ilog2(int x) { return x > 1 ? 1 + ilog2(x / 2) : 0; }
template <int N, int GL>
struct ScatterShape {
    static_assert(GL > 0 && (GL & (GL - 1)) == 0, "reduce-scatter: power-of-two group");
    static constexpr int M = 1 << ilog2(2 * N - 1), K = M > GL ? M / GL : 1, H = ilog2(M / K);     // H: halving rounds
};
template <int N, int GL>
__device__ __forceinline__ int group_scatter_sum(const double (&v)[N], int lg, double (&s)[ScatterShape<N, GL>::K]) {
    constexpr int M = ScatterShape<N, GL>::M, K = ScatterShape<N, GL>::K, H = ScatterShape<N, GL>::H;
    double c[M];
    UNROLL for (int i = 0; i < M; ++i) c[i] = i < N ? v[i] : 0.0;
    int first = 0;
    UNROLL for (int r = 0; r < H; ++r) {                 // all sends of a round are independent: one shuffle latency per round
        const int half = M >> (r + 1);
        const bool hi = (lg >> r) & 1;
        double g[M > 1 ? M / 2 : 1];
        UNROLL for (int i = 0; i < half; ++i) g[i] = __shfl_xor_sync(0xffffffffu, hi ? c[i] : c[half + i], 1 << r);
        UNROLL for (int i = 0; i < half; ++i) c[i] = (hi ? c[half + i] : c[i]) + g[i];
        if (hi) first += half;
    }
    UNROLL for (int o = 1 << H; o < GL; o <<= 1) {
        double g[K];
        UNROLL for (int i = 0; i < K; ++i) g[i] = __shfl_xor_sync(0xffffffffu, c[i], o);
        UNROLL for (int i = 0; i < K; ++i) c[i] += g[i];
    }
    UNROLL for (int i = 0; i < K; ++i) s[i] = c[i];
    return first;
}

// (H0 x)_e for the lane's element e: diagonal entry times x_e, plus the off-diagonal drift product x0 in HX layouts.
template <class LaneT>
__device__ __forceinline__ double kdiag(const LaneT &L, int e, double xe, double x0) {
    if constexpr (LaneT::HX != 0) return fma(L.d0[e], xe, x0);
    else return L.d0[e] * xe;
}

// X = sum_{j<=J} (h/2)^j S^j B   (src/linear_solvers.jl:94-106), evaluated in Horner form  X <- B + ((h/2) S) X,  J times from
// X = B -- the same polynomial in S applied to B (it is the reference's own Jacobi sweep, linear_solvers.jl:118-124, run for
// exactly J sweeps), with the factor h/2 folded into the coefficients: one FMA per element and term less than accumulating
// the terms one by one.  `sc` = S(level) prescaled by the control values; SCALED: already multiplied by h/2.  B is preserved.
template <int JT, bool SCALED = false, class LaneT>
__device__ __forceinline__ void neumann(LaneT &L, typename LaneT::SC &sc, int J, double h, double (&B)[LaneT::E], double (&X)[LaneT::E]) {
    constexpr int E = LaneT::E;
    if (!SCALED) L.s_scale(sc, 0.5 * h);
    UNROLL for (int e = 0; e < E; ++e) X[e] = B[e];
    const int JJ = JT > 0 ? JT : J;          // JT > 0: number of Neumann terms known at compile time (fully unrolled)
#pragma unroll
    for (int it = 0; it < JJ; ++it) {
        double T[E];
        L.s_pass_add(sc, X, B, T);
        UNROLL for (int e = 0; e < E; ++e) X[e] = T[e];
    }
}

// JACOBI_SOLVER (src/linear_solvers.jl:110-152): X = B; T = B + (h/2) S X; err = ||T - X||_F over the whole n x m block;
// X = T; stop when err < tol or after J sweeps.  The block of a trajectory is one group here (the planner only admits
// GPT == 1), so the norm is one group reduction; groups of a warp that have converged keep exchanging (the passes need
// the whole warp) but stop updating, and the warp leaves the loop when all its groups are done.  B is preserved.
template <class LaneT>
__device__ __forceinline__ void jacobi(LaneT &L, const typename LaneT::SC &sc, int maxit, double h, double (&B)[LaneT::E], double (&X)[LaneT::E]) {
    constexpr int E = LaneT::E;
    UNROLL for (int e = 0; e < E; ++e) X[e] = B[e];
    bool active = true;
    for (int it = 0; it < maxit; ++it) {
        double T[E], err = 0.0;
        L.s_pass(sc, X, T);
        UNROLL for (int e = 0; e < E; ++e) { T[e] = fma(0.5 * h, T[e], B[e]); const double d = T[e] - X[e]; err = fma(d, d, err); }
        err = group_sum(err, L.sGL, L.sbase);
        if (active) { UNROLL for (int e = 0; e < E; ++e) X[e] = T[e]; }
        active = active && !(sqrt(err) < L.stol);
        if (!__any_sync(0xffffffffu, active)) break;
    }
}

// linear_solver.solve of the steppers: JT >= 0 truncated Neumann series (JT > 0: compile-time J), JT < 0 Jacobi sweeps.
template <int JT, bool SCALED = false, class LaneT>
__device__ __forceinline__ void solve(LaneT &L, typename LaneT::SC &sc, int J, double h, double (&B)[LaneT::E], double (&X)[LaneT::E]) {
    if constexpr (JT < 0) jacobi(L, sc, J, h, B, X);
    else neumann<JT, SCALED>(L, sc, J, h, B, X);
}

// Weighted layouts: the boundary products of a state step, bp[0] = K05 u and bp[1] = S0 u of the state u it starts from.
template <class LaneT>
__device__ __forceinline__ void step_open(LaneT &L, const double (&u)[LaneT::E], const double (&p05)[LaneT::NC], const double (&q0)[LaneT::NC],
                                          double (&bp)[2][LaneT::E]) {
    typename LaneT::SC w[2];
    L.template w_prescale<false>(p05, w[0]);
    L.template w_prescale<true>(q0, w[1]);
    typename LaneT::Nbr nb;
    L.exchange(u, nb);
    L.template w_from<2, 2u, 1u, 0u>(w, u, nb, u, bp);
}

// src/StormerVerlet.jl:461-504 for the weighted layouts, entered with the boundary products bp of u (step_open).  SHARE: the last
// product pass also forms those of the outgoing u for the next step (p05 of the next step = pn; its S0 is this step's S1) and leaves
// them in bp, so consecutive steps share one exchange of u.
template <int JT, bool SHARE, class LaneT>
__device__ __forceinline__ void state_step_w(LaneT &L, int J, double h, double (&u)[LaneT::E], double (&v)[LaneT::E], double (&v05)[LaneT::E],
                                             double (&bp)[2][LaneT::E], const double (&pn)[LaneT::NC]) {
    constexpr int E = LaneT::E;
    double rhs[E], l1[E];
    typename LaneT::SC sc;
    typename LaneT::Nbr nb;
    L.s_prescale(1, sc);
    L.s_pass_add(sc, v, bp[0], rhs);                                                           // K05 u + S05 v
    solve<JT>(L, sc, J, h, rhs, l1);
    UNROLL for (int e = 0; e < E; ++e) v05[e] = fma(0.5 * h, l1[e], v[e]);
    double k1v[E], s05v[E];
    {
        typename LaneT::SC w[3];
        L.template w_prescale<false>(L.p[0], w[0]);
        L.template w_prescale<false>(L.p[2], w[1]);
        L.template w_prescale<true>(L.q[1], w[2]);
        double t[3][E];                                                                        // kappa1 = S0 u - K0 v05, -K1 v05, S05 v05
        L.exchange(v05, nb);
        L.template w_from<3, 4u, 3u, 1u, 3u>(w, v05, nb, bp[1], t);
        UNROLL for (int e = 0; e < E; ++e) {
            k1v[e] = t[1][e];
            s05v[e] = t[2][e];
            u[e] = fma(0.5 * h, t[0][e], u[e]);            // u + (h/2) kappa1
        }
    }
    constexpr int NO = SHARE ? 3 : 1;
    typename LaneT::SC w[NO];
    L.s_prescale(2, sc);
    if constexpr (SHARE) w[2] = sc;                                                            // the next step's S0
    L.s_pass_add(sc, u, k1v, rhs);                                                             // S1 (u + (h/2) kappa1) - K1 v05
    double k2[E];
    solve<JT>(L, sc, J, h, rhs, k2);
    UNROLL for (int e = 0; e < E; ++e) u[e] = fma(0.5 * h, k2[e], u[e]);
    L.template w_prescale<false>(L.p[1], w[0]);
    if constexpr (SHARE) L.template w_prescale<false>(pn, w[1]);
    double t[NO][E];                                                                           // l2 = K05 u + S05 v05 (, next K05 u, S0 u)
    L.exchange(u, nb);
    L.template w_from<NO, 4u, 3u, 1u>(w, u, nb, s05v, t);
    UNROLL for (int e = 0; e < E; ++e) v[e] = fma(0.5 * h, t[0][e], v05[e]);                   // v + (h/2)(l1 + l2) = v05 + (h/2) l2
    if constexpr (SHARE) { UNROLL for (int e = 0; e < E; ++e) { bp[0][e] = t[1][e]; bp[1][e] = t[2][e]; } }
}

// src/StormerVerlet.jl:461-504.  u, v updated in place; v05 returned.
template <int JT, class LaneT>
__device__ __forceinline__ void state_step(LaneT &L, int J, double h, double (&u)[LaneT::E], double (&v)[LaneT::E], double (&v05)[LaneT::E]) {
    constexpr int E = LaneT::E, NC = LaneT::NC;
    if constexpr (LaneWeighted<LaneT>::value) {
        double bp[2][E];
        step_open(L, u, L.p[1], L.q[0], bp);
        state_step_w<JT, false>(L, J, h, u, v, v05, bp, L.p[1]);
        return;
    }
    double rhs[E], l1[E], s0u[E];
    L.sync_reset();        // buffer parity restarts at 0: with compile-time J every exchange address is a constant offset
    L.template pass_each<true, true>(u, [&](int e, const double (&Ae)[NC + 1], const double (&De)[NC]) {
        double r = kdiag(L, e, u[e], Ae[NC]), s = 0.0;
        UNROLL for (int qq = 0; qq < NC; ++qq) { r = fma(L.p[1][qq], Ae[qq], r); s = fma(L.q[0][qq], De[qq], s); }
        rhs[e] = r;            // K05 u
        s0u[e] = s;            // S0 u
    });
    typename LaneT::SC sc;
    L.s_prescale(1, sc);
    L.s_pass_add(sc, v, rhs, rhs);                                                             // + S05 v
    solve<JT>(L, sc, J, h, rhs, l1);
    UNROLL for (int e = 0; e < E; ++e) v05[e] = fma(0.5 * h, l1[e], v[e]);
    double k1v[E], s05v[E];
    L.template pass_each<true, true>(v05, [&](int e, const double (&Ae)[NC + 1], const double (&De)[NC]) {
        double k0 = kdiag(L, e, v05[e], Ae[NC]), k1 = k0, s = 0.0;
        UNROLL for (int qq = 0; qq < NC; ++qq) {
            k0 = fma(L.p[0][qq], Ae[qq], k0);
            k1 = fma(L.p[2][qq], Ae[qq], k1);
            s = fma(L.q[1][qq], De[qq], s);
        }
        k1v[e] = -k1;                                  // -K1 v05 (the sign rides on the FMA that consumes it)
        s05v[e] = s;                                   // S05 v05
        u[e] = fma(0.5 * h, s0u[e] - k0, u[e]);        // u + (h/2) kappa1,  kappa1 = S0 u - K0 v05
    });
    L.s_prescale(2, sc);
    L.s_pass_add(sc, u, k1v, rhs);                                                             // S1 (u + (h/2) kappa1) - K1 v05
    double k2[E];
    solve<JT>(L, sc, J, h, rhs, k2);
    UNROLL for (int e = 0; e < E; ++e) u[e] = fma(0.5 * h, k2[e], u[e]);
    L.template pass_each<true, false>(u, [&](int e, const double (&Ae)[NC + 1], const double (&)[NC]) {
        double l2 = kdiag(L, e, u[e], Ae[NC]) + s05v[e];
        UNROLL for (int qq = 0; qq < NC; ++qq) l2 = fma(L.p[1][qq], Ae[qq], l2);
        v[e] = fma(0.5 * h, l1[e] + l2, v[e]);
    });
}

// src/StormerVerlet.jl:255-303 with the diagonal-W forcing of src/evalobjgrad.jl:862,882-888, fused with the five
// traces per control of adjoint_grad_calc! (src/evalobjgrad.jl:2578-2618):
//   T[q][0] = tr(vr0,Ha,lr05)  T[q][1] = tr(vi05,Hs,lr05)  T[q][2] = tr(vr,Ha,lr05)
//   T[q][3] = tr(vr,Hs,li)+tr(vr0,Hs,li0)                   T[q][4] = tr(vi05,Ha,li)+tr(vi05,Ha,li0)
// The group-reduced traces are left in shared memory at tred[q*5 + a] (written by lane 0 of the group, or with RS by their
// owners).
// DEFER: the lane's partial traces are returned in tpart[q*5 + a] instead of being reduced over the group (pipelined
// instantiations hand them to the gradient role).
// RS > 0: the traces are reduce-scattered over the group of RS lanes (group_scatter_sum), and `writer` only says that the lane
// belongs to a group.
// tcar: the lane-partial tr(vr0,Hs,li0) of this step on entry -- the tr(vr,Hs,li) of the step before (trace_hs before the first) --
// and tr(vr,Hs,li) on return, so that every boundary trace is summed once.
template <int JT, bool FORCING, class LaneT, bool DEFER = false, int RS = 0>
__device__ __forceinline__ void adjoint_step(LaneT &L, int J, double h, double (&mu)[LaneT::E], double (&nu)[LaneT::E],
                                             const double (&vr0)[LaneT::E], const double (&vi05)[LaneT::E],
                                             const double (&vr)[LaneT::E], double *tred, int GL, int gbase_lane, bool writer,
                                             double *tpart = nullptr, double *tcar = nullptr) {
    constexpr int E = LaneT::E, NC = LaneT::NC;
    // the group's reduced traces into tred: v holds A of the five traces per control, starting at trace a0
    auto reduce = [&](auto &v, auto a0c) {
        constexpr int A = std::extent_v<std::remove_reference_t<decltype(v)>> / NC, a0 = decltype(a0c)::value;
        if constexpr (RS > 0) {
            constexpr int K = ScatterShape<NC * A, RS>::K, H = ScatterShape<NC * A, RS>::H;
            const int lg = (threadIdx.x & 31) & (RS - 1);
            double sv[K];
            const int first = group_scatter_sum<NC * A, RS>(v, lg, sv);
            if (writer && (lg >> H) == 0) {
                UNROLL for (int i = 0; i < K; ++i) {
                    const int j = first + i;
                    if (j < NC * A) tred[(j / A) * 5 + a0 + j % A] = sv[i];
                }
            }
        } else {
            group_sum_n(v, GL, gbase_lane);
            if (writer) { UNROLL for (int qq = 0; qq < NC; ++qq) UNROLL for (int a = 0; a < A; ++a) tred[qq * 5 + a0 + a] = v[qq * A + a]; }
        }
    };
    double rhs[E], s05n[E], Tb[NC][2];
    typename LaneT::SC sc;
    L.sync_reset();
    L.s_prescale(0, sc);
    L.s_pass(sc, mu, rhs);
    UNROLL for (int qq = 0; qq < NC; ++qq) { Tb[qq][0] = 0.0; Tb[qq][1] = 0.0; }
    L.template pass_each<true, true>(nu, [&](int e, const double (&Ae)[NC + 1], const double (&De)[NC]) {
        double kk = kdiag(L, e, nu[e], Ae[NC]), s = 0.0;
        UNROLL for (int qq = 0; qq < NC; ++qq) {
            kk = fma(L.p[1][qq], Ae[qq], kk);
            s = fma(L.q[1][qq], De[qq], s);
            if (!tcar) Tb[qq][0] = fma(vr0[e], Ae[qq], Tb[qq][0]);      // tr(vr0, Hs, li0)
            Tb[qq][1] = fma(vi05[e], De[qq], Tb[qq][1]);     // tr(vi05, Ha, li0)
        }
        rhs[e] = (FORCING ? fma(L.w[e], vr0[e], rhs[e]) : rhs[e]) - kk;   // S0 mu + hr0 - K05 nu
        s05n[e] = s;                                         // S05 nu
    });
    double k2[E];
    solve<JT>(L, sc, J, h, rhs, k2);
    UNROLL for (int e = 0; e < E; ++e) mu[e] = fma(0.5 * h, k2[e], mu[e]);   // X = lr05
    double l2[E], r0[E], mu2[E];
    {
        double Ta[NC][3];
        UNROLL for (int qq = 0; qq < NC; ++qq) UNROLL for (int a = 0; a < 3; ++a) Ta[qq][a] = 0.0;
        L.template pass_each<true, true>(mu, [&](int e, const double (&Ae)[NC + 1], const double (&De)[NC]) {
            double k0 = kdiag(L, e, mu[e], Ae[NC]), k1 = k0, s = 0.0;
            UNROLL for (int qq = 0; qq < NC; ++qq) {
                k0 = fma(L.p[0][qq], Ae[qq], k0);
                k1 = fma(L.p[2][qq], Ae[qq], k1);
                s = fma(L.q[2][qq], De[qq], s);
                Ta[qq][0] = fma(vr0[e], De[qq], Ta[qq][0]);
                Ta[qq][1] = fma(vi05[e], Ae[qq], Ta[qq][1]);
                Ta[qq][2] = fma(vr[e], De[qq], Ta[qq][2]);
            }
            const double hi0 = FORCING ? L.w[e] * vi05[e] : 0.0;
            l2[e] = k0 + s05n[e] + hi0;                              // K0 X + S05 nu + hi0
            r0[e] = s05n[e] + k1 + hi0;                              // S05 nu + K1 X + hi1
            mu2[e] = fma(0.5 * h, FORCING ? fma(L.w[e], vr[e], s) : s, mu[e]);     // X + (h/2)(S1 X + hr1)
        });
        // the three traces that only involve lr05 = X are complete: reduce them now, overlapped with the next products
        double tv3[NC * 3];
        UNROLL for (int qq = 0; qq < NC; ++qq) UNROLL for (int a = 0; a < 3; ++a) tv3[qq * 3 + a] = Ta[qq][a];
        if constexpr (LaneSigned<LaneT>::value) { UNROLL for (int qq = 0; qq < NC; ++qq) { tv3[qq * 3] *= L.dsign(qq); tv3[qq * 3 + 2] *= L.dsign(qq); } }
        if constexpr (DEFER) { UNROLL for (int qq = 0; qq < NC; ++qq) UNROLL for (int a = 0; a < 3; ++a) tpart[qq * 5 + a] = tv3[qq * 3 + a]; }
        else reduce(tv3, std::integral_constant<int, 0>{});
    }
    L.s_prescale(1, sc);
    double l1[E];
    if constexpr (JT >= 0) {
        L.s_scale(sc, 0.5 * h);
        L.s_pass_add(sc, l2, r0, rhs);                                            // S05 nu + (h/2) S05 l2 + K1 X + hi1
        solve<JT, true>(L, sc, J, h, rhs, l1);
    } else {
        double tv[E];
        L.s_pass(sc, l2, tv);
        UNROLL for (int e = 0; e < E; ++e) rhs[e] = fma(0.5 * h, tv[e], r0[e]);
        solve<JT>(L, sc, J, h, rhs, l1);
    }
    UNROLL for (int e = 0; e < E; ++e) nu[e] = fma(0.5 * h, l2[e] + l1[e], nu[e]);
    L.template pass_each<true, true>(nu, [&](int e, const double (&Ae)[NC + 1], const double (&De)[NC]) {
        double kk = kdiag(L, e, nu[e], Ae[NC]);
        UNROLL for (int qq = 0; qq < NC; ++qq) {
            kk = fma(L.p[1][qq], Ae[qq], kk);
            Tb[qq][0] = fma(vr[e], Ae[qq], Tb[qq][0]);       // + tr(vr, Hs, li)
            Tb[qq][1] = fma(vi05[e], De[qq], Tb[qq][1]);     // + tr(vi05, Ha, li)
        }
        mu[e] = fma(-0.5 * h, kk, mu2[e]);                   // mu + (h/2) kappa1, kappa1 = S1 X - K05 nu + hr1
    });
    {
        double tv2[NC * 2];
        UNROLL for (int qq = 0; qq < NC; ++qq) UNROLL for (int a = 0; a < 2; ++a) tv2[qq * 2 + a] = Tb[qq][a];
        if (tcar) { UNROLL for (int qq = 0; qq < NC; ++qq) { tv2[qq * 2] += tcar[qq]; tcar[qq] = Tb[qq][0]; } }
        if constexpr (LaneSigned<LaneT>::value) { UNROLL for (int qq = 0; qq < NC; ++qq) tv2[qq * 2 + 1] *= L.dsign(qq); }
        if constexpr (DEFER) { UNROLL for (int qq = 0; qq < NC; ++qq) UNROLL for (int a = 0; a < 2; ++a) tpart[qq * 5 + 3 + a] = tv2[qq * 2 + a]; }
        else reduce(tv2, std::integral_constant<int, 3>{});
    }
    if constexpr (!DEFER) __syncwarp();
}

// Lane-partial tr(v, Hs_q, x) for every control q: the boundary trace adjoint_step carries from step to step (tcar).
template <class LaneT>
__device__ __forceinline__ void trace_hs(LaneT &L, const double (&v)[LaneT::E], const double (&x)[LaneT::E], double (&tc)[LaneT::NC]) {
    constexpr int NC = LaneT::NC;
    UNROLL for (int qq = 0; qq < NC; ++qq) tc[qq] = 0.0;
    L.sync_reset();
    L.template pass_each<true, false>(x, [&](int e, const double (&Ae)[NC + 1], const double (&)[NC]) {
        UNROLL for (int qq = 0; qq < NC; ++qq) tc[qq] = fma(v[e], Ae[qq], tc[qq]);
    });
}

// ---- pipelined instantiations: hand-over between the state role and the adjoint role of one CTA through two step counters per
// warp pair in shared memory (st.release.cta / ld.acquire.cta; an mbarrier try_wait version was no faster, and its wake-ups are
// coarser than the step they synchronise)
__device__ __forceinline__ void pipe_post(volatile int *cnt, int value, int lane) {      // after the warp's shared-memory traffic
    __syncwarp();
    if (lane == 0) asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(const_cast<int *>(cnt))), "r"(value) : "memory");
}
__device__ __forceinline__ void pipe_wait(volatile int *cnt, int at_least) {
    const unsigned a = (unsigned)__cvta_generic_to_shared(const_cast<int *>(cnt));
    int v;
    do { asm volatile("ld.acquire.cta.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); } while (v < at_least);
}
// SYNC 0: all threads of the CTA; 1: the calling warp; 2: the nthr threads of the gradient role (named barrier 2)
template <int SYNC>
__device__ __forceinline__ void role_sync(int nthr) {
    if constexpr (SYNC == 1) __syncwarp();
    else if constexpr (SYNC == 2) asm volatile("bar.sync 2, %0;" ::"r"(nthr) : "memory");
    else __syncthreads();
}

// Fill the control table for `nst` steps starting at time t: all threads of the CTA into the table at offset 0 (SYNC = 0), or the
// 32 lanes of the table warp (SYNC = 1) / the rnthr threads of the gradient role (SYNC = 2) into the table buffer at offset `toff`.
// XPT: one extra point, the midpoint of the step after the chunk (the shared boundary pass of the chunk's last forward step needs
// its p05): the same recurrence, so the same value as the next chunk's row 1.
template <int NC, int SYNC = 0, bool XPT = false>
__device__ void fill_table(const TrajParams &S, double *sm, double t, double dt, int nst, double dtknot, int toff = 0, int rtid = 0, int rnthr = 0) {
    if (SYNC == 0) { rtid = threadIdx.x; rnthr = blockDim.x; toff = 0; }
    double *times = sm + S.o_times + toff, *tabb = sm + S.o_tabb + toff, *tabph = sm + S.o_tabph + toff, *tabpq = sm + S.o_tabpq + toff;
    int *tabk = reinterpret_cast<int *>(sm + S.o_tabk + toff);
    const int npts = 2 * nst + 1 + XPT, Nfreq = S.P.Nfreq, D1 = S.A.D1;
    role_sync<SYNC>(rnthr);          // the previous chunk's table is no longer in use
    if (rtid == 0) {
        double tt = t;
        times[0] = tt;
        for (int i = 0; i < nst; ++i) {    // same recurrence as the reference: t + 0.5 dt, then t = t + dt
            times[2 * i + 1] = tt + 0.5 * dt;
            tt = tt + dt;
            times[2 * i + 2] = tt;
        }
        if (XPT) times[2 * nst + 1] = tt + 0.5 * dt;
    }
    role_sync<SYNC>(rnthr);
    const double width = 3.0 * dtknot;
    for (int idx = rtid; idx < npts * (NC * Nfreq + 1); idx += rnthr) {
        const int i = idx / (NC * Nfreq + 1), j = idx % (NC * Nfreq + 1);
        const double tt = times[i];
        if (j == NC * Nfreq) {             // src/bsplines.jl:224-253
            long long k = (long long)ceil(tt / dtknot + 2.0);
            k = k < 3 ? 3 : (k > D1 ? D1 : k);
            tabk[i] = (int)k;
            double tau = (tt - dtknot * ((double)k - 1.5)) / width;
            tabb[3 * i + 0] = 9.0 / 8 + 4.5 * tau + 4.5 * tau * tau;
            tau = (tt - dtknot * ((double)(k - 1) - 1.5)) / width;
            tabb[3 * i + 1] = 0.75 - 9.0 * tau * tau;
            tau = (tt - dtknot * ((double)(k - 2) - 1.5)) / width;
            tabb[3 * i + 2] = 9.0 / 8 - 4.5 * tau + 4.5 * tau * tau;
        } else {
            const int qq = j / Nfreq, fr = j % Nfreq;
            double sn, cs;
            sincos(S.P.cfreq[qq + NC * fr] * tt, &sn, &cs);
            tabph[2 * (i * NC * Nfreq + j)] = cs;
            tabph[2 * (i * NC * Nfreq + j) + 1] = sn;
        }
    }
    role_sync<SYNC>(rnthr);
    const double *pcof = sm + S.o_pcof;
    for (int idx = rtid; idx < npts * S.TPC * NC; idx += rnthr) {
        const int i = idx / (S.TPC * NC), rem = idx % (S.TPC * NC), tr = rem / NC, qq = rem % NC;
        const int k = tabk[i];
        const double b0 = tabb[3 * i], b1 = tabb[3 * i + 1], b2 = tabb[3 * i + 2];
        const double *pc = pcof + tr * S.NparS;
        double pv = 0.0, qv = 0.0;
        for (int fr = 0; fr < Nfreq; ++fr) {   // src/bsplines.jl:229-261
            const int off1 = 2 * qq * Nfreq * D1 + fr * 2 * D1 - 1, off2 = off1 + D1;
            const double fbs1 = pc[off1 + k] * b0 + pc[off1 + k - 1] * b1 + pc[off1 + k - 2] * b2;
            const double fbs2 = pc[off2 + k] * b0 + pc[off2 + k - 1] * b1 + pc[off2 + k - 2] * b2;
            const double cs = tabph[2 * (i * NC * Nfreq + qq * Nfreq + fr)], sn = tabph[2 * (i * NC * Nfreq + qq * Nfreq + fr) + 1];
            pv += fbs1 * cs - fbs2 * sn;
            qv += fbs1 * sn + fbs2 * cs;
        }
        tabpq[(i * S.TPC + tr) * 2 * NC + 2 * qq] = pv;
        tabpq[(i * S.TPC + tr) * 2 * NC + 2 * qq + 1] = qv;
    }
    role_sync<SYNC>(rnthr);
}

// Gradient scatter role: (control, frequency, alpha) with a 3-knot register window.
struct Updater {
    bool on;
    int uq, uf, ua, gbase, kw;
    double acc0, acc1, acc2;
};

// One step's contribution to the gradient windows of this lane's roles (src/evalobjgrad.jl:2578-2618, bsplines.jl:321-381).
// Time points in decreasing order: t0 (table row 2ls), t0 + dt/2 (2ls+1), t0 + dt (2ls+2).
template <int NC, int UPL>
__device__ __forceinline__ void grad_scatter(Updater (&U)[UPL], double *gsm, const double *tred, const double *tabb, const double *tabph,
                                             const int *tabk, int ls, int Nfreq) {
    UNROLL for (int j = 0; j < UPL; ++j) {
        if (U[j].on) {
            double Tq[5];
            UNROLL for (int a = 0; a < 5; ++a) Tq[a] = tred[U[j].uq * 5 + a];
            UNROLL for (int tp = 0; tp < 3; ++tp) {
                const int i = 2 * ls + tp;
                const double Pc = tp == 1 ? Tq[3] : -Tq[1];
                const double Qc = tp == 0 ? -Tq[0] : (tp == 1 ? -Tq[4] : -Tq[2]);
                const int ph = 2 * (i * NC * Nfreq + U[j].uq * Nfreq + U[j].uf);
                const double cs = tabph[ph], sn = tabph[ph + 1];
                const double X = U[j].ua == 0 ? Pc * cs + Qc * sn : Qc * cs - Pc * sn;
                const int k = tabk[i];
                while (U[j].kw > k) { gsm[U[j].gbase + U[j].kw] += U[j].acc0; U[j].acc0 = U[j].acc1; U[j].acc1 = U[j].acc2; U[j].acc2 = 0.0; --U[j].kw; }
                U[j].acc0 = fma(tabb[3 * i], X, U[j].acc0);
                U[j].acc1 = fma(tabb[3 * i + 1], X, U[j].acc1);
                U[j].acc2 = fma(tabb[3 * i + 2], X, U[j].acc2);
            }
        }
    }
    __syncwarp();                        // the roles have read tred before anything overwrites it
}

// OBJ = 1: objFuncType 2/3 — a second adjoint set without forcing gives the infidelity-only gradient
// (src/evalobjgrad.jl:848-855, :905-918; step_no_forcing! src/StormerVerlet.jl:365-406).
//
// PIPE = 1 (latency instantiations, small launches): the CTA has 3 NW warps in three ROLES with the same lane layout, plus one
// table warp that computes the control tables (B-spline values, carrier phases, p_q, q_q of the next TRAJ_CH steps) ahead of all of
// them into a ring of TRAJ_TABS buffers, so no role ever stops for the table (measured: ~20% of a lone trajectory's time).  The state
// role runs the forward sweep and then recomputes the states backwards, handing (vr0, vi05, vr) of every step to its twin lane in
// the adjoint role through a TRAJ_RING-slot ring in shared memory (two step counters per warp pair); the adjoint role runs the
// adjoint steps one or more steps behind and hands its lane-partial traces to the gradient role, which does the group
// reductions and the B-spline scatter.  A single trajectory has no other parallelism beyond its n x m elements: the recomputed
// state does not depend on the adjoint, and the gradient accumulation feeds nothing back, so the backward sweep costs the
// longest of the three per-step chains instead of their sum.  Same arithmetic on the same values as PIPE = 0.
//
// SEG = true (time-parallel evaluation, jq_seg.cu): every CTA sweeps ONE segment of the time axis in one of the modes of SegArgs --
// forward from a block of unit vectors or from the true boundary state, adjoint without forcing from unit vectors, or the backward
// sweep between two known boundaries -- with the same steppers on the same lane layout.
//
// HIST = true (segment sweeps of the history VJP, jq_seg_vjp_launch with a SegHist): mode 2 also saves the states, mode 7 sweeps the
// particular solutions with the cotangent jumps, mode 5 applies the jumps to the second adjoint set.  Separate instantiations, so that
// the ones kernel 7's evaluation and the final-state VJP run keep their code.
template <class LaneT, int UPL, int MINB = 1, int JT = 0, int OBJ = 0, int GLT = 0, int NW = TRAJ_WARPS, int PIPE_ = 0, bool SEG = false,
          bool HIST = false>
__global__ void __launch_bounds__((PIPE_ == 1 ? 3 * NW + 1 : PIPE_ == 2 ? 2 * NW : NW) * 32, MINB) jq_traj_kernel(const __grid_constant__ TrajParams S) {
    constexpr int E = LaneT::E, NC = LaneT::NC;
    constexpr bool PIPE = PIPE_ != 0;
    static_assert(!SEG || PIPE_ == 0, "segment sweeps: plain layout");
    static_assert(!HIST || SEG, "history paths: segment sweeps only");
    // PIPE_ = 1: roles state | adjoint | gradient + one table warp; PIPE_ = 2 (shapes whose register budget allows 8 warps only):
    // state and adjoint in one role, and the gradient role also produces the control tables in the slack of its own steps
    constexpr int NR = PIPE_ == 1 ? 3 : PIPE_ == 2 ? 2 : 1, R_ADJ = PIPE_ == 1 ? 1 : 0, R_GRAD = NR - 1;
    extern __shared__ double sm[];
    const DevProblem &P = S.P;
    const LaunchArgs &A = S.A;
    Geo g;
    g.lane = threadIdx.x & 31; g.warp = threadIdx.x >> 5;
    const int role = PIPE ? g.warp / NW : 0;                 // 0: state role (and everything when PIPE = 0), 1: adjoint role, 2: gradient role, 3: table warp
    const int pwarp = g.warp;                                // warp in the CTA
    if constexpr (PIPE) g.warp = role < NR ? g.warp - role * NW : 0;
    const int rtid = PIPE ? (int)threadIdx.x - role * NW * 32 : (int)threadIdx.x, rnthr = PIPE ? NW * 32 : (int)blockDim.x;
    const int GL = GLT > 0 ? GLT : S.GL;       // GLT: group size known at compile time (reductions unroll and overlap)
    g.lg = g.lane % GL;
    const int gw = g.lane / GL;                              // group inside the warp; lanes past GPW*GL are idle
    const bool lane_on = gw < S.GPW;
    g.group = g.warp * S.GPW + (lane_on ? gw : 0);
    g.tloc = g.group / S.GPT; g.gi = g.group % S.GPT;
    const int gbase_lane = (lane_on ? gw : 0) * GL;          // first lane of this group
    // SEG: the CTA's mode and segment, its first sub-trajectory; sub-trajectory = (block of unit vectors, trajectory)
    int smode = 0, seg = 0, sq0 = 0, sper = 0;
    if constexpr (SEG) {
        int b = blockIdx.x;
        const int part = b >= A.seg.ctas0 ? 1 : 0;
        if (part) b -= A.seg.ctas0;
        smode = A.seg.mode[part];
        if constexpr (HIST) { if (S.H.mode2 != 0 && (int)blockIdx.x >= S.H.ctas1) { smode = S.H.mode2; b = (int)blockIdx.x - S.H.ctas1; } }
        sper = (smode == 1 || smode == 3) ? ((2 * P.n + P.m - 1) / P.m) * A.ntraj : A.ntraj;
        const int cps = (sper + S.TPC - 1) / S.TPC;
        seg = A.seg.seg_lo + b / cps; sq0 = (b % cps) * S.TPC;
        // refinement pass of the defect sweep: nothing to do when the previous pass left no defect above the tolerance
        if (smode == 6 && A.seg.pass > 0 && A.seg.flags[A.seg.pass - 1] == 0) return;
    }
    auto cta_traj = [&](int tloc) -> int {       // trajectory (candidate x sample) of the CTA's tloc-th resident one, -1 if none
        if constexpr (SEG) { const int q = sq0 + tloc; return q < sper ? q % A.ntraj : -1; }
        else { const int tg = blockIdx.x * S.TPC + tloc; return tg < A.ntraj ? tg : -1; }
    };
    const int traj_ = g.tloc < S.TPC ? cta_traj(g.tloc) : -1;
    const int traj = traj_ < 0 ? 0 : traj_;
    const int sblk = SEG && traj_ >= 0 ? (sq0 + g.tloc) / A.ntraj : 0;       // SEG: which block of m unit vectors
    const bool live_t = lane_on && traj_ >= 0;                          // dead groups compute on zeros and write nothing
    const int s = live_t ? traj % A.nsamples : 0;
    const int n = P.n, m = P.m, Npar = A.Npar, D1 = A.D1, Nfreq = P.Nfreq, J = P.J;
    const double tinv = 1.0 / P.T, dtknot = P.T / (D1 - 2);
    const int tl = g.tloc < S.TPC ? g.tloc : 0;              // table row used by this group

    LaneT L;
    L.setup(S, sm, g);
    L.sGL = GL; L.sbase = gbase_lane; L.stol = P.tol;
    bool ok[E];
    UNROLL for (int e = 0; e < E; ++e) {
        const int r = L.row(e);
        ok[e] = live_t && r < n && L.col(e) < m;
        L.d0[e] = ok[e] ? S.plan_d0[r] + (A.shift ? A.shift[(size_t)s * n + r] : 0.0) : 0.0;
        L.w[e] = ok[e] ? S.plan_w[r] * tinv : 0.0;
    }
    // stage this CTA's pcof vectors and zero the per-group gradient accumulators
    for (int idx = threadIdx.x; idx < S.TPC * Npar; idx += blockDim.x) {
        const int tr = idx / Npar, k = idx % Npar, tg = cta_traj(tr);
        sm[S.o_pcof + tr * S.NparS + k] = tg >= 0 ? A.pcof[(size_t)(tg / A.nsamples) * A.pstride + k] : 0.0;
    }
    for (int idx = threadIdx.x; idx < S.ngroups * Npar; idx += blockDim.x) { sm[S.o_gsm + idx] = 0.0; if (OBJ) sm[S.o_gsm2 + idx] = 0.0; }
    volatile int *pcnt = reinterpret_cast<volatile int *>(sm + S.o_cnt);     // [warp][states produced, consumed, traces produced, consumed]
    volatile int *cdone = pcnt + NW * 4, *tabs_ready = cdone + NR * NW;        // chunks finished per consumer warp; table chunks produced
    const int nch = (int)((P.nsteps + TRAJ_CH - 1) / TRAJ_CH);                // global chunk ids: forward c, backward nch + c
    if constexpr (PIPE) {
        if (threadIdx.x < NW * 4) pcnt[threadIdx.x] = 0;
        if (threadIdx.x < NR * NW) cdone[threadIdx.x] = threadIdx.x < NW ? 0 : nch;     // only the state role consumes forward tables
        if (threadIdx.x == 0) *tabs_ready = 0;
        __syncthreads();                                     // pcof staged and counters cleared before the roles part ways
    }
    // table production (PIPE): chunk k of the forward (k < nch) or backward sweep into buffer k % TRAJ_TABS, by the table warp
    // (PIPE_ = 1) or by all warps of the gradient role (PIPE_ = 2), once every consumer warp has finished chunk k - TRAJ_TABS
    double ptt = 0.0, pdt = P.T / (double)P.nsteps;
    int kprod = 0;
    const int ktotal = A.evaladjoint ? 2 * nch : nch;
    auto produce_table = [&]() {
        if constexpr (!PIPE) return;
        const int k = kprod++;
        if (k == nch) { ptt = P.T; pdt = -pdt; }
        const long long s0 = (long long)(k < nch ? k : k - nch) * TRAJ_CH;
        const int nst = (int)((P.nsteps - s0) < TRAJ_CH ? (P.nsteps - s0) : TRAJ_CH);
        constexpr int NCONS = PIPE_ == 1 ? NR * NW : NW;                              // PIPE_ = 2: the gradient role trails its own tables by construction
        if (g.lane < NCONS) pipe_wait(cdone + g.lane, k - TRAJ_TABS + 1);             // buffer k % TRAJ_TABS no longer in use
        __syncwarp();
        if constexpr (PIPE_ == 1) fill_table<NC, 1>(S, sm, ptt, pdt, nst, dtknot, (k % TRAJ_TABS) * S.tab_role_stride, g.lane, 32);
        else if constexpr (PIPE_ == 2) fill_table<NC, 2>(S, sm, ptt, pdt, nst, dtknot, (k % TRAJ_TABS) * S.tab_role_stride, rtid, rnthr);
        for (int i = 0; i < nst; ++i) ptt = ptt + pdt;                                // the consumers' own recurrence
        if (PIPE_ == 1 || g.warp == 0) pipe_post(tabs_ready, k + 1, g.lane);
    };
    if constexpr (PIPE_ == 1) {
        if (role == NR) {               // table warp: runs ahead of every role; the roles meet at named barrier 1, which does not count it
            while (kprod < ktotal) produce_table();
            return;
        }
    }
    if constexpr (PIPE_ == 2) {
        if (role == R_GRAD) { while (kprod < nch) produce_table(); }                  // forward sweep: the gradient role has nothing else to do
    }
    // every thread of the CTA (PIPE: of the trajectory roles)
    auto consumer_sync = [&]() {
        if constexpr (PIPE) asm volatile("bar.sync 1, %0;" ::"r"(NR * NW * 32) : "memory");
        else __syncthreads();
    };

    // SEG: steps [k0, k1) of the time axis
    long long k0 = 0, k1 = P.nsteps;
    if constexpr (SEG) { k0 = (long long)seg * P.nsteps / A.seg.nseg; k1 = (long long)(seg + 1) * P.nsteps / A.seg.nseg; }
    const long long nstl = k1 - k0;
    const size_t nm = (size_t)n * m, sbt = SEG ? ((size_t)seg * A.ntraj + traj) : 0;     // SEG: (segment, trajectory) index of the outputs
    double vr[E], vi[E], vi05[E];
    UNROLL for (int e = 0; e < E; ++e) {
        const size_t ix = L.row(e) + (size_t)n * L.col(e);
        const size_t bx = L.row(e) + (size_t)2 * n * L.col(e);           // SEG boundary vectors: [column][u rows, then v rows]
        if constexpr (!SEG) { vr[e] = ok[e] ? P.uinit[ix] : 0.0; vi[e] = 0.0; }
        else {
            const int j = sblk * m + L.col(e);                           // unit vector of this column: u_j (j < n) or v_{j-n}
            if (smode == 1) { vr[e] = ok[e] && L.row(e) == j ? 1.0 : 0.0; vi[e] = ok[e] && L.row(e) + n == j ? 1.0 : 0.0; }
            else if (smode == 2) { vr[e] = ok[e] ? A.seg.X[sbt * 2 * nm + bx] : 0.0; vi[e] = ok[e] ? A.seg.X[sbt * 2 * nm + bx + n] : 0.0; }
            else if (smode >= 4 && (!HIST || smode != 7)) {              // backward sweeps: Xb = X + J' Eta at the segment end (6: X itself)
                const size_t b1 = (sbt + A.ntraj) * 2 * nm + bx;
                const bool plain = smode == 6 && A.seg.pass == 0;       // first defect sweep: from the forward boundary state
                vr[e] = ok[e] ? A.seg.X[b1] - (plain ? 0.0 : A.seg.Eta[b1 + n]) : 0.0;
                vi[e] = ok[e] ? A.seg.X[b1 + n] + (plain ? 0.0 : A.seg.Eta[b1]) : 0.0;
            }
            else { vr[e] = 0.0; vi[e] = 0.0; }
        }
        vi05[e] = 0.0;
    }
    const double *tabpq = sm + S.o_tabpq;                     // PIPE: re-pointed at the chunk's table buffer

#define LOAD_LEVELS(ls)                                                                                              \
    UNROLL for (int qq = 0; qq < NC; ++qq) {                                                                         \
        L.p[0][qq] = L.p[2][qq]; L.q[0][qq] = L.q[2][qq];                                                            \
        const double *r1 = tabpq + ((2 * (ls) + 1) * S.TPC + tl) * 2 * NC, *r2 = tabpq + ((2 * (ls) + 2) * S.TPC + tl) * 2 * NC; \
        L.p[1][qq] = r1[2 * qq]; L.q[1][qq] = r1[2 * qq + 1];                                                        \
        L.p[2][qq] = r2[2 * qq]; L.q[2][qq] = r2[2 * qq + 1];                                                        \
        if constexpr (LaneSigned<LaneT>::value) { L.q[1][qq] *= L.dsign(qq); L.q[2][qq] *= L.dsign(qq); }            \
    }
#define LOAD_LEVEL0()                                                                                                \
    UNROLL for (int qq = 0; qq < NC; ++qq) {                                                                         \
        L.p[2][qq] = tabpq[tl * 2 * NC + 2 * qq]; L.q[2][qq] = tabpq[tl * 2 * NC + 2 * qq + 1];                      \
        if constexpr (LaneSigned<LaneT>::value) L.q[2][qq] *= L.dsign(qq);                                           \
    }

    // ------------------------------------------------------------ forward sweep (src/evalobjgrad.jl:698-753)
    double dt = P.T / (double)P.nsteps, t = 0.0, pen = 0.0;
    if constexpr (SEG) t = A.seg.times[seg];
    // forward history (jq_eval_forward; src/evalobjgrad.jl:2847-2849): Re = vr, Im = -vi after every save_every-th step
    const bool hist = A.hist_r != nullptr && (!HIST || smode == 2);
    size_t hpos = hist ? (size_t)(live_t ? traj : 0) * A.nsave * ((size_t)n * m) : 0;      // start of the next saved block
    int hcount = hist ? A.save_every : 0;                                                // steps until the next save
    if constexpr (HIST) {
        // mode 2: the saves in (k0, k1] -- the first is j1 = k0 / save_every + 1 -- and block 0 in segment 0, written by one trajectory
        // per history row; the others start at hcount = 0, which the countdown never reaches again
        if (hist) {
            const long long q0 = (long long)seg * P.nsteps / A.seg.nseg, j1 = q0 / A.save_every + 1;
            hpos = ((size_t)(traj / S.H.hist_nc) * A.nsave + (seg == 0 ? 0 : j1)) * ((size_t)n * m);
            hcount = live_t && traj % S.H.hist_nc == 0 ? (int)(j1 * A.save_every - q0) : 0;
        }
    }
    auto save_state = [&]() {
        UNROLL for (int e = 0; e < E; ++e)
            if (ok[e]) {
                const size_t ix = hpos + L.row(e) + (size_t)n * L.col(e);
                A.hist_r[ix] = vr[e]; A.hist_i[ix] = -vi[e];
            }
        hpos += (size_t)n * m;
    };
    if (hist && (!HIST || (seg == 0 && hcount != 0))) save_state();
    // two copies of the loop (generic lambda, both inlined): the evaluation path carries no per-step history test
    // SHARE (weighted layouts, not pipelined): a step's last product pass also gives the next step's boundary products (bp, with
    // the next p05 from the table row past the step: the table carries one extra point for the last step of a chunk).  The penalty
    // (penalf2aTrap + penalf2a), the sum over the steps of w.*(vr_k^2 + vr_k+1^2 + 2 vi05^2), is then evaluated as twice
    // (w.*vr_0^2 / 2 + sum of w.*(vr_k+1^2 + vi05^2) - w.*vr_N^2 / 2), so that every state is squared once.  The other layouts keep
    // the step-by-step form: several of them spill, and the end terms would add spill loads to their forward loops.
    constexpr bool SHARE = LaneWeighted<LaneT>::value && !PIPE;
    auto forward_sweep = [&](auto with_hist) {
        if constexpr (SHARE) { UNROLL for (int e = 0; e < E; ++e) pen = fma(0.5 * L.w[e], vr[e] * vr[e], pen); }
        double bp[SHARE ? 2 : 1][SHARE ? E : 1];
        for (long long s0 = 0; s0 < (SEG ? nstl : P.nsteps); s0 += TRAJ_CH) {
            const int nst = (int)(((SEG ? nstl : P.nsteps) - s0) < TRAJ_CH ? ((SEG ? nstl : P.nsteps) - s0) : TRAJ_CH);
            if constexpr (PIPE) {
                const int gk = (int)(s0 / TRAJ_CH);
                pipe_wait(tabs_ready, gk + 1);
                tabpq = sm + S.o_tabpq + (gk % TRAJ_TABS) * S.tab_role_stride;
            } else fill_table<NC, 0, SHARE>(S, sm, t, dt, nst, dtknot);
            LOAD_LEVEL0();
            if constexpr (SHARE) {
                if (s0 == 0) {
                    double p05[NC];
                    UNROLL for (int qq = 0; qq < NC; ++qq) p05[qq] = tabpq[(S.TPC + tl) * 2 * NC + 2 * qq];
                    step_open(L, vr, p05, L.q[2], bp);
                }
            }
            for (int ls = 0; ls < nst; ++ls) {
                LOAD_LEVELS(ls);
                if constexpr (SHARE) {
                    double pn[NC];
                    UNROLL for (int qq = 0; qq < NC; ++qq) pn[qq] = tabpq[((2 * ls + 3) * S.TPC + tl) * 2 * NC + 2 * qq];
                    state_step_w<JT, true>(L, J, dt, vr, vi, vi05, bp, pn);
                    UNROLL for (int e = 0; e < E; ++e) pen = fma(L.w[e], fma(vr[e], vr[e], vi05[e] * vi05[e]), pen);
                } else {
                    UNROLL for (int e = 0; e < E; ++e) pen = fma(L.w[e], vr[e] * vr[e], pen);                              // penalf2aTrap
                    state_step<JT>(L, J, dt, vr, vi, vi05);
                    UNROLL for (int e = 0; e < E; ++e) pen = fma(L.w[e], vr[e] * vr[e] + 2.0 * vi05[e] * vi05[e], pen);   // penalf2a
                }
                t = t + dt;
                if constexpr (decltype(with_hist)::value) { if (--hcount == 0) { hcount = A.save_every; save_state(); } }
            }
            if constexpr (PIPE) pipe_post(cdone + pwarp, (int)(s0 / TRAJ_CH) + 1, g.lane);
        }
        if constexpr (SHARE) {
            UNROLL for (int e = 0; e < E; ++e) pen = fma(-0.5 * L.w[e], vr[e] * vr[e], pen);
            pen *= 2.0;
        }
    };
    double *red = sm + S.o_red;
    double lr[E], li[E], vr0[E];
    if constexpr (SEG) {
        if (smode <= 2) {
            if constexpr (HIST && OBJ == 0) { if (hist) forward_sweep(std::true_type{}); else forward_sweep(std::false_type{}); }
            else forward_sweep(std::false_type{});
            if (smode == 1) {                                // column j of the segment's propagator
                UNROLL for (int e = 0; e < E; ++e) {
                    const int j = sblk * m + L.col(e);
                    if (ok[e] && j < 2 * n) {
                        double *o = A.seg.Phi + (sbt * A.seg.ld + j) * A.seg.ld + L.row(e);
                        o[0] = vr[e]; o[n] = vi[e];
                    }
                }
                return;
            }
            double pv[1] = {pen};
            group_sum_n(pv, GL, gbase_lane);
            if (lane_on && g.lg == 0) red[g.group * 4 + 2] = pv[0];
            __syncthreads();
            if (live_t && g.gi == 0 && g.lg == 0) {
                double pens = 0.0;
                for (int j = 0; j < S.GPT; ++j) pens += red[(tl * S.GPT + j) * 4 + 2];
                if (!HIST || A.seg.penpart) A.seg.penpart[sbt] = 0.5 * dt * pens;      // the history VJP has no penalty shares
            }
            return;
        }
        // backward modes: terminal adjoint = unit vectors (3), zero (4) or the boundary value Lam[seg + 1] (5)
        UNROLL for (int e = 0; e < E; ++e) {
            const size_t bx = L.row(e) + (size_t)2 * n * L.col(e);
            const int j = sblk * m + L.col(e);
            if (smode == 3) { lr[e] = ok[e] && L.row(e) == j ? 1.0 : 0.0; li[e] = ok[e] && L.row(e) + n == j ? 1.0 : 0.0; }
            else if (smode == 5) { lr[e] = ok[e] ? A.seg.Lam[(sbt + A.ntraj) * 2 * nm + bx] : 0.0; li[e] = ok[e] ? A.seg.Lam[(sbt + A.ntraj) * 2 * nm + bx + n] : 0.0; }
            else { lr[e] = 0.0; li[e] = 0.0; }
        }
    } else {
    if (PIPE && role != 0) {}                                // the adjoint and gradient roles wait at the barrier below
    else if (hist) forward_sweep(std::true_type{});
    else forward_sweep(std::false_type{});
    // infidelity (pFidType 2) and leak: group partials -> shared -> per-trajectory sums in group order
    {
        double re = 0.0, im = 0.0;
        UNROLL for (int e = 0; e < E; ++e) {
            const size_t ix = L.row(e) + (size_t)n * L.col(e);
            const double tr_ = ok[e] ? P.vtr[ix] : 0.0, ti_ = ok[e] ? P.vti[ix] : 0.0;
            re += vr[e] * tr_ - vi[e] * ti_;
            im += vr[e] * ti_ + vi[e] * tr_;
        }
        double rip[3] = {re, im, pen};
        group_sum_n(rip, GL, gbase_lane);
        re = rip[0]; im = rip[1]; pen = rip[2];
        consumer_sync();
        if (lane_on && g.lg == 0 && role == 0) { red[g.group * 4] = re; red[g.group * 4 + 1] = im; red[g.group * 4 + 2] = pen; }
        consumer_sync();
    }
    double rs = 0.0, is = 0.0, pens = 0.0;
    for (int j = 0; j < S.GPT; ++j) {
        const int gg = tl * S.GPT + j;
        rs += red[gg * 4]; is += red[gg * 4 + 1]; pens += red[gg * 4 + 2];
    }
    rs /= m; is /= m;
    // primary objective by pFidType (src/evalobjgrad.jl:755-763) with s = rs + i is: 1: 1 + |s|^2 - 2 Re(s e^{-i phase});
    // 2: 1 - |s|^2; 3, 4: 1 - tracefidreal(v, e^{i phase} Vtg) = 1 - (rs cos(phase) - is sin(phase)).  pFidType 3 carries the
    // phase as the last entry of the pcof vector (:591-596).
    const int pfid = P.pFidType;
    double sph = 0.0, cph = 1.0;
    if (pfid != 2) sincos(pfid == 3 ? A.pcof[(size_t)((live_t ? traj : 0) / A.nsamples) * A.pstride + Npar] : P.globalPhase, &sph, &cph);
    const double abs2 = rs * rs + is * is;
    const double infid = pfid == 1 ? 1.0 + abs2 - 2.0 * (rs * cph + is * sph) : pfid == 2 ? 1.0 - abs2 : 1.0 - (rs * cph - is * sph);
    if (live_t && g.gi == 0 && g.lg == 0 && role == 0) {
        double *o = A.scal + (size_t)traj * 4;
        o[0] = infid; o[1] = 0.5 * dt * pens; o[2] = 1.0 - abs2; o[3] = 0.0;   // w already carries 1/T; traceInfidelity = 1 - |s|^2 (:792)
        if (pfid == 3 && A.evaladjoint) {        // gradient with respect to the global phase (:923-945), last entry of both gradients
            const double pg = rs * sph + is * cph;
            A.grad[(size_t)traj * A.gstride + Npar] = pg;
            if (OBJ) A.infidgrad[(size_t)traj * A.gstride + Npar] = pg;
        }
    }
    if (!A.evaladjoint) return;

    // ------------------------------------------------------------ backward sweep (src/evalobjgrad.jl:810-921)
    // terminal condition (init_adjoint!, :2026-2059): types 1 and 2 share the formula, type 1 on scomplex0 = e^{i phase} - s (:825-826);
    // types 3, 4: lambda_r = Re(rot) / 2N, lambda_i = -Im(rot) / 2N, rot = e^{i phase} (Vtr + i Vti)
    const double rs_ = pfid == 1 ? cph - rs : rs, is_ = pfid == 1 ? sph - is : is;
    UNROLL for (int e = 0; e < E; ++e) {
        const size_t ix = L.row(e) + (size_t)n * L.col(e);
        const double tr_ = ok[e] ? P.vtr[ix] : 0.0, ti_ = ok[e] ? P.vti[ix] : 0.0;
        if (pfid <= 2) {
            lr[e] = (rs_ * tr_ + is_ * ti_) / m;     // init_adjoint!, src/evalobjgrad.jl:2029-2042
            li[e] = (is_ * tr_ - rs_ * ti_) / m;
        } else {
            lr[e] = 0.5 * (cph * tr_ - sph * ti_) / m;
            li[e] = -0.5 * (sph * tr_ + cph * ti_) / m;
        }
    }
    }   // !SEG
    double lrn[OBJ ? E : 1], lin[OBJ ? E : 1];
    if constexpr (OBJ != 0) {
        UNROLL for (int e = 0; e < E; ++e) { lrn[e] = lr[e]; lin[e] = li[e]; }
        if constexpr (SEG) {                 // second adjoint set (no forcing): its own boundary values Lam2[seg + 1]
            if (smode == 5) {
                UNROLL for (int e = 0; e < E; ++e) {
                    const size_t b1 = (sbt + A.ntraj) * 2 * nm + L.row(e) + (size_t)2 * n * L.col(e);
                    lrn[e] = ok[e] ? A.seg.Lam2[b1] : 0.0; lin[e] = ok[e] ? A.seg.Lam2[b1 + n] : 0.0;
                }
            }
        }
    }
    // gradient scatter roles: role u = lg + j*GL < NU owns (control, frequency, alpha)
    const int NU = NC * Nfreq * 2;
    Updater U[UPL], U2[OBJ ? UPL : 1];
    UNROLL for (int j = 0; j < UPL; ++j) {
        const int u = g.lg + j * GL;
        U[j].on = lane_on && u < NU && (!PIPE || role == R_GRAD);
        U[j].uq = U[j].on ? u / (2 * Nfreq) : 0;
        U[j].uf = U[j].on ? (u >> 1) % Nfreq : 0;
        U[j].ua = u & 1;
        U[j].gbase = 2 * U[j].uq * Nfreq * D1 + U[j].uf * 2 * D1 + U[j].ua * D1 - 1;
        U[j].kw = D1; U[j].acc0 = 0.0; U[j].acc1 = 0.0; U[j].acc2 = 0.0;
        if constexpr (OBJ != 0) U2[j] = U[j];
    }
    double *gsm = sm + S.o_gsm + g.group * Npar;
    double *tred = sm + S.o_tred + g.group * (NC * 5);
    double *gsm2 = sm + S.o_gsm2 + g.group * Npar;
    const double *tabb = sm + S.o_tabb, *tabph = sm + S.o_tabph;
    const int *tabk = reinterpret_cast<const int *>(sm + S.o_tabk);

    t = P.T;
    if constexpr (SEG) t = A.seg.times[A.seg.nseg + seg];
    dt = -dt;
    if constexpr (!PIPE) {
        // weighted layouts carry the boundary trace from step to step; in the other layouts' backward loops, several of which
        // spill, the carried sums would be more live registers
        constexpr bool CARRY = LaneWeighted<LaneT>::value;
        // the same layouts reduce-scatter the traces when the group size is known at compile time
        constexpr int RSG = CARRY && GLT > 0 ? GLT : 0;
        double tcar[NC], tcar2[OBJ ? NC : 1];
        if constexpr (CARRY) {
            trace_hs(L, vr, li, tcar);
            if constexpr (OBJ != 0) trace_hs(L, vr, lin, tcar2);
        }
        // history VJP (modes 5 and 7): the cotangent of save j = K / save_every >= 1 jumps into the unforced set after the iteration
        // that recomputes state K; the block of the next save is prefetched into L1 then, so that its loads stay off the critical path
        // of the steps in between.  Derived from the loop position (warp-uniform), so the sweeps carry no extra state.
        auto jump = [&](double (&xr)[E], double (&xi)[E], int K) -> bool {
            if (!(S.H.cot_r || S.H.cot_i) || K == 0 || K % A.save_every != 0) return false;      // save 0 is Uinit: no effect
            const size_t j = (size_t)(K / A.save_every), base = ((size_t)traj * A.nsave + j) * nm;
            UNROLL for (int e = 0; e < E; ++e)
                if (ok[e]) {
                    const size_t ix = base + L.row(e) + (size_t)n * L.col(e);
                    if (S.H.cot_r) { xr[e] = fma(-0.5, S.H.cot_r[ix], xr[e]); if (j > 1) asm volatile("prefetch.global.L1 [%0];" ::"l"(S.H.cot_r + ix - nm)); }
                    if (S.H.cot_i) { xi[e] = fma(0.5, S.H.cot_i[ix], xi[e]); if (j > 1) asm volatile("prefetch.global.L1 [%0];" ::"l"(S.H.cot_i + ix - nm)); }
                }
            return true;
        };
        for (long long s0 = 0; s0 < (SEG ? nstl : P.nsteps); s0 += TRAJ_CH) {
            const int nst = (int)(((SEG ? nstl : P.nsteps) - s0) < TRAJ_CH ? ((SEG ? nstl : P.nsteps) - s0) : TRAJ_CH);
            fill_table<NC>(S, sm, t, dt, nst, dtknot);
            LOAD_LEVEL0();
            for (int ls = 0; ls < nst; ++ls) {
                LOAD_LEVELS(ls);
                if constexpr (SEG) {
                    if (smode != 5) {        // no gradient: the traces are dead code (DEFER leaves them in registers nobody reads)
                        double tp[NC * 5];
                        if (smode == 3 || (HIST && smode == 7)) {
                            adjoint_step<JT, false, LaneT, true>(L, J, dt, lr, li, vr, vi05, vr, nullptr, GL, gbase_lane, false, tp);
                            if constexpr (HIST && OBJ == 0) { if (smode == 7) jump(lr, li, (int)(k1 - 1 - s0) - ls); }      // particular solution
                        }
                        else if (smode == 6) state_step<JT>(L, J, dt, vr, vi, vi05);
                        else {
                            UNROLL for (int e = 0; e < E; ++e) vr0[e] = vr[e];
                            state_step<JT>(L, J, dt, vr, vi, vi05);
                            adjoint_step<JT, true, LaneT, true>(L, J, dt, lr, li, vr0, vi05, vr, nullptr, GL, gbase_lane, false, tp);
                        }
                        t = t + dt;
                        continue;
                    }
                }
                UNROLL for (int e = 0; e < E; ++e) vr0[e] = vr[e];
                state_step<JT>(L, J, dt, vr, vi, vi05);
                adjoint_step<JT, true, LaneT, false, RSG>(L, J, dt, lr, li, vr0, vi05, vr, tred, GL, gbase_lane, RSG > 0 ? lane_on : lane_on && g.lg == 0, nullptr, CARRY ? tcar : nullptr);   // traces -> tred
                grad_scatter<NC, UPL>(U, gsm, tred, tabb, tabph, tabk, ls, Nfreq);
                if constexpr (OBJ != 0) {
                    adjoint_step<JT, false, LaneT, false, RSG>(L, J, dt, lrn, lin, vr0, vi05, vr, tred, GL, gbase_lane, RSG > 0 ? lane_on : lane_on && g.lg == 0, nullptr, CARRY ? tcar2 : nullptr);
                    grad_scatter<NC, UPL>(U2, gsm2, tred, tabb, tabph, tabk, ls, Nfreq);
                    if constexpr (HIST) {                    // after this step's traces; the carried trace is tr(vr, Hs, lin) of the jumped lin
                        if (jump(lrn, lin, (int)(k1 - 1 - s0) - ls)) { if constexpr (CARRY) trace_hs(L, vr, lin, tcar2); }
                    }
                }
                t = t + dt;
            }
        }
    } else {
        // hand-over ring: slot = step % TRAJ_RING; element k of (vr0, vi05, vr) of this lane at ring[(slot * 3E + k) * rnthr + rtid]
        double *ring = sm + S.o_ring;
        volatile int *produced = pcnt + g.warp * 4, *consumed = produced + 1, *tproduced = produced + 2, *tconsumed = produced + 3;
        double *tring = ring + (size_t)TRAJ_RING * 3 * E * rnthr;      // lane-partial traces: [slot][NC * 5][rnthr]
        int step = 0;
        for (long long s0 = 0; s0 < P.nsteps; s0 += TRAJ_CH) {
            const int nst = (int)((P.nsteps - s0) < TRAJ_CH ? (P.nsteps - s0) : TRAJ_CH);
            const int gk = nch + (int)(s0 / TRAJ_CH);
            if constexpr (PIPE_ == 2) {
                if (role == R_GRAD) { while (kprod < ktotal && kprod < gk + 3) produce_table(); }     // stay two chunks ahead of the own steps
            }
            pipe_wait(tabs_ready, gk + 1);
            {
                const int toff = (gk % TRAJ_TABS) * S.tab_role_stride;
                tabpq = sm + S.o_tabpq + toff; tabb = sm + S.o_tabb + toff; tabph = sm + S.o_tabph + toff;
                tabk = reinterpret_cast<const int *>(sm + S.o_tabk + toff);
            }
            LOAD_LEVEL0();
            for (int ls = 0; ls < nst; ++ls, ++step) {
                LOAD_LEVELS(ls);
                const int slot = step % TRAJ_RING;
                double *rs_ = ring + (size_t)slot * 3 * E * rnthr + rtid;
                double *ts_ = tring + (size_t)slot * NC * 5 * rnthr + rtid;
                if (role == 0) {
                    UNROLL for (int e = 0; e < E; ++e) vr0[e] = vr[e];
                    state_step<JT>(L, J, dt, vr, vi, vi05);
                    if constexpr (PIPE_ == 1) {
                        pipe_wait(consumed, step - TRAJ_RING + 1);                 // the slot's previous content has been read
                        UNROLL for (int e = 0; e < E; ++e) { rs_[e * rnthr] = vr0[e]; rs_[(E + e) * rnthr] = vi05[e]; rs_[(2 * E + e) * rnthr] = vr[e]; }
                        pipe_post(produced, step + 1, g.lane);
                    }
                }
                if (role == R_ADJ) {
                    if constexpr (PIPE_ == 1) {
                        pipe_wait(produced, step + 1);
                        UNROLL for (int e = 0; e < E; ++e) { vr0[e] = rs_[e * rnthr]; vi05[e] = rs_[(E + e) * rnthr]; vr[e] = rs_[(2 * E + e) * rnthr]; }
                        pipe_post(consumed, step + 1, g.lane);
                    }
                    double tp[NC * 5];
                    adjoint_step<JT, true, LaneT, true>(L, J, dt, lr, li, vr0, vi05, vr, nullptr, GL, gbase_lane, false, tp);
                    pipe_wait(tconsumed, step - TRAJ_RING + 1);
                    UNROLL for (int k = 0; k < NC * 5; ++k) ts_[k * rnthr] = tp[k];
                    pipe_post(tproduced, step + 1, g.lane);
                }
                if (role == R_GRAD) {
                    pipe_wait(tproduced, step + 1);
                    double tp[NC * 5];
                    UNROLL for (int k = 0; k < NC * 5; ++k) tp[k] = ts_[k * rnthr];
                    pipe_post(tconsumed, step + 1, g.lane);
                    group_sum_n(tp, GL, gbase_lane);
                    if (lane_on && g.lg == 0) { UNROLL for (int k = 0; k < NC * 5; ++k) tred[k] = tp[k]; }
                    __syncwarp();
                    grad_scatter<NC, UPL>(U, gsm, tred, tabb, tabph, tabk, ls, Nfreq);
                }
                t = t + dt;
            }
            pipe_post(cdone + pwarp, gk + 1, g.lane);
        }
    }
    UNROLL for (int j = 0; j < UPL; ++j) {
        if (U[j].on) { gsm[U[j].gbase + U[j].kw] += U[j].acc0; gsm[U[j].gbase + U[j].kw - 1] += U[j].acc1; gsm[U[j].gbase + U[j].kw - 2] += U[j].acc2; }
        if constexpr (OBJ != 0) if (U2[j].on) { gsm2[U2[j].gbase + U2[j].kw] += U2[j].acc0; gsm2[U2[j].gbase + U2[j].kw - 1] += U2[j].acc1; gsm2[U2[j].gbase + U2[j].kw - 2] += U2[j].acc2; }
    }
    if constexpr (SEG) {
        if (smode != 5) {                    // adjoint at the segment start: column j of Adj, or the particular solution
            UNROLL for (int e = 0; e < E; ++e) {
                const int j = sblk * m + L.col(e);
                if (smode == 3) {
                    if (ok[e] && j < 2 * n) { double *o = A.seg.Adj + (sbt * A.seg.ld + j) * A.seg.ld + L.row(e); o[0] = lr[e]; o[n] = li[e]; }
                } else if (ok[e]) {
                    const size_t b0 = sbt * 2 * nm + L.row(e) + (size_t)2 * n * L.col(e);
                    if (smode == 4 || (HIST && smode == 7)) { A.seg.cpart[b0] = lr[e]; A.seg.cpart[b0 + n] = li[e]; }
                    else {
                        // defect of the backward recomputation against the current boundary state X_p (+ J' Eta_p in a refinement pass)
                        const bool plain = A.seg.pass == 0;
                        const double du = vr[e] - (A.seg.X[b0] - (plain ? 0.0 : A.seg.Eta[b0 + n]));
                        const double dv = vi[e] - (A.seg.X[b0 + n] + (plain ? 0.0 : A.seg.Eta[b0]));
                        A.seg.dpart[b0] = dv; A.seg.dpart[b0 + n] = -du;
                        if (fabs(du) > A.seg.refine_tol || fabs(dv) > A.seg.refine_tol) A.seg.flags[A.seg.pass] = 1;      // benign race: every writer stores 1
                    }
                }
            }
            return;
        }
    }
    consumer_sync();
    // total gradient of each resident trajectory = dt * sum of its groups' partial gradients, in group order
    for (int idx = threadIdx.x; idx < S.TPC * Npar; idx += (PIPE ? NR * NW * 32 : (int)blockDim.x)) {
        const int tr = idx / Npar, k = idx % Npar, tg = cta_traj(tr);
        if (tg < 0) continue;
        double gs = 0.0;
        for (int j = 0; j < S.GPT; ++j) gs += sm[S.o_gsm + (tr * S.GPT + j) * Npar + k];
        if constexpr (SEG) {
            A.seg.gpart[((size_t)seg * A.ntraj + tg) * Npar + k] = dt * gs;
            if constexpr (OBJ != 0) {
                double g2 = 0.0;
                for (int j = 0; j < S.GPT; ++j) g2 += sm[S.o_gsm2 + (tr * S.GPT + j) * Npar + k];
                A.seg.gpart2[((size_t)seg * A.ntraj + tg) * Npar + k] = dt * g2;
            }
            continue;
        }
        A.grad[(size_t)tg * A.gstride + k] = dt * gs;
        if (OBJ) {
            double g2 = 0.0;
            for (int j = 0; j < S.GPT; ++j) g2 += sm[S.o_gsm2 + (tr * S.GPT + j) * Npar + k];
            A.infidgrad[(size_t)tg * A.gstride + k] = dt * g2;
        }
    }
}

// Table entry of one instantiation: the key is derived from the template arguments, so it cannot disagree with the kernel.
template <class LaneT, int UPL, int MINB = 1, int JT = 0, int OBJ = 0, int GLT = 0, int NW = TRAJ_WARPS, int PIPE = 0, bool SEG = false,
          bool HIST = false>
constexpr Inst traj_inst() {
    return {{LaneT::KIND, LaneT::R, LaneT::C, LaneT::NC, LaneT::WQ, LaneT::LMASK, UPL, OBJ != 0, JT < 0, LaneT::HX != 0, !LaneT::AS,
             GLT, JT > 0 ? JT : 0, NW, PIPE, SEG, LaneT::NF, HIST},
            jq_traj_kernel<LaneT, UPL, MINB, JT, OBJ, GLT, NW, PIPE, SEG, HIST>};
}
}  // namespace
