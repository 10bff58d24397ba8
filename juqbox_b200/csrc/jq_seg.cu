// Time-parallel evaluation of a few trajectories (kernel id 7).
//
// One evaluation of traceobjgrad is a serial recurrence over nsteps time steps (src/evalobjgrad.jl:698-753 forward, :810-921 backward);
// a single trajectory occupies one or two warps of one SM for the whole sweep.  Every one-step map of the scheme is LINEAR: the
// Stormer-Verlet state step (src/StormerVerlet.jl:461-504, truncated Neumann solves included) is a real-linear map of (u, v) in R^2n,
// applied column by column, and the adjoint step (:255-303) is affine in (mu, nu) with a forcing that is linear in the state.  So the
// time axis is cut into nseg segments that are swept concurrently and joined exactly (up to rounding) through their propagators:
//
//   launch 1  per segment: forward sweeps of the 2n unit vectors (blocks of m columns on the register-resident layouts) -> Phi_p,
//             adjoint sweeps without forcing of the 2n unit vectors -> Adj_p
//   join X    X_{p+1} = Phi_p X_p from X_0 = Uinit; objective terms and the terminal adjoint from X_nseg (init_adjoint!, :2026-2059)
//   launch 2  per segment: forward sweep of the true state from X_p -> penalty share (penalf2aTrap / penalf2a, :2170-2208);
//             backward state sweep from X_{p+1} -> defect d_p of the backward recomputation (the reference recomputes the states with
//             the times of ITS backward recurrence t = t - dt from T, :810-919, which the rounding of nsteps additions shifts against
//             the forward ones by ~1e-10: its backward states are not the forward ones, and its gradient sees that at ~5e-11 relative)
//   join Eta  Xb_p = X_p + eps_p, eps_p = Psi_p eps_{p+1} + d_p: the boundary states the reference's backward sweep passes through
//             (+ two refinement passes, defect sweep and join, that return at once unless the time steps are coarse)
//   launch 3  per segment: backward sweep from Xb_{p+1} with zero terminal adjoint -> particular adjoint solution c_p
//   join Lam  Lam_p = Adj_p Lam_{p+1} + c_p   (objFuncType 2/3: and Lam2_p = Adj_p Lam2_{p+1} for the second, unforced adjoint set)
//   launch 4  per segment: the reference's backward sweep (state recomputed backwards, adjoint with forcing, gradient traces and
//             B-spline scatter) between the known boundaries -> gradient share
//   sum       grad = sum_p gradient shares, leak = sum_p penalty shares, in a fixed order
//
// The critical path is ~4 nsteps / nseg steps + 3 nseg small products instead of 3 nsteps steps; the extra work (4n/m forward-
// equivalents) runs on SMs that a lone trajectory leaves idle.  Results agree with the plain kernels to rounding
// (tests/test_gpu_timeparallel.py: 1e-12 relative asserted, 5e-15 ... 3e-14 measured) and are bit-reproducible.
#include <algorithm>
#include <cmath>
#include <cstdlib>

#include <cooperative_groups.h>

#include "jq_common.h"

namespace cg = cooperative_groups;

namespace {

// ---- joins -----------------------------------------------------------------------------------------------------------------------
// kind 0: X_{p+1} = Phi_p X_p, p = 0 .. nseg-1, from X_0 = Uinit
// kind 1: Lam_p = Adj_p Lam_{p+1} + c_p, p = nseg-1 .. 1, from the terminal adjoint Lam_nseg (jq_seg_objective_kernel)
// kind 2: Eta_p = Adj_p Eta_{p+1} + J d_p from Eta_nseg = 0: the backward-recomputed boundary states are Xb_p = X_p + eps_p with
//         eps_p = Psi_p eps_{p+1} + d_p, Psi_p the backward propagator ~ Phi_p^-1 = J' Phi_p^T J (symplectic up to the Neumann truncation,
//         ~1e-4 relative, acting on eps ~ 1e-10: exact to rounding); Eta = J eps, and Phi_p^T is the adjoint propagator Adj_p (the adjoint
//         scheme is the exact discrete adjoint of the state scheme: |Adj_p - Phi_p^T| ~ 1e-14 measured).
// kind 4: Lam2_p = Adj_p Lam2_{p+1} from the same terminal value: the second adjoint set of objFuncType 2/3 (no forcing,
//         src/evalobjgrad.jl:848-855), whose gradient is the infidelity-only one.
// kind 3: refinement of Eta.  With coarse time steps the Neumann truncation breaks the symplectic identity at more than rounding (a
//         12-step Rabi problem: 1e-3), and the Eta of kind 2 is off by that factor times eps.  The defect sweep is then repeated from
//         X + J' Eta (SegArgs::pass), its new defect d' chained the same way and added: each pass gains the same factor.  The passes
//         are launched unconditionally and return at once unless the previous defect exceeded refine_tol (SegArgs::flags).
// The columns of a boundary vector are independent chains of nseg dependent matrix-vector products: ONE WARP per (trajectory, column)
// and no block barrier in the small case -- a first version with one CTA per trajectory paid 1.5-2.5 us per segment in __syncthreads
// round trips and generic-to-shared address arithmetic for a 0.1 us product.  M[j][i] (unit vector j, row i) is contiguous in i and
// was just written (L2 resident).

struct ChainArgs {
    const double *M;       // [seg][traj][2n][2n]
    double *V;             // [nseg + 1][traj][m][2n]
    const double *C;       // [seg][traj][m][2n] or nullptr
    int kind;
    bool accumulate;       // kind 3: the chain runs on the correction Delta_p = Adj_p Delta_{p+1} + d'_p from 0, and Eta_p += Delta_p
};

__device__ __forceinline__ ChainArgs chain_args(const LaunchArgs &A, int kind) {
    ChainArgs c;
    c.kind = kind;
    c.M = kind == 0 ? A.seg.Phi : A.seg.Adj;
    c.V = kind == 0 ? A.seg.X : kind == 1 ? A.seg.Lam : kind == 4 ? A.seg.Lam2 : A.seg.Eta;
    c.C = kind == 0 || kind == 4 ? nullptr : kind == 1 ? A.seg.cpart : A.seg.dpart;
    c.accumulate = kind == 3;
    return c;
}

// 2n <= 32: lane i owns entry i of the vector.  The matrices are stored with leading dimension NV (8, 16 or 32; rows and columns past
// 2n are zero) and, with the segment's c_p / d_p, stream through a warp-private ring of D shared-memory slots by cp.async (16-byte
// copies, one commit group per segment): the loads of segment s + D are in flight while segment s is multiplied, so the chain of nseg
// dependent products does not wait for L2 (register prefetch two segments ahead left ~0.4 us of a 0.65 us step exposed).  The vector is
// broadcast through a warp-private strip of shared memory: on one warp (tools/microbench_chain.cu) 32 shuffle broadcasts of a double
// cost ~550 cycles, the 32 FMAs in 8 chains + tree ~100 -- so no shuffles.  sh: per warp [D][NV * NV + 32] | strip[32]
template <int NV, int D>
__global__ void __launch_bounds__(256) jq_seg_chain_small_kernel(const DevProblem P, const LaunchArgs A, int kind) {
    extern __shared__ __align__(16) double sh[];
    constexpr int SLOT = NV * NV + 32;                       // matrix, then the segment's c_p / d_p (32 entries, 2n used)
    const ChainArgs c = chain_args(A, kind);
    const int n = P.n, m = P.m, n2 = 2 * n, nseg = A.seg.nseg, nt = A.ntraj, lane = threadIdx.x & 31;
    const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);          // warp = (trajectory, column)
    if (w >= nt * m) return;
    if (kind == 3 && A.seg.flags[A.seg.pass - 1] == 0) return;
    double *ring = sh + (size_t)(threadIdx.x >> 5) * (D * SLOT + 32), *xs = ring + D * SLOT;
    const int tr = w / m, col = w % m;
    const size_t nv = (size_t)n2 * m;
    const bool on = lane < n2;
    const int lc = lane & (NV - 1);                          // lanes past NV repeat work, write nothing
    const int nstep = kind == 0 ? nseg : nseg - 1;
    const int sgn = kind == 0 ? 1 : -1, p0 = kind == 0 ? 0 : nseg - 1;      // segment of step s: p0 + sgn s
    const double *Mbase = c.M + ((size_t)p0 * nt + tr) * (NV * NV);
    const long long Mstep = (long long)sgn * nt * (NV * NV);
    const double *Cbase = c.C ? c.C + ((size_t)p0 * nt + tr) * nv + (size_t)col * n2 : nullptr;       // 16-byte aligned: 2n is even
    double *Vbase = c.V + ((size_t)(kind == 0 ? 1 : nseg - 1) * nt + tr) * nv + (size_t)col * n2 + (on ? lane : 0);
    const long long Vstep = (long long)sgn * nt * (long long)nv;
    auto issue = [&](int s) {                                // one commit group per step, empty past the last one
        if (s < nstep) {
            const double *M = Mbase + (long long)s * Mstep;
            double *dst = ring + (s % D) * SLOT;
#pragma unroll
            for (int q = 0; q < NV * NV / 64; ++q) {         // NV * NV / 2 chunks of 16 bytes over 32 lanes
                const int ch = lane + 32 * q;
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(dst + 2 * ch)), "l"(M + 2 * ch) : "memory");
            }
            if (Cbase && 2 * lane < n2)
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(dst + NV * NV + 2 * lane)), "l"(Cbase + (long long)s * Vstep + 2 * lane) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    double x = 0.0;
    if (kind == 0) {
        x = on && lane < n ? P.uinit[lane + (size_t)n * col] : 0.0;
        if (on) c.V[(size_t)tr * nv + (size_t)col * n2 + lane] = x;
    } else if (kind == 1 || kind == 4) x = on ? c.V[((size_t)nseg * nt + tr) * nv + (size_t)col * n2 + lane] : 0.0;
    else if (kind == 2 && on) c.V[((size_t)nseg * nt + tr) * nv + (size_t)col * n2 + lane] = 0.0;
    for (int s = 0; s < D; ++s) issue(s);
    const double2 *xv = reinterpret_cast<const double2 *>(xs);
    for (int s = 0; s < nstep; ++s) {
        asm volatile("cp.async.wait_group %0;" ::"n"(D - 1) : "memory");        // this lane's copies of step s have landed ...
        xs[lane] = x;
        __syncwarp();                                        // ... and so have the other lanes'
        const double *Ms = ring + (s % D) * SLOT;
        double acc[8];
#pragma unroll
        for (int k = 0; k < 8; k += 2) { const double2 v = xv[k >> 1]; acc[k] = Ms[k * NV + lc] * v.x; acc[k + 1] = Ms[(k + 1) * NV + lc] * v.y; }
#pragma unroll
        for (int k = 8; k < NV; k += 2) {
            const double2 v = xv[k >> 1];
            acc[k & 7] = fma(Ms[k * NV + lc], v.x, acc[k & 7]);
            acc[(k + 1) & 7] = fma(Ms[(k + 1) * NV + lc], v.y, acc[(k + 1) & 7]);
        }
        const double cp = Cbase && on ? Ms[NV * NV + lane] : 0.0;
        x = (((acc[0] + acc[1]) + (acc[2] + acc[3])) + ((acc[4] + acc[5]) + (acc[6] + acc[7]))) + cp;
        __syncwarp();                                        // the strip and the slot have been read by every lane
        if (on) { if (c.accumulate) Vbase[(long long)s * Vstep] += x; else Vbase[(long long)s * Vstep] = x; }
        issue(s + D);
    }
}

// 2n > 32: one CTA per (trajectory, column), NJ groups of W = roundup32(2n) threads: thread (jq, i) forms the share
// sum_k M[jq + NJ k][i] x[jq + NJ k] of entry i in four independent chains; the NJ shares meet in shared memory.  CNT > 0: the thread's
// CNT matrix entries of the current segment sit in registers, the next segment's are requested as soon as the products are formed and
// fly during the reduction (1024 threads, 16 entries each for 2n = 128: measured faster than 512 threads with 32 entries in 128
// registers, 390 vs 470 us per join of 129 segments); CNT = 0 (2n > 128): plain loads.  sh: xs[W] | part[NJ * W]
template <int CNT>
__global__ void __launch_bounds__(1024) jq_seg_chain_block_kernel(const DevProblem P, const LaunchArgs A, int kind, int W, int NJ) {
    extern __shared__ double sh[];
    const ChainArgs c = chain_args(A, kind);
    const int n = P.n, m = P.m, n2 = 2 * n, nseg = A.seg.nseg, nt = A.ntraj, tid = threadIdx.x;
    if (kind == 3 && A.seg.flags[A.seg.pass - 1] == 0) return;
    const int tr = blockIdx.x / m, col = blockIdx.x % m;
    const size_t nv = (size_t)n2 * m;
    const int jq = tid / W, i = tid % W, PART = W;
    const bool on = i < n2;
    const int nstep = kind == 0 ? nseg : nseg - 1;
    const int cnt = (n2 + NJ - 1) / NJ;
    auto seg_of = [&](int s) { return kind == 0 ? s : nseg - 1 - s; };
    constexpr int HALF = CNT > 0 ? (CNT + 1) / 2 : 1;       // two arrays of CNT / 2, one per pair of partial sums
    double a0[HALF], a1[HALF];
    auto fetch = [&](int s) {
        if constexpr (CNT > 0) {
            const double *M = c.M + ((size_t)seg_of(s) * nt + tr) * n2 * n2 + i;   // leading dimension 2n here (jq_seg_ld)
#pragma unroll
            for (int k = 0; k < HALF; ++k) { const int j = jq + NJ * k; a0[k] = on && j < n2 ? M[(size_t)j * n2] : 0.0; }
#pragma unroll
            for (int k = 0; k < HALF; ++k) { const int j = jq + NJ * (k + HALF); a1[k] = on && j < n2 ? M[(size_t)j * n2] : 0.0; }
        }
    };
    if (tid < W) {
        double x0 = 0.0;
        if (tid < n2) {
            if (kind == 0) { x0 = tid < n ? P.uinit[tid + (size_t)n * col] : 0.0; c.V[(size_t)tr * nv + (size_t)col * n2 + tid] = x0; }
            else if (kind == 1 || kind == 4) x0 = c.V[((size_t)nseg * nt + tr) * nv + (size_t)col * n2 + tid];
            else if (kind == 2) c.V[((size_t)nseg * nt + tr) * nv + (size_t)col * n2 + tid] = 0.0;
        }
        sh[tid] = x0;
    }
    if (nstep > 0) fetch(0);
    for (int s = 0; s < nstep; ++s) {
        const int p = seg_of(s);
        __syncthreads();                                   // xs of this step is in place
        double cp = 0.0;
        if (c.C && tid < n2) cp = c.C[((size_t)p * nt + tr) * nv + (size_t)col * n2 + tid];
        double t[4] = {0.0, 0.0, 0.0, 0.0};
        if constexpr (CNT > 0) {
#pragma unroll
            for (int k = 0; k < HALF; ++k) { const int j = jq + NJ * k; t[k & 1] = fma(a0[k], sh[j < n2 ? j : 0], t[k & 1]); }
#pragma unroll
            for (int k = 0; k < HALF; ++k) { const int j = jq + NJ * (k + HALF); t[2 + (k & 1)] = fma(a1[k], sh[j < n2 ? j : 0], t[2 + (k & 1)]); }
            if (s + 1 < nstep) fetch(s + 1);
        } else {
            const double *M = c.M + ((size_t)p * nt + tr) * n2 * n2;
            if (on) {
#pragma unroll 4
                for (int k = 0; k < cnt; ++k) { const int j = jq + NJ * k; if (j < n2) t[k & 3] = fma(M[(size_t)j * n2 + i], sh[j], t[k & 3]); }
            }
        }
        sh[PART + jq * W + i] = (t[0] + t[1]) + (t[2] + t[3]);
        __syncthreads();
        double v = 0.0;
        if (tid < W) {
            double u[4] = {0.0, 0.0, 0.0, 0.0};
            for (int q = 0; q < NJ; ++q) u[q & 3] += sh[PART + q * W + tid];
            v = ((u[0] + u[1]) + (u[2] + u[3])) + cp;
        }
        __syncthreads();                                   // every share and every xs entry has been read
        if (tid < W) sh[tid] = v;
        if (tid < n2) {
            double *o = c.V + ((size_t)(kind == 0 ? p + 1 : p) * nt + tr) * nv + (size_t)col * n2 + tid;
            if (c.accumulate) *o += v; else *o = v;
        }
    }
}

// 2n > 32, spread over a thread-block cluster: one SM streams a freshly written 131 KB matrix (2n = 128) at ~45 GB/s only -- 3 us per
// segment in the kernel above -- so the chain of one (trajectory, column) runs on a CLUSTER of CS CTAs (CS SMs).  Each CTA owns EPC =
// 2n / CS entries of the vector: it reads only its EPC columns of every matrix (EPC * 8 bytes of each row), thread (jq, i) forms the
// share sum_k M[jq + NG k][i] x[jq + NG k] of its entry in registers that were filled NB segments ahead, the NG shares meet in shared
// memory, and the new entries are written into the vector copy of EVERY CTA of the cluster through distributed shared memory (an
// all-gather); one cluster.sync per segment (~380 cycles), double-buffered vector.  sh: xs[2][2n] | part[NG * EPC]
template <int KPT, int NB>
__global__ void __launch_bounds__(256) jq_seg_chain_cluster_kernel(const DevProblem P, const LaunchArgs A, int kind, int EPC, int NG) {
    extern __shared__ double sh[];
    cg::cluster_group cluster = cg::this_cluster();
    const int CS = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
    const ChainArgs c = chain_args(A, kind);
    const int n = P.n, m = P.m, n2 = 2 * n, nseg = A.seg.nseg, nt = A.ntraj, tid = threadIdx.x;
    if (kind == 3 && A.seg.flags[A.seg.pass - 1] == 0) return;          // uniform over the cluster
    const int chain = blockIdx.x / CS, tr = chain / m, col = chain % m;
    const size_t nv = (size_t)n2 * m;
    const int jq = tid / EPC, i = tid % EPC, gi = rank * EPC + i;       // this thread's entry of the vector
    const bool worker = jq < NG && gi < n2;
    double *xs = sh, *part = sh + 2 * n2;
    const int nstep = kind == 0 ? nseg : nseg - 1;
    const int sgn = kind == 0 ? 1 : -1, p0 = kind == 0 ? 0 : nseg - 1;
    const double *Mbase = c.M + ((size_t)p0 * nt + tr) * n2 * n2 + (size_t)jq * n2 + (worker ? gi : 0);     // leading dimension 2n (jq_seg_ld)
    const long long Mstep = (long long)sgn * nt * n2 * n2;
    auto fetch = [&](int s, double (&a)[KPT]) {
        const double *M = Mbase + (long long)s * Mstep;
#pragma unroll
        for (int k = 0; k < KPT; ++k) a[k] = worker && jq + NG * k < n2 ? M[(size_t)NG * k * n2] : 0.0;
    };
    for (int idx = tid; idx < n2; idx += blockDim.x) {       // every CTA starts from its own copy of the whole vector
        double x0 = 0.0;
        if (kind == 0) x0 = idx < n ? P.uinit[idx + (size_t)n * col] : 0.0;
        else if (kind == 1 || kind == 4) x0 = c.V[((size_t)nseg * nt + tr) * nv + (size_t)col * n2 + idx];
        xs[idx] = x0;
        if (rank == 0 && kind == 0) c.V[(size_t)tr * nv + (size_t)col * n2 + idx] = x0;
        if (rank == 0 && kind == 2) c.V[((size_t)nseg * nt + tr) * nv + (size_t)col * n2 + idx] = 0.0;
    }
    double a[NB][KPT];
#pragma unroll
    for (int u = 0; u < NB; ++u) {
        if (u < nstep) fetch(u, a[u]);
    }
    cluster.sync();
    int cur = 0;
    for (int s0 = 0; s0 < nstep; s0 += NB) {
#pragma unroll
        for (int u = 0; u < NB; ++u) {
            const int s = s0 + u;
            if (s < nstep) {                                 // uniform over the cluster
                const int p = p0 + sgn * s;
                const double *x = xs + cur * n2;
                double t0 = 0.0, t1 = 0.0;
#pragma unroll
                for (int k = 0; k < KPT; k += 2) {
                    const int j0 = jq + NG * k, j1 = jq + NG * (k + 1);
                    t0 = fma(a[u][k], x[j0 < n2 ? j0 : 0], t0);
                    if (k + 1 < KPT) t1 = fma(a[u][k + 1], x[j1 < n2 ? j1 : 0], t1);
                }
                if (jq < NG) part[jq * EPC + i] = t0 + t1;
                if (s + NB < nstep) fetch(s + NB, a[u]);
                __syncthreads();
                if (tid < EPC && rank * EPC + tid < n2) {
                    const int ge = rank * EPC + tid;
                    double w[4] = {0.0, 0.0, 0.0, 0.0};
                    for (int q = 0; q < NG; ++q) w[q & 3] += part[q * EPC + tid];
                    double v = (w[0] + w[1]) + (w[2] + w[3]);
                    if (c.C) v += c.C[((size_t)p * nt + tr) * nv + (size_t)col * n2 + ge];
                    double *xn = xs + (cur ^ 1) * n2 + ge;
                    for (int r = 0; r < CS; ++r) *cluster.map_shared_rank(xn, r) = v;          // all-gather through distributed shared memory
                    double *o = c.V + ((size_t)(kind == 0 ? p + 1 : p) * nt + tr) * nv + (size_t)col * n2 + ge;
                    if (c.accumulate) *o += v; else *o = v;
                }
                cluster.sync();                              // the new vector is complete in every CTA; part and the old vector are free
                cur ^= 1;
            }
        }
    }
}

// Objective terms of the final state X_nseg (src/evalobjgrad.jl:755-792) and the terminal adjoint (init_adjoint!, :2026-2059): the same
// formulas as the trajectory kernels (jq_traj_kernels.cuh).  One CTA per trajectory, one warp-ordered reduction.
__global__ void __launch_bounds__(256) jq_seg_objective_kernel(const DevProblem P, const LaunchArgs A) {
    __shared__ double red[16];
    const int n = P.n, m = P.m, n2 = 2 * n, nseg = A.seg.nseg, nt = A.ntraj, tid = threadIdx.x, tr = blockIdx.x;
    const size_t nv = (size_t)n2 * m;
    const double *xs = A.seg.X + ((size_t)nseg * nt + tr) * nv;
    double re = 0.0, im = 0.0;
    for (int idx = tid; idx < n * m; idx += blockDim.x) {
        const int r = idx % n, c = idx / n;
        const double vr = xs[c * n2 + r], vi = xs[c * n2 + n + r], tr_ = P.vtr[idx], ti_ = P.vti[idx];
        re += vr * tr_ - vi * ti_;
        im += vr * ti_ + vi * tr_;
    }
    for (int o = 16; o > 0; o >>= 1) { re += __shfl_xor_sync(0xffffffffu, re, o); im += __shfl_xor_sync(0xffffffffu, im, o); }
    if ((tid & 31) == 0) { red[2 * (tid >> 5)] = re; red[2 * (tid >> 5) + 1] = im; }
    __syncthreads();
    double rs = 0.0, is = 0.0;
    for (int w = 0; w < (int)(blockDim.x + 31) / 32; ++w) { rs += red[2 * w]; is += red[2 * w + 1]; }
    rs /= m; is /= m;
    const int pfid = P.pFidType;
    double sph = 0.0, cph = 1.0;
    if (pfid != 2) sincos(pfid == 3 ? A.pcof[(size_t)(tr / A.nsamples) * A.pstride + A.Npar] : P.globalPhase, &sph, &cph);
    const double abs2 = rs * rs + is * is;
    const double infid = pfid == 1 ? 1.0 + abs2 - 2.0 * (rs * cph + is * sph) : pfid == 2 ? 1.0 - abs2 : 1.0 - (rs * cph - is * sph);
    if (tid == 0) {
        double *o = A.scal + (size_t)tr * 4;
        o[0] = infid; o[2] = 1.0 - abs2; o[3] = 0.0;          // o[1] (leak) is the sum of the penalty shares (jq_seg_sum_kernel)
        if (pfid == 3 && A.evaladjoint) {
            A.grad[(size_t)tr * A.gstride + A.Npar] = rs * sph + is * cph;
            if (A.infidgrad) A.infidgrad[(size_t)tr * A.gstride + A.Npar] = rs * sph + is * cph;
        }
    }
    if (!A.evaladjoint) return;
    const double rs_ = pfid == 1 ? cph - rs : rs, is_ = pfid == 1 ? sph - is : is;
    double *LT = A.seg.Lam + ((size_t)nseg * nt + tr) * nv;
    for (int idx = tid; idx < n * m; idx += blockDim.x) {
        const double tr_ = P.vtr[idx], ti_ = P.vti[idx];
        const int bx = (idx / n) * n2 + idx % n;             // boundary vectors: [column][u rows, then v rows]
        if (pfid <= 2) { LT[bx] = (rs_ * tr_ + is_ * ti_) / m; LT[bx + n] = (is_ * tr_ - rs_ * ti_) / m; }
        else { LT[bx] = 0.5 * (cph * tr_ - sph * ti_) / m; LT[bx + n] = -0.5 * (sph * tr_ + cph * ti_) / m; }
        if (A.seg.Lam2) { double *L2 = A.seg.Lam2 + ((size_t)nseg * nt + tr) * nv; L2[bx] = LT[bx]; L2[bx + n] = LT[bx + n]; }
    }
}

// grad[tr][k] = sum_p gpart[p][tr][k], leak[tr] = sum_p penpart[p][tr]: one warp per output, lane l sums the segments l, l + 32, ... in
// order, then a butterfly -- a fixed order, independent of the launch geometry
__global__ void __launch_bounds__(256) jq_seg_sum_kernel(const LaunchArgs A) {
    const int nseg = A.seg.nseg, nt = A.ntraj, Npar = A.Npar, lane = threadIdx.x & 31;
    const long long total = (long long)nt * (Npar + 1), nwarps = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long idx = blockIdx.x * (long long)(blockDim.x >> 5) + (threadIdx.x >> 5); idx < total; idx += nwarps) {
        const int tr = (int)(idx / (Npar + 1)), k = (int)(idx % (Npar + 1));
        if (k < Npar && !A.evaladjoint) continue;
        double s = 0.0;
        if (k == Npar) { for (int p = lane; p < nseg; p += 32) s += A.seg.penpart[(size_t)p * nt + tr]; }
        else { for (int p = lane; p < nseg; p += 32) s += A.seg.gpart[((size_t)p * nt + tr) * Npar + k]; }
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) {
            if (k == Npar) A.scal[(size_t)tr * 4 + 1] = s;
            else A.grad[(size_t)tr * A.gstride + k] = s;
        }
        if (k < Npar && A.seg.gpart2) {                      // objFuncType 2/3: the infidelity-only gradient
            double s2 = 0.0;
            for (int p = lane; p < nseg; p += 32) s2 += A.seg.gpart2[((size_t)p * nt + tr) * Npar + k];
            for (int o = 16; o > 0; o >>= 1) s2 += __shfl_xor_sync(0xffffffffu, s2, o);
            if (lane == 0) A.infidgrad[(size_t)tr * A.gstride + k] = s2;
        }
    }
}

// VJP (jq_seg_vjp_launch): the terminal value of the unforced adjoint set from the cotangent c of trajectory tr (cot_r + tr * cstride,
// the last block of a cotangent history), kernel 9's terminal condition lambda_r(T) = -c_r / 2, lambda_i(T) = c_i / 2 (NULL part: zero)
// in the boundary layout, Lam2_nseg = [column][u rows, then v rows]; and U(T) of X_nseg in the ABI layout (Re U = vr, Im U = -vi,
// column-major n x m), written by cotangent 0 of every (candidate, sample): trajectory tr = t * nc + k.
__global__ void __launch_bounds__(256) jq_seg_vjp_terminal_kernel(const DevProblem P, const LaunchArgs A, int nc, const double *cot_r,
                                                                  const double *cot_i, size_t cstride, double *state_r, double *state_i) {
    const int n = P.n, nseg = A.seg.nseg;
    const size_t nm = (size_t)n * P.m, nv = 2 * nm, total = (size_t)A.ntraj * nm;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const size_t tr = idx / nm, e = idx % nm;
        const size_t bx = ((size_t)nseg * A.ntraj + tr) * nv + (e / n) * 2 * n + e % n;
        if (A.seg.Lam2) {
            const size_t c = tr * cstride + e;
            A.seg.Lam2[bx] = cot_r ? -0.5 * cot_r[c] : 0.0;
            A.seg.Lam2[bx + n] = cot_i ? 0.5 * cot_i[c] : 0.0;
        }
        if (tr % nc == 0) {
            const size_t o = (tr / nc) * nm + e;
            if (state_r) state_r[o] = A.seg.X[bx];
            if (state_i) state_i[o] = -A.seg.X[bx + n];
        }
    }
}

// vjp[tr][k] = sum_p gpart2[p][tr][k] in jq_seg_sum_kernel's fixed order (one warp per entry, lane l sums the segments l, l + 32, ...,
// then a butterfly); with pFidType 3 the phase entry k = Npar of the pstride-long rows is 0: U(T) does not depend on it
__global__ void __launch_bounds__(256) jq_seg_vjp_sum_kernel(const LaunchArgs A, double *vjp) {
    const int nseg = A.seg.nseg, nt = A.ntraj, Npar = A.Npar, lane = threadIdx.x & 31;
    const long long total = (long long)nt * A.pstride, nwarps = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long idx = blockIdx.x * (long long)(blockDim.x >> 5) + (threadIdx.x >> 5); idx < total; idx += nwarps) {
        const int tr = (int)(idx / A.pstride), k = (int)(idx % A.pstride);
        double s = 0.0;
        if (k < Npar) { for (int p = lane; p < nseg; p += 32) s += A.seg.gpart2[((size_t)p * nt + tr) * Npar + k]; }
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) vjp[idx] = s;
    }
}

// Join `kind` of the segment boundaries of A (see the kinds above): one warp per (trajectory, column); small matrices: the columns of a
// trajectory share a CTA, large ones: a CTA (an SM) each
void run_join(const DevProblem &P, const LaunchArgs &A, int kind, cudaStream_t st) {
    const size_t n2 = 2 * (size_t)P.n;
    const long long nwarps = (long long)A.ntraj * P.m;
    if (n2 <= 32) {
        // ring of 8 segments per warp: 8 (NV^2 + 32) + 32 doubles -- one warp per CTA for 2n > 16 (68 KB), up to four otherwise
        constexpr int D = 8;
        const int NV = n2 <= 8 ? 8 : n2 <= 16 ? 16 : 32;
        const int wpb = (int)std::min<long long>(NV == 32 ? 1 : 4, nwarps);
        const unsigned grid = (unsigned)((nwarps + wpb - 1) / wpb);
        const size_t sm = (size_t)wpb * (D * (NV * NV + 32) + 32) * sizeof(double);
        void (*k)(const DevProblem, const LaunchArgs, int) =
            NV == 8 ? jq_seg_chain_small_kernel<8, D> : NV == 16 ? jq_seg_chain_small_kernel<16, D> : jq_seg_chain_small_kernel<32, D>;
        if (sm > 48 * 1024) cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
        k<<<grid, wpb * 32, sm, st>>>(P, A, kind);
    } else {
        // cluster version: CS = 8 CTAs per chain, EPC entries each, NG = 256 / EPC row groups, at most 8 matrix entries per thread
        {
            const int CS = 8, EPC = (int)((n2 + CS - 1) / CS), NG = EPC <= 256 ? 256 / EPC : 0, kpt = NG ? (int)((n2 + NG - 1) / NG) : 99;
            const char *cenv = getenv("JQ_SEG_CLUSTER");
            if ((cenv ? atoi(cenv) != 0 : true) && kpt <= 8) {
                cudaLaunchConfig_t cfg = {};
                cfg.gridDim = dim3((unsigned)(nwarps * CS)); cfg.blockDim = dim3(256);
                cfg.dynamicSmemBytes = (size_t)(2 * n2 + NG * EPC) * sizeof(double); cfg.stream = st;
                cudaLaunchAttribute at[1];
                at[0].id = cudaLaunchAttributeClusterDimension;
                at[0].val.clusterDim.x = CS; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
                cfg.attrs = at; cfg.numAttrs = 1;
                cudaError_t ce = kpt <= 4 ? cudaLaunchKernelEx(&cfg, jq_seg_chain_cluster_kernel<4, 4>, P, A, kind, EPC, NG)
                                          : cudaLaunchKernelEx(&cfg, jq_seg_chain_cluster_kernel<8, 4>, P, A, kind, EPC, NG);
                if (ce == cudaSuccess) return;
                cudaGetLastError();                     // fall through to the one-CTA kernel
            }
        }
        const int W = (int)((n2 + 31) / 32 * 32), NJ = std::max(1, 1024 / W), cnt = (int)((n2 + NJ - 1) / NJ);
        const unsigned grid = (unsigned)nwarps, thr = (unsigned)(W * NJ);
        const size_t sm = (size_t)(W + NJ * W) * sizeof(double);
        if (cnt <= 8) jq_seg_chain_block_kernel<8><<<grid, thr, sm, st>>>(P, A, kind, W, NJ);
        else if (cnt <= 16) jq_seg_chain_block_kernel<16><<<grid, thr, sm, st>>>(P, A, kind, W, NJ);
        else jq_seg_chain_block_kernel<0><<<grid, thr, sm, st>>>(P, A, kind, W, NJ);
    }
}

// development: JQ_SEG_TIMING=1 prints the CUDA-event time of every stage of a time-parallel launch
struct StageTimer {
    cudaEvent_t ev[12];
    int nev = 0;
    const bool on = getenv("JQ_SEG_TIMING") != nullptr;
    cudaStream_t st;
    explicit StageTimer(cudaStream_t s) : st(s) {}
    void mark() { if (on && nev < 12) { cudaEventCreate(&ev[nev]); cudaEventRecord(ev[nev], st); ++nev; } }
    void print(const char *what) {
        if (!on) return;
        cudaStreamSynchronize(st);
        printf("%s (us):", what);
        for (int k = 1; k < nev; ++k) { float ms = 0.f; cudaEventElapsedTime(&ms, ev[k - 1], ev[k]); printf(" %.1f", ms * 1e3); }
        printf("\n");
    }
    ~StageTimer() { for (int k = 0; k < nev; ++k) cudaEventDestroy(ev[k]); }
};

}   // namespace

// Number of segments for a launch of ntraj trajectories.  Per evaluation the sweeps between boundaries cost ~ nsteps / nseg steps of one
// lane's instruction stream (three times in a row), the joins ~ nseg dependent products (three times), the propagator launch a fixed
// amount of work: nseg ~ sqrt(nsteps * step / product); the measured optimum is flat (profiles/r02_timeparallel.md).  When the propagator
// launch fills the GPU, its CTA count is rounded to whole waves of one CTA per SM.  tpc = trajectories per CTA of the propagator plan.
int jq_seg_auto_segments(const DevProblem &P, int ntraj, int evaladjoint, int tpc, int sms) {
    const int nblk = (2 * P.n + P.m - 1) / P.m;
    const double kappa = 2 * P.n <= 32 ? 1.6 : 0.5;
    double nseg = sqrt((double)P.nsteps * kappa);
    // CTAs per segment in the propagator launch -- counted as for an evaluation with gradient also for objective-only calls, so that both
    // cut the time axis the same way and return bit-identical objectives (a line search mixes the two)
    (void)evaladjoint;
    const long long cps = 2 * (((long long)nblk * ntraj + tpc - 1) / tpc);
    const double waves = nseg * (double)cps / sms;
    if (waves >= 0.75 && cps <= sms) nseg = floor(floor(waves + 0.5) * sms / (double)cps);
    nseg = std::min<double>(nseg, (double)(P.nsteps / 16));
    nseg = std::min<double>(nseg, 1024.0);
    return (int)std::max<double>(nseg, 1.0);
}

// Leading dimension of the segment propagators: 8, 16 or 32 for the one-warp joins (zero padded), 2n for the block join.
int jq_seg_ld(const DevProblem &P) { const int n2 = 2 * P.n; return n2 <= 8 ? 8 : n2 <= 16 ? 16 : n2 <= 32 ? 32 : n2; }

// The segment workspace of a driver, counted and, given `work`, carved into S's arrays in that driver's order.
// Every array is rounded to an even number of doubles, so that each starts 16-byte aligned.
//   evaluation (vjp false): Phi, X, penpart; with `adjoint` also Adj, Lam, Eta, cpart, dpart, gpart and, for objFuncType 2/3, Lam2, gpart2
//   VJP: Phi, X; with `adjoint` (cotangents) also Adj, Lam2, Eta, dpart, gpart, gpart2 and, with `jumps` (a history), cpart
size_t jq_seg_workspace(const DevProblem &P, int ntraj, int Npar, int nseg, bool vjp, bool adjoint, bool jumps, double *work, SegArgs *S) {
    const size_t ld = (size_t)jq_seg_ld(P), nm2 = 2 * (size_t)P.n * P.m, nt = (size_t)ntraj, ns = (size_t)nseg;
    const size_t prop = ns * nt * ld * ld, bound = (ns + 1) * nt * nm2, part = ns * nt * nm2, grad = ns * nt * (size_t)Npar;
    SegArgs count{};
    SegArgs &A = S ? *S : count;
    size_t tot = 0;
    auto take = [&](double *&dst, size_t cnt) { dst = work ? work + tot : nullptr; tot += (cnt + 1) & ~(size_t)1; };
    take(A.Phi, prop);
    take(A.X, bound);
    if (!vjp) take(A.penpart, ns * nt);
    if (adjoint) {
        take(A.Adj, prop);
        take(vjp ? A.Lam2 : A.Lam, bound);
        take(A.Eta, bound);
        if (!vjp) take(A.cpart, part);
        take(A.dpart, part);
        take(A.gpart, grad);
        if (!vjp && P.objFuncType != 1) take(A.Lam2, bound);
        if (vjp || P.objFuncType != 1) take(A.gpart2, grad);
        if (vjp && jumps) take(A.cpart, part);
    }
    return tot;
}

// Segment p covers steps [p nsteps / nseg, (p + 1) nsteps / nseg).  The reference advances the time by t = t + dt from 0 in the forward
// sweep (src/evalobjgrad.jl:745) and by t = t - dt from T in the backward sweep (:810, :919); the segment sweeps start from the values
// those recurrences reach, not from k dt, so that every control is evaluated at bit-identical times.
void jq_seg_times(const DevProblem &P, int nseg, double *times) {
    const double dt = P.T / (double)P.nsteps;
    double t = 0.0;
    int p = 0;
    for (long long k = 0; k < P.nsteps && p < nseg; ++k) {
        while (p < nseg && (long long)p * P.nsteps / nseg == k) times[p++] = t;
        t = t + dt;
    }
    t = P.T;
    p = nseg - 1;
    const double mdt = -dt;
    for (long long k = P.nsteps; k > 0 && p >= 0; --k) {
        while (p >= 0 && (long long)(p + 1) * P.nsteps / nseg == k) times[nseg + p--] = t;
        t = t + mdt;
    }
}

// The segment set-up of both drivers: A's segment count, times, propagator stride and refinement state, the workspace arrays of
// jq_seg_workspace (with the adjoint sets when A.evaladjoint), the refinement flags cleared and the padding of the propagators zeroed
static void seg_setup(const DevProblem &P, LaunchArgs &A, int nseg, const double *times, int *flags, double *work, bool vjp, bool jumps,
                      cudaStream_t st) {
    const size_t ld = (size_t)jq_seg_ld(P), nt = (size_t)A.ntraj, ns = (size_t)nseg;
    A.seg.nseg = nseg;
    A.seg.times = times;
    A.seg.ld = (int)ld;
    A.seg.pass = 0;
    A.seg.flags = flags;
    A.seg.refine_tol = 1.0e-9 / (double)nseg;              // |eps| <~ nseg |d|: below 1e-9 the first-order join is exact to 1e-12 and better
    jq_seg_workspace(P, A.ntraj, A.Npar, nseg, vjp, A.evaladjoint, jumps, work, &A.seg);
    cudaMemsetAsync(flags, 0, 4 * sizeof(int), st);
    if (ld != 2 * (size_t)P.n) {            // the padding of the propagators must read as zero
        cudaMemsetAsync(A.seg.Phi, 0, ns * nt * ld * ld * sizeof(double), st);
        if (A.evaladjoint) cudaMemsetAsync(A.seg.Adj, 0, ns * nt * ld * ld * sizeof(double), st);
    }
}

cudaError_t jq_seg_launch(TrajPlan *plan_prop, TrajPlan *plan, TrajPlan *plan_obj, const DevProblem &P, const LaunchArgs &A0, int nseg, const double *times, int *flags, double *work, cudaStream_t st, const SegCoop *coop,
                          int *nctas, int *regs, size_t *smem, int *traj_per_cta, int *nlaunch) {
    if (nseg < 1 || nseg > P.nsteps) return cudaErrorInvalidValue;
    if (P.solver != 1 || A0.hist_r || (P.objFuncType != 1 && (!plan_obj || (A0.evaladjoint && !A0.infidgrad)))) return cudaErrorNotSupported;
    const size_t nt = (size_t)A0.ntraj, ld = (size_t)jq_seg_ld(P);
    if (2 * P.n > 512) return cudaErrorNotSupported;
    LaunchArgs A = A0;
    seg_setup(P, A, nseg, times, flags, work, false, false, st);
    int launches = 0;
    StageTimer timer(st);
    timer.mark();
    // launch 1: propagators
    A.seg.mode[0] = 1; A.seg.mode[1] = A.evaladjoint ? 3 : 0;
    const bool shared = coop && coop->nranks > 1 && nseg % coop->nranks == 0;
    if (shared) { A.seg.seg_cnt = nseg / coop->nranks; A.seg.seg_lo = coop->rank * A.seg.seg_cnt; }
    cudaError_t e = jq_traj_launch(plan_prop ? plan_prop : plan, P, A, st, nctas, regs, smem, traj_per_cta);
    if (e != cudaSuccess) return e;
    if (shared) {               // every rank swept its share of the segments: complete Phi and Adj everywhere
        const size_t per_rank = (size_t)A.seg.seg_cnt * nt * ld * ld;
        if (coop->allgather(coop->ctx, A.seg.Phi, per_rank, st) != 0) return cudaErrorUnknown;
        if (A.evaladjoint && coop->allgather(coop->ctx, A.seg.Adj, per_rank, st) != 0) return cudaErrorUnknown;
        A.seg.seg_lo = 0; A.seg.seg_cnt = 0;
        launches += A.evaladjoint ? 2 : 1;
    }
    timer.mark();
    run_join(P, A, 0, st);
    timer.mark();
    jq_seg_objective_kernel<<<(unsigned)nt, 256, 0, st>>>(P, A);
    timer.mark();
    // launch 2: penalty shares; defects of the backward state recomputation
    A.seg.mode[0] = 2; A.seg.mode[1] = A.evaladjoint ? 6 : 0;
    e = jq_traj_launch(plan, P, A, st, nullptr, nullptr, nullptr, nullptr);
    if (e != cudaSuccess) return e;
    launches += 4;
    timer.mark();
    if (A.evaladjoint) {
        run_join(P, A, 2, st);
        // refinement passes of the boundary states of the backward sweep: no-ops unless the defects are large (coarse time steps)
        for (int r = 1; r <= 2; ++r) {
            A.seg.pass = r; A.seg.mode[0] = 6; A.seg.mode[1] = 0;
            e = jq_traj_launch(plan, P, A, st, nullptr, nullptr, nullptr, nullptr);
            if (e != cudaSuccess) return e;
            run_join(P, A, 3, st);
            launches += 2;
        }
        A.seg.pass = 0;
        timer.mark();
        // launch 3: particular adjoint solutions
        A.seg.mode[0] = 4; A.seg.mode[1] = 0;
        e = jq_traj_launch(plan, P, A, st, nullptr, nullptr, nullptr, nullptr);
        if (e != cudaSuccess) return e;
        timer.mark();
        run_join(P, A, 1, st);
        if (P.objFuncType != 1) { run_join(P, A, 4, st); ++launches; }
        timer.mark();
        // launch 4: gradient shares (objFuncType 2/3: with the second adjoint set, on the plan that has it)
        A.seg.mode[0] = 5; A.seg.mode[1] = 0;
        e = jq_traj_launch(P.objFuncType != 1 ? plan_obj : plan, P, A, st, nullptr, nullptr, nullptr, nullptr);
        if (e != cudaSuccess) return e;
        launches += 4;
        timer.mark();
    }
    const long long total = (long long)nt * (A.Npar + 1);
    jq_seg_sum_kernel<<<(unsigned)std::min<long long>((total + 7) / 8, 148 * 8), 256, 0, st>>>(A);
    ++launches;
    timer.mark();
    timer.print("seg stages");
    if (nlaunch) *nlaunch = launches;
    return cudaGetLastError();
}

// Vector-Jacobian products of the saved states on the segment sweeps (DESIGN.md §4.9, §4.10): the stages of jq_seg_launch that the
// unforced adjoint set (kind 4, Lam2) needs, started from the callers' cotangents instead of the objective's terminal adjoint --
//   launch 1  Phi_p (mode 1) and, with cotangents, Adj_p (mode 3)
//   join X    X_{p+1} = Phi_p X_p, then jq_seg_vjp_terminal_kernel: Lam2_nseg from the last cotangent block, U(T) from X_nseg
//   launch 2  the saved states (mode 2, with a history; no penalty shares: penpart is nullptr), defect sweeps (mode 6, pass 0; the penalty plays no part) and, with jumps,
//             the particular solutions of the unforced set (mode 7): adjoint sweeps from zero with the segment's cotangent jumps
//   join Eta  and the two refinement passes (mode 6 only)
//   join Lam2 Lam2_p = Adj_p Lam2_{p+1} (kind 4), with jumps Lam2_p = Adj_p Lam2_{p+1} + c_p (kind 1 with Lam = Lam2, cpart = c)
//   launch 4  gradient sweeps (mode 5) on plan_obj, the two-set instantiation, jumps applied to the second set: gpart2 is the VJP's
//             share of segment p
//   sum       vjp = sum_p gpart2 (jq_seg_vjp_sum_kernel)
// Launch 3 and join Lam (the forced set's particular solutions) are not run: mode 5 still sweeps the forced set next to the unforced
// one, from Lam = Lam2 (a finite input), and its gpart is discarded.  A save at global step k belongs to the segment p with
// k0 <= k < k1: its jump is in c_p, so Lam2_p contains it; save nsave - 1 is the terminal value, save 0 has no effect.
// ncot = 0: launch 1 (Phi only), join X, then U(T) and / or the history.
// P.objFuncType must be 2 or 3, so that mode 5 selects the two-set instantiation (the other modes select the plain ones whatever it is).
// Trajectory tr = t * nc + k of A, nc = max(ncot, 1), pulls back cotangent k (cot_r, cot_i [tr][nsave][n*m], NULL: zero) of
// candidate x sample t; nsave = 1 (save_every = nsteps): the final-state VJP, whose stages and arithmetic do not depend on this
// function's history arguments.  vjp [tr][A.pstride]; state_r, state_i [t][n*m] or NULL; hist_r, hist_i [t][nsave][n*m] or NULL.
cudaError_t jq_seg_vjp_launch(TrajPlan *plan_prop, TrajPlan *plan, TrajPlan *plan_obj, const DevProblem &P, const LaunchArgs &A0, int nseg,
                              const double *times, int *flags, double *work, cudaStream_t st, int ncot, int save_every, long long nsave,
                              const double *cot_r, const double *cot_i, double *vjp, double *state_r, double *state_i, double *hist_r,
                              double *hist_i, int *nctas, int *regs, size_t *smem, int *traj_per_cta, int *nlaunch) {
    if (nseg < 1 || nseg > P.nsteps) return cudaErrorInvalidValue;
    if (save_every < 1 || nsave < 1) return cudaErrorInvalidValue;
    const bool cot = ncot > 0, jumps = cot && nsave > 1 && (cot_r || cot_i), hist = hist_r || hist_i;
    if (P.solver != 1 || P.objFuncType == 1 || A0.hist_r || 2 * P.n > 512 || (cot && !plan_obj)) return cudaErrorNotSupported;
    if (hist && !(hist_r && hist_i)) return cudaErrorInvalidValue;
    const size_t nm2 = 2 * (size_t)P.n * P.m, nt = (size_t)A0.ntraj;
    LaunchArgs A = A0;
    A.evaladjoint = cot ? 1 : 0;
    seg_setup(P, A, nseg, times, flags, work, true, jumps, st);
    if (cot) A.seg.Lam = A.seg.Lam2;        // mode 5 sweeps the forced set from Lam2 (its gradient shares are discarded)
    // the history VJP's additions to the launches: the saves of mode 2 (cotangent 0 of every (candidate, sample)), the third mode of
    // launch 2 and the cotangent jumps of modes 7 and 5
    SegHist H{};
    H.hist_nc = std::max(ncot, 1);
    if (jumps) { H.cot_r = cot_r; H.cot_i = cot_i; }
    const size_t nm = nm2 / 2;
    int launches = 0;
    // Eta_0, which no join writes, enters the refinement passes' defect of segment 0 (dpart_0 feeds nothing, but the flag does): zero,
    // so that a stale workspace cannot start a pass
    if (cot) cudaMemsetAsync(A.seg.Eta, 0, nt * nm2 * sizeof(double), st);
    StageTimer timer(st);
    timer.mark();
    A.seg.mode[0] = 1; A.seg.mode[1] = cot ? 3 : 0;
    cudaError_t e = jq_traj_launch(plan_prop ? plan_prop : plan, P, A, st, nctas, regs, smem, traj_per_cta);
    if (e != cudaSuccess) return e;
    timer.mark();
    run_join(P, A, 0, st);
    launches += 2;
    timer.mark();
    if (cot || state_r || state_i) {
        const size_t nel = nt * nm;
        jq_seg_vjp_terminal_kernel<<<(unsigned)std::min<size_t>((nel + 255) / 256, 148 * 8), 256, 0, st>>>(
            P, A, std::max(ncot, 1), cot_r ? cot_r + (size_t)(nsave - 1) * nm : nullptr, cot_i ? cot_i + (size_t)(nsave - 1) * nm : nullptr,
            (size_t)nsave * nm, state_r, state_i);
        ++launches;
        timer.mark();
    }
    if (hist || cot) {         // launch 2: the modes of this call, in the order 2, 6, 7
        int modes[3] = {0, 0, 0}, k = 0;
        if (hist) modes[k++] = 2;
        if (cot) modes[k++] = 6;
        if (jumps) modes[k++] = 7;
        A.seg.mode[0] = modes[0]; A.seg.mode[1] = modes[1]; H.mode2 = modes[2];
        if (hist) { A.hist_r = hist_r; A.hist_i = hist_i; A.save_every = save_every; A.nsave = nsave; }
        if (jumps) { A.save_every = save_every; A.nsave = nsave; }
        e = jq_traj_launch(plan, P, A, st, nullptr, nullptr, nullptr, nullptr, hist || jumps ? &H : nullptr);
        if (e != cudaSuccess) return e;
        A.hist_r = A.hist_i = nullptr;
        H.mode2 = 0;
        ++launches;
        timer.mark();
    }
    if (cot) {
        run_join(P, A, 2, st);
        ++launches;
        A.seg.mode[0] = 6; A.seg.mode[1] = 0;
        for (int r = 1; r <= 2; ++r) {         // refinement passes: no-ops unless the defects are large (coarse time steps)
            A.seg.pass = r;
            e = jq_traj_launch(plan, P, A, st, nullptr, nullptr, nullptr, nullptr);
            if (e != cudaSuccess) return e;
            run_join(P, A, 3, st);
            launches += 2;
        }
        A.seg.pass = 0;
        timer.mark();
        run_join(P, A, jumps ? 1 : 4, st);
        timer.mark();
        A.seg.mode[0] = 5;
        e = jq_traj_launch(plan_obj, P, A, st, nullptr, nullptr, nullptr, nullptr, jumps ? &H : nullptr);
        if (e != cudaSuccess) return e;
        timer.mark();
        const long long total = (long long)nt * A.pstride;
        jq_seg_vjp_sum_kernel<<<(unsigned)std::min<long long>((total + 7) / 8, 148 * 8), 256, 0, st>>>(A, vjp);
        launches += 3;
        timer.mark();
    }
    timer.print("seg vjp stages");
    if (nlaunch) *nlaunch = launches;
    return cudaGetLastError();
}
