// Planners, launch and instantiation lookup of the register-resident trajectory kernels; the kernels themselves are in
// jq_traj_kernels.cuh (shared with the jq_traj_inst_*.cu files, which hold the other parts of the table).
#include "jq_traj_kernels.cuh"

namespace {

const Inst kInst[] = {
    traj_inst<FiberLane<2, 1, 1>, 1, 4>(), traj_inst<FiberLane<4, 1, 1>, 1, 3>(), traj_inst<FiberLane<4, 1, 1>, 2, 3>(), traj_inst<FiberLane<6, 1, 1>, 2>(),
    traj_inst<FiberLane<3, 1, 1>, 1, 3>(), traj_inst<FiberLane<3, 1, 1>, 2, 3>(), traj_inst<FiberLane<4, 2, 1>, 1>(), traj_inst<FiberLane<3, 2, 1>, 1>(),
    traj_inst<FiberLane<2, 2, 1>, 1>(), traj_inst<FiberLane<4, 3, 1>, 1>(), traj_inst<FiberLane<3, 3, 1>, 1>(), traj_inst<FiberLane<2, 3, 1>, 1>(),
    traj_inst<FiberLane<5, 2, 1>, 1>(), traj_inst<FiberLane<5, 3, 1>, 1>(), traj_inst<FiberLane<6, 2, 1>, 1>(), traj_inst<FiberLane<5, 1, 1>, 2>(),   // 5- and 6-level fastest subsystem
    traj_inst<FiberLane<5, 2, 1>, 1, 1, 0, 1>(),
};
const InstPart kInstA = inst_part(kInst);

// The entry for `want` with J Neumann terms compiled in, else its run-time-J entry.  Every field matches exactly except: an entry
// with glt == 0 serves any group size, a query with nw == 0 takes the entry's own warp count, pipe is compared as zero / non-zero.
const Inst *find_inst(const InstKey &want, int J) {
    for (int jt : {J, 0})
        for (const InstPart *part : {&kInstA, &kInstB, &kInstC, &kInstD, &kInstE, &kInstF, &kInstG})
            for (const Inst *i = part->inst; i < part->inst + part->count; ++i) {
                const InstKey &k = i->key;
                if (k.kind == want.kind && k.R == want.R && k.C == want.C && k.NC == want.NC && k.WQ == want.WQ && k.LMASK == want.LMASK &&
                    k.UPL == want.UPL && k.obj2 == want.obj2 && k.jacobi == want.jacobi && k.hx == want.hx &&
                    k.general_hanti == want.general_hanti && k.NF == want.NF && k.jt == jt && (k.glt == 0 || k.glt == want.glt) &&
                    (want.nw == 0 || k.nw == want.nw) && (k.pipe != 0) == (want.pipe != 0) && k.seg == want.seg && k.hist == want.hist) return i;
            }
    return nullptr;
}

// The query of a plan on problem P: the layout comes from the plan, what the kernel must compute from the problem.
InstKey query(const InstKey &layout, const DevProblem &P) {
    InstKey q = layout;
    q.obj2 = P.objFuncType != 1;
    q.jacobi = P.solver != 1;
    return q;
}

double value_at(const HostOps &H, int o, int r, int c) {
    const int *rp = H.rowptr + o * (H.n + 1);
    double v = 0.0;
    for (int p = rp[r]; p < rp[r + 1]; ++p) if (H.col[p] == c) v += H.val[p];
    return v;
}

bool upload_plan(TrajPlan *pl, const std::vector<int> &pi, const std::vector<double> &pd, const std::vector<double> &d0,
                 const std::vector<double> &w) {
    bool ok = cudaMalloc(&pl->d_i, (pi.size() + 1) * sizeof(int)) == cudaSuccess && cudaMalloc(&pl->d_d, (pd.size() + 1) * sizeof(double)) == cudaSuccess &&
              cudaMalloc(&pl->d_d0, d0.size() * sizeof(double)) == cudaSuccess && cudaMalloc(&pl->d_w, w.size() * sizeof(double)) == cudaSuccess;
    if (!ok) return false;
    cudaMemcpy(pl->d_i, pi.data(), pi.size() * sizeof(int), cudaMemcpyHostToDevice);
    cudaMemcpy(pl->d_d, pd.data(), pd.size() * sizeof(double), cudaMemcpyHostToDevice);
    cudaMemcpy(pl->d_d0, d0.data(), d0.size() * sizeof(double), cudaMemcpyHostToDevice);
    cudaMemcpy(pl->d_w, w.data(), w.size() * sizeof(double), cudaMemcpyHostToDevice);
    return true;
}

// Diagonal of H0; returns false when H0 has off-diagonal entries (listed in `off` as (row, col, value) if given).
struct OffDiag { int r, c; double v; };
bool h0_diagonal(const HostOps &H, std::vector<double> &d0, std::vector<OffDiag> *off = nullptr) {
    d0.assign(H.n, 0.0);
    bool diag = true;
    for (int r = 0; r < H.n; ++r)
        for (int p = H.rowptr[r]; p < H.rowptr[r + 1]; ++p) {
            if (H.col[p] == r) d0[r] = H.val[p];
            else if (H.val[p] != 0.0) { diag = false; if (off) off->push_back({r, H.col[p], H.val[p]}); else return false; }
        }
    return diag;
}

int pow2ceil(int x) { int p = 1; while (p < x) p <<= 1; return p; }

}  // namespace

// ------------------------------------------------------------------------------------------------ planners
TrajPlan *jq_slot_plan_create(const DevProblem &P, const HostOps &H, const double *wdiag, char *err, size_t errlen) {
    const int n = H.n, m = H.m, Nc = H.Nc;
    auto no = [&](const char *why) { snprintf(err, errlen, "%s", why); return (TrajPlan *)nullptr; };
    if (P.wreal || P.any_unc) return no("dense forbidden-state weights / uncoupled controls run on the generic kernel");
    if (P.solver != 1) return no("Jacobi solver (data-dependent sweep count) runs on the generic kernel");
    if (n > 128) return no("n > 128");
    std::vector<double> d0;
    if (!h0_diagonal(H, d0)) return no("Hconst has off-diagonal entries");
    int WQ = 0;
    std::vector<std::vector<std::vector<int>>> cols(n, std::vector<std::vector<int>>(Nc));
    for (int q = 0; q < Nc; ++q)
        for (int r = 0; r < n; ++r) {
            std::vector<int> &cc = cols[r][q];
            for (int o : {1 + q, 1 + Nc + q}) {
                const int *rp = H.rowptr + o * (n + 1);
                for (int p = rp[r]; p < rp[r + 1]; ++p) {
                    bool have = false;
                    for (int x : cc) have |= (x == H.col[p]);
                    if (!have) cc.push_back(H.col[p]);
                }
            }
            WQ = (int)cc.size() > WQ ? (int)cc.size() : WQ;
        }
    if (WQ > 2) return no("more than 2 entries per row and control (not a ladder-type control Hamiltonian)");
    WQ = 2;
    int NL = 2;
    while (NL < 32 && NL < n) NL <<= 1;
    while (NL < 32 && NL < Nc * H.Nfreq * 2) NL <<= 1;
    if (NL < Nc * H.Nfreq * 2) return no("more (control, frequency) pairs than lanes");
    const int R = (n + NL - 1) / NL;
    InstKey key{2, R, 1, Nc, WQ, 0, 1};
    key.glt = NL;
    for (int c = 1; c <= 4; ++c) if (m % c == 0 && R * c <= 4) key.C = c;
    while (key.C >= 1 && (m % key.C != 0 || !find_inst(query(key, P), 0))) --key.C;     // the widest instantiated C that divides m
    if (key.C < 1) return no("no slot instantiation for this (rows per lane, columns per lane, controls, objFuncType)");
    const int C = key.C;

    TrajPlan *pl = new TrajPlan();
    pl->key = key;
    pl->NL = NL; pl->NLR = NL * R; pl->GPT = m / C; pl->CPG = C;
    pl->ngroups = TRAJ_WARPS * (32 / NL);
    pl->TPC = pl->ngroups / pl->GPT;
    pl->exch_per_unit = 4 * pl->NLR * C;      // 2 parities x 2 blocks per round
    if (pl->TPC < 1) { delete pl; return no("a trajectory does not fit in one CTA"); }
    const int NLR = pl->NLR;
    std::vector<int> pos((size_t)NLR * Nc * WQ);
    std::vector<double> hv((size_t)NLR * Nc * WQ * 2, 0.0), d0p(NLR, 0.0), wp(NLR, 0.0);
    for (int r = 0; r < NLR; ++r) {
        if (r < n) { d0p[r] = d0[r]; wp[r] = wdiag[r]; }
        for (int q = 0; q < Nc; ++q)
            for (int e = 0; e < WQ; ++e) {
                const size_t ix = ((size_t)r * Nc + q) * WQ + e;
                pos[ix] = r;                                     // padding: own position, zero coefficients
                if (r < n && e < (int)cols[r][q].size()) {
                    const int c = cols[r][q][e];
                    pos[ix] = c;
                    hv[2 * ix] = value_at(H, 1 + q, r, c);
                    hv[2 * ix + 1] = value_at(H, 1 + Nc + q, r, c);
                }
            }
    }
    if (!upload_plan(pl, pos, hv, d0p, wp)) { jq_traj_plan_destroy(pl); return no("cudaMalloc failed for the slot plan"); }
    err[0] = 0;
    return pl;
}

// Fibre layout: find R such that control q is either "local" (couples only rows r, r+-1 inside a block of R
// consecutive rows) or "remote" (couples row k of fibre rho only to row k of <= 2 other fibres, with a coefficient
// that does not depend on k).  True for Kronecker ladder operators with the first subsystem of size R.
TrajPlan *jq_fiber_plan_create(const DevProblem &P, const HostOps &H, const double *wdiag, char *err, size_t errlen, int pipe) {
    const int n = H.n, m = H.m, Nc = H.Nc;
    auto no = [&](const char *why) { snprintf(err, errlen, "%s", why); return (TrajPlan *)nullptr; };
    if (P.wreal || P.any_unc) return no("dense forbidden-state weights / uncoupled controls run on the generic kernel");
    std::vector<double> d0;
    std::vector<OffDiag> h0off;
    const bool h0diag = h0_diagonal(H, d0, &h0off);
    // block size: first break of control 0's first off-diagonals
    int R = n;
    for (int r = 0; r + 1 < n; ++r) {
        bool any = false;
        for (int o : {1, 1 + Nc}) any |= value_at(H, o, r, r + 1) != 0.0 || value_at(H, o, r + 1, r) != 0.0;
        if (!any) { R = r + 1; break; }
    }
    if (n % R != 0) return no("rows do not split into equal fibres");
    if (R < 2 || R > 6) return no("fibre length not instantiated");
    const int nfib = n / R;
    int LMASK = 0;
    struct Rem { int off[2]; double hs[2], ha[2]; };
    std::vector<std::vector<Rem>> rem(nfib, std::vector<Rem>(Nc));
    for (int q = 0; q < Nc; ++q) {
        bool local = false, remote = false;
        for (int o : {1 + q, 1 + Nc + q}) {
            const int *rp = H.rowptr + o * (n + 1);
            for (int r = 0; r < n; ++r)
                for (int p = rp[r]; p < rp[r + 1]; ++p) {
                    if (H.val[p] == 0.0) continue;
                    const int c = H.col[p];
                    if (r / R == c / R) { if (c != r + 1 && c != r - 1) return no("control couples inside a fibre beyond nearest neighbours"); local = true; }
                    else { if (r % R != c % R) return no("control couples different levels of different fibres"); remote = true; }
                }
        }
        if (local && remote) return no("control is neither purely local nor purely remote");
        if (local || !remote) LMASK |= 1 << q;       // an all-zero control is trivially local
        if (remote) {
            for (int f = 0; f < nfib; ++f) {
                Rem &x = rem[f][q];
                x.off[0] = x.off[1] = 0; x.hs[0] = x.hs[1] = x.ha[0] = x.ha[1] = 0.0;
                for (int f2 = 0; f2 < nfib; ++f2) {
                    if (f2 == f) continue;
                    const double s0 = value_at(H, 1 + q, f * R, f2 * R), a0 = value_at(H, 1 + Nc + q, f * R, f2 * R);
                    bool nz = s0 != 0.0 || a0 != 0.0;
                    for (int k = 1; k < R; ++k) {
                        const double sk = value_at(H, 1 + q, f * R + k, f2 * R + k), ak = value_at(H, 1 + Nc + q, f * R + k, f2 * R + k);
                        if (sk != s0 || ak != a0) return no("remote coupling is not uniform along the fibre");
                    }
                    if (!nz) continue;
                    const int side = f2 < f ? 0 : 1;             // entry 0 = lower neighbour fibre, entry 1 = upper
                    if (x.off[side] != 0) return no("more than one neighbour fibre on one side");
                    x.off[side] = f2 - f; x.hs[side] = s0; x.ha[side] = a0;
                }
            }
        }
    }
    // AS: Hanti = upper(Hsym) - lower(Hsym) for every control (the a - a' / a + a' pair of ladder operators)
    bool AS = true;
    for (int q = 0; q < Nc && AS; ++q) {
        if ((LMASK >> q) & 1) {
            for (int r = 0; r + 1 < n && AS; ++r) {
                if ((r + 1) % R == 0) continue;
                AS = value_at(H, 1 + Nc + q, r, r + 1) == value_at(H, 1 + q, r, r + 1) &&
                     value_at(H, 1 + Nc + q, r + 1, r) == -value_at(H, 1 + q, r + 1, r);
            }
        } else {
            for (int f = 0; f < nfib && AS; ++f) AS = rem[f][q].ha[0] == -rem[f][q].hs[0] && rem[f][q].ha[1] == rem[f][q].hs[1];
        }
    }
    // off-diagonal drift: only exchange couplings between the fibre subsystem and a remote one, i.e. entries
    // (fibre f, level k) <- (lower neighbour fibre of control q, level k+1) or (upper neighbour fibre, level k-1)
    int HX = 0;
    std::vector<double> xco;                       // [fibre][control][R-1][lo, hi]
    if (!h0diag) {
        if (P.objFuncType != 1 || P.solver != 1) return no("off-diagonal Hconst: only objFuncType 1 with the Neumann solver is instantiated");
        xco.assign((size_t)nfib * Nc * (R - 1) * 2, 0.0);
        for (const OffDiag &e : h0off) {
            const int f = e.r / R, k = e.r % R, f2 = e.c / R, k2 = e.c % R;
            int hit = -1, side = f2 < f ? 0 : 1;
            for (int q = 0; q < Nc && hit < 0; ++q)
                if (!((LMASK >> q) & 1) && f2 != f && rem[f][q].off[side] == f2 - f) hit = q;
            if (hit < 0 || k2 != (side == 0 ? k + 1 : k - 1))
                return no("Hconst has off-diagonal entries that are not exchange couplings with the fibre subsystem");
            xco[(((size_t)f * Nc + hit) * (R - 1) + (side == 0 ? k : k - 1)) * 2 + side] += e.v;
            HX |= 1 << hit;
        }
        HX = ((1 << Nc) - 1) & ~LMASK;             // one instantiation per shape: every remote control carries (possibly zero) coefficients
    }
    if (LMASK != 1 && LMASK != (1 << Nc) - 1) return no("only control 1 local (or all local) is instantiated");
    if (Nc > 1 && LMASK == (1 << Nc) - 1) return no("several local controls are not instantiated");
    const int NL = pow2ceil(nfib);
    if (NL > 32) return no("more than 32 fibres per column");
    int GL = pow2ceil(NL * m) > 32 ? 32 : pow2ceil(NL * m);
    if (NL == 1 && (32 / m) * m > (32 / GL) * m) GL = m;     // one lane per column: pack m-lane groups without padding
    const int CPG = GL / NL, GPT = (m + CPG - 1) / CPG;
    const int NU = Nc * H.Nfreq * 2, UPL = (NU + GL - 1) / GL;
    if (UPL > 2) return no("too many (control, frequency) pairs for the group size");
    InstKey key{3, R, 1, Nc, 2, LMASK, UPL};
    key.hx = HX != 0; key.general_hanti = !AS; key.glt = GL;
    const bool found = find_inst(query(key, P), 0) != nullptr;
    // Jacobi: residual norm over the whole block = one group reduction -> one group per trajectory only
    if (P.solver != 1 && (!found || GPT != 1)) return no("Jacobi solver: no fibre instantiation for this shape (or the trajectory spans several groups)");
    if (HX && !found) return no("off-diagonal (exchange) Hconst: no fibre instantiation for this shape");
    if (!found) return no("no fibre instantiation for this (fibre length, controls, updaters per lane, Hanti form, objFuncType)");
    // lane offsets of remote neighbours must stay inside the column block of NL lanes
    TrajPlan *pl = new TrajPlan();
    pl->key = key;
    pl->NL = NL; pl->NLR = NL * R; pl->GPT = GPT; pl->CPG = CPG;
    pl->ngroups = TRAJ_WARPS * (32 / GL);
    pl->TPC = pl->ngroups / GPT;
    pl->exch_per_unit = 4 * R * 32;           // 2 parities x 2 fibres per round
    if (pl->TPC < 1) {
        // a trajectory wider than 4 warps (e.g. 45 x 12): the 8-warp instantiations (plain problems only)
        InstKey wide = query(key, P);
        wide.nw = 8;
        if (GPT <= 8 && find_inst(wide, 0)) { pl->key.nw = 8; pl->ngroups = 8 * (32 / GL); pl->TPC = pl->ngroups / GPT; }
        else { delete pl; return no("a trajectory does not fit in one CTA"); }
    }
    const int perq = 4 * (R - 1) + 4 + (HX ? 2 * (R - 1) : 0), per = Nc * perq;
    std::vector<int> pi((size_t)NL * Nc * 2, 0);
    std::vector<double> pd((size_t)NL * per, 0.0), d0p((size_t)NL * R, 0.0), wp((size_t)NL * R, 0.0);
    for (int f = 0; f < NL; ++f) {
        if (f >= nfib) continue;                       // padding fibres: zero coefficients, own lane
        for (int k = 0; k < R; ++k) { d0p[f * R + k] = d0[f * R + k]; wp[f * R + k] = wdiag[f * R + k]; }
        for (int q = 0; q < Nc; ++q) {
            double *c = pd.data() + (size_t)f * per + q * perq;
            if (HX)
                for (int k = 0; k < R - 1; ++k)
                    for (int sd = 0; sd < 2; ++sd) c[4 * (R - 1) + 4 + 2 * k + sd] = xco[(((size_t)f * Nc + q) * (R - 1) + k) * 2 + sd];
            if ((LMASK >> q) & 1) {
                for (int k = 0; k < R - 1; ++k) {
                    const int r = f * R + k;
                    c[4 * k] = value_at(H, 1 + q, r, r + 1);        // Hs[r, r+1]: x_{k+1} -> row k
                    c[4 * k + 1] = value_at(H, 1 + q, r + 1, r);    // Hs[r+1, r]: x_k -> row k+1
                    c[4 * k + 2] = value_at(H, 1 + Nc + q, r, r + 1);
                    c[4 * k + 3] = value_at(H, 1 + Nc + q, r + 1, r);
                }
            } else {
                for (int e = 0; e < 2; ++e) {
                    pi[((size_t)f * Nc + q) * 2 + e] = rem[f][q].off[e];
                    c[4 * (R - 1) + 2 * e] = rem[f][q].hs[e];
                    c[4 * (R - 1) + 2 * e + 1] = rem[f][q].ha[e];
                }
            }
        }
    }
    if (pipe) {      // pipelined roles: single-fibre columns only (no exchange buffer), plain problems; NW = warps that hold one group set
        const int nwp = (GPT * GL + 31) / 32;
        pl->key.pipe = 1; pl->key.nw = nwp;
        if (LMASK != (1 << Nc) - 1 || !find_inst(query(pl->key, P), P.J)) { delete pl; return no("no pipelined fibre instantiation for this shape"); }
        pl->ngroups = nwp * (32 / GL); pl->TPC = pl->ngroups / GPT;
    }
    if (!upload_plan(pl, pi, pd, d0p, wp)) { jq_traj_plan_destroy(pl); return no("cudaMalloc failed for the fibre plan"); }
    err[0] = 0;
    return pl;
}


// Tile layout: every subsystem has 4 levels, control q is the ladder pair (a_q + a_q', a_q - a_q') of subsystem q (row stride
// 4^q), Hconst diagonal.  NF in-lane directions, then NT tiled directions cut in mirrored halves, the others remote (see TileLane).
TrajPlan *jq_tile_plan_create(const DevProblem &P, const HostOps &H, const double *wdiag, int NT, int NF, char *err, size_t errlen, int pipe,
                              bool seg) {
    const int n = H.n, m = H.m, Nc = H.Nc;
    auto no = [&](const char *why) { snprintf(err, errlen, "%s", why); return (TrajPlan *)nullptr; };
    if (P.wreal || P.any_unc) return no("dense forbidden-state weights / uncoupled controls run on the generic kernel");
    if (P.solver != 1 || P.objFuncType != 1) return no("tile layout: only objFuncType 1 with the Neumann solver is instantiated");
    if (Nc < 2 || Nc > 3) return no("tile layout: 2 or 3 controls");
    if (NT < 0 || NF < 0 || NF + NT > Nc) return no("tile layout: bad number of in-lane / tiled directions");
    int n4 = 1;
    for (int q = 0; q < Nc; ++q) n4 *= 4;
    if (n != n4) return no("tile layout: every subsystem must have 4 levels");
    std::vector<double> d0;
    if (!h0_diagonal(H, d0)) return no("tile layout: Hconst has off-diagonal entries");
    std::vector<double> sq((size_t)Nc * 3, 0.0);        // ladder coefficient between levels l and l+1 of subsystem q
    for (int q = 0, stride = 1; q < Nc; ++q, stride *= 4) {
        for (int o : {1 + q, 1 + Nc + q}) {
            const int *rp = H.rowptr + o * (n + 1);
            for (int r = 0; r < n; ++r)
                for (int p = rp[r]; p < rp[r + 1]; ++p) {
                    if (H.val[p] == 0.0) continue;
                    const int c = H.col[p], lo = r < c ? r : c, hi = r < c ? c : r;
                    if (hi - lo != stride || (lo / stride) % 4 == 3) return no("tile layout: control is not a ladder operator of its subsystem");
                }
        }
        for (int l = 0; l < 3; ++l) sq[q * 3 + l] = value_at(H, 1 + q, l * stride, (l + 1) * stride);
        for (int r = 0; r < n; ++r) {
            const int l = (r / stride) % 4;
            if (l == 3) continue;
            const double s = sq[q * 3 + l];
            if (value_at(H, 1 + q, r, r + stride) != s || value_at(H, 1 + q, r + stride, r) != s ||
                value_at(H, 1 + Nc + q, r, r + stride) != s || value_at(H, 1 + Nc + q, r + stride, r) != -s)
                return no("tile layout: control is not the (a + a', a - a') pair with level-only coefficients");
        }
    }
    int NL = 1 << NT;
    for (int q = NF + NT; q < Nc; ++q) NL *= 4;
    const int GL = pow2ceil(NL * m) > 32 ? 32 : pow2ceil(NL * m);
    if (NL > 32) return no("tile layout: more than 32 lanes per column");
    const int CPG = GL / NL, GPT = (m + CPG - 1) / CPG;
    const int NU = Nc * H.Nfreq * 2, UPL = (NU + GL - 1) / GL;
    if (UPL > 1) return no("tile layout: too many (control, frequency) pairs for the group size");
    const int nwp = pipe ? (GPT * GL + 31) / 32 : 0;
    InstKey key{4, NT, 1, Nc, 0, 0, UPL};
    key.glt = GL; key.nw = nwp; key.pipe = pipe ? 1 : 0;      // nw = 0: the 4 x 4 x 4 tiles run 8 warps per CTA
    key.NF = NF;
    InstKey want = query(key, P);
    want.seg = seg;
    if (!find_inst(want, P.J)) return no("tile layout: no instantiation");
    TrajPlan *pl = new TrajPlan();
    pl->key = key;
    pl->NL = NL; pl->NLR = n; pl->GPT = GPT; pl->CPG = CPG;
    pl->ngroups = TRAJ_WARPS * (32 / GL);
    pl->TPC = pl->ngroups / GPT;
    pl->exch_per_unit = 0;                         // shuffles only
    if (pipe) { pl->ngroups = nwp * (32 / GL); pl->TPC = pl->ngroups / GPT; }
    if (pl->TPC < 1) { delete pl; return no("a trajectory does not fit in one CTA"); }
    const int nrem = Nc - NF - NT, per = 3 * NF + 3 * NT + 2 * nrem;
    std::vector<int> pi((size_t)NL * (nrem > 0 ? nrem : 1) * 2, 0);
    std::vector<double> pd((size_t)NL * per, 0.0), d0p(n), wp(n);
    for (int r = 0; r < n; ++r) { d0p[r] = d0[r]; wp[r] = wdiag[r]; }
    for (int rho = 0; rho < NL; ++rho) {
        double *c = pd.data() + (size_t)rho * per;
        for (int d = 0; d < NF; ++d)
            for (int l = 0; l < 3; ++l) c[3 * d + l] = sq[d * 3 + l];
        c += 3 * NF;
        for (int d = 0; d < NT; ++d) {
            const int hb = (rho >> d) & 1, q = NF + d;
            c[3 * d] = sq[q * 3 + (hb ? 2 : 0)];
            c[3 * d + 1] = sq[q * 3 + 1];
            c[3 * d + 2] = hb ? -1.0 : 1.0;
        }
        for (int r = 0, gs = 1; r < nrem; ++r, gs *= 4) {
            const int g = ((rho >> NT) / gs) % 4, q = NF + NT + r;
            if (g > 0) { pi[((size_t)rho * nrem + r) * 2] = -(gs << NT); c[3 * NT + 2 * r] = sq[q * 3 + g - 1]; }
            if (g < 3) { pi[((size_t)rho * nrem + r) * 2 + 1] = gs << NT; c[3 * NT + 2 * r + 1] = sq[q * 3 + g]; }
        }
    }
    if (!upload_plan(pl, pi, pd, d0p, wp)) { jq_traj_plan_destroy(pl); return no("cudaMalloc failed for the tile plan"); }
    err[0] = 0;
    return pl;
}

void jq_traj_plan_destroy(TrajPlan *pl) {
    if (!pl) return;
    for (void *p : {(void *)pl->d_i, (void *)pl->d_d, (void *)pl->d_d0, (void *)pl->d_w}) if (p) cudaFree(p);
    delete pl;
}

// Segment-sweep instantiations exist only for Neumann problems on non-pipelined 4-warp (tile: their own) plans without drift
// couplings and with the ladder form of Hanti.
bool jq_seg_supported(const TrajPlan *pl, const DevProblem &P, bool second_adjoint, bool hist) {
    if (!pl || 2 * P.n > 512) return false;
    InstKey want = query(pl->key, P);
    want.seg = 1;
    want.obj2 = second_adjoint;
    want.hist = hist;
    return find_inst(want, P.J) != nullptr;
}

int jq_traj_plan_tpc(const TrajPlan *pl) { return pl ? pl->TPC : 0; }
int jq_traj_plan_lanes(const TrajPlan *pl) { return pl ? pl->GPT * pl->key.glt : 0; }

cudaError_t jq_traj_launch(TrajPlan *pl, const DevProblem &P, const LaunchArgs &A, cudaStream_t st, int *nctas, int *regs,
                           size_t *smem, int *traj_per_cta, const SegHist *hist) {
    // never substitute: Neumann for Jacobi, one adjoint set for two, no drift couplings
    InstKey want = query(pl->key, P);
    const bool seg = A.seg.nseg > 0;
    if (seg) {                  // segment sweeps of the time-parallel evaluation
        if (A.hist_r && !hist) return cudaErrorNotSupported;
        want.seg = 1;
        want.hist = hist != nullptr;        // the history VJP's paths live in their own instantiations
        // objFuncType 2/3: only the gradient sweep (mode 5) carries the second adjoint set; every other mode is the plain one
        want.obj2 = want.obj2 && A.seg.mode[0] == 5;
    }
    if (want.pipe && P.nsteps > 0x7ffffff0LL) return cudaErrorNotSupported;      // the hand-over counters are ints
    const Inst *inst = find_inst(want, P.J);
    if (!inst || (inst->key.jt != 0 && inst->key.jt != P.J)) return cudaErrorNotSupported;
    TrajParams S{};
    S.P = P; S.A = A;
    if (seg && hist) S.H = *hist;
    S.NL = pl->NL; S.NLR = pl->NLR; S.GL = pl->key.glt; S.GPT = pl->GPT; S.CPG = pl->CPG;
    S.plan_i = pl->d_i; S.plan_d = pl->d_d; S.plan_d0 = pl->d_d0; S.plan_w = pl->d_w;
    S.exch_per_unit = pl->exch_per_unit;
    S.NparS = A.Npar | 1;
    S.GPW = 32 / pl->key.glt;
    const int npts = 2 * TRAJ_CH + 2, NC = pl->key.NC;     // control-table points per chunk, with fill_table's extra point
    // warps per CTA: 4 normally; fewer when the per-CTA gradient windows / pcof staging of very long coefficient
    // vectors would not fit in shared memory (the kernel only uses blockDim.x and the counts below)
    int nw = inst->key.nw, TPC = 0, ngroups = 0;
    size_t bytes = 0;
    const int pipe = inst->key.pipe;
    const int kind = pl->key.kind, Eper = kind == 4 ? (1 << (2 * pl->key.NF + pl->key.R)) : kind == 3 ? pl->key.R : pl->key.R * pl->key.C;      // elements per lane
    for (; nw >= 1; nw >>= 1) {
        ngroups = nw * S.GPW;
        TPC = ngroups / pl->GPT;
        if (TPC < 1) return cudaErrorInvalidConfiguration;
        int o = 0;
        auto take = [&](int cnt) { int at = o; o += (cnt + 1) & ~1; return at; };   // keep 16-byte alignment
        S.o_exch = take(pl->exch_per_unit * (kind == 2 ? ngroups : nw));
        S.o_pcof = take(TPC * S.NparS);
        S.o_gsm = take(ngroups * A.Npar);
        S.o_times = take(npts);                              // control table: one contiguous block per role
        S.o_tabb = take(3 * npts);
        S.o_tabph = take(2 * npts * NC * P.Nfreq);
        S.o_tabpq = take(npts * TPC * 2 * NC);
        S.o_tabk = take((npts + 1) / 2);
        S.tab_role_stride = o - S.o_times;
        if (pipe) take((TRAJ_TABS - 1) * S.tab_role_stride);   // the other table buffers of the table warp's ring
        S.o_red = take(ngroups * 4);
        S.o_tred = take(ngroups * NC * 5);
        S.o_gsm2 = take(P.objFuncType != 1 ? ngroups * A.Npar : 0);
        S.o_ring = take(pipe ? TRAJ_RING * (3 * Eper + 5 * NC) * nw * 32 : 0);      // state hand-over ring, then the trace ring
        S.o_cnt = take(pipe ? 2 * nw + (3 * nw + 2) / 2 + 1 : 0);       // int counters: 4 per warp triple, 1 per consumer warp, 1 for the tables
        bytes = (size_t)o * sizeof(double);
        if (bytes <= 227 * 1024 || pipe) break;              // pipelined instantiations have a fixed number of warps
    }
    if (nw < 1) return cudaErrorInvalidConfiguration;       // does not fit even with one warp per CTA: caller falls back
    S.TPC = TPC; S.ngroups = ngroups;
    if (bytes > 227 * 1024) return cudaErrorInvalidConfiguration;
    cudaError_t e = cudaFuncSetAttribute(inst->fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return e;
    cudaFuncAttributes fa;
    e = cudaFuncGetAttributes(&fa, inst->fn);
    if (e != cudaSuccess) return e;
    int grid = (A.ntraj + TPC - 1) / TPC;
    if (seg) {                  // CTAs per (mode, segment): sub-trajectories = blocks of m unit vectors x trajectories, or the trajectories
        const int nblk = (2 * P.n + P.m - 1) / P.m;
        auto ctas = [&](int mode) {
            if (mode == 0) return 0LL;
            const long long per = (mode == 1 || mode == 3) ? (long long)nblk * A.ntraj : (long long)A.ntraj;
            return (long long)(A.seg.seg_cnt > 0 ? A.seg.seg_cnt : A.seg.nseg) * ((per + TPC - 1) / TPC);
        };
        const long long c0 = ctas(A.seg.mode[0]), c1 = ctas(A.seg.mode[1]), c2 = ctas(S.H.mode2);
        if (c0 + c1 + c2 > 0x7fffffffLL || c0 + c1 + c2 < 1) return cudaErrorInvalidConfiguration;
        S.A.seg.ctas0 = (int)c0;
        S.H.ctas1 = (int)(c0 + c1);
        grid = (int)(c0 + c1 + c2);
    }
    inst->fn<<<grid, (pipe == 1 ? 3 * nw + 1 : pipe == 2 ? 2 * nw : nw) * 32, bytes, st>>>(S);
    if (nctas) *nctas = grid;
    if (regs) *regs = fa.numRegs;
    if (smem) *smem = bytes;
    if (traj_per_cta) *traj_per_cta = TPC;
    return cudaGetLastError();
}
