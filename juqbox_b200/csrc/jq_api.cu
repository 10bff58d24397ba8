// C-ABI layer (include/juqbox_b200.h): problem upload, operator tables, kernel selection, launches and the
// per-candidate weighted reduction.  No torch types, no CPU fallback.
#include "jq_common.h"
#include "../../include/juqbox_b200.h"

#include <dlfcn.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

static thread_local char g_err[512] = "";

static int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
#define CU(call)                                                                                       \
    do {                                                                                               \
        cudaError_t e_ = (call);                                                                       \
        if (e_ != cudaSuccess) return fail(JQ_ERR_CUDA, "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

// ---- NCCL through dlopen: only the five entry points the sample-sharded all-reduce needs ----
typedef struct ncclComm *nccl_comm_t;
typedef struct { char internal[128]; } nccl_uid_t;
struct NcclApi {
    int (*GetUniqueId)(nccl_uid_t *) = nullptr;
    int (*CommInitRank)(nccl_comm_t *, int, nccl_uid_t, int) = nullptr;
    int (*CommDestroy)(nccl_comm_t) = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, nccl_comm_t, cudaStream_t) = nullptr;
    int (*AllGather)(const void *, void *, size_t, int, nccl_comm_t, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    bool ok = false;
};
static NcclApi g_nccl;
static int load_nccl();

struct jq_handle {
    nccl_comm_t comm = nullptr;
    int comm_rank = 0, comm_size = 1;
    bool cooperative = false;           // jq_comm_set_cooperative: every rank passes the same arguments, the time segments of kernel 7 are shared out
    int device = 0;
    DevProblem P{};
    int n = 0, m = 0, Nc = 0, Nfreq = 0, pfid = 2;       // Nc: coupled + uncoupled controls
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaEvent_t ev_done = nullptr;      // end of the last evaluation: calls on another stream wait for it (shared scratch buffers)
    cudaStream_t last_stream = nullptr;
    bool have_last = false;
    std::vector<void *> owned;          // device allocations freed at destroy
    double *d_vtr = nullptr, *d_vti = nullptr;
    // host copies of the row-wise operators (for the planners)
    std::vector<int> rowptr, col;
    std::vector<double> val;
    TrajPlan *slot = nullptr, *fiber = nullptr, *tile = nullptr, *tile_lat = nullptr;     // tile_lat: fewest elements per lane (small batches)
    bool dense_ok = false;              // the dense (FP64 MMA) kernel can serve this problem
    bool dense_auto = false;            // ... and the operators are dense enough for it to beat the row-wise generic kernel
    char dense_reason[128] = "";
    int lat_ntraj = 0;                  // automatic mode: launches with at most this many trajectories use the latency layout
    // time-parallel evaluation (jq_seg.cu, kernel id 7): plan whose instantiations have segment sweeps (the non-pipelined latency
    // tile layout, else the fibre plan -- then shared with `fiber`), workspace, segments (0 = automatic)
    TrajPlan *seg_plan = nullptr, *seg_prop = nullptr, *seg_obj = nullptr;      // seg_prop: plan of the propagator launch (nullptr: seg_plan); seg_obj: of the gradient sweep for objFuncType 2/3
    double *d_seg = nullptr; size_t cap_seg = 0;
    double *d_segt = nullptr; size_t cap_segt = 0; int segt_nseg = 0; std::vector<double> segt;
    int seg_nseg = 0, seg_ntraj = 0, sms = 148, last_nseg = 0;
    char slot_reason[256] = "", fiber_reason[256] = "", tile_reason[256] = "";
    int kernel_pref = 0;
    bool prefer_tile = true;            // automatic mode: tile layout before the fibre layout
    // growable scratch
    double *d_scal = nullptr, *d_grad = nullptr, *d_igrad = nullptr;
    size_t cap_traj = 0, cap_grad = 0, cap_igrad = 0;
    double *d_in = nullptr;  size_t cap_in = 0;    // staged host inputs
    double *d_out = nullptr; size_t cap_out = 0;   // staged host outputs
    // last-evaluation cache of the fused callback entry (jq_eval_f_grad; src/ipopt_interface.jl:27-31)
    bool cache_valid = false;
    std::vector<double> c_pcof, c_shift, c_w, c_igrad, c_lgrad;
    double c_infid = 0.0, c_leak = 0.0;
    // last-evaluation facts
    int last_kernel = 0, last_launches = 0, last_ctas = 0, last_regs = 0, last_tpc = 1, last_traj_launches = 1;
    size_t last_smem = 0;
    bool timed = false;
};

template <class T>
static int upload(jq_handle *h, const T *src, size_t count, T **dst) {
    void *p = nullptr;
    CU(cudaMalloc(&p, std::max<size_t>(count, 1) * sizeof(T)));
    h->owned.push_back(p);
    if (count) CU(cudaMemcpy(p, src, count * sizeof(T), cudaMemcpyHostToDevice));
    *dst = (T *)p;
    return 0;
}

static int grow(double **buf, size_t *cap, size_t need) {
    if (need <= *cap) return 0;
    if (*buf) cudaFree(*buf);
    *buf = nullptr;
    *cap = 0;
    CU(cudaMalloc((void **)buf, need * sizeof(double)));
    *cap = need;
    return 0;
}

// operator -> sorted CSR rows appended to (rowptr, col, val); `force_diag` inserts missing diagonal entries.
static int append_rows(const jq_operator &op, int n, bool force_diag, std::vector<int> &rowptr, std::vector<int> &col,
                       std::vector<double> &val, const char *name) {
    std::vector<std::vector<std::pair<int, double>>> rows(n);
    if (op.format == JQ_DENSE) {
        if (!op.nzval) return fail(JQ_ERR_ARG, "%s: dense operator without values", name);
        for (int c = 0; c < n; ++c)
            for (int r = 0; r < n; ++r) {
                const double v = op.nzval[(size_t)c * n + r];
                if (v != 0.0) rows[r].push_back({c, v});
            }
    } else if (op.format == JQ_CSC) {
        if (!op.colptr || (op.nnz > 0 && (!op.rowval || !op.nzval))) return fail(JQ_ERR_ARG, "%s: CSC operator with null arrays", name);
        if (op.colptr[0] != 0 || op.colptr[n] != op.nnz) return fail(JQ_ERR_ARG, "%s: CSC colptr must be 0-based and end at nnz", name);
        for (int c = 0; c < n; ++c)
            for (int64_t p = op.colptr[c]; p < op.colptr[c + 1]; ++p) {
                const int64_t r = op.rowval[p];
                if (r < 0 || r >= n) return fail(JQ_ERR_ARG, "%s: CSC row index %lld out of range", name, (long long)r);
                rows[r].push_back({c, op.nzval[p]});
            }
    } else {
        return fail(JQ_ERR_ARG, "%s: unknown operator format %d", name, op.format);
    }
    for (int r = 0; r < n; ++r) {
        auto &row = rows[r];
        std::sort(row.begin(), row.end(), [](const std::pair<int, double> &a, const std::pair<int, double> &b) { return a.first < b.first; });
        if (force_diag) {
            bool has = false;
            for (auto &e : row) has |= (e.first == r);
            if (!has) {
                row.push_back({r, 0.0});
                std::sort(row.begin(), row.end(), [](const std::pair<int, double> &a, const std::pair<int, double> &b) { return a.first < b.first; });
            }
        }
        rowptr.push_back((int)col.size());
        for (auto &e : row) { col.push_back(e.first); val.push_back(e.second); }
    }
    rowptr.push_back((int)col.size());
    return 0;
}

static int load_nccl() {
    if (g_nccl.ok) return 0;
    void *lib = nullptr;
    for (const char *name : {"libnccl.so.2", "libnccl.so"}) {
        lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
        if (lib) break;
    }
    if (!lib) return fail(JQ_ERR_ARG, "NCCL not found (dlopen libnccl.so.2): %s", dlerror());
#define SYM(field, name)                                                              \
    *(void **)(&g_nccl.field) = dlsym(lib, name);                                     \
    if (!g_nccl.field) return fail(JQ_ERR_ARG, "NCCL symbol %s missing", name)
    SYM(GetUniqueId, "ncclGetUniqueId");
    SYM(CommInitRank, "ncclCommInitRank");
    SYM(CommDestroy, "ncclCommDestroy");
    SYM(AllReduce, "ncclAllReduce");
    SYM(AllGather, "ncclAllGather");
    SYM(GroupStart, "ncclGroupStart");
    SYM(GroupEnd, "ncclGroupEnd");
    SYM(GetErrorString, "ncclGetErrorString");
#undef SYM
    g_nccl.ok = true;
    return 0;
}
#define NC(call)                                                                                           \
    do {                                                                                                   \
        int r_ = (call);                                                                                   \
        if (r_ != 0) return fail(JQ_ERR_CUDA, "%s: %s", #call, g_nccl.GetErrorString ? g_nccl.GetErrorString(r_) : "nccl error"); \
    } while (0)

extern "C" int jq_comm_unique_id(void *id128) {
    if (!id128) return fail(JQ_ERR_ARG, "jq_comm_unique_id: null argument");
    int rc = load_nccl();
    if (rc) return rc;
    NC(g_nccl.GetUniqueId((nccl_uid_t *)id128));
    return 0;
}

extern "C" int jq_comm_init(jq_handle *h, int32_t rank, int32_t nranks, const void *id128) {
    if (!h || !id128 || nranks < 1 || rank < 0 || rank >= nranks) return fail(JQ_ERR_ARG, "jq_comm_init: bad argument");
    int rc = load_nccl();
    if (rc) return rc;
    if (h->comm) { g_nccl.CommDestroy(h->comm); h->comm = nullptr; }
    CU(cudaSetDevice(h->device));
    nccl_uid_t id;
    memcpy(&id, id128, sizeof(id));
    NC(g_nccl.CommInitRank(&h->comm, nranks, id, rank));
    h->comm_rank = rank; h->comm_size = nranks;
    return 0;
}

// In-place all-gather of `count` doubles per rank (rank r's share already sits at buf + r * count).
static int seg_allgather(void *ctx, double *buf, size_t count, cudaStream_t st) {
    jq_handle *h = static_cast<jq_handle *>(ctx);
    return g_nccl.AllGather(buf + (size_t)h->comm_rank * count, buf, count, 8 /*ncclDouble*/, h->comm, st);
}

extern "C" int jq_comm_set_cooperative(jq_handle *h, int32_t on) {
    if (!h) return fail(JQ_ERR_ARG, "jq_comm_set_cooperative: null handle");
    if (on && !h->comm) return fail(JQ_ERR_ARG, "jq_comm_set_cooperative: attach a communicator first (jq_comm_init)");
    h->cooperative = on != 0;
    return 0;
}

extern "C" int jq_comm_destroy(jq_handle *h) {
    if (!h) return fail(JQ_ERR_ARG, "jq_comm_destroy: null handle");
    if (h->comm) { CU(cudaSetDevice(h->device)); cudaStreamSynchronize(h->stream); g_nccl.CommDestroy(h->comm); h->comm = nullptr; }
    h->comm_size = 1; h->comm_rank = 0; h->cooperative = false;
    return 0;
}

extern "C" const char *jq_last_error(void) { return g_err; }
extern "C" const char *jq_version(void) { return "juqbox_b200 0.1 (sm_100a)"; }

extern "C" int jq_create(const jq_problem *pb, int device, jq_handle **out) {
    if (!pb || !out) return fail(JQ_ERR_ARG, "jq_create: null argument");
    *out = nullptr;
    if (pb->n < 1 || pb->m < 1 || pb->m > pb->n) return fail(JQ_ERR_ARG, "jq_create: need 1 <= m <= n (n=%d, m=%d)", pb->n, pb->m);
    if (pb->ncoupled < 0 || pb->nuncoupled < 0 || pb->ncoupled + pb->nuncoupled < 1)
        return fail(JQ_ERR_ARG, "jq_create: need at least one control Hamiltonian (ncoupled + nuncoupled >= 1)");
    if (pb->ncoupled + pb->nuncoupled > JQ_MAX_CTRL) return fail(JQ_ERR_ARG, "jq_create: at most %d control Hamiltonians", JQ_MAX_CTRL);
    if (pb->nfreq < 1 || pb->nsteps < 1 || !(pb->T > 0.0) || pb->neumann_terms < 0)
        return fail(JQ_ERR_ARG, "jq_create: need nfreq >= 1, nsteps >= 1, T > 0, neumann_terms >= 0");
    if (pb->linear_solver < 0 || pb->linear_solver > 2)
        return fail(JQ_ERR_ARG, "jq_create: linear_solver must be NEUMANN_SOLVER (1) or JACOBI_SOLVER (2), got %d", pb->linear_solver);
    if (pb->pfid_type < 1 || pb->pfid_type > 4) return fail(JQ_ERR_ARG, "jq_create: pFidType must be 1, 2, 3 or 4 (got %d)", pb->pfid_type);
    if (pb->obj_func_type < 1 || pb->obj_func_type > 3) return fail(JQ_ERR_ARG, "jq_create: objFuncType must be 1, 2 or 3");
    if (!pb->uinit || !pb->vtarget_r || !pb->vtarget_i || !pb->wdiag || !pb->cfreq || (pb->ncoupled > 0 && (!pb->hsym || !pb->hanti)))
        return fail(JQ_ERR_ARG, "jq_create: null problem array");
    if (pb->nuncoupled > 0 && (!pb->hunc || !pb->unc_is_symm || !pb->unc_rfreq)) return fail(JQ_ERR_ARG, "jq_create: null uncoupled-control array");
    if (pb->wmat_imag && !pb->wmat_real) return fail(JQ_ERR_ARG, "jq_create: wmat_imag needs wmat_real");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) return fail(JQ_ERR_CUDA, "jq_create: no CUDA device (there is no CPU fallback)");
    if (device < 0 || device >= ndev) return fail(JQ_ERR_ARG, "jq_create: device %d out of range (%d devices)", device, ndev);
    CU(cudaSetDevice(device));

    jq_handle *h = new jq_handle();
    h->device = device;
    // Controls as the kernels see them: the coupled pairs first, then one entry per uncoupled control with its operator in the
    // Hsym slot (symmetric, added to K) or in the Hanti slot (antisymmetric, added to S) and an empty partner (KS!, :2372-2387).
    const int n = pb->n, m = pb->m, Nc = pb->ncoupled + pb->nuncoupled;
    h->n = n; h->m = m; h->Nc = Nc; h->Nfreq = pb->nfreq; h->pfid = pb->pfid_type;
    const jq_operator empty{JQ_DENSE, 0, nullptr, nullptr, nullptr};
    std::vector<double> zeros((size_t)n * n, 0.0);
    jq_operator zero_op = empty;
    zero_op.nnz = (int64_t)n * n; zero_op.nzval = zeros.data();
    int rc = append_rows(pb->h0, n, true, h->rowptr, h->col, h->val, "Hconst");
    for (int q = 0; q < Nc && rc == 0; ++q) {
        const bool unc = q >= pb->ncoupled;
        const int u = q - pb->ncoupled;
        rc = append_rows(!unc ? pb->hsym[q] : (pb->unc_is_symm[u] ? pb->hunc[u] : zero_op), n, false, h->rowptr, h->col, h->val, unc ? "Hunc_ops" : "Hsym_ops");
    }
    for (int q = 0; q < Nc && rc == 0; ++q) {
        const bool unc = q >= pb->ncoupled;
        const int u = q - pb->ncoupled;
        rc = append_rows(!unc ? pb->hanti[q] : (pb->unc_is_symm[u] ? zero_op : pb->hunc[u]), n, false, h->rowptr, h->col, h->val, unc ? "Hunc_ops" : "Hanti_ops");
    }
    if (rc) { delete h; return rc; }
    std::vector<int> h0diag(n);
    for (int r = 0; r < n; ++r)
        for (int p = h->rowptr[r]; p < h->rowptr[r + 1]; ++p)
            if (h->col[p] == r) h0diag[r] = p;

    DevProblem &P = h->P;
    P.n = n; P.m = m; P.Nc = Nc; P.Nfreq = pb->nfreq; P.J = pb->neumann_terms; P.objFuncType = pb->obj_func_type;
    P.pFidType = pb->pfid_type; P.globalPhase = pb->global_phase; P.any_unc = pb->nuncoupled > 0;
    for (int q = 0; q < JQ_MAX_CTRL; ++q) { P.ctrl_kind[q] = 0; P.ctrl_rfreq[q] = 0.0; }
    for (int u = 0; u < pb->nuncoupled; ++u) {
        P.ctrl_kind[pb->ncoupled + u] = pb->unc_is_symm[u] ? 1 : 2;
        P.ctrl_rfreq[pb->ncoupled + u] = pb->unc_rfreq[u];
    }
    P.solver = pb->linear_solver == 2 ? 2 : 1; P.tol = pb->solver_tol;
    P.nsteps = pb->nsteps; P.T = pb->T;
    double *tmp = nullptr;
    int *itmp = nullptr;
#define UP(src, cnt, field)                                                        \
    do {                                                                           \
        if ((rc = upload(h, src, (size_t)(cnt), &tmp)) != 0) { jq_destroy(h); return rc; } \
        field = tmp;                                                               \
    } while (0)
#define UPI(src, cnt, field)                                                        \
    do {                                                                            \
        if ((rc = upload(h, src, (size_t)(cnt), &itmp)) != 0) { jq_destroy(h); return rc; } \
        field = itmp;                                                               \
    } while (0)
    UP(pb->uinit, n * m, P.uinit);
    UP(pb->vtarget_r, n * m, h->d_vtr);
    UP(pb->vtarget_i, n * m, h->d_vti);
    P.vtr = h->d_vtr; P.vti = h->d_vti;
    UP(pb->wdiag, n, P.wdiag);
    UP(pb->cfreq, Nc * pb->nfreq, P.cfreq);
    P.wreal = P.wimag = nullptr;
    if (pb->wmat_real) UP(pb->wmat_real, (size_t)n * n, P.wreal);
    if (pb->wmat_imag) UP(pb->wmat_imag, (size_t)n * n, P.wimag);
    UP(h->val.data(), h->val.size(), P.val);
    UPI(h->rowptr.data(), h->rowptr.size(), P.rowptr);
    UPI(h->col.data(), h->col.size(), P.col);
    UPI(h0diag.data(), n, P.h0diag);
    {   // packed copy of the operator table for the generic kernel's bulk copy
        const size_t nrp = h->rowptr.size(), nnz = h->col.size();
        const size_t off_col = nrp * sizeof(int), off_val = (off_col + nnz * sizeof(int) + 15) & ~(size_t)15;
        const size_t total = (off_val + nnz * sizeof(double) + 15) & ~(size_t)15;
        std::vector<unsigned char> blob(total, 0);
        memcpy(blob.data(), h->rowptr.data(), nrp * sizeof(int));
        memcpy(blob.data() + off_col, h->col.data(), nnz * sizeof(int));
        memcpy(blob.data() + off_val, h->val.data(), nnz * sizeof(double));
        unsigned char *dblob = nullptr;
        if ((rc = upload(h, blob.data(), total, &dblob)) != 0) { jq_destroy(h); return rc; }
        P.csr_blob = dblob; P.csr_bytes = (int)total; P.csr_off_col = (int)off_col; P.csr_off_val = (int)off_val;
    }
    P.dense_ops = nullptr;
    if (n <= 64) {   // dense row-major copies for the tensor-core kernel
        int n8 = 0, ldk = 0;
        jq_dense_padding(n, &n8, &ldk);
        std::vector<double> dn((size_t)(1 + 2 * Nc) * n8 * ldk, 0.0);
        for (int o = 0; o < 1 + 2 * Nc; ++o)
            for (int r = 0; r < n; ++r)
                for (int p2 = h->rowptr[(size_t)o * (n + 1) + r]; p2 < h->rowptr[(size_t)o * (n + 1) + r + 1]; ++p2)
                    dn[((size_t)o * n8 + r) * ldk + h->col[p2]] += h->val[p2];
        double *ddn = nullptr;
        if ((rc = upload(h, dn.data(), dn.size(), &ddn)) != 0) { jq_destroy(h); return rc; }
        P.dense_ops = ddn;
    }
#undef UP
#undef UPI
    if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess || cudaEventCreate(&h->ev0) != cudaSuccess ||
        cudaEventCreate(&h->ev1) != cudaSuccess || cudaEventCreateWithFlags(&h->ev_done, cudaEventDisableTiming) != cudaSuccess) {
        jq_destroy(h);
        return fail(JQ_ERR_CUDA, "jq_create: stream/event creation failed");
    }
    HostOps H{n, m, Nc, pb->nfreq, h->rowptr.data(), h->col.data(), h->val.data()};
    h->slot = jq_slot_plan_create(P, H, pb->wdiag, h->slot_reason, sizeof(h->slot_reason));
    h->fiber = jq_fiber_plan_create(P, H, pb->wdiag, h->fiber_reason, sizeof(h->fiber_reason));
    {
        const char *nt = getenv("JQ_TILE_NT");      // development: number of tiled directions of the tile layout (default: all)
        h->tile = jq_tile_plan_create(P, H, pb->wdiag, nt ? atoi(nt) : Nc, h->tile_reason, sizeof(h->tile_reason));
        // Latency layout: a trajectory spread over as many lanes as the warp-local exchange allows (one element per lane for two
        // subsystems, two for three).  A lone evaluation (the reference's own call pattern, one pcof per Ipopt callback) is bound
        // by the instruction stream of ONE lane, so fewer elements per lane is what shortens it; throughput layouts win once the
        // SMs are full.
        char why[256];
        const char *lnt = getenv("JQ_TILE_LAT_NT");
        const char *lp = getenv("JQ_LAT_PIPE");        // development: 0 = latency layout without the pipelined roles
        const int pipe = lp ? atoi(lp) : 1;
        h->tile_lat = jq_tile_plan_create(P, H, pb->wdiag, lnt ? atoi(lnt) : (Nc == 2 ? 0 : 1), why, sizeof(why), pipe);
        if (!h->tile_lat && pipe) h->tile_lat = jq_fiber_plan_create(P, H, pb->wdiag, why, sizeof(why), 1);     // single-fibre shapes: same layout, pipelined roles
        int sms = 148;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
        const char *lt = getenv("JQ_LAT_NTRAJ");
        // one latency CTA per SM: beyond that the throughput layouts win (measured)
        h->dense_ok = jq_dense_supported(P, h->dense_reason, sizeof(h->dense_reason));
        // a dense contraction executes n^2 multiply-adds per product and column whatever the sparsity: worth it from ~20% fill
        // (measured: 5%-filled ladder operators with remote exchange run 1.6x faster on the row-wise generic kernel)
        size_t nnz = 0;
        for (double v : h->val) nnz += v != 0.0;
        h->dense_auto = h->dense_ok && n >= 8 && (double)nnz >= 0.2 * (double)(1 + 2 * Nc) * n * n;
        h->lat_ntraj = lt ? atoi(lt) : sms * (h->tile_lat ? jq_traj_plan_tpc(h->tile_lat) : 1);
        // Time-parallel evaluation for launches of very few trajectories (one pcof per Ipopt callback): segments of the time axis
        // swept concurrently and joined through their propagators
        h->sms = sms;
        h->seg_plan = jq_tile_plan_create(P, H, pb->wdiag, Nc == 2 ? 0 : 1, why, sizeof(why), 0);
        if (!h->seg_plan) h->seg_plan = h->fiber;
        if (h->seg_plan && !jq_seg_supported(h->seg_plan, P)) { if (h->seg_plan != h->fiber) jq_traj_plan_destroy(h->seg_plan); h->seg_plan = nullptr; }
        // objFuncType 2/3: the gradient sweep needs the second adjoint set, which the fibre layout has
        if (h->seg_plan && P.objFuncType != 1) {
            if (h->fiber && jq_seg_supported(h->fiber, P, true)) h->seg_obj = h->fiber;
            else { if (h->seg_plan != h->fiber) jq_traj_plan_destroy(h->seg_plan); h->seg_plan = nullptr; }
        }
        // propagator launch (many independent unit-vector sweeps): the throughput tile layout when the problem has one
        const char *pe = getenv("JQ_SEG_PROP_TILE");
        if (h->seg_plan && h->tile && jq_seg_supported(h->tile, P) && (pe ? atoi(pe) != 0 : true)) h->seg_prop = h->tile;
        // automatic mode: time-parallel while the propagator launch (2 x 2n/m unit-vector sweeps per trajectory and segment) stays within
        // about four warps per SM -- measured cross-overs against the other kernels: cnot2 ~60 candidates, cnot3 ~30, risk-neutral ~1100
        // samples (profiles/r02_timeparallel.md)
        const char *sn = getenv("JQ_SEG_NTRAJ");
        if (h->seg_plan) {
            const int lanes = std::max(1, jq_traj_plan_lanes(h->seg_prop ? h->seg_prop : h->seg_plan)), nblk = (2 * n + m - 1) / m;
            h->seg_ntraj = std::max(1, (4 * sms * 32) / (2 * nblk * lanes));
        }
        if (sn) h->seg_ntraj = atoi(sn);
    }
    *out = h;
    return 0;
}

extern "C" int jq_destroy(jq_handle *h) {
    if (!h) return 0;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (h->comm && g_nccl.ok) { g_nccl.CommDestroy(h->comm); h->comm = nullptr; }
    for (void *p : h->owned) cudaFree(p);
    for (double *p : {h->d_scal, h->d_grad, h->d_igrad, h->d_in, h->d_out}) if (p) cudaFree(p);
    if (h->slot) jq_traj_plan_destroy(h->slot);
    if (h->tile) jq_traj_plan_destroy(h->tile);
    if (h->tile_lat) jq_traj_plan_destroy(h->tile_lat);
    if (h->seg_plan && h->seg_plan != h->fiber) jq_traj_plan_destroy(h->seg_plan);
    if (h->fiber) jq_traj_plan_destroy(h->fiber);
    if (h->d_seg) cudaFree(h->d_seg);
    if (h->d_segt) cudaFree(h->d_segt);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->ev_done) cudaEventDestroy(h->ev_done);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return 0;
}

extern "C" int jq_update_target(jq_handle *h, const double *vr, const double *vi) {
    if (!h || !vr || !vi) return fail(JQ_ERR_ARG, "jq_update_target: null argument");
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaMemcpy(h->d_vtr, vr, sizeof(double) * h->n * h->m, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(h->d_vti, vi, sizeof(double) * h->n * h->m, cudaMemcpyHostToDevice));
    h->cache_valid = false;
    return 0;
}

extern "C" int jq_cache_invalidate(jq_handle *h) {
    if (!h) return fail(JQ_ERR_ARG, "jq_cache_invalidate: null handle");
    h->cache_valid = false;
    return 0;
}

extern "C" int64_t jq_abi_info(int32_t what) {
    switch (what) {
    case 0: return 2;                                   // ABI version (2: jq_eval_f_grad, jq_abi_info, pFidType / dense weights / uncoupled controls)
    case 1: return (int64_t)sizeof(jq_problem);
    case 2: return (int64_t)sizeof(jq_operator);
    case 3: return (int64_t)offsetof(jq_problem, nsteps);
    case 4: return (int64_t)offsetof(jq_problem, T);
    case 5: return (int64_t)offsetof(jq_problem, uinit);
    case 6: return (int64_t)offsetof(jq_problem, h0);
    case 7: return (int64_t)offsetof(jq_problem, hsym);
    case 8: return (int64_t)offsetof(jq_problem, solver_tol);
    case 9: return (int64_t)offsetof(jq_operator, nnz);
    case 10: return (int64_t)offsetof(jq_operator, nzval);
    default: return -1;
    }
}

extern "C" int jq_set_kernel(jq_handle *h, int32_t kernel) {
    if (!h || kernel < 0 || kernel > 7) return fail(JQ_ERR_ARG, "jq_set_kernel: kernel must be 0 ... 7");
    if (kernel == 7 && !h->seg_plan) return fail(JQ_ERR_ARG, "jq_set_kernel: no time-parallel evaluation for this problem (needs a tile / fibre layout, the Neumann solver, diagonal weights)");
    if (kernel == 6 && !h->dense_ok) return fail(JQ_ERR_ARG, "jq_set_kernel: the dense (tensor-core) kernel cannot serve this problem (%s)", h->dense_reason);
    if (kernel == 5 && !h->tile_lat) return fail(JQ_ERR_ARG, "jq_set_kernel: no latency layout for this problem");
    if (kernel == 4 && !h->tile) return fail(JQ_ERR_ARG, "jq_set_kernel: no tile-layout instantiation for this problem (%s)", h->tile_reason);
    if (kernel == 2 && !h->slot) return fail(JQ_ERR_ARG, "jq_set_kernel: no slot-layout instantiation for this problem (%s)", h->slot_reason);
    if (kernel == 3 && !h->fiber) return fail(JQ_ERR_ARG, "jq_set_kernel: no fibre-layout instantiation for this problem (%s)", h->fiber_reason);
    h->kernel_pref = kernel;
    return 0;
}

extern "C" int jq_set_time_segments(jq_handle *h, int32_t nseg) {
    if (!h || nseg < 0) return fail(JQ_ERR_ARG, "jq_set_time_segments: need a handle and nseg >= 0 (0 = automatic)");
    h->seg_nseg = nseg;
    return 0;
}

extern "C" int64_t jq_time_segments(double T, int64_t nsteps, int32_t nseg, double *t_first, double *t_last) {
    if (nseg < 1 || nsteps < nseg || !t_first || !t_last) { fail(JQ_ERR_ARG, "jq_time_segments: need 1 <= nseg <= nsteps and two output arrays"); return -1; }
    DevProblem P{};
    P.T = T; P.nsteps = nsteps;
    std::vector<double> t(2 * (size_t)nseg);
    jq_seg_times(P, nseg, t.data());
    int64_t longest = 0;
    for (int p = 0; p < nseg; ++p) {
        t_first[p] = t[p]; t_last[p] = t[(size_t)nseg + p];
        longest = std::max<int64_t>(longest, (int64_t)(p + 1) * nsteps / nseg - (int64_t)p * nsteps / nseg);
    }
    return longest;
}

extern "C" int jq_query(jq_handle *h, int32_t what, double *value) {
    if (!h || !value) return fail(JQ_ERR_ARG, "jq_query: null argument");
    switch (what) {
    case 0: *value = h->last_kernel; break;
    case 1: {
        if (!h->timed) return fail(JQ_ERR_ARG, "jq_query: no evaluation has run yet");
        CU(cudaEventSynchronize(h->ev1));
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
        *value = ms;
        break;
    }
    case 2: *value = h->last_launches; break;
    case 3: *value = h->last_tpc; break;
    case 4: *value = h->last_ctas; break;
    case 5: *value = h->last_regs; break;
    case 6: *value = (double)h->last_smem; break;
    case 7: *value = h->last_kernel == 7 ? h->last_nseg : 0; break;
    default: return fail(JQ_ERR_ARG, "jq_query: unknown item %d", what);
    }
    return 0;
}

// Per-candidate outputs: copies (weights == nullptr) or weighted sums over the samples of each candidate
// (src/ipopt_interface.jl:48-59) in sample order (few samples; jq_weighted_sum_kernel takes over from 64 samples).
__global__ void jq_finalize_kernel(int nbatch, int nsamples, int Npar, int objFuncType, int evaladjoint, const double *w,
                                   const double *scal, const double *gt, const double *igt, double *infid, double *leak,
                                   double *tinfid, double *grad, double *infidgrad, double *leakgrad) {
    const int nout = w ? nbatch : nbatch * nsamples;
    const long long total = (long long)nout * (Npar + 1);
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int o = (int)(idx / (Npar + 1)), k = (int)(idx % (Npar + 1));
        const int t0 = w ? o * nsamples : o, cnt = w ? nsamples : 1;
        if (k == Npar) {
            double a = 0.0, b = 0.0, c = 0.0;
            for (int s = 0; s < cnt; ++s) {
                const double ws = w ? w[s] : 1.0;
                const double *sc = scal + (size_t)(t0 + s) * 4;
                a += ws * sc[0]; b += ws * sc[1]; c += ws * sc[2];
            }
            if (infid) infid[o] = a;
            if (leak) leak[o] = b;
            if (tinfid) tinfid[o] = c;
        } else if (evaladjoint) {
            double g = 0.0, ig = 0.0;
            for (int s = 0; s < cnt; ++s) {
                const double ws = w ? w[s] : 1.0;
                g += ws * gt[(size_t)(t0 + s) * Npar + k];
                if (objFuncType != 1) ig += ws * igt[(size_t)(t0 + s) * Npar + k];
            }
            if (grad) grad[(size_t)o * Npar + k] = g;
            if (objFuncType != 1) {
                if (infidgrad) infidgrad[(size_t)o * Npar + k] = ig;
                if (leakgrad) leakgrad[(size_t)o * Npar + k] = g - ig;   // src/evalobjgrad.jl:947
            } else if (infidgrad) {
                infidgrad[(size_t)o * Npar + k] = g;                      // infidelgrad = totalgrad, :951
            }
        }
    }
}

// Weighted sums over many samples of one candidate (risk-neutral quadrature / noise sweeps with thousands of nodes):
// block (candidate, tile of 32 output columns); thread (column c, sample lane l) sums samples l, l+32, ... in order,
// the 32 lane partials are then added in lane order -> deterministic for a given nsamples.  Columns 0..Npar-1 are the
// gradient entries, Npar..Npar+2 the three scalars.
#define WS_LANES 32
__global__ void __launch_bounds__(32 * WS_LANES) jq_weighted_sum_kernel(int nsamples, int Npar, int objFuncType, int evaladjoint,
                                   const double *w, const double *scal, const double *gt, const double *igt, double *infid, double *leak,
                                   double *tinfid, double *grad, double *infidgrad, double *leakgrad) {
    __shared__ double part[2][WS_LANES][33];
    const int c = threadIdx.x & 31, l = threadIdx.x >> 5, k = blockIdx.y * 32 + c, o = blockIdx.x;   // candidates on grid.x (no 65535 limit)
    const size_t t0 = (size_t)o * nsamples;
    double g = 0.0, ig = 0.0;
    if (k < Npar) {
        if (evaladjoint)
            for (int s = l; s < nsamples; s += WS_LANES) {
                g += w[s] * gt[(t0 + s) * Npar + k];
                if (objFuncType != 1) ig += w[s] * igt[(t0 + s) * Npar + k];
            }
    } else if (k < Npar + 3) {
        for (int s = l; s < nsamples; s += WS_LANES) g += w[s] * scal[(t0 + s) * 4 + (k - Npar)];
    }
    part[0][l][c] = g; part[1][l][c] = ig;
    __syncthreads();
    if (l != 0 || k >= Npar + 3) return;
    g = 0.0; ig = 0.0;
    for (int j = 0; j < WS_LANES; ++j) { g += part[0][j][c]; ig += part[1][j][c]; }
    if (k >= Npar) {
        double *dst = k == Npar ? infid : k == Npar + 1 ? leak : tinfid;
        if (dst) dst[o] = g;
    } else if (evaladjoint) {
        if (grad) grad[(size_t)o * Npar + k] = g;
        if (objFuncType != 1) {
            if (infidgrad) infidgrad[(size_t)o * Npar + k] = ig;
            if (leakgrad) leakgrad[(size_t)o * Npar + k] = g - ig;
        } else if (infidgrad) {
            infidgrad[(size_t)o * Npar + k] = g;
        }
    }
}


// Launch the trajectory kernel for `A`: the register-resident layouts in order of preference (tile, fibre, slot), then the
// generic kernel.  In automatic mode a layout that cannot serve this launch (no instantiation for the variant, shared-memory
// layout does not fit, out of launch resources) hands over to the next one; an explicitly requested kernel fails instead.
static int launch_trajectories(jq_handle *h, const LaunchArgs &A, cudaStream_t st) {
    TrajPlan *cands[4] = {nullptr, nullptr, nullptr, nullptr};
    int ncand = 0;
    const int pref = h->kernel_pref;
    const bool small = A.ntraj <= h->lat_ntraj;
    if (pref == 5 || (pref == 0 && h->tile_lat && small)) cands[ncand++] = h->tile_lat;
    if (pref == 0 && small && h->fiber && h->tile && h->Nc >= 3) cands[ncand++] = h->fiber;     // three subsystems: the fibre layout (4 elements per lane) before the 8-element tiles
    if (pref == 4 || (pref == 0 && h->tile && h->prefer_tile)) cands[ncand++] = h->tile;
    if (pref == 3 || (pref == 0 && h->fiber && !(ncand && cands[ncand - 1] == h->fiber) && !(ncand > 1 && cands[ncand - 2] == h->fiber))) cands[ncand++] = h->fiber;
    if (pref == 2 || (pref == 0 && h->slot)) cands[ncand++] = h->slot;
    TrajPlan *plan = nullptr;
    int ctas = 0, regs = 0, tpc = 1;
    size_t smem = 0;
    CU(cudaEventRecord(h->ev0, st));
    // very few trajectories: time-parallel evaluation (segments of the time axis swept concurrently)
    const bool seg_able = h->seg_plan && h->P.solver == 1 && !A.hist_r;
    if (pref == 7 || (pref == 0 && seg_able && A.ntraj <= h->seg_ntraj && h->P.nsteps >= 256)) {
        if (!seg_able) return fail(JQ_ERR_ARG, "time-parallel evaluation: Neumann solver, no state history");
        TrajPlan *prop = h->seg_prop ? h->seg_prop : h->seg_plan;
        int nseg = h->seg_nseg > 0 ? h->seg_nseg : jq_seg_auto_segments(h->P, A.ntraj, A.evaladjoint, jq_traj_plan_tpc(prop), h->sms);
        if (nseg > h->P.nsteps) nseg = (int)h->P.nsteps;
        // cooperative evaluation: the segments are shared out evenly over the ranks (every rank computes the same nseg)
        // ... when the propagator launch is at least two waves of CTAs: below that its collective costs more than it saves
        const long long l1_ctas = 2LL * nseg * (((long long)((2 * h->n + h->m - 1) / h->m) * A.ntraj + jq_traj_plan_tpc(prop) - 1) / jq_traj_plan_tpc(prop));
        const char *cf = getenv("JQ_SEG_COOP_FORCE");     // tests: share out small problems too
        const bool coop_on = h->cooperative && h->comm && h->comm_size > 1 && h->P.nsteps >= h->comm_size &&
                             (l1_ctas >= 2LL * h->sms || (cf && atoi(cf)));
        if (coop_on) {
            nseg = std::max(h->comm_size, (nseg + h->comm_size - 1) / h->comm_size * h->comm_size);
            if (nseg > h->P.nsteps) nseg = (int)(h->P.nsteps / h->comm_size) * h->comm_size;       // >= comm_size by the test above
        }
        SegCoop coop{h->comm_rank, h->comm_size, seg_allgather, h};
        int rc = grow(&h->d_seg, &h->cap_seg, jq_seg_workspace_doubles(h->P, A.ntraj, A.Npar, nseg, A.evaladjoint));
        if (rc) return rc;
        if (h->segt_nseg != nseg) {           // segment start / end times: host recurrence, once per segment count
            h->segt.resize(2 * (size_t)nseg);
            jq_seg_times(h->P, nseg, h->segt.data());
            if ((rc = grow(&h->d_segt, &h->cap_segt, 2 * (size_t)nseg + 2)) != 0) return rc;      // times, then the four refinement flags
            CU(cudaMemcpyAsync(h->d_segt, h->segt.data(), 2 * (size_t)nseg * sizeof(double), cudaMemcpyHostToDevice, st));
            h->segt_nseg = nseg;
        }
        int nl = 0;
        cudaError_t e = jq_seg_launch(h->seg_prop, h->seg_plan, h->seg_obj, h->P, A, nseg, h->d_segt, reinterpret_cast<int *>(h->d_segt + 2 * (size_t)nseg), h->d_seg, st, coop_on && nseg >= h->comm_size ? &coop : nullptr, &ctas, &regs, &smem, &tpc, &nl);
        if (e == cudaSuccess) {
            CU(cudaEventRecord(h->ev1, st));
            h->timed = true;
            h->last_kernel = 7; h->last_nseg = nseg; h->last_traj_launches = nl;
            h->last_ctas = ctas; h->last_regs = regs; h->last_smem = smem; h->last_tpc = tpc;
            return 0;
        }
        cudaGetLastError();
        const bool soft = e == cudaErrorInvalidConfiguration || e == cudaErrorNotSupported || e == cudaErrorLaunchOutOfResources;
        if (!soft || pref != 0) return fail(JQ_ERR_CUDA, "time-parallel evaluation failed: %s", cudaGetErrorString(e));
    }
    h->last_traj_launches = 1;
    for (int i = 0; i < ncand && !plan; ++i) {
        cudaError_t e = jq_traj_launch(cands[i], h->P, A, st, &ctas, &regs, &smem, &tpc);
        if (e == cudaSuccess) { plan = cands[i]; break; }
        cudaGetLastError();                                   // clear the (non-sticky) launch error before trying the next kernel
        const bool soft = e == cudaErrorInvalidConfiguration || e == cudaErrorNotSupported || e == cudaErrorLaunchOutOfResources;
        if (!soft || pref != 0) return fail(JQ_ERR_CUDA, "trajectory kernel launch failed: %s", cudaGetErrorString(e));
    }
    bool dense = false;
    if (!plan && (pref == 6 || (pref == 0 && h->dense_auto && !A.hist_r))) {
        // unstructured operators: the products are real contractions -> FP64 tensor-core kernel, samples of a candidate batched
        cudaError_t e = jq_dense_launch(h->P, A, st, &ctas, &regs, &smem, &tpc);
        if (e == cudaSuccess) dense = true;
        else {
            cudaGetLastError();
            if (pref == 6) return fail(JQ_ERR_CUDA, "dense kernel launch failed: %s", cudaGetErrorString(e));
        }
    }
    if (!plan && !dense) {
        if (pref > 1) return fail(JQ_ERR_ARG, "requested kernel is not available for this problem");
        if (jq_generic_smem_bytes(h->P, A.Npar) > 227 * 1024)
            return fail(JQ_ERR_ARG, "problem too large for the generic kernel's shared memory (n*m = %d)", h->n * h->m);
        tpc = 1;
        CU(jq_generic_launch(h->P, A, st, &ctas, &regs, &smem));
    }
    CU(cudaEventRecord(h->ev1, st));
    h->timed = true;
    h->last_kernel = plan ? (plan == h->tile_lat ? 5 : jq_traj_plan_kind(plan)) : dense ? 6 : 1;
    h->last_ctas = ctas; h->last_regs = regs; h->last_smem = smem; h->last_tpc = tpc;
    return 0;
}

static int check_batch_args(jq_handle *h, int nbatch, const double *pcof, int npar, int nsamples, const double *shift,
                            bool empty_shard_ok = false) {
    if (!h) return fail(JQ_ERR_ARG, "null handle");
    if (nbatch < 1 || !pcof) return fail(JQ_ERR_ARG, "need nbatch >= 1 and a pcof array");
    const int nsig = 2 * h->Nc;
    npar -= h->pfid == 3 ? 1 : 0;              // pFidType 3: the last entry is the global phase (src/evalobjgrad.jl:591-596)
    if (npar % nsig != 0 || npar < 3 * nsig)   // src/evalobjgrad.jl:604-606
        return fail(JQ_ERR_PCOF_LENGTH, "pcof must have an even number of elements >= %d, not %d", 3 * nsig, npar);
    if (npar % (nsig * h->Nfreq) != 0 || npar / (nsig * h->Nfreq) < 3)   // src/bsplines.jl:177-181 (and k >= 3 needs D1 >= 3)
        return fail(JQ_ERR_PCOF_LENGTH, "Inconsistent number of coefficients and size of parameter vector (nCoeff = %d, Nfreq = %d, Ncoupled + Nunc = %d)", npar, h->Nfreq, h->Nc);
    // an empty sample shard (more ranks than quadrature nodes) contributes zeros and still joins the all-reduce
    if (nsamples < (empty_shard_ok ? 0 : 1)) return fail(JQ_ERR_ARG, "nsamples must be >= 1 (0 only with weights: an empty sample shard)");
    if ((long long)nbatch * nsamples > 0x7fffffffLL) return fail(JQ_ERR_ARG, "nbatch * nsamples exceeds 2^31 - 1 trajectories per call");
    if (!shift && nsamples > 1) return fail(JQ_ERR_ARG, "nsamples > 1 needs h0_diag_shift");
    return 0;
}

extern "C" int jq_traceobjgrad_batch_device(jq_handle *h, int32_t nbatch, const double *pcof, int32_t npar, int32_t nsamples,
                                            const double *shift, const double *weights, int32_t evaladjoint, double *infid,
                                            double *leak, double *trace_infid, double *grad, double *infidgrad, double *leakgrad,
                                            void *cuda_stream) {
    int rc = check_batch_args(h, nbatch, pcof, npar, nsamples, shift, weights != nullptr);
    if (rc) return rc;
    CU(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    const size_t ntraj = (size_t)nbatch * nsamples;
    // the handle's scratch (d_scal, d_grad, d_igrad) is shared by every call: a call on a different stream than the previous one
    // (host-pointer entry = the handle's own stream, device entry = the caller's) first waits for that one to finish
    if (h->have_last && h->last_stream != st) CU(cudaStreamWaitEvent(st, h->ev_done, 0));
    if ((rc = grow(&h->d_scal, &h->cap_traj, ntraj * 4)) != 0) return rc;
    if (evaladjoint && (rc = grow(&h->d_grad, &h->cap_grad, ntraj * npar)) != 0) return rc;
    if (evaladjoint && h->P.objFuncType != 1 && (rc = grow(&h->d_igrad, &h->cap_igrad, ntraj * npar)) != 0) return rc;

    // npar is the caller's vector length: the spline coefficients, plus the global phase as last entry for pFidType 3; gradients
    // have the same length, so the finalize kernels just see npar columns
    const int nspl = npar - (h->pfid == 3 ? 1 : 0);
    LaunchArgs A{};
    A.ntraj = (int)ntraj; A.nsamples = nsamples; A.Npar = nspl; A.D1 = nspl / (2 * h->Nc * h->Nfreq); A.evaladjoint = evaladjoint ? 1 : 0;
    A.pstride = npar; A.gstride = npar;
    A.pcof = pcof; A.shift = shift; A.scal = h->d_scal; A.grad = h->d_grad; A.infidgrad = h->P.objFuncType != 1 ? h->d_igrad : nullptr;

    if (ntraj > 0 && (rc = launch_trajectories(h, A, st)) != 0) return rc;
    const int nout = weights ? nbatch : (int)ntraj;
    const long long total = (long long)nout * (npar + 1);
    const int fb = 256, fg = (int)std::min<long long>((total + fb - 1) / fb, 148 * 8);
    if (weights && nsamples >= 64)
        jq_weighted_sum_kernel<<<dim3(nbatch, (npar + 3 + 31) / 32), 32 * WS_LANES, 0, st>>>(nsamples, npar, h->P.objFuncType, A.evaladjoint,
                                          weights, h->d_scal, h->d_grad, h->d_igrad, infid, leak, trace_infid, grad, infidgrad, leakgrad);
    else
        jq_finalize_kernel<<<fg, fb, 0, st>>>(nbatch, nsamples, npar, h->P.objFuncType, A.evaladjoint, weights, h->d_scal, h->d_grad,
                                              h->d_igrad, infid, leak, trace_infid, grad, infidgrad, leakgrad);
    CU(cudaGetLastError());
    h->last_launches = 1 + h->last_traj_launches;
    if (h->comm && weights && h->comm_size > 1) {
        // the path's one exchange step: weighted sums over the sample shards of all ranks (sum, FP64), one grouped call
        const size_t nb = (size_t)nbatch, ng = (size_t)nbatch * npar;
        // every call between GroupStart and GroupEnd is attempted and the group is always closed, so an error on one rank
        // cannot leave the communicator inside an open group
        int nrc = g_nccl.GroupStart();
        auto red = [&](double *buf, size_t cnt) { if (buf && nrc == 0) nrc = g_nccl.AllReduce(buf, buf, cnt, 8 /*ncclDouble*/, 0 /*ncclSum*/, h->comm, st); };
        red(infid, nb); red(leak, nb); red(trace_infid, nb);
        if (A.evaladjoint) {
            red(grad, ng); red(infidgrad, ng);
            if (h->P.objFuncType != 1) red(leakgrad, ng);
        }
        const int erc = g_nccl.GroupEnd();
        if (nrc == 0) nrc = erc;
        if (nrc != 0) return fail(JQ_ERR_CUDA, "ncclAllReduce of the weighted sample sums: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(nrc) : "nccl error");
        h->last_launches += 1;
    }
    CU(cudaEventRecord(h->ev_done, st));
    h->last_stream = st; h->have_last = true;
    return 0;
}


// Tikhonov + packing of the fused callback entry: out = [f, infid, leak, grad_f[npar], leakgrad[npar], infidgrad[npar]]; one block, the
// squared norm summed in a fixed order (thread-strided partials, then thread order) so that f is bit-reproducible.
__global__ void __launch_bounds__(256) jq_tikhonov_kernel(int npar, int objFuncType, double tik0, const double *pcof, const double *prior,
                                                          const double *infid, const double *leak, const double *igrad, const double *lgrad, double *out) {
    __shared__ double part[256];
    double s = 0.0;
    for (int k = threadIdx.x; k < npar; k += blockDim.x) {
        const double d = prior ? pcof[k] - prior[k] : pcof[k];
        s += d * d;
        out[3 + k] = igrad[k] + (2.0 * tik0 / npar) * d;                   // src/evalobjgrad.jl:2339-2349, ipopt_interface.jl:136-141
        out[3 + npar + k] = objFuncType != 1 ? lgrad[k] : 0.0;
        out[3 + 2 * npar + k] = igrad[k];                                  // last_infidelity_grad as the reference stores it (cache)
    }
    part[threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double pen = 0.0;
        for (int j = 0; j < blockDim.x; ++j) pen += part[j];
        const double f = objFuncType == 1 ? infid[0] + leak[0] : infid[0];  // ipopt_interface.jl:89-93
        out[0] = f + tik0 * pen / npar;                                    // :96-98, evalobjgrad.jl:2291-2316
        out[1] = infid[0];
        out[2] = leak[0];
    }
}

extern "C" int jq_eval_f_grad(jq_handle *h, const double *pcof, int32_t npar, int32_t nsamples, const double *shift, const double *weights,
                              double tik0, const double *prior, double *f, double *grad_f, double *infid, double *leak, double *leakgrad,
                              int32_t *evaluated) {
    int rc = check_batch_args(h, 1, pcof, npar, nsamples, shift, weights != nullptr);
    if (rc) return rc;
    const size_t n_shift = shift ? (size_t)nsamples * h->n : 0, n_w = weights ? (size_t)nsamples : 0;
    // the reference's cache test (src/ipopt_interface.jl:84): norm(pcof - last_pcof) > 1e-15; shards / weights compared exactly
    bool hit = h->cache_valid && h->c_pcof.size() == (size_t)npar && h->c_shift.size() == n_shift && h->c_w.size() == n_w;
    if (hit) {
        double d2 = 0.0;
        for (int k = 0; k < npar; ++k) { const double d = pcof[k] - h->c_pcof[k]; d2 += d * d; }
        hit = !(sqrt(d2) > 1.0e-15) && (n_shift == 0 || memcmp(shift, h->c_shift.data(), n_shift * sizeof(double)) == 0) &&
              (n_w == 0 || memcmp(weights, h->c_w.data(), n_w * sizeof(double)) == 0);
    }
    if (evaluated) *evaluated = hit ? 0 : 1;
    if (!hit) {
        CU(cudaSetDevice(h->device));
        h->cache_valid = false;
        const bool two = h->P.objFuncType != 1;
        const size_t n_in = (size_t)npar + n_shift + (n_w ? n_w : 1) + (prior ? npar : 0);
        const size_t n_out = 3 + (size_t)npar * (two ? 3 : 1) + 3 + 3 * (size_t)npar;
        if ((rc = grow(&h->d_in, &h->cap_in, n_in)) != 0) return rc;
        if ((rc = grow(&h->d_out, &h->cap_out, n_out)) != 0) return rc;
        cudaStream_t st = h->stream;
        double *d_pcof = h->d_in, *d_shift = shift ? d_pcof + npar : nullptr, *d_w = d_pcof + npar + n_shift;
        double *d_prior = prior ? d_w + (n_w ? n_w : 1) : nullptr;
        CU(cudaMemcpyAsync(d_pcof, pcof, (size_t)npar * sizeof(double), cudaMemcpyHostToDevice, st));
        if (n_shift) CU(cudaMemcpyAsync(d_shift, shift, n_shift * sizeof(double), cudaMemcpyHostToDevice, st));
        const double one = 1.0;
        if (n_w) CU(cudaMemcpyAsync(d_w, weights, n_w * sizeof(double), cudaMemcpyHostToDevice, st));
        else CU(cudaMemcpyAsync(d_w, &one, sizeof(double), cudaMemcpyHostToDevice, st));      // no weights: the single sample has weight 1
        if (prior) CU(cudaMemcpyAsync(d_prior, prior, (size_t)npar * sizeof(double), cudaMemcpyHostToDevice, st));
        double *o_infid = h->d_out, *o_leak = o_infid + 1, *o_tinf = o_leak + 1, *o_g = o_tinf + 1;
        double *o_ig = two ? o_g + npar : nullptr, *o_lg = two ? o_ig + npar : nullptr;
        double *o_pack = o_g + (size_t)npar * (two ? 3 : 1);
        rc = jq_traceobjgrad_batch_device(h, 1, d_pcof, npar, nsamples, d_shift, d_w, 1, o_infid, o_leak, o_tinf, o_g, o_ig, o_lg, st);
        if (rc) return rc;
        jq_tikhonov_kernel<<<1, 256, 0, st>>>(npar, h->P.objFuncType, tik0, d_pcof, d_prior, o_infid, o_leak, two ? o_ig : o_g, o_lg, o_pack);
        CU(cudaGetLastError());
        h->last_launches += 1;
        std::vector<double> pack(3 + 3 * (size_t)npar);
        CU(cudaMemcpyAsync(pack.data(), o_pack, pack.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        // store what the reference stores (last_infidelity, last_leak, last_infidelity_grad, last_leak_grad): the Tikhonov terms are
        // re-applied on a cache hit because tik0 / prior are inputs of every call
        h->c_pcof.assign(pcof, pcof + npar);
        h->c_shift.assign(shift ? shift : pcof, shift ? shift + n_shift : pcof);
        h->c_w.assign(weights ? weights : pcof, weights ? weights + n_w : pcof);
        h->c_infid = pack[1]; h->c_leak = pack[2];
        h->c_lgrad.assign(pack.begin() + 3 + npar, pack.begin() + 3 + 2 * (size_t)npar);
        h->c_igrad.assign(pack.begin() + 3 + 2 * (size_t)npar, pack.end());
        h->cache_valid = true;
        if (f) *f = pack[0];
        if (infid) *infid = pack[1];
        if (leak) *leak = pack[2];
        if (grad_f) memcpy(grad_f, pack.data() + 3, (size_t)npar * sizeof(double));
        if (leakgrad && two) memcpy(leakgrad, pack.data() + 3 + npar, (size_t)npar * sizeof(double));
        return 0;
    }
    // cache hit: no launch, no transfer
    double pen = 0.0;
    for (int k = 0; k < npar; ++k) { const double d = prior ? pcof[k] - prior[k] : pcof[k]; pen += d * d; }
    if (f) *f = (h->P.objFuncType == 1 ? h->c_infid + h->c_leak : h->c_infid) + tik0 * pen / npar;
    if (infid) *infid = h->c_infid;
    if (leak) *leak = h->c_leak;
    if (grad_f)
        for (int k = 0; k < npar; ++k) grad_f[k] = h->c_igrad[k] + (2.0 * tik0 / npar) * (prior ? pcof[k] - prior[k] : pcof[k]);
    if (leakgrad && h->P.objFuncType != 1) memcpy(leakgrad, h->c_lgrad.data(), (size_t)npar * sizeof(double));
    return 0;
}

extern "C" int jq_eval_forward(jq_handle *h, int32_t nbatch, const double *pcof, int32_t npar, int32_t nsamples, const double *shift,
                               int32_t save_every, double *hist_r, double *hist_i, double *infid, double *leak) {
    int rc = check_batch_args(h, nbatch, pcof, npar, nsamples, shift);
    if (rc) return rc;
    if (!hist_r || !hist_i) return fail(JQ_ERR_ARG, "jq_eval_forward: null history buffer");
    if (save_every < 1 || h->P.nsteps % save_every != 0)     // src/evalobjgrad.jl:2797-2799
        return fail(JQ_ERR_ARG, "nsteps must be divisible by saveEvery. nsteps=%lld, saveEvery=%d", (long long)h->P.nsteps, save_every);
    CU(cudaSetDevice(h->device));
    const size_t ntraj = (size_t)nbatch * nsamples, len = (size_t)h->n * h->m;
    const long long nsave = h->P.nsteps / save_every + 1;
    const size_t n_pcof = (size_t)nbatch * npar, n_shift = shift ? (size_t)nsamples * h->n : 0, n_hist = ntraj * (size_t)nsave * len;
    if ((rc = grow(&h->d_in, &h->cap_in, n_pcof + n_shift)) != 0) return rc;
    if ((rc = grow(&h->d_out, &h->cap_out, 2 * n_hist)) != 0) return rc;
    if ((rc = grow(&h->d_scal, &h->cap_traj, ntraj * 4)) != 0) return rc;
    cudaStream_t st = h->stream;
    double *d_pcof = h->d_in, *d_shift = shift ? h->d_in + n_pcof : nullptr;
    CU(cudaMemcpyAsync(d_pcof, pcof, n_pcof * sizeof(double), cudaMemcpyHostToDevice, st));
    if (shift) CU(cudaMemcpyAsync(d_shift, shift, n_shift * sizeof(double), cudaMemcpyHostToDevice, st));
    const int nspl = npar - (h->pfid == 3 ? 1 : 0);
    LaunchArgs A{};
    A.ntraj = (int)ntraj; A.nsamples = nsamples; A.Npar = nspl; A.D1 = nspl / (2 * h->Nc * h->Nfreq); A.evaladjoint = 0;
    A.pstride = npar; A.gstride = npar;
    A.pcof = d_pcof; A.shift = d_shift; A.scal = h->d_scal; A.grad = nullptr; A.infidgrad = nullptr;
    A.hist_r = h->d_out; A.hist_i = h->d_out + n_hist; A.save_every = save_every; A.nsave = nsave;
    if ((rc = launch_trajectories(h, A, st)) != 0) return rc;      // same kernel choice as jq_traceobjgrad_batch
    h->last_launches = 1;
    CU(cudaMemcpyAsync(hist_r, A.hist_r, n_hist * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(hist_i, A.hist_i, n_hist * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (infid || leak) {
        std::vector<double> sc(ntraj * 4);
        CU(cudaMemcpy(sc.data(), h->d_scal, sc.size() * sizeof(double), cudaMemcpyDeviceToHost));
        for (size_t t = 0; t < ntraj; ++t) { if (infid) infid[t] = sc[4 * t]; if (leak) leak[t] = sc[4 * t + 1]; }
    }
    return 0;
}

extern "C" int jq_eval_controls(jq_handle *h, const double *pcof, int32_t npar, int32_t ntimes, const double *times, double *p, double *q) {
    int rc = check_batch_args(h, 1, pcof, npar, 1, nullptr);
    if (rc) return rc;
    if (ntimes < 0 || (ntimes > 0 && (!times || !p || !q))) return fail(JQ_ERR_ARG, "jq_eval_controls: null time or output array");
    if (ntimes == 0) return 0;
    CU(cudaSetDevice(h->device));
    const size_t nout = (size_t)h->Nc * ntimes;
    if ((rc = grow(&h->d_in, &h->cap_in, (size_t)npar + ntimes)) != 0) return rc;
    if ((rc = grow(&h->d_out, &h->cap_out, 2 * nout)) != 0) return rc;
    cudaStream_t st = h->stream;
    CU(cudaMemcpyAsync(h->d_in, pcof, (size_t)npar * sizeof(double), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(h->d_in + npar, times, (size_t)ntimes * sizeof(double), cudaMemcpyHostToDevice, st));
    CU(jq_controls_launch(h->P, (npar - (h->pfid == 3 ? 1 : 0)) / (2 * h->Nc * h->Nfreq), h->d_in, ntimes, h->d_in + npar, h->d_out, h->d_out + nout, st));
    CU(cudaMemcpyAsync(p, h->d_out, nout * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(q, h->d_out + nout, nout * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return 0;
}

extern "C" int jq_traceobjgrad_batch(jq_handle *h, int32_t nbatch, const double *pcof, int32_t npar, int32_t nsamples,
                                     const double *shift, const double *weights, int32_t evaladjoint, double *infid, double *leak,
                                     double *trace_infid, double *grad, double *infidgrad, double *leakgrad) {
    int rc = check_batch_args(h, nbatch, pcof, npar, nsamples, shift, weights != nullptr);
    if (rc) return rc;
    CU(cudaSetDevice(h->device));
    const size_t ntraj = (size_t)nbatch * nsamples, nout = weights ? (size_t)nbatch : ntraj;
    const size_t n_pcof = (size_t)nbatch * npar, n_shift = shift ? (size_t)nsamples * h->n : 0, n_w = weights ? (size_t)nsamples : 0;
    if ((rc = grow(&h->d_in, &h->cap_in, n_pcof + n_shift + n_w + 1)) != 0) return rc;      // + 1: a valid weights pointer for an empty shard
    const bool want_g = evaladjoint && grad, want_ig = evaladjoint && infidgrad, want_lg = evaladjoint && leakgrad && h->P.objFuncType != 1;
    const size_t n_outs = 3 * nout + (size_t)(want_g + want_ig + want_lg) * nout * npar;
    if ((rc = grow(&h->d_out, &h->cap_out, n_outs)) != 0) return rc;
    cudaStream_t st = h->stream;
    double *d_pcof = h->d_in, *d_shift = shift ? h->d_in + n_pcof : nullptr, *d_w = weights ? h->d_in + n_pcof + n_shift : nullptr;
    CU(cudaMemcpyAsync(d_pcof, pcof, n_pcof * sizeof(double), cudaMemcpyHostToDevice, st));
    if (shift && n_shift) CU(cudaMemcpyAsync(d_shift, shift, n_shift * sizeof(double), cudaMemcpyHostToDevice, st));
    if (weights && n_w) CU(cudaMemcpyAsync(d_w, weights, n_w * sizeof(double), cudaMemcpyHostToDevice, st));
    double *o_infid = h->d_out, *o_leak = o_infid + nout, *o_tinf = o_leak + nout, *cur = o_tinf + nout;
    double *o_g = nullptr, *o_ig = nullptr, *o_lg = nullptr;
    if (want_g) { o_g = cur; cur += nout * npar; }
    if (want_ig) { o_ig = cur; cur += nout * npar; }
    if (want_lg) { o_lg = cur; cur += nout * npar; }
    rc = jq_traceobjgrad_batch_device(h, nbatch, d_pcof, npar, nsamples, d_shift, d_w, evaladjoint, o_infid, o_leak, o_tinf, o_g, o_ig,
                                      o_lg, st);
    if (rc) return rc;
    if (infid) CU(cudaMemcpyAsync(infid, o_infid, nout * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (leak) CU(cudaMemcpyAsync(leak, o_leak, nout * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (trace_infid) CU(cudaMemcpyAsync(trace_infid, o_tinf, nout * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (want_g) CU(cudaMemcpyAsync(grad, o_g, nout * npar * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (want_ig) CU(cudaMemcpyAsync(infidgrad, o_ig, nout * npar * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (want_lg) CU(cudaMemcpyAsync(leakgrad, o_lg, nout * npar * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return 0;
}

extern "C" int jq_forward_sensitivity(jq_handle *h, int32_t nbatch, const double *pcof, int32_t npar, int32_t nsamples,
                                      const double *shift, const double *weights, int32_t ndir, const double *dirs, double *infid,
                                      double *leak, double *dinfid, double *dleak, double *dstate_r, double *dstate_i) {
    int rc = check_batch_args(h, nbatch, pcof, npar, nsamples, shift);
    if (rc) return rc;
    if (ndir < 1 || !dirs) return fail(JQ_ERR_ARG, "jq_forward_sensitivity: need ndir >= 1 and a dirs array");
    if ((long long)nbatch * nsamples * ndir > 0x7fffffffLL)
        return fail(JQ_ERR_ARG, "jq_forward_sensitivity: nbatch * nsamples * ndir exceeds 2^31 - 1 trajectories per call");
    if (h->P.solver == 2) return fail(JQ_ERR_ARG, "jq_forward_sensitivity: the Jacobi solver has no tangent sweep (use the Neumann solver)");
    if (weights && (dstate_r || dstate_i))
        return fail(JQ_ERR_ARG, "jq_forward_sensitivity: a weighted sum of final-state tangents is not defined (pass weights or dstate, not both)");
    if (weights && h->comm && h->comm_size > 1)
        return fail(JQ_ERR_ARG, "jq_forward_sensitivity: never communicates; with a communicator attached shard the directions, not the samples (no weights)");
    const int nspl = npar - (h->pfid == 3 ? 1 : 0);
    if (jq_fwdsens_smem_bytes(h->P, nspl) > 227 * 1024)
        return fail(JQ_ERR_ARG, "jq_forward_sensitivity: problem too large for the tangent kernel's shared memory (n*m = %d)", h->n * h->m);
    CU(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    if (h->have_last && h->last_stream != st) CU(cudaStreamWaitEvent(st, h->ev_done, 0));      // shared scratch, see jq_traceobjgrad_batch_device
    const size_t nt = (size_t)nbatch * nsamples, ntraj = nt * ndir, len = (size_t)h->n * h->m;
    const size_t nout = weights ? (size_t)nbatch : nt, ndout = nout * ndir;
    const size_t n_pcof = (size_t)nbatch * npar, n_dirs = (size_t)nbatch * ndir * npar;
    const size_t n_shift = shift ? (size_t)nsamples * h->n : 0, n_w = weights ? (size_t)nsamples : 0;
    const bool want_state = dstate_r || dstate_i;
    const size_t n_state = want_state ? ntraj * len : 0;
    if ((rc = grow(&h->d_in, &h->cap_in, n_pcof + n_dirs + n_shift + n_w)) != 0) return rc;
    if ((rc = grow(&h->d_out, &h->cap_out, 2 * nout + 2 * ndout + 2 * n_state)) != 0) return rc;
    if ((rc = grow(&h->d_scal, &h->cap_traj, nt * 4)) != 0) return rc;
    if ((rc = grow(&h->d_grad, &h->cap_grad, ntraj)) != 0) return rc;
    if ((rc = grow(&h->d_igrad, &h->cap_igrad, ntraj)) != 0) return rc;
    double *d_pcof = h->d_in, *d_dirs = d_pcof + n_pcof, *d_shift = shift ? d_dirs + n_dirs : nullptr;
    double *d_w = weights ? d_dirs + n_dirs + n_shift : nullptr;
    CU(cudaMemcpyAsync(d_pcof, pcof, n_pcof * sizeof(double), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_dirs, dirs, n_dirs * sizeof(double), cudaMemcpyHostToDevice, st));
    if (n_shift) CU(cudaMemcpyAsync(d_shift, shift, n_shift * sizeof(double), cudaMemcpyHostToDevice, st));
    if (n_w) CU(cudaMemcpyAsync(d_w, weights, n_w * sizeof(double), cudaMemcpyHostToDevice, st));
    double *o_infid = h->d_out, *o_leak = o_infid + nout, *o_dinf = o_leak + nout, *o_dleak = o_dinf + ndout;
    double *o_sr = want_state ? o_dleak + ndout : nullptr, *o_si = want_state ? o_sr + n_state : nullptr;

    SensArgs S{};
    S.ntraj = (int)ntraj; S.nsamples = nsamples; S.ndir = ndir; S.Npar = nspl; S.D1 = nspl / (2 * h->Nc * h->Nfreq); S.pstride = npar;
    S.pcof = d_pcof; S.dirs = d_dirs; S.shift = d_shift;
    S.scal = h->d_scal; S.dinfid = h->d_grad; S.dleak = h->d_igrad; S.dstate_r = o_sr; S.dstate_i = o_si;
    int ctas = 0, regs = 0, gpc = 1;
    size_t smem = 0;
    CU(cudaEventRecord(h->ev0, st));
    CU(jq_fwdsens_launch(h->P, S, st, &ctas, &regs, &smem, &gpc));
    CU(cudaEventRecord(h->ev1, st));
    h->timed = true;
    h->last_kernel = 8; h->last_ctas = ctas; h->last_regs = regs; h->last_smem = smem; h->last_tpc = gpc; h->last_traj_launches = 1;
    // per-trajectory outputs or the weighted sums over the samples, in the fixed order of the evaluation path's reductions: the
    // directions take the place of the gradient columns (dinfid as `grad`, dleak as `infidgrad`)
    if (weights && nsamples >= 64)
        jq_weighted_sum_kernel<<<dim3(nbatch, (ndir + 3 + 31) / 32), 32 * WS_LANES, 0, st>>>(nsamples, ndir, 2, 1, d_w, h->d_scal, h->d_grad,
                                          h->d_igrad, o_infid, o_leak, nullptr, o_dinf, o_dleak, nullptr);
    else {
        const long long total = (long long)nout * (ndir + 1);
        const int fb = 256, fg = (int)std::min<long long>((total + fb - 1) / fb, 148 * 8);
        jq_finalize_kernel<<<fg, fb, 0, st>>>(nbatch, nsamples, ndir, 2, 1, d_w, h->d_scal, h->d_grad, h->d_igrad, o_infid, o_leak, nullptr,
                                              o_dinf, o_dleak, nullptr);
    }
    CU(cudaGetLastError());
    h->last_launches = 2;
    CU(cudaEventRecord(h->ev_done, st));
    h->last_stream = st; h->have_last = true;
    if (infid) CU(cudaMemcpyAsync(infid, o_infid, nout * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (leak) CU(cudaMemcpyAsync(leak, o_leak, nout * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (dinfid) CU(cudaMemcpyAsync(dinfid, o_dinf, ndout * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (dleak) CU(cudaMemcpyAsync(dleak, o_dleak, ndout * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (dstate_r) CU(cudaMemcpyAsync(dstate_r, o_sr, n_state * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (dstate_i) CU(cudaMemcpyAsync(dstate_i, o_si, n_state * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return 0;
}
