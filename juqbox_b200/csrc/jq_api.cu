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
#include <initializer_list>
#include <memory>
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

struct PlanFree { void operator()(TrajPlan *p) const { jq_traj_plan_destroy(p); } };
using PlanPtr = std::unique_ptr<TrajPlan, PlanFree>;

// A way to serve a launch: a kernel (jq_set_kernel / jq_query(0) id) and, for the register-resident layouts, its plan (for the
// time-parallel evaluation the plan of its segment sweeps).  Indices 0-6 are the routes of kernel ids 1-7; the in-lane tiles are a
// second route of id 4.
enum RouteId { GENERIC, SLOT, FIBER, TILE, LATENCY, DENSE, TIME_PARALLEL, TILE_INLANE, NROUTES };
struct Route {
    int kernel = 0;
    TrajPlan *plan = nullptr;
    bool ok = false;
    char why[300] = "";     // !ok: why jq_set_kernel refuses the kernel id
};

// What the last evaluation ran (jq_query items 0 and 3-7)
struct Ran {
    int kernel = 0, ctas = 0, regs = 0, tpc = 1;
    size_t smem = 0;
    int nseg = 0;           // time segments (kernel 7)
    int launches = 1;       // kernel launches of the trajectory work (the time-parallel evaluation makes several)
};

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
    std::vector<PlanPtr> plans;         // every trajectory plan; the routes and the roles below point into it
    Route route[NROUTES];
    int tile_in_ntraj = 0;              // automatic mode: launches with at least this many trajectories use the in-lane tiles
    bool dense_auto = false;            // the dense kernel can serve this problem and the operators are dense enough for it to beat the
                                        // row-wise generic kernel
    int lat_ntraj = 0;                  // automatic mode: launches with at most this many trajectories use the latency layout
    // time-parallel evaluation (jq_seg.cu, kernel id 7): its route's plan runs the segment sweeps (the tile layout with the fewest
    // elements per lane, else the fibre plan); seg_prop: plan of the propagator launch; seg_obj: of the gradient sweep for
    // objFuncType 2/3.  Workspace, segments (0 = automatic)
    TrajPlan *seg_prop = nullptr, *seg_obj = nullptr;
    double *d_seg = nullptr; size_t cap_seg = 0;
    double *d_segt = nullptr; size_t cap_segt = 0; int segt_nseg = 0; std::vector<double> segt;
    int seg_nseg = 0, seg_ntraj = 0, sms = 148;
    int kernel_pref = 0;
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
    Ran ran;
    int last_launches = 0;              // every launch of the last entry (jq_query(2)): the trajectory work, reductions, all-reduce
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

// grow() for the buffers of the history derivatives, which reach hundreds of MB (cnot3 at save_every = 1: ~128 MB per trajectory and
// cotangent or direction): a request larger than the device, or one cudaMalloc cannot satisfy, is JQ_ERR_ALLOC with the size
static int grow_history(double **buf, size_t *cap, double need, const char *who) {
    size_t free_b = 0, total_b = 0;
    CU(cudaMemGetInfo(&free_b, &total_b));
    if (need * sizeof(double) > (double)total_b)
        return fail(JQ_ERR_ALLOC, "%s: needs %.1f GB in one device buffer, the device has %.1f GB", who, need * sizeof(double) / 1e9,
                    total_b / 1e9);
    if ((size_t)need <= *cap) return 0;
    if (*buf) cudaFree(*buf);
    *buf = nullptr;
    *cap = 0;
    const cudaError_t e = cudaMalloc((void **)buf, (size_t)need * sizeof(double));
    if (e != cudaSuccess) {
        *buf = nullptr;
        cudaGetLastError();
        return fail(e == cudaErrorMemoryAllocation ? JQ_ERR_ALLOC : JQ_ERR_CUDA, "%s: cudaMalloc of %.1f GB: %s", who,
                    need * sizeof(double) / 1e9, cudaGetErrorString(e));
    }
    *cap = (size_t)need;
    return 0;
}

// The host arrays of an entry, staged through the handle's d_in / d_out: n doubles at *dev.  An input takes space and a device pointer
// when the caller gave it (src) and is copied there before the launch; an output takes them when it has entries and is copied to dst,
// when given, after the launch.  Counts are doubles because history sizes can overflow size_t; grow_history rejects them by size.
struct In { double **dev; double n; const double *src; };
struct Out { double **dev; double n; double *dst; };

// Size d_in and d_out for an entry's arrays (grow(), or grow_history() for the history entries, `history` naming the entry), hand out
// the device pointers in list order and copy the inputs to the device
static int stage(jq_handle *h, const char *history, std::initializer_list<In> in, std::initializer_list<Out> out, cudaStream_t st) {
    double n_in = 0.0, n_out = 0.0;
    for (const In &a : in) n_in += a.src ? a.n : 0.0;
    for (const Out &a : out) n_out += a.n;
    int rc = history ? grow_history(&h->d_in, &h->cap_in, n_in, history) : grow(&h->d_in, &h->cap_in, (size_t)n_in);
    if (rc || (rc = history ? grow_history(&h->d_out, &h->cap_out, n_out, history) : grow(&h->d_out, &h->cap_out, (size_t)n_out)) != 0)
        return rc;
    double *p = h->d_in;
    for (const In &a : in) {
        *a.dev = a.src ? p : nullptr;
        if (a.src) p += (size_t)a.n;
    }
    p = h->d_out;
    for (const Out &a : out) {
        *a.dev = a.n > 0 ? p : nullptr;
        p += (size_t)a.n;
    }
    for (const In &a : in)
        if (a.src && a.n > 0) CU(cudaMemcpyAsync(*a.dev, a.src, (size_t)a.n * sizeof(double), cudaMemcpyHostToDevice, st));
    return 0;
}

// Copy an entry's outputs back to the host and wait for them
static int read_back(std::initializer_list<Out> out, cudaStream_t st) {
    for (const Out &a : out)
        if (a.dst && a.n > 0) CU(cudaMemcpyAsync(a.dst, *a.dev, (size_t)a.n * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return 0;
}

// Run `launch(ran)`, the trajectory work of an entry on kernel `kernel` (jq_query(0)), between the timing events, and record what ran:
// jq_query reports it, and the entry's launch count starts from it
template <class Launch>
static int record_launch(jq_handle *h, int kernel, cudaStream_t st, Launch &&launch) {
    CU(cudaEventRecord(h->ev0, st));
    Ran ran;
    ran.kernel = kernel;
    if (int rc = launch(ran)) return rc;
    CU(cudaEventRecord(h->ev1, st));
    h->timed = true;
    h->ran = ran;
    h->last_launches = ran.launches;
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
    auto own = [h](TrajPlan *p) { if (p) h->plans.emplace_back(p); return p; };
    auto set_route = [h](RouteId id, int kernel, TrajPlan *plan, bool ok, const char *missing, const char *reason) {
        Route &r = h->route[id];
        r.kernel = kernel; r.plan = plan; r.ok = ok;
        if (!ok) snprintf(r.why, sizeof(r.why), reason ? "%s (%s)" : "%s", missing, reason);
    };
    char why[256];
    set_route(GENERIC, 1, nullptr, true, "", nullptr);
    TrajPlan *slot = own(jq_slot_plan_create(P, H, pb->wdiag, why, sizeof(why)));
    set_route(SLOT, 2, slot, slot, "no slot-layout instantiation for this problem", why);
    TrajPlan *fiber = own(jq_fiber_plan_create(P, H, pb->wdiag, why, sizeof(why)));
    set_route(FIBER, 3, fiber, fiber, "no fibre-layout instantiation for this problem", why);
    TrajPlan *tile = own(jq_tile_plan_create(P, H, pb->wdiag, Nc, 0, why, sizeof(why)));
    set_route(TILE, 4, tile, tile, "no tile-layout instantiation for this problem", why);
    // Two subsystems, first one whole in the lane (TileLane<2,1,1>): half the exchange shuffles per element of the 2 x 2 tiles
    // and twice the independent element chains per lane, but 4 instead of 2 trajectories per warp
    const char *ti = getenv("JQ_TILE_INLANE");      // development: 0 = never, 1 = for every launch, unset = automatic
    TrajPlan *tile_in = tile && !(ti && atoi(ti) == 0) ? own(jq_tile_plan_create(P, H, pb->wdiag, 1, 1, why, sizeof(why))) : nullptr;
    set_route(TILE_INLANE, 4, tile_in, tile_in, "no in-lane tile instantiation for this problem", nullptr);
    // Latency layout: a trajectory spread over as many lanes as the warp-local exchange allows (one element per lane for two
    // subsystems, two for three), with pipelined roles.  A lone evaluation (the reference's own call pattern, one pcof per Ipopt
    // callback) is bound by the instruction stream of ONE lane, so fewer elements per lane is what shortens it; throughput layouts
    // win once the SMs are full.
    TrajPlan *lat = own(jq_tile_plan_create(P, H, pb->wdiag, Nc == 2 ? 0 : 1, 0, why, sizeof(why), 1));
    if (!lat) lat = own(jq_fiber_plan_create(P, H, pb->wdiag, why, sizeof(why), 1));     // single-fibre shapes: same layout, pipelined roles
    set_route(LATENCY, 5, lat, lat, "no latency layout for this problem", nullptr);
    const bool dense_ok = jq_dense_supported(P, why, sizeof(why));
    set_route(DENSE, 6, nullptr, dense_ok, "the dense (tensor-core) kernel cannot serve this problem", why);
    // a dense contraction executes n^2 multiply-adds per product and column whatever the sparsity: worth it from ~20% fill
    // (measured: 5%-filled ladder operators with remote exchange run 1.6x faster on the row-wise generic kernel)
    size_t nnz = 0;
    for (double v : h->val) nnz += v != 0.0;
    h->dense_auto = dense_ok && n >= 8 && (double)nnz >= 0.2 * (double)(1 + 2 * Nc) * n * n;
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    h->sms = sms;
    // one latency CTA per SM: beyond that the throughput layouts win (measured)
    h->lat_ntraj = sms * (lat ? jq_traj_plan_tpc(lat) : 1);
    // in-lane tiles from one full resident wave of them (2 CTAs of 16 trajectories per SM, 4736 on 148 SMs): below it their
    // CTAs leave SMs half empty where the 2 x 2 tiles (wave 2368) fill them.  Measured cnot2 speed-up over the 2 x 2 tiles (B200,
    // 1000 W; profiles/r03_tile_inlane.md): 0.88x at 2368 and 0.85x at 3552 candidates; 1.09x at 4736, 1.06x at 7104, 1.10x at
    // 9472 and 16384, 1.12x at 32768.
    if (tile_in) h->tile_in_ntraj = ti && atoi(ti) == 1 ? 0 : 2 * sms * jq_traj_plan_tpc(tile_in);
    // Time-parallel evaluation for launches of very few trajectories (one pcof per Ipopt callback): segments of the time axis
    // swept concurrently and joined through their propagators.  The segment sweeps run on the tile layout with the fewest elements
    // per lane, else on the fibre plan; objFuncType 2/3: the gradient sweep needs the second adjoint set, which the fibre layout has
    TrajPlan *seg = own(jq_tile_plan_create(P, H, pb->wdiag, Nc == 2 ? 0 : 1, 0, why, sizeof(why), 0, true));
    if (!seg) seg = fiber;
    if (!jq_seg_supported(seg, P) || (P.objFuncType != 1 && !jq_seg_supported(fiber, P, true))) seg = nullptr;
    set_route(TIME_PARALLEL, 7, seg, seg,
              "no time-parallel evaluation for this problem (needs a tile / fibre layout, the Neumann solver, diagonal weights)", nullptr);
    if (seg) {
        h->seg_obj = P.objFuncType != 1 ? fiber : nullptr;
        // propagator launch (many independent unit-vector sweeps): the throughput tile layout when the problem has one
        h->seg_prop = jq_seg_supported(tile, P) ? tile : seg;
        // automatic mode: time-parallel while the propagator launch (2 x 2n/m unit-vector sweeps per trajectory and segment) stays
        // within about four warps per SM -- measured cross-overs against the other kernels: cnot2 ~60 candidates, cnot3 ~30,
        // risk-neutral ~1100 samples (profiles/r02_timeparallel.md)
        const int lanes = std::max(1, jq_traj_plan_lanes(h->seg_prop)), nblk = (2 * n + m - 1) / m;
        h->seg_ntraj = std::max(1, (4 * sms * 32) / (2 * nblk * lanes));
    }
    if (const char *sn = getenv("JQ_SEG_NTRAJ")) h->seg_ntraj = atoi(sn);
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
    h->plans.clear();
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
    if (kernel > 0 && !h->route[kernel - 1].ok) return fail(JQ_ERR_ARG, "jq_set_kernel: %s", h->route[kernel - 1].why);
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
    case 0: *value = h->ran.kernel; break;
    case 1: {
        if (!h->timed) return fail(JQ_ERR_ARG, "jq_query: no evaluation has run yet");
        CU(cudaEventSynchronize(h->ev1));
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
        *value = ms;
        break;
    }
    case 2: *value = h->last_launches; break;
    case 3: *value = h->ran.tpc; break;
    case 4: *value = h->ran.ctas; break;
    case 5: *value = h->ran.regs; break;
    case 6: *value = (double)h->ran.smem; break;
    case 7: *value = h->ran.nseg; break;
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


// Per-candidate outputs of `ncol` columns (gradient entries or directions) and the three scalars of every trajectory: copies
// (w == nullptr) or weighted sums over the samples, with jq_weighted_sum_kernel from 64 samples on.  The two kernels add in
// different orders, so the rule that picks one fixes the bits of the sums.
static void launch_finalize(int nbatch, int nsamples, int ncol, int objFuncType, int evaladjoint, const double *w, const double *scal,
                            const double *gt, const double *igt, double *infid, double *leak, double *tinfid, double *grad,
                            double *infidgrad, double *leakgrad, cudaStream_t st) {
    if (w && nsamples >= 64) {
        jq_weighted_sum_kernel<<<dim3(nbatch, (ncol + 3 + 31) / 32), 32 * WS_LANES, 0, st>>>(nsamples, ncol, objFuncType, evaladjoint, w, scal,
                                          gt, igt, infid, leak, tinfid, grad, infidgrad, leakgrad);
        return;
    }
    const long long total = (long long)(w ? nbatch : nbatch * nsamples) * (ncol + 1);
    const int fb = 256, fg = (int)std::min<long long>((total + fb - 1) / fb, 148 * 8);
    jq_finalize_kernel<<<fg, fb, 0, st>>>(nbatch, nsamples, ncol, objFuncType, evaladjoint, w, scal, gt, igt, infid, leak, tinfid, grad,
                                          infidgrad, leakgrad);
}

// The handle's scratch (d_scal, d_grad, d_igrad) is shared by every call: a call on a different stream than the previous one
// (host-pointer entries = the handle's own stream, device entry = the caller's) first waits for that one to finish
static int scratch_acquire(jq_handle *h, cudaStream_t st) {
    if (h->have_last && h->last_stream != st) CU(cudaStreamWaitEvent(st, h->ev_done, 0));
    return 0;
}

static int scratch_release(jq_handle *h, cudaStream_t st) {
    CU(cudaEventRecord(h->ev_done, st));
    h->last_stream = st; h->have_last = true;
    return 0;
}

// The spline coefficients of a caller's vector of npar entries (pFidType 3: the last entry is the global phase, src/evalobjgrad.jl:591-596)
// and D1, their number per control function and carrier
struct Splines { int nspl, D1; };
static Splines splines(const jq_handle *h, int npar) {
    const int nspl = npar - (h->pfid == 3 ? 1 : 0);
    return {nspl, nspl / (2 * h->Nc * h->Nfreq)};
}

// Arguments of a launch over nbatch x nsamples trajectories.  npar is the caller's vector length: the spline coefficients, plus the
// global phase as last entry for pFidType 3; gradients have the same length.
static LaunchArgs launch_args(const jq_handle *h, int nbatch, int npar, int nsamples, const double *pcof, const double *shift) {
    const Splines s = splines(h, npar);
    LaunchArgs A{};
    A.ntraj = nbatch * nsamples; A.nsamples = nsamples; A.Npar = s.nspl; A.D1 = s.D1;
    A.pstride = npar; A.gstride = npar;
    A.pcof = pcof; A.shift = shift; A.scal = h->d_scal;
    return A;
}

// The routes a launch tries, in order.  An explicit preference has only its own routes; automatic mode lists every route that may
// serve the launch, the fastest for its size first.
static int launch_routes(const jq_handle *h, const LaunchArgs &A, int pref, const Route *out[NROUTES]) {
    int n = 0;
    auto add = [&](RouteId id) {
        if (!h->route[id].ok) return;
        for (int i = 0; i < n; ++i) if (out[i] == &h->route[id]) return;
        out[n++] = &h->route[id];
    };
    auto tiles = [&]() { if (A.ntraj >= h->tile_in_ntraj) add(TILE_INLANE); add(TILE); };
    if (pref == 4) tiles();
    else if (pref > 0) add(RouteId(pref - 1));
    if (pref != 0) return n;
    // very few trajectories: time-parallel evaluation (segments of the time axis swept concurrently)
    if (h->P.solver == 1 && !A.hist_r && A.ntraj <= h->seg_ntraj && h->P.nsteps >= 256) add(TIME_PARALLEL);
    const bool small = A.ntraj <= h->lat_ntraj;
    if (small) add(LATENCY);
    if (small && h->route[TILE].ok && h->Nc >= 3) add(FIBER);     // three subsystems: the fibre layout (4 elements per lane) before the 8-element tiles
    tiles();
    add(FIBER);
    add(SLOT);
    // unstructured operators: the products are real contractions -> FP64 tensor-core kernel, samples of a candidate batched
    if (h->dense_auto && !A.hist_r) add(DENSE);
    add(GENERIC);
    return n;
}

// Outcome of a route's launch: 0, HANDED_OVER for an error after which automatic mode tries the next route (the route cannot serve
// this launch: no instantiation for the variant, shared-memory layout does not fit, out of launch resources), else the error
static const int HANDED_OVER = 1;
static int launched(cudaError_t e, bool hand_over, const char *what) {
    if (e == cudaSuccess) return 0;
    cudaGetLastError();                                   // clear the (non-sticky) launch error before trying the next route
    const bool soft = e == cudaErrorInvalidConfiguration || e == cudaErrorNotSupported || e == cudaErrorLaunchOutOfResources;
    return soft && hand_over ? HANDED_OVER : fail(JQ_ERR_CUDA, "%s failed: %s", what, cudaGetErrorString(e));
}

// Segments of a time-parallel launch of ntraj trajectories: jq_set_time_segments, or automatic (jq_seg_auto_segments)
static int seg_count(const jq_handle *h, int ntraj, int evaladjoint) {
    const int nseg = h->seg_nseg > 0 ? h->seg_nseg : jq_seg_auto_segments(h->P, ntraj, evaladjoint, jq_traj_plan_tpc(h->seg_prop), h->sms);
    return nseg > h->P.nsteps ? (int)h->P.nsteps : nseg;
}

// Segment start / end times of nseg segments on the device, then the four refinement flags (int): host recurrence, uploaded once per
// segment count
static int seg_times_upload(jq_handle *h, int nseg, cudaStream_t st) {
    if (h->segt_nseg == nseg) return 0;
    h->segt.resize(2 * (size_t)nseg);
    jq_seg_times(h->P, nseg, h->segt.data());
    int rc = grow(&h->d_segt, &h->cap_segt, 2 * (size_t)nseg + 2);
    if (rc) return rc;
    CU(cudaMemcpyAsync(h->d_segt, h->segt.data(), 2 * (size_t)nseg * sizeof(double), cudaMemcpyHostToDevice, st));
    h->segt_nseg = nseg;
    return 0;
}

// The time-parallel evaluation of `A`
static int launch_time_parallel(jq_handle *h, const LaunchArgs &A, cudaStream_t st, Ran &ran, bool hand_over) {
    if (h->P.solver != 1 || A.hist_r) return fail(JQ_ERR_ARG, "time-parallel evaluation: Neumann solver, no state history");
    const int tpc = jq_traj_plan_tpc(h->seg_prop);
    int nseg = seg_count(h, A.ntraj, A.evaladjoint);
    // cooperative evaluation: the segments are shared out evenly over the ranks (every rank computes the same nseg)
    // ... when the propagator launch is at least two waves of CTAs: below that its collective costs more than it saves
    const long long l1_ctas = 2LL * nseg * (((long long)((2 * h->n + h->m - 1) / h->m) * A.ntraj + tpc - 1) / tpc);
    const char *cf = getenv("JQ_SEG_COOP_FORCE");     // tests: share out small problems too
    const bool coop_on = h->cooperative && h->comm && h->comm_size > 1 && h->P.nsteps >= h->comm_size &&
                         (l1_ctas >= 2LL * h->sms || (cf && atoi(cf)));
    if (coop_on) {
        nseg = std::max(h->comm_size, (nseg + h->comm_size - 1) / h->comm_size * h->comm_size);
        if (nseg > h->P.nsteps) nseg = (int)(h->P.nsteps / h->comm_size) * h->comm_size;       // >= comm_size by the test above
    }
    SegCoop coop{h->comm_rank, h->comm_size, seg_allgather, h};
    int rc = grow(&h->d_seg, &h->cap_seg, jq_seg_workspace(h->P, A.ntraj, A.Npar, nseg, false, A.evaladjoint, false));
    if (rc) return rc;
    if ((rc = seg_times_upload(h, nseg, st)) != 0) return rc;
    ran.nseg = nseg;
    return launched(jq_seg_launch(h->seg_prop, h->route[TIME_PARALLEL].plan, h->seg_obj, h->P, A, nseg, h->d_segt,
                                  reinterpret_cast<int *>(h->d_segt + 2 * (size_t)nseg), h->d_seg, st, coop_on && nseg >= h->comm_size ? &coop : nullptr,
                                  &ran.ctas, &ran.regs, &ran.smem, &ran.tpc, &ran.launches),
                    hand_over, "time-parallel evaluation");
}

// Launch route `r` for `A`, recording what ran in `ran`
static int launch_route(jq_handle *h, const Route &r, const LaunchArgs &A, cudaStream_t st, Ran &ran, bool hand_over) {
    switch (r.kernel) {
    case 7: return launch_time_parallel(h, A, st, ran, hand_over);
    case 6: return launched(jq_dense_launch(h->P, A, st, &ran.ctas, &ran.regs, &ran.smem, &ran.tpc), hand_over, "dense kernel launch");
    case 1:
        if (jq_generic_smem_bytes(h->P, A.Npar) > 227 * 1024)
            return fail(JQ_ERR_ARG, "problem too large for the generic kernel's shared memory (n*m = %d)", h->n * h->m);
        return launched(jq_generic_launch(h->P, A, st, &ran.ctas, &ran.regs, &ran.smem), hand_over, "generic kernel launch");
    default: return launched(jq_traj_launch(r.plan, h->P, A, st, &ran.ctas, &ran.regs, &ran.smem, &ran.tpc), hand_over, "trajectory kernel launch");
    }
}

// Launch the trajectory work for `A` on the first of its routes that serves it: automatic mode hands over to the next route, an
// explicitly requested kernel fails instead.
static int launch_trajectories(jq_handle *h, const LaunchArgs &A, cudaStream_t st) {
    const int pref = h->kernel_pref;
    const Route *routes[NROUTES];
    const int n = launch_routes(h, A, pref, routes);
    return record_launch(h, 0, st, [&](Ran &ran) {
        int rc = HANDED_OVER;
        for (int i = 0; i < n && rc == HANDED_OVER; ++i) {
            ran = Ran();
            ran.kernel = routes[i]->kernel;
            rc = launch_route(h, *routes[i], A, st, ran, pref == 0 && i + 1 < n);
        }
        return rc;
    });
}

// The batch arguments every entry checks.  The derivative entries run `per_traj` trajectories (directions or cotangents) per candidate
// and sample; `who` names the entry in the trajectory-count message.
static int check_batch_args(jq_handle *h, int nbatch, const double *pcof, int npar, int nsamples, const double *shift,
                            bool empty_shard_ok = false, int per_traj = 1, const char *who = nullptr) {
    if (!h) return fail(JQ_ERR_ARG, "null handle");
    if (nbatch < 1 || !pcof) return fail(JQ_ERR_ARG, "need nbatch >= 1 and a pcof array");
    const int nsig = 2 * h->Nc, nspl = splines(h, npar).nspl;
    if (nspl % nsig != 0 || nspl < 3 * nsig)   // src/evalobjgrad.jl:604-606
        return fail(JQ_ERR_PCOF_LENGTH, "pcof must have an even number of elements >= %d, not %d", 3 * nsig, nspl);
    if (nspl % (nsig * h->Nfreq) != 0 || nspl / (nsig * h->Nfreq) < 3)   // src/bsplines.jl:177-181 (and k >= 3 needs D1 >= 3)
        return fail(JQ_ERR_PCOF_LENGTH, "Inconsistent number of coefficients and size of parameter vector (nCoeff = %d, Nfreq = %d, Ncoupled + Nunc = %d)", nspl, h->Nfreq, h->Nc);
    // an empty sample shard (more ranks than quadrature nodes) contributes zeros and still joins the all-reduce
    if (nsamples < (empty_shard_ok ? 0 : 1)) return fail(JQ_ERR_ARG, "nsamples must be >= 1 (0 only with weights: an empty sample shard)");
    if ((long long)nbatch * nsamples * per_traj > 0x7fffffffLL)
        return fail(JQ_ERR_ARG, "%s%snbatch * nsamples%s exceeds 2^31 - 1 trajectories per call", who ? who : "", who ? ": " : "",
                    per_traj > 1 ? " * (directions or cotangents)" : "");
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
    if ((rc = scratch_acquire(h, st)) != 0) return rc;
    if ((rc = grow(&h->d_scal, &h->cap_traj, ntraj * 4)) != 0) return rc;
    if (evaladjoint && (rc = grow(&h->d_grad, &h->cap_grad, ntraj * npar)) != 0) return rc;
    if (evaladjoint && h->P.objFuncType != 1 && (rc = grow(&h->d_igrad, &h->cap_igrad, ntraj * npar)) != 0) return rc;

    LaunchArgs A = launch_args(h, nbatch, npar, nsamples, pcof, shift);
    A.evaladjoint = evaladjoint ? 1 : 0;
    A.grad = h->d_grad; A.infidgrad = h->P.objFuncType != 1 ? h->d_igrad : nullptr;
    if (ntraj > 0 && (rc = launch_trajectories(h, A, st)) != 0) return rc;
    launch_finalize(nbatch, nsamples, npar, h->P.objFuncType, A.evaladjoint, weights, h->d_scal, h->d_grad, h->d_igrad, infid, leak,
                    trace_infid, grad, infidgrad, leakgrad, st);
    CU(cudaGetLastError());
    h->last_launches = 1 + h->ran.launches;
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
    return scratch_release(h, st);
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
        cudaStream_t st = h->stream;
        const double one = 1.0;                 // no weights: the single sample has weight 1
        std::vector<double> pack(3 + 3 * (size_t)npar);
        double *d_pcof, *d_shift, *d_w, *d_prior, *o_infid, *o_leak, *o_tinf, *o_g, *o_ig, *o_lg, *o_pack;
        const std::initializer_list<Out> out = {{&o_infid, 1, nullptr}, {&o_leak, 1, nullptr}, {&o_tinf, 1, nullptr}, {&o_g, (double)npar, nullptr},
                                                {&o_ig, two ? (double)npar : 0.0, nullptr}, {&o_lg, two ? (double)npar : 0.0, nullptr},
                                                {&o_pack, (double)pack.size(), pack.data()}};
        rc = stage(h, nullptr, {{&d_pcof, (double)npar, pcof}, {&d_shift, (double)n_shift, shift}, {&d_w, n_w ? (double)n_w : 1.0, n_w ? weights : &one},
                                {&d_prior, (double)npar, prior}}, out, st);
        if (rc) return rc;
        rc = jq_traceobjgrad_batch_device(h, 1, d_pcof, npar, nsamples, d_shift, d_w, 1, o_infid, o_leak, o_tinf, o_g, o_ig, o_lg, st);
        if (rc) return rc;
        jq_tikhonov_kernel<<<1, 256, 0, st>>>(npar, h->P.objFuncType, tik0, d_pcof, d_prior, o_infid, o_leak, two ? o_ig : o_g, o_lg, o_pack);
        CU(cudaGetLastError());
        h->last_launches += 1;
        if ((rc = read_back(out, st)) != 0) return rc;
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

// the saving stride of the history entries (jq_eval_forward, jq_history_vjp, jq_history_jvp)
static int check_save_every(const jq_handle *h, int save_every) {
    if (save_every < 1 || h->P.nsteps % save_every != 0)     // src/evalobjgrad.jl:2797-2799
        return fail(JQ_ERR_ARG, "nsteps must be divisible by saveEvery. nsteps=%lld, saveEvery=%d", (long long)h->P.nsteps, save_every);
    return 0;
}

extern "C" int jq_eval_forward(jq_handle *h, int32_t nbatch, const double *pcof, int32_t npar, int32_t nsamples, const double *shift,
                               int32_t save_every, double *hist_r, double *hist_i, double *infid, double *leak) {
    int rc = check_batch_args(h, nbatch, pcof, npar, nsamples, shift);
    if (rc) return rc;
    if (!hist_r || !hist_i) return fail(JQ_ERR_ARG, "jq_eval_forward: null history buffer");
    if ((rc = check_save_every(h, save_every)) != 0) return rc;
    CU(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const size_t ntraj = (size_t)nbatch * nsamples;
    const long long nsave = h->P.nsteps / save_every + 1;
    const double n_hist = (double)ntraj * nsave * h->n * h->m;
    double *d_pcof, *d_shift, *o_hr, *o_hi;
    const std::initializer_list<Out> out = {{&o_hr, n_hist, hist_r}, {&o_hi, n_hist, hist_i}};
    if ((rc = stage(h, nullptr, {{&d_pcof, (double)nbatch * npar, pcof}, {&d_shift, (double)nsamples * h->n, shift}}, out, st)) != 0) return rc;
    if ((rc = grow(&h->d_scal, &h->cap_traj, ntraj * 4)) != 0) return rc;
    LaunchArgs A = launch_args(h, nbatch, npar, nsamples, d_pcof, d_shift);
    A.hist_r = o_hr; A.hist_i = o_hi; A.save_every = save_every; A.nsave = nsave;
    if ((rc = launch_trajectories(h, A, st)) != 0) return rc;      // same kernel choice as jq_traceobjgrad_batch
    if ((rc = read_back(out, st)) != 0) return rc;
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
    cudaStream_t st = h->stream;
    const double nout = (double)h->Nc * ntimes;
    double *d_pcof, *d_times, *o_p, *o_q;
    const std::initializer_list<Out> out = {{&o_p, nout, p}, {&o_q, nout, q}};
    if ((rc = stage(h, nullptr, {{&d_pcof, (double)npar, pcof}, {&d_times, (double)ntimes, times}}, out, st)) != 0) return rc;
    CU(jq_controls_launch(h->P, splines(h, npar).D1, d_pcof, ntimes, d_times, o_p, o_q, st));
    return read_back(out, st);
}

extern "C" int jq_traceobjgrad_batch(jq_handle *h, int32_t nbatch, const double *pcof, int32_t npar, int32_t nsamples,
                                     const double *shift, const double *weights, int32_t evaladjoint, double *infid, double *leak,
                                     double *trace_infid, double *grad, double *infidgrad, double *leakgrad) {
    int rc = check_batch_args(h, nbatch, pcof, npar, nsamples, shift, weights != nullptr);
    if (rc) return rc;
    CU(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const double nout = weights ? nbatch : (double)nbatch * nsamples, ngrad = nout * npar;
    const bool want_g = evaladjoint && grad, want_ig = evaladjoint && infidgrad, want_lg = evaladjoint && leakgrad && h->P.objFuncType != 1;
    double *d_pcof, *d_shift, *d_w, *o_infid, *o_leak, *o_tinf, *o_g, *o_ig, *o_lg;
    const std::initializer_list<Out> out = {{&o_infid, nout, infid}, {&o_leak, nout, leak}, {&o_tinf, nout, trace_infid},
                                            {&o_g, want_g ? ngrad : 0.0, grad}, {&o_ig, want_ig ? ngrad : 0.0, infidgrad},
                                            {&o_lg, want_lg ? ngrad : 0.0, leakgrad}};
    // an empty sample shard's weights take no space but keep a valid pointer
    rc = stage(h, nullptr, {{&d_pcof, (double)nbatch * npar, pcof}, {&d_shift, (double)nsamples * h->n, shift}, {&d_w, (double)nsamples, weights}},
               out, st);
    if (rc) return rc;
    rc = jq_traceobjgrad_batch_device(h, nbatch, d_pcof, npar, nsamples, d_shift, d_w, evaladjoint, o_infid, o_leak, o_tinf, o_g, o_ig,
                                      o_lg, st);
    if (rc) return rc;
    return read_back(out, st);
}

// The tangent kernel's (kernel 8) checks that both forward-mode entries make
static int check_tangent_kernel(const jq_handle *h, const char *who, int npar) {
    if (h->P.solver == 2) return fail(JQ_ERR_ARG, "%s: the Jacobi solver has no tangent sweep (use the Neumann solver)", who);
    if (jq_fwdsens_smem_bytes(h->P, splines(h, npar).nspl) > 227 * 1024)
        return fail(JQ_ERR_ARG, "%s: problem too large for the tangent kernel's shared memory (n*m = %d)", who, h->n * h->m);
    return 0;
}

// The tangent kernel's arguments for ndir directions per (candidate, sample) of staged inputs.  Its scalars and directional derivatives
// go to the handle's scratch (d_scal, d_grad, d_igrad), grown here.
static int tangent_args(jq_handle *h, int nbatch, int npar, int nsamples, int ndir, const double *pcof, const double *dirs,
                        const double *shift, SensArgs *S) {
    const size_t nt = (size_t)nbatch * nsamples, ntraj = nt * ndir;
    int rc = grow(&h->d_scal, &h->cap_traj, nt * 4);
    if (rc || (rc = grow(&h->d_grad, &h->cap_grad, ntraj)) != 0 || (rc = grow(&h->d_igrad, &h->cap_igrad, ntraj)) != 0) return rc;
    const Splines s = splines(h, npar);
    *S = SensArgs{};
    S->ntraj = (int)ntraj; S->nsamples = nsamples; S->ndir = ndir; S->Npar = s.nspl; S->D1 = s.D1; S->pstride = npar;
    S->pcof = pcof; S->dirs = dirs; S->shift = shift;
    S->scal = h->d_scal; S->dinfid = h->d_grad; S->dleak = h->d_igrad;
    return 0;
}

extern "C" int jq_forward_sensitivity(jq_handle *h, int32_t nbatch, const double *pcof, int32_t npar, int32_t nsamples,
                                      const double *shift, const double *weights, int32_t ndir, const double *dirs, double *infid,
                                      double *leak, double *dinfid, double *dleak, double *dstate_r, double *dstate_i) {
    const char *who = "jq_forward_sensitivity";
    int rc = check_batch_args(h, nbatch, pcof, npar, nsamples, shift, false, ndir, who);
    if (rc) return rc;
    if (ndir < 1 || !dirs) return fail(JQ_ERR_ARG, "%s: need ndir >= 1 and a dirs array", who);
    if ((rc = check_tangent_kernel(h, who, npar)) != 0) return rc;
    if (weights && (dstate_r || dstate_i))
        return fail(JQ_ERR_ARG, "%s: a weighted sum of final-state tangents is not defined (pass weights or dstate, not both)", who);
    if (weights && h->comm && h->comm_size > 1)
        return fail(JQ_ERR_ARG, "%s: never communicates; with a communicator attached shard the directions, not the samples (no weights)", who);
    CU(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    if ((rc = scratch_acquire(h, st)) != 0) return rc;
    const double nout = weights ? nbatch : (double)nbatch * nsamples, ndout = nout * ndir;
    const double n_state = dstate_r || dstate_i ? (double)nbatch * nsamples * ndir * h->n * h->m : 0.0;
    double *d_pcof, *d_dirs, *d_shift, *d_w, *o_infid, *o_leak, *o_dinf, *o_dleak, *o_sr, *o_si;
    const std::initializer_list<Out> out = {{&o_infid, nout, infid}, {&o_leak, nout, leak}, {&o_dinf, ndout, dinfid}, {&o_dleak, ndout, dleak},
                                            {&o_sr, n_state, dstate_r}, {&o_si, n_state, dstate_i}};
    rc = stage(h, nullptr, {{&d_pcof, (double)nbatch * npar, pcof}, {&d_dirs, (double)nbatch * ndir * npar, dirs},
                            {&d_shift, (double)nsamples * h->n, shift}, {&d_w, (double)nsamples, weights}}, out, st);
    SensArgs S;
    if (rc || (rc = tangent_args(h, nbatch, npar, nsamples, ndir, d_pcof, d_dirs, d_shift, &S)) != 0) return rc;
    S.dstate_r = o_sr; S.dstate_i = o_si;
    rc = record_launch(h, 8, st, [&](Ran &r) {
        CU(jq_fwdsens_launch(h->P, S, st, &r.ctas, &r.regs, &r.smem, &r.tpc));
        return 0;
    });
    if (rc) return rc;
    // per-trajectory outputs or the weighted sums over the samples, in the fixed order of the evaluation path's reductions: the
    // directions take the place of the gradient columns (dinfid as `grad`, dleak as `infidgrad`)
    launch_finalize(nbatch, nsamples, ndir, 2, 1, d_w, h->d_scal, h->d_grad, h->d_igrad, o_infid, o_leak, nullptr, o_dinf, o_dleak, nullptr, st);
    CU(cudaGetLastError());
    h->last_launches += 1;
    if ((rc = scratch_release(h, st)) != 0) return rc;
    return read_back(out, st);
}

extern "C" int jq_history_jvp(jq_handle *h, int32_t nbatch, const double *pcof, int32_t npar, int32_t nsamples, const double *shift,
                              int32_t save_every, int32_t ndir, const double *dirs, double *dhist_r, double *dhist_i) {
    const char *who = "jq_history_jvp";
    int rc = check_batch_args(h, nbatch, pcof, npar, nsamples, shift, false, ndir, who);
    if (rc) return rc;
    if ((rc = check_save_every(h, save_every)) != 0) return rc;
    if (ndir < 1 || !dirs) return fail(JQ_ERR_ARG, "%s: need ndir >= 1 and a dirs array", who);
    if (!dhist_r || !dhist_i) return fail(JQ_ERR_ARG, "%s: null tangent-history output", who);
    if ((rc = check_tangent_kernel(h, who, npar)) != 0) return rc;
    CU(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    if ((rc = scratch_acquire(h, st)) != 0) return rc;
    const long long nsave = h->P.nsteps / save_every + 1;
    const double n_hist = (double)nbatch * nsamples * ndir * nsave * h->n * h->m;
    double *d_pcof, *d_dirs, *d_shift, *o_hr, *o_hi;
    const std::initializer_list<Out> out = {{&o_hr, n_hist, dhist_r}, {&o_hi, n_hist, dhist_i}};
    // tangent histories reach hundreds of MB: JQ_ERR_ALLOC with the size when they do not fit
    rc = stage(h, who, {{&d_pcof, (double)nbatch * npar, pcof}, {&d_dirs, (double)nbatch * ndir * npar, dirs}, {&d_shift, (double)nsamples * h->n, shift}},
               out, st);
    SensArgs S;
    if (rc || (rc = tangent_args(h, nbatch, npar, nsamples, ndir, d_pcof, d_dirs, d_shift, &S)) != 0) return rc;
    S.dhist_r = o_hr; S.dhist_i = o_hi; S.save_every = save_every; S.nsave = nsave;     // dinfid, dleak: written, not returned
    rc = record_launch(h, 8, st, [&](Ran &r) {
        CU(jq_fwdsens_launch(h->P, S, st, &r.ctas, &r.regs, &r.smem, &r.tpc));
        return 0;
    });
    if (rc || (rc = scratch_release(h, st)) != 0) return rc;
    return read_back(out, st);
}

// The serial VJP entries (kernel 9): cotangents [traj][nsave][n*m] of the saved states.  The final-state entry has one save, U(T)
// (save_every = nsteps), returned in state_r / state_i; `history`: the history entry, nsave saves returned in hist_r / hist_i, its
// buffers grown with grow_history.
static int vjp_serial(jq_handle *h, const char *who, bool history, int32_t nbatch, const double *pcof, int32_t npar, int32_t nsamples,
                      const double *shift, int32_t save_every, int32_t ncot, const double *cot_r, const double *cot_i, double *vjp,
                      double *save_r, double *save_i) {
    int rc = check_batch_args(h, nbatch, pcof, npar, nsamples, shift, false, ncot, who);
    if (rc) return rc;
    if (history && (rc = check_save_every(h, save_every)) != 0) return rc;
    if (ncot < 1 || (!cot_r && !cot_i)) return fail(JQ_ERR_ARG, "%s: need ncot >= 1 and at least one of cot_r, cot_i", who);
    if (!vjp) return fail(JQ_ERR_ARG, "%s: null vjp output", who);
    const Splines s = splines(h, npar);
    if (jq_vjp_smem_bytes(h->P, s.nspl) > 227 * 1024)
        return fail(JQ_ERR_ARG, "%s: problem too large for the VJP kernel's shared memory (n*m = %d)", who, h->n * h->m);
    CU(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const long long nsave = history ? h->P.nsteps / save_every + 1 : 1;
    const double nt = (double)nbatch * nsamples, len = (double)h->n * h->m, n_cot = nt * ncot * nsave * len;
    const double n_save = save_r || save_i ? nt * nsave * len : 0.0;
    double *d_pcof, *d_shift, *d_cr, *d_ci, *o_vjp, *o_sr, *o_si;
    const std::initializer_list<Out> out = {{&o_vjp, nt * ncot * npar, vjp}, {&o_sr, n_save, save_r}, {&o_si, n_save, save_i}};
    rc = stage(h, history ? who : nullptr, {{&d_pcof, (double)nbatch * npar, pcof}, {&d_shift, (double)nsamples * h->n, shift},
                                            {&d_cr, n_cot, cot_r}, {&d_ci, n_cot, cot_i}}, out, st);
    if (rc) return rc;
    VjpArgs V{};
    V.ntraj = nbatch * nsamples * ncot; V.nsamples = nsamples; V.ncot = ncot; V.Npar = s.nspl; V.D1 = s.D1; V.pstride = npar;
    V.pcof = d_pcof; V.shift = d_shift; V.cot_r = d_cr; V.cot_i = d_ci; V.save_every = history ? save_every : h->P.nsteps; V.nsave = nsave;
    V.vjp = o_vjp;
    (history ? V.hist_r : V.state_r) = o_sr;
    (history ? V.hist_i : V.state_i) = o_si;
    rc = record_launch(h, 9, st, [&](Ran &r) {
        CU(jq_vjp_launch(h->P, V, st, &r.ctas, &r.regs, &r.smem, &r.tpc));
        return 0;
    });
    if (rc) return rc;
    return read_back(out, st);
}

extern "C" int jq_final_state_vjp(jq_handle *h, int32_t nbatch, const double *pcof, int32_t npar, int32_t nsamples, const double *shift,
                                  int32_t ncot, const double *cot_r, const double *cot_i, double *vjp, double *state_r, double *state_i) {
    return vjp_serial(h, "jq_final_state_vjp", false, nbatch, pcof, npar, nsamples, shift, 0, ncot, cot_r, cot_i, vjp, state_r, state_i);
}

extern "C" int jq_history_vjp(jq_handle *h, int32_t nbatch, const double *pcof, int32_t npar, int32_t nsamples, const double *shift,
                              int32_t save_every, int32_t ncot, const double *cot_r, const double *cot_i, double *vjp, double *hist_r,
                              double *hist_i) {
    return vjp_serial(h, "jq_history_vjp", true, nbatch, pcof, npar, nsamples, shift, save_every, ncot, cot_r, cot_i, vjp, hist_r, hist_i);
}

// The VJP entries on the time-parallel path: cotangents [traj][nsave][n*m] of the saved states (nsave = 1, save_every = nsteps: of U(T),
// whose stages jq_seg_vjp_launch runs unchanged); ncot = 0 returns U(T) (state) and / or the history alone.  `history`: the history
// entry's rejections and buffers, sized by nsave.
static int vjp_time_parallel(jq_handle *h, const char *who, bool history, int32_t nbatch, const double *pcof, int32_t npar, int32_t nsamples,
                             const double *shift, int32_t save_every, int32_t ncot, const double *cot_r, const double *cot_i, double *vjp,
                             double *state_r, double *state_i, double *hist_r, double *hist_i) {
    const int nc = std::max<int>(ncot, 1);
    int rc = check_batch_args(h, nbatch, pcof, npar, nsamples, shift, false, nc, who);
    if (rc) return rc;
    if (history && (rc = check_save_every(h, save_every)) != 0) return rc;
    if (ncot < 0) return fail(JQ_ERR_ARG, "%s: need ncot >= 0 (0: %s only)", who, history ? "the history" : "U(T)");
    if (ncot == 0 && !history && !state_r && !state_i) return fail(JQ_ERR_ARG, "%s: ncot = 0 returns U(T) only and needs state_r or state_i", who);
    if (ncot == 0 && history && !hist_r && !hist_i) return fail(JQ_ERR_ARG, "%s: ncot = 0 returns the history only and needs hist_r or hist_i", who);
    if (ncot > 0 && !cot_r && !cot_i) return fail(JQ_ERR_ARG, "%s: need at least one of cot_r, cot_i", who);
    if (ncot > 0 && !vjp) return fail(JQ_ERR_ARG, "%s: null vjp output", who);
    if (!h->route[TIME_PARALLEL].ok) return fail(JQ_ERR_ARG, "%s: %s", who, h->route[TIME_PARALLEL].why);
    // the pulled-back adjoint is the unforced second set of objFuncType 2/3: every launch sees objFuncType 2, whatever the problem's
    DevProblem P = h->P;
    P.objFuncType = 2;
    TrajPlan *fiber = h->route[FIBER].plan;
    if (ncot > 0 && !jq_seg_supported(fiber, P, true, history))
        return fail(JQ_ERR_ARG, "%s: no segment gradient sweep with the second adjoint set (fibre layout) for this problem", who);
    if (history && !jq_seg_supported(h->route[TIME_PARALLEL].plan, P, false, true))
        return fail(JQ_ERR_ARG, "%s: no segment sweep with the history paths for this problem's layout", who);
    CU(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    if ((rc = scratch_acquire(h, st)) != 0) return rc;       // the segment workspace is shared with the evaluation entries
    // trajectory (b, s, k) is kernel-7 trajectory b * nsamples * nc + s * nc + k: sample s * nc + k of candidate b, whose shift row is s
    const int ns2 = nsamples * nc;
    const long long nsave = history ? h->P.nsteps / save_every + 1 : 1;
    const size_t nt = (size_t)nbatch * nsamples, ntraj = nt * nc;
    const double len = (double)h->n * h->m, n_cot = ncot > 0 ? (double)ntraj * nsave * len : 0.0;
    const double n_vjp = ncot > 0 ? (double)ntraj * npar : 0.0, n_state = state_r || state_i ? nt * len : 0.0;
    const double n_hist = hist_r || hist_i ? nt * nsave * len : 0.0;
    const int nseg = seg_count(h, (int)ntraj, 1);
    const size_t need = jq_seg_workspace(P, (int)ntraj, splines(h, npar).nspl, nseg, true, ncot > 0, nsave > 1);
    if (need > h->cap_seg && (rc = grow_history(&h->d_seg, &h->cap_seg, (double)need, who)) != 0) return rc;
    if ((rc = seg_times_upload(h, nseg, st)) != 0) return rc;
    std::vector<double> shifts(shift ? (size_t)ns2 * h->n : 0);
    for (size_t r = 0; r < (shift ? (size_t)ns2 : 0); ++r) memcpy(&shifts[r * h->n], shift + (r / nc) * h->n, h->n * sizeof(double));
    double *d_pcof, *d_shift, *d_cr, *d_ci, *o_vjp, *o_sr, *o_si, *o_hr, *o_hi;
    const std::initializer_list<Out> out = {{&o_vjp, n_vjp, vjp}, {&o_sr, n_state, state_r}, {&o_si, n_state, state_i},
                                            {&o_hr, n_hist, hist_r}, {&o_hi, n_hist, hist_i}};
    // histories reach hundreds of MB: JQ_ERR_ALLOC with the size when they do not fit
    rc = stage(h, history ? who : nullptr, {{&d_pcof, (double)nbatch * npar, pcof}, {&d_shift, (double)shifts.size(), shift ? shifts.data() : nullptr},
                                            {&d_cr, n_cot, ncot > 0 ? cot_r : nullptr}, {&d_ci, n_cot, ncot > 0 ? cot_i : nullptr}}, out, st);
    if (rc) return rc;
    const LaunchArgs A = launch_args(h, nbatch, npar, ns2, d_pcof, d_shift);
    rc = record_launch(h, 7, st, [&](Ran &r) {
        r.nseg = nseg;
        return launched(jq_seg_vjp_launch(h->seg_prop, h->route[TIME_PARALLEL].plan, fiber, P, A, nseg, h->d_segt,
                                          reinterpret_cast<int *>(h->d_segt + 2 * (size_t)nseg), h->d_seg, st, ncot,
                                          history ? save_every : (int)h->P.nsteps, nsave, d_cr, d_ci, o_vjp, state_r ? o_sr : nullptr,
                                          state_i ? o_si : nullptr, o_hr, o_hi, &r.ctas, &r.regs, &r.smem, &r.tpc, &r.launches),
                        false, who);
    });
    if (rc || (rc = scratch_release(h, st)) != 0) return rc;
    return read_back(out, st);
}

extern "C" int jq_final_state_vjp_time_parallel(jq_handle *h, int32_t nbatch, const double *pcof, int32_t npar, int32_t nsamples,
                                                const double *shift, int32_t ncot, const double *cot_r, const double *cot_i, double *vjp,
                                                double *state_r, double *state_i) {
    return vjp_time_parallel(h, "jq_final_state_vjp_time_parallel", false, nbatch, pcof, npar, nsamples, shift, 0, ncot, cot_r, cot_i, vjp,
                             state_r, state_i, nullptr, nullptr);
}

extern "C" int jq_history_vjp_time_parallel(jq_handle *h, int32_t nbatch, const double *pcof, int32_t npar, int32_t nsamples,
                                            const double *shift, int32_t save_every, int32_t ncot, const double *cot_r, const double *cot_i,
                                            double *vjp, double *hist_r, double *hist_i) {
    return vjp_time_parallel(h, "jq_history_vjp_time_parallel", true, nbatch, pcof, npar, nsamples, shift, save_every, ncot, cot_r, cot_i,
                             vjp, nullptr, nullptr, hist_r, hist_i);
}
