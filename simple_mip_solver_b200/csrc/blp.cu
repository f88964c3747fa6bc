// libblp.so — host side of the batched node-LP bound step and its C ABI (include/blp.h).
//
// One handle = one GPU + one CUDA stream + the shared LP data (A, A', c, b, scaling, step size).
// blp_solve_batch runs restarted Halpern PDHG for a whole batch of node LPs:
//   set-up kernels -> [ period graph: K x (k_primal, k_dual) | evaluation graph: k_tick,
//   k_eval_cols, k_eval_rows, k_decide, k_apply_restart | harvest / refill of finished slots |
//   wide batches: k_freeze_cols/rows (frozen flags per 32-node block), k_fold_cols, k_work_* (the tiles'
//   work lists of the step kernels), k_pow_A/AT/finish (step of the block that still moves), k_freeze_count ]
//   repeated until every node has a status -> output kernels.  The host reads 13 ints per period
//   (nodes running / finished / restarting, frozen counts, watchdog resets).
#include "../../include/blp.h"

#include <cuda_runtime.h>
#include <dlfcn.h>

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <type_traits>
#include <vector>

#include "blp_kernels.cuh"
#include "blp_prep.hpp"
#include "blp_simplex.cuh"

using namespace blp;

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CK(call)                                                                           \
    do {                                                                                   \
        cudaError_t e_ = (call);                                                           \
        if (e_ != cudaSuccess)                                                             \
            return fail(BLP_ERR_CUDA, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__, \
                        cudaGetErrorString(e_));                                           \
    } while (0)

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

template <class T>
cudaError_t upload(DevBuf& b, const std::vector<T>& v, cudaStream_t s) {
    cudaError_t e = b.ensure(std::max<size_t>(v.size(), 1) * sizeof(T));
    if (e != cudaSuccess) return e;
    if (v.empty()) return cudaSuccess;
    return cudaMemcpyAsync(b.p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, s);
}

struct Plan {
    int NT, tiles, chunks, rows_per_cta;
    int V = 1;                // nodes per lane: 2 selects the k_primal2 / k_dual2 kernels
    int cap = 0;              // slab entries staged in shared memory per CTA (step kernels, spmv)
    size_t smem = 0;          // dynamic shared memory bytes of those kernels
    const int* chunk_ptr = nullptr;   // device: row range of every CTA (step kernels)
};

constexpr int kMaxSlabEntries = 2816;       // 44 KB of entries + row pointers stay under 48 KB

// Row ranges of the step-kernel CTAs: at most rows_per_cta rows and about 4x the average entry
// count per chunk; a long row (dense cut row) gets a chunk of its own and is then gathered by all
// warps of the CTA together. Also sizes the shared-memory slab (largest chunk, capped).
// Output: pairs (first row, end row), one per chunk, the chunks with the most entries first — CTAs
// are dispatched in blockIdx order, so the slow long-row chunks (appended cut rows sit at the END of
// the matrix) start at once instead of forming the tail of every launch.
void plan_chunks(Plan& p, const std::vector<int32_t>& ptr, int rows, std::vector<int32_t>& pairs) {
    std::vector<int32_t> bounds;
    const long nnz = ptr[rows];
    const long budget = std::max<long>(4 * ((nnz * p.rows_per_cta + rows - 1) / std::max(rows, 1)), kLongRow);
    bounds.clear();
    bounds.push_back(0);
    int worst = 0;
    int r = 0;
    while (r < rows) {
        int r1 = r;
        long cnt = 0;
        while (r1 < rows && r1 - r < p.rows_per_cta) {
            const long len = ptr[r1 + 1] - ptr[r1];
            if (len > kLongRow) {                 // long row: alone in its chunk
                if (r1 == r) { cnt = len; ++r1; }
                break;
            }
            if (r1 > r && cnt + len > budget) break;
            cnt += len;
            ++r1;
        }
        worst = std::max<long>(worst, cnt);
        bounds.push_back(r1);
        r = r1;
    }
    p.chunks = (int)bounds.size() - 1;
    std::vector<int32_t> order(p.chunks);
    for (int q = 0; q < p.chunks; ++q) order[q] = q;
    auto weight = [&](int q) { return ptr[bounds[q + 1]] - ptr[bounds[q]]; };
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) {      // long-row chunks first, the rest in row order
        const bool la = bounds[a + 1] - bounds[a] == 1 && weight(a) > kLongRow;
        const bool lb = bounds[b + 1] - bounds[b] == 1 && weight(b) > kLongRow;
        if (la != lb) return la;
        return la ? weight(a) > weight(b) : false;
    });
    pairs.resize(2 * (size_t)p.chunks);
    for (int q = 0; q < p.chunks; ++q) {
        pairs[2 * q] = bounds[order[q]];
        pairs[2 * q + 1] = bounds[order[q] + 1];
    }
    const int ptr_slots = (p.rows_per_cta + 4) / 4;
    p.cap = std::max(0, std::min(worst, kMaxSlabEntries - ptr_slots));
    p.smem = 16 * ((size_t)ptr_slots + (size_t)p.cap);
}

// spmv keeps uniform chunks
void plan_slab(Plan& p, const std::vector<int32_t>& ptr, int rows) {
    int worst = 0;
    for (int r0 = 0; r0 < rows; r0 += p.rows_per_cta) {
        const int r1 = std::min(rows, r0 + p.rows_per_cta);
        worst = std::max(worst, ptr[r1] - ptr[r0]);
    }
    const int ptr_slots = (p.rows_per_cta + 4) / 4;
    p.cap = std::max(0, std::min(worst, kMaxSlabEntries - ptr_slots));
    p.smem = 16 * ((size_t)ptr_slots + (size_t)p.cap);
}

// Tuning constants of the restart / primal-weight logic and of the launch plans. A production build
// compiles the defaults in; only a library built with -DBLP_TUNING (python -m simple_mip_solver_b200._build
// --tuning, used by the sweep tools under tools/) reads BLP_* environment variables, so that two values
// can be A/B-ed in one process.
#ifdef BLP_TUNING
int env_int(const char* name, int dflt) {
    const char* s = getenv(name);
    return (s && *s) ? atoi(s) : dflt;
}

double env_dbl(const char* name, double dflt) {
    const char* s = getenv(name);
    return (s && *s) ? atof(s) : dflt;
}
#else
constexpr int env_int(const char*, int dflt) { return dflt; }
constexpr double env_dbl(const char*, double dflt) { return dflt; }
#endif

int pick_nt(int B) {
    int nt = 1;
    while (nt < 32 && nt < B) nt <<= 1;
    return nt;
}

// Calls f(std::integral_constant<int, NT>{}) for a nodes-per-warp width nt from pick_nt: the kernels that keep one
// node per lane are instantiated for these six widths.
template <class F>
void with_nt(int nt, F&& f) {
    switch (nt) {
        case 1: f(std::integral_constant<int, 1>{}); break;
        case 2: f(std::integral_constant<int, 2>{}); break;
        case 4: f(std::integral_constant<int, 4>{}); break;
        case 8: f(std::integral_constant<int, 8>{}); break;
        case 16: f(std::integral_constant<int, 16>{}); break;
        default: f(std::integral_constant<int, 32>{}); break;
    }
}

// Step kernels: many small CTAs in tile-major order, so the CTAs resident at one moment work on
// one or two node tiles and the gathered vector of those tiles stays in L2 (blp_kernels.cuh).
// width: nodes of the batch, nt: nodes per warp.
Plan plan_rows(int rows, int width, int nt, int rows_per_warp, int max_chunks) {
    Plan p;
    p.NT = nt;
    p.tiles = (width + nt - 1) / nt;
    const int pass = kWarps * (32 / p.NT);
    int rpc = pass * std::max(rows_per_warp, 1);
    if (max_chunks > 0) {
        const int need = (rows + max_chunks - 1) / max_chunks;
        rpc = std::max(rpc, ((need + pass - 1) / pass) * pass);
    } else {
        while (rpc > 512 && rpc > pass) rpc -= pass;      // step kernels: slab pointers stay small
    }
    p.rows_per_cta = rpc;
    p.chunks = std::max(1, (rows + rpc - 1) / rpc);
    return p;
}

constexpr int kEvalChunks = 48;

struct GraphKey {
    DevProb P;
    DevState S;
    DecideArgs D;
    int K, rpw;
};

}  // namespace

struct blp_handle_s {
    int device = 0;
    int num_sms = 0, coop_ok = 0;      // SM count; cooperative launch supported
    cudaStream_t stream = nullptr;
    int m_base = 0, n = 0;
    HostCsr A0;                        // unscaled rows (base + appended cuts)
    std::vector<int32_t> hptrA, hptrAT; // host copies of the row pointers of A and A' (slab sizing)
    std::vector<double> c0, b0;
    std::vector<double> dr, dc;
    // device copies
    DevBuf rowptr, ent, cptr, cent, c, b, rowscale, colscale, d_dr, d_dc;
    DevBuf uent, ucent;                // unscaled entries, same patterns (blp_spmv)
    DevBuf uc, ub;                     // unscaled objective / row lower bounds (simplex path)
    // dual simplex path (blp_simplex_*): factor stores of the current and the previous call, staging
    DevBuf sx_binv[2], sx_head[2], sx_stat[2], sx_wts[2], sx_work, sx_in, sx_out, sx_wide;
    DevBuf sx_bnd[2];                  // each store's node bounds [B][n] x 2 and row masks [B][m - m_base]
    int sx_bnd_mask[2] = {0, 0};       // ... whether that call had row masks (else every pool row was on)
    DevBuf sx_gmi;                     // blp_simplex_gmi_cuts_host: requests and results
    int sx_cur = 0;                    // store the NEXT call writes; the other one holds the last call
    int sx_last_B = 0, sx_last_m = -1; // nodes / rows of the last call's store (-1: none)
    DevBuf chunkC, chunkR;             // row ranges of the step-kernel CTAs (primal / dual)
    std::vector<int32_t> h_chunkC, h_chunkR;
    DevProb P{};
    // staging of the host-buffer entry points
    DevBuf s_lb, s_ub, s_x0, s_y0, s_mask, s_x, s_y, s_tmp, s_ws, s_node, s_int, s_delta, s_par;
    int32_t* h_counters = nullptr;     // pinned, 16 entries
    double frz_c = 0.0, frz_r = 0.0;   // units of the freezing margins: rms of the scaled objective / right-hand side
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    // node tiles are independent chains of launches: inside a period graph they run as up to
    // kLanes parallel branches, so the tail of one branch's kernel overlaps the next kernel of another
    static constexpr int kLanes = 4;
    cudaStream_t side[kLanes - 1] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev_fork = nullptr, ev_join[kLanes - 1] = {nullptr, nullptr, nullptr};
    std::vector<cudaEvent_t> prof_ev;
    // multi-GPU exchange (blp_comm_init): NCCL communicator of this rank and a 16-byte device buffer
    void* comm = nullptr;
    int comm_ranks = 1;
    double* d_pair = nullptr;
    // cached period graphs
    bool graph_valid = false;
    GraphKey gkey{};
    cudaGraphExec_t g_steps = nullptr, g_eval = nullptr;

    void drop_graphs() {
        if (g_steps) cudaGraphExecDestroy(g_steps);
        if (g_eval) cudaGraphExecDestroy(g_eval);
        g_steps = g_eval = nullptr;
        graph_valid = false;
    }
};

namespace {

// ---- NCCL, bound at run time -----------------------------------------------------------------
// The only collective of the path is the 16-byte all-reduce(min) of [incumbent, dual bound]
// (SURVEY section 8e). libnccl is opened with dlopen so that libblp.so has no link-time
// dependency on it: a process that has torch loaded gets torch's copy, any other host the system one.
struct NcclId { char internal[128]; };
struct NcclApi {
    void* lib = nullptr;
    int (*GetUniqueId)(NcclId*) = nullptr;
    int (*CommInitRank)(void**, int, NcclId, int) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};
constexpr int kNcclFloat64 = 8, kNcclMin = 3;      // ncclDataType_t / ncclRedOp_t values (nccl.h)

NcclApi* nccl_api() {
    static NcclApi api;
    static bool tried = false;
    if (tried) return api.lib ? &api : nullptr;
    tried = true;
    const char* names[] = {getenv("BLP_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) {
        if (!nm || !*nm) continue;
        api.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
        if (api.lib) break;
    }
    if (!api.lib) return nullptr;
    api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(dlsym(api.lib, "ncclGetUniqueId"));
    api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(dlsym(api.lib, "ncclCommInitRank"));
    api.AllReduce = reinterpret_cast<decltype(api.AllReduce)>(dlsym(api.lib, "ncclAllReduce"));
    api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(dlsym(api.lib, "ncclCommDestroy"));
    api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(dlsym(api.lib, "ncclGetErrorString"));
    if (!api.GetUniqueId || !api.CommInitRank || !api.AllReduce || !api.CommDestroy) {
        dlclose(api.lib);
        api.lib = nullptr;
        return nullptr;
    }
    return &api;
}

int nccl_fail(const NcclApi* a, const char* what, int rc) {
    return fail(BLP_ERR_CUDA, "%s: NCCL error %d (%s)", what, rc,
                (a && a->GetErrorString) ? a->GetErrorString(rc) : "?");
}

// (re)build scaling, transpose, step size and the device copies of the shared LP data
int prepare(blp_handle h) {
    const int m = h->A0.rows, n = h->n, mb = h->m_base;
    HostCsr As = h->A0;
    // Diagonal scaling over ALL rows currently in the matrix (base + appended cut rows). It only
    // conditions the iteration: residuals, tolerances and certificates are evaluated in the unscaled
    // problem, and the tolerance scale ||b|| is taken per node over the rows of ITS LP (k_decide), so what
    // a node is held to does not depend on cuts only other nodes carry. (Equilibrating appended rows
    // against a column scaling frozen at the base problem was measured: config 4's cut rounds needed
    // 14-33 % more iterations, profiles/r2g_configs_3_4.json — dense cut rows want their say in dc.)
    h->dr.assign(m, 1.0);
    h->dc.assign(n, 1.0);
    ruiz_pc(As, h->dr, h->dc, 10, 0);
    std::vector<double> bs(m), cs(n), rowscale(m), colscale(n);
    for (int i = 0; i < m; ++i) bs[i] = h->b0[i] * h->dr[i];
    for (int j = 0; j < n; ++j) cs[j] = h->c0[j] * h->dc[j];
    const std::vector<double> b0_base(h->b0.begin(), h->b0.begin() + mb);
    const double sb = 1.0 / (norm2(bs) + 1.0), sc = 1.0 / (norm2(cs) + 1.0);
    double cinf = 0.0;
    for (int i = 0; i < m; ++i) bs[i] *= sb;
    for (int j = 0; j < n; ++j) {
        cs[j] *= sc;
        cinf = std::max(cinf, std::fabs(cs[j]));
    }
    for (int i = 0; i < m; ++i) rowscale[i] = 1.0 / (h->dr[i] * sb);
    for (int j = 0; j < n; ++j) colscale[j] = 1.0 / (h->dc[j] * sc);
    HostCsr At = transpose(As);
    HostCsr A0t = transpose(h->A0);
    const double eta = 0.998 / sigma_max(As, At);
    h->hptrA = As.ptr;
    h->hptrAT = At.ptr;
    const double nb = norm2(bs), nc = norm2(cs);
    h->frz_c = nc / std::sqrt((double)std::max(n, 1));
    h->frz_r = nb / std::sqrt((double)std::max(m, 1));

    cudaStream_t s = h->stream;
    auto pack = [](const HostCsr& a) {
        std::vector<Ent> e(a.idx.size());
        for (size_t p = 0; p < e.size(); ++p) e[p] = Ent{a.idx[p], 0, a.val[p]};
        return e;
    };
    const std::vector<Ent> eA = pack(As), eAt = pack(At), eA0 = pack(h->A0), eA0t = pack(A0t);
    CK(upload(h->rowptr, As.ptr, s));
    CK(upload(h->ent, eA, s));
    CK(upload(h->cptr, At.ptr, s));
    CK(upload(h->cent, eAt, s));
    CK(upload(h->uent, eA0, s));
    CK(upload(h->ucent, eA0t, s));
    CK(upload(h->uc, h->c0, s));
    CK(upload(h->ub, h->b0, s));
    h->sx_last_m = -1;                 // the rows changed: stored factors are void
    CK(upload(h->c, cs, s));
    CK(upload(h->b, bs, s));
    CK(upload(h->rowscale, rowscale, s));
    CK(upload(h->colscale, colscale, s));
    CK(upload(h->d_dr, h->dr, s));
    CK(upload(h->d_dc, h->dc, s));
    CK(cudaStreamSynchronize(s));      // host vectors go out of scope

    DevProb& P = h->P;
    P.m = m;
    P.m_base = h->m_base;
    P.n = n;
    P.nnz = (int)As.ptr.back();
    P.rowptr = h->rowptr.as<int32_t>();
    P.ent = h->ent.as<Ent>();
    P.cptr = h->cptr.as<int32_t>();
    P.cent = h->cent.as<Ent>();
    P.c = h->c.as<double>();
    P.b = h->b.as<double>();
    P.rowscale = h->rowscale.as<double>();
    P.colscale = h->colscale.as<double>();
    P.dr = h->d_dr.as<double>();
    P.dc = h->d_dc.as<double>();
    P.eta = eta;
    P.sb = sb;
    P.sc = sc;
    P.objscale = 1.0 / (sb * sc);
    P.bnorm0 = norm2(b0_base);
    P.bcut2 = 0.0;
    for (int i = mb; i < m; ++i) P.bcut2 += h->b0[i] * h->b0[i];
    P.cnorm0 = norm2(h->c0);
    P.cinf_s = cinf;
    P.omega0 = ((nb > 1e-12 && nc > 1e-12) ? nc / nb : 1.0) * env_dbl("BLP_OMEGA0_SCALE", 1.0);
    h->drop_graphs();
    return BLP_OK;
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct Carve {
    char* base;
    size_t off = 0;
    template <class T> T* take(size_t count) {
        off = align_up(off, 256);
        T* p = reinterpret_cast<T*>(base + off);
        off += count * sizeof(T);
        return p;
    }
};

size_t carve_state(const blp_handle h, int B, void* ws, DevState* S) {
    const int ld = blp_ld(B);
    const size_t n = h->n, m = h->A0.rows;
    Carve cv{reinterpret_cast<char*>(ws)};
    DevState s{};
    s.B = B;
    s.ld = ld;
    s.xbar = cv.take<double>(n * ld);
    s.xa = cv.take<anc_t>(n * ld);
    s.l = cv.take<double>(n * ld);
    s.u = cv.take<double>(n * ld);
    s.X1 = cv.take<double>(n * ld);
    s.DX = cv.take<double>(n * ld);
    s.G = cv.take<double>(n * ld);
    s.y = cv.take<double>(m * ld);
    s.ya = cv.take<anc_t>(m * ld);
    s.Y1 = cv.take<double>(m * ld);
    s.DY = cv.take<double>(m * ld);
    s.omega = cv.take<double>(ld);
    s.fpe0 = cv.take<double>(ld);
    s.fpe_prev = cv.take<double>(ld);
    s.pobj = cv.take<double>(ld);
    s.dobj = cv.take<double>(ld);
    s.sbase = cv.take<int32_t>(ld);
    s.fin = cv.take<int32_t>(ld);
    s.status = cv.take<int32_t>(ld);
    s.iters = cv.take<int32_t>(ld);
    s.restart = cv.take<int32_t>(ld);
    s.origin = cv.take<int32_t>(ld);
    s.newpos = cv.take<int32_t>(ld);
    s.start = cv.take<int32_t>(ld);
    s.fresh = cv.take<int32_t>(ld);
    s.newlist = cv.take<int32_t>(ld);
    s.partC = cv.take<double>((size_t)kEvalChunks * C_N * ld);
    s.partR = cv.take<double>((size_t)kEvalChunks * R_N * ld);
    s.fracD = cv.take<double>((size_t)kEvalChunks * ld);
    s.fracI = cv.take<int32_t>((size_t)kEvalChunks * ld);
    s.isint = cv.take<uint8_t>(n);
    s.rowmask = cv.take<uint8_t>((m - h->m_base) * (size_t)ld + 1);
    s.dbg = cv.take<double>((size_t)ld * 8);
    s.lref = cv.take<double>(n * (size_t)(ld / 32));
    s.uref = cv.take<double>(n * (size_t)(ld / 32));
    s.lumask = cv.take<uint32_t>(n * (size_t)(ld / 32));
    s.counters = cv.take<int32_t>(16);
    s.cfrz = cv.take<uint8_t>(n * (size_t)(ld / 32));
    s.rfrz = cv.take<uint8_t>(m * (size_t)(ld / 32));
    {   // folded matrices of every 64-node tile (k_fold_cols, k_work_*): 32 bytes per stored entry and tile
        const size_t tiles = ld / kBlk, nnz = h->A0.ptr.empty() ? 0 : (size_t)h->A0.ptr.back();
        s.cval = cv.take<double>(n * (size_t)(ld / 32));
        s.fcol = cv.take<uint8_t>(n * tiles);
        s.fval = cv.take<double>(n * tiles);
        auto work_list = [&](const size_t rows, const int rec_bytes) {
            WorkList w;
            w.row = cv.take<int2>((rows + 1) * tiles);
            w.ent = cv.take<Ent>(nnz * tiles);
            w.rec = cv.take<int4>(rows * tiles * (rec_bytes / 16));
            w.chunk = cv.take<int4>(rows * tiles);
            w.kept = cv.take<int32_t>(rows * tiles);
            w.count = cv.take<int32_t>(tiles);
            return w;
        };
        s.wlC = work_list(n, kPrimalRowBytes);
        s.wlR = work_list(m, kDualRowBytes);
        s.ftc = cv.take<uint8_t>(n * tiles);
        s.ftr = cv.take<uint8_t>(m * tiles);
        s.pv = cv.take<double>(n * tiles);
        s.pw = cv.take<double>(m * tiles);
        s.ppart = cv.take<double>((size_t)kPowChunks * tiles);
        s.eta_tile = cv.take<double>(tiles);
    }
    s.eta = cv.take<double>(ld);
    s.eta_lock = cv.take<int32_t>(ld);
    if (S) *S = s;
    return align_up(cv.off, 256);
}

// which: 0 primal only, 1 dual only, 2 both. The two-nodes-per-lane kernels can be launched for a
// sub-range of node tiles [tile0, tile0 + ntiles) (ntiles < 0: all), see ensure_graphs.
void launch_steps(const DevProb& P, const DevState& S, const Plan& pc, const Plan& pr, int it,
                  bool major, cudaStream_t st, int which = 2, int tile0 = 0, int ntiles = -1) {
    if (pc.V == 2) {
        const int nt = ntiles < 0 ? pc.tiles : ntiles;
        const dim3 gc(pc.chunks, nt), gr(pr.chunks, nt);
        if (which != 1) {
            if (major) k_primal2<true><<<gc, kCtaThreads, pc.smem, st>>>(P, S, it, pc.rows_per_cta, pc.cap, pc.chunk_ptr, tile0);
            else k_primal2<false><<<gc, kCtaThreads, pc.smem, st>>>(P, S, it, pc.rows_per_cta, pc.cap, pc.chunk_ptr, tile0);
        }
        if (which != 0) {
            if (major) k_dual2<true><<<gr, kCtaThreads, pr.smem, st>>>(P, S, it, pr.rows_per_cta, pr.cap, pr.chunk_ptr, tile0);
            else k_dual2<false><<<gr, kCtaThreads, pr.smem, st>>>(P, S, it, pr.rows_per_cta, pr.cap, pr.chunk_ptr, tile0);
        }
        return;
    }
    with_nt(pc.NT, [&](auto nt) {
        const dim3 gc(pc.chunks, pc.tiles), gr(pr.chunks, pr.tiles);
        if (which != 1) {
            if (major) k_primal<nt, true><<<gc, kCtaThreads, pc.smem, st>>>(P, S, it, pc.rows_per_cta, pc.cap, pc.chunk_ptr);
            else k_primal<nt, false><<<gc, kCtaThreads, pc.smem, st>>>(P, S, it, pc.rows_per_cta, pc.cap, pc.chunk_ptr);
        }
        if (which != 0) {
            if (major) k_dual<nt, true><<<gr, kCtaThreads, pr.smem, st>>>(P, S, it, pr.rows_per_cta, pr.cap, pr.chunk_ptr);
            else k_dual<nt, false><<<gr, kCtaThreads, pr.smem, st>>>(P, S, it, pr.rows_per_cta, pr.cap, pr.chunk_ptr);
        }
    });
}

// Recompute the frozen-coordinate flags of every 32-node block (mode: see k_freeze_cols) and their count.
struct StepArgs {
    double safety, cap;      // step of a tile = min(cap / ||A||, safety / ||A_UU||); safety 0 = keep 0.998 / ||A||
    int passes_first, passes;
};
// pc / pr: the step plans, whose chunks the work lists are split over.
int launch_freeze(const DevProb& P, const DevState& S, const FreezeArgs& F, const StepArgs& T, const Plan& pc,
                  const Plan& pr, int mode, cudaStream_t st) {
    const int halves = (S.B + 31) / 32;
    auto rows_per_cta = [&](int rows) {
        const int want_chunks = std::max(1, 148 * 8 / halves);
        const int r = (rows + want_chunks - 1) / want_chunks;
        return std::max(kWarps, (r + kWarps - 1) / kWarps * kWarps);
    };
    const int rc = rows_per_cta(P.n), rr = rows_per_cta(P.m);
    k_freeze_cols<<<dim3((P.n + rc - 1) / rc, halves), kCtaThreads, 0, st>>>(P, S, F, rc, mode);
    k_freeze_rows<<<dim3((P.m + rr - 1) / rr, halves), kCtaThreads, 0, st>>>(P, S, F, rr, mode);
    const int tiles = (S.B + kBlk - 1) / kBlk;
    auto per_tile = [&](int rows) { return dim3(std::max(1, std::min((rows + kCtaThreads - 1) / kCtaThreads, 148 * 4 / tiles + 1)), tiles); };
    k_fold_cols<<<per_tile(P.n), kCtaThreads, 0, st>>>(P, S);
    k_work_count<true><<<per_tile(P.n), kCtaThreads, 0, st>>>(P, S);
    k_work_count<false><<<per_tile(P.m), kCtaThreads, 0, st>>>(P, S);
    k_work_scan<true><<<tiles, 1024, 0, st>>>(P, S, pc.chunks, pc.rows_per_cta);
    k_work_scan<false><<<tiles, 1024, 0, st>>>(P, S, pr.chunks, pr.rows_per_cta);
    k_work_fill<true><<<per_tile(P.n), kCtaThreads, 0, st>>>(P, S);
    k_work_fill<false><<<per_tile(P.m), kCtaThreads, 0, st>>>(P, S);
    int launched = 10;
    if (T.safety > 0.0) {
        const dim3 gp(std::min(kPowChunks, std::max(1, (std::max(P.n, P.m) + 4 * kCtaThreads - 1) / (4 * kCtaThreads))), tiles);
        if (mode == 2) k_pow_init<<<gp, kCtaThreads, 0, st>>>(P, S);
        const int passes = mode == 2 ? T.passes_first : T.passes;
        for (int q = 0; q < passes; ++q) {
            k_pow_A<<<gp, kCtaThreads, 0, st>>>(P, S);
            k_pow_AT<<<gp, kCtaThreads, 0, st>>>(P, S);
        }
        k_pow_finish<<<tiles, kBlk, 0, st>>>(P, S, T.safety, T.cap, mode);
        launched += 2 * passes + 1 + (mode == 2 ? 1 : 0);
    }
    k_freeze_count<<<tiles, kCtaThreads, 0, st>>>(P, S);
    return launched;
}

void launch_eval(const DevProb& P, const DevState& S, const Plan& ec, const Plan& er,
                 const DecideArgs& D, int K, cudaStream_t st) {
    k_tick<<<1, 1, 0, st>>>(S, K);
    with_nt(ec.NT, [&](auto nt) {
        k_eval_cols<nt><<<dim3(ec.chunks, ec.tiles), kCtaThreads, 0, st>>>(P, S, ec.rows_per_cta);
        k_eval_rows<nt><<<dim3(er.chunks, er.tiles), kCtaThreads, 0, st>>>(P, S, er.rows_per_cta);
    });
    k_decide<<<(S.B + 127) / 128, 128, 0, st>>>(P, S, D);
    const int rchunks = std::min(64, std::max(1, (std::max(P.n, P.m) + 63) / 64));
    k_apply_restart<<<dim3(rchunks, (S.ld + 31) / 32), kCtaThreads, 0, st>>>(P, S);
}

void launch_check_rows(const DevProb& P, const DevState& S, const Plan& er, int only_fresh,
                       cudaStream_t st) {
    with_nt(er.NT, [&](auto nt) {
        k_check_rows<nt><<<dim3(er.chunks, er.tiles), kCtaThreads, 0, st>>>(P, S, er.rows_per_cta, only_fresh);
    });
}

void launch_harvest(const DevProb& P, const DevState& S, const DevOut& O, const Plan& ec,
                    const Plan& er, bool want_frac, cudaStream_t st, int* launches) {
    const double eps = 1e-4;      // variable_epsilon of the reference (utils/tolerance.py:2)
    if (O.x || want_frac) {
        with_nt(ec.NT, [&](auto nt) {
            k_harvest_x<nt><<<dim3(ec.chunks, ec.tiles), kCtaThreads, 0, st>>>(P, S, O, eps, ec.rows_per_cta);
        });
        ++*launches;
    }
    if (O.y) {
        with_nt(er.NT, [&](auto nt) {
            k_harvest_y<nt><<<dim3(er.chunks, er.tiles), kCtaThreads, 0, st>>>(P, S, O, er.rows_per_cta);
        });
        ++*launches;
    }
    k_harvest_nodes<<<(S.B + 127) / 128, 128, 0, st>>>(P, S, O, ec.chunks, eps, want_frac ? 1 : 0);
    ++*launches;
}

// One evaluation period of a narrow batch (one-node-per-lane kernels) as ONE cooperative launch.
// Returns cudaErrorNotSupported when the grid cannot be made co-resident.
cudaError_t launch_period_coop(blp_handle h, const DevProb& P, const DevState& S, const Plan& pc,
                               const Plan& pr, int K, cudaStream_t st) {
    const void* fn = nullptr;
    with_nt(pc.NT, [&](auto nt) { fn = (const void*)k_period_coop<nt>; });
    const size_t smem = pc.smem + pr.smem;        // both slabs stay resident for the whole period
    if (smem > 200 * 1024) return cudaErrorNotSupported;
    if (smem > 48 * 1024) {
        cudaError_t ea = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (ea != cudaSuccess) return ea;
    }
    int occ = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, kCtaThreads, smem);
    if (e != cudaSuccess) return e;
    if (occ < 1) return cudaErrorNotSupported;
    const int items = std::max(pc.chunks, pr.chunks) * pc.tiles;
    // worth it only for small LPs, where every CTA gets at most one work item per phase; with
    // more rows than that (the tail of a large batch) two graph launches are as fast (measured)
    if (items > occ * h->num_sms) return cudaErrorNotSupported;
    const int grid = std::max(1, items);
    CoopPlan C{pc.rows_per_cta, pc.cap, pc.chunks, pr.rows_per_cta, pr.cap, pr.chunks, pc.tiles,
               pc.chunk_ptr, pr.chunk_ptr};
    DevProb Pc = P;
    DevState Sc = S;
    int Kc = K;
    void* args[] = {&Pc, &Sc, &Kc, &C};
    return cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(kCtaThreads), args, smem, st);
}

int elementwise_grid(size_t total) {
    size_t g = (total + kCtaThreads - 1) / kCtaThreads;
    return (int)std::min<size_t>(std::max<size_t>(g, 1), 148 * 16);
}

int check_opts(const blp_opts* in, blp_opts* o) {
    blp_default_opts(o);
    if (in) *o = *in;
    if (!(o->eps_rel > 0.0) || !(o->eps_infeas > 0.0) || o->max_iters < 1 || o->eval_every < 1 ||
        o->max_active < 0 || std::isnan(o->obj_cutoff) || !(o->freeze_margin >= 0.0) || !(o->step_safety >= 0.0) ||
        o->step_safety > 1.0)
        return fail(BLP_ERR_ARG, "blp_opts: eps_rel/eps_infeas must be > 0, max_iters/eval_every >= 1, "
                                 "max_active >= 0, freeze_margin >= 0, 0 <= step_safety <= 1");
    return BLP_OK;
}

}  // namespace

// ================================================================================================
extern "C" {

void blp_default_opts(blp_opts* o) {
    if (!o) return;
    o->eps_rel = 1e-7;
    o->eps_infeas = 1e-9;
    o->max_iters = 2000000;
    o->eval_every = 64;
    o->use_graph = 1;
    o->compact = 1;
    o->verbose = 0;
    o->profile = 0;
    o->max_active = 0;
    o->obj_cutoff = INFINITY;
    o->freeze = 1;
    o->freeze_margin = 0.05;
    o->step_safety = 0.98;
}

int blp_slots(int B, const blp_opts* o) {
    return (o && o->max_active > 0 && o->max_active < B) ? o->max_active : B;
}

int blp_ld(int B) { return B <= 0 ? 0 : (B + kBlk - 1) / kBlk * kBlk; }

const char* blp_last_error(void) { return g_err.c_str(); }

const char* blp_version(void) {
#ifdef BLP_TUNING
    return "blp 0.2 sm_100a (tuning build: BLP_* environment variables are read)";
#else
    return "blp 0.2 sm_100a";
#endif
}

int blp_create(int device, int m, int n, int64_t nnz, const int32_t* rowptr, const int32_t* colidx,
               const double* val, const double* c, const double* row_lb, blp_handle* out) {
    if (!out) return fail(BLP_ERR_ARG, "blp_create: out is NULL");
    *out = nullptr;
    if (m < 1 || n < 1 || nnz < 0 || !rowptr || !c || !row_lb || (nnz > 0 && (!colidx || !val)))
        return fail(BLP_ERR_ARG, "blp_create: need m >= 1, n >= 1, nnz >= 0 and non-NULL arrays");
    if (rowptr[0] != 0 || rowptr[m] != nnz)
        return fail(BLP_ERR_ARG, "blp_create: rowptr[0] must be 0 and rowptr[m] must equal nnz");
    for (int i = 0; i < m; ++i) {
        if (rowptr[i + 1] < rowptr[i]) return fail(BLP_ERR_ARG, "blp_create: rowptr not monotone at row %d", i);
        if (!(std::fabs(row_lb[i]) < 1e30))
            return fail(BLP_ERR_ARG, "blp_create: row_lb[%d] is not finite (rows are 'a.x >= b')", i);
    }
    for (int64_t p = 0; p < nnz; ++p)
        if (colidx[p] < 0 || colidx[p] >= n || !std::isfinite(val[p]))
            return fail(BLP_ERR_ARG, "blp_create: entry %lld has column %d / non-finite value", (long long)p, colidx[p]);
    for (int j = 0; j < n; ++j)
        if (!std::isfinite(c[j])) return fail(BLP_ERR_ARG, "blp_create: c[%d] is not finite", j);
    int ndev = 0;
    CK(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev)
        return fail(BLP_ERR_ARG, "blp_create: device %d out of range (%d visible)", device, ndev);
    CK(cudaSetDevice(device));
    blp_handle h = new (std::nothrow) blp_handle_s;
    if (!h) return fail(BLP_ERR_NOMEM, "blp_create: out of host memory");
    h->device = device;
    h->m_base = m;
    h->n = n;
    h->A0.rows = m;
    h->A0.cols = n;
    h->A0.ptr.assign(rowptr, rowptr + m + 1);
    h->A0.idx.assign(colidx, colidx + nnz);
    h->A0.val.assign(val, val + nnz);
    h->c0.assign(c, c + n);
    h->b0.assign(row_lb, row_lb + m);
    cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, device);
    cudaDeviceGetAttribute(&h->coop_ok, cudaDevAttrCooperativeLaunch, device);
    cudaError_t e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
    // the wide step kernels carry ~8 KB of static shared memory next to a slab of up to 44 KB and the scalars of up
    // to kMaxChunkRows rows (24 KB): opt in above 48 KB
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_primal2<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 72 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_primal2<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 72 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_dual2<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 72 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_dual2<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 72 * 1024);
    if (e == cudaSuccess) e = cudaMallocHost(&h->h_counters, 16 * sizeof(int32_t));
    for (int q = 0; q < 4 && e == cudaSuccess; ++q) e = cudaEventCreate(&h->ev[q]);
    for (int q = 0; q < blp_handle_s::kLanes - 1 && e == cudaSuccess; ++q) {
        e = cudaStreamCreateWithFlags(&h->side[q], cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_join[q], cudaEventDisableTiming);
    }
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming);
    if (e != cudaSuccess) {
        blp_destroy(h);
        return fail(BLP_ERR_CUDA, "blp_create: %s", cudaGetErrorString(e));
    }
    int rc = prepare(h);
    if (rc != BLP_OK) {
        blp_destroy(h);
        return rc;
    }
    *out = h;
    return BLP_OK;
}

int blp_append_rows(blp_handle h, int k, const int32_t* rowptr, const int32_t* colidx,
                    const double* val, const double* rhs, int* first_row_id) {
    if (!h) return fail(BLP_ERR_ARG, "blp_append_rows: NULL handle");
    if (k < 1 || !rowptr || !rhs) return fail(BLP_ERR_ARG, "blp_append_rows: need k >= 1 rows");
    if (rowptr[0] != 0) return fail(BLP_ERR_ARG, "blp_append_rows: rowptr[0] must be 0");
    const int64_t nnz = rowptr[k];
    for (int i = 0; i < k; ++i) {
        if (rowptr[i + 1] < rowptr[i]) return fail(BLP_ERR_ARG, "blp_append_rows: rowptr not monotone");
        if (!(std::fabs(rhs[i]) < 1e30)) return fail(BLP_ERR_ARG, "blp_append_rows: rhs[%d] not finite", i);
    }
    for (int64_t p = 0; p < nnz; ++p)
        if (colidx[p] < 0 || colidx[p] >= h->n || !std::isfinite(val[p]))
            return fail(BLP_ERR_ARG, "blp_append_rows: bad entry %lld", (long long)p);
    CK(cudaSetDevice(h->device));
    const int first = h->A0.rows;
    const int32_t base = h->A0.ptr.back();
    for (int i = 0; i < k; ++i) h->A0.ptr.push_back(base + rowptr[i + 1]);
    h->A0.idx.insert(h->A0.idx.end(), colidx, colidx + nnz);
    h->A0.val.insert(h->A0.val.end(), val, val + nnz);
    h->b0.insert(h->b0.end(), rhs, rhs + k);
    h->A0.rows += k;
    if (first_row_id) *first_row_id = first;
    return prepare(h);
}

int blp_truncate_rows(blp_handle h, int m_keep) {
    if (!h) return fail(BLP_ERR_ARG, "blp_truncate_rows: NULL handle");
    if (m_keep < h->m_base || m_keep > h->A0.rows)
        return fail(BLP_ERR_ARG, "blp_truncate_rows: m_keep %d outside [%d, %d]", m_keep, h->m_base, h->A0.rows);
    if (m_keep == h->A0.rows) return BLP_OK;
    CK(cudaSetDevice(h->device));
    h->A0.rows = m_keep;
    h->A0.ptr.resize(m_keep + 1);
    h->A0.idx.resize(h->A0.ptr.back());
    h->A0.val.resize(h->A0.ptr.back());
    h->b0.resize(m_keep);
    return prepare(h);
}

int blp_num_rows(blp_handle h) { return h ? h->A0.rows : 0; }
int blp_num_base_rows(blp_handle h) { return h ? h->m_base : 0; }
int blp_num_cols(blp_handle h) { return h ? h->n : 0; }
void* blp_stream(blp_handle h) { return h ? (void*)h->stream : nullptr; }

size_t blp_workspace_bytes(blp_handle h, int B) {
    if (!h || B < 1) return 0;
    return carve_state(h, B, nullptr, nullptr) + 256;
}

int blp_solve_batch(blp_handle h, int B, const double* lb, const double* ub,
                    const uint8_t* row_mask, const double* x0, const double* y0,
                    const int32_t* int_idx, int n_int, const blp_opts* opts_in,
                    void* workspace, size_t workspace_bytes,
                    double* obj, double* lower_bound, int32_t* status, int32_t* iters,
                    double* x, double* y, int32_t* frac_idx, blp_stats* stats) {
    if (!h) return fail(BLP_ERR_ARG, "blp_solve_batch: NULL handle");
    if (B < 1 || !lb || !ub) return fail(BLP_ERR_ARG, "blp_solve_batch: need B >= 1 and lb/ub");
    if (frac_idx && int_idx == nullptr && n_int > 0)
        return fail(BLP_ERR_ARG, "blp_solve_batch: n_int > 0 with int_idx NULL");
    blp_opts o;
    int rc = check_opts(opts_in, &o);
    if (rc != BLP_OK) return rc;
    // W node slots are resident at once; with W < B (blp_opts.max_active) the other nodes wait
    // in the caller's arrays and take over the slots of finished ones (continuous batching)
    const int W = blp_slots(B, &o);
    const bool refill_mode = W < B;
    const int ld_in = blp_ld(B);
    if (!workspace || workspace_bytes < blp_workspace_bytes(h, W))
        return fail(BLP_ERR_NOMEM, "blp_solve_batch: workspace of %zu bytes, need %zu", workspace_bytes,
                    blp_workspace_bytes(h, W));
    CK(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const DevProb& P = h->P;

    void* ws = reinterpret_cast<void*>(align_up(reinterpret_cast<size_t>(workspace), 256));
    DevState S;
    carve_state(h, W, ws, &S);
    const bool have_mask = (P.m > P.m_base) && row_mask != nullptr;
    uint8_t* mask_ws = S.rowmask;
    if (!have_mask) S.rowmask = nullptr;
    // frozen coordinates (k_freeze_cols): margins in units of the scaled problem's rms cost / right-hand side
    const bool freeze = o.freeze != 0 && o.freeze_margin > 0.0 && env_int("BLP_FREEZE", 1) != 0;
    const double fm = env_dbl("BLP_FREEZE_MARGIN", o.freeze_margin), fl = env_dbl("BLP_FREEZE_RELEASE", 1.0 / 3.0);
    const FreezeArgs F{h->frz_c > 0.0 ? fl * fm * h->frz_c : INFINITY, h->frz_c > 0.0 ? fm * h->frz_c : INFINITY,
                       h->frz_r > 0.0 ? fl * fm * h->frz_r : INFINITY, h->frz_r > 0.0 ? fm * h->frz_r : INFINITY};
    const StepArgs T{freeze ? env_dbl("BLP_STEP_SAFETY", o.step_safety) : 0.0, env_dbl("BLP_STEP_CAP", 4.0),
                     env_int("BLP_POW_FIRST", 40), env_int("BLP_POW_PASSES", 3)};
    uint8_t* const cfrz_ws = S.cfrz;
    const size_t frz_bytes = (size_t)(S.rfrz - S.cfrz) + (size_t)P.m * (S.ld / 32);
    if (!freeze) S.cfrz = S.rfrz = nullptr;
    const bool want_frac = frac_idx != nullptr && int_idx != nullptr && n_int > 0;
    if (o.verbose < 2) S.dbg = nullptr;
    uint8_t* isint_ws = const_cast<uint8_t*>(S.isint);
    if (!want_frac) S.isint = nullptr;
    DevOut O{obj, lower_bound, x, y, status, iters, frac_idx, ld_in};

    // evaluation period: eval_every at first, 4x that once a node batch has run 32 periods (an
    // evaluation costs about three iterations; late in a solve nothing changes within 64 of them)
    const int K0 = std::min(o.eval_every, o.max_iters);
    int K = K0;
    const int rpw = env_int("BLP_ROWS_PER_WARP", 8);
    int NT = pick_nt(W);     // nodes per warp; re-picked when compaction narrows the batch
    // evaluation / check / harvest plans: one node per lane, re-made when compaction narrows the batch
    Plan ec = plan_rows(P.n, W, NT, 1, kEvalChunks), er = plan_rows(P.m, W, NT, 1, kEvalChunks);
    DecideArgs D{ec.chunks, er.chunks, K, o.max_iters, o.eps_rel, o.eps_infeas,
                 env_dbl("BLP_BETA_SUFF", 0.2), env_dbl("BLP_BETA_NEC", 0.8), env_dbl("BLP_BETA_ART", 0.36),
                 env_dbl("BLP_OMEGA_THETA", 0.05), env_dbl("BLP_OMEGA_BALANCE", 0.3),
                 env_dbl("BLP_OMEGA_DEADZONE", 0.25), o.obj_cutoff};
    int launches = 0;

    CK(cudaEventRecord(h->ev[0], st));
    CK(cudaMemsetAsync(S.counters, 0, 16 * sizeof(int32_t), st));
    if (freeze) CK(cudaMemsetAsync(cfrz_ws, 0, frz_bytes, st));
    if (have_mask)
        CK(cudaMemcpy2DAsync(mask_ws, S.ld, row_mask, ld_in, S.ld, P.m - P.m_base, cudaMemcpyDeviceToDevice, st));
    if (want_frac) {
        CK(cudaMemsetAsync(isint_ws, 0, P.n, st));
        k_set_isint<<<(n_int + 255) / 256, 256, 0, st>>>(int_idx, n_int, P.n, isint_ws);
        ++launches;
    }
    if (x) CK(cudaMemsetAsync(x, 0, (size_t)P.n * ld_in * sizeof(double), st));
    if (y) CK(cudaMemsetAsync(y, 0, (size_t)P.m * ld_in * sizeof(double), st));
    if (ld_in > B) {
        k_out_pad<<<(ld_in - B + 127) / 128, 128, 0, st>>>(O, B, ld_in);
        ++launches;
    }
    k_init_nodes<<<(S.ld + 127) / 128, 128, 0, st>>>(P, S);
    k_init_cols<<<elementwise_grid((size_t)P.n * S.ld), kCtaThreads, 0, st>>>(P, S, lb, ub, x0, ld_in);
    k_init_rows<<<elementwise_grid((size_t)P.m * S.ld), kCtaThreads, 0, st>>>(P, S, y0, ld_in);
    launch_check_rows(P, S, er, 0, st);
    k_build_lumask<<<elementwise_grid((size_t)P.n * (S.ld / 32) * 32), kCtaThreads, 0, st>>>(P, S);
    k_count_active<<<(W + 127) / 128, 128, 0, st>>>(S);
    launches += 6;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(h->h_counters, S.counters, 13 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    int active = h->h_counters[0];

    // step kernels: fewer rows per warp when the batch is narrow, so that a handful of running
    // nodes still spreads over all SMs (the per-iteration latency floor of the solve's tail)
    const bool allow_v2 = env_int("BLP_V2", 1) != 0;
    const int graph_lanes = env_int("BLP_GRAPH_LANES", 2);
    const int rpw2 = std::min(env_int("BLP_ROWS_PER_WARP2", 16), kMaxChunkRows / kWarps);   // two-nodes-per-lane kernels: 128 rows per CTA
    // primal step with frozen coordinates: a third of a chunk's rows are left, 192-row chunks amortise the slab better
    // (profiles/r2v_variant_sweep.log: -2.7 %; 5 or 4 CTAs per SM, 8 gathers in flight, 4 graph lanes all lose)
    const int rpw2p = std::min(env_int("BLP_ROWS_PER_WARP2P", freeze ? 24 : rpw2), kMaxChunkRows / kWarps);
    auto step_plan = [&](int rows, int width, bool primal = false) {
        // two nodes per lane pay off when a launch has real work; tiny LPs stay on the
        // one-node-per-lane kernels, which can run a whole period as one cooperative launch
        // (k_primal2 / k_dual2 index the state with 32 bits)
        const bool v2 = allow_v2 && width >= kBlk && (long)std::max(P.n, P.m) * width >= (1L << 20) &&
                        (size_t)std::max(P.n, P.m) * S.ld < ((size_t)1 << 32);
        int r = v2 ? (primal ? rpw2p : rpw2) : rpw;
        Plan p = plan_rows(rows, width, NT, r, 0);
        auto shape = [&](Plan& q, int rr) {
            if (!v2) return;
            q.V = 2;                                   // a warp = one row x 64 nodes
            q.tiles = (width + kBlk - 1) / kBlk;
            q.rows_per_cta = kWarps * std::max(rr, 1);
            q.chunks = std::max(1, (rows + q.rows_per_cta - 1) / q.rows_per_cta);
        };
        shape(p, r);
        while (r > 1 && (long)p.chunks * p.tiles < 148L * 12) {
            r /= 2;
            p = plan_rows(rows, width, NT, r, 0);
            shape(p, r);
        }
        return p;
    };
    Plan pc = step_plan(P.n, W, true), pr = step_plan(P.m, W);
    auto finish_step_plans = [&]() -> int {
        plan_chunks(pc, h->hptrAT, P.n, h->h_chunkC);
        plan_chunks(pr, h->hptrA, P.m, h->h_chunkR);
        if (pc.V == 2) {                           // k_primal2 / k_dual2 stage their rows' scalars behind the slab
            pc.smem += (size_t)kPrimalRowBytes * pc.rows_per_cta;
            pr.smem += (size_t)kDualRowBytes * pr.rows_per_cta;
        }
        CK(upload(h->chunkC, h->h_chunkC, st));
        CK(upload(h->chunkR, h->h_chunkR, st));
        pc.chunk_ptr = h->chunkC.as<int32_t>();
        pr.chunk_ptr = h->chunkR.as<int32_t>();
        return BLP_OK;
    };
    if ((rc = finish_step_plans()) != BLP_OK) return rc;

    if (active < W) launch_harvest(P, S, O, ec, er, want_frac, st, &launches);    // decided at set-up

    // continuous batching: pending nodes next .. B-1 take over the slots of harvested ones
    int next = W, refills = 0;
    auto refill = [&]() -> int {
        while (next < B && active < S.B) {
            const int nnew = std::min(B - next, S.B - active);
            k_refill_plan<<<1, 1024, 0, st>>>(P, S, next, nnew);
            k_refill_cols<<<elementwise_grid((size_t)P.n * nnew), kCtaThreads, 0, st>>>(P, S, lb, ub, x0, ld_in, nnew);
            k_refill_rows<<<elementwise_grid((size_t)P.m * nnew), kCtaThreads, 0, st>>>(P, S, y0, row_mask, ld_in, nnew);
            launch_check_rows(P, S, er, 1, st);
            k_build_lumask<<<elementwise_grid((size_t)P.n * ((S.B + 31) / 32) * 32), kCtaThreads, 0, st>>>(P, S);
            k_count_active<<<(S.B + 127) / 128, 128, 0, st>>>(S);
            launches += 6;
            CK(cudaGetLastError());
            CK(cudaMemcpyAsync(h->h_counters, S.counters, 13 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            next += nnew;
            refills += nnew;
            active = h->h_counters[0];
            if (h->h_counters[3] > 0) launch_harvest(P, S, O, ec, er, want_frac, st, &launches);
        }
        return BLP_OK;
    };
    if ((rc = refill()) != BLP_OK) return rc;
    // frozen coordinates exist for the two-nodes-per-lane step kernels only (wide batches)
    auto refreeze = [&](int mode) {
        if (!freeze || pc.V != 2) return;
        launches += launch_freeze(P, S, F, T, pc, pr, mode, st);
    };
    refreeze(2);

    const bool profile = o.profile == 1;
    const bool use_graph = o.use_graph && !profile;
    if (profile)
        while ((int)h->prof_ev.size() < 2 * 4 * K0 + 1) {
            cudaEvent_t e;
            CK(cudaEventCreate(&e));
            h->prof_ev.push_back(e);
        }

    bool coop = false;          // this period's steps run as one cooperative launch
    bool coop_rejected = false; // the current plan does not fit a cooperative grid
    const bool allow_coop = h->coop_ok && env_int("BLP_COOP", 1) != 0;
    auto ensure_graphs = [&]() -> int {
        GraphKey key;
        memset(&key, 0, sizeof key);
        key.P = P;
        key.S = S;
        key.D = D;
        key.K = K;
        key.rpw = rpw | (rpw2 << 8) | (rpw2p << 24) | (allow_v2 ? 1 << 16 : 0) | (coop ? 1 << 17 : 0) | (graph_lanes << 20);
        if (h->graph_valid && memcmp(&key, &h->gkey, sizeof key) == 0) return BLP_OK;
        h->drop_graphs();
        cudaGraph_t g = nullptr;
        cudaError_t e = cudaSuccess;
        if (!coop) {
            CK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
            const int lanes = pc.V == 2 ? std::max(1, std::min({graph_lanes, pc.tiles, (int)blp_handle_s::kLanes})) : 1;
            if (lanes == 1) {
                for (int it = 0; it < K; ++it) launch_steps(P, S, pc, pr, it, it == K - 1, st);
            } else {
                // branch b owns the node tiles [b*T/lanes, (b+1)*T/lanes): its 2K launches depend
                // only on each other, the branches meet again at the end of the period
                CK(cudaEventRecord(h->ev_fork, st));
                for (int b = 0; b < lanes; ++b) {
                    cudaStream_t sb = b == 0 ? st : h->side[b - 1];
                    if (b) CK(cudaStreamWaitEvent(sb, h->ev_fork, 0));
                    const int t0 = (int)((long)pc.tiles * b / lanes), t1 = (int)((long)pc.tiles * (b + 1) / lanes);
                    for (int it = 0; it < K; ++it) launch_steps(P, S, pc, pr, it, it == K - 1, sb, 2, t0, t1 - t0);
                    if (b) {
                        CK(cudaEventRecord(h->ev_join[b - 1], sb));
                        CK(cudaStreamWaitEvent(st, h->ev_join[b - 1], 0));
                    }
                }
            }
            CK(cudaStreamEndCapture(st, &g));
            e = cudaGraphInstantiate(&h->g_steps, g, 0);
            cudaGraphDestroy(g);
            if (e != cudaSuccess) return fail(BLP_ERR_CUDA, "graph instantiate: %s", cudaGetErrorString(e));
        }
        CK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
        launch_eval(P, S, ec, er, D, K, st);
        CK(cudaStreamEndCapture(st, &g));
        e = cudaGraphInstantiate(&h->g_eval, g, 0);
        cudaGraphDestroy(g);
        if (e != cudaSuccess) return fail(BLP_ERR_CUDA, "graph instantiate: %s", cudaGetErrorString(e));
        h->gkey = key;
        h->graph_valid = true;
        return BLP_OK;
    };

    int total = 0, evals = 0, compactions = 0;
    double step_ms = 0.0, primal_ms = 0.0, dual_ms = 0.0, node_iters = 0.0, skipped_cols = 0.0, skipped_rows = 0.0;
    while (active > 0 && (refill_mode || total < o.max_iters)) {
        // retire finished nodes: pack the running ones to the front when that frees node tiles
        // (while nodes are pending, freed slots are refilled instead)
        if (o.compact && active < S.B && next >= B) {
            const int cur_tiles = (S.B + NT - 1) / NT, new_tiles = (active + NT - 1) / NT;
            if ((new_tiles < cur_tiles && (new_tiles * 8 <= cur_tiles * 7 || cur_tiles <= 16)) ||
                pick_nt(active) < NT) {
                const int oldB = S.B;
                k_compact_plan<<<1, 1024, 0, st>>>(S);
                k_compact_vecs<<<elementwise_grid((size_t)(5 * P.n + 3 * P.m) * 32), kCtaThreads, 0, st>>>(P, S, oldB);
                CK(cudaGetLastError());
                S.B = active;
                k_build_lumask<<<elementwise_grid((size_t)P.n * ((S.B + 31) / 32) * 32), kCtaThreads, 0, st>>>(P, S);
                launches += 3;
                ++compactions;
                NT = pick_nt(S.B);
                pc = step_plan(P.n, S.B, true);
                pr = step_plan(P.m, S.B);
                if ((rc = finish_step_plans()) != BLP_OK) return rc;
                if (freeze) {
                    // the slots moved: the tiles are new sets of nodes and their flags start afresh (x', y' travelled
                    // with the nodes); a batch that has become too narrow for the freezing kernels updates every
                    // coordinate again, so its nodes return to the step of the full matrix
                    if (pc.V == 2) launches += launch_freeze(P, S, F, T, pc, pr, 2, st);
                    else k_eta_reset<<<(S.ld + 127) / 128, 128, 0, st>>>(P, S), ++launches;
                }
                coop_rejected = false;
                ec = plan_rows(P.n, S.B, NT, 1, kEvalChunks);
                er = plan_rows(P.m, S.B, NT, 1, kEvalChunks);
                D.chunksC = ec.chunks;
                D.chunksR = er.chunks;
            }
        }
        {
            int want = (total >= 32 * K0 && env_int("BLP_ADAPTIVE_EVAL", 1)) ? 4 * K0 : K0;
            if (!refill_mode) want = std::min(want, o.max_iters - total);
            if (want != K) {
                K = want;
                D.steps_in_period = K;
            }
        }
        coop = use_graph && allow_coop && pc.V == 1 && !coop_rejected;
        if (use_graph) {
            int rcg = ensure_graphs();
            if (rcg != BLP_OK) return rcg;
        }
        CK(cudaEventRecord(h->ev[2], st));
        if (coop) {
            cudaError_t ce = launch_period_coop(h, P, S, pc, pr, K, st);
            if (ce != cudaSuccess) {                      // too many rows / not co-resident: graph path
                cudaGetLastError();
                coop = false;
                coop_rejected = true;
                int rcg = ensure_graphs();
                if (rcg != BLP_OK) return rcg;
                CK(cudaGraphLaunch(h->g_steps, st));
            }
        } else if (use_graph) {
            CK(cudaGraphLaunch(h->g_steps, st));
        } else if (profile) {
            CK(cudaEventRecord(h->prof_ev[0], st));
            for (int it = 0; it < K; ++it) {
                launch_steps(P, S, pc, pr, it, it == K - 1, st, 0);
                CK(cudaEventRecord(h->prof_ev[2 * it + 1], st));
                launch_steps(P, S, pc, pr, it, it == K - 1, st, 1);
                CK(cudaEventRecord(h->prof_ev[2 * it + 2], st));
            }
        } else {
            for (int it = 0; it < K; ++it) launch_steps(P, S, pc, pr, it, it == K - 1, st);
        }
        CK(cudaEventRecord(h->ev[3], st));
        if (use_graph) {
            CK(cudaGraphLaunch(h->g_eval, st));
        } else {
            launch_eval(P, S, ec, er, D, K, st);
        }
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(h->h_counters, S.counters, 13 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, h->ev[2], h->ev[3]));
        step_ms += ms;
        if (profile)
            for (int it = 0; it < K; ++it) {
                float t = 0.f;
                CK(cudaEventElapsedTime(&t, h->prof_ev[2 * it], h->prof_ev[2 * it + 1]));
                primal_ms += t;
                CK(cudaEventElapsedTime(&t, h->prof_ev[2 * it + 1], h->prof_ev[2 * it + 2]));
                dual_ms += t;
            }
        node_iters += (double)active * K;
        if (freeze && pc.V == 2) {      // counts of the flags that were in force during this period
            unsigned long long fc[2];
            memcpy(fc, h->h_counters + 8, sizeof fc);
            skipped_cols += (double)fc[0] * (K - 1);
            skipped_rows += (double)fc[1] * (K - 1);
        }
        total += K;
        evals += 1;
        launches += (coop ? 1 : 2 * K) + 5;
        active = h->h_counters[0];
        const int finished_now = h->h_counters[3], restarting = h->h_counters[1];
        const int refills_before = refills;
        if (finished_now > 0) {
            launch_harvest(P, S, O, ec, er, want_frac, st, &launches);
            CK(cudaGetLastError());
            if ((rc = refill()) != BLP_OK) return rc;
        }
        if (active > 0) refreeze(refills > refills_before ? 1 : 0);
        if (o.verbose >= 2) {
            double t[8 * 4];
            const int kshow = std::min(4, S.B);
            CK(cudaMemcpy(t, S.dbg, sizeof(double) * 8 * kshow, cudaMemcpyDeviceToHost));
            for (int k = 0; k < kshow; ++k)
                fprintf(stderr, "[blp]   col %d: rp %.2e rd %.2e gap %.2e fpe %.2e omega %.3e since_restart %.0f pobj %.9e dobj %.9e\n",
                        k, t[8 * k], t[8 * k + 1], t[8 * k + 2], t[8 * k + 3], t[8 * k + 4], t[8 * k + 5], t[8 * k + 6], t[8 * k + 7]);
        }
        if (o.verbose)
            fprintf(stderr, "[blp] iters %d  width %d  running %d  restarting %d  finished now %d  steps_ms %.3f\n",
                    total, S.B, active, restarting, finished_now, ms);
    }
    CK(cudaEventRecord(h->ev[1], st));
    CK(cudaStreamSynchronize(st));
    if (stats) {
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]));
        stats->iterations = total;
        stats->evaluations = evals;
        stats->kernel_launches = launches;
        stats->compactions = compactions;
        stats->step_kernel_ms = step_ms;
        stats->total_ms = ms;
        stats->node_iterations = node_iters;
        stats->primal_kernel_ms = primal_ms;
        stats->dual_kernel_ms = dual_ms;
        stats->refills = refills;
        stats->skipped_col_updates = skipped_cols;
        stats->skipped_row_updates = skipped_rows;
        stats->step_resets = h->h_counters[12];
    }
    return BLP_OK;
}

// ---- host-buffer entry points -------------------------------------------------------------------
namespace {

int stage_in(blp_handle h, DevBuf& dst, const double* src, int B, int rows, int ld) {
    cudaStream_t st = h->stream;
    CK(dst.ensure((size_t)rows * ld * sizeof(double)));
    CK(h->s_tmp.ensure((size_t)rows * B * sizeof(double)));
    CK(cudaMemcpyAsync(h->s_tmp.p, src, (size_t)rows * B * sizeof(double), cudaMemcpyHostToDevice, st));
    k_transpose_in<<<dim3((rows + 31) / 32, (ld + 31) / 32), dim3(32, 8), 0, st>>>(
        h->s_tmp.as<double>(), B, rows, ld, dst.as<double>());
    CK(cudaGetLastError());
    // s_tmp is reused by the next stage_in on the same stream: ordering is by the stream
    return BLP_OK;
}

int stage_out(blp_handle h, const DevBuf& src, double* dst, int B, int rows, int ld) {
    cudaStream_t st = h->stream;
    CK(h->s_tmp.ensure((size_t)rows * B * sizeof(double)));
    k_transpose_out<<<dim3((rows + 31) / 32, (ld + 31) / 32), dim3(32, 8), 0, st>>>(
        src.as<double>(), B, rows, ld, h->s_tmp.as<double>());
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(dst, h->s_tmp.p, (size_t)rows * B * sizeof(double), cudaMemcpyDeviceToHost, st));
    return BLP_OK;
}

struct NodeOut {
    double *obj, *lower;
    int32_t *status, *iters, *frac;
};

NodeOut node_out(blp_handle h, int ld) {
    char* p = h->s_node.as<char>();
    NodeOut o;
    o.obj = reinterpret_cast<double*>(p);
    o.lower = o.obj + ld;
    o.status = reinterpret_cast<int32_t*>(o.lower + ld);
    o.iters = o.status + ld;
    o.frac = o.iters + ld;
    return o;
}

int finish_host(blp_handle h, int B, int ld, const NodeOut& no, bool want_x, bool want_y,
                double* obj, double* lower_bound, int32_t* status, int32_t* iters, double* x,
                double* y, int32_t* frac_idx) {
    cudaStream_t st = h->stream;
    if (want_x) { int rc = stage_out(h, h->s_x, x, B, h->n, ld); if (rc) return rc; }
    if (want_y) { int rc = stage_out(h, h->s_y, y, B, h->A0.rows, ld); if (rc) return rc; }
    if (obj) CK(cudaMemcpyAsync(obj, no.obj, B * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (lower_bound) CK(cudaMemcpyAsync(lower_bound, no.lower, B * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (status) CK(cudaMemcpyAsync(status, no.status, B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (iters) CK(cudaMemcpyAsync(iters, no.iters, B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (frac_idx) CK(cudaMemcpyAsync(frac_idx, no.frac, B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return BLP_OK;
}

int stage_common(blp_handle h, int B, int W, int ld, const uint8_t* row_mask, const int32_t* int_idx,
                 int n_int, bool want_x, bool want_y, const uint8_t** d_mask,
                 const int32_t** d_int) {
    cudaStream_t st = h->stream;
    const int m = h->A0.rows, n = h->n, mc = m - h->m_base;
    *d_mask = nullptr;
    *d_int = nullptr;
    if (row_mask && mc > 0) {
        CK(h->s_mask.ensure((size_t)mc * ld + (size_t)mc * B));
        uint8_t* raw = h->s_mask.as<uint8_t>() + (size_t)mc * ld;
        CK(cudaMemcpyAsync(raw, row_mask, (size_t)mc * B, cudaMemcpyHostToDevice, st));
        k_transpose_in_u8<<<elementwise_grid((size_t)mc * ld), kCtaThreads, 0, st>>>(
            raw, B, mc, ld, h->s_mask.as<uint8_t>());
        *d_mask = h->s_mask.as<uint8_t>();
    }
    if (int_idx && n_int > 0) {
        CK(h->s_int.ensure((size_t)n_int * sizeof(int32_t)));
        CK(cudaMemcpyAsync(h->s_int.p, int_idx, (size_t)n_int * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        *d_int = h->s_int.as<int32_t>();
    }
    if (want_x) CK(h->s_x.ensure((size_t)n * ld * sizeof(double)));
    if (want_y) CK(h->s_y.ensure((size_t)m * ld * sizeof(double)));
    CK(h->s_node.ensure((size_t)ld * (2 * sizeof(double) + 3 * sizeof(int32_t))));
    CK(h->s_ws.ensure(blp_workspace_bytes(h, W)));
    CK(cudaGetLastError());
    return BLP_OK;
}

// blp_solve_batch on the bounds and starts staged in h->s_lb, s_ub (s_x0, s_y0 if given), results to the host
int solve_staged(blp_handle h, int B, int ld, bool have_x0, bool have_y0, const uint8_t* row_mask,
                 const int32_t* int_idx, int n_int, const blp_opts* opts, double* obj, double* lower_bound,
                 int32_t* status, int32_t* iters, double* x, double* y, int32_t* frac_idx, blp_stats* stats) {
    const uint8_t* d_mask;
    const int32_t* d_int;
    int rc;
    if ((rc = stage_common(h, B, blp_slots(B, opts), ld, row_mask, int_idx, n_int, x != nullptr, y != nullptr,
                           &d_mask, &d_int)))
        return rc;
    NodeOut no = node_out(h, ld);
    rc = blp_solve_batch(h, B, h->s_lb.as<double>(), h->s_ub.as<double>(), d_mask,
                         have_x0 ? h->s_x0.as<double>() : nullptr, have_y0 ? h->s_y0.as<double>() : nullptr,
                         d_int, n_int, opts, h->s_ws.p, h->s_ws.cap, no.obj, no.lower, no.status,
                         no.iters, x ? h->s_x.as<double>() : nullptr,
                         y ? h->s_y.as<double>() : nullptr, no.frac, stats);
    if (rc) return rc;
    return finish_host(h, B, ld, no, x != nullptr, y != nullptr, obj, lower_bound, status, iters, x, y, frac_idx);
}

// Bound changes of B children against their parent: child k sets the bounds of variables
// delta_var[delta_ptr[k] .. delta_ptr[k + 1]) to delta_lb / delta_ub. `who` names the entry point in the errors.
int check_deltas(blp_handle h, int B, const int32_t* delta_ptr, const int32_t* delta_var, const double* delta_lb,
                 const double* delta_ub, const char* who) {
    const int nd = delta_ptr[B];
    if (delta_ptr[0] != 0 || nd < 0 || (nd > 0 && (!delta_var || !delta_lb || !delta_ub)))
        return fail(BLP_ERR_ARG, "%s: bad delta arrays", who);
    for (int k = 0; k < B; ++k)
        if (delta_ptr[k + 1] < delta_ptr[k]) return fail(BLP_ERR_ARG, "%s: delta_ptr not monotone", who);
    for (int p = 0; p < nd; ++p)
        if (delta_var[p] < 0 || delta_var[p] >= h->n)
            return fail(BLP_ERR_ARG, "%s: delta_var[%d] = %d out of range", who, p, delta_var[p]);
    return BLP_OK;
}

struct DevDeltas {
    const int32_t* ptr;
    const int32_t* var;
    const double *lb, *ub;
};

// Uploads checked delta arrays with nd = delta_ptr[B] > 0 entries into h->s_delta.
int stage_deltas(blp_handle h, int B, const int32_t* delta_ptr, const int32_t* delta_var, const double* delta_lb,
                 const double* delta_ub, DevDeltas* out) {
    cudaStream_t st = h->stream;
    const int nd = delta_ptr[B];
    const size_t ip = align_up((size_t)(B + 1) * sizeof(int32_t), 8), iv = align_up((size_t)nd * sizeof(int32_t), 8);
    CK(h->s_delta.ensure(ip + iv + 2 * (size_t)nd * sizeof(double) + 64));
    char* d = h->s_delta.as<char>();
    out->ptr = reinterpret_cast<const int32_t*>(d);
    out->var = reinterpret_cast<const int32_t*>(d + ip);
    out->lb = reinterpret_cast<const double*>(d + ip + iv);
    out->ub = out->lb + nd;
    CK(cudaMemcpyAsync(d, delta_ptr, (B + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d + ip, delta_var, nd * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d + ip + iv, delta_lb, nd * sizeof(double), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d + ip + iv + nd * sizeof(double), delta_ub, nd * sizeof(double), cudaMemcpyHostToDevice, st));
    return BLP_OK;
}

}  // namespace

int blp_solve_batch_host(blp_handle h, int B, const double* lb, const double* ub,
                         const uint8_t* row_mask, const double* x0, const double* y0,
                         const int32_t* int_idx, int n_int, const blp_opts* opts,
                         double* obj, double* lower_bound, int32_t* status, int32_t* iters,
                         double* x, double* y, int32_t* frac_idx, blp_stats* stats) {
    if (!h) return fail(BLP_ERR_ARG, "blp_solve_batch_host: NULL handle");
    if (B < 1 || !lb || !ub) return fail(BLP_ERR_ARG, "blp_solve_batch_host: need B >= 1 and lb/ub");
    CK(cudaSetDevice(h->device));
    const int ld = blp_ld(B), n = h->n, m = h->A0.rows;
    int rc;
    if ((rc = stage_in(h, h->s_lb, lb, B, n, ld))) return rc;
    if ((rc = stage_in(h, h->s_ub, ub, B, n, ld))) return rc;
    if (x0 && (rc = stage_in(h, h->s_x0, x0, B, n, ld))) return rc;
    if (y0 && (rc = stage_in(h, h->s_y0, y0, B, m, ld))) return rc;
    return solve_staged(h, B, ld, x0 != nullptr, y0 != nullptr, row_mask, int_idx, n_int, opts, obj, lower_bound,
                        status, iters, x, y, frac_idx, stats);
}

int blp_solve_children_host(blp_handle h, int B, const double* parent_lb, const double* parent_ub,
                            const int32_t* delta_ptr, const int32_t* delta_var,
                            const double* delta_lb, const double* delta_ub,
                            const uint8_t* row_mask, const double* x0, const double* y0,
                            const int32_t* int_idx, int n_int, const blp_opts* opts,
                            double* obj, double* lower_bound, int32_t* status, int32_t* iters,
                            double* x, double* y, int32_t* frac_idx, blp_stats* stats) {
    if (!h) return fail(BLP_ERR_ARG, "blp_solve_children_host: NULL handle");
    if (B < 1 || !parent_lb || !parent_ub || !delta_ptr)
        return fail(BLP_ERR_ARG, "blp_solve_children_host: need B >= 1, parent bounds and delta_ptr");
    int rc = check_deltas(h, B, delta_ptr, delta_var, delta_lb, delta_ub, "blp_solve_children_host");
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const int ld = blp_ld(B), n = h->n, m = h->A0.rows;
    // parent vectors: [lb | ub | x0 | y0]
    CK(h->s_par.ensure((size_t)(3 * n + m) * sizeof(double)));
    double* par = h->s_par.as<double>();
    CK(cudaMemcpyAsync(par, parent_lb, n * sizeof(double), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(par + n, parent_ub, n * sizeof(double), cudaMemcpyHostToDevice, st));
    if (x0) CK(cudaMemcpyAsync(par + 2 * n, x0, n * sizeof(double), cudaMemcpyHostToDevice, st));
    if (y0) CK(cudaMemcpyAsync(par + 3 * n, y0, m * sizeof(double), cudaMemcpyHostToDevice, st));
    CK(h->s_lb.ensure((size_t)n * ld * sizeof(double)));
    CK(h->s_ub.ensure((size_t)n * ld * sizeof(double)));
    const int gcol = elementwise_grid((size_t)n * ld), grow = elementwise_grid((size_t)m * ld);
    k_broadcast_rows<<<gcol, kCtaThreads, 0, st>>>(par, n, ld, h->s_lb.as<double>());
    k_broadcast_rows<<<gcol, kCtaThreads, 0, st>>>(par + n, n, ld, h->s_ub.as<double>());
    if (x0) {
        CK(h->s_x0.ensure((size_t)n * ld * sizeof(double)));
        k_broadcast_rows<<<gcol, kCtaThreads, 0, st>>>(par + 2 * n, n, ld, h->s_x0.as<double>());
    }
    if (y0) {
        CK(h->s_y0.ensure((size_t)m * ld * sizeof(double)));
        k_broadcast_rows<<<grow, kCtaThreads, 0, st>>>(par + 3 * n, m, ld, h->s_y0.as<double>());
    }
    if (delta_ptr[B] > 0) {
        DevDeltas d;
        if ((rc = stage_deltas(h, B, delta_ptr, delta_var, delta_lb, delta_ub, &d))) return rc;
        k_patch_bounds<<<(B + 127) / 128, 128, 0, st>>>(B, ld, d.ptr, d.var, d.lb, d.ub, h->s_lb.as<double>(),
                                                         h->s_ub.as<double>());
    }
    CK(cudaGetLastError());
    return solve_staged(h, B, ld, x0 != nullptr, y0 != nullptr, row_mask, int_idx, n_int, opts, obj, lower_bound,
                        status, iters, x, y, frac_idx, stats);
}

int blp_spmv(blp_handle h, int B, int transpose, const double* X, double* Y) {
    if (!h || B < 1 || !X || !Y) return fail(BLP_ERR_ARG, "blp_spmv: bad arguments");
    CK(cudaSetDevice(h->device));
    const int ld = blp_ld(B);
    const int rows = transpose ? h->n : h->A0.rows;
    const int32_t* ptr = transpose ? h->P.cptr : h->P.rowptr;
    const Ent* ent = transpose ? h->ucent.as<Ent>() : h->uent.as<Ent>();
    cudaStream_t st = h->stream;
    if (B >= kBlk && env_int("BLP_V2", 1) != 0) {               // two nodes per lane
        Plan p;
        p.rows_per_cta = kWarps * env_int("BLP_ROWS_PER_WARP2", 16);
        p.chunks = std::max(1, (rows + p.rows_per_cta - 1) / p.rows_per_cta);
        p.tiles = ld / kBlk;
        plan_slab(p, transpose ? h->hptrAT : h->hptrA, rows);
        k_spmv2<<<dim3(p.chunks, p.tiles), kCtaThreads, p.smem, st>>>(ptr, ent, rows, B, ld, X, Y, p.rows_per_cta, p.cap);
        CK(cudaGetLastError());
        return BLP_OK;
    }
    Plan p = plan_rows(rows, B, pick_nt(B), env_int("BLP_ROWS_PER_WARP", 8), 0);
    plan_slab(p, transpose ? h->hptrAT : h->hptrA, rows);
    with_nt(p.NT, [&](auto nt) {
        k_spmv<nt><<<dim3(p.chunks, p.tiles), kCtaThreads, p.smem, st>>>(ptr, ent, rows, B, ld, X, Y, p.rows_per_cta, p.cap);
    });
    CK(cudaGetLastError());
    return BLP_OK;
}

// ---- dual simplex path for small node LPs (blp_simplex.cuh) ---------------------------------------
namespace {

__global__ void k_sx_expand_children(const int B, const int n, const int m, const double* __restrict__ plb,
                                     const double* __restrict__ pub, const int8_t* __restrict__ pcs,
                                     const int8_t* __restrict__ prs, const uint8_t* __restrict__ pmask, const int mc,
                                     double* __restrict__ lb, double* __restrict__ ub, int8_t* __restrict__ cs,
                                     int8_t* __restrict__ rs, uint8_t* __restrict__ mask) {
    const size_t tot = (size_t)B * n;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < tot; e += (size_t)gridDim.x * blockDim.x) {
        const int j = (int)(e % n);
        lb[e] = plb[j];
        ub[e] = pub[j];
        if (cs) cs[e] = pcs[j];
    }
    if (rs)
        for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < (size_t)B * m; e += (size_t)gridDim.x * blockDim.x)
            rs[e] = prs[e % m];
    if (mask)
        for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < (size_t)B * mc; e += (size_t)gridDim.x * blockDim.x)
            mask[e] = pmask[e % mc];
}

__global__ void k_sx_patch_children(const int B, const int n, const int32_t* __restrict__ dptr,
                                    const int32_t* __restrict__ dvar, const double* __restrict__ dlb,
                                    const double* __restrict__ dub, double* __restrict__ lb, double* __restrict__ ub) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= B) return;
    for (int p = dptr[k]; p < dptr[k + 1]; ++p) {
        lb[(size_t)k * n + dvar[p]] = dlb[p];
        ub[(size_t)k * n + dvar[p]] = dub[p];
    }
}

struct SxStage {           // device pointers carved from h->sx_in / h->sx_out
    double *lb, *ub;
    uint8_t* mask;
    int8_t *cs, *rs;
    int32_t* parent;
    double *obj, *x, *y, *rc;
    int32_t *status, *pivots, *flips;
    int8_t *cso, *rso;
};

int sx_carve(blp_handle h, int B, bool want_mask, bool want_status, bool want_parent, SxStage* S) {
    const size_t n = h->n, m = h->A0.rows, mc = m - h->m_base;
    {
        size_t need = 2 * B * n * sizeof(double) + 256 * 8 + B * mc + B * n + B * m + B * sizeof(int32_t);
        CK(h->sx_in.ensure(need));
        Carve cv{h->sx_in.as<char>()};
        S->lb = cv.take<double>(B * n);
        S->ub = cv.take<double>(B * n);
        S->mask = (want_mask && mc > 0) ? cv.take<uint8_t>(B * mc) : nullptr;
        S->cs = want_status ? cv.take<int8_t>(B * n) : nullptr;
        S->rs = want_status ? cv.take<int8_t>(B * m) : nullptr;
        S->parent = want_parent ? cv.take<int32_t>(B) : nullptr;
    }
    {
        size_t need = (size_t)B * (1 + 2 * n + m) * sizeof(double) + 256 * 10 + 3 * B * sizeof(int32_t) + B * (n + m);
        CK(h->sx_out.ensure(need));
        Carve cv{h->sx_out.as<char>()};
        S->obj = cv.take<double>(B);
        S->x = cv.take<double>(B * n);
        S->y = cv.take<double>(B * m);
        S->rc = cv.take<double>(B * n);
        S->status = cv.take<int32_t>(B);
        S->pivots = cv.take<int32_t>(B);
        S->flips = cv.take<int32_t>(B);
        S->cso = cv.take<int8_t>(B * n);
        S->rso = cv.take<int8_t>(B * m);
    }
    return BLP_OK;
}

// Groups of SMs that k_simplex_wide runs side by side for a batch of B mid-size LPs of m rows: G = min(B,
// Gmax(m)), S = SMs / G CTAs per group. A group's pivot is bound by its barriers and by the rows every CTA
// scans for its own decisions, not by bandwidth, so small LPs gain from many groups and large ones, whose
// inverses compete for HBM, from few. Gmax(m) is fitted from the sweep of tools/gpu_simplex_groups.py
// (profiles/simplex_groups_sweep.json, DESIGN section 2b).
int sx_groups(int m, int B) {
    const int gmax = m <= 5000 ? 64 : 16;
    return std::min(B, gmax);
}

// launch the simplex kernel on staged inputs, copy the results back to the host
int sx_run(blp_handle h, int B, const SxStage& S, bool use_parent, int max_pivots, double* obj,
           int32_t* status, int32_t* pivots, double* x, double* y, double* rc, int8_t* cso, int8_t* rso,
           blp_stats* stats) {
    cudaStream_t st = h->stream;
    const int n = h->n, m = h->A0.rows, N = n + m;
    const int ldm = (m + 31) / 32 * 32;
    const int cur = h->sx_cur, prev = cur ^ 1;
    CK(h->sx_binv[cur].ensure((size_t)B * m * ldm * sizeof(double)));
    CK(h->sx_head[cur].ensure((size_t)B * m * sizeof(int32_t)));
    CK(h->sx_stat[cur].ensure((size_t)B * N));
    CK(h->sx_wts[cur].ensure((size_t)B * m * sizeof(double)));
    const size_t stride = (size_t)6 * N + 6 * m + (5 * (size_t)N + 7) / 8 + 2;
    CK(h->sx_work.ensure((size_t)B * stride * sizeof(double)));
    SxProb P{m, h->m_base, n, ldm, h->P.rowptr, h->uent.as<Ent>(), h->P.cptr, h->ucent.as<Ent>(),
             h->uc.as<double>(), h->ub.as<double>()};
    SxBatch Q{};
    Q.B = B;
    Q.max_pivots = max_pivots;
    // test knobs of a tuning build: a negative mismatch threshold refuses every pivot that does not directly
    // follow a factorisation, a small interval forces the periodic refactorisation
    Q.pivot_mismatch = env_dbl("BLP_SX_MISMATCH", kSxPivotMismatch);
    Q.refactor_every = env_int("BLP_SX_REFACTOR_EVERY", 0);
    Q.lb = S.lb; Q.ub = S.ub; Q.rowon = S.mask; Q.cstat_in = S.cs; Q.rstat_in = S.rs;
    Q.parent = use_parent ? S.parent : nullptr;
    Q.Binv = h->sx_binv[cur].as<double>(); Q.head = h->sx_head[cur].as<int32_t>();
    Q.stat = h->sx_stat[cur].as<int8_t>(); Q.wts = h->sx_wts[cur].as<double>();
    Q.pBinv = h->sx_binv[prev].as<double>(); Q.phead = h->sx_head[prev].as<int32_t>();
    Q.pstat = h->sx_stat[prev].as<int8_t>(); Q.pwts = h->sx_wts[prev].as<double>();
    Q.work = h->sx_work.as<double>(); Q.work_stride = stride;
    // The bounds and row masks stay with the store: blp_simplex_gmi_cuts_host reads a node's final bounds there.
    // Copied on every call, asked for or not: 2 B n doubles plus B (m - m_base) bytes, device to device, against
    // the B m^2 doubles of inverses the same call writes (at m = n = 500: 8 KB per node against 2 MB).
    const size_t mc = (size_t)(m - h->m_base);
    CK(h->sx_bnd[cur].ensure((size_t)2 * B * n * sizeof(double) + (size_t)B * mc));
    {
        double* bl = h->sx_bnd[cur].as<double>();
        CK(cudaMemcpyAsync(bl, S.lb, (size_t)B * n * sizeof(double), cudaMemcpyDeviceToDevice, st));
        CK(cudaMemcpyAsync(bl + (size_t)B * n, S.ub, (size_t)B * n * sizeof(double), cudaMemcpyDeviceToDevice, st));
        if (S.mask) CK(cudaMemcpyAsync(bl + (size_t)2 * B * n, S.mask, (size_t)B * mc, cudaMemcpyDeviceToDevice, st));
        h->sx_bnd_mask[cur] = S.mask != nullptr;
    }
    Q.obj = S.obj; Q.status = S.status; Q.pivots = S.pivots; Q.flips = S.flips;
    Q.x = S.x; Q.y = S.y; Q.rc = S.rc; Q.cstat_out = S.cso; Q.rstat_out = S.rso;
    CK(cudaEventRecord(h->ev[2], st));
    if (m <= kSxMaxRows) {
        const int threads = m <= 128 ? 128 : 512;
        k_simplex<<<B, threads, 0, st>>>(P, Q);
    } else {
        // one cooperative grid, one CTA per SM, split into G groups of S CTAs; group g solves nodes g, g + G, ...
        if (!h->coop_ok) return fail(BLP_ERR_STATE, "blp_simplex: LPs of more than %d rows need cooperative launches", kSxMaxRows);
        int occ = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_simplex_wide, 512, 0));
        if (occ < 1) return fail(BLP_ERR_STATE, "blp_simplex: k_simplex_wide does not fit an SM");
        // a tuning build forces G through BLP_SX_GROUPS, clamped to [1, min(B, SMs)]
        const int G = std::max(1, std::min(env_int("BLP_SX_GROUPS", sx_groups(m, B)), std::min(B, h->num_sms)));
        const int grid = G * (h->num_sms / G);
        if (grid > occ * h->num_sms) return fail(BLP_ERR_STATE, "blp_simplex: %d CTAs are not co-resident", grid);
        CK(h->sx_wide.ensure((size_t)G * kSxBarrierStride * sizeof(unsigned)));
        unsigned* counters = h->sx_wide.as<unsigned>();
        CK(cudaMemsetAsync(counters, 0, (size_t)G * kSxBarrierStride * sizeof(unsigned), st));  // the groups' arrival counters
        void* args[] = {(void*)&P, (void*)&Q, (void*)&G, (void*)&counters};
        CK(cudaLaunchCooperativeKernel((const void*)k_simplex_wide, dim3(grid), dim3(512), args, 0, st));
    }
    CK(cudaGetLastError());
    CK(cudaEventRecord(h->ev[3], st));
    if (obj) CK(cudaMemcpyAsync(obj, S.obj, B * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (status) CK(cudaMemcpyAsync(status, S.status, B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (pivots) CK(cudaMemcpyAsync(pivots, S.pivots, B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (x) CK(cudaMemcpyAsync(x, S.x, (size_t)B * n * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (y) CK(cudaMemcpyAsync(y, S.y, (size_t)B * m * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (rc) CK(cudaMemcpyAsync(rc, S.rc, (size_t)B * n * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (cso) CK(cudaMemcpyAsync(cso, S.cso, (size_t)B * n, cudaMemcpyDeviceToHost, st));
    if (rso) CK(cudaMemcpyAsync(rso, S.rso, (size_t)B * m, cudaMemcpyDeviceToHost, st));
    std::vector<int32_t> hp;
    if (stats) {
        hp.resize(2 * (size_t)B);
        CK(cudaMemcpyAsync(hp.data(), S.pivots, B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(hp.data() + B, S.flips, B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    }
    CK(cudaEventRecord(h->ev[1], st));
    CK(cudaStreamSynchronize(st));
    h->sx_cur = prev;                  // the store just written becomes "the last call"
    h->sx_last_B = B;
    h->sx_last_m = m;
    if (stats) {
        memset(stats, 0, sizeof *stats);
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]));
        stats->total_ms = ms;
        CK(cudaEventElapsedTime(&ms, h->ev[2], h->ev[3]));
        stats->step_kernel_ms = ms;
        double tot = 0.0;
        int mx = 0;
        for (int k = 0; k < B; ++k) { tot += hp[k]; mx = std::max(mx, hp[k]); }
        stats->iterations = mx;
        stats->node_iterations = tot;
        stats->kernel_launches = 1;
        int fl = 0;
        for (int k = 0; k < B; ++k) fl += hp[B + k];
        stats->refills = fl;           // bound flips of the ratio test (reported, not a refill count)
    }
    return BLP_OK;
}

int sx_check(blp_handle h, int B, const char* who) {
    if (!h) return fail(BLP_ERR_ARG, "%s: NULL handle", who);
    if (B < 1) return fail(BLP_ERR_ARG, "%s: need B >= 1", who);
    if (h->A0.rows > kSxMaxRowsWide)
        return fail(BLP_ERR_STATE, "%s: %d rows, the dense-inverse simplex takes at most %d (use blp_solve_batch)",
                    who, h->A0.rows, kSxMaxRowsWide);
    return BLP_OK;
}

}  // namespace

int blp_simplex_max_rows(void) { return kSxMaxRowsWide; }
int blp_simplex_batch_rows(void) { return kSxMaxRows; }

int blp_simplex_batch_host(blp_handle h, int B, const double* lb, const double* ub, const uint8_t* row_mask,
                           const int8_t* col_status, const int8_t* row_status, const int32_t* parent_slot,
                           int max_pivots, double* obj, int32_t* status, int32_t* pivots, double* x,
                           double* y, double* rc, int8_t* col_status_out, int8_t* row_status_out,
                           blp_stats* stats) {
    int rcode = sx_check(h, B, "blp_simplex_batch_host");
    if (rcode) return rcode;
    if (!lb || !ub) return fail(BLP_ERR_ARG, "blp_simplex_batch_host: lb/ub are NULL");
    if ((col_status == nullptr) != (row_status == nullptr))
        return fail(BLP_ERR_ARG, "blp_simplex_batch_host: col_status and row_status come together");
    if (max_pivots < 0) return fail(BLP_ERR_ARG, "blp_simplex_batch_host: max_pivots < 0");
    const size_t n = h->n, m = h->A0.rows, mc = m - h->m_base;
    bool use_parent = false;
    if (parent_slot) {
        for (int k = 0; k < B; ++k) {
            if (parent_slot[k] >= 0) use_parent = true;
            if (parent_slot[k] >= 0 && ((int)m != h->sx_last_m || parent_slot[k] >= h->sx_last_B))
                return fail(BLP_ERR_STATE, "blp_simplex_batch_host: parent_slot[%d] = %d does not name a node of the "
                                           "previous simplex call on this matrix", k, parent_slot[k]);
        }
    }
    CK(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    CK(cudaEventRecord(h->ev[0], st));
    SxStage S;
    if ((rcode = sx_carve(h, B, row_mask != nullptr, col_status != nullptr, use_parent, &S))) return rcode;
    CK(cudaMemcpyAsync(S.lb, lb, B * n * sizeof(double), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(S.ub, ub, B * n * sizeof(double), cudaMemcpyHostToDevice, st));
    if (S.mask) CK(cudaMemcpyAsync(S.mask, row_mask, B * mc, cudaMemcpyHostToDevice, st));
    if (S.cs) {
        CK(cudaMemcpyAsync(S.cs, col_status, B * n, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(S.rs, row_status, B * m, cudaMemcpyHostToDevice, st));
    }
    if (use_parent) CK(cudaMemcpyAsync(S.parent, parent_slot, B * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    return sx_run(h, B, S, use_parent, max_pivots, obj, status, pivots, x, y, rc, col_status_out, row_status_out, stats);
}

int blp_simplex_children_host(blp_handle h, int B, const double* parent_lb, const double* parent_ub,
                              const int32_t* delta_ptr, const int32_t* delta_var, const double* delta_lb,
                              const double* delta_ub, const uint8_t* row_mask, const int8_t* col_status,
                              const int8_t* row_status, int parent_slot, int max_pivots, double* obj,
                              int32_t* status, int32_t* pivots, double* x, double* y, double* rc,
                              int8_t* col_status_out, int8_t* row_status_out, blp_stats* stats) {
    int rcode = sx_check(h, B, "blp_simplex_children_host");
    if (rcode) return rcode;
    if (!parent_lb || !parent_ub || !delta_ptr)
        return fail(BLP_ERR_ARG, "blp_simplex_children_host: need parent bounds and delta_ptr");
    if ((col_status == nullptr) != (row_status == nullptr))
        return fail(BLP_ERR_ARG, "blp_simplex_children_host: col_status and row_status come together");
    if ((rcode = check_deltas(h, B, delta_ptr, delta_var, delta_lb, delta_ub, "blp_simplex_children_host"))) return rcode;
    const int nd = delta_ptr[B];
    if (max_pivots < 0) return fail(BLP_ERR_ARG, "blp_simplex_children_host: max_pivots < 0");
    const size_t n = h->n, m = h->A0.rows, mc = m - h->m_base;
    const bool use_parent = parent_slot >= 0;
    if (use_parent && ((int)m != h->sx_last_m || parent_slot >= h->sx_last_B))
        return fail(BLP_ERR_STATE, "blp_simplex_children_host: parent_slot %d does not name a node of the previous "
                                   "simplex call on this matrix", parent_slot);
    CK(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    CK(cudaEventRecord(h->ev[0], st));
    SxStage S;
    if ((rcode = sx_carve(h, B, row_mask != nullptr, col_status != nullptr, use_parent, &S))) return rcode;
    // parent vectors [lb | ub | cs | rs | mask] and deltas go up once, the per-node arrays are built on the device
    const size_t pbytes = 2 * n * sizeof(double) + n + m + mc + 64;
    CK(h->s_par.ensure(pbytes));
    char* pp = h->s_par.as<char>();
    double* d_plb = reinterpret_cast<double*>(pp);
    double* d_pub = d_plb + n;
    int8_t* d_pcs = reinterpret_cast<int8_t*>(d_pub + n);
    int8_t* d_prs = d_pcs + n;
    uint8_t* d_pmask = reinterpret_cast<uint8_t*>(d_prs + m);
    CK(cudaMemcpyAsync(d_plb, parent_lb, n * sizeof(double), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_pub, parent_ub, n * sizeof(double), cudaMemcpyHostToDevice, st));
    if (col_status) {
        CK(cudaMemcpyAsync(d_pcs, col_status, n, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(d_prs, row_status, m, cudaMemcpyHostToDevice, st));
    }
    if (S.mask) CK(cudaMemcpyAsync(d_pmask, row_mask, mc, cudaMemcpyHostToDevice, st));
    k_sx_expand_children<<<elementwise_grid((size_t)B * n), kCtaThreads, 0, st>>>(
        B, (int)n, (int)m, d_plb, d_pub, d_pcs, d_prs, d_pmask, (int)mc, S.lb, S.ub, S.cs, S.rs, S.mask);
    if (nd > 0) {
        DevDeltas d;
        if ((rcode = stage_deltas(h, B, delta_ptr, delta_var, delta_lb, delta_ub, &d))) return rcode;
        k_sx_patch_children<<<(B + 127) / 128, 128, 0, st>>>(B, (int)n, d.ptr, d.var, d.lb, d.ub, S.lb, S.ub);
    }
    if (use_parent) {
        std::vector<int32_t> par(B, parent_slot);
        CK(cudaMemcpyAsync(S.parent, par.data(), B * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        CK(cudaStreamSynchronize(st));      // `par` goes out of scope
    }
    CK(cudaGetLastError());
    rcode = sx_run(h, B, S, use_parent, max_pivots, obj, status, pivots, x, y, rc, col_status_out, row_status_out, stats);
    if (rcode == BLP_OK && stats) stats->kernel_launches += nd > 0 ? 2 : 1;
    return rcode;
}

int blp_simplex_tableau_rows_host(blp_handle h, int slot, int nrows, const int32_t* vars, double* out) {
    if (!h) return fail(BLP_ERR_ARG, "blp_simplex_tableau_rows_host: NULL handle");
    if (nrows < 1 || !vars || !out) return fail(BLP_ERR_ARG, "blp_simplex_tableau_rows_host: need nrows >= 1, vars, out");
    const int n = h->n, m = h->A0.rows, N = n + m;
    if (h->sx_last_m != m || slot < 0 || slot >= h->sx_last_B)
        return fail(BLP_ERR_STATE, "blp_simplex_tableau_rows_host: slot %d does not name a node of the previous simplex "
                                   "call on this matrix", slot);
    for (int t = 0; t < nrows; ++t)
        if (vars[t] < 0 || vars[t] >= N) return fail(BLP_ERR_ARG, "blp_simplex_tableau_rows_host: vars[%d] out of range", t);
    CK(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const int ldm = (m + 31) / 32 * 32;
    const int last = h->sx_cur ^ 1;
    CK(h->s_int.ensure((size_t)nrows * sizeof(int32_t)));
    CK(h->s_tmp.ensure((size_t)nrows * N * sizeof(double)));
    CK(cudaMemcpyAsync(h->s_int.p, vars, (size_t)nrows * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    SxProb P{m, h->m_base, n, ldm, h->P.rowptr, h->uent.as<Ent>(), h->P.cptr, h->ucent.as<Ent>(),
             h->uc.as<double>(), h->ub.as<double>()};
    k_simplex_tableau_rows<<<nrows, 256, 0, st>>>(P, h->sx_binv[last].as<double>() + (size_t)slot * m * ldm,
                                                  h->sx_head[last].as<int32_t>() + (size_t)slot * m, nrows,
                                                  h->s_int.as<int32_t>(), h->s_tmp.as<double>());
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, h->s_tmp.p, (size_t)nrows * N * sizeof(double), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return BLP_OK;
}

int blp_simplex_gmi_cuts_host(blp_handle h, int ncuts, const int32_t* slots, const int32_t* vars, const double* f0,
                              const uint8_t* col_is_int, double* pi, double* pi0, int32_t* code) {
    if (!h) return fail(BLP_ERR_ARG, "blp_simplex_gmi_cuts_host: NULL handle");
    if (ncuts < 1 || !slots || !vars || !f0 || !col_is_int || !pi || !pi0 || !code)
        return fail(BLP_ERR_ARG, "blp_simplex_gmi_cuts_host: need ncuts >= 1 and every array");
    const int n = h->n, m = h->A0.rows, N = n + m;
    if (h->sx_last_m != m)
        return fail(BLP_ERR_STATE, "blp_simplex_gmi_cuts_host: no simplex call on this matrix has its factors stored");
    for (int t = 0; t < ncuts; ++t) {
        if (slots[t] < 0 || slots[t] >= h->sx_last_B)
            return fail(BLP_ERR_STATE, "blp_simplex_gmi_cuts_host: slots[%d] = %d does not name a node of the previous "
                                       "simplex call", t, slots[t]);
        if (vars[t] < 0 || vars[t] >= N) return fail(BLP_ERR_ARG, "blp_simplex_gmi_cuts_host: vars[%d] out of range", t);
        if (!(f0[t] > 0.0 && f0[t] < 1.0)) return fail(BLP_ERR_ARG, "blp_simplex_gmi_cuts_host: f0[%d] not in (0, 1)", t);
    }
    CK(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const int ldm = (m + 31) / 32 * 32;
    const int last = h->sx_cur ^ 1;
    const size_t B = (size_t)h->sx_last_B;
    CK(h->sx_gmi.ensure((size_t)ncuts * (2 * sizeof(int32_t) + sizeof(double)) + (size_t)n + (size_t)ncuts * (n + 1) * sizeof(double) +
                        (size_t)ncuts * sizeof(int32_t) + 256 * 8));
    Carve cv{h->sx_gmi.as<char>()};
    int32_t* d_slot = cv.take<int32_t>(ncuts);
    int32_t* d_var = cv.take<int32_t>(ncuts);
    double* d_f0 = cv.take<double>(ncuts);
    uint8_t* d_int = cv.take<uint8_t>(n);
    double* d_pi = cv.take<double>((size_t)ncuts * n);
    double* d_pi0 = cv.take<double>(ncuts);
    int32_t* d_code = cv.take<int32_t>(ncuts);
    CK(cudaMemcpyAsync(d_slot, slots, ncuts * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_var, vars, ncuts * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_f0, f0, ncuts * sizeof(double), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_int, col_is_int, n, cudaMemcpyHostToDevice, st));
    SxProb P{m, h->m_base, n, ldm, h->P.rowptr, h->uent.as<Ent>(), h->P.cptr, h->ucent.as<Ent>(),
             h->uc.as<double>(), h->ub.as<double>()};
    const double* bnd = h->sx_bnd[last].as<double>();
    GmiArgs G{ncuts, h->sx_binv[last].as<double>(), h->sx_head[last].as<int32_t>(), h->sx_stat[last].as<int8_t>(),
              bnd, bnd + B * n, h->sx_bnd_mask[last] ? reinterpret_cast<const uint8_t*>(bnd + 2 * B * n) : nullptr,
              d_slot, d_var, d_f0, d_int, d_pi, d_pi0, d_code};
    const size_t smem = (size_t)2 * m * sizeof(double);
    if (smem > 48 * 1024) CK(cudaFuncSetAttribute(k_simplex_gmi_cuts, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_simplex_gmi_cuts<<<ncuts, kGmiThreads, smem, st>>>(P, G);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(pi, d_pi, (size_t)ncuts * n * sizeof(double), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(pi0, d_pi0, ncuts * sizeof(double), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(code, d_code, ncuts * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return BLP_OK;
}

int blp_stream_sync(blp_handle h) {
    if (!h) return fail(BLP_ERR_ARG, "blp_stream_sync: NULL handle");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    return BLP_OK;
}

int blp_comm_unique_id(char id[128]) {
    if (!id) return fail(BLP_ERR_ARG, "blp_comm_unique_id: id is NULL");
    NcclApi* a = nccl_api();
    if (!a) return fail(BLP_ERR_STATE, "blp_comm_unique_id: libnccl.so.2 not found (set BLP_NCCL_LIB)");
    NcclId u;
    const int rc = a->GetUniqueId(&u);
    if (rc) return nccl_fail(a, "ncclGetUniqueId", rc);
    memcpy(id, u.internal, 128);
    return BLP_OK;
}

int blp_comm_probe(blp_handle h) {
    if (!h) return fail(BLP_ERR_ARG, "blp_comm_probe: NULL handle");
    if (h->comm) return fail(BLP_ERR_STATE, "blp_comm_probe: the handle already has a communicator");
    if (!nccl_api()) return fail(BLP_ERR_STATE, "blp_comm_probe: libnccl.so.2 not found (set BLP_NCCL_LIB)");
    CK(cudaSetDevice(h->device));
    return BLP_OK;
}

int blp_comm_init(blp_handle h, int nranks, int rank, const char id[128]) {
    if (!h || !id) return fail(BLP_ERR_ARG, "blp_comm_init: NULL handle or id");
    if (nranks < 1 || rank < 0 || rank >= nranks) return fail(BLP_ERR_ARG, "blp_comm_init: rank %d of %d", rank, nranks);
    if (h->comm) return fail(BLP_ERR_STATE, "blp_comm_init: the handle already has a communicator");
    NcclApi* a = nccl_api();
    if (!a) return fail(BLP_ERR_STATE, "blp_comm_init: libnccl.so.2 not found (set BLP_NCCL_LIB)");
    CK(cudaSetDevice(h->device));
    NcclId u;
    memcpy(u.internal, id, 128);
    const int rc = a->CommInitRank(&h->comm, nranks, u, rank);
    if (rc) {
        h->comm = nullptr;
        return nccl_fail(a, "ncclCommInitRank", rc);
    }
    h->comm_ranks = nranks;
    if (!h->d_pair) CK(cudaMalloc(&h->d_pair, 2 * sizeof(double)));
    return BLP_OK;
}

int blp_allreduce_min(blp_handle h, double* two_vals) {
    if (!h || !two_vals) return fail(BLP_ERR_ARG, "blp_allreduce_min: NULL handle or values");
    if (!h->comm || h->comm_ranks == 1) return BLP_OK;        // a world of one rank: identity
    NcclApi* a = nccl_api();
    CK(cudaSetDevice(h->device));
    CK(cudaMemcpyAsync(h->d_pair, two_vals, 2 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    const int rc = a->AllReduce(h->d_pair, h->d_pair, 2, kNcclFloat64, kNcclMin, h->comm, h->stream);
    if (rc) return nccl_fail(a, "ncclAllReduce", rc);
    CK(cudaMemcpyAsync(two_vals, h->d_pair, 2 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return BLP_OK;
}

int blp_comm_destroy(blp_handle h) {
    if (!h) return fail(BLP_ERR_ARG, "blp_comm_destroy: NULL handle");
    if (h->comm) {
        cudaSetDevice(h->device);
        cudaStreamSynchronize(h->stream);
        NcclApi* a = nccl_api();
        if (a) a->CommDestroy(h->comm);
        h->comm = nullptr;
        h->comm_ranks = 1;
    }
    return BLP_OK;
}

int blp_destroy(blp_handle h) {
    if (!h) return BLP_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    blp_comm_destroy(h);
    if (h->d_pair) cudaFree(h->d_pair);
    h->drop_graphs();
    DevBuf* bufs[] = {&h->rowptr, &h->ent, &h->cptr, &h->cent, &h->c, &h->b,
                      &h->rowscale, &h->colscale, &h->d_dr, &h->d_dc, &h->uent, &h->ucent, &h->chunkC, &h->chunkR, &h->s_lb,
                      &h->s_ub, &h->s_x0, &h->s_y0, &h->s_mask, &h->s_x, &h->s_y, &h->s_tmp,
                      &h->s_ws, &h->s_node, &h->s_int, &h->s_delta, &h->s_par, &h->uc, &h->ub,
                      &h->sx_binv[0], &h->sx_binv[1], &h->sx_head[0], &h->sx_head[1], &h->sx_stat[0],
                      &h->sx_stat[1], &h->sx_wts[0], &h->sx_wts[1], &h->sx_work, &h->sx_in, &h->sx_out, &h->sx_wide,
                      &h->sx_bnd[0], &h->sx_bnd[1], &h->sx_gmi};
    for (DevBuf* b : bufs) b->release();
    for (cudaEvent_t e : h->ev) if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : h->ev_join) if (e) cudaEventDestroy(e);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    for (cudaStream_t s : h->side) if (s) cudaStreamDestroy(s);
    for (cudaEvent_t e : h->prof_ev) cudaEventDestroy(e);
    if (h->h_counters) cudaFreeHost(h->h_counters);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return BLP_OK;
}

}  // extern "C"
