// Device kernels of the batched node-LP bound step (sm_100a, fp64, no tensor cores).
//
// Layout: the CALLER's batched vectors are node-fastest, V[row][ld]. The solver's own state is
// tile-major: nodes are grouped in blocks of 64 and element (row j, node k) lives at
// ((k / 64) * rows + j) * 64 + k % 64 (tix()), so the 512-byte segments a node block touches in
// consecutive rows are contiguous in HBM. A warp owns one matrix row (or 32/NT rows) for a tile of
// nodes, so every state access of a warp is one contiguous segment and the CSR entries of a row
// are warp-uniform. Work is ordered tile-major (blockIdx.y = tile, blockIdx.x = row chunk) so the
// CTAs resident at any moment share a few node tiles and the gathered vector of those tiles is
// served from L2 after its first (compulsory) read from HBM.
//
// Algorithm: reflected, restarted Halpern PDHG. With T the PDHG map
//     x' = clip(x - tau (c - A'y), l, u),   y' = max(0, y + sigma (b - A (2x' - x)))
// one step is  z+ = w (2 T(z) - z) + (1 - w) z_anchor,  w = (s+1)/(s+2), s = steps since restart.
// State kept per node column: xbar = 2x' - x (gathered by the dual step; the next primal step
// rebuilds x = w xbar + (1-w) xa from it), xa, l, u (+ block reference bounds and masks), y, ya.
#pragma once
#include <cstdint>
#include <cooperative_groups.h>
#include <cuda_runtime.h>

namespace blp {

#ifndef BLP_U
#define BLP_U 4          // gathers issued back to back per row batch
#endif
#ifndef BLP_MINB
#define BLP_MINB 6       // resident CTAs per SM the step kernels are compiled for
#endif
// Halpern anchors xa, ya are stored in fp32 (BLP_ANCHOR32=1). Any fixed point a is a valid Halpern
// anchor (z+ = w R(z) + (1-w) a converges to a fixed point of R for every a); a restart therefore
// sets the anchor to the fp32 rounding of the restart point and keeps the current point in fp64.
// The iterates stay within |a - z0| / (k+1) of the sequence anchored at z0 itself. Saves 4 of the
// 8 anchor bytes read per state element and iteration.
#ifndef BLP_ANCHOR32
#define BLP_ANCHOR32 1
#endif
#if BLP_ANCHOR32
using anc_t = float;
using anc2_t = float2;
#else
using anc_t = double;
using anc2_t = double2;
#endif
constexpr int kCtaThreads = 256;
constexpr int kBlk = 64;      // nodes per layout block (row stride of a lane's column, in doubles)
constexpr int kWarps = kCtaThreads / 32;

// column-pass accumulators (sums first, then maxima)
enum { C_DX2, C_CROSS, C_DRES2, C_CX, C_BND, C_DXA2, C_BOX, C_BOXABS, C_CD, C_DBOX, C_DBOXABS, C_NSUM,
       C_DMAX = C_NSUM, C_DVIOL, C_RAYVIOL, C_DRAYVIOL, C_N };
// row-pass accumulators
enum { R_PRES2, R_BY, R_DY2, R_DYA2, R_BYABS, R_BD, R_BDABS, R_NSUM,
       R_ADNEG = R_NSUM, R_YMAX, R_DYMAX, R_DYNEG, R_N };

// one stored matrix entry; 16 bytes so that a row walk is one 128-bit load per nonzero
struct __align__(16) Ent {
    int32_t idx;
    int32_t pad;
    double val;
};

struct DevProb {
    int m, m_base, n, nnz;
    const int32_t* rowptr; const Ent* ent;       // scaled A   (m x n), CSR
    const int32_t* cptr;   const Ent* cent;      // scaled A^T (n x m), CSR
    const double* c; const double* b;            // scaled objective / row lower bounds
    const double* rowscale; const double* colscale;   // scaled residual -> unscaled
    const double* dr; const double* dc;
    double eta, sb, sc, objscale, bnorm0, cnorm0, cinf_s, omega0;
    double bcut2;          // sum of squares of the (unscaled) right-hand sides of ALL appended rows
};

// Work list of a frozen-path step kernel for every 64-node tile (k_work_*, rebuilt once per evaluation period): the
// rows that are not frozen for the tile (ACTIVE rows), those of more than kLongRow stored entries first, then the
// others, each group in ascending row order; their kept entries packed in that order; one record of row scalars per
// active row; and one header per (tile, chunk) of the launch grid. Rows of the step kernel: columns of A (primal,
// rows = n) or rows of A (dual, rows = m).
struct WorkList {
    int2* row;       // [tile][rows + 1] active row k: {row id, start of its entries in ent}; k = count: {-1, end}
    Ent* ent;        // [tile][nnz]
    int4* rec;       // [tile][rows][kPrimalRowBytes / 16 or kDualRowBytes / 16] row scalars (primal_rec / dual_rec)
    int4* chunk;     // [tile][rows] chunk header {first active row, rows (-1: one long row), first entry, end entry}
    int32_t* kept;   // [tile][rows] kept entries of a row, -1 = frozen (k_work_count; k_work_scan's scratch)
    int32_t* count;  // [tile] active rows
};

struct DevState {
    int B, ld;
    double *xbar, *l, *u, *X1, *DX, *G;            // [n][ld]
    double *y, *Y1, *DY;                           // [m][ld]
    anc_t *xa, *ya;                                // [n][ld], [m][ld] Halpern anchors
    uint8_t* rowmask;                              // [m - m_base][ld] (workspace copy) or null
    double *omega, *fpe0, *fpe_prev, *pobj, *dobj; // [ld]
    int32_t *sbase, *fin, *status, *iters, *restart;   // [ld]
    int32_t *origin, *newpos;                      // [ld] caller's node id of a column; compaction map
    int32_t *start, *fresh, *newlist;              // [ld] iteration count at which the slot's node was loaded;
                                                   //      1 = loaded by the last refill; slots of that refill
    double *partC, *partR;                         // [chunks][C_N][ld], [chunks][R_N][ld]
    double* fracD; int32_t* fracI;                 // [chunks][ld] most-fractional partials
    const uint8_t* isint;                          // [n] 1 = integer column, or null
    double* dbg;                                   // [ld][8] per-node trace of the last evaluation, or null
    // bounds of a 32-node block are mostly identical (nodes differ from the root in a few entries):
    // lref/uref hold the block's reference bound per row, lumask the nodes that deviate from it;
    // the primal step reads the dense l,u of a row only for those nodes. Layout [block][row].
    double *lref, *uref;
    uint32_t* lumask;
    int32_t* counters;                             // see k_tick; [8..11] = two 64-bit counts of k_freeze_count
    // Frozen coordinates (k_freeze_cols / k_freeze_rows): one byte per (32-node block, row), layout
    // [block][row] like lref; 1 = every running node of the block agrees that the coordinate rests.
    uint8_t *cfrz, *rfrz;
    // Folded matrices of a 64-node tile: the entries the step kernels still have to gather once the frozen
    // coordinates are taken out, as work lists (k_work_*). A folded column's contribution to a row of A is summed
    // into the row's rconst (the dual record's second scalar) once per evaluation period.
    double* cval;                                  // [block][n] x' of a frozen column if the block's nodes agree on it
    uint8_t* fcol; double* fval;                   // [tile][n] column folded into rconst, with the value it rests at
    WorkList wlC, wlR;                             // primal step (rows of A'), dual step (rows of A)
    // Step size of a node (k_pow_*): eta = P.eta = 0.998 / ||A|| unless its tile has frozen coordinates, then up to
    // safety / ||A_UU||, A_UU = the rows and columns of the tile that still move.
    double* eta; int32_t* eta_lock;                // [ld] current step; 1 = the watchdog sent the node back to P.eta
    uint8_t *ftc, *ftr;                            // [tile][n], [tile][m] 1 = frozen for the tile
    double *pv, *pw;                               // [tile][n], [tile][m] power-iteration vectors
    double *ppart, *eta_tile;                      // [tile][kPowChunks] partial ||v||^2; [tile] step the tile allows
};
constexpr int kPowChunks = 32;

// Margins of the freezing rule in the scaled problem's units (blp.cu: solve set-up).
struct FreezeArgs {
    double c_lo, c_hi;      // reduced-cost margin below which a frozen column is released / above which it freezes
    double r_lo, r_hi;      // the same for the slack of a row with zero multiplier
};

// caller-side output arrays (node-fastest, leading dimension ld; entries indexed by ORIGINAL node)
struct DevOut {
    double *obj, *lower, *x, *y;
    int32_t *status, *iters, *frac_idx;
    int ld;                                        // leading dimension of the caller's arrays
};

__device__ __forceinline__ bool is_inf(double v) { return fabs(v) >= 1e30; }

// tile-major index of (row, node) in an internal [rows] x [ld] state array
__device__ __forceinline__ size_t tix(const int row, const int node, const int rows) {
    return ((size_t)(node >> 6) * rows + row) * kBlk + (node & (kBlk - 1));
}

// ---------------------------------------------------------------------------------------------
// gather-dot of one CSR row with a batched vector: sum_p val[p] * V[idx[p]][node]
// NT == 32: the row is warp-uniform, so every lane issues the same 128-bit entry load (one
// broadcast wavefront) and then its own coalesced 8-byte gather; 4 entries are in flight at once.
// NT < 32: every lane walks the row of its own sub-group.
template <int NT>
__device__ __forceinline__ double row_dot(const int32_t* __restrict__ ptr,
                                          const Ent* __restrict__ ent, int row, bool row_ok,
                                          const double* __restrict__ Vn, bool node_ok) {
    // Vn: the lane's column inside a tile-major state array (row stride 32 doubles)
    constexpr int ld = kBlk;
    double acc = 0.0;
    if (NT == 32 || (row_ok && node_ok)) {
        const int p0 = __ldg(ptr + row), p1 = __ldg(ptr + row + 1);
        int p = p0;
        for (; p + 4 <= p1; p += 4) {
            const int4 e0 = __ldg(reinterpret_cast<const int4*>(ent + p));
            const int4 e1 = __ldg(reinterpret_cast<const int4*>(ent + p + 1));
            const int4 e2 = __ldg(reinterpret_cast<const int4*>(ent + p + 2));
            const int4 e3 = __ldg(reinterpret_cast<const int4*>(ent + p + 3));
            double v0 = 0, v1 = 0, v2 = 0, v3 = 0;
            if (node_ok) {
                v0 = Vn[(size_t)e0.x * ld];
                v1 = Vn[(size_t)e1.x * ld];
                v2 = Vn[(size_t)e2.x * ld];
                v3 = Vn[(size_t)e3.x * ld];
            }
            acc = fma(__hiloint2double(e0.w, e0.z), v0, acc);
            acc = fma(__hiloint2double(e1.w, e1.z), v1, acc);
            acc = fma(__hiloint2double(e2.w, e2.z), v2, acc);
            acc = fma(__hiloint2double(e3.w, e3.z), v3, acc);
        }
        for (; p < p1; ++p) {
            const int4 e = __ldg(reinterpret_cast<const int4*>(ent + p));
            const double v = node_ok ? Vn[(size_t)e.x * ld] : 0.0;
            acc = fma(__hiloint2double(e.w, e.z), v, acc);
        }
    }
    return acc;
}

// The same walk for TWO batched vectors at once (the evaluation's A x' and A d): one pass over the
// row's entries, eight gathers in flight, so a 400-entry cut row costs 50 dependent round trips
// per evaluation instead of 200.
template <int NT>
__device__ __forceinline__ void row_dot_pair(const int32_t* __restrict__ ptr, const Ent* __restrict__ ent,
                                             int row, bool row_ok, const double* __restrict__ Vn,
                                             const double* __restrict__ Wn, bool node_ok, double& accv,
                                             double& accw) {
    constexpr int ld = kBlk;
    accv = 0.0;
    accw = 0.0;
    if (NT == 32 || (row_ok && node_ok)) {
        const int p0 = __ldg(ptr + row), p1 = __ldg(ptr + row + 1);
        for (int p = p0; p < p1; p += 4) {
            int4 e[4];
            double v[4], w[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                v[q] = 0.0;
                w[q] = 0.0;
                e[q] = make_int4(0, 0, 0, 0);
                if (p + q < p1) {
                    e[q] = __ldg(reinterpret_cast<const int4*>(ent + p + q));
                    if (node_ok) {
                        v[q] = Vn[(size_t)e[q].x * ld];
                        w[q] = Wn[(size_t)e[q].x * ld];
                    }
                }
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const double cf = __hiloint2double(e[q].w, e[q].z);
                accv = fma(cf, v[q], accv);
                accw = fma(cf, w[q], accw);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Row slab of a CTA in shared memory. The step kernels give every CTA a contiguous chunk of CSR
// rows; all 256 threads first copy the chunk's row pointers and (when they fit) its entries with
// coalesced 128-bit loads. A row walk then costs one shared-memory read per nonzero, and the only
// global round trip on a warp's critical path is the one that matters: the streaming loads and
// the gathers of the batched vector, all issued together.
struct Slab {
    const int* sp;       // shared: absolute row pointers of rows r0 .. r1
    const int4* se;      // shared: entries [sp[0], sp[nrows]) or nullptr if they did not fit
    int base;
};

extern __shared__ int4 dyn_smem[];

// Per-row scalars a slab stage can copy to shared memory along with the row pointers: rs(j, slot) loads
// those of global row j and stores them at `slot` (the row's place in the CTA's work list).
struct NoRowScalars {
    __device__ __forceinline__ void operator()(int, int) const {}
};

template <class RS = NoRowScalars>
__device__ __forceinline__ Slab stage_slab(const int32_t* __restrict__ ptr,
                                           const Ent* __restrict__ ent, const int r0, const int r1,
                                           const int rows_per_cta, const int cap,
                                           int4* const smem_base = dyn_smem, const RS rs = RS()) {
    int* sp = reinterpret_cast<int*>(smem_base);
    int4* se = smem_base + (rows_per_cta + 4) / 4;
    const int nrows = r1 - r0;
    for (int t = threadIdx.x; t <= nrows; t += kCtaThreads) {
        sp[t] = __ldg(ptr + r0 + t);
        if (t < nrows) rs(r0 + t, t);
    }
    __syncthreads();
    Slab s;
    s.sp = sp;
    s.base = sp[0];
    s.se = nullptr;
    const int cnt = sp[nrows] - s.base;
    if (cnt <= cap) {
        const int4* __restrict__ src = reinterpret_cast<const int4*>(ent) + s.base;
        for (int t = threadIdx.x; t < cnt; t += kCtaThreads) se[t] = __ldg(src + t);
        __syncthreads();
        s.se = se;
    }
    return s;
}

template <bool SHARED>
__device__ __forceinline__ double dot_entries(const int4* __restrict__ E, const int p0, const int p1,
                                              const double* __restrict__ Vn, const int ld,
                                              const bool node_ok) {
    // ld: distance (in doubles) between consecutive rows of the gathered vector for this lane.
    // kU gathers are issued back to back before the first one is consumed: the row's critical
    // path is one memory round trip per kU nonzeros. Only the column index is kept in a register
    // while the gathers fly; the coefficient is re-read (shared memory / L1) at the multiply.
    constexpr int kU = BLP_U;
    double acc = 0.0;
    for (int p = p0; p < p1; p += kU) {
        double v[kU];
#pragma unroll
        for (int q = 0; q < kU; ++q) {
            v[q] = 0.0;
            if (p + q < p1) {
                const int col = SHARED ? E[p + q].x : __ldg(&E[p + q].x);
                if (node_ok) v[q] = Vn[(size_t)col * ld];
            }
        }
#pragma unroll
        for (int q = 0; q < kU; ++q)
            if (p + q < p1) {
                const int2 c = SHARED ? *reinterpret_cast<const int2*>(&E[p + q].z)
                                      : __ldg(reinterpret_cast<const int2*>(&E[p + q].z));
                acc = fma(__hiloint2double(c.y, c.x), v[q], acc);
            }
    }
    return acc;
}

// gather-dot of local row lr of the slab; NT == 32: warp-uniform row, NT < 32: one row per sub-group
template <int NT>
__device__ __forceinline__ double slab_dot(const Slab& sl, const Ent* __restrict__ ent, const int lr,
                                           const bool row_ok, const double* __restrict__ Vn,
                                           const int ld, const bool node_ok) {
    if (NT != 32 && !(row_ok && node_ok)) return 0.0;
    const int p0 = sl.sp[lr], p1 = sl.sp[lr + 1];
    if (sl.se) return dot_entries<true>(sl.se - sl.base, p0, p1, Vn, ld, node_ok);
    return dot_entries<false>(reinterpret_cast<const int4*>(ent), p0, p1, Vn, ld, node_ok);
}

// A chunk that consists of ONE long row (a dense cut row, typically) is shared by all threads of
// the CTA in the one-node-per-lane kernels too: thread t gathers the entries p0 + t / NT,
// p0 + t / NT + 256 / NT, ... for node t % NT (the NT threads of a slice read NT consecutive
// doubles), the partial sums meet in shared memory and are folded in slice order, so the result is
// deterministic. Without it one warp walks the row alone: 400 entries = 100 dependent round trips,
// which made every iteration of a NARROW batch with cut rows 1.5x slower (BASELINE.md, config 4).
// Returns the dot for node (cy * NT + t % NT) in the threads t < NT, which are the lanes that own
// row r0 in the regular mapping (warp 0, sub-group 0).
constexpr int kLongRow = 96;

template <int NT>
__device__ __forceinline__ double coop_dot_nt(const Slab& sl, const Ent* __restrict__ ent,
                                              const double* __restrict__ V, const int rows_v,
                                              const int cy, const DevState& S) {
    constexpr int NS = kCtaThreads / NT;                      // slices of the row
    __shared__ double red[kCtaThreads];
    const int nl = threadIdx.x % NT, slice = threadIdx.x / NT;
    const int node = cy * NT + nl;
    const bool ok = node < S.B && S.fin[node] == 0;
    const double* __restrict__ Vn = V + tix(0, ok ? node : cy * NT, rows_v);
    const int p0 = sl.sp[0], p1 = sl.sp[1];
    const int4* __restrict__ E = sl.se ? sl.se - sl.base : reinterpret_cast<const int4*>(ent);
    double acc = 0.0;
    for (int p = p0 + slice; p < p1; p += 4 * NS) {            // four independent gathers in flight
        double v[4], cf[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int pq = p + q * NS;
            v[q] = 0.0;
            cf[q] = 0.0;
            if (pq < p1) {
                const int4 e = sl.se ? E[pq] : __ldg(E + pq);
                cf[q] = __hiloint2double(e.w, e.z);
                v[q] = Vn[(size_t)e.x * kBlk];
            }
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) acc = fma(cf[q], v[q], acc);
    }
    red[threadIdx.x] = acc;
    __syncthreads();
    double r = 0.0;
    if (threadIdx.x < NT)
        for (int q = 0; q < NS; ++q) r += red[q * NT + threadIdx.x];
    return r;
}

// ---------------------------------------------------------------------------------------------
// Primal half step, fused  G = A'y  ->  x' = clip(x - tau (c - G), l, u)  ->  xbar = 2x' - x.
template <int NT, bool MAJOR>
__device__ __forceinline__ void primal_chunk(const DevProb& P, const DevState& S, const int it,
                                             const int rows_per_cta, const int cap,
                                             const int* __restrict__ chunk_ptr, const int cx, const int cy,
                                             const Slab* pre = nullptr) {
    constexpr int RW = 32 / NT;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int node = cy * NT + (lane % NT);
    const int sub = lane / NT;
    const bool node_ok = node < S.B && S.fin[node] == 0;
    if (__ballot_sync(0xffffffffu, node_ok) == 0) return;     // whole node tile retired
    double w = 0.0, tau = 0.0;
    if (node_ok) {
        const int s = S.sbase[node] + it;
        w = (double)s / (double)(s + 1);
        tau = S.eta[node] / S.omega[node];
    }
    const int r0 = __ldg(chunk_ptr + 2 * cx);              // chunk cx = rows [r0, r1); heaviest chunks first
    const int r1 = __ldg(chunk_ptr + 2 * cx + 1);
    const Slab sl = pre ? *pre : stage_slab(P.cptr, P.cent, r0, r1, rows_per_cta, cap);
    const double* __restrict__ yn = S.y + tix(0, node, P.m);
    const bool coop = (r1 - r0 == 1) && (sl.sp[1] - sl.sp[0] > kLongRow);
    double cg = 0.0;
    if (coop) {
        cg = coop_dot_nt<NT>(sl, P.cent, S.y, P.m, cy, S);
        if (threadIdx.x >= NT) return;
    }
    for (int jb = r0 + warp * RW; jb < r1; jb += kWarps * RW) {
        const int j = jb + sub;
        const bool row_ok = j < r1;
        const size_t e = tix(j, node, P.n);
        double xb = 0, a = 0, lo = 0, hi = 0;
        if (row_ok && node_ok) {       // streaming loads first, the gathers follow at once
            xb = S.xbar[e];
            a = (double)__ldcs(S.xa + e);
            const size_t fi = (size_t)(node >> 5) * P.n + j;
            const uint32_t mk = __ldg(S.lumask + fi);
            if ((mk >> (node & 31)) & 1u) {
                lo = __ldcs(S.l + e);
                hi = __ldcs(S.u + e);
            } else {
                lo = __ldg(S.lref + fi);
                hi = __ldg(S.uref + fi);
            }
        }
        const double g = coop ? cg : slab_dot<NT>(sl, P.cent, row_ok ? j - r0 : 0, row_ok, yn, kBlk, node_ok && row_ok);
        if (row_ok && node_ok) {
            const double xc = fma(w, xb - a, a);                  // w xbar + (1-w) xa
            const double xp = fmin(fmax(xc - tau * (__ldg(P.c + j) - g), lo), hi);
            S.xbar[e] = 2.0 * xp - xc;
            if constexpr (MAJOR) {
                S.X1[e] = xp;
                S.DX[e] = xp - xc;
                S.G[e] = g;
            }
        }
    }
}

template <int NT, bool MAJOR>
__global__ void __launch_bounds__(kCtaThreads, BLP_MINB)
k_primal(const DevProb P, const DevState S, const int it, const int rows_per_cta, const int cap,
         const int* __restrict__ chunk_ptr) {
    primal_chunk<NT, MAJOR>(P, S, it, rows_per_cta, cap, chunk_ptr, blockIdx.x, blockIdx.y);
}

// Dual half step, fused  s = A xbar  ->  y' = max(0, y + sigma (b - s))  ->  Halpern update of y.
template <int NT, bool MAJOR>
__device__ __forceinline__ void dual_chunk(const DevProb& P, const DevState& S, const int it,
                                           const int rows_per_cta, const int cap,
                                           const int* __restrict__ chunk_ptr, const int cx, const int cy,
                                           const Slab* pre = nullptr) {
    constexpr int RW = 32 / NT;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int node = cy * NT + (lane % NT);
    const int sub = lane / NT;
    const bool node_ok = node < S.B && S.fin[node] == 0;
    if (__ballot_sync(0xffffffffu, node_ok) == 0) return;     // whole node tile retired
    double w = 0.0, sig = 0.0;
    if (node_ok) {
        const int s = S.sbase[node] + it;
        w = (double)(s + 1) / (double)(s + 2);
        sig = S.eta[node] * S.omega[node];
    }
    const int r0 = __ldg(chunk_ptr + 2 * cx);              // chunk cx = rows [r0, r1); heaviest chunks first
    const int r1 = __ldg(chunk_ptr + 2 * cx + 1);
    const Slab sl = pre ? *pre : stage_slab(P.rowptr, P.ent, r0, r1, rows_per_cta, cap);
    const double* __restrict__ xn = S.xbar + tix(0, node, P.n);
    const bool coop = (r1 - r0 == 1) && (sl.sp[1] - sl.sp[0] > kLongRow);
    double cg = 0.0;
    if (coop) {
        cg = coop_dot_nt<NT>(sl, P.ent, S.xbar, P.n, cy, S);
        if (threadIdx.x >= NT) return;
    }
    for (int ib = r0 + warp * RW; ib < r1; ib += kWarps * RW) {
        const int i = ib + sub;
        const bool row_ok = i < r1;
        const size_t e = tix(i, node, P.m);
        double yc = 0, a = 0;
        bool on = true;
        if (row_ok && node_ok) {
            yc = S.y[e];
            a = (double)__ldcs(S.ya + e);
            if (i >= P.m_base && S.rowmask) on = S.rowmask[(size_t)(i - P.m_base) * S.ld + node] != 0;
        }
        const double ax = coop ? cg : slab_dot<NT>(sl, P.ent, row_ok ? i - r0 : 0, row_ok, xn, kBlk, node_ok && row_ok);
        if (row_ok && node_ok) {
            const double yp = on ? fmax(0.0, yc + sig * (__ldg(P.b + i) - ax)) : 0.0;
            S.y[e] = fma(w, (2.0 * yp - yc) - a, a);
            if constexpr (MAJOR) {
                S.Y1[e] = yp;
                S.DY[e] = yp - yc;
            }
        }
    }
}

template <int NT, bool MAJOR>
__global__ void __launch_bounds__(kCtaThreads, BLP_MINB)
k_dual(const DevProb P, const DevState S, const int it, const int rows_per_cta, const int cap,
       const int* __restrict__ chunk_ptr) {
    dual_chunk<NT, MAJOR>(P, S, it, rows_per_cta, cap, chunk_ptr, blockIdx.x, blockIdx.y);
}

// One whole evaluation period (K iterations) of a NARROW batch as a single cooperative launch:
// the grid loops over the (row chunk, node tile) work items of the primal step, meets at a grid
// barrier, does the dual step, meets again. Two launches per iteration cost ~20 us when only a
// few nodes are running (tiny LPs, the tail of a batch); two grid barriers cost a few.
// The gpu-scope fence inside grid.sync() also drops stale L1 lines of the vectors other CTAs wrote.
struct CoopPlan {
    int rpcC, capC, nchC, rpcR, capR, nchR, tiles;
    const int* chunkC;
    const int* chunkR;
};

template <int NT>
__global__ void __launch_bounds__(kCtaThreads, 4)
k_period_coop(const DevProb P, const DevState S, const int K, const CoopPlan C) {
    cooperative_groups::grid_group grid = cooperative_groups::this_grid();
    // the launch gives every CTA at most one primal and one dual work item; their row slabs are
    // staged in shared memory once and serve all K iterations
    const int w = blockIdx.x;
    const bool hasC = w < C.nchC * C.tiles, hasR = w < C.nchR * C.tiles;
    const int cxC = w % C.nchC, cyC = w / C.nchC, cxR = w % C.nchR, cyR = w / C.nchR;
    Slab slC{nullptr, nullptr, 0}, slR{nullptr, nullptr, 0};
    int4* const baseR = dyn_smem + (C.rpcC + 4) / 4 + C.capC;
    if (hasC) slC = stage_slab(P.cptr, P.cent, __ldg(C.chunkC + 2 * cxC), __ldg(C.chunkC + 2 * cxC + 1), C.rpcC, C.capC);
    if (hasR) slR = stage_slab(P.rowptr, P.ent, __ldg(C.chunkR + 2 * cxR), __ldg(C.chunkR + 2 * cxR + 1), C.rpcR, C.capR, baseR);
    for (int it = 0; it < K; ++it) {
        const bool major = it == K - 1;
        if (hasC) {
            if (major) primal_chunk<NT, true>(P, S, it, C.rpcC, C.capC, C.chunkC, cxC, cyC, &slC);
            else primal_chunk<NT, false>(P, S, it, C.rpcC, C.capC, C.chunkC, cxC, cyC, &slC);
        }
        grid.sync();
        if (hasR) {
            if (major) dual_chunk<NT, true>(P, S, it, C.rpcR, C.capR, C.chunkR, cxR, cyR, &slR);
            else dual_chunk<NT, false>(P, S, it, C.rpcR, C.capR, C.chunkR, cxR, cyR, &slR);
        }
        grid.sync();
    }
}

// ---------------------------------------------------------------------------------------------
// Two-nodes-per-lane step kernels (batches of >= 64 nodes). A warp owns one matrix row for a
// whole 64-node block: every state access is one 128-bit load/store per lane (512 contiguous
// bytes per warp), and the per-row instruction overhead (index arithmetic, entry reads, loop
// control) is spent once per 64 nodes instead of once per 32 — the one-node-per-lane kernels
// issue ~170 instructions per row and are issue-bound, not bandwidth-bound
// (profiles/r1b_full_step_kernels.md).
#ifndef BLP_MINB2
#define BLP_MINB2 5
#endif

__device__ __forceinline__ double2 ld2(const double* p) { return *reinterpret_cast<const double2*>(p); }
__device__ __forceinline__ double2 ldcs2(const double* p) {
    return __ldcs(reinterpret_cast<const double2*>(p));
}
__device__ __forceinline__ double2 ldcs2(const float* p) {     // two fp32 anchors, widened
    const float2 v = __ldcs(reinterpret_cast<const float2*>(p));
    return make_double2((double)v.x, (double)v.y);
}
__device__ __forceinline__ void st2(double* p, const double2 v, const bool k0, const bool k1) {
    if (k0 && k1) *reinterpret_cast<double2*>(p) = v;
    else if (k0) p[0] = v.x;
    else if (k1) p[1] = v.y;
}

// ld: distance (in doubles) between consecutive rows of the gathered vector (kBlk for the solver's
// tile-major state, the caller's leading dimension for blp_spmv). Row col of the lane's column is at
// Vn + off + col * ld, computed in the index type I (the step kernels use 32 bits, see k_primal2).
// PAD = false leaves the slots of a batch past the row's end unset (they are never read): at 48 registers that
// is what lets the step kernels keep a full batch of gathers in flight (k_spmv2 spills without the padding).
template <bool SHARED, class I = size_t, bool PAD = true>
__device__ __forceinline__ void dot2_entries(const int4* __restrict__ E, const int p0, const int p1,
                                             const double* __restrict__ Vn, double& g0, double& g1,
                                             const int ld = kBlk, const I off = 0) {
    constexpr int kU = BLP_U;
#pragma unroll 1
    for (int p = p0; p < p1; p += kU) {
        double2 v[kU];
#pragma unroll
        for (int q = 0; q < kU; ++q) {
            if (PAD) v[q] = make_double2(0.0, 0.0);
            if (p + q < p1) {
                const int col = SHARED ? E[p + q].x : __ldg(&E[p + q].x);
                v[q] = ld2(Vn + (off + (I)col * (I)ld));
            }
        }
#pragma unroll
        for (int q = 0; q < kU; ++q)
            if (p + q < p1) {
                const int2 c = SHARED ? *reinterpret_cast<const int2*>(&E[p + q].z)
                                      : __ldg(reinterpret_cast<const int2*>(&E[p + q].z));
                const double cf = __hiloint2double(c.y, c.x);
                g0 = fma(cf, v[q].x, g0);
                g1 = fma(cf, v[q].y, g1);
            }
    }
}

__device__ __forceinline__ void slab_dot2(const Slab& sl, const Ent* __restrict__ ent, const int lr,
                                          const double* __restrict__ Vn, double& g0, double& g1,
                                          const int ld = kBlk) {
    const int p0 = sl.sp[lr], p1 = sl.sp[lr + 1];
    if (sl.se) dot2_entries<true>(sl.se - sl.base, p0, p1, Vn, g0, g1, ld);
    else dot2_entries<false>(reinterpret_cast<const int4*>(ent), p0, p1, Vn, g0, g1, ld);
}

// A chunk that consists of ONE long row (a dense cut row, typically) is shared by all warps of the
// CTA: each warp gathers a slice of the row's entries, the partial sums meet in shared memory.

__device__ __forceinline__ void coop_dot2(const Slab& sl, const Ent* __restrict__ ent, const int p0, const int p1,
                                          const double* __restrict__ Vn, const int warp, const int lane,
                                          double& g0, double& g1) {
    __shared__ double2 red[kWarps][32];
    const int seg = ((p1 - p0 + kWarps - 1) / kWarps + BLP_U - 1) / BLP_U * BLP_U;
    const int a = min(p1, p0 + warp * seg), b = min(p1, a + seg);
    double s0 = 0.0, s1 = 0.0;
    if (sl.se) dot2_entries<true>(sl.se - sl.base, a, b, Vn, s0, s1);
    else dot2_entries<false>(reinterpret_cast<const int4*>(ent), a, b, Vn, s0, s1);
    red[warp][lane] = make_double2(s0, s1);
    __syncthreads();
    g0 = 0.0;
    g1 = 0.0;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) {
        g0 += red[w][lane].x;
        g1 += red[w][lane].y;
    }
}

// Rows of a frozen-path CTA's chunk as in its work list, {row id, start of its entries} (stage_work): a trip reads
// both with one 64-bit load, and the end of its entries from the next row.
constexpr int kMaxChunkRows = 512;
__shared__ int2 s_row[kMaxChunkRows + 1];

// What a warp's trip over one row reads besides the row's state and gathers, staged with the slab (no round trip of
// its own) and read from shared memory after the gathers are issued. At 48 registers (5 CTAs per SM) the compiler
// can only keep a full BLP_U batch of gathers in flight when nothing else is live across them: with these scalars
// loaded from global memory inside the trip it issued one gather at a time in the primal step and two in the dual
// step, and the trip waited on the bound mask before its first gather (DESIGN §4).
// Per-lane loop invariants of the two-nodes-per-lane steps: (w0, w1) and (tau0, tau1) / (sigma0, sigma1).
__shared__ double2 s_wv[32], s_sv[32];

// Dynamic shared memory behind a step kernel's slab (row pointers, `cap` entries) that holds its row scalars.
__device__ __forceinline__ int4* row_scalar_smem(const int rows_per_cta, const int cap) {
    return dyn_smem + (rows_per_cta + 4) / 4 + cap;
}
// Bytes per chunk row (host side sizes the launch with them).
constexpr int kPrimalRowBytes = 48, kDualRowBytes = 16;

// One record of row scalars per chunk row, the same in shared memory and in a work list (WorkList::rec).
// primal step: (lref, uref) of row j in the tile's two 32-node blocks h0, h0 + 1, c_j, and the blocks' lumask words
struct PrimalRec {
    double2 lu[2];
    double c;
    uint32_t mk[2];
};
// dual step: b_i, and rconst of row i in the tile (frozen coordinates) or 0
struct DualRec {
    double b, rc;
};
static_assert(sizeof(PrimalRec) == kPrimalRowBytes && sizeof(DualRec) == kDualRowBytes, "row record sizes");

// rs(j, slot) of stage_slab: loads the primal record of row j, stores it at rec[slot]
struct PrimalRowScalars {
    const double* c; const double* lref; const double* uref; const uint32_t* lumask;   // at block h0
    size_t rows;                                                                    // block stride
    PrimalRec* rec;
    __device__ PrimalRowScalars(const DevProb& P, const DevState& S, const int h0, PrimalRec* dst) : rec(dst) {
        const size_t f = (size_t)h0 * P.n;
        c = P.c; lref = S.lref + f; uref = S.uref + f; lumask = S.lumask + f; rows = P.n;
    }
    __device__ __forceinline__ void operator()(const int j, const int slot) const {
        PrimalRec r;
        r.lu[0] = make_double2(__ldg(lref + j), __ldg(uref + j));
        r.lu[1] = make_double2(__ldg(lref + rows + j), __ldg(uref + rows + j));
        r.c = __ldg(c + j);
        r.mk[0] = __ldg(lumask + j);
        r.mk[1] = __ldg(lumask + rows + j);
        rec[slot] = r;
    }
};

// the same for the dual step without frozen coordinates (rconst 0)
struct DualRowScalars {
    const double* b;
    DualRec* rec;
    __device__ __forceinline__ void operator()(const int i, const int slot) const { rec[slot] = DualRec{__ldg(b + i), 0.0}; }
};

// Slab of a frozen-path CTA: chunk `hd` of its tile's work list W (k_work_scan). Every address is known from the
// header, so the chunk's rows (s_row), its row records (row_scalar_smem) and, when they fit in `cap`, its kept entries
// are copied in one round trip. The slab has no row pointers: a trip finds its entries through s_row.
template <class Rec>
__device__ __forceinline__ Slab stage_work(const WorkList& W, const int rows, const int nnz, const int tile,
                                           const int4 hd, const int rows_per_cta, const int cap) {
    constexpr int RQ = sizeof(Rec) / sizeof(int4);
    int4* se = dyn_smem + (rows_per_cta + 4) / 4;
    int4* sr = row_scalar_smem(rows_per_cta, cap);
    const int nk = hd.y < 0 ? 1 : hd.y, cnt = hd.w - hd.z;
    const bool fits = cnt <= cap;
    const int2* __restrict__ rw = W.row + (size_t)tile * (rows + 1) + hd.x;
    const int4* __restrict__ rr = W.rec + ((size_t)tile * rows + hd.x) * RQ;
    const int4* __restrict__ re = reinterpret_cast<const int4*>(W.ent + (size_t)tile * nnz) + hd.z;
    const int units = max(max(nk + 1, nk * RQ), fits ? cnt : 0);
    for (int t0 = threadIdx.x; t0 < units; t0 += 2 * kCtaThreads) {
        int2 r[2];
        int4 s[2], e[2];
#pragma unroll
        for (int q = 0; q < 2; ++q) {                          // all loads first, then the stores
            const int t = t0 + q * kCtaThreads;
            if (t <= nk) r[q] = __ldg(rw + t);
            if (t < nk * RQ) s[q] = __ldg(rr + t);
            if (fits && t < cnt) e[q] = __ldg(re + t);
        }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int t = t0 + q * kCtaThreads;
            if (t <= nk) s_row[t] = r[q];
            if (t < nk * RQ) sr[t] = s[q];
            if (fits && t < cnt) se[t] = e[q];
        }
    }
    __syncthreads();
    Slab s;
    s.sp = nullptr;
    s.base = hd.z;
    s.se = fits ? se : nullptr;
    return s;
}

// Frozen-path CTAs (iterations 0 .. K-2 of a period with frozen coordinates) walk a chunk of their tile's work list:
// its active rows only, each with its kept entries. The last iteration of a period (MAJOR) and batches without
// frozen coordinates walk rows [r0, r1) of the full matrix (chunk_ptr).
template <bool MAJOR>
__global__ void __launch_bounds__(kCtaThreads, BLP_MINB2)
k_primal2(const DevProb P, const DevState S, const int it, const int rows_per_cta, const int cap,
          const int* __restrict__ chunk_ptr, const int tile0) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int tile = tile0 + blockIdx.y;
    const int node = tile * kBlk + lane * 2;                   // this lane: nodes node, node + 1
    const bool frz = !MAJOR && S.cfrz != nullptr;
    // the chunk header and the nodes' scalars are loaded together: one round trip
    const int4 hd = frz ? __ldg(S.wlC.chunk + (size_t)tile * P.n + blockIdx.x)
                        : make_int4(__ldg(chunk_ptr + 2 * blockIdx.x), __ldg(chunk_ptr + 2 * blockIdx.x + 1), 0, 0);
    const int2 sb = *reinterpret_cast<const int2*>(S.sbase + node);
    const double2 et = ld2(S.eta + node), om = ld2(S.omega + node);
    const bool k0 = node < S.B && S.fin[node] == 0;
    const bool k1 = node + 1 < S.B && S.fin[node + 1] == 0;
    const unsigned live = __ballot_sync(0xffffffffu, k0 || k1);
    if (live == 0) return;                                     // whole block retired
    // which lanes store node / node + 1: warp-uniform masks, so that the trip keeps no predicate registers for them
    // (the gather batch needs them). The MAJOR step keeps k0 / k1: with the masks it spills.
    const unsigned run0 = __ballot_sync(0xffffffffu, k0), run1 = __ballot_sync(0xffffffffu, k1);
    auto st0 = [&] { return MAJOR ? k0 : ((run0 >> (threadIdx.x & 31)) & 1u) != 0; };
    auto st1 = [&] { return MAJOR ? k1 : ((run1 >> (threadIdx.x & 31)) & 1u) != 0; };
    if (warp == 0) {                                           // every warp has the same; read back after the stage
        const int s0 = sb.x + it, s1 = sb.y + it;
        s_wv[lane] = make_double2(k0 ? (double)s0 / (double)(s0 + 1) : 0.0, k1 ? (double)s1 / (double)(s1 + 1) : 0.0);
        s_sv[lane] = make_double2(k0 ? et.x / om.x : 0.0, k1 ? et.y / om.y : 0.0);
    }
    if (frz && hd.y == 0) return;                              // no active row left for this chunk
    const int r0 = hd.x, r1 = hd.y;                            // rows of the full matrix (not frz)
    // with frozen coordinates: the tile's kept entries of A' (entries of frozen rows, whose multiplier is zero, taken out)
    const Ent* __restrict__ cent = frz ? S.wlC.ent + (size_t)tile * P.nnz : P.cent;
    PrimalRec* const recs = reinterpret_cast<PrimalRec*>(row_scalar_smem(rows_per_cta, cap));
    const Slab sl = frz ? stage_work<PrimalRec>(S.wlC, P.n, P.nnz, tile, hd, rows_per_cta, cap)
                        : stage_slab(P.cptr, P.cent, r0, r1, rows_per_cta, cap, dyn_smem,
                                     PrimalRowScalars(P, S, tile * 2, recs));
    // 32-bit element indices: the host picks these kernels only for state arrays of fewer than 2^32 elements
    const unsigned base = (unsigned)tix(0, node, P.n);
    const double* __restrict__ yn = S.y + tix(0, node, P.m);
    const unsigned yoff = (unsigned)tix(0, node, P.m);
    const unsigned bit = node & 31;
    const int half = lane >> 4;                                // lanes 16-31: nodes of block h0 + 1
    const bool coop = frz ? hd.y < 0 : (r1 - r0 == 1) && (sl.sp[1] - sl.sp[0] > kLongRow);
    // row slot k of the chunk: {row, start of its entries}; its entries end where row k + 1's start
    auto row_at = [&](const int k) { return frz ? s_row[k] : make_int2(r0 + k, sl.sp[k]); };
    double cg0 = 0.0, cg1 = 0.0;
    int2 rc = make_int2(0, 0);
    if (coop) {
        rc = row_at(0);
        coop_dot2(sl, cent, rc.y, row_at(1).y, yn, warp, lane, cg0, cg1);
        if (warp != 0) return;
    }
    // one warp trip: row slot k of the chunk (rk = row_at(k)); gather(p0, p1, g0, g1) adds the gather-dot of entries
    // [p0, p1) to (g0, g1)
    auto trip = [&](const int k, const int2 rk, double g0, double g1, auto gather) {
        const int p1 = row_at(k + 1).y;
        const unsigned e = base + (unsigned)rk.x * kBlk;
        const double2 xb = ld2(S.xbar + e);
        const double2 a = ldcs2(S.xa + e);
        gather(rk.y, p1, g0, g1);
        // the rest of the row's inputs come from shared memory once the gathers fly; the dense bounds of nodes
        // that deviate from their block's reference (about 1 % of rows) only after them
        const PrimalRec* rv = reinterpret_cast<const PrimalRec*>(row_scalar_smem(rows_per_cta, cap)) + k;
        const uint32_t mk = (rv->mk[half] >> bit) & 3u;
        const double2 lh = rv->lu[half];
        double lo0 = lh.x, hi0 = lh.y, lo1 = lh.x, hi1 = lh.y;
        if (mk & 1u) {                                         // node deviates from its block's reference
            lo0 = __ldcs(S.l + e);
            hi0 = __ldcs(S.u + e);
        }
        if (mk & 2u) {
            lo1 = __ldcs(S.l + e + 1);
            hi1 = __ldcs(S.u + e + 1);
        }
        const double cj = rv->c;
        const double2 w = s_wv[lane], tau = s_sv[lane];
        const double xc0 = fma(w.x, xb.x - a.x, a.x), xc1 = fma(w.y, xb.y - a.y, a.y);
        const double xp0 = fmin(fmax(xc0 - tau.x * (cj - g0), lo0), hi0);
        const double xp1 = fmin(fmax(xc1 - tau.y * (cj - g1), lo1), hi1);
        st2(S.xbar + e, make_double2(2.0 * xp0 - xc0, 2.0 * xp1 - xc1), st0(), st1());
        if constexpr (MAJOR) {
            st2(S.X1 + e, make_double2(xp0, xp1), st0(), st1());
            st2(S.DX + e, make_double2(xp0 - xc0, xp1 - xc1), st0(), st1());
            st2(S.G + e, make_double2(g0, g1), st0(), st1());
        }
    };
    if (coop) {                                                // warp 0, the chunk's one row
        trip(0, rc, cg0, cg1, [](int, int, double&, double&) {});
        return;
    }
    // Whether the entries sit in shared memory is the same for the whole CTA: choosing the loop here keeps the
    // choice (and its pointer) out of the registers that are live across a trip's gathers.
    const int ntrips = frz ? hd.y : r1 - r0;                   // frozen columns rest at their bound for the whole tile
    if (sl.se) {
        const int4* const E = sl.se - sl.base;
        for (int k = warp; k < ntrips; k += kWarps)
            trip(k, row_at(k), 0.0, 0.0, [&](const int p0, const int p1, double& g0, double& g1) {
                dot2_entries<true, unsigned, false>(E, p0, p1, S.y, g0, g1, kBlk, yoff);
            });
    } else {
        const int4* const E = reinterpret_cast<const int4*>(cent);
        for (int k = warp; k < ntrips; k += kWarps)
            trip(k, row_at(k), 0.0, 0.0, [&](const int p0, const int p1, double& g0, double& g1) {
                dot2_entries<false, unsigned, false>(E, p0, p1, S.y, g0, g1, kBlk, yoff);
            });
    }
}

template <bool MAJOR>
__global__ void __launch_bounds__(kCtaThreads, BLP_MINB2)
k_dual2(const DevProb P, const DevState S, const int it, const int rows_per_cta, const int cap,
        const int* __restrict__ chunk_ptr, const int tile0) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int tile = tile0 + blockIdx.y;
    const int node = tile * kBlk + lane * 2;
    const bool frz = !MAJOR && S.rfrz != nullptr;
    const int4 hd = frz ? __ldg(S.wlR.chunk + (size_t)tile * P.m + blockIdx.x)     // as in k_primal2
                        : make_int4(__ldg(chunk_ptr + 2 * blockIdx.x), __ldg(chunk_ptr + 2 * blockIdx.x + 1), 0, 0);
    const int2 sb = *reinterpret_cast<const int2*>(S.sbase + node);
    const double2 et = ld2(S.eta + node), om = ld2(S.omega + node);
    const bool k0 = node < S.B && S.fin[node] == 0;
    const bool k1 = node + 1 < S.B && S.fin[node + 1] == 0;
    const unsigned live = __ballot_sync(0xffffffffu, k0 || k1);
    if (live == 0) return;
    const unsigned run0 = __ballot_sync(0xffffffffu, k0), run1 = __ballot_sync(0xffffffffu, k1);   // as in k_primal2
    auto st0 = [&] { return ((run0 >> (threadIdx.x & 31)) & 1u) != 0; };
    auto st1 = [&] { return ((run1 >> (threadIdx.x & 31)) & 1u) != 0; };
    if (warp == 0) {                                           // every warp has the same; read back after the stage
        const int s0 = sb.x + it, s1 = sb.y + it;
        s_wv[lane] = make_double2(k0 ? (double)(s0 + 1) / (double)(s0 + 2) : 0.0,
                                  k1 ? (double)(s1 + 1) / (double)(s1 + 2) : 0.0);
        s_sv[lane] = make_double2(k0 ? et.x * om.x : 0.0, k1 ? et.y * om.y : 0.0);
    }
    if (frz && hd.y == 0) return;
    const int r0 = hd.x, r1 = hd.y;
    // with frozen coordinates: the tile's kept entries of A (columns that rest at one value for the whole tile are
    // summed into the row's rconst once per evaluation period instead of being gathered every iteration)
    const Ent* __restrict__ aent = frz ? S.wlR.ent + (size_t)tile * P.nnz : P.ent;
    DualRec* const recs = reinterpret_cast<DualRec*>(row_scalar_smem(rows_per_cta, cap));
    const Slab sl = frz ? stage_work<DualRec>(S.wlR, P.m, P.nnz, tile, hd, rows_per_cta, cap)
                        : stage_slab(P.rowptr, P.ent, r0, r1, rows_per_cta, cap, dyn_smem, DualRowScalars{P.b, recs});
    const unsigned base = (unsigned)tix(0, node, P.m);      // 32-bit element indices, as in k_primal2
    const double* __restrict__ xn = S.xbar + tix(0, node, P.n);
    const unsigned xoff = (unsigned)tix(0, node, P.n);
    const bool coop = frz ? hd.y < 0 : (r1 - r0 == 1) && (sl.sp[1] - sl.sp[0] > kLongRow);
    auto row_at = [&](const int k) { return frz ? s_row[k] : make_int2(r0 + k, sl.sp[k]); };   // as in k_primal2
    double cg0 = 0.0, cg1 = 0.0;
    int2 rc = make_int2(0, 0);
    if (coop) {
        rc = row_at(0);
        coop_dot2(sl, aent, rc.y, row_at(1).y, xn, warp, lane, cg0, cg1);
        if (warp != 0) return;
        if (frz) {
            const double rc = recs[0].rc;
            cg0 += rc;
            cg1 += rc;
        }
    }
    // one warp trip: row slot k of the chunk (rk = row_at(k)); gather(k, p0, p1, ax0, ax1) sets (ax0, ax1) to the
    // row's A x
    auto trip = [&](const int k, const int2 rk, auto gather) {
        const int p1 = row_at(k + 1).y;
        const int i = rk.x;
        const unsigned e = base + (unsigned)i * kBlk;
        const double2 yc = ld2(S.y + e);
        const double2 a = ldcs2(S.ya + e);
        bool on0 = true, on1 = true;
        if (i >= P.m_base && S.rowmask) {
            const uint8_t* mrow = S.rowmask + (size_t)(i - P.m_base) * S.ld + node;
            on0 = mrow[0] != 0;
            on1 = mrow[1] != 0;
        }
        double ax0, ax1;
        gather(k, rk.y, p1, ax0, ax1);
        const double bi = reinterpret_cast<const DualRec*>(row_scalar_smem(rows_per_cta, cap))[k].b;
        const double2 w = s_wv[lane], sig = s_sv[lane];
        const double yp0 = on0 ? fmax(0.0, yc.x + sig.x * (bi - ax0)) : 0.0;
        const double yp1 = on1 ? fmax(0.0, yc.y + sig.y * (bi - ax1)) : 0.0;
        st2(S.y + e, make_double2(fma(w.x, (2.0 * yp0 - yc.x) - a.x, a.x),
                                  fma(w.y, (2.0 * yp1 - yc.y) - a.y, a.y)), st0(), st1());
        if constexpr (MAJOR) {
            st2(S.Y1 + e, make_double2(yp0, yp1), st0(), st1());
            st2(S.DY + e, make_double2(yp0 - yc.x, yp1 - yc.y), st0(), st1());
        }
    };
    if (coop) {                                                // warp 0, the chunk's one row
        trip(0, rc, [&](int, int, int, double& ax0, double& ax1) { ax0 = cg0; ax1 = cg1; });
        return;
    }
    // as in k_primal2: the shared / global choice of the entries is made once per CTA
    const int ntrips = frz ? hd.y : r1 - r0;                   // a frozen row's multiplier rests at zero for the whole tile
    if (sl.se) {
        const int4* const E = sl.se - sl.base;
        for (int k = warp; k < ntrips; k += kWarps)
            trip(k, row_at(k), [&](const int k_, const int p0, const int p1, double& ax0, double& ax1) {
                ax0 = ax1 = reinterpret_cast<const DualRec*>(row_scalar_smem(rows_per_cta, cap))[k_].rc;   // 0 without frozen coordinates
                dot2_entries<true, unsigned, false>(E, p0, p1, S.xbar, ax0, ax1, kBlk, xoff);
            });
    } else {
        const int4* const E = reinterpret_cast<const int4*>(aent);
        for (int k = warp; k < ntrips; k += kWarps)
            trip(k, row_at(k), [&](const int k_, const int p0, const int p1, double& ax0, double& ax1) {
                ax0 = ax1 = reinterpret_cast<const DualRec*>(row_scalar_smem(rows_per_cta, cap))[k_].rc;
                dot2_entries<false, unsigned, false>(E, p0, p1, S.xbar, ax0, ax1, kBlk, xoff);
            });
    }
}

// k_primal2 / k_dual2 walk one row x one 64-node tile per warp trip. They are bound by how many independent
// row walks an SM holds: variants that buy per-warp parallelism with registers (two rows per trip, two node
// tiles per warp) lose more in resident warps than they gain (DESIGN §4).

// ---------------------------------------------------------------------------------------------
// CTA-level, order-fixed reduction of per-thread accumulators into the chunk's partial slot.
template <int NT, int NACC, int NSUM>
__device__ __forceinline__ void cta_reduce_store(double (&acc)[NACC], double* __restrict__ part,
                                                 int ld, int node_base) {
    __shared__ double sm[NACC][kCtaThreads];
#pragma unroll
    for (int a = 0; a < NACC; ++a) sm[a][threadIdx.x] = acc[a];
    __syncthreads();
    // thread t < NT*NACC reduces accumulator (t / NT) of local node (t % NT)
    for (int t = threadIdx.x; t < NT * NACC; t += kCtaThreads) {
        const int a = t / NT, nl = t % NT;
        double r = sm[a][nl];
        for (int q = nl + NT; q < kCtaThreads; q += NT)
            r = (a < NSUM) ? r + sm[a][q] : fmax(r, sm[a][q]);
        part[((size_t)blockIdx.x * NACC + a) * ld + node_base + nl] = r;
    }
}

// Column pass of an evaluation: G' = A'y', reduced costs, dual residual, objectives, Farkas box
// term, ray direction d = x' - xa (left in G for the row pass).
template <int NT>
__global__ void __launch_bounds__(kCtaThreads)
k_eval_cols(const DevProb P, const DevState S, const int rows_per_cta) {
    constexpr int RW = 32 / NT;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int node = blockIdx.y * NT + (lane % NT);
    const int sub = lane / NT;
    const bool node_ok = node < S.B && S.fin[node] == 0;
    if (__ballot_sync(0xffffffffu, node_ok) == 0) return;     // uniform over the CTA
    double acc[C_N];
#pragma unroll
    for (int a = 0; a < C_N; ++a) acc[a] = 0.0;
    const int r0 = blockIdx.x * rows_per_cta;
    const int r1 = min(P.n, r0 + rows_per_cta);
    for (int jb = r0 + warp * RW; jb < r1; jb += kWarps * RW) {
        const int j = jb + sub;
        const bool row_ok = j < r1;
        const size_t e = tix(j, node, P.n);
        const double gp = row_dot<NT>(P.cptr, P.cent, row_ok ? j : 0, row_ok, S.Y1 + tix(0, node, P.m),
                                      node_ok && row_ok);
        if (row_ok && node_ok) {
            const double xp = S.X1[e], dx = S.DX[e], g = S.G[e];
            const double lo = S.l[e], hi = S.u[e], xa = (double)S.xa[e];
            const double cj = __ldg(P.c + j), cs = __ldg(P.colscale + j);
            const bool fl = !is_inf(lo), fu = !is_inf(hi);
            acc[C_DX2] = fma(dx, dx, acc[C_DX2]);
            acc[C_CROSS] = fma(dx, gp - g, acc[C_CROSS]);
            const double r = cj - gp;
            const double lam = (r > 0.0) ? (fl ? r : 0.0) : (fu ? r : 0.0);
            const double dres = (r - lam) * cs;
            acc[C_DRES2] = fma(dres, dres, acc[C_DRES2]);
            acc[C_CX] = fma(cj, xp, acc[C_CX]);
            if (lam > 0.0) acc[C_BND] = fma(lo, lam, acc[C_BND]);
            else if (lam < 0.0) acc[C_BND] = fma(hi, lam, acc[C_BND]);
            const double d = xp - xa;
            acc[C_DXA2] = fma(d, d, acc[C_DXA2]);
            double box = 0.0;
            if (gp > 0.0) { if (fu) box = gp * hi; else acc[C_RAYVIOL] = fmax(acc[C_RAYVIOL], gp); }
            else if (gp < 0.0) { if (fl) box = gp * lo; else acc[C_RAYVIOL] = fmax(acc[C_RAYVIOL], -gp); }
            acc[C_BOX] += box;
            acc[C_BOXABS] += fabs(box);
            // the same Farkas box term for the dual STEP dy = y' - y (A'dy = gp - g): on an
            // infeasible LP the step converges to the certificate ray, free of the offset y' carries
            const double gd = gp - g;
            double dbox = 0.0;
            if (gd > 0.0) { if (fu) dbox = gd * hi; else acc[C_DRAYVIOL] = fmax(acc[C_DRAYVIOL], gd); }
            else if (gd < 0.0) { if (fl) dbox = gd * lo; else acc[C_DRAYVIOL] = fmax(acc[C_DRAYVIOL], -gd); }
            acc[C_DBOX] += dbox;
            acc[C_DBOXABS] += fabs(dbox);
            acc[C_CD] = fma(cj, d, acc[C_CD]);
            acc[C_DMAX] = fmax(acc[C_DMAX], fabs(d));
            if (fl) acc[C_DVIOL] = fmax(acc[C_DVIOL], -d);
            if (fu) acc[C_DVIOL] = fmax(acc[C_DVIOL], d);
            S.G[e] = d;
        }
    }
    cta_reduce_store<NT, C_N, C_NSUM>(acc, S.partC, S.ld, blockIdx.y * NT);
}

// Row pass of an evaluation: A x' and A d, primal residual, b.y', iterate movement.
template <int NT>
__global__ void __launch_bounds__(kCtaThreads)
k_eval_rows(const DevProb P, const DevState S, const int rows_per_cta) {
    constexpr int RW = 32 / NT;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int node = blockIdx.y * NT + (lane % NT);
    const int sub = lane / NT;
    const bool node_ok = node < S.B && S.fin[node] == 0;
    if (__ballot_sync(0xffffffffu, node_ok) == 0) return;     // uniform over the CTA
    double acc[R_N];
#pragma unroll
    for (int a = 0; a < R_N; ++a) acc[a] = 0.0;
    const int r0 = blockIdx.x * rows_per_cta;
    const int r1 = min(P.m, r0 + rows_per_cta);
    for (int ib = r0 + warp * RW; ib < r1; ib += kWarps * RW) {
        const int i = ib + sub;
        const bool row_ok = i < r1;
        const size_t e = tix(i, node, P.m);
        const bool ok = row_ok && node_ok;
        double ax, ad;
        row_dot_pair<NT>(P.rowptr, P.ent, row_ok ? i : 0, row_ok, S.X1 + tix(0, node, P.n), S.G + tix(0, node, P.n),
                         ok, ax, ad);
        if (ok) {
            bool on = true;
            if (i >= P.m_base && S.rowmask) on = S.rowmask[(size_t)(i - P.m_base) * S.ld + node] != 0;
            if (on) {
                const double yp = S.Y1[e], dy = S.DY[e], ya = (double)S.ya[e];
                const double bi = __ldg(P.b + i);
                const double pr = fmax(bi - ax, 0.0) * __ldg(P.rowscale + i);
                acc[R_PRES2] = fma(pr, pr, acc[R_PRES2]);
                acc[R_BY] = fma(bi, yp, acc[R_BY]);
                acc[R_BYABS] += fabs(bi * yp);
                acc[R_DY2] = fma(dy, dy, acc[R_DY2]);
                const double t = yp - ya;
                acc[R_DYA2] = fma(t, t, acc[R_DYA2]);
                acc[R_ADNEG] = fmax(acc[R_ADNEG], -ad);
                acc[R_YMAX] = fmax(acc[R_YMAX], yp);
                acc[R_BD] = fma(bi, dy, acc[R_BD]);
                acc[R_BDABS] += fabs(bi * dy);
                acc[R_DYMAX] = fmax(acc[R_DYMAX], fabs(dy));
                acc[R_DYNEG] = fmax(acc[R_DYNEG], -dy);
            }
        }
    }
    cta_reduce_store<NT, R_N, R_NSUM>(acc, S.partR, S.ld, blockIdx.y * NT);
}

// ---------------------------------------------------------------------------------------------
// One thread per node: fold the chunk partials in fixed order, test termination and the
// infeasibility / unboundedness certificates, decide restarts, update the primal weight.
struct DecideArgs {
    int chunksC, chunksR, steps_in_period, max_iters;
    double eps, eps_inf;
    double beta_suff, beta_nec, beta_art, theta;    // restart thresholds, primal-weight smoothing
    double balance, balance_dead;   // primal-weight feedback on the lagging criterion (0 = off), see k_decide
    double cutoff;                  // blp_opts.obj_cutoff: retire a node whose dual bound reaches it (status 5)
};

// counters: [0] nodes still running after the evaluation, [1] nodes restarting,
//           [2] PDHG iterations executed so far (advanced by k_tick at the start of a period,
//               so one captured period graph can be replayed unchanged),
//           [3] nodes that got a status in this evaluation (to be harvested)
__global__ void k_tick(const DevState S, const int steps) {
    S.counters[0] = 0;
    S.counters[1] = 0;
    S.counters[2] += steps;
    S.counters[3] = 0;
}

__global__ void k_decide(const DevProb P, const DevState S, const DecideArgs D) {
    const int node = blockIdx.x * blockDim.x + threadIdx.x;
    if (node >= S.B) return;
    S.restart[node] = 0;
    if (S.fin[node] != 0) return;
    double c[C_N], r[R_N];
#pragma unroll
    for (int a = 0; a < C_N; ++a) c[a] = 0.0;
#pragma unroll
    for (int a = 0; a < R_N; ++a) r[a] = 0.0;
    for (int ch = 0; ch < D.chunksC; ++ch)
#pragma unroll
        for (int a = 0; a < C_N; ++a) {
            const double v = S.partC[((size_t)ch * C_N + a) * S.ld + node];
            c[a] = (a < C_NSUM) ? c[a] + v : fmax(c[a], v);
        }
    for (int ch = 0; ch < D.chunksR; ++ch)
#pragma unroll
        for (int a = 0; a < R_N; ++a) {
            const double v = S.partR[((size_t)ch * R_N + a) * S.ld + node];
            r[a] = (a < R_NSUM) ? r[a] + v : fmax(r[a], v);
        }
    const double omega = S.omega[node];
    const double eta = S.eta[node];
    const double tau = eta / omega, sig = eta * omega;
    const double fpe = sqrt(fmax(c[C_DX2] / tau + r[R_DY2] / sig + 2.0 * c[C_CROSS], 0.0));
    const double pobj = c[C_CX] * P.objscale;
    const double dobj = (r[R_BY] + c[C_BND]) * P.objscale;
    // the primal tolerance is relative to ||b|| over the rows of THIS node's LP: the base rows plus the
    // appended rows its mask switches on — not over rows that only other nodes hold
    double bn2 = P.bnorm0 * P.bnorm0;
    if (P.m > P.m_base) {
        if (S.rowmask) {
            for (int i = P.m_base; i < P.m; ++i)
                if (S.rowmask[(size_t)(i - P.m_base) * S.ld + node]) {
                    const double b0 = P.b[i] * P.rowscale[i];
                    bn2 = fma(b0, b0, bn2);
                }
        } else {
            bn2 += P.bcut2;
        }
    }
    const double rp = sqrt(r[R_PRES2]) / (1.0 + sqrt(bn2));
    const double rd = sqrt(c[C_DRES2]) / (1.0 + P.cnorm0);
    const double rg = fabs(pobj - dobj) / (1.0 + fabs(pobj) + fabs(dobj));
    S.pobj[node] = pobj;
    S.dobj[node] = dobj;
    if (S.dbg) {
        double* t = S.dbg + (size_t)node * 8;
        t[0] = rp; t[1] = rd; t[2] = rg; t[3] = fpe; t[4] = omega; t[5] = (double)S.sbase[node];
        t[6] = pobj; t[7] = dobj;
    }
    const int total = S.counters[2] - S.start[node];      // iterations this node has run
    const bool last = total >= D.max_iters;
    int st = -1;
    if (rp <= D.eps && rd <= D.eps && rg <= D.eps) {
        st = 0;
    } else {
        // Farkas certificate of primal infeasibility from the dual iterate y' >= 0:
        //   b.y' > max_{l<=x<=u} (A'y').x     (columns with an infinite bound must not need it)
        const double farkas = r[R_BY] - c[C_BOX];
        if (farkas > 0.0 && farkas > D.eps_inf * (r[R_BYABS] + c[C_BOXABS]) &&
            c[C_RAYVIOL] <= 1e-8 * r[R_YMAX])
            st = 1;
        // ... and from the dual step dy >= 0 (it reaches the ray long before y' is dominated by it)
        const double fstep = r[R_BD] - c[C_DBOX];
        if (st < 0 && r[R_DYMAX] > 0.0 && fstep > 1e-6 * (r[R_BDABS] + c[C_DBOXABS]) &&
            c[C_DRAYVIOL] <= 1e-8 * r[R_DYMAX] && r[R_DYNEG] <= 1e-8 * r[R_DYMAX])
            st = 1;
        // primal ray d = x' - xa: c.d < 0, A d >= 0, d respects finite bounds => unbounded
        const double dmax = c[C_DMAX];
        if (st < 0 && dmax > 0.0 && c[C_CD] < -1e-6 * dmax * P.cinf_s &&
            r[R_ADNEG] <= 1e-8 * dmax && c[C_DVIOL] <= 1e-8 * dmax)
            st = 2;
    }
    // objective limit: the dual objective is a valid lower bound of the node LP whenever the dual
    // iterate is feasible (rd: the part of the reduced costs no finite bound can absorb)
    if (st < 0 && rd <= D.eps && dobj >= D.cutoff) st = 5;
    if (st < 0 && last) st = 3;
    if (st >= 0) {
        S.status[node] = st;
        S.fin[node] = 1;
        S.iters[node] = total;
        if (st == 1) S.pobj[node] = INFINITY;
        atomicAdd(S.counters + 3, 1);
        return;
    }
    atomicAdd(S.counters + 0, 1);
    // restart test on the fixed-point error (sufficient / necessary / artificial)
    const int s_now = S.sbase[node] + D.steps_in_period;
    const double f0 = S.fpe0[node], fprev = S.fpe_prev[node];
    const bool first = !(f0 < INFINITY);
    // a step above 1 / ||A|| rests on the frozen set staying frozen and on a power-iteration estimate; if the
    // fixed-point error grows by half within a phase the node goes back to 1 / ||A|| for good and restarts
    const bool runaway = eta > P.eta && !first && fpe > 1.5 * fmin(f0, fprev);
    if (runaway) {
        S.eta[node] = P.eta;
        S.eta_lock[node] = 1;
        atomicAdd(S.counters + 12, 1);
    }
    const bool do_restart = first || runaway || fpe <= D.beta_suff * f0 || (fpe <= D.beta_nec * f0 && fpe > fprev) ||
                            (double)s_now >= D.beta_art * (double)total;
    if (do_restart) {
        const double ddx = sqrt(c[C_DXA2]), ddy = sqrt(r[R_DYA2]);
        double om = omega;
        if (!first && ddx > 1e-10 && ddy > 1e-10)
            om = exp(D.theta * log(ddy / ddx) + (1.0 - D.theta) * log(omega));
        // residual balancing: the primal residual shrinks with the dual step (omega up), the
        // duality gap with the primal step (omega down); push towards whichever criterion lags
        // (bench fixtures: same mean iteration count, slowest node of a 256-node batch 12-25 % earlier;
        // the feedback alone may move omega at most 1e4 either way from its initial value;
        // criteria within a factor exp(dead zone) of each other count as balanced)
        if (!first && D.balance > 0.0 && rp > 0.0 && rg > 0.0) {
            const double lr = log(rp / rg);
            const double ex = copysign(fmin(fmax(fabs(lr) - D.balance_dead, 0.0), 1.0), lr);
            const double fb = om * exp(D.balance * ex);
            if (fb <= 1e4 * P.omega0 && fb >= 1e-4 * P.omega0) om = fb;
        }
        S.omega[node] = om;
        S.fpe0[node] = runaway ? INFINITY : fpe;
        S.fpe_prev[node] = INFINITY;
        S.sbase[node] = 0;
        S.restart[node] = 1;
        atomicAdd(S.counters + 1, 1);
    } else {
        S.fpe_prev[node] = fpe;
        S.sbase[node] = s_now;
    }
}

// Restart: the anchor and the current point both become T(z) of the evaluated iterate.
// grid = (row chunks, ceil(ld/32)); a warp owns 32 node columns and strides over the rows.
__global__ void __launch_bounds__(kCtaThreads)
k_apply_restart(const DevProb P, const DevState S) {
    if (S.counters[1] == 0) return;
    const int lane = threadIdx.x & 31;
    const int node = blockIdx.y * 32 + lane;
    const bool mine = node < S.B && S.restart[node] != 0;
    if (__ballot_sync(0xffffffffu, mine) == 0) return;
    if (!mine) return;
    const int gwarp = (blockIdx.x * kCtaThreads + threadIdx.x) >> 5;
    const int nwarps = (gridDim.x * kCtaThreads) >> 5;
    for (int j = gwarp; j < P.n; j += nwarps) {
        const size_t e = tix(j, node, P.n);
        const double v = S.X1[e];
        S.xa[e] = (anc_t)v;
        S.xbar[e] = v;
    }
    for (int i = gwarp; i < P.m; i += nwarps) {
        const size_t e = tix(i, node, P.m);
        const double v = S.Y1[e];
        S.ya[e] = (anc_t)v;
        S.y[e] = v;
    }
}

// ---------------------------------------------------------------------------------------------
// Freezing of settled coordinates. Most columns of a node LP rest on a bound with a reduced cost of the right
// sign, and the rows with slack keep a zero multiplier, from the warm start to the end of the solve (C5 frontier:
// 60 % of the columns, 24 % of the rows); the iteration recomputes the same values for them, 20 bytes of HBM
// stream per coordinate, node and iteration. A coordinate is FROZEN for a 64-node tile when, for every running
// node of the tile,
//   column:  x' = x_iterate = anchor = the bound (lower with r_j >= margin, upper with r_j <= -margin; or l == u),
//   row:     y' = y_iterate = anchor = 0 and (A x' - b)_i >= margin (or the row is masked off for the node),
// i.e. exactly when the full iteration would reproduce the coordinate. The step kernels skip frozen coordinates
// (k_primal2 / k_dual2, all iterations of a period but the last); the last iteration of a period updates
// everything, so the evaluation — KKT test on the FULL problem, certificates, restart rule — sees exact x', y',
// A'y, and whatever the frozen set was, a status is only ever assigned by the full test. The flags are recomputed
// after every evaluation with hysteresis (freeze above *_hi, release below *_lo; a node loaded by the last refill
// is held to *_hi), per 32-node block; a tile's two blocks must agree. Screened on the host first
// (tests/tools/cpu_freeze_lab.py: same iteration counts, half the coordinate updates skipped on C4 and C5).
//   mode 0: after an evaluation; 1: after a refill (S.fresh marks the new nodes); 2: ignore the stored flags
__device__ __forceinline__ bool rests_on(const double v, const double bound, const double width) {
    return fabs(v - bound) <= 1e-6 * width;      // fp32 anchors and the Halpern average leave ~1e-8 relative
}

__global__ void __launch_bounds__(kCtaThreads)
k_freeze_cols(const DevProb P, const DevState S, const FreezeArgs F, const int rows_per_cta, const int mode) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int node = blockIdx.y * 32 + lane;
    const bool live = node < S.B && S.fin[node] == 0;
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x < 4) S.counters[8 + threadIdx.x] = 0;   // k_freeze_count follows
    const unsigned running = __ballot_sync(0xffffffffu, live);
    if (running == 0) return;                                 // uniform over the CTA
    const bool strict = mode == 2 || (mode == 1 && live && S.fresh[node] != 0);
    uint8_t* __restrict__ flags = S.cfrz + (size_t)blockIdx.y * P.n;
    double* __restrict__ cval = S.cval + (size_t)blockIdx.y * P.n;
    const double* __restrict__ yn = S.Y1 + tix(0, node, P.m);
    const int r0 = blockIdx.x * rows_per_cta;
    const int r1 = min(P.n, r0 + rows_per_cta);
    for (int j = r0 + warp; j < r1; j += kWarps) {
        const uint8_t stored = flags[j], prev = mode == 2 ? 0 : stored;
        const double gp = row_dot<32>(P.cptr, P.cent, j, true, yn, live);
        bool ok = true;
        double xp = 0.0;
        if (live) {
            const size_t e = tix(j, node, P.n);
            const double lo = S.l[e], hi = S.u[e];
            xp = S.X1[e];
            ok = false;
            if (xp == lo || xp == hi) {
                const double r = __ldg(P.c + j) - gp;
                const double th = (prev && !strict) ? F.c_lo : F.c_hi;
                const double width = is_inf(hi - lo) ? fabs(xp) : fmax(hi - lo, fabs(xp));
                const bool settled = lo >= hi || (xp == lo ? r >= th : -r >= th);
                ok = settled && rests_on(S.xbar[e], xp, width) && (anc_t)xp == S.xa[e];
            }
        }
        const bool all = __all_sync(0xffffffffu, ok);
        // 3: frozen, and every running node of the block rests at the same value (the column can be folded)
        const double ref = __shfl_sync(0xffffffffu, xp, __ffs(running) - 1);
        const bool uniform = __all_sync(0xffffffffu, !live || xp == ref);
        const uint8_t flag = all ? (uniform ? 3 : 1) : 0;
        if (lane == 0) {
            if (flag != stored) flags[j] = flag;
            if (flag == 3) cval[j] = ref;
        }
    }
}

__global__ void __launch_bounds__(kCtaThreads)
k_freeze_rows(const DevProb P, const DevState S, const FreezeArgs F, const int rows_per_cta, const int mode) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int node = blockIdx.y * 32 + lane;
    const bool live = node < S.B && S.fin[node] == 0;
    if (__ballot_sync(0xffffffffu, live) == 0) return;
    const bool strict = mode == 2 || (mode == 1 && live && S.fresh[node] != 0);
    uint8_t* __restrict__ flags = S.rfrz + (size_t)blockIdx.y * P.m;
    const double* __restrict__ xn = S.X1 + tix(0, node, P.n);
    const int r0 = blockIdx.x * rows_per_cta;
    const int r1 = min(P.m, r0 + rows_per_cta);
    for (int i = r0 + warp; i < r1; i += kWarps) {
        const uint8_t stored = flags[i], prev = mode == 2 ? 0 : stored;
        const double ax = row_dot<32>(P.rowptr, P.ent, i, true, xn, live);
        bool ok = true;
        if (live) {
            const size_t e = tix(i, node, P.m);
            const bool zero = S.Y1[e] == 0.0 && S.y[e] == 0.0 && S.ya[e] == (anc_t)0;
            const bool off = i >= P.m_base && S.rowmask && S.rowmask[(size_t)(i - P.m_base) * S.ld + node] == 0;
            const double th = (prev && !strict) ? F.r_lo : F.r_hi;
            ok = zero && (off || ax - __ldg(P.b + i) >= th);
        }
        const bool all = __all_sync(0xffffffffu, ok);
        if (lane == 0 && (uint8_t)all != stored) flags[i] = all;
    }
}

// Folded matrices of every tile with a running node, from the flags (see DevState). One thread per column / row.
//   k_fold_cols: which columns rest at ONE value for the whole tile (both blocks flag 3 with equal values, a block
//                without a running node agrees) — their contribution to A x is a per-row constant of the tile —
//                and which columns (ftc) and rows (ftr) are frozen for the tile; the work lists (k_work_*) follow
// running nodes of the tile's two 32-node blocks -> s_l[0], s_l[1] (all threads of the CTA call; ends with a barrier)
__device__ __forceinline__ void tile_running(const DevState& S, const int tile, int* s_l) {
    if (threadIdx.x < kBlk) {
        const int node = tile * kBlk + threadIdx.x;
        const unsigned bal = __ballot_sync(0xffffffffu, node < S.B && S.fin[node] == 0);
        if ((threadIdx.x & 31) == 0) s_l[threadIdx.x >> 5] = __popc(bal);
    }
    __syncthreads();
}

__global__ void __launch_bounds__(kCtaThreads)
k_fold_cols(const DevProb P, const DevState S) {
    __shared__ int s_l[2];
    const int tile = blockIdx.y;
    tile_running(S, tile, s_l);
    const int l0 = s_l[0], l1 = s_l[1];
    if (l0 + l1 == 0) return;
    const uint8_t* __restrict__ f0 = S.cfrz + (size_t)(2 * tile) * P.n;
    const double* __restrict__ v0 = S.cval + (size_t)(2 * tile) * P.n;
    for (int j = blockIdx.x * kCtaThreads + threadIdx.x; j < P.n; j += gridDim.x * kCtaThreads) {
        const bool a = l0 == 0 || f0[j] == 3, b = l1 == 0 || f0[P.n + j] == 3;
        const double va = l0 ? v0[j] : v0[P.n + j], vb = l1 ? v0[P.n + j] : va;
        const bool fold = a && b && va == vb;
        S.fcol[(size_t)tile * P.n + j] = fold;
        S.fval[(size_t)tile * P.n + j] = fold ? va : 0.0;
        S.ftc[(size_t)tile * P.n + j] = (l0 == 0 || f0[j] != 0) && (l1 == 0 || f0[P.n + j] != 0);
    }
    const uint8_t* __restrict__ g0 = S.rfrz + (size_t)(2 * tile) * P.m;
    for (int i = blockIdx.x * kCtaThreads + threadIdx.x; i < P.m; i += gridDim.x * kCtaThreads)
        S.ftr[(size_t)tile * P.m + i] = (l0 == 0 || g0[i] != 0) && (l1 == 0 || g0[P.m + i] != 0);
}

// Work lists of the frozen-path step kernels (WorkList), built after k_fold_cols for every tile with a running node.
// PRIMAL: rows of A' (columns j, active unless ftc, entry (j, i) kept unless row i is frozen: its multiplier is zero);
// dual: rows of A (rows i, active unless ftr, entry (i, j) kept unless column j is folded into rconst).
//   k_work_count: kept entries of every row, -1 for a frozen one. One thread per row.
//   k_work_scan:  one CTA per tile: the active rows' places and entry starts, then the chunk headers.
//   k_work_fill:  the kept entries (in the row's order) and the record of every active row. One thread per row.
template <bool PRIMAL>
__device__ __forceinline__ bool work_row_active(const DevState& S, const int rows, const int tile, const int r) {
    return !(PRIMAL ? S.ftc : S.ftr)[(size_t)tile * rows + r];
}
template <bool PRIMAL>
__device__ __forceinline__ bool work_entry_kept(const DevProb& P, const DevState& S, const int tile, const int col) {
    return PRIMAL ? !S.ftr[(size_t)tile * P.m + col] : !S.fcol[(size_t)tile * P.n + col];
}

template <bool PRIMAL>
__global__ void __launch_bounds__(kCtaThreads)
k_work_count(const DevProb P, const DevState S) {
    __shared__ int s_l[2];
    const int tile = blockIdx.y;
    tile_running(S, tile, s_l);
    if (s_l[0] + s_l[1] == 0) return;
    const int rows = PRIMAL ? P.n : P.m;
    const int32_t* __restrict__ ptr = PRIMAL ? P.cptr : P.rowptr;
    const Ent* __restrict__ ent = PRIMAL ? P.cent : P.ent;
    int32_t* __restrict__ kept = (PRIMAL ? S.wlC : S.wlR).kept + (size_t)tile * rows;
    for (int r = blockIdx.x * kCtaThreads + threadIdx.x; r < rows; r += gridDim.x * kCtaThreads) {
        int cnt = -1;
        if (work_row_active<PRIMAL>(S, rows, tile, r)) {
            cnt = 0;
            for (int p = __ldg(ptr + r); p < __ldg(ptr + r + 1); ++p) cnt += work_entry_kept<PRIMAL>(P, S, tile, __ldg(&ent[p].idx));
        }
        kept[r] = cnt;
    }
}

// Chunk headers: the long active rows (more than kLongRow stored entries, the rows the full-matrix plan gives a chunk
// of their own) take chunks 0 .. L-1, one each; the N other active rows are split over the remaining Q chunks in row
// order, chunk q holding the rows whose weight prefix P_s (kept entries + cw per row) lies in [q W / Q, (q+1) W / Q),
// W the total. A row's trip costs about one round trip per BLP_U kept entries plus one for its state, hence
// cw >= BLP_U; cw >= E / (Q rows_per_cta - N) (E: kept entries of the N rows) bounds every chunk to rows_per_cta rows.
// Q >= N / rows_per_cta and Q >= 1 when N > 0: the full-matrix plan has at least that many chunks of short rows.
template <bool PRIMAL>
__global__ void __launch_bounds__(1024)
k_work_scan(const DevProb P, const DevState S, const int chunks, const int rows_per_cta) {
    __shared__ int s_l[2];
    __shared__ int4 s_part[32];
    const int tile = blockIdx.x;
    tile_running(S, tile, s_l);
    if (s_l[0] + s_l[1] == 0) return;
    const WorkList& W = PRIMAL ? S.wlC : S.wlR;
    const int rows = PRIMAL ? P.n : P.m;
    const int32_t* __restrict__ ptr = PRIMAL ? P.cptr : P.rowptr;
    int32_t* const kept = W.kept + (size_t)tile * rows;
    int2* const out = W.row + (size_t)tile * (rows + 1);
    int4* const hdr = W.chunk + (size_t)tile * rows;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int seg = (rows + blockDim.x - 1) / blockDim.x;
    const int r0 = min(rows, (int)threadIdx.x * seg), r1 = min(rows, r0 + seg);
    // (long rows, their kept entries, other rows, their kept entries) of the thread's segment
    int4 c = make_int4(0, 0, 0, 0);
#pragma unroll 4
    for (int r = r0; r < r1; ++r) {
        const int k = kept[r];
        const bool lng = __ldg(ptr + r + 1) - __ldg(ptr + r) > kLongRow;
        if (k >= 0 && lng) c.x += 1, c.y += k;
        if (k >= 0 && !lng) c.z += 1, c.w += k;
    }
    // exclusive scan over the threads, in thread (= row) order
    int4 inc = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int x = __shfl_up_sync(0xffffffffu, inc.x, d), y = __shfl_up_sync(0xffffffffu, inc.y, d);
        const int z = __shfl_up_sync(0xffffffffu, inc.z, d), w = __shfl_up_sync(0xffffffffu, inc.w, d);
        if (lane >= d) inc.x += x, inc.y += y, inc.z += z, inc.w += w;
    }
    if (lane == 31) s_part[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        int4 v = lane < (int)(blockDim.x >> 5) ? s_part[lane] : make_int4(0, 0, 0, 0);
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int x = __shfl_up_sync(0xffffffffu, v.x, d), y = __shfl_up_sync(0xffffffffu, v.y, d);
            const int z = __shfl_up_sync(0xffffffffu, v.z, d), w = __shfl_up_sync(0xffffffffu, v.w, d);
            if (lane >= d) v.x += x, v.y += y, v.z += z, v.w += w;
        }
        s_part[lane] = v;                                      // inclusive over warps 0 .. lane
    }
    __syncthreads();
    const int4 tot = s_part[31];
    int4 run = make_int4(inc.x - c.x, inc.y - c.y, inc.z - c.z, inc.w - c.w);
    if (warp > 0) {
        const int4 b = s_part[warp - 1];
        run.x += b.x, run.y += b.y, run.z += b.z, run.w += b.w;
    }
    const int L = tot.x, EL = tot.y, N = tot.z;
    for (int r = r0; r < r1; ++r) {
        const int k = kept[r];
        if (k < 0) continue;
        if (__ldg(ptr + r + 1) - __ldg(ptr + r) > kLongRow) {
            out[run.x] = make_int2(r, run.y);
            run.x += 1, run.y += k;
        } else {
            out[L + run.z] = make_int2(r, EL + run.w);
            run.z += 1, run.w += k;
        }
    }
    if (threadIdx.x == 0) {
        out[L + N] = make_int2(-1, EL + tot.w);
        W.count[tile] = L + N;
    }
    __syncthreads();                                           // out[] complete, kept[] free: it holds chunk starts now
    for (int q = threadIdx.x; q < L; q += blockDim.x) hdr[q] = make_int4(q, -1, out[q].y, out[q + 1].y);
    const int Q = chunks - L;
    if (Q < 1) return;
    const long long ES = tot.w, room = (long long)Q * rows_per_cta - N;
    const bool by_count = room <= 0 || ES / room >= (1 << 16);   // then every row weighs the same (Q rows_per_cta >= N)
    const long long cw = by_count ? 1 : max((long long)BLP_U, (ES + room - 1) / room);
    const unsigned long long Wt = (by_count ? 0 : ES) + cw * N;
    auto chunk_of = [&](const int s) -> int {                  // s < N
        const unsigned long long pw = (by_count ? 0 : out[L + s].y - EL) + cw * s;
        return (int)((unsigned __int128)pw * Q / Wt);
    };
    // chunk q starts at the first row s with chunk_of(s) >= q
    for (int s = threadIdx.x; s <= N; s += blockDim.x) {
        const int qs = s < N ? chunk_of(s) : Q, qp = s > 0 ? chunk_of(s - 1) : -1;
        for (int q = qp + 1; q <= qs && q < Q; ++q) kept[q] = s;
    }
    __syncthreads();
    for (int q = threadIdx.x; q < Q; q += blockDim.x) {
        const int k0 = L + kept[q], k1 = L + (q + 1 < Q ? kept[q + 1] : N);
        hdr[L + q] = make_int4(k0, k1 - k0, out[k0].y, out[k1].y);
    }
}

template <bool PRIMAL>
__global__ void __launch_bounds__(kCtaThreads)
k_work_fill(const DevProb P, const DevState S) {
    __shared__ int s_l[2];
    const int tile = blockIdx.y;
    tile_running(S, tile, s_l);
    if (s_l[0] + s_l[1] == 0) return;
    const WorkList& W = PRIMAL ? S.wlC : S.wlR;
    const int rows = PRIMAL ? P.n : P.m;
    const int32_t* __restrict__ ptr = PRIMAL ? P.cptr : P.rowptr;
    const int4* __restrict__ in = reinterpret_cast<const int4*>(PRIMAL ? P.cent : P.ent);
    const int2* __restrict__ act = W.row + (size_t)tile * (rows + 1);
    int4* __restrict__ out = reinterpret_cast<int4*>(W.ent + (size_t)tile * P.nnz);
    const int nact = W.count[tile];
    for (int k = blockIdx.x * kCtaThreads + threadIdx.x; k < nact; k += gridDim.x * kCtaThreads) {
        const int2 v = act[k];
        const int r = v.x, p0 = __ldg(ptr + r), p1 = __ldg(ptr + r + 1);
        int w = v.y;
        if constexpr (PRIMAL) {
            for (int p = p0; p < p1; ++p) {
                const int4 e = __ldg(in + p);
                if (work_entry_kept<true>(P, S, tile, e.x)) out[w++] = e;
            }
            PrimalRowScalars(P, S, 2 * tile, reinterpret_cast<PrimalRec*>(W.rec) + (size_t)tile * rows)(r, k);
        } else {
            const uint8_t* __restrict__ fcol = S.fcol + (size_t)tile * P.n;
            const double* __restrict__ fval = S.fval + (size_t)tile * P.n;
            double c = 0.0;                                    // rconst: sum over the folded columns, in row order
            for (int p = p0; p < p1; ++p) {
                const int4 e = __ldg(in + p);
                if (fcol[e.x]) c = fma(__hiloint2double(e.w, e.z), fval[e.x], c);
                else out[w++] = e;
            }
            reinterpret_cast<DualRec*>(W.rec)[(size_t)tile * rows + k] = DualRec{__ldg(P.b + r), c};
        }
    }
}

// Step size of a tile with frozen coordinates. While the frozen coordinates rest, the iteration of the tile's
// nodes is PDHG on the rows and columns that still move, A_UU, whose norm bounds the step: eta <= 1 / ||A_UU||_2.
// (Round 1 looked for a larger step under the FULL matrix' norm and found none that converges on C5; the norm of
// the active block is the rigorous version: C4 0.47 ||A||, C5 0.86 ||A||, tests/tools/cpu_freeze_lab.py.)
// Power iteration on A_UU' A_UU per tile, warm-started from the tile's previous vector (the sets change slowly):
//   k_pow_A:  w = M_r A M_c (v / ||v||)      one thread per row, ||v||^2 = sum of the previous pass' partials
//   k_pow_AT: v = M_c A' w, partial ||v||^2  one thread per column, fixed-order reductions (deterministic)
//   k_pow_finish: sigma = ||v||^(1/2); eta_tile = min(cap * P.eta, safety / sigma); a node takes a LARGER step only at
//                 a restart or when it was just loaded, a smaller one at once; nodes the watchdog locked stay at P.eta
__global__ void __launch_bounds__(kCtaThreads)
k_pow_init(const DevProb P, const DevState S) {
    const int tile = blockIdx.y;
    for (int j = blockIdx.x * kCtaThreads + threadIdx.x; j < P.n; j += gridDim.x * kCtaThreads)
        S.pv[(size_t)tile * P.n + j] = 1.0;
    if (blockIdx.x == 0 && threadIdx.x < kPowChunks)
        S.ppart[(size_t)tile * kPowChunks + threadIdx.x] = threadIdx.x == 0 ? (double)P.n : 0.0;
}

__global__ void __launch_bounds__(kCtaThreads)
k_pow_A(const DevProb P, const DevState S) {
    const int tile = blockIdx.y;
    double tot = 0.0;
    for (int q = 0; q < kPowChunks; ++q) tot += S.ppart[(size_t)tile * kPowChunks + q];
    const double scale = tot > 0.0 ? rsqrt(tot) : 0.0;
    const uint8_t* __restrict__ ftc = S.ftc + (size_t)tile * P.n;
    const uint8_t* __restrict__ ftr = S.ftr + (size_t)tile * P.m;
    const double* __restrict__ v = S.pv + (size_t)tile * P.n;
    const int4* __restrict__ E = reinterpret_cast<const int4*>(P.ent);
    for (int i = blockIdx.x * kCtaThreads + threadIdx.x; i < P.m; i += gridDim.x * kCtaThreads) {
        double acc = 0.0;
        if (!ftr[i])
            for (int p = __ldg(P.rowptr + i); p < __ldg(P.rowptr + i + 1); ++p) {
                const int4 e = __ldg(E + p);
                if (!ftc[e.x]) acc = fma(__hiloint2double(e.w, e.z), v[e.x], acc);
            }
        S.pw[(size_t)tile * P.m + i] = acc * scale;
    }
}

__global__ void __launch_bounds__(kCtaThreads)
k_pow_AT(const DevProb P, const DevState S) {
    __shared__ double red[kCtaThreads];
    const int tile = blockIdx.y;
    const uint8_t* __restrict__ ftc = S.ftc + (size_t)tile * P.n;
    const double* __restrict__ w = S.pw + (size_t)tile * P.m;
    const int4* __restrict__ E = reinterpret_cast<const int4*>(P.cent);
    double sq = 0.0;
    for (int j = blockIdx.x * kCtaThreads + threadIdx.x; j < P.n; j += gridDim.x * kCtaThreads) {
        double acc = 0.0;
        if (!ftc[j])
            for (int p = __ldg(P.cptr + j); p < __ldg(P.cptr + j + 1); ++p) {
                const int4 e = __ldg(E + p);
                acc = fma(__hiloint2double(e.w, e.z), w[e.x], acc);     // w is zero on frozen rows
            }
        S.pv[(size_t)tile * P.n + j] = acc;
        sq = fma(acc, acc, sq);
    }
    red[threadIdx.x] = sq;
    __syncthreads();
    for (int h = kCtaThreads / 2; h > 0; h >>= 1) {
        if (threadIdx.x < h) red[threadIdx.x] += red[threadIdx.x + h];
        __syncthreads();
    }
    if (threadIdx.x == 0) S.ppart[(size_t)tile * kPowChunks + blockIdx.x] = red[0];
}

__global__ void __launch_bounds__(kBlk)
k_pow_finish(const DevProb P, const DevState S, const double safety, const double cap, const int mode) {
    const int tile = blockIdx.x, node = tile * kBlk + threadIdx.x;
    double tot = 0.0;
    for (int q = 0; q < kPowChunks; ++q) tot += S.ppart[(size_t)tile * kPowChunks + q];
    const double sigma = sqrt(sqrt(tot));          // ||A_UU' A_UU v|| for a unit v: the largest singular value, squared
    double et = cap * P.eta;
    if (sigma > 0.0) et = fmin(et, safety / sigma);
    et = fmax(et, P.eta);
    if (threadIdx.x == 0) S.eta_tile[tile] = et;
    if (node >= S.B || S.fin[node] != 0) return;
    const bool may_raise = S.restart[node] != 0 || mode == 2 || (mode == 1 && S.fresh[node] != 0);
    const double cur = S.eta[node];
    const double nxt = (may_raise && !S.eta_lock[node]) ? et : fmin(cur, et);
    if (nxt != cur) {
        // the fixed-point error is measured in the step's own metric, ~ sqrt(eta) for the same move: keep the
        // restart rule's and the watchdog's references comparable across the change
        const double f = sqrt(nxt / cur);
        S.eta[node] = nxt;
        S.fpe0[node] *= f;
        S.fpe_prev[node] *= f;
    }
}

__global__ void k_eta_reset(const DevProb P, const DevState S) {
    const int node = blockIdx.x * blockDim.x + threadIdx.x;
    if (node >= S.ld) return;
    const double cur = S.eta[node];
    if (cur != P.eta) {
        const double f = sqrt(P.eta / cur);
        S.fpe0[node] *= f;
        S.fpe_prev[node] *= f;
    }
    S.eta[node] = P.eta;
}

// Frozen (coordinate, running node) pairs of the whole batch, as the step kernels will see them (both 32-node
// blocks of a tile agree): counters[8..9] = columns, counters[10..11] = rows, as two 64-bit counts. One CTA per tile.
__global__ void __launch_bounds__(kCtaThreads)
k_freeze_count(const DevProb P, const DevState S) {
    __shared__ int s_live[2];
    __shared__ unsigned long long s_cnt[2];
    const int tile = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x < 2) s_cnt[threadIdx.x] = 0ull;
    if (warp < 2) {
        const int node = tile * kBlk + warp * 32 + lane;
        const unsigned bal = __ballot_sync(0xffffffffu, node < S.B && S.fin[node] == 0);
        if (lane == 0) s_live[warp] = __popc(bal);
    }
    __syncthreads();
    const int l0 = s_live[0], l1 = s_live[1];
    if (l0 + l1 == 0) return;
    unsigned long long cnt[2] = {0ull, 0ull};
#pragma unroll
    for (int a = 0; a < 2; ++a) {
        const int rows = a == 0 ? P.n : P.m;
        const uint8_t* __restrict__ f0 = (a == 0 ? S.cfrz : S.rfrz) + (size_t)(2 * tile) * rows;
        const uint8_t* __restrict__ f1 = f0 + rows;
        int c = 0;
        for (int r = threadIdx.x; r < rows; r += kCtaThreads)
            c += ((l0 == 0 || f0[r] != 0) && (l1 == 0 || f1[r] != 0)) ? 1 : 0;
        cnt[a] = (unsigned long long)c * (unsigned long long)(l0 + l1);
    }
    atomicAdd(&s_cnt[0], cnt[0]);
    atomicAdd(&s_cnt[1], cnt[1]);
    __syncthreads();
    if (threadIdx.x < 2)
        atomicAdd(reinterpret_cast<unsigned long long*>(S.counters + 8) + threadIdx.x, s_cnt[threadIdx.x]);
}

// ---------------------------------------------------------------------------------------------
// Set-up: scale the per-node bounds into the solver's space and build the start point.
__global__ void __launch_bounds__(kCtaThreads)
k_init_cols(const DevProb P, const DevState S, const double* __restrict__ lb,
            const double* __restrict__ ub, const double* __restrict__ x0, const int ld_in) {
    const size_t total = (size_t)P.n * S.ld;
    for (size_t e = (size_t)blockIdx.x * kCtaThreads + threadIdx.x; e < total;
         e += (size_t)gridDim.x * kCtaThreads) {
        const int j = (int)(e / S.ld), node = (int)(e % S.ld);
        double lo = 0.0, hi = 0.0, x = 0.0;
        if (node < S.B) {
            const double f = P.sb / P.dc[j];
            const size_t ei = (size_t)j * ld_in + node;
            const double a = lb[ei], b = ub[ei];
            lo = is_inf(a) ? (a > 0 ? INFINITY : -INFINITY) : a * f;
            hi = is_inf(b) ? (b > 0 ? INFINITY : -INFINITY) : b * f;
            x = x0 ? x0[ei] * f : 0.0;
            x = fmin(fmax(x, lo), hi);
        }
        if (lo > hi) {              // empty box: primal infeasible without any iteration
            S.fin[node] = 1; S.status[node] = 1; S.pobj[node] = INFINITY; S.dobj[node] = INFINITY;
        }
        const size_t t = tix(j, node, P.n);
        S.l[t] = lo; S.u[t] = hi; S.xa[t] = (anc_t)x; S.xbar[t] = x; S.X1[t] = x;
        S.DX[t] = 0.0; S.G[t] = 0.0;
    }
}

__global__ void __launch_bounds__(kCtaThreads)
k_init_rows(const DevProb P, const DevState S, const double* __restrict__ y0, const int ld_in) {
    const size_t total = (size_t)P.m * S.ld;
    for (size_t e = (size_t)blockIdx.x * kCtaThreads + threadIdx.x; e < total;
         e += (size_t)gridDim.x * kCtaThreads) {
        const int i = (int)(e / S.ld), node = (int)(e % S.ld);
        double y = 0.0;
        if (node < S.B && y0) {
            y = fmax(0.0, y0[(size_t)i * ld_in + node] * P.sc / P.dr[i]);
            if (i >= P.m_base && S.rowmask && S.rowmask[(size_t)(i - P.m_base) * S.ld + node] == 0)
                y = 0.0;
        }
        const size_t t = tix(i, node, P.m);
        S.y[t] = y; S.ya[t] = (anc_t)y; S.Y1[t] = y; S.DY[t] = 0.0;
    }
}

// Row-activity bound test (the cheap infeasibility screen for branching children, e.g. the
// right child x2 >= 2 of small_branch against x0 + x2 <= 1.5): a row whose largest possible
// activity over the node's box stays below its lower bound proves the node LP infeasible.
template <int NT>
__global__ void __launch_bounds__(kCtaThreads)
k_check_rows(const DevProb P, const DevState S, const int rows_per_cta, const int only_fresh) {
    constexpr int RW = 32 / NT;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int node = blockIdx.y * NT + (lane % NT);
    const int sub = lane / NT;
    const bool node_ok = node < S.B && (!only_fresh || S.fresh[node] != 0);
    if (__ballot_sync(0xffffffffu, node_ok) == 0) return;
    const int r0 = blockIdx.x * rows_per_cta;
    const int r1 = min(P.m, r0 + rows_per_cta);
    for (int ib = r0 + warp * RW; ib < r1; ib += kWarps * RW) {
        const int i = ib + sub;
        if (i >= r1 || !node_ok) continue;
        if (i >= P.m_base && S.rowmask && S.rowmask[(size_t)(i - P.m_base) * S.ld + node] == 0)
            continue;
        double act = 0.0, mag = 0.0;
        for (int p = __ldg(P.rowptr + i); p < __ldg(P.rowptr + i + 1); ++p) {
            const double a = P.ent[p].val;
            const size_t e = tix(P.ent[p].idx, node, P.n);
            const double t = a * (a > 0.0 ? S.u[e] : S.l[e]);
            act += t;
            mag += fabs(t);
        }
        const double bi = __ldg(P.b + i);
        if (bi - act > 1e-9 * (fabs(bi) + mag) + 1e-300) {
            S.fin[node] = 1; S.status[node] = 1; S.pobj[node] = INFINITY; S.dobj[node] = INFINITY;
        }
    }
}

// (re)build the per-block reference bounds and deviation masks from the dense l,u state
__global__ void __launch_bounds__(kCtaThreads)
k_build_lumask(const DevProb P, const DevState S) {
    const int lane = threadIdx.x & 31;
    const size_t gwarp = ((size_t)blockIdx.x * kCtaThreads + threadIdx.x) >> 5;
    const size_t nwarps = ((size_t)gridDim.x * kCtaThreads) >> 5;
    const int blocks = (S.B + 31) >> 5;
    const size_t total = (size_t)blocks * P.n;
    for (size_t w = gwarp; w < total; w += nwarps) {
        const int blk = (int)(w / P.n), j = (int)(w % P.n);
        const int node = blk * 32 + lane;
        const size_t e = tix(j, node, P.n);
        const double lo = S.l[e], hi = S.u[e];
        const double lr = __shfl_sync(0xffffffffu, lo, 0), ur = __shfl_sync(0xffffffffu, hi, 0);
        const bool dev = node < S.B && (lo != lr || hi != ur);
        const unsigned mk = __ballot_sync(0xffffffffu, dev);
        if (lane == 0) {
            S.lumask[w] = mk;
            S.lref[w] = lr;
            S.uref[w] = ur;
        }
    }
}

// counters[0] += running nodes, counters[3] += nodes decided at set-up and not yet harvested
__global__ void k_count_active(const DevState S) {
    const int node = blockIdx.x * blockDim.x + threadIdx.x;
    if (node >= S.B) return;
    const int f = S.fin[node];
    if (f == 0) atomicAdd(S.counters + 0, 1);
    else if (f == 1) atomicAdd(S.counters + 3, 1);
}

__global__ void k_init_nodes(const DevProb P, const DevState S) {
    const int node = blockIdx.x * blockDim.x + threadIdx.x;
    if (node >= S.ld) return;
    S.omega[node] = P.omega0;
    S.fpe0[node] = INFINITY;
    S.fpe_prev[node] = INFINITY;
    S.pobj[node] = 0.0;
    S.dobj[node] = -INFINITY;
    S.sbase[node] = 0;
    S.fin[node] = node < S.B ? 0 : 2;
    S.status[node] = 3;
    S.iters[node] = 0;
    S.restart[node] = 0;
    S.origin[node] = node;
    S.start[node] = 0;
    S.fresh[node] = 0;
    S.eta[node] = P.eta;
    S.eta_lock[node] = 0;
}

// ---------------------------------------------------------------------------------------------
// Refill (continuous batching, blp_opts.max_active < B): the batch holds S.B node SLOTS; a slot
// whose node has been harvested (fin == 2) takes the next pending node of the caller's batch, so
// the step kernels keep sweeping a full-width batch while a long frontier drains, instead of
// narrowing towards the slowest node of every slice.
//   k_refill_plan (one CTA): free slots in ascending order get nodes next, next+1, ... (nnew of
//                 them); per-slot scalars are reset; newlist[q] = slot of the q-th new node
//   k_refill_cols / k_refill_rows: the new slots' state columns, as k_init_cols / k_init_rows
__global__ void __launch_bounds__(1024) k_refill_plan(const DevProb P, const DevState S, const int next,
                                                      const int nnew) {
    __shared__ int wsum[32];
    __shared__ int base_s;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) base_s = 0;
    __syncthreads();
    const int now = S.counters[2];
    for (int c0 = 0; c0 < S.B; c0 += 1024) {
        const int k = c0 + tid;
        const bool free_slot = k < S.B && S.fin[k] == 2;
        const unsigned bal = __ballot_sync(0xffffffffu, free_slot);
        if (lane == 0) wsum[warp] = __popc(bal);
        __syncthreads();
        int before = base_s;
        for (int w = 0; w < warp; ++w) before += wsum[w];
        const int q = before + __popc(bal & ((1u << lane) - 1u));
        int total = 0;
        for (int w = 0; w < 32; ++w) total += wsum[w];
        __syncthreads();
        const bool take = free_slot && q < nnew;
        if (k < S.B) S.fresh[k] = take ? 1 : 0;
        if (take) {
            S.newlist[q] = k;
            S.origin[k] = next + q;
            S.start[k] = now;
            S.omega[k] = P.omega0;
            S.fpe0[k] = INFINITY;
            S.fpe_prev[k] = INFINITY;
            S.pobj[k] = 0.0;
            S.dobj[k] = -INFINITY;
            S.sbase[k] = 0;
            S.fin[k] = 0;
            S.status[k] = 3;
            S.iters[k] = 0;
            S.restart[k] = 0;
            S.eta[k] = P.eta;
            S.eta_lock[k] = 0;
        }
        if (tid == 0) base_s += total;
        __syncthreads();
    }
    if (tid == 0) {
        S.counters[0] = 0;
        S.counters[3] = 0;
    }
}

__global__ void __launch_bounds__(kCtaThreads)
k_refill_cols(const DevProb P, const DevState S, const double* __restrict__ lb,
              const double* __restrict__ ub, const double* __restrict__ x0, const int ld_in,
              const int nnew) {
    const size_t total = (size_t)P.n * nnew;
    for (size_t e = (size_t)blockIdx.x * kCtaThreads + threadIdx.x; e < total;
         e += (size_t)gridDim.x * kCtaThreads) {
        const int j = (int)(e / nnew), slot = S.newlist[e % nnew];
        const size_t ei = (size_t)j * ld_in + S.origin[slot];
        const double f = P.sb / P.dc[j];
        const double a = lb[ei], b = ub[ei];
        const double lo = is_inf(a) ? (a > 0 ? INFINITY : -INFINITY) : a * f;
        const double hi = is_inf(b) ? (b > 0 ? INFINITY : -INFINITY) : b * f;
        const double x = fmin(fmax(x0 ? x0[ei] * f : 0.0, lo), hi);
        if (lo > hi) {
            S.fin[slot] = 1; S.status[slot] = 1; S.pobj[slot] = INFINITY; S.dobj[slot] = INFINITY;
        }
        const size_t t = tix(j, slot, P.n);
        S.l[t] = lo; S.u[t] = hi; S.xa[t] = (anc_t)x; S.xbar[t] = x; S.X1[t] = x;
        S.DX[t] = 0.0; S.G[t] = 0.0;
    }
}

__global__ void __launch_bounds__(kCtaThreads)
k_refill_rows(const DevProb P, const DevState S, const double* __restrict__ y0,
              const uint8_t* __restrict__ row_mask, const int ld_in, const int nnew) {
    const size_t total = (size_t)P.m * nnew;
    for (size_t e = (size_t)blockIdx.x * kCtaThreads + threadIdx.x; e < total;
         e += (size_t)gridDim.x * kCtaThreads) {
        const int i = (int)(e / nnew), slot = S.newlist[e % nnew];
        const int org = S.origin[slot];
        bool on = true;
        if (i >= P.m_base && S.rowmask) {
            const uint8_t v = row_mask[(size_t)(i - P.m_base) * ld_in + org];
            S.rowmask[(size_t)(i - P.m_base) * S.ld + slot] = v;
            on = v != 0;
        }
        const double y = (y0 && on) ? fmax(0.0, y0[(size_t)i * ld_in + org] * P.sc / P.dr[i]) : 0.0;
        const size_t t = tix(i, slot, P.m);
        S.y[t] = y; S.ya[t] = (anc_t)y; S.Y1[t] = y; S.DY[t] = 0.0;
    }
}

// Harvest: nodes that received a status in the last evaluation (fin == 1) hand their results to
// the caller's arrays at their ORIGINAL node index; afterwards they are marked fin = 2 and the next
// compaction drops their columns.
//   k_harvest_x: x = X1 * dc / sb, plus per-chunk partials of the most fractional integer column
//   k_harvest_y: y = Y1 * dr / sc
//   k_harvest_nodes: per-node scalars, fold of the fractionality partials (ties -> smaller index)
template <int NT>
__global__ void __launch_bounds__(kCtaThreads)
k_harvest_x(const DevProb P, const DevState S, const DevOut O, const double frac_eps,
            const int rows_per_cta) {
    constexpr int RW = 32 / NT;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int node = blockIdx.y * NT + (lane % NT);
    const int sub = lane / NT;
    const bool node_ok = node < S.B && S.fin[node] == 1;
    if (__ballot_sync(0xffffffffu, node_ok) == 0) return;     // uniform over the CTA
    const int org = node_ok ? S.origin[node] : 0;
    const double inv = 1.0 / P.sb;
    double best = frac_eps;
    int besti = 0x7fffffff;
    const int r0 = blockIdx.x * rows_per_cta;
    const int r1 = min(P.n, r0 + rows_per_cta);
    for (int jb = r0 + warp * RW; jb < r1; jb += kWarps * RW) {
        const int j = jb + sub;
        if (j < r1 && node_ok) {
            const double v = S.X1[tix(j, node, P.n)] * __ldg(P.dc + j) * inv;
            if (O.x) O.x[(size_t)j * O.ld + org] = v;
            if (S.isint && S.isint[j]) {
                const double dist = fmin(v - floor(v), ceil(v) - v);
                if (dist > best) { best = dist; besti = j; }      // ascending j per lane: first wins
            }
        }
    }
    __shared__ double sd[kCtaThreads];
    __shared__ int si[kCtaThreads];
    sd[threadIdx.x] = best;
    si[threadIdx.x] = besti;
    __syncthreads();
    if (threadIdx.x < NT) {
        double bd = sd[threadIdx.x];
        int bi = si[threadIdx.x];
        for (int q = threadIdx.x + NT; q < kCtaThreads; q += NT)
            if (sd[q] > bd || (sd[q] == bd && si[q] < bi)) { bd = sd[q]; bi = si[q]; }
        const int nd = blockIdx.y * NT + threadIdx.x;
        if (nd < S.ld) {
            S.fracD[(size_t)blockIdx.x * S.ld + nd] = bd;
            S.fracI[(size_t)blockIdx.x * S.ld + nd] = bi;
        }
    }
}

template <int NT>
__global__ void __launch_bounds__(kCtaThreads)
k_harvest_y(const DevProb P, const DevState S, const DevOut O, const int rows_per_cta) {
    constexpr int RW = 32 / NT;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int node = blockIdx.y * NT + (lane % NT);
    const int sub = lane / NT;
    const bool node_ok = node < S.B && S.fin[node] == 1;
    if (__ballot_sync(0xffffffffu, node_ok) == 0) return;
    const int org = node_ok ? S.origin[node] : 0;
    const double inv = 1.0 / P.sc;
    const int r0 = blockIdx.x * rows_per_cta;
    const int r1 = min(P.m, r0 + rows_per_cta);
    for (int ib = r0 + warp * RW; ib < r1; ib += kWarps * RW) {
        const int i = ib + sub;
        if (i < r1 && node_ok)
            O.y[(size_t)i * O.ld + org] = S.Y1[tix(i, node, P.m)] * __ldg(P.dr + i) * inv;
    }
}

__global__ void k_harvest_nodes(const DevProb P, const DevState S, const DevOut O, const int chunks,
                                const double frac_eps, const int have_frac) {
    const int node = blockIdx.x * blockDim.x + threadIdx.x;
    if (node >= S.B || S.fin[node] != 1) return;
    const int org = S.origin[node];
    const int st = S.status[node];
    if (O.obj) O.obj[org] = S.pobj[node];
    if (O.lower) O.lower[org] = S.dobj[node];
    if (O.status) O.status[org] = st;
    if (O.iters) O.iters[org] = S.iters[node];
    if (O.frac_idx) {
        int bi = -1;
        if (st == 0 && have_frac) {
            double bd = frac_eps;
            int cand = 0x7fffffff;
            for (int ch = 0; ch < chunks; ++ch) {
                const double d = S.fracD[(size_t)ch * S.ld + node];
                const int i = S.fracI[(size_t)ch * S.ld + node];
                if (d > bd || (d == bd && i < cand)) { bd = d; cand = i; }
            }
            if (cand != 0x7fffffff) bi = cand;
        }
        O.frac_idx[org] = bi;
    }
    S.fin[node] = 2;
}

// output slots of the padding columns B..ld-1
__global__ void k_out_pad(const DevOut O, const int B, const int ld) {
    const int k = B + blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= ld) return;
    if (O.obj) O.obj[k] = 0.0;
    if (O.lower) O.lower[k] = 0.0;
    if (O.status) O.status[k] = -1;
    if (O.iters) O.iters[k] = 0;
    if (O.frac_idx) O.frac_idx[k] = -1;
}

// Compaction: running nodes (fin == 0) move to the front of the batch, keeping their order, so
// that retired node columns stop costing bandwidth. One CTA plans the move and permutes the
// per-node scalars; k_compact_vecs then moves every state row in place (a column only ever moves
// to a smaller index, and each warp sweeps its row in ascending order, so nothing unread is
// overwritten).
__global__ void __launch_bounds__(1024) k_compact_plan(const DevState S) {
    __shared__ int wsum[32];
    __shared__ int base_s;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) base_s = 0;
    __syncthreads();
    for (int c0 = 0; c0 < S.B; c0 += 1024) {
        const int k = c0 + tid;
        const bool keep = k < S.B && S.fin[k] == 0;
        double om = 0, f0 = 0, fp = 0, po = 0, dq = 0, et = 0;
        int sb = 0, stt = 0, itr = 0, org = 0, beg = 0, lck = 0;
        if (keep) {
            om = S.omega[k]; f0 = S.fpe0[k]; fp = S.fpe_prev[k]; po = S.pobj[k]; dq = S.dobj[k];
            sb = S.sbase[k]; stt = S.status[k]; itr = S.iters[k]; org = S.origin[k]; beg = S.start[k];
            et = S.eta[k]; lck = S.eta_lock[k];
        }
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) wsum[warp] = __popc(bal);
        __syncthreads();
        int before = base_s;
        for (int w = 0; w < warp; ++w) before += wsum[w];
        const int pos = before + __popc(bal & ((1u << lane) - 1u));
        int total = 0;
        for (int w = 0; w < 32; ++w) total += wsum[w];
        __syncthreads();
        if (k < S.B) S.newpos[k] = keep ? pos : -1;
        if (keep) {
            S.omega[pos] = om; S.fpe0[pos] = f0; S.fpe_prev[pos] = fp; S.pobj[pos] = po; S.dobj[pos] = dq;
            S.sbase[pos] = sb; S.status[pos] = stt; S.iters[pos] = itr; S.origin[pos] = org;
            S.start[pos] = beg;
            S.eta[pos] = et; S.eta_lock[pos] = lck;
        }
        if (tid == 0) base_s += total;
        __syncthreads();
    }
    const int nb = base_s;
    for (int k = tid; k < S.ld; k += 1024) {
        S.fin[k] = k < nb ? 0 : 2;
        S.restart[k] = 0;
    }
    if (tid == 0) S.counters[4] = nb;
}

__global__ void __launch_bounds__(kCtaThreads)
k_compact_vecs(const DevProb P, const DevState S, const int oldB) {
    const int lane = threadIdx.x & 31;
    const int gwarp = (blockIdx.x * kCtaThreads + threadIdx.x) >> 5;
    const int nwarps = (gridDim.x * kCtaThreads) >> 5;
    const int mc = S.rowmask ? P.m - P.m_base : 0;
    const int ncol = 5 * P.n, nrow = 3 * P.m;         // xbar, xa, l, u, X1; y, ya, Y1 (x', y' feed the freezing rule)
    const int total = ncol + nrow + mc;
    // one state row (512-byte segments of all node blocks) per warp and pass
    auto move_row = [&](auto* arr, const int row, const int rows) {
        for (int c0 = 0; c0 < oldB; c0 += 32) {
            const int k = c0 + lane;
            const int p = k < oldB ? S.newpos[k] : -1;
            const auto v = p >= 0 ? arr[tix(row, k, rows)] : 0;
            __syncwarp();
            if (p >= 0) arr[tix(row, p, rows)] = v;
        }
    };
    for (int r = gwarp; r < total; r += nwarps) {
        if (r < ncol + nrow) {
            if (r < ncol) {
                const int a = r / P.n, row = r % P.n;
                if (a == 1) move_row(S.xa, row, P.n);
                else move_row(a == 0 ? S.xbar : a == 2 ? S.l : a == 3 ? S.u : S.X1, row, P.n);
            } else {
                const int q = r - ncol, a = q / P.m, row = q % P.m;
                if (a == 1) move_row(S.ya, row, P.m);
                else move_row(a == 0 ? S.y : S.Y1, row, P.m);
            }
        } else {
            uint8_t* base = S.rowmask + (size_t)(r - ncol - nrow) * S.ld;
            for (int c0 = 0; c0 < oldB; c0 += 32) {
                const int k = c0 + lane;
                const int p = k < oldB ? S.newpos[k] : -1;
                const uint8_t v = p >= 0 ? base[k] : 0;
                __syncwarp();
                if (p >= 0) base[p] = v;
            }
        }
    }
}

__global__ void k_set_isint(const int32_t* __restrict__ int_idx, const int n_int, const int n,
                            uint8_t* __restrict__ isint) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q < n_int) {
        const int j = int_idx[q];
        if (j >= 0 && j < n) isint[j] = 1;
    }
}

// ---------------------------------------------------------------------------------------------
// Plain batched SpMV on the unscaled matrix (parity tests, SpMV roofline measurement).
template <int NT>
__global__ void __launch_bounds__(kCtaThreads)
k_spmv(const int32_t* __restrict__ ptr, const Ent* __restrict__ ent, const int rows, const int B,
       const int ld,
       const double* __restrict__ X, double* __restrict__ Y, const int rows_per_cta, const int cap) {
    constexpr int RW = 32 / NT;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int node = blockIdx.y * NT + (lane % NT);
    const int sub = lane / NT;
    const bool node_ok = node < B;
    const int r0 = blockIdx.x * rows_per_cta;
    const int r1 = min(rows, r0 + rows_per_cta);
    const Slab sl = stage_slab(ptr, ent, r0, r1, rows_per_cta, cap);
    for (int ib = r0 + warp * RW; ib < r1; ib += kWarps * RW) {
        const int i = ib + sub;
        const bool row_ok = i < r1;
        const double s = slab_dot<NT>(sl, ent, row_ok ? i - r0 : 0, row_ok, X + node, ld,
                                      node_ok && row_ok);
        if (row_ok && node_ok) Y[(size_t)i * ld + node] = s;
    }
}

// The same with two nodes per lane (B >= 64): a warp owns one matrix row for 64 nodes, every access is
// one 128-bit load / store per lane, the CSR chunk of the CTA is staged in shared memory.
__global__ void __launch_bounds__(kCtaThreads, BLP_MINB2)
k_spmv2(const int32_t* __restrict__ ptr, const Ent* __restrict__ ent, const int rows, const int B,
        const int ld, const double* __restrict__ X, double* __restrict__ Y, const int rows_per_cta,
        const int cap) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int node = blockIdx.y * kBlk + lane * 2;
    const int r0 = blockIdx.x * rows_per_cta;
    const int r1 = min(rows, r0 + rows_per_cta);
    const Slab sl = stage_slab(ptr, ent, r0, r1, rows_per_cta, cap);
    const bool k0 = node < B, k1 = node + 1 < B;
    if (node >= ld) return;                                    // ld is a multiple of 64: never taken
    for (int i = r0 + warp; i < r1; i += kWarps) {
        double g0 = 0.0, g1 = 0.0;
        slab_dot2(sl, ent, i - r0, X + node, g0, g1, ld);
        st2(Y + (size_t)i * ld + node, make_double2(g0, g1), k0, k1);
    }
}

// node-major host order [B][rows]  <->  node-fastest device order [rows][ld] (tiled transpose)
__global__ void k_transpose_in(const double* __restrict__ src, const int B, const int rows,
                               const int ld, double* __restrict__ dst) {
    __shared__ double tile[32][33];
    const int r0 = blockIdx.x * 32, k0 = blockIdx.y * 32;
    for (int q = threadIdx.y; q < 32; q += blockDim.y) {
        const int k = k0 + q, r = r0 + threadIdx.x;
        tile[q][threadIdx.x] = (k < B && r < rows) ? src[(size_t)k * rows + r] : 0.0;
    }
    __syncthreads();
    for (int q = threadIdx.y; q < 32; q += blockDim.y) {
        const int r = r0 + q, k = k0 + threadIdx.x;
        if (r < rows && k < ld) dst[(size_t)r * ld + k] = tile[threadIdx.x][q];
    }
}

__global__ void k_transpose_out(const double* __restrict__ src, const int B, const int rows,
                                const int ld, double* __restrict__ dst) {
    __shared__ double tile[32][33];
    const int r0 = blockIdx.x * 32, k0 = blockIdx.y * 32;
    for (int q = threadIdx.y; q < 32; q += blockDim.y) {
        const int r = r0 + q, k = k0 + threadIdx.x;
        tile[q][threadIdx.x] = (r < rows && k < ld) ? src[(size_t)r * ld + k] : 0.0;
    }
    __syncthreads();
    for (int q = threadIdx.y; q < 32; q += blockDim.y) {
        const int k = k0 + q, r = r0 + threadIdx.x;
        if (k < B && r < rows) dst[(size_t)k * rows + r] = tile[threadIdx.x][q];
    }
}

__global__ void k_transpose_in_u8(const uint8_t* __restrict__ src, const int B, const int rows,
                                  const int ld, uint8_t* __restrict__ dst) {
    const size_t total = (size_t)rows * ld;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total;
         e += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(e / ld), k = (int)(e % ld);
        dst[e] = k < B ? src[(size_t)k * rows + r] : 0;
    }
}

// children-of-one-parent bounds: broadcast the parent's vectors, then patch the deltas
__global__ void k_broadcast_rows(const double* __restrict__ v, const int rows, const int ld,
                                 double* __restrict__ dst) {
    const size_t total = (size_t)rows * ld;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total;
         e += (size_t)gridDim.x * blockDim.x)
        dst[e] = v[e / ld];
}

__global__ void k_patch_bounds(const int B, const int ld, const int32_t* __restrict__ dptr,
                               const int32_t* __restrict__ dvar, const double* __restrict__ dlb,
                               const double* __restrict__ dub, double* __restrict__ lb,
                               double* __restrict__ ub) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= B) return;
    for (int p = dptr[k]; p < dptr[k + 1]; ++p) {
        lb[(size_t)dvar[p] * ld + k] = dlb[p];
        ub[(size_t)dvar[p] * ld + k] = dub[p];
    }
}

}  // namespace blp
