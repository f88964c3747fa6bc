// Batched bounded dual simplex for SMALL node LPs (rows <= kSxMaxRows): one CTA per node LP.
//
// Why it exists next to the PDHG kernels: the reference's Node API reads a simplex VERTEX and a
// BASIS (integrality test base_node.py:281-283, most fractional index :544-562, tableau :513-530,
// getBasisStatus/setBasisStatus :589, 608, "maxNumIteration pivots" :645-646). A first-order method
// converges to a point of the optimal face; for the LP sizes of configs 1-3 a dense-inverse dual
// simplex per node is both exact and faster. A batch (frontier, strong-branching children) is one
// launch: blockIdx.x = node, the CTA's threads share the node's O(m^2) work.
//
// LP of a node:  min c.x,  A x - s = b,  l <= x <= u,  s >= 0  (s free where the row is masked off).
// State per node in global memory: Binv (m x m, ROW major, leading dimension ldm: a warp streams a whole
// row of it in the update sweep, and the row the ratio test needs is one contiguous read),
// x_B, reduced costs d, basis head, status, DSE weights. Pivoting rules, tolerances and the ORDER OF
// EVERY FLOATING-POINT OPERATION are those of oracle/dual_simplex.py (the numpy restatement the tests
// compare against pivot for pivot): single rounded operations only (__dmul_rn/__dadd_rn, no FMA
// contraction), sums in ascending index order, row norms in 16 interleaved partial sums.
#pragma once
#include <cstdint>
#include <cooperative_groups.h>
#include <cuda_runtime.h>

#include "blp_kernels.cuh"

namespace blp {

constexpr int kSxMaxRows = 1024;          // one CTA per node (k_simplex)
constexpr int kSxMaxRowsWide = 8192;      // a group of SMs per node (k_simplex_wide, cooperative launch)
constexpr int kSxWeightLanes = 16;
constexpr int SX_BASIC = 1, SX_UPPER = 2, SX_LOWER = 3;
constexpr double kSxPrimalTol = 1e-9, kSxDualTol = 1e-9, kSxPivTol = 1e-9, kSxTieRel = 1e-12;
constexpr double kSxRatioBin = 68719476736.0;      // 2^36
constexpr double kSxBig = 1e8;
constexpr int kSxRefactorEvery = 1000;     // ... or 2 m pivots if that is more
constexpr double kSxPivotMismatch = 1e-7; // |alpha_q[r] - alpha_r[q]| relative: refactorise before pivoting

struct SxProb {
    int m, m_base, n, ldm;
    const int32_t* rowptr; const Ent* ent;     // unscaled A, CSR (entries ascending by column)
    const int32_t* cptr;   const Ent* cent;    // unscaled A', CSR (entries ascending by row)
    const double* c; const double* b;          // unscaled objective / row lower bounds
};

// per-call arrays; node k uses slice k of each
struct SxBatch {
    int B, max_pivots;
    double pivot_mismatch;                     // kSxPivotMismatch (a tuning build reads BLP_SX_MISMATCH)
    int refactor_every;                        // 0: max(kSxRefactorEvery, 2 m) (BLP_SX_REFACTOR_EVERY)
    const double* lb; const double* ub;        // [B][n] node major
    const uint8_t* rowon;                      // [B][m - m_base] or null (all pool rows on)
    const int8_t* cstat_in; const int8_t* rstat_in;   // [B][n], [B][m] CLP codes, or null = slack basis
    const int32_t* parent;                     // [B] slot of the source store to start from (-1: from status), or null
    // factor stores: this call's (written) and the previous call's (read when parent >= 0)
    double* Binv; int32_t* head; int8_t* stat; double* wts;
    const double* pBinv; const int32_t* phead; const int8_t* pstat; const double* pwts;
    double* work;                              // [B][work_stride] doubles
    size_t work_stride;
    // outputs
    double* obj; int32_t* status; int32_t* pivots; int32_t* flips;
    double* x; double* y; double* rc;          // [B][n], [B][m], [B][n]
    int8_t* cstat_out; int8_t* rstat_out;      // [B][n], [B][m]
};

__device__ __forceinline__ double sx_mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double sx_add(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double sx_sub(double a, double b) { return __dsub_rn(a, b); }

// ---- block reductions (deterministic: max / min are order independent) ---------------------------
struct SxRed {
    double d[32];
    int i[32];
    double bd;
    int bi;
};

__device__ __forceinline__ double sx_block_max(double v, SxRed& s) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    __syncthreads();
    if (lane == 0) s.d[warp] = v;
    __syncthreads();
    if (warp == 0) {
        double t = lane < nw ? s.d[lane] : -INFINITY;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t = fmax(t, __shfl_xor_sync(0xffffffffu, t, o));
        if (lane == 0) s.bd = t;
    }
    __syncthreads();
    return s.bd;
}

__device__ __forceinline__ int sx_block_min_int(int v, SxRed& s) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
    __syncthreads();
    if (lane == 0) s.i[warp] = v;
    __syncthreads();
    if (warp == 0) {
        int t = lane < nw ? s.i[lane] : 2147483647;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t = min(t, __shfl_xor_sync(0xffffffffu, t, o));
        if (lane == 0) s.bi = t;
    }
    __syncthreads();
    return s.bi;
}

// lexicographic minimum of (key ascending, |alpha| descending, index ascending)
struct SxCand {
    double key, mag;
    int j;
};
__device__ __forceinline__ bool sx_better(const SxCand& a, const SxCand& b) {
    if (a.key != b.key) return a.key < b.key;
    if (a.mag != b.mag) return a.mag > b.mag;
    return a.j < b.j;
}
__device__ __forceinline__ SxCand sx_shfl(const SxCand& c, int o) {
    SxCand r;
    r.key = __shfl_xor_sync(0xffffffffu, c.key, o);
    r.mag = __shfl_xor_sync(0xffffffffu, c.mag, o);
    r.j = __shfl_xor_sync(0xffffffffu, c.j, o);
    return r;
}
struct SxCandRed {
    SxCand w[32];
    SxCand best;
};
__device__ __forceinline__ SxCand sx_block_best(SxCand c, SxCandRed& s) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const SxCand t = sx_shfl(c, o);
        if (sx_better(t, c)) c = t;
    }
    __syncthreads();
    if (lane == 0) s.w[warp] = c;
    __syncthreads();
    if (warp == 0) {
        SxCand t;
        t.key = INFINITY; t.mag = 0.0; t.j = 2147483647;
        if (lane < nw) t = s.w[lane];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const SxCand q = sx_shfl(t, o);
            if (sx_better(q, t)) t = q;
        }
        if (lane == 0) s.best = t;
    }
    __syncthreads();
    return s.best;
}


// ---- the team that works on ONE node: a CTA (k_simplex) or a group of CTAs of the cooperative grid (k_simplex_wide) ----
// Array work (the O(m^2) sweep, row / column dots, vector updates) is split over the team's threads and
// followed by a team barrier. DECISIONS (pricing, ratio test, pivot row of a factorisation step) are
// taken by every CTA for itself from the shared arrays: the reductions are max / min / lexicographic min
// over all m or n+m elements — cheap, order independent, so every CTA reaches the same decision and the
// scalars live in its own shared memory; no cross-CTA reduction, no barrier per decision. A group team
// therefore needs 5 barriers per pivot (8 with bound flips) and both teams compute bit-identical results.
struct SxCtrl {            // per-CTA scalars: one thread decides, the CTA reads them after __syncthreads
    int r, q, nflip, status, par_ok;
    double slope;
};

struct SxGroupBar {        // per-CTA view of its group's barrier (shared memory)
    unsigned* counter;     // the group's arrival counter (zeroed before the launch)
    unsigned gen;          // this CTA's barrier generation; carries over from one node of the group to the next
    unsigned nctas;        // CTAs of the group
};

template <bool WIDE>
struct SxTeam {
    int tid, nth, lane, warp, nwarps;
    SxRed* red;            // shared memory of this CTA
    SxCandRed* cred;
    SxCtrl* ctrl;
    SxGroupBar* bar;       // group team only

    // Barrier over the team. Group team: every CTA of the group arrives once per generation on the group's
    // counter; thread 0 spins until all have (the cooperative launch guarantees co-residency). The gpu-scope
    // fences order the CTA's earlier global writes before the arrival and drop its stale L1 lines after it.
    __device__ __forceinline__ void sync() const {
        if (!WIDE) { __syncthreads(); return; }
        __syncthreads();
        if (threadIdx.x == 0) {
            const unsigned target = (bar->gen + 1u) * bar->nctas;
            __threadfence();
            atomicAdd(bar->counter, 1u);
            while (*reinterpret_cast<volatile unsigned*>(bar->counter) < target) __nanosleep(32);
            __threadfence();
            bar->gen += 1u;
        }
        __syncthreads();
    }
    // CTA-local reductions over values every CTA computes for ALL elements
    __device__ __forceinline__ double max(double v) const { return sx_block_max(v, *red); }
    __device__ __forceinline__ int min_int(int v) const { return sx_block_min_int(v, *red); }
    __device__ __forceinline__ SxCand best(SxCand c) const { return sx_block_best(c, *cred); }
};

// ---- the node's view ---------------------------------------------------------------------------
struct SxNode {
    int m, n, N, ldm;
    double* Binv;        // [m][ldm] row major: (i, k) at i * ldm + k
    int32_t* head;       // [m]
    int8_t* stat;        // [N]
    double* w;           // [m] DSE weights
    double *lo, *hi, *d, *ar, *key;      // [N]
    double *xB, *rho, *aq, *col, *y, *rhs;   // [m]
    double* xfull;       // [N]
    int8_t *artlo, *arthi, *want, *flip, *artdone; // [N]
};


// Ordered sparse dot  sum_p val[p] * vec(idx[p])  over the CSR/CSC entries [p0, p1): the sum runs in
// entry order with single rounded operations (oracle order), but the loads of 8 entries and of the 8
// gathered values are issued together — a chain of dependent global loads per entry was most of the
// time of the pricing / FTRAN loops. Terms with a zero factor are skipped (value preserving).
constexpr int kSxDotBatch = 8;
template <class Vec>
__device__ __forceinline__ double sx_dot_entries(const Ent* __restrict__ ent, const int p0, const int p1, Vec vec) {
    double acc = 0.0;
    for (int p = p0; p < p1; p += kSxDotBatch) {
        double a[kSxDotBatch], v[kSxDotBatch];
        int id[kSxDotBatch];
#pragma unroll
        for (int u = 0; u < kSxDotBatch; ++u) {
            a[u] = 0.0;
            id[u] = 0;
            if (p + u < p1) {
                const int4 raw = *reinterpret_cast<const int4*>(ent + p + u);
                id[u] = raw.x;
                a[u] = __hiloint2double(raw.w, raw.z);
            }
        }
#pragma unroll
        for (int u = 0; u < kSxDotBatch; ++u) v[u] = (p + u < p1) ? vec(id[u]) : 0.0;
#pragma unroll
        for (int u = 0; u < kSxDotBatch; ++u)
            if (a[u] != 0.0 && v[u] != 0.0) acc = sx_add(acc, sx_mul(v[u], a[u]));
    }
    return acc;
}

// acc_i = sum_k Binv(i,k) v[k], ascending k, zeros of v skipped (thread per row)
template <class Team>
__device__ __forceinline__ void sx_matvec(const Team& T, const SxNode& nd, const double* v, double* out) {
    for (int i = T.tid; i < nd.m; i += T.nth) {
        double acc = 0.0;
        for (int k0 = 0; k0 < nd.m; k0 += kSxDotBatch) {
            double bv[kSxDotBatch], vk[kSxDotBatch];
#pragma unroll
            for (int u = 0; u < kSxDotBatch; ++u) {
                const int k = k0 + u;
                vk[u] = k < nd.m ? v[k] : 0.0;
                bv[u] = (k < nd.m && vk[u] != 0.0) ? nd.Binv[(size_t)i * nd.ldm + k] : 0.0;
            }
#pragma unroll
            for (int u = 0; u < kSxDotBatch; ++u)
                if (vk[u] != 0.0) acc = sx_add(acc, sx_mul(bv[u], vk[u]));
        }
        out[i] = acc;
    }
}

// alpha = Binv a_j for column j of [A, -I] (thread per row; entries of a_j ascending by row)
template <class Team>
__device__ __forceinline__ void sx_ftran_col(const Team& T, const SxProb& P, const SxNode& nd, int j, double* out) {
    if (j < nd.n) {
        const int p0 = P.cptr[j], p1 = P.cptr[j + 1];
        for (int i = T.tid; i < nd.m; i += T.nth) {
            const double* Bi = nd.Binv + (size_t)i * nd.ldm;
            out[i] = sx_dot_entries(P.cent, p0, p1, [&](int k) { return Bi[k]; });
        }
    } else {
        const int k = j - nd.n;
        for (int i = T.tid; i < nd.m; i += T.nth)
            out[i] = sx_add(0.0, sx_mul(nd.Binv[(size_t)i * nd.ldm + k], -1.0));
    }
}

// Ordered row norm while a warp walks row i of Binv 32 columns at a time: the oracle sums the squares of
// the columns k = g, g + 16, g + 32, ... (ascending) into partial sum g, then adds the 16 partial sums in
// order. In a chunk of 32 consecutive columns lane g < 16 holds column 32t + g and lane g + 16 holds column
// 32t + g + 16, i.e. the next term of the same partial sum: lane g adds its own square, then the one its
// partner hands over. sq = -1 marks a column beyond m (no term).
__device__ __forceinline__ void sx_norm_step(double& acc, const double sq, const int lane) {
    const double other = __shfl_down_sync(0xffffffffu, sq, 16);
    if (lane < 16) {
        if (sq >= 0.0) acc = sx_add(acc, sq);
        if (other >= 0.0) acc = sx_add(acc, other);
    }
}
__device__ __forceinline__ double sx_norm_finish(const double acc) {
    double w = 0.0;
#pragma unroll
    for (int g = 0; g < kSxWeightLanes; ++g) w = sx_add(w, __shfl_sync(0xffffffffu, acc, g));
    return w;
}

// Binv <- E Binv for a basis change in row position r; rowr[k] = old Binv(r,k) / pivot must be ready.
// A warp owns a row: Binv(i,k) <- Binv(i,k) - alpha_i rowr[k] (row r <- rowr), streamed 32 columns per
// trip, 8 trips of loads issued before the first store (the compiler cannot prove that a store to Binv
// does not alias the next load). With WEIGHTS the row norm is rebuilt in the same sweep.
template <bool WEIGHTS, class Team>
__device__ __forceinline__ void sx_update_inverse(const Team& T, const SxNode& nd, const double* alpha,
                                                  const double* rowr, const int r) {
    constexpr int kTrips = 8;
    const int lane = T.lane, m = nd.m;
    for (int i = T.warp; i < m; i += T.nwarps) {
        double* row = nd.Binv + (size_t)i * nd.ldm;
        const double ai = alpha[i];
        double acc = 0.0;
        for (int k0 = 0; k0 < m; k0 += 32 * kTrips) {
            double v[kTrips], rk[kTrips];
#pragma unroll
            for (int u = 0; u < kTrips; ++u) {
                const int k = k0 + 32 * u + lane;
                v[u] = (k < m) ? row[k] : 0.0;
                rk[u] = (k < m) ? rowr[k] : 0.0;
            }
#pragma unroll
            for (int u = 0; u < kTrips; ++u) {
                const int k = k0 + 32 * u + lane;
                double sq = -1.0;
                if (k < m) {
                    const double nv = (i == r) ? rk[u] : sx_sub(v[u], sx_mul(ai, rk[u]));
                    row[k] = nv;
                    sq = sx_mul(nv, nv);
                }
                if (WEIGHTS && k0 + 32 * u < m) sx_norm_step(acc, sq, lane);
            }
        }
        if (WEIGHTS) {
            const double w = sx_norm_finish(acc);
            if (lane == 0) nd.w[i] = w;
        }
    }
    T.sync();
}

template <class Team>
__device__ __forceinline__ void sx_weights(const Team& T, const SxNode& nd) {
    constexpr int kTrips = 8;
    const int lane = T.lane, m = nd.m;
    for (int i = T.warp; i < m; i += T.nwarps) {
        const double* row = nd.Binv + (size_t)i * nd.ldm;
        double acc = 0.0;
        for (int k0 = 0; k0 < m; k0 += 32 * kTrips) {
            double v[kTrips];
#pragma unroll
            for (int u = 0; u < kTrips; ++u) {
                const int k = k0 + 32 * u + lane;
                v[u] = (k < m) ? row[k] : 0.0;
            }
#pragma unroll
            for (int u = 0; u < kTrips; ++u) {
                const int k = k0 + 32 * u + lane;
                if (k0 + 32 * u < m) sx_norm_step(acc, (k < m) ? sx_mul(v[u], v[u]) : -1.0, lane);
            }
        }
        const double w = sx_norm_finish(acc);
        if (lane == 0) nd.w[i] = w;
    }
    T.sync();
}

// Slack basis, then the wanted structurals pivoted in one by one (start and refactorisation).
// nd.want[j] != 0 marks the columns that should be basic; nd.stat holds the nonbasic sides.
template <class Team>
__device__ void sx_factor(const Team& T, const SxProb& P, const SxNode& nd) {
    const int m = nd.m, n = nd.n, N = nd.N;
    for (size_t e = T.tid; e < (size_t)m * nd.ldm; e += T.nth) {
        const int i = (int)(e / nd.ldm), k = (int)(e % nd.ldm);
        nd.Binv[e] = (i == k) ? -1.0 : 0.0;
    }
    for (int i = T.tid; i < m; i += T.nth) nd.head[i] = n + i;
    for (int j = T.tid; j < N; j += T.nth) {
        const int8_t s = nd.stat[j];
        nd.key[j] = (double)s;                              // "keep": the status before this factorisation
        if (j >= n) nd.stat[j] = SX_BASIC;
        else if (s == SX_BASIC) nd.stat[j] = SX_LOWER;
    }
    T.sync();
    for (int j = 0; j < n; ++j) {
        if (!nd.want[j]) continue;                          // uniform: same data for every thread
        sx_ftran_col(T, P, nd, j, nd.aq);
        T.sync();
        // pivot row: every CTA for itself, over all rows
        double best = kSxPivTol;
        for (int i = threadIdx.x; i < m; i += blockDim.x) {
            const int hv = nd.head[i];
            if (hv >= n && !nd.want[hv]) best = fmax(best, fabs(nd.aq[i]));
        }
        best = T.max(best);
        int r = 2147483647;
        if (best > kSxPivTol)
            for (int i = threadIdx.x; i < m; i += blockDim.x) {
                const int hv = nd.head[i];
                if (hv >= n && !nd.want[hv] && fabs(nd.aq[i]) == best) r = min(r, i);
            }
        r = T.min_int(r);
        if (r == 2147483647) continue;
        const double piv = nd.aq[r];
        const int s_old = nd.head[r];
        const int keep = (int)nd.key[s_old];
        for (int k = T.tid; k < m; k += T.nth) nd.rho[k] = nd.Binv[(size_t)r * nd.ldm + k] / piv;
        T.sync();                                           // rho staged, everybody has read head[r] / key
        sx_update_inverse<false>(T, nd, nd.aq, nd.rho, r);  // ends with a team barrier
        if (T.tid == 0) {
            nd.stat[s_old] = keep != SX_BASIC ? (int8_t)keep : (int8_t)SX_LOWER;
            nd.head[r] = j;
            nd.stat[j] = SX_BASIC;
        }
        T.sync();
    }
}

__device__ __forceinline__ double sx_nonbasic_value(const SxNode& nd, int j) {
    const int8_t s = nd.stat[j];
    return s == SX_BASIC ? 0.0 : (s == SX_UPPER ? nd.hi[j] : nd.lo[j]);
}

// y = c_B Binv (ascending row position, zeros of c_B skipped); d = c - A'y, d_slack = y, d_basic = 0
template <class Team>
__device__ void sx_duals(const Team& T, const SxProb& P, const SxNode& nd) {
    const int m = nd.m, n = nd.n;
    // c_B is gathered once (xfull is free here); thread k then walks its own column of Binv
    for (int p = T.tid; p < m; p += T.nth) {
        const int hv = nd.head[p];
        nd.col[p] = hv < n ? P.c[hv] : 0.0;
    }
    T.sync();
    for (int k = T.tid; k < m; k += T.nth) {
        double acc = 0.0;
        const double* colk = nd.Binv + k;                     // element (p, k) at p * ldm + k: coalesced over k
        const size_t ldm = nd.ldm;
        for (int p0 = 0; p0 < m; p0 += kSxDotBatch) {
            double cb[kSxDotBatch], bv[kSxDotBatch];
#pragma unroll
            for (int u = 0; u < kSxDotBatch; ++u) {
                const int p = p0 + u;
                cb[u] = p < m ? nd.col[p] : 0.0;
                bv[u] = (p < m && cb[u] != 0.0) ? colk[(size_t)p * ldm] : 0.0;
            }
#pragma unroll
            for (int u = 0; u < kSxDotBatch; ++u)
                if (cb[u] != 0.0) acc = sx_add(acc, sx_mul(cb[u], bv[u]));
        }
        nd.y[k] = acc;
    }
    T.sync();
    for (int j = T.tid; j < nd.N; j += T.nth) {
        double dj;
        if (j < n) {
            const double* yv = nd.y;
            dj = sx_sub(P.c[j], sx_dot_entries(P.cent, P.cptr[j], P.cptr[j + 1], [&](int i) { return yv[i]; }));
        } else {
            dj = nd.y[j - n];
        }
        nd.d[j] = nd.stat[j] == SX_BASIC ? 0.0 : dj;
    }
    T.sync();
}

// rhs = b - A x_N + x_N(slack);  x_B = Binv rhs
template <class Team>
__device__ void sx_primal(const Team& T, const SxProb& P, const SxNode& nd) {
    const int m = nd.m, n = nd.n;
    for (int i = T.tid; i < m; i += T.nth) {
        const double acc = sx_dot_entries(P.ent, P.rowptr[i], P.rowptr[i + 1],
                                          [&](int j) { return sx_nonbasic_value(nd, j); });
        nd.rhs[i] = sx_add(sx_sub(P.b[i], acc), sx_nonbasic_value(nd, n + i));
    }
    T.sync();
    sx_matvec(T, nd, nd.rhs, nd.xB);
    T.sync();
}

template <class Team>
__device__ void sx_make_dual_feasible(const Team& T, const SxNode& nd) {
    for (int j = T.tid; j < nd.N; j += T.nth) {
        int8_t s = nd.stat[j];
        if (s == SX_BASIC) continue;
        double lo = nd.lo[j], hi = nd.hi[j];
        if (lo == hi) { nd.stat[j] = SX_LOWER; continue; }
        const double dj = nd.d[j];
        if (dj < -kSxDualTol) s = SX_UPPER;
        else if (dj > kSxDualTol) s = SX_LOWER;
        else if (s == SX_LOWER && isinf(lo)) s = SX_UPPER;
        else if (s == SX_UPPER && isinf(hi)) s = SX_LOWER;
        if (s == SX_UPPER && isinf(hi)) { nd.hi[j] = kSxBig; nd.arthi[j] = 1; }
        if (s == SX_LOWER && isinf(lo)) { nd.lo[j] = -kSxBig; nd.artlo[j] = 1; }
        nd.stat[j] = s;
    }
    T.sync();
}

// ------------------------------------------------------------------------------------------------
// The dual simplex of one node, run by a team (see SxTeam).
template <bool WIDE>
__device__ void sx_solve_node(const SxProb& P, const SxBatch& Q, const int node, const SxTeam<WIDE>& T) {
    SxCtrl& C = *T.ctrl;
    const int m = P.m, n = P.n, N = n + m;
    SxNode nd;
    nd.m = m; nd.n = n; nd.N = N; nd.ldm = P.ldm;
    nd.Binv = Q.Binv + (size_t)node * m * P.ldm;
    nd.head = Q.head + (size_t)node * m;
    nd.stat = Q.stat + (size_t)node * N;
    nd.w = Q.wts + (size_t)node * m;
    {
        double* wk = Q.work + (size_t)node * Q.work_stride;
        nd.lo = wk; wk += N; nd.hi = wk; wk += N; nd.d = wk; wk += N; nd.ar = wk; wk += N; nd.key = wk; wk += N;
        nd.xfull = wk; wk += N;
        nd.xB = wk; wk += m; nd.rho = wk; wk += m; nd.aq = wk; wk += m; nd.col = wk; wk += m;
        nd.y = wk; wk += m; nd.rhs = wk; wk += m;
        int8_t* fl = reinterpret_cast<int8_t*>(wk);
        nd.artlo = fl; nd.arthi = fl + N; nd.want = fl + 2 * N; nd.flip = fl + 3 * N; nd.artdone = fl + 4 * N;
    }
    const double* lbk = Q.lb + (size_t)node * n;
    const double* ubk = Q.ub + (size_t)node * n;
    const int mc = m - P.m_base;
    const uint8_t* onk = Q.rowon ? Q.rowon + (size_t)node * mc : nullptr;
    const int par = Q.parent ? Q.parent[node] : -1;
    const bool from_status = Q.cstat_in != nullptr && Q.rstat_in != nullptr;
    // can the parent's factor be continued? Only if every row that is masked off here has its slack
    // basic there (every CTA checks all pool rows for itself)
    if (threadIdx.x == 0) C.par_ok = 1;
    __syncthreads();
    if (par >= 0 && onk)
        for (int i = threadIdx.x; i < mc; i += blockDim.x)
            if (onk[i] == 0 && Q.pstat[(size_t)par * N + n + P.m_base + i] != SX_BASIC) C.par_ok = 0;
    __syncthreads();

    // ---- bounds, starting status ------------------------------------------------------------
    for (int j = T.tid; j < N; j += T.nth) {
        double lo, hi;
        bool on = true;
        if (j < n) {
            lo = lbk[j]; hi = ubk[j];
            lo = (lo <= -1e30) ? -INFINITY : lo;
            hi = (hi >= 1e30) ? INFINITY : hi;
        } else {
            const int i = j - n;
            on = !(i >= P.m_base && onk && onk[i - P.m_base] == 0);
            lo = on ? 0.0 : -INFINITY;
            hi = INFINITY;
        }
        nd.lo[j] = lo; nd.hi[j] = hi;
        nd.artlo[j] = 0; nd.arthi[j] = 0; nd.flip[j] = 0; nd.artdone[j] = 0;
        int8_t st = SX_LOWER, want = 0;
        if (par >= 0) {
            st = Q.pstat[(size_t)par * N + j];
            want = st == SX_BASIC || !on;
        } else if (from_status) {
            if (j < n) {
                const int8_t cs = Q.cstat_in[(size_t)node * n + j];
                st = cs == SX_UPPER ? SX_UPPER : SX_LOWER;
                want = cs == SX_BASIC;
            } else {
                want = (Q.rstat_in[(size_t)node * m + (j - n)] == SX_BASIC) || !on;
            }
        } else {
            want = j >= n;
        }
        nd.stat[j] = st;
        nd.want[j] = want;
    }
    T.sync();
    const bool use_parent = par >= 0 && C.par_ok != 0;
    if (par >= 0 && !use_parent) {                       // fall back: factorise from the parent's status
        for (int j = T.tid; j < N; j += T.nth)
            if (nd.stat[j] == SX_BASIC) nd.stat[j] = SX_LOWER;
        T.sync();
    }
    if (use_parent) {
        const double* src = Q.pBinv + (size_t)par * m * P.ldm;
        for (size_t e = T.tid; e < (size_t)m * P.ldm; e += T.nth) nd.Binv[e] = src[e];
        for (int i = T.tid; i < m; i += T.nth) {
            nd.head[i] = Q.phead[(size_t)par * m + i];
            nd.w[i] = Q.pwts[(size_t)par * m + i];
        }
        T.sync();
    } else {
        sx_factor(T, P, nd);
    }
    sx_duals(T, P, nd);
    sx_make_dual_feasible(T, nd);
    sx_primal(T, P, nd);
    if (!use_parent) sx_weights(T, nd);

    int pivots = 0, flips_total = 0, since_factor = 0, status = 0;
    // no anti-cycling rule: a hard cap far above any pivot count seen ends a cycling node with status 3
    const int pivot_cap = min(Q.max_pivots, 50 * N + 1000);
    const int refactor_every = Q.refactor_every > 0 ? Q.refactor_every : max(kSxRefactorEvery, 2 * m);
    auto score_of = [&](const int i) {
        const int hv = nd.head[i];
        const double xb = nd.xB[i];
        const double inf = fmax(sx_sub(nd.lo[hv], xb), sx_sub(xb, nd.hi[hv]));
        return inf > sx_mul(kSxPrimalTol, sx_add(1.0, fabs(xb))) ? sx_mul(inf, inf) / nd.w[i] : -1.0;
    };
    while (true) {
        // ---- leaving row: dual steepest edge; every CTA decides for itself over all rows -----------
        double local = -1.0;
        for (int i = threadIdx.x; i < m; i += blockDim.x) local = fmax(local, score_of(i));
        const double best = T.max(local);
        if (best < 0.0) {
            // optimal for the bounded problem. A nonbasic variable resting on an ARTIFICIAL bound with a
            // zero reduced cost does not make the LP unbounded: move it to its real bound once and let
            // the dual simplex repair what that breaks (every CTA scans all variables for itself)
            auto goes_back = [&](const int j) {
                const int8_t st = nd.stat[j];
                return st != SX_BASIC && fabs(nd.d[j]) <= kSxDualTol && !nd.artdone[j] &&
                       ((st == SX_UPPER && nd.arthi[j] && isfinite(nd.lo[j])) ||
                        (st == SX_LOWER && nd.artlo[j] && isfinite(nd.hi[j])));
            };
            double any = -1.0;
            for (int j = threadIdx.x; j < N; j += blockDim.x)
                if (goes_back(j)) any = 1.0;
            if (T.max(any) < 0.0) { status = 0; break; }
            T.sync();                                      // everybody has scanned before anything moves
            for (int j = T.tid; j < N; j += T.nth)
                if (goes_back(j)) {
                    nd.stat[j] = nd.stat[j] == SX_UPPER ? SX_LOWER : SX_UPPER;
                    nd.artdone[j] = 1;
                }
            T.sync();
            sx_primal(T, P, nd);
            continue;
        }
        if (pivots >= pivot_cap) { status = 3; break; }
        if (since_factor >= refactor_every) {
            T.sync();                                      // nobody still reads the state being rebuilt
            for (int j = T.tid; j < N; j += T.nth) nd.want[j] = nd.stat[j] == SX_BASIC;
            T.sync();
            sx_factor(T, P, nd);
            sx_duals(T, P, nd);
            sx_primal(T, P, nd);
            sx_weights(T, nd);
            since_factor = 0;
            continue;
        }
        {
            const double thr = sx_mul(best, sx_sub(1.0, kSxTieRel));
            int hmin = 2147483647;
            for (int i = threadIdx.x; i < m; i += blockDim.x)
                if (score_of(i) >= thr) hmin = min(hmin, nd.head[i]);
            hmin = T.min_int(hmin);
            for (int i = threadIdx.x; i < m; i += blockDim.x)
                if (nd.head[i] == hmin) C.r = i;
            __syncthreads();
        }
        const int r = C.r;
        const int leaving = nd.head[r];
        const double xbr = nd.xB[r];
        const bool below = xbr < nd.lo[leaving];
        const double infr = fmax(sx_sub(nd.lo[leaving], xbr), sx_sub(xbr, nd.hi[leaving]));
        // ---- row r of the tableau, eligibility and ratio keys (split over the team) ----------------
        {
            const double* rv = nd.Binv + (size_t)r * nd.ldm;      // row r of Binv, read in place
            for (int j = T.tid; j < N; j += T.nth) {
                double a;
                if (j < n) a = sx_dot_entries(P.cent, P.cptr[j], P.cptr[j + 1], [&](int i) { return rv[i]; });
                else a = -rv[j - n];
                nd.ar[j] = a;
                const int8_t st = nd.stat[j];
                const double sa = below ? -a : a;
                const bool elig = st != SX_BASIC && nd.lo[j] < nd.hi[j] &&
                                  ((st == SX_LOWER && sa > kSxPivTol) || (st == SX_UPPER && sa < -kSxPivTol));
                nd.key[j] = elig ? rint(sx_mul(fabs(nd.d[j]) / fabs(a), kSxRatioBin)) : INFINITY;
            }
        }
        if (threadIdx.x == 0) { C.slope = infr; C.nflip = 0; C.q = -1; }
        T.sync();                                          // barrier 1: ar, key complete
        // ---- bound flipping ratio test: every CTA walks the candidates in order for itself ----------
        const double flip_tol = sx_mul(kSxPrimalTol, sx_add(1.0, fabs(xbr)));
        SxCand prev;
        prev.key = -1.0; prev.mag = INFINITY; prev.j = -1;  // before every candidate (keys are >= 0)
        while (true) {
            SxCand c;
            c.key = INFINITY; c.mag = 0.0; c.j = 2147483647;
            for (int j = threadIdx.x; j < N; j += blockDim.x) {
                SxCand t;
                t.key = nd.key[j]; t.mag = fabs(nd.ar[j]); t.j = j;
                if (t.key < INFINITY && sx_better(prev, t) && sx_better(t, c)) c = t;
            }
            c = T.best(c);
            if (!(c.key < INFINITY)) break;                  // no candidate left: C.q stays -1
            const int j = c.j;
            const double rng = sx_sub(nd.hi[j], nd.lo[j]);
            bool flipped = false;
            if (isfinite(rng)) {
                const double rest = sx_sub(C.slope, sx_mul(c.mag, rng));
                if (rest > flip_tol) {
                    flipped = true;
                    __syncthreads();
                    if (threadIdx.x == 0) {
                        C.slope = rest;
                        C.nflip += 1;
                        nd.flip[j] = 1;                  // every CTA sets the same marks
                    }
                    __syncthreads();
                    prev = c;
                }
            }
            if (!flipped) {
                if (threadIdx.x == 0) C.q = j;
                break;
            }
        }
        __syncthreads();
        const int q = C.q;
        if (q < 0) { status = 1; break; }
        const int nflip = C.nflip;
        // ---- entering column; the mismatch check comes before anything of the pivot is applied -------
        sx_ftran_col(T, P, nd, q, nd.aq);
        T.sync();                                          // barrier 2: alpha_q complete, every CTA has set its flip marks
        const double piv = nd.aq[r];
        if (since_factor > 0 && fabs(sx_sub(piv, nd.ar[q])) > sx_mul(Q.pivot_mismatch, sx_add(1.0, fabs(nd.ar[q])))) {
            // the two ways to the pivot element disagree: refactorise and price again with nothing applied.
            // Flipping first would leave the flipped columns on the bound their reduced costs say is wrong.
            if (nflip > 0)
                for (int j = T.tid; j < N; j += T.nth) nd.flip[j] = 0;   // read again after the refactorisation's barriers
            since_factor = refactor_every;
            continue;
        }
        if (nflip > 0) {
            // xfull <- bound moves of the flipped columns; col = A delta - delta_slack; x_B -= Binv col
            for (int j = T.tid; j < N; j += T.nth) {
                double dl = 0.0;
                if (nd.flip[j]) {
                    const bool atlo = nd.stat[j] == SX_LOWER;
                    dl = atlo ? sx_sub(nd.hi[j], nd.lo[j]) : sx_sub(nd.lo[j], nd.hi[j]);
                    nd.stat[j] = atlo ? SX_UPPER : SX_LOWER;
                    nd.flip[j] = 0;
                }
                nd.xfull[j] = dl;
            }
            T.sync();
            for (int i = T.tid; i < m; i += T.nth) {
                const double* dv = nd.xfull;
                const double acc = sx_dot_entries(P.ent, P.rowptr[i], P.rowptr[i + 1], [&](int j) { return dv[j]; });
                nd.col[i] = sx_sub(acc, nd.xfull[n + i]);
            }
            T.sync();
            sx_matvec(T, nd, nd.col, nd.rho);              // rho is free until the pivot row is staged below;
            for (int i = T.tid; i < m; i += T.nth) nd.xB[i] = sx_sub(nd.xB[i], nd.rho[i]);   // thread i wrote rho[i]
            T.sync();                                      // the flipped x_B complete
            flips_total += nflip;
        }
        // ---- step lengths, updates ----------------------------------------------------------------
        const double target = below ? nd.lo[leaving] : nd.hi[leaving];
        const double theta_p = sx_sub(nd.xB[r], target) / piv;
        const double xq_new = sx_add(nd.stat[q] == SX_UPPER ? nd.hi[q] : nd.lo[q], theta_p);
        const double theta_d = nd.d[q] / nd.ar[q];
        T.sync();                                          // barrier 3: everybody has read the old x_B, d
        for (int i = T.tid; i < m; i += T.nth)
            nd.xB[i] = (i == r) ? xq_new : sx_sub(nd.xB[i], sx_mul(theta_p, nd.aq[i]));
        for (int j = T.tid; j < N; j += T.nth) {
            double dj = sx_sub(nd.d[j], sx_mul(theta_d, nd.ar[j]));
            if (j == leaving) dj = -theta_d;
            if (j == q) dj = 0.0;
            nd.d[j] = dj;
        }
        for (int k = T.tid; k < m; k += T.nth) nd.rho[k] = nd.Binv[(size_t)r * nd.ldm + k] / piv;
        T.sync();                                          // barrier 4: scaled pivot row staged
        sx_update_inverse<true>(T, nd, nd.aq, nd.rho, r);  // ends with barrier 5
        if (threadIdx.x == 0) {                            // every CTA writes the same three values
            nd.stat[leaving] = below ? SX_LOWER : SX_UPPER;
            nd.stat[q] = SX_BASIC;
            nd.head[r] = q;
        }
        __syncthreads();
        ++pivots;
        ++since_factor;
    }

    // ---- finish: fresh x_B with one refinement step, duals, outputs ----------------------------
    T.sync();
    sx_primal(T, P, nd);
    for (int j = T.tid; j < N; j += T.nth) nd.xfull[j] = sx_nonbasic_value(nd, j);
    T.sync();
    for (int i = T.tid; i < m; i += T.nth) nd.xfull[nd.head[i]] = nd.xB[i];
    T.sync();
    for (int i = T.tid; i < m; i += T.nth) {     // resid = rhs - B x_B
        double res = nd.rhs[i];
        for (int p = P.rowptr[i]; p < P.rowptr[i + 1]; ++p) {
            const Ent e = P.ent[p];
            if (nd.stat[e.idx] == SX_BASIC) res = sx_sub(res, sx_mul(e.val, nd.xfull[e.idx]));
        }
        if (nd.stat[n + i] == SX_BASIC) res = sx_add(res, nd.xfull[n + i]);
        nd.col[i] = res;
    }
    T.sync();
    sx_matvec(T, nd, nd.col, nd.aq);
    T.sync();
    for (int i = T.tid; i < m; i += T.nth) {
        const double v = sx_add(nd.xB[i], nd.aq[i]);
        nd.xB[i] = v;
        nd.xfull[nd.head[i]] = v;
    }
    T.sync();
    sx_duals(T, P, nd);
    if (threadIdx.x == 0) C.status = status;
    __syncthreads();
    if (status == 0) {                                     // every CTA scans all variables for itself
        bool bad = false;
        for (int j = threadIdx.x; j < N; j += blockDim.x) {
            const int8_t st = nd.stat[j];
            if ((st == SX_UPPER && nd.arthi[j]) || (st == SX_LOWER && nd.artlo[j])) bad = true;
            if (fabs(nd.xfull[j]) >= 0.5 * kSxBig) bad = true;
        }
        if (bad) C.status = 2;                              // benign race: every writer stores 2
        __syncthreads();
    }
    for (int j = T.tid; j < n; j += T.nth) {
        if (Q.x) Q.x[(size_t)node * n + j] = nd.xfull[j];
        if (Q.rc) Q.rc[(size_t)node * n + j] = nd.d[j];
        if (Q.cstat_out) Q.cstat_out[(size_t)node * n + j] = nd.stat[j];
    }
    for (int i = T.tid; i < m; i += T.nth) {
        if (Q.y) Q.y[(size_t)node * m + i] = nd.y[i];
        if (Q.rstat_out) Q.rstat_out[(size_t)node * m + i] = nd.stat[n + i];
    }
    if (T.tid == 0) {
        double obj = 0.0;
        for (int j = 0; j < n; ++j) obj = sx_add(obj, sx_mul(P.c[j], nd.xfull[j]));
        if (Q.obj) Q.obj[node] = obj;
        if (Q.status) Q.status[node] = C.status;
        if (Q.pivots) Q.pivots[node] = pivots;
        if (Q.flips) Q.flips[node] = flips_total;
    }
}

// One CTA per node: blockIdx.x = node of the batch.
__global__ void __launch_bounds__(512, 1)
k_simplex(const SxProb P, const SxBatch Q) {
    __shared__ SxRed red;
    __shared__ SxCandRed cred;
    __shared__ SxCtrl ctrl;
    SxTeam<false> T;
    T.tid = threadIdx.x; T.nth = blockDim.x; T.lane = threadIdx.x & 31; T.warp = threadIdx.x >> 5;
    T.nwarps = blockDim.x >> 5;
    T.red = &red; T.cred = &cred; T.ctrl = &ctrl; T.bar = nullptr;
    sx_solve_node<false>(P, Q, blockIdx.x, T);
}

// G groups of S CTAs in one cooperative launch (one CTA per SM, grid = G S): LPs of up to kSxMaxRowsWide rows,
// whose dense inverse (m^2 doubles: 200 MB at m = 5000) is swept by the S SMs of a group at once. Group g
// solves nodes g, g + G, g + 2G, ... one after the other; G = 1 is the whole GPU on each node. Same code,
// same results. Each group's arrival counter sits on its own 128-byte line (kSxBarrierStride unsigneds).
constexpr int kSxBarrierStride = 32;
__global__ void __launch_bounds__(512, 1)
k_simplex_wide(const SxProb P, const SxBatch Q, const int groups, unsigned* const barrier_counters) {
    __shared__ SxRed red;
    __shared__ SxCandRed cred;
    __shared__ SxCtrl ctrl;
    __shared__ SxGroupBar bar;
    const int S = gridDim.x / groups, g = blockIdx.x / S;
    if (threadIdx.x == 0) {
        bar.counter = barrier_counters + (size_t)g * kSxBarrierStride;
        bar.gen = 0u;
        bar.nctas = (unsigned)S;
    }
    __syncthreads();
    SxTeam<true> T;
    T.tid = (blockIdx.x % S) * blockDim.x + threadIdx.x; T.nth = S * blockDim.x; T.lane = threadIdx.x & 31;
    T.warp = T.tid >> 5; T.nwarps = T.nth >> 5;
    T.red = &red; T.cred = &cred; T.ctrl = &ctrl; T.bar = &bar;
    for (int node = g; node < Q.B; node += groups) sx_solve_node<true>(P, Q, node, T);
}

// Rows of the simplex tableau Binv [A, -I] of a node whose factor is in a store (device-side GMI
// input, base_node.py:513-530): out[t][:] = row of the basic variable vars[t] (or zeros if not basic).
// grid = (rows requested), block = 256.
__global__ void k_simplex_tableau_rows(const SxProb P, const double* __restrict__ Binv,
                                       const int32_t* __restrict__ head, const int nrows,
                                       const int32_t* __restrict__ vars, double* __restrict__ out) {
    __shared__ int s_pos;
    const int t = blockIdx.x;
    const int m = P.m, n = P.n, N = n + m;
    if (threadIdx.x == 0) s_pos = -1;
    __syncthreads();
    for (int i = threadIdx.x; i < m; i += blockDim.x)
        if (head[i] == vars[t]) s_pos = i;
    __syncthreads();
    const int r = s_pos;
    double* o = out + (size_t)t * N;
    for (int j = threadIdx.x; j < N; j += blockDim.x) {
        double a = 0.0;
        if (r >= 0) {
            if (j < n) {
                double acc = 0.0;
                for (int p = P.cptr[j]; p < P.cptr[j + 1]; ++p) {
                    const Ent e = P.cent[p];
                    const double ri = Binv[(size_t)r * P.ldm + e.idx];
                    if (ri != 0.0) acc = sx_add(acc, sx_mul(ri, e.val));
                }
                a = acc;
            } else {
                a = -Binv[(size_t)r * P.ldm + (j - n)];
            }
        }
        o[j] = a;
    }
}

// ---- GMI cuts of stored factors (BaseNode._gomory_cuts_of_basis + numerically_safe_cut, on the device) ----
constexpr int kGmiThreads = 256;           // also the lane count of the two ordered dot products
constexpr int GMI_OK = 0, GMI_NOT_BASIC = 1, GMI_NONFINITE = 2, GMI_ZERO = 3;
constexpr double kGmiMaxTerm = 1e3;        // utils/tolerance.py max_term
constexpr double kGmiGoodEps = 1e-2;       // good_coefficient_approximation_epsilon
constexpr double kGmiExactEps = 1e-14;     // exact_coefficient_approximation_epsilon

// utils/floating_point.get_fraction(x, estimate): est = +1 'over', -1 'under', 0 nearest. The convergents
// h / k are kept in doubles: a returned one has |h|, k <= max_term (|x| + 1) and is exact, and the partial
// sums never cancel (h_i, h_{i-1}, h_{i-2} share a sign from i = 1 on, k_i > 0), so the comparison with
// max_term decides as on Python's integers; a convergent beyond it (even an infinite one) is only compared.
__device__ __forceinline__ void gmi_fraction(const double x, const int est, double& num, double& den) {
    if (fabs(x) > kGmiMaxTerm) {
        num = est > 0 ? ceil(x) : (est < 0 ? floor(x) : rint(x));
        den = 1.0;
        return;
    }
    double h2 = 0.0, k2 = 1.0, h1 = 1.0, k1 = 0.0, h, k;
    double value = x;
    int last = 0;
    for (;; ++last) {
        const double a = floor(value);
        h = sx_add(sx_mul(a, h1), h2);
        k = sx_add(sx_mul(a, k1), k2);
        if (h > kGmiMaxTerm || k > kGmiMaxTerm) break;
        const double rest = sx_sub(value, a);
        if (rest == 0.0) { num = h; den = k; return; }        // exact
        value = __ddiv_rn(1.0, rest);
        h2 = h1; k2 = k1; h1 = h; k1 = k;
    }
    // h1 / k1 is convergent last - 1, h2 / k2 convergent last - 2 (last >= 1 here); odd ones lie above x
    const bool odd = last & 1;
    if (est > 0) {
        if (!odd) { num = h1; den = k1; }
        else if (last >= 2) { num = h2; den = k2; }
        else { num = ceil(x); den = 1.0; }
    } else if (est < 0) {
        if (odd) { num = h1; den = k1; }
        else { num = h2; den = k2; }
    } else {
        num = h1; den = k1;
    }
}

// numerically_safe_cut's rounding of one scaled coefficient (estimate 'over')
__device__ __forceinline__ double gmi_safe_coef(const double coef) {
    double n, d;
    gmi_fraction(coef, 1, n, d);
    if (coef != 0.0 && fabs(sx_sub(1.0, __ddiv_rn(__ddiv_rn(n, d), coef))) > kGmiGoodEps) {
        double n2, d2;
        gmi_fraction(coef, 0, n2, d2);
        if (fabs(sx_sub(__ddiv_rn(n2, d2), coef)) < kGmiExactEps) { n = n2; d = d2; }
    }
    return __ddiv_rn(n, d);
}

struct GmiArgs {
    int ncuts;
    const double* Binv; const int32_t* head; const int8_t* stat;   // the last call's store
    const double* lb; const double* ub; const uint8_t* rowon;       // its bounds / row masks (rowon may be null)
    const int32_t* slot; const int32_t* var; const double* f0; const uint8_t* col_is_int;
    double* pi; double* pi0; int32_t* code;                          // [ncuts][n], [ncuts], [ncuts]
};

// One CTA (kGmiThreads threads) per request t: the GMI cut of the tableau row of basic variable var[t] of node
// slot[t], mapped to x-space and rounded as numerically_safe_cut(estimate='over'). Restated in numpy by
// oracle/gmi_device.py, which the results match bit for bit. Order of the floating-point work:
//   tableau row   as k_simplex_tableau_rows: structural j = sum over the entries of column j ascending by row
//                 of Binv(r, i) a_ij (terms with Binv(r, i) = 0 skipped), slack n + i = -Binv(r, i)
//   GMI           row_j = tab_j sign_j (sign -1 at an upper bound), f = row - floor(row), integer:
//                 f <= f0 ? f / f0 : (1 - f) / (1 - f0), else row > 0 ? row / f0 : -row / (1 - f0); basic -> 0;
//                 a column is integer if col_is_int and its offset is within 1e-9 of an integer
//   x-space       pi_j = pi'_j sign_j + sum over the entries of column j ascending by row of pi_s(i) a_ij
//                 (pi_s(i) = 0 skipped; rows masked off for the node carry pi_s = 0)
//   right side    (1 + sum_j pi_x(j) offset_j) + sum_i pi_s(i) b_i, each sum in 256 lanes: lane t adds the
//                 terms t, t + 256, t + 512, ... in order, then the 256 lane sums are added in lane order
//   rounding      scale by 1 / max|pi|, coefficients rounded over, the right side under (gmi_fraction)
// Shared memory: row r of Binv and pi_s, 2 m doubles (dynamic, up to 128 KB at m = 8192).
__global__ void __launch_bounds__(kGmiThreads)
k_simplex_gmi_cuts(const SxProb P, const GmiArgs G) {
    extern __shared__ double gmi_smem[];
    double* rowr = gmi_smem;                 // [m]
    double* pis = gmi_smem + P.m;            // [m]
    __shared__ double part[kGmiThreads];
    __shared__ int s_pos, s_bad;
    __shared__ double s_max;
    const int t = blockIdx.x, tid = threadIdx.x;
    const int m = P.m, n = P.n, N = n + m, mc = m - P.m_base;
    const int slot = G.slot[t], v = G.var[t];
    const double f0 = G.f0[t];
    const int8_t* st = G.stat + (size_t)slot * N;
    const int32_t* hd = G.head + (size_t)slot * m;
    const double* lb = G.lb + (size_t)slot * n;
    const double* ub = G.ub + (size_t)slot * n;
    const uint8_t* on = G.rowon ? G.rowon + (size_t)slot * mc : nullptr;
    double* pi = G.pi + (size_t)t * n;
    if (tid == 0) { s_pos = -1; s_bad = 0; }
    __syncthreads();
    for (int i = tid; i < m; i += kGmiThreads)
        if (hd[i] == v) s_pos = i;
    // nonbasic structurals sit at a bound (|bound| >= 1e30 is none), slacks at 0
    for (int j = tid; j < n; j += kGmiThreads) {
        if (st[j] == SX_BASIC) continue;
        const double o = st[j] == SX_UPPER ? ub[j] : lb[j];
        if (!isfinite(o) || fabs(o) >= 1e30) s_bad = 1;
    }
    __syncthreads();
    const int r = s_pos;
    if (r < 0 || s_bad) {
        for (int j = tid; j < n; j += kGmiThreads) pi[j] = 0.0;
        if (tid == 0) { G.pi0[t] = 0.0; G.code[t] = r < 0 ? GMI_NOT_BASIC : GMI_NONFINITE; }
        return;
    }
    const double* Br = G.Binv + (size_t)slot * m * P.ldm + (size_t)r * P.ldm;
    for (int i = tid; i < m; i += kGmiThreads) rowr[i] = Br[i];
    __syncthreads();
    const double omf0 = sx_sub(1.0, f0);
    // slacks: offset 0, sign +1, never integer
    double acc_b = 0.0;
    for (int i = tid; i < m; i += kGmiThreads) {
        double ps = 0.0;
        const bool carried = !(i >= P.m_base && on && on[i - P.m_base] == 0);
        if (st[n + i] != SX_BASIC) {
            const double row = sx_mul(-rowr[i], 1.0);
            ps = row > 0.0 ? __ddiv_rn(row, f0) : __ddiv_rn(-row, omf0);
        }
        if (!carried) ps = 0.0;
        pis[i] = ps;
        acc_b = sx_add(acc_b, sx_mul(ps, P.b[i]));
    }
    __syncthreads();
    // structurals
    double acc_o = 0.0, big = 0.0;
    for (int j = tid; j < n; j += kGmiThreads) {
        const int8_t s = st[j];
        const int p0 = P.cptr[j], p1 = P.cptr[j + 1];
        double px = 0.0, off = 0.0, sign = 1.0;
        if (s != SX_BASIC) {
            sign = s == SX_UPPER ? -1.0 : 1.0;
            off = s == SX_UPPER ? ub[j] : lb[j];
            double tab = 0.0;
            for (int p = p0; p < p1; ++p) {
                const Ent e = P.cent[p];
                const double ri = rowr[e.idx];
                if (ri != 0.0) tab = sx_add(tab, sx_mul(ri, e.val));
            }
            const double row = sx_mul(tab, sign);
            const bool is_int = G.col_is_int[j] && fabs(sx_sub(off, rint(off))) <= 1e-9;
            double ps;
            if (is_int) {
                const double f = sx_sub(row, floor(row));
                ps = f <= f0 ? __ddiv_rn(f, f0) : __ddiv_rn(sx_sub(1.0, f), omf0);
            } else {
                ps = row > 0.0 ? __ddiv_rn(row, f0) : __ddiv_rn(-row, omf0);
            }
            px = sx_mul(ps, sign);
        }
        acc_o = sx_add(acc_o, sx_mul(px, off));
        double as = 0.0;
        for (int p = p0; p < p1; ++p) {
            const Ent e = P.cent[p];
            const double ps = pis[e.idx];
            if (ps != 0.0) as = sx_add(as, sx_mul(ps, e.val));
        }
        const double coef = sx_add(px, as);
        pi[j] = coef;
        if (!isfinite(coef)) s_bad = 1;
        big = fmax(big, fabs(coef));
    }
    // right-hand side: lane sums in lane order
    part[tid] = acc_o;
    __syncthreads();
    double dot_o = 0.0;
    if (tid == 0)
        for (int l = 0; l < kGmiThreads; ++l) dot_o = sx_add(dot_o, part[l]);
    __syncthreads();
    part[tid] = acc_b;
    __syncthreads();
    if (tid == 0) {
        double dot_b = 0.0;
        for (int l = 0; l < kGmiThreads; ++l) dot_b = sx_add(dot_b, part[l]);
        part[0] = sx_add(sx_add(1.0, dot_o), dot_b);
    }
    __syncthreads();
    const double rhs = part[0];
    // a non-finite coefficient or right-hand side (a factor that is not a clean solve's) gives no cut: the
    // rounding below is only defined on finite values
    if (s_bad || !isfinite(rhs)) {
        for (int j = tid; j < n; j += kGmiThreads) pi[j] = 0.0;
        if (tid == 0) { G.pi0[t] = 0.0; G.code[t] = GMI_NONFINITE; }
        return;
    }
    // largest |coefficient| (order independent)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) big = fmax(big, __shfl_xor_sync(0xffffffffu, big, o));
    if (tid == 0) s_max = 0.0;
    __syncthreads();
    if ((tid & 31) == 0) atomicMax(reinterpret_cast<unsigned long long*>(&s_max), __double_as_longlong(big));
    __syncthreads();
    const double biggest = s_max;            // >= 0, so the bit patterns order as the values
    if (biggest == 0.0) {                    // numerically_safe_cut returns a zero cut unchanged
        if (tid == 0) { G.pi0[t] = rhs; G.code[t] = GMI_ZERO; }
        return;
    }
    const double factor = __ddiv_rn(1.0, biggest);
    for (int j = tid; j < n; j += kGmiThreads) pi[j] = gmi_safe_coef(sx_mul(pi[j], factor));
    if (tid == 0) {
        double nu, de;
        gmi_fraction(sx_mul(rhs, factor), -1, nu, de);
        G.pi0[t] = __ddiv_rn(nu, de);
        G.code[t] = GMI_OK;
    }
}

}  // namespace blp
