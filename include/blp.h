/*
 * blp.h — C ABI of the batched node-LP bound step (libblp.so, sm_100a).
 *
 * The reference (spkelle2/simple_mip_solver) has no FFI: its LP arithmetic is reached through the
 * CyClpSimplex object held in node.lp. Each entry point below names the reference call it replaces
 * (paths relative to the reference root). INTEGRATION.md shows the ctypes binding a maintainer
 * would add on the reference side.
 *
 * Problem solved for every node k of a batch (the reference's canonical form, base_node.py:34,111):
 *
 *     min c.x   s.t.   A x >= row_lb  (rows >= m_base are cut rows, enabled per node by row_mask)
 *                      lb_k <= x <= ub_k
 *
 * Conventions
 *   - plain C types only; no C++ exceptions cross the boundary.
 *   - return value 0 = ok, negative = blp_status error; text via blp_last_error() (thread local).
 *   - per-node solver outcomes are DATA (status[]), not errors. CLP codes are kept
 *     (base_node.py:274-275, pseudo_cost.py:86): 0 optimal, 1 primal infeasible,
 *     2 dual infeasible (unbounded), 3 iteration limit; 5 = stopped by blp_opts.obj_cutoff (opt-in).
 *   - "device" pointers are CUDA device pointers owned by the caller (torch tensors in the Python
 *     host layer) and borrowed for the duration of the call. Batched vectors are stored
 *     node-fastest: element (j, k) of an [rows][ld] array lives at j*ld + k, ld = blp_ld(B)
 *     (B rounded up to a multiple of 64).
 *   - a handle is bound to one GPU and one CUDA stream and is not thread safe.
 *   - infinite bounds: any |v| >= 1e30 (CLP's getCoinInfinity() is DBL_MAX) or IEEE inf.
 */
#ifndef BLP_H
#define BLP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct blp_handle_s* blp_handle;

enum blp_status {
    BLP_OK = 0,
    BLP_ERR_ARG = -1,      /* bad argument */
    BLP_ERR_CUDA = -2,     /* CUDA runtime error (message has the CUDA string) */
    BLP_ERR_NOMEM = -3,    /* workspace too small / allocation failed */
    BLP_ERR_STATE = -4     /* call not valid in this handle state */
};

typedef struct blp_opts {
    double eps_rel;        /* relative KKT tolerance (primal, dual, gap); default 1e-7: bounds the objective
                              error by ~5e-7 relative (DESIGN.md section 2); 1e-8 is SURVEY 8d's figure */
    double eps_infeas;     /* relative size a Farkas certificate must reach; default 1e-9 */
    int max_iters;         /* PDHG iteration cap per call (the analogue of lp.maxNumIteration,
                              base_node.py:645); nodes still running get status 3. default 2000000 */
    int eval_every;        /* iterations between KKT / restart evaluations; default 64 */
    int use_graph;         /* 1: replay each evaluation period as one CUDA graph; default 1 */
    int compact;           /* 1: retire finished nodes by compacting the batch; default 1 */
    int verbose;           /* 1: print one line per evaluation to stderr */
    int profile;           /* 1: no graphs; time every k_primal / k_dual launch with CUDA events
                              (blp_stats.primal_kernel_ms / dual_kernel_ms). default 0 */
    int max_active;        /* node slots resident at once (continuous batching). 0 or >= B: all B nodes
                              are resident. With 0 < max_active < B the first max_active nodes start,
                              and whenever nodes finish the next pending ones take over their slots, so
                              a long frontier (branch_and_bound.py:215-266 evaluates it one node at a
                              time) is swept at constant batch width with state for max_active nodes
                              only. max_iters then counts per node from its own start and may be
                              overshot by less than one evaluation period. default 0 */
    double obj_cutoff;     /* objective limit (the analogue of CLP's dual objective limit): a node whose dual
                              objective b.y + sum_j min(r_j l_j, r_j u_j) — a valid lower bound of its LP at
                              every evaluation — reaches obj_cutoff is retired with status 5, its lower_bound
                              being that bound. The reference prunes such a node after the full solve
                              (branch_and_bound.py:251, 261): with the incumbent's value as the cutoff the
                              search tree is the same, only the node's LP value is a bound instead of the
                              optimum, which is why this is opt-in. default +inf (off) */
    int freeze;            /* 1: wide batches skip the update of coordinates that rest — a column on a bound with a
                              reduced cost of the right sign, a row with zero multiplier and slack — for every node
                              of a 64-node tile. The last iteration of every evaluation period updates everything
                              and the KKT test is always the full problem's, so a status never depends on the
                              frozen set; what is saved is HBM stream (blp_stats.skipped_*). default 1 */
    double freeze_margin;  /* safety margin of that rule in units of the scaled problem's rms cost / right-hand
                              side: freeze above it, release below a third of it. default 0.05 */
    double step_safety;    /* with frozen coordinates the iteration of a tile is PDHG on the rows and columns that
                              still move, A_UU, and its step may be step_safety / ||A_UU||_2 (power iteration per
                              tile, re-estimated after every evaluation) instead of 0.998 / ||A||_2; a node whose
                              fixed-point error grows under the larger step returns to 0.998 / ||A||_2 for good.
                              0 keeps 0.998 / ||A||_2. In [0, 1]; default 0.98 */
} blp_opts;

typedef struct blp_stats {
    int iterations;            /* PDHG iterations executed by the call (max over nodes) */
    int evaluations;           /* KKT evaluations */
    int kernel_launches;       /* kernels of this library launched by the call */
    int compactions;
    double step_kernel_ms;     /* device time spent in the two step kernels (CUDA events) */
    double total_ms;           /* device time of the whole call (CUDA events) */
    double node_iterations;    /* sum over iterations of the number of node columns swept */
    double primal_kernel_ms;   /* profile mode: device time of all k_primal launches */
    double dual_kernel_ms;     /* profile mode: device time of all k_dual launches */
    int refills;               /* nodes that entered through a freed slot (max_active < B) */
    double skipped_col_updates;/* (column, node, iteration) updates skipped because the column was frozen */
    double skipped_row_updates;/* the same for rows; node_iterations * (n + m) is the total without freezing */
    int step_resets;           /* nodes the watchdog sent back from step_safety / ||A_UU|| to 0.998 / ||A|| */
} blp_stats;

/* default options */
void blp_default_opts(blp_opts* o);

/* leading dimension (in elements) of every [rows][ld] batched array for a batch of B nodes */
int blp_ld(int B);

/* node slots a call with B nodes and these options keeps resident: max_active if 0 < max_active < B,
 * else B (opts may be NULL) */
int blp_slots(int B, const blp_opts* opts);

/* bytes of device workspace blp_solve_batch needs for W = blp_slots(B, opts) resident nodes
 * (depends on m incl. appended rows) */
size_t blp_workspace_bytes(blp_handle h, int W);

/*
 * Build the shared part of all node LPs on GPU `device`: CSR of A (m x n), its transpose, the
 * diagonal scaling and the step size. Host pointers, copied.
 * Replaces: model construction for the solver — MILPInstance(...).lp handed to
 * Node(lp=model.lp, ...) (algorithms/base_algorithm.py:18-29) and the per-child rebuild in
 * BaseNode._base_branch (nodes/base_node.py:592-608), which here is paid once per instance.
 */
int blp_create(int device, int m, int n, int64_t nnz, const int32_t* rowptr, const int32_t* colidx,
               const double* val, const double* c, const double* row_lb, blp_handle* out);

/*
 * Append k cut rows (CSR, host pointers) "row . x >= rhs" to the shared pool; they become rows
 * m .. m+k-1 and are enabled per node through row_mask. Returns the id of the first new row.
 * Replaces: lp.addConstraint(pi * x >= pi0, name) in BaseNode._select_cuts (base_node.py:459-460).
 */
int blp_append_rows(blp_handle h, int k, const int32_t* rowptr, const int32_t* colidx,
                    const double* val, const double* rhs, int* first_row_id);

/* Drop every appended row with id >= m_keep (m_keep >= m_base).
 * Replaces: lp.removeConstraint(name) in BaseNode._remove_slack_cuts (base_node.py:337-338). */
int blp_truncate_rows(blp_handle h, int m_keep);

/* current row counts */
int blp_num_rows(blp_handle h);
int blp_num_base_rows(blp_handle h);
int blp_num_cols(blp_handle h);

/*
 * Solve B node LPs that share the handle's matrix. All array arguments are DEVICE pointers in the
 * node-fastest layout with ld = blp_ld(B); optional ones may be NULL.
 *   lb, ub      [n][ld]        per-node variable bounds (the only thing _base_branch changes,
 *                               base_node.py:595-600)
 *   row_mask    [m-m_base][ld] uint8, 1 = cut row present in node k's LP; NULL = all present
 *   x0, y0      [n][ld],[m][ld] warm start (parent's primal / row duals), NULL = cold
 *   int_idx     [n_int]        int32 integer column ids in ascending order (for frac_idx), or NULL
 *   workspace   blp_workspace_bytes(h, blp_slots(B, opts)) bytes
 * outputs (each may be NULL):
 *   obj         [ld]  primal objective c.x at termination (+inf where status == 1)
 *   lower_bound [ld]  Lagrangian bound b.y + sum_j min((c-A'y)_j l_j, (c-A'y)_j u_j)
 *   status      [ld]  CLP code per node
 *   iters       [ld]  PDHG iterations the node ran
 *   x, y        [n][ld], [m][ld]  primal solution and row duals (y >= 0 for rows "a.x >= b")
 *   frac_idx    [ld]  most fractional integer column (first wins ties, distance > 1e-4), -1 if
 *                     the node is integral or not solved  (BaseNode._most_fractional_index,
 *                     base_node.py:544-562; the integrality test of _bound_lp :281-283)
 * Replaces: self.lp.dual() + getStatusCode/objectiveValue/primalVariableSolution/
 * dualConstraintSolution in BaseNode._bound_lp (base_node.py:273-283), and n.lp.dual() for every
 * strong-branching child in BaseNode._strong_branch (base_node.py:644-646), for a whole batch.
 */
int blp_solve_batch(blp_handle h, int B, const double* lb, const double* ub,
                    const uint8_t* row_mask, const double* x0, const double* y0,
                    const int32_t* int_idx, int n_int, const blp_opts* opts,
                    void* workspace, size_t workspace_bytes,
                    double* obj, double* lower_bound, int32_t* status, int32_t* iters,
                    double* x, double* y, int32_t* frac_idx, blp_stats* stats);

/*
 * Host-buffer form of the same call: the form the reference's Python would bind. Inputs are HOST
 * arrays in node-major order (one contiguous bound vector per node, as each node.lp holds them):
 *   lb, ub [B][n]; row_mask [B][m-m_base] or NULL; x0 [B][n], y0 [B][m] or NULL.
 * Outputs are HOST arrays: obj/lower_bound/status/iters/frac_idx [B]; x [B][n], y [B][m] or NULL.
 * The library stages through its own device memory (grown on demand, released by blp_destroy);
 * host<->device copies are part of the call.
 */
int blp_solve_batch_host(blp_handle h, int B, const double* lb, const double* ub,
                         const uint8_t* row_mask, const double* x0, const double* y0,
                         const int32_t* int_idx, int n_int, const blp_opts* opts,
                         double* obj, double* lower_bound, int32_t* status, int32_t* iters,
                         double* x, double* y, int32_t* frac_idx, blp_stats* stats);

/*
 * Children-of-one-parent form (the strong-branching batch, pseudo_cost.py:57-62): node k has the
 * parent's bounds parent_lb/parent_ub [n] (host) except for delta entries
 * delta_ptr[k] .. delta_ptr[k+1]-1, each (delta_var, delta_lb, delta_ub). Host inputs/outputs as
 * in blp_solve_batch_host; x0/y0 are ONE parent vector ([n], [m], host) broadcast to all nodes.
 */
int blp_solve_children_host(blp_handle h, int B, const double* parent_lb, const double* parent_ub,
                            const int32_t* delta_ptr, const int32_t* delta_var,
                            const double* delta_lb, const double* delta_ub,
                            const uint8_t* row_mask, const double* x0, const double* y0,
                            const int32_t* int_idx, int n_int, const blp_opts* opts,
                            double* obj, double* lower_bound, int32_t* status, int32_t* iters,
                            double* x, double* y, int32_t* frac_idx, blp_stats* stats);

/*
 * Dual simplex path for small and mid-size node LPs (at most blp_simplex_max_rows() rows incl. appended cut
 * rows): one CTA per node — for LPs of more than blp_simplex_batch_rows() rows a group of SMs per node, the
 * groups side by side in one cooperative launch, each through its share of the batch — runs a bounded dual simplex with a dense basis inverse (dual steepest edge pricing,
 * bound flipping ratio test; csrc/blp_simplex.cuh, restated in numpy in oracle/dual_simplex.py). It
 * returns what the reference reads from CLP after lp.dual(): a VERTEX and its BASIS, so that the
 * integrality test (base_node.py:281-283), the most fractional index (:544-562), the tableau
 * (:513-530) and get/setBasisStatus (:589, 608) mean what they mean in the reference, and max_pivots is
 * literally lp.maxNumIteration (:645, the 5 pivots of strong branching, pseudo_cost.py:22).
 * All arrays are HOST arrays, node major (one contiguous vector per node):
 *   lb, ub            [B][n]
 *   row_mask          [B][m-m_base] uint8 or NULL (all appended rows present)
 *   col_status,       [B][n], [B][m] int8 in CLP's coding (1 basic, 2 at upper, 3 at lower; anything else
 *   row_status        counts as "at lower") = lp.setBasisStatus of the parent's basis; both NULL = slack
 *                     basis. A status that is not a basis is repaired (rows without a pivot keep their slack).
 *   parent_slot       [B] or NULL: node k starts from the FACTORISED basis node parent_slot[k] of the
 *                     previous blp_simplex_* call on this handle ended with (-1: factorise from the status).
 *                     The store is dropped when rows are appended or truncated.
 * outputs (each may be NULL): obj [B] (c.x of the final basic solution: the dual objective when status
 * is 3, which is a valid lower bound as in pseudo_cost.py:86-92), status [B] CLP codes, pivots [B],
 * x [B][n], y [B][m] row duals, rc [B][n] reduced costs, col_status_out [B][n], row_status_out [B][m].
 * stats (may be NULL): iterations = max pivots of a node, node_iterations = sum of pivots, total_ms,
 * step_kernel_ms = the simplex kernel, kernel_launches, refills = bound flips of the ratio tests.
 */
int blp_simplex_max_rows(void);        /* 8192: above blp_simplex_batch_rows() a group of SMs works on each node */
int blp_simplex_batch_rows(void);      /* 1024: up to here one CTA per node */
int blp_simplex_batch_host(blp_handle h, int B, const double* lb, const double* ub, const uint8_t* row_mask,
                           const int8_t* col_status, const int8_t* row_status, const int32_t* parent_slot,
                           int max_pivots, double* obj, int32_t* status, int32_t* pivots, double* x,
                           double* y, double* rc, int8_t* col_status_out, int8_t* row_status_out,
                           blp_stats* stats);

/* Children of ONE parent (pseudo_cost.py:57-62, base_node.py:592-608): bounds as deltas against the
 * parent's (as in blp_solve_children_host), ONE row_mask [m-m_base], ONE parent basis col_status [n] /
 * row_status [m] (or NULL) and ONE parent_slot (or -1) shared by all B children. */
int blp_simplex_children_host(blp_handle h, int B, const double* parent_lb, const double* parent_ub,
                              const int32_t* delta_ptr, const int32_t* delta_var, const double* delta_lb,
                              const double* delta_ub, const uint8_t* row_mask, const int8_t* col_status,
                              const int8_t* row_status, int parent_slot, int max_pivots, double* obj,
                              int32_t* status, int32_t* pivots, double* x, double* y, double* rc,
                              int8_t* col_status_out, int8_t* row_status_out, blp_stats* stats);

/* Rows of the simplex tableau inv(B) [A, -I] of node `slot` of the previous blp_simplex_* call:
 * out[t][0..n+m) is the row of the basic variable vars[t] (structural j < n, slack of row i = n + i),
 * zeros if vars[t] is not basic. Replaces the dense inverse of BaseNode.tableau (base_node.py:513-526)
 * for the rows _find_gomory_cuts needs (:468-511). */
int blp_simplex_tableau_rows_host(blp_handle h, int slot, int nrows, const int32_t* vars, double* out);

/* Gomory mixed integer cuts of the previous blp_simplex_* call, one per request t: the tableau row of the
 * basic variable vars[t] (numbered as above) in the stored factor of node slots[t] (either team: one CTA per
 * node or a group of SMs per node), shifted / complemented to the node's final nonbasic bounds (slacks at 0),
 * turned into a GMI cut with fractional part f0[t] in (0, 1) (col_is_int [n]: 1 for integer structurals;
 * a shifted column stays integer only if its bound is integral), mapped back to x-space over the rows the
 * node's LP carried (base rows and the pool rows its row mask switched on) and rounded as
 * numerically_safe_cut(..., estimate='over'). Outputs: pi [ncuts][n], pi0 [ncuts] (the cut pi.x >= pi0) and
 * code [ncuts]: BLP_GMI_OK, BLP_GMI_NOT_BASIC (vars[t] is not basic; pi = 0), BLP_GMI_NONFINITE (a nonbasic
 * column sits at an infinite bound, or the cut has a non-finite coefficient or right-hand side, as a node that
 * did not end optimal can leave behind; pi = 0) or BLP_GMI_ZERO (every coefficient is 0: pi and the unrounded
 * pi0 are returned as numerically_safe_cut returns them). Replaces, for many nodes in one launch, the host
 * work per cut of the reference's _find_gomory_cuts / tableau (base_node.py:468-526) and its rounding
 * (floating_point.py:40). The arithmetic is restated in oracle/gmi_device.py, which the results match bit
 * for bit. A slot beyond the previous call, or no stored factors on this matrix, is BLP_ERR_STATE. Slots are meant to
 * name nodes that ended optimal (status 0); any other slot is answered too, under the rules above. */
enum { BLP_GMI_OK = 0, BLP_GMI_NOT_BASIC = 1, BLP_GMI_NONFINITE = 2, BLP_GMI_ZERO = 3 };
int blp_simplex_gmi_cuts_host(blp_handle h, int ncuts, const int32_t* slots, const int32_t* vars, const double* f0,
                              const uint8_t* col_is_int, double* pi, double* pi0, int32_t* code);

/* Batched SpMV on the handle's (unscaled) matrix, device pointers, node-fastest layout:
 * transpose == 0: Y[m][ld] = A X[n][ld];  transpose == 1: Y[n][ld] = A' X[m][ld].
 * Exposed for parity tests and for the SpMV roofline measurement. */
int blp_spmv(blp_handle h, int B, int transpose, const double* X, double* Y);

/* cudaStream_t (as void*) the handle launches on; for CUDA-event timing by the caller. */
void* blp_stream(blp_handle h);

/* Block until everything queued on the handle's stream has finished (blp_spmv is asynchronous). */
int blp_stream_sync(blp_handle h);

int blp_destroy(blp_handle h);

const char* blp_last_error(void);

/*
 * Multi-GPU exchange (SURVEY section 8e). Node LPs are independent, so a frontier is split by node
 * over one process per GPU and the data path has no collective; after a batch the ranks agree on
 *   two_vals[0] = best integer-feasible objective found (the incumbent, branch_and_bound.py:258-262)
 *   two_vals[1] = smallest lower bound of the nodes still open (BranchAndBound.dual_bound, :199-201)
 * with one 16-byte ncclAllReduce(min) over NVLink on the handle's stream. NCCL is bound at run time
 * (dlopen of libnccl.so.2, or $BLP_NCCL_LIB).
 *   blp_comm_probe      0 when blp_comm_init can be entered on this rank (libnccl bound, the handle has no
 *                       communicator yet, its device can be selected). ncclCommInitRank is itself a
 *                       collective: the ranks agree on their probes BEFORE any of them enters it
 *   blp_comm_unique_id  rank 0 creates the 128-byte NCCL id; the host distributes it to all ranks
 *   blp_comm_init       every rank joins with (nranks, rank, id); collective
 *   blp_allreduce_min   two_vals: HOST pointer, in/out; identity on a handle without communicator
 */
int blp_comm_probe(blp_handle h);
int blp_comm_unique_id(char id[128]);
int blp_comm_init(blp_handle h, int nranks, int rank, const char id[128]);
int blp_allreduce_min(blp_handle h, double* two_vals);
int blp_comm_destroy(blp_handle h);

/* library / build identification, e.g. "blp 0.1 sm_100a" */
const char* blp_version(void);

/*
 * MPS reader (host only, no GPU needed). Replaces: MILPInstance(file_name=...) of the reference's
 * tests (test_simple_mip_solver/helpers.py:42, example_models.py:43-48), which reads the model through
 * CLP's MPS reader. Dialect: what CLP writes — free whitespace-separated fields, sections NAME / ROWS /
 * COLUMNS / RHS / BOUNDS / ENDATA, integer columns flagged by UI / LI / BV bounds or MARKER lines,
 * optional set names; RANGES are ignored; empty rows and columns are kept.
 * The model is returned as written: rows with their sense 'L' / 'G' / 'E' and right-hand side (the caller
 * brings it into the solver's ">=" form as base_algorithm.py:53-59 does), objective c with offset,
 * bounds l, u (IEEE +-inf for missing ones), ascending integer column ids.
 *   blp_mps_read   parse `path`; on error returns BLP_ERR_ARG and blp_mps_last_error() has the text
 *   blp_mps_dims   row / column / nonzero / integer-column counts
 *   blp_mps_copy   fill caller arrays: CSR rowptr[m+1], colidx[nnz], val[nnz] (columns ascending within
 *                  a row, duplicates summed), rhs[m], sense[m], c[n], *obj_offset, l[n], u[n],
 *                  int_idx[n_int]; any pointer may be NULL
 */
typedef struct blp_mps_s* blp_mps;
int blp_mps_read(const char* path, blp_mps* out);
int blp_mps_dims(blp_mps mps, int32_t* m, int32_t* n, int64_t* nnz, int32_t* n_int);
int blp_mps_copy(blp_mps mps, int32_t* rowptr, int32_t* colidx, double* val, double* rhs, char* sense,
                 double* c, double* obj_offset, double* l, double* u, int32_t* int_idx);
const char* blp_mps_name(blp_mps mps);
const char* blp_mps_row_name(blp_mps mps, int32_t i);
const char* blp_mps_col_name(blp_mps mps, int32_t j);
int blp_mps_free(blp_mps mps);
const char* blp_mps_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* BLP_H */
