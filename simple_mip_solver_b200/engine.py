"""ctypes binding of libblp.so (include/blp.h): the batched node-LP bound step on one B200.

This is the thin layer between the Python branch-and-bound control flow and the CUDA kernels.
PyTorch is used for device-buffer ownership only. There is no CPU fallback: if the shared
library is missing or the call fails, an exception is raised.

Replaces, for a whole batch of nodes at once, what the reference does one node at a time through
CyClpSimplex: ``self.lp.dual()`` and the status/objective/solution reads of
``BaseNode._bound_lp`` (simple_mip_solver/nodes/base_node.py:259-286) and the per-child
``n.lp.dual()`` of ``BaseNode._strong_branch`` (base_node.py:629-647).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from pathlib import Path
from typing import Optional, Sequence

import numpy as np
import scipy.sparse as sp

import os as _os
_LIB_PATH = Path(_os.environ.get('BLP_LIB') or Path(__file__).resolve().parent / 'csrc' / 'libblp.so')
_lib = None

INF = 1e30   # |bound| >= INF means "no bound" on the device side


class BlpError(RuntimeError):
    pass


class BlpOpts(C.Structure):
    _fields_ = [('eps_rel', C.c_double), ('eps_infeas', C.c_double), ('max_iters', C.c_int),
                ('eval_every', C.c_int), ('use_graph', C.c_int), ('compact', C.c_int),
                ('verbose', C.c_int), ('profile', C.c_int), ('max_active', C.c_int), ('obj_cutoff', C.c_double),
                ('freeze', C.c_int), ('freeze_margin', C.c_double), ('step_safety', C.c_double)]


class BlpStats(C.Structure):
    _fields_ = [('iterations', C.c_int), ('evaluations', C.c_int), ('kernel_launches', C.c_int),
                ('compactions', C.c_int), ('step_kernel_ms', C.c_double), ('total_ms', C.c_double),
                ('node_iterations', C.c_double), ('primal_kernel_ms', C.c_double),
                ('dual_kernel_ms', C.c_double), ('refills', C.c_int),
                ('skipped_col_updates', C.c_double), ('skipped_row_updates', C.c_double), ('step_resets', C.c_int)]

    def as_dict(self):
        return {f: getattr(self, f) for f, _ in self._fields_}


_P = C.c_void_p
_SIGNATURES = {
    'blp_default_opts': (None, [C.POINTER(BlpOpts)]),
    'blp_ld': (C.c_int, [C.c_int]),
    'blp_slots': (C.c_int, [C.c_int, C.POINTER(BlpOpts)]),
    'blp_workspace_bytes': (C.c_size_t, [_P, C.c_int]),
    'blp_create': (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int64, _P, _P, _P, _P, _P, C.POINTER(_P)]),
    'blp_append_rows': (C.c_int, [_P, C.c_int, _P, _P, _P, _P, C.POINTER(C.c_int)]),
    'blp_truncate_rows': (C.c_int, [_P, C.c_int]),
    'blp_num_rows': (C.c_int, [_P]),
    'blp_num_base_rows': (C.c_int, [_P]),
    'blp_num_cols': (C.c_int, [_P]),
    'blp_solve_batch': (C.c_int, [_P, C.c_int, _P, _P, _P, _P, _P, _P, C.c_int, C.POINTER(BlpOpts),
                                  _P, C.c_size_t, _P, _P, _P, _P, _P, _P, _P, C.POINTER(BlpStats)]),
    'blp_solve_batch_host': (C.c_int, [_P, C.c_int, _P, _P, _P, _P, _P, _P, C.c_int,
                                       C.POINTER(BlpOpts), _P, _P, _P, _P, _P, _P, _P,
                                       C.POINTER(BlpStats)]),
    'blp_solve_children_host': (C.c_int, [_P, C.c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                                          C.c_int, C.POINTER(BlpOpts), _P, _P, _P, _P, _P, _P, _P,
                                          C.POINTER(BlpStats)]),
    'blp_simplex_max_rows': (C.c_int, []),
    'blp_simplex_batch_rows': (C.c_int, []),
    'blp_simplex_batch_host': (C.c_int, [_P, C.c_int, _P, _P, _P, _P, _P, _P, C.c_int, _P, _P, _P, _P, _P, _P,
                                         _P, _P, C.POINTER(BlpStats)]),
    'blp_simplex_children_host': (C.c_int, [_P, C.c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P, C.c_int, C.c_int,
                                            _P, _P, _P, _P, _P, _P, _P, _P, C.POINTER(BlpStats)]),
    'blp_simplex_tableau_rows_host': (C.c_int, [_P, C.c_int, C.c_int, _P, _P]),
    'blp_spmv': (C.c_int, [_P, C.c_int, C.c_int, _P, _P]),
    'blp_stream': (_P, [_P]),
    'blp_stream_sync': (C.c_int, [_P]),
    'blp_destroy': (C.c_int, [_P]),
    'blp_last_error': (C.c_char_p, []),
    'blp_version': (C.c_char_p, []),
    'blp_comm_probe': (C.c_int, [_P]),
    'blp_comm_unique_id': (C.c_int, [C.c_char_p]),
    'blp_comm_init': (C.c_int, [_P, C.c_int, C.c_int, C.c_char_p]),
    'blp_allreduce_min': (C.c_int, [_P, C.POINTER(C.c_double)]),
    'blp_comm_destroy': (C.c_int, [_P]),
    'blp_mps_read': (C.c_int, [C.c_char_p, C.POINTER(_P)]),
    'blp_mps_dims': (C.c_int, [_P, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int64),
                               C.POINTER(C.c_int32)]),
    'blp_mps_copy': (C.c_int, [_P] * 11),
    'blp_mps_name': (C.c_char_p, [_P]),
    'blp_mps_row_name': (C.c_char_p, [_P, C.c_int32]),
    'blp_mps_col_name': (C.c_char_p, [_P, C.c_int32]),
    'blp_mps_free': (C.c_int, [_P]),
    'blp_mps_last_error': (C.c_char_p, []),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)


def load_library():
    """Load libblp.so. Raises BlpError when it has not been built — there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not _LIB_PATH.exists():
        raise BlpError(f'{_LIB_PATH} is missing: build it with `python -m simple_mip_solver_b200._build` '
                       '(nvcc, sm_100a). The bound step has no CPU fallback.')
    lib = C.CDLL(str(_LIB_PATH))
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _check(rc: int, what: str):
    if rc != 0:
        raise BlpError(f'{what} failed ({rc}): {load_library().blp_last_error().decode()}')


def _np_ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(_P)


def _f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None and a.shape != shape:
        raise ValueError(f'expected array of shape {shape}, got {a.shape}')
    return a


def default_opts(**kw) -> BlpOpts:
    o = BlpOpts()
    load_library().blp_default_opts(C.byref(o))
    for k, v in kw.items():
        if not hasattr(o, k):
            raise TypeError(f'unknown solver option {k!r}')
        setattr(o, k, v)
    return o


def leading_dim(B: int) -> int:
    return (B + 63) // 64 * 64


@dataclass
class BatchResult:
    """Per-node results of one batched bound call (host arrays)."""
    objective: np.ndarray         # [B] c.x (inf where infeasible)
    lower_bound: np.ndarray       # [B] dual objective (a valid lower bound at optimality)
    status: np.ndarray            # [B] CLP codes: 0 optimal, 1 infeasible, 2 unbounded, 3 iteration limit
    iterations: np.ndarray        # [B]
    frac_idx: np.ndarray          # [B] most fractional integer column or -1
    x: Optional[np.ndarray]       # [B, n]
    y: Optional[np.ndarray]       # [B, m] row duals (>= 0)
    stats: dict


@dataclass
class SimplexBatchResult:
    """Per-node results of one batched dual simplex call (host arrays)."""
    objective: np.ndarray         # [B] c.x of the final basic solution
    status: np.ndarray            # [B] CLP codes
    pivots: np.ndarray            # [B]
    x: np.ndarray                 # [B, n] the vertex
    y: np.ndarray                 # [B, m] row duals
    reduced_costs: np.ndarray     # [B, n]
    col_status: np.ndarray        # [B, n] int8, CLP coding: 1 basic, 2 at upper, 3 at lower
    row_status: np.ndarray        # [B, m]
    stats: dict


class BatchLP:
    """Shared part (A, c, row lower bounds) of all node LPs of one MILP, resident on one GPU.

    Canonical form of the reference (base_node.py:683-710): ``min c.x, A x >= b, l <= x <= u``.
    """

    def __init__(self, A, b, c, device: int = 0):
        lib = load_library()
        A = sp.csr_matrix(A, dtype=np.float64)
        A.sort_indices()
        self.m_base, self.n = A.shape
        self.device = int(device)
        b = _f64(b, (self.m_base,))
        c = _f64(c, (self.n,))
        rowptr = np.ascontiguousarray(A.indptr, dtype=np.int32)
        colidx = np.ascontiguousarray(A.indices, dtype=np.int32)
        val = np.ascontiguousarray(A.data, dtype=np.float64)
        h = _P()
        _check(lib.blp_create(self.device, self.m_base, self.n, int(A.nnz), _np_ptr(rowptr),
                              _np_ptr(colidx), _np_ptr(val), _np_ptr(c), _np_ptr(b), C.byref(h)),
               'blp_create')
        self._h = h
        self._lib = lib
        self._ws = None          # torch tensor owning the device workspace

    # -- bookkeeping ------------------------------------------------------------------------
    @property
    def m(self) -> int:
        return self._lib.blp_num_rows(self._h)

    @property
    def num_cut_rows(self) -> int:
        return self.m - self.m_base

    def close(self):
        if getattr(self, '_h', None):
            self._lib.blp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def append_rows(self, rows, rhs) -> int:
        """Append cut rows ``rows . x >= rhs`` (lp.addConstraint, base_node.py:459-460).
        Returns the id of the first new row."""
        R = sp.csr_matrix(np.atleast_2d(rows) if not sp.issparse(rows) else rows, dtype=np.float64)
        R.sort_indices()
        k = R.shape[0]
        if R.shape[1] != self.n:
            raise ValueError(f'cut rows have {R.shape[1]} columns, the LP has {self.n}')
        rhs = _f64(np.atleast_1d(rhs), (k,))
        first = C.c_int(-1)
        rowptr = np.ascontiguousarray(R.indptr, dtype=np.int32)
        colidx = np.ascontiguousarray(R.indices, dtype=np.int32)
        val = np.ascontiguousarray(R.data, dtype=np.float64)
        _check(self._lib.blp_append_rows(self._h, k, _np_ptr(rowptr), _np_ptr(colidx), _np_ptr(val),
                                         _np_ptr(rhs), C.byref(first)), 'blp_append_rows')
        return first.value

    def truncate_rows(self, m_keep: int):
        """Drop appended rows with id >= m_keep (lp.removeConstraint, base_node.py:337-338)."""
        _check(self._lib.blp_truncate_rows(self._h, int(m_keep)), 'blp_truncate_rows')

    # -- host-buffer calls (what the Node classes use) --------------------------------------------
    def solve_batch(self, lb, ub, row_mask=None, x0=None, y0=None,
                    integer_indices: Optional[Sequence[int]] = None, opts: Optional[BlpOpts] = None,
                    want_x: bool = True, want_y: bool = True) -> BatchResult:
        """Solve B node LPs given per-node bounds ``lb, ub`` of shape [B, n] (host arrays)."""
        lb = np.ascontiguousarray(np.atleast_2d(lb), dtype=np.float64)
        B = lb.shape[0]
        lb = _f64(lb, (B, self.n))
        ub = _f64(np.atleast_2d(ub), (B, self.n))
        m, mc = self.m, self.num_cut_rows
        mask = None
        if row_mask is not None and mc > 0:
            mask = np.ascontiguousarray(np.atleast_2d(row_mask), dtype=np.uint8)
            if mask.shape != (B, mc):
                raise ValueError(f'row_mask must have shape {(B, mc)}, got {mask.shape}')
        x0 = None if x0 is None else _f64(np.atleast_2d(x0), (B, self.n))
        y0 = None if y0 is None else _f64(np.atleast_2d(y0), (B, m))
        ii = None if integer_indices is None else np.ascontiguousarray(sorted(integer_indices), dtype=np.int32)
        out = self._alloc_out(B, m, want_x, want_y)
        st = BlpStats()
        o = opts if opts is not None else default_opts()
        _check(self._lib.blp_solve_batch_host(
            self._h, B, _np_ptr(lb), _np_ptr(ub), _np_ptr(mask), _np_ptr(x0), _np_ptr(y0), _np_ptr(ii),
            0 if ii is None else len(ii), C.byref(o), _np_ptr(out['obj']), _np_ptr(out['lower']),
            _np_ptr(out['status']), _np_ptr(out['iters']), _np_ptr(out['x']), _np_ptr(out['y']),
            _np_ptr(out['frac']), C.byref(st)), 'blp_solve_batch_host')
        return self._result(out, st)

    def solve_children(self, parent_lb, parent_ub, deltas, row_mask=None, x0=None, y0=None,
                       integer_indices=None, opts: Optional[BlpOpts] = None, want_x: bool = True,
                       want_y: bool = True) -> BatchResult:
        """Solve B children of one parent. ``deltas[k]`` is a list of ``(var, lb, ub)`` bound
        changes of child k against the parent's bounds (base_node.py:595-600); ``x0, y0`` are the
        parent's primal / row-dual vectors used as the common warm start."""
        B = len(deltas)
        if B < 1:
            raise ValueError('need at least one child')
        parent_lb = _f64(parent_lb, (self.n,))
        parent_ub = _f64(parent_ub, (self.n,))
        m, mc = self.m, self.num_cut_rows
        dptr = np.zeros(B + 1, dtype=np.int32)
        for k, d in enumerate(deltas):
            dptr[k + 1] = dptr[k] + len(d)
        flat = [t for d in deltas for t in d]
        dvar = np.ascontiguousarray([t[0] for t in flat], dtype=np.int32)
        dlb = np.ascontiguousarray([t[1] for t in flat], dtype=np.float64)
        dub = np.ascontiguousarray([t[2] for t in flat], dtype=np.float64)
        mask = None
        if row_mask is not None and mc > 0:
            mask = np.ascontiguousarray(np.atleast_2d(row_mask), dtype=np.uint8)
            if mask.shape != (B, mc):
                raise ValueError(f'row_mask must have shape {(B, mc)}, got {mask.shape}')
        x0 = None if x0 is None else _f64(x0, (self.n,))
        y0 = None if y0 is None else _f64(y0, (m,))
        ii = None if integer_indices is None else np.ascontiguousarray(sorted(integer_indices), dtype=np.int32)
        out = self._alloc_out(B, m, want_x, want_y)
        st = BlpStats()
        o = opts if opts is not None else default_opts()
        _check(self._lib.blp_solve_children_host(
            self._h, B, _np_ptr(parent_lb), _np_ptr(parent_ub), _np_ptr(dptr), _np_ptr(dvar),
            _np_ptr(dlb), _np_ptr(dub), _np_ptr(mask), _np_ptr(x0), _np_ptr(y0), _np_ptr(ii),
            0 if ii is None else len(ii), C.byref(o), _np_ptr(out['obj']), _np_ptr(out['lower']),
            _np_ptr(out['status']), _np_ptr(out['iters']), _np_ptr(out['x']), _np_ptr(out['y']),
            _np_ptr(out['frac']), C.byref(st)), 'blp_solve_children_host')
        return self._result(out, st)

    def _alloc_out(self, B, m, want_x, want_y):
        return dict(obj=np.empty(B), lower=np.empty(B), status=np.empty(B, dtype=np.int32),
                    iters=np.empty(B, dtype=np.int32), frac=np.empty(B, dtype=np.int32),
                    x=np.empty((B, self.n)) if want_x else None,
                    y=np.empty((B, m)) if want_y else None)

    @staticmethod
    def _result(out, st) -> BatchResult:
        return BatchResult(objective=out['obj'], lower_bound=out['lower'], status=out['status'],
                           iterations=out['iters'], frac_idx=out['frac'], x=out['x'], y=out['y'],
                           stats=st.as_dict())

    # -- dual simplex path for small LPs: a vertex and a basis per node ----------------------------
    @property
    def simplex_capable(self) -> bool:
        """True when the LP (with its appended rows) is small enough for blp_simplex_*."""
        return self.m <= self._lib.blp_simplex_max_rows()

    @property
    def simplex_batched(self) -> bool:
        """True when a simplex batch runs one CTA per node; beyond blp_simplex_batch_rows() rows a group
        of SMs works on each node (one cooperative launch, the groups side by side, each through its share of
        the batch), so a batch takes longer per node and a whole strong-branching round may not fit in memory."""
        return self.m <= self._lib.blp_simplex_batch_rows()

    def _simplex_out(self, B, m):
        return dict(obj=np.empty(B), status=np.empty(B, dtype=np.int32), pivots=np.empty(B, dtype=np.int32),
                    x=np.empty((B, self.n)), y=np.empty((B, m)), rc=np.empty((B, self.n)),
                    cs=np.empty((B, self.n), dtype=np.int8), rs=np.empty((B, m), dtype=np.int8))

    @staticmethod
    def _simplex_result(out, st) -> 'SimplexBatchResult':
        return SimplexBatchResult(objective=out['obj'], status=out['status'], pivots=out['pivots'], x=out['x'],
                                  y=out['y'], reduced_costs=out['rc'], col_status=out['cs'],
                                  row_status=out['rs'], stats=st.as_dict())

    def _mask_arg(self, row_mask, shape):
        if row_mask is None or self.num_cut_rows == 0:
            return None
        mask = np.ascontiguousarray(row_mask, dtype=np.uint8)
        if mask.shape != shape:
            raise ValueError(f'row_mask must have shape {shape}, got {mask.shape}')
        return mask

    def simplex_batch(self, lb, ub, row_mask=None, col_status=None, row_status=None, parent_slot=None,
                      max_pivots: int = 2147483647) -> 'SimplexBatchResult':
        """Dual simplex for B node LPs (blp_simplex_batch_host): per-node bounds [B, n], optional
        per-node starting basis in CLP's coding (lp.setBasisStatus, base_node.py:608) or the slot of
        the previous simplex call whose factorised basis to continue from."""
        lb = np.ascontiguousarray(np.atleast_2d(lb), dtype=np.float64)
        B = lb.shape[0]
        lb = _f64(lb, (B, self.n))
        ub = _f64(np.atleast_2d(ub), (B, self.n))
        m = self.m
        mask = self._mask_arg(None if row_mask is None else np.atleast_2d(row_mask), (B, self.num_cut_rows))
        cs = rs = None
        if col_status is not None:
            cs = np.ascontiguousarray(np.atleast_2d(col_status), dtype=np.int8)
            rs = np.ascontiguousarray(np.atleast_2d(row_status), dtype=np.int8)
            if cs.shape != (B, self.n) or rs.shape != (B, m):
                raise ValueError(f'basis status must have shapes {(B, self.n)} and {(B, m)}')
        par = None if parent_slot is None else np.ascontiguousarray(parent_slot, dtype=np.int32).reshape(B)
        out = self._simplex_out(B, m)
        st = BlpStats()
        _check(self._lib.blp_simplex_batch_host(
            self._h, B, _np_ptr(lb), _np_ptr(ub), _np_ptr(mask), _np_ptr(cs), _np_ptr(rs), _np_ptr(par),
            int(min(max_pivots, 2147483647)), _np_ptr(out['obj']), _np_ptr(out['status']), _np_ptr(out['pivots']),
            _np_ptr(out['x']), _np_ptr(out['y']), _np_ptr(out['rc']), _np_ptr(out['cs']), _np_ptr(out['rs']),
            C.byref(st)), 'blp_simplex_batch_host')
        return self._simplex_result(out, st)

    def simplex_children(self, parent_lb, parent_ub, deltas, row_mask=None, col_status=None,
                         row_status=None, parent_slot: int = -1,
                         max_pivots: int = 2147483647) -> 'SimplexBatchResult':
        """Dual simplex for B children of one parent (blp_simplex_children_host): ``deltas[k]`` lists the
        ``(var, lb, ub)`` bound changes of child k (base_node.py:595-600); the parent's basis comes as
        CLP status arrays or as the slot it had in the previous simplex call."""
        B = len(deltas)
        if B < 1:
            raise ValueError('need at least one child')
        parent_lb = _f64(parent_lb, (self.n,))
        parent_ub = _f64(parent_ub, (self.n,))
        m = self.m
        dptr = np.zeros(B + 1, dtype=np.int32)
        for k, d in enumerate(deltas):
            dptr[k + 1] = dptr[k] + len(d)
        flat = [t for d in deltas for t in d]
        dvar = np.ascontiguousarray([t[0] for t in flat], dtype=np.int32)
        dlb = np.ascontiguousarray([t[1] for t in flat], dtype=np.float64)
        dub = np.ascontiguousarray([t[2] for t in flat], dtype=np.float64)
        mask = self._mask_arg(row_mask, (self.num_cut_rows,))
        cs = rs = None
        if col_status is not None:
            cs = np.ascontiguousarray(col_status, dtype=np.int8)
            rs = np.ascontiguousarray(row_status, dtype=np.int8)
            if cs.shape != (self.n,) or rs.shape != (m,):
                raise ValueError(f'basis status must have shapes {(self.n,)} and {(m,)}')
        out = self._simplex_out(B, m)
        st = BlpStats()
        _check(self._lib.blp_simplex_children_host(
            self._h, B, _np_ptr(parent_lb), _np_ptr(parent_ub), _np_ptr(dptr), _np_ptr(dvar), _np_ptr(dlb),
            _np_ptr(dub), _np_ptr(mask), _np_ptr(cs), _np_ptr(rs), int(parent_slot),
            int(min(max_pivots, 2147483647)), _np_ptr(out['obj']), _np_ptr(out['status']), _np_ptr(out['pivots']),
            _np_ptr(out['x']), _np_ptr(out['y']), _np_ptr(out['rc']), _np_ptr(out['cs']), _np_ptr(out['rs']),
            C.byref(st)), 'blp_simplex_children_host')
        return self._simplex_result(out, st)

    def simplex_tableau_rows(self, slot: int, variables) -> np.ndarray:
        """Rows of inv(B) [A, -I] that belong to the basic ``variables`` of node ``slot`` of the
        previous simplex call (blp_simplex_tableau_rows_host; base_node.py:513-526)."""
        v = np.ascontiguousarray(variables, dtype=np.int32).ravel()
        out = np.empty((len(v), self.n + self.m))
        _check(self._lib.blp_simplex_tableau_rows_host(self._h, int(slot), len(v), _np_ptr(v), _np_ptr(out)),
               'blp_simplex_tableau_rows_host')
        return out

    # -- device-buffer calls (torch tensors own the memory) --------------------------------------
    def solve_batch_device(self, lb, ub, row_mask=None, x0=None, y0=None, int_idx=None,
                           opts: Optional[BlpOpts] = None, want_x=True, want_y=True):
        """Device-resident form. ``lb, ub``: torch float64 CUDA tensors of shape [n, ld] in the
        node-fastest layout (ld = leading_dim(B)); ``B`` is taken from ``lb.B`` if present, else
        from ``ub.shape[1]``. Returns a dict of torch tensors plus 'stats'."""
        import torch
        B = int(getattr(lb, 'B', lb.shape[1]))
        ld = leading_dim(B)
        m = self.m
        dev = torch.device('cuda', self.device)
        for name, t, rows in (('lb', lb, self.n), ('ub', ub, self.n), ('x0', x0, self.n), ('y0', y0, m)):
            if t is None:
                continue
            if t.dtype != torch.float64 or not t.is_cuda or not t.is_contiguous() or tuple(t.shape) != (rows, ld):
                raise ValueError(f'{name} must be a contiguous float64 CUDA tensor of shape {(rows, ld)}')
        o = opts if opts is not None else default_opts()
        need = self._lib.blp_workspace_bytes(self._h, self._lib.blp_slots(B, C.byref(o)))
        if self._ws is None or self._ws.numel() < need:
            self._ws = None
            self._ws = torch.empty(need, dtype=torch.uint8, device=dev)
        out = dict(obj=torch.empty(ld, dtype=torch.float64, device=dev),
                   lower=torch.empty(ld, dtype=torch.float64, device=dev),
                   status=torch.empty(ld, dtype=torch.int32, device=dev),
                   iters=torch.empty(ld, dtype=torch.int32, device=dev),
                   frac=torch.empty(ld, dtype=torch.int32, device=dev),
                   x=torch.empty((self.n, ld), dtype=torch.float64, device=dev) if want_x else None,
                   y=torch.empty((m, ld), dtype=torch.float64, device=dev) if want_y else None)
        p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        st = BlpStats()
        torch.cuda.current_stream(dev).synchronize()     # inputs were produced on torch's stream
        _check(self._lib.blp_solve_batch(
            self._h, B, p(lb), p(ub), p(row_mask), p(x0), p(y0), p(int_idx),
            0 if int_idx is None else int(int_idx.numel()), C.byref(o), p(self._ws), self._ws.numel(),
            p(out['obj']), p(out['lower']), p(out['status']), p(out['iters']), p(out['x']), p(out['y']),
            p(out['frac']), C.byref(st)), 'blp_solve_batch')
        out['stats'] = st.as_dict()
        return out

    def spmv_device(self, X, transpose: bool = False, B: Optional[int] = None, out=None):
        """Y = A X (or A' X) on the unscaled matrix; X: [n or m, ld] float64 CUDA tensor."""
        import torch
        B = int(X.shape[1] if B is None else B)
        ld = leading_dim(B)
        rows_in = self.m if transpose else self.n
        rows_out = self.n if transpose else self.m
        if tuple(X.shape) != (rows_in, ld) or X.dtype != torch.float64 or not X.is_contiguous():
            raise ValueError(f'X must be contiguous float64 of shape {(rows_in, ld)}')
        Y = out if out is not None else torch.empty((rows_out, ld), dtype=torch.float64, device=X.device)
        torch.cuda.current_stream(X.device).synchronize()
        _check(self._lib.blp_spmv(self._h, B, 1 if transpose else 0, C.c_void_p(X.data_ptr()),
                                  C.c_void_p(Y.data_ptr())), 'blp_spmv')
        _check(self._lib.blp_stream_sync(self._h), 'blp_stream_sync')
        return Y

    def spmv_async(self, X, Y, B: int, transpose: bool = False):
        """Queue one batched SpMV on the handle's stream without synchronising (benchmarks)."""
        _check(self._lib.blp_spmv(self._h, B, 1 if transpose else 0, C.c_void_p(X.data_ptr()),
                                  C.c_void_p(Y.data_ptr())), 'blp_spmv')

    # -- multi-GPU exchange (one process per GPU) -------------------------------------------------
    def comm_init(self):
        """Join the NCCL communicator of the library with the ranks of the initialised
        ``torch.distributed`` process group: rank 0 creates the id (blp_comm_unique_id), the group
        broadcasts its 128 bytes, every rank calls blp_comm_init. No-op for a single rank."""
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
            return False
        rank, world = dist.get_rank(), dist.get_world_size()
        buf = C.create_string_buffer(128)
        box = [None]
        if rank == 0:       # a failure here must still reach the broadcast, or the other ranks wait forever
            rc = self._lib.blp_comm_unique_id(buf)
            box = [buf.raw if rc == 0 else (self._lib.blp_last_error() or b'?').decode(errors='replace')]
        dist.broadcast_object_list(box, src=0)
        if not isinstance(box[0], bytes):
            raise RuntimeError(f'blp_comm_unique_id failed on rank 0: {box[0]}')
        _check(self._lib.blp_comm_init(self._h, world, rank, box[0]), 'blp_comm_init')
        return True

    def comm_probe(self) -> bool:
        """True when this rank can enter blp_comm_init (libnccl bound, no communicator yet)."""
        return self._lib.blp_comm_probe(self._h) == 0

    def comm_destroy(self):
        """Leave the library's communicator (blp_comm_destroy); ``close()`` does it as well."""
        _check(self._lib.blp_comm_destroy(self._h), 'blp_comm_destroy')

    def allreduce_min(self, incumbent: float, dual_bound: float):
        """Global (min incumbent, min open lower bound) through blp_allreduce_min."""
        v = (C.c_double * 2)(float(incumbent), float(dual_bound))
        _check(self._lib.blp_allreduce_min(self._h, v), 'blp_allreduce_min')
        return float(v[0]), float(v[1])

    def stream_sync(self):
        _check(self._lib.blp_stream_sync(self._h), 'blp_stream_sync')

    @property
    def stream_ptr(self) -> int:
        return int(self._lib.blp_stream(self._h) or 0)


class MultiGpuBatchLP:
    """The same node LPs on several GPUs of one box from ONE process: one ``BatchLP`` handle (its own
    replica of the matrix, its own CUDA stream) per device, one host thread per handle — ctypes
    releases the GIL for the duration of a C call, so the devices run concurrently.

    Node LPs are independent, so a batch is split by node into contiguous shards
    (``parallel.shard_bounds``) and the data path has no collective. The one exchange of the path —
    the all-reduce(min) of ``[best integral objective, smallest open lower bound]`` — runs over the
    library's NCCL communicator between the handles (``blp_allreduce_min``, NVLink) when the devices
    are distinct; every result carries it in ``stats['global_incumbent'/'global_lower_bound']``.

    Same call surface as ``BatchLP`` (the part the Node layer uses). The stored simplex factors of a
    call live on the device that solved the node, so ``parent_slot`` is not offered here: children
    start from the parent's basis status, as with ``lp.setBasisStatus`` in the reference.
    The reference is single process, single device (SURVEY.md section 5); the callers that form the
    batches are BranchAndBound.solve (branch_and_bound.py:226-232) and
    PseudoCostBranchNode._update_pseudo_costs (pseudo_cost.py:57-62)."""

    def __init__(self, A, b, c, devices: Sequence[int]):
        from concurrent.futures import ThreadPoolExecutor
        if len(devices) < 1:
            raise ValueError('need at least one device')
        self.devices = [int(dv) for dv in devices]
        self.parts = [BatchLP(A, b, c, device=dv) for dv in self.devices]
        self.n, self.m_base = self.parts[0].n, self.parts[0].m_base
        self._pool = ThreadPoolExecutor(max_workers=len(self.parts))
        self._comm = False
        if len(set(self.devices)) == len(self.devices) and len(self.devices) > 1:
            self._comm = self._comm_init()

    # -- bookkeeping ---------------------------------------------------------------------------------
    @property
    def m(self) -> int:
        return self.parts[0].m

    @property
    def num_cut_rows(self) -> int:
        return self.parts[0].num_cut_rows

    @property
    def simplex_capable(self) -> bool:
        return self.parts[0].simplex_capable

    @property
    def simplex_batched(self) -> bool:
        return self.parts[0].simplex_batched

    @property
    def uses_nccl(self) -> bool:
        return self._comm

    def _comm_init(self) -> bool:
        """All handles join one NCCL communicator (rank = position in ``devices``); ncclCommInitRank is
        collective, so every handle enters it from its own thread. All or none."""
        lib = self.parts[0]._lib
        if not all(p.comm_probe() for p in self.parts):
            return False
        buf = C.create_string_buffer(128)
        if lib.blp_comm_unique_id(buf) != 0:
            return False
        ident = buf.raw
        world = len(self.parts)
        rcs = list(self._pool.map(lambda rp: lib.blp_comm_init(rp[1]._h, world, rp[0], ident), enumerate(self.parts)))
        if any(rcs):
            for p, rc in zip(self.parts, rcs):
                if rc == 0:
                    p.comm_destroy()
            return False
        return True

    def append_rows(self, rows, rhs) -> int:
        first = [p.append_rows(rows, rhs) for p in self.parts]
        return first[0]

    def truncate_rows(self, m_keep: int):
        for p in self.parts:
            p.truncate_rows(m_keep)

    def close(self):
        for p in self.parts:
            p.close()
        self._pool.shutdown(wait=True)

    # -- sharded calls -------------------------------------------------------------------------------
    def _shards(self, B: int):
        from .parallel import shard_bounds
        world = min(len(self.parts), B)
        return [shard_bounds(B, r, world) for r in range(world)]

    def _run(self, B, call):
        """``call(part, begin, end)`` on every shard concurrently; then the bound exchange."""
        shards = self._shards(B)
        futs = [self._pool.submit(call, self.parts[r], b, e) for r, (b, e) in enumerate(shards)]
        return [f.result() for f in futs]

    def _exchange(self, pairs):
        """Global (incumbent, lower bound): over NCCL between the handles, else a host min."""
        if self._comm and len(pairs) == len(self.parts):
            got = list(self._pool.map(lambda pp: pp[0].allreduce_min(*pp[1]), zip(self.parts, pairs)))
            return got[0]
        return min(p[0] for p in pairs), min(p[1] for p in pairs)

    @staticmethod
    def _pair(obj, lower, status, frac):
        integral = (status == 0) & (frac < 0)
        open_ = (status == 0) & ~integral
        inc = float(obj[integral].min()) if integral.any() else float('inf')
        low = float(lower[open_].min()) if open_.any() else float('inf')
        return inc, low

    @staticmethod
    def _cat(parts, name):
        vals = [getattr(p, name) for p in parts]
        return None if vals[0] is None else np.concatenate(vals)

    def _merge_stats(self, parts, pairs):
        st = dict(parts[0].stats)
        for k in ('kernel_launches', 'node_iterations', 'refills', 'compactions', 'evaluations',
                  'skipped_col_updates', 'skipped_row_updates', 'step_resets'):
            st[k] = sum(p.stats.get(k, 0) for p in parts)
        for k in ('iterations', 'total_ms', 'step_kernel_ms'):
            st[k] = max(p.stats.get(k, 0) for p in parts)
        st['devices'] = self.devices[:len(parts)]
        st['global_incumbent'], st['global_lower_bound'] = self._exchange(pairs)
        st['bound_exchange'] = 'blp_allreduce_min (NCCL)' if self._comm and len(pairs) == len(self.parts) else 'host'
        return st

    def _merge(self, parts):
        pairs = [self._pair(p.objective, p.lower_bound, p.status, p.frac_idx) for p in parts]
        return BatchResult(objective=self._cat(parts, 'objective'), lower_bound=self._cat(parts, 'lower_bound'),
                           status=self._cat(parts, 'status'), iterations=self._cat(parts, 'iterations'),
                           frac_idx=self._cat(parts, 'frac_idx'), x=self._cat(parts, 'x'), y=self._cat(parts, 'y'),
                           stats=self._merge_stats(parts, pairs))

    def _merge_simplex(self, parts, integer_indices=None):
        pairs = []
        for p in parts:
            ok = p.status == 0
            inc = low = float('inf')
            if ok.any():
                if integer_indices is not None and len(integer_indices):
                    xi = p.x[:, list(integer_indices)]
                    integral = ok & (np.max(np.abs(xi - np.round(xi)), axis=1) <= 1e-4)
                else:
                    integral = ok
                inc = float(p.objective[integral].min()) if integral.any() else float('inf')
                low = float(p.objective[ok & ~integral].min()) if (ok & ~integral).any() else float('inf')
            pairs.append((inc, low))
        return SimplexBatchResult(objective=self._cat(parts, 'objective'), status=self._cat(parts, 'status'),
                                  pivots=self._cat(parts, 'pivots'), x=self._cat(parts, 'x'), y=self._cat(parts, 'y'),
                                  reduced_costs=self._cat(parts, 'reduced_costs'),
                                  col_status=self._cat(parts, 'col_status'), row_status=self._cat(parts, 'row_status'),
                                  stats=self._merge_stats(parts, pairs))

    @staticmethod
    def _rows(a, b, e):
        return None if a is None else np.atleast_2d(a)[b:e]

    def solve_batch(self, lb, ub, row_mask=None, x0=None, y0=None, integer_indices=None, opts=None,
                    want_x=True, want_y=True) -> BatchResult:
        lb, ub = np.atleast_2d(lb), np.atleast_2d(ub)
        R = self._rows
        return self._merge(self._run(lb.shape[0], lambda p, b, e: p.solve_batch(
            lb[b:e], ub[b:e], row_mask=R(row_mask, b, e), x0=R(x0, b, e), y0=R(y0, b, e),
            integer_indices=integer_indices, opts=opts, want_x=want_x, want_y=want_y)))

    def solve_children(self, parent_lb, parent_ub, deltas, row_mask=None, x0=None, y0=None,
                       integer_indices=None, opts=None, want_x=True, want_y=True) -> BatchResult:
        R = self._rows
        return self._merge(self._run(len(deltas), lambda p, b, e: p.solve_children(
            parent_lb, parent_ub, deltas[b:e], row_mask=R(row_mask, b, e), x0=x0, y0=y0,
            integer_indices=integer_indices, opts=opts, want_x=want_x, want_y=want_y)))

    def simplex_batch(self, lb, ub, row_mask=None, col_status=None, row_status=None, parent_slot=None,
                      max_pivots: int = 2147483647, integer_indices=None) -> SimplexBatchResult:
        if parent_slot is not None and (np.asarray(parent_slot) >= 0).any():
            raise BlpError('stored simplex factors are per device: MultiGpuBatchLP takes no parent_slot')
        lb, ub = np.atleast_2d(lb), np.atleast_2d(ub)
        R = self._rows
        return self._merge_simplex(self._run(lb.shape[0], lambda p, b, e: p.simplex_batch(
            lb[b:e], ub[b:e], row_mask=R(row_mask, b, e), col_status=R(col_status, b, e),
            row_status=R(row_status, b, e), max_pivots=max_pivots)), integer_indices)

    def simplex_children(self, parent_lb, parent_ub, deltas, row_mask=None, col_status=None, row_status=None,
                         parent_slot: int = -1, max_pivots: int = 2147483647,
                         integer_indices=None) -> SimplexBatchResult:
        if parent_slot >= 0:
            raise BlpError('stored simplex factors are per device: MultiGpuBatchLP takes no parent_slot')
        return self._merge_simplex(self._run(len(deltas), lambda p, b, e: p.simplex_children(
            parent_lb, parent_ub, deltas[b:e], row_mask=row_mask, col_status=col_status, row_status=row_status,
            max_pivots=max_pivots)), integer_indices)

    def simplex_tableau_rows(self, slot: int, variables):
        raise BlpError('stored simplex factors are per device: MultiGpuBatchLP offers no tableau rows')
