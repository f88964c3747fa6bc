"""Look-alikes of the CyLP objects the reference's Node API touches, backed by the GPU engine.

The reference keeps a ``CyClpSimplex`` in ``node.lp`` and calls ``lp.dual()`` on it, one node at a
time (simple_mip_solver/nodes/base_node.py:273, 646). CyLP/CLP are not part of the reference repo
and are absent here; this module provides the subset of that object protocol the reference uses
(listed in SURVEY.md section 8b) with a different engine underneath:

* every LP of one MILP shares one ``SharedLP`` — the matrix, objective, row bounds, the pool of
  appended cut rows and the ``engine.BatchLP`` handle that lives on the GPU;
* a ``CyClpSimplex`` here is only the per-node part: variable bounds, which cut rows are present,
  a warm start, an iteration budget and the last solution;
* ``dual()`` solves one node through the batched CUDA bound step; ``solve_lps([...])`` solves many
  node LPs of the same MILP in ONE call and leaves each result in its object, so that a later
  ``dual()`` on an unchanged LP is a cache hit. That is how a frontier of open nodes, or all
  strong-branching children, reach the kernels as a batch while the search code stays sequential.

There is no CPU solve here: without libblp.so / a GPU, ``dual()`` raises.
"""
from __future__ import annotations

from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import copy
import types

import numpy as np
import scipy.sparse as sp

COIN_INFINITY = 1.7976931348623157e308      # what CyClpSimplex.getCoinInfinity() returns (DBL_MAX)

# PDHG iterations granted per unit of ``lp.maxNumIteration`` (the reference counts dual simplex
# pivots, base_node.py:645; a first-order iteration is far cheaper than a pivot)
PDHG_ITERS_PER_PIVOT = 512

# device memory the dense basis inverses of one simplex call may take: 'auto' sends a larger batch to PDHG,
# 'simplex' splits it into consecutive calls
SIMPLEX_MEMORY_BUDGET = 16 << 30
SIMPLEX_WIDE_MAX_BATCH = 2

BASIC, AT_UPPER, AT_LOWER = 1, 2, 3      # CLP's getBasisStatus coding


class CyLPArray(np.ndarray):
    """ndarray subclass with the name the reference imports from cylp.py.modeling.CyLPModel."""
    __array_priority__ = 5.0

    def __new__(cls, data, info=None):
        return np.array(data, dtype=np.float64).view(cls)


# ------------------------------------------------------------------------------------------------
# a very small modelling layer: x = lp.addVariable('x', n); lp += l <= x <= u;
# lp.addConstraint(pi * x >= pi0, name); lp.objective = c * x  (base_node.py:459-460, 592-608)
class CyLPVar:
    __array_ufunc__ = None          # make ndarray * var defer to CyLPVar.__rmul__

    def __init__(self, name: str, dim: int):
        self.name = name
        self.dim = int(dim)
        self.lower = CyLPArray(np.zeros(self.dim))
        self.upper = CyLPArray(np.full(self.dim, COIN_INFINITY))
        self.indices = np.arange(self.dim)
        self._pending_lower = None

    def __repr__(self):
        return f'CyLPVar({self.name!r}, {self.dim})'

    def __hash__(self):
        return id(self)

    def __eq__(self, other):
        return self is other

    # coefficient products
    def __rmul__(self, coefs):
        return CyLPExpr(self, coefs)

    def __mul__(self, coefs):
        return CyLPExpr(self, coefs)

    # bounds: "l <= x <= u" evaluates as (l <= x) and (x <= u); the first half parks the lower
    # bound on the variable, the second half returns the combined bound statement
    def __ge__(self, lower):
        self._pending_lower = np.broadcast_to(np.asarray(lower, dtype=float), (self.dim,)).copy()
        return CyLPBounds(self, self._pending_lower, None)

    def __le__(self, upper):
        lower, self._pending_lower = self._pending_lower, None
        upper = np.broadcast_to(np.asarray(upper, dtype=float), (self.dim,)).copy()
        return CyLPBounds(self, lower, upper)


class CyLPBounds:
    def __init__(self, var, lower, upper):
        self.var, self.lower, self.upper = var, lower, upper

    def __bool__(self):
        return True


class CyLPExpr:
    """coefs * x with coefs a vector (one row) or a matrix (several rows)."""
    __array_ufunc__ = None

    def __init__(self, var: CyLPVar, coefs):
        self.var = var
        if sp.issparse(coefs):
            M = sp.csr_matrix(coefs, dtype=float)
        else:
            M = sp.csr_matrix(np.atleast_2d(np.asarray(coefs, dtype=float)))
        if M.shape[1] != var.dim:
            raise ValueError(f'coefficients have {M.shape[1]} columns, variable has {var.dim}')
        self.coefs = M
        self._pending_lower = None

    def __sub__(self, constant):
        """``pi * x - pi0``: an expression keeps only its linear part (a constant moves no optimum;
        the reference writes objectives this way, test_floating_point.py)."""
        assert np.isscalar(constant) or np.asarray(constant).size == 1, 'only a constant can be subtracted'
        return self

    __add__ = __sub__

    def __ge__(self, lower):
        k = self.coefs.shape[0]
        lo = np.broadcast_to(np.asarray(lower, dtype=float), (k,)).copy()
        self._pending_lower = lo
        return CyLPConstraint(self, lo, np.full(k, COIN_INFINITY))

    def __le__(self, upper):
        k = self.coefs.shape[0]
        lo, self._pending_lower = self._pending_lower, None
        if lo is None:
            lo = np.full(k, -COIN_INFINITY)
        up = np.broadcast_to(np.asarray(upper, dtype=float), (k,)).copy()
        return CyLPConstraint(self, lo, up)


class CyLPConstraint:
    def __init__(self, expr: CyLPExpr, lower, upper, name: Optional[str] = None):
        self.name = name
        self.lower = CyLPArray(lower)
        self.upper = CyLPArray(upper)
        self.variables = [expr.var]
        self.varCoefs = {expr.var: expr.coefs}
        self.nRows = expr.coefs.shape[0]
        self.isRange = False

    def __bool__(self):
        return True


# ------------------------------------------------------------------------------------------------
class RoundMemo:
    """Results of speculative cut rounds (``BranchAndBound(frontier_cut_rounds=True)``) for the real nodes to find.

    ``lps``: (LP state key, digest of the starting basis) -> what a simplex solve of that LP from that basis
    returns (status, objective, x, y, reduced costs, basis, pivots): a node LP's simplex solve depends on nothing
    else. ``cuts``: (solve key, node idx, cut round, max_gomory_cuts) -> the device GMI cuts of that solve, as
    ``BaseNode._device_gomory_cuts`` makes them while the solve's factor is in the store. A frontier prefetch
    empties it once it holds more than ``BranchAndBound.MEMO_LPS`` LP results."""

    def __init__(self):
        self.lps: Dict[tuple, tuple] = {}
        self.cuts: Dict[tuple, dict] = {}
        self.lp_hits = 0
        self.cut_hits = 0
        self.speculative_lps = 0
        self.cut_round_resolves = 0     # real nodes that re-solved an LP to get its factor back for cuts

    def clear(self):
        self.lps.clear()
        self.cuts.clear()


def _start_digest(start) -> tuple:
    if start is None:
        return ()
    return (np.asarray(start[0]).tobytes(), np.asarray(start[1]).tobytes(), tuple(start[2].items()))


# ------------------------------------------------------------------------------------------------
class SharedLP:
    """What all node LPs of one MILP have in common: ``min c.x, A x >= b`` plus a pool of cut rows.

    Owns the GPU handle. Cut rows are appended to the device matrix the first time an LP that
    contains them is solved and are switched on per node through the row mask of the batched call.
    """
    default_method = 'auto'         # 'auto' | 'simplex' | 'pdhg' for models created from now on
    default_devices = None          # e.g. [0, 1, 2, 3]: shard every batch of node LPs over these GPUs

    def __init__(self, A, b, c, device: int = 0):
        self.A = sp.csr_matrix(A, dtype=np.float64)
        self.m, self.n = self.A.shape
        self.b = np.asarray(b, dtype=np.float64).reshape(self.m).copy()
        self.c = np.asarray(c, dtype=np.float64).reshape(self.n).copy()
        self.device = device
        self.devices = None             # set to a list of GPU ids before the first solve to use several
        self._engine = None
        self.cut_names: List[str] = []                     # pool order = device row order
        self.cut_index: Dict[Tuple[str, int], int] = {}     # (name, content digest) -> pool row
        self.cut_rows: List[Tuple[np.ndarray, float]] = []
        self._on_device = 0                                # how many pool rows the device has
        self.solve_calls = 0
        self.lps_solved = 0
        self.kernel_launches = 0
        # which device path solves the node LPs: 'auto' = the dual simplex (a vertex and a basis, as
        # the reference gets from CLP) while the LP is small enough for it, PDHG beyond
        self.method = SharedLP.default_method
        self.simplex_calls = 0          # id of the last simplex call (its factors are the engine's store)
        self.simplex_pivots = 0
        self.pool_cap = 256             # appended cut rows the device matrix may hold before it is rebuilt
        self.pool_rebuilds = 0
        # [best integral objective, smallest open lower bound] of the last batch, reduced over the GPUs
        # that shared it (blp_allreduce_min); (None, None) on a single device
        self.last_global_bounds = (None, None)
        # root of the model: its bounds (every node is the root plus a few changed bounds,
        # base_node.py:595-600) and, once solved, its primal/dual pair (the common warm start of a frontier)
        self.root_bounds = None
        self.root_xy = None
        self.max_abs_coef = None        # max |A_ij| (BaseNode.max_term), computed on first use
        self.memo: Optional[RoundMemo] = None   # speculative cut rounds of a frontier (BranchAndBound)

    @property
    def engine(self):
        if self._engine is None:
            from simple_mip_solver_b200 import engine as _engine
            devices = self.devices if self.devices is not None else SharedLP.default_devices
            if devices is not None and len(devices) > 1:
                self._engine = _engine.MultiGpuBatchLP(self.A, self.b, self.c, devices=devices)
            else:
                self._engine = _engine.BatchLP(self.A, self.b, self.c,
                                               device=self.device if not devices else devices[0])
        return self._engine

    def register_cut(self, key: Tuple[str, int], pi: np.ndarray, pi0: float) -> int:
        """Pool row of the cut ``key = (name, digest of its coefficients)``. Two runs on one model can
        produce the same NAME for different rows (cut_gomory_<node>_<round>_<row>): the content is
        part of the identity, so a re-used name never resolves to a stale device row."""
        k = self.cut_index.get(key)
        if k is None:
            k = len(self.cut_names)
            self.cut_names.append(key[0])
            self.cut_index[key] = k
            self.cut_rows.append((np.asarray(pi, dtype=np.float64).copy(), float(pi0)))
        return k

    def make_room(self, needed) -> None:
        """Garbage collection of the device cut pool. Rows stay in the pool after the node that
        added them is done (another open node may hold the same cut); when the pool would outgrow
        ``pool_cap`` rows (and twice what the batch about to be solved needs) it is emptied
        (blp_truncate_rows) and the batch re-appends what it uses. Stored simplex factors refer to the
        old row numbering and are dropped with it."""
        new = sum(1 for key in needed if key not in self.cut_index)
        if len(self.cut_names) + new <= max(self.pool_cap, 2 * len(needed)):
            return
        self.cut_names, self.cut_index, self.cut_rows = [], {}, []
        self._on_device = 0
        self.pool_rebuilds += 1
        self.simplex_calls += 1
        if self._engine is not None:
            self._engine.truncate_rows(self.m)

    def pool_row(self, lp: 'CyClpSimplex', name: str) -> int:
        return self.cut_index[lp._cut_keys[name]]

    def use_simplex(self, n_lps: int = 1) -> bool:
        if self.method == 'pdhg':
            return False
        eng = self.engine
        ok = bool(getattr(eng, 'simplex_capable', False))
        if ok and self.method == 'auto':
            m = self.m + len(self.cut_rows)
            ok = n_lps * m * m * 8 <= SIMPLEX_MEMORY_BUDGET
            # mid-size LPs (a group of SMs per node): only where the vertex is what the caller is after —
            # a single node's bound / cut round; batches go to PDHG
            if ok and not getattr(eng, 'simplex_batched', True):
                ok = n_lps <= SIMPLEX_WIDE_MAX_BATCH
        if not ok and self.method == 'simplex':
            raise RuntimeError('the LP is too large for the dual simplex path')
        return ok

    def simplex_call_size(self, n_lps: int) -> int:
        """LPs per simplex call: as many as SIMPLEX_MEMORY_BUDGET holds dense basis inverses of, at least one."""
        m = self.m + len(self.cut_rows)
        return max(1, min(n_lps, SIMPLEX_MEMORY_BUDGET // (m * m * 8)))

    def sync_cuts(self):
        if self._on_device < len(self.cut_rows):
            new = self.cut_rows[self._on_device:]
            self.engine.append_rows(np.vstack([p for p, _ in new]), np.array([r for _, r in new]))
            self._on_device = len(self.cut_rows)

    def close(self):
        if self._engine is not None:
            self._engine.close()
            self._engine = None
            self._on_device = 0


_EMPTY_ROWS: Dict[int, Tuple[sp.csr_matrix, np.ndarray, np.ndarray]] = {}


def _empty_rows(n: int):
    """(0 x n matrix, no lower bounds, no upper bounds), one shared instance per width."""
    if n not in _EMPTY_ROWS:
        _EMPTY_ROWS[n] = (sp.csr_matrix((0, n)), np.zeros(0), np.zeros(0))
    return _EMPTY_ROWS[n]


class CyClpSimplex:
    """Per-node LP with the attribute/method names of cylp.cy.CyClpSimplex that the reference uses."""

    def __init__(self, shared: Optional[SharedLP] = None, lower=None, upper=None):
        self._shared = shared
        self._vars: List[CyLPVar] = []
        self._l = None if lower is None else CyLPArray(lower)
        self._u = None if upper is None else CyLPArray(upper)
        self._cuts: Dict[str, Tuple[np.ndarray, float]] = {}      # cut rows present in this LP
        self._cut_keys: Dict[str, Tuple[str, int]] = {}            # their pool identities
        self._pending_rows = []                                    # rows added before `shared` exists
        # Modelling-only state. The device solves `A x >= b` over ONE variable vector; CyLP models can hold
        # more (rows with an upper bound, further variables, no base rows). Such a model is kept so
        # that the Node layer can inspect and REJECT it exactly as the reference does (`_sense`,
        # `_x_only_variable`, base_node.py:111-112, 683-710); it cannot be solved.
        self._foreign_rows: Dict[str, Tuple[np.ndarray, float, float]] = {}   # name -> (pi, lower, upper)
        self._base_off = False                                     # the base rows were removed by name
        self._foreign_base = None                                  # (A csr, lower, upper): base rows of a "<=" model
        self._objective = None
        self.logLevel = 0
        self.maxNumIteration = 2147483647
        self.iteration = 0
        self._status = -1
        self._obj = 0.0
        self._x = None
        self._y = None
        self._rc = None
        self._lower_bound = -np.inf
        self._solved_key = None
        self._warm: Optional[Tuple[np.ndarray, Dict[str, float], np.ndarray]] = None
        self._basis = None              # (cols, rows) handed over by setBasisStatus, rows in this LP's order
        self._basis_out = None          # (cols, base rows, {cut name: status}) of the last simplex solve
        self._basis_exact = False       # _basis_out is a basis of the LP as it is now
        self._basis_kept = None         # the last exact basis minus slack cuts removed since (see removeConstraint)
        self._basis_guess = None        # (solved key, cols, rows): active-set status of the last first-order solve
        self._factor_ref = None         # (simplex call id, slot, cut names) of the last simplex solve
        self._parent_ref = None         # the parent's _factor_ref (copy_for_child)
        self._parent_bounds = (None, None)   # the parent's bound arrays (children of one parent share them)
        self._basis_start = None        # setBasisStatus by row NAME: (cols, base rows, {cut name: status})
        self._solve_start = None        # the starting basis of the last simplex solve (its RoundMemo key part)
        self.integer_indices_hint: Optional[Sequence[int]] = None
        self.integer_index_set = None           # frozenset of the hint once a node has checked it
        self.solver_opts: Dict[str, float] = {}
        if shared is not None:
            v = CyLPVar('x', shared.n)
            self._vars.append(v)
            if self._l is None:
                self._l = CyLPArray(np.zeros(shared.n))
            if self._u is None:
                self._u = CyLPArray(np.full(shared.n, COIN_INFINITY))

    # ---- model building (the subset the reference exercises) -------------------------------
    def addVariable(self, name: str, dim: int, isInt: bool = False):
        v = CyLPVar(name, dim)
        self._vars.append(v)
        if len(self._vars) == 1:
            self._l = CyLPArray(np.zeros(dim))
            self._u = CyLPArray(np.full(dim, COIN_INFINITY))
        else:
            self._solved_key = None         # a second variable vector: modelling-only from here on
        return v

    def getVarByName(self, name: str):
        for v in self._vars:
            if v.name == name:
                return v
        raise KeyError(name)

    def __iadd__(self, stmt):
        if isinstance(stmt, CyLPBounds):
            if self._vars and stmt.var.name != self._vars[0].name:
                if stmt.lower is not None:
                    stmt.var.lower = CyLPArray(stmt.lower)
                if stmt.upper is not None:
                    stmt.var.upper = CyLPArray(stmt.upper)
                return self
            if stmt.lower is not None:
                self._l = CyLPArray(stmt.lower)
            if stmt.upper is not None:
                self._u = CyLPArray(stmt.upper)
            self._solved_key = None
            self._basis_exact = False
            self._basis_kept = None
        elif isinstance(stmt, CyLPConstraint):
            self.addConstraint(stmt)
        else:
            raise TypeError(f'cannot add {type(stmt)} to the LP')
        return self

    def addConstraint(self, cons: CyLPConstraint, name: Optional[str] = None, addMpsNames: bool = True):
        assert isinstance(cons, CyLPConstraint), 'constraint must come from an expression like pi * x >= pi0'
        cons.name = name if name is not None else (cons.name or f'R_{id(cons)}')
        M = cons.varCoefs[cons.variables[0]]
        if self._shared is None:
            # base rows of a model under construction: A x >= b only (the canonical form)
            assert (np.asarray(cons.upper) >= 1e300).all(), 'rows must be one sided: a.x >= b'
            self._pending_rows.append(cons)
            return
        one_sided = (np.asarray(cons.upper) >= 1e300).all() and cons.variables[0].name == self._vars[0].name
        for r in range(M.shape[0]):
            nm = cons.name if M.shape[0] == 1 else f'{cons.name}_{r}'
            pi, pi0 = np.asarray(M.getrow(r).todense()).ravel(), float(cons.lower[r])
            if one_sided:
                self._cuts[nm] = (pi, pi0)
                self._cut_keys[nm] = (nm, hash((pi.tobytes(), pi0)))
            else:
                self._foreign_rows[nm] = (pi, pi0, float(cons.upper[r]))
        self._solved_key = None
        self._basis_exact = False
        self._basis_kept = None

    def removeConstraint(self, name: str):
        if name in self._foreign_rows:
            del self._foreign_rows[name]
        elif name == 'R_base' and self._foreign_base is not None:
            self._foreign_base = None
        elif name == 'R_base' and not self._base_off and self._shared is not None:
            self._base_off = True
        elif name in self._cuts:
            del self._cuts[name]
            del self._cut_keys[name]
            kept = self._basis_out if self._basis_exact else self._basis_kept
            if kept is not None and kept[2].get(name) == BASIC:
                # the row's slack was basic: without the row the same x is the basic solution of the same
                # basis minus that slack (CLP keeps its statuses across the removal of a slack cut too,
                # base_node.py:326-341 followed by the tableau of :513-530). Kept as a second opinion for
                # `kept_basis_status`; getBasisStatus() itself answers from the solution as before
                self._basis_kept = (kept[0], kept[1], {nm: st for nm, st in kept[2].items() if nm != name})
            else:
                self._basis_kept = None
        else:
            raise KeyError(f'Constraint "{name}" does not exist')       # CyLP's wording
        self._solved_key = None
        self._basis_exact = False

    @property
    def solvable(self) -> bool:
        """False for a model the device form cannot express (see ``_foreign_rows``)."""
        return len(self._vars) == 1 and not self._foreign_rows and not self._base_off and self._foreign_base is None

    def _finalize(self, device: int = 0):
        """Turn a model built with addVariable/addConstraint/objective into a shared LP."""
        if self._shared is not None:
            return
        n = self._vars[0].dim
        rows = [c.varCoefs[c.variables[0]] for c in self._pending_rows]
        A = sp.vstack(rows, format='csr') if rows else sp.csr_matrix((0, n))
        b = np.concatenate([np.asarray(c.lower) for c in self._pending_rows]) if rows else np.zeros(0)
        c = np.zeros(n) if self._objective is None else np.asarray(self._objective, dtype=float).ravel()
        self._base_names = [c_.name for c_ in self._pending_rows]
        self._shared = SharedLP(A, b, c, device=device)
        self._pending_rows = []

    # ---- attributes read by the reference ------------------------------------------------------
    @property
    def variables(self):
        v = self._vars[0]
        v.lower, v.upper = self._l, self._u
        return self._vars

    @property
    def constraints(self):
        sh = self._need_shared()
        x = self._vars[0]
        out = []
        if not self._base_off:
            out.append(CyLPConstraint(CyLPExpr(x, sh.A), sh.b, np.full(sh.m, COIN_INFINITY), name='R_base'))
        for nm, (pi, pi0) in self._cuts.items():
            out.append(CyLPConstraint(CyLPExpr(x, pi), [pi0], [COIN_INFINITY], name=nm))
        if self._foreign_base is not None:
            A, lo, up = self._foreign_base
            out.append(CyLPConstraint(CyLPExpr(x, A), lo, up, name='R_base'))
        for nm, (pi, lo, up) in self._foreign_rows.items():
            out.append(CyLPConstraint(CyLPExpr(x, pi[:x.dim]), [lo], [up], name=nm))
        return out

    def _foreign(self):
        """(rows as csr, lower, upper) of everything the device form does not hold."""
        n = self._vars[0].dim
        if self._foreign_base is None and not self._foreign_rows:
            return _empty_rows(n)
        mats, los, ups = [], [], []
        if self._foreign_base is not None:
            A, lo, up = self._foreign_base
            mats.append(A), los.append(lo), ups.append(up)
        for pi, lo, up in self._foreign_rows.values():
            mats.append(sp.csr_matrix(pi[None, :n])), los.append([lo]), ups.append([up])
        return sp.vstack(mats, format='csr'), np.concatenate(los), np.concatenate(ups)

    def first_constraint_max_term(self) -> float:
        """max |coefficient| of the first constraint object (what BaseNode keeps as ``max_term``,
        base_node.py:104), without building the constraint list: for the base rows it is a property of the
        shared matrix, computed once per model."""
        sh = self._need_shared()
        if not self._base_off and sh.m:
            if sh.max_abs_coef is None:
                sh.max_abs_coef = float(np.max(np.abs(sh.A.data))) if sh.A.nnz else 0.0
            return sh.max_abs_coef
        cons = self.constraints
        if not cons:
            return 0.0
        M = cons[0].varCoefs[cons[0].variables[0]]
        return float(np.max(np.abs(M.data))) if M.nnz else 0.0

    @property
    def nVariables(self):
        return sum(v.dim for v in self._vars)

    nCols = nVariables

    @property
    def _base_rows(self) -> int:
        return 0 if self._base_off else self._need_shared().m

    @property
    def nConstraints(self):
        return self._base_rows + len(self._cuts) + self._foreign()[0].shape[0]

    nRows = nConstraints

    @property
    def variablesLower(self):
        if len(self._vars) > 1:
            return CyLPArray(np.concatenate([self._l] + [v.lower for v in self._vars[1:]]))
        return self._l

    @variablesLower.setter
    def variablesLower(self, v):
        self._l = CyLPArray(v)
        self._solved_key = None
        self._basis_exact = False
        self._basis_kept = None

    @property
    def variablesUpper(self):
        if len(self._vars) > 1:
            return CyLPArray(np.concatenate([self._u] + [v.upper for v in self._vars[1:]]))
        return self._u

    @variablesUpper.setter
    def variablesUpper(self, v):
        self._u = CyLPArray(v)
        self._solved_key = None
        self._basis_exact = False
        self._basis_kept = None

    @property
    def constraintsLower(self):
        sh = self._need_shared()
        return CyLPArray(np.concatenate([sh.b[:self._base_rows], [p0 for _, p0 in self._cuts.values()],
                                         self._foreign()[1]]))

    @property
    def constraintsUpper(self):
        return CyLPArray(np.concatenate([np.full(self._base_rows + len(self._cuts), COIN_INFINITY),
                                         self._foreign()[2]]))

    @property
    def coefMatrix(self):
        sh = self._need_shared()
        if not self._cuts and self.solvable:
            return sh.A.tocsc()
        base = sh.A if self._base_rows == sh.m else sh.A[:self._base_rows]
        return sp.vstack([base] + [sp.csr_matrix(p[None, :]) for p, _ in self._cuts.values()] +
                         [self._foreign()[0]]).tocsc()

    @property
    def objective(self):
        if self._shared is not None:
            return CyLPArray(self._shared.c)
        return self._objective

    @objective.setter
    def objective(self, value):
        if isinstance(value, CyLPExpr):
            value = np.asarray(value.coefs.todense()).ravel()
        value = CyLPArray(np.asarray(value, dtype=float).ravel())
        if self._shared is not None:
            assert np.array_equal(value, self._shared.c), \
                'the objective is shared by all node LPs of a model and cannot change per node'
        self._objective = value

    objectiveCoefficients = objective

    @property
    def matrix(self):
        """CLP's packed column-major matrix; the reference's tests read ``lp.matrix.elements``."""
        A = self.coefMatrix.tocsc()
        A.sort_indices()
        return types.SimpleNamespace(elements=A.data.copy(), indices=A.indices.copy(), vectorStarts=A.indptr.copy())

    @staticmethod
    def getCoinInfinity():
        return COIN_INFINITY

    def setInteger(self, idx):
        pass

    # ---- results ---------------------------------------------------------------------------------
    def getStatusCode(self):
        return self._status

    @property
    def objectiveValue(self):
        return self._obj

    @property
    def primalVariableSolution(self):
        return {'x': self._x}

    @property
    def dualConstraintSolution(self):
        sh = self._need_shared()
        if self._y is None:
            return {}
        out = {'R_base': CyLPArray(self._y[:sh.m])}
        for k, nm in enumerate(self._cuts):
            out[nm] = CyLPArray([self._y[sh.m + k]])
        return out

    @property
    def dualVariableSolution(self):
        return {'x': self._rc}

    @property
    def lagrangianBound(self):
        """Dual objective of the last solve: a valid lower bound on the LP value (new; the
        iteration-limited dual simplex objective plays this role in the reference, pseudo_cost.py:86)."""
        return self._lower_bound

    def getBasisStatus(self):
        """(column status, row status) in CLP's coding (1 basic, 2 at upper, 3 at lower), rows in this
        LP's order (base rows, then its cut rows). After a dual simplex solve this is the optimal
        BASIS, as in the reference (base_node.py:589). After a PDHG solve (large LPs) it is the active
        set of the primal-dual pair: a column strictly inside its bounds, or a row with slack, counts
        as basic; away from a non-degenerate vertex that is not a basis and ``BaseNode.tableau``
        returns None as the reference does for an inconsistent basis (base_node.py:518-519)."""
        if self._basis_out is not None and self._basis_exact:
            cols, base, cuts = self._basis_out
            rows = np.concatenate([base, [cuts.get(nm, BASIC) for nm in self._cuts]]).astype(np.int32)
            return cols.astype(np.int32), rows
        n, m = self.nVariables, self.nConstraints
        unsolved = self._solved_key is None or self._solved_key != self._state_key()
        if unsolved and self._basis is not None and len(self._basis[0]) == n and len(self._basis[1]) == m:
            # not solved since setBasisStatus: CLP hands back what it was given (a child right after
            # _base_branch carries its parent's basis, base_node.py:608)
            return self._basis[0].astype(np.int32), self._basis[1].astype(np.int32)
        if self._x is None:
            return np.full(n, 3, dtype=np.int32), np.full(m, 1, dtype=np.int32)
        key = self._solved_key
        if self._basis_guess is not None and self._basis_guess[0] == key and key is not None and not unsolved:
            return self._basis_guess[1].copy(), self._basis_guess[2].copy()      # asked once per strong-branching child
        tol = 1e-6
        x = self._x
        scale = 1.0 + np.abs(x)
        at_l = x - self._l <= tol * scale
        at_u = self._u - x <= tol * scale
        cols = np.where(at_l, 3, np.where(at_u, 2, 1)).astype(np.int32)
        # row activities without the CSC copy `coefMatrix` makes for its callers: base rows, then this LP's cuts
        sh = self._need_shared()
        act = [(sh.A if self._base_rows == sh.m else sh.A[:self._base_rows]) @ x]
        act += [[float(np.dot(p, x))] for p, _ in self._cuts.values()]
        act.append(self._foreign()[0] @ x)
        lower = np.asarray(self.constraintsLower)
        rows = np.where(np.concatenate(act) - lower > tol * (1.0 + np.abs(lower)), 1, 3).astype(np.int32)
        if not unsolved:
            self._basis_guess = (key, cols.copy(), rows.copy())
        return cols, rows

    def kept_basis_status(self):
        """(cols, rows) of the last simplex basis with the slack cuts removed since taken out, or None
        if anything else changed the LP after that solve."""
        kept = self._basis_kept
        if kept is None or self._x is None or set(kept[2]) != set(self._cuts):
            return None
        rows = np.concatenate([kept[1], [kept[2][nm] for nm in self._cuts]]).astype(np.int32)
        return kept[0].astype(np.int32), rows

    @property
    def has_exact_basis(self) -> bool:
        """True when getBasisStatus() is the basis of a dual simplex solve of the current LP."""
        return self._basis_out is not None and self._basis_exact

    def setBasisStatus(self, cols, rows):
        """Starting basis of the next dual simplex solve (base_node.py:608); rows in this LP's
        current order, remembered by row name so that later cut rounds cannot shift them."""
        cols, rows = np.asarray(cols).copy(), np.asarray(rows).copy()
        self._basis = (cols, rows)
        m = self._need_shared().m
        if len(cols) == self.nVariables and len(rows) == m + len(self._cuts):
            self._basis_start = (cols.astype(np.int8), rows[:m].astype(np.int8),
                                 {nm: int(rows[m + t]) for t, nm in enumerate(self._cuts)})
        else:
            self._basis_start = None

    def tableau_rows(self, variables) -> Optional[np.ndarray]:
        """Rows of the simplex tableau inv(B) [A, -I] for the given basic variables (LP numbering:
        structurals, then the slack of every row in this LP's order), computed on the device from the
        factorised basis of the last simplex solve; None when that factor is gone (another batch was
        solved since) or the LP was not solved by the simplex path."""
        found = self._stored_factor()
        if found is None:
            return None
        slot, to_pool = found
        rows = self._shared.engine.simplex_tableau_rows(slot, to_pool[np.asarray(variables, dtype=int)])
        return rows[:, to_pool]

    def gmi_cuts(self, variables, f0, col_is_int) -> Optional[Tuple[np.ndarray, np.ndarray, np.ndarray]]:
        """Rounded GMI cuts of the basic ``variables`` (LP numbering, as ``tableau_rows``) with fractional
        parts ``f0``, computed on the device from the factorised basis of the last simplex solve in one call
        (engine.simplex_gmi_cuts): (pi [k, n], pi0 [k], code [k]), or None when that factor is gone."""
        found = self._stored_factor()
        if found is None:
            return None
        slot, to_pool = found
        v = to_pool[np.asarray(variables, dtype=int)]
        return self._shared.engine.simplex_gmi_cuts(np.full(len(v), slot), v, f0, col_is_int)

    @property
    def has_stored_factor(self) -> bool:
        """True while the engine's factor store holds the factorised basis of this LP's last simplex solve."""
        return self._stored_factor() is not None

    def clone(self) -> 'CyClpSimplex':
        """An independent copy of this LP with its last solve (a speculative cut round works on it)."""
        c = copy.copy(self)
        c._l, c._u = self._l.copy(), self._u.copy()
        c._cuts, c._cut_keys = dict(self._cuts), dict(self._cut_keys)
        c._foreign_rows, c._vars = dict(self._foreign_rows), list(self._vars)
        return c

    @property
    def solve_key(self):
        """RoundMemo key of the current solve: None unless the LP is solved as it stands by the simplex path."""
        if self._solve_start is None or not self.has_exact_basis or self._solved_key != self._state_key():
            return None
        return self._solved_key, _start_digest(self._solve_start)

    def memo_cuts(self, idx, cut_round, max_gomory_cuts):
        """Device GMI cuts a speculative round made of this very solve, or None."""
        sh = self._shared
        key = self.solve_key
        if sh is None or sh.memo is None or key is None:
            return None
        got = sh.memo.cuts.get((key, idx, cut_round, max_gomory_cuts))
        if got is None:
            return None
        sh.memo.cut_hits += 1
        return {r: (CyLPArray(pi), pi0) for r, (pi, pi0) in got.items()}

    def restore_factor(self) -> bool:
        """Put this LP's factor back in the store by solving it again from the basis its last solve started from
        (the same solve, so the same result). Only while speculative cut rounds are on: a solve answered by the
        RoundMemo, or one of an earlier chunk of a batch, left no factor where the one-node-per-call run has one."""
        sh = self._shared
        if sh is None or sh.memo is None or self.solve_key is None or hasattr(sh.engine, 'parts'):
            return False
        start = self._basis_start
        self._basis_out, self._basis_start = None, self._solve_start
        try:
            solve_lps([self], force=True)
        finally:
            self._basis_start = start
        return self.has_stored_factor

    def _stored_factor(self):
        """(slot of this LP in the engine's factor store, map from LP numbering to the device's pool numbering)
        while the store still holds the factor of this LP's last solve, else None."""
        sh = self._need_shared()
        ref = self._factor_ref
        if ref is None or self._solved_key != self._state_key() or ref[0] != sh.simplex_calls \
                or hasattr(sh.engine, 'parts'):          # several GPUs: the factor lives on one of them
            return None
        n, m = sh.n, sh.m
        pool = [m + sh.pool_row(self, nm) for nm in self._cuts]      # pool row of every cut row of this LP
        return ref[1], np.concatenate([np.arange(n + m), n + np.asarray(pool, dtype=int)]).astype(int)

    def set_warm_start(self, x, duals_by_row: Dict[str, float], y_base):
        """Parent's primal vector and row duals; the analogue of handing the parent's basis to
        the child (base_node.py:589, 608)."""
        self._warm = (np.asarray(x, dtype=float).copy(), dict(duals_by_row),
                      np.asarray(y_base, dtype=float).copy())

    # ---- solving -----------------------------------------------------------------------------------
    def _need_shared(self) -> SharedLP:
        if self._shared is None:
            self._finalize()
        return self._shared

    def _state_key(self):
        return (self._l.tobytes(), self._u.tobytes(), tuple(self._cut_keys.values()), int(self.maxNumIteration))

    def dual(self):
        if self._solved_key is None or self._solved_key != self._state_key():
            solve_lps([self])
        return self._status

    primal = dual

    def copy_for_child(self) -> 'CyClpSimplex':
        """New per-node LP on the same shared data with copies of bounds and cut membership
        (what the per-child rebuild of base_node.py:592-608 amounts to)."""
        child = CyClpSimplex(self._need_shared(), self._l.copy(), self._u.copy())
        child._cuts = dict(self._cuts)
        child._cut_keys = dict(self._cut_keys)
        child._foreign_rows, child._foreign_base, child._base_off = dict(self._foreign_rows), self._foreign_base, self._base_off
        child._vars += self._vars[1:]
        child._objective = self._objective
        child.integer_indices_hint = self.integer_indices_hint
        child.integer_index_set = self.integer_index_set
        child.solver_opts = self.solver_opts
        if self._factor_ref is not None and self._solved_key == self._state_key():
            child._parent_ref = self._factor_ref
        child._parent_bounds = (self._l, self._u)
        if self._x is not None and self._y is not None:
            sh = self._shared
            child.set_warm_start(self._x, {nm: self._y[sh.m + k] for k, nm in enumerate(self._cuts)},
                                 self._y[:sh.m])
        return child


def solve_lps(lps: Iterable[CyClpSimplex], force: bool = False) -> int:
    """Solve every not-yet-solved LP in ``lps`` with ONE batched GPU call per shared model.

    Results are stored in each object (status, objective, x, row duals, reduced costs); LPs whose
    state is unchanged since their last solve are skipped unless ``force``. Returns the number
    of LPs actually sent to the GPU."""
    from simple_mip_solver_b200.engine import default_opts
    groups: Dict[int, List[CyClpSimplex]] = {}
    for lp in lps:
        sh = lp._need_shared()
        assert lp.solvable, 'the device solves A x >= b over one variable vector: this model has rows with an ' \
                            'upper bound, further variables or no base rows (BaseAlgorithm converts "<=" models)'
        if force or lp._solved_key is None or lp._solved_key != lp._state_key():
            if not force and sh.memo is not None and _from_memo(sh, lp):
                continue
            groups.setdefault(id(sh), []).append(lp)
    sent = 0
    for todo in groups.values():
        sh = todo[0]._shared
        # distinct iteration budgets cannot share a call: split by budget
        by_budget: Dict[int, List[CyClpSimplex]] = {}
        for lp in todo:
            by_budget.setdefault(int(lp.maxNumIteration), []).append(lp)
        for budget, batch in by_budget.items():
            _solve_group(sh, batch, budget, default_opts)
            sent += len(batch)
    return sent


def _memo_start(lp: CyClpSimplex):
    """The basis a simplex solve of ``lp`` starts from (what _solve_group_simplex's start_of picks), or None when
    the solve also depends on something else (a stored parent factor, a first-order crossover start)."""
    if lp.solver_opts.get('factor_cache', False):
        return None
    return lp._basis_out if lp._basis_out is not None else lp._basis_start


def _from_memo(sh: SharedLP, lp: CyClpSimplex) -> bool:
    start = _memo_start(lp)
    if start is None:
        return False
    got = sh.memo.lps.get((lp._state_key(), _start_digest(start)))
    if got is None:
        return False
    sh.memo.lp_hits += 1
    status, obj, x, y, rc, basis, pivots = got
    lp._status, lp.iteration = status, pivots
    lp._basis_out = basis
    lp._basis_exact, lp._basis_kept, lp._factor_ref = True, None, None
    lp._solve_start = start
    if status == 1:
        lp._obj, lp._x, lp._y, lp._rc, lp._lower_bound = float('inf'), None, None, None, float('inf')
    else:
        lp._x, lp._y, lp._rc = CyLPArray(x), y.copy(), CyLPArray(rc)
        lp._obj = lp._lower_bound = obj
    lp._solved_key = lp._state_key()
    return True


def _solve_group(sh: SharedLP, batch: List[CyClpSimplex], budget: int, default_opts):
    sh.make_room({lp._cut_keys[nm] for lp in batch for nm in lp._cuts})
    for lp in batch:
        for nm, (pi, pi0) in lp._cuts.items():
            sh.register_cut(lp._cut_keys[nm], pi, pi0)
    sh.sync_cuts()
    if sh.use_simplex(len(batch)):
        # a later call starts its LPs from their basis status: the store holds the factors of the last call only
        step = sh.simplex_call_size(len(batch))
        for k0 in range(0, len(batch), step):
            _solve_group_simplex(sh, batch[k0:k0 + step], budget, default_opts)
    else:
        _solve_group_pdhg(sh, batch, budget, default_opts)
    for lp in batch:
        lp._solved_key = lp._state_key()


def _child_deltas(batch: List[CyClpSimplex]):
    """If every LP of the batch differs from the first one's PARENT bounds in a few entries only
    — the children of one strong-branching round (base_node.py:592-608) — return those parent
    bounds and the per-LP ``(var, lb, ub)`` changes; else None."""
    first = batch[0]
    pl, pu = getattr(first, '_parent_bounds', (None, None))
    if pl is None or len(batch) < 2:
        return None
    deltas = []
    for lp in batch:
        if getattr(lp, '_parent_bounds', (None, None))[0] is not pl:
            return None
        idx = np.flatnonzero((lp._l != pl) | (lp._u != pu))
        if len(idx) > 8:
            return None
        deltas.append([(int(j), float(lp._l[j]), float(lp._u[j])) for j in idx])
    return pl, pu, deltas


def _solve_group_simplex(sh: SharedLP, batch: List[CyClpSimplex], budget: int, default_opts=None):
    """One batched dual simplex call: vertex, duals, reduced costs and the optimal basis per node LP."""
    eng = sh.engine
    if not getattr(eng, 'simplex_batched', True) and default_opts is not None and budget >= 2147483647:
        # Mid-size LP (the whole GPU per node), no basis to start from: CROSSOVER. A cold dual simplex needs
        # tens of thousands of pivots here (41 116 at the C4 root); the first-order solve finds the optimal
        # face in a second or two, its active set is the starting status (repaired where it is not a
        # basis, made dual feasible by bound flips) and the dual simplex only cleans up.
        cold = [lp for lp in batch if lp._basis_out is None and lp._basis_start is None]
        if cold:
            _solve_group_pdhg(sh, cold, budget, default_opts)
            m0 = sh.m
            for lp in cold:
                if lp._status == 0 and lp._x is not None:
                    cols, rows = lp.getBasisStatus()
                    lp._basis_start = (cols.astype(np.int8), rows[:m0].astype(np.int8),
                                       {nm: int(rows[m0 + t]) for t, nm in enumerate(lp._cuts)})
    B, n, m, mc = len(batch), sh.n, sh.m, len(sh.cut_names)
    use_cache = bool(batch[0].solver_opts.get('factor_cache', False)) and not hasattr(eng, 'parts')
    same_cuts = all(lp._cut_keys == batch[0]._cut_keys for lp in batch)

    def start_of(lp):
        # a re-solve continues from the LP's own last basis (CLP keeps it inside the object), a first
        # solve from what setBasisStatus handed over (base_node.py:608)
        return lp._basis_out if lp._basis_out is not None else lp._basis_start

    def status_rows(lp):
        """starting status of the pool rows: base rows and this LP's cuts from the starting basis,
        everything else basic (new cut rows enter with their slack basic)"""
        rows = np.full(m + mc, BASIC, dtype=np.int8)
        cols = np.full(n, AT_LOWER, dtype=np.int8)
        start = start_of(lp)
        if start is not None:
            cols = np.asarray(start[0], dtype=np.int8)
            rows[:m] = start[1]
            for nm in lp._cuts:
                rows[m + sh.pool_row(lp, nm)] = start[2].get(nm, BASIC)
        return cols, rows

    def parent_slot(lp):
        keys = tuple(lp._cut_keys.values())
        for ref in (lp._factor_ref, lp._parent_ref):
            if use_cache and ref is not None and ref[0] == sh.simplex_calls and ref[2] == keys:
                return ref[1]
        return -1

    def same_start(a, b):
        sa, sb = start_of(a), start_of(b)
        if sa is None or sb is None:
            return sa is sb
        return sa is sb or (np.array_equal(sa[0], sb[0]) and np.array_equal(sa[1], sb[1]) and sa[2] == sb[2])

    same_basis = all(same_start(lp, batch[0]) and parent_slot(lp) == parent_slot(batch[0]) for lp in batch)

    kids = _child_deltas(batch) if (same_cuts and same_basis) else None
    if kids is not None:
        pl, pu, deltas = kids
        lp0 = batch[0]
        mask = None
        if mc:
            mask = np.zeros(mc, dtype=np.uint8)
            for nm in lp0._cuts:
                mask[sh.pool_row(lp0, nm)] = 1
        cols, rows = status_rows(lp0)
        slot = parent_slot(lp0)
        res = eng.simplex_children(np.where(pl <= -1e30, -np.inf, pl), np.where(pu >= 1e30, np.inf, pu), deltas,
                                   row_mask=mask, col_status=cols, row_status=rows, parent_slot=slot,
                                   max_pivots=budget)
    else:
        lb = np.empty((B, n))
        ub = np.empty((B, n))
        mask = np.zeros((B, mc), dtype=np.uint8) if mc else None
        cs = np.empty((B, n), dtype=np.int8)
        rs = np.empty((B, m + mc), dtype=np.int8)
        par = np.full(B, -1, dtype=np.int32)
        for k, lp in enumerate(batch):
            lb[k] = np.where(lp._l <= -1e30, -np.inf, lp._l)
            ub[k] = np.where(lp._u >= 1e30, np.inf, lp._u)
            for nm in lp._cuts:
                mask[k, sh.pool_row(lp, nm)] = 1
            cs[k], rs[k] = status_rows(lp)
            par[k] = parent_slot(lp)
        res = eng.simplex_batch(lb, ub, row_mask=mask, col_status=cs, row_status=rs,
                                parent_slot=par if (par >= 0).any() else None, max_pivots=budget)
    sh.solve_calls += 1
    sh.simplex_calls += 1
    sh.last_global_bounds = (res.stats.get('global_incumbent'), res.stats.get('global_lower_bound'))
    sh.lps_solved += B
    sh.kernel_launches += int(res.stats.get('kernel_launches', 1))
    sh.simplex_pivots += int(res.pivots.sum())
    starts = [start_of(lp) for lp in batch]
    for k, lp in enumerate(batch):
        st = int(res.status[k])
        lp._status = st
        lp.iteration = int(res.pivots[k])
        lp._solve_start = None if use_cache else starts[k]
        rows = [m + sh.pool_row(lp, nm) for nm in lp._cuts]
        lp._basis_out = (res.col_status[k].copy(), res.row_status[k, :m].copy(),
                         {nm: int(res.row_status[k, r]) for nm, r in zip(lp._cuts, rows)})
        lp._factor_ref = (sh.simplex_calls, k, tuple(lp._cut_keys.values()))
        lp._basis_exact = True
        lp._basis_kept = None
        if st == 1:
            lp._obj, lp._x, lp._y, lp._rc, lp._lower_bound = float('inf'), None, None, None, float('inf')
            continue
        lp._x = CyLPArray(res.x[k])
        lp._y = np.concatenate([res.y[k, :m], res.y[k, rows]]) if rows else res.y[k, :m].copy()
        lp._rc = CyLPArray(res.reduced_costs[k])
        lp._obj = float(res.objective[k])
        lp._lower_bound = lp._obj          # a dual feasible basis: c.x of the basic solution is the dual objective
    if sh.memo is not None:
        for lp in batch:
            if lp._solve_start is not None:
                key = (lp._state_key(), _start_digest(lp._solve_start))
                sh.memo.lps[key] = (lp._status, lp._obj, None if lp._x is None else np.asarray(lp._x).copy(),
                                    None if lp._y is None else lp._y.copy(),
                                    None if lp._rc is None else np.asarray(lp._rc).copy(), lp._basis_out, lp.iteration)


def _deltas_against(lp: CyClpSimplex, l0, u0, limit: int):
    idx = np.flatnonzero((lp._l != l0) | (lp._u != u0))
    if len(idx) > limit:
        return None
    fin = lambda v, s: float(np.inf * s) if abs(v) >= 1e30 else float(v)
    return [(int(j), fin(lp._l[j], -1), fin(lp._u[j], 1)) for j in idx]


def _solve_group_pdhg(sh: SharedLP, batch: List[CyClpSimplex], budget: int, default_opts):
    """One batched PDHG call. Nodes go to the device as the reference creates them
    (base_node.py:592-608): a parent's bounds plus the few bounds each node has moved, with ONE
    primal/dual pair as the common warm start (blp_solve_children_host) — the parent's for the
    children of a strong-branching round, the root's for a frontier of open nodes. No per-node dense
    vector is built on the host. (The first solve of a model, and a node that has moved more than
    256 bounds, take the dense form blp_solve_batch_host.)"""
    eng = sh.engine
    B, n, m, mc = len(batch), sh.n, sh.m, len(sh.cut_names)
    okw = {k: v for k, v in batch[0].solver_opts.items() if k not in ('factor_cache', 'method')}
    if budget < 2147483647:
        okw['max_iters'] = int(min(budget * PDHG_ITERS_PER_PIVOT, 2_000_000_000))
    opts = default_opts(**okw)
    ints = batch[0].integer_indices_hint
    mask = None
    if mc:
        mask = np.zeros((B, mc), dtype=np.uint8)
        for k, lp in enumerate(batch):
            for nm in lp._cuts:
                mask[k, sh.pool_row(lp, nm)] = 1

    def warm_vectors(lp):
        wx, wcuts, wy = lp._warm
        y0 = np.zeros(m + mc)
        y0[:m] = wy
        for nm, v in wcuts.items():
            if nm in lp._cuts:
                y0[m + sh.pool_row(lp, nm)] = v
        return wx, y0

    # a large iteration-limited batch is a strong-branching round: only status and objective of the
    # children are read (pseudo_cost.py:68-100), so their primal/dual vectors stay on the device
    want_xy = budget >= 2147483647 or B * (n + m) <= (1 << 22)
    res = None
    kids = _child_deltas(batch)
    same_warm = all(lp._warm is batch[0]._warm or
                    (lp._warm is not None and batch[0]._warm is not None and lp._warm[0] is batch[0]._warm[0])
                    for lp in batch)
    if kids is not None and same_warm:                    # children of one parent
        pl, pu, deltas = kids
        x0 = y0 = None
        if batch[0]._warm is not None:
            x0, y0 = warm_vectors(batch[0])
        res = eng.solve_children(np.where(pl <= -1e30, -np.inf, pl), np.where(pu >= 1e30, np.inf, pu), deltas,
                                 row_mask=mask, x0=x0, y0=y0, integer_indices=ints, opts=opts,
                                 want_x=want_xy, want_y=want_xy)
    elif sh.root_bounds is not None and sh.root_xy is not None and B > 1:      # a frontier of open nodes
        l0, u0 = sh.root_bounds
        deltas = [_deltas_against(lp, l0, u0, 256) for lp in batch]
        if all(dl is not None for dl in deltas):
            x0, ybase = sh.root_xy
            y0 = np.concatenate([ybase, np.zeros(mc)])
            res = eng.solve_children(np.where(l0 <= -1e30, -np.inf, l0), np.where(u0 >= 1e30, np.inf, u0), deltas,
                                     row_mask=mask, x0=x0, y0=y0, integer_indices=ints, opts=opts,
                                     want_x=want_xy, want_y=want_xy)
    if res is None:
        lb = np.empty((B, n))
        ub = np.empty((B, n))
        any_warm = any(lp._warm is not None for lp in batch)
        x0 = np.zeros((B, n)) if any_warm else None
        y0 = np.zeros((B, m + mc)) if any_warm else None
        for k, lp in enumerate(batch):
            lb[k] = np.where(lp._l <= -1e30, -np.inf, lp._l)
            ub[k] = np.where(lp._u >= 1e30, np.inf, lp._u)
            if lp._warm is not None:
                x0[k], y0[k] = warm_vectors(lp)
        res = eng.solve_batch(lb, ub, row_mask=mask, x0=x0, y0=y0, integer_indices=ints, opts=opts,
                              want_x=want_xy, want_y=want_xy)
    if sh.root_bounds is None:
        sh.root_bounds = (np.asarray(batch[0]._l).copy(), np.asarray(batch[0]._u).copy())
    if sh.root_xy is None and B == 1 and not batch[0]._cuts and int(res.status[0]) == 0 and \
            np.array_equal(batch[0]._l, sh.root_bounds[0]) and np.array_equal(batch[0]._u, sh.root_bounds[1]):
        sh.root_xy = (res.x[0].copy(), res.y[0, :m].copy())
    sh.solve_calls += 1
    sh.last_global_bounds = (res.stats.get('global_incumbent'), res.stats.get('global_lower_bound'))
    sh.lps_solved += B
    sh.kernel_launches += int(res.stats['kernel_launches'])
    for k, lp in enumerate(batch):
        st = int(res.status[k])
        lp._status = st
        lp.iteration = int(res.iterations[k])
        lp._lower_bound = float(res.lower_bound[k])
        lp._basis_out = None
        lp._basis_exact = False
        lp._basis_kept = None
        lp._factor_ref = None
        rows = [sh.pool_row(lp, nm) + m for nm in lp._cuts]
        if st == 1:
            lp._obj, lp._x, lp._y, lp._rc = float('inf'), None, None, None
        elif not want_xy:
            lp._x = lp._y = lp._rc = None
            lp._obj = float(res.objective[k]) if st not in (3, 5) else float(res.lower_bound[k])
        else:
            ysel = np.concatenate([res.y[k, :m], res.y[k, rows]]) if rows else res.y[k, :m].copy()
            x = res.x[k].copy()
            lp._x = CyLPArray(x)
            lp._y = ysel
            full_y = res.y[k]
            lp._rc = CyLPArray(sh.c - sh.A.T @ full_y[:m] -
                               (np.vstack([sh.cut_rows[j - m][0] for j in rows]).T @ full_y[rows] if rows else 0.0))
            # status 3 = budget exhausted: report the Lagrangian bound, the analogue of the
            # dual-feasible objective an iteration-limited dual simplex returns
            lp._obj = float(res.objective[k]) if st not in (3, 5) else float(res.lower_bound[k])
