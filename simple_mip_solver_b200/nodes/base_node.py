"""BaseNode — best-first search, most-fractional branching, LP bound with cut rounds.

Same Node API as the reference's ``simple_mip_solver/nodes/base_node.py`` (attributes, method
names, argument meaning, assertion messages), so ``BranchAndBound(model, Node).solve()`` and user
subclasses work unchanged. What differs is how the LP work is done:

* a child is the parent's shared LP plus one changed bound (``lp.copy_for_child()``) instead of a
  rebuilt model (reference :592-608);
* ``_bound_lp`` asks the GPU engine, and ``BaseNode.prefetch`` / ``_strong_branch_batch`` hand many
  node LPs to it in one call (the reference solves one LP per ``lp.dual()``, :273, :646).
"""
from __future__ import annotations

import copy
import re
import time
from math import acos, ceil, degrees, floor
from statistics import median
from typing import Any, Dict, Iterable, List, Sequence, Set, Tuple, TypeVar, Union

import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from simple_mip_solver_b200.compat.cylp_like import CyClpSimplex, CyLPArray, solve_lps
from simple_mip_solver_b200.engine import GMI_OK, GMI_ZERO
from simple_mip_solver_b200.utils.floating_point import numerically_safe_cut
from simple_mip_solver_b200.utils.tolerance import (
    cutting_plane_progress_tolerance, good_coefficient_approximation_epsilon,
    max_cut_generation_iterations, max_nonzero_coefs, max_relative_cut_term_ratio, min_cut_depth,
    parallel_cut_tolerance, variable_epsilon)

T = TypeVar('T', bound='BaseNode')

_COUNTER_KEYS = ('total_cut_generation_iterations', 'total_iterations_gmic_created',
                 'total_number_gmic_created', 'total_iterations_gmic_added',
                 'total_number_gmic_added', 'total_iterations_gmic_removed',
                 'total_number_gmic_removed')


class BaseNode:
    """A node of the branch and bound tree; other node types subclass it."""

    def __init__(self: T, lp: CyClpSimplex, integer_indices: List[int], idx: int = None,
                 dual_bound: Union[float, int] = -float('inf'), b_idx: int = None,
                 b_dir: str = None, b_val: float = None, depth: int = 0,
                 ancestors: tuple = None, *args, **kwargs):
        # argument checks: messages as in the reference (base_node.py:49-71)
        assert isinstance(lp, CyClpSimplex), 'lp must be CyClpSimplex instance'
        # a child carries the very list its parent was checked with (lp.copy_for_child hands it on): the
        # O(|I|) checks run once per model, not once per node (24 ms a node at 10 000 integer variables)
        index_set = getattr(lp, 'integer_index_set', None) if lp.integer_indices_hint is integer_indices else None
        if index_set is None:
            n_vars = lp.nVariables
            assert all(isinstance(i, int) and 0 <= i < n_vars for i in integer_indices), \
                'indices must match variables'
        assert idx is None or isinstance(idx, int), 'node idx must be integer if provided'
        if index_set is None:
            index_set = frozenset(integer_indices)
            assert len(index_set) == len(integer_indices), 'indices must be distinct'
        assert isinstance(dual_bound, (float, int)), 'dual bound must be a float or an int'
        assert (b_dir is None) == (b_idx is None) == (b_val is None), 'none are none or all are none'
        assert b_idx is None or b_idx in index_set, \
            'branch index corresponds to integer variable if it exists'
        assert b_dir in ['right', 'left'] or b_dir is None, 'we can only branch right or left'
        if b_val is not None:
            good_left = 0 < b_val - lp.variablesUpper[b_idx] < 1
            good_right = 0 < lp.variablesLower[b_idx] - b_val < 1
            assert (b_dir == 'left' and good_left) or (b_dir == 'right' and good_right), \
                'branch val should be within 1 of both bounds'
        assert isinstance(depth, int) and depth >= 0, 'depth is a positive integer'
        if ancestors is not None:
            assert isinstance(ancestors, tuple), 'ancestors must be a tuple if provided'
            assert idx not in ancestors, 'idx cannot be an ancestor of itself'

        lp.logLevel = 0
        lp.integer_indices_hint = integer_indices
        lp.integer_index_set = index_set
        self.lp = lp
        self._integer_indices = integer_indices
        self.idx = idx
        self.dual_bound = dual_bound
        self.objective_value = None
        self.solution = None
        self.lp_feasible = None
        self.lp_unsolved = False
        self.lp_cut_off = False
        self.unbounded = None
        self.mip_feasible = None
        self._b_dir, self._b_idx, self._b_val = b_dir, b_idx, b_val
        self.depth = depth
        self.search_method = 'best first'
        self.branch_method = 'most fractional'
        self.is_leaf = True
        self.lineage = ((ancestors or tuple()) + ((idx,) if idx is not None else tuple())) or None
        self.children = None
        # cut bookkeeping (reference :99-114)
        self.cut_name_pattern = re.compile('^cut_')
        self.gmic_name_pattern = re.compile('^cut_gomory_')
        self._cut_pool = {}
        self._status_override = None    # (cols, rows) to read the basis from instead of lp.getBasisStatus()
        self.cut_generation_iterations = 0
        self.cut_generation_stalled = False
        self.cut_generation_terminator = None
        self.cut_generation_dual_bound = {}
        self.tracked_cut_generation_iterations = 0
        for op in ('created', 'added', 'removed'):
            setattr(self, f'iterations_gmic_{op}', 0)
            setattr(self, f'number_gmic_{op}', 0)
        # largest |coefficient| of the first constraint object (reference :104); a 0-d CyLPArray, as CyLP's
        # coefficient matrices make it (the reference's tests check the type)
        self.max_term = CyLPArray(self.lp.first_constraint_max_term())

        assert self._sense == '>=', 'must have Ax >= b'
        assert self._variables_nonnegative, 'must have x >= 0 for all variables'

    # ---------------------------------------------------------------- cut pool
    @property
    def cut_pool(self):
        return self._cut_pool

    @cut_pool.setter
    def cut_pool(self, cuts: Dict[str, Tuple[CyLPArray, float]]):
        for name, (pi, pi0) in cuts.items():
            assert self.cut_name_pattern.match(name), 'idx should start with "cut_"'
            assert isinstance(pi, CyLPArray), 'pi should be CyLPArray'
            assert isinstance(pi0, (int, float)), 'pi0 should be number'
        self._cut_pool = cuts

    # ---------------------------------------------------------------- bounding
    def bound(self: T, **kwargs: Any) -> Dict[str, Any]:
        return self._base_bound(**kwargs)

    @staticmethod
    def prefetch(nodes: Iterable['BaseNode']) -> int:
        """Solve the LP relaxations of many nodes of one model in a single batched GPU call.

        New relative to the reference, which has no batched entry point. The results stay cached
        in each ``node.lp``; a later ``node.bound()`` finds its first LP already solved. Returns
        the number of LPs sent to the GPU."""
        return solve_lps([n.lp for n in nodes])

    def _base_bound(self: T, max_cut_generation_iterations: int = max_cut_generation_iterations,
                    total_cut_generation_iterations: int = 0, total_iterations_gmic_created: int = 0,
                    total_number_gmic_created: int = 0, total_iterations_gmic_added: int = 0,
                    total_number_gmic_added: int = 0, total_iterations_gmic_removed: int = 0,
                    total_number_gmic_removed: int = 0,
                    cut_generation_dual_bound_dict: Dict[int, Dict[int, float]] = None,
                    max_cut_generation_run_time: int = None, max_dual_bound: float = float('inf'),
                    **kwargs) -> Dict[str, Any]:
        """Solve the LP relaxation, then run cut rounds while they help (reference :137-230)."""
        totals = dict(zip(_COUNTER_KEYS, (
            total_cut_generation_iterations, total_iterations_gmic_created,
            total_number_gmic_created, total_iterations_gmic_added, total_number_gmic_added,
            total_iterations_gmic_removed, total_number_gmic_removed)))
        cut_generation_dual_bound_dict = cut_generation_dual_bound_dict or {}
        assert isinstance(max_cut_generation_iterations, (int, float)) and \
            max_cut_generation_iterations > 0, 'max_cut_generation_iterations must be a positive number'
        for key, value in totals.items():
            assert isinstance(value, int) and value >= 0, f"{key} is nonnegative integer"
        if cut_generation_dual_bound_dict:
            good, msg = self._good_cut_generation_dual_bound_dict(cut_generation_dual_bound_dict)
            assert good, msg
        if max_cut_generation_run_time is None:
            max_cut_generation_run_time = float('inf')
        assert isinstance(max_cut_generation_run_time, (float, int)) and \
            max_cut_generation_run_time >= 0, 'max_cut_generation_run_time is nonnegative'
        assert isinstance(max_dual_bound, (float, int)), 'max_dual_bound is a number'

        self._bound_lp()
        start = time.process_time()

        def out_of_time():
            return time.process_time() - start >= max_cut_generation_run_time

        while self.lp_feasible and not self.lp_unsolved and not self.lp_cut_off and not self.mip_feasible and not self.cut_generation_stalled \
                and self.cut_generation_iterations < max_cut_generation_iterations \
                and not out_of_time() and self.objective_value < max_dual_bound:
            self._cut_generation_iteration(**kwargs)
        if self.cut_generation_iterations == max_cut_generation_iterations:
            self.cut_generation_terminator = 'max iterations'
        elif out_of_time():
            self.cut_generation_terminator = 'time'
        elif self.objective_value > max_dual_bound:
            self.cut_generation_terminator = 'dual bound'

        mine = (self.cut_generation_iterations, self.iterations_gmic_created,
                self.number_gmic_created, self.iterations_gmic_added, self.number_gmic_added,
                self.iterations_gmic_removed, self.number_gmic_removed)
        rtn = {key: totals[key] + inc for key, inc in zip(_COUNTER_KEYS, mine)}
        if self.idx is not None and self.cut_generation_dual_bound:
            cut_generation_dual_bound_dict[self.idx] = self.cut_generation_dual_bound
            rtn['cut_generation_dual_bound_dict'] = cut_generation_dual_bound_dict
        return rtn

    def _good_cut_generation_dual_bound_dict(self, d) -> Tuple[bool, Union[str, None]]:
        """(ok, message) for a ``{node idx: {cut round: dual bound}}`` record travelling on the kwargs
        bus. The messages are part of the reference's API contract (its tests match on them,
        test_base_node.py:176-313); the checks are written as a first-failure search."""
        def first_problem():
            if not isinstance(d, dict):
                yield 'cut_generation_dual_bound_dict should be a dictionary'
                return
            for idx, rounds in d.items():
                problems = (
                    (not isinstance(idx, int), f'index {idx} should be integer'),
                    (idx == self.idx, f'index {idx} has already been processed'),
                    (not isinstance(rounds, dict), f'index {idx} should have dictionary value'),
                )
                yield from (msg for bad, msg in problems if bad)
                if not isinstance(rounds, dict):
                    continue
                yield from (f'cut index {k} for node {idx} should be integer'
                            for k in rounds if not isinstance(k, int))
                yield from (f'dual bound for node {idx} cut index {k} should be a number'
                            for k, v in rounds.items() if not isinstance(v, (int, float)))
                if sorted(rounds) != list(range(len(rounds))):          # rounds 0, 1, ..., no gaps
                    yield f'index {idx} should have dictionary keyed by range of ints'
        msg = next(first_problem(), None)
        return msg is None, msg

    def _bound_lp(self: T, track_dual_bound: bool = False) -> None:
        """Solve this node's LP relaxation and record status, objective, solution and the
        integrality verdict (reference :259-286). A cached batched solve counts as the solve."""
        assert self._x_only_variable, 'x must be our only variable'
        assert isinstance(track_dual_bound, bool), 'track_dual_bound is boolean'
        if track_dual_bound:
            assert self.tracked_cut_generation_iterations not in self.cut_generation_dual_bound, \
                'lp is only bound once per cut generation iteration'
        self.lp.dual()
        self._read_lp()
        if track_dual_bound:
            self.cut_generation_dual_bound[self.tracked_cut_generation_iterations] = self.objective_value

    def _read_lp(self: T) -> None:
        code = self.lp.getStatusCode()
        # CLP never stops a normal bound on an iteration count; the device solvers can (PDHG's
        # iteration budget on a degenerate LP, the simplex kernel's anti-cycling cap). Such a node
        # is NOT infeasible: it stays an open leaf whose value is the dual bound the solve reached,
        # and the search reports 'stopped on iterations or time' unless the incumbent closes it.
        self.lp_unsolved = code == 3 and self.lp.maxNumIteration >= 2147483647
        self.lp_feasible = code in [0, 2] or self.lp_unsolved     # optimal or dual infeasible (:274)
        self.unbounded = code == 2
        self.objective_value = self.lp.objectiveValue if self.lp_feasible else float('inf')
        # status 5: the solve was stopped by the objective limit (blp_opts.obj_cutoff, opt-in through
        # BranchAndBound(lp_cutoff=True)): the node's value is a lower bound that already reaches the
        # incumbent, so the search prunes it exactly where the reference would (branch_and_bound.py:261)
        self.lp_cut_off = code == 5
        if self.lp_cut_off:
            self.lp_feasible = True
        if self.lp_unsolved or self.lp_cut_off:
            self.objective_value = float(self.lp.lagrangianBound)
            self.solution = self.lp.primalVariableSolution['x']
            self.mip_feasible = False
            return
        sol = self.lp.primalVariableSolution
        self.solution = None if not self.lp_feasible else sol['x'] if isinstance(sol, dict) else sol
        if self.lp_feasible and len(self._integer_indices):
            vals = self.solution[self._integer_indices]
            self.mip_feasible = bool(np.max(np.abs(np.round(vals) - vals)) <= variable_epsilon)
            if self.mip_feasible and not self.unbounded:
                # A simplex vertex that passes this test is integral to machine precision; a
                # first-order solution is integral to the solve tolerance. Snap the integer
                # variables so that an incumbent's objective is the objective of an integral point.
                x = np.array(self.solution, dtype=float)
                x[self._integer_indices] = np.round(vals)
                self.solution = CyLPArray(x)
                self.objective_value = float(np.dot(np.asarray(self.lp.objective), x))
        else:
            self.mip_feasible = bool(self.lp_feasible)

    # ---------------------------------------------------------------- cut rounds
    def _cut_generation_iteration(self: T, cutting_plane_progress_tolerance: float =
                                  cutting_plane_progress_tolerance, track_dual_bound: bool = False,
                                  **kwargs: Any) -> None:
        """One round: drop slack cuts, generate, select and append, re-solve (reference :292-324)."""
        before = self._cut_round_prepare(cutting_plane_progress_tolerance, track_dual_bound, **kwargs)
        self._bound_lp(track_dual_bound=track_dual_bound)
        self._cut_round_finish(before, cutting_plane_progress_tolerance)

    def _cut_round_prepare(self: T, cutting_plane_progress_tolerance: float = cutting_plane_progress_tolerance,
                           track_dual_bound: bool = False, **kwargs: Any) -> float:
        """First half of a cut round, up to the re-solve: returns the objective before it. Shared by
        ``_cut_generation_iteration`` and the lock-step rounds of ``BranchAndBound(frontier_cut_rounds=True)``."""
        assert all(self.solution > -variable_epsilon), 'we must have x >= 0'
        assert isinstance(cutting_plane_progress_tolerance, float) and \
            cutting_plane_progress_tolerance > 0, 'cutting_plane_progress_tolerance must be positive'
        assert isinstance(track_dual_bound, bool), 'track_dual_bound is boolean'
        self.solution = np.maximum(self.solution, 0)
        self.cut_generation_iterations += 1
        if track_dual_bound:
            self.tracked_cut_generation_iterations += 1
        before = self.objective_value
        self._remove_slack_cuts(**kwargs)
        self.cut_pool = {**self.cut_pool, **self._generate_cuts(**kwargs)}
        self._select_cuts(**kwargs)
        return before

    def _cut_round_finish(self: T, before: float,
                          cutting_plane_progress_tolerance: float = cutting_plane_progress_tolerance) -> None:
        """Second half of a cut round, after the re-solve: the stall test."""
        if before == 0 or abs(before - self.objective_value) / abs(before) < cutting_plane_progress_tolerance:
            self.cut_generation_stalled = True
            self.cut_generation_terminator = self.cut_generation_terminator or 'cuts not deep enough'

    def _remove_slack_cuts(self: T, **kwargs) -> List[str]:
        """Remove cut rows whose dual is zero (reference :326-341). A first-order dual is zero
        only up to the solve tolerance, so 'zero' means below 1e-9 of the largest row dual."""
        removable = self._slack_cut_names()
        for name in removable:
            self.lp.removeConstraint(name)
        self._update_gmic_counts(cut_idxs=removable, operation='removed')
        return removable

    def _slack_cut_names(self: T) -> List[str]:
        duals = self.lp.dualConstraintSolution
        biggest = max((float(np.max(np.abs(v))) for v in duals.values() if len(v)), default=0.0)
        thresh = 1e-9 * max(1.0, biggest)
        return [name for name, v in duals.items() if self.cut_name_pattern.match(name) and np.all(np.abs(v) <= thresh)]

    def _update_gmic_counts(self, cut_idxs: Union[Set[str], List[str], Dict[str, Any]],
                            operation: str) -> None:
        assert isinstance(cut_idxs, (set, list, dict)), \
            "cut_idxs should be an iterable of strings, but not a single string itself"
        for name in cut_idxs:
            assert isinstance(name, str), "each item in cut_idx should be str type"
        assert operation in ['added', 'created', 'removed'], \
            'operation must be "added", "created", or "removed"'
        hits = sum(1 for name in cut_idxs if self.gmic_name_pattern.match(name))
        setattr(self, f'iterations_gmic_{operation}',
                getattr(self, f'iterations_gmic_{operation}') + (1 if hits else 0))
        setattr(self, f'number_gmic_{operation}', getattr(self, f'number_gmic_{operation}') + hits)

    def _generate_cuts(self: T, gomory_cuts: bool = True, max_gomory_cuts: int = None,
                       device_gomory: bool = False, **kwargs) -> Dict[str, Tuple[CyLPArray, float]]:
        """``max_gomory_cuts`` (new; default None = one cut per fractional basic integer variable, as
        the reference :365-385): only the rows of the most fractional ones — a root with thousands of
        fractional variables would otherwise spend its time rounding thousands of dense cuts on the host.
        ``device_gomory`` (new; default False): while the factorised basis of this LP's simplex solve is in
        the engine's store, the cuts of the same rows are formed and rounded on the device in one call
        (``_device_gomory_cuts``); their round-off is the device's, not the host's. Otherwise, and with the
        option off, the host path."""
        assert isinstance(gomory_cuts, bool), 'gomory_cuts is boolean'
        assert max_gomory_cuts is None or (isinstance(max_gomory_cuts, int) and max_gomory_cuts > 0), \
            'max_gomory_cuts is a positive integer if provided'
        assert isinstance(device_gomory, bool), 'device_gomory is boolean'
        pool = {}
        if gomory_cuts:
            safe = None
            if device_gomory:
                safe = self.lp.memo_cuts(self.idx, self.cut_generation_iterations, max_gomory_cuts) \
                    if self._status_override is None else None
                if safe is None:
                    safe = self._device_gomory_cuts(max_rows=max_gomory_cuts)
            if safe is None:
                safe = {row_idx: numerically_safe_cut(pi=pi, pi0=pi0, estimate='over')
                        for row_idx, (pi, pi0) in self._find_gomory_cuts(max_rows=max_gomory_cuts).items()}
            for row_idx, cut in safe.items():
                pool[f'cut_gomory_{self.idx}_{self.cut_generation_iterations}_{row_idx}'] = cut
            self._update_gmic_counts(cut_idxs=pool, operation='created')
        return pool

    def _select_cuts(self, max_nonzero_coefs: int = max_nonzero_coefs,
                     min_cut_depth: float = min_cut_depth,
                     parallel_cut_tolerance: float = parallel_cut_tolerance,
                     max_relative_cut_term_ratio: float = max_relative_cut_term_ratio,
                     **kwargs) -> Dict[str, Tuple[CyLPArray, float]]:
        """Append the deepest, mutually non-parallel cuts of the pool to the LP (reference
        :387-466); appended rows reach the GPU as masked rows of the shared matrix."""
        assert isinstance(max_nonzero_coefs, int) and 0 < max_nonzero_coefs, \
            'max_nonzero_coefs must be positive int'
        assert isinstance(min_cut_depth, (float, int)) and 0 < min_cut_depth, 'min_cut_depth must be > 0'
        assert 0 < parallel_cut_tolerance <= 90, 'parallel_cut_tolerance must be number in (0, 90]'
        assert isinstance(max_relative_cut_term_ratio, (int, float)) and \
            0 < max_relative_cut_term_ratio, 'max_relative_cut_term_ratio must be positive'
        eps = good_coefficient_approximation_epsilon
        depth = {}
        for name, (pi, pi0) in self.cut_pool.items():
            nnz = int(np.count_nonzero(np.abs(pi) > eps))
            if 0 < nnz <= max_nonzero_coefs:
                depth[name] = (float(np.dot(pi, self.solution)) - pi0) / float(np.linalg.norm(pi))
        if not depth:
            self.cut_generation_terminator = 'no cuts'
        elif min(depth.values()) >= 0:
            self.cut_generation_terminator = 'no improving cuts'
        elif min(depth.values()) >= -min_cut_depth:
            self.cut_generation_terminator = 'no sufficient cuts'

        added = {}
        x = self.lp.getVarByName('x')
        for name in sorted(depth, key=depth.get):
            if depth[name] >= -min_cut_depth:
                break
            pi, pi0 = self.cut_pool[name]
            if np.max(np.abs(pi)) > max_relative_cut_term_ratio * self.max_term:
                continue
            too_parallel = False
            for other, _ in added.values():
                cos_t = median([-1, np.dot(pi, other) / (np.linalg.norm(pi) * np.linalg.norm(other)), 1])
                if degrees(acos(cos_t)) < parallel_cut_tolerance:
                    too_parallel = True
                    break
            if not too_parallel:
                self.lp.addConstraint(pi * x >= pi0, name)
                added[name] = (pi, pi0)
                del self.cut_pool[name]
        self._update_gmic_counts(cut_idxs=added, operation='added')
        return added

    def _find_gomory_cuts(self: T, max_rows: int = None) -> Dict[int, Tuple[CyLPArray, float]]:
        """GMI cuts of the current solution (reference :468-511). The basis is what ``getBasisStatus``
        reports; when that is not a basis of this solution (after slack cuts were removed the LP has no
        solve of its own yet, and the active set of a degenerate vertex need not be one), the basis of the
        last solve minus the removed slack rows is tried — what CLP keeps across ``removeConstraint``."""
        cuts = self._gomory_cuts_of_basis(max_rows)
        kept = getattr(self.lp, 'kept_basis_status', lambda: None)() if cuts is None else None
        if kept is not None:
            self._status_override = kept
            try:
                cuts = self._gomory_cuts_of_basis(max_rows)
            finally:
                self._status_override = None
        return cuts if cuts is not None else {}

    def _basis_status(self):
        return self._status_override if self._status_override is not None else self.lp.getBasisStatus()

    def _gomory_cuts_of_basis(self: T, max_rows: int = None) -> Union[None, Dict[int, Tuple[CyLPArray, float]]]:
        """Gomory mixed integer cuts from the rows of the LP tableau that belong to fractional
        basic integer variables (reference :468-511; Conforti et al. 5.31), vectorised.

        The tableau rows come from the device: ``lp.tableau_rows`` multiplies the rows of the
        factorised basis inverse the dual simplex kernel left behind into ``[A, -I]`` (only the rows
        that are needed; the reference inverts the whole dense basis matrix, :513-526). Nonbasic
        variables sitting at a nonzero bound (a branching bound, an upper bound) are
        shifted/complemented to zero first; the reference's formula assumes nonbasics at zero and is
        the special case without shifts (its pinned ``cut3`` example, test_base_node.py:654-684,
        gives the same cut). When the LP was solved by the first-order path (LPs too large for the
        simplex kernels) the basis is the active set of the solution and is used only if the basic
        solution it defines reproduces the solver's x. Returns None when the status at hand
        (``_basis_status``) is not a basis of this solution."""
        sel = self._gomory_rows(max_rows)
        if sel is None:
            return None
        basic, wanted, is_basic, is_int, offset, sign, A, b = sel
        cuts = {}
        if not wanted:
            return cuts
        n = self.lp.nVariables
        rows = self._tableau_rows([int(basic[r]) for r, _ in wanted])
        if rows is None:
            return None
        for (row_idx, f0), trow in zip(wanted, rows):
            row = np.where(is_basic, 0.0, trow * sign)               # coefficients of the shifted nonbasics
            f = row - np.floor(row)
            pi_int = np.where(f <= f0, f / f0, (1 - f) / (1 - f0))
            pi_cont = np.where(row > 0, row / f0, -row / (1 - f0))
            pi_shift = np.where(is_int, pi_int, pi_cont)
            pi_shift[is_basic] = 0.0
            # sum pi' x' >= 1 with x'_j = sign_j (x_j - offset_j) for structurals, slack = A x - b
            pi_x, pi_s = pi_shift[:n] * sign[:n], pi_shift[n:]
            coefs = pi_x + A.T @ pi_s
            rhs = 1.0 + float(np.dot(pi_x, offset[:n])) + float(np.dot(pi_s, b))
            cuts[row_idx] = (CyLPArray(coefs), rhs)
        return cuts

    def _device_gomory_cuts(self: T, max_rows: int = None) -> Union[None, Dict[int, Tuple[CyLPArray, float]]]:
        """The cuts ``_gomory_cuts_of_basis`` makes of the same rows, already rounded as
        ``numerically_safe_cut(..., estimate='over')``, from ONE device call on the stored factor of this LP's
        last simplex solve (``lp.gmi_cuts``, blp_simplex_gmi_cuts_host). None when that factor is gone, the
        status at hand is not that solve's basis, or the device declines a row (a nonbasic column at an
        infinite bound): the caller then takes the host path, which decides those cases as always."""
        if self._status_override is not None:
            return None
        if not self.lp.has_stored_factor:
            # with speculative cut rounds on, a solve the memo answered left no factor where the one-node-per-call
            # run has one: solve it again (same start, same result) rather than take the host path
            if not self.lp.restore_factor():
                return None
            if not getattr(self, '_speculative', False):
                self.lp._shared.memo.cut_round_resolves += 1
        req = self._gomory_requests(max_rows)
        if req is None:
            return None
        if not req[0]:
            return {}
        got = self.lp.gmi_cuts(*req[1:])
        return None if got is None else self._cuts_of_device(req[0], *got)

    def _gomory_requests(self: T, max_rows: int = None):
        """(wanted [(row position, f0)], basic variables, f0s, integer mask) of the rows ``_gomory_cuts_of_basis``
        picks, or None when the status at hand is not a basis of this solution."""
        sel = self._gomory_rows(max_rows)
        if sel is None:
            return None
        basic, wanted = sel[0], sel[1]
        int_mask = np.zeros(self.lp.nVariables, dtype=np.uint8)
        int_mask[self._integer_indices] = 1
        return wanted, [int(basic[r]) for r, _ in wanted], [f0 for _, f0 in wanted], int_mask

    @staticmethod
    def _cuts_of_device(wanted, pi, pi0, code) -> Union[None, Dict[int, Tuple[CyLPArray, float]]]:
        """Cuts by row position from simplex_gmi_cuts' answer; None if the device declined a row."""
        if not np.isin(code, (GMI_OK, GMI_ZERO)).all():
            return None
        return {row_idx: (CyLPArray(pi[t]), float(pi0[t])) for t, (row_idx, _) in enumerate(wanted)}

    def _speculative_copy(self: T) -> T:
        """A copy of this not yet bounded node for a speculative cut round (same idx, bounds, cuts, basis, cut
        pool and last solve; its own LP object), so that no method of the real node runs."""
        c = copy.copy(self)
        c.lp = self.lp.clone()
        c._cut_pool = dict(self._cut_pool)
        c.cut_generation_dual_bound = dict(self.cut_generation_dual_bound)
        c._speculative = True
        return c

    def _gomory_rows(self: T, max_rows: int = None):
        """Which tableau rows ``_gomory_cuts_of_basis`` turns into cuts: (basic, wanted = [(row position, f0)],
        is_basic, is_int, offset, sign over the n + m variables, A, b), or None when the status at hand is not a
        basis of this solution."""
        n, m = self.lp.nVariables, self.lp.nConstraints
        col_stat, row_stat = self._basis_status()
        basic = self.basic_variable_indices
        if len(basic) != m:
            return None
        is_basic = np.zeros(n + m, dtype=bool)
        is_basic[basic] = True
        is_int = np.zeros(n + m, dtype=bool)
        is_int[self._integer_indices] = True
        A = self.lp.coefMatrix
        b = np.asarray(self.lp.constraintsLower, dtype=float)
        l = np.asarray(self.lp.variablesLower, dtype=float)
        u = np.asarray(self.lp.variablesUpper, dtype=float)
        # nonbasic values: structural at lower / upper bound, slack (A x - b) at zero
        at_upper = np.concatenate([col_stat == 2, np.zeros(m, dtype=bool)])
        offset = np.concatenate([np.where(col_stat == 2, u, l), np.zeros(m)])
        offset[is_basic] = 0.0
        if not np.isfinite(offset).all():
            return None
        sign = np.where(at_upper, -1.0, 1.0)
        x = np.asarray(self.solution, dtype=float)
        if self._status_override is None and self.lp.has_exact_basis:
            x_basic = np.concatenate([x, A @ x - b])[basic]
        elif m <= 512:
            full = np.concatenate((A.toarray(), -np.identity(m)), axis=1)
            try:
                x_basic = np.linalg.solve(full[:, basic], b - full @ offset)
            except np.linalg.LinAlgError:
                return None
        else:
            lu = self._sparse_basis_factor(basic)
            if lu is None:
                return None
            A_full = sp.hstack([sp.csr_matrix(A), -sp.identity(m, format='csr')], format='csr')
            x_basic = lu.solve(b - A_full @ offset)
        if self._status_override is not None or not self.lp.has_exact_basis:
            z = offset.copy()
            z[basic] = x_basic
            if np.max(np.abs(z[:n] - x) / (1.0 + np.abs(x))) > 1e-5:
                return None                      # the active set is not the basis of this solution
        is_int &= np.abs(offset - np.round(offset)) <= 1e-9          # shifted variable stays integer
        eps = good_coefficient_approximation_epsilon
        wanted = []
        for row_idx, j in enumerate(basic):
            if j >= n or j not in self._integer_indices or not self._is_fractional(float(x_basic[row_idx])):
                continue
            f0 = self._get_fraction(float(x_basic[row_idx]))
            if f0 < eps or f0 + eps > 1:
                continue
            wanted.append((row_idx, f0))
        if max_rows is not None and len(wanted) > max_rows:
            keep = sorted(wanted, key=lambda t: -min(t[1], 1 - t[1]))[:max_rows]      # most fractional first (stable)
            wanted = sorted(keep)
        return basic, wanted, is_basic, is_int, offset, sign, A, b

    def _tableau_rows(self, variables: Sequence[int]):
        """Rows of inv([A, -I]_B) [A, -I] for the given basic variables: from the device when the
        factorised basis of this LP's solve is still in the engine's store, else from a dense solve on
        the host (what the reference does for every row, :513-526)."""
        rows = self.lp.tableau_rows(variables) if self._status_override is None else None
        if rows is not None:
            return rows
        basic = self.basic_variable_indices
        m = self.lp.nConstraints
        if len(basic) != m:
            return None
        pos = {int(j): p for p, j in enumerate(basic)}
        if m <= 512:
            # small LPs: the reference's own dense computation (:513-526); its round-off is what the
            # reference's pinned cut rounds (test_base_node.py:316-337) were recorded with
            full = np.concatenate((self.lp.coefMatrix.toarray(), -np.identity(m)), axis=1)
            try:
                T_ = np.linalg.solve(full[:, basic], full)
            except np.linalg.LinAlgError:
                return None
            return np.array([T_[pos[int(v)]] if int(v) in pos else np.zeros(full.shape[1]) for v in variables])
        lu = self._sparse_basis_factor(basic)
        if lu is None:
            return None
        # row of basic variable at position p: z' [A, -I] with B' z = e_p (one sparse solve per row,
        # SURVEY 8f #1) — never the dense m x (n+m) tableau
        A_full = sp.hstack([sp.csr_matrix(self.lp.coefMatrix), -sp.identity(m, format='csr')], format='csc')
        out = np.zeros((len(variables), A_full.shape[1]))
        for t, v in enumerate(variables):
            if int(v) in pos:
                e = np.zeros(m)
                e[pos[int(v)]] = 1.0
                out[t] = A_full.T @ lu.solve(e, trans='T')
        return out

    def _sparse_basis_factor(self, basic):
        """Sparse LU of the basis matrix [A, -I]_B (host; used when the factor is not on the device)."""
        m = self.lp.nConstraints
        A_full = sp.hstack([sp.csr_matrix(self.lp.coefMatrix), -sp.identity(m, format='csr')], format='csc')
        try:
            with np.errstate(all='ignore'):
                import warnings
                with warnings.catch_warnings():
                    warnings.simplefilter('error')
                    return spla.splu(A_full[:, basic].tocsc())
        except Exception:          # singular (RuntimeError) or near-singular (MatrixRankWarning)
            return None

    @property
    def tableau(self):
        """Simplex tableau inv([A, -I]_B) [A, -I] of ``A x - s = b``, one row per basic variable in
        ascending variable order (reference :513-526), or None when the status is not a basis."""
        basic = self.basic_variable_indices
        if len(basic) != self.lp.nConstraints:
            return None
        return self._tableau_rows([int(j) for j in basic])

    @property
    def basic_variable_indices(self):
        return np.where(np.concatenate(self._basis_status()) == 1)[0]

    # ---------------------------------------------------------------- branching
    def branch(self: T, **kwargs: Any) -> Dict[str, T]:
        return self._base_branch(self._most_fractional_index, **kwargs)

    @property
    def _most_fractional_index(self: T) -> int:
        """Integer variable furthest from an integer, first one on ties (reference :544-562)."""
        if not self.lp_feasible or not len(self._integer_indices):
            return None
        ints = np.asarray(self._integer_indices)
        vals = np.asarray(self.solution)[ints]
        dist = np.minimum(vals - np.floor(vals), np.ceil(vals) - vals)
        k = int(np.argmax(dist))            # argmax returns the first maximiser
        return int(ints[k]) if dist[k] > variable_epsilon else None

    def _base_branch(self: T, branch_idx: int, next_node_idx: int = None, **kwargs: Any) -> Dict[str, T]:
        """Two children: ``x[idx] <= floor(v)`` (left) and ``x[idx] >= ceil(v)`` (right), each the
        parent's LP with one bound moved and the parent's primal/dual pair as warm start
        (reference :564-627)."""
        assert self._x_only_variable, 'x must be our only variable'
        assert next_node_idx is None or isinstance(next_node_idx, int), \
            'next node index should be integer if provided'
        assert self.lp_feasible, 'must solve before branching'
        assert branch_idx in self._integer_indices, 'must branch on integer index'
        b_val = float(self.solution[branch_idx])
        assert self._is_fractional(b_val), "index branched on must be fractional"
        self.is_leaf = False
        basis = self.lp.getBasisStatus()
        lps = {}
        for direction in ('right', 'left'):
            lp = self.lp.copy_for_child()
            if direction == 'left':
                lp.variablesUpper[branch_idx] = floor(b_val)
            else:
                lp.variablesLower[branch_idx] = ceil(b_val)
            lp.setBasisStatus(*basis)
            lps[direction] = lp
        self.children = (next_node_idx, next_node_idx + 1) if next_node_idx is not None else None
        common = dict(integer_indices=self._integer_indices, dual_bound=self.objective_value,
                      b_idx=branch_idx, b_val=b_val, depth=self.depth + 1, ancestors=self.lineage)
        return {
            'left': type(self)(lp=lps['left'], idx=next_node_idx, b_dir='left', **common, **kwargs),
            'right': type(self)(lp=lps['right'], b_dir='right',
                                idx=next_node_idx + 1 if next_node_idx is not None else None,
                                **common, **kwargs),
            'next_node_idx': next_node_idx + 2 if next_node_idx is not None else None,
        }

    def _strong_branch(self: T, idx: int, iterations: int = 5) -> Dict[str, T]:
        """Both children of a branch on ``idx`` with an iteration-limited LP solve each
        (reference :629-647)."""
        return self._strong_branch_batch([idx], iterations)[idx]

    def _strong_branch_batch(self: T, indices: Sequence[int], iterations: int = 5) -> Dict[int, Dict[str, T]]:
        """Strong branching on several variables at once: all 2*len(indices) child LPs go to the
        GPU in ONE batched call. The reference loops over ``_strong_branch`` (pseudo_cost.py:60-62)."""
        assert isinstance(iterations, int) and iterations > 0, 'iterations must be positive integer'
        out = {}
        for idx in indices:
            out[idx] = {k: v for k, v in self._base_branch(idx).items() if k in ('left', 'right')}
            for child in out[idx].values():
                child.lp.maxNumIteration = iterations
        solve_lps([child.lp for pair in out.values() for child in pair.values()])
        return out

    def _is_fractional(self: T, value: Union[int, float]) -> bool:
        assert isinstance(value, (int, float)), 'value should be a number'
        return min(value - floor(value), ceil(value) - value) > variable_epsilon

    @staticmethod
    def _get_fraction(value: Union[int, float]) -> Union[int, float]:
        assert isinstance(value, (int, float)), 'value should be a number'
        return value - floor(value)

    # ---------------------------------------------------------------- best-first order
    def __eq__(self: T, other):
        if isinstance(other, BaseNode):
            return self.dual_bound == other.dual_bound
        raise TypeError('A Node can only be compared with another Node')

    def __lt__(self: T, other):
        if isinstance(other, BaseNode):
            return self.dual_bound < other.dual_bound
        raise TypeError('A Node can only be compared with another Node')

    __hash__ = object.__hash__

    def __repr__(self):
        return f'node {self.idx}'

    # ---------------------------------------------------------------- form checks
    @property
    def _sense(self: T):
        inf = self.lp.getCoinInfinity()
        lower_bounded = self.lp.constraintsLower.max() > -inf
        upper_bounded = self.lp.constraintsUpper.min() < inf
        assert not (lower_bounded and upper_bounded), "all constraints should be bounded same way"
        return '<=' if upper_bounded else '>='

    @property
    def _variables_nonnegative(self: T):
        return bool((self.lp.variablesLower >= 0).all())

    @property
    def _x_only_variable(self: T):
        return len(self.lp.variables) == 1 and self.lp.variables[0].name == 'x'
