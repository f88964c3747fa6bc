"""BranchAndBound — the search loop, with a batched LP frontier.

Interface and decisions follow the reference's ``simple_mip_solver/algorithms/branch_and_bound.py``
(constructor :123-213, ``solve`` :215-241, ``_evaluate_node`` :243-266, return processing
:268-306): nodes are taken from the queue one at a time, pruned against the incumbent, bounded,
and either update the incumbent or branch. That order-dependent control flow stays in Python.

New here: before a node is bounded, the LP relaxations of the ``frontier_batch`` best open nodes
are solved together in one GPU call (``BaseNode.prefetch``) and cached in their LP objects; the
loop then proceeds exactly as the sequential one, most ``lp.dual()`` calls being cache hits. The
prefetch is speculative — a prefetched node may later be pruned — and never changes which node is
evaluated next or what any node's bound is, so the tree is the one the sequential loop builds.
"""
from __future__ import annotations

import heapq
import time
from queue import PriorityQueue
from typing import Any, Dict, Iterable, List, Tuple, Type, Union

import numpy as np

from simple_mip_solver_b200.algorithms.base_algorithm import BaseAlgorithm
from simple_mip_solver_b200.compat.binary_tree import BinaryTree
from simple_mip_solver_b200.compat.milp_instance import MILPInstance
from simple_mip_solver_b200.compat.cylp_like import RoundMemo, solve_lps
from simple_mip_solver_b200.nodes.base_node import BaseNode
from simple_mip_solver_b200.utils.tolerance import cutting_plane_progress_tolerance, max_cut_generation_iterations


class BranchAndBoundTree(BinaryTree):
    """Tree of evaluated and open nodes; vertex attribute 'node' holds the Node instance."""

    def get_leaves(self, subtree_root_id: int, depth: int = None, keep: str = 'all') -> List[BaseNode]:
        """Leaves of the subtree under ``subtree_root_id``, optionally after cutting the subtree
        ``depth`` edges below its root (reference :22-61)."""
        assert subtree_root_id in self, 'subtree_root_id must belong to the tree'
        assert keep in ['all', 'feasible', 'not infeasible'], \
            "keep is one of 'all', 'feasible', or 'not infeasible'"
        everyone = [v.attr['node'] for v in self.nodes.values()]
        if depth is None:
            found = [n for n in everyone if n.is_leaf and subtree_root_id in n.lineage]
        else:
            assert isinstance(depth, int) and depth >= 0, 'depth is a nonnegative integer'
            if depth == 0:
                found = self.get_node_instances([subtree_root_id])
            elif depth == 1:
                found = self.get_node_instances(self.get_children(subtree_root_id))
            else:
                shallow = [n for n in everyone if n.is_leaf and subtree_root_id in n.lineage[-depth:]]
                at_depth = [n for n in everyone if len(n.lineage) >= depth + 1 and
                            n.lineage[-(depth + 1)] == subtree_root_id]
                found = shallow + at_depth
        if keep == 'feasible':
            return [n for n in found if n.lp_feasible]
        if keep == 'not infeasible':
            return [n for n in found if n.lp_feasible is not False]
        return found

    def get_disjunction(self, subtree_root_id: int) -> Dict[int, Tuple[np.ndarray, np.ndarray]]:
        return {n.idx: (n.lp.variablesLower.copy(), n.lp.variablesUpper.copy())
                for n in self.get_leaves(subtree_root_id, keep='not infeasible')}

    def get_node_instances(self, node_ids: Union[int, Iterable[int]]):
        single = isinstance(node_ids, int)
        if single:
            node_ids = [node_ids]
        else:
            assert isinstance(node_ids, Iterable) and not isinstance(node_ids, str), \
                'node_ids must be an integer or iterable (that is not a string)'
            node_ids = list(node_ids)
        missing = set(node_ids) - set(self.nodes)
        assert not missing, f'the following node_ids are not in the tree: {missing}'
        found = [self.nodes[i].attr.get('node') for i in node_ids]
        assert all(n is not None for n in found), \
            'each vertex in the branch and bound tree must have an attribute for a node instance'
        return found[0] if single else found

    def subtree_dual_bound(self, subtree_root_id: int, depth: int = None) -> Union[float, int]:
        assert subtree_root_id in self, 'subtree_root_id must belong to the tree'
        return min(n.objective_value if n.objective_value is not None else n.dual_bound
                   for n in self.get_leaves(subtree_root_id, depth=depth))


class BranchAndBound(BaseAlgorithm):
    """Solve a MILP by branch and bound with the search/branch/bound methods of ``Node``."""

    _node_attributes = ['dual_bound', 'objective_value', 'solution', 'lp_feasible', 'mip_feasible',
                        'search_method', 'branch_method', 'idx', 'lp', 'is_leaf', 'lineage']
    _node_funcs = ['bound', 'branch', '__lt__', '__eq__']
    _queue_funcs = ['put', 'get', 'empty']

    def __init__(self, model: MILPInstance, Node: Type[BaseNode] = BaseNode, node_queue: Any = None,
                 node_limit: int = float('inf'), mip_gap: float = .0001, logging: bool = False,
                 max_run_time: float = float('inf'), initial_primal_bound: float = float('inf'),
                 frontier_batch: int = 32, lp_cutoff: bool = False, frontier_cut_rounds: bool = False,
                 **kwargs: Any):
        """``frontier_batch``: how many open nodes have their LP relaxation solved per GPU call
        (1 = one LP per call, as the reference). ``lp_cutoff``: hand the incumbent's value to the LP solver as
        an objective limit, so that a node whose dual bound already reaches it stops iterating (the
        reference solves it to the end and prunes it then, :251, :261; the tree is the same, the node's
        recorded LP value is a bound). ``frontier_cut_rounds``: after a frontier's LPs are solved, run the cut rounds
        of its nodes speculatively in lock step (one batched re-solve and one batched device GMI call per round,
        ``device_gomory`` on) and keep the results for the nodes' own ``bound()`` to find; the search computes what
        it computes with ``frontier_batch=1, device_gomory=True``. All other arguments as in the reference."""
        node_queue = node_queue or PriorityQueue()
        super().__init__(model=model, Node=Node, node_attributes=self._node_attributes,
                         node_funcs=self._node_funcs, **kwargs)
        for func in self._queue_funcs:
            assert callable(getattr(node_queue, func, None)), f'node_queue needs a {func} function'
        assert node_limit == float('inf') or (isinstance(node_limit, int) and node_limit > 0), \
            "node limit must be positive integer or infinity"
        assert 0 <= mip_gap < 1, 'mip_gap is a ratio between 0 and 1'
        assert isinstance(logging, bool), 'logging is boolean'
        assert max_run_time > 0, 'max_run_time is positive value'
        assert initial_primal_bound > -float('inf'), 'initial_primal_bound is real or infinite'
        assert isinstance(frontier_batch, int) and frontier_batch >= 1, 'frontier_batch is a positive integer'
        assert isinstance(frontier_cut_rounds, bool), 'frontier_cut_rounds is boolean'
        special_keys = {'right', 'left', 'cuts'}
        assert set(kwargs.keys()).isdisjoint(special_keys), f'keys {special_keys} are saved for later use'
        assert all(isinstance(k, str) for k in kwargs), 'kwargs keys must be strings'

        self._node_queue = node_queue
        self._unbounded = None
        self._best_solution = None
        self.solution = None
        self.status = 'unsolved'
        self.objective_value = None
        self.primal_bound = initial_primal_bound
        self.node_limit = node_limit
        self.tree = BranchAndBoundTree()
        self.tree.add_root(self.root_node.idx, node=self.root_node)
        self.solve_time = 0
        self.mip_gap = mip_gap
        self.logging = logging
        self.max_run_time = max_run_time
        self.frontier_batch = frontier_batch
        self.lp_cutoff = bool(lp_cutoff)
        self.prefetch_calls = 0
        self.prefetched_lps = 0
        self.unsolved_nodes = 0         # nodes whose LP stopped on the solver's iteration budget
        self.frontier_bounds = (None, None)
        self.frontier_cut_rounds = frontier_cut_rounds
        if frontier_cut_rounds:
            self._kwargs['device_gomory'] = True          # on the bus: the rounds the memo answers are device rounds
            self.root_node.lp._need_shared().memo = RoundMemo()

    @property
    def _memo(self):
        return getattr(self.root_node.lp._shared, 'memo', None)

    @property
    def speculative_lps(self) -> int:
        """LPs the speculative cut rounds solved (frontier_cut_rounds)."""
        return self._memo.speculative_lps if self._memo is not None else 0

    @property
    def memo_hits(self) -> int:
        """LP solves and cut generations of real nodes answered by the speculative rounds."""
        return self._memo.lp_hits + self._memo.cut_hits if self._memo is not None else 0

    @property
    def cut_round_resolves(self) -> int:
        """Real nodes that solved an LP again to get its factor back for device cuts."""
        return self._memo.cut_round_resolves if self._memo is not None else 0

    @property
    def dual_bound(self):
        return self.tree.subtree_dual_bound(self.root_node.idx)

    @property
    def current_gap(self):
        if self.primal_bound == self.dual_bound == 0:
            return 0
        if self.primal_bound == 0:
            return float('inf')
        if self.primal_bound == float('inf'):
            return None
        return abs(self.primal_bound - self.dual_bound) / abs(self.primal_bound)

    def solve(self) -> None:
        start = time.process_time()
        if self.status == 'unsolved':
            self._node_queue.put(self.root_node)

        def finished():
            gap = self.current_gap
            return (self._node_queue.empty() or self._unbounded or
                    self.evaluated_nodes >= self.node_limit or
                    (gap is not None and gap <= self.mip_gap) or
                    time.process_time() - start > self.max_run_time)

        while not finished():
            if self.logging and self.evaluated_nodes % 100 == 0:
                print(f'{self.evaluated_nodes} nodes evaluated gap: {self.current_gap}')
            node = self._node_queue.get()
            if self.lp_cutoff and self.primal_bound < float('inf') and hasattr(node.lp, 'solver_opts'):
                node.lp.solver_opts['obj_cutoff'] = float(self.primal_bound)     # shared by the model's LPs
            self._prefetch_frontier(node)
            self._evaluate_node(node)

        self.solve_time += time.process_time() - start
        if self._unbounded:
            self.status = 'unbounded'
        elif self._node_queue.empty() and self.primal_bound == float('inf') and not self.unsolved_nodes:
            self.status = 'infeasible'
        elif self.primal_bound < float('inf') and self.current_gap is not None and self.current_gap <= self.mip_gap:
            self.status = 'optimal'
        else:
            self.status = 'stopped on iterations or time'
        self.solution = self._best_solution
        self.objective_value = self.primal_bound

    def _prefetch_frontier(self, node: BaseNode) -> None:
        """If ``node``'s LP is not solved yet, solve it together with the LPs of the best open
        nodes still in the queue (those that would not be pruned right now) in one GPU call."""
        if self.frontier_batch <= 1 or node.lp._solved_key is not None:
            return
        if not node.dual_bound < self.primal_bound:
            return
        pending = getattr(self._node_queue, 'queue', None)
        batch = [node]
        if pending:
            want = self.frontier_batch - 1
            open_nodes = [n for n in pending if n.lp._solved_key is None and
                          n.dual_bound < self.primal_bound]
            batch += heapq.nsmallest(want, open_nodes)
        memo = self._memo
        if memo is not None and len(memo.lps) > self.MEMO_LPS:
            memo.clear()            # bounded: what is dropped is solved again by its node, as without the memo
        sent = type(node).prefetch(batch)
        self.prefetch_calls += 1
        self.prefetched_lps += sent
        if memo is not None:
            self._speculate_cut_rounds(batch)
        # with several GPUs the shards of the batch agree on [incumbent, dual bound] through
        # blp_allreduce_min; kept for monitoring — pruning stays in the reference's node order
        self.frontier_bounds = getattr(getattr(node.lp, '_shared', None), 'last_global_bounds', (None, None))

    def _evaluate_node(self, node: BaseNode) -> None:
        """Bound the node unless the incumbent prunes it; then record a new incumbent or branch
        (reference :243-266)."""
        if not node.dual_bound < self.primal_bound:
            return
        self.evaluated_nodes += 1
        self._process_bound_rtn(node.bound(**self._kwargs))
        if node.unbounded:
            self._unbounded = True
        if getattr(node, 'lp_unsolved', False):
            # the LP hit the solver's iteration budget: the node stays an open leaf carrying the dual
            # bound it reached (never dropped as infeasible, never branched on an unconverged point)
            self.unsolved_nodes += 1
            return
        if node.lp_feasible and node.objective_value < self.primal_bound:
            if node.mip_feasible:
                self._best_solution = node.solution
                self.primal_bound = node.objective_value
            else:
                self._process_branch_rtn(node.idx, node.branch(**self._kwargs))

    def _process_branch_rtn(self, parent_id: int, rtn: Dict[str, Any]):
        assert isinstance(rtn, dict), 'rtn must be a dictionary'
        assert isinstance(parent_id, int), 'parent_id must be integer'
        assert parent_id in self.tree, 'parent must already exist in tree'
        for direction in ['left', 'right']:
            assert direction in rtn, f'{direction} must be in the returned dict'
            child = rtn[direction]
            assert isinstance(child, self._Node), f'{direction} value must be type {type(self._Node)}'
            assert child.idx not in self.tree, 'please give unique node ID'
            del rtn[direction]          # only a child that was accepted leaves the caller's dict
            self._node_queue.put(child)
            getattr(self.tree, f'add_{direction}_child')(child.idx, parent_id, node=child)
        self._process_rtn(rtn)

    def _process_bound_rtn(self, rtn: Dict[str, Any]):
        """Cuts returned under key 'cuts' are shared with every queued node's cut pool
        (reference :291-306); the rest goes on the kwargs bus."""
        assert isinstance(rtn, dict), 'rtn must be a dictionary'
        cuts = rtn.pop('cuts', None) if 'cuts' in rtn else None
        if cuts:
            for name, (pi, pi0) in cuts.items():
                for queued in self._node_queue.queue:
                    queued.cut_pool[name] = (pi, pi0)
        self._process_rtn(rtn)

    # ---------------------------------------------------------------- speculative cut rounds
    MEMO_LPS = 1024         # LP results the RoundMemo holds before the next frontier prefetch empties it
    _BOUND_ARGS = frozenset(('max_cut_generation_iterations', 'cut_generation_dual_bound_dict',
                             'max_cut_generation_run_time', 'max_dual_bound', 'pseudo_costs', 'strong_branch_iters',
                             'total_cut_generation_iterations', 'total_iterations_gmic_created',
                             'total_number_gmic_created', 'total_iterations_gmic_added', 'total_number_gmic_added',
                             'total_iterations_gmic_removed', 'total_number_gmic_removed'))

    def _speculate_cut_rounds(self, batch: List[BaseNode]) -> None:
        """The cut rounds of a freshly prefetched frontier, run ahead on copies of its nodes in lock step: each round
        prepares every copy whose ``_base_bound`` loop would go on, re-solves their LPs together and forms the next
        round's cuts of all of them in one device call. What the copies solve and cut lands in the RoundMemo; a real
        node's ``bound()`` then runs unchanged and finds its rounds answered where its state is the copy's (a 'cuts'
        broadcast into its pool, or a pool rebuild, makes it differ and it solves for itself)."""
        from simple_mip_solver_b200.nodes.nodes import (DepthFirstSearchNode, PseudoCostBranchDepthFirstSearchNode,
                                                        PseudoCostBranchNode)
        kw = self._kwargs
        # the package's own node classes only: a subclass may override a round. A time limit is not deterministic.
        own = (BaseNode, DepthFirstSearchNode, PseudoCostBranchNode, PseudoCostBranchDepthFirstSearchNode)
        if kw.get('max_cut_generation_run_time') is not None or not kw.get('gomory_cuts', True):
            return
        # simplex-path LPs only: a batched first-order solve depends on the batch it was in
        copies = [n._speculative_copy() for n in batch if type(n) in own and n.lp.solve_key is not None]
        if not copies:
            return
        max_rounds = kw.get('max_cut_generation_iterations', max_cut_generation_iterations)
        max_dual = kw.get('max_dual_bound', float('inf'))
        track = kw.get('track_dual_bound', False)
        tol = kw.get('cutting_plane_progress_tolerance', cutting_plane_progress_tolerance)
        rkw = {k: v for k, v in kw.items() if k not in self._BOUND_ARGS}

        def goes_on(s):          # the loop condition of BaseNode._base_bound (no time limit)
            return s.lp_feasible and not s.lp_unsolved and not s.lp_cut_off and not s.mip_feasible and \
                not s.cut_generation_stalled and s.cut_generation_iterations < max_rounds and \
                s.objective_value < max_dual

        for s in copies:
            s._bound_lp()                                    # the prefetched solve
        self._memo_cuts(copies, kw.get('max_gomory_cuts'))
        active = [s for s in copies if goes_on(s)]
        while active:
            before = [s._cut_round_prepare(**rkw) for s in active]
            for chunk in self._simplex_chunks(active):
                solve_lps([s.lp for s in chunk])
                self._memo.speculative_lps += len(chunk)
                for s in chunk:
                    s._bound_lp(track_dual_bound=track)
                # each call replaces the factor store: this chunk's cuts before the next chunk's call
                self._memo_cuts(chunk, kw.get('max_gomory_cuts'))
            for s, b in zip(active, before):
                s._cut_round_finish(b, tol)
            active = [s for s in active if goes_on(s)]

    @staticmethod
    def _simplex_chunks(nodes: List[BaseNode]):
        """Chunks that reach the engine as one simplex call each, as a single node's solve would (under 'auto' a
        larger batch of mid-size LPs would go to the first-order path)."""
        sh = nodes[0].lp._shared
        k = len(nodes)
        while k > 1 and not sh.use_simplex(k):
            k //= 2
        k = max(1, min(k, sh.simplex_call_size(k)))
        return [nodes[i:i + k] for i in range(0, len(nodes), k)]

    def _memo_cuts(self, nodes: List[BaseNode], max_gomory_cuts) -> None:
        """Device GMI cuts of the next round of every node whose solve is feasible, fractional and still in the factor
        store, all in one simplex_gmi_cuts call, into the RoundMemo: not only for the rounds the copies' loops reach,
        because the real node may go on where its copy stopped."""
        todo = []
        for s in nodes:
            key = s.lp.solve_key
            # a round that first removes slack cuts changes the LP: its cuts come from the host path, as always
            if key is None or not s.lp_feasible or s.mip_feasible or s.lp_unsolved or s.lp_cut_off or \
                    not s.lp.has_stored_factor or s._slack_cut_names():
                continue
            sol = s.solution
            s.solution = np.maximum(sol, 0)               # what _cut_round_prepare hands to _generate_cuts
            try:
                req = s._gomory_requests(max_gomory_cuts)
            finally:
                s.solution = sol
            if req is not None:
                todo.append((s, key, req))
        calls = [(s, key, req) for s, key, req in todo if req[0]]
        for s, key, req in todo:
            if not req[0]:
                self._memo.cuts[(key, s.idx, s.cut_generation_iterations + 1, max_gomory_cuts)] = {}
        if not calls:
            return
        slots, variables, f0s = [], [], []
        for s, key, req in calls:
            slot, to_pool = s.lp._stored_factor()
            variables += list(to_pool[np.asarray(req[1], dtype=int)])
            slots += [slot] * len(req[1])
            f0s += req[2]
        pi, pi0, code = calls[0][0].lp._shared.engine.simplex_gmi_cuts(slots, variables, f0s, calls[0][2][3])
        t = 0
        for s, key, req in calls:
            k = len(req[1])
            cuts = BaseNode._cuts_of_device(req[0], pi[t:t + k], pi0[t:t + k], code[t:t + k])
            t += k
            if cuts is not None:
                self._memo.cuts[(key, s.idx, s.cut_generation_iterations + 1, max_gomory_cuts)] = \
                    {r: (np.asarray(p).copy(), p0) for r, (p, p0) in cuts.items()}
