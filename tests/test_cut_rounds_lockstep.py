"""BranchAndBound(frontier_cut_rounds=True) on the CPU: the speculative lock-step cut rounds of a prefetched frontier
must leave the search exactly as ``frontier_batch=1, device_gomory=True`` runs it — node for node and bit for bit —
while reaching the engine in fewer calls. The stand-in engine solves and forms cuts on each LP's own rows only, in
a canonical row order, so that its answers do not depend on where a cut sits in the device pool (which the two
runs fill in different orders)."""
import json
import os

import numpy as np
import pytest

import simple_mip_solver_b200.engine as engine
from oracle import gmi_device
from oracle.dual_simplex import BASIC, dual_simplex
from simple_mip_solver_b200 import (BaseNode, BranchAndBound, DepthFirstSearchNode, PseudoCostBranchDepthFirstSearchNode,
                                    PseudoCostBranchNode)
from simple_mip_solver_b200.compat.cylp_like import CyLPArray, SharedLP
from test_gmi_device_cuts import GmiOracleBatchLP
from test_gomory import EXAMPLES, SCALE1, model_from
from helpers import use_oracle_engine

GOLD = os.path.join(os.path.dirname(__file__), 'golden')
FUZZ = json.load(open(os.path.join(GOLD, 'fuzz_models.json')))
CLASSES = {'BaseNode': (BaseNode, {}), 'DepthFirstSearchNode': (DepthFirstSearchNode, {}),
           'PseudoCostBranchNode': (PseudoCostBranchNode, {'pseudo_costs': {}}),
           'PseudoCostBranchDepthFirstSearchNode': (PseudoCostBranchDepthFirstSearchNode, {'pseudo_costs': {}})}


class OwnRowsBatchLP(GmiOracleBatchLP):
    """Each LP is solved on its base rows plus its own cut rows sorted by content; results are mapped back to the
    pool numbering. Factors are kept per slot in that reduced form."""

    def _simplex(self, lbs, ubs, masks, css, rss, parents, max_pivots):
        from simple_mip_solver_b200.engine import SimplexBatchResult
        A, b = self._full()
        m, B, n = A.shape[0], len(lbs), self.n
        type(self).calls += 1
        type(self).lps += B
        type(self).batch_sizes.append(B)
        out, store = [], []
        for k in range(B):
            pool = [j for j in range(m - self.m_base) if masks is None or masks[k][j]]
            pool.sort(key=lambda j: (A[self.m_base + j].tobytes(), b[self.m_base + j]))
            rows = list(range(self.m_base)) + [self.m_base + j for j in pool]
            cs = None if css is None else css[k]
            rs = None if rss is None else np.asarray(rss[k])[rows]
            r = dual_simplex(A[rows], b[rows], self.c, lbs[k], ubs[k], col_status=cs, row_status=rs,
                             max_pivots=max_pivots)
            y = np.zeros(m)
            y[rows] = r.y
            rso = np.full(m, BASIC, np.int8)
            rso[rows] = r.row_status
            out.append((r, y, rso))
            store.append((r, rows))
        self._store = tuple(store)
        self._bounds = (np.array(lbs, float), np.array(ubs, float), None)
        return SimplexBatchResult(
            objective=np.array([r.objective for r, _, _ in out]), status=np.array([r.status for r, _, _ in out], np.int32),
            pivots=np.array([r.pivots for r, _, _ in out], np.int32), x=np.array([r.x for r, _, _ in out]),
            y=np.array([y for _, y, _ in out]), reduced_costs=np.array([r.rc for r, _, _ in out]),
            col_status=np.array([r.col_status for r, _, _ in out], np.int8), row_status=np.array([s for _, _, s in out]),
            stats=dict(kernel_launches=0))

    def simplex_gmi_cuts(self, slots, variables, f0, int_mask):
        type(self).gmi_calls += 1
        type(self).gmi_cuts += len(variables)
        A, b = self._full()
        lbs, ubs, _ = self._bounds
        n = self.n
        pis, pi0s, codes = [], [], []
        for s, v, f in zip(slots, variables, f0):
            r, rows = self._store[s]
            v = int(v)
            local = v if v < n else (n + rows.index(v - n) if (v - n) in rows else -1)
            pi, pi0, code = gmi_device.gmi_cut(r, A[rows], b[rows], self.m_base, lbs[s], ubs[s],
                                               np.ones(len(rows), bool), local, float(f), int_mask)
            pis.append(pi)
            pi0s.append(pi0)
            codes.append(code)
        return np.array(pis), np.array(pi0s), np.array(codes, np.int32)

    def simplex_tableau_rows(self, slot, variables):
        r, rows = self._store[slot]
        A, _ = self._full()
        n, m = self.n, A.shape[0]
        full = np.concatenate([A[rows], -np.eye(len(rows))], axis=1)
        pos = {int(v): i for i, v in enumerate(r.head)}
        out = np.zeros((len(variables), n + m))
        for t, v in enumerate(np.asarray(variables).ravel()):
            v = int(v)
            local = v if v < n else (n + rows.index(v - n) if (v - n) in rows else -1)
            if local in pos:
                row = r.Binv[pos[local]] @ full
                out[t, :n] = row[:n]
                out[t, n + np.asarray(rows)] = row[n:]
        return out


@pytest.fixture
def own_rows_engine(monkeypatch):
    use_oracle_engine(monkeypatch)
    OwnRowsBatchLP.gmi_calls = OwnRowsBatchLP.gmi_cuts = 0
    monkeypatch.setattr(engine, 'BatchLP', OwnRowsBatchLP)
    return OwnRowsBatchLP


def run(rec, label, engine_cls, **kw):
    Node, extra = CLASSES[label]
    engine_cls.calls = engine_cls.lps = 0
    engine_cls.batch_sizes = []
    engine_cls.gmi_calls = 0
    bb = BranchAndBound(model_from(rec), Node, **{k: (dict(v) if isinstance(v, dict) else v) for k, v in extra.items()},
                        **kw)
    bb.solve()
    return bb, engine_cls.calls + engine_cls.gmi_calls, list(engine_cls.batch_sizes)


def bits(a):
    return None if a is None else np.asarray(a, dtype=np.float64).tobytes()


def snapshot(bb):
    nodes = {}
    for idx, vert in bb.tree.nodes.items():
        n = vert.attr['node']
        cuts = {nm: (bits(pi), float(pi0)) for nm, (pi, pi0) in n.lp._cuts.items()}
        pool = {nm: (bits(pi), float(pi0)) for nm, (pi, pi0) in n.cut_pool.items()}
        nodes[idx] = (n.objective_value, bits(n.solution), n.lp_feasible, n.mip_feasible, n.is_leaf,
                      n.cut_generation_iterations, n.cut_generation_terminator, cuts, pool)
    kw = {k: v for k, v in bb._kwargs.items() if k not in ('device_gomory',)}
    return bb.status, bb.objective_value, bits(bb.solution), nodes, repr(kw)


def cases():
    return (list(SCALE1.items()) + [(k, EXAMPLES[k]) for k in ('small_branch', 'cut1', 'cut2', 'cut3', 'square')]
            + list(FUZZ.items()))


@pytest.mark.parametrize('label', list(CLASSES))
def test_lock_step_equals_one_node_per_call(own_rows_engine, label):
    total_one = total_lock = batched = 0
    for name, rec in cases():
        one, calls_one, _ = run(rec, label, own_rows_engine, frontier_batch=1, device_gomory=True)
        lock, calls_lock, sizes = run(rec, label, own_rows_engine, frontier_batch=32, frontier_cut_rounds=True)
        assert snapshot(lock) == snapshot(one), name
        assert lock.cut_round_resolves == 0, name
        total_one, total_lock = total_one + calls_one, total_lock + calls_lock
        batched += lock.speculative_lps > 0 and max(sizes) > 1
    print(f'{label}: engine calls {total_one} one node per call, {total_lock} in lock step')
    assert total_lock < total_one and batched > 0


def test_memo_is_used_and_reported(own_rows_engine):
    rec = FUZZ['random_12x6_seed3']
    bb, _, _ = run(rec, 'BaseNode', own_rows_engine, frontier_cut_rounds=True)
    assert bb.speculative_lps > 0 and bb.memo_hits > 0 and bb.cut_round_resolves == 0


def _broadcast_before(monkeypatch, idx):
    """A 'cuts' broadcast into node ``idx``'s pool right before it is bounded (after its frontier was speculated
    on): an objective cut just above the node's dual bound."""
    orig = BranchAndBound._evaluate_node

    def wrapped(self, node):
        if node.idx == idx:
            c = np.asarray(self.root_node.lp.objective, dtype=float)
            node.cut_pool['cut_extra_0'] = (CyLPArray(c), float(node.dual_bound) + 1.0)
        return orig(self, node)
    monkeypatch.setattr(BranchAndBound, '_evaluate_node', wrapped)


@pytest.mark.parametrize('what', ['cuts_broadcast', 'make_room', 'pruned'])
def test_memo_misses_fall_back_and_still_match(own_rows_engine, monkeypatch, what):
    """A node whose state differs from its speculative copy's solves for itself and the search stays the one-node-
    per-call search: a 'cuts' broadcast into a prefetched node's pool, a pool rebuild (make_room) between rounds,
    and prefetched nodes pruned by the incumbent before they are bounded."""
    rebuilds = 0
    for name, rec in cases()[:24]:
        extra = {}
        if what == 'cuts_broadcast':
            _broadcast_before(monkeypatch, 2)
        if what == 'pruned':
            gold = float(rec['reference']['BaseNode_gomory']['objective']) if 'reference' in rec and \
                'BaseNode_gomory' in rec['reference'] else None
            if gold is None or not np.isfinite(gold):
                continue
            extra['initial_primal_bound'] = gold + 1e-6 * max(1.0, abs(gold))
        if what == 'make_room':
            monkeypatch.setattr(SharedLP, 'pool_cap', 0, raising=False)
        runs = []
        for kw in (dict(frontier_batch=1, device_gomory=True), dict(frontier_batch=32, frontier_cut_rounds=True)):
            bb = BranchAndBound(model_from(rec), BaseNode, **extra, **kw)
            if what == 'make_room':
                bb.root_node.lp._need_shared().pool_cap = 0
            bb.solve()
            runs.append(bb)
        assert snapshot(runs[1]) == snapshot(runs[0]), (what, name)
        rebuilds += runs[1].root_node.lp._shared.pool_rebuilds
    assert what != 'make_room' or rebuilds > 0


def test_status_and_optimum_equal_the_goldens(own_rows_engine):
    for name, rec in list(SCALE1.items()) + [(k, EXAMPLES[k]) for k in ('small_branch', 'cut1', 'cut2', 'cut3', 'square')]:
        gold = rec['reference']['BaseNode_gomory']
        bb, _, _ = run(rec, 'BaseNode', own_rows_engine, frontier_cut_rounds=True)
        assert bb.status == gold['status'], name
        want = float(gold['objective'])
        assert abs(bb.objective_value - want) <= 1e-6 * max(1.0, abs(want)), name
