"""GPU: GMI cuts of stored simplex factors (blp_simplex_gmi_cuts_host, BatchLP.simplex_gmi_cuts) and the Node
layer's device_gomory path. Every cut must match the numpy restatement of the kernel (oracle/gmi_device.py) bit
for bit; the restatement is given the device's own basis row, read back through blp_simplex_tableau_rows_host
(the slack part of a tableau row is -Binv(r, :)), so this file checks the cut kernel and not the pivoting."""
import json
import os
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import gmi_device
from simple_mip_solver_b200 import BaseNode, BranchAndBound, CyLPArray, MILPInstance, engine
from simple_mip_solver_b200.compat import solve_lps
from simple_mip_solver_b200.instances import grumpy_random_mip
from simple_mip_solver_b200.utils.floating_point import numerically_safe_cut

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), 'golden')
SCALE1 = json.load(open(os.path.join(GOLD, 'scale_1_models.json')))
EXAMPLES = json.load(open(os.path.join(GOLD, 'example_models.json')))


def model_from(rec):
    return MILPInstance(A=np.array(rec['A']), b=CyLPArray(rec['b']), c=CyLPArray(rec['c']),
                        l=CyLPArray(rec['l']), u=CyLPArray(rec['u']), sense=['Min', '>='],
                        integerIndices=list(rec['integer_indices']), numVars=len(rec['c']))


def _requests(d, res, per_slot):
    """(slot, var, f0): the fractional basic integers of every node, plus one nonbasic structural and one basic
    slack per node."""
    n = len(d.c)
    out = []
    for k in range(len(res.status)):
        if res.status[k] != 0:
            continue
        x = res.x[k]
        basic = np.flatnonzero(res.col_status[k] == 1)
        frac = [j for j in basic if j in d.integer_indices and 1e-2 < x[j] - np.floor(x[j]) < 1 - 1e-2]
        out += [(k, int(j), float(x[j] - np.floor(x[j]))) for j in frac[:per_slot]]
        nonbasic = np.flatnonzero(res.col_status[k] != 1)
        if len(nonbasic):
            out.append((k, int(nonbasic[0]), 0.5))
        slacks = np.flatnonzero(res.row_status[k] == 1)
        if len(slacks):
            out.append((k, n + int(slacks[-1]), 0.25))
    return out


def _check_against_restatement(lp, A, b, m_base, lb, ub, masks, res, reqs, int_mask):
    slots, vars_, f0 = (np.array(v) for v in zip(*reqs))
    pi, pi0, code = lp.simplex_gmi_cuts(slots, vars_, f0, int_mask)
    n, m = A.shape[1], A.shape[0]
    assert pi.shape == (len(reqs), n)
    for t, (s, v, f) in enumerate(reqs):
        status = np.concatenate([res.col_status[s], res.row_status[s]])
        if status[v] == 1:
            row = -lp.simplex_tableau_rows(s, [v])[0][n:]
            node = SimpleNamespace(head=np.array([v]), Binv=row[None, :], col_status=res.col_status[s],
                                   row_status=res.row_status[s])
        else:
            node = SimpleNamespace(head=np.array([-1]), Binv=np.zeros((1, m)), col_status=res.col_status[s],
                                   row_status=res.row_status[s])
        on = np.ones(m, bool)
        if masks is not None:
            on[m_base:] = masks[s].astype(bool)
        want_pi, want_pi0, want_code = gmi_device.gmi_cut(node, A, b, m_base, lb[s], ub[s], on, v, f, int_mask)
        assert code[t] == want_code, (t, s, v)
        assert np.array_equal(pi[t], want_pi), (t, s, v, np.max(np.abs(pi[t] - want_pi)))
        assert pi0[t] == want_pi0, (t, s, v)
    return code


def test_one_cta_batch_with_pool_rows_masked_per_node(blp_lib):
    d = grumpy_random_mip(40, 30, density=0.2, rand_seed=5)
    n = len(d.c)
    lp = engine.BatchLP(d.A, d.b, d.c)
    root = lp.simplex_batch(d.l[None], d.u[None])
    x = root.x[0]
    rng = np.random.default_rng(0)
    rows = -rng.integers(0, 4, size=(3, n)).astype(float)
    lp.append_rows(rows, rows @ x - 1.0)                 # loose rows, switched on per node
    A = np.vstack([d.A.toarray(), rows])
    b = np.concatenate([d.b, rows @ x - 1.0])
    ints = np.asarray(d.integer_indices)
    frac = np.abs(x[ints] - np.round(x[ints]))
    branch = ints[np.argsort(-frac, kind='stable')][:6]
    B = 12
    lb, ub = np.tile(d.l, (B, 1)), np.tile(d.u, (B, 1))
    for k in range(B):                                   # branching bounds: down (at upper) and up (at lower)
        j = branch[k % len(branch)]
        if k % 2:
            lb[k, j] = np.ceil(x[j])
        else:
            ub[k, j] = np.floor(x[j])
    masks = (rng.random((B, 3)) < 0.6).astype(np.uint8)
    res = lp.simplex_batch(lb, ub, row_mask=masks)
    int_mask = np.zeros(n, np.uint8)
    int_mask[ints] = 1
    reqs = _requests(d, res, per_slot=8)
    code = _check_against_restatement(lp, A, b, d.A.shape[0], lb, ub, masks, res, reqs, int_mask)
    assert (code == gmi_device.GMI_OK).sum() >= B and (code == gmi_device.GMI_NOT_BASIC).any()
    assert (res.col_status == 2).any()                   # some nonbasics sit at an upper bound
    lp.close()


def test_grouped_wide_batch(blp_lib):
    d = grumpy_random_mip(500, 1100, density=0.02, maxObjCoeff=10, maxConsCoeff=10, tightness=2, rand_seed=7)
    n = len(d.c)
    lp = engine.BatchLP(d.A, d.b, d.c)
    assert not lp.simplex_batched
    root = lp.simplex_batch(d.l[None], d.u[None])
    x = root.x[0]
    ints = np.asarray(d.integer_indices)
    j = int(ints[np.argmax(np.abs(x[ints] - np.round(x[ints])))])
    B = 3
    lb, ub = np.tile(d.l, (B, 1)), np.tile(d.u, (B, 1))
    ub[1, j] = np.floor(x[j])
    lb[2, j] = np.ceil(x[j])
    res = lp.simplex_batch(lb, ub)
    int_mask = np.ones(n, np.uint8)
    reqs = _requests(d, res, per_slot=6)
    code = _check_against_restatement(lp, d.A.toarray(), d.b, d.A.shape[0], lb, ub, None, res, reqs, int_mask)
    assert (code == gmi_device.GMI_OK).sum() >= 3
    lp.close()


def test_bad_requests_are_refused(blp_lib):
    d = grumpy_random_mip(20, 10, density=0.3, rand_seed=3)
    n, m = len(d.c), d.A.shape[0]
    lp = engine.BatchLP(d.A, d.b, d.c)
    ones = np.ones(n, np.uint8)
    with pytest.raises(engine.BlpError, match=r'\(-4\)'):            # no simplex call yet
        lp.simplex_gmi_cuts([0], [0], [0.5], ones)
    lp.simplex_batch(np.tile(d.l, (2, 1)), np.tile(d.u, (2, 1)))
    with pytest.raises(engine.BlpError, match=r'\(-4\)'):
        lp.simplex_gmi_cuts([2], [0], [0.5], ones)
    with pytest.raises(engine.BlpError, match=r'\(-4\)'):
        lp.simplex_gmi_cuts([-1], [0], [0.5], ones)
    with pytest.raises(engine.BlpError, match=r'\(-1\)'):
        lp.simplex_gmi_cuts([0], [n + m], [0.5], ones)
    with pytest.raises(engine.BlpError, match=r'\(-1\)'):
        lp.simplex_gmi_cuts([0], [0], [1.0], ones)
    lp.append_rows(np.ones((1, n)), [0.0])                # the rows changed: the store is void
    with pytest.raises(engine.BlpError, match=r'\(-4\)'):
        lp.simplex_gmi_cuts([0], [0], [0.5], ones)
    lp.close()


@pytest.mark.parametrize('name', ['cut1', 'cut2', 'cut3', 'square', 'small_branch', 'random'])
def test_device_cuts_are_valid_at_integer_points(blp_lib, name):
    import itertools
    rec = EXAMPLES[name]
    A, b = np.array(rec['A']), np.array(rec['b'])
    bb = BranchAndBound(model_from(rec), BaseNode, node_limit=12, gomory_cuts=False)
    bb.solve()
    checked = separated = 0
    for vert in bb.tree.nodes.values():
        node = vert.attr['node']
        if not node.lp_feasible or node.mip_feasible or node.solution is None:
            continue
        solve_lps([node.lp], force=True)
        cuts = node._device_gomory_cuts()
        assert cuts is not None
        host = {k: numerically_safe_cut(pi, pi0, estimate='over') for k, (pi, pi0) in node._find_gomory_cuts().items()}
        assert list(host) == list(cuts)
        for k, (pi, pi0) in cuts.items():
            # cuts off the LP vertex wherever the host path's rounded cut does (rounding towards safety can
            # weaken a cut until it no longer does, on either path)
            if float(np.dot(host[k][0], node.solution)) < host[k][1] - 1e-9:
                assert float(np.dot(pi, node.solution)) < pi0 - 1e-9, (name, node.idx, k)
                separated += 1
        lo = np.asarray(node.lp.variablesLower)
        hi = np.minimum(np.asarray(node.lp.variablesUpper), lo + 12)
        pts = []
        if len(rec['c']) <= 3:
            for p in itertools.product(*[range(int(np.ceil(a)), int(c) + 1) for a, c in zip(lo, hi)]):
                p = np.array(p, dtype=float)
                if (A @ p >= b - 1e-9).all():
                    pts.append(p)
        for pi, pi0 in cuts.values():
            for p in pts:
                assert float(np.dot(pi, p)) >= pi0 - 1e-7, (name, node.idx, p)
            checked += 1
    assert checked > 0 and separated > 0
    bb.model.lp._shared.close()


def test_device_gomory_branch_and_bound_matches_goldens(blp_lib, monkeypatch):
    calls = []
    original = engine.BatchLP.simplex_gmi_cuts

    def counted(self, slots, variables, f0, int_mask):
        calls.append(len(variables))
        return original(self, slots, variables, f0, int_mask)

    monkeypatch.setattr(engine.BatchLP, 'simplex_gmi_cuts', counted)
    for name, rec in list(SCALE1.items()) + [(k, EXAMPLES[k]) for k in ('small_branch', 'cut1', 'cut2', 'cut3', 'square')]:
        gold = rec['reference']['BaseNode_gomory']
        bb = BranchAndBound(model_from(rec), BaseNode, device_gomory=True)
        bb.solve()
        assert bb.status == gold['status'] == 'optimal', name
        want = float(gold['objective'])
        assert abs(bb.objective_value - want) <= 1e-6 * max(1.0, abs(want)), (name, bb.objective_value, want)
        bb.model.lp._shared.close()
    assert len(calls) > 0 and max(calls) > 1              # several cuts in one call


def test_frontier_cut_rounds_match_the_goldens(blp_lib):
    """BranchAndBound(frontier_cut_rounds=True) with the default Gomory options: status and optimum are the
    reference's, the real nodes find their rounds in the memo, and a node costs fewer engine calls than with the
    option off."""
    hits = calls_on = calls_off = nodes_on = nodes_off = 0
    for name, rec in list(SCALE1.items()) + [(k, EXAMPLES[k]) for k in ('small_branch', 'cut1', 'cut2', 'cut3', 'square')]:
        gold = rec['reference']['BaseNode_gomory']
        want = float(gold['objective'])
        for on in (False, True):
            bb = BranchAndBound(model_from(rec), BaseNode, frontier_cut_rounds=on)
            bb.solve()
            assert bb.status == gold['status'] == 'optimal', (name, on)
            assert abs(bb.objective_value - want) <= 1e-6 * max(1.0, abs(want)), (name, on, bb.objective_value, want)
            sh = bb.model.lp._shared
            if on:
                hits += bb.memo_hits
                calls_on += sh.solve_calls
                nodes_on += bb.evaluated_nodes
            else:
                calls_off += sh.solve_calls
                nodes_off += bb.evaluated_nodes
            sh.close()
    print(f'memo hits {hits}; LP calls per evaluated node: off {calls_off / nodes_off:.2f}, on {calls_on / nodes_on:.2f}')
    assert hits > 0 and calls_on / nodes_on < calls_off / nodes_off
