"""GPU: the BASELINE.json configurations 3 and 4 at reduced or full size, through the Node API.

config 3: synthetic random MILP 500 vars x 300 rows, 10 % density; strong branching on up to 64
          candidates x 2 children handed to the kernels as ONE batch by PseudoCostBranchNode.
config 4: sparse MILP with a cutting-plane bound: cut rows appended per node batch (shared pool,
          per-node row masks), three rounds; here 2000 x 1000 so that the CPU oracle stays fast.
"""
import numpy as np
import pytest
import scipy.sparse as sp

from oracle.highs_lp import HIGHS_INF, HighsLP
from simple_mip_solver_b200 import CyLPArray, MILPInstance, PseudoCostBranchNode
from simple_mip_solver_b200.instances import frontier_nodes, grumpy_random_mip, numpy_random_mip

pytestmark = pytest.mark.gpu


def rel(a, b):
    return abs(a - b) / max(1.0, abs(b))


def test_config3_strong_branching_batch(blp_lib):
    d = grumpy_random_mip(500, 300, density=0.1, maxObjCoeff=10, maxConsCoeff=10, tightness=2, rand_seed=2)
    model = MILPInstance(A=d.A.toarray(), b=CyLPArray(d.b), c=CyLPArray(d.c), l=CyLPArray(d.l), u=CyLPArray(d.u),
                         sense=['Min', '>='], integerIndices=d.integer_indices, numVars=d.n)
    node = PseudoCostBranchNode(model.lp, model.integerIndices, idx=0)
    # 100 "pivots" = 51 200 PDHG iterations: enough for every child to reach the 1e-8 tolerance
    rtn = node.bound(pseudo_costs={}, strong_branch_iters=100, gomory_cuts=False)
    ref_root = HighsLP(d.A, d.c, d.b, np.full(d.m, HIGHS_INF), d.l, d.u).solve()
    assert rel(node.objective_value, ref_root.objective) <= 1e-6
    pcs = rtn['pseudo_costs']
    sh = model.lp._shared
    assert sh.solve_calls == 2 and sh.lps_solved == 1 + 2 * len(pcs)      # root, then ALL children at once
    assert len(pcs) >= 32
    x = node.solution
    checked = 0
    for j, entry in list(pcs.items())[:24]:
        for direction in ('left', 'right'):
            l, u = d.l.copy(), d.u.copy()
            if direction == 'left':
                u[j] = np.floor(x[j])
                change = x[j] - u[j]
            else:
                l[j] = np.ceil(x[j])
                change = l[j] - x[j]
            ref = HighsLP(d.A, d.c, d.b, np.full(d.m, HIGHS_INF), l, u).solve()
            want = max(ref.objective - node.objective_value, 0) / change if ref.status == 0 else 0.0
            assert entry[direction]['times'] == 1
            # a pseudo cost is a difference quotient of two objectives that are each right to 1e-6
            # relative: the admissible error is 2e-6 |obj| / (change of the variable)
            assert entry[direction]['cost'] == pytest.approx(want, rel=1e-3, abs=2e-6 * abs(ref_root.objective) / change)
            checked += 1
    assert checked == 48
    # the branching decision the reference would take from these costs (pseudo_cost.py:118-133)
    assert node._best_pseudo_costs_index(pcs) in pcs


def test_config4_cut_rounds_with_row_masks(blp_lib):
    from simple_mip_solver_b200 import engine
    d = numpy_random_mip(2000, 1000, density=0.01, seed=2)
    root = HighsLP(d.A, d.c, d.b, np.full(d.m, HIGHS_INF), d.l, d.u).solve()
    B = 32
    lbs, ubs, _ = frontier_nodes(d, root.x, 0, B, 8, seed=3)
    lp = engine.BatchLP(d.A, d.b, d.c)
    rng = np.random.default_rng(5)
    cuts, rhs = [], []
    masks = np.zeros((B, 0), dtype=np.uint8)
    res = lp.solve_batch(lbs, ubs, x0=np.tile(root.x, (B, 1)), y0=np.tile(np.maximum(root.row_dual, 0), (B, 1)))
    prev = res.objective.copy()
    for rnd in range(3):
        # each round appends 8 dense knapsack-cover style rows  -sum_{j in S} x_j >= -floor(sum x*_S)
        # built from one node's current solution; a row is switched on for a random half of the nodes
        new_rows, new_rhs = [], []
        for k in range(8):
            S = rng.choice(d.n, size=200, replace=False)
            xs = res.x[k % B]
            row = np.zeros(d.n)
            row[S] = -1.0
            new_rows.append(row)
            new_rhs.append(-np.floor(xs[S].sum()))
        first = lp.append_rows(np.array(new_rows), np.array(new_rhs))
        assert first == d.m + 8 * rnd
        cuts += new_rows
        rhs += new_rhs
        masks = np.hstack([masks, (rng.random((B, 8)) < 0.5).astype(np.uint8)])
        res = lp.solve_batch(lbs, ubs, row_mask=masks, x0=res.x,
                             y0=np.hstack([res.y, np.zeros((B, 8))]))
        for k in range(0, B, 5):
            h = HighsLP(d.A, d.c, d.b, np.full(d.m, HIGHS_INF), lbs[k], ubs[k])
            for t in np.flatnonzero(masks[k]):
                h.add_row(cuts[t], rhs[t])
            ref = h.solve()
            assert res.status[k] == ref.status, (rnd, k)
            if ref.status == 0:
                assert rel(res.objective[k], ref.objective) <= 1e-6, (rnd, k, res.objective[k], ref.objective)
                assert res.objective[k] >= prev[k] - 1e-6 * abs(prev[k])      # cuts only tighten
        ok = res.status == 0
        assert (res.y[ok][:, d.m:][masks[ok] == 0] == 0).all()                 # masked rows carry no dual
        prev = np.where(ok, res.objective, prev)
    lp.truncate_rows(d.m)
    assert lp.m == d.m
    lp.close()


def test_config3_default_five_pivot_strong_branching(blp_lib):
    """Config 3 with the reference's DEFAULT budget, strong_branch_iters=5 (pseudo_cost.py:22): on the
    dual simplex path that is literally 5 dual simplex pivots per child from the parent's basis, the
    objective of an unfinished child being the dual objective of its last basis (a valid lower bound,
    pseudo_cost.py:86-92). Checked against the numpy restatement pivot for pivot, and the branching
    variable the costs select (:118-133) against the one the restatement's costs select."""
    from oracle.dual_simplex import dual_simplex
    d = grumpy_random_mip(500, 300, density=0.1, maxObjCoeff=10, maxConsCoeff=10, tightness=2, rand_seed=2)
    model = MILPInstance(A=d.A.toarray(), b=CyLPArray(d.b), c=CyLPArray(d.c), l=CyLPArray(d.l), u=CyLPArray(d.u),
                         sense=['Min', '>='], integerIndices=d.integer_indices, numVars=d.n)
    node = PseudoCostBranchNode(model.lp, model.integerIndices, idx=0)
    rtn = node.bound(pseudo_costs={}, gomory_cuts=False)            # strong_branch_iters defaults to 5
    pcs = rtn['pseudo_costs']
    sh = model.lp._shared
    assert sh.solve_calls == 2 and sh.lps_solved == 1 + 2 * len(pcs) and len(pcs) >= 100
    A = d.A.toarray()
    root = dual_simplex(A, d.b, d.c, d.l, d.u)
    assert np.array_equal(np.asarray(node.solution), root.x) and node.objective_value == root.objective
    x = root.x
    want = {}
    limited = 0
    for j in pcs:
        want[j] = {}
        for direction in ('left', 'right'):
            l, u = d.l.copy(), d.u.copy()
            if direction == 'left':
                u[j] = np.floor(x[j]); change = x[j] - u[j]
            else:
                l[j] = np.ceil(x[j]); change = l[j] - x[j]
            r = dual_simplex(A, d.b, d.c, l, u, col_status=root.col_status, row_status=root.row_status, max_pivots=5)
            limited += r.status == 3
            cost = max(r.objective - root.objective, 0) / change if r.status in (0, 3) else 0.0
            want[j][direction] = cost
            assert pcs[j][direction]['cost'] == cost, (j, direction)          # exact: same pivots, same arithmetic
    assert limited > len(pcs)                    # most children do stop at the 5-pivot budget
    gold = {j: {dr: dict(cost=c, times=1) for dr, c in v.items()} for j, v in want.items()}
    assert node._best_pseudo_costs_index(pcs) == node._best_pseudo_costs_index(gold)
    # against HiGHS under the same 5-iteration limit: a different simplex takes different 5 pivots, so
    # the costs are not comparable one by one; report how the selected variable ranks there
    h = HighsLP(d.A, d.c, d.b, np.full(d.m, HIGHS_INF), d.l, d.u)
    hr = h.solve()
    hcost = {}
    for j in pcs:
        hcost[j] = {}
        for direction in ('left', 'right'):
            h.set_col_bounds(d.l, d.u)
            if direction == 'left':
                h.set_one_col_bound(j, d.l[j], np.floor(x[j])); change = x[j] - np.floor(x[j])
            else:
                h.set_one_col_bound(j, np.ceil(x[j]), d.u[j]); change = np.ceil(x[j]) - x[j]
            h.set_basis(hr.col_basis, hr.row_basis)
            r = h.solve(iteration_limit=5)
            hcost[j][direction] = dict(cost=max(r.objective - hr.objective, 0) / change if r.status in (0, 3) else 0.0, times=1)
    pick, hpick = node._best_pseudo_costs_index(pcs), node._best_pseudo_costs_index(hcost)

    def score(costs, j):
        return min(costs[j]['right']['cost'] * (np.ceil(x[j]) - x[j]), costs[j]['left']['cost'] * (x[j] - np.floor(x[j])))
    rank = sorted(hcost, key=lambda j: -score(hcost, j)).index(pick)
    print(f'5-pivot strong branching, {len(pcs)} candidates: device picks x{pick}, HiGHS-5-iteration costs pick x{hpick}; '
          f'the device pick ranks {rank + 1} of {len(pcs)} under the HiGHS costs')


def _write_mps(path, d):
    """Free-format MPS of ``min c.x, A x >= b, l <= x <= u`` with integer columns (what CLP writes)."""
    A = d.A.tocsc()
    with open(path, 'w') as f:
        f.write('NAME bench\nROWS\n N OBJ\n')
        for i in range(d.m):
            f.write(f' G R{i}\n')
        f.write('COLUMNS\n')
        for j in range(d.n):
            f.write(f' C{j} OBJ {d.c[j]:.17g}\n')
            for p in range(A.indptr[j], A.indptr[j + 1]):
                f.write(f' C{j} R{A.indices[p]} {A.data[p]:.17g}\n')
        f.write('RHS\n')
        for i in range(d.m):
            f.write(f' RHS R{i} {d.b[i]:.17g}\n')
        f.write('BOUNDS\n')
        for j in range(d.n):
            f.write(f' UI BND C{j} {d.u[j]:.17g}\n')
        f.write('ENDATA\n')


def test_config4_shape_through_the_node_api(blp_lib, tmp_path):
    """The Node API at the C4 shape (10 000 x 5 000), from an MPS file, in a fresh process so that its
    peak resident set is its own: BaseNode.bound() with the reference's default cut loop, and
    BranchAndBound(PseudoCostBranchNode) for a few nodes — the root's strong-branching round hands
    thousands of children to the GPU in one call. The model stays sparse on the host (no dense A, no
    dense [B, n] bound arrays): resident set under 2 GB."""
    import json
    import os
    import subprocess
    import sys
    d = numpy_random_mip(10000, 5000, density=2e-3, seed=2)
    path = str(tmp_path / 'c4.mps')
    _write_mps(path, d)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, 'tests', 'tools', 'c4_node_api.py'), path],
                         capture_output=True, text=True, timeout=1500, cwd=root)
    assert out.returncode == 0, out.stderr[-3000:]
    r = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith('{')][-1])
    print(r)
    gold = float(np.load(os.path.join(root, 'bench_data', 'c4_root.npz'))['objective'])
    assert r['sparse_model'] and r['n'] == 10000 and r['n_int'] == 10000
    assert r['bound_feasible'] and r['bound_objective'] >= gold - 1e-6 * abs(gold)      # cut rounds only raise it
    assert r['bb_status'] == 'stopped on iterations or time' and r['bb_nodes'] == 3
    assert rel(r['bb_root_objective'], gold) <= 1e-6
    assert r['bb_dual_bound'] >= gold - 1e-6 * abs(gold)
    assert r['pseudo_costs'] > 1000 and r['lps_solved'] > 2000
    assert r['peak_rss_gb'] < 2.0, r['peak_rss_gb']


def test_config4_shape_exact_vertex_and_gomory_round(blp_lib):
    """SURVEY 8f #1 at the C4 shape (10 000 x 5 000): a single node's LP goes to the wide dual simplex
    (the whole GPU on one node), so BaseNode gets an exact vertex and basis, GMI cuts are generated from
    tableau rows computed on the device, appended, and the LP is re-solved from the previous basis."""
    import os
    import time
    from simple_mip_solver_b200 import BaseNode
    d = numpy_random_mip(10000, 5000, density=2e-3, seed=2)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    gold = float(np.load(os.path.join(root, 'bench_data', 'c4_root.npz'))['objective'])
    model = MILPInstance(A=d.A, b=CyLPArray(d.b), c=CyLPArray(d.c), l=CyLPArray(d.l), u=CyLPArray(d.u),
                         sense=['Min', '>='], integerIndices=d.integer_indices, numVars=d.n)
    node = BaseNode(model.lp, model.integerIndices, idx=0)
    t = time.perf_counter()
    node._bound_lp()
    t_root = time.perf_counter() - t
    assert node.lp.has_exact_basis and rel(node.objective_value, gold) <= 1e-9
    cols, rows = node.lp.getBasisStatus()
    assert int((cols == 1).sum() + (rows == 1).sum()) == 5000                  # a basis: exactly m basics
    x = np.asarray(node.solution)
    assert (d.A @ x >= d.b - 1e-7).all() and (x >= d.l - 1e-9).all() and (x <= d.u + 1e-9).all()
    frac = np.minimum(x - np.floor(x), np.ceil(x) - x)
    n_frac = int((frac > 1e-4).sum())
    assert n_frac <= 5000                                                       # a vertex: at most m fractional
    before = node.objective_value
    t = time.perf_counter()
    node._cut_generation_iteration(max_gomory_cuts=16, track_dual_bound=False)
    t_round = time.perf_counter() - t
    assert node.number_gmic_created == 16 and node.number_gmic_added >= 1
    assert node.lp.nConstraints == 5000 + node.number_gmic_added
    assert node.objective_value >= before - 1e-9 * abs(before)
    x2 = np.asarray(node.solution)
    for name, (pi, pi0) in node.lp._cuts.items():
        assert float(np.dot(pi, x2)) >= pi0 - 1e-7 * max(1.0, abs(pi0)), name    # the new vertex satisfies the cuts
        assert float(np.dot(pi, x)) < pi0                                        # ... which cut off the old one
    print(f'C4 root by the wide dual simplex: {node.lp.iteration if False else ""} {t_root:.2f} s, {n_frac} fractional; one GMI round '
          f'(16 cuts created, {node.number_gmic_added} added): {t_round:.2f} s, bound {before:.6f} -> {node.objective_value:.6f}')
    model.lp._shared.close()
