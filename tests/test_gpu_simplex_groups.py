"""GPU: batches of mid-size LPs (1025-8192 rows) on the grouped grid kernel. k_simplex_wide splits one cooperative
launch into G groups of S CTAs, group g solving nodes g, g + G, ... with its own barrier. Every node must match the
numpy restatement (oracle/dual_simplex.py) bit for bit, whatever G is.

A library built with -DBLP_TUNING reads BLP_SX_GROUPS to force G; those cases run in a subprocess that loads such a
library (see test_gpu_simplex_paths._run_with_knobs). The production library picks G from m, B and the SM count.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle.dual_simplex import BASIC, dual_simplex
from simple_mip_solver_b200.instances import grumpy_random_mip
from test_gpu_simplex import _children, same

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UNLIMITED = 2147483647
FORCED_GROUPS = (1, 2, 3, 7, 16)


def _lp_1100():
    return grumpy_random_mip(500, 1100, density=0.02, maxObjCoeff=10, maxConsCoeff=10, tightness=2, rand_seed=7)


def _mixed_batch(d, ref_root, B):
    """Node 0 the root from the slack basis, then children of the root alternately from its basis status and
    from its stored factor (slot 0 of the previous call)."""
    deltas = [[]] + _children(d, ref_root.x, B)[:B - 1]
    lb, ub = np.tile(d.l, (B, 1)), np.tile(d.u, (B, 1))
    for k, dl in enumerate(deltas):
        for j, lo, hi in dl:
            lb[k, j], ub[k, j] = lo, hi
    cs = np.tile(ref_root.col_status, (B, 1))
    rs = np.tile(ref_root.row_status, (B, 1))
    cs[0] = 3
    rs[0] = BASIC
    parent = np.array([-1] + [(k % 2) - 1 for k in range(1, B)], np.int32)      # -1 status, 0 stored factor
    return lb, ub, cs, rs, parent


def _mixed_refs(d, ref_root, batch, limit, **kw):
    A = d.A.toarray()
    lb, ub, cs, rs, parent = batch
    return [dual_simplex(A, d.b, d.c, lb[k], ub[k], col_status=cs[k], row_status=rs[k], max_pivots=limit,
                         start=ref_root if parent[k] >= 0 else None, **kw) for k in range(len(lb))]


def _run_batch(lp, d, batch, limit):
    lb, ub, cs, rs, parent = batch
    lp.simplex_batch(d.l[None], d.u[None])                                 # the root is the stored call
    return lp.simplex_batch(lb, ub, col_status=cs, row_status=rs, parent_slot=parent, max_pivots=limit)


# ---- cases run on a tuning library (in a subprocess) -------------------------------------------------------
def _forced_groups_cases():
    """The 1100 x 500 LP in batches of 9 and 16, 5 pivots and unlimited, under every G of FORCED_GROUPS;
    then per-node pool-row masks with a stored factor continued or refactorised."""
    from simple_mip_solver_b200 import engine
    d = _lp_1100()
    A = d.A.toarray()
    ref_root = dual_simplex(A, d.b, d.c, d.l, d.u)
    lp = engine.BatchLP(d.A, d.b, d.c)
    assert not lp.simplex_batched
    batch = _mixed_batch(d, ref_root, 16)
    for limit in (5, UNLIMITED):
        refs = _mixed_refs(d, ref_root, batch, limit)
        for B in (9, 16):
            sub = tuple(a[:B] for a in batch)
            for G in FORCED_GROUPS:
                os.environ['BLP_SX_GROUPS'] = str(G)
                res = _run_batch(lp, d, sub, limit)
                for k in range(B):
                    same(res, k, refs[k], ('1100 x 500', limit, B, G, k))
    lp.close()
    # pool rows switched off per node: row 1 is slack basic in the parent (its factor is continued), row 0 is
    # tight there (the kernel factorises the parent's status again)
    d = grumpy_random_mip(48, 1025, density=0.15, rand_seed=1025)
    A = d.A.toarray()
    x0 = dual_simplex(A, d.b, d.c, d.l, d.u).x
    S = np.argsort(-(x0 - np.floor(x0)))[:6]
    cuts = np.zeros((2, d.n))
    cuts[0, S] = -1.0
    cuts[1, :] = -1.0
    rhs = np.array([-np.floor(x0[S].sum() - 1e-9), -10.0 * (x0.sum() + 1.0)])
    Afull, bfull = np.vstack([A, cuts]), np.concatenate([d.b, rhs])
    ref_parent = dual_simplex(Afull, bfull, d.c, d.l, d.u)
    assert ref_parent.row_status[d.m] != BASIC and ref_parent.row_status[d.m + 1] == BASIC
    lp = engine.BatchLP(d.A, d.b, d.c)
    lp.append_rows(cuts, rhs)
    deltas = _children(d, ref_parent.x, 4)
    B = len(deltas)
    masks = np.array([[1, 1], [1, 0], [0, 1], [0, 0]] * 2, np.uint8)[:B]
    lb, ub = np.tile(d.l, (B, 1)), np.tile(d.u, (B, 1))
    for k, dl in enumerate(deltas):
        for j, lo, hi in dl:
            lb[k, j], ub[k, j] = lo, hi
    cs, rs = np.tile(ref_parent.col_status, (B, 1)), np.tile(ref_parent.row_status, (B, 1))
    for G in (3, 7):
        os.environ['BLP_SX_GROUPS'] = str(G)
        lp.simplex_batch(d.l[None], d.u[None], row_mask=np.ones((1, 2), np.uint8))
        res = lp.simplex_batch(lb, ub, row_mask=masks, col_status=cs, row_status=rs,
                               parent_slot=np.zeros(B, np.int32))
        for k in range(B):
            on = np.concatenate([np.ones(d.m, bool), masks[k].astype(bool)])
            ref = dual_simplex(Afull, bfull, d.c, lb[k], ub[k], row_on=on, col_status=cs[k], row_status=rs[k],
                               start=ref_parent)
            same(res, k, ref, ('masked', G, k))
    lp.close()
    return len(FORCED_GROUPS)


def _refused_pivot_groups_case():
    """Every pivot that does not follow a factorisation refused (BLP_SX_MISMATCH=-1), 3 groups: a refused pivot
    costs each node a refactorisation with its own number of barriers, which must not desynchronise a group."""
    from simple_mip_solver_b200 import engine
    d = grumpy_random_mip(48, 1025, density=0.15, rand_seed=1025)
    A = d.A.toarray()
    kw = dict(pivot_mismatch=float(os.environ['BLP_SX_MISMATCH']))
    ref_root = dual_simplex(A, d.b, d.c, d.l, d.u, **kw)
    assert ref_root.refused > 0
    lp = engine.BatchLP(d.A, d.b, d.c)
    batch = _mixed_batch(d, ref_root, 9)
    refused = 0
    for limit in (5, UNLIMITED):
        refs = _mixed_refs(d, ref_root, batch, limit, **kw)
        lp.simplex_batch(d.l[None], d.u[None])
        lb, ub, cs, rs, parent = batch
        res = lp.simplex_batch(lb, ub, col_status=cs, row_status=rs, parent_slot=parent, max_pivots=limit)
        for k, ref in enumerate(refs):
            same(res, k, ref, ('refused', limit, k))
            refused += ref.refused
    lp.close()
    return refused


@pytest.fixture(scope='module')
def tuning_lib(blp_lib, tmp_path_factory):
    from simple_mip_solver_b200 import _build
    return _build.build_extension(tuning=True, out=tmp_path_factory.mktemp('tuning') / 'libblp_tuning.so')


def _run_with_knobs(tuning_lib, cases, **knobs):
    code = ("import sys, json; sys.path[:0] = [%r, %r]\n"
            "import test_gpu_simplex_groups as t\n"
            "print(json.dumps(t.%s()))\n") % (ROOT, os.path.join(ROOT, 'tests'), cases)
    env = dict(os.environ, BLP_LIB=str(tuning_lib), **knobs)
    res = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, env=env, timeout=1800)
    assert res.returncode == 0, res.stdout[-1000:] + res.stderr[-4000:]
    return json.loads(res.stdout.strip().splitlines()[-1])


def test_forced_group_counts_bit_identical(tuning_lib):
    """G = 1, 2, 3, 7, 16 (3 and 7 divide neither the SM count nor the batch): every node of batches of 9 and 16
    mid-size LPs, and of a batch with per-node pool-row masks, is the restatement's to the bit."""
    _run_with_knobs(tuning_lib, '_forced_groups_cases')


def test_refused_pivots_keep_groups_in_step(tuning_lib):
    refused = _run_with_knobs(tuning_lib, '_refused_pivot_groups_case', BLP_SX_MISMATCH='-1', BLP_SX_GROUPS='3')
    assert refused > 0


# ---- production library (G chosen by the library) ----------------------------------------------------------
@pytest.mark.parametrize('m', [1025, 2048])
def test_automatic_groups_bit_identical(blp_lib, m):
    """Batches of 1, 5 and 16 LPs with 48 columns: every node is the restatement's, and the tableau rows of a
    node other than the first equal inv(B) [A, -I]."""
    from simple_mip_solver_b200 import engine
    d = grumpy_random_mip(48, m, density=0.15, rand_seed=m)
    A = d.A.toarray()
    ref_root = dual_simplex(A, d.b, d.c, d.l, d.u)
    lp = engine.BatchLP(d.A, d.b, d.c)
    assert not lp.simplex_batched
    for B in (1, 5, 16):
        batch = _mixed_batch(d, ref_root, B)
        refs = _mixed_refs(d, ref_root, batch, UNLIMITED)
        res = _run_batch(lp, d, batch, UNLIMITED)
        for k in range(B):
            same(res, k, refs[k], (m, B, k))
    slot = 3
    basic = np.flatnonzero(np.concatenate([res.col_status[slot], res.row_status[slot]]) == BASIC)
    rows = lp.simplex_tableau_rows(slot, basic)
    full = np.concatenate([A, -np.eye(m)], axis=1)
    want = np.linalg.solve(full[:, basic], full)
    assert np.allclose(rows, want, rtol=1e-9, atol=1e-9), np.abs(rows - want).max()
    lp.close()


def test_automatic_groups_on_the_1100_row_lp(blp_lib):
    from simple_mip_solver_b200 import engine
    d = _lp_1100()
    ref_root = dual_simplex(d.A.toarray(), d.b, d.c, d.l, d.u)
    lp = engine.BatchLP(d.A, d.b, d.c)
    batch = _mixed_batch(d, ref_root, 12)
    refs = _mixed_refs(d, ref_root, batch, 5)
    res = _run_batch(lp, d, batch, 5)
    for k in range(12):
        same(res, k, refs[k], ('1100 x 500 auto', k))
    lp.close()


def test_node_api_strong_branching_on_a_mid_size_model(blp_lib, monkeypatch):
    """SharedLP.default_method = 'simplex' on a 1100-row model: the root's strong-branching round (5 pivots per
    child from the root's basis) goes to the grouped kernel as one batch, and its pseudo costs are the
    restatement's exactly."""
    from simple_mip_solver_b200 import CyLPArray, MILPInstance, PseudoCostBranchNode
    from simple_mip_solver_b200.compat.cylp_like import SharedLP
    monkeypatch.setattr(SharedLP, 'default_method', 'simplex')
    d = grumpy_random_mip(48, 1100, density=0.15, rand_seed=11)
    model = MILPInstance(A=d.A.toarray(), b=CyLPArray(d.b), c=CyLPArray(d.c), l=CyLPArray(d.l), u=CyLPArray(d.u),
                         sense=['Min', '>='], integerIndices=d.integer_indices, numVars=d.n)
    node = PseudoCostBranchNode(model.lp, model.integerIndices, idx=0)
    rtn = node.bound(pseudo_costs={}, gomory_cuts=False)
    pcs = rtn['pseudo_costs']
    sh = model.lp._shared
    assert len(pcs) >= 4 and sh.lps_solved >= 1 + 2 * len(pcs)
    A = d.A.toarray()
    cols, rows = model.lp.getBasisStatus()
    cols, rows = np.array(cols, np.int8), np.array(rows, np.int8)
    x, root_obj = np.asarray(node.solution), node.objective_value
    for j in pcs:
        for direction in ('left', 'right'):
            l, u = d.l.copy(), d.u.copy()
            if direction == 'left':
                u[j] = np.floor(x[j]); change = x[j] - u[j]
            else:
                l[j] = np.ceil(x[j]); change = l[j] - x[j]
            r = dual_simplex(A, d.b, d.c, l, u, col_status=cols, row_status=rows, max_pivots=5)
            cost = max(r.objective - root_obj, 0) / change if r.status in (0, 3) else 0.0
            assert pcs[j][direction]['cost'] == cost, (j, direction)
