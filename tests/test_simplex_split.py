"""CPU: with method='simplex', a batch of node LPs whose dense basis inverses exceed SIMPLEX_MEMORY_BUDGET is sent
as consecutive simplex calls of at most as many LPs as the budget holds, and every LP ends exactly where the
unsplit call leaves it. The engine is the numpy restatement of the device kernels (tests/helpers.OracleBatchLP)."""
import numpy as np
import pytest

from helpers import use_oracle_engine
from simple_mip_solver_b200 import CyLPArray, MILPInstance, PseudoCostBranchNode
from simple_mip_solver_b200.compat import cylp_like
from simple_mip_solver_b200.instances import grumpy_random_mip


def _strong_branching_round(iterations):
    d = grumpy_random_mip(40, 20, density=0.2, rand_seed=3)
    model = MILPInstance(A=d.A.toarray(), b=CyLPArray(d.b), c=CyLPArray(d.c), l=CyLPArray(d.l), u=CyLPArray(d.u),
                         sense=['Min', '>='], integerIndices=d.integer_indices, numVars=d.n)
    node = PseudoCostBranchNode(model.lp, model.integerIndices, idx=0)
    node._bound_lp()
    x = np.asarray(node.solution)
    frac = [j for j in d.integer_indices if node._is_fractional(float(x[j]))]
    assert len(frac) >= 4
    kids = node._strong_branch_batch(frac, iterations)
    out = []
    for j in frac:
        for direction in ('left', 'right'):
            lp = kids[j][direction].lp
            cols, rows = lp.getBasisStatus()
            out.append((lp.getStatusCode(), lp.objectiveValue, np.array(lp.primalVariableSolution['x']), np.array(cols), np.array(rows)))
    return out, d.m


@pytest.mark.parametrize('iterations', [5, 2147483647])
def test_oversized_simplex_batch_is_split_into_calls(monkeypatch, iterations):
    eng = use_oracle_engine(monkeypatch, 'simplex')
    whole, m = _strong_branching_round(iterations)
    assert eng.batch_sizes[-1] == len(whole)
    per_call = 3
    monkeypatch.setattr(cylp_like, 'SIMPLEX_MEMORY_BUDGET', per_call * m * m * 8 + 7)
    eng = use_oracle_engine(monkeypatch, 'simplex')
    split, _ = _strong_branching_round(iterations)
    calls = -(-len(split) // per_call)
    assert eng.batch_sizes[1:] == [per_call] * (calls - 1) + [len(split) - per_call * (calls - 1)]
    assert len(split) == len(whole)
    for k, (a, b) in enumerate(zip(whole, split)):
        assert a[0] == b[0], k
        if a[0] != 1:
            assert a[1] == b[1], k
            assert np.array_equal(a[2], b[2]), k
        assert np.array_equal(a[3], b[3]) and np.array_equal(a[4], b[4]), k
