"""Device GMI cuts (blp_simplex_gmi_cuts_host, BaseNode(device_gomory=True)) on the CPU: the numpy restatement of
the kernel (oracle/gmi_device.py) against the reference's rounding, and the Node layer's device path on a stand-in
engine that answers simplex_gmi_cuts with that restatement."""
import numpy as np
import pytest

import simple_mip_solver_b200.engine as engine
from helpers import OracleBatchLP, use_oracle_engine
from oracle import gmi_device
from simple_mip_solver_b200 import BaseNode, BranchAndBound, CyLPArray
from simple_mip_solver_b200.compat import solve_lps
from simple_mip_solver_b200.utils.floating_point import numerically_safe_cut
from test_gomory import EXAMPLES, SCALE1, integer_points, model_from


class GmiOracleBatchLP(OracleBatchLP):
    """OracleBatchLP plus simplex_gmi_cuts: the restatement on the stored oracle factors, with the bounds and
    row masks of the call that stored them (as the device keeps them with its store)."""
    gmi_calls = 0
    gmi_cuts = 0

    def _simplex(self, lbs, ubs, masks, css, rss, parents, max_pivots):
        res = super()._simplex(lbs, ubs, masks, css, rss, parents, max_pivots)
        self._bounds = (np.array(lbs, float), np.array(ubs, float), None if masks is None else np.array(masks))
        return res

    def simplex_gmi_cuts(self, slots, variables, f0, int_mask):
        type(self).gmi_calls += 1
        type(self).gmi_cuts += len(variables)
        A, b = self._full()
        lbs, ubs, masks = self._bounds
        pis, pi0s, codes = [], [], []
        for s, v, f in zip(slots, variables, f0):
            on = np.ones(A.shape[0], bool)
            if masks is not None:
                on[self.m_base:] = np.asarray(masks[s], bool)
            pi, pi0, code = gmi_device.gmi_cut(self._store[s], A, b, self.m_base, lbs[s], ubs[s], on, int(v),
                                               float(f), int_mask)
            pis.append(pi)
            pi0s.append(pi0)
            codes.append(code)
        return np.array(pis), np.array(pi0s), np.array(codes, np.int32)


@pytest.fixture
def gmi_engine(monkeypatch):
    use_oracle_engine(monkeypatch)
    GmiOracleBatchLP.gmi_calls = GmiOracleBatchLP.gmi_cuts = 0
    monkeypatch.setattr(engine, 'BatchLP', GmiOracleBatchLP)
    return GmiOracleBatchLP


def bits(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64)).view(np.int64)


def reference_rounding(pi, pi0):
    safe, safe0 = numerically_safe_cut(CyLPArray(pi), float(pi0), estimate='over')
    return np.asarray(safe, dtype=np.float64), float(safe0)


EDGE_CUTS = [
    ([0.0, 0.0, 0.0], 1.5),                              # zero cut: returned unchanged
    ([0.0, -0.0, 2.0], 0.0),
    ([1.0, -1.0, 0.5], -3.25),                           # exact fractions, negatives
    ([3.0, 1.0, 1.0 / 3.0], 1.0),                        # 1/9 after scaling: exact-fraction fallback
    ([1.0, 1e-5, -1e-5], 0.1),                           # tiny coefficients: one-sided convergent is poor
    ([1.0, 0.3333333333333333, 0.6666666666666666], 0.7),
    ([1e-3, 2e-3, 1.0], 2500.0),                         # |pi0| > max_term after scaling
    ([1.0, 0.999999, 1e-3 + 1e-12], -2500.5),
    ([7.0, 3.0, np.pi], np.e),
    ([-1.0, 0.123456789, 0.000999], 1e-9),
]


def test_restated_rounding_is_the_reference_rounding_bit_for_bit():
    rng = np.random.default_rng(3)
    cases = list(EDGE_CUTS)
    for _ in range(300):
        k = int(rng.integers(1, 12))
        pi = rng.normal(size=k) * 10.0 ** rng.integers(-4, 4, size=k)
        pi[rng.random(k) < 0.2] = 0.0
        if rng.random() < 0.3:
            pi = np.round(pi * 8) / 8                     # exact binary fractions
        cases.append((pi, float(rng.normal() * 10.0 ** rng.integers(-3, 5))))
    for pi, pi0 in cases:
        want, want0 = reference_rounding(np.asarray(pi, float), pi0)
        got, got0, code = gmi_device.safe_cut(np.asarray(pi, float), pi0)
        assert np.array_equal(bits(got), bits(want)), (pi, pi0, got, want)
        assert bits([got0])[0] == bits([want0])[0], (pi, pi0, got0, want0)
        assert code == (gmi_device.GMI_ZERO if not np.any(pi) else gmi_device.GMI_OK)


def test_option_off_never_asks_the_device(gmi_engine):
    bb = BranchAndBound(model_from(EXAMPLES['cut2']), BaseNode)
    bb.solve()
    assert bb.status == 'optimal'
    assert gmi_engine.gmi_calls == 0


@pytest.mark.parametrize('name', ['cut1', 'cut2', 'cut3', 'square', 'small_branch', 'random'])
def test_device_cuts_are_valid_and_match_the_host_path(gmi_engine, name):
    """Below branching bounds, every cut of the device path keeps every integer point of its node, is the host
    path's rounded cut up to round-off, and cuts off the node's LP vertex wherever that one does (rounding
    towards safety can weaken a cut until it no longer does, on either path)."""
    rec = EXAMPLES[name]
    bb = BranchAndBound(model_from(rec), BaseNode, node_limit=12, gomory_cuts=False)
    bb.solve()
    checked = 0
    for vert in bb.tree.nodes.values():
        node = vert.attr['node']
        if not node.lp_feasible or node.mip_feasible or node.solution is None:
            continue
        solve_lps([node.lp], force=True)             # its factor back in the store
        cuts = node._device_gomory_cuts()
        host = {k: reference_rounding(pi, pi0) for k, (pi, pi0) in node._find_gomory_cuts().items()}
        assert cuts is not None and list(cuts) == list(host)
        lo = np.asarray(node.lp.variablesLower)
        hi = np.minimum(np.asarray(node.lp.variablesUpper), lo + 12)
        pts = list(integer_points(rec, lo, hi)) if len(rec['c']) <= 3 else []
        for k, (pi, pi0) in cuts.items():
            assert np.allclose(pi, host[k][0], rtol=0, atol=1e-9) and abs(pi0 - host[k][1]) <= 1e-9
            if float(np.dot(host[k][0], node.solution)) < host[k][1] - 1e-9:
                assert float(np.dot(pi, node.solution)) < pi0 - 1e-9
            for p in pts:
                assert float(np.dot(pi, p)) >= pi0 - 1e-7, (name, node.idx, p)
            checked += 1
    assert checked > 0 and gmi_engine.gmi_calls > 0


def test_device_path_falls_back_when_the_factor_is_gone(gmi_engine):
    m = model_from(EXAMPLES['cut2'])
    node = BaseNode(m.lp, m.integerIndices, idx=0)
    node._bound_lp()
    assert node.lp.has_stored_factor
    other = m.lp.copy_for_child()
    other.variablesUpper[0] = 1.0
    solve_lps([other])                               # replaces the store
    assert not node.lp.has_stored_factor and node._device_gomory_cuts() is None
    host = node._generate_cuts()
    again = node._generate_cuts(device_gomory=True)
    assert gmi_engine.gmi_calls == 0
    assert list(host) == list(again)
    for name in host:
        assert np.array_equal(host[name][0], again[name][0]) and host[name][1] == again[name][1]


def test_device_gomory_bound_reaches_the_golden_optimum(gmi_engine):
    """BranchAndBound(BaseNode, device_gomory=True) with the default cut rounds: status and optimum are the
    reference's (BaseNode_gomory goldens) on the scale_1 fixtures and the example models."""
    cases = list(SCALE1.items()) + [(k, EXAMPLES[k]) for k in ('small_branch', 'cut1', 'cut2', 'cut3', 'square')]
    for name, rec in cases:
        gold = rec['reference']['BaseNode_gomory']
        bb = BranchAndBound(model_from(rec), BaseNode, device_gomory=True)
        bb.solve()
        assert bb.status == gold['status'], name
        assert abs(bb.objective_value - float(gold['objective'])) <= 1e-6 * max(1.0, abs(float(gold['objective']))), name
    assert gmi_engine.gmi_calls > 0
