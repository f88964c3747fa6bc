"""The numpy restatement of the device's dual simplex (oracle/dual_simplex.py) on the paths that small,
well-conditioned LPs with zero lower bounds never take, checked against HiGHS:

* a pivot refused because the two ways to the pivot element disagree (``pivot_mismatch=-1`` refuses every
  pivot that does not directly follow a factorisation; a natural mismatch needs cancellation in the inverse);
* the periodic refactorisation (``refactor_every`` of a few pivots instead of max(1000, 2 m));
* lower bounds other than zero: negative and positive finite ones, free columns, columns fixed at a nonzero
  value, columns with only an upper bound.

The restatement is what the CUDA kernels are compared with bit for bit (tests/test_gpu_simplex_paths.py), so a
wrong answer here is a wrong answer of the device.
"""
import numpy as np
import pytest

from oracle.dual_simplex import dual_simplex
from oracle.highs_lp import HIGHS_INF, HighsLP
from simple_mip_solver_b200.instances import grumpy_random_mip
from test_oracle_pins import _random_lp

UNB = 1e308                      # "no bound", as HighsLP and the restatement read it


def _random_bounded_lp(rng):
    """Like _random_lp, with every kind of column bound: boxed with a negative or positive lower bound,
    only a lower bound, only an upper bound, free, fixed at a nonzero value."""
    n = int(rng.integers(1, 9))
    m = int(rng.integers(1, 9))
    A = rng.integers(-4, 5, size=(m, n)).astype(float) * (rng.random((m, n)) < 0.6)
    b = rng.integers(-6, 7, size=m).astype(float)
    c = rng.integers(-5, 6, size=n).astype(float)
    kind = rng.choice(5, size=n, p=[0.4, 0.2, 0.15, 0.1, 0.15])
    lo = rng.integers(-5, 6, size=n).astype(float)
    l = np.where(kind == 0, lo, 0.0)
    u = np.where(kind == 0, lo + rng.integers(0, 7, size=n), 0.0)
    l = np.where(kind == 1, lo, l)                      # [lo, inf)
    u = np.where(kind == 1, UNB, u)
    l = np.where(kind == 2, -UNB, l)                    # (-inf, hi]
    u = np.where(kind == 2, lo, u)
    l = np.where(kind == 3, -UNB, l)                    # free
    u = np.where(kind == 3, UNB, u)
    fixed = np.where(lo == 0.0, 3.0, lo)                # fixed at a nonzero value
    l = np.where(kind == 4, fixed, l)
    u = np.where(kind == 4, fixed, u)
    return A, b, c, l, u


def _agrees_with_highs(A, b, c, l, u, r, what):
    """Status and value of a restatement result against HiGHS; an optimal answer must be a basis and a
    feasible vertex. HiGHS reports 'unbounded or infeasible' as 2 and gives up with -1 on a few unbounded
    LPs; those count as agreeing with 1 / 2."""
    h = HighsLP(A, c, b, np.full(len(b), HIGHS_INF), l, u).solve()
    assert r.status == h.status or (h.status in (2, -1) and r.status in (1, 2)), (what, r.status, h.status)
    if r.status == 0:
        assert abs(r.objective - h.objective) <= 1e-7 * max(1.0, abs(h.objective)), (what, r.objective, h.objective)
        assert int((r.col_status == 1).sum() + (r.row_status == 1).sum()) == len(b), what
        lo, hi = np.where(l <= -1e30, -np.inf, l), np.where(u >= 1e30, np.inf, u)
        assert (A @ r.x >= b - 1e-7 * (1.0 + np.abs(b))).all(), what
        assert (r.x >= lo - 1e-9 * (1.0 + np.abs(lo))).all() and (r.x <= hi + 1e-9 * (1.0 + np.abs(hi))).all(), what
    return r.status


def _random_lps(gen, seed, count=1500):
    rng = np.random.default_rng(seed)
    for t in range(count):
        yield (t,) + gen(rng)


KNOBS = [dict(pivot_mismatch=-1.0), dict(refactor_every=1), dict(refactor_every=3), dict(refactor_every=7)]
KNOB_IDS = ['mismatch', 'refactor1', 'refactor3', 'refactor7']


@pytest.mark.parametrize('knobs', KNOBS, ids=KNOB_IDS)
def test_forced_refactorisations_on_random_lps(knobs):
    """1500 random small LPs (infeasible, unbounded, degenerate, fixed variables) with every pivot refused
    once or a refactorisation every few pivots: the same statuses and values as HiGHS. Before the mismatch
    check ran ahead of the bound flips, LPs 232 and 692 of this seed stopped 'optimal' above the optimum."""
    seen = {0: 0, 1: 0, 2: 0}
    refused = 0
    for t, A, b, c, l, u in _random_lps(_random_lp, 7):
        r = dual_simplex(A, b, c, l, u, **knobs)
        seen[_agrees_with_highs(A, b, c, l, u, r, t)] += 1
        refused += r.refused
    assert min(seen.values()) > 100, seen
    if 'pivot_mismatch' in knobs:
        assert refused > 300, refused


@pytest.mark.parametrize('knobs', KNOBS, ids=KNOB_IDS)
def test_forced_refactorisations_on_grumpy_roots(knobs):
    """Root LPs of GrUMPy's 40 x 20 packing MIPs: every pivot after the first needs a bound flip or two, so a
    refused pivot that left its flips behind ended 'optimal' at a primal feasible, dual infeasible point
    (seed 0: -420.95 instead of -464.58)."""
    for seed in range(6):
        d = grumpy_random_mip(40, 20, density=0.2, rand_seed=seed)
        A = d.A.toarray()
        r = dual_simplex(A, d.b, d.c, d.l, d.u, **knobs)
        assert r.status == 0, seed
        _agrees_with_highs(A, d.b, d.c, d.l, d.u, r, seed)
        assert r.flips > 0, seed
        if 'pivot_mismatch' in knobs:
            assert r.refused > 0, seed
        # the knobs change the path, not the answer
        ref = dual_simplex(A, d.b, d.c, d.l, d.u)
        assert r.objective == pytest.approx(ref.objective, rel=1e-12), seed


# LPs of _random_lps(_random_bounded_lp, 11) that the restatement (and so the device) gets wrong through the
# artificial bound +-1e8 of an infinite bound (DESIGN section 8 item 8): a free column with a zero reduced cost
# ends on it (status 2 instead of optimal), or the round-off it leaves in x_B makes a row look infeasible at
# the optimal basis (LP 188, status 1 instead of optimal; without an upper bound on three of its columns).
ARTIFICIAL_BOUND_LPS = {188, 228, 332, 483, 570, 1000, 1024, 1136, 1340, 1425}


@pytest.mark.parametrize('knobs', [{}] + KNOBS[:2], ids=['default'] + KNOB_IDS[:2])
def test_every_kind_of_column_bound(knobs):
    """1500 random LPs whose columns have negative and positive finite lower bounds, no lower bound, no upper
    bound, no bound at all, or are fixed at a nonzero value: statuses and values equal HiGHS's, an optimal
    answer is a basis and a feasible vertex."""
    seen = {0: 0, 1: 0, 2: 0}
    for t, A, b, c, l, u in _random_lps(_random_bounded_lp, 11):
        if t in ARTIFICIAL_BOUND_LPS:
            continue
        r = dual_simplex(A, b, c, l, u, **knobs)
        seen[_agrees_with_highs(A, b, c, l, u, r, t)] += 1
    assert min(seen.values()) > 50, seen


@pytest.mark.xfail(strict=True, reason='DESIGN section 8 item 8: the artificial bound of an infinite bound')
@pytest.mark.parametrize('which', [188, 228])
def test_artificial_bound_reproducers(which):
    """Optimal LPs the dual simplex calls infeasible (188) or unbounded (228). Fixing section 8 item 8 turns
    this into a pass: then drop these LPs from ARTIFICIAL_BOUND_LPS."""
    for t, A, b, c, l, u in _random_lps(_random_bounded_lp, 11, count=which + 1):
        pass
    _agrees_with_highs(A, b, c, l, u, dual_simplex(A, b, c, l, u), t)
