"""GPU: the dual simplex kernels on the paths that test_gpu_simplex.py does not take on purpose — refused
pivots, the periodic refactorisation, every kind of column bound, row counts at the edges of a warp, a CTA and
the grid launch, and a stored factor continued under a row mask. Each result is compared bit for bit with the
numpy restatement (oracle/dual_simplex.py) run with the same parameters, and its value with HiGHS's.

The refused pivot and the refactorisation interval are test knobs that only a library built with -DBLP_TUNING
reads (BLP_SX_MISMATCH, BLP_SX_REFACTOR_EVERY); those cases run in a subprocess that loads such a library.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle.dual_simplex import BASIC, dual_simplex
from oracle.highs_lp import HIGHS_INF, HighsLP
from simple_mip_solver_b200.instances import grumpy_random_mip
from test_gpu_simplex import _children, same
from test_oracle_pins import _random_lp
from test_simplex_paths import ARTIFICIAL_BOUND_LPS, _random_bounded_lp, _random_lps

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UNLIMITED = 2147483647


def _device_bounds(v):
    return np.clip(v, -1e300, 1e300)


def _value_is_highs(A, b, c, l, u, obj, what):
    h = HighsLP(A, c, b, np.full(len(b), HIGHS_INF), l, u).solve()
    assert h.status == 0, what
    assert abs(obj - h.objective) <= 1e-7 * max(1.0, abs(h.objective)), (what, obj, h.objective)


def _child_bounds(d, dl):
    l, u = d.l.copy(), d.u.copy()
    for j, lo, hi in dl:
        l[j], u[j] = lo, hi
    return l, u


# ---- cases run on a tuning library (in a subprocess, see _run_with_knobs) ---------------------------------
def _knobs_from_env():
    kw = {}
    if os.environ.get('BLP_SX_MISMATCH'):
        kw['pivot_mismatch'] = float(os.environ['BLP_SX_MISMATCH'])
    if os.environ.get('BLP_SX_REFACTOR_EVERY'):
        kw['refactor_every'] = int(os.environ['BLP_SX_REFACTOR_EVERY'])
    return kw


def _cta_cases():
    """The CTA kernel under the knobs of the environment: random LPs, the grumpy 40 x 20 roots and their
    strong-branching children, from the status and from the stored factor, 5 pivots and unlimited."""
    from simple_mip_solver_b200 import engine
    kw = _knobs_from_env()
    refused = 0
    rng = np.random.default_rng(7)
    for t in range(1500):
        A, b, c, l, u = _random_lp(rng)
        if not A.any():
            continue
        lp = engine.BatchLP(A, b, c)
        res = lp.simplex_batch(l[None], _device_bounds(u)[None])
        lp.close()
        ref = dual_simplex(A, b, c, l, u, **kw)
        same(res, 0, ref, ('random', t))
        refused += ref.refused
        if ref.status == 0:
            _value_is_highs(A, b, c, l, u, res.objective[0], ('random', t))
    differs = 0
    for seed in range(3):
        d = grumpy_random_mip(40, 20, density=0.2, rand_seed=seed)
        A = d.A.toarray()
        lp = engine.BatchLP(d.A, d.b, d.c)
        root = lp.simplex_batch(d.l[None], d.u[None])
        ref_root = dual_simplex(A, d.b, d.c, d.l, d.u, **kw)
        same(root, 0, ref_root, ('root', seed))
        _value_is_highs(A, d.b, d.c, d.l, d.u, root.objective[0], ('root', seed))
        refused += ref_root.refused
        # the knobs really change the path: the default run ends with other bits
        differs += not np.array_equal(dual_simplex(A, d.b, d.c, d.l, d.u).x, ref_root.x)
        deltas = _children(d, ref_root.x, 4)
        for limit in (5, UNLIMITED):
            for cached in (False, True):
                if cached:
                    lp.simplex_batch(d.l[None], d.u[None])
                res = lp.simplex_children(d.l, d.u, deltas, col_status=root.col_status[0], row_status=root.row_status[0],
                                          parent_slot=0 if cached else -1, max_pivots=limit)
                for k, dl in enumerate(deltas):
                    l, u = _child_bounds(d, dl)
                    ref = dual_simplex(A, d.b, d.c, l, u, col_status=ref_root.col_status,
                                       row_status=ref_root.row_status, max_pivots=limit,
                                       start=ref_root if cached else None, **kw)
                    same(res, k, ref, ('child', seed, limit, cached, k))
                    refused += ref.refused
                    if limit == UNLIMITED and ref.status == 0:
                        _value_is_highs(A, d.b, d.c, l, u, res.objective[k], ('child', seed, cached, k))
        lp.close()
    assert differs > 0
    if 'pivot_mismatch' in kw:
        assert refused > 300, refused
    return refused


def _grid_cases():
    """The grid kernel under the knobs of the environment: root cold, children from the status and from the
    stored factor. A refused pivot costs the restatement a refactorisation, so that case runs on a 1025 x 48 LP
    (root: 94 pivots, 58 bound flips), the others on the 500 x 1100 LP of test_wide_kernel_is_bit_identical_too."""
    from simple_mip_solver_b200 import engine
    kw = _knobs_from_env()
    if 'pivot_mismatch' in kw:
        d, limits = grumpy_random_mip(48, 1025, density=0.15, rand_seed=1025), (5, UNLIMITED)
    else:
        d, limits = grumpy_random_mip(500, 1100, density=0.02, maxObjCoeff=10, maxConsCoeff=10, tightness=2,
                                      rand_seed=7), (5,)
    A = d.A.toarray()
    lp = engine.BatchLP(d.A, d.b, d.c)
    assert not lp.simplex_batched
    root = lp.simplex_batch(d.l[None], d.u[None])
    ref_root = dual_simplex(A, d.b, d.c, d.l, d.u, **kw)
    same(root, 0, ref_root, 'wide root')
    _value_is_highs(A, d.b, d.c, d.l, d.u, root.objective[0], 'wide root')
    assert ref_root.flips > 0 and (ref_root.refused > 0 or 'pivot_mismatch' not in kw)
    deltas = _children(d, ref_root.x, 1)
    for limit in limits:
        for cached in (False, True):
            if cached:
                lp.simplex_batch(d.l[None], d.u[None])
            res = lp.simplex_children(d.l, d.u, deltas, col_status=root.col_status[0], row_status=root.row_status[0],
                                      parent_slot=0 if cached else -1, max_pivots=limit)
            for k, dl in enumerate(deltas):
                l, u = _child_bounds(d, dl)
                ref = dual_simplex(A, d.b, d.c, l, u, col_status=ref_root.col_status, row_status=ref_root.row_status,
                                   max_pivots=limit, start=ref_root if cached else None, **kw)
                same(res, k, ref, ('wide child', limit, cached, k))
                if limit == UNLIMITED and ref.status == 0:
                    _value_is_highs(A, d.b, d.c, l, u, res.objective[k], ('wide child', cached, k))
    lp.close()
    return int(root.pivots[0])


@pytest.fixture(scope='module')
def tuning_lib(blp_lib, tmp_path_factory):
    from simple_mip_solver_b200 import _build
    return _build.build_extension(tuning=True, out=tmp_path_factory.mktemp('tuning') / 'libblp_tuning.so')


def _run_with_knobs(tuning_lib, cases, **knobs):
    code = ("import sys, json; sys.path[:0] = [%r, %r]\n"
            "import test_gpu_simplex_paths as t\n"
            "print(json.dumps(t.%s()))\n") % (ROOT, os.path.join(ROOT, 'tests'), cases)
    env = dict(os.environ, BLP_LIB=str(tuning_lib), **knobs)
    res = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, env=env, timeout=1200)
    assert res.returncode == 0, res.stdout[-1000:] + res.stderr[-4000:]
    return json.loads(res.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize('knobs', [dict(BLP_SX_MISMATCH='-1'), dict(BLP_SX_REFACTOR_EVERY='3')],
                         ids=['mismatch', 'refactor3'])
def test_cta_kernel_with_refused_pivots_and_refactorisations(tuning_lib, knobs):
    """A refused pivot leaves nothing behind (its bound flips included), and a refactorisation every 3 pivots
    continues where the updated inverse left off: the device follows the restatement bit for bit and ends at
    HiGHS's optimum on every LP and child."""
    refused = _run_with_knobs(tuning_lib, '_cta_cases', **knobs)
    print('refused pivots', refused)


@pytest.mark.parametrize('knobs', [dict(BLP_SX_MISMATCH='-1'), dict(BLP_SX_REFACTOR_EVERY='300')],
                         ids=['mismatch', 'refactor300'])
def test_grid_kernel_with_refused_pivots_and_refactorisations(tuning_lib, knobs):
    """The same on the cooperative grid kernel, whose team barriers the refused pivot must not skip."""
    pivots = _run_with_knobs(tuning_lib, '_grid_cases', **knobs)
    print('wide root pivots', pivots)


# ---- production library -----------------------------------------------------------------------------------
def test_every_kind_of_column_bound_bit_exact(blp_lib):
    """1500 LPs with negative and positive lower bounds, free columns, columns fixed at a nonzero value and
    infinite upper bounds: bit for bit the restatement's answers, HiGHS's value where the restatement has it
    (ARTIFICIAL_BOUND_LPS: DESIGN section 8 item 8)."""
    from simple_mip_solver_b200 import engine
    seen = {0: 0, 1: 0, 2: 0}
    for t, A, b, c, l, u in _random_lps(_random_bounded_lp, 11):
        if not A.any():
            continue
        lp = engine.BatchLP(A, b, c)
        res = lp.simplex_batch(_device_bounds(l)[None], _device_bounds(u)[None])
        lp.close()
        ref = dual_simplex(A, b, c, l, u)
        same(res, 0, ref, t)
        seen[ref.status] += 1
        if ref.status == 0 and t not in ARTIFICIAL_BOUND_LPS:
            _value_is_highs(A, b, c, l, u, res.objective[0], t)
    assert min(seen.values()) > 50, seen


def _tableau_is_inverse_times_matrix(lp, res, A, what):
    basic = np.flatnonzero(np.concatenate([res.col_status[0], res.row_status[0]]) == BASIC)
    assert len(basic) == A.shape[0], what
    rows = lp.simplex_tableau_rows(0, basic)
    full = np.concatenate([A, -np.eye(A.shape[0])], axis=1)
    want = np.linalg.solve(full[:, basic], full)
    assert np.allclose(rows, want, rtol=1e-9, atol=1e-9), (what, np.abs(rows - want).max())


@pytest.mark.parametrize('m', [31, 32, 33, 255, 256, 257, 1024, 1025])
def test_row_counts_at_the_kernel_edges(blp_lib, m):
    """Row counts around a warp, the 128-thread CTA, the 512-thread CTA's sweep and the last CTA-kernel size,
    and 1025 (the first grid launch): bit for bit the restatement, HiGHS's value, and tableau rows equal to
    inv(B) [A, -I]."""
    from simple_mip_solver_b200 import engine
    d = grumpy_random_mip(48, m, density=0.15, rand_seed=m)
    A = d.A.toarray()
    lp = engine.BatchLP(d.A, d.b, d.c)
    assert lp.simplex_batched == (m <= 1024)
    res = lp.simplex_batch(d.l[None], d.u[None])
    ref = dual_simplex(A, d.b, d.c, d.l, d.u)
    assert ref.status == 0 and ref.pivots > 0
    same(res, 0, ref, m)
    _value_is_highs(A, d.b, d.c, d.l, d.u, res.objective[0], m)
    _tableau_is_inverse_times_matrix(lp, res, A, m)
    lp.close()


def test_wide_kernel_tableau_rows(blp_lib):
    """Tableau rows of the 500 x 1100 root (grid kernel) against inv(B) [A, -I], every basic variable."""
    from simple_mip_solver_b200 import engine
    d = grumpy_random_mip(500, 1100, density=0.02, maxObjCoeff=10, maxConsCoeff=10, tightness=2, rand_seed=7)
    lp = engine.BatchLP(d.A, d.b, d.c)
    res = lp.simplex_batch(d.l[None], d.u[None])
    assert res.status[0] == 0
    _tableau_is_inverse_times_matrix(lp, res, d.A.toarray(), 'wide root')
    lp.close()


def test_stored_factor_with_masked_rows(blp_lib):
    """Children that start from the parent's stored factor (parent_slot) and switch a pool row off: if that row's
    slack is basic in the parent the factor is continued; if the row is tight there the kernel factorises the
    parent's status again. Both bit for bit the restatement (start=, row_on=), both at HiGHS's value."""
    from simple_mip_solver_b200 import engine
    d = grumpy_random_mip(30, 15, density=0.3, rand_seed=5)
    A = d.A.toarray()
    x0 = dual_simplex(A, d.b, d.c, d.l, d.u).x
    # pool row 0 cuts the root optimum off (tight in the parent), pool row 1 is far from binding (slack basic)
    S = np.argsort(-(x0 - np.floor(x0)))[:6]
    cuts = np.zeros((2, d.n))
    cuts[0, S] = -1.0
    cuts[1, :] = -1.0
    rhs = np.array([-np.floor(x0[S].sum() - 1e-9), -10.0 * (x0.sum() + 1.0)])
    assert cuts[0] @ x0 < rhs[0]
    Afull, bfull = np.vstack([A, cuts]), np.concatenate([d.b, rhs])
    lp = engine.BatchLP(d.A, d.b, d.c)
    lp.append_rows(cuts, rhs)
    parent = lp.simplex_batch(d.l[None], d.u[None], row_mask=np.ones((1, 2), np.uint8))
    ref_parent = dual_simplex(Afull, bfull, d.c, d.l, d.u)
    same(parent, 0, ref_parent, 'parent')
    assert ref_parent.row_status[d.m] != BASIC and ref_parent.row_status[d.m + 1] == BASIC
    deltas = _children(d, ref_parent.x, 2)
    for off, continued in ((1, True), (0, False)):
        mask = np.ones(2, np.uint8)
        mask[off] = 0
        on = np.concatenate([np.ones(d.m, bool), mask.astype(bool)])
        lp.simplex_batch(d.l[None], d.u[None], row_mask=np.ones((1, 2), np.uint8))     # the parent is the last call
        res = lp.simplex_children(d.l, d.u, deltas, row_mask=mask, col_status=parent.col_status[0],
                                  row_status=parent.row_status[0], parent_slot=0)
        assert ((~on & (ref_parent.row_status != BASIC)).any()) != continued
        for k, dl in enumerate(deltas):
            l, u = _child_bounds(d, dl)
            ref = dual_simplex(Afull, bfull, d.c, l, u, row_on=on, col_status=ref_parent.col_status,
                               row_status=ref_parent.row_status, start=ref_parent)
            same(res, k, ref, (off, k))
            if ref.status == 0:
                _value_is_highs(Afull[on], bfull[on], d.c, l, u, res.objective[k], (off, k))
    lp.close()
