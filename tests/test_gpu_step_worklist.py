"""GPU: the work lists of the frozen-path step kernels (k_work_*) must not depend on how a tile's active rows are split
into chunks.

Every active row of a tile is walked by exactly one warp trip per iteration, over its kept entries in the same order,
whatever chunk it lands in. So the same LPs solved with different rows per CTA (BLP_ROWS_PER_WARP2P for the primal
step, BLP_ROWS_PER_WARP2 for the dual step; only a -DBLP_TUNING build reads them) give bit-identical statuses,
iteration counts, objectives, x and y. A row dropped from a work list or walked twice would change them.
"""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from simple_mip_solver_b200.instances import frontier_nodes, numpy_random_mip

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (primal, dual) rows per warp before the launch plan halves them to fill the GPU: with the 8 node tiles of these
# batches the primal chunks end at 40, 32 and 24 rows, the dual chunks at 16, 8 and 16
SETTINGS = [('5', '2'), ('4', '1'), ('3', '16')]


def _c4():
    z = np.load(os.path.join(ROOT, 'bench_data', 'c4_root.npz'))
    d = numpy_random_mip(int(z['n']), int(z['m']), density=float(z['density']), seed=int(z['seed']))
    return d, z['x'], np.maximum(z['y'], 0.0)


def _digest(r):
    out = dict(status=r.status.tolist(), iters=r.iterations.tolist(),
               obj=hashlib.sha256(np.ascontiguousarray(r.objective).tobytes()).hexdigest())
    for name in ('x', 'y'):
        out[name] = hashlib.sha256(np.ascontiguousarray(getattr(r, name)).tobytes()).hexdigest()
    return out


def _cases():
    """Run in a subprocess on the tuning library: a C4 frontier slice through fewer slots than nodes (refills), and a
    batch of 450 nodes (not a multiple of 64) with pool cut rows of 300 entries (more than kLongRow) switched on per
    node."""
    from simple_mip_solver_b200 import engine as eng
    d, x0, y0 = _c4()
    res = {}
    lbs, ubs, _ = frontier_nodes(d, x0, 0, 640, 16, seed=0)
    B = lbs.shape[0]
    lp = eng.BatchLP(d.A, d.b, d.c)
    r = lp.solve_batch(lbs, ubs, x0=np.tile(x0, (B, 1)), y0=np.tile(y0, (B, 1)), opts=eng.default_opts(max_active=512))
    res['refill'] = _digest(r)
    res['refill_solved'] = int((r.status == 0).sum())
    lbs, ubs = lbs[:450], ubs[:450]
    B, k = 450, 6
    rng = np.random.default_rng(5)
    rows = np.zeros((k, d.n))
    for i in range(k):
        idx = rng.choice(d.n, 300, replace=False)
        rows[i, idx] = rng.integers(1, 10, 300)
    lp.append_rows(rows, rows @ x0 + np.array([0.5, 1.0, 0.25, 2.0, 0.1, 0.75]))
    mask = np.zeros((B, k), dtype=np.uint8)
    mask[:64, 0] = 1                      # on for the first tile only
    mask[::2, 1] = 1                      # on for every other node
    mask[:, 2] = 1                        # on everywhere
    mask[200:, 3] = 1                     # on for the last tiles; rows 4, 5 off everywhere
    r = lp.solve_batch(lbs, ubs, row_mask=mask, x0=np.tile(x0, (B, 1)),
                       y0=np.tile(np.concatenate([y0, np.zeros(k)]), (B, 1)))
    lp.close()
    res['cuts'] = _digest(r)
    res['cuts_solved'] = int((r.status == 0).sum())
    res['cuts_skipped_rows'] = float(r.stats['skipped_row_updates'])
    return res


@pytest.fixture(scope='module')
def tuning_lib(blp_lib, tmp_path_factory):
    from simple_mip_solver_b200 import _build
    return _build.build_extension(tuning=True, out=tmp_path_factory.mktemp('tuning') / 'libblp_tuning.so')


def _run(tuning_lib, primal, dual):
    code = ("import sys, json; sys.path[:0] = [%r, %r]\n"
            "import test_gpu_step_worklist as t\n"
            "print(json.dumps(t._cases()))\n") % (ROOT, os.path.join(ROOT, 'tests'))
    env = dict(os.environ, BLP_LIB=str(tuning_lib), BLP_ROWS_PER_WARP2P=primal, BLP_ROWS_PER_WARP2=dual)
    res = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, env=env, timeout=1800)
    assert res.returncode == 0, res.stdout[-1000:] + res.stderr[-4000:]
    return json.loads(res.stdout.strip().splitlines()[-1])


def test_chunk_splits_do_not_change_results(tuning_lib):
    runs = [_run(tuning_lib, p, q) for p, q in SETTINGS]
    base = runs[0]
    assert base['refill_solved'] >= 600 and base['cuts_solved'] >= 440, base
    assert base['cuts_skipped_rows'] > 0
    for (p, q), r in zip(SETTINGS[1:], runs[1:]):
        for case in ('refill', 'cuts'):
            for key in ('status', 'iters', 'obj', 'x', 'y'):
                assert r[case][key] == base[case][key], (case, key, p, q)
