"""Sweep of the grouped mid-size dual simplex (k_simplex_wide, G groups of S = SMs / G CTAs in one launch).

For m in {1100, 2048, 5000 (the C4 shape), 8192}, batches B in {1, 2, 4, ..., 64} and forced G (BLP_SX_GROUPS on a
-DBLP_TUNING library, G = 1 being the whole GPU on each node in turn) plus the library's own rule, it times two
workloads on strong-branching children of the root:
  five   5 pivots per child from the root's stored factor (parent_slot 0),
  full   unlimited pivots from the root's basis status (factorisation included),
and the same children on PDHG with the 512 * 5 iteration budget that 'auto' routing gives them today.
Each point is the simplex kernel time (CUDA events, stats step_kernel_ms) over REPS repetitions, the G values
alternating within a repetition. Outputs (status, pivots, objective, x) must be bit-identical across G.
Writes the points to --out (default simplex_groups_sweep.json in the working directory); device name and power
limit are read in the same run.

    python tools/gpu_simplex_groups.py [--reps 3] [--shapes 1100,2048,5000,8192]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

import _tuning  # noqa: F401  (builds and selects the tuning library before the engine is imported)
from simple_mip_solver_b200 import engine
from simple_mip_solver_b200.instances import grumpy_random_mip, numpy_random_mip

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BATCHES = (1, 2, 4, 8, 16, 32, 64)
FULL_MAX_B = {5000: 8}          # full solves at the C4 shape factorise ~5000 columns per child


def _shape(m):
    if m == 1100:
        return grumpy_random_mip(500, 1100, density=0.02, maxObjCoeff=10, maxConsCoeff=10, tightness=2, rand_seed=7), None
    if m == 5000:
        z = np.load(os.path.join(ROOT, 'bench_data', 'c4_root.npz'))
        return numpy_random_mip(10000, 5000, density=float(z['density']), seed=int(z['seed'])), z
    return grumpy_random_mip(48, m, density=0.15, rand_seed=m), None


def _children(d, x, B):
    ints = np.asarray(d.integer_indices)
    frac = np.minimum(x[ints] - np.floor(x[ints]), np.ceil(x[ints]) - x[ints])
    cand = ints[np.argsort(-frac, kind='stable')]
    out = []
    for j in cand:
        out.append([(int(j), float(d.l[j]), float(np.floor(x[j])))])
        out.append([(int(j), float(np.ceil(x[j])), float(d.u[j]))])
        if len(out) >= B:
            break
    return out[:B]


def _groups(B):
    return [g for g in (1, 2, 4, 8, 16, 32, 64) if g <= B] + ['auto']


def _set_groups(g):
    if g == 'auto':
        os.environ.pop('BLP_SX_GROUPS', None)
    else:
        os.environ['BLP_SX_GROUPS'] = str(g)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--shapes', default='1100,2048,5000,8192')
    ap.add_argument('--batches', default=','.join(map(str, BATCHES)))
    ap.add_argument('--out', default='simplex_groups_sweep.json')
    a = ap.parse_args()
    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip()
    rec = dict(device=smi, reps=a.reps, points=[])
    print('device:', smi, flush=True)
    for m in map(int, a.shapes.split(',')):
        d, z = _shape(m)
        lp = engine.BatchLP(d.A, d.b, d.c)
        t = time.perf_counter()
        if z is not None:            # the C4 root: its optimal basis is stored, factorise it (no pivot needed)
            root = lp.simplex_batch(d.l[None], d.u[None], col_status=z['col_basis'][None], row_status=z['row_basis'][None])
        else:
            _set_groups(1)
            root = lp.simplex_batch(d.l[None], d.u[None])
        assert root.status[0] == 0, root.status
        cs, rs = root.col_status[0], root.row_status[0]
        print(f'm {m} n {d.n}: root {root.pivots[0]} pivots, {time.perf_counter() - t:.1f} s', flush=True)

        def store_root():
            lp.simplex_batch(d.l[None], d.u[None], col_status=cs[None], row_status=rs[None], max_pivots=0)

        for B in map(int, a.batches.split(',')):
            if B * m * m * 8 > 60e9:
                continue
            deltas = _children(d, root.x[0], B)
            if len(deltas) < B:
                continue
            for work in ('five', 'full'):
                if work == 'full' and B > FULL_MAX_B.get(m, 64):
                    continue
                times, first = {g: [] for g in _groups(B)}, None
                for rep in range(a.reps):
                    for g in _groups(B):
                        _set_groups(g)
                        if work == 'five':
                            store_root()
                        r = lp.simplex_children(d.l, d.u, deltas, col_status=cs, row_status=rs,
                                                parent_slot=0 if work == 'five' else -1,
                                                max_pivots=5 if work == 'five' else 2147483647)
                        times[g].append(r.stats['step_kernel_ms'])
                        got = (r.status.copy(), r.pivots.copy(), r.objective.copy(), r.x.copy())
                        if first is None:
                            first = got
                        else:
                            assert all(np.array_equal(u, v) for u, v in zip(first, got)), (m, B, work, g)
                point = dict(m=m, n=d.n, B=B, work=work, ms={str(g): v for g, v in times.items()},
                             pivots_sum=int(first[1].sum()))
                if work == 'five':
                    _set_groups('auto')
                    opts = engine.default_opts(max_iters=5 * 512)
                    pd = []
                    for rep in range(a.reps):
                        pr = lp.solve_children(d.l, d.u, deltas, x0=root.x[0], y0=root.y[0],
                                               integer_indices=d.integer_indices, opts=opts, want_x=False, want_y=False)
                        pd.append(pr.stats['total_ms'])
                    point['pdhg_ms'] = pd
                rec['points'].append(point)
                med = {g: float(np.median(v)) for g, v in times.items()}
                print(json.dumps(dict(m=m, B=B, work=work, median_ms=med, pdhg=point.get('pdhg_ms'))), flush=True)
                os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
                with open(a.out, 'w') as f:
                    json.dump(rec, f, indent=1)
        lp.close()
    _set_groups('auto')


if __name__ == '__main__':
    sys.exit(main())
