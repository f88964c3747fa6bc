"""Cut rounds of BranchAndBound(BaseNode) with the default Gomory options: host cut generation (the default),
device GMI cuts (device_gomory=True, blp_simplex_gmi_cuts_host), and lock-step speculative cut rounds of each
prefetched frontier (frontier_cut_rounds=True).

Models: seeded instances.numpy_random_mip of the C3 shape (500 rows x 300 columns) and one of 1 000 rows,
each solved to a node limit. Per configuration: wall time, time spent in BaseNode._generate_cuts (host work plus,
with the device options, the device calls), engine calls (LP solves and GMI calls), LPs per solve call, evaluated nodes
and objective. The configurations alternate and repeat; the card's name and power limit are read in the same
run. Usage: python tools/gpu_cut_rounds.py --out FILE [--nodes 20] [--repeats 2]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from simple_mip_solver_b200 import BaseNode, BranchAndBound, CyLPArray, MILPInstance, engine  # noqa: E402
from simple_mip_solver_b200.instances import numpy_random_mip  # noqa: E402

MODELS = {'c3_500x300': dict(numVars=300, numCons=500, density=0.1, seed=3),
          'r1000x500': dict(numVars=500, numCons=1000, density=0.05, seed=4)}
CONFIGS = {'host_cuts': {}, 'device_gomory': dict(device_gomory=True),
           'frontier_cut_rounds': dict(frontier_cut_rounds=True)}


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else 'unknown'


def run(spec, kwargs, nodes):
    d = numpy_random_mip(**spec)
    model = MILPInstance(A=d.A.toarray(), b=CyLPArray(d.b), c=CyLPArray(d.c), l=CyLPArray(d.l), u=CyLPArray(d.u),
                         sense=['Min', '>='], integerIndices=list(d.integer_indices), numVars=len(d.c))
    spent = [0.0]
    gmi = [0]
    gen, gmi_call = BaseNode._generate_cuts, engine.BatchLP.simplex_gmi_cuts

    def timed_gen(self, **kw):
        t = time.perf_counter()
        try:
            return gen(self, **kw)
        finally:
            spent[0] += time.perf_counter() - t

    def counted_gmi(self, *a):
        gmi[0] += 1
        return gmi_call(self, *a)

    BaseNode._generate_cuts, engine.BatchLP.simplex_gmi_cuts = timed_gen, counted_gmi
    try:
        bb = BranchAndBound(model, BaseNode, node_limit=nodes, **kwargs)
        t = time.perf_counter()
        bb.solve()
        wall = time.perf_counter() - t
    finally:
        BaseNode._generate_cuts, engine.BatchLP.simplex_gmi_cuts = gen, gmi_call
    sh = bb.model.lp._shared
    out = dict(wall_s=wall, cut_generation_s=spent[0], solve_calls=sh.solve_calls, gmi_calls=gmi[0],
               device_calls=sh.solve_calls + gmi[0], lps=sh.lps_solved,
               lps_per_solve_call=sh.lps_solved / max(1, sh.solve_calls), evaluated_nodes=bb.evaluated_nodes,
               objective=bb.objective_value if np.isfinite(bb.objective_value) else str(bb.objective_value),
               status=bb.status, gmic_added=bb._kwargs.get('total_number_gmic_added', 0),
               speculative_lps=bb.speculative_lps, memo_hits=bb.memo_hits, cut_round_resolves=bb.cut_round_resolves)
    sh.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--nodes', type=int, default=20)
    ap.add_argument('--repeats', type=int, default=2)
    args = ap.parse_args()
    result = dict(card=card(), nodes=args.nodes, runs=[])
    print(result['card'], flush=True)
    for name, spec in MODELS.items():
        run(spec, {}, 2)                                  # warm-up: module load, first allocations
        for rep in range(args.repeats):
            for cname, kw in CONFIGS.items():
                r = dict(model=name, config=cname, repeat=rep, **run(spec, kw, args.nodes))
                print(json.dumps(r), flush=True)
                result['runs'].append(r)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(result, f, indent=1)


if __name__ == '__main__':
    main()
