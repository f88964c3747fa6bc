import os, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from simple_mip_solver_b200 import engine
from simple_mip_solver_b200.instances import grumpy_random_mip
from oracle.highs_lp import HIGHS_INF, HighsLP
d = grumpy_random_mip(500, 300, density=0.1, maxObjCoeff=10, maxConsCoeff=10, tightness=2, rand_seed=2)
h = HighsLP(d.A, d.c, d.b, np.full(d.m, HIGHS_INF), d.l, d.u); root = h.solve(); x = root.x
ints = np.asarray(d.integer_indices)
frac = np.minimum(x[ints] - np.floor(x[ints]), np.ceil(x[ints]) - x[ints])
cand = ints[np.argsort(-frac, kind='stable')][:64]
deltas = []
for j in cand:
    deltas.append([(int(j), d.l[j], float(np.floor(x[j])))]); deltas.append([(int(j), float(np.ceil(x[j])), d.u[j])])
lp = engine.BatchLP(d.A, d.b, d.c)
rr = lp.solve_batch(d.l[None], d.u[None])
for rep in range(4):
    t = time.perf_counter(); r = lp.solve_children(d.l, d.u, deltas, x0=rr.x[0], y0=rr.y[0], integer_indices=d.integer_indices); dt = time.perf_counter() - t
    print(rep, 'gpu_s', round(dt, 4), 'iters max', r.iterations.max(), 'mean', int(r.iterations.mean()), 'status', np.unique(r.status, return_counts=True), 'launches', r.stats['kernel_launches'], 'total_ms', round(r.stats['total_ms'],1), 'step_ms', round(r.stats['step_kernel_ms'],1))
objs = []
for dl in deltas:
    l, u = d.l.copy(), d.u.copy(); l[dl[0][0]], u[dl[0][0]] = dl[0][1], dl[0][2]
    h.set_col_bounds(l, u); h.set_basis(root.col_basis, root.row_basis); s = h.solve(); objs.append((s.status, s.objective))
print('max rel err', max(abs(a - b[1]) / max(1, abs(b[1])) for a, b, s in zip(r.objective, objs, r.status) if s == 0 and b[0] == 0), 'status match', all(int(s) == b[0] for s, b in zip(r.status, objs)))
