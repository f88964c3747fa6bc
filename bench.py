#!/usr/bin/env python
"""bench.py — node-LP solves/sec of the batched bound step (BASELINE.json metric).

A *step* is one pass of the hot path over one batch: ``--batch`` open nodes (a slice of the
synthetic frontier of the named workload, default C5: 50 000 vars x 20 000 rows, ~200k nonzeros)
are solved to the parity tolerance (rel. KKT 1e-7, see DESIGN.md section 2; --eps 1e-8 for SURVEY 8d's figure) by one ``blp_solve_batch`` call per GPU.
``--slots`` of them are resident at a time (blp_opts.max_active): a node that finishes hands its
slot to the next pending node of the slice, so the step kernels sweep a constant batch width.
With N GPUs every rank solves its own slice of the frontier (weak scaling: per-GPU batch fixed)
and the only collective is the 16-byte all-reduce(min) of [incumbent, dual bound] per step.

  value   device-resident inputs (bounds and warm start already in HBM), CUDA-event time on the
          library's stream, max over ranks;
  e2e     same metric through the host-buffer plugin call (``BatchLP.solve_children`` =
          blp_solve_children_host: the root's bounds, per node its changed bounds, the root's primal/dual
          pair as warm start): host arrays in, H2D + solve + D2H of objective/status/x/y of every node
          inside the timed region;
  roofline  k_primal / k_dual per-launch time from CUDA events around every launch of the timed
          steps (blp_opts.profile) against the measured HBM copy peak;
  cpu_baseline  the HiGHS dual-simplex stand-in for the reference's CLP path (oracle/highs_lp.py),
          warm-started from the root basis, one LP per task on all host cores, bounded sample.

  named_config  BASELINE.json config 5 AS NAMED, timed in the same run after the steps above: ``--named-batch``
          (4096) concurrent node LPs per step split over the N GPUs (strong scaling: 4096/N per GPU), device
          resident, CUDA events, max over ranks, golden nodes validated — so that the driver's 1/2/4/8-GPU
          runs carry the weak-scaling curve (`value`) and the strong-scaling curve of the named frontier.

``--impl reference`` times only that CPU path (rank 0).

``--dump-outputs DIR`` writes what the last timed step of `value` returned (see dump_outputs), so that two
builds can be compared output for output on the same inputs.

bench.py writes nothing into the repository (it may be read-only): no bytecode caches, and a library whose
sources changed since build() is recompiled into a temporary directory.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (n, m, density, max dive depth, fixture)
    'c5': (50000, 20000, 2e-4, 32, 'c5_root.npz'),
    'c4': (10000, 5000, 2e-3, 16, 'c4_root.npz'),
    'c3': (500, 300, 0.1, 8, 'c3_root.npz'),
}
METRIC = 'node_lp_solves_per_sec'
UNIT = 'node-LPs/s'


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def load_instance(name):
    from simple_mip_solver_b200.instances import grumpy_random_mip, numpy_random_mip
    n, m, dens, depth, fixture = WORKLOADS[name]
    if name == 'c3':
        d = grumpy_random_mip(n, m, density=dens, maxObjCoeff=10, maxConsCoeff=10, tightness=2, rand_seed=2)
    else:
        d = numpy_random_mip(n, m, density=dens, seed=2)
    root = None
    if fixture and os.path.exists(os.path.join(ROOT, 'bench_data', fixture)):
        z = np.load(os.path.join(ROOT, 'bench_data', fixture))
        root = dict(x=z['x'], y=np.maximum(z['y'], 0.0), col_basis=z['col_basis'].astype(np.int32),
                    row_basis=z['row_basis'].astype(np.int32), objective=float(z['objective']))
    return d, depth, root


def load_child_goldens(name):
    """Committed HiGHS answers for the frontier nodes GOLD_FIRST.. (tests/tools/make_child_goldens.py)."""
    path = os.path.join(ROOT, 'bench_data', f'{name}_children.npz')
    if not os.path.exists(path):
        return None
    z = np.load(path)
    return dict(node_ids=z['node_ids'], status=z['status'], objective=z['objective'])


GOLD_PER_STEP = 8          # nodes with committed golden answers that ride in every step


def step_nodes(d, root, depth, seed, slice_index, B, gold):
    """Nodes of one step: B - 8 nodes of the frontier slice plus 8 of the 64 nodes whose HiGHS answers
    are committed (the same generator, ids from the reserved range), rotating with the slice. They are
    solved and timed like every other node; bench.py compares them with the goldens afterwards.
    A node is its list of ``(var, lb, ub)`` changes against the root bounds (base_node.py:595-600)."""
    from simple_mip_solver_b200.instances import GOLD_COUNT, GOLD_FIRST, frontier_nodes
    g = GOLD_PER_STEP if (gold is not None and B > GOLD_PER_STEP) else 0
    _, _, deltas = frontier_nodes(d, root['x'], slice_index * B, B - g, depth, seed=seed, dense=False)
    gold_ids = []
    if g:
        gold_ids = [(slice_index * g + t) % GOLD_COUNT for t in range(g)]
        for i in gold_ids:
            deltas = deltas + frontier_nodes(d, root['x'], GOLD_FIRST + i, 1, depth, seed=0, dense=False)[2]
    return deltas, gold_ids


class Validator:
    """Collects (golden id, status, objective) of the golden nodes of every timed step."""

    def __init__(self, gold):
        self.gold, self.rows = gold, []

    def add(self, gold_ids, status, objective):
        for i, st, ob in zip(gold_ids, status, objective):
            self.rows.append((int(i), int(st), float(ob)))

    def report(self, tol=1e-6):
        if self.gold is None:
            return {'checked': 0, 'ok': 0, 'note': 'no committed child goldens for this workload'}
        ok, worst = 0, 0.0
        for i, st, ob in self.rows:
            gs, go = int(self.gold['status'][i]), float(self.gold['objective'][i])
            err = abs(ob - go) / max(1.0, abs(go)) if (gs == 0 and st == 0) else 0.0
            worst = max(worst, err)
            ok += int(st == gs and err <= tol)
        return {'checked': len(self.rows), 'ok': ok, 'max_rel_objective_error': worst, 'tolerance': tol,
                'against': 'bench_data/*_children.npz (HiGHS dual simplex, made offline), compared after the timed region'}


DUMP_NODES = 1 << 19          # per-node values of at most this many nodes (4 MB per array)
DUMP_SAMPLE = 1 << 20         # (coordinate, node) entries of x and of y (8 MB each)


def dump_outputs(out_dir, r, B):
    """Write the result of one solve_batch_device call as float64 DIR/<name>.npy: obj, lower, status, iters
    and frac of the first min(B, DUMP_NODES) nodes, and x_sample / y_sample, the primal and dual solutions at
    DUMP_SAMPLE (coordinate, node) pairs drawn with a fixed seed (the full x and y of 2048 C5 nodes take
    1.2 GB). At most 36 MB in all."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    k = min(B, DUMP_NODES)
    out = {name: r[name][:k] for name in ('obj', 'lower', 'status', 'iters', 'frac')}
    rng = np.random.default_rng(0)
    for name in ('x', 'y'):
        rows = r[name].shape[0]
        idx = rng.integers(0, rows, DUMP_SAMPLE), rng.integers(0, B, DUMP_SAMPLE)
        out[name + '_sample'] = r[name][tuple(torch.from_numpy(i).to(r[name].device) for i in idx)]
    for name, t in out.items():
        np.save(os.path.join(out_dir, name + '.npy'), t.double().cpu().numpy())
    log(f'wrote {len(out)} arrays of the last timed step to {out_dir}')


def root_by_oracle(d):
    """Root vertex/basis from the HiGHS oracle (only when no fixture is committed)."""
    from oracle.highs_lp import HIGHS_INF, HighsLP
    r = HighsLP(d.A, d.c, d.b, np.full(d.m, HIGHS_INF), d.l, d.u).solve()
    return dict(x=r.x, y=np.maximum(r.row_dual, 0.0), col_basis=r.col_basis, row_basis=r.row_basis,
                objective=r.objective)


# ------------------------------------------------------------------------------------- CPU arm
_W = {}


def _cpu_init(A, b, c, l, u, col_basis, row_basis, tol=1e-9):
    from oracle.highs_lp import HIGHS_INF, HighsLP
    _W['lp'] = HighsLP(A, c, b, np.full(A.shape[0], HIGHS_INF), l, u, tol=tol)
    _W['basis'] = (col_basis, row_basis)
    _W['l'], _W['u'] = l, u


def _cpu_solve(deltas):
    """One node LP on one core: root bounds + deltas, warm start from the root basis (the
    reference hands the parent's basis to the child, base_node.py:589,608)."""
    lp = _W['lp']
    l, u = _W['l'].copy(), _W['u'].copy()
    for j, lo, hi in deltas:
        l[j], u[j] = lo, hi
    lp.set_col_bounds(l, u)
    lp.set_basis(*_W['basis'])
    t = time.perf_counter()
    r = lp.solve()
    return r.status, r.objective, time.perf_counter() - t


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


class CpuArm:
    def __init__(self, d, root, cores, tol=1e-9):
        import multiprocessing as mp
        self.cores = cores
        ctx = mp.get_context('fork')
        self.pool = ctx.Pool(cores, initializer=_cpu_init,
                             initargs=(d.A, d.b, d.c, d.l, d.u, root['col_basis'], root['row_basis'], tol))

    def run(self, deltas_list):
        t = time.perf_counter()
        out = self.pool.map(_cpu_solve, deltas_list, chunksize=1)
        return out, time.perf_counter() - t

    def close(self):
        self.pool.close()
        self.pool.join()


# ------------------------------------------------------------------------------------- helpers
class ClockSampler:
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.idx = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', f'--id={self.idx}', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                 '-lms', '200'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([t.strip() for t in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for nm, v in zip(names, r[3:7]):
                    if v.lower().startswith('active'):
                        reasons.add(nm)
            except (ValueError, IndexError):
                pass
        # samples under load: the upper half of the observed clocks
        sm.sort()
        load = sm[len(sm) // 2:] if sm else []
        return {'sm_mhz': float(np.median(load)) if load else None,
                'sm_max_mhz': max(mx) if mx else None, 'reasons': sorted(reasons),
                'samples': len(sm)}


def node_bytes(n, m):
    """Algorithmic HBM bytes per node and iteration, as the kernels' state representation requires
    them. SURVEY.md section 8d counts 8(6n+3m) with dense per-node bounds and 8(4n+3m) with bounds
    kept as deltas, which is what the kernels do (one reference bound per row and 32-node block plus
    a deviation mask); since the Halpern anchors are stored in fp32 the count is
      primal launch: xbar read + write (16n), anchor xa (4n), gathered y (8m)
      dual launch:   y read + write (16m), anchor ya (4m), gathered xbar (8n)
    = 28(n+m) per node and iteration (1.96 MB at C5; 8(4n+3m) would be 2.08 MB)."""
    return 20 * n + 8 * m, 8 * n + 20 * m


# ------------------------------------------------------------------------------------- main
def run_reference(args, d, depth, root, rank):
    """The reference's CPU path (HiGHS-DS stand-in for CLP) on all host cores."""
    from simple_mip_solver_b200.instances import frontier_nodes
    if rank != 0:
        return
    cores = host_cores()
    if root is None:
        root = root_by_oracle(d)
    per_step = args.cpu_nodes or cores
    arm = CpuArm(d, root, cores, tol=args.eps)
    steps = args.warmup + args.steps
    times, solved = [], 0
    for s in range(steps):
        _, _, deltas = frontier_nodes(d, root['x'], s * per_step, per_step, depth, seed=args.seed)
        out, dt = arm.run(deltas)
        if s >= args.warmup:
            times.append(dt)
            solved += sum(1 for st, _, _ in out if st in (0, 1, 2))
    arm.close()
    total = sum(times)
    value = solved / total
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * total / max(args.steps, 1),
        'higher_is_better': True, 'scaling': args.scaling, 'vs_baseline': None, 'dtype': 'f64',
        'data': 'synthetic',
        'config': workload_config(args, d, per_step),
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                         'sample': f'{per_step} frontier nodes per step on {cores} processes, HiGHS 1.12 dual '
                                   f'simplex (stand-in for CLP), presolve off, feasibility tolerances {args.eps:g} (the GPU arm\'s eps_rel), warm start from the root basis'},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, d, batch):
    n, m, dens, depth, _ = WORKLOADS[args.workload]
    return {'workload': f'{args.workload}: frontier of open-node LPs of a synthetic sparse MILP, {n} vars x {m} rows, '
                        f'{d.A.nnz} nonzeros, dive depth U{{1..{depth}}}, solved to rel. KKT {args.eps:g}; '
                        f'{batch} nodes per step per GPU ({args.scaling} scaling; the 4096-node frontier of the named config '
                        f'is swept in slices), '
                        f'{min(args.slots, batch) if args.slots > 0 else batch} of them resident at a time '
                        f'(finished nodes hand their slot to pending ones)',
            'batch_per_gpu': batch, 'resident_slots': min(args.slots, batch) if args.slots > 0 else batch,
            'eps_rel': args.eps, 'seed': args.seed,
            'l2_policy': 'solver state per step exceeds L2 (see state_mb); no flush needed'}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=2)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='blp', choices=['blp', 'reference'])
    ap.add_argument('--workload', default='c5', choices=list(WORKLOADS))
    ap.add_argument('--batch', type=int, default=2048,
                    help='open nodes per step: per GPU with --scaling weak, in total with --scaling strong')
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'],
                    help='weak: every GPU solves --batch nodes per step; strong: --batch nodes per step are '
                         'split over the GPUs (BASELINE.json config 5 as named: --batch 4096 --scaling strong)')
    ap.add_argument('--e2e-steps', type=int, default=3)
    ap.add_argument('--slots', type=int, default=512,
                    help='nodes resident at a time (blp_opts.max_active); 0 = the whole batch')
    ap.add_argument('--eps', type=float, default=1e-7)
    ap.add_argument('--max-iters', type=int, default=2000000)
    ap.add_argument('--seed', type=int, default=0)
    ap.add_argument('--cpu-nodes', type=int, default=0, help='CPU arm: nodes per step (default: one per core)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--named-batch', type=int, default=4096,
                    help='weak-scaling runs also time BASELINE.json config 5 AS NAMED in the same process: this many '
                         'concurrent node LPs per step split over the GPUs (strong scaling); 0 = skip')
    ap.add_argument('--named-steps', type=int, default=1)
    ap.add_argument('--named-warmup', type=int, default=0,
                    help='extra warm-up steps of the named leg (it runs warm: after the W + K steps behind `value`)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last timed step returned as DIR/<name>.npy '
                         '(float64, about 17 MB at the default batch; rank 0\'s slice)')
    args = ap.parse_args()
    sys.dont_write_bytecode = True

    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))

    d, depth, root = load_instance(args.workload)
    if args.impl == 'reference':
        run_reference(args, d, depth, root, rank)
        return

    if args.scaling == 'strong':
        if args.batch % world:
            raise SystemExit(f'--scaling strong: --batch {args.batch} is not a multiple of {world} GPUs')
        args.batch //= world
    from simple_mip_solver_b200.instances import frontier_nodes
    n, m, B = d.n, d.m, args.batch
    gold = load_child_goldens(args.workload)
    checker = Validator(gold)
    checker_e2e = Validator(gold)
    if root is None:      # the product arm never runs the oracle, not even to define its workload
        raise SystemExit(f'bench_data/{WORKLOADS[args.workload][4]} is missing: make it with '
                         f'tests/tools/make_bench_fixture.py')

    # ---- CPU baseline first (fork pool before CUDA is initialised), rank 0 at N=1 only ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = host_cores()
        k = args.cpu_nodes or cores
        _, _, deltas = frontier_nodes(d, root['x'], 10_000_000, k, depth, seed=args.seed)
        arm = CpuArm(d, root, cores, tol=args.eps)
        out, dt = arm.run(deltas)
        arm.close()
        ok = sum(1 for st, _, _ in out if st in (0, 1, 2))
        cpu = {'value': ok / dt, 'unit': UNIT, 'cores': cores, 'kind': 'port',
               'sample': f'{k} frontier nodes of the same workload, one LP per process on {cores} processes, '
                         f'HiGHS 1.12 dual simplex (stand-in for CLP), presolve off, feasibility tolerances {args.eps:g}, '
                         f'warm start from the root basis; {dt:.1f} s wall, mean {np.mean([t for _, _, t in out]):.2f} s per LP per core'}
        log('cpu_baseline', cpu)

    import torch
    import torch.distributed as dist
    from simple_mip_solver_b200 import _build, engine, parallel
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    if _build.is_stale():
        # sources changed since build(): this run's library goes to a directory that lives as long as main()
        lib_dir = tempfile.TemporaryDirectory(prefix='blp_bench_')
        engine._LIB_PATH = _build.build_extension(out=Path(lib_dir.name) / 'libblp.so')

    lp = engine.BatchLP(d.A, d.b, d.c, device=local_rank)
    # blp_allreduce_min over the library's own NCCL communicator when world > 1; all ranks or none
    # (parallel.join_library_comm): the node LPs, which are what is timed, do not depend on it
    use_comm = parallel.join_library_comm(lp, device=dev, log=lambda msg: print(msg, file=sys.stderr))
    ld = engine.leading_dim(B)
    W = min(args.slots, B) if args.slots > 0 else B           # resident node slots
    ldW = engine.leading_dim(W)
    ext = torch.cuda.ExternalStream(lp.stream_ptr, device=dev)
    opts = engine.default_opts(eps_rel=args.eps, max_iters=args.max_iters, max_active=W)
    opts_prof = engine.default_opts(eps_rel=args.eps, max_iters=min(args.max_iters, 1024), profile=1)
    int_idx = torch.arange(n, dtype=torch.int32, device=dev)

    def node_slice(step):
        return step_nodes(d, root, depth, args.seed, step * world + rank, B, gold)

    root_l = torch.from_numpy(d.l).to(dev)
    root_u = torch.from_numpy(d.u).to(dev)

    def pack(deltas):
        """host side of a slice: (node, var, lb, ub) of every bound change, pinned"""
        node = np.concatenate([np.full(len(dl), k, dtype=np.int64) for k, dl in enumerate(deltas)])
        flat = [t for dl in deltas for t in dl]
        arr = lambda v, dt: torch.from_numpy(np.asarray(v, dtype=dt)).pin_memory()
        return (arr(node, np.int64), arr([t[0] for t in flat], np.int64), arr([t[1] for t in flat], np.float64),
                arr([t[2] for t in flat], np.float64))

    def to_device(packed, count=B):
        """root bounds broadcast over the node columns, then the slice's bound changes scattered in"""
        ldc = engine.leading_dim(count)
        lb = root_l[:, None].expand(n, ldc).contiguous()
        ub = root_u[:, None].expand(n, ldc).contiguous()
        node, var, lo, hi = (t.to(dev, non_blocking=True) for t in packed)
        keep = node < count
        lb[var[keep], node[keep]] = lo[keep]
        ub[var[keep], node[keep]] = hi[keep]
        return lb, ub

    x0 = torch.from_numpy(root['x']).to(dev)[:, None].expand(n, ld).contiguous()
    y0 = torch.from_numpy(root['y']).to(dev)[:, None].expand(m, ld).contiguous()

    def exchange(res_obj, res_lower, res_status, res_frac, count=B):
        """16-byte all-reduce(min) of [best integral objective in slice, min open lower bound]."""
        st = res_status[:count]
        integral = (st == 0) & (res_frac[:count] < 0)
        inc = float(res_obj[:count][integral].min().item()) if bool(integral.any()) else float('inf')
        open_ = (st == 0) & ~integral
        lowb = float(res_lower[:count][open_].min().item()) if bool(open_.any()) else float('inf')
        return parallel.allreduce_bounds(inc, lowb, device=dev, lp=lp if use_comm else None)

    total_steps = args.warmup + args.steps
    slices = [node_slice(s) for s in range(total_steps)]
    packed = [pack(sl[0]) for sl in slices]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        lp.stream_sync()

    # ---- device-resident arm ----
    iters_all = []
    agg = dict(launches=0, solved=0, unsolved=0, infeasible=0, node_iters=0.0, iters=0,
               primal_ms=0.0, dual_ms=0.0, step_ms=0.0, total_ms=0.0, refills=0, skipped_cols=0.0, skipped_rows=0.0)
    sampler = ClockSampler(local_rank)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for s in range(total_steps):
        lb, ub = to_device(packed[s])
        if s == args.warmup:
            barrier()
            if rank == 0:
                sampler.start()
            ev0.record(ext)
        r = lp.solve_batch_device(lb, ub, x0=x0, y0=y0, int_idx=int_idx, opts=opts, want_x=True, want_y=True)
        exchange(r['obj'], r['lower'], r['status'], r['frac'])
        if s >= args.warmup:
            st = r['status'][:B]
            agg['solved'] += int(((st == 0) | (st == 1) | (st == 2)).sum().item())
            agg['unsolved'] += int((st == 3).sum().item())
            agg['infeasible'] += int((st == 1).sum().item())
            iters_all.append(r['iters'][:B].cpu().numpy())
            g = len(slices[s][1])
            if g:
                checker.add(slices[s][1], st[B - g:B].cpu().numpy(), r['obj'][B - g:B].cpu().numpy())
            sdict = r['stats']
            agg['launches'] += sdict['kernel_launches']
            agg['node_iters'] += sdict['node_iterations']
            agg['iters'] += sdict['iterations']
            agg['primal_ms'] += sdict['primal_kernel_ms']
            agg['dual_ms'] += sdict['dual_kernel_ms']
            agg['step_ms'] += sdict['step_kernel_ms']
            agg['total_ms'] += sdict['total_ms']
            agg['refills'] += sdict['refills']
            agg['skipped_cols'] += sdict['skipped_col_updates']
            agg['skipped_rows'] += sdict['skipped_row_updates']
        log(f'[rank {rank}] step {s} iters {r["stats"]["iterations"]} total_ms {r["stats"]["total_ms"]:.0f}')
        del lb, ub
    ev1.record(ext)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, r, B)
    # per-kernel split: the first 1024 iterations of the first W nodes of the last timed slice once
    # more (full batch width) with CUDA events around every k_primal / k_dual launch
    # (blp_opts.profile: no CUDA graph; not part of `value`)
    prof = None
    if rank == 0:
        lb, ub = to_device(packed[-1], W)
        prof = lp.solve_batch_device(lb, ub, x0=x0[:, :ldW].contiguous(), y0=y0[:, :ldW].contiguous(),
                                     int_idx=int_idx, opts=opts_prof, want_x=False, want_y=False)['stats']
        del lb, ub
    # plain batched SpMV (BASELINE.json's second figure): Y = A X and G = A' Y at the resident width,
    # CUDA events on the library stream, operands larger than L2; not part of `value`
    spmv = None
    if rank == 0:
        spmv = {}
        for name, tr, rin, rout in (('A', False, n, m), ('AT', True, m, n)):
            X = torch.randn((rin, ldW), dtype=torch.float64, device=dev)
            Y = torch.empty((rout, ldW), dtype=torch.float64, device=dev)
            torch.cuda.synchronize(dev)
            for _ in range(3):
                lp.spmv_async(X, Y, W, transpose=tr)
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record(ext)
            for _ in range(20):
                lp.spmv_async(X, Y, W, transpose=tr)
            s1.record(ext)
            lp.stream_sync()
            spmv[name] = s0.elapsed_time(s1) / 20.0
            del X, Y
    dev_ms = ev0.elapsed_time(ev1)
    dev_ms = parallel.allreduce_max(dev_ms, device=dev)
    sums = parallel.allreduce_sum([agg['solved'], agg['unsolved'], agg['launches'], agg['infeasible']], device=dev)
    value = sums[0] / (dev_ms * 1e-3)

    # ---- end-to-end arm: pinned host buffers through the plugin call ----
    e2e_steps = max(1, args.e2e_steps)
    e2e_slices = [node_slice(total_steps + s) for s in range(1 + e2e_steps)]
    # The nodes of a frontier are children of the root: the plugin call takes them as the reference
    # creates them (base_node.py:592-608) — the parent's bounds, per node the changed bounds, the
    # parent's primal/dual pair as the common warm start (blp_solve_children_host).
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()
    hl, hu, hx0, hy0 = pin(d.l), pin(d.u), pin(root['x']), pin(root['y'])
    opts_e = engine.default_opts(eps_rel=args.eps, max_iters=args.max_iters, max_active=W)
    ints = list(range(n))
    h2d = d2h = 0
    e2e_solved = 0
    t0 = None
    for s in range(1 + e2e_steps):
        deltas_s = e2e_slices[s][0]
        if s == 1:
            barrier()
            t0 = time.perf_counter()
        rr = lp.solve_children(hl, hu, deltas_s, x0=hx0, y0=hy0, integer_indices=ints, opts=opts_e)
        integral = (rr.status == 0) & (rr.frac_idx < 0)
        inc = float(rr.objective[integral].min()) if integral.any() else float('inf')
        open_ = (rr.status == 0) & ~integral
        lowb = float(rr.lower_bound[open_].min()) if open_.any() else float('inf')
        parallel.allreduce_bounds(inc, lowb, device=dev, lp=lp if use_comm else None)
        if s >= 1:
            g = len(e2e_slices[s][1])
            if g:
                checker_e2e.add(e2e_slices[s][1], rr.status[B - g:], rr.objective[B - g:])
            e2e_solved += int(np.isin(rr.status, (0, 1, 2)).sum())
            nd = sum(len(dl) for dl in deltas_s)
            h2d = hl.nbytes + hu.nbytes + hx0.nbytes + hy0.nbytes + 4 * n + 4 * (B + 1) + 20 * nd
            d2h = rr.x.nbytes + rr.y.nbytes + rr.objective.nbytes + rr.lower_bound.nbytes + \
                rr.status.nbytes + rr.iterations.nbytes + rr.frac_idx.nbytes
    barrier()
    e2e_s = parallel.allreduce_max(time.perf_counter() - t0, device=dev)
    e2e_total = parallel.allreduce_sum([e2e_solved], device=dev)[0]

    # ---- BASELINE.json config 5 as named, in the same run: --named-batch concurrent node LPs per step split
    # over the GPUs (strong scaling), device-resident and timed like `value`. Only next to a weak-scaling run of the
    # named workload; every rank takes the same branches, so the collectives inside line up.
    named = None
    Bn = args.named_batch // world if args.named_batch > 0 else 0
    if args.scaling == 'weak' and args.workload == 'c5' and args.named_steps > 0 and Bn >= 64 and \
            Bn * world == args.named_batch and Bn % 64 == 0:
        del x0, y0
        ldn = engine.leading_dim(Bn)
        Wn = min(args.slots, Bn) if args.slots > 0 else Bn
        xn = torch.from_numpy(root['x']).to(dev)[:, None].expand(n, ldn).contiguous()
        yn = torch.from_numpy(root['y']).to(dev)[:, None].expand(m, ldn).contiguous()
        opts_n = engine.default_opts(eps_rel=args.eps, max_iters=args.max_iters, max_active=Wn)
        checker_n = Validator(gold)
        n_steps = args.named_warmup + args.named_steps
        # slices of the same frontier generator, far from the ones timed above
        n_slices = [step_nodes(d, root, depth, args.seed, 100_000 + s * world + rank, Bn, gold) for s in range(n_steps)]
        n_packed = [pack(sl[0]) for sl in n_slices]
        n0, n1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n_solved = n_iters = 0
        n_node_iters = 0.0
        if args.named_warmup == 0:
            barrier()
            n0.record(ext)
        for s in range(n_steps):
            lb, ub = to_device(n_packed[s], Bn)
            if s == args.named_warmup and s > 0:
                barrier()
                n0.record(ext)
            r = lp.solve_batch_device(lb, ub, x0=xn, y0=yn, int_idx=int_idx, opts=opts_n, want_x=True, want_y=True)
            exchange(r['obj'], r['lower'], r['status'], r['frac'], count=Bn)
            if s >= args.named_warmup:
                st = r['status'][:Bn]
                n_solved += int(((st == 0) | (st == 1) | (st == 2)).sum().item())
                n_iters += r['stats']['iterations']
                n_node_iters += r['stats']['node_iterations']
                g = len(n_slices[s][1])
                if g:
                    checker_n.add(n_slices[s][1], st[Bn - g:Bn].cpu().numpy(), r['obj'][Bn - g:Bn].cpu().numpy())
            log(f'[rank {rank}] named step {s} iters {r["stats"]["iterations"]} total_ms {r["stats"]["total_ms"]:.0f}')
            del lb, ub
        n1.record(ext)
        barrier()
        n_ms = parallel.allreduce_max(n0.elapsed_time(n1), device=dev)
        n_total = parallel.allreduce_sum([n_solved], device=dev)[0]
        named = {'value': n_total / (n_ms * 1e-3), 'unit': UNIT, 'scaling': 'strong',
                 'nodes_per_step': args.named_batch, 'nodes_per_gpu': Bn, 'resident_slots': Wn,
                 'steps': args.named_steps, 'warmup': args.named_warmup, 'ms_per_step': n_ms / args.named_steps,
                 'slot_utilisation': n_node_iters / max(n_iters * Wn, 1), 'validated': checker_n.report(),
                 'note': 'BASELINE.json config 5 as named (this many concurrent node LPs, sharded by node over the GPUs), '
                         'timed in the same run, warm, after the W + K steps behind `value`: CUDA events on the library stream, '
                         'barrier + synchronize on both sides, max over ranks; slot_utilisation is rank 0\'s'}
        del xn, yn

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        except Exception:
            pass
        peak = float(peaks.get('hbm_gbs', 6650.0))
        peak_src = 'measured (MEASURED_PEAKS.json hbm_gbs)' if 'hbm_gbs' in peaks else 'fallback 6650 GB/s'
        pb, db = node_bytes(n, m)
        bytes_A = 12 * d.A.nnz + 4 * (m + 1)
        bytes_AT = 12 * d.A.nnz + 4 * (n + 1)
        # iteration pair over the TIMED steps (CUDA events around each period's step graph)
        it_timed = max(agg['iters'], 1)
        # a coordinate the kernels skipped as frozen (blp_opts.freeze) costs neither its 20 stream bytes nor, its entries
        # being folded out of the tile's matrices, the 8 bytes of its gathered value: 28 bytes per ACTIVE coordinate
        pair_bytes = ((pb + db) * agg['node_iters'] - 28 * (agg['skipped_cols'] + agg['skipped_rows'])
                      + (bytes_A + bytes_AT) * it_timed) / it_timed
        pair_s = agg['step_ms'] * 1e-3 / it_timed
        pair_gbs = pair_bytes / pair_s / 1e9
        # per-kernel split from the profile step (same slice as the last timed step)
        it_prof = max(prof['iterations'], 1)
        primal_bytes = (pb * prof['node_iterations'] - 20 * prof['skipped_col_updates'] - 8 * prof['skipped_row_updates']
                        + bytes_AT * it_prof) / it_prof
        dual_bytes = (db * prof['node_iterations'] - 20 * prof['skipped_row_updates'] - 8 * prof['skipped_col_updates']
                      + bytes_A * it_prof) / it_prof
        primal_s = prof['primal_kernel_ms'] * 1e-3 / it_prof
        dual_s = prof['dual_kernel_ms'] * 1e-3 / it_prof
        prim_gbs = primal_bytes / primal_s / 1e9 if primal_s > 0 else 0.0
        dual_gbs = dual_bytes / dual_s / 1e9 if dual_s > 0 else 0.0
        traffic = None
        try:
            tr = json.load(open(os.path.join(ROOT, 'profiles', 'r2z_traffic.json')))
            if tr['workload'] == args.workload and tr['batch'] == W:
                # DRAM read+write bytes of one k_primal2 + one k_dual2 launch at full batch width (ncu)
                traffic = tr['k_primal2_dram_bytes_per_launch'] + tr['k_dual2_dram_bytes_per_launch']
        except Exception:
            pass
        state_mb = 8 * ldW * (7 * n + 4 * m) / 1e6
        cfg = workload_config(args, d, B)
        cfg['state_mb'] = round(state_mb, 1)
        cfg['timing'] = 'value: CUDA events on the library stream around the K timed steps, max over ranks'
        if world > 1:
            cfg['bound_exchange'] = ('blp_allreduce_min (library NCCL communicator), 16 bytes per step' if use_comm
                                     else 'torch.distributed all_reduce (library communicator unavailable)')
        line = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': dev_ms / max(args.steps, 1), 'higher_is_better': True,
            'scaling': args.scaling, 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic', 'config': cfg,
            'validated': {'device_arm': checker.report(), 'e2e_arm': checker_e2e.report()},
            'e2e': {'value': e2e_total / e2e_s, 'unit': UNIT, 'h2d_bytes_per_step': int(h2d),
                    'd2h_bytes_per_step': int(d2h), 'steps': e2e_steps},
            'gpu_launches': int(sums[2]),
            'clocks': clocks,
            'roofline': {'bound': 'hbm', 'kernel': 'PDHG iteration = k_primal + k_dual (one launch each)',
                         'achieved': pair_gbs, 'peak': peak, 'unit': 'GB/s', 'frac': pair_gbs / peak,
                         'traffic': traffic, 'traffic_note': 'ncu dram read+write of one iteration at FULL batch width early in a solve '
                         '(profiles/r2z_traffic.json: 66 % of the columns, 27 % of the rows frozen; algorithmic bytes of that '
                         'launch pair: 450 MB); bytes_per_launch is the average over the timed steps, '
                         'where slots of finished nodes are refilled while nodes are pending and the tail of a step is compacted', 'full_width_bytes': (pb + db) * W + bytes_A + bytes_AT,
                         'peak_source': peak_src, 'bytes_per_launch': pair_bytes,
                         'ms_per_launch': pair_s * 1e3,
                         'measured': 'CUDA events around every period graph (64 iterations) of the timed steps; '
                                     'bytes = 28 per ACTIVE (coordinate, node) and iteration — 20 streamed + 8 gathered; frozen coordinates '
                                     '(nodes.frozen_*_share) are neither updated nor gathered — '
                                     '+ both matrices (bounds kept as block reference + mask, fp32 anchors)',
                         'k_primal': {'achieved': prim_gbs, 'frac': prim_gbs / peak, 'bytes_per_launch': primal_bytes,
                                      'ms_per_launch': primal_s * 1e3},
                         'k_dual': {'achieved': dual_gbs, 'frac': dual_gbs / peak, 'bytes_per_launch': dual_bytes,
                                    'ms_per_launch': dual_s * 1e3},
                         'split_measured': 'first 1024 iterations of the last timed slice (full batch width) re-run with CUDA events around every launch'},
            'spmv': {'unit': 'GB/s', 'batch': W, 'note': 'plain batched SpMV on the unscaled matrix, node-fastest '
                     'operands [rows][ld]; bytes = 12 nnz + 4(rows+1) + 8 B (n + m); CUDA events over 20 launches',
                     'A': {'ms': spmv['A'], 'achieved': (bytes_A + 8 * W * (n + m)) / spmv['A'] / 1e6,
                           'frac': (bytes_A + 8 * W * (n + m)) / spmv['A'] / 1e6 / peak},
                     'AT': {'ms': spmv['AT'], 'achieved': (bytes_AT + 8 * W * (n + m)) / spmv['AT'] / 1e6,
                            'frac': (bytes_AT + 8 * W * (n + m)) / spmv['AT'] / 1e6 / peak}},
            'cpu_baseline': cpu,
            'named_config': named,
            'nodes': {'solved': int(sums[0]), 'iteration_limit': int(sums[1]), 'infeasible': int(sums[3]),
                      'pdhg_iterations_per_step': agg['iters'] / max(args.steps, 1),
                      'refills_per_step': agg['refills'] / max(args.steps, 1),
                      'mean_iterations_per_node': agg['node_iters'] / max(agg['solved'] + agg['unsolved'], 1),
                      # how full the resident slots were over the timed steps: 1 - this is the tail of a step (slots
                      # idle once nothing is pending and the slowest nodes finish), rank 0
                      'slot_utilisation': agg['node_iters'] / max(agg['iters'] * W, 1),
                      # share of the (column, node, iteration) / (row, node, iteration) updates skipped as frozen
                      'frozen_col_share': agg['skipped_cols'] / max(agg['node_iters'] * n, 1),
                      'frozen_row_share': agg['skipped_rows'] / max(agg['node_iters'] * m, 1),
                      'iterations_p50_p90_max': [float(np.percentile(np.concatenate(iters_all), q)) for q in (50, 90, 100)]},
        }
        print(json.dumps(line), flush=True)
    lp.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
