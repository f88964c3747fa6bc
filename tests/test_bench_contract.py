"""bench.py contract that can be checked without a GPU: the reference arm's JSON line (the driver
computes its ratio from it), the committed root fixtures every workload branches from, and the
refusal of the product arm to define its workload with the oracle."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench                                                     # noqa: E402


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--workload', 'c3',
                          '--steps', '2', '--warmup', '1'], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith('{')]
    assert len(lines) == 1
    j = json.loads(lines[0])
    assert j['impl'] == 'reference' and j['metric'] == bench.METRIC and j['unit'] == bench.UNIT
    assert j['n_gpus'] == 1 and j['steps'] == 2 and j['warmup'] == 1 and j['higher_is_better'] is True
    assert j['value'] > 0 and j['ms_per_step'] > 0 and j['vs_baseline'] is None and j['dtype'] == 'f64'
    assert j['gpu_launches'] == 0
    assert j['e2e'] == {'value': j['value'], 'unit': j['unit'], 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    cb = j['cpu_baseline']
    assert cb['kind'] == 'port' and cb['cores'] >= 1 and cb['value'] == j['value'] and 'HiGHS' in cb['sample']
    assert j['config']['workload'].startswith('c3:')


def test_other_ranks_of_the_reference_arm_exit_without_work():
    env = dict(os.environ, RANK='1', LOCAL_RANK='1', WORLD_SIZE='2')
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--workload', 'c3',
                          '--gpus', '2', '--steps', '1', '--warmup', '1'], capture_output=True, text=True,
                         timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0 and not [ln for ln in out.stdout.splitlines() if ln.startswith('{')]


@pytest.mark.parametrize('name', list(bench.WORKLOADS))
def test_root_fixture_is_the_lp_optimum_of_its_workload(name):
    """x is feasible, y >= 0 prices it out (reduced costs have the right sign at the bounds), the
    objective equals c.x = the dual objective: the fixture is an optimal primal-dual pair."""
    d, depth, root = bench.load_instance(name)
    assert root is not None, 'every workload ships its root fixture'
    x, y = root['x'], root['y']
    assert x.shape == (d.n,) and y.shape == (d.m,)
    scale = 1.0 + abs(root['objective'])
    assert (x >= d.l - 1e-7).all() and (x <= d.u + 1e-7).all()
    assert (d.A @ x >= d.b - 1e-6).all() and (y >= 0).all()
    r = d.c - d.A.T @ y
    dual = d.b @ y + np.maximum(r, 0) @ d.l + np.minimum(r, 0) @ d.u
    assert abs(d.c @ x - root['objective']) <= 1e-9 * scale
    assert abs(dual - root['objective']) <= 1e-7 * scale


def test_dump_outputs_is_seeded_float64_and_bounded(tmp_path):
    """--dump-outputs writes the same sample of the same result twice, in float64, within 64 MB."""
    import torch
    n, m, B, ld = 3000, 1000, 100, 128
    r = dict(obj=torch.randn(ld, dtype=torch.float64), lower=torch.randn(ld, dtype=torch.float64),
             status=torch.zeros(ld, dtype=torch.int32), iters=torch.arange(ld, dtype=torch.int32),
             frac=torch.full((ld,), -1, dtype=torch.int32),
             x=torch.arange(n * ld, dtype=torch.float64).reshape(n, ld),
             y=torch.arange(m * ld, dtype=torch.float64).reshape(m, ld))
    bench.dump_outputs(str(tmp_path / 'a'), r, B)
    bench.dump_outputs(str(tmp_path / 'b'), r, B)
    names = sorted(os.listdir(tmp_path / 'a'))
    assert names == sorted(f'{k}.npy' for k in ('obj', 'lower', 'status', 'iters', 'frac', 'x_sample', 'y_sample'))
    total = 0
    for f in names:
        a, b = np.load(tmp_path / 'a' / f), np.load(tmp_path / 'b' / f)
        assert a.dtype == np.float64 and np.array_equal(a, b), f
        total += os.path.getsize(tmp_path / 'a' / f)
    assert total <= 64 << 20
    assert np.array_equal(np.load(tmp_path / 'a' / 'obj.npy'), r['obj'][:B].numpy())
    x = np.load(tmp_path / 'a' / 'x_sample.npy')
    assert x.size == bench.DUMP_SAMPLE and (x % ld < B).all()     # only columns of real nodes


def test_product_arm_never_defines_its_workload_with_the_oracle():
    src = open(os.path.join(ROOT, 'bench.py')).read()
    gpu_arm = src[src.index("    from simple_mip_solver_b200.instances import frontier_nodes\n    n, m, B = d.n"):]
    head = gpu_arm[:gpu_arm.index('# ---- CPU baseline first')]
    assert 'root_by_oracle' not in head and 'SystemExit' in head
