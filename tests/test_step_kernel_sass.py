"""What the compiler made of the frozen-path step kernels k_primal2<false> / k_dual2<false> (CPU only: nvcc and
cuobjdump cross-compile for sm_100a without a GPU).

They are latency bound: a warp's trip over one matrix row costs as many dependent memory round trips as the
compiled code serialises. The source asks for BLP_U gathers in flight per batch; at the 48-register budget of
5 CTAs per SM the compiler used to issue them one (primal) or two (dual) at a time. These tests pin the budget
and the batch depth of the shared-slab gather loop.
"""
from __future__ import annotations

import re
import shutil
import subprocess
from pathlib import Path

import pytest

from simple_mip_solver_b200 import _build

KERNELS = {
    'k_primal2<false>': '_ZN3blp9k_primal2ILb0EEEvNS_7DevProbENS_8DevStateEiiiPKii',
    'k_dual2<false>': '_ZN3blp7k_dual2ILb0EEEvNS_7DevProbENS_8DevStateEiiiPKii',
}
BLP_U = 4


def _tool(name):
    exe = shutil.which(name) or f'/usr/local/cuda/bin/{name}'
    if not Path(exe).exists():
        pytest.skip(f'{name} not available')
    return exe


@pytest.fixture(scope='module')
def compiled(tmp_path_factory):
    nvcc, cuobjdump = _tool('nvcc'), _tool('cuobjdump')
    out = tmp_path_factory.mktemp('sass') / 'blp.cubin'
    # the flags of _build.build_extension, with -cubin instead of -shared
    cmd = [nvcc, '-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
           '-cubin', '-Xptxas', '-v', '-o', str(out), str(_build.CSRC / 'blp.cu')]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    sass = {}
    for name, sym in KERNELS.items():
        r = subprocess.run([cuobjdump, '-sass', '-fun', sym, str(out)], capture_output=True, text=True)
        assert r.returncode == 0 and sym in r.stdout, r.stderr
        sass[name] = r.stdout
    return res.stdout + res.stderr, sass


def ptxas_usage(log, sym):
    """(registers, spill store bytes, spill load bytes) from the -Xptxas -v report of one kernel."""
    m = re.search(r"Function properties for %s\s*\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, "
                  r"(\d+) bytes spill loads\s*\n[^\n]*Used (\d+) registers" % re.escape(sym), log)
    assert m, 'no ptxas report for ' + sym
    return int(m.group(4)), int(m.group(2)), int(m.group(3))


_INS = re.compile(r'/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;')
_REG = re.compile(r'\bR(\d+)\b')


def _instructions(sass):
    for line in sass.splitlines():
        m = _INS.search(line)
        if m:
            yield re.sub(r'^@!?U?P[T\d]+\s+', '', m.group(1))


def gather_batches(sass):
    """Shared-slab gathers issued before the first DFMA that reads one of them, per batch.

    A shared-slab gather is a 128-bit global load whose address derives from a 32-bit LDS (the entry's column
    index read from the CTA's slab). The walk is linear: the loop bodies of these kernels have no inner branches.
    """
    tainted, pending, batches, issued = set(), set(), [], 0
    for ins in _instructions(sass):
        op, _, rest = ins.partition(' ')
        ops = [o.strip() for o in rest.split(',')]
        dst = _REG.match(ops[0]) if ops and ops[0] else None
        width = 2 if ('.WIDE' in op or '.64' in op) else (4 if '.128' in op else 1)
        dregs = set(range(int(dst.group(1)), int(dst.group(1)) + width)) if dst else set()
        srcs = {int(r) for o in ops[1:] for r in _REG.findall(o)}
        if op.startswith('LDG') and '.128' in op and 'CONSTANT' not in op:
            addr = {int(r) for r in _REG.findall(ops[1])} if len(ops) > 1 else set()
            if addr & tainted:
                pending |= dregs
                issued += 1
            else:
                pending -= dregs
            tainted -= dregs
            continue
        if op.startswith('DFMA') and srcs & pending:
            batches.append(issued)
            pending, issued = set(), 0
        if op == 'LDS':
            tainted |= dregs
        elif op.startswith(('LD', 'ST', 'ATOM', 'RED', 'BAR', 'BRA', 'EXIT', 'BSSY', 'BSYNC')):
            tainted -= dregs
        elif srcs & tainted:
            tainted |= dregs
        else:
            tainted -= dregs
        pending -= dregs if not op.startswith('DFMA') else set()
    return batches


@pytest.mark.parametrize('kernel', sorted(KERNELS))
def test_register_budget_without_spills(compiled, kernel):
    log, _ = compiled
    regs, st, ld = ptxas_usage(log, KERNELS[kernel])
    assert regs <= 48, f'{kernel}: {regs} registers, 5 CTAs of 256 threads per SM need <= 48'
    assert st == 0 and ld == 0, f'{kernel}: {st} bytes of spill stores, {ld} of spill loads'


@pytest.mark.parametrize('kernel', sorted(KERNELS))
def test_full_gather_batch_in_flight(compiled, kernel):
    _, sass = compiled
    batches = gather_batches(sass[kernel])
    assert batches, f'{kernel}: no shared-slab gather loop found'
    assert min(batches) >= BLP_U, f'{kernel}: gathers in flight before the first use, per batch: {batches}'
