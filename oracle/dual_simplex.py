"""TEST INFRASTRUCTURE — numpy restatement of the bounded dual simplex the device runs for small LPs.

The reference solves every node LP with CLP's dual simplex from the parent's basis
(``simple_mip_solver/nodes/base_node.py:273`` ``self.lp.dual()``, ``:589, 608`` get/setBasisStatus,
``:645-646`` ``maxNumIteration`` pivots for strong branching). CLP is third party and absent from
/root/reference and from this image, so the pivoting rules are the textbook ones (Koberstein, "The
dual simplex method", 2005: dual steepest edge pricing, bound flipping ratio test), stated completely
here so that the CUDA kernel (simple_mip_solver_b200/csrc/blp_simplex.cuh) can be checked against this
file PIVOT FOR PIVOT. Every floating-point operation below is a single rounded IEEE operation (no
fused multiply-add) and every sum runs in a fixed order, which the kernel reproduces, so basis,
pivot count and solution agree bit for bit.

  LP        min c.x,  A x - s = b,  l <= x <= u,  s >= 0 (s free for a row that is masked off)
  basis     explicit dense inverse Binv of the m basic columns of [A, -I]
  start     the given CLP-coded status (1 basic, 2 at upper, 3 at lower) or the slack basis. Basic
            structurals are pivoted into the slack basis one by one in index order; the pivot row
            is the largest |alpha_i| among the rows still owned by a slack that is to leave
            (smallest row on ties); without a pivot > PIV_TOL the column stays nonbasic and its
            row keeps its slack (basis repair). Nonbasic columns with a wrong-signed reduced cost
            are moved to their other bound, to an artificial bound +-BIG if that one is infinite.
  leaving   dual steepest edge: largest infeasibility^2 / ||row of Binv||^2; ties (relative
            TIE_REL) -> smallest variable index
  entering  bound flipping ratio test: candidates in order of (ratio rounded to 2^-36, larger
            |alpha| first, smaller index first); a boxed candidate whose flip leaves the row
            infeasible is flipped, the first one that cannot be flipped enters
  pivot     alpha_q = Binv a_q first; if it disagrees with alpha_r[q] (PIVOT_MISMATCH), refactorise
            and price again with nothing applied; otherwise the flips, then the basis change
  stop      0 optimal, 1 primal infeasible (no entering column), 3 pivot limit,
            2 unbounded (a variable ends at an artificial bound)
  finish    x_B, y, d recomputed from Binv, one step of iterative refinement on x_B

Pinned against: the reference's known answers (small_branch root x == [0, 1.25, 1.5],
test_base_node.py:406-416; no_branch, infeasible, unbounded, cut2) and HiGHS optimal values on every
fixture (tests/test_oracle_pins.py). The choice among alternative optimal vertices beyond those
pins is CLP's and unpinned (SURVEY.md section 8c).

Only tests/ and tests/golden/make_goldens.py may import this module; the product never does.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

BASIC, AT_UPPER, AT_LOWER = 1, 2, 3
PRIMAL_TOL = 1e-9
DUAL_TOL = 1e-9
PIV_TOL = 1e-9
TIE_REL = 1e-12
RATIO_BIN = 2.0 ** 36
BIG = 1e8
INF = 1e30
WEIGHT_LANES = 16            # the kernel sums a row's squares in 16 interleaved partial sums
REFACTOR_EVERY = 1000        # ... or 2 m pivots if that is more (a refactorisation costs about as many pivots as there are basic structurals)
PIVOT_MISMATCH = 1e-7        # |alpha_q[r] - alpha_r[q]| relative: the inverse has drifted, refactorise before pivoting


@dataclass
class SimplexResult:
    status: int
    objective: float
    x: np.ndarray
    y: np.ndarray            # row duals (>= 0 for an active row a.x >= b)
    rc: np.ndarray           # reduced costs of the structurals
    col_status: np.ndarray   # CLP codes
    row_status: np.ndarray
    pivots: int
    head: np.ndarray         # basic variable of every row position
    Binv: np.ndarray
    flips: int = 0
    weights: np.ndarray = None
    refused: int = 0         # pivots refused by the mismatch check (each followed by a refactorisation)


def _weights(Binv):
    m = Binv.shape[0]
    sq = Binv * Binv
    w = np.zeros(m)
    for lane in range(WEIGHT_LANES):
        part = np.zeros(m)
        for k in range(lane, m, WEIGHT_LANES):
            part = part + sq[:, k]
        w = w + part
    return w


def _update_inverse(Binv, alpha, r):
    """Binv <- E Binv for the basis change in row position r (alpha = Binv a_q)."""
    row = Binv[r] / alpha[r]
    Binv -= np.outer(alpha, row)          # elementwise: one multiply, one subtract
    Binv[r] = row


def _matvec_cols(M, v):
    """sum_k M[:, k] * v[k] in ascending k, skipping zeros of v (value preserving)."""
    acc = np.zeros(M.shape[0])
    for k in np.flatnonzero(v):
        acc = acc + M[:, k] * v[k]
    return acc


def _vecmat_rows(v, M):
    """sum_i v[i] * M[i, :] in ascending i, skipping zeros of v."""
    acc = np.zeros(M.shape[1])
    for i in np.flatnonzero(v):
        acc = acc + v[i] * M[i, :]
    return acc


def dual_simplex(A, b, c, l, u, row_on=None, col_status=None, row_status=None,
                 max_pivots: int = 2147483647, dse: bool = True, bfrt: bool = True,
                 start: 'SimplexResult' = None, pivot_mismatch: float = PIVOT_MISMATCH,
                 refactor_every: int = 0) -> SimplexResult:
    """``pivot_mismatch`` and ``refactor_every`` (0: max(REFACTOR_EVERY, 2 m)) are the two knobs a library
    built with -DBLP_TUNING reads from BLP_SX_MISMATCH and BLP_SX_REFACTOR_EVERY: a negative threshold refuses
    every pivot that does not directly follow a factorisation."""
    A = np.asarray(A, dtype=float)
    m, n = A.shape
    N = n + m
    b = np.asarray(b, dtype=float)
    row_on = np.ones(m, bool) if row_on is None else np.asarray(row_on, bool)
    l = np.asarray(l, dtype=float)
    u = np.asarray(u, dtype=float)
    lo = np.concatenate([np.where(l <= -INF, -np.inf, l), np.where(row_on, 0.0, -np.inf)])
    hi = np.concatenate([np.where(u >= INF, np.inf, u), np.full(m, np.inf)])
    cost = np.concatenate([np.asarray(c, dtype=float), np.zeros(m)])
    art_lo = np.zeros(N, bool)
    art_hi = np.zeros(N, bool)
    art_done = np.zeros(N, bool)
    stat = np.full(N, AT_LOWER, dtype=np.int32)
    want_basic = np.zeros(N, bool)
    if col_status is None or row_status is None:
        want_basic[n:] = True
    else:
        cs, rs = np.asarray(col_status), np.asarray(row_status)
        stat[:n] = np.where(cs == AT_UPPER, AT_UPPER, AT_LOWER)
        want_basic[:n] = cs == BASIC
        want_basic[n:] = (rs == BASIC) | ~row_on

    head = np.arange(n, N)
    Binv = -np.eye(m)

    def factor(want):
        """Slack basis, then the wanted structurals pivoted in one by one (also the refactorisation)."""
        nonlocal head, Binv
        head = np.arange(n, N)
        Binv = -np.eye(m)
        keep = stat.copy()
        stat[n:] = BASIC
        stat[:n] = np.where(keep[:n] == BASIC, AT_LOWER, keep[:n])
        for j in np.flatnonzero(want[:n]):
            alpha = _matvec_cols(Binv, A[:, j])
            best, r = PIV_TOL, -1
            for i in range(m):
                if head[i] >= n and not want[head[i]] and abs(alpha[i]) > best:
                    best, r = abs(alpha[i]), i
            if r < 0:
                continue
            _update_inverse(Binv, alpha, r)
            s = head[r]
            stat[s] = keep[s] if keep[s] != BASIC else AT_LOWER
            head[r] = j
            stat[j] = BASIC

    def nonbasic_values():
        v = np.where(stat == AT_UPPER, hi, lo)
        v[stat == BASIC] = 0.0
        return v

    def duals():
        cB = cost[head]
        y = _vecmat_rows(cB, Binv)
        d = cost.copy()
        d[:n] = cost[:n] - _vecmat_rows(y, A)
        d[n:] = y
        d[stat == BASIC] = 0.0
        return y, d

    def primal():
        xN = nonbasic_values()
        rhs = b - _matvec_cols(A, xN[:n]) + xN[n:]
        return _matvec_cols(Binv, rhs), rhs

    def make_dual_feasible(d):
        for j in range(N):
            if stat[j] == BASIC:
                continue
            if lo[j] == hi[j]:
                stat[j] = AT_LOWER
                continue
            if d[j] < -DUAL_TOL:
                stat[j] = AT_UPPER
            elif d[j] > DUAL_TOL:
                stat[j] = AT_LOWER
            elif stat[j] == AT_LOWER and np.isinf(lo[j]):
                stat[j] = AT_UPPER
            elif stat[j] == AT_UPPER and np.isinf(hi[j]):
                stat[j] = AT_LOWER
            if stat[j] == AT_UPPER and np.isinf(hi[j]):
                hi[j] = BIG
                art_hi[j] = True
            if stat[j] == AT_LOWER and np.isinf(lo[j]):
                lo[j] = -BIG
                art_lo[j] = True

    if start is not None:
        # continue from the factorised basis another solve ended with (blp_simplex_*'s parent_slot)
        stat[:n] = start.col_status
        stat[n:] = start.row_status
        if (~row_on & (stat[n:] != BASIC)).any():
            want_basic[:] = stat == BASIC
            want_basic[n:] |= ~row_on
            start = None
        else:
            head = start.head.copy()
            Binv = start.Binv.copy()
    if start is None:
        factor(want_basic)
    y, d = duals()
    make_dual_feasible(d)
    xB, _ = primal()
    w = (start.weights.copy() if start is not None else _weights(Binv)) if dse else np.ones(m)

    pivots = flips_total = refused = 0
    since_factor = 0
    refactor_every = refactor_every if refactor_every > 0 else max(REFACTOR_EVERY, 2 * m)
    status = 0
    while True:
        infeas = np.maximum(lo[head] - xB, xB - hi[head])
        cand = infeas > PRIMAL_TOL * (1.0 + np.abs(xB))
        if not cand.any():
            # optimal for the bounded problem. A nonbasic variable resting on an ARTIFICIAL bound with a zero
            # reduced cost does not make the LP unbounded (the objective does not care where it sits): move
            # it to its real bound once and let the dual simplex repair what that breaks.
            back = np.flatnonzero((stat != BASIC) & (np.abs(d) <= DUAL_TOL) & ~art_done &
                                  (((stat == AT_UPPER) & art_hi & np.isfinite(lo)) |
                                   ((stat == AT_LOWER) & art_lo & np.isfinite(hi))))
            if len(back):
                for j in back:
                    stat[j] = AT_LOWER if stat[j] == AT_UPPER else AT_UPPER
                    art_done[j] = True
                xB, _ = primal()
                continue
            status = 0
            break
        if pivots >= min(max_pivots, 50 * N + 1000):     # the cap ends a cycling node (no anti-cycling rule)
            status = 3
            break
        if since_factor >= refactor_every:
            wb = np.zeros(N, bool)
            wb[head] = True
            factor(wb)
            y, d = duals()
            xB, _ = primal()
            w = _weights(Binv) if dse else np.ones(m)
            since_factor = 0
            continue
        score = np.where(cand, infeas * infeas / w, -1.0)
        best = score.max()
        tied = np.flatnonzero(score >= best * (1.0 - TIE_REL))
        r = int(tied[np.argmin(head[tied])])
        below = xB[r] < lo[head[r]]                      # the leaving variable goes to its lower bound
        rho = Binv[r].copy()
        alpha_r = np.empty(N)
        alpha_r[:n] = _vecmat_rows(rho, A)
        alpha_r[n:] = -rho
        nb = stat != BASIC
        movable = lo < hi
        sa = -alpha_r if below else alpha_r              # x_Br must move against sa_j * (move of x_j)
        elig = nb & movable & (((stat == AT_LOWER) & (sa > PIV_TOL)) | ((stat == AT_UPPER) & (sa < -PIV_TOL)))
        cand_j = np.flatnonzero(elig)
        ratio = np.abs(d[cand_j]) / np.abs(alpha_r[cand_j])
        key = np.rint(ratio * RATIO_BIN)
        order = sorted(range(len(cand_j)), key=lambda k: (key[k], -abs(alpha_r[cand_j[k]]), cand_j[k]))
        slope = infeas[r]
        q = -1
        flips = []
        for k in order:
            j = int(cand_j[k])
            rng = hi[j] - lo[j]
            if bfrt and np.isfinite(rng):
                rest = slope - abs(alpha_r[j]) * rng
                if rest > PRIMAL_TOL * (1.0 + abs(xB[r])):
                    slope = rest
                    flips.append(j)
                    continue
            q = j
            break
        if q < 0:
            status = 1
            break
        aq = A[:, q] if q < n else -np.eye(m)[:, q - n]
        alpha_q = _matvec_cols(Binv, aq)
        if since_factor > 0 and abs(alpha_q[r] - alpha_r[q]) > pivot_mismatch * (1.0 + abs(alpha_r[q])):
            # the two ways to the pivot element disagree: refactorise and price again. Nothing of this
            # pivot is applied, the bound flips included: a flipped column would rest on the bound its
            # reduced cost says is wrong, and nothing after the refactorisation would move it back.
            since_factor = refactor_every
            refused += 1
            continue
        if flips:
            delta = np.zeros(N)
            for j in flips:
                delta[j] = (hi[j] - lo[j]) if stat[j] == AT_LOWER else (lo[j] - hi[j])
                stat[j] = AT_UPPER if stat[j] == AT_LOWER else AT_LOWER
            col = _matvec_cols(A, delta[:n]) - delta[n:]
            xB = xB - _matvec_cols(Binv, col)
            flips_total += len(flips)
        target = lo[head[r]] if below else hi[head[r]]
        theta_p = (xB[r] - target) / alpha_q[r]
        xB = xB - theta_p * alpha_q
        xq_new = (hi[q] if stat[q] == AT_UPPER else lo[q]) + theta_p
        theta_d = d[q] / alpha_r[q]
        d = d - theta_d * alpha_r
        leaving = head[r]
        d[leaving] = -theta_d
        d[q] = 0.0
        _update_inverse(Binv, alpha_q, r)
        stat[leaving] = AT_LOWER if below else AT_UPPER
        stat[q] = BASIC
        head[r] = q
        xB[r] = xq_new
        if dse:
            w = _weights(Binv)
        pivots += 1
        since_factor += 1

    # finish: fresh x_B (one refinement step), duals and reduced costs from the final inverse
    xB, rhs = primal()
    x_all = nonbasic_values()
    x_all[head] = xB
    resid = rhs.copy()                                  # rhs - B x_B: basic structurals in index order, then the slack
    for j in range(n):
        if stat[j] == BASIC:
            resid = resid - A[:, j] * x_all[j]
    resid = np.where(stat[n:] == BASIC, resid + x_all[n:], resid)
    xB = xB + _matvec_cols(Binv, resid)
    y, d = duals()
    x_all = nonbasic_values()
    x_all[head] = xB
    if status == 0:
        at_art = ((stat == AT_UPPER) & art_hi) | ((stat == AT_LOWER) & art_lo)
        if at_art.any() or (np.abs(x_all) >= 0.5 * BIG).any():
            status = 2
    obj = 0.0
    for j in range(n):
        obj = obj + cost[j] * x_all[j]
    return SimplexResult(status=status, objective=float(obj), x=x_all[:n].copy(), y=y.copy(), rc=d[:n].copy(),
                         col_status=stat[:n].copy(), row_status=stat[n:].copy(), pivots=pivots,
                         head=head.copy(), Binv=Binv, flips=flips_total, weights=w.copy(), refused=refused)
