"""TEST INFRASTRUCTURE — numpy restatement of the device GMI cut kernel (k_simplex_gmi_cuts,
simple_mip_solver_b200/csrc/blp_simplex.cuh; C ABI blp_simplex_gmi_cuts_host).

What it computes is the reference's cut of a tableau row (``_find_gomory_cuts``, base_node.py:468-511, as
``BaseNode._gomory_cuts_of_basis`` states it with shifted / complemented nonbasics) followed by
``numerically_safe_cut(..., estimate='over')`` (floating_point.py:40). What is restated here is HOW the device
computes it, so that the kernel can be checked against this file BIT FOR BIT: every floating-point operation is
one rounded IEEE double operation (no fused multiply-add) and every sum runs in the kernel's fixed order:

  tableau row   structural j: sum over rows i ascending of Binv(r, i) a_ij, terms with Binv(r, i) = 0 skipped
                (k_simplex_tableau_rows, oracle/dual_simplex._vecmat_rows); slack n + i: -Binv(r, i)
  x-space       pi_j = pi_x(j) + (sum over rows i ascending of pi_s(i) a_ij, pi_s(i) = 0 skipped)
  right side    (1 + lane_dot(pi_x, offset)) + lane_dot(pi_s, b): LANES partial sums, lane t takes the terms
                t, t + LANES, ... in order, then the lane sums are added in lane order
  rounding      the continued-fraction convergents of get_fraction in doubles (a returned convergent is exact)

Only tests/ may import this module; the product never does.
"""
from __future__ import annotations

import numpy as np

from oracle.dual_simplex import BASIC, AT_UPPER, _vecmat_rows

LANES = 256                  # kGmiThreads: the kernel's block size
MAX_TERM = 1e3               # utils/tolerance.py
GOOD_EPS = 1e-2
EXACT_EPS = 1e-14
GMI_OK, GMI_NOT_BASIC, GMI_NONFINITE, GMI_ZERO = 0, 1, 2, 3


def get_fraction(x: float, est: int):
    """gmi_fraction: (numerator, denominator) as floats; est = +1 over, -1 under, 0 nearest."""
    x = np.float64(x)
    if abs(x) > MAX_TERM:
        return (np.ceil(x) if est > 0 else np.floor(x) if est < 0 else np.rint(x)), np.float64(1.0)
    h2, k2, h1, k1 = np.float64(0.0), np.float64(1.0), np.float64(1.0), np.float64(0.0)
    value = x
    last = 0
    with np.errstate(all='ignore'):
        while True:
            a = np.floor(value)
            h = a * h1 + h2
            k = a * k1 + k2
            if h > MAX_TERM or k > MAX_TERM:
                break
            rest = value - a
            if rest == 0.0:
                return h, k
            value = np.float64(1.0) / rest
            h2, k2, h1, k1 = h1, k1, h, k
            last += 1
    odd = last % 2 == 1
    if est > 0:
        if not odd:
            return h1, k1
        return (h2, k2) if last >= 2 else (np.ceil(x), np.float64(1.0))
    if est < 0:
        return (h1, k1) if odd else (h2, k2)
    return h1, k1


def safe_coef(coef: float) -> float:
    coef = np.float64(coef)
    n, d = get_fraction(coef, 1)
    if coef != 0.0 and abs(np.float64(1.0) - (n / d) / coef) > GOOD_EPS:
        n2, d2 = get_fraction(coef, 0)
        if abs(n2 / d2 - coef) < EXACT_EPS:
            n, d = n2, d2
    return float(n / d)


def safe_cut(pi: np.ndarray, pi0: float):
    """(pi, pi0, code) as the kernel's last step: scaled to unit max, rounded over / under."""
    pi = np.asarray(pi, dtype=np.float64)
    biggest = float(np.max(np.abs(pi))) if pi.size else 0.0
    if biggest == 0.0:
        return pi.copy(), float(pi0), GMI_ZERO
    factor = 1.0 / biggest
    out = np.array([safe_coef(c) for c in pi * factor])
    n, d = get_fraction(float(pi0) * factor, -1)
    return out, float(n / d), GMI_OK


def lane_dot(u: np.ndarray, w: np.ndarray) -> float:
    prod = np.asarray(u, dtype=np.float64) * np.asarray(w, dtype=np.float64)
    part = np.zeros(LANES)
    for s in range(0, len(prod), LANES):
        seg = prod[s:s + LANES]
        part[:len(seg)] = part[:len(seg)] + seg
    total = 0.0
    for v in part:
        total = total + float(v)
    return total


def gmi_cut(res, A, b, m_base: int, lb, ub, row_on, var: int, f0: float, col_is_int):
    """One request of blp_simplex_gmi_cuts_host. ``res``: the node's oracle.dual_simplex.SimplexResult (head,
    Binv, final status); ``A`` [m, n] dense with every pool row, ``b`` [m]; ``lb, ub`` the node's bounds as
    the solve had them; ``row_on`` [m] the rows its LP carries. Returns (pi [n], pi0, code)."""
    A = np.asarray(A, dtype=np.float64)
    m, n = A.shape
    stat = np.concatenate([res.col_status, res.row_status])
    lb, ub = np.asarray(lb, dtype=np.float64), np.asarray(ub, dtype=np.float64)
    nb = stat[:n] != BASIC
    off_x = np.where(stat[:n] == AT_UPPER, ub, lb)
    bad = bool((nb & (~np.isfinite(off_x) | (np.abs(off_x) >= 1e30))).any())
    pos = np.flatnonzero(res.head == var)
    if len(pos) == 0 or bad:
        return np.zeros(n), 0.0, (GMI_NOT_BASIC if len(pos) == 0 else GMI_NONFINITE)
    rho = res.Binv[int(pos[0])]
    f0 = float(f0)
    omf0 = 1.0 - f0
    # slacks: offset 0, sign +1, never integer; rows the node does not carry contribute nothing
    row_s = -rho * 1.0
    pis = np.where(row_s > 0.0, row_s / f0, -row_s / omf0)
    pis[stat[n:] == BASIC] = 0.0
    pis[~np.asarray(row_on, bool)] = 0.0
    # structurals
    sign = np.where(stat[:n] == AT_UPPER, -1.0, 1.0)
    off = np.where(nb, off_x, 0.0)
    row = _vecmat_rows(rho, A) * sign
    with np.errstate(all='ignore'):
        f = row - np.floor(row)
        p_int = np.where(f <= f0, f / f0, (1.0 - f) / omf0)
        p_cont = np.where(row > 0.0, row / f0, -row / omf0)
    is_int = np.asarray(col_is_int, bool) & (np.abs(off - np.rint(off)) <= 1e-9)
    px = np.where(is_int, p_int, p_cont) * sign
    px[~nb] = 0.0
    coef = px + _vecmat_rows(pis, A)
    rhs = (1.0 + lane_dot(px, off)) + lane_dot(pis, b)
    if not (np.isfinite(coef).all() and np.isfinite(rhs)):
        return np.zeros(n), 0.0, GMI_NONFINITE
    return safe_cut(coef, rhs)
