"""Exact rational references for the NW permanent kernel (test infrastructure).

The kernel (permanent_kernel.cu) evaluates permanentExact by the Nijenhuis-Wilf / Ryser sum over Gray-code column
subsets of the ones-padded square matrix:

    perm(A) = (4(n&1) - 2) * sum_{i < 2^(n-1)} (-1)^i prod_j x_j(gray(i)),
    x_j(S)  = a[j, n-1] - rs_j / 2 + sum_{k in S} a[j, k],        rs_j = sum_k a[j, k].

On dense real input one missing, repeated or sign-flipped Gray step moves that sum by one term out of 2^(n-1), far
below any floating-point tolerance.  This module makes such errors visible:

* nw_range_exact(A, begin, end) is the partial sum over Gray indices [begin, end) as an exact Fraction -- what
  pda_permanent_range returns as hi + lo -- together with sum |terms|.
* perm_exact(A) is the exact permanent of an integer matrix (permanentExact semantics: for a rectangular matrix the
  sum over injective maps of the short side, which is perm(ones-padded) / (|rows - cols|)! exactly).
* exact_matrix(...) draws integer matrices on which the kernel has no rounding to do.  Every row has an odd sum and a
  small absolute row sum r_j, so every 2 x_j is an odd integer with |2 x_j| <= r_j: no NW term is ever zero, and
  every product is exact when prod r_j < 2^53.

  - "exact" regime, 2^(n-1) prod r_j < 2^53: every term and every partial sum, in any order, is a multiple of 2^-n
    below 2^53 * 2^-n.  The kernel's double-double sum then carries lo == 0 throughout and its result must equal
    perm_exact bit for bit.
  - "wide" regime, prod r_j < 2^53 and 2^(2(n-1)) prod r_j < 2^105: products are still exact, but the running sums
    round.  Every two-sum error, and every sum of them the kernel forms (lo), is then a multiple of 2^-n below
    2^(n-1) * ulp(2^(n-1) prod r_j 2^-n) <= 2^53 * 2^-n, so lo stays exact and hi + lo is the exact sum.  The kernel's
    result must be the correctly rounded exact permanent, and hi + lo of a range the exact partial sum; a lost lo
    shows.
"""
from __future__ import annotations

import itertools
import math
from fractions import Fraction

import numpy as np

EXACT_BITS = 53


def gray(i: int) -> int:
    return i ^ (i >> 1)


def _as_int_matrix(A) -> tuple[list[list[int]], int]:
    """A as integers times 2^-s (every finite double is dyadic)."""
    A = np.asarray(A, dtype=np.float64)
    s = 0
    for v in A.reshape(-1):
        if not np.isfinite(v):
            raise ValueError("non-finite entry")
        d = float(v).as_integer_ratio()[1]
        s = max(s, d.bit_length() - 1)
    return [[int(Fraction(float(v)) * (1 << s)) for v in row] for row in A], s


def _padded(A) -> tuple[list[list[int]], int, int]:
    """Ones-padded square of A (nwPerm.cpp:226-228) as integers times 2^-s, and s, n."""
    M, s = _as_int_matrix(A)
    rows = len(M)
    cols = len(M[0]) if rows else np.asarray(A).shape[1]
    n = max(rows, cols)
    one = 1 << s
    P = [[(M[j][k] if (j < rows and k < cols) else one) for k in range(n)] for j in range(n)]
    return P, s, n


def nw_range_exact(A, begin: int, end: int) -> tuple[Fraction, Fraction]:
    """NW partial sum over Gray indices [begin, end) of the ones-padded square of A, exactly, and sum |terms|.
    Multiply the first by (4(n&1) - 2) for the permanent of the padded square over the full range."""
    P, s, n = _padded(A)
    if n < 1 or not 0 <= begin <= end <= (1 << (n - 1)):
        raise ValueError("bad Gray range")
    den = 1 << (n * (s + 1))                       # term = prod_j (2 x_j 2^s) / 2^(n (s + 1))
    rs = [sum(r) for r in P]
    base2 = [2 * P[j][n - 1] - rs[j] for j in range(n)]  # 2 x_j of the empty subset, in units of 2^-s
    absrow = [sum(abs(v) for v in r) for r in P]         # |2 x_j| <= absrow_j
    bound = math.prod(absrow) if n else 1
    tot, tot_abs = 0, 0
    if bound < (1 << 62) and max(absrow, default=0) < (1 << 30):
        A2 = 2 * np.array(P, dtype=np.int64)[:, : n - 1]  # (n, n-1)
        b2 = np.array(base2, dtype=np.int64)
        chunk = int(max(1, min(1 << 16, (1 << 62) // max(bound, 1))))
        cols = np.arange(n - 1, dtype=np.uint64)
        for c0 in range(begin, end, chunk):
            idx = np.arange(c0, min(end, c0 + chunk), dtype=np.uint64)
            g = idx ^ (idx >> np.uint64(1))
            bits = ((g[:, None] >> cols[None, :]) & np.uint64(1)).astype(np.int64)
            Y = b2[None, :] + bits @ A2.T                # (len, n) int64, |Y| <= absrow
            prod = np.prod(Y, axis=1)
            sign = np.where((idx & np.uint64(1)) == 1, -1, 1).astype(np.int64)
            tot += int(np.sum(sign * prod))
            tot_abs += int(np.sum(np.abs(prod)))
    else:  # large entries: Python integers (slow, small ranges only)
        for i in range(begin, end):
            g = gray(i)
            p = 1
            for j in range(n):
                p *= base2[j] + 2 * sum(P[j][k] for k in range(n - 1) if (g >> k) & 1)
            tot += -p if i & 1 else p
            tot_abs += abs(p)
    return Fraction(tot, den), Fraction(tot_abs, den)


def perm_exact(A) -> int:
    """Exact permanentExact of an integer matrix: sum over injective maps of the short side into the long side of the
    products.  DP over used long-side lines as bitmasks with Python ints, short-side lines with the fewest nonzeros
    first; a long-side line that no later short-side line touches is dropped from the mask (its states merge)."""
    A = np.asarray(A)
    if A.size and not np.all(A == np.round(A)):
        raise ValueError("perm_exact takes integer matrices")
    M = [[int(v) for v in row] for row in (A if A.shape[0] <= A.shape[1] else A.T)]
    m = len(M)
    if m == 0:
        return 1
    nz = [[(k, v) for k, v in enumerate(row) if v] for row in M]
    order = sorted(range(m), key=lambda j: (len(nz[j]), j))
    last_use = {}
    for t, j in enumerate(order):
        for k, _ in nz[j]:
            last_use[k] = t
    f = {0: 1}
    for t, j in enumerate(order):
        g: dict[int, int] = {}
        dead = 0
        for k, _ in nz[j]:
            if last_use[k] == t:
                dead |= 1 << k
        for mask, val in f.items():
            for k, a in nz[j]:
                bit = 1 << k
                if mask & bit:
                    continue
                key = (mask | bit) & ~dead
                g[key] = g.get(key, 0) + val * a
        f = {k: v for k, v in g.items() if v}
        if not f:
            return 0
    return sum(f.values())


def perm_brute(A) -> int:
    """Sum over injective maps by enumeration (small matrices only)."""
    A = np.asarray(A)
    if A.shape[0] > A.shape[1]:
        A = A.T
    m, n = A.shape
    return sum(math.prod(int(A[i, p[i]]) for i in range(m)) for p in itertools.permutations(range(n), m))


def nw_factor(n: int) -> int:
    return 4 * (n & 1) - 2


def log2_budget(n: int, regime: str) -> float:
    """Largest sum of log2(r_j) a matrix of size n may have in the regime (strict upper bound)."""
    if regime == "exact":
        return EXACT_BITS - (n - 1)
    if regime == "wide":
        return min(EXACT_BITS, 2 * EXACT_BITS - 1 - 2 * (n - 1))
    raise ValueError(regime)


def regime_ok(A, regime: str) -> bool:
    """Every row sum odd and prod r_j inside the regime's budget."""
    A = np.asarray(A, dtype=np.int64)
    n = A.shape[0]
    if A.shape != (n, n) or n == 0:
        return False
    if np.any(A.sum(axis=1) % 2 == 0):
        return False
    r = np.abs(A).sum(axis=1)
    return sum(math.log2(int(v)) for v in r) < log2_budget(n, regime) - 1e-9


def _row(rng, r: int, first: int, n: int, signed: bool) -> dict[int, int]:
    """Integer entries with absolute sum r spread over at most three columns, one of them `first`."""
    parts = [r]
    if r > 1 and n > 1:
        k = int(rng.integers(1, min(3, r, n) + 1))
        if k > 1:
            cuts = sorted(rng.choice(np.arange(1, r), size=k - 1, replace=False).tolist())
            parts = [b - a for a, b in zip([0] + cuts, cuts + [r])]
    others = [c for c in rng.permutation(n).tolist() if c != first][: len(parts) - 1]
    row = {}
    for c, v in zip([first] + others, parts):
        row[c] = -v if (signed and rng.random() < 0.5) else v
    return row


def exact_matrix(rng, n: int, *, signed: bool = False, regime: str = "exact", rmax: int = 3) -> np.ndarray:
    """An n x n integer matrix in the regime (see the module docstring).  Row j has an odd absolute sum r_j <= rmax
    (r_j = 1 once the budget is spent) and a nonzero in column sigma(j) for a random permutation sigma, so every column
    is used; rows and columns come in random order."""
    if n == 0:
        return np.zeros((0, 0))
    budget = log2_budget(n, regime)
    sigma = rng.permutation(n)
    A = np.zeros((n, n), dtype=np.int64)
    spent = 0.0
    for j in rng.permutation(n).tolist():
        choices = [r for r in range(3, rmax + 1, 2) if spent + math.log2(r) < budget - 1e-9]
        r = int(rng.choice(choices)) if choices and rng.random() < 0.85 else 1
        spent += math.log2(r)
        for c, v in _row(rng, r, int(sigma[j]), n, signed).items():
            A[j, c] = v
    A = A[rng.permutation(n)][:, rng.permutation(n)]
    assert regime_ok(A, regime)
    return A.astype(np.float64)


def sum_abs_terms_bound(A) -> float:
    """2^(n-1) prod_j (r_j / 2) over the ones-padded square: a bound on sum |terms| that needs no walk."""
    P, s, n = _padded(A)
    return math.ldexp(float(math.prod(sum(abs(v) for v in r) for r in P)), n - 1 - n * (s + 1))


def nw_error_bound(A, exact) -> float:
    """Rigorous bound on |kernel - permanentExact| for any (ones-padded) input: each term is a product of n exactly
    formed factors (n - 1 roundings), the double-double sum adds at most a few roundings more, the NW factor 2 is exact
    and the rectangular division by k! rounds once more:
        4 (n + 2) 2^-53 * 2 sum|terms| / k!  +  2^-52 |permanent|."""
    A = np.asarray(A)
    n = max(A.shape)
    k = abs(A.shape[0] - A.shape[1])
    u = 2.0 ** -53
    return 4 * (n + 2) * u * 2 * sum_abs_terms_bound(A) / math.factorial(k) + 2 * u * abs(float(exact))


def nw_error_estimate(A, rng, per_k: int = 256) -> float:
    """Estimate (not a bound) of the kernel's error on a dense square matrix, for which neither an exact value nor a
    useful rigorous bound is affordable: 4 (n + 2) 2^-53 * 2 sum|terms|, with sum |terms| estimated by sampling
    per_k subsets of every size |S| = k and weighting each size by C(n-1, k).  On U(0,1) input the NW sum cancels
    (sum |terms| / perm grows like (e/2)^n), so this tracks the kernel's real accuracy where a fixed rtol cannot."""
    A = np.asarray(A, dtype=np.float64)
    n = A.shape[0]
    base = A[:, n - 1] - A.sum(axis=1) / 2
    tot = 0.0
    for k in range(n):
        idx = np.argsort(rng.random((per_k, n - 1)), axis=1)[:, :k]
        X = base[None, :] + A[:, idx].sum(axis=-1).T
        tot += math.comb(n - 1, k) * float(np.mean(np.abs(np.prod(X, axis=1))))
    return 4 * (n + 2) * 2.0 ** -53 * 2 * tot


def to_float(x) -> float:
    """Correctly rounded double of an int or Fraction."""
    return float(Fraction(x))
