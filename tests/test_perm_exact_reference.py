"""CPU self-tests of the exact permanent references in tests/perm_exact.py (no GPU needed).  The GPU tests in
test_gpu_permanent_exact.py demand bit-for-bit agreement with these references, so the references themselves are
pinned here: against enumeration, against the cancellation-free DP of truth.py, against the CPU oracle's own NW walk
and against each other."""
import math
from fractions import Fraction

import numpy as np
import pytest

import perm_exact as pe
from truth import perm_injective


@pytest.mark.parametrize("signed", [False, True])
def test_perm_exact_matches_enumeration(signed):
    rng = np.random.default_rng(11 + signed)
    for n in range(0, 8):
        for _ in range(4):
            A = pe.exact_matrix(rng, n, signed=signed)
            assert pe.perm_exact(A) == pe.perm_brute(A)
    # rectangular: the sum over injective maps of the short side, either orientation, and dense integer entries
    for r, c in [(1, 4), (2, 5), (3, 6), (4, 7), (5, 3), (6, 2), (0, 3), (3, 0)]:
        A = rng.integers(-3 if signed else 0, 4, size=(r, c)).astype(np.float64)
        assert pe.perm_exact(A) == pe.perm_brute(A)
    assert pe.perm_exact(np.zeros((0, 0))) == 1


def test_perm_exact_matches_truth_and_oracle(oracle):
    rng = np.random.default_rng(5)
    # non-negative input: truth.perm_injective adds non-negative terms only (relative error ~ (m + n) ulp)
    for r, c in [(4, 4), (6, 9), (9, 6), (10, 12), (12, 12), (3, 20)]:
        A = rng.integers(0, 5, size=(r, c)).astype(np.float64)
        want = pe.perm_exact(A)
        assert abs(perm_injective(A) - want) <= 4 * (r + c) * 2.0 ** -53 * want
    # the oracle's NW walk is one running double: inside the exact regime it has nothing to round either
    for n in (1, 2, 5, 9, 12, 17, 20):
        for signed in (False, True):
            A = pe.exact_matrix(rng, n, signed=signed)
            got, st = oracle.permanent_exact(A)
            assert st == 0 and got == pe.perm_exact(A)


@pytest.mark.parametrize("regime", ["exact", "wide"])
def test_nw_range_exact_full_range_is_the_permanent(regime):
    rng = np.random.default_rng(23)
    for n in range(1, 17):
        for signed in (False, True):
            A = pe.exact_matrix(rng, n, signed=signed, regime=regime, rmax=3 if regime == "exact" else 15)
            total = 1 << (n - 1)
            s, s_abs = pe.nw_range_exact(A, 0, total)
            assert pe.nw_factor(n) * s == pe.perm_exact(A)
            assert s_abs <= pe.sum_abs_terms_bound(A)
            # any split adds up, whatever the cut points
            cuts = sorted({0, total, *rng.integers(0, total + 1, size=3).tolist()})
            assert sum(pe.nw_range_exact(A, a, b)[0] for a, b in zip(cuts, cuts[1:])) == s


def test_nw_range_exact_rectangular_and_dyadic():
    rng = np.random.default_rng(29)
    # ones-padded rectangle: full NW sum * factor / k! is the injective sum
    for r, c in [(2, 5), (5, 3), (4, 7)]:
        A = rng.integers(-2, 3, size=(r, c)).astype(np.float64)
        n, k = max(r, c), abs(r - c)
        s, _ = pe.nw_range_exact(A, 0, 1 << (n - 1))
        assert pe.nw_factor(n) * s / math.factorial(k) == pe.perm_exact(A)
    # dyadic entries scale out exactly: perm(A / 4) = perm(A) / 4^n
    A = pe.exact_matrix(rng, 6, signed=True)
    s, _ = pe.nw_range_exact(A / 4, 0, 32)
    assert pe.nw_factor(6) * s == Fraction(pe.perm_exact(A), 4 ** 6)
    # the Python-integer path (large entries) agrees with the vectorised one
    B = rng.integers(-(1 << 20), 1 << 20, size=(5, 5)).astype(np.float64)
    s, s_abs = pe.nw_range_exact(B, 3, 13)
    want = sum((-1) ** i * math.prod(Fraction(int(B[j, 4])) - Fraction(int(B[j].sum()), 2)
                                     + sum(int(B[j, k]) for k in range(4) if (pe.gray(i) >> k) & 1) for j in range(5))
               for i in range(3, 13))
    assert s == want


def test_nw_range_exact_far_into_the_range():
    """Starts near 2^31 at n = 32 (unsigned indices, no int64 overflow of the Gray code)."""
    rng = np.random.default_rng(31)
    A = pe.exact_matrix(rng, 32, signed=True)
    b = (1 << 31) - 5
    s, _ = pe.nw_range_exact(A, b, 1 << 31)
    P = A.astype(np.int64)
    want = Fraction(0)
    for i in range(b, 1 << 31):
        S = [k for k in range(31) if (pe.gray(i) >> k) & 1]
        x = [Fraction(int(P[j, 31])) - Fraction(int(P[j].sum()), 2) + sum(int(P[j, k]) for k in S) for j in range(32)]
        want += (-1) ** i * math.prod(x)
    assert s == want


@pytest.mark.parametrize("regime", ["exact", "wide"])
def test_generator_stays_in_its_regime(regime):
    rng = np.random.default_rng(37)
    for n in range(1, 33):
        for signed in (False, True):
            A = pe.exact_matrix(rng, n, signed=signed, regime=regime, rmax=3 if regime == "exact" else 31)
            assert pe.regime_ok(A, regime)
            Ai = A.astype(np.int64)
            assert np.all(Ai.sum(axis=1) % 2 != 0)                # every 2 x_j odd: no NW term is zero
            assert np.all(np.any(Ai != 0, axis=0))                # every column is flipped with effect
            r = np.abs(Ai).sum(axis=1)
            bits = sum(math.log2(int(v)) for v in r)
            if regime == "exact":
                assert (n - 1) + bits < 53                         # every partial sum is an exact double
            else:
                assert bits < 53 and 2 * (n - 1) + bits < 105
    # the regime test rejects what it must
    assert not pe.regime_ok(np.array([[2.0]]), "exact")                # even row sum: a zero term
    assert not pe.regime_ok(np.full((32, 32), 1.0) * np.eye(32) * 3, "exact")  # 2^31 * 3^32 > 2^53
    # and no term of a full walk is zero
    A = pe.exact_matrix(rng, 9, signed=True)
    for i in range(1 << 8):
        assert pe.nw_range_exact(A, i, i + 1)[1] > 0
