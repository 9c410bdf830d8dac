"""CPU checks of the exactly factorable Schur matrices of tests/dd_exact.py: the construction is exact, the float64 products
stay below 2^53, and the (hi, lo) pairs loaded into the library are normalised double-doubles."""
from fractions import Fraction

import mpmath as mp
import numpy as np
import pytest

import dd_exact as dx

LARGEST_N = 4200                                            # the largest n of tests/test_gpu_dd_kernels.py


@pytest.mark.parametrize("E", [0, 40])
def test_h_is_l0_l0t_exactly(E):
    """with Python integers: H = L0 L0' and H y0 = h hold exactly at n = 40"""
    n = 40
    p = dx.problem(n, E)
    A = [[int(v) for v in row] for row in np.ldexp(p.L0, p.e[:, None])]       # back to the integers of A
    assert all(A[i][i] == 2 ** 17 for i in range(n)) and all(A[i][k] == 0 for i in range(n) for k in range(i + 1, n))
    for i in range(n):
        for k in range(n):
            exact = Fraction(sum(A[i][m] * A[k][m] for m in range(n)), 2 ** int(p.e[i] + p.e[k]))
            assert Fraction(float(p.H[i, k])) == exact, (i, k)
        assert Fraction(float(p.L0[i, i])) == Fraction(2 ** 17, 2 ** int(p.e[i]))
    for i in range(n):
        assert sum(Fraction(float(p.H[i, k])) * Fraction(float(p.y0[k])) for k in range(n)) == Fraction(float(p.h[i]))


def test_integer_products_stay_below_2_53():
    """at the largest n every partial sum of P = A A', A' z and A (A' z) is an integer below 2^53: exact in any order"""
    bP, bh, bz = dx.bounds(LARGEST_N)
    assert max(bP, bh, bz) < 2.0 ** 53
    p = dx.problem(LARGEST_N, 40)
    assert np.all(np.diag(p.L0) == np.ldexp(2.0 ** 17, -p.e))
    # A is diagonally dominant with a margin: the off-diagonal row sums are at most 8 (n - 1) < 2^17
    assert 8 * (LARGEST_N - 1) < 2 ** 17


def test_lo_words_are_normalised():
    """(H, H 2^-60): |lo| <= ulp(hi) / 2, so hi + lo rounds to hi; the same for h.  T_LO is sqrt(1 + 2^-60) - 1"""
    p = dx.problem(300, 40)
    for x in (p.H, p.h):
        hi, lo = dx.dd_pair(x, True)
        assert np.all(np.abs(lo) <= np.spacing(np.abs(hi)) / 2)
        assert np.array_equal(hi + lo, hi)
        assert np.abs(lo[hi != 0]).min() > 0
    with mp.workprec(256):
        assert abs((1 + mp.mpf(dx.T_LO)) ** 2 - (1 + mp.mpf(2) ** -60)) < mp.mpf(2) ** -110
    assert dx.T_LO > 4e-19


def test_graded_problem_is_the_plain_one_scaled():
    """E = 40 is E = 0 scaled by D on both sides: the bit-identity the GPU test relies on starts from identical integers"""
    a, b = dx.problem(97, 0), dx.problem(97, 40)
    assert b.e.max() > 30 and np.array_equal(a.y0, np.ldexp(b.y0, -b.e))
    assert np.array_equal(b.L0, a.L0 * b.d[:, None]) and np.array_equal(b.H, a.H * b.d[:, None] * b.d[None, :])
