"""The NumPy model of the Ozaki INT8 Cholesky update (tests/chol_i8_model.py) against exact rational arithmetic: digit ranges,
the INT32 headroom of the level sums and the truncation bound.  No GPU needed."""
from fractions import Fraction

import numpy as np
import pytest

import chol_i8_model as m


def exact_digit_value(digits, s, i):
    return [Fraction(s[i]) * sum(Fraction(int(digits[t, i, k]), 128 ** (t + 1)) for t in range(m.PLANES))
            for k in range(digits.shape[2])]


def test_digits_fit_and_reconstruct():
    rng = np.random.default_rng(1)
    near = [1.0, 255 / 256, np.nextafter(255 / 256, 0), np.nextafter(1.0, 0), 0.5, np.nextafter(0.5, 1), 127.5 / 128]
    rows = [rng.standard_normal(40) * 2.0 ** rng.integers(-200, 200) for _ in range(12)]
    for v in near:
        r = rng.uniform(-1, 1, 40) * v
        r[3] = v
        r[7] = -v
        rows.append(r * 2.0 ** 37)
    rows.append(np.full(40, 5e-324))                      # subnormal row
    P = np.array(rows)
    digits, s = m.slice_rows(P)
    assert np.all(np.abs(digits[0].astype(int)) <= 127)
    assert np.all(np.abs(digits[1:].astype(int)) <= 64)
    for i in range(P.shape[0]):
        mx = np.max(np.abs(P[i]))
        assert mx <= s[i] * 255 / 256 and s[i] <= 2 * mx * 256 / 255
        rec = exact_digit_value(digits, s, i)
        for k in range(P.shape[1]):
            assert abs(Fraction(P[i, k]) - rec[k]) <= Fraction(s[i]) / 2 ** 57


def test_zero_nan_inf_rows():
    P = np.ones((4, 8))
    P[0] = 0.0
    P[1, 3] = np.nan
    P[2, 5] = -np.inf
    digits, s = m.slice_rows(P)
    assert s[0] == 0.0 and np.isnan(s[1]) and np.isnan(s[2]) and s[3] == 2.0
    assert not digits[:, :3].any()
    out = m.update(P, 0, 0, np.zeros((4, 4)))
    assert np.all(np.isnan(out[1])) and np.all(np.isnan(out[:, 2])) and np.all(out[0, [0, 3]] == 0.0)
    assert out[3, 3] == -8.0


def test_level_sums_fit_int32_at_k1024():
    """Worst case: |d_1| = 127 and |d_t| = 64 for t >= 2, all of one sign, K = 1024."""
    K = 1024
    d = np.empty((m.PLANES, 1, K), dtype=np.int8)
    d[0] = 127
    d[1:] = 64
    lv = m.level_sums(d, d)
    assert lv.max() < 2 ** 31
    assert 8 * 1024 * 127 ** 2 < 2 ** 31
    dn = -d
    assert m.level_sums(dn, d).min() > -2 ** 31


@pytest.mark.parametrize("K", [1, 7, 32, 45])
def test_update_error_bound_against_exact(K):
    """Truncation: |sum_l C_l 2^-7l sigma_i sigma_j - P_i . P_j| <= 1.5 * 2^-55 K sigma_i sigma_j (dropped digit pairs
    a + b >= 10: 7 * 2^-58 per k, plus 2 * 2^-57 from the digits beyond the eighth); the float64 fold then adds at most
    2^-52 of the exact digit sum."""
    rng = np.random.default_rng(K)
    rows = 9
    P = rng.standard_normal((rows, K)) * 2.0 ** rng.integers(-60, 60, size=(rows, 1))
    P[2] = rng.uniform(0.99, 1.0, K) * 2.0 ** 10            # rows whose entries sit just below a power of two
    P[3] = -P[2]
    digits, s = m.slice_rows(P)
    lv = m.level_sums(digits, digits)
    C0 = np.zeros((rows, rows))
    out = m.fold(lv, s, s, C0)
    for i in range(rows):
        for j in range(rows):
            exact = sum(Fraction(P[i, k]) * Fraction(P[j, k]) for k in range(K))
            digit_sum = Fraction(s[i]) * Fraction(s[j]) * sum(Fraction(int(lv[l, i, j]), 128 ** (l + 2)) for l in range(m.PLANES))
            assert abs(digit_sum - exact) <= Fraction(3, 2) * Fraction(K) * Fraction(s[i]) * Fraction(s[j]) / 2 ** 55
            assert abs(Fraction(-out[i, j]) - digit_sum) <= abs(digit_sum) / 2 ** 52


def test_computed_tiles_mask():
    mask = m.computed_tiles(300, 200, 0, 0, True)
    assert mask[:128, :64].all() and not mask[:128, 128:].any() and mask[128:256, 128:192].all()
    assert m.computed_tiles(10, 10, 0, 500, True).sum() == 0
    assert m.computed_tiles(10, 10, 0, 500, False).all()
