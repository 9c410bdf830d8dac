"""Schur matrices whose double-double Cholesky factor is known exactly (plain NumPy; used by tests/test_gpu_dd_kernels.py and
pinned on the CPU by tests/test_dd_exact_cpu.py).

A is lower triangular with integer entries: the diagonal is 2^17, the strict lower part is uniform in [-8, 8].  D = diag(2^-e_i)
with integers e_i in [0, E].  Then L0 = D A and H = L0 L0' are exact doubles:
  * P = A A' is a float64 product of integer matrices whose partial sums stay below 2^53 (checked by bounds()), so it is
    exact in any summation order, with or without FMA;
  * H_ik = P_ik 2^(-e_i - e_k) is a power-of-two scaling of an exact double;
  * chol(H) = L0 exactly, because the Cholesky factor is unique.
The right-hand side: z has integer entries in [-2^10, 2^10], y0 = D^-1 z and h = D (A (A' z)), again exact, so H y0 = h.

Non-zero lo words: (H, H 2^-60) is a normalised double-double of H (1 + 2^-60), whose factor is L0 sqrt(1 + 2^-60) =
L0 + L0 t with t = sqrt(1 + 2^-60) - 1; loading h the same way keeps the solution y0.  A kernel that drops a lo word is off
by about t = 4e-19 relative, far above the tolerances of the tests.

Well conditioned at every size used: the off-diagonal row and column sums of A are at most 8 (n - 1) < 2^17 for n < 16384, so
A = 2^17 (I + N) with ||N|| <= 8 (n - 1) / 2^17 (0.26 at n = 4200) and cond(A) <= 1.7.  Errors of the double-double
factorisation and solves then stay at a small multiple of n 2^-104 relative to each row's scale (the tolerances below).

Scaling by powers of two commutes with every double-double operation as long as nothing overflows or underflows, so the
graded problem (E = 40) is factored and solved with exactly the rounding of the plain one (E = 0): its L equals D L(E = 0) and
its dely equals D^-1 dely(E = 0) bit for bit.
"""
from functools import lru_cache
from types import SimpleNamespace

import mpmath as mp
import numpy as np

DIAG = 2.0 ** 17
OFF = 8
ZMAX = 2 ** 10
LO_SCALE = 2.0 ** -60
with mp.workprec(256):
    T_LO = float(mp.sqrt(1 + mp.mpf(2) ** -60) - 1)        # L0 sqrt(1 + 2^-60) = L0 + L0 T_LO

# |error_ij| <= TOL_L max_k |L0_ik| for the factor, |error_i| <= TOL_Y 2^e_i ||z||_inf for dely.  Both from n 2^-104
# (= 2.1e-28 at the largest n = 4200, about 2^-106 per double-double operation along the longest dependent chain of n
# multiply-adds): TOL_L = 1e-27 is five times that bound, TOL_Y = 1e-26 adds the two triangular solves (another n 2^-104
# each) and cond(A)^2 <= 3 of the equilibrated problem on top.  Dropping a lo word costs about 4e-19, eight orders above.
TOL_L = 1e-27
TOL_Y = 1e-26


@lru_cache(maxsize=2)
def _base(n, seed):
    rng = np.random.default_rng(seed)
    A = np.tril(rng.integers(-OFF, OFF + 1, size=(n, n)).astype(np.float64), -1)
    A[np.diag_indices(n)] = DIAG
    z = rng.integers(-ZMAX, ZMAX + 1, size=n).astype(np.float64)
    P = A @ A.T                                             # exact: integer partial sums below 2^53
    hp = A @ (A.T @ z)                                      # exact as well (bounds())
    return A, P, z, hp


def problem(n, E, seed=None):
    """The exact problem of size n and grading E: L0 (lower), H (full, symmetric), h, y0, the exponents e and ||z||_inf."""
    seed = 1000 + n if seed is None else seed
    A, P, z, hp = _base(n, seed)
    e = np.random.default_rng(seed + 7).integers(0, E + 1, size=n) if E > 0 else np.zeros(n, dtype=np.int64)
    d = np.ldexp(1.0, -e)                                   # D, exact powers of two
    return SimpleNamespace(n=n, E=E, e=e, d=d, L0=A * d[:, None], H=P * d[:, None] * d[None, :], h=hp * d, y0=z / d,
                           zinf=float(np.abs(z).max()))


def dd_pair(x, lo):
    """(hi, lo) of x (lo = False) or of x (1 + 2^-60) (lo = True), as float64 arrays in x's memory order"""
    return x, (x * LO_SCALE if lo else np.zeros_like(x))


def factor_error(Lhi, Llo, p, lo):
    """entrywise error of a double-double factor (lower triangles) against L0 (1 + T_LO), scaled by the row tolerance;
    computed in float64 as (L_hi - L0) + (L_lo - L0 t), both differences far below the tolerance in rounding"""
    t = T_LO if lo else 0.0
    err = (np.tril(Lhi) - p.L0) + (np.tril(Llo) - p.L0 * t)
    return np.abs(err) / (TOL_L * np.abs(p.L0).max(axis=1))[:, None]


def solve_error(yhi, ylo, p):
    """entrywise error of a double-double dely against y0, scaled by its tolerance"""
    return np.abs((yhi - p.y0) + ylo) / (TOL_Y * p.zinf / p.d)


def bounds(n, seed=None):
    """largest partial sum (in absolute value) of the integer products behind P = A A' and h = A (A' z)"""
    A, _, z, _ = _base(n, 1000 + n if seed is None else seed)
    Aa = np.abs(A)
    return float((Aa @ Aa.T).max()), float((Aa @ (Aa.T @ np.abs(z))).max()), float((Aa.T @ np.abs(z)).max())
