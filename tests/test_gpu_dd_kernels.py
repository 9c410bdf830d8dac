"""GPU tests of the double-double Schur factorisation and solves (k_dd_potrf_tile, k_dd_trsm_tile, k_dd_syrk_tile in
csrc/ddlp.cuh, k_dd_trsv_multi / k_dd_trsv_fwd / k_dd_trsv_bwd in csrc/ddlp.cu, the row-block-cyclic factorisation of
csrc/dddist.cu) against Schur matrices whose factor is known exactly (tests/dd_exact.py), at every tile and launch shape: one to
132 tiles, ragged last tiles of width 1 to 32, one CTA solving several row tiles, the single-CTA solves, row blocks of 64 / 128
/ 256 rows on a one-rank communicator and over 2 and all visible GPUs.  The matrices go straight into the handle (lrn_dd_dbg_set_array), so no LP model is
needed and the reference costs O(n^2).  Also the Schur assembly, the residuals and find_mu against exact rational values."""
import ctypes as C
import math
from fractions import Fraction

import numpy as np
import pytest

import dd_exact as dx

pytestmark = pytest.mark.gpu
PD = C.POINTER(C.c_double)
PI = C.POINTER(C.c_int64)
LRN_ERR_STATE = -4
U2 = Fraction(1, 2 ** 106)                                 # unit roundoff of one double-double operation, squared u = 2^-53


@pytest.fixture(scope="module")
def lib(pkg):
    from loraine_jl_b200 import _lib
    L = _lib.lib()
    i32 = C.c_int32
    L.lrn_dd_dbg_set_array.restype = i32
    L.lrn_dd_dbg_set_array.argtypes = [C.c_void_p, i32, PD, PD]
    L.lrn_dd_dbg_set_trsv_ctas.restype = i32
    L.lrn_dd_dbg_set_trsv_ctas.argtypes = [C.c_void_p, i32]
    return L


def _dp(a):
    return a.ctypes.data_as(PD)


class Handle:
    """a lrn_dd handle driven through the C ABI: n multipliers, one LP row unless a model is loaded"""

    def __init__(self, lib, n, nlin=1, ngpus=1, world1=False):
        """ngpus > 1: lrn_dd_create_multi; world1: a one-rank NCCL communicator (the distributed path on one GPU)"""
        self.lib, self.n = lib, n
        self.h = C.c_void_p()
        if ngpus > 1 or world1:
            import torch  # noqa: F401  (loads the bundled libnccl into the process)
        if ngpus == 1:
            rc = lib.lrn_dd_create(C.byref(self.h), n, nlin, -1)
        else:
            rc = lib.lrn_dd_create_multi(C.byref(self.h), n, nlin, ngpus, None)
        assert rc == 0 and self.h.value
        if world1:
            buf = C.create_string_buffer(128)
            assert lib.lrn_dist_unique_id(buf) == 0
            assert lib.lrn_dd_dist_init(self.h, 0, 1, buf) == 0

    def close(self):
        if self.h:
            self.lib.lrn_dd_destroy(self.h)
            self.h = C.c_void_p()

    def call(self, name, *args):
        return getattr(self.lib, name)(self.h, *args)

    def set_array(self, which, x, lo):
        hi, lw = dx.dd_pair(np.asfortranarray(x, dtype=np.float64), lo)
        assert self.lib.lrn_dd_dbg_set_array(self.h, which, _dp(hi), _dp(np.asfortranarray(lw))) == 0

    def factor(self):
        return self.call("lrn_dd_schur_factor")

    def get(self, which, size):
        hi, lo = np.zeros(size), np.zeros(size)
        assert self.call("lrn_dd_get_array", which, _dp(hi), _dp(lo)) == 0
        return hi, lo

    def factor_L(self):
        """tril of L (the strict upper triangle is not part of the contract)"""
        hi, lo = self.get(2, self.n * self.n)
        return np.tril(hi.reshape(self.n, self.n, order="F")), np.tril(lo.reshape(self.n, self.n, order="F"))

    def solve(self, h, lo, which=3):
        self.set_array(5, h, lo)
        assert self.call("lrn_dd_schur_solve", which) == 0
        return self.get(6, self.n)


def _check_L(L, p, lo):
    worst = dx.factor_error(L[0], L[1], p, lo).max()
    assert worst <= 1.0, "L off L0 by %.3g x tolerance" % worst


def _check_y(y, p):
    worst = dx.solve_error(y[0], y[1], p).max()
    assert worst <= 1.0, "dely off y0 by %.3g x tolerance" % worst


def _same(a, b):
    return np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


# ---- the factor at tile edges -------------------------------------------------------------------------------------------
# 1, 2, 3 tiles (with and without the second-stream update of the rest), ragged last tiles of width 1, 31, 32; 4097 and
# 4200 have 129 and 132 tiles, more than the 128 CTAs of the multi-CTA solve
NS = [1, 2, 31, 32, 33, 63, 64, 65, 96, 97, 300, 1100, 4097, 4200]


@pytest.mark.parametrize("n,lo", [(n, lo) for n in NS for lo in (False, True)])
def test_factor_and_solve_match_the_exact_factor(lib, n, lo):
    """L = L0 (1 + t) and dely = y0 for the plain (E = 0) and the graded (E = 40) problem, and the graded results are the plain
    ones scaled by D and D^-1 bit for bit (solves with the production CTA count)"""
    h = Handle(lib, n)
    try:
        got = {}
        for E in (0, 40):
            p = dx.problem(n, E)
            h.set_array(1, p.H, lo)
            assert h.factor() == 0
            L = h.factor_L()
            _check_L(L, p, lo)
            y = h.solve(p.h, lo)
            _check_y(y, p)
            got[E] = (L, y, p.d)
        (L0, y0, _), (L40, y40, d) = got[0], got[40]
        assert _same(L40, (L0[0] * d[:, None], L0[1] * d[:, None]))
        assert _same(y40, (y0[0] / d, y0[1] / d))
    finally:
        h.close()


# ---- the solves at every launch shape -----------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [65, 97, 300, 1100])
@pytest.mark.parametrize("ctas", [0, 1, 2, 3, 7, -1])
def test_solves_at_every_launch_shape(lib, n, ctas):
    """lrn_dd_schur_solve with the single-CTA kernels (ctas = 0), with fewer CTAs than row tiles (one CTA solves several tiles
    and reuses its shared memory) and with the production count (-1): dely = y0, graded = plain scaled bit for bit, and
    which = 6 is bit for bit two which = 3 solves, the first dely loaded as the second right-hand side"""
    h = Handle(lib, n)
    try:
        assert lib.lrn_dd_dbg_set_trsv_ctas(h.h, ctas) == 0
        got = {}
        for E in (0, 40):
            p = dx.problem(n, E)
            h.set_array(1, p.H, True)
            assert h.factor() == 0
            y = h.solve(p.h, True)
            _check_y(y, p)
            got[E] = y
            y6 = h.solve(p.h, True, which=6)
            assert lib.lrn_dd_dbg_set_array(h.h, 5, _dp(y[0]), _dp(y[1])) == 0
            assert h.call("lrn_dd_schur_solve", 3) == 0
            assert _same(h.get(6, n), y6)
        d = dx.problem(n, 40).d
        assert _same(got[40], (got[0][0] / d, got[0][1] / d))
    finally:
        h.close()


def test_trsv_cta_hook_arguments(lib):
    h = Handle(lib, 40)
    try:
        assert lib.lrn_dd_dbg_set_trsv_ctas(h.h, -2) == -1
        assert lib.lrn_dd_dbg_set_trsv_ctas(h.h, 1 << 20) == 0      # clamped to what lrn_dd_create chose
        x = np.zeros(40)
        for which in (0, 2, 3, 4, 6):
            assert lib.lrn_dd_dbg_set_array(h.h, which, _dp(x), _dp(x)) == -1
        assert lib.lrn_dd_dbg_set_array(h.h, 1, None, None) == -1
        assert h.call("lrn_dd_schur_solve", 3) == LRN_ERR_STATE        # no factor yet
    finally:
        h.close()


# ---- pivot failure ------------------------------------------------------------------------------------------------------
def _fails_at(h, H, p, j, lo):
    """factor H: the failure must be reported at pivot j (LAPACK-style j + 1), and the failed factor must not be used"""
    h.set_array(1, H, lo)
    assert h.factor() == j + 1
    assert h.call("lrn_dd_schur_solve", 3) == LRN_ERR_STATE


@pytest.mark.parametrize("j", [0, 31, 32, 33, 295, 299])
def test_pivot_failure_index(lib, j):
    """n = 300 (ten tiles, the last one rows 288 .. 299): pivot j made negative (H_jj -= 2 L0_jj^2 -> pivot -L0_jj^2), a NaN on
    the diagonal at j, a NaN at (j, c) for c < j (it reaches pivot j first) all report j + 1; the unmodified H factors to L0
    on the same handle afterwards"""
    n, lo = 300, True
    p = dx.problem(n, 40)
    H = p.H.copy()
    h = Handle(lib, n)
    try:
        H[j, j] -= 2 * p.L0[j, j] ** 2
        _fails_at(h, H, p, j, lo)
        H[j, j] = p.H[j, j]
        h.set_array(1, H, lo)
        assert h.factor() == 0
        _check_L(h.factor_L(), p, lo)
        H[j, j] = np.nan
        _fails_at(h, H, p, j, lo)
        H[j, j] = p.H[j, j]
        for c in sorted({0, j // 2, j - 1}) if j > 0 else []:
            H[j, c] = H[c, j] = np.nan
            _fails_at(h, H, p, j, lo)
            H[j, c] = H[c, j] = p.H[j, c]
        h.set_array(1, H, lo)
        assert h.factor() == 0
        _check_L(h.factor_L(), p, lo)
        _check_y(h.solve(p.h, lo), p)
    finally:
        h.close()


# ---- several GPUs -------------------------------------------------------------------------------------------------------
def _visible_gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.parametrize("n", [300, 1100, 4200])
@pytest.mark.parametrize("gpus", ["world1", "two", "all"])
def test_distributed_factor_matches_the_exact_factor(lib, pkg, n, gpus):
    """The row-block-cyclic factorisation: row blocks of 64 / 128 / 256 rows (n = 4200: 17 blocks, the last one 104 rows, so
    with 8 GPUs the last steps have ranks that own no row).  world1: a one-rank communicator runs every step of it (diagonal
    block broadcast, padded all-gather, panel solves and trailing updates) on one GPU; two / all: lrn_dd_create_multi.  L
    equals the single-GPU L bit for bit and L0 to the tolerance, dely = y0; a pivot failure in block 1, in a block of the
    last rank and in the last block reports j + 1.  (A multi-GPU handle reports rank 0's index, which for blocks of other
    ranks arrives with the broadcast of the diagonal block.)"""
    if gpus == "world1":
        ng = 1
    else:
        ndev = _visible_gpus()
        if ndev < 2:
            pytest.skip("needs 2 GPUs")
        if gpus == "all" and ndev == 2:
            pytest.skip("only 2 GPUs visible: same as 'two'")
        ng = 2 if gpus == "two" else ndev
    lo = True
    p = dx.problem(n, 40)
    s = Handle(lib, n)
    try:
        s.set_array(1, p.H, lo)
        assert s.factor() == 0
        L1, y1 = s.factor_L(), s.solve(p.h, lo)
    finally:
        s.close()
    pw = pkg.dist.dd_block_rows(n)
    nblk = -(-n // pw)
    assert pw == {300: 64, 1100: 128, 4200: 256}[n]
    m = Handle(lib, n, ngpus=ng, world1=(gpus == "world1"))
    try:
        m.set_array(1, p.H, lo)
        assert m.factor() == 0
        L = m.factor_L()
        assert _same(L, L1)
        _check_L(L, p, lo)
        y = m.solve(p.h, lo)
        assert _same(y, y1)
        _check_y(y, p)
        H = p.H.copy()
        js = {pw + 5, (nblk - 1) * pw + 3, n - 1}
        if ng - 1 < nblk:
            js.add((ng - 1) * pw + pw // 2)
        for j in sorted(js):
            H[j, j] -= 2 * p.L0[j, j] ** 2
            _fails_at(m, H, p, j, lo)
            H[j, j] = p.H[j, j]
        m.set_array(1, H, lo)
        assert m.factor() == 0
        assert _same(m.factor_L(), L1)
    finally:
        m.close()


# ---- assembly, residuals and find_mu against exact rational values --------------------------------------------------------
def _dd_random(rng, hi):
    """normalised double-doubles with the given hi words and random lo words of about 2^-60 relative"""
    return hi, hi * np.ldexp(rng.uniform(-1, 1, size=hi.shape), -60)


def _F(hi, lo):
    return Fraction(float(hi)) + Fraction(float(lo))


def test_schur_assembly_and_residuals_are_exact_to_the_last_words(lib):
    """one LP, n = 300 multipliers, 360 LP rows: a dense LP column (299 entries: the j loop of k_dd_lp_schur strides), a
    multiplier row in 41 LP columns (the lanes of k_dd_spmv loop), a row with a single entry, non-zero lo words in C_lin, d,
    b, x and y, and s a power of two (w = x / s exact).  H, Rp and Rd against exact rationals."""
    n, m = 300, 360
    rng = np.random.default_rng(2026)
    others = [r for r in range(n) if r != 7]
    cols = [others]                                                      # dense column
    cols += [sorted({5} | set(rng.choice(others, 2, replace=False).tolist())) for _ in range(40)]
    cols.append([7, 100])                                                # row 7 has this single entry
    cols += [sorted(set(rng.choice(others, int(rng.integers(1, 5)), replace=False).tolist())) for _ in range(m - 42)]
    assert len(cols[0]) > 256 and sum(5 in c for c in cols) > 32 and sum(7 in c for c in cols) == 1
    colptr = np.cumsum([1] + [len(c) for c in cols]).astype(np.int64)
    rowval = np.array([r + 1 for c in cols for r in c], dtype=np.int64)
    nnz = len(rowval)
    c_hi, c_lo = _dd_random(rng, np.ldexp(rng.integers(1, 2 ** 20, size=nnz) * rng.choice([-1.0, 1.0], size=nnz), -10))
    d_hi, d_lo = _dd_random(rng, rng.uniform(-2, 2, size=m))
    b_hi, b_lo = _dd_random(rng, rng.uniform(-2, 2, size=n))
    x_hi, x_lo = _dd_random(rng, rng.uniform(0.5, 2, size=m))
    s_hi = np.ldexp(1.0, rng.integers(-3, 4, size=m))
    y_hi, y_lo = _dd_random(rng, rng.uniform(-1, 1, size=n))
    h = Handle(lib, n, nlin=m)
    try:
        assert h.call("lrn_dd_set_lin", colptr.ctypes.data_as(PI), rowval.ctypes.data_as(PI), _dp(c_hi), _dp(c_lo), _dp(d_hi),
                      _dp(d_lo)) == 0
        assert h.call("lrn_dd_set_b", _dp(b_hi), _dp(b_lo)) == 0
        assert h.call("lrn_dd_finalize") == 0
        assert h.call("lrn_dd_set_iterate", _dp(y_hi), _dp(y_lo), _dp(x_hi), _dp(x_lo), _dp(s_hi), None) == 0
        assert h.call("lrn_dd_residuals") == 0
        assert h.call("lrn_dd_schur_assemble") == 0
        Hh, Hl = h.get(1, n * n)
        Hh, Hl = Hh.reshape(n, n, order="F"), Hl.reshape(n, n, order="F")
        rp, rd = h.get(3, n), h.get(4, m)
    finally:
        h.close()
    assert np.array_equal(Hh, Hh.T) and np.array_equal(Hl, Hl.T)
    Cv = [_F(a, b) for a, b in zip(c_hi, c_lo)]
    w = [_F(x_hi[k], x_lo[k]) / Fraction(float(s_hi[k])) for k in range(m)]
    # H_ji (j >= i) = sum_k C_ik w_k C_jk.  Each term takes two double-double products (<= 6 u^2 relative each, u = 2^-53)
    # and each of the m - 1 sequential additions of k_dd_lp_schur adds <= 3 u^2 of the partial sum (the accurate
    # double-double sum): |error| <= (3 m + 12) u^2 sum |terms|, which is <= 2^-100 sum |terms| up to m = 17 terms.
    val, mag, cnt = {}, {}, {}
    for k, c in enumerate(cols):
        ents = [(r, Cv[colptr[k] - 1 + q]) for q, r in enumerate(c)]
        for a, (i, ci) in enumerate(ents):
            cw = ci * w[k]
            for j, cj in ents[a:]:
                t = cw * cj
                val[j, i] = val.get((j, i), 0) + t
                mag[j, i] = mag.get((j, i), 0) + abs(t)
                cnt[j, i] = cnt.get((j, i), 0) + 1
    lower = np.tril(np.ones((n, n), dtype=bool))
    nz = np.zeros((n, n), dtype=bool)
    for (j, i), v in val.items():
        nz[j, i] = True
        err = abs(_F(Hh[j, i], Hl[j, i]) - v)
        assert err <= (3 * cnt[j, i] + 12) * U2 * mag[j, i], (j, i, float(err / mag[j, i]))
    assert not Hh[lower & ~nz].any() and not Hl[lower & ~nz].any()
    # Rp = b - C x (k_dd_spmv by rows), Rd = d - s - C' y (by columns, then two subtractions).  A term: one product (6 u^2); the
    # additions it goes through: ceil(len / 32) in its lane, 5 in the warp sum and at most 2 more; with len <= 300 that is
    # (6 + 3 * 17) u^2 < 2^-100 of the sum of |terms| (b, d and s included).
    rows = [[] for _ in range(n)]
    for k, c in enumerate(cols):
        for q, r in enumerate(c):
            rows[r].append((k, Cv[colptr[k] - 1 + q]))
    tol = Fraction(1, 2 ** 100)
    for i in range(n):
        terms = [_F(b_hi[i], b_lo[i])] + [-cv * _F(x_hi[k], x_lo[k]) for k, cv in rows[i]]
        assert abs(_F(*[a[i] for a in rp]) - sum(terms)) <= tol * sum(abs(t) for t in terms), ("Rp", i)
    for k, c in enumerate(cols):
        terms = [_F(d_hi[k], d_lo[k]), -Fraction(float(s_hi[k]))]
        terms += [-Cv[colptr[k] - 1 + q] * _F(y_hi[r], y_lo[r]) for q, r in enumerate(c)]
        assert abs(_F(*[a[k] for a in rd]) - sum(terms)) <= tol * sum(abs(t) for t in terms), ("Rd", k)


@pytest.mark.parametrize("nlin", [1, 31, 32, 33, 1023, 1024, 1025, 5000])
def test_find_mu_against_the_exact_sum(lib, nlin):
    """mu = x's / nlin (k_dd_dot, one CTA of 1024 threads): terms from 1 to 2^40 that cancel in pairs down to ~2^-40 of their
    size, with lo words.  A term takes one product (6 u^2) and at most ceil(nlin / 1024) + 10 additions (its thread, then two
    warp sums), 3 u^2 each: <= 51 u^2 < 2^-100 of sum |terms| at nlin = 5000; the division by nlin adds < 2^-100 |mu|."""
    rng = np.random.default_rng(nlin)
    xh = np.ldexp(rng.uniform(1, 2, size=nlin), rng.integers(0, 41, size=nlin)) * rng.choice([-1.0, 1.0], size=nlin)
    sh = rng.uniform(0.5, 2, size=nlin)
    half = nlin // 2
    xh[half:2 * half] = -xh[:half]                                       # x_i s_i + x_i' s_i' = x_i (s_i - s_i')
    sh[half:2 * half] = sh[:half] * (1 + np.ldexp(rng.uniform(-1, 1, size=half), -40))
    xh, xl = _dd_random(rng, xh)
    sh, sl = _dd_random(rng, sh)
    h = Handle(lib, 1, nlin=nlin)
    try:
        colptr = np.arange(1, nlin + 2, dtype=np.int64)
        rowval = np.ones(nlin, dtype=np.int64)
        one = np.ones(nlin)
        assert h.call("lrn_dd_set_lin", colptr.ctypes.data_as(PI), rowval.ctypes.data_as(PI), _dp(one), None, _dp(one), None) == 0
        assert h.call("lrn_dd_set_b", _dp(np.ones(1)), None) == 0
        assert h.call("lrn_dd_finalize") == 0
        assert h.call("lrn_dd_set_iterate", _dp(np.zeros(1)), None, _dp(xh), _dp(xl), _dp(sh), _dp(sl)) == 0
        mu = np.zeros(2)
        assert h.call("lrn_dd_find_mu", _dp(mu)) == 0
    finally:
        h.close()
    terms = [_F(xh[i], xl[i]) * _F(sh[i], sl[i]) for i in range(nlin)]
    exact = sum(terms) / nlin
    tol = Fraction(1, 2 ** 100)
    assert abs(_F(mu[0], mu[1]) - exact) <= tol * sum(abs(t) for t in terms) / nlin + tol * abs(exact)
    if nlin >= 1000 and nlin % 2 == 0:
        assert abs(exact) < Fraction(1, 2 ** 20) * sum(abs(t) for t in terms) / nlin       # the cancellation is real
