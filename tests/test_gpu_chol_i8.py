"""Ozaki INT8 trailing update of the Cholesky factorisation on the GPU: the tcgen05 kernel bit for bit against the NumPy model
(tests/chol_i8_model.py), and whole factorisations through the forced path against the DMMA path."""
import ctypes as C

import numpy as np
import pytest

import chol_i8_model as m

pytestmark = pytest.mark.gpu

PD = C.POINTER(C.c_double)


def dp(a):
    return a.ctypes.data_as(PD)


@pytest.fixture(scope="module")
def L(pkg):
    from loraine_jl_b200 import _lib
    lib = _lib.lib()
    lib.lrn_dbg_cholesky.argtypes = [C.c_int32, PD, PD, C.c_int32, C.POINTER(C.c_int32), C.c_int32, PD]
    yield lib
    lib.lrn_dbg_chol_int8(0)


def kernel_update(L, P, a_row0, b_row0, C0, row0=0, col0=0, lower=0):
    P = np.asfortranarray(P, dtype=np.float64)
    out = np.asfortranarray(C0.copy())
    M, N = out.shape
    sig = np.zeros(P.shape[0])
    rc = L.lrn_dbg_syrk_i8(P.shape[0], P.shape[1], dp(P), a_row0, b_row0, M, N, row0, col0, lower, dp(out), dp(sig), 0, None)
    assert rc == 0
    return out, sig


def expected(P, a_row0, b_row0, C0, row0=0, col0=0, lower=0):
    want = m.update(P, a_row0, b_row0, C0)
    return np.where(m.computed_tiles(*C0.shape, row0, col0, lower), want, C0)


def same_bits(a, b):
    return np.array_equal(a.view(np.int64), b.view(np.int64)) or np.array_equal(a, b, equal_nan=True)


@pytest.mark.parametrize("MN", [(1, 1), (63, 64), (64, 65), (65, 127), (127, 129), (129, 63), (1037, 1037)])
@pytest.mark.parametrize("K", [1, 31, 32, 512, 1000, 1024])
def test_kernel_bits_ragged(L, MN, K):
    M, N = MN
    if M * N * K > 1037 * 1037 * 32 and K != 1024:
        pytest.skip("large shapes are covered at K = 32 and K = 1024")
    rng = np.random.default_rng(M * 7 + N * 3 + K)
    rows = max(M, N)
    P = rng.standard_normal((rows, K))
    C0 = rng.standard_normal((M, N))
    got, sig = kernel_update(L, P, 0, 0, C0)
    assert same_bits(sig, m.row_scales(P))
    assert same_bits(got, expected(P, 0, 0, C0))


@pytest.mark.parametrize("a_row0,b_row0,M,N,row0,col0", [(1024, 1024, 700, 700, 0, 0), (0, 0, 1300, 256, 0, 0),
                                                         (8, 64, 500, 300, 64, 0), (0, 0, 300, 400, 0, 130)])
def test_kernel_bits_lower_offsets(L, a_row0, b_row0, M, N, row0, col0):
    rng = np.random.default_rng(a_row0 + M + col0)
    rows = max(a_row0 + M, b_row0 + N)
    P = rng.standard_normal((rows, 256))
    C0 = rng.standard_normal((M, N))
    got, _ = kernel_update(L, P, a_row0, b_row0, C0, row0, col0, 1)
    assert same_bits(got, expected(P, a_row0, b_row0, C0, row0, col0, 1))


def test_kernel_bits_exponents_zero_subnormal_nan_inf(L):
    rng = np.random.default_rng(11)
    rows, K = 200, 96
    P = rng.standard_normal((rows, K)) * 2.0 ** rng.integers(-200, 201, size=(rows, 1))
    P[5] = 0.0
    P[9] = rng.standard_normal(K) * 5e-324 * 1e3           # subnormal entries
    P[10, 7] = 3e-320
    P[17, 40] = np.nan
    P[23, 3] = np.inf
    P[31] = rng.uniform(0.996, 1.0, K) * 2.0 ** 100        # entries just below a power of two
    C0 = rng.standard_normal((rows, rows))
    got, _ = kernel_update(L, P, 0, 0, C0)
    want = expected(P, 0, 0, C0)
    assert same_bits(got, want)
    for r in (17, 23):
        assert np.isnan(got[r]).all() and np.isnan(got[:, r]).all()
    assert np.array_equal(got[5, :5], C0[5, :5])


def spd(n, seed, graded=False):
    import torch
    rng = np.random.default_rng(seed)
    G = torch.from_numpy(rng.standard_normal((n, n)) / np.sqrt(n)).to("cuda")
    A = (G @ G.T).cpu().numpy() + np.eye(n)
    A = (A + A.T) / 2
    if graded:
        d = 10.0 ** rng.uniform(-20, 20, n)
        A = A * d[:, None] * d[None, :]
    return np.asfortranarray(A)


def factor(L, A, mode, x=None, which=0):
    assert L.lrn_dbg_chol_int8(mode) == 0
    out = np.asfortranarray(A.copy())
    info = C.c_int32(-1)
    rc = L.lrn_dbg_cholesky(A.shape[0], dp(out), dp(x) if x is not None else None, which, C.byref(info), 0, None)
    L.lrn_dbg_chol_int8(0)
    assert rc == 0
    return out, info.value


def backward_error(A, Lf):
    import torch
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    At, Lt = torch.from_numpy(A).to(dev), torch.from_numpy(Lf).to(dev)
    R = torch.tril(At - Lt @ Lt.T)
    d = torch.sqrt(torch.diagonal(At))
    return float((R.abs() / (d[:, None] * d[None, :])).max())


@pytest.mark.parametrize("n,graded", [(2048, False), (2048, True), (5000, False), (5000, True), (20000, True)])
def test_forced_factorisation_matches_dmma_accuracy(L, n, graded):
    A = spd(n, n + graded, graded)
    b = np.random.default_rng(n).standard_normal(n)
    x8 = b.copy()
    L8, info8 = factor(L, A, 2, x8, 3)
    Ld, infod = factor(L, A, 0)
    assert info8 == 0 and infod == 0
    e8, ed = backward_error(A, L8), backward_error(A, Ld)
    assert e8 <= 1e-12 and e8 <= 4.0 * ed, (e8, ed)
    if n <= 5000 and not graded:                              # the tolerance of test_cholesky_and_solves
        xref = np.linalg.solve(A, b)
        assert np.linalg.norm(x8 - xref) <= 1e-11 * np.linalg.norm(xref)
    else:                                                     # scaled residual of the solve
        r = A @ x8 - b
        d = np.sqrt(np.diag(A))
        assert np.linalg.norm(r / d) <= 1e-11 * np.linalg.norm(d * x8) * np.sqrt(n)
    L8b, _ = factor(L, A, 2)
    assert np.array_equal(L8.view(np.int64), L8b.view(np.int64))          # deterministic


def test_natural_threshold_uses_int8_and_stays_accurate(L):
    """mode 1 (the Schur factor's default) takes the INT8 path at n >= 16384 and gives the same bits as the forced path."""
    n = 16384 + 1000
    A = spd(n, 3)
    L1, i1 = factor(L, A, 1)
    L2, i2 = factor(L, A, 2)
    assert i1 == 0 and i2 == 0
    assert np.array_equal(L1.view(np.int64), L2.view(np.int64))
    assert backward_error(A, L1) <= 1e-12


def test_forced_factorisation_info_bad_pivot_and_nan(L):
    n = 2048                                                  # panels of 256 columns
    A = spd(n, 5)
    bad = A.copy()
    bad[600, 600] = -1.0                                      # third panel
    _, info8 = factor(L, bad, 2)
    _, infod = factor(L, bad, 0)
    assert info8 == infod == 601
    nan = A.copy()
    nan[1500, 300] = np.nan                                   # lower triangle, second panel's columns
    _, info8 = factor(L, nan, 2)
    _, infod = factor(L, nan, 0)
    assert info8 == infod == 1501
