"""Host helpers of the own-rows layout of the kit = 0 Schur matrix (loraine_jl_b200.dist, mirroring RowOwner::local and
local_rows in csrc/ops.cuh and the footprint in csrc/solver.cu / csrc/dist.cu) against brute-force enumeration, and a NumPy
restatement of the fan-out forward / fan-in backward triangular solves over emulated ranks."""
import numpy as np
import pytest
import scipy.linalg as sl


@pytest.fixture(scope="module")
def dist(pkg):
    return pkg.dist


def _enumerate(n, pw, rank, world):
    """global rows of `rank`, in the order the own-rows layout stacks them"""
    return [r for r in range(n) if world <= 1 or (r // pw) % world == rank]


@pytest.mark.parametrize("world", range(1, 9))
@pytest.mark.parametrize("n,pw", [(1, 64), (21, 8), (104, 64), (300, 128), (1100, 128), (5000, 256), (17001, 512), (1024, 512),
                                  (2048, 256)])
def test_local_rows_and_index_against_enumeration(dist, world, n, pw):
    seen = np.zeros(n, dtype=int)
    for rank in range(world):
        rows = _enumerate(n, pw, rank, world)
        assert dist.local_rows(n, pw, rank, world) == len(rows)
        for i, r in enumerate(rows):
            assert dist.row_owner(r, pw, world) == rank
            assert dist.local_row(r, pw, world) == i
            seen[r] += 1
    assert (seen == 1).all()


def test_ranks_without_rows_and_ragged_last_block(dist):
    assert dist.local_rows(300, 128, 3, 4) == 0                # 3 blocks, rank 3 holds none
    assert dist.local_rows(300, 128, 2, 4) == 300 - 256          # the ragged last block
    assert dist.local_rows(104, 128, 1, 2) == 0


@pytest.mark.parametrize("world", [1, 2, 3, 8])
@pytest.mark.parametrize("n,pw", [(300, 128), (17001, 512), (140000, 512)])
def test_footprint_of_both_layouts(dist, world, n, pw):
    nblk = -(-n // pw)
    for rank in range(world):
        rows = len(_enumerate(n, pw, rank, world)) if n < 20000 else dist.local_rows(n, pw, rank, world)
        ld = -(-max(rows, 1) // 8) * 8
        want = 2 * ld * n * 8 + (4 * (-(-n // 8) * 8) * pw + nblk * pw * pw + pw) * 8
        assert dist.schur_bytes(n, pw, rank, world, True) == want
        assert dist.schur_bytes(n, pw, rank, world, False) == 2 * (-(-n // 8) * 8) * n * 8
    if world == 2 and n == 140000:
        # two ranks: H and L of rank 0 (137 blocks of 512 rows) 157.1 GB, the extras 2.87 GB (4 panel slots 2.29 GB + 274 stored inverses 0.57 GB)
        extra = dist.schur_bytes(n, pw, 0, 2, True) - 2 * dist.local_rows(n, pw, 0, 2) * n * 8
        assert 2.86e9 < extra < 2.88e9
        assert 157.0e9 < 2 * dist.local_rows(n, pw, 0, 2) * n * 8 < 157.2e9


def _solve_dist(L, b, pw, world):
    """fan-out forward and fan-in backward solves with L split into the ranks' own row blocks (L' x = y with y = L^-1 b)"""
    n = L.shape[0]
    nblk = -(-n // pw)
    own = [np.array([r for r in range(n) if (r // pw) % world == k], dtype=int) for k in range(world)]
    Lr = [L[o, :] for o in own]                                  # each rank's rows only
    X = [np.linalg.inv(L[p * pw:(p + 1) * pw, p * pw:(p + 1) * pw]) for p in range(nblk)]
    xs = [b.copy() for _ in range(world)]                        # every rank's copy of the right-hand side
    for p in range(nblk):
        c0, c1 = p * pw, min(n, (p + 1) * pw)
        owner = p % world
        y = X[p] @ xs[owner][c0:c1]
        for k in range(world):                                    # broadcast, then each rank updates its rows below block p
            xs[k][c0:c1] = y
            sel = own[k] >= c1
            xs[k][own[k][sel]] -= Lr[k][sel, c0:c1] @ y
    y = xs[0].copy()
    assert all(np.array_equal(v, y) for v in xs)
    x = [y.copy() for _ in range(world)]
    for p in reversed(range(nblk)):
        c0, c1 = p * pw, min(n, (p + 1) * pw)
        s = np.zeros(c1 - c0)
        for k in range(world):                                    # all-reduce of the partial sums of segment p
            sel = own[k] >= c1
            s += Lr[k][sel, c0:c1].T @ x[k][own[k][sel]]
        for k in range(world):
            x[k][c0:c1] = X[p].T @ (x[k][c0:c1] - s)
    assert all(np.array_equal(v, x[0]) for v in x)
    return y, x[0]


@pytest.mark.parametrize("world", [1, 2, 3, 5])
@pytest.mark.parametrize("n,pw", [(37, 8), (130, 16), (64, 64), (200, 32)])
def test_fan_out_fan_in_solves_match_solve_triangular(world, n, pw):
    rng = np.random.default_rng(n * 10 + world)
    A = rng.standard_normal((n, n))
    L = np.linalg.cholesky(A @ A.T + n * np.eye(n))
    b = rng.standard_normal(n)
    y, x = _solve_dist(L, b, pw, world)
    y_ref = sl.solve_triangular(L, b, lower=True)
    x_ref = sl.solve_triangular(L.T, y_ref, lower=False)
    assert np.linalg.norm(y - y_ref) <= 1e-12 * np.linalg.norm(y_ref)
    assert np.linalg.norm(x - x_ref) <= 1e-12 * np.linalg.norm(x_ref)
