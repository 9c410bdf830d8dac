"""The matrix-completion generator of the large CG-path tests (no GPU needed)."""
import numpy as np
import pytest

import mc_instances as mc


@pytest.mark.parametrize("r,c,k,n_obs,lp", [(12, 12, 1, 101, 0), (7, 9, 2, 40, 0), (20, 15, 3, 150, 6)])
def test_generator_invariants(r, c, k, n_obs, lp):
    inst = mc.matrix_completion(r, c, k, n_obs, seed=3, lp_rows=lp)
    m = r + c
    assert inst.n == n_obs and inst.bs == ([m] + ([-lp] if lp else []))
    assert np.linalg.matrix_rank(inst.M) == k and inst.M.shape == (r, c)
    # Omega: distinct entries, sorted, inside the matrix
    flat = inst.obs_i * c + inst.obs_j
    assert np.all(np.diff(flat) > 0) and flat.min() >= 0 and flat.max() < r * c
    np.testing.assert_array_equal(inst.c, inst.M[inst.obs_i, inst.obs_j])
    assert abs(inst.nuclear_norm - np.linalg.svd(inst.M, compute_uv=False).sum()) <= 1e-10 * inst.nuclear_norm
    b = inst.body
    psd = b[b[:, 1] == 1]
    f0 = psd[psd[:, 0] == 0]
    np.testing.assert_array_equal(f0[:, 2], np.arange(1, m + 1))
    np.testing.assert_array_equal(f0[:, 2], f0[:, 3])
    assert np.all(f0[:, 4] == -0.5)
    fe = psd[psd[:, 0] > 0]
    # one upper-triangle entry per constraint (two stored entries after symmetrisation): F_e = (E_{i,r+j} + E_{r+j,i}) / 2
    np.testing.assert_array_equal(fe[:, 0], np.arange(1, n_obs + 1))
    np.testing.assert_array_equal(fe[:, 2], inst.obs_i + 1)
    np.testing.assert_array_equal(fe[:, 3], r + inst.obs_j + 1)
    assert np.all(fe[:, 4] == 0.5) and np.all(fe[:, 2] < fe[:, 3])
    # y = 0 is strictly feasible: I/2 > 0; so is X = [a I  M~; M~' a I] with M~ = M on Omega, 0 elsewhere, for a > ||M~||
    Mt = np.zeros((r, c))
    Mt[inst.obs_i, inst.obs_j] = inst.M[inst.obs_i, inst.obs_j]
    a = np.linalg.norm(Mt, 2) + 1.0
    X = np.block([[a * np.eye(r), Mt], [Mt.T, a * np.eye(c)]])
    assert np.linalg.eigvalsh(X)[0] > 0
    # the optimum is attained by X* = [U S U'  M; M'  V S V'] (rank k): feasible, and -tr(X*)/2 = -||M||_*
    U, s, Vt = np.linalg.svd(inst.M, full_matrices=False)
    Xs = np.block([[U @ np.diag(s) @ U.T, inst.M], [inst.M.T, Vt.T @ np.diag(s) @ Vt]])
    assert np.linalg.eigvalsh(Xs)[0] >= -1e-9 * s[0] and np.linalg.matrix_rank(Xs, tol=1e-8 * s[0]) == k
    assert abs(-np.trace(Xs) / 2 - inst.optimum) <= 1e-10 * inst.nuclear_norm
    if lp:
        lpb = b[b[:, 1] == 2]
        assert np.all(lpb[lpb[:, 0] == 0][:, 4] == -1.0e3) and np.all(lpb[lpb[:, 0] > 0][:, 4] == 1.0)


def test_seed_reproducible():
    a, b = mc.matrix_completion(30, 20, 2, 300, seed=11), mc.matrix_completion(30, 20, 2, 300, seed=11)
    np.testing.assert_array_equal(a.body, b.body)
    np.testing.assert_array_equal(a.M, b.M)


def test_oracle_recovers_nuclear_norm():
    """kit = 0 NumPy oracle on a 12 x 12 rank-1 instance at 70 % sampling: exact recovery, the optimum is -||M||_*."""
    from oracle import loraine_oracle as lo, sdpa_io
    inst = mc.matrix_completion(12, 12, 1, round(0.7 * 144), seed=1)
    r = lo.solve_raw(sdpa_io.raw_from_sdpa_arrays(*inst.arrays), dict(kit=0, eDIMACS=1e-7, verb=0))
    assert r.status == 1
    assert abs(r.primal_obj - inst.optimum) <= 1e-6 * abs(inst.optimum)
    Y = r.X[0][:12, 12:]
    assert np.linalg.norm(Y - inst.M) <= 1e-5 * np.linalg.norm(inst.M)
