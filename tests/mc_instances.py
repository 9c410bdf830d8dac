"""Seeded nuclear-norm matrix-completion SDPs: a model with a known optimum and a low-rank solution at any number of
constraints, which is what the CG path (kit = 1) with the H_alpha preconditioner is for.

M = P Q' (r x c, rank k, Gaussian factors) is observed on a uniform sample Omega of its entries.  In SDPA form, with one
PSD block of side m = r + c:
    variables   y_e, one per observed entry e = (i, j)
    F_e         = (E_{i, r+j} + E_{r+j, i}) / 2          (two stored entries)
    F_0         = -I / 2,   c_e = M_ij
so the primal is  min sum_e M_ij y_e  s.t.  I/2 + sum_e y_e F_e >= 0  and the dual is
    max -tr(X)/2  s.t.  X = [W1 Y; Y' W2] >= 0,  Y_ij = M_ij on Omega.
When nuclear-norm minimisation recovers M exactly, both optima are -||M||_* and the optimal X has rank k (Y = M).
Both sides are strictly feasible: y = 0, and X = [a I  M~; M~' a I] for large a.

`lp_rows > 0` appends a diagonal (LP) block of the bounds y_e >= -lp_bound for the first lp_rows entries; with a loose
bound it does not change the optimum.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np


@dataclass
class MCInstance:
    n: int                  # number of constraints (observed entries)
    bs: list                # SDPA block sizes
    c: np.ndarray           # objective (M on Omega)
    body: np.ndarray        # SDPA entries [k, blk, i, j, v], 1-based, upper triangle
    M: np.ndarray           # the r x c matrix
    obs_i: np.ndarray       # row of each observed entry (0-based)
    obs_j: np.ndarray       # column of each observed entry (0-based)
    nuclear_norm: float     # ||M||_*

    @property
    def arrays(self):
        return self.n, self.bs, self.c, self.body

    @property
    def optimum(self):
        return -self.nuclear_norm


def matrix_completion(r, c, k, n_obs, seed=0, lp_rows=0, lp_bound=1.0e3):
    rng = np.random.default_rng(seed)
    P = rng.standard_normal((r, k))
    Q = rng.standard_normal((c, k))
    M = P @ Q.T
    flat = np.sort(rng.choice(r * c, size=n_obs, replace=False))
    oi, oj = flat // c, flat % c
    # ||P Q'||_* from the k x k core: P = U_P R_P, Q = U_Q R_Q  ->  singular values of R_P R_Q'
    nuc = float(np.linalg.svd(np.linalg.qr(P)[1] @ np.linalg.qr(Q)[1].T, compute_uv=False).sum())
    m = r + c
    d = np.arange(1, m + 1)
    e = np.arange(1, n_obs + 1)
    parts = [np.column_stack([np.zeros(m), np.ones(m), d, d, np.full(m, -0.5)]),
             np.column_stack([e, np.ones(n_obs), oi + 1, r + oj + 1, np.full(n_obs, 0.5)])]
    bs = [m]
    if lp_rows > 0:
        t = np.arange(1, lp_rows + 1)
        parts.append(np.column_stack([np.zeros(lp_rows), np.full(lp_rows, 2), t, t, np.full(lp_rows, -lp_bound)]))
        parts.append(np.column_stack([t, np.full(lp_rows, 2), t, t, np.ones(lp_rows)]))
        bs.append(-lp_rows)
    body = np.concatenate(parts).astype(np.float64)
    return MCInstance(n=n_obs, bs=bs, c=M[oi, oj].copy(), body=body, M=M, obs_i=oi, obs_j=oj, nuclear_norm=nuc)
