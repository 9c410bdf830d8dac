"""NumPy model of the Ozaki INT8 trailing update of the Cholesky factorisation (loraine.jl_b200/csrc/chol_i8.cu).

It performs the same float64 operations in the same order as the kernels, so the GPU result must match it bit for bit:
slicing into 8 int8 digit planes with per-row power-of-two scales, exact level sums (int64 here, exact int32 on the tensor
cores), then the fixed Horner fold."""
import numpy as np

PLANES = 8


def row_scales(P):
    """sigma_i = 2^e with max_k |P_ik| / sigma_i in [1/2, 255/256); 0 for a zero row, NaN for a row with a NaN or an Inf."""
    P = np.asarray(P, dtype=np.float64)
    bad = ~np.all(np.isfinite(P), axis=1)
    m = np.max(np.abs(np.where(np.isfinite(P), P, 0.0)), axis=1, initial=0.0)
    f, e = np.frexp(m)
    s = np.ldexp(1.0, np.where(f < 255.0 / 256.0, e, e + 1))
    s = np.where(m == 0.0, 0.0, s)
    return np.where(bad, np.nan, s)


def slice_rows(P):
    """(digits, sigma): digits[t] (t = 0..7) is the int8 plane of digit d_{t+1}, P_ik ~ sigma_i sum_t d_t 2^-7t."""
    P = np.asarray(P, dtype=np.float64)
    s = row_scales(P)
    live = s > 0.0                                     # False for zero and NaN rows
    with np.errstate(invalid="ignore", divide="ignore"):
        r = np.where(live[:, None], P / np.where(live, s, 1.0)[:, None], 0.0)
    digits = np.empty((PLANES,) + P.shape, dtype=np.int8)
    for t in range(PLANES):
        y = r * 128.0
        d = np.rint(y)
        r = y - d
        digits[t] = d.astype(np.int8)
    return digits, s


def level_sums(dA, dB):
    """C_l (l = 2..9, index l - 2) = sum_{a+b=l} dA_a dB_b^T, exact in int64."""
    A64, B64 = dA.astype(np.int64), dB.astype(np.int64)
    out = np.zeros((PLANES, dA.shape[1], dB.shape[1]), dtype=np.int64)
    for a in range(PLANES):
        for b in range(PLANES - a):
            out[a + b] += A64[a] @ B64[b].T
    return out


def fold(levels, sa, sb, C):
    """C - (acc 2^-14) (sigma_i sigma_j) with acc = C_9; acc = C_l + acc 2^-7 for l = 8..2 (float64, no fused operations)."""
    acc = levels[PLANES - 1].astype(np.float64)
    for l in range(PLANES - 2, -1, -1):
        acc = levels[l].astype(np.float64) + acc * 2.0 ** -7
    with np.errstate(invalid="ignore", over="ignore"):
        return C - (acc * 2.0 ** -14) * (sa[:, None] * sb[None, :])


def update(P, a_row0, b_row0, C):
    """C (M x N) - P[a_row0 + i] . P[b_row0 + j] the way the INT8 kernel computes it (all tiles)."""
    M, N = C.shape
    digits, s = slice_rows(P)
    dA, dB = digits[:, a_row0:a_row0 + M], digits[:, b_row0:b_row0 + N]
    return fold(level_sums(dA, dB), s[a_row0:a_row0 + M], s[b_row0:b_row0 + N], np.asarray(C, dtype=np.float64))


def computed_tiles(M, N, row0, col0, lower):
    """Boolean M x N mask of the entries the kernel writes: 128 x 64 tiles, lower mode skips tiles wholly above the diagonal."""
    mask = np.ones((M, N), dtype=bool)
    if lower:
        for bm in range(0, M, 128):
            for bn in range(0, N, 64):
                if row0 + bm + 127 < col0 + bn:
                    mask[bm:bm + 128, bn:bn + 64] = False
    return mask
