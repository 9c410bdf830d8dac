// State of the double-double LP path (ddlp.cu) and the Cholesky tile arithmetic shared by the single-GPU factorisation
// (ddlp.cu) and the row-block-cyclic multi-GPU one (dddist.cu).  Both run the same tile bodies in the same order, so the
// factor of a sharded handle equals the single-GPU factor bit for bit.
#pragma once
#include "common.cuh"
#include "dd.cuh"
#include "../../include/loraine_b200.h"
#include "../../include/loraine_b200_dd.h"
#include <algorithm>

struct lrn_dd_solver {
    int device = 0;
    cudaStream_t st = nullptr, st2 = nullptr;
    cudaEvent_t evP = nullptr, evR = nullptr;
    std::string err;
    int n = 0, nlin = 0;
    long long nnz = 0;
    // C_lin by LP column (CSC) and by multiplier row (CSR): the transposed product and the Schur rows each want one of them
    lrn::DevBuf<int> cptr, cidx, rptr, ridx;
    lrn::DevBuf<lrn::dd> cval, rval;
    lrn::DevBuf<lrn::dd> d, b, x, s, si, y, rp, rd, rhs, dely, dx, ds, xn, sn, rnt, w, tl, tn;
    lrn::DevBuf<lrn::dd> H, L, red, rdiag;
    lrn::DevBuf<int> info, flags;      // info[0]: Cholesky pivot, info[1]: time-out of the flag wait in the multi-CTA solves
    int trsv_ctas = 0, trsv_ctas_max = 0, trsv_epoch = 0;     // (trsv_ctas_max: the lrn_dd_create value)
    bool have_lin = false, have_b = false, finalized = false, have_iterate = false, have_H = false, have_factor = false;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    double t_ms[4] = {0, 0, 0, 0};
    // ---- multi-GPU (dddist.cu) ----------------------------------------------------------------------------------------------
    // Row-block-cyclic ownership of the Schur rows: row block g (height pw) belongs to rank g % world.  world > 1 or a
    // communicator makes the handle "sharded": the assembly writes the rank's own rows of the lower triangle only and the
    // factorisation runs the distributed Cholesky.  H and L stay full n x n on every rank.
    int rank = 0, world = 1, pw = 64;
    void* nccl = nullptr;              // lrn::DistCtx* (lrn_dd_dist_init / lrn_dd_create_multi)
    void* group = nullptr;             // lrn::GroupOf<lrn_dd_solver>*: facade of an in-process group (lrn_dd_create_multi)
    bool H_gathered = false;           // the row shards of H have been summed over the ranks (lrn_dd_get_array(1))
    lrn::DevBuf<lrn::dd> xb, sendbuf, recvbuf;   // factorisation: broadcast diagonal block, solved row blocks mine / all
    lrn::DevBuf<int> tiles;            // my 32-row tiles, increasing
};

namespace lrn {

// height of a row block of the dd Schur distribution (mirrored by dist.dd_block_rows)
inline int dd_block_rows(long long n) { return n >= 4096 ? 256 : (n >= 1024 ? 128 : 64); }
inline bool dd_sharded(const lrn_dd_solver* h) { return h->world > 1 || h->nccl != nullptr; }

// dddist.cu, used by ddlp.cu on a sharded handle with a communicator (collectives: every rank calls them in the same order)
int dd_factor_dist(lrn_dd_solver* h);                   // L := chol(H) on every rank; returns the LAPACK-style info, agreed
void dd_gather_H(lrn_dd_solver* h);                     // sum the row shards of H over the ranks, in place

}  // namespace lrn

namespace {
using namespace lrn;

constexpr int DD_TS = 32;          // Cholesky tile
constexpr int TRSM_CB = 8;

// ------------------------------------------------------------------------------------------------------------------------
// tiled right-looking Cholesky (32 x 32 tiles): factor the diagonal tile, solve the tiles below it, update the trailing tiles
// ------------------------------------------------------------------------------------------------------------------------
// (the reciprocals of the pivots go to rdiag: the solves below multiply by them instead of dividing -- a double-double division
// is ~10 times a multiplication)
__global__ void __launch_bounds__(DD_TS * DD_TS) k_dd_potrf_tile(dd* __restrict__ A, int n, int k0, int w, int* __restrict__ info,
                                                                 dd* __restrict__ rdiag) {
    constexpr int TS = DD_TS;
    __shared__ dd t[TS][TS + 1];
    __shared__ dd rinv[TS];
    __shared__ int bad;
    const int r = threadIdx.x, c = threadIdx.y;           // r fastest: coalesced along a column
    if (r == 0 && c == 0) bad = 0;
    if (r < w && c < w) t[r][c] = A[(size_t)(k0 + c) * n + k0 + r];
    __syncthreads();
    if (*info != 0) return;                                // an earlier tile already failed
    for (int j = 0; j < w; j++) {
        if (r == j && c == j) {
            if (dd_le_zero(t[j][j]) || !(t[j][j].hi == t[j][j].hi)) bad = 1;
            else {
                const dd rs = dd_rsqrt(t[j][j]);            // pivot = a * rsqrt(a), its reciprocal = rsqrt(a)
                t[j][j] = dd_mul(t[j][j], rs);
                rinv[j] = rs;
                rdiag[k0 + j] = rs;
            }
        }
        __syncthreads();
        if (bad) {
            if (r == 0 && c == 0) *info = k0 + j + 1;
            return;
        }
        if (c == j && r > j && r < w) t[r][j] = dd_mul(t[r][j], rinv[j]);
        __syncthreads();
        if (c > j && c < w && r >= c && r < w) t[r][c] = dd_fms(t[r][j], t[c][j], t[r][c]);
        __syncthreads();
    }
    if (r < w && c < w) A[(size_t)(k0 + c) * n + k0 + r] = (r >= c) ? t[r][c] : dd_make(0.0);
}

// X Lkk' = A for the 32-row tile starting at row i0 below the diagonal tile k0.  Eight warps per tile, lane = row of the tile.
// The 32 columns are solved in four blocks of eight: first all warps subtract the contribution of the finished blocks from
// the eight columns of the current block (warp = column: independent dot products), then warp 0 runs the short substitution
// inside the block.  The dependent chain per row is 4 x 28 multiply-adds instead of 496 (a single warp doing the whole
// substitution took 41 us per step at n = 2000 and was the longest kernel of the panel chain).
__device__ __forceinline__ void dd_trsm_tile_body(dd* __restrict__ A, int n, int k0, int w, const dd* __restrict__ rdiag, int i0) {
    constexpr int TS = DD_TS;
    __shared__ dd l[TS][TS + 1];
    __shared__ dd xr[TS][TS + 1];
    __shared__ dd rd[TS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int row = i0 + lane;
    if (warp == 0 && lane < w) rd[lane] = rdiag[k0 + lane];
    for (int c = warp; c < w; c += TRSM_CB) {
        if (lane < w) l[lane][c] = A[(size_t)(k0 + c) * n + k0 + lane];
        xr[lane][c] = (row < n) ? A[(size_t)(k0 + c) * n + row] : dd_make(0.0);
    }
    __syncthreads();
    for (int c0 = 0; c0 < w; c0 += TRSM_CB) {
        const int c = c0 + warp;
        if (c0 > 0 && c < w) {
            dd a0 = xr[lane][c], a1 = dd_make(0.0), a2 = dd_make(0.0), a3 = dd_make(0.0);
            for (int p = 0; p < c0; p += 4) {                       // c0 is a multiple of 8
                a0 = dd_fms(xr[lane][p], l[c][p], a0);
                a1 = dd_fms(xr[lane][p + 1], l[c][p + 1], a1);
                a2 = dd_fms(xr[lane][p + 2], l[c][p + 2], a2);
                a3 = dd_fms(xr[lane][p + 3], l[c][p + 3], a3);
            }
            xr[lane][c] = dd_add(dd_add(a0, a1), dd_add(a2, a3));
        }
        __syncthreads();
        if (warp == 0) {
            const int c1 = min(w, c0 + TRSM_CB);
            for (int cc = c0; cc < c1; cc++) {
                dd v = xr[lane][cc];
                for (int p = c0; p < cc; p++) v = dd_fms(xr[lane][p], l[cc][p], v);
                xr[lane][cc] = dd_mul(v, rd[cc]);
            }
        }
        __syncthreads();
    }
    if (row < n)
        for (int c = warp; c < w; c += TRSM_CB) A[(size_t)(k0 + c) * n + row] = xr[lane][c];
}

// tile blockIdx.x below the diagonal tile
__global__ void __launch_bounds__(DD_TS * TRSM_CB) k_dd_trsm_tile(dd* __restrict__ A, int n, int k0, int w, const dd* __restrict__ rdiag) {
    dd_trsm_tile_body(A, n, k0, w, rdiag, k0 + w + blockIdx.x * DD_TS);
}

// A(I, J) -= X_I X_J' for the tile at rows i0, columns j0 of the trailing matrix (K = w, the panel columns k0 .. k0 + w)
__device__ __forceinline__ void dd_syrk_tile_body(dd* __restrict__ A, int n, int k0, int w, int i0, int j0) {
    constexpr int TS = DD_TS;
    __shared__ dd xi[TS][TS + 1];
    __shared__ dd xj[TS][TS + 1];
    const int r = threadIdx.x, c = threadIdx.y;
    // thread (r, c) loads column c of the panel for row r of both tiles
    if (c < w) {
        xi[r][c] = (i0 + r < n) ? A[(size_t)(k0 + c) * n + i0 + r] : dd_make(0.0);
        xj[r][c] = (j0 + r < n) ? A[(size_t)(k0 + c) * n + j0 + r] : dd_make(0.0);
    }
    __syncthreads();
    const int gi = i0 + r, gj = j0 + c;
    if (gi < n && gj < n && gi >= gj) {
        dd acc = A[(size_t)gj * n + gi];
        for (int p = 0; p < w; p++) acc = dd_fms(xi[r][p], xj[c][p], acc);
        A[(size_t)gj * n + gi] = acc;
    }
}

// tile pairs I >= J of the trailing matrix
// (column tiles jt0 + blockIdx.y: the first tile column of the trailing matrix is updated on the panel stream, the rest on a
// second stream -- see lrn_dd_schur_factor)
__global__ void __launch_bounds__(DD_TS * DD_TS) k_dd_syrk_tile(dd* __restrict__ A, int n, int k0, int w, int jt0) {
    const int jt = jt0 + blockIdx.y;
    if (jt > (int)blockIdx.x) return;
    const int base = k0 + w;
    dd_syrk_tile_body(A, n, k0, w, base + blockIdx.x * DD_TS, base + jt * DD_TS);
}

}  // namespace
