// Blocked right-looking Cholesky with one-step look-ahead on two streams.  One cooperative launch per column panel
// (panel_factor_kernel) factors the diagonal block -- 64 x 64 tiles factored AND inverted in registers -- and solves all rows
// below it with DMMA tile products; the trailing update is a lower-only SYRK-shaped product with K = panel width on the TMA-fed
// kernel (panels of 256 / 512 / 2 x 512 columns).  Triangular solves advance 256 unknowns per step through pre-built
// inverses of the 256 x 256 diagonal blocks and are replayed as CUDA graphs (see chol_solve).
#include "chol.cuh"
#include "gemm.cuh"
#include <cooperative_groups.h>
#include <algorithm>

namespace lrn {
namespace {

constexpr int DB = CHOL_DB;
constexpr int SLD = DB + 1;
constexpr size_t POTRF_SMEM = (2 * DB * SLD + DB + 2 + 4 * DB) * sizeof(double);

// One CTA factors a 64x64 diagonal block held in REGISTERS (each of the 256 threads owns a cyclic 4x4 sub-tile: rows
// ti+16a, columns tj+16b), two barriers per column; the inverse of the factor is then built row by row in shared memory
// (4 partial dot products per entry).  ~15 us instead of ~100 us for the previous shared-memory version.
// 16 consecutive columns j = 16*JA + jm of the register-resident 64x64 factorisation.  JA is a compile-time constant so that
// every "is this my row / column block" test folds away and the triangular structure skips whole 16x16 register sub-blocks.
template <int JA>
__device__ __forceinline__ void potrf64_steps(double (&r)[4][4], double (&z)[4][4], double* colbuf, double* rowbuf, int ti, int tj,
                                              int nb, int* __restrict__ info, int base) {
    for (int jm = 0; jm < 16; jm++) {
        const int j = JA * 16 + jm;
        double* cb = colbuf + (j & 1) * DB;
        double* rb = rowbuf + (j & 1) * DB;
        if (tj == jm) {                                   // owners of column j publish the raw column a(j:,j)
#pragma unroll
            for (int a = JA; a < 4; a++) cb[ti + 16 * a] = r[a][JA];
        }
        if (ti == jm) {                                   // owners of row j publish Z(j,0:j)
#pragma unroll
            for (int b = 0; b <= JA; b++) rb[tj + 16 * b] = z[JA][b];
        }
        __syncthreads();
        double d = cb[j];
        if (!(d > 0.0)) {                                  // also catches NaN; every thread substitutes the same value
            if (threadIdx.x == 0 && j < nb && *info == 0) *info = base + j + 1;
            d = 1.0;
        }
        const double rs = rsqrt(d), rd = rs * rs;           // 1/l_jj and 1/d
        double ck[4], rk[4];
#pragma unroll
        for (int b = JA; b < 4; b++) ck[b] = (b > JA || tj > jm) ? cb[tj + 16 * b] : 0.0;
#pragma unroll
        for (int b = 0; b <= JA; b++) rk[b] = rb[tj + 16 * b];
#pragma unroll
        for (int a = JA; a < 4; a++) {
            const double ci = cb[ti + 16 * a];
            const double li = (a > JA || ti > jm) ? ci * rd : 0.0;
#pragma unroll
            for (int b = JA; b < 4; b++) r[a][b] = fma(-li, ck[b], r[a][b]);       // trailing matrix
#pragma unroll
            for (int b = 0; b <= JA; b++) z[a][b] = fma(-li, rk[b], z[a][b]);      // Z(i,:) -= (a_ij / d) Z(j,:)
        }
        if (ti == jm) {                                   // E(j,:) = Z(j,:) / l_jj
#pragma unroll
            for (int b = 0; b <= JA; b++) z[JA][b] *= rs;
        }
        if (tj == jm) {                                   // column j is final: l_ij = a_ij / l_jj, l_jj = d / l_jj
#pragma unroll
            for (int a = JA; a < 4; a++) {
                if (a > JA || ti > jm) r[a][JA] = cb[ti + 16 * a] * rs;
                else if (ti == jm) r[a][JA] = d * rs;
            }
        }
    }
}

// Factor a 64x64 block held in REGISTERS (each of the 256 threads owns the cyclic 4x4 sub-tile rows ti+16a, columns tj+16b)
// and build the inverse of the factor in the same sweep: with Z = I,  step j:  E(j,:) = Z(j,:)/l_jj ;  Z(i,:) -= l_ij E(j,:)
// for i > j (forward substitution on the identity, right-looking) -- one block barrier and one rsqrt per column, no
// separate inversion phase.
__device__ __forceinline__ void potrf64_block(double* __restrict__ A, int lda, int nb, double* __restrict__ dinv,
                                              int* __restrict__ info, int base, double* sm) {
    double* colbuf = sm;                  // [2][DB]  raw column j of the trailing matrix   (double buffered)
    double* rowbuf = sm + 2 * DB;         // [2][DB]  row j of Z
    const int tid = threadIdx.x, ti = tid & 15, tj = tid >> 4;
    double r[4][4], z[4][4];
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
        for (int b = 0; b < 4; b++) {
            const int i = ti + 16 * a, k = tj + 16 * b;
            double v = 0.0;
            if (i < nb && k < nb) v = (i >= k) ? A[(size_t)k * lda + i] : A[(size_t)i * lda + k];   // symmetric fill from the lower part
            else if (i == k) v = 1.0;                                                            // identity padding
            r[a][b] = v;
            z[a][b] = (i == k) ? 1.0 : 0.0;
        }
    potrf64_steps<0>(r, z, colbuf, rowbuf, ti, tj, nb, info, base);
    potrf64_steps<1>(r, z, colbuf, rowbuf, ti, tj, nb, info, base);
    potrf64_steps<2>(r, z, colbuf, rowbuf, ti, tj, nb, info, base);
    potrf64_steps<3>(r, z, colbuf, rowbuf, ti, tj, nb, info, base);
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
        for (int b = 0; b < 4; b++) {
            const int i = ti + 16 * a, k = tj + 16 * b;
            if (i < nb && k < nb && i >= k) A[(size_t)k * lda + i] = r[a][b];
            dinv[(size_t)k * DB + i] = (i < nb && k < nb && i >= k) ? z[a][b] : 0.0;
        }
}

__global__ void __launch_bounds__(256)
    potrf_diag_kernel(double* __restrict__ A, int lda, int nb, double* __restrict__ dinv, int* __restrict__ info, int base) {
    extern __shared__ double sm[];
    potrf64_block(A, lda, nb, dinv, info, base, sm);
}

// ---------------------------------------------------------------------------------------------------------------------
// Cooperative small-matrix Cholesky (64 < n <= 512): ONE launch factors the whole block, produces the inverted 64x64
// diagonal blocks and (optionally) the full inverse of the factor.  Replaces ~60 dependent tiny launches per 512-block
// (the latency chain that bounded the factorisation of mid-size Schur matrices and of the PSD blocks).
// Grid-wide barriers (cooperative launch) separate: diagonal block factorisation (CTA 0) | row-block solves | trailing tiles.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int TLD = DB + 1;     // padded k-stride of the shared-memory tiles

// s[k*TLD + i] = G[i + k*ld]  (i < rows, k < cols; zero elsewhere)
__device__ __forceinline__ void tile_load(double* s, const double* __restrict__ G, int ld, int rows, int cols) {
    for (int idx = threadIdx.x; idx < DB * DB; idx += 256) {
        const int i = idx & 63, k = idx >> 6;
        s[k * TLD + i] = (i < rows && k < cols) ? G[(size_t)k * ld + i] : 0.0;
    }
}
// s[k*TLD + j] = G[k + j*ld]  (k < rows, j < cols): the transposed placement
__device__ __forceinline__ void tile_load_t(double* s, const double* __restrict__ G, int ld, int rows, int cols) {
    for (int idx = threadIdx.x; idx < DB * DB; idx += 256) {
        const int k = idx & 63, j = idx >> 6;
        s[k * TLD + j] = (k < rows && j < cols) ? G[(size_t)j * ld + k] : 0.0;
    }
}
// acc[a][b] += sum_k As[k][ti+16a] * Bs[k][tj+16b]
__device__ __forceinline__ void tile_prod(const double* __restrict__ As, const double* __restrict__ Bs, double (&acc)[4][4]) {
    const int ti = threadIdx.x & 15, tj = threadIdx.x >> 4;
#pragma unroll 8
    for (int k = 0; k < DB; k++) {
        double a[4], b[4];
#pragma unroll
        for (int t = 0; t < 4; t++) { a[t] = As[k * TLD + ti + 16 * t]; b[t] = Bs[k * TLD + tj + 16 * t]; }
#pragma unroll
        for (int x = 0; x < 4; x++)
#pragma unroll
            for (int y = 0; y < 4; y++) acc[x][y] = fma(a[x], b[y], acc[x][y]);
    }
}

__global__ void __launch_bounds__(256)
    potrf_coop_kernel(double* __restrict__ A, int lda, int n, double* __restrict__ dinv, double* __restrict__ X, int ldx,
                      int* __restrict__ info, int base) {
    extern __shared__ double sm[];
    cooperative_groups::grid_group grid = cooperative_groups::this_grid();
    double* As = sm;
    double* Bs = sm + DB * TLD;
    const int G = gridDim.x, c = blockIdx.x, tid = threadIdx.x, ti = tid & 15, tj = tid >> 4;
    const int nb = (n + DB - 1) / DB;
    for (int j = 0; j < nb; j++) {
        const int j0 = j * DB, jb = min(DB, n - j0);
        if (c == 0) potrf64_block(A + (size_t)j0 * lda + j0, lda, jb, dinv + (size_t)j * DB * DB, info, base + j0, sm);
        __threadfence();
        grid.sync();
        for (int i = j + 1 + c; i < nb; i += G) {                      // P_i <- P_i * inv(L_jj)^T
            const int i0 = i * DB, ib = min(DB, n - i0);
            __syncthreads();
            tile_load(As, A + (size_t)j0 * lda + i0, lda, ib, jb);
            tile_load(Bs, dinv + (size_t)j * DB * DB, DB, DB, DB);     // Bs[k][cc] = dinv[cc + k*64] = inv(L_jj)[cc][k]
            __syncthreads();
            double acc[4][4] = {};
            tile_prod(As, Bs, acc);
#pragma unroll
            for (int x = 0; x < 4; x++)
#pragma unroll
                for (int y = 0; y < 4; y++) {
                    const int a = ti + 16 * x, b = tj + 16 * y;
                    if (a < ib && b < jb) A[(size_t)(j0 + b) * lda + i0 + a] = acc[x][y];
                }
        }
        __threadfence();
        grid.sync();
        const int t = nb - 1 - j, ntile = t * (t + 1) / 2;
        for (int tile = c; tile < ntile; tile += G) {                  // A_rc -= P_r P_c^T   (j < cc <= r)
            int rr = (int)((sqrt(8.0 * tile + 1.0) - 1.0) * 0.5);
            while ((rr + 1) * (rr + 2) / 2 <= tile) rr++;
            while (rr * (rr + 1) / 2 > tile) rr--;
            const int cc = tile - rr * (rr + 1) / 2;
            const int r0 = (j + 1 + rr) * DB, c0 = (j + 1 + cc) * DB, rb = min(DB, n - r0), cb = min(DB, n - c0);
            __syncthreads();
            tile_load(As, A + (size_t)j0 * lda + r0, lda, rb, jb);
            tile_load(Bs, A + (size_t)j0 * lda + c0, lda, cb, jb);
            __syncthreads();
            double acc[4][4] = {};
            tile_prod(As, Bs, acc);
#pragma unroll
            for (int x = 0; x < 4; x++)
#pragma unroll
                for (int y = 0; y < 4; y++) {
                    const int a = ti + 16 * x, b = tj + 16 * y;
                    if (a < rb && b < cb) A[(size_t)(c0 + b) * lda + r0 + a] -= acc[x][y];
                }
        }
        __threadfence();
        grid.sync();
    }
    if (!X) return;
    // full inverse of the factor: X_ii = inv(L_ii);  X_ic = -inv(L_ii) * sum_{k=c}^{i-1} L_ik X_kc   (block row after block row)
    for (int i = c; i < nb; i += G) {
        const int i0 = i * DB, ib = min(DB, n - i0);
        for (int idx = tid; idx < DB * DB; idx += 256) {
            const int a = idx & 63, b = idx >> 6;
            if (a < ib && b < ib) X[(size_t)(i0 + b) * ldx + i0 + a] = dinv[(size_t)i * DB * DB + (size_t)b * DB + a];
        }
    }
    __threadfence();
    grid.sync();
    for (int i = 1; i < nb; i++) {
        const int i0 = i * DB, ib = min(DB, n - i0);
        for (int cc = c; cc < i; cc += G) {
            const int c0 = cc * DB;
            double acc[4][4] = {};
            for (int k = cc; k < i; k++) {
                const int k0 = k * DB;
                __syncthreads();
                tile_load(As, A + (size_t)k0 * lda + i0, lda, ib, DB);          // As[t][a] = L_ik[a][t]
                tile_load_t(Bs, X + (size_t)c0 * ldx + k0, ldx, DB, DB);        // Bs[t][b] = X_kc[t][b]
                __syncthreads();
                tile_prod(As, Bs, acc);
            }
            __syncthreads();
#pragma unroll
            for (int x = 0; x < 4; x++)
#pragma unroll
                for (int y = 0; y < 4; y++) Bs[(ti + 16 * x) * TLD + tj + 16 * y] = acc[x][y];   // Bs[t][b] = acc[t][b]
            tile_load(As, dinv + (size_t)i * DB * DB, DB, DB, DB);              // As[t][a] = inv(L_ii)[a][t]
            __syncthreads();
            double acc2[4][4] = {};
            tile_prod(As, Bs, acc2);
#pragma unroll
            for (int x = 0; x < 4; x++)
#pragma unroll
                for (int y = 0; y < 4; y++) {
                    const int a = ti + 16 * x, b = tj + 16 * y;
                    if (a < ib) X[(size_t)(c0 + b) * ldx + i0 + a] = -acc2[x][y];
                }
        }
        __threadfence();
        grid.sync();
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Whole-panel factorisation in ONE cooperative launch: the (rows x w) column panel whose top w x w block is the current
// diagonal block is factored right-looking in 64-column steps,
//     step j :  CTA 0 factors + inverts the 64 x 64 diagonal block (registers)          | grid barrier
//               every row tile below:  P_i <- A_ij inv(L_jj)^T        (64 x 64 x 64 DMMA) | grid barrier
//               remaining panel columns k > j:  A_ik -= P_i P_k^T      (64 x 64 x 64 DMMA) | grid barrier
// so that the diagonal block AND the rows below it leave the kernel solved.  Replaces, per panel, the cooperative diagonal
// kernel + its explicit w x w inverse + memset + the rows x w x w panel GEMM + the copy back (5 dependent launches and an
// m^3-class inversion on the critical path of mid-size factorisations).  Tiles are staged in shared memory [k][m] with a +4
// padded stride (conflict-free m8n8k4 fragment loads, same layout as gemm.cu).
// ---------------------------------------------------------------------------------------------------------------------
constexpr int PLD = DB + 4;
constexpr size_t PANEL_SMEM = (size_t)2 * DB * PLD * sizeof(double);

__device__ __forceinline__ void dmma884p(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}
// s[k*PLD + i] = G[i + k*ld]  (i < rows, k < cols; zero elsewhere)
__device__ __forceinline__ void ptile_load(double* s, const double* __restrict__ G, int ld, int rows, int cols) {
    for (int idx = threadIdx.x; idx < DB * DB; idx += 256) {
        const int i = idx & 63, k = idx >> 6;
        s[k * PLD + i] = (i < rows && k < cols) ? G[(size_t)k * ld + i] : 0.0;
    }
}
// acc += A B^T with As[k][m], Bs[k][n]; 8 warps as 2 x 4, warp tile 32 x 16.  Element (i, j, t) of acc is row
// wm0 + 8 i + (lane >> 2), column wn0 + 8 j + 2 (lane & 3) + t.
__device__ __forceinline__ void ptile_mma(const double* __restrict__ As, const double* __restrict__ Bs, double (&acc)[4][2][2]) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int wm0 = (warp >> 2) * 32, wn0 = (warp & 3) * 16, lr = lane >> 2, lk = lane & 3;
#pragma unroll 4
    for (int kk = 0; kk < DB; kk += 4) {
        double a[4], b[2];
#pragma unroll
        for (int i = 0; i < 4; i++) a[i] = As[(kk + lk) * PLD + wm0 + i * 8 + lr];
#pragma unroll
        for (int j = 0; j < 2; j++) b[j] = Bs[(kk + lk) * PLD + wn0 + j * 8 + lr];
#pragma unroll
        for (int i = 0; i < 4; i++)
#pragma unroll
            for (int j = 0; j < 2; j++) dmma884p(acc[i][j][0], acc[i][j][1], a[i], b[j]);
    }
}

// s[k*PLD + n] = G[k + n*ld]  (k < rows, n < cols): the transposed placement (B operand given as a K x N column-major block)
__device__ __forceinline__ void ptile_load_t(double* s, const double* __restrict__ G, int ld, int rows, int cols) {
    for (int idx = threadIdx.x; idx < DB * DB; idx += 256) {
        const int k = idx & 63, n = idx >> 6;
        s[k * PLD + n] = (k < rows && n < cols) ? G[(size_t)n * ld + k] : 0.0;
    }
}

// X (optional, rows == w <= 512 only): the full inverse of the factor of the diagonal block, built after the factorisation by
// recursive doubling from the inverted 64 x 64 diagonal blocks:  inv([L11 0; L21 L22]) = [X11 0; -X22 (L21 X11) X22]  for
// block sizes 64 -> 128 -> 256 -> 512 (two grid-wide phases per level: T = L21 X11, then X21 = -X22 T; 6 dependent phases for a
// 512 block instead of 7 block-row levels of a forward substitution).  T is a w x w scratch (leading dimension ldx).
__global__ void __launch_bounds__(256)
    panel_factor_kernel(double* __restrict__ A, int lda, int rows, int w, double* __restrict__ dinv, int* __restrict__ info, int base,
                        double* __restrict__ X, int ldx, double* __restrict__ T) {
    extern __shared__ double sm[];
    cooperative_groups::grid_group grid = cooperative_groups::this_grid();
    double* As = sm;
    double* Bs = sm + DB * PLD;
    const int G = gridDim.x, c = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int wm0 = (warp >> 2) * 32, wn0 = (warp & 3) * 16, lr = lane >> 2, lk = lane & 3;
    const int nbj = (w + DB - 1) / DB, nt = (rows + DB - 1) / DB;
    // The 64 x 64 diagonal block of step j + 1 is factored by CTA 0 DURING the update phase of step j (right after it has applied
    // step j to that block), so a step costs two grid barriers and the register factorisation hides behind the tile updates.
    if (c == 0) potrf64_block(A, lda, min(DB, w), dinv, info, base, sm);
    __threadfence();
    grid.sync();
    for (int j = 0; j < nbj; j++) {
        const int j0 = j * DB, jb = min(DB, w - j0);
        // ---- row tiles below the diagonal block of this step: P_i <- A_ij inv(L_jj)^T -------------------------------
        for (int i = j + 1 + c; i < nt; i += G) {
            const int i0 = i * DB, ib = min(DB, rows - i0);
            __syncthreads();
            ptile_load(As, A + (size_t)j0 * lda + i0, lda, ib, jb);
            ptile_load(Bs, dinv + (size_t)j * DB * DB, DB, DB, DB);      // Bs[k][b] = inv(L_jj)[b][k]
            __syncthreads();
            double acc[4][2][2] = {};
            ptile_mma(As, Bs, acc);
#pragma unroll
            for (int x = 0; x < 4; x++)
#pragma unroll
                for (int y = 0; y < 2; y++)
#pragma unroll
                    for (int t = 0; t < 2; t++) {
                        const int a = wm0 + x * 8 + lr, b = wn0 + y * 8 + lk * 2 + t;
                        if (a < ib && b < jb) A[(size_t)(j0 + b) * lda + i0 + a] = acc[x][y][t];
                    }
        }
        __threadfence();
        grid.sync();
        // ---- the panel columns to the right of step j: A_ik -= P_i P_k^T for block columns k > j, row tiles i >= k -----------
        const int nk = nbj - 1 - j;
        if (nk > 0) {
            const long long ntask = (long long)(nt - 1 - j) * nk;
            // task 0 is the next diagonal tile (j+1, j+1): CTA 0 takes it, factors that tile, and (only when it is alone) the rest;
            // the other CTAs share tasks 1 .. ntask-1
            const long long tfirst = (c == 0) ? 0 : c, tstride = (G > 1) ? (c == 0 ? ntask : G - 1) : 1;
            for (long long task = tfirst; task < ntask; task += tstride) {
                const int i = j + 1 + (int)(task / nk), k = j + 1 + (int)(task % nk);
                if (k > i) continue;                                   // block-uniform: above the diagonal of the panel
                const int i0 = i * DB, k0 = k * DB, ib = min(DB, rows - i0), kb = min(DB, w - k0);
                __syncthreads();
                ptile_load(As, A + (size_t)j0 * lda + i0, lda, ib, jb);
                ptile_load(Bs, A + (size_t)j0 * lda + k0, lda, kb, jb);
                __syncthreads();
                double acc[4][2][2] = {};
                ptile_mma(As, Bs, acc);
#pragma unroll
                for (int x = 0; x < 4; x++)
#pragma unroll
                    for (int y = 0; y < 2; y++)
#pragma unroll
                        for (int t = 0; t < 2; t++) {
                            const int a = wm0 + x * 8 + lr, b = wn0 + y * 8 + lk * 2 + t;
                            if (a < ib && b < kb) A[(size_t)(k0 + b) * lda + i0 + a] -= acc[x][y][t];
                        }
                if (task == 0) {                                       // (CTA 0 only) the next diagonal tile is final: factor it now
                    const int n0 = (j + 1) * DB;
                    __threadfence_block();
                    __syncthreads();
                    potrf64_block(A + (size_t)n0 * lda + n0, lda, min(DB, w - n0), dinv + (size_t)(j + 1) * DB * DB, info, base + n0, sm);
                }
            }
            __threadfence();
            grid.sync();
        }
    }
    if (!X) return;
    // ---- inverse of the factor (diagonal block only) ---------------------------------------------------------------------
    for (int i = c; i < nbj; i += G) {                                   // X_ii = inv(L_ii); the rest of X starts as zero
        const int i0 = i * DB, ib = min(DB, w - i0);
        for (int idx = threadIdx.x; idx < DB * DB; idx += 256) {
            const int a = idx & 63, b = idx >> 6;
            if (a < ib && b < ib) X[(size_t)(i0 + b) * ldx + i0 + a] = dinv[(size_t)i * DB * DB + (size_t)b * DB + a];
        }
    }
    __threadfence();
    grid.sync();
    for (int sblk = 1; sblk < nbj; sblk *= 2) {                          // sblk 64-tiles per half: halves of size 64 * sblk
        const int npair = (nbj + 2 * sblk - 1) / (2 * sblk);
        // phase A: T = L21 X11 for every pair block (tiles (i, j) of the lower-left quarter; X11 is lower triangular: k >= j)
        // phase B: X21 = -X22 T                                        (X22 is lower triangular: k <= i)
        for (int phase = 0; phase < 2; phase++) {
            const int ntask = npair * sblk * sblk;
            for (int task = c; task < ntask; task += G) {
                const int pb = task / (sblk * sblk), rem = task - pb * sblk * sblk;
                const int ti = rem / sblk, tj = rem - ti * sblk;          // tile inside the quarter
                const int t0 = pb * 2 * sblk;                             // first 64-tile of the pair block
                const int gi = t0 + sblk + ti, gj = t0 + tj;              // global 64-tile coordinates of the output tile
                if (gi >= nbj) continue;                                  // the second half does not exist (w not a power of two)
                const int i0 = gi * DB, j0 = gj * DB, ib = min(DB, w - i0), jb = min(DB, w - j0);
                double acc[4][2][2] = {};
                const int kbeg = phase == 0 ? tj : 0, kend = phase == 0 ? sblk : ti + 1;
                for (int kt = kbeg; kt < kend; kt++) {
                    __syncthreads();
                    if (phase == 0) {
                        const int k0 = (t0 + kt) * DB, kb = min(DB, w - k0);
                        ptile_load(As, A + (size_t)k0 * lda + i0, lda, ib, kb);                 // L21 tile (gi, t0 + kt)
                        ptile_load_t(Bs, X + (size_t)j0 * ldx + k0, ldx, kb, jb);               // X11 tile (t0 + kt, gj)
                    } else {
                        const int k0 = (t0 + sblk + kt) * DB, kb = min(DB, w - k0);
                        ptile_load(As, X + (size_t)k0 * ldx + i0, ldx, ib, kb);                 // X22 tile (gi, t0 + sblk + kt)
                        ptile_load_t(Bs, T + (size_t)j0 * ldx + k0, ldx, kb, jb);               // T tile (t0 + sblk + kt, gj)
                    }
                    __syncthreads();
                    ptile_mma(As, Bs, acc);
                }
                double* out = (phase == 0 ? T : X) + (size_t)j0 * ldx + i0;
                const double sgn = phase == 0 ? 1.0 : -1.0;
#pragma unroll
                for (int x = 0; x < 4; x++)
#pragma unroll
                    for (int y = 0; y < 2; y++)
#pragma unroll
                        for (int t = 0; t < 2; t++) {
                            const int a = wm0 + x * 8 + lr, b = wn0 + y * 8 + lk * 2 + t;
                            if (a < ib && b < jb) out[(size_t)b * ldx + a] = sgn * acc[x][y][t];
                        }
            }
            __threadfence();
            grid.sync();
        }
    }
}

constexpr int COOP_MAXN = 512;

// panel width: 256 for mid-size matrices (the panel chain is the critical path), 512 above 8192, 1024 (factored as two 512-wide
// halves) from 16384 on: the trailing update then runs with K = 1024, which halves the number of C-tile read-modify-write
// epilogues and pipeline fills of the TMA-fed kernel per flop
int pick_nb(int n) { return n >= 16384 ? 1024 : (n > 8192 ? 512 : 256); }

void potrf_launch_config() {
    static PerDeviceOnce once;
    once.run([&] {
        LRN_CUDA(cudaFuncSetAttribute(potrf_diag_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)POTRF_SMEM));
        LRN_CUDA(cudaFuncSetAttribute(potrf_coop_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)POTRF_SMEM));
        LRN_CUDA(cudaFuncSetAttribute(panel_factor_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)std::max(POTRF_SMEM, PANEL_SMEM)));
    });
}

// factor a block of side n <= 512 with one launch; X (optional, n x n, ldx) receives the full inverse of the factor
void potrf_small(double* A, int lda, int n, double* dinv, double* X, int ldx, int* info, int base, cudaStream_t st) {
    potrf_launch_config();
    if (n <= DB && !X) {
        potrf_diag_kernel<<<1, 256, POTRF_SMEM, st>>>(A, lda, n, dinv, info, base);
        LRN_CHECK_LAUNCH();
        return;
    }
    LRN_REQUIRE(n <= COOP_MAXN, "potrf_small handles n <= 512");
    if (X) LRN_CUDA(cudaMemsetAsync(X, 0, (size_t)ldx * n * sizeof(double), st));
    const int nb = (int)cdiv(n, DB);
    int G = nb * (nb - 1) / 2;
    G = G < 1 ? 1 : (G > 28 ? 28 : G);
    void* args[] = {&A, &lda, &n, &dinv, &X, &ldx, &info, &base};
    LRN_CUDA(cudaLaunchCooperativeKernel((void*)potrf_coop_kernel, dim3(G), dim3(256), args, POTRF_SMEM, st));
    g_kernel_launches.fetch_add(1, std::memory_order_relaxed);
}

// Factor the kb x kb diagonal block at the top of a column panel AND solve the `rows_below` rows under it, in one cooperative
// launch (panel_factor_kernel).  `gcap` bounds the grid: all SMs for mid-size matrices (the panel chain is the critical path),
// a third of them for very large ones (the chain hides behind the trailing update; the panel must not evict its CTAs).
void factor_panel(double* Akk, int kb, int rows_below, int lda, double* dk, int* info, int base, int gcap, cudaStream_t st) {
    potrf_launch_config();
    if (kb > COOP_MAXN) {
        // wide panel = two halves: left half (all rows), update of the right half with it (one DMMA GEMM), right half
        const int k1 = (kb / 2 + DB - 1) / DB * DB, k2 = kb - k1;
        const int below1 = k2 + (rows_below > 0 ? rows_below : 0);
        factor_panel(Akk, k1, below1, lda, dk, info, base, gcap, st);
        const double* P = Akk + k1;                                          // rows below the left diagonal block
        GemmParams g;
        g.A = P; g.B = P; g.C = Akk + (size_t)k1 * lda + k1;
        g.M = below1; g.N = k2; g.K = k1; g.lda = lda; g.ldb = lda; g.ldc = lda;
        g.transB = true; g.alpha = -1.0; g.beta = 1.0; g.lower = 1;
        gemm(g, st);
        factor_panel(Akk + (size_t)k1 * lda + k1, k2, rows_below, lda, dk + (size_t)(k1 / DB) * DB * DB, info, base + k1, gcap, st);
        return;
    }
    int rows = kb + (rows_below > 0 ? rows_below : 0);
    const int nt = (int)cdiv(rows, DB), nbj = (int)cdiv(kb, DB);
    long long tasks = std::max<long long>(nt - 1, (long long)(nt - 1) * std::max(nbj - 1, 1));
    int G = (int)std::min<long long>(std::max(gcap, 1), std::max<long long>(tasks, 1));
    const size_t smem = std::max(POTRF_SMEM, PANEL_SMEM);
    double* X = nullptr; int ldx = 0; double* T = nullptr;
    void* args[] = {&Akk, &lda, &rows, &kb, &dk, &info, &base, &X, &ldx, &T};
    LRN_CUDA(cudaLaunchCooperativeKernel((void*)panel_factor_kernel, dim3(G), dim3(256), args, smem, st));
    g_kernel_launches.fetch_add(1, std::memory_order_relaxed);
}

// diagonal block (w <= 512) + full inverse of its factor into X (w x w, ldx, zero above the diagonal), one cooperative launch;
// T: w x ldx scratch
void factor_diag_with_inverse(double* Akk, int lda, int w, double* dk, double* X, int ldx, double* T, int* info, int base,
                              cudaStream_t st) {
    potrf_launch_config();
    LRN_REQUIRE(w <= COOP_MAXN, "diagonal block wider than 512");
    LRN_CUDA(cudaMemsetAsync(X, 0, (size_t)ldx * w * sizeof(double), st));
    const int nbj = (int)cdiv(w, DB);
    int G = std::max(1, std::min(device_sm_count(), nbj * nbj / 2 + 1));
    const size_t smem = std::max(POTRF_SMEM, PANEL_SMEM);
    int rows = w;
    void* args[] = {&Akk, &lda, &rows, &w, &dk, &info, &base, &X, &ldx, &T};
    LRN_CUDA(cudaLaunchCooperativeKernel((void*)panel_factor_kernel, dim3(G), dim3(256), args, smem, st));
    g_kernel_launches.fetch_add(1, std::memory_order_relaxed);
}

int panel_grid_cap(int n) { return n >= 16384 ? std::max(16, device_sm_count() / 3) : device_sm_count(); }

void chol_rec(double* A, int n, int lda, double* dinv, int* info, int base, CholWork& work, cudaStream_t st) {
    if (n <= COOP_MAXN) {
        potrf_small(A, lda, n, dinv, nullptr, 0, info, base, st);
        return;
    }
    const int NB = pick_nb(n), gcap = panel_grid_cap(n);
    for (int k = 0; k < n; k += NB) {
        const int kb = (n - k < NB) ? (n - k) : NB;
        double* Akk = A + (size_t)k * lda + k;
        double* dk = dinv + (size_t)(k / DB) * DB * DB;
        const int rows = n - k - kb;
        factor_panel(Akk, kb, rows, lda, dk, info, base + k, gcap, st);
        if (rows <= 0) break;
        double* P = A + (size_t)k * lda + (k + kb);          // rows x kb panel below the diagonal block
        // trailing update, lower triangle only
        GemmParams p;
        p.A = P; p.B = P; p.C = A + (size_t)(k + kb) * lda + (k + kb);
        p.M = rows; p.N = rows; p.K = kb; p.lda = lda; p.ldb = lda; p.ldc = lda;
        p.transB = true; p.alpha = -1.0; p.beta = 1.0; p.lower = 1;
        gemm(p, st);
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Triangular solves with 256-wide steps.  After a factorisation the inverses of the 256 x 256 diagonal blocks of L are
// built once (chol_build_tinv: block forward substitution on the stored 64 x 64 inverses, batched DMMA GEMMs over all
// blocks), so a step is two launches: y_b = inv(L_bb) x_b (one CTA, 1024 threads, 256 KB from L2/HBM) and the update of the
// remaining right-hand side with the (n - j) x 256 panel (forward: 64 rows x 4 column quarters per CTA, 16 loads in flight
// per thread; backward: one column of L per warp pass, coalesced along the column).  L is read once per direction.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int SW = 256;

__global__ void tinv_diag_kernel(const double* __restrict__ dinv, double* __restrict__ X, int nsb_total) {
    // X block b = sb / 4, sub-block i = sb % 4: X_ii = D_i (lower triangle)
    const int sb = blockIdx.x;
    if (sb >= nsb_total) return;
    const double* d = dinv + (size_t)sb * DB * DB;
    double* x = X + (size_t)(sb / 4) * SW * SW + (size_t)(sb % 4) * DB * SW + (sb % 4) * DB;
    for (int idx = threadIdx.x; idx < DB * DB; idx += blockDim.x) {
        const int r = idx & 63, c = idx >> 6;
        x[r + (size_t)c * SW] = (r >= c) ? d[idx] : 0.0;
    }
}

__global__ void __launch_bounds__(1024)
    trsv_diag_kernel(const double* __restrict__ X, int jb, const double* __restrict__ rhs, double* __restrict__ sol, int dir,
                     const double* __restrict__ Xnext) {
    __shared__ double xs[SW], red[4][SW];
    const int tid = threadIdx.x;
    if (tid < SW) xs[tid] = (tid < jb) ? rhs[tid] : 0.0;
    if (Xnext) {   // pull the next step's inverse block (512 KB) towards L2 while this step runs
        const char* pn = reinterpret_cast<const char*>(Xnext) + (size_t)tid * 512;
#pragma unroll
        for (int u = 0; u < 4; u++) asm volatile("prefetch.global.L2 [%0];" ::"l"(pn + u * 128));
    }
    __syncthreads();
    if (!dir) {
        // y_r = sum_{c <= r} X(r, c) x_c : thread (r, part) takes the columns c = part (mod 4), 16 loads in flight
        const int r = tid & 255, part = tid >> 8;
        double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
        if (r < jb) {
            const double* Xr = X + r;
#pragma unroll 1
            for (int t0 = 0; t0 < 64; t0 += 16) {
                if (part + 4 * t0 > r) break;
                double v[16];
#pragma unroll
                for (int u = 0; u < 16; u++) {
                    const int c = part + 4 * (t0 + u);
                    v[u] = (c <= r) ? Xr[(size_t)c * SW] : 0.0;
                }
#pragma unroll
                for (int u = 0; u < 16; u += 4) {
                    a0 += v[u] * xs[part + 4 * (t0 + u)];
                    a1 += v[u + 1] * xs[part + 4 * (t0 + u + 1)];
                    a2 += v[u + 2] * xs[part + 4 * (t0 + u + 2)];
                    a3 += v[u + 3] * xs[part + 4 * (t0 + u + 3)];
                }
            }
        }
        red[part][r] = (a0 + a1) + (a2 + a3);
        __syncthreads();
        if (tid < jb) sol[tid] = (red[0][tid] + red[1][tid]) + (red[2][tid] + red[3][tid]);
    } else {
        // y_r = sum_{c >= r} X(c, r) x_c : one column of X per warp pass, the 8 rows of a warp are loaded together
        const int lane = tid & 31, warp = tid >> 5;
        double acc[8];
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const int r = warp + 32 * k;
            const double* col = X + (size_t)r * SW;
            double a = 0.0;
#pragma unroll
            for (int u = 0; u < 8; u++) {
                const int c = 32 * u + lane;
                if (c >= r && c < jb) a += col[c] * xs[c];
            }
            acc[k] = a;
        }
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const double a = warp_sum(acc[k]);
            const int r = warp + 32 * k;
            if (lane == 0 && r < jb) sol[r] = a;
        }
    }
}

__global__ void __launch_bounds__(256)
    trsv_update_fwd_kernel(const double* __restrict__ L, int lda, int n, int j0, int jb, const double* __restrict__ y,
                           double* __restrict__ rhs) {
    __shared__ double ys[SW], red[4][64];
    const int tid = threadIdx.x, r = tid & 63, q = tid >> 6;
    ys[tid] = (tid < jb) ? y[tid] : 0.0;
    __syncthreads();
    const int i = j0 + jb + blockIdx.x * 64 + r;
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    if (i < n) {
        const int c0 = q * 64, c1 = min(jb, c0 + 64);
        const double* Lp = L + (size_t)j0 * lda + i;
        int c = c0;
        for (; c + 15 < c1; c += 16) {           // 16 independent loads in flight per thread
            double v[16];
#pragma unroll
            for (int u = 0; u < 16; u++) v[u] = Lp[(size_t)(c + u) * lda];
#pragma unroll
            for (int u = 0; u < 16; u += 4) {
                a0 += v[u] * ys[c + u];
                a1 += v[u + 1] * ys[c + u + 1];
                a2 += v[u + 2] * ys[c + u + 2];
                a3 += v[u + 3] * ys[c + u + 3];
            }
        }
        for (; c < c1; c++) a0 += Lp[(size_t)c * lda] * ys[c];
    }
    red[q][r] = (a0 + a1) + (a2 + a3);
    __syncthreads();
    if (q == 0 && i < n) rhs[i] -= (red[0][r] + red[1][r]) + (red[2][r] + red[3][r]);
}

__global__ void __launch_bounds__(256)
    trsv_update_bwd_kernel(const double* __restrict__ L, int lda, int j0, int jb, const double* __restrict__ y,
                           double* __restrict__ rhs) {
    __shared__ double ys[SW];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    ys[tid] = (tid < jb) ? y[tid] : 0.0;
    __syncthreads();
    // 32 columns of L per CTA, 4 per warp, two at a time
    const int ibase = blockIdx.x * 32 + warp * 4;
    for (int u = 0; u < 4; u += 2) {
        const int i0 = ibase + u, i1 = i0 + 1;
        if (i0 >= j0) break;
        const double* L0 = L + (size_t)i0 * lda + j0;
        const double* L1 = (i1 < j0) ? L + (size_t)i1 * lda + j0 : L0;
        double a0 = 0.0, a1 = 0.0;
#pragma unroll 8
        for (int c = lane; c < jb; c += 32) { a0 += L0[c] * ys[c]; a1 += L1[c] * ys[c]; }
        a0 = warp_sum(a0);
        a1 = warp_sum(a1);
        if (lane == 0) {
            rhs[i0] -= a0;
            if (i1 < j0) rhs[i1] -= a1;
        }
    }
}

__global__ void zero_upper_kernel(double* A, int n, int lda) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    int j = blockIdx.y + gridDim.y * blockIdx.z;        // y/z split: n may exceed the 65535 limit of grid.y
    if (j < n && i < n && i < j) A[(size_t)j * lda + i] = 0.0;
}

}  // namespace

void chol_diag_block(double* Akk, int lda, int w, double* dinv, double* X, int ldx, double* T, int* info, int base, cudaStream_t st) {
    if (X && T) factor_diag_with_inverse(Akk, lda, w, dinv, X, ldx, T, info, base, st);
    else potrf_small(Akk, lda, w, dinv, X, ldx, info, base, st);
}

void ensure_aux(CholWork& work) {
    if (work.aux) return;
    int lo = 0, hi = 0;
    LRN_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    LRN_CUDA(cudaStreamCreateWithPriority(&work.aux, cudaStreamNonBlocking, hi));
    LRN_CUDA(cudaStreamCreateWithPriority(&work.aux2, cudaStreamNonBlocking, hi));
    for (auto& e : work.ev) LRN_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
}

// the two trailing-update products of a panel run as Ozaki INT8 products (chol_i8.cu) when the caller opted in: the solved
// panel is sliced into digit planes once, on the panel stream, and both products read the planes
static bool lookahead_i8(int n, int int8) {
    static const bool env_off = [] { const char* e = getenv("LRN_CHOL_INT8"); return e && atoi(e) == 0; }();
    const int NB = pick_nb(n);
    return n > NB && (int8 == 2 || (int8 == 1 && NB == 1024 && !env_off));
}
static int slice_rows(int rows) { return round_up(rows, 128) + 128; }   // room for the 128-row tiles at row offset wq

// Right-looking factorisation with one-step look-ahead on two streams.  The high-priority panel stream runs the whole
// dependency chain -- panel p (one cooperative launch: diagonal block + rows below), then the update of the NEXT panel's
// columns -- while the main stream applies the rest of the trailing update of panel p (columns behind the next panel) on the
// TMA-fed kernel.  Events: evP[p] "panel p is factored" (main stream may update with it), evR[p] "rest update p is done" (the
// panel stream may touch the columns it wrote: the next-columns update of step p+1 also receives rest(p)).
void chol_lookahead(double* A, int n, int lda, CholWork& work, cudaStream_t st) {
    ensure_aux(work);
    cudaStream_t sp = work.aux;
    cudaEvent_t evStart = work.ev[0], evP[2] = {work.ev[1], work.ev[2]}, evR[2] = {work.ev[3], work.ev[4]};
    int* info = work.info_ptr();
    const int NB = pick_nb(n), npan = (int)cdiv(n, NB), gcap = panel_grid_cap(n);
    const bool i8 = lookahead_i8(n, work.int8);
    if (i8) {
        const int r0 = slice_rows(n - NB);
        for (int b = 0; b < 2; b++) {
            if (work.i8_slices[b].n < i8_slice_bytes(r0, NB)) work.i8_slices[b].alloc(i8_slice_bytes(r0, NB));
            if (work.i8_sigma[b].n < (size_t)r0) work.i8_sigma[b].alloc((size_t)r0);
        }
    }
    LRN_CUDA(cudaEventRecord(evStart, st));
    LRN_CUDA(cudaStreamWaitEvent(sp, evStart, 0));
    int last = 0;
    for (int p = 0; p < npan; p++) {
        const int c0 = p * NB, w = (n - c0 < NB) ? (n - c0) : NB, rows = n - c0;
        double* Ap = A + (size_t)c0 * lda + c0;
        double* dk = work.dinv.p + (size_t)(c0 / DB) * DB * DB;
        factor_panel(Ap, w, rows - w, lda, dk, info, c0, gcap, sp);
        const int q0 = c0 + w;
        const double* P = Ap + w;                                           // rows below the diagonal block, lda
        // set p & 1 was last read by the products of panel p - 2; the next-columns update of panel p - 1, which precedes this
        // slicing on the panel stream, waited for rest(p - 2)
        const int rpad = slice_rows(n - q0);
        int8_t* sl = work.i8_slices[p & 1].p;
        const double* sg = work.i8_sigma[p & 1].p;
        if (i8 && q0 < n) i8_slice(P, lda, n - q0, w, rpad, sl, work.i8_sigma[p & 1].p, sp);
        LRN_CUDA(cudaEventRecord(evP[p & 1], sp));
        last = p & 1;
        if (q0 >= n) break;
        const int wq = (n - q0 < NB) ? (n - q0) : NB;
        const int q1 = q0 + wq;
        // rest of the trailing matrix (lower triangle, columns behind the next panel) on the main stream
        LRN_CUDA(cudaStreamWaitEvent(st, evP[p & 1], 0));
        if (q1 < n) {
            if (i8) {
                syrk_update_i8(sl, sg, rpad, w, wq, wq, n - q1, n - q1, A + (size_t)q1 * lda + q1, lda, 0, 0, true, st);
            } else {
                GemmParams g;
                g.A = P + wq; g.B = P + wq; g.C = A + (size_t)q1 * lda + q1;
                g.M = n - q1; g.N = n - q1; g.K = w; g.lda = lda; g.ldb = lda; g.ldc = lda;
                g.transB = true; g.alpha = -1.0; g.beta = 1.0; g.lower = 1;
                gemm(g, st);
            }
        }
        LRN_CUDA(cudaEventRecord(evR[p & 1], st));
        // the next panel's columns on the panel stream (they also received rest(p-1), which must have completed)
        if (p >= 1) LRN_CUDA(cudaStreamWaitEvent(sp, evR[(p - 1) & 1], 0));
        if (i8) syrk_update_i8(sl, sg, rpad, w, 0, 0, n - q0, wq, A + (size_t)q0 * lda + q0, lda, 0, 0, true, sp);
        else gemm_nt(sp, n - q0, wq, w, -1.0, P, lda, P, lda, 1.0, A + (size_t)q0 * lda + q0, lda);
    }
    LRN_CUDA(cudaStreamWaitEvent(st, evP[last], 0));
}

void cholesky_lower(double* A, int n, int lda, CholWork& work, cudaStream_t st) {
    work.ensure(n);
    work.tinv_for = nullptr;
    LRN_CUDA(cudaMemsetAsync(work.info_ptr(), 0, sizeof(int), st));
    if (n <= 0) return;
    if (n >= 1024) chol_lookahead(A, n, lda, work, st);
    else chol_rec(A, n, lda, work.dinv.p, work.info_ptr(), 0, work, st);
}

size_t chol_work_bytes(int n, int int8) {
    const size_t d = sizeof(double);
    size_t bytes = (size_t)cdiv(n, DB) * DB * DB * d + sizeof(int);             // dinv, info
    bytes += (size_t)cdiv(n, SW) * (SW * SW + DB * DB) * d;                     // tinv, tscr (chol_build_tinv)
    if (n >= 1024 && lookahead_i8(n, int8)) {                                   // two slice sets (chol_lookahead)
        const int r0 = slice_rows(n - pick_nb(n));
        bytes += 2 * (i8_slice_bytes(r0, pick_nb(n)) + (size_t)r0 * d);
    }
    return bytes;
}

// inverses of the 256 x 256 diagonal blocks of L: X_ii = D_i, X_ij = -D_i (L[i, j:i] X[j:i, j]) for sub-blocks i > j
void chol_build_tinv(const double* L, int n, int lda, CholWork& work, cudaStream_t st) {
    const int nblk = (int)cdiv(n, SW), nfull = n / SW, tail = n - nfull * SW;
    if (work.tinv.n < (size_t)nblk * SW * SW) work.tinv.alloc((size_t)nblk * SW * SW);
    if (work.tscr.n < (size_t)nblk * DB * DB) work.tscr.alloc((size_t)nblk * DB * DB);
    const int nsb_total = (int)cdiv(n, DB);
    tinv_diag_kernel<<<nsb_total, 256, 0, st>>>(work.dinv.p, work.tinv.p, nsb_total);
    LRN_CHECK_LAUNCH();
    for (int grp = 0; grp < 2; grp++) {
        // group 0: all full blocks in one batch; group 1: the partial last block
        const int b0 = grp ? nfull : 0, cnt = grp ? (tail > 0 ? 1 : 0) : nfull, jb = grp ? tail : SW;
        if (cnt <= 0) continue;
        const int nsb = (int)cdiv(jb, DB);
        const double* Lb = L + (size_t)b0 * SW * lda + (size_t)b0 * SW;
        double* Xb = work.tinv.p + (size_t)b0 * SW * SW;
        const double* Db = work.dinv.p + (size_t)b0 * 4 * DB * DB;
        for (int j = 0; j + 1 < nsb; j++)
            for (int i = j + 1; i < nsb; i++) {
                const int rb = std::min(DB, jb - i * DB), K = DB * (i - j);
                GemmParams g;                       // S = L[i, j:i] X[j:i, j]
                g.A = Lb + (size_t)j * DB * lda + i * DB; g.lda = lda; g.sA = (long long)SW * lda + SW;
                g.B = Xb + (size_t)j * DB * SW + j * DB; g.ldb = SW; g.sB = (long long)SW * SW;
                g.C = work.tscr.p; g.ldc = DB; g.sC = DB * DB;
                g.M = rb; g.N = DB; g.K = K; g.batch = cnt;
                gemm(g, st);
                GemmParams f;                       // X_ij = -D_i S
                f.A = Db + (size_t)i * DB * DB; f.lda = DB; f.sA = 4LL * DB * DB;
                f.B = work.tscr.p; f.ldb = DB; f.sB = DB * DB;
                f.C = Xb + (size_t)j * DB * SW + i * DB; f.ldc = SW; f.sC = (long long)SW * SW;
                f.M = rb; f.N = DB; f.K = rb; f.alpha = -1.0; f.batch = cnt;
                gemm(f, st);
            }
    }
    work.tinv_for = L;
}

static void chol_solve_enqueue(const double* L, int n, int lda, CholWork& work, double* x, double* tmp, int which, cudaStream_t st) {
    const int nstep = (int)cdiv(n, SW);
    for (int dir = 0; dir < 2; dir++) {
        if (!(which & (dir ? 2 : 1))) continue;
        for (int s = 0; s < nstep; s++) {
            const int b = dir ? nstep - 1 - s : s;
            const int j0 = b * SW, jb = (n - j0 < SW) ? (n - j0) : SW;
            const int bn = dir ? b - 1 : b + 1;
            const double* Xn = (bn >= 0 && bn < nstep && (size_t)(bn + 1) * SW * SW <= work.tinv.n) ? work.tinv.p + (size_t)bn * SW * SW : nullptr;
            trsv_diag_kernel<<<1, 1024, 0, st>>>(work.tinv.p + (size_t)b * SW * SW, jb, x + j0, tmp + j0, dir, Xn);
            LRN_CHECK_LAUNCH();
            const int rest = dir ? j0 : n - j0 - jb;
            if (rest <= 0) continue;
            if (!dir) trsv_update_fwd_kernel<<<(unsigned)cdiv(rest, 64), 256, 0, st>>>(L, lda, n, j0, jb, tmp + j0, x);
            else trsv_update_bwd_kernel<<<(unsigned)cdiv(rest, 32), 256, 0, st>>>(L, lda, j0, jb, tmp + j0, x);
            LRN_CHECK_LAUNCH();
        }
        LRN_CUDA(cudaMemcpyAsync(x, tmp, (size_t)n * sizeof(double), cudaMemcpyDeviceToDevice, st));
    }
}

void chol_solve(const double* L, int n, int lda, CholWork& work, double* x, double* tmp, int which, cudaStream_t st) {
    if (n <= 0) return;
    if (work.tinv_for != L) chol_build_tinv(L, n, lda, work, st);
    CholWork::SolveGraph& G = work.sgraph[which & 3];
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (st != nullptr && st != cudaStreamLegacy && st != cudaStreamPerThread) cudaStreamIsCapturing(st, &cap);
    if (cap != cudaStreamCaptureStatusNone) {        // already inside somebody else's capture (the PCG body): plain launches
        chol_solve_enqueue(L, n, lda, work, x, tmp, which, st);
        return;
    }
    const bool capturable = st != nullptr && st != cudaStreamLegacy && st != cudaStreamPerThread && !gemm_profile_active() &&
                            n >= 4 * SW && !G.broken;
    const bool same = G.exec && G.L == L && G.tinv == work.tinv.p && G.x == x && G.tmp == tmp && G.n == n && G.lda == lda;
    if (capturable && same) {
        LRN_CUDA(cudaGraphLaunch(G.exec, st));
        g_kernel_launches.fetch_add(G.nodes);
        return;
    }
    if (!capturable || !G.warm) {                    // small systems, uncapturable streams, and the first solve (eager warm-up)
        chol_solve_enqueue(L, n, lda, work, x, tmp, which, st);
        G.warm = true;
        return;
    }
    if (G.exec) { cudaGraphExecDestroy(G.exec); G.exec = nullptr; }
    bool ok = cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
    if (ok) {
        cudaGraph_t graph = nullptr;
        const long long before = g_kernel_launches.load();
        try { chol_solve_enqueue(L, n, lda, work, x, tmp, which, st); } catch (...) { ok = false; }
        if (cudaStreamEndCapture(st, &graph) != cudaSuccess || !graph) ok = false;
        G.nodes = g_kernel_launches.load() - before;
        g_kernel_launches.fetch_sub(G.nodes);
        if (ok && cudaGraphInstantiate(&G.exec, graph, 0) != cudaSuccess) { ok = false; G.exec = nullptr; }
        if (graph) cudaGraphDestroy(graph);
    }
    if (!ok) {
        cudaGetLastError();
        G.broken = true;
        chol_solve_enqueue(L, n, lda, work, x, tmp, which, st);
        return;
    }
    G.L = L; G.tinv = work.tinv.p; G.x = x; G.tmp = tmp; G.n = n; G.lda = lda;
    LRN_CUDA(cudaGraphLaunch(G.exec, st));
    g_kernel_launches.fetch_add(G.nodes);
}

void trsm_left_lower_trans(const double* L, int n, int lda, const CholWork& work, double* Y, int ldy, int ncols, cudaStream_t st) {
    if (n <= 0 || ncols <= 0) return;
    const int nblk = (int)cdiv(n, DB);
    for (int b = nblk - 1; b >= 0; b--) {
        const int j0 = b * DB, jb = (n - j0 < DB) ? (n - j0) : DB;
        double* Yj = Y + j0;
        // X_j = inv(L_jj)^T Y_j   (in place: one M tile, every CTA reads exactly the columns it writes)
        gemm_tn(st, jb, ncols, jb, 1.0, work.dinv.p + (size_t)b * DB * DB, DB, Yj, ldy, 0.0, Yj, ldy);
        // Y[0:j0, :] -= L[j0:j0+jb, 0:j0]^T X_j
        if (j0 > 0) gemm_tn(st, j0, ncols, jb, -1.0, L + j0, lda, Yj, ldy, 1.0, Y, ldy);
    }
}

void zero_strict_upper(double* A, int n, int lda, cudaStream_t st) {
    if (n <= 1) return;
    const unsigned gy = (unsigned)std::min(n, 32768);
    dim3 grid((unsigned)cdiv(n, 256), gy, (unsigned)cdiv(n, gy));
    zero_upper_kernel<<<grid, 256, 0, st>>>(A, n, lda);
    LRN_CHECK_LAUNCH();
}

}  // namespace lrn
