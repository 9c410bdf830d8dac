/* loraine_b200 -- test / benchmark hooks onto the library's dense primitives (not part of the drop-in boundary).
 * All pointers are HOST pointers (column-major, leading dimension = rows); the hooks stage through device memory
 * with the library's padded leading dimensions so that the tests exercise the same code paths as the solver. */
#ifndef LORAINE_B200_DEBUG_H
#define LORAINE_B200_DEBUG_H
#include <stdint.h>
#include "loraine_b200.h"
#include "loraine_b200_dd.h"
#ifdef __cplusplus
extern "C" {
#endif

/* C = alpha*op(A)*op(B)[.*colscale] + beta*C (mode 0) or C = beta*C + alpha*(op(A)op(B)).^2 (mode 1); mode | 2: the caller
 * promises op(A)(i,k) = 0 for k < i and op(B)(k,j) = 0 for k < j (tiles skip that part of the K loop); lower != 0 computes
 * only tiles that intersect the lower triangle.  misalign != 0 offsets the device buffers by 8 bytes (exercises the
 * unaligned cp.async path).  reps > 0: the kernel is timed over `reps` launches (CUDA events) into *ms_per_launch. */
int32_t lrn_dbg_gemm(int32_t M, int32_t N, int32_t K, int32_t transA, int32_t transB, double alpha, const double* A,
                     const double* B, double beta, double* C, int32_t mode, int32_t lower, const double* colscale,
                     int32_t misalign, int32_t reps, double* ms_per_launch);
/* A (n x n, symmetric, lower used) -> L in the lower triangle (upper zeroed); x (n) <- solve per `which` (0 = skip) */
int32_t lrn_dbg_cholesky(int32_t n, double* A, double* x, int32_t which, int32_t* info, int32_t reps, double* ms_factor);
/* trailing updates of lrn_dbg_cholesky: 0 = DMMA (default), 1 = Ozaki INT8 products when the panels are 1024 wide (n >= 16384;
 * the Schur factor's default, off under LRN_CHOL_INT8=0), 2 = Ozaki INT8 products at every panel width (n >= 1024) */
int32_t lrn_dbg_chol_int8(int32_t mode);
/* the Ozaki INT8 product alone: P (rows x K, K <= 1024) is sliced into digit planes and C (M x N) -= P[a_row0 + i, :] P[b_row0 + j, :]^T
 * (a_row0, b_row0 multiples of 8; rows beyond `rows` read as zero).  lower != 0: only 128 x 64 tiles that meet the lower triangle
 * of a symmetric matrix in which C(0, 0) sits at (row0, col0).  sigma (optional, rows) receives the row scales.  reps > 0: the
 * update is timed over `reps` further launches (they keep subtracting from the device copy of C) into *ms_per_launch. */
int32_t lrn_dbg_syrk_i8(int32_t rows, int32_t K, const double* P, int32_t a_row0, int32_t b_row0, int32_t M, int32_t N, int64_t row0,
                        int64_t col0, int32_t lower, double* C, double* sigma, int32_t reps, double* ms_per_launch);
/* symmetric n <= 64: eigenvalues (descending) and eigenvectors */
int32_t lrn_dbg_eig_small(int32_t n, const double* A, double* evals, double* V, int32_t relative);
/* one-sided block Jacobi SVD of the m x m matrix A: UD = U*diag(sigma), V (NULL: not accumulated), sigma (descending) */
int32_t lrn_dbg_svd(int32_t m, const double* A, double* UD, double* V, double* sigma, double tol, int32_t* sweeps, double* ms);
/* Lanczos extreme eigenpairs of the symmetric m x m matrix T */
int32_t lrn_dbg_lanczos(int32_t m, const double* T, int32_t nev_top, double tol, double* lmin, double* lmax,
                        double* top_vals, double* top_vecs, int32_t* iters, int32_t* converged);
/* batched smallest eigenvalue of `count` symmetric m x m matrices stored one after the other (tridiagonalisation kernel) */
int32_t lrn_dbg_batched_lambda_min(int32_t count, int32_t m, const double* mats, double* out);
/* device micro-benchmarks: kind 0 = DMMA (mma.sync m8n8k4 f64) register-resident peak, 1 = DFMA peak, 2 = HBM copy GB/s */
int32_t lrn_dbg_peak(int32_t kind, double* value);

/* per-launch timing of the DMMA GEMM kernel (roofline bookkeeping of bench.py): mode 1 starts recording one CUDA-event pair
 * per launch on the launching stream, mode 0 stops and returns total kernel milliseconds, algorithmic flops and launches;
 * modes 10 / 11 / 12 return the same totals of the last stopped profile for the cp.async kernel / the TMA-fed kernel / the
 * block-Jacobi panel-rotation kernel alone */
int32_t lrn_dbg_gemm_profile(int32_t mode, double* ms, double* flops, int64_t* launches);

/* test hook (runs WITHOUT a device): the host-side model preparation of lrn_create_from_triplets; hands one prepared matrix back
 * as 0-based CSC.  which: 0 = AA_iblk (n_var x m^2), 1 = C_iblk (m x m), 2 = B_iblk (n_var x m, datarank = -1), 3 = C_lin
 * (n_var x nlin); vec_out (optional) receives b (which 0..2) or d_lin (which 3).  Returns the number of stored entries or < 0. */
int64_t lrn_dbg_model_block(int64_t n_var, int64_t nblocks, const int64_t* blocksizes, int64_t ntrip, const int64_t* tk,
                            const int64_t* tblk, const int64_t* ti, const int64_t* tj, const double* tv, const double* c,
                            int32_t datarank, int64_t iblk, int32_t which, int64_t cap, int64_t* colptr_out, int64_t* rowval_out,
                            double* nzval_out, double* vec_out);
/* test hook: give a single-GPU handle the Schur-row ownership of `rank` out of `world` (row blocks of `block_rows` rows, 0 =
 * the library's default for n_var) WITHOUT a communicator: lrn_schur_assemble then fills only the owned row blocks, so a test
 * on one GPU can check that the shards of all ranks add up to the full matrix.  lrn_schur_factor refuses to run in that state. */
int32_t lrn_dbg_set_shard(lrn_handle_t h, int32_t rank, int32_t world, int32_t block_rows);
/* the same for a double-double LP handle (loraine_b200_dd.h): block_rows a multiple of 32 (0 = the library's default for n_var).
 * lrn_dd_schur_assemble then writes the owned rows of the lower triangle only (zeros elsewhere, no upper mirror),
 * lrn_dd_get_array(h, 1, ...) returns that shard, and lrn_dd_schur_factor fails with LRN_ERR_STATE. */
int32_t lrn_dd_dbg_set_shard(lrn_dd_handle_t h, int32_t rank, int32_t world, int32_t block_rows);
/* test hook: load an array of a double-double LP handle directly, so that the factorisation and the solves can be checked on
 * matrices whose factor is known exactly.  Ids as in lrn_dd_get_array; lo may be NULL (exact doubles).
 *   which = 1: the Schur matrix H (n_var x n_var, symmetric, column-major, full).  No iterate is needed; the handle then holds
 *              a Schur matrix and no factor.  A sharded handle keeps only its own rows of the lower triangle (zeros
 *              elsewhere), the state lrn_dd_schur_assemble leaves, so lrn_dd_schur_factor runs the distributed path.
 *   which = 5: the right-hand side h of lrn_dd_schur_solve (n_var).
 * On a lrn_dd_create_multi handle every device receives the same array.  Any other id: LRN_ERR_ARG. */
int32_t lrn_dd_dbg_set_array(lrn_dd_handle_t h, int32_t which, const double* hi, const double* lo);
/* test hook: the number of CTAs of the multi-CTA triangular solves of lrn_dd_schur_solve.  0 = the single-CTA kernels,
 * -1 = the value lrn_dd_create chose, >= 1 = that many, clamped to the lrn_dd_create value (every CTA must stay resident:
 * the CTAs wait on each other's results).  Fewer CTAs than row tiles make one CTA solve several tiles. */
int32_t lrn_dd_dbg_set_trsv_ctas(lrn_dd_handle_t h, int32_t ctas);
/* test hook for the kit = 1 H_alpha preconditioner, whose build forms T (n_var x erank sum m_i) and A_j u_r (n_var x max m_i)
 * `rows` rows at a time: set_rows > 0 forces that slab height (clamped to n_var; 1 and odd heights are allowed), 0 restores the
 * automatic height (n_var when both whole arrays fit 2 GiB, otherwise the largest multiple of 8 that does).  *rows_used
 * (optional) receives the height the last lrn_prec_prepare(h, 1) used (0 before the first).  A lrn_create_multi handle sets
 * every member and reports member 0. */
int32_t lrn_dbg_prec_slab(lrn_handle_t h, int64_t set_rows, int64_t* rows_used);
/* relative Frobenius distance ||A_a - A_b||_F / ||A_b||_F over the LOWER triangles of the n_var x n_var Schur matrices
 * (which = LRN_ARR_H) or Cholesky factors (LRN_ARR_L) of two handles living on the same device; computed on the device
 * (bench.py's dist_parity: sharded handle against a single-GPU handle at n_var = 40000 without a 12.8 GB download) */
int32_t lrn_dbg_compare(lrn_handle_t a, lrn_handle_t b, int32_t which, double* relerr);
/* multi-GPU: sum the row-block shards of the Schur matrix over all ranks in place (collective; every rank calls).
 * LRN_ERR_STATE on a handle in the own-rows layout (it holds no full matrix); so does lrn_dbg_compare. */
int32_t lrn_dbg_gather_H(lrn_handle_t h);
/* test hook: storage layout of the kit = 0 Schur matrix H and its factor L.  force (before lrn_finalize): -1 lrn_finalize
 * decides (default), 0 replicated (n_var rows on every rank), 1 own rows (only the rank's own row blocks, stacked; the sharded
 * assembly, lrn_dist_init / lrn_dbg_set_shard ownership, must be set before lrn_finalize); -2 leaves the setting.  *layout
 * (optional) receives the layout in use: 0, 1, or -1 before lrn_finalize.  A group handle sets every member, reports member 0. */
int32_t lrn_dbg_schur_layout(lrn_handle_t h, int32_t force, int32_t* layout);
/* test hook: layout of the PSD block state.  force (before lrn_finalize): -1 lrn_finalize decides (default: distributed when
 * kit = 0, nlmi >= 2 and the handle has a communicator with world > 1), 0 replicated (every rank holds every block), 1
 * distributed (block i on rank block_owner(msizes, world)[i]; needs kit = 0 and such a communicator, or lrn_finalize fails);
 * -2 leaves the setting.  *layout (optional) receives the layout in use: 0, 1, or -1 before lrn_finalize.  A group handle
 * sets every member and reports member 0. */
int32_t lrn_dbg_block_layout(lrn_handle_t h, int32_t force, int32_t* layout);
/* test hook: the device bytes lrn_finalize counts for the kit = 0 state of group member `member` (0 for a plain handle) in its
 * Schur layout, with the PSD blocks replicated (sharded = 0) or distributed (1), into *bytes (optional); held (optional, nlmi
 * entries) receives per block the bytes of the m x m arrays and m-vectors the member holds for it: a block of another rank
 * keeps only its gathered W (G when datarank = -1). */
int32_t lrn_dbg_block_footprint(lrn_handle_t h, int32_t member, int32_t sharded, int64_t* bytes, int64_t* held);
/* test hook: group member `member`'s own device copy (0 for a plain handle) of W (which = LRN_ARR_W) or G (LRN_ARR_G) of block
 * iblk, m x m into out, without any collective: with distributed blocks a non-owner holds the copy the all-gather of
 * lrn_prepare_W gave it (W, or G when datarank = -1); LRN_ERR_ARG when the member holds no such array. */
int32_t lrn_dbg_member_block(lrn_handle_t h, int32_t member, int64_t iblk, int32_t which, double* out);
/* test hook: the device bytes lrn_finalize counts for the kit = 0 state of this handle (its rank, world and block height)
 * in the replicated (rows_local = 0) or the own-rows layout (1).  A group handle reports member 0. */
int32_t lrn_dbg_schur_footprint(lrn_handle_t h, int32_t rows_local, int64_t* bytes);
/* test hook: load the kit = 0 Schur matrix H (n_var x n_var, column-major, host; the lower triangle is used) into the
 * handle's layout: a replicated handle takes all of it, an own-rows handle its own row blocks; every member of a group
 * handle reads the same array.  lrn_schur_factor then factors it (checks of the factorisation on known matrices). */
int32_t lrn_dbg_set_H(lrn_handle_t h, const double* H);
/* test hook: the lrn_create_multi facade with `world` (1..8) members that all live on the CURRENT device and exchange data
 * through an in-process loopback transport instead of NCCL (host rendezvous of the member threads, device-to-device copies;
 * a member that does not arrive within 120 s makes the collective fail).  The peer-memory exchange is off.  block_rows: row
 * block height of the Schur distribution (a multiple of 64, at most 512; 0 = the library's default for n_var).  Lets world =
 * 2 or 3 of the distributed factorisation and solves run on one GPU. */
int32_t lrn_dbg_create_loopback(lrn_handle_t* out, int64_t n_var, int64_t nlmi, const int64_t* msizes, int64_t nlin,
                                const lrn_options_t* opt, int32_t world, int32_t block_rows);

#ifdef __cplusplus
}
#endif
#endif
