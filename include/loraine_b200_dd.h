/* loraine_b200_dd.h -- C ABI of the double-double ("Float64x2") LP path of libloraine_b200.so  (SURVEY.md section 8(f), row N4).
 *
 * Scope: `Loraine.Optimizer{Float64x2}` (README.md:37-54 of the reference) on models WITHOUT semidefinite blocks
 * (nlmi = 0, the shape of examples/k.jl:8-38): every array expression of the interior-point iteration runs on the GPU in
 * double-double arithmetic (two doubles per number, ~106 bits; the element type MultiFloats.jl calls Float64x2).
 * Models with PSD blocks are still rejected for element types other than Float64 (no fallback).
 *
 * Conventions: a double-double scalar crosses the boundary as `double v[2]` = {hi, lo} with value hi + lo -- the two limbs of
 * MultiFloats' `Float64x2` (`x._limbs`); a vector as two parallel arrays hi[], lo[] (lo may be NULL on input: exact doubles).
 * Index arrays are 1-based CSC like in loraine_b200.h.  Return codes as in loraine_b200.h (0 ok, < 0 error with
 * lrn_dd_last_error(), > 0 pivot index of a failed Cholesky).  Each entry point cites the reference lines it replaces.
 */
#ifndef LORAINE_B200_DD_H
#define LORAINE_B200_DD_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct lrn_dd_solver* lrn_dd_handle_t;

/* MySolver{Float64x2} state for nlmi = 0: n_var multipliers y, nlin LP rows (src/Solvers.jl:363-446).  device < 0: current */
int32_t lrn_dd_create(lrn_dd_handle_t* out, int64_t n_var, int64_t nlin, int32_t device);
/* Multi-GPU, in-process: one host thread drives `ngpus` devices (devices[r], or 0 .. ngpus-1 when devices is NULL); the NCCL
 * communicator is made inside the library (ncclCommInitAll).  Returns a facade that every other lrn_dd_* entry point accepts:
 * each call runs on every device, host-visible outputs come from the first.  The Schur matrix is assembled and factored
 * row-block-cyclically over the devices (row blocks of 256 rows for n_var >= 4096, 128 for n_var >= 1024, 64 otherwise), the
 * rest of the iteration is replicated; results equal the single-GPU ones bit for bit.  ngpus == 1: same as lrn_dd_create;
 * ngpus <= 0: every visible device; more than visible: LRN_ERR_ARG; no device: LRN_ERR_NO_DEVICE (no CPU fallback). */
int32_t lrn_dd_create_multi(lrn_dd_handle_t* out, int64_t n_var, int64_t nlin, int32_t ngpus, const int32_t* devices);
/* Multi-GPU, one process per GPU: attach the handle to rank `rank` of a `world`-rank NCCL communicator; unique_id128 comes
 * from lrn_dist_unique_id (loraine_b200.h) on rank 0 and is passed to every rank.  Call after lrn_dd_create, before the
 * first lrn_dd_schur_assemble.  From then on lrn_dd_schur_factor is a collective (every rank calls it, in the same order as
 * the others), and so is lrn_dd_get_array(h, 1, ...).  world = 1 runs the distributed code path on one GPU. */
int32_t lrn_dd_dist_init(lrn_dd_handle_t h, int32_t rank, int32_t world, const void* unique_id128);
/* C_lin (n_var x nlin, CSC, 1-based) and d_lin, src/model.jl:70-84 */
int32_t lrn_dd_set_lin(lrn_dd_handle_t h, const int64_t* colptr, const int64_t* rowval, const double* nz_hi, const double* nz_lo,
                       const double* d_hi, const double* d_lo);
int32_t lrn_dd_set_b(lrn_dd_handle_t h, const double* b_hi, const double* b_lo);
int32_t lrn_dd_finalize(lrn_dd_handle_t h);
int32_t lrn_dd_destroy(lrn_dd_handle_t h);
const char* lrn_dd_last_error(lrn_dd_handle_t h);

/* iterate after initial_point (src/initial_point.jl:48-73): y, X_lin, S_lin */
int32_t lrn_dd_set_iterate(lrn_dd_handle_t h, const double* y_hi, const double* y_lo, const double* x_hi, const double* x_lo,
                           const double* s_hi, const double* s_lo);
int32_t lrn_dd_get_solution(lrn_dd_handle_t h, double* y_hi, double* y_lo, double* x_hi, double* x_lo, double* s_hi, double* s_lo);

/* find_mu, src/Solvers.jl:480-494: mu = dot(X_lin, S_lin) / nlin */
int32_t lrn_dd_find_mu(lrn_dd_handle_t h, double mu[2]);
/* prepare_W for the LP block, src/prepare_W.jl:88-92: Si_lin = 1 ./ S_lin */
int32_t lrn_dd_prepare_W(lrn_dd_handle_t h);
/* Rp = b - C_lin X_lin, Rd_lin = d_lin - S_lin - C_lin' y, src/predictor_corrector.jl:8-22 */
int32_t lrn_dd_residuals(lrn_dd_handle_t h);
/* BBBB = C_lin spdiagm(X_lin .* S_lin_inv) C_lin', src/predictor_corrector.jl:36-39 */
int32_t lrn_dd_schur_assemble(lrn_dd_handle_t h);
/* h = Rp + C_lin ((X_lin .* Si_lin) .* Rd_lin + X_lin), src/predictor_corrector.jl:43-50 */
int32_t lrn_dd_rhs_predictor(lrn_dd_handle_t h);
/* corrector right-hand side, src/predictor_corrector.jl:183-192 */
int32_t lrn_dd_rhs_corrector(lrn_dd_handle_t h, const double sigma[2], const double mu[2]);
/* cholesky(Hermitian(BBBB,:L)), src/predictor_corrector.jl:57,85; k > 0: pivot k not positive */
int32_t lrn_dd_schur_factor(lrn_dd_handle_t h);
/* BBBB += delta I, src/predictor_corrector.jl:74 */
int32_t lrn_dd_schur_shift(lrn_dd_handle_t h, double delta);
/* dely = L' \ (L \ h) (which = 3) or (L L')^-1 (L L')^-1 h (which = 6, the regularised-path quirk), src/predictor_corrector.jl:85-90,199.
 * LRN_ERR_STATE when there is no valid factor (no lrn_dd_schur_factor since the Schur matrix changed, or it failed). */
int32_t lrn_dd_schur_solve(lrn_dd_handle_t h, int32_t which);
/* find_step_lin, src/predictor_corrector.jl:329-364.  predict != 0: Xn_lin, Sn_lin, RNT_lin; else the iterate is updated. */
int32_t lrn_dd_find_step(lrn_dd_handle_t h, int32_t predict, const double sigma[2], const double mu[2], double tau,
                         double alpha_lin[2], double beta_lin[2]);
/* dot(Xn_lin, Sn_lin) for sigma_update, src/predictor_corrector.jl:163-166 */
int32_t lrn_dd_sigma_trace(lrn_dd_handle_t h, double dot_lin[2]);
/* check_convergence arithmetic for nlmi = 0, src/Solvers.jl:496-523: err[6][2], b'y, d'x */
int32_t lrn_dd_dimacs(lrn_dd_handle_t h, double err6[12], double by[2], double dx[2]);

/* parity hook: which = 1 H (n x n, column-major, lower mirrored), 2 L (lower), 3 Rp, 4 Rd_lin, 5 rhs h, 6 dely, 7 delX_lin,
 * 8 delS_lin, 9 Xn_lin, 10 Sn_lin, 11 RNT_lin, 12 Si_lin.  On a multi-GPU handle H is gathered from the row shards of all
 * ranks (exact: the shards are disjoint); with lrn_dd_dist_init that makes which = 1 a collective that every rank must call
 * (hi may be NULL on the ranks that do not want the copy). */
int32_t lrn_dd_get_array(lrn_dd_handle_t h, int32_t which, double* hi, double* lo);
/* device milliseconds since the last reset: [0] schur_assemble, [1] schur_factor, [2] schur_solve, [3] everything else */
int32_t lrn_dd_timers(lrn_dd_handle_t h, double ms[4], int32_t reset);

#ifdef __cplusplus
}
#endif
#endif
