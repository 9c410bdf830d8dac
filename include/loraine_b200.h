/* loraine_b200 -- C ABI of the B200-native replacement of Loraine.jl's per-iteration linear-algebra hot path.
 *
 * The reference (kocvara/Loraine.jl v0.2.5, pure Julia) has no FFI boundary; the seams this ABI replaces are the Julia
 * method bodies listed next to every entry point below (paths relative to the reference root).  The Julia host keeps the
 * control flow of src/predictor_corrector.jl and src/Solvers.jl:304-361,448-478 and calls these functions with `ccall`
 * (see INTEGRATION.md and julia/LoraineB200.jl).
 *
 * Conventions
 *   - every function returns int32: 0 = ok; > 0 = LAPACK-style "leading minor of order k is not positive definite"
 *     (maps to Julia's PosDefException(k)); < 0 = argument / CUDA / NCCL error, message via lrn_last_error().
 *   - dense matrices are column-major Float64 with leading dimension = number of rows (Julia `Matrix{Float64}`).
 *   - sparse matrices are Julia `SparseMatrixCSC{Float64,Int64}` fields passed raw: 1-based colptr (ncol+1), 1-based
 *     rowval, nzval.  vec index of entry (p,q) of an m x m block is p + (q-1) m (src/model.jl:219).
 *   - host pointers are only read/written during the call; the library keeps no host pointer.  All device memory is owned
 *     by the handle.  Calls are synchronous with respect to every host-visible output.
 *   - Float64 is the only element type (Optimizer{Float64xN} must be rejected on the Julia side before reaching the ABI).
 *   - there is NO CPU fallback: lrn_create fails with LRN_ERR_NO_DEVICE when no sm_100 GPU is usable.
 */
#ifndef LORAINE_B200_H
#define LORAINE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct lrn_solver* lrn_handle_t;

#define LRN_OK 0
#define LRN_ERR_ARG (-1)
#define LRN_ERR_CUDA (-2)
#define LRN_ERR_NO_DEVICE (-3)
#define LRN_ERR_STATE (-4)
#define LRN_ERR_NCCL (-5)
#define LRN_ERR_UNSUPPORTED (-6)

/* Options = the subset of DEFAULT_OPTIONS (src/Solvers.jl:169-185) that selects hot-path branches. */
typedef struct lrn_options {
    int32_t kit;            /* 0 direct (Cholesky), 1 CG                                   */
    int32_t datarank;       /* 0 general Schur assembly, -1 rank-one path (makeBBBB_rank1) */
    int32_t preconditioner; /* 0 none, 1 H_alpha, 2 H_beta, 4 hybrid (starts as H_beta)    */
    int32_t erank;          /* expected rank for H_alpha                                   */
    int32_t aamat;          /* 0..3, tau / AAAATtau variant (src/Solvers.jl:646-655,715-739) */
    int32_t datasparsity;   /* kappa of prep_sparse! (src/model.jl:153-174); only used when schur_split = 1 */
    int32_t schur_split;    /* 0 = cost model picks F1/F3 per matrix (default), 1 = reference rule nnz > kappa -> F1 */
    int32_t rank1_mode;     /* 0 = SpMM + DMMA SYRK with squared epilogue (reference formulation) */
    double svd_tol;         /* block-Jacobi stopping level of max |u_i.u_j|/(|u_i||u_j|) over the rotated columns (0 -> default 1e-8), measured
                             * at the START of the last sweep (quadratic convergence: ~1e-14 after it).  Blocks with m >= 1024 may stop one
                             * sweep earlier when a Gram product shows the columns are already orthogonal to 1e4 svd_tol^2 */
    double lanczos_tol;     /* relative Ritz residual for lambda_min (0 -> default 1e-8) */
    int32_t device;         /* CUDA device ordinal, -1 = current / LOCAL_RANK */
    int32_t reserved;
} lrn_options_t;

void lrn_default_options(lrn_options_t* opt);

/* ---- construction: replaces MyModel / MySolver storage (src/model.jl:34-87, src/Solvers.jl:18-147, :363-446) ---- */
/* Limits on n_var: kit = 0 forms the dense n_var x n_var Schur matrix and its factor on every GPU, so 1 <= n_var <= 140 000
 * (LRN_ERR_ARG "n_var out of range (1..140000)"), and lrn_finalize returns LRN_ERR_ARG, naming the bytes needed and the bytes
 * free, when they, the Cholesky workspace and the model do not fit the device's free memory (near n_var = 100 000 on a
 * 180 GB B200, for any number of GPUs).  kit = 1 forms neither: 1 <= n_var <= 2^31 - 1, and lrn_finalize returns
 * LRN_ERR_ARG, naming the bytes needed and the bytes free, when the CG state does not fit the device's free memory.  With an
 * LP block and n_var > 140 000, lrn_prec_prepare(h, 1) (H_alpha) returns LRN_ERR_UNSUPPORTED; kinds 2 and 4 run. */
int32_t lrn_create(lrn_handle_t* out, int64_t n_var, int64_t nlmi, const int64_t* msizes, int64_t nlin,
                   const lrn_options_t* opt);
/* AA[i] (n_var x m_i^2, row k = vec(calA_{i,k}), math sign), as built by prep_AA! (src/model.jl:199-229) */
int32_t lrn_set_block_AA(lrn_handle_t h, int64_t iblk, const int64_t* colptr, const int64_t* rowval, const double* nzval);
/* C[i] (m_i x m_i sparse, = -A[i,1], src/model.jl:133) */
int32_t lrn_set_block_C(lrn_handle_t h, int64_t iblk, const int64_t* colptr, const int64_t* rowval, const double* nzval);
/* B[i] (n_var x m_i, row k = b_k with A[i,k+1] = b_k b_k', src/model.jl:176-197); only for datarank = -1 */
int32_t lrn_set_block_B(lrn_handle_t h, int64_t iblk, const int64_t* colptr, const int64_t* rowval, const double* nzval);
/* C_lin (n_var x nlin) and d_lin (src/MOI_wrapper.jl:149,217) */
int32_t lrn_set_lin(lrn_handle_t h, const int64_t* colptr, const int64_t* rowval, const double* nzval, const double* d_lin);
int32_t lrn_set_b(lrn_handle_t h, const double* b);
/* builds the device-side sparse structures; must be called once after the setters */
int32_t lrn_finalize(lrn_handle_t h);
int32_t lrn_destroy(lrn_handle_t h);
/* problem dimensions of a handle (a host that loaded the model with lrn_load_sdpa has no other way to know them):
 * msizes (optional) receives nlmi block sizes */
int32_t lrn_get_dims(lrn_handle_t h, int64_t* n_var, int64_t* nlmi, int64_t* nlin, int64_t* msizes);
const char* lrn_last_error(lrn_handle_t h);

/* ---- model preparation inside the library (replaces the per-nonzero triplet builder of MOI.copy_to, src/MOI_wrapper.jl:152-209,
 * and _prepare_A / prep_AA! / prep_B / prep_sparse!, src/model.jl:120-229) ----
 * Triplets in SDPA convention: problem  min c'y  s.t.  sum_k F_k y_k - F_0 >= 0 ; entry t says F_{tk[t]} (0 = F_0) has value
 * tv[t] at (ti[t], tj[t]) (1-based, ONE triangle given, mirrored by the library) of block tblk[t] (1-based); blocksizes[b] > 0 is
 * a PSD block, < 0 a diagonal (LP) block of -blocksizes[b] rows.  The handle comes back finalized (no lrn_set_* / lrn_finalize
 * calls needed).  opt->datarank = -1 runs the rank-one conversion of prep_B and fails with LRN_ERR_ARG when a matrix is not
 * rank one within 5e-6 (the reference throws).  ngpus: 1 = one device, otherwise as lrn_create_multi. */
int32_t lrn_create_from_triplets(lrn_handle_t* out, int64_t n_var, int64_t nblocks, const int64_t* blocksizes, int64_t ntrip,
                                 const int64_t* tk, const int64_t* tblk, const int64_t* ti, const int64_t* tj, const double* tv,
                                 const double* c, const lrn_options_t* opt, int32_t ngpus);
/* the same from an SDPA sparse file (.dat-s), as examples/solve_sdpa.jl:14-34 does through MOI.FileFormats.SDPA */
int32_t lrn_load_sdpa(lrn_handle_t* out, const char* path, const lrn_options_t* opt, int32_t ngpus);
/* find_initial!, src/initial_point.jl:17-81: X_i = Eps_i I, S_i = Eta_i I, y = 0, x_lin = Epss, s_lin = Etaa on the device
 * (the norms of the model data it needs are recorded by lrn_finalize); initpoint as in DEFAULT_OPTIONS */
int32_t lrn_initial_point(lrn_handle_t h, int32_t initpoint);

/* ---- iterate upload / download (initial_point.jl output in; MOI getters out, src/MOI_wrapper.jl:315-354) ---- */
int32_t lrn_set_iterate(lrn_handle_t h, const double* const* X, const double* const* S, const double* y,
                        const double* x_lin, const double* s_lin);
/* With the PSD blocks distributed over the ranks (kit = 0, several blocks, a communicator attached before lrn_finalize) each
 * block lives on one owner rank: lrn_set_iterate reads every block and keeps the owned ones; on a one-process-per-GPU handle
 * lrn_get_solution, lrn_get_slack and the per-block ids of lrn_get_array are collectives (every rank calls them with the same
 * blocks requested; the owner broadcasts each block), a lrn_create_multi handle reads each block from its owner. */
int32_t lrn_get_solution(lrn_handle_t h, double* y, double* const* X, double* x_lin);
int32_t lrn_get_slack(lrn_handle_t h, double* const* S, double* s_lin);

/* ---- per-iteration hot path ---- */
/* find_mu, src/Solvers.jl:480-494 */
int32_t lrn_find_mu(lrn_handle_t h, double* mu);
/* prepare_W + try_cholesky, src/prepare_W.jl:5-94.  *status4 = 1 when X or S could not be made positive definite */
int32_t lrn_prepare_W(lrn_handle_t h, int32_t* status4);
/* residuals Rp, Rd_i, Rd_lin, src/predictor_corrector.jl:8-22 */
int32_t lrn_residuals(lrn_handle_t h);
/* makeBBBB_rank1 | makeBBBBs (+ LP term), src/predictor_corrector.jl:24-40, src/makeBBBB.jl:1-218 */
int32_t lrn_schur_assemble(lrn_handle_t h);
/* predictor right-hand side: makeRHS + LP part, src/predictor_corrector.jl:43-50, src/makeBBBB.jl:221-228 */
int32_t lrn_rhs_predictor(lrn_handle_t h);
/* corrector right-hand side, src/predictor_corrector.jl:183-192 */
int32_t lrn_rhs_corrector(lrn_handle_t h, double sigma, double mu);
/* cholesky(Hermitian(BBBB,:L)), src/predictor_corrector.jl:57,85.  Returns k > 0 when not positive definite. */
int32_t lrn_schur_factor(lrn_handle_t h);
/* BBBB += delta*I, src/predictor_corrector.jl:74 */
int32_t lrn_schur_shift(lrn_handle_t h, double delta);
/* dely = op(h): which = 1: L\h, 2: L'\h, 3: L'\(L\h), 6: (LL')^-1 (LL')^-1 h (the reference's regularised-path quirk,
 * src/predictor_corrector.jl:85-90 with a `Cholesky` object whose adjoint is itself) */
int32_t lrn_schur_solve(lrn_handle_t h, int32_t which);
/* Prec_for_CG_tilS_prep (kind 1) / Prec_for_CG_beta (kind 2 or 4), src/Solvers.jl:624-663, 674-864 */
int32_t lrn_prec_prepare(lrn_handle_t h, int32_t kind);
/* dely = cg(MyA, h; tol, maxIter, precon), src/predictor_corrector.jl:134,235 (ConjugateGradients.jl recurrence),
 * operator src/Solvers.jl:572-614, preconditioners :616-622, :665-672, :866-904.  kind 0 none, 1 H_alpha, 2/4 H_beta */
int32_t lrn_pcg(lrn_handle_t h, double tol, int64_t max_iter, int32_t kind, int64_t* num_iters, int32_t* exit_code);
/* find_step + find_step_lin, src/predictor_corrector.jl:248-364.  predict != 0: computes Xn, Sn, RNT; else updates y, X, S.
 * alpha/beta: per-block step lengths (length nlmi); *_lin as in the reference (1.0 when nlin = 0). */
int32_t lrn_find_step(lrn_handle_t h, int32_t predict, double sigma, double mu, double tau, double* alpha, double* beta,
                      double* alpha_lin, double* beta_lin);
/* btrace(Xn,Sn) and dot(Xn_lin,Sn_lin) for sigma_update, src/predictor_corrector.jl:159-168 */
int32_t lrn_sigma_trace(lrn_handle_t h, double* tr_XnSn, double* dot_lin);
/* check_convergence arithmetic, src/Solvers.jl:496-523: err[6], b'y, <C,X>, d'x */
int32_t lrn_dimacs(lrn_handle_t h, double* err6, double* by, double* trCX, double* dx);

/* ---- parity hooks (tests) ---- */
#define LRN_ARR_H 1      /* Schur matrix, n_var x n_var, lower mirrored to full   */
#define LRN_ARR_L 2      /* Cholesky factor (lower, upper zeroed)                 */
#define LRN_ARR_RHS 3    /* current right-hand side h (n_var)                     */
#define LRN_ARR_DELY 4
#define LRN_ARR_RP 5
#define LRN_ARR_W 10     /* per block m x m: */
#define LRN_ARR_G 11
#define LRN_ARR_GI 12
#define LRN_ARR_SI 13
#define LRN_ARR_D 14     /* per block m */
#define LRN_ARR_DDSI 15
#define LRN_ARR_RD 16
#define LRN_ARR_DELX 17
#define LRN_ARR_DELS 18
#define LRN_ARR_RNT 19
#define LRN_ARR_XN 20
#define LRN_ARR_SN 21
int32_t lrn_get_array(lrn_handle_t h, int32_t which, int64_t iblk, double* out);
/* apply the CG operator / preconditioner once: out = A x (kind -1) or out = M^-1 x (kind 0,1,2) */
int32_t lrn_apply_operator(lrn_handle_t h, int32_t kind, const double* x, double* out);

/* ---- instrumentation ---- */
#define LRN_T_PREPARE_W 0
#define LRN_T_RESIDUALS 1
#define LRN_T_ASSEMBLE 2
#define LRN_T_RHS 3
#define LRN_T_FACTOR 4
#define LRN_T_SOLVE 5
#define LRN_T_FIND_STEP 6
#define LRN_T_PREC 7
#define LRN_T_CG 8
#define LRN_T_DIMACS 9
#define LRN_T_SVD 10
#define LRN_T_EIGMIN 11
#define LRN_T_COUNT 12
/* accumulated device milliseconds (CUDA events on the library stream) and call counts per phase; reset != 0 clears */
int32_t lrn_timers(lrn_handle_t h, double* ms, int64_t* calls, int32_t reset);
/* name of a phase under the reference's TimerOutputs section names where one exists ("prep W", "BBBBs" -- "BBBB_rank1" when
 * rank1 != 0 --, "prep W SVD", "prec", src/makeBBBB.jl:2,30, src/prepare_W.jl:37, src/Solvers.jl:676); NULL when out of range */
const char* lrn_timer_name(int32_t phase, int32_t rank1);
/* number of kernels launched by the library through this handle's process so far */
int64_t lrn_kernel_launches(void);
/* change an option after creation (the reference mutates solver.aamat / solver.preconditioner in the hybrid switch,
 * src/Solvers.jl:339-347): name in {"aamat", "erank", "svd_tol", "lanczos_tol", "sparse_op"}; sparse_op: 0 = dense W M W form of the
 * kit = 1 Schur operator, 1 = sparse-aware form wherever the data is stored symmetrically, -1 = automatic (default) */
int32_t lrn_set_option(lrn_handle_t h, const char* name, double value);
/* diagnostic counters of the last calls: [0] svd sweeps, [1] lanczos iterations (sum), [2] lanczos not converged count */
int32_t lrn_stats(lrn_handle_t h, int64_t* out3);

/* ---- multi-GPU, in-process: ONE host thread drives `ngpus` devices through one handle (SURVEY 8(b): the unchanged
 * single-process Loraine.Optimizer, src/MOI_wrapper.jl:136-140, can use the whole box).  The library creates one solver per
 * device (devices[r], or 0..ngpus-1 when devices is NULL) and their NCCL communicators with ncclCommInitAll; every other
 * entry point accepts the returned handle unchanged and fans the call out to the devices (Schur rows and the Cholesky
 * factorisation are sharded block-cyclically, the m x m work of the iteration is replicated).  ngpus <= 0: all devices. ---- */
int32_t lrn_create_multi(lrn_handle_t* out, int64_t n_var, int64_t nlmi, const int64_t* msizes, int64_t nlin,
                         const lrn_options_t* opt, int32_t ngpus, const int32_t* devices);

/* ---- multi-GPU (one process per GPU; NCCL over NVLink) ---- */
/* unique id: 128 bytes generated on rank 0 with lrn_dist_unique_id and broadcast by the host (torch.distributed / MPI) */
int32_t lrn_dist_unique_id(void* out128);
/* Collective.  On a finalized kit = 0 handle every rank also checks that the exchange buffers of the distributed
 * factorisation fit its free device memory; if any rank is short, every rank returns LRN_ERR_ARG (lrn_last_error names
 * the byte counts) and the handle stays single-GPU. */
int32_t lrn_dist_init(lrn_handle_t h, int32_t rank, int32_t world, const void* unique_id128);

#ifdef __cplusplus
}
#endif
#endif
