// Dense blocked FP64 Cholesky (lower) + blocked triangular solves.
// Replaces LAPACK dpotrf/dtrsv behind `cholesky(Hermitian(BBBB,:L))` and `L' \ (L \ h)` (src/predictor_corrector.jl:57,89-90,199)
// and behind `cholesky(X[i])` / `cholesky(S[i])` (src/prepare_W.jl:7,24), `cholesky(S)` (src/Solvers.jl:805).
#pragma once
#include "common.cuh"

namespace lrn {

constexpr int CHOL_DB = 64;   // diagonal block size (one CTA, shared memory)

// Workspace: inverses of the 64x64 diagonal blocks of L (used by the panel TRSM and by the triangular solves).
struct CholWork {
    DevBuf<double> dinv;      // cdiv(n,64) blocks of 64x64 (ld 64), zero above the diagonal
    DevBuf<int> info;         // [0] = 0 ok, >0 = 1-based index of the first non-positive pivot (LAPACK convention)
    int* info_ext = nullptr;  // optional external flag location (lets the caller gather many flags with one copy)
    DevBuf<double> tinv, tscr; // inverses of the 256 x 256 diagonal blocks of L (triangular solves) + 64 x 64 scratch per block
    const double* tinv_for = nullptr;   // factor the inverses belong to (reset by every factorisation)
    // the launch sequence of a triangular solve (2 launches per 256 unknowns) only depends on (L, n, lda, x, tmp, which): it is
    // captured once as a CUDA graph and replayed (the solves are bound by launch latency, not by HBM)
    struct SolveGraph {
        cudaGraphExec_t exec = nullptr;
        const double* L = nullptr; const double* tinv = nullptr; double* x = nullptr; double* tmp = nullptr;
        int n = 0, lda = 0;
        long long nodes = 0;
        bool warm = false, broken = false;
    } sgraph[4];                  // indexed by `which` (1 forward, 2 backward, 3 both)
    cudaStream_t aux = nullptr;   // high-priority side stream (panel factorisation + broadcast look-ahead in multi-GPU runs)
    cudaStream_t aux2 = nullptr;  // second high-priority stream (distributed path: early factorisation of the next diagonal block)
    cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    // trailing updates as Ozaki INT8 products (chol_i8.cu): 0 never (DMMA), 1 when the panels are 1024 wide (n >= 16384) unless the
    // environment sets LRN_CHOL_INT8=0, 2 at every panel width (tests).  Only the Schur factor opts in.
    int int8 = 0;
    // digit planes + row scales of the solved panel, two sets: panel p + 1 is sliced while the rest update of panel p still
    // reads panel p's set
    DevBuf<int8_t> i8_slices[2];
    DevBuf<double> i8_sigma[2];
    int n = 0;
    void ensure(int n_) {
        if (n_ > n || !dinv.p) { dinv.alloc((size_t)cdiv(n_, CHOL_DB) * CHOL_DB * CHOL_DB); n = n_; }
        if (!info.p) info.alloc(1);
    }
    int* info_ptr() const { return info_ext ? info_ext : info.p; }
};

// Factor the lower triangle of A (n x n, column-major, lda) in place: A = L L^T. The strict upper triangle is ignored
// (inside diagonal 128-tiles it may be overwritten with don't-care values). Enqueues only; read `work.info` after a sync.
void cholesky_lower(double* A, int n, int lda, CholWork& work, cudaStream_t st);

// Factor ONE diagonal block (w <= 512) in place with a single launch; `dinv` receives its inverted 64 x 64 diagonal blocks and
// X (w x w, leading dimension ldx, optional) the full inverse of the factor (lower triangular, zero above the diagonal);
// T: w x ldx scratch for the recursive-doubling inversion (null: the older block forward substitution is used).
void chol_diag_block(double* Akk, int lda, int w, double* dinv, double* X, int ldx, double* T, int* info, int base, cudaStream_t st);

// creates the high-priority side stream and the events of `work` on first use
void ensure_aux(CholWork& work);

// x <- L^{-1} x (which=1), x <- L^{-T} x (which=2), both (which=3). `tmp` has n doubles. Uses work.dinv of the same factor;
// the first solve after a factorisation builds the inverses of the 256 x 256 diagonal blocks (work.tinv).
void chol_solve(const double* L, int n, int lda, CholWork& work, double* x, double* tmp, int which, cudaStream_t st);

// Y <- L^{-T} Y for an n x ncols right-hand-side block (in place), blocked with the inverted diagonal blocks of `work`:
// used for G = L_S^{-T} (U D^{1/2}) in the NT scaling (no accumulated right singular vectors needed).
void trsm_left_lower_trans(const double* L, int n, int lda, const CholWork& work, double* Y, int ldy, int ncols, cudaStream_t st);

// Zero the strict upper triangle (so the factor can be used as a dense GEMM operand).
void zero_strict_upper(double* A, int n, int lda, cudaStream_t st);

// ---- Ozaki INT8 products (chol_i8.cu) ----
// bytes of the digit planes of rows_pad rows x K columns
size_t i8_slice_bytes(int rows_pad, int K);
// slice P (rows x K, leading dimension ldp, 1 <= K <= 1024) into 8 int8 digit planes and per-row power-of-two scales sigma;
// rows [rows, rows_pad) get zero digits and sigma 0 (rows_pad % 8 == 0)
void i8_slice(const double* P, int ldp, int rows, int K, int rows_pad, int8_t* slices, double* sigma, cudaStream_t st);
// C (M x N, ldc) -= P[a_row0 + i, :] P[b_row0 + j, :]^T from the slices (a_row0, b_row0 multiples of 8).  lower: only tiles
// (128 x 64) that meet the lower triangle, with (row0, col0) the position of C(0, 0) in the symmetric matrix; entries above the
// diagonal inside such tiles are updated too (don't-care for the factorisation)
void syrk_update_i8(const int8_t* slices, const double* sigma, int rows_pad, int K, int a_row0, int b_row0, int M, int N, double* C,
                    int ldc, long long row0, long long col0, bool lower, cudaStream_t st);

}  // namespace lrn
