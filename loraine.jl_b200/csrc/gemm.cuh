// FP64 tensor-core (DMMA) GEMM family -- the dense workhorse of the library.
//   C = alpha * op(A) op(B) [.* colscale] + beta * C      (mode 0)
//   C = beta * C + alpha * (op(A) op(B)).^2               (mode 1, rank-one Schur epilogue, src/makeBBBB.jl:10-14)
// Column-major, arbitrary sizes, optional batching over blockIdx.z with element strides.
#pragma once
#include "common.cuh"

namespace lrn {

struct GemmParams {
    const double* A = nullptr;
    const double* B = nullptr;
    double* C = nullptr;
    int M = 0, N = 0, K = 0;
    int lda = 0, ldb = 0, ldc = 0;
    long long sA = 0, sB = 0, sC = 0;   // batch strides (elements)
    int batch = 1;
    bool transA = false, transB = false;
    double alpha = 1.0, beta = 0.0;
    int mode = 0;                       // 0 plain, 1 squared-accumulate
    int lower = 0;                      // 1: skip tiles strictly above the diagonal (symmetric outputs)
    const double* colscale = nullptr;   // optional length-N scale applied to product columns
    long long sScale = 0;               // batch stride of colscale
    // second (inner) batch level: z = z1*batch2 + z2, offsets z1*s? + z2*s?2 (split-K partial products, etc.)
    int batch2 = 1;
    long long sA2 = 0, sB2 = 0, sC2 = 0;
    int K_last = 0;                     // if >0: K used by the last inner index (z2 == batch2-1)
    // optional scatter of output columns in blocks of 32 (block-Jacobi round-robin re-arrangement):
    // dest column = cblkmap[z1*(N/32) + col/32]*32 + col%32, C batch strides ignored. N must be a multiple of 32.
    const int* cblkmap = nullptr;
    // global offsets of the sub-problem (only used by the lower-triangle tile test when a product is split into regions)
    int row0 = 0, col0 = 0;
    long long row0z = 0;      // the outer batch index z1 adds z1 * row0z to row0 (row blocks of a block-cyclic distribution are a
                              // strided batch: sA = sC = row0z rows further down the same matrix)
    bool no_bulk = false;     // keep this product off the TMA-fed kernel (edge strips / remainders issued by gemm() itself)
    int ktri = 0;             // 1: op(A) (M x K) and op(B) (K x N) vanish for k < row resp. k < column (product of a transposed
                              // lower-triangular factor with a lower-triangular factor): tiles start their K loop at max(m0, n0)
};

// Enqueue on `stream`. Never synchronises.
void gemm(const GemmParams& p, cudaStream_t stream);

// Convenience wrappers (single problem).
inline void gemm_nn(cudaStream_t s, int M, int N, int K, double alpha, const double* A, int lda, const double* B, int ldb,
                    double beta, double* C, int ldc) {
    GemmParams p; p.A = A; p.B = B; p.C = C; p.M = M; p.N = N; p.K = K; p.lda = lda; p.ldb = ldb; p.ldc = ldc;
    p.alpha = alpha; p.beta = beta; gemm(p, s);
}
inline void gemm_nt(cudaStream_t s, int M, int N, int K, double alpha, const double* A, int lda, const double* B, int ldb,
                    double beta, double* C, int ldc) {
    GemmParams p; p.A = A; p.B = B; p.C = C; p.M = M; p.N = N; p.K = K; p.lda = lda; p.ldb = ldb; p.ldc = ldc;
    p.alpha = alpha; p.beta = beta; p.transB = true; gemm(p, s);
}
inline void gemm_tn(cudaStream_t s, int M, int N, int K, double alpha, const double* A, int lda, const double* B, int ldb,
                    double beta, double* C, int ldc) {
    GemmParams p; p.A = A; p.B = B; p.C = C; p.M = M; p.N = N; p.K = K; p.lda = lda; p.ldb = ldb; p.ldc = ldc;
    p.alpha = alpha; p.beta = beta; p.transA = true; gemm(p, s);
}

// Number of DMMA GEMM kernel launches issued so far by this process (bench `gpu_launches` bookkeeping).
long long gemm_launch_count();
// enable / disable the TMA (cp.async.bulk) fed kernel for large A*B^T products (default on; tests compare both paths)
void gemm_set_bulk(bool on);
// number of SMs of the current device (cached per device)
int device_sm_count();

// Block-Jacobi panel rotation (see panel_rotate_kernel): cur / nxt are column-major work buffers with leading dimension
// ldw >= 128 * tiles whose padding rows are zero; pair z owns columns [64 z, 64 z + 64) of cur and its rotated halves go
// to the 32-column slots slotmap[2z], slotmap[2z+1] of nxt.  rot holds the 64 x 64 rotations (ld 64) one after the other.
struct PanelRotateParams {
    const double* cur = nullptr;
    double* nxt = nullptr;
    const double* rot = nullptr;
    const int* slotmap = nullptr;
    int ldw = 0;
    int tiles = 0;            // 128-row tiles per panel
    long long total = 0;      // pairs * tiles
};
void panel_rotate(const PanelRotateParams& p, cudaStream_t stream);
// mode 1: start recording one CUDA-event pair per GEMM launch; mode 0: stop, synchronise and report the totals
// modes 10 / 11 / 12 / 13 return the totals of one kernel family of the last stopped profile; family 3 (the INT8 Ozaki update of
// chol_i8.cu) is kept out of the mode 0 totals, which describe the DMMA kernels only
void gemm_profile(int mode, double* ms, double* flops, long long* launches);
bool gemm_profile_active();   // per-launch event timing is on (stream capture must not be used meanwhile)
// per-launch records of kernels outside gemm.cu: begin records a start event on `st` when the profile is on (returns false
// otherwise); end records the stop event and files the launch under family `fam` with its algorithmic flops
bool gemm_prof_begin(cudaStream_t st, cudaEvent_t& start);
void gemm_prof_end(cudaEvent_t start, cudaStream_t st, double flops, int fam);

}  // namespace lrn
