// Elementwise / reduction / sparse kernels of the IP hot path (HBM- or L2-bound work; no tensor cores).
#pragma once
#include "common.cuh"
#include <algorithm>

namespace lrn {

// ---- dense m x m elementwise (column-major, separate leading dimensions) -----------------------------------------
// out = a*A + b*B + c*C   (B, C optional)
void mat_lincomb(cudaStream_t st, int rows, int cols, double* out, int ldo, double a, const double* A, int lda, double b,
                 const double* B, int ldb, double c, const double* C, int ldc);
// out = sym(a*A + b*B + c*C + d*D)  :  out[i,j] = (t[i,j] + t[j,i]) / 2   (square)
void mat_sym_lincomb(cudaStream_t st, int m, double* out, int ldo, double a, const double* A, int lda, double b,
                     const double* B, int ldb, double c, const double* C, int ldc, double d, const double* D, int ldd);
// A <- (A + A^T)/2 in place
void mat_symmetrize(cudaStream_t st, int m, double* A, int lda);
// out[i,j] = dd[i] * dd[j] * (T[i,j] + T[j,i]) / 2           (src/predictor_corrector.jl:268-269, :281-282)
void mat_scaled_sym(cudaStream_t st, int m, double* out, int ldo, const double* T, int ldt, const double* dd);
// RNT[i,j] = -(T[i,j] + T[j,i]) / (D[i] + D[j])               (src/predictor_corrector.jl:308-309)
void mat_rnt(cudaStream_t st, int m, double* out, int ldo, const double* T, int ldt, const double* D);
// T[i,i] += D[i] - sigmamu / D[i];  T -= RNT                  (src/predictor_corrector.jl:186)
void mat_corr_inner(cudaStream_t st, int m, double* T, int ldt, const double* D, double sigmamu, const double* RNT, int ldr);
// out[:,j] = in[:,j] * s[j]
void mat_scale_cols(cudaStream_t st, int rows, int cols, double* out, int ldo, const double* in, int ldi, const double* s);
// out = in^T
void mat_transpose(cudaStream_t st, int m, double* out, int ldo, const double* in, int ldi);
void mat_add_diag(cudaStream_t st, int m, double* A, int lda, double v);
// A[i,i] += a * D[i] + b / D[i]
void mat_add_diag_vec(cudaStream_t st, int m, double* A, int lda, double a, double b, const double* D);
void mat_set_identity(cudaStream_t st, int m, double* A, int lda, double v);
// d[j] = sum_i A[i,j] * B[i,j]
void mat_coldot(cudaStream_t st, int rows, int cols, const double* A, int lda, const double* B, int ldb, double* d);
// mirror the lower triangle into the upper triangle
void mat_mirror_lower(cudaStream_t st, int n, double* A, int lda);

// ---- vectors -----------------------------------------------------------------------------------------------------
enum VecOp {
    VEC_RECIP = 0,        // out = 1 / a
    VEC_RSQRT = 1,        // out = 1 / sqrt(a)
    VEC_POW_M32 = 2,      // out = a^(-3/2)
    VEC_MUL = 3,          // out = a * b
    VEC_DIV = 4,          // out = a / b
    VEC_COPY = 5,
};
void vec_op(cudaStream_t st, int n, VecOp op, double* out, const double* a, const double* b);
// out = alpha*a + beta*b (b optional)
void vec_axpby(cudaStream_t st, int n, double* out, double alpha, const double* a, double beta, const double* b);

// ---- reductions into a device scalar slot (deterministic two-stage) -------------------------------------------------
struct Reducer {
    DevBuf<double> partial;       // per-CTA partials
    DevBuf<double> slots;         // device result slots
    double* h_slots = nullptr;    // pinned host mirror
    int nslots = 0;
    void init(int nslots_);
    ~Reducer();
    // slot += / = result (accumulate flag)
    void dot_mat(cudaStream_t st, int rows, int cols, const double* A, int lda, const double* B, int ldb, int slot, bool accumulate);
    void dot_vec(cudaStream_t st, int n, const double* a, const double* b, int slot, bool accumulate) {
        dot_mat(st, n, 1, a, n, b, n, slot, accumulate);
    }
    // slot = min_i a[i]/b[i] (b optional -> min a[i]); combined with previous content when `accumulate`
    void min_ratio(cudaStream_t st, int n, const double* a, const double* b, int slot, bool accumulate);
    void zero(cudaStream_t st);
    // copy all slots to the host mirror and synchronise
    const double* fetch(cudaStream_t st);
};

// Row ownership of the Schur matrix in multi-GPU runs: 1-D block-cyclic by ROW blocks of height `pw`
// (row block g -> rank g % world); a rank assembles and factors the part of the lower triangle that lies in its rows
// (entry (r, c), c <= r, belongs to the owner of row r).  world <= 1: everything is owned.
// Storage of H and L: replicated (n_var rows on every rank, rows_local = false) or "own rows" (rows_local = true: only the
// rank's own row blocks, stacked in block order into local_rows(...) rows; local(row) maps a global row to its local one).
struct RowOwner {
    int rank = 0, world = 1, pw = 512;
    bool rows_local = false;
#ifdef __CUDACC__
    __host__ __device__
#endif
    bool owns(int row) const { return world <= 1 || ((row / pw) % world) == rank; }
    // local row of an owned global row: block g = row / pw is the (g / world)-th block of its owner
#ifdef __CUDACC__
    __host__ __device__
#endif
    int local(int row) const { return rows_local && world > 1 ? (row / pw / world) * pw + row % pw : row; }
};
// rows of `rank` in the own-rows layout (its blocks g = rank, rank + world, ...; a ragged last block counts its real rows)
inline int local_rows(int n, int pw, int rank, int world) {
    if (world <= 1) return n;
    const int nblk = (n + pw - 1) / pw;
    if (rank >= nblk) return 0;
    const int cnt = (nblk - 1 - rank) / world + 1, glast = rank + (cnt - 1) * world;
    return (cnt - 1) * pw + (n - glast * pw < pw ? n - glast * pw : pw);
}

// Owner rank of every PSD block when the blocks are distributed over the ranks (lrn_finalize: kit = 0, nlmi >= 2 and a
// communicator with world > 1).  Greedy balance of m_i^3: blocks by decreasing m_i^3 (ties: lower index first), each to the
// least-loaded rank (ties: lowest rank).  Every rank computes the same assignment; a rank may own no block.
inline std::vector<int> block_owner(const std::vector<int>& msizes, int world) {
    const int nb = (int)msizes.size();
    std::vector<int> order(nb), owner(nb, 0);
    for (int i = 0; i < nb; i++) order[i] = i;
    auto cube = [&](int i) { return (long long)msizes[i] * msizes[i] * msizes[i]; };
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return cube(a) > cube(b); });
    std::vector<long long> load(world > 1 ? world : 1, 0);
    for (int i : order) {
        const int r = (int)(std::min_element(load.begin(), load.end()) - load.begin());
        owner[i] = r;
        load[r] += cube(i);
    }
    return owner;
}

// ---- staged sparse-pair Schur assembly (pairs.cu) ------------------------------------------------------------------
// Plan of the shared-memory staged pair kernel: constraints are taken in INDEX order in groups of up to 8 consecutive COLUMNS
// of H whose distinct matrix indices (at most PAIR_MAXC per constraint) fit one CTA's shared memory as rows W[x, I] of the
// symmetric scaling matrix; the row side streams the lower-triangle entry lists of all constraints j >= k, bucketed by
// their entry count so that the lanes of a warp do the same amount of work.
constexpr int PAIR_MAXC = 8;      // distinct indices per constraint matrix handled by the staged kernel
constexpr int PAIR_ROWS = 8;      // columns of H per group (consecutive constraints)
struct PairPlan {
    bool ok = false;
    int ngroups = 0, nbuckets = 0, smax = 0;
    size_t smem = 0;
    // groups (descending row order = descending work): first row, rows, staged doubles per W row, offsets into gidx / rowA
    DevBuf<int> g_r0, g_cnt, g_S, g_idx0;
    DevBuf<int> gidx;              // per group: the S staged column indices of W (padding repeats a valid index)
    DevBuf<int> row_off, row_c;    // per group row (ngroups * PAIR_ROWS): offset of its indices inside the staged row, count
    DevBuf<double> rowA;           // per group row: dense symmetric PAIR_MAXC x PAIR_MAXC coefficient block (local indices)
    // column side, bucket-major: members (constraint ids ascending inside a bucket), entry ranges, entries (p, q, weight)
    DevBuf<int> b_first, b_ids, b_eptr;      // nbuckets + 1 ; members ; members + 1
    std::vector<int> h_b_first;
    DevBuf<int2> e_pq;
    DevBuf<double> e_w;
};

// ---- sparse data of one PSD block --------------------------------------------------------------------------------
struct SparseBlock {
    int m = 0, n_var = 0;
    long long nnz = 0;
    // by-constraint CSR of AA_i (row j = vec(calA_{i,j}), math sign), entries as (p, q, value)
    DevBuf<int> rowptr, ep, eq;
    std::vector<int> h_rowptr, h_part;   // host copies (launch sizing, F1 loop)
    DevBuf<double> ev;
    // by-position CSC: distinct (p,q) positions with the list of (constraint, value) that touch them
    int npos = 0;
    DevBuf<int> pos_p, pos_q, posptr, pos_row;
    DevBuf<double> pos_val;
    // sparse-aware Schur operator (kit = 1): positions grouped by column (pcolptr, m + 1), values of mat(AA' y) per position;
    // usable when every calA_j is stored symmetrically and the union pattern is sparse
    DevBuf<int> pcolptr;
    DevBuf<int> longrows;            // rows of the union pattern with more than 32 entries (handled warp-per-row)
    int nlong = 0;
    DevBuf<double> mval;
    DevBuf<double> eval;             // one partial result per stored entry (entry-parallel kernels + deterministic row sums)
    bool sparse_ok = false;          // structurally possible (symmetric storage, bounded rows)
    bool sparse_op = false;          // in use (sparse_ok and union pattern density <= 5 %, or forced through lrn_set_option)
    // participating constraints (nnz > 0) in nnz-descending (sigmaA) order
    int npart = 0, nF1 = 0;
    DevBuf<int> part;
    int max_row_nnz = 0;
    bool all_single_diag = false;    // every participating matrix is v * e_a e_a^T
    PairPlan pairs;                  // staged pair kernel (used when every matrix of the block goes through the F3 formula)
    // rank-one factors (datarank == -1): CSR n_var x m
    bool has_B = false;
    long long nnzB = 0;
    DevBuf<int> b_rowptr, b_col;
    DevBuf<double> b_val;
};

// out[p + q*ld] += scale * sum_{(j,v) at (p,q)} v * y[j]        (mat(AA' y), src/predictor_corrector.jl:13,252; src/Solvers.jl:595)
void sp_scatter_ATy(cudaStream_t st, const SparseBlock& sb, const double* y, double scale, double* out, int ld);
// out[j] += scale * sum_e ev * M[ep + eq*ld]                    (AA * vec(M), src/makeBBBB.jl:225 etc.)
void sp_A_vec(cudaStream_t st, const SparseBlock& sb, const double* M, int ld, double scale, double* out);
// Sparse-aware Schur operator pieces (MyA functor, src/Solvers.jl:572-614, without the two dense m^3 products):
//   sp_pos_values : mval[t] = sum_{(j,v) at position t} v * y[j]                      (the nonzeros of M = mat(AA' y))
//   sp_M_times_W  : Z = M W  (column q: gather from W(:,q) staged in shared memory, M row r = M column r by symmetry)
//   sp_A_sampled  : out[j] += scale * sum_{(p,q,v) in calA_j} v * <W(:,p), Z(:,q)>     (= <calA_j, W M W>, W symmetric)
void sp_pos_values(cudaStream_t st, SparseBlock& sb, const double* y);
void sp_M_times_W(cudaStream_t st, const SparseBlock& sb, const double* W, int ldw, double* Z, int ldz);
void sp_A_sampled(cudaStream_t st, SparseBlock& sb, const double* W, int ldw, const double* Z, int ldz, double scale,
                  double* out);
//   sp_M_times_cols : Y(:, c) = M X(:, c) for a thin X (m x k)                          (mat(AA' y) * U in the H_alpha apply)
//   sp_A_rank       : out[j] += sum_{(p,q,v) in calA_j} v * sum_r ZY[p,r] U[q,r]        (AA * kron(U, Z y), src/Solvers.jl:891-896)
//   sp_row_sums     : out[j] += scale * sum of sb.eval over the entries of row j        (second half of the entry-parallel kernels)
void sp_M_times_cols(cudaStream_t st, const SparseBlock& sb, const double* X, int ldx, int k, double* Y, int ldy);
void sp_A_rank(cudaStream_t st, SparseBlock& sb, const double* ZY, int ldz, const double* U, int ldu, int k, double* out);
void sp_row_sums(cudaStream_t st, const SparseBlock& sb, double scale, double* out);
// BG[j + c*ldo] = sum_t B[j,t] G[t,c]                           (B_i * G_i, src/makeBBBB.jl:7)
void sp_B_times_G(cudaStream_t st, const SparseBlock& sb, const double* G, int ldg, double* BG, int ldo);
// Sparse-pair Schur term (F3 formula, src/makeBBBB.jl:139-213 / _dot :39-64): for participating positions jj <= kk, both >= first,
//   H[max(j,k), min(j,k)] += tr(calA_j W calA_k W)
void sp_schur_pairs(cudaStream_t st, const SparseBlock& sb, int first, const double* W, int ldw, double* H, int ldh,
                    RowOwner own = RowOwner());
// The same Schur term through the shared-memory staged kernel (pairs.cu); requires sb.pairs.ok.  All pairs of the block.
// accumulate = false: H holds zeros where this block writes (first block of an assembly): plain stores instead of read-modify-write
void sp_schur_pairs_staged(cudaStream_t st, const SparseBlock& sb, const double* W, int ldw, double* H, int ldh,
                           RowOwner own = RowOwner(), bool accumulate = true);
// host: build sb.pairs from the by-constraint entry lists (0-based rowptr / p / q / value, symmetric storage required)
void sp_build_pair_plan(SparseBlock& sb, const std::vector<int>& rowptr, const std::vector<int>& ep, const std::vector<int>& eq,
                        const std::vector<double>& ev, cudaStream_t st);
// F1 column (src/makeBBBB.jl:81-104): given U = W calA_j W dense, H[max(j,k),min(j,k)] += <calA_k, U> for positions kk >= jj
void sp_schur_f1_column(cudaStream_t st, const SparseBlock& sb, int jj, const double* U, int ldu, double* H, int ldh,
                        RowOwner own = RowOwner());
// densify calA_j into a zeroed m x m buffer
void sp_densify(cudaStream_t st, const SparseBlock& sb, int j, double* out, int ld);

// ---- LP block (C_lin is n_var x nlin) ----------------------------------------------------------------------------
struct SparseLin {
    int n_var = 0, nlin = 0;
    long long nnz = 0;
    DevBuf<int> r_ptr, r_col;     // CSR by variable j
    DevBuf<double> r_val;
    DevBuf<int> c_ptr, c_row;     // CSC by LP row r
    DevBuf<double> c_val;
};
// out[r] = a*base[r] (base optional) + scale * sum_j C[j,r] y[j]
void lin_CT_y(cudaStream_t st, const SparseLin& L, const double* y, double scale, double a, const double* base, double* out);
// out[j] += scale * sum_r C[j,r] x[r]
void lin_C_x(cudaStream_t st, const SparseLin& L, const double* x, double scale, double* out);
// H[j,k] += sum_r C[j,r] d[r] C[k,r]   for k <= j              (src/predictor_corrector.jl:36-38)
void lin_schur(cudaStream_t st, const SparseLin& L, const double* d, double* H, int ldh, RowOwner own = RowOwner());
// diag[j] += sum_r C[j,r]^2 d[r]
void lin_schur_diag(cudaStream_t st, const SparseLin& L, const double* d, double* diag);

}  // namespace lrn
