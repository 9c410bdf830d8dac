#include "ops.cuh"
#include <algorithm>

namespace lrn {
namespace {

constexpr int TB = 256;
inline dim3 grid2(int rows, int cols) {
    LRN_REQUIRE(cols <= 65535, "matrix dimension above 65535 is not supported by the elementwise kernels");
    return dim3((unsigned)cdiv(rows, TB), (unsigned)cols);
}

__global__ void k_lincomb(int rows, double* out, int ldo, double a, const double* A, int lda, double b, const double* B,
                          int ldb, double c, const double* C, int ldc) {
    int i = blockIdx.x * TB + threadIdx.x, j = blockIdx.y;
    if (i >= rows) return;
    double v = a * A[(size_t)j * lda + i];
    if (B) v += b * B[(size_t)j * ldb + i];
    if (C) v += c * C[(size_t)j * ldc + i];
    out[(size_t)j * ldo + i] = v;
}
__device__ __forceinline__ double lc4(int i, int j, double a, const double* A, int lda, double b, const double* B, int ldb,
                                      double c, const double* C, int ldc, double d, const double* D, int ldd) {
    double v = a * A[(size_t)j * lda + i];
    if (B) v += b * B[(size_t)j * ldb + i];
    if (C) v += c * C[(size_t)j * ldc + i];
    if (D) v += d * D[(size_t)j * ldd + i];
    return v;
}
__global__ void k_sym_lincomb(int m, double* out, int ldo, double a, const double* A, int lda, double b, const double* B,
                              int ldb, double c, const double* C, int ldc, double d, const double* D, int ldd) {
    int i = blockIdx.x * TB + threadIdx.x, j = blockIdx.y;
    if (i >= m) return;
    double v = lc4(i, j, a, A, lda, b, B, ldb, c, C, ldc, d, D, ldd);
    double w = lc4(j, i, a, A, lda, b, B, ldb, c, C, ldc, d, D, ldd);
    out[(size_t)j * ldo + i] = 0.5 * (v + w);
}
__global__ void k_symmetrize(int m, double* A, int lda) {
    int i = blockIdx.x * TB + threadIdx.x, j = blockIdx.y;
    if (i >= m || i <= j) return;
    double v = 0.5 * (A[(size_t)j * lda + i] + A[(size_t)i * lda + j]);
    A[(size_t)j * lda + i] = v;
    A[(size_t)i * lda + j] = v;
}
__global__ void k_scaled_sym(int m, double* out, int ldo, const double* T, int ldt, const double* dd) {
    int i = blockIdx.x * TB + threadIdx.x, j = blockIdx.y;
    if (i >= m) return;
    double a = dd[i] * dd[j];
    // reference: XXX = DDsi' .* T .* DDsi ; XXX = (XXX + XXX')/2
    out[(size_t)j * ldo + i] = 0.5 * (a * T[(size_t)j * ldt + i] + a * T[(size_t)i * ldt + j]);
}
__global__ void k_rnt(int m, double* out, int ldo, const double* T, int ldt, const double* D) {
    int i = blockIdx.x * TB + threadIdx.x, j = blockIdx.y;
    if (i >= m) return;
    out[(size_t)j * ldo + i] = -(T[(size_t)j * ldt + i] + T[(size_t)i * ldt + j]) / (D[i] + D[j]);
}
__global__ void k_corr_inner(int m, double* T, int ldt, const double* D, double sigmamu, const double* R, int ldr) {
    int i = blockIdx.x * TB + threadIdx.x, j = blockIdx.y;
    if (i >= m) return;
    double v = T[(size_t)j * ldt + i];
    if (i == j) v += D[i] - sigmamu / D[i];
    v -= R[(size_t)j * ldr + i];
    T[(size_t)j * ldt + i] = v;
}
__global__ void k_scale_cols(int rows, double* out, int ldo, const double* in, int ldi, const double* s) {
    int i = blockIdx.x * TB + threadIdx.x, j = blockIdx.y;
    if (i >= rows) return;
    out[(size_t)j * ldo + i] = in[(size_t)j * ldi + i] * s[j];
}
__global__ void k_transpose(int m, double* out, int ldo, const double* in, int ldi) {
    __shared__ double tile[32][33];
    int bx = blockIdx.x * 32, by = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += 8) {
        int i = bx + threadIdx.x, j = by + r;
        if (i < m && j < m) tile[r][threadIdx.x] = in[(size_t)j * ldi + i];
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += 8) {
        int i = by + threadIdx.x, j = bx + r;        // out[i,j] = in[j,i]
        if (i < m && j < m) out[(size_t)j * ldo + i] = tile[threadIdx.x][r];
    }
}
__global__ void k_add_diag(int m, double* A, int lda, double v) {
    int i = blockIdx.x * TB + threadIdx.x;
    if (i < m) A[(size_t)i * lda + i] += v;
}
__global__ void k_add_diag_vec(int m, double* A, int lda, double a, double b, const double* D) {
    int i = blockIdx.x * TB + threadIdx.x;
    if (i < m) A[(size_t)i * lda + i] += a * D[i] + b / D[i];
}
__global__ void k_set_identity(int m, double* A, int lda, double v) {
    int i = blockIdx.x * TB + threadIdx.x, j = blockIdx.y;
    if (i < m) A[(size_t)j * lda + i] = (i == j) ? v : 0.0;
}
__global__ void k_coldot(int rows, int cols, const double* A, int lda, const double* B, int ldb, double* d) {
    int warp = (blockIdx.x * TB + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= cols) return;
    double s = 0.0;
    for (int i = lane; i < rows; i += 32) s += A[(size_t)warp * lda + i] * B[(size_t)warp * ldb + i];
    s = warp_sum(s);
    if (lane == 0) d[warp] = s;
}
// columns are spread over blockIdx.y and blockIdx.z so that n_var may exceed the 65535 limit of grid.y
__global__ void k_mirror_lower(int n, double* A, int lda) {
    int i = blockIdx.x * TB + threadIdx.x, j = blockIdx.y + gridDim.y * blockIdx.z;
    if (j < n && i < n && i > j) A[(size_t)i * lda + j] = A[(size_t)j * lda + i];
}
__global__ void k_vec_op(int n, int op, double* out, const double* a, const double* b) {
    int i = blockIdx.x * TB + threadIdx.x;
    if (i >= n) return;
    double x = a[i], r;
    switch (op) {
        case VEC_RECIP: r = 1.0 / x; break;
        case VEC_RSQRT: r = 1.0 / sqrt(x); break;
        case VEC_POW_M32: r = 1.0 / (x * sqrt(x)); break;
        case VEC_MUL: r = x * b[i]; break;
        case VEC_DIV: r = x / b[i]; break;
        default: r = x;
    }
    out[i] = r;
}
__global__ void k_vec_axpby(int n, double* out, double alpha, const double* a, double beta, const double* b) {
    int i = blockIdx.x * TB + threadIdx.x;
    if (i >= n) return;
    double v = alpha * a[i];
    if (b) v += beta * b[i];
    out[i] = v;
}

// ---- reductions ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(TB) k_dot_partial(int rows, long long total, const double* A, int lda, const double* B,
                                                    int ldb, double* partial) {
    __shared__ double red[32];
    double s = 0.0;
    for (long long idx = (long long)blockIdx.x * TB + threadIdx.x; idx < total; idx += (long long)gridDim.x * TB) {
        long long j = idx / rows;
        int i = (int)(idx - j * rows);
        s += A[(size_t)j * lda + i] * B[(size_t)j * ldb + i];
    }
    s = block_sum(s, red);
    if (threadIdx.x == 0) partial[blockIdx.x] = s;
}
__global__ void __launch_bounds__(TB) k_sum_finish(const double* partial, int n, double* slot, int accumulate) {
    __shared__ double red[32];
    double s = 0.0;
    for (int i = threadIdx.x; i < n; i += TB) s += partial[i];
    s = block_sum(s, red);
    if (threadIdx.x == 0) *slot = (accumulate ? *slot : 0.0) + s;
}
__global__ void __launch_bounds__(TB) k_minratio_partial(int n, const double* a, const double* b, double* partial) {
    __shared__ double red[32];
    double m = 1.0e300;
    for (int i = blockIdx.x * TB + threadIdx.x; i < n; i += gridDim.x * TB) {
        double v = b ? a[i] / b[i] : a[i];
        m = fmin(m, v);
    }
    m = warp_min(m);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < TB / 32; w++) m = fmin(m, red[w]);
        partial[blockIdx.x] = m;
    }
}
__global__ void k_min_finish(const double* partial, int n, double* slot, int accumulate) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        double m = accumulate ? *slot : 1.0e300;
        for (int i = 0; i < n; i++) m = fmin(m, partial[i]);
        *slot = m;
    }
}

// ---- sparse ----------------------------------------------------------------------------------------------------
__global__ void k_scatter_ATy(int npos, const int* __restrict__ pos_p, const int* __restrict__ pos_q,
                              const int* __restrict__ posptr, const int* __restrict__ pos_row,
                              const double* __restrict__ pos_val, const double* __restrict__ y, double scale,
                              double* __restrict__ out, int ld) {
    int t = blockIdx.x * TB + threadIdx.x;
    if (t >= npos) return;
    double s = 0.0;
    for (int e = posptr[t]; e < posptr[t + 1]; e++) s += pos_val[e] * y[pos_row[e]];
    out[(size_t)pos_q[t] * ld + pos_p[t]] += scale * s;
}
// The three gather kernels below give one WARP to a position / row and let the lanes stride its list: lists are short on
// average but skewed (a theta problem has one row with m entries), and a thread-per-row loop would serialise on it.
__global__ void __launch_bounds__(256) k_pos_values(int npos, const int* __restrict__ posptr, const int* __restrict__ pos_row,
                                                    const double* __restrict__ pos_val, const double* __restrict__ y,
                                                    double* __restrict__ mval) {
    const int t = (blockIdx.x * 256 + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (t >= npos) return;
    double s = 0.0;
    for (int e = posptr[t] + lane; e < posptr[t + 1]; e += 32) s += pos_val[e] * y[pos_row[e]];
    s = warp_sum(s);
    if (lane == 0) mval[t] = s;
}
// Z = M W (row r of the symmetric M is read as its column r).  Short rows: one thread per (r, q), gathering down column q
// of W (L1/L2-resident).  The few long rows (a theta problem has one with m entries) get one warp per (r, q) in a second
// launch, so no thread ever walks a long list alone.
constexpr int MW_LONG = 32;
__global__ void __launch_bounds__(256) k_M_times_W_short(int m, const int* __restrict__ pcolptr, const int* __restrict__ pos_p,
                                                         const double* __restrict__ mval, const double* __restrict__ W, int ldw,
                                                         double* __restrict__ Z, int ldz) {
    const int r = blockIdx.x * 256 + threadIdx.x, q = blockIdx.y;
    if (r >= m) return;
    const int t0 = pcolptr[r], t1 = pcolptr[r + 1];
    if (t1 - t0 > MW_LONG) return;
    const double* Wq = W + (size_t)q * ldw;
    double s = 0.0;
    for (int t = t0; t < t1; t++) s += mval[t] * Wq[pos_p[t]];
    Z[(size_t)q * ldz + r] = s;
}
__global__ void __launch_bounds__(256) k_M_times_W_long(int m, int nlong, const int* __restrict__ longrows,
                                                        const int* __restrict__ pcolptr, const int* __restrict__ pos_p,
                                                        const double* __restrict__ mval, const double* __restrict__ W, int ldw,
                                                        double* __restrict__ Z, int ldz) {
    const int q = (blockIdx.x * 256 + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (q >= m) return;
    const int r = longrows[blockIdx.y];
    const double* Wq = W + (size_t)q * ldw;
    double s = 0.0;
    for (int t = pcolptr[r] + lane; t < pcolptr[r + 1]; t += 32) s += mval[t] * Wq[pos_p[t]];
    s = warp_sum(s);
    if (lane == 0) Z[(size_t)q * ldz + r] = s;
}
// one warp per stored entry: eval[e] = v_e <W(:, p_e), Z(:, q_e)>.  Entry-parallel, so one dense constraint (e.g. the trace
// constraint of a theta problem, m entries) does not serialise on a single warp; the per-constraint sums follow in k_row_sums
__global__ void __launch_bounds__(256) k_A_sampled(long long nnz, int m, const int* __restrict__ ep, const int* __restrict__ eq,
                                                   const double* __restrict__ ev, const double* __restrict__ W, int ldw,
                                                   const double* __restrict__ Z, int ldz, double* __restrict__ eval) {
    const long long e = ((long long)blockIdx.x * 256 + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (e >= nnz) return;
    const double* wp = W + (size_t)ep[e] * ldw;
    const double* zq = Z + (size_t)eq[e] * ldz;
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    int i = lane;
    for (; i + 96 < m; i += 128) {
        a0 += wp[i] * zq[i];
        a1 += wp[i + 32] * zq[i + 32];
        a2 += wp[i + 64] * zq[i + 64];
        a3 += wp[i + 96] * zq[i + 96];
    }
    for (; i < m; i += 32) a0 += wp[i] * zq[i];
    const double s = warp_sum((a0 + a1) + (a2 + a3));
    if (lane == 0) eval[e] = ev[e] * s;
}
// one thread per stored entry: eval[e] = v_e sum_r ZY[p_e, r] U[q_e, r]
__global__ void k_A_rank_entries(long long nnz, const int* __restrict__ ep, const int* __restrict__ eq,
                                 const double* __restrict__ ev, const double* __restrict__ ZY, int ldz,
                                 const double* __restrict__ U, int ldu, int k, double* __restrict__ eval) {
    const long long e = (long long)blockIdx.x * TB + threadIdx.x;
    if (e >= nnz) return;
    double t = 0.0;
    for (int r = 0; r < k; r++) t += ZY[(size_t)r * ldz + ep[e]] * U[(size_t)r * ldu + eq[e]];
    eval[e] = ev[e] * t;
}
// one warp per constraint, fixed summation order: out[j] += scale * sum_{e in row j} eval[e]
__global__ void __launch_bounds__(256) k_row_sums(int n_var, const int* __restrict__ rowptr, const double* __restrict__ eval,
                                                  double scale, double* __restrict__ out) {
    const int j = (blockIdx.x * 256 + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (j >= n_var) return;
    const int e0 = rowptr[j], e1 = rowptr[j + 1];
    if (e0 == e1) return;
    double s = 0.0;
    for (int e = e0 + lane; e < e1; e += 32) s += eval[e];
    s = warp_sum(s);
    if (lane == 0) out[j] += scale * s;
}
// Y(r, c) = sum_{t in column r of M} mval[t] X(pos_p[t], c)   (M symmetric: row r read as column r); one warp per (r, c)
__global__ void __launch_bounds__(256) k_M_times_cols(int m, int k, const int* __restrict__ pcolptr, const int* __restrict__ pos_p,
                                                      const double* __restrict__ mval, const double* __restrict__ X, int ldx,
                                                      double* __restrict__ Y, int ldy) {
    const int r = (blockIdx.x * 256 + threadIdx.x) >> 5, lane = threadIdx.x & 31, c = blockIdx.y;
    if (r >= m || c >= k) return;
    const double* Xc = X + (size_t)c * ldx;
    double s = 0.0;
    for (int t = pcolptr[r] + lane; t < pcolptr[r + 1]; t += 32) s += mval[t] * Xc[pos_p[t]];
    s = warp_sum(s);
    if (lane == 0) Y[(size_t)c * ldy + r] = s;
}
__global__ void k_A_vec_thread(int n_var, const int* __restrict__ rowptr, const int* __restrict__ ep,
                               const int* __restrict__ eq, const double* __restrict__ ev, const double* __restrict__ M,
                               int ld, double scale, double* __restrict__ out) {
    int j = blockIdx.x * TB + threadIdx.x;
    if (j >= n_var) return;
    int e0 = rowptr[j], e1 = rowptr[j + 1];
    if (e0 == e1) return;
    double s = 0.0;
    for (int e = e0; e < e1; e++) s += ev[e] * M[(size_t)eq[e] * ld + ep[e]];
    out[j] += scale * s;
}
__global__ void k_A_vec_warp(int n_var, const int* __restrict__ rowptr, const int* __restrict__ ep,
                             const int* __restrict__ eq, const double* __restrict__ ev, const double* __restrict__ M, int ld,
                             double scale, double* __restrict__ out) {
    int j = (blockIdx.x * TB + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (j >= n_var) return;
    int e0 = rowptr[j], e1 = rowptr[j + 1];
    double s = 0.0;
    for (int e = e0 + lane; e < e1; e += 32) s += ev[e] * M[(size_t)eq[e] * ld + ep[e]];
    s = warp_sum(s);
    if (lane == 0 && e1 > e0) out[j] += scale * s;
}
__global__ void k_B_times_G(int n_var, int m, const int* __restrict__ b_rowptr, const int* __restrict__ b_col,
                            const double* __restrict__ b_val, const double* __restrict__ G, int ldg, double* __restrict__ BG,
                            int ldo) {
    int j = blockIdx.x * TB + threadIdx.x, c = blockIdx.y;
    if (j >= n_var) return;
    double s = 0.0;
    for (int t = b_rowptr[j]; t < b_rowptr[j + 1]; t++) s += b_val[t] * G[(size_t)c * ldg + b_col[t]];
    BG[(size_t)c * ldo + j] = s;
}
// one thread per ordered pair of participating positions (jj <= kk); W symmetric so both gathers walk down columns a and b
__global__ void __launch_bounds__(256) k_schur_pairs(int npart, int first, const int* __restrict__ part,
                                                     const int* __restrict__ rowptr, const int* __restrict__ ep,
                                                     const int* __restrict__ eq, const double* __restrict__ ev,
                                                     const double* __restrict__ W, int ldw, double* __restrict__ H, int ldh,
                                                     RowOwner own) {
    const int kk = first + blockIdx.x * 16 + threadIdx.x;
    const int jj = first + blockIdx.y * 16 + threadIdx.y;
    if (blockIdx.x < blockIdx.y) return;
    if (kk >= npart || jj >= npart || kk < jj) return;
    const int j = part[jj], k = part[kk];
    if (!own.owns(j > k ? j : k)) return;
    const int e0 = rowptr[j], e1 = rowptr[j + 1], f0 = rowptr[k], f1 = rowptr[k + 1];
    double acc = 0.0;
    for (int e = e0; e < e1; e++) {
        const double va = ev[e];
        const double* Wa = W + (size_t)ep[e] * ldw;     // column a
        const double* Wb = W + (size_t)eq[e] * ldw;     // column b
        double s = 0.0;
        for (int f = f0; f < f1; f++) s += ev[f] * __ldg(Wb + ep[f]) * __ldg(Wa + eq[f]);   // W[p,b] * W[q,a]
        acc += va * s;
    }
    const int r = j > k ? j : k, c = j > k ? k : j;
    H[(size_t)c * ldh + own.local(r)] += acc;
}
__global__ void k_schur_f1_column(int npart, int jj, const int* __restrict__ part, const int* __restrict__ rowptr,
                                  const int* __restrict__ ep, const int* __restrict__ eq, const double* __restrict__ ev,
                                  const double* __restrict__ U, int ldu, double* __restrict__ H, int ldh, RowOwner own) {
    int kk = jj + ((blockIdx.x * TB + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (kk >= npart) return;
    const int j = part[jj], k = part[kk];
    if (!own.owns(j > k ? j : k)) return;
    double s = 0.0;
    for (int f = rowptr[k] + lane; f < rowptr[k + 1]; f += 32) s += ev[f] * U[(size_t)eq[f] * ldu + ep[f]];
    s = warp_sum(s);
    if (lane == 0) {
        const int r = j > k ? j : k, c = j > k ? k : j;
        H[(size_t)c * ldh + own.local(r)] += s;
    }
}
__global__ void k_densify(int e0, int e1, const int* __restrict__ ep, const int* __restrict__ eq, const double* __restrict__ ev,
                          double* __restrict__ out, int ld) {
    int e = e0 + blockIdx.x * TB + threadIdx.x;
    if (e < e1) out[(size_t)eq[e] * ld + ep[e]] = ev[e];
}

// ---- LP ----------------------------------------------------------------------------------------------------------
__global__ void k_lin_CT_y(int nlin, const int* __restrict__ c_ptr, const int* __restrict__ c_row,
                           const double* __restrict__ c_val, const double* __restrict__ y, double scale, double a,
                           const double* __restrict__ base, double* __restrict__ out) {
    int r = blockIdx.x * TB + threadIdx.x;
    if (r >= nlin) return;
    double s = 0.0;
    for (int t = c_ptr[r]; t < c_ptr[r + 1]; t++) s += c_val[t] * y[c_row[t]];
    out[r] = (base ? a * base[r] : 0.0) + scale * s;
}
__global__ void k_lin_C_x(int n_var, const int* __restrict__ r_ptr, const int* __restrict__ r_col,
                          const double* __restrict__ r_val, const double* __restrict__ x, double scale, double* __restrict__ out) {
    int j = blockIdx.x * TB + threadIdx.x;
    if (j >= n_var) return;
    double s = 0.0;
    for (int t = r_ptr[j]; t < r_ptr[j + 1]; t++) s += r_val[t] * x[r_col[t]];
    out[j] += scale * s;
}
__global__ void k_lin_schur(int n_var, const int* __restrict__ r_ptr, const int* __restrict__ r_col,
                            const double* __restrict__ r_val, const int* __restrict__ c_ptr, const int* __restrict__ c_row,
                            const double* __restrict__ c_val, const double* __restrict__ d, double* __restrict__ H, int ldh,
                            double* __restrict__ diag, RowOwner own) {
    int j = blockIdx.x * TB + threadIdx.x;
    if (j >= n_var) return;
    if (H && !own.owns(j)) return;          // thread j writes row j of the lower triangle
    const int jl = own.local(j);
    for (int t = r_ptr[j]; t < r_ptr[j + 1]; t++) {
        const int r = r_col[t];
        const double w = r_val[t] * d[r];
        if (H) {
            for (int u = c_ptr[r]; u < c_ptr[r + 1]; u++) {
                const int k = c_row[u];
                if (k <= j) H[(size_t)k * ldh + jl] += w * c_val[u];
            }
        } else {
            diag[j] += w * r_val[t];
        }
    }
}

}  // namespace

void mat_lincomb(cudaStream_t st, int rows, int cols, double* out, int ldo, double a, const double* A, int lda, double b,
                 const double* B, int ldb, double c, const double* C, int ldc) {
    if (rows <= 0 || cols <= 0) return;
    k_lincomb<<<grid2(rows, cols), TB, 0, st>>>(rows, out, ldo, a, A, lda, b, B, ldb, c, C, ldc);
    LRN_CHECK_LAUNCH();
}
void mat_sym_lincomb(cudaStream_t st, int m, double* out, int ldo, double a, const double* A, int lda, double b,
                     const double* B, int ldb, double c, const double* C, int ldc, double d, const double* D, int ldd) {
    if (m <= 0) return;
    k_sym_lincomb<<<grid2(m, m), TB, 0, st>>>(m, out, ldo, a, A, lda, b, B, ldb, c, C, ldc, d, D, ldd);
    LRN_CHECK_LAUNCH();
}
void mat_symmetrize(cudaStream_t st, int m, double* A, int lda) {
    if (m <= 1) return;
    k_symmetrize<<<grid2(m, m), TB, 0, st>>>(m, A, lda);
    LRN_CHECK_LAUNCH();
}
void mat_scaled_sym(cudaStream_t st, int m, double* out, int ldo, const double* T, int ldt, const double* dd) {
    k_scaled_sym<<<grid2(m, m), TB, 0, st>>>(m, out, ldo, T, ldt, dd);
    LRN_CHECK_LAUNCH();
}
void mat_rnt(cudaStream_t st, int m, double* out, int ldo, const double* T, int ldt, const double* D) {
    k_rnt<<<grid2(m, m), TB, 0, st>>>(m, out, ldo, T, ldt, D);
    LRN_CHECK_LAUNCH();
}
void mat_corr_inner(cudaStream_t st, int m, double* T, int ldt, const double* D, double sigmamu, const double* RNT, int ldr) {
    k_corr_inner<<<grid2(m, m), TB, 0, st>>>(m, T, ldt, D, sigmamu, RNT, ldr);
    LRN_CHECK_LAUNCH();
}
void mat_scale_cols(cudaStream_t st, int rows, int cols, double* out, int ldo, const double* in, int ldi, const double* s) {
    k_scale_cols<<<grid2(rows, cols), TB, 0, st>>>(rows, out, ldo, in, ldi, s);
    LRN_CHECK_LAUNCH();
}
void mat_transpose(cudaStream_t st, int m, double* out, int ldo, const double* in, int ldi) {
    dim3 grid((unsigned)cdiv(m, 32), (unsigned)cdiv(m, 32)), block(32, 8);
    k_transpose<<<grid, block, 0, st>>>(m, out, ldo, in, ldi);
    LRN_CHECK_LAUNCH();
}
void mat_add_diag(cudaStream_t st, int m, double* A, int lda, double v) {
    k_add_diag<<<(unsigned)cdiv(m, TB), TB, 0, st>>>(m, A, lda, v);
    LRN_CHECK_LAUNCH();
}
void mat_add_diag_vec(cudaStream_t st, int m, double* A, int lda, double a, double b, const double* D) {
    k_add_diag_vec<<<(unsigned)cdiv(m, TB), TB, 0, st>>>(m, A, lda, a, b, D);
    LRN_CHECK_LAUNCH();
}
void mat_set_identity(cudaStream_t st, int m, double* A, int lda, double v) {
    k_set_identity<<<grid2(m, m), TB, 0, st>>>(m, A, lda, v);
    LRN_CHECK_LAUNCH();
}
void mat_coldot(cudaStream_t st, int rows, int cols, const double* A, int lda, const double* B, int ldb, double* d) {
    k_coldot<<<(unsigned)cdiv((long long)cols * 32, TB), TB, 0, st>>>(rows, cols, A, lda, B, ldb, d);
    LRN_CHECK_LAUNCH();
}
void mat_mirror_lower(cudaStream_t st, int n, double* A, int lda) {
    if (n <= 1) return;
    const unsigned gy = (unsigned)std::min(n, 32768);
    k_mirror_lower<<<dim3((unsigned)cdiv(n, TB), gy, (unsigned)cdiv(n, gy)), TB, 0, st>>>(n, A, lda);
    LRN_CHECK_LAUNCH();
}
void vec_op(cudaStream_t st, int n, VecOp op, double* out, const double* a, const double* b) {
    if (n <= 0) return;
    k_vec_op<<<(unsigned)cdiv(n, TB), TB, 0, st>>>(n, (int)op, out, a, b);
    LRN_CHECK_LAUNCH();
}
void vec_axpby(cudaStream_t st, int n, double* out, double alpha, const double* a, double beta, const double* b) {
    if (n <= 0) return;
    k_vec_axpby<<<(unsigned)cdiv(n, TB), TB, 0, st>>>(n, out, alpha, a, beta, b);
    LRN_CHECK_LAUNCH();
}

// ---- Reducer -----------------------------------------------------------------------------------------------------
constexpr int RED_BLOCKS = 592;   // 4 x 148

void Reducer::init(int nslots_) {
    nslots = nslots_;
    partial.alloc(RED_BLOCKS);
    slots.alloc(nslots);
    if (!h_slots) LRN_CUDA(cudaMallocHost(&h_slots, nslots * sizeof(double)));
}
Reducer::~Reducer() {
    if (h_slots) cudaFreeHost(h_slots);
}
void Reducer::dot_mat(cudaStream_t st, int rows, int cols, const double* A, int lda, const double* B, int ldb, int slot,
                      bool accumulate) {
    long long total = (long long)rows * cols;
    if (total <= 0) {
        if (!accumulate) LRN_CUDA(cudaMemsetAsync(slots.p + slot, 0, sizeof(double), st));
        return;
    }
    int nb = (int)std::min<long long>(RED_BLOCKS, cdiv(total, TB * 4));
    k_dot_partial<<<nb, TB, 0, st>>>(rows, total, A, lda, B, ldb, partial.p);
    k_sum_finish<<<1, TB, 0, st>>>(partial.p, nb, slots.p + slot, accumulate ? 1 : 0);
    LRN_CHECK_LAUNCH();
}
void Reducer::min_ratio(cudaStream_t st, int n, const double* a, const double* b, int slot, bool accumulate) {
    if (n <= 0) return;
    int nb = (int)std::min<long long>(RED_BLOCKS, cdiv(n, TB * 4));
    k_minratio_partial<<<nb, TB, 0, st>>>(n, a, b, partial.p);
    k_min_finish<<<1, 32, 0, st>>>(partial.p, nb, slots.p + slot, accumulate ? 1 : 0);
    LRN_CHECK_LAUNCH();
}
void Reducer::zero(cudaStream_t st) { LRN_CUDA(cudaMemsetAsync(slots.p, 0, nslots * sizeof(double), st)); }
const double* Reducer::fetch(cudaStream_t st) {
    LRN_CUDA(cudaMemcpyAsync(h_slots, slots.p, nslots * sizeof(double), cudaMemcpyDeviceToHost, st));
    LRN_CUDA(cudaStreamSynchronize(st));
    return h_slots;
}

// ---- sparse launchers ----------------------------------------------------------------------------------------------
void sp_scatter_ATy(cudaStream_t st, const SparseBlock& sb, const double* y, double scale, double* out, int ld) {
    if (sb.npos == 0) return;
    k_scatter_ATy<<<(unsigned)cdiv(sb.npos, TB), TB, 0, st>>>(sb.npos, sb.pos_p.p, sb.pos_q.p, sb.posptr.p, sb.pos_row.p,
                                                              sb.pos_val.p, y, scale, out, ld);
    LRN_CHECK_LAUNCH();
}
void sp_A_vec(cudaStream_t st, const SparseBlock& sb, const double* M, int ld, double scale, double* out) {
    if (sb.nnz == 0) return;
    if (sb.nnz > 16LL * sb.n_var || sb.max_row_nnz > 64)      // long rows: lanes stride the row instead of one serial thread
        k_A_vec_warp<<<(unsigned)cdiv((long long)sb.n_var * 32, TB), TB, 0, st>>>(sb.n_var, sb.rowptr.p, sb.ep.p, sb.eq.p,
                                                                                  sb.ev.p, M, ld, scale, out);
    else
        k_A_vec_thread<<<(unsigned)cdiv(sb.n_var, TB), TB, 0, st>>>(sb.n_var, sb.rowptr.p, sb.ep.p, sb.eq.p, sb.ev.p, M, ld,
                                                                    scale, out);
    LRN_CHECK_LAUNCH();
}
void sp_pos_values(cudaStream_t st, SparseBlock& sb, const double* y) {
    if (sb.npos == 0) return;
    k_pos_values<<<(unsigned)cdiv((long long)sb.npos * 32, 256), 256, 0, st>>>(sb.npos, sb.posptr.p, sb.pos_row.p, sb.pos_val.p, y,
                                                                              sb.mval.p);
    LRN_CHECK_LAUNCH();
}
void sp_M_times_W(cudaStream_t st, const SparseBlock& sb, const double* W, int ldw, double* Z, int ldz) {
    dim3 grid((unsigned)cdiv(sb.m, 256), (unsigned)sb.m);
    k_M_times_W_short<<<grid, 256, 0, st>>>(sb.m, sb.pcolptr.p, sb.pos_p.p, sb.mval.p, W, ldw, Z, ldz);
    LRN_CHECK_LAUNCH();
    if (sb.nlong > 0) {
        dim3 gl((unsigned)cdiv((long long)sb.m * 32, 256), (unsigned)sb.nlong);
        k_M_times_W_long<<<gl, 256, 0, st>>>(sb.m, sb.nlong, sb.longrows.p, sb.pcolptr.p, sb.pos_p.p, sb.mval.p, W, ldw, Z, ldz);
        LRN_CHECK_LAUNCH();
    }
}
void sp_row_sums(cudaStream_t st, const SparseBlock& sb, double scale, double* out) {
    k_row_sums<<<(unsigned)cdiv((long long)sb.n_var * 32, 256), 256, 0, st>>>(sb.n_var, sb.rowptr.p, sb.eval.p, scale, out);
    LRN_CHECK_LAUNCH();
}
void sp_A_sampled(cudaStream_t st, SparseBlock& sb, const double* W, int ldw, const double* Z, int ldz, double scale,
                  double* out) {
    if (sb.nnz == 0) return;
    k_A_sampled<<<(unsigned)cdiv(sb.nnz * 32, 256), 256, 0, st>>>(sb.nnz, sb.m, sb.ep.p, sb.eq.p, sb.ev.p, W, ldw, Z, ldz,
                                                                  sb.eval.p);
    LRN_CHECK_LAUNCH();
    sp_row_sums(st, sb, scale, out);
}
void sp_M_times_cols(cudaStream_t st, const SparseBlock& sb, const double* X, int ldx, int k, double* Y, int ldy) {
    dim3 grid((unsigned)cdiv((long long)sb.m * 32, 256), (unsigned)k);
    k_M_times_cols<<<grid, 256, 0, st>>>(sb.m, k, sb.pcolptr.p, sb.pos_p.p, sb.mval.p, X, ldx, Y, ldy);
    LRN_CHECK_LAUNCH();
}
void sp_A_rank(cudaStream_t st, SparseBlock& sb, const double* ZY, int ldz, const double* U, int ldu, int k, double* out) {
    if (sb.nnz == 0) return;
    k_A_rank_entries<<<(unsigned)cdiv(sb.nnz, TB), TB, 0, st>>>(sb.nnz, sb.ep.p, sb.eq.p, sb.ev.p, ZY, ldz, U, ldu, k, sb.eval.p);
    LRN_CHECK_LAUNCH();
    sp_row_sums(st, sb, 1.0, out);
}
void sp_B_times_G(cudaStream_t st, const SparseBlock& sb, const double* G, int ldg, double* BG, int ldo) {
    dim3 grid((unsigned)cdiv(sb.n_var, TB), (unsigned)sb.m);
    k_B_times_G<<<grid, TB, 0, st>>>(sb.n_var, sb.m, sb.b_rowptr.p, sb.b_col.p, sb.b_val.p, G, ldg, BG, ldo);
    LRN_CHECK_LAUNCH();
}
void sp_schur_pairs(cudaStream_t st, const SparseBlock& sb, int first, const double* W, int ldw, double* H, int ldh,
                    RowOwner own) {
    int cnt = sb.npart - first;
    if (cnt <= 0) return;
    unsigned g = (unsigned)cdiv(cnt, 16);
    LRN_REQUIRE(g <= 65535u, "more than 1048560 participating constraints in one block are not supported");
    dim3 grid(g, g), block(16, 16);
    k_schur_pairs<<<grid, block, 0, st>>>(sb.npart, first, sb.part.p, sb.rowptr.p, sb.ep.p, sb.eq.p, sb.ev.p, W, ldw, H, ldh, own);
    LRN_CHECK_LAUNCH();
}
void sp_schur_f1_column(cudaStream_t st, const SparseBlock& sb, int jj, const double* U, int ldu, double* H, int ldh,
                        RowOwner own) {
    int cnt = sb.npart - jj;
    if (cnt <= 0) return;
    k_schur_f1_column<<<(unsigned)cdiv((long long)cnt * 32, TB), TB, 0, st>>>(sb.npart, jj, sb.part.p, sb.rowptr.p, sb.ep.p,
                                                                              sb.eq.p, sb.ev.p, U, ldu, H, ldh, own);
    LRN_CHECK_LAUNCH();
}
void sp_densify(cudaStream_t st, const SparseBlock& sb, int j, double* out, int ld) {
    const int e0 = sb.h_rowptr[j], e1 = sb.h_rowptr[j + 1];
    if (e1 > e0) {
        k_densify<<<(unsigned)cdiv(e1 - e0, TB), TB, 0, st>>>(e0, e1, sb.ep.p, sb.eq.p, sb.ev.p, out, ld);
        LRN_CHECK_LAUNCH();
    }
}

void lin_CT_y(cudaStream_t st, const SparseLin& L, const double* y, double scale, double a, const double* base, double* out) {
    if (L.nlin <= 0) return;
    k_lin_CT_y<<<(unsigned)cdiv(L.nlin, TB), TB, 0, st>>>(L.nlin, L.c_ptr.p, L.c_row.p, L.c_val.p, y, scale, a, base, out);
    LRN_CHECK_LAUNCH();
}
void lin_C_x(cudaStream_t st, const SparseLin& L, const double* x, double scale, double* out) {
    if (L.nlin <= 0) return;
    k_lin_C_x<<<(unsigned)cdiv(L.n_var, TB), TB, 0, st>>>(L.n_var, L.r_ptr.p, L.r_col.p, L.r_val.p, x, scale, out);
    LRN_CHECK_LAUNCH();
}
void lin_schur(cudaStream_t st, const SparseLin& L, const double* d, double* H, int ldh, RowOwner own) {
    if (L.nlin <= 0) return;
    k_lin_schur<<<(unsigned)cdiv(L.n_var, TB), TB, 0, st>>>(L.n_var, L.r_ptr.p, L.r_col.p, L.r_val.p, L.c_ptr.p, L.c_row.p,
                                                            L.c_val.p, d, H, ldh, nullptr, own);
    LRN_CHECK_LAUNCH();
}
void lin_schur_diag(cudaStream_t st, const SparseLin& L, const double* d, double* diag) {
    if (L.nlin <= 0) return;
    k_lin_schur<<<(unsigned)cdiv(L.n_var, TB), TB, 0, st>>>(L.n_var, L.r_ptr.p, L.r_col.p, L.r_val.p, L.c_ptr.p, L.c_row.p,
                                                            L.c_val.p, d, nullptr, 0, diag, RowOwner());
    LRN_CHECK_LAUNCH();
}

}  // namespace lrn
