// kit = 1 path: preconditioned conjugate gradients on the Schur system without forming it.
//   operator        : MyA functor            src/Solvers.jl:572-614   (solver.cu: apply_A)
//   preconditioners : MyM_no :616-622, H_beta Prec_for_CG_beta/MyM_beta :624-672,
//                     H_alpha Prec_for_CG_tilS_prep/prec_alpha_S!/MyM :674-904
//   recurrence      : ConjugateGradients.jl `cg` (un-vendored; call sites src/predictor_corrector.jl:134,235)
// The whole recurrence keeps its scalars on the device; the host reads one residual norm per iteration.
#include "solver.cuh"
#include "group.cuh"
#include "../../include/loraine_b200_debug.h"
#include <algorithm>
#include <cmath>

using namespace lrn;

namespace lrn {
void solver_apply_A(lrn_solver* h, const double* x, double* out);
}

namespace {

constexpr int TBK = 256;
inline unsigned nb(long long n) { return (unsigned)cdiv(n, TBK); }

enum { S_GAMMA = 8, S_PAP = 9, S_ALPHA = 10, S_RR = 11, S_ZR = 12, S_BETA = 13, S_FLAG = 14 };

__global__ void k_cg_alpha(double* s) {
    double a = s[S_GAMMA] / s[S_PAP];
    s[S_ALPHA] = a;
    if (isinf(a) || a < 0.0) s[S_FLAG] = 1.0;
}
__global__ void k_cg_update(int n, const double* __restrict__ s, const double* __restrict__ p, const double* __restrict__ Ap,
                            double* __restrict__ x, double* __restrict__ r) {
    int i = blockIdx.x * TBK + threadIdx.x;
    if (i >= n) return;
    const double a = s[S_ALPHA];
    x[i] += a * p[i];
    r[i] -= a * Ap[i];
}
__global__ void k_cg_beta(double* s) { s[S_BETA] = s[S_ZR] / s[S_GAMMA]; }
__global__ void k_cg_p(int n, const double* __restrict__ s, const double* __restrict__ z, double* __restrict__ p) {
    int i = blockIdx.x * TBK + threadIdx.x;
    if (i < n) p[i] = z[i] + s[S_BETA] * p[i];
}
__global__ void k_fill2(int n, double* a, double v) {
    int i = blockIdx.x * TBK + threadIdx.x;
    if (i < n) a[i] = v;
}
__global__ void k_set_diag(int n, double* A, int lda, const double* d) {
    int i = blockIdx.x * TBK + threadIdx.x;
    if (i < n) A[(size_t)i * lda + i] = d[i];
}
// AU[j - r0, p] = rowscale[j] * sum_q calA_j[p,q] U[q] for the constraints j of the slab [r0, r0 + rows)
//                                                        (prec_alpha_S!, src/Solvers.jl:833-841)
__global__ void k_build_AU(int r0, int rows, const int* __restrict__ rowptr, const int* __restrict__ ep, const int* __restrict__ eq,
                           const double* __restrict__ ev, const double* __restrict__ U, const double* __restrict__ rowscale,
                           double* __restrict__ AU, int ld) {
    const int i = blockIdx.x * TBK + threadIdx.x;
    if (i >= rows) return;
    const int j = r0 + i;
    const double sc = rowscale ? rowscale[j] : 1.0;
    for (int e = rowptr[j]; e < rowptr[j + 1]; e++) AU[(size_t)ep[e] * ld + i] += sc * ev[e] * U[eq[e]];
}
// Thin products of the H_alpha apply (k = erank <= 8 columns): the DMMA tiles would be 1/64 full, these are plain
// bandwidth-bound kernels instead.
constexpr int THIN_K = 8;
// out(i, c) = sum_r A(r, i) B(r, c): one warp per column i of A (coalesced along the column), shuffle reduction
__global__ void __launch_bounds__(256) k_AtB_thin(const double* __restrict__ A, int lda, int rows, int cols,
                                                  const double* __restrict__ B, int ldb, int k, double* __restrict__ out,
                                                  int ldo) {
    const int i = (blockIdx.x * 256 + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (i >= cols) return;
    const double* a = A + (size_t)i * lda;
    double acc[THIN_K];
#pragma unroll
    for (int c = 0; c < THIN_K; c++) acc[c] = 0.0;
    for (int r = lane; r < rows; r += 32) {
        const double av = a[r];
#pragma unroll
        for (int c = 0; c < THIN_K; c++)
            if (c < k) acc[c] += av * B[(size_t)c * ldb + r];
    }
#pragma unroll
    for (int c = 0; c < THIN_K; c++) {
        if (c >= k) break;
        const double v = warp_sum(acc[c]);
        if (lane == 0) out[(size_t)c * ldo + i] = v;
    }
}
// out(r, c) = sum_i A(r, i) B(i, c): 32 rows x 8 column slices per CTA (coalesced 256 B row segments), shared-memory reduction
__global__ void __launch_bounds__(256) k_AB_thin(const double* __restrict__ A, int lda, int rows, int cols,
                                                 const double* __restrict__ B, int ldb, int k, double* __restrict__ out,
                                                 int ldo) {
    __shared__ double red[8][32];
    const int rl = threadIdx.x & 31, sl = threadIdx.x >> 5;
    const int r = blockIdx.x * 32 + rl;
    const int chunk = (cols + 7) / 8, i0 = sl * chunk, i1 = min(cols, i0 + chunk);
    for (int c = 0; c < k; c++) {
        double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
        if (r < rows) {
            const double* Bc = B + (size_t)c * ldb;
            int i = i0;
            for (; i + 3 < i1; i += 4) {
                a0 += A[(size_t)i * lda + r] * Bc[i];
                a1 += A[(size_t)(i + 1) * lda + r] * Bc[i + 1];
                a2 += A[(size_t)(i + 2) * lda + r] * Bc[i + 2];
                a3 += A[(size_t)(i + 3) * lda + r] * Bc[i + 3];
            }
            for (; i < i1; i++) a0 += A[(size_t)i * lda + r] * Bc[i];
        }
        red[sl][rl] = (a0 + a1) + (a2 + a3);
        __syncthreads();
        if (sl == 0 && r < rows) {
            double t = 0.0;
#pragma unroll
            for (int u = 0; u < 8; u++) t += red[u][rl];
            out[(size_t)c * ldo + r] = t;
        }
        __syncthreads();
    }
}
void AtB_thin(cudaStream_t st, const double* A, int lda, int rows, int cols, const double* B, int ldb, int k, double* out, int ldo) {
    if (k > THIN_K) { gemm_tn(st, cols, k, rows, 1.0, A, lda, B, ldb, 0.0, out, ldo); return; }
    k_AtB_thin<<<(unsigned)cdiv((long long)cols * 32, 256), 256, 0, st>>>(A, lda, rows, cols, B, ldb, k, out, ldo);
    LRN_CHECK_LAUNCH();
}
void AB_thin(cudaStream_t st, const double* A, int lda, int rows, int cols, const double* B, int ldb, int k, double* out, int ldo) {
    if (k > THIN_K) { gemm_nn(st, rows, k, cols, 1.0, A, lda, B, ldb, 0.0, out, ldo); return; }
    k_AB_thin<<<(unsigned)cdiv(rows, 32), 256, 0, st>>>(A, lda, rows, cols, B, ldb, k, out, ldo);
    LRN_CHECK_LAUNCH();
}

struct PhaseT {   // minimal event timer (same bookkeeping as solver.cu)
    lrn_solver* h; PhaseEvt e;
    PhaseT(lrn_solver* h_, int phase) : h(h_) {
        e.phase = phase;
        auto take = [&]() {
            if (h->evpool.empty()) { cudaEvent_t ev; LRN_CUDA(cudaEventCreate(&ev)); return ev; }
            cudaEvent_t ev = h->evpool.back(); h->evpool.pop_back(); return ev;
        };
        e.a = take(); e.b = take();
        LRN_CUDA(cudaEventRecord(e.a, h->st));
    }
    ~PhaseT() { cudaEventRecord(e.b, h->st); h->pending.push_back(e); h->t_calls[e.phase]++; }
};

template <typename F>
int32_t guarded(lrn_solver* h, F&& f) {
    if (!h) return LRN_ERR_ARG;
    try {
        LRN_CUDA(cudaSetDevice(h->device));
        return f();
    } catch (const std::invalid_argument& e) { h->err = e.what(); return LRN_ERR_ARG;
    } catch (const CudaError& e) { h->err = e.what(); return LRN_ERR_CUDA;
    } catch (const std::exception& e) { h->err = e.what(); return LRN_ERR_STATE; }
}

// out = D^{-1} x   (AAAATtau \ x, src/Solvers.jl:874,900)
void d_solve(lrn_solver* h, const double* x, double* out) {
    cudaStream_t st = h->st;
    if (h->pDense) {
        LRN_CUDA(cudaMemcpyAsync(out, x, h->n_var * sizeof(double), cudaMemcpyDeviceToDevice, st));
        chol_solve(h->pDd.p(), h->n_var, h->pDd.ld, h->cholD, out, h->tn1.p, 3, st);
    } else {
        vec_op(st, h->n_var, VEC_DIV, out, x, h->pDiag.p);
    }
}

// tau of one block from the extreme eigenvalues of W (src/Solvers.jl:642-650, :706-719)
int block_tau(lrn_solver* h, Block& B, int k, std::vector<double>& top_vals) {
    cudaStream_t st = h->st;
    const int m = B.m, ld = B.ld;
    if (!B.U.p()) { B.U.init(m, k); B.MU.init(m, k); B.ZY.init(m, k); B.Zf.init(m, m); }
    top_vals.assign(k, 0.0);
    const double tol = h->opt.lanczos_tol > 0 ? h->opt.lanczos_tol : 1e-8;
    LanczosResult r = lanczos_extreme(B.W.p(), m, ld, 3, k, top_vals.data(), B.U.p(), B.U.ld, tol, h->lan, st);
    h->stat_lanczos_iters += r.iters;
    if (!r.converged) h->stat_lanczos_fail++;
    h->red.dot_mat(st, 1, m, B.W.p(), ld + 1, h->ones.p, 1, 15, false);    // trace(W)
    const double* s = h->red.fetch(st);
    const double tr = s[15];
    double sum_l = 0.0;
    for (double v : top_vals) sum_l += v;
    const double min_s = r.lmin, mean_s = (tr - sum_l) / (double)(m - k);
    B.tau = (h->opt.aamat == 0) ? min_s : (min_s + mean_s) / 2.0 - 1.0e-14;
    return 0;
}

void prec_beta(lrn_solver* h) {
    cudaStream_t st = h->st;
    const int n = h->n_var, k = h->opt.erank;
    if (!h->pDiag.p) { h->pDiag.alloc(n); h->pDsq.alloc(n); }
    double shift = 0.0;
    std::vector<double> tv;
    for (auto& B : h->blk) {
        block_tau(h, B, k, tv);
        if (h->opt.aamat < 3) shift += B.tau * B.tau;
    }
    k_fill2<<<nb(n), TBK, 0, st>>>(n, h->pDiag.p, shift);
    if (h->nlmi > 0 && h->nlin > 0) {
        vec_op(st, h->nlin, VEC_MUL, h->tl1.p, h->x_lin.p, h->si_lin.p);
        lin_schur_diag(st, h->lin, h->tl1.p, h->pDiag.p);
    }
    h->pDense = false;
}

int32_t prec_alpha(lrn_solver* h) {
    cudaStream_t st = h->st;
    const int n = h->n_var, k = h->opt.erank;
    LRN_REQUIRE(k >= 1, "erank must be >= 1 for the H_alpha preconditioner");
    if (!h->pDiag.p) { h->pDiag.alloc(n); h->pDsq.alloc(n); }
    int kS = 0, maxm = 1;
    for (auto& B : h->blk) { kS += k * B.m; maxm = std::max(maxm, B.m); }
    if (h->kS != kS || !h->pS.p) {
        h->kS = kS;
        h->pS.alloc((size_t)pad_ld(kS) * kS);
        h->pY.alloc(kS);
        h->pYw.alloc(kS);
    }
    double shift = 0.0;
    std::vector<double> tv, sc(k);
    for (auto& B : h->blk) {
        const int m = B.m, ld = B.ld;
        block_tau(h, B, k, tv);
        if (h->opt.aamat < 3) shift += B.tau * B.tau;
        // Umat = vect_l * sqrt(lambda_l - tau)                                   (src/Solvers.jl:721-722)
        for (int r = 0; r < k; r++) sc[r] = std::sqrt(std::max(tv[r] - B.tau, 0.0));
        LRN_CUDA(cudaMemcpyAsync(B.vtmp.p, sc.data(), k * sizeof(double), cudaMemcpyHostToDevice, st));
        mat_scale_cols(st, m, k, B.U.p(), B.U.ld, B.U.p(), B.U.ld, B.vtmp.p);
        // Z = chol(2 W0 + U U').L with W0 = W - U U'                             (src/Solvers.jl:725-731)
        mat_lincomb(st, m, m, B.Zf.p(), ld, 2.0, B.W.p(), ld, 0.0, nullptr, 0, 0.0, nullptr, 0);
        gemm_nt(st, m, m, k, -1.0, B.U.p(), B.U.ld, B.U.p(), B.U.ld, 1.0, B.Zf.p(), ld);
        cholesky_lower(B.Zf.p(), m, ld, B.cholX, st);     // cholX workspace is free between prepare_W calls
        int info = 0;
        LRN_CUDA(cudaMemcpyAsync(&info, B.cholX.info_ptr(), sizeof(int), cudaMemcpyDeviceToHost, st));
        LRN_CUDA(cudaStreamSynchronize(st));
        B.chol_cached = false;
        if (info != 0) return info;
        zero_strict_upper(B.Zf.p(), m, ld, st);
    }
    // AAAATtau = sum tau_i^2 I (+ C_lin diag(x./s) C_lin')                        (src/Solvers.jl:734-745)
    k_fill2<<<nb(n), TBK, 0, st>>>(n, h->pDiag.p, shift);
    h->pDense = false;
    if (h->nlin > 0) {
        vec_op(st, h->nlin, VEC_MUL, h->tl1.p, h->x_lin.p, h->si_lin.p);
        if (!h->pDd.p()) h->pDd.init(n, n);
        LRN_CUDA(cudaMemsetAsync(h->pDd.p(), 0, h->pDd.bytes(), st));
        lin_schur(st, h->lin, h->tl1.p, h->pDd.p(), h->pDd.ld);
        lin_schur_diag(st, h->lin, h->tl1.p, h->pDiag.p);
        k_set_diag<<<nb(n), TBK, 0, st>>>(n, h->pDd.p(), h->pDd.ld, h->pDiag.p);
        cholesky_lower(h->pDd.p(), n, h->pDd.ld, h->cholD, st);
        int info = 0;
        LRN_CUDA(cudaMemcpyAsync(&info, h->cholD.info_ptr(), sizeof(int), cudaMemcpyDeviceToHost, st));
        LRN_CUDA(cudaStreamSynchronize(st));
        if (info != 0) return info;
        h->pDense = true;
    }
    vec_op(st, n, VEC_RSQRT, h->pDsq.p, h->pDiag.p, nullptr);
    // t = [AA_i kron(U_i, Z_i)]_i ; fast formula scales rows by diag(AAAATtau)^{-1/2}   (src/Solvers.jl:752-801, :819-864)
    const bool fast = (!h->pDense) || k == 1;
    // The fast formula needs T only through S = T'T, so T and A_j u_r are built `R` rows at a time and S accumulates the slab
    // products.  The other formula needs whole columns of T (only reachable with an LP block, i.e. below KIT0_MAX_NVAR).
    const int R = fast ? prec_slab_rows(n, kS, maxm, h->slab_force) : n;
    const int ldt = pad_ld(R);
    if (h->slab_rows != R || h->pT.n != (size_t)ldt * kS) {
        h->pT.alloc((size_t)ldt * kS);
        h->pAU.alloc((size_t)ldt * maxm);
        h->slab_rows = R;
    }
    const int lds = pad_ld(kS);
    for (int r0 = 0; r0 < n; r0 += R) {
        const int rows = std::min(R, n - r0);
        int off = 0;
        for (auto& B : h->blk) {
            const int m = B.m;
            for (int r = 0; r < k; r++) {
                LRN_CUDA(cudaMemsetAsync(h->pAU.p, 0, (size_t)ldt * m * sizeof(double), st));
                k_build_AU<<<nb(rows), TBK, 0, st>>>(r0, rows, B.sp.rowptr.p, B.sp.ep.p, B.sp.eq.p, B.sp.ev.p,
                                                     B.U.p() + (size_t)r * B.U.ld, fast ? h->pDsq.p : nullptr, h->pAU.p, ldt);
                gemm_nn(st, rows, m, m, 1.0, h->pAU.p, ldt, B.Zf.p(), B.ld, 0.0, h->pT.p + (size_t)(off + r * m) * ldt, ldt);
            }
            off += k * m;
        }
        if (fast) gemm_tn(st, kS, kS, rows, 1.0, h->pT.p, ldt, h->pT.p, ldt, r0 > 0 ? 1.0 : 0.0, h->pS.p, lds);
    }
    if (!fast) {
        // S = t' * (AAAATtau \ t), column by column (only for erank > 1 together with an LP block)
        DevBuf<double> DT((size_t)ldt * kS);
        for (int c = 0; c < kS; c++) d_solve(h, h->pT.p + (size_t)c * ldt, DT.p + (size_t)c * ldt);
        gemm_tn(st, kS, kS, n, 1.0, h->pT.p, ldt, DT.p, ldt, 0.0, h->pS.p, lds);
        LRN_CUDA(cudaStreamSynchronize(st));
    }
    // S = (S + S')/2 + I ; cholS = cholesky(S)                                    (src/Solvers.jl:804-805)
    mat_symmetrize(st, kS, h->pS.p, lds);
    mat_add_diag(st, kS, h->pS.p, lds, 1.0);
    cholesky_lower(h->pS.p, kS, lds, h->cholS, st);
    int info = 0;
    LRN_CUDA(cudaMemcpyAsync(&info, h->cholS.info_ptr(), sizeof(int), cudaMemcpyDeviceToHost, st));
    LRN_CUDA(cudaStreamSynchronize(st));
    return info;
}

// Mx = M^{-1} x for the H_alpha preconditioner (MyM functor, src/Solvers.jl:866-904)
void apply_alpha(lrn_solver* h, const double* x, double* out) {
    cudaStream_t st = h->st;
    const int n = h->n_var, k = h->opt.erank;
    double* v = h->tn2.p;
    d_solve(h, x, v);
    int off = 0;
    for (auto& B : h->blk) {
        const int m = B.m, ld = B.ld;
        if (B.sp.sparse_ok) {
            // mat(AA' v) U without densifying: values per stored position, then a gather product with the thin U
            sp_pos_values(st, B.sp, v);
            sp_M_times_cols(st, B.sp, B.U.p(), B.U.ld, k, B.MU.p(), B.MU.ld);
        } else {
            LRN_CUDA(cudaMemsetAsync(B.T1.p(), 0, B.T1.bytes(), st));
            sp_scatter_ATy(st, B.sp, v, 1.0, B.T1.p(), ld);
            AB_thin(st, B.T1.p(), ld, m, m, B.U.p(), B.U.ld, k, B.MU.p(), B.MU.ld);
        }
        AtB_thin(st, B.Zf.p(), ld, m, m, B.MU.p(), B.MU.ld, k, h->pY.p + off, m);
        off += k * m;
    }
    chol_solve(h->pS.p, h->kS, pad_ld(h->kS), h->cholS, h->pY.p, h->pYw.p, 3, st);
    double* yy2 = h->cg_Ap.p;     // free while the preconditioner runs
    LRN_CUDA(cudaMemsetAsync(yy2, 0, n * sizeof(double), st));
    off = 0;
    for (auto& B : h->blk) {
        const int m = B.m, ld = B.ld;
        AB_thin(st, B.Zf.p(), ld, m, m, h->pY.p + off, m, k, B.ZY.p(), B.ZY.ld);
        sp_A_rank(st, B.sp, B.ZY.p(), B.ZY.ld, B.U.p(), B.U.ld, k, yy2);
        off += k * m;
    }
    d_solve(h, yy2, out);
    vec_axpby(st, n, out, 1.0, v, -1.0, out);
}

void apply_prec(lrn_solver* h, int kind, const double* r, double* z) {
    cudaStream_t st = h->st;
    if (kind == 0) LRN_CUDA(cudaMemcpyAsync(z, r, h->n_var * sizeof(double), cudaMemcpyDeviceToDevice, st));
    else if (kind == 1) apply_alpha(h, r, z);
    else vec_op(st, h->n_var, VEC_DIV, z, r, h->pDiag.p);
}

void ensure_cg(lrn_solver* h) {
    if (!h->cg_r.p) {
        for (auto* v : {&h->cg_r, &h->cg_z, &h->cg_p, &h->cg_Ap}) v->alloc(h->n_var);
    }
}

}  // namespace

namespace lrn {
// Above this many bytes for the whole T and A_j u_r the H_alpha build runs in row slabs.
constexpr size_t PREC_SLAB_BUDGET = (size_t)2 << 30;

size_t prec_slab_bytes(int rows, int kS, int maxm) { return (size_t)pad_ld(rows) * ((size_t)kS + (size_t)maxm) * sizeof(double); }

int prec_slab_rows(int n_var, int kS, int maxm, int64_t force) {
    if (force > 0) return (int)std::min<int64_t>(force, n_var);
    if (prec_slab_bytes(n_var, kS, maxm) <= PREC_SLAB_BUDGET) return n_var;
    const size_t per_row = ((size_t)kS + (size_t)maxm) * sizeof(double);
    const size_t R = (PREC_SLAB_BUDGET / per_row) & ~(size_t)7;
    return (int)std::max<size_t>(R, 8);
}
}  // namespace lrn

extern "C" {

int32_t lrn_prec_prepare(lrn_handle_t h, int32_t kind) {
    LRN_GROUP(h, lrn_prec_prepare(m_, kind));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(h->finalized && h->nlmi > 0, "preconditioners need at least one PSD block");
        if (kind == 1 && h->nlin > 0 && h->n_var > KIT0_MAX_NVAR) {
            h->err = "H_alpha with an LP block forms the dense n_var x n_var matrix AAAATtau and factors it; above n_var = " +
                     std::to_string(KIT0_MAX_NVAR) + " it does not fit one GPU (use preconditioner 2, H_beta, which needs only its diagonal)";
            return LRN_ERR_UNSUPPORTED;
        }
        PhaseT ph(h, LRN_T_PREC);
        for (auto& Bk : h->blk) Bk.ud_valid = false;
        ensure_cg(h);
        int32_t rc = LRN_OK;
        if (kind == 1) rc = prec_alpha(h);
        else if (kind == 2 || kind == 4) prec_beta(h);
        else if (kind != 0) { h->err = "preconditioner kind must be 0, 1, 2 or 4"; return LRN_ERR_ARG; }
        h->prec_ready = kind;
        return rc;
    });
}

int32_t lrn_pcg(lrn_handle_t h, double tol, int64_t max_iter, int32_t kind, int64_t* num_iters, int32_t* exit_code) {
    LRN_GROUP(h, lrn_pcg(m_, tol, max_iter, kind, r_ == 0 ? num_iters : group_scratch().i64, r_ == 0 ? exit_code : group_scratch().i32));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(num_iters && exit_code, "null outputs");
        LRN_REQUIRE(kind == 0 || kind == 1 || kind == 2 || kind == 4, "bad preconditioner kind");
        LRN_REQUIRE(kind == 0 || h->prec_ready == kind || (kind != 1 && (h->prec_ready == 2 || h->prec_ready == 4)),
                    "preconditioner not prepared (lrn_prec_prepare)");
        PhaseT ph(h, LRN_T_CG);
        for (auto& Bk : h->blk) Bk.ud_valid = false;
        ensure_cg(h);
        cudaStream_t st = h->st;
        const int n = h->n_var;
        Reducer& R = h->red;
        double* x = h->dely.p;
        double *r = h->cg_r.p, *z = h->cg_z.p, *p = h->cg_p.p, *Ap = h->cg_Ap.p;
        const double* b = h->rhs.p;
        LRN_CUDA(cudaMemsetAsync(x, 0, n * sizeof(double), st));
        R.zero(st);
        R.dot_vec(st, n, b, b, S_RR, false);
        const double* s = R.fetch(st);
        *num_iters = 0;
        if (std::sqrt(s[S_RR]) == 0.0) { *exit_code = 1; return LRN_OK; }
        // r = b - A*0 = b
        LRN_CUDA(cudaMemcpyAsync(r, b, n * sizeof(double), cudaMemcpyDeviceToDevice, st));
        const double res0 = std::sqrt(s[S_RR]);
        if (res0 <= tol) { *exit_code = 2; return LRN_OK; }
        apply_prec(h, kind, r, z);
        LRN_CUDA(cudaMemcpyAsync(p, z, n * sizeof(double), cudaMemcpyDeviceToDevice, st));
        // One CG iteration is ~25 small launches (operator, preconditioner, vector updates) followed by ONE host read of the
        // residual norm.  All operands live at fixed device addresses, so from the second iteration on the whole body
        // -- z = M r, beta, p, Ap = A p, alpha, x, r, |r|^2 -- is replayed as a CUDA graph captured once per call (the first
        // iteration runs eagerly and warms every lazily configured kernel / workspace).
        auto part_a = [&]() {
            solver_apply_A(h, p, Ap);
            R.dot_vec(st, n, r, z, S_GAMMA, false);
            R.dot_vec(st, n, p, Ap, S_PAP, false);
            k_cg_alpha<<<1, 1, 0, st>>>(R.slots.p);
            k_cg_update<<<nb(n), TBK, 0, st>>>(n, R.slots.p, p, Ap, x, r);
            R.dot_vec(st, n, r, r, S_RR, false);
            LRN_CHECK_LAUNCH();
        };
        auto part_b = [&]() {
            apply_prec(h, kind, r, z);
            R.dot_vec(st, n, z, r, S_ZR, false);
            k_cg_beta<<<1, 1, 0, st>>>(R.slots.p);
            k_cg_p<<<nb(n), TBK, 0, st>>>(n, R.slots.p, z, p);
            LRN_CHECK_LAUNCH();
        };
        cudaGraph_t graph = nullptr;
        cudaGraphExec_t gexec = nullptr;
        long long graph_nodes = 0;
        bool use_graph = !gemm_profile_active() && max_iter >= 3;
        auto release = [&]() {
            if (gexec) cudaGraphExecDestroy(gexec);
            if (graph) cudaGraphDestroy(graph);
            gexec = nullptr; graph = nullptr;
        };
        for (int64_t it = 1; it <= max_iter; it++) {
            if (it == 1) {
                part_a();
            } else if (it == 2 || !use_graph) {
                part_b();          // eager once more: the preconditioner's second application still sees first-use set-up
                part_a();
            } else {
                if (!gexec) {
                    bool ok = cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
                    if (ok) {
                        const long long before = g_kernel_launches.load();
                        try { part_b(); part_a(); } catch (...) { ok = false; }
                        cudaGraph_t gcap = nullptr;
                        if (cudaStreamEndCapture(st, &gcap) != cudaSuccess || !gcap) ok = false;
                        graph = gcap;
                        if (ok && cudaGraphInstantiate(&gexec, graph, 0) != cudaSuccess) ok = false;
                        graph_nodes = g_kernel_launches.load() - before;
                        g_kernel_launches.fetch_sub(graph_nodes);       // counted per replay below
                    }
                    if (!ok) {                                            // fall back to eager launches for the rest of the call
                        cudaGetLastError();
                        release();
                        use_graph = false;
                        part_b();
                        part_a();
                    }
                }
                if (gexec) {
                    LRN_CUDA(cudaGraphLaunch(gexec, st));
                    g_kernel_launches.fetch_add(graph_nodes);
                }
            }
            s = R.fetch(st);
            if (s[S_FLAG] != 0.0 || std::isnan(s[S_ALPHA])) { *exit_code = -13; *num_iters = it; release(); return LRN_OK; }
            if (std::sqrt(s[S_RR]) / res0 <= tol) { *exit_code = 30; *num_iters = it; release(); return LRN_OK; }
        }
        release();
        *exit_code = -2;
        *num_iters = max_iter;
        LRN_CUDA(cudaStreamSynchronize(st));
        return LRN_OK;
    });
}

int32_t lrn_apply_operator(lrn_handle_t h, int32_t kind, const double* x, double* out) {
    if (h && h->group) return lrn_apply_operator(static_cast<Group*>(h->group)->members[0], kind, x, out);
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(x && out, "null pointers");
        ensure_cg(h);
        cudaStream_t st = h->st;
        const int n = h->n_var;
        h->cg_p.upload(x, n, st);
        if (kind == -1) solver_apply_A(h, h->cg_p.p, h->cg_z.p);
        else apply_prec(h, kind, h->cg_p.p, h->cg_z.p);
        LRN_CUDA(cudaMemcpyAsync(out, h->cg_z.p, n * sizeof(double), cudaMemcpyDeviceToHost, st));
        LRN_CUDA(cudaStreamSynchronize(st));
        return LRN_OK;
    });
}

int32_t lrn_dbg_prec_slab(lrn_handle_t h, int64_t set_rows, int64_t* rows_used) {
    if (h && h->group) {
        Group* g = static_cast<Group*>(h->group);
        for (auto* m : g->members) {
            const int32_t rc = lrn_dbg_prec_slab(m, set_rows, nullptr);
            if (rc != LRN_OK) return rc;
        }
        return lrn_dbg_prec_slab(g->members[0], set_rows, rows_used);
    }
    if (!h || set_rows < 0) return LRN_ERR_ARG;
    h->slab_force = set_rows;
    if (rows_used) *rows_used = h->slab_rows;
    return LRN_OK;
}

}  // extern "C"
