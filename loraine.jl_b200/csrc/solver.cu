// C ABI + device-resident interior-point state.  Every entry point cites the reference lines it replaces in
// include/loraine_b200.h.  No CPU fallback: all arithmetic of the hot path runs in the kernels of gemm.cu / chol.cu /
// eig.cu / ops.cu and in the small kernels below.
#include "solver.cuh"
#include "dist.cuh"
#include "group.cuh"
#include <algorithm>
#include <cmath>
#include <numeric>
#include <thread>

using namespace lrn;

namespace lrn {
void record_model_norms(lrn_solver* h, const std::vector<double>& b_host);   // model.cu
}

namespace {

constexpr int TBK = 256;

// ---- small LP-block kernels (vectors of length nlin) -------------------------------------------------------------------
// predictor: t = (x .* si) .* rd + x                                             (src/predictor_corrector.jl:49)
// corrector: t = (x .* si) .* rd + x + (dx .* ds) .* si - sigmamu .* si          (src/predictor_corrector.jl:190-191)
__global__ void k_lp_rhs(int n, int corr, double sigmamu, const double* x, const double* si, const double* rd,
                         const double* dx, const double* ds, double* t) {
    int i = blockIdx.x * TBK + threadIdx.x;
    if (i >= n) return;
    double v = (x[i] * si[i]) * rd[i] + x[i];
    if (corr) v += (dx[i] * ds[i]) * si[i] - sigmamu * si[i];
    t[i] = v;
}
// find_step_lin, src/predictor_corrector.jl:330-335:  dx = -x - x.*si.*ds [+ sigmamu.*si + rnt]
__global__ void k_lp_dx(int n, int corr, double sigmamu, const double* x, const double* si, const double* ds,
                        const double* rnt, double* dx) {
    int i = blockIdx.x * TBK + threadIdx.x;
    if (i >= n) return;
    double v = -x[i] - x[i] * si[i] * ds[i];
    if (corr) v += sigmamu * si[i] + rnt[i];
    dx[i] = v;
}
// src/predictor_corrector.jl:351-354
__global__ void k_lp_pred_update(int n, double a, double b, const double* x, const double* s, const double* dx,
                                 const double* ds, const double* si, double* xn, double* sn, double* rnt) {
    int i = blockIdx.x * TBK + threadIdx.x;
    if (i >= n) return;
    xn[i] = x[i] + a * dx[i];
    sn[i] = s[i] + b * ds[i];
    rnt[i] = -(dx[i] * ds[i]) * si[i];
}
// CG operator LP part: t = (x .* sinv) .* t                                       (src/Solvers.jl:609)
__global__ void k_mul3(int n, const double* a, const double* b, double* t) {
    int i = blockIdx.x * TBK + threadIdx.x;
    if (i < n) t[i] = (a[i] * b[i]) * t[i];
}
__global__ void k_fill(int n, double* a, double v) {
    int i = blockIdx.x * TBK + threadIdx.x;
    if (i < n) a[i] = v;
}

inline unsigned nb(long long n) { return (unsigned)cdiv(n, TBK); }

// ---- error / timer plumbing ------------------------------------------------------------------------------------------
struct Phase {
    lrn_solver* h;
    PhaseEvt e;
    Phase(lrn_solver* h_, int phase) : h(h_) {
        e.phase = phase;
        auto take = [&]() {
            if (h->evpool.empty()) {
                cudaEvent_t ev;
                LRN_CUDA(cudaEventCreate(&ev));
                return ev;
            }
            cudaEvent_t ev = h->evpool.back();
            h->evpool.pop_back();
            return ev;
        };
        e.a = take();
        e.b = take();
        LRN_CUDA(cudaEventRecord(e.a, h->st));
    }
    ~Phase() {
        cudaEventRecord(e.b, h->st);
        h->pending.push_back(e);
        h->t_calls[e.phase]++;
    }
};

void flush_timers(lrn_solver* h) {
    if (h->pending.empty()) return;
    LRN_CUDA(cudaStreamSynchronize(h->st));
    for (auto& e : h->pending) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, e.a, e.b) == cudaSuccess) h->t_ms[e.phase] += ms;
        h->evpool.push_back(e.a);
        h->evpool.push_back(e.b);
    }
    h->pending.clear();
}

template <typename F>
int32_t guarded(lrn_solver* h, F&& f) {
    if (!h) return LRN_ERR_ARG;
    try {
        LRN_CUDA(cudaSetDevice(h->device));
        int32_t r = f();
        if (h->pending.size() > 512) flush_timers(h);
        return r;
    } catch (const std::invalid_argument& e) {
        h->err = e.what();
        return LRN_ERR_ARG;
    } catch (const CudaError& e) {
        h->err = e.what();
        return LRN_ERR_CUDA;
    } catch (const std::exception& e) {
        h->err = e.what();
        return LRN_ERR_STATE;
    }
}

void upload_dense(lrn_solver* h, DMat& M, const double* host) {
    LRN_CUDA(cudaMemcpy2DAsync(M.p(), (size_t)M.ld * sizeof(double), host, (size_t)M.rows * sizeof(double),
                               (size_t)M.rows * sizeof(double), M.cols, cudaMemcpyHostToDevice, h->st));
}
void download_dense(lrn_solver* h, const double* dev, int ld, int rows, int cols, double* host) {
    LRN_CUDA(cudaMemcpy2DAsync(host, (size_t)rows * sizeof(double), dev, (size_t)ld * sizeof(double),
                               (size_t)rows * sizeof(double), cols, cudaMemcpyDeviceToHost, h->st));
}

void copy_csc(HostCSC& dst, int64_t ncol, const int64_t* colptr, const int64_t* rowval, const double* nzval) {
    LRN_REQUIRE(colptr && colptr[0] == 1, "colptr must be 1-based (Julia SparseMatrixCSC)");
    dst.colptr.assign(colptr, colptr + ncol + 1);
    const int64_t nnz = colptr[ncol] - 1;
    LRN_REQUIRE(nnz >= 0 && nnz < 2000000000LL, "nnz out of range");
    LRN_REQUIRE(nnz == 0 || (rowval && nzval), "null rowval/nzval");
    dst.rowval.assign(rowval, rowval + nnz);
    dst.nzval.assign(nzval, nzval + nnz);
    for (auto& c : dst.colptr) c -= 1;
    for (auto& r : dst.rowval) r -= 1;
    dst.set = true;
}

// Build the device structures of one PSD block from the staged Julia CSC of AA_i (n_var x m^2).
void build_block(lrn_solver* h, Block& B) {
    const int m = B.m, n = h->n_var;
    SparseBlock& sp = B.sp;
    sp.m = m;
    sp.n_var = n;
    LRN_REQUIRE(B.hAA.set, "lrn_set_block_AA was not called for every block");
    const auto& cp = B.hAA.colptr;
    const auto& rv = B.hAA.rowval;
    const auto& nz = B.hAA.nzval;
    const int64_t nnz = (int64_t)rv.size();
    sp.nnz = nnz;
    std::vector<int> rowptr(n + 1, 0);
    for (int64_t e = 0; e < nnz; e++) {
        LRN_REQUIRE(rv[e] >= 0 && rv[e] < n, "AA row index out of range");
        rowptr[rv[e] + 1]++;
    }
    for (int j = 0; j < n; j++) rowptr[j + 1] += rowptr[j];
    std::vector<int> ep(nnz), eq(nnz), fill(rowptr.begin(), rowptr.end() - 1);
    std::vector<double> ev(nnz);
    std::vector<int> pos_p, pos_q, posptr, pos_row((size_t)nnz);
    std::vector<double> pos_val((size_t)nnz);
    posptr.push_back(0);
    const int64_t ncol = (int64_t)m * m;
    int64_t w = 0;
    for (int64_t c = 0; c < ncol; c++) {
        if (cp[c + 1] == cp[c]) continue;
        const int p = (int)(c % m), q = (int)(c / m);
        for (int64_t e = cp[c]; e < cp[c + 1]; e++) {
            const int j = (int)rv[e];
            const int dst = fill[j]++;
            ep[dst] = p; eq[dst] = q; ev[dst] = nz[e];
            pos_row[w] = j; pos_val[w] = nz[e];
            w++;
        }
        pos_p.push_back(p); pos_q.push_back(q); posptr.push_back((int)w);
    }
    sp.npos = (int)pos_p.size();
    {
        // sparse-aware Schur operator (kit = 1): needs symmetric storage of every calA_j (entry (p,q,v) <=> (q,p,v)) and a
        // sparse union pattern; otherwise the operator keeps the dense W M W form
        std::vector<int> pcol(m + 1, 0);
        for (size_t t = 0; t < pos_q.size(); t++) pcol[pos_q[t] + 1]++;
        for (int q = 0; q < m; q++) pcol[q + 1] += pcol[q];
        bool sym = true;
        {
            // positions are sorted by (q, p); (p,q) and (q,p) must carry identical (constraint, value) lists
            auto find = [&](int p, int q) -> long long {
                int lo = pcol[q], hi = pcol[q + 1];
                while (lo < hi) { int mid = (lo + hi) >> 1; if (pos_p[mid] < p) lo = mid + 1; else hi = mid; }
                return (lo < pcol[q + 1] && pos_p[lo] == p) ? lo : -1;
            };
            for (size_t t = 0; t < pos_p.size() && sym; t++) {
                if (pos_p[t] <= pos_q[t]) continue;
                long long u = find(pos_q[t], pos_p[t]);
                if (u < 0 || posptr[u + 1] - posptr[u] != posptr[t + 1] - posptr[t]) { sym = false; break; }
                for (int a = posptr[t], b2 = posptr[u]; a < posptr[t + 1]; a++, b2++)
                    if (pos_row[a] != pos_row[b2] || pos_val[a] != pos_val[b2]) { sym = false; break; }
            }
            // every strictly-upper position needs its mirror too: count check
            long long lower = 0, upper = 0;
            for (size_t t = 0; t < pos_p.size(); t++) { if (pos_p[t] > pos_q[t]) lower++; else if (pos_p[t] < pos_q[t]) upper++; }
            if (lower != upper) sym = false;
        }
        int maxrow = 0;
        for (int j = 0; j < n; j++) maxrow = std::max(maxrow, rowptr[j + 1] - rowptr[j]);
        (void)maxrow;
        sp.sparse_ok = sym && sp.npos > 0;
        sp.sparse_op = sp.sparse_ok && (double)sp.npos <= 0.05 * (double)m * m;
        if (sp.sparse_ok) {
            sp.pcolptr.upload(pcol, h->st);
            std::vector<int> longrows;
            for (int r = 0; r < m; r++) if (pcol[r + 1] - pcol[r] > 32) longrows.push_back(r);
            sp.nlong = (int)longrows.size();
            if (sp.nlong > 0) sp.longrows.upload(longrows, h->st);
            sp.mval.alloc((size_t)std::max(sp.npos, 1));
        }
        sp.eval.alloc((size_t)std::max<int64_t>(nnz, 1));
        if (getenv("LRN_DEBUG_BUILD"))
            fprintf(stderr, "[lrn build] block m=%d nnz=%lld npos=%d symmetric=%d sparse_ok=%d sparse_op=%d\n", m, (long long)nnz,
                    sp.npos, (int)sym, (int)sp.sparse_ok, (int)sp.sparse_op);
    }
    // participating constraints in nnz-descending stable order (= sigmaA restricted to nnz > 0, src/model.jl:157-160)
    std::vector<int> part;
    for (int j = 0; j < n; j++) if (rowptr[j + 1] > rowptr[j]) part.push_back(j);
    std::stable_sort(part.begin(), part.end(), [&](int a, int b2) {
        return (rowptr[a + 1] - rowptr[a]) > (rowptr[b2 + 1] - rowptr[b2]);
    });
    sp.npart = (int)part.size();
    sp.max_row_nnz = sp.npart ? rowptr[part[0] + 1] - rowptr[part[0]] : 0;
    // F1 / F3 split: a prefix of the nnz-sorted list uses the dense formula
    int nF1 = 0;
    if (h->opt.schur_split == 1) {
        for (int jj = 0; jj < sp.npart; jj++) {
            int nzj = rowptr[part[jj] + 1] - rowptr[part[jj]];
            if (nzj > h->opt.datasparsity) nF1 = jj + 1; else break;
        }
    } else {
        // cost model (SURVEY 8(d)): F3_j ~ nnz_j * sum_{k>=j} nnz_k gathered pairs, F1_j ~ 4 m^3 tensor flops + launches
        double suffix = 0.0;
        std::vector<double> suf(sp.npart + 1, 0.0);
        for (int jj = sp.npart - 1; jj >= 0; jj--) {
            suffix += rowptr[part[jj] + 1] - rowptr[part[jj]];
            suf[jj] = suffix;
        }
        for (int jj = 0; jj < sp.npart; jj++) {
            double nzj = rowptr[part[jj] + 1] - rowptr[part[jj]];
            if (nzj * suf[jj] > 0.13 * (double)m * m * m + 2.0e7) nF1 = jj + 1; else break;
        }
    }
    sp.nF1 = nF1;
    if (h->opt.kit == 0) sp_build_pair_plan(sp, rowptr, ep, eq, ev, h->st);   // staged pair kernel of the Schur assembly
    sp.h_rowptr = rowptr;
    sp.h_part = part;
    sp.rowptr.upload(rowptr, h->st); sp.ep.upload(ep, h->st); sp.eq.upload(eq, h->st); sp.ev.upload(ev, h->st);
    sp.pos_p.upload(pos_p, h->st); sp.pos_q.upload(pos_q, h->st); sp.posptr.upload(posptr, h->st);
    sp.pos_row.upload(pos_row, h->st); sp.pos_val.upload(pos_val, h->st);
    sp.part.upload(part, h->st);
    // rank-one factors: Julia CSC n_var x m  ->  CSR by constraint
    if (B.hB.set) {
        const auto& bc = B.hB.colptr;
        const int64_t bn = (int64_t)B.hB.rowval.size();
        std::vector<int> brp(n + 1, 0), bcol(bn);
        std::vector<double> bval(bn);
        for (int64_t e = 0; e < bn; e++) brp[B.hB.rowval[e] + 1]++;
        for (int j = 0; j < n; j++) brp[j + 1] += brp[j];
        std::vector<int> f2(brp.begin(), brp.end() - 1);
        for (int c = 0; c < m; c++)
            for (int64_t e = bc[c]; e < bc[c + 1]; e++) {
                int dst = f2[B.hB.rowval[e]]++;
                bcol[dst] = c; bval[dst] = B.hB.nzval[e];
            }
        sp.has_B = bn > 0;
        sp.nnzB = bn;
        sp.b_rowptr.upload(brp, h->st); sp.b_col.upload(bcol, h->st); sp.b_val.upload(bval, h->st);
    }
    // dense C_i
    B.C.init(m, m);
    double nc = 0.0;
    if (B.hC.set) {
        std::vector<double> Cd((size_t)B.C.ld * m, 0.0);
        for (int c = 0; c < m; c++)
            for (int64_t e = B.hC.colptr[c]; e < B.hC.colptr[c + 1]; e++) {
                Cd[(size_t)c * B.C.ld + B.hC.rowval[e]] += B.hC.nzval[e];
            }
        for (int c = 0; c < m; c++)
            for (int r = 0; r < m; r++) nc += Cd[(size_t)c * B.C.ld + r] * Cd[(size_t)c * B.C.ld + r];
        B.C.buf.upload(Cd.data(), Cd.size(), h->st);
    }
    B.normC = std::sqrt(nc);
    LRN_CUDA(cudaStreamSynchronize(h->st));
    B.hAA = HostCSC(); B.hB = HostCSC(); B.hC = HostCSC();
    for (DMat* M : {&B.X, &B.S, &B.dX, &B.dS, &B.Xn, &B.Sn, &B.G, &B.Gi, &B.W, &B.Si, &B.Rd, &B.RNT, &B.LX, &B.LS, &B.T1, &B.T2, &B.T3, &B.T4})
        M->init(m, m);
    B.ld = B.X.ld;
    B.D.alloc(m); B.DDsi.alloc(m); B.dm12.alloc(m); B.dm32.alloc(m); B.vtmp.alloc(m);
}

// row-wise Gershgorin bounds of sign * T:  g[i] = sign T_ii - sum_{j != i} |T_ij|   (lambda_min(sign T) >= min_i g[i])
__global__ void k_gershgorin(int m, const double* __restrict__ T, int ld, double sign, double* __restrict__ g) {
    const int i = (blockIdx.x * 256 + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (i >= m) return;
    double s = 0.0;
    for (int j = lane; j < m; j += 32) if (j != i) s += fabs(T[(size_t)i * ld + j]);     // T symmetric: column i read contiguously
    s = warp_sum(s);
    if (lane == 0) g[i] = sign * T[(size_t)i * ld + i] - s;
}
__global__ void k_shifted_copy(int m, const double* __restrict__ T, int ldt, double sign, double shift, double* __restrict__ out, int ldo) {
    const int i = blockIdx.x * 256 + threadIdx.x, j = blockIdx.y;
    if (i < m) out[(size_t)j * ldo + i] = sign * T[(size_t)j * ldt + i] - (i == j ? shift : 0.0);
}

// Guaranteed fallback for an extreme eigenvalue when Lanczos did not converge (ADVICE r1: an unconverged Ritz value lies
// ABOVE lambda_min, so the step length would be overestimated and the iterate could leave the cone silently):
// lambda_min(sign T) by bisection on "sign T - t I is positive definite" (one Cholesky per step), between the Gershgorin
// lower bound and the Ritz value `hi` (an upper bound of lambda_min).  Returns a value t with t <= lambda_min < t + tol_abs.
double extreme_by_bisection(lrn_solver* h, const double* T, int m, int ld, double sign, double hi) {
    cudaStream_t st = h->st;
    if (h->eig_scratch.rows != m) h->eig_scratch.init(m, m);
    DevBuf<double> g((size_t)m);
    k_gershgorin<<<nb((long long)m * 32), TBK, 0, st>>>(m, T, ld, sign, g.p);
    LRN_CHECK_LAUNCH();
    h->red.min_ratio(st, m, g.p, nullptr, 7, false);
    double lo = h->red.fetch(st)[7];
    const double scale = std::max(std::fabs(lo), std::fabs(hi));
    const double tol_abs = 1e-9 * (scale > 0 ? scale : 1.0);
    if (!(lo < hi)) return std::min(lo, hi);
    for (int it = 0; it < 80 && hi - lo > tol_abs; it++) {
        const double t = 0.5 * (lo + hi);
        k_shifted_copy<<<dim3(nb(m), (unsigned)m), TBK, 0, st>>>(m, T, ld, sign, t, h->eig_scratch.p(), h->eig_scratch.ld);
        LRN_CHECK_LAUNCH();
        cholesky_lower(h->eig_scratch.p(), m, h->eig_scratch.ld, h->eig_chol, st);
        int info = 0;
        LRN_CUDA(cudaMemcpyAsync(&info, h->eig_chol.info_ptr(), sizeof(int), cudaMemcpyDeviceToHost, st));
        LRN_CUDA(cudaStreamSynchronize(st));
        if (info == 0) lo = t; else hi = t;          // positive definite  <=>  t < lambda_min
        h->stat_bisect++;
    }
    return lo;
}

// smallest (and optionally largest) eigenvalue of the symmetric m x m matrix T (device)
double lambda_min(lrn_solver* h, const double* T, int m, int ld, double* lmax = nullptr) {
    Phase ph(h, LRN_T_EIGMIN);
    double tol = h->opt.lanczos_tol > 0 ? h->opt.lanczos_tol : 1e-8;
    LanczosResult r = lanczos_extreme(T, m, ld, lmax ? 3 : 1, 0, nullptr, nullptr, 0, tol, h->lan, h->st, h->lanczos_kmax);
    h->stat_lanczos_iters += r.iters;
    if (!r.converged) {
        // not converged within the Krylov budget: replace the Ritz values by guaranteed bounds (bisection on Cholesky tests)
        h->stat_lanczos_fail++;
        const double sc = std::max(std::fabs(r.lmin), std::fabs(r.lmax));
        if (r.resid_min > tol * (sc > 0 ? sc : 1.0)) r.lmin = extreme_by_bisection(h, T, m, ld, 1.0, r.lmin);
        if (lmax && r.resid_max > tol * (sc > 0 ? sc : 1.0)) r.lmax = -extreme_by_bisection(h, T, m, ld, -1.0, -r.lmax);
    }
    if (lmax) *lmax = r.lmax;
    return r.lmin;
}

// lambda_min of two symmetric matrices at once (see the corrector branch of lrn_find_step)
void lambda_min_pair(lrn_solver* h, const double* Ta, const double* Tb, int m, int ld, double* la, double* lb) {
    Phase ph(h, LRN_T_EIGMIN);
    const double tol = h->opt.lanczos_tol > 0 ? h->opt.lanczos_tol : 1e-8;
    if (!h->st2) {
        LRN_CUDA(cudaStreamCreateWithFlags(&h->st2, cudaStreamNonBlocking));
        LRN_CUDA(cudaEventCreateWithFlags(&h->ev2, cudaEventDisableTiming));
    }
    LRN_CUDA(cudaEventRecord(h->ev2, h->st));               // both matrices were produced on the main stream
    LRN_CUDA(cudaStreamWaitEvent(h->st2, h->ev2, 0));
    LanczosResult ra, rb;
    std::string err_a;
    const int dev = h->device, kmax = h->lanczos_kmax;
    std::thread ta([&] {
        try {
            LRN_CUDA(cudaSetDevice(dev));
            ra = lanczos_extreme(Ta, m, ld, 1, 0, nullptr, nullptr, 0, tol, h->lan2, h->st2, kmax);
        } catch (const std::exception& e) { err_a = e.what(); }
    });
    try {
        rb = lanczos_extreme(Tb, m, ld, 1, 0, nullptr, nullptr, 0, tol, h->lan, h->st, kmax);
    } catch (...) { ta.join(); throw; }
    ta.join();
    if (!err_a.empty()) throw CudaError(err_a);
    h->stat_lanczos_iters += ra.iters + rb.iters;
    for (int k = 0; k < 2; k++) {                           // non-converged runs: guaranteed bounds instead of Ritz values
        LanczosResult& r = k ? rb : ra;
        if (r.converged) continue;
        h->stat_lanczos_fail++;
        const double sc = std::max(std::fabs(r.lmin), std::fabs(r.lmax));
        if (r.resid_min > tol * (sc > 0 ? sc : 1.0)) r.lmin = extreme_by_bisection(h, k ? Tb : Ta, m, ld, 1.0, r.lmin);
    }
    *la = ra.lmin;
    *lb = rb.lmin;
}

inline double steplen(double mimi, double tau) { return (mimi > -1e-6) ? 0.99 : std::min(1.0, -tau / mimi); }

// Factor X (or S) of block `B` into L with the reference's try_cholesky retry loop (src/prepare_W.jl:5-26).
bool try_cholesky(lrn_solver* h, DMat& X, DMat& L, CholWork& cw) {
    const int m = X.rows;
    for (int icount = 0;; icount++) {
        LRN_CUDA(cudaMemcpyAsync(L.p(), X.p(), X.bytes(), cudaMemcpyDeviceToDevice, h->st));
        cholesky_lower(L.p(), m, L.ld, cw, h->st);
        int info = 0;
        LRN_CUDA(cudaMemcpyAsync(&info, cw.info_ptr(), sizeof(int), cudaMemcpyDeviceToHost, h->st));
        LRN_CUDA(cudaStreamSynchronize(h->st));
        if (info == 0) return true;
        if (icount >= 1000) {
            mat_set_identity(h->st, m, L.p(), L.ld, 1.0);
            cholesky_lower(L.p(), m, L.ld, cw, h->st);   // keeps dinv consistent with the identity factor
            return false;
        }
        mat_add_diag(h->st, m, X.p(), X.ld, 1e-5);
    }
}

// out = A x  (MyA functor, src/Solvers.jl:582-614)
void apply_A(lrn_solver* h, const double* x, double* out) {
    cudaStream_t st = h->st;
    LRN_CUDA(cudaMemsetAsync(out, 0, (size_t)h->n_var * sizeof(double), st));
    for (auto& B : h->blk) {
        const int m = B.m, ld = B.ld;
        if (B.sp.sparse_op) {
            // M = mat(AA' x) is sparse: Z = M W by gathers, then <calA_j, W Z> sampled at the stored positions (HBM/L2-bound,
            // 2 (npos + nnz) m flops instead of 4 m^3)
            sp_pos_values(st, B.sp, x);
            sp_M_times_W(st, B.sp, B.W.p(), ld, B.T2.p(), ld);
            sp_A_sampled(st, B.sp, B.W.p(), ld, B.T2.p(), ld, 1.0, out);
            continue;
        }
        LRN_CUDA(cudaMemsetAsync(B.T1.p(), 0, B.T1.bytes(), st));
        sp_scatter_ATy(st, B.sp, x, 1.0, B.T1.p(), ld);
        gemm_nn(st, m, m, m, 1.0, B.W.p(), ld, B.T1.p(), ld, 0.0, B.T2.p(), ld);
        gemm_nn(st, m, m, m, 1.0, B.T2.p(), ld, B.W.p(), ld, 0.0, B.T3.p(), ld);
        sp_A_vec(st, B.sp, B.T3.p(), ld, 1.0, out);
    }
    if (h->nlin > 0) {
        lin_CT_y(st, h->lin, x, 1.0, 0.0, nullptr, h->tl1.p);
        k_mul3<<<nb(h->nlin), TBK, 0, st>>>(h->nlin, h->x_lin.p, h->si_lin.p, h->tl1.p);
        lin_C_x(st, h->lin, h->tl1.p, 1.0, out);
    }
}

}  // namespace

// =======================================================================================================================
//  C ABI
// =======================================================================================================================
extern "C" {

void lrn_default_options(lrn_options_t* o) {
    if (!o) return;
    std::memset(o, 0, sizeof(*o));
    o->kit = 0; o->datarank = 0; o->preconditioner = 1; o->erank = 1; o->aamat = 1; o->datasparsity = 8;
    o->schur_split = 0; o->rank1_mode = 0; o->svd_tol = 0.0; o->lanczos_tol = 0.0; o->device = -1;
}

int32_t lrn_create(lrn_handle_t* out, int64_t n_var, int64_t nlmi, const int64_t* msizes, int64_t nlin,
                   const lrn_options_t* opt) {
    if (!out) return LRN_ERR_ARG;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return LRN_ERR_NO_DEVICE;
    lrn_solver* h = new lrn_solver();
    if (opt) h->opt = *opt; else lrn_default_options(&h->opt);
    int32_t rc = guarded(h, [&]() -> int32_t {
        int dev = h->opt.device;
        if (dev < 0) {
            const char* lr = getenv("LOCAL_RANK");
            dev = lr ? atoi(lr) % ndev : 0;
        }
        LRN_REQUIRE(dev < ndev, "device ordinal out of range");
        h->device = dev;
        LRN_CUDA(cudaSetDevice(dev));
        cudaDeviceProp prop;
        LRN_CUDA(cudaGetDeviceProperties(&prop, dev));
        if (prop.major < 10) {
            h->err = "loraine_b200 requires an sm_100 (Blackwell) GPU; there is no fallback path";
            return LRN_ERR_NO_DEVICE;
        }
        // kit = 0: the Schur matrix and its factor are dense n_var x n_var FP64 (2 x 8 n_var^2 bytes): 140 000 is what 180 GB
        // of HBM holds.  kit = 1 forms neither; its limit is the device memory lrn_finalize checks (indices stay int).
        if (h->opt.kit == 1) LRN_REQUIRE(n_var >= 1 && n_var <= INT32_MAX, "n_var out of range (1..2147483647 for kit = 1)");
        else LRN_REQUIRE(n_var >= 1 && n_var <= KIT0_MAX_NVAR, "n_var out of range (1..140000)");
        LRN_REQUIRE(nlmi >= 0 && nlin >= 0 && nlin < 2000000000LL, "nlmi/nlin out of range");
        LRN_REQUIRE(nlmi == 0 || msizes, "msizes is null");
        h->n_var = (int)n_var; h->nlmi = (int)nlmi; h->nlin = (int)nlin;
        LRN_CUDA(cudaStreamCreateWithFlags(&h->st, cudaStreamNonBlocking));
        h->blk.resize(nlmi);
        for (int i = 0; i < nlmi; i++) {
            LRN_REQUIRE(msizes[i] >= 1 && msizes[i] <= 46000, "block size out of range");
            h->blk[i].m = (int)msizes[i];
            h->sum_m += msizes[i];
        }
        return LRN_OK;
    });
    if (rc != LRN_OK && rc != LRN_ERR_NO_DEVICE) { *out = h; return rc; }
    if (rc == LRN_ERR_NO_DEVICE) { delete h; return rc; }
    *out = h;
    return LRN_OK;
}

int32_t lrn_set_block_AA(lrn_handle_t h, int64_t i, const int64_t* colptr, const int64_t* rowval, const double* nzval) {
    LRN_GROUP(h, lrn_set_block_AA(m_, i, colptr, rowval, nzval));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(i >= 0 && i < h->nlmi && !h->finalized, "bad block index / already finalized");
        copy_csc(h->blk[i].hAA, (int64_t)h->blk[i].m * h->blk[i].m, colptr, rowval, nzval);
        return LRN_OK;
    });
}
int32_t lrn_set_block_C(lrn_handle_t h, int64_t i, const int64_t* colptr, const int64_t* rowval, const double* nzval) {
    LRN_GROUP(h, lrn_set_block_C(m_, i, colptr, rowval, nzval));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(i >= 0 && i < h->nlmi && !h->finalized, "bad block index / already finalized");
        copy_csc(h->blk[i].hC, h->blk[i].m, colptr, rowval, nzval);
        return LRN_OK;
    });
}
int32_t lrn_set_block_B(lrn_handle_t h, int64_t i, const int64_t* colptr, const int64_t* rowval, const double* nzval) {
    LRN_GROUP(h, lrn_set_block_B(m_, i, colptr, rowval, nzval));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(i >= 0 && i < h->nlmi && !h->finalized, "bad block index / already finalized");
        copy_csc(h->blk[i].hB, h->blk[i].m, colptr, rowval, nzval);
        return LRN_OK;
    });
}
int32_t lrn_set_lin(lrn_handle_t h, const int64_t* colptr, const int64_t* rowval, const double* nzval, const double* d_lin) {
    LRN_GROUP(h, lrn_set_lin(m_, colptr, rowval, nzval, d_lin));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(!h->finalized, "already finalized");
        if (h->nlin == 0) return LRN_OK;
        LRN_REQUIRE(d_lin, "d_lin is null");
        copy_csc(h->hClin, h->nlin, colptr, rowval, nzval);
        h->d_lin.upload(d_lin, h->nlin, h->st);
        double s = 0;
        for (int r = 0; r < h->nlin; r++) s += d_lin[r] * d_lin[r];
        h->normd = std::sqrt(s);
        LRN_CUDA(cudaStreamSynchronize(h->st));
        return LRN_OK;
    });
}
int32_t lrn_set_b(lrn_handle_t h, const double* b) {
    LRN_GROUP(h, lrn_set_b(m_, b));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(b, "b is null");
        h->b.upload(b, h->n_var, h->st);
        h->hb.assign(b, b + h->n_var);
        double s = 0;
        for (int j = 0; j < h->n_var; j++) s += b[j] * b[j];
        h->normb = std::sqrt(s);
        LRN_CUDA(cudaStreamSynchronize(h->st));
        return LRN_OK;
    });
}

// Device bytes of the kit = 1 state, from the staged model: model data, the n_var-long vectors, the m x m block arrays, and
// for H_alpha the kS x kS matrix S and one slab of its row-slab build (the dense AAAATtau of an LP block below KIT0_MAX_NVAR).
static size_t cg_footprint(const lrn_solver* h) {
    const size_t n = (size_t)h->n_var, d = sizeof(double), ix = sizeof(int);
    size_t bytes = 14 * n * d;                                    // y, dely, rhs, Rp, tn1, tn2, ones, b, 4 CG vectors, pDiag, pDsq
    int kS = 0, maxm = 1;
    for (const auto& B : h->blk) {
        const size_t nnz = B.hAA.rowval.size(), nnzB = B.hB.rowval.size(), mm = (size_t)pad_ld(B.m) * B.m;
        bytes += nnz * (3 * ix + 3 * d) + nnz * (3 * ix + d);     // by-constraint (p, q, v, values), by-position lists
        bytes += 2 * (n + 1) * ix + nnzB * (ix + d);              // row pointers, constraint order, rank-one factors
        bytes += 24 * mm * d;                                     // X, S, W, G, ... T1-T4, C, Z, work of the m x m kernels
        kS += h->opt.erank * B.m;
        maxm = std::max(maxm, B.m);
    }
    if (h->nlin > 0) bytes += 2 * h->hClin.rowval.size() * (ix + d) + (n + h->nlin + 2) * ix + 12 * (size_t)h->nlin * d;
    if (h->opt.preconditioner == 1 || h->opt.preconditioner == 4) {
        bytes += ((size_t)pad_ld(kS) * kS + 2 * (size_t)kS) * d;
        bytes += prec_slab_bytes(prec_slab_rows(h->n_var, kS, maxm, h->slab_force), kS, maxm);
        if (h->nlin > 0 && h->n_var <= KIT0_MAX_NVAR) bytes += (size_t)pad_ld(h->n_var) * n * d;
    }
    return bytes;
}

int32_t lrn_finalize(lrn_handle_t h) {
    LRN_GROUP(h, lrn_finalize(m_));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(!h->finalized, "already finalized");
        LRN_REQUIRE(h->b.p, "lrn_set_b was not called");
        if (h->opt.kit == 1) {
            // refuse a model whose CG state cannot fit before anything is allocated, instead of failing partway through a solve
            size_t free_b = 0, total_b = 0;
            LRN_CUDA(cudaMemGetInfo(&free_b, &total_b));
            const size_t need = cg_footprint(h);
            if (need > free_b)
                throw std::invalid_argument("kit = 1 state needs " + std::to_string(need) + " bytes of device memory, " +
                                            std::to_string(free_b) + " bytes are free");
        }
        const int n = h->n_var;
        int maxm = 1;
        record_model_norms(h, h->hb);          // norms of AA_i, b, C_lin rows for lrn_initial_point (host copies still exist)
        for (auto& B : h->blk) { build_block(h, B); maxm = std::max(maxm, B.m); }
        if (h->nlin > 0) {
            LRN_REQUIRE(h->hClin.set, "lrn_set_lin was not called");
            SparseLin& L = h->lin;
            L.n_var = n; L.nlin = h->nlin;
            const auto& cp = h->hClin.colptr;
            const int64_t nnz = (int64_t)h->hClin.rowval.size();
            L.nnz = nnz;
            std::vector<int> cptr(cp.begin(), cp.end()), crow(h->hClin.rowval.begin(), h->hClin.rowval.end());
            std::vector<int> rptr(n + 1, 0), rcol(nnz);
            std::vector<double> rval(nnz);
            for (int64_t e = 0; e < nnz; e++) {
                LRN_REQUIRE(crow[e] >= 0 && crow[e] < n, "C_lin row index out of range");
                rptr[crow[e] + 1]++;
            }
            for (int j = 0; j < n; j++) rptr[j + 1] += rptr[j];
            std::vector<int> f(rptr.begin(), rptr.end() - 1);
            for (int r = 0; r < h->nlin; r++)
                for (int64_t e = cp[r]; e < cp[r + 1]; e++) {
                    int dst = f[crow[e]]++;
                    rcol[dst] = r; rval[dst] = h->hClin.nzval[e];
                }
            L.c_ptr.upload(cptr, h->st); L.c_row.upload(crow, h->st); L.c_val.upload(h->hClin.nzval, h->st);
            L.r_ptr.upload(rptr, h->st); L.r_col.upload(rcol, h->st); L.r_val.upload(rval, h->st);
            LRN_CUDA(cudaStreamSynchronize(h->st));
            h->hClin = HostCSC();
            for (auto* v : {&h->x_lin, &h->s_lin, &h->si_lin, &h->dx_lin, &h->ds_lin, &h->xn_lin, &h->sn_lin, &h->rnt_lin,
                            &h->rd_lin, &h->tl1, &h->tl2})
                v->alloc(h->nlin);
        }
        for (auto* v : {&h->y, &h->dely, &h->rhs, &h->Rp, &h->tn1, &h->tn2}) v->alloc(n);
        const int nones = std::max(std::max(n, h->nlin), maxm);
        h->ones.alloc(nones);
        k_fill<<<nb(nones), TBK, 0, h->st>>>(nones, h->ones.p, 1.0);
        h->blk_info.alloc(2 * std::max(1, h->nlmi));
        for (int i = 0; i < h->nlmi; i++) {
            h->blk[i].cholX.info_ext = h->blk_info.p + 2 * i;
            h->blk[i].cholS.info_ext = h->blk_info.p + 2 * i + 1;
        }
        h->red.init(16 + 4 * std::max(1, h->nlmi));
        {   // equal-sized blocks share a batched SVD
            std::vector<std::pair<int, std::vector<int>>> bym;
            for (int i = 0; i < h->nlmi; i++) {
                bool found = false;
                for (auto& g : bym) if (g.first == h->blk[i].m) { g.second.push_back(i); found = true; }
                if (!found) bym.push_back({h->blk[i].m, {i}});
            }
            h->svd_group_of.assign(h->nlmi, -1);
            for (auto& g : bym) {
                if (g.second.size() < 2) continue;
                auto G = std::make_unique<SvdGroup>();
                G->m = g.first; G->blocks = g.second;
                std::vector<const double*> a; std::vector<double*> ud, sg;
                for (int i : g.second) {
                    a.push_back(h->blk[i].T1.p()); ud.push_back(h->blk[i].T2.p()); sg.push_back(h->blk[i].D.p);
                    h->svd_group_of[i] = (int)h->svd_groups.size();
                }
                G->A.upload(a, h->st); G->UD.upload(ud, h->st); G->sig.upload(sg, h->st);
                h->svd_groups.push_back(std::move(G));
            }
        }
        {   // small blocks get their two eigmin's per find_step from one batched launch
            std::vector<double*> ptrs; std::vector<int> ms, lds;
            for (int i = 0; i < h->nlmi; i++) {
                Block& B = h->blk[i];
                if (B.m > 64 && B.m <= 384) {
                    h->eig_small.push_back(i);
                    ptrs.push_back(B.T4.p()); ptrs.push_back(B.T1.p());
                    ms.push_back(B.m); ms.push_back(B.m); lds.push_back(B.ld); lds.push_back(B.ld);
                }
            }
            if (!ptrs.empty()) {
                h->eig_ptrs.upload(ptrs, h->st); h->eig_ms.upload(ms, h->st); h->eig_lds.upload(lds, h->st);
                h->eig_out.alloc(ptrs.size());
            }
        }
        bool rank1 = (h->opt.datarank == -1) && h->nlmi > 0;
        for (auto& B : h->blk) rank1 = rank1 && B.sp.has_B;
        if (h->opt.datarank == -1 && !rank1) h->opt.datarank = 0;      // src/Solvers.jl:435-444
        if (h->opt.kit == 0) {
            h->H.init(n, n);
            h->L.init(n, n);
            if (rank1) h->BG.init(n, round_up(maxm, 32));   // K padded to a multiple of 32 (zero columns) for the TMA-fed SYRK
        }
        LRN_CUDA(cudaStreamSynchronize(h->st));
        h->finalized = true;
        return LRN_OK;
    });
}

int32_t lrn_destroy(lrn_handle_t h) {
    if (!h) return LRN_OK;
    if (h->group) {
        Group* g = static_cast<Group*>(h->group);
        // the communicators of one ncclCommInitAll clique are destroyed from concurrent threads (ncclCommDestroy may wait for peers)
        std::vector<std::thread> th;
        for (auto* m : g->members) th.emplace_back([m] { lrn_destroy(m); });
        for (auto& t : th) t.join();
        delete g;
        delete h;
        return LRN_OK;
    }
    cudaSetDevice(h->device);
    if (h->st) cudaStreamSynchronize(h->st);
    for (auto& e : h->pending) { cudaEventDestroy(e.a); cudaEventDestroy(e.b); }
    for (auto& e : h->evpool) cudaEventDestroy(e);
    cudaStream_t st = h->st;
    for (auto& s_ : h->side) if (s_) { cudaStreamSynchronize(s_); cudaStreamDestroy(s_); }
    if (h->evFork) cudaEventDestroy(h->evFork);
    for (auto& e : h->evJoin) if (e) cudaEventDestroy(e);
    if (h->st2) { cudaStreamSynchronize(h->st2); cudaStreamDestroy(h->st2); }
    if (h->ev2) cudaEventDestroy(h->ev2);
    if (h->nccl) { delete static_cast<DistCtx*>(h->nccl); h->nccl = nullptr; }
    delete h;
    if (st) cudaStreamDestroy(st);
    return LRN_OK;
}

int32_t lrn_get_dims(lrn_handle_t h, int64_t* n_var, int64_t* nlmi, int64_t* nlin, int64_t* msizes) {
    if (!h) return LRN_ERR_ARG;
    if (h->group) return lrn_get_dims(static_cast<Group*>(h->group)->members[0], n_var, nlmi, nlin, msizes);
    if (n_var) *n_var = h->n_var;
    if (nlmi) *nlmi = h->nlmi;
    if (nlin) *nlin = h->nlin;
    if (msizes) for (int i = 0; i < h->nlmi; i++) msizes[i] = h->blk[i].m;
    return LRN_OK;
}

const char* lrn_last_error(lrn_handle_t h) {
    if (!h) return "null handle";
    if (h->group && h->err.empty() && !static_cast<Group*>(h->group)->members.empty())
        return static_cast<Group*>(h->group)->members[0]->err.c_str();
    return h->err.c_str();
}

// ---- iterate ----------------------------------------------------------------------------------------------------------
int32_t lrn_set_iterate(lrn_handle_t h, const double* const* X, const double* const* S, const double* y, const double* x_lin,
                        const double* s_lin) {
    LRN_GROUP(h, lrn_set_iterate(m_, X, S, y, x_lin, s_lin));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(h->finalized, "lrn_finalize first");
        for (int i = 0; i < h->nlmi; i++) {
            LRN_REQUIRE(X && S && X[i] && S[i], "null X/S block");
            upload_dense(h, h->blk[i].X, X[i]);
            upload_dense(h, h->blk[i].S, S[i]);
            h->blk[i].chol_cached = false;
            h->blk[i].rdb_valid = false;
        }
        LRN_REQUIRE(y, "null y");
        h->y.upload(y, h->n_var, h->st);
        if (h->nlin > 0) {
            LRN_REQUIRE(x_lin && s_lin, "null x_lin/s_lin");
            h->x_lin.upload(x_lin, h->nlin, h->st);
            h->s_lin.upload(s_lin, h->nlin, h->st);
            vec_op(h->st, h->nlin, VEC_RECIP, h->si_lin.p, h->s_lin.p, nullptr);
        }
        LRN_CUDA(cudaStreamSynchronize(h->st));
        h->have_factor = false;
        return LRN_OK;
    });
}

int32_t lrn_get_solution(lrn_handle_t h, double* y, double* const* X, double* x_lin) {
    if (h && h->group) return lrn_get_solution(static_cast<Group*>(h->group)->members[0], y, X, x_lin);
    return guarded(h, [&]() -> int32_t {
        if (y) LRN_CUDA(cudaMemcpyAsync(y, h->y.p, h->n_var * sizeof(double), cudaMemcpyDeviceToHost, h->st));
        if (X)
            for (int i = 0; i < h->nlmi; i++)
                if (X[i]) download_dense(h, h->blk[i].X.p(), h->blk[i].ld, h->blk[i].m, h->blk[i].m, X[i]);
        if (x_lin && h->nlin > 0)
            LRN_CUDA(cudaMemcpyAsync(x_lin, h->x_lin.p, h->nlin * sizeof(double), cudaMemcpyDeviceToHost, h->st));
        LRN_CUDA(cudaStreamSynchronize(h->st));
        return LRN_OK;
    });
}

int32_t lrn_get_slack(lrn_handle_t h, double* const* S, double* s_lin) {
    if (h && h->group) return lrn_get_slack(static_cast<Group*>(h->group)->members[0], S, s_lin);
    return guarded(h, [&]() -> int32_t {
        if (S)
            for (int i = 0; i < h->nlmi; i++)
                if (S[i]) download_dense(h, h->blk[i].S.p(), h->blk[i].ld, h->blk[i].m, h->blk[i].m, S[i]);
        if (s_lin && h->nlin > 0)
            LRN_CUDA(cudaMemcpyAsync(s_lin, h->s_lin.p, h->nlin * sizeof(double), cudaMemcpyDeviceToHost, h->st));
        LRN_CUDA(cudaStreamSynchronize(h->st));
        return LRN_OK;
    });
}

// symmetric m x m product op(A) op(B): only the tiles that meet the lower triangle are computed, then mirrored
static void gemm_sym(cudaStream_t st, bool ta, bool tb, int m, const double* A, int lda, const double* B, int ldb, double* C,
                     int ldc) {
    GemmParams p;
    p.A = A; p.B = B; p.C = C; p.M = m; p.N = m; p.K = m; p.lda = lda; p.ldb = ldb; p.ldc = ldc;
    p.transA = ta; p.transB = tb; p.lower = 1;
    gemm(p, st);
    mat_mirror_lower(st, m, C, ldc);
}

// Sparse data: delS = Rd - M with a sparse M = mat(AA' dely), so G' delS G = G' Rd G - G' (M G).  G' Rd G is formed once per
// iteration (Rd and G are fixed between lrn_residuals / lrn_prepare_W calls); M G is a gather product.
static bool use_rdb(const Block& B) { return B.sp.sparse_ok && (double)B.sp.npos <= 0.05 * (double)B.m * B.m; }
static void ensure_rdb(lrn_solver* h, Block& B, cudaStream_t st) {
    if (B.rdb_valid) return;
    const int m = B.m, ld = B.ld;
    if (!B.RdB.p()) {
        LRN_CUDA(cudaStreamSynchronize(st));       // DevBuf allocation synchronises the device anyway; keep the order explicit
        B.RdB.init(m, m);
    }
    gemm_nn(st, m, m, m, 1.0, B.Rd.p(), ld, B.G.p(), ld, 0.0, B.T1.p(), ld);
    gemm_sym(st, true, false, m, B.G.p(), ld, B.T1.p(), ld, B.RdB.p(), B.RdB.ld);
    B.rdb_valid = true;
}

// fork / join of the side streams around a loop over independent PSD blocks
static void side_fork(lrn_solver* h) {
    if (!h->side[0]) {
        for (auto& s_ : h->side) LRN_CUDA(cudaStreamCreateWithFlags(&s_, cudaStreamNonBlocking));
        LRN_CUDA(cudaEventCreateWithFlags(&h->evFork, cudaEventDisableTiming));
        for (auto& e : h->evJoin) LRN_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    LRN_CUDA(cudaEventRecord(h->evFork, h->st));
    for (auto& s_ : h->side) LRN_CUDA(cudaStreamWaitEvent(s_, h->evFork, 0));
}
static void side_join(lrn_solver* h) {
    for (int k = 0; k < lrn_solver::NSIDE; k++) {
        LRN_CUDA(cudaEventRecord(h->evJoin[k], h->side[k]));
        LRN_CUDA(cudaStreamWaitEvent(h->st, h->evJoin[k], 0));
    }
}

// ---- hot path -------------------------------------------------------------------------------------------------------
int32_t lrn_find_mu(lrn_handle_t h, double* mu) {
    LRN_GROUP(h, lrn_find_mu(m_, r_ == 0 ? mu : group_scratch().d));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(mu, "null output");
        cudaStream_t st = h->st;
        h->red.zero(st);
        for (auto& B : h->blk) h->red.dot_mat(st, B.m, B.m, B.X.p(), B.ld, B.S.p(), B.ld, 0, true);
        if (h->nlin > 0) h->red.dot_vec(st, h->nlin, h->x_lin.p, h->s_lin.p, 0, true);
        const double* r = h->red.fetch(st);
        *mu = r[0] / (double)(h->sum_m + h->nlin);
        return LRN_OK;
    });
}

int32_t lrn_prepare_W(lrn_handle_t h, int32_t* status4) {
    LRN_GROUP(h, lrn_prepare_W(m_, r_ == 0 ? status4 : group_scratch().i32));
    return guarded(h, [&]() -> int32_t {
        Phase ph(h, LRN_T_PREPARE_W);
        cudaStream_t st = h->st;
        if (status4) *status4 = 0;
        const double svd_tol = h->opt.svd_tol > 0 ? h->opt.svd_tol : 1e-8;
        for (auto& B : h->blk) {
            const int m = B.m, ld = B.ld;
            if (!B.chol_cached) {
                bool okx = try_cholesky(h, B.X, B.LX, B.cholX);
                bool oks = try_cholesky(h, B.S, B.LS, B.cholS);
                if ((!okx || !oks) && status4) *status4 = 1;
            }
            B.chol_cached = false;
            B.rdb_valid = false;
            zero_strict_upper(B.LX.p(), m, ld, st);
            zero_strict_upper(B.LS.p(), m, ld, st);
            // CC = L_S' L_X                                                   (src/prepare_W.jl:39)
            {
                GemmParams p;                    // both factors are lower triangular: the K loop of a tile starts at max(m0, n0)
                p.A = B.LS.p(); p.B = B.LX.p(); p.C = B.T1.p(); p.M = m; p.N = m; p.K = m; p.lda = ld; p.ldb = ld; p.ldc = ld;
                p.transA = true; p.ktri = 1;
                gemm(p, st);
            }
        }
        // U*D, D = svd(CC) without accumulating V                                (src/prepare_W.jl:42)
        {
            Phase ps(h, LRN_T_SVD);
            for (auto& G : h->svd_groups)
                h->stat_svd_sweeps = svd_block_jacobi_batched(G->A.p, h->blk[G->blocks[0]].ld, G->m, (int)G->blocks.size(), G->UD.p,
                                                              h->blk[G->blocks[0]].ld, G->sig.p, G->w, svd_tol, 30, st);
            for (int i = 0; i < h->nlmi; i++) {
                if (h->svd_group_of[i] >= 0) continue;
                Block& B = h->blk[i];
                h->stat_svd_sweeps = svd_block_jacobi(B.T1.p(), B.ld, B.m, B.T2.p(), B.ld, nullptr, 0, B.D.p, B.svd, svd_tol, 30, st);
            }
        }
        const bool fanw = h->nlmi >= 4;          // independent per-block post-processing chains -> side streams
        if (fanw) side_fork(h);
        cudaStream_t st_main = st;
        for (int ib = 0; ib < h->nlmi; ib++) {
            Block& B = h->blk[ib];
            const int m = B.m, ld = B.ld;
            cudaStream_t st = fanw ? h->side[ib % lrn_solver::NSIDE] : st_main;
            vec_op(st, m, VEC_RSQRT, B.dm12.p, B.D.p, nullptr);
            vec_op(st, m, VEC_POW_M32, B.dm32.p, B.D.p, nullptr);
            // G = L_X V D^{-1/2} = L_S^{-T} (U D) D^{-1/2}   (CC V = U D with CC = L_S' L_X)   (src/prepare_W.jl:60)
            mat_scale_cols(st, m, m, B.G.p(), ld, B.T2.p(), ld, B.dm12.p);
            trsm_left_lower_trans(B.LS.p(), m, ld, B.cholS, B.G.p(), ld, m, st);
            // Gi = inv(G) (src/prepare_W.jl:63) is never multiplied with anything on the device (find_step uses the closed
            // forms of the scaled directions); it is produced on demand for the LRN_ARR_GI parity hook from U D kept in T2.
            // W = G G'                                                        (src/prepare_W.jl:64)
            gemm_sym(st, false, true, m, B.G.p(), ld, B.G.p(), ld, B.W.p(), ld);
            // Si = S^{-1} = (G D^{-1/2}) (G D^{-1/2})'                        (src/prepare_W.jl:68; G'SG = D)
            mat_scale_cols(st, m, m, B.T1.p(), ld, B.G.p(), ld, B.dm12.p);
            gemm_sym(st, false, true, m, B.T1.p(), ld, B.T1.p(), ld, B.Si.p(), ld);
            // DDsi = 1 ./ sqrt(diag(G' S G))  (src/prepare_W.jl:71-74).  With G = L_S^{-T} (U D) D^{-1/2} the p-th diagonal entry
            // of G' S G is ||(U D)(:,p)||^2 / D_p = D_p exactly (D_p IS that column norm), so DDsi = D^{-1/2} without a GEMM.
            LRN_CUDA(cudaMemcpyAsync(B.DDsi.p, B.dm12.p, m * sizeof(double), cudaMemcpyDeviceToDevice, st));
            B.ud_valid = true;        // T2 = U D and LS stay intact until the next call that uses the scratch matrices
        }
        if (fanw) side_join(h);
        if (h->nlin > 0) vec_op(st, h->nlin, VEC_RECIP, h->si_lin.p, h->s_lin.p, nullptr);
        return LRN_OK;
    });
}

int32_t lrn_residuals(lrn_handle_t h) {
    LRN_GROUP(h, lrn_residuals(m_));
    return guarded(h, [&]() -> int32_t {
        Phase ph(h, LRN_T_RESIDUALS);
        cudaStream_t st = h->st;
        const int n = h->n_var;
        LRN_CUDA(cudaMemcpyAsync(h->Rp.p, h->b.p, n * sizeof(double), cudaMemcpyDeviceToDevice, st));
        for (auto& B : h->blk) {
            B.rdb_valid = false;
            sp_A_vec(st, B.sp, B.X.p(), B.ld, -1.0, h->Rp.p);
            mat_lincomb(st, B.m, B.m, B.Rd.p(), B.ld, 1.0, B.C.p(), B.C.ld, -1.0, B.S.p(), B.ld, 0.0, nullptr, 0);
            sp_scatter_ATy(st, B.sp, h->y.p, -1.0, B.Rd.p(), B.ld);
        }
        if (h->nlin > 0) {
            lin_C_x(st, h->lin, h->x_lin.p, -1.0, h->Rp.p);
            vec_axpby(st, h->nlin, h->tl1.p, 1.0, h->d_lin.p, -1.0, h->s_lin.p);
            lin_CT_y(st, h->lin, h->y.p, -1.0, 1.0, h->tl1.p, h->rd_lin.p);
        }
        return LRN_OK;
    });
}

int32_t lrn_schur_assemble(lrn_handle_t h) {
    LRN_GROUP(h, lrn_schur_assemble(m_));
    return guarded(h, [&]() -> int32_t {
        for (auto& Bk : h->blk) Bk.ud_valid = false;
        LRN_REQUIRE(h->H.p(), "Schur matrix is only allocated for kit = 0");
        Phase ph(h, LRN_T_ASSEMBLE);
        cudaStream_t st = h->st;
        const int n = h->n_var;
        LRN_CUDA(cudaMemsetAsync(h->H.p(), 0, h->H.bytes(), st));
        h->H_gathered = false;
        RowOwner own;                                  // multi-GPU: every rank assembles only the row blocks it owns
        own.rank = h->rank; own.world = h->world; own.pw = h->dist_pw;
        bool first_block = true;                       // H is still all zeros
        for (auto& B : h->blk) {
            const int m = B.m, ld = B.ld;
            const bool h_is_zero = first_block;
            first_block = false;
            if (h->opt.datarank == -1) {
                // BBBB += ((B G)(B G)').^2                                    (src/makeBBBB.jl:7-14)
                sp_B_times_G(st, B.sp, B.G.p(), ld, h->BG.p(), h->BG.ld);
                const int Kp = round_up(m, 32);          // zero padding columns: K % 32 == 0 selects the TMA-fed kernel
                if (Kp > m)
                    LRN_CUDA(cudaMemsetAsync(h->BG.p() + (size_t)m * h->BG.ld, 0, (size_t)(Kp - m) * h->BG.ld * sizeof(double), st));
                GemmParams p;
                p.A = h->BG.p(); p.B = h->BG.p(); p.C = h->H.p();
                p.M = n; p.N = n; p.K = Kp; p.lda = h->BG.ld; p.ldb = h->BG.ld; p.ldc = h->H.ld;
                p.transB = true; p.alpha = 1.0; p.beta = 1.0; p.mode = 1; p.lower = 1;
                if (h->world <= 1) gemm(p, st);
                else syrk_sq_row_blocks(h->BG.p(), h->BG.ld, n, Kp, h->H.p(), h->H.ld, own.rank, own.world, own.pw, st);
            } else {
                for (int jj = 0; jj < B.sp.nF1; jj++) {
                    // F1: U = W calA_j W, column of <calA_k, U>                (src/makeBBBB.jl:81-104)
                    LRN_CUDA(cudaMemsetAsync(B.T1.p(), 0, B.T1.bytes(), st));
                    sp_densify(st, B.sp, B.sp.h_part[jj], B.T1.p(), ld);
                    gemm_nn(st, m, m, m, 1.0, B.W.p(), ld, B.T1.p(), ld, 0.0, B.T2.p(), ld);
                    gemm_nn(st, m, m, m, 1.0, B.T2.p(), ld, B.W.p(), ld, 0.0, B.T3.p(), ld);
                    sp_schur_f1_column(st, B.sp, jj, B.T3.p(), ld, h->H.p(), h->H.ld, own);
                }
                // F3 for the remaining (sparse) matrices                       (src/makeBBBB.jl:139-213)
                if (B.sp.pairs.ok && (h->use_staged_pairs == 1 || (h->use_staged_pairs < 0 && B.sp.npart >= 1024)))
                    sp_schur_pairs_staged(st, B.sp, B.W.p(), ld, h->H.p(), h->H.ld, own, !(h_is_zero && B.sp.nF1 == 0));
                else sp_schur_pairs(st, B.sp, B.sp.nF1, B.W.p(), ld, h->H.p(), h->H.ld, own);
            }
        }
        if (h->nlin > 0) {
            // BBBB += C_lin * spdiagm(X_lin .* S_lin_inv) * C_lin'             (src/predictor_corrector.jl:36-38)
            vec_op(st, h->nlin, VEC_MUL, h->tl1.p, h->x_lin.p, h->si_lin.p);
            lin_schur(st, h->lin, h->tl1.p, h->H.p(), h->H.ld, own);
        }
        h->have_factor = false;
        return LRN_OK;
    });
}

static void add_lp_rhs(lrn_solver* h, int corr, double sigmamu) {
    if (h->nlin <= 0) return;
    k_lp_rhs<<<nb(h->nlin), TBK, 0, h->st>>>(h->nlin, corr, sigmamu, h->x_lin.p, h->si_lin.p, h->rd_lin.p, h->dx_lin.p,
                                              h->ds_lin.p, h->tl1.p);
    lin_C_x(h->st, h->lin, h->tl1.p, 1.0, h->rhs.p);
}

int32_t lrn_rhs_predictor(lrn_handle_t h) {
    LRN_GROUP(h, lrn_rhs_predictor(m_));
    return guarded(h, [&]() -> int32_t {
        for (auto& Bk : h->blk) Bk.ud_valid = false;
        Phase ph(h, LRN_T_RHS);
        cudaStream_t st = h->st;
        LRN_CUDA(cudaMemcpyAsync(h->rhs.p, h->Rp.p, h->n_var * sizeof(double), cudaMemcpyDeviceToDevice, st));
        for (auto& B : h->blk) {
            const int m = B.m, ld = B.ld;
            // h += AA * vec(W (Rd + S) W)                                     (src/makeBBBB.jl:225)
            mat_lincomb(st, m, m, B.T1.p(), ld, 1.0, B.Rd.p(), ld, 1.0, B.S.p(), ld, 0.0, nullptr, 0);
            if ((double)B.sp.nnz <= 0.05 * (double)m * m) {
                // sparse data: <calA_j, W T W> is only needed at the stored positions -- Z = T W (one product), then one
                // m-long inner product <W(:,p), Z(:,q)> per stored entry instead of the second m^3 product
                gemm_nn(st, m, m, m, 1.0, B.T1.p(), ld, B.W.p(), ld, 0.0, B.T2.p(), ld);
                sp_A_sampled(st, B.sp, B.W.p(), ld, B.T2.p(), ld, 1.0, h->rhs.p);
            } else {
                gemm_nn(st, m, m, m, 1.0, B.W.p(), ld, B.T1.p(), ld, 0.0, B.T2.p(), ld);
                gemm_sym(st, false, false, m, B.T2.p(), ld, B.W.p(), ld, B.T3.p(), ld);
                sp_A_vec(st, B.sp, B.T3.p(), ld, 1.0, h->rhs.p);
            }
        }
        add_lp_rhs(h, 0, 0.0);
        return LRN_OK;
    });
}

int32_t lrn_rhs_corrector(lrn_handle_t h, double sigma, double mu) {
    LRN_GROUP(h, lrn_rhs_corrector(m_, sigma, mu));
    return guarded(h, [&]() -> int32_t {
        for (auto& Bk : h->blk) Bk.ud_valid = false;
        Phase ph(h, LRN_T_RHS);
        cudaStream_t st = h->st;
        const double sm = sigma * mu;
        LRN_CUDA(cudaMemcpyAsync(h->rhs.p, h->Rp.p, h->n_var * sizeof(double), cudaMemcpyDeviceToDevice, st));
        for (auto& B : h->blk) {
            const int m = B.m, ld = B.ld;
            // h += AA * vec(G (G' Rd G + diag(D) - diag(sigma mu ./ D) - RNT) G')      (src/predictor_corrector.jl:186)
            if (use_rdb(B)) {
                ensure_rdb(h, B, st);
                LRN_CUDA(cudaMemcpyAsync(B.T2.p(), B.RdB.p(), B.RdB.bytes(), cudaMemcpyDeviceToDevice, st));
            } else {
                gemm_nn(st, m, m, m, 1.0, B.Rd.p(), ld, B.G.p(), ld, 0.0, B.T1.p(), ld);
                gemm_sym(st, true, false, m, B.G.p(), ld, B.T1.p(), ld, B.T2.p(), ld);
            }
            mat_corr_inner(st, m, B.T2.p(), ld, B.D.p, sm, B.RNT.p(), ld);
            if ((double)B.sp.nnz <= 0.05 * (double)m * m) {
                // sparse data: (G K G')(p,q) = <(K G')(:,p), G'(:,q)> (K symmetric) is only needed at the stored positions:
                // one product K G', an explicit G' (T4 is free here) and one m-long inner product per stored entry
                gemm_nt(st, m, m, m, 1.0, B.T2.p(), ld, B.G.p(), ld, 0.0, B.T1.p(), ld);
                mat_transpose(st, m, B.T4.p(), ld, B.G.p(), ld);
                sp_A_sampled(st, B.sp, B.T1.p(), ld, B.T4.p(), ld, 1.0, h->rhs.p);
            } else {
                gemm_nn(st, m, m, m, 1.0, B.G.p(), ld, B.T2.p(), ld, 0.0, B.T1.p(), ld);
                gemm_sym(st, false, true, m, B.T1.p(), ld, B.G.p(), ld, B.T3.p(), ld);
                sp_A_vec(st, B.sp, B.T3.p(), ld, 1.0, h->rhs.p);
            }
        }
        add_lp_rhs(h, 1, sm);
        return LRN_OK;
    });
}

int32_t lrn_schur_factor(lrn_handle_t h) {
    LRN_GROUP(h, lrn_schur_factor(m_));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(h->H.p(), "Schur matrix is only allocated for kit = 0");
        int info = 0;
        {
            Phase ph(h, LRN_T_FACTOR);
            cudaStream_t st = h->st;
            LRN_CUDA(cudaMemcpyAsync(h->L.p(), h->H.p(), h->H.bytes(), cudaMemcpyDeviceToDevice, st));
            LRN_REQUIRE(h->world <= 1 || (h->nccl && static_cast<DistCtx*>(h->nccl)->comm),
                        "the Schur rows are sharded but the handle has no NCCL communicator (lrn_dist_init / lrn_create_multi)");
            if (h->nccl && static_cast<DistCtx*>(h->nccl)->comm)
                cholesky_dist(h->L.p(), h->n_var, h->L.ld, h->cholH, *static_cast<DistCtx*>(h->nccl), h->dist_pw, st);
            else {
                h->cholH.int8 = h->chol_int8;
                cholesky_lower(h->L.p(), h->n_var, h->L.ld, h->cholH, st);
            }
            LRN_CUDA(cudaMemcpyAsync(&info, h->cholH.info_ptr(), sizeof(int), cudaMemcpyDeviceToHost, st));
            LRN_CUDA(cudaStreamSynchronize(st));
        }
        LRN_REQUIRE(info >= 0, "distributed factorisation: a peer did not deliver its part of a panel in time (peer-memory exchange)");
        h->have_factor = (info == 0);
        return info;
    });
}

int32_t lrn_schur_shift(lrn_handle_t h, double delta) {
    LRN_GROUP(h, lrn_schur_shift(m_, delta));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(h->H.p(), "Schur matrix is only allocated for kit = 0");
        if (h->world > 1 && !h->H_gathered) {
            // sharded rows: every rank shifts the diagonal entries of its own row blocks only
            const int pw = h->dist_pw, n = h->n_var;
            for (int g = h->rank; g * pw < n; g += h->world) {
                const int r0 = g * pw, rb = std::min(pw, n - r0);
                mat_add_diag(h->st, rb, h->H.p() + (size_t)r0 * h->H.ld + r0, h->H.ld, delta);
            }
        } else {
            mat_add_diag(h->st, h->n_var, h->H.p(), h->H.ld, delta);
        }
        h->have_factor = false;
        return LRN_OK;
    });
}

int32_t lrn_schur_solve(lrn_handle_t h, int32_t which) {
    LRN_GROUP(h, lrn_schur_solve(m_, which));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(h->have_factor, "no valid Cholesky factor (call lrn_schur_factor)");
        LRN_REQUIRE(which == 1 || which == 2 || which == 3 || which == 6, "which must be 1, 2, 3 or 6");
        Phase ph(h, LRN_T_SOLVE);
        cudaStream_t st = h->st;
        LRN_CUDA(cudaMemcpyAsync(h->dely.p, h->rhs.p, h->n_var * sizeof(double), cudaMemcpyDeviceToDevice, st));
        const int reps = (which == 6) ? 2 : 1;
        const int w = (which == 6) ? 3 : which;
        for (int r = 0; r < reps; r++) chol_solve(h->L.p(), h->n_var, h->L.ld, h->cholH, h->dely.p, h->tn1.p, w, st);
        return LRN_OK;
    });
}

int32_t lrn_find_step(lrn_handle_t h, int32_t predict, double sigma, double mu, double tau, double* alpha, double* beta,
                      double* alpha_lin, double* beta_lin) {
    if (h && h->group)
        return group_call(h, [&](lrn_solver* m_, int r_) -> int32_t {
            if (r_ == 0) return lrn_find_step(m_, predict, sigma, mu, tau, alpha, beta, alpha_lin, beta_lin);
            GroupScratch& g = group_scratch();
            g.a.assign(std::max(1, m_->nlmi), 0.0);
            g.b.assign(std::max(1, m_->nlmi), 0.0);
            return lrn_find_step(m_, predict, sigma, mu, tau, g.a.data(), g.b.data(), g.d, g.d + 1);
        });
    return guarded(h, [&]() -> int32_t {
        for (auto& Bk : h->blk) Bk.ud_valid = false;
        LRN_REQUIRE((h->nlmi == 0 || (alpha && beta)) && alpha_lin && beta_lin, "null outputs");
        Phase ph(h, LRN_T_FIND_STEP);
        cudaStream_t st = h->st;
        const double sm = sigma * mu;
        // multi-block problems whose blocks all go to the batched lambda_min kernel have no host synchronisation inside the
        // loop: the independent per-block chains of small kernels are spread over the side streams
        bool fan = h->nlmi >= 4 && h->eig_small.size() == (size_t)h->nlmi;
        if (fan) side_fork(h);
        cudaStream_t st_main = st;
        for (int i = 0; i < h->nlmi; i++) {
            Block& B = h->blk[i];
            const int m = B.m, ld = B.ld;
            cudaStream_t st = fan ? h->side[i % lrn_solver::NSIDE] : st_main;
            // delS = Rd - mat(AA' dely)                                        (src/predictor_corrector.jl:252)
            LRN_CUDA(cudaMemcpyAsync(B.dS.p(), B.Rd.p(), B.Rd.bytes(), cudaMemcpyDeviceToDevice, st));
            sp_scatter_ATy(st, B.sp, h->dely.p, -1.0, B.dS.p(), ld);
            // delSb = G' delS G                                                (:263)
            if (use_rdb(B)) {
                ensure_rdb(h, B, st);
                sp_pos_values(st, B.sp, h->dely.p);
                sp_M_times_W(st, B.sp, B.G.p(), ld, B.T1.p(), ld);                      // T1 = M G
                LRN_CUDA(cudaMemcpyAsync(B.T2.p(), B.RdB.p(), B.RdB.bytes(), cudaMemcpyDeviceToDevice, st));
                GemmParams p;                                                            // T2 = G'RdG - G'(M G), lower + mirror
                p.A = B.G.p(); p.B = B.T1.p(); p.C = B.T2.p(); p.M = m; p.N = m; p.K = m; p.lda = ld; p.ldb = ld; p.ldc = ld;
                p.transA = true; p.alpha = -1.0; p.beta = 1.0; p.lower = 1;
                gemm(p, st);
                mat_mirror_lower(st, m, B.T2.p(), ld);
            } else {
                gemm_nn(st, m, m, m, 1.0, B.dS.p(), ld, B.G.p(), ld, 0.0, B.T1.p(), ld);
                gemm_sym(st, true, false, m, B.G.p(), ld, B.T1.p(), ld, B.T2.p(), ld);
            }
            // delX = mat(-X - W delS W)                         (predictor, :255)
            //      = mat(sigma mu Si - X - W delS W + G RNT G') (corrector, :257)
            // with W = G G' both congruences collapse into ONE:  delX = mat([sigma mu Si] - X + G (RNT - delSb) G')
            if (predict) mat_lincomb(st, m, m, B.T3.p(), ld, -1.0, B.T2.p(), ld, 0.0, nullptr, 0, 0.0, nullptr, 0);
            else mat_lincomb(st, m, m, B.T3.p(), ld, -1.0, B.T2.p(), ld, 1.0, B.RNT.p(), ld, 0.0, nullptr, 0);
            gemm_nn(st, m, m, m, 1.0, B.G.p(), ld, B.T3.p(), ld, 0.0, B.T1.p(), ld);
            gemm_sym(st, false, true, m, B.T1.p(), ld, B.G.p(), ld, B.T4.p(), ld);
            if (predict)
                mat_sym_lincomb(st, m, B.dX.p(), ld, -1.0, B.X.p(), ld, 1.0, B.T4.p(), ld, 0.0, nullptr, 0, 0.0, nullptr, 0);
            else
                mat_sym_lincomb(st, m, B.dX.p(), ld, sm, B.Si.p(), ld, -1.0, B.X.p(), ld, 1.0, B.T4.p(), ld, 0.0, nullptr, 0);
            // delXb = Gi delX Gi' (:264) in closed form (Gi X Gi' = D, Gi Si Gi' = D^-1, Gi W = G'):
            //   delXb = (RNT - delSb) - diag(D) [+ sigma mu diag(1/D)]       -> T3
            mat_add_diag_vec(st, m, B.T3.p(), ld, -1.0, predict ? 0.0 : sm, B.D.p);
            if (predict) {
                // RNT = -(Gi delX delS G + G' delS delX Gi') ./ (D_p + D_q) = -(P + P') ./ (...), P = delXb delSb   (:308-309)
                gemm_nn(st, m, m, m, 1.0, B.T3.p(), ld, B.T2.p(), ld, 0.0, B.T1.p(), ld);
                mat_rnt(st, m, B.RNT.p(), ld, B.T1.p(), ld, B.D.p);
            }
            // XXX = sym(DDsi' .* delXb .* DDsi), sym(DDsi' .* delSb .* DDsi) ; eigmin                   (:268-285)
            mat_scaled_sym(st, m, B.T4.p(), ld, B.T3.p(), ld, B.DDsi.p);
            mat_scaled_sym(st, m, B.T1.p(), ld, B.T2.p(), ld, B.DDsi.p);
            const bool batched = (m > 64 && m <= 384);
            if (!batched && predict) {
                // predictor: XXX_X = DDsi (-D - delSb) DDsi = -I - XXX_S  (diag(G'SG) = D), so eigmin(XXX_X) = -1 - eigmax(XXX_S):
                // one Lanczos run delivers both step lengths
                double lmax = 0.0;
                const double lmin = lambda_min(h, B.T1.p(), m, ld, &lmax);
                beta[i] = steplen(lmin, tau);
                alpha[i] = steplen(-1.0 - lmax, tau);
            } else if (!batched) {
                // corrector: the two smallest eigenvalues are independent Lanczos runs, each a chain of small latency-bound
                // kernels with host check points: the X part runs on a second stream driven by a second host thread
                double lx = 0.0, ls = 0.0;
                lambda_min_pair(h, B.T4.p(), B.T1.p(), m, ld, &lx, &ls);
                alpha[i] = steplen(lx, tau);
                beta[i] = steplen(ls, tau);
            }
        }
        if (fan) side_join(h);
        if (!h->eig_small.empty()) {
            Phase pe(h, LRN_T_EIGMIN);
            const int cnt = 2 * (int)h->eig_small.size();
            batched_lambda_min(h->eig_ptrs.p, h->eig_ms.p, h->eig_lds.p, cnt, h->eig_out.p, st);
            std::vector<double> lam(cnt);
            LRN_CUDA(cudaMemcpyAsync(lam.data(), h->eig_out.p, cnt * sizeof(double), cudaMemcpyDeviceToHost, st));
            LRN_CUDA(cudaStreamSynchronize(st));
            for (size_t t = 0; t < h->eig_small.size(); t++) {
                alpha[h->eig_small[t]] = steplen(lam[2 * t], tau);
                beta[h->eig_small[t]] = steplen(lam[2 * t + 1], tau);
            }
        }
        *alpha_lin = 1.0;
        *beta_lin = 1.0;
        if (h->nlin > 0) {
            // find_step_lin                                                    (:329-347)
            const int nl = h->nlin;
            lin_CT_y(st, h->lin, h->dely.p, -1.0, 1.0, h->rd_lin.p, h->ds_lin.p);
            k_lp_dx<<<nb(nl), TBK, 0, st>>>(nl, predict ? 0 : 1, sm, h->x_lin.p, h->si_lin.p, h->ds_lin.p, h->rnt_lin.p, h->dx_lin.p);
            h->red.min_ratio(st, nl, h->dx_lin.p, h->x_lin.p, 0, false);
            h->red.min_ratio(st, nl, h->ds_lin.p, h->s_lin.p, 1, false);
            const double* r = h->red.fetch(st);
            *alpha_lin = steplen(r[0], tau);
            *beta_lin = steplen(r[1], tau);
        }
        if (predict) {
            for (int i = 0; i < h->nlmi; i++) {
                Block& B = h->blk[i];
                const int m = B.m, ld = B.ld;
                // Xn, Sn, RNT                                                   (:306-309)
                mat_lincomb(st, m, m, B.Xn.p(), ld, 1.0, B.X.p(), ld, alpha[i], B.dX.p(), ld, 0.0, nullptr, 0);
                mat_lincomb(st, m, m, B.Sn.p(), ld, 1.0, B.S.p(), ld, beta[i], B.dS.p(), ld, 0.0, nullptr, 0);
            }
            if (h->nlin > 0)
                k_lp_pred_update<<<nb(h->nlin), TBK, 0, st>>>(h->nlin, *alpha_lin, *beta_lin, h->x_lin.p, h->s_lin.p, h->dx_lin.p,
                                                              h->ds_lin.p, h->si_lin.p, h->xn_lin.p, h->sn_lin.p, h->rnt_lin.p);
        } else {
            double amin = *alpha_lin, bmin = *beta_lin;
            for (int i = 0; i < h->nlmi; i++) { amin = std::min(amin, alpha[i]); bmin = std::min(bmin, beta[i]); }
            // y, X, S update                                                    (:313-321, :358-360)
            vec_axpby(st, h->n_var, h->y.p, 1.0, h->y.p, bmin, h->dely.p);
            for (auto& B : h->blk) {
                const int m = B.m, ld = B.ld;
                mat_lincomb(st, m, m, B.X.p(), ld, 1.0, B.X.p(), ld, amin, B.dX.p(), ld, 0.0, nullptr, 0);
                mat_symmetrize(st, m, B.X.p(), ld);
                mat_lincomb(st, m, m, B.S.p(), ld, 1.0, B.S.p(), ld, bmin, B.dS.p(), ld, 0.0, nullptr, 0);
                mat_symmetrize(st, m, B.S.p(), ld);
                B.chol_cached = false;
            }
            if (h->nlin > 0) {
                vec_axpby(st, h->nlin, h->x_lin.p, 1.0, h->x_lin.p, amin, h->dx_lin.p);
                vec_axpby(st, h->nlin, h->s_lin.p, 1.0, h->s_lin.p, bmin, h->ds_lin.p);
                // S_lin_inv is refreshed; Si_lin (same values) is refreshed by the next prepare_W like in the reference
                vec_op(st, h->nlin, VEC_RECIP, h->si_lin.p, h->s_lin.p, nullptr);
            }
        }
        LRN_CUDA(cudaStreamSynchronize(st));
        return LRN_OK;
    });
}

int32_t lrn_sigma_trace(lrn_handle_t h, double* tr, double* dl) {
    LRN_GROUP(h, lrn_sigma_trace(m_, r_ == 0 ? tr : group_scratch().d, r_ == 0 ? dl : group_scratch().d + 1));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(tr && dl, "null outputs");
        cudaStream_t st = h->st;
        h->red.zero(st);
        for (auto& B : h->blk) h->red.dot_mat(st, B.m, B.m, B.Xn.p(), B.ld, B.Sn.p(), B.ld, 0, true);
        if (h->nlin > 0) h->red.dot_vec(st, h->nlin, h->xn_lin.p, h->sn_lin.p, 1, false);
        const double* r = h->red.fetch(st);
        *tr = r[0];
        *dl = r[1];
        return LRN_OK;
    });
}

int32_t lrn_dimacs(lrn_handle_t h, double* err6, double* by_out, double* trCX_out, double* dx_out) {
    LRN_GROUP(h, r_ == 0 ? lrn_dimacs(m_, err6, by_out, trCX_out, dx_out)
                       : lrn_dimacs(m_, group_scratch().d, nullptr, nullptr, nullptr));
    return guarded(h, [&]() -> int32_t {
        for (auto& Bk : h->blk) Bk.ud_valid = false;
        LRN_REQUIRE(err6, "null output");
        Phase ph(h, LRN_T_DIMACS);
        cudaStream_t st = h->st;
        Reducer& R = h->red;
        R.zero(st);
        // slots: 0 Rp.Rp, 1 b.y, 2 min x_lin, 3 rd_lin.rd_lin, 4 min s_lin, 5 d.x, 6 s.x ; per block 16+4i: Rd.Rd, S.X, C.X
        R.dot_vec(st, h->n_var, h->Rp.p, h->Rp.p, 0, false);
        R.dot_vec(st, h->n_var, h->b.p, h->y.p, 1, false);
        for (int i = 0; i < h->nlmi; i++) {
            Block& B = h->blk[i];
            R.dot_mat(st, B.m, B.m, B.Rd.p(), B.ld, B.Rd.p(), B.ld, 16 + 4 * i, false);
            R.dot_mat(st, B.m, B.m, B.S.p(), B.ld, B.X.p(), B.ld, 16 + 4 * i + 1, false);
            R.dot_mat(st, B.m, B.m, B.C.p(), B.C.ld, B.X.p(), B.ld, 16 + 4 * i + 2, false);
        }
        {
            // eigmin(X), eigmin(S) only enter as max(0, -eigmin): a successful Cholesky proves eigmin > 0; the factors
            // are kept for the next prepare_W (X and S do not change in between).  The 2 nlmi factorisations are independent
            // and, for small blocks, latency-bound single-CTA-group kernels: multi-block problems spread them over side
            // streams (fork / join with events) so that they overlap.
            const bool fan = h->nlmi >= 4;
            if (fan && !h->side[0]) {
                for (auto& s_ : h->side) LRN_CUDA(cudaStreamCreateWithFlags(&s_, cudaStreamNonBlocking));
                LRN_CUDA(cudaEventCreateWithFlags(&h->evFork, cudaEventDisableTiming));
                for (auto& e : h->evJoin) LRN_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            }
            if (fan) {
                LRN_CUDA(cudaEventRecord(h->evFork, st));
                for (auto& s_ : h->side) LRN_CUDA(cudaStreamWaitEvent(s_, h->evFork, 0));
            }
            for (int i = 0; i < h->nlmi; i++) {
                Block& B = h->blk[i];
                cudaStream_t sx = fan ? h->side[(2 * i) % lrn_solver::NSIDE] : st;
                cudaStream_t ss = fan ? h->side[(2 * i + 1) % lrn_solver::NSIDE] : st;
                LRN_CUDA(cudaMemcpyAsync(B.LX.p(), B.X.p(), B.X.bytes(), cudaMemcpyDeviceToDevice, sx));
                cholesky_lower(B.LX.p(), B.m, B.ld, B.cholX, sx);
                LRN_CUDA(cudaMemcpyAsync(B.LS.p(), B.S.p(), B.S.bytes(), cudaMemcpyDeviceToDevice, ss));
                cholesky_lower(B.LS.p(), B.m, B.ld, B.cholS, ss);
            }
            if (fan)
                for (int k = 0; k < lrn_solver::NSIDE; k++) {
                    LRN_CUDA(cudaEventRecord(h->evJoin[k], h->side[k]));
                    LRN_CUDA(cudaStreamWaitEvent(st, h->evJoin[k], 0));
                }
        }
        if (h->nlin > 0) {
            R.min_ratio(st, h->nlin, h->x_lin.p, nullptr, 2, false);
            R.dot_vec(st, h->nlin, h->rd_lin.p, h->rd_lin.p, 3, false);
            R.min_ratio(st, h->nlin, h->s_lin.p, nullptr, 4, false);
            R.dot_vec(st, h->nlin, h->d_lin.p, h->x_lin.p, 5, false);
            R.dot_vec(st, h->nlin, h->s_lin.p, h->x_lin.p, 6, false);
        }
        std::vector<int> infos(2 * std::max(1, h->nlmi), 0);
        if (h->nlmi > 0)
            LRN_CUDA(cudaMemcpyAsync(infos.data(), h->blk_info.p, 2 * h->nlmi * sizeof(int), cudaMemcpyDeviceToHost, st));
        const double* r = R.fetch(st);
        std::vector<double> v(r, r + R.nslots);
        const double nb_ = h->normb, by = v[1];
        double e1 = std::sqrt(v[0]) / (1 + nb_), e2 = 0, e3 = 0, e4 = 0, e5 = 0, e6 = 0, trCX = 0;
        for (int i = 0; i < h->nlmi; i++) {
            Block& B = h->blk[i];
            const double CX = v[16 + 4 * i + 2];
            trCX += CX;
            double lx = 1.0, ls = 1.0;
            if (infos[2 * i] != 0) lx = lambda_min(h, B.X.p(), B.m, B.ld);
            if (infos[2 * i + 1] != 0) ls = lambda_min(h, B.S.p(), B.m, B.ld);
            B.chol_cached = (infos[2 * i] == 0 && infos[2 * i + 1] == 0);
            e2 += std::max(0.0, -lx / (1 + nb_));
            e3 += std::sqrt(v[16 + 4 * i]) / (1 + B.normC);
            e4 += std::max(0.0, -ls / (1 + B.normC));
            e6 += v[16 + 4 * i + 1] / (1 + std::fabs(CX) + std::fabs(by));
        }
        e5 = (trCX - by) / (1 + std::fabs(trCX) + std::fabs(by));
        double dx = 0.0;
        if (h->nlin > 0) {
            dx = v[5];
            e2 += std::max(0.0, -v[2] / (1 + nb_));
            e3 += std::sqrt(v[3]) / (1 + h->normd);
            e4 += std::max(0.0, -v[4] / (1 + h->normd));
            e5 = (trCX + dx - by) / (1 + std::fabs(trCX) + std::fabs(by));
            e6 += v[6] / (1 + std::fabs(dx) + std::fabs(by));
        }
        err6[0] = e1; err6[1] = e2; err6[2] = e3; err6[3] = e4; err6[4] = e5; err6[5] = e6;
        if (by_out) *by_out = by;
        if (trCX_out) *trCX_out = trCX;
        if (dx_out) *dx_out = dx;
        return LRN_OK;
    });
}

// ---- parity hooks -------------------------------------------------------------------------------------------------------
int32_t lrn_get_array(lrn_handle_t h, int32_t which, int64_t iblk, double* out) {
    // Schur matrix: a collective (every member contributes its row blocks); everything else is replicated -> member 0
    if (h && h->group && which != LRN_ARR_H) return lrn_get_array(static_cast<Group*>(h->group)->members[0], which, iblk, out);
    LRN_GROUP(h, lrn_get_array(m_, which, iblk, r_ == 0 ? out : nullptr));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(out || which == LRN_ARR_H, "null output");
        cudaStream_t st = h->st;
        const int n = h->n_var;
        auto vec_out = [&](const double* p, int len) {
            LRN_CUDA(cudaMemcpyAsync(out, p, (size_t)len * sizeof(double), cudaMemcpyDeviceToHost, st));
        };
        if (which == LRN_ARR_H || which == LRN_ARR_L) {
            LRN_REQUIRE(h->H.p(), "Schur matrix is only allocated for kit = 0");
            DMat& M = (which == LRN_ARR_H) ? h->H : h->L;
            // work on a copy in tn-sized chunks is not possible: use the spare matrix of the other kind only when safe
            if (which == LRN_ARR_H && h->world > 1 && h->nccl && static_cast<DistCtx*>(h->nccl)->comm && !h->H_gathered) {
                // every rank holds only its own row blocks: sum them up (once per assembly)
                dist_allreduce_sum(M.p(), (size_t)M.ld * n, *static_cast<DistCtx*>(h->nccl), st);
                h->H_gathered = true;
            }
            if (which == LRN_ARR_H) mat_mirror_lower(st, n, M.p(), M.ld);
            else zero_strict_upper(M.p(), n, M.ld, st);
            if (out) download_dense(h, M.p(), M.ld, n, n, out);
        } else if (which == LRN_ARR_RHS) vec_out(h->rhs.p, n);
        else if (which == LRN_ARR_DELY) vec_out(h->dely.p, n);
        else if (which == LRN_ARR_RP) vec_out(h->Rp.p, n);
        else {
            LRN_REQUIRE(iblk >= 0 && iblk < h->nlmi, "bad block index");
            Block& B = h->blk[iblk];
            const DMat* M = nullptr;
            switch (which) {
                case LRN_ARR_W: M = &B.W; break;
                case LRN_ARR_G: M = &B.G; break;
                case LRN_ARR_GI: {
                    // Gi = D^{-1/2} U' L_S' = (L_S (U D) D^{-3/2})'  -- valid until the next prepare_W / find_step scratch reuse
                    LRN_REQUIRE(B.ud_valid, "Gi is only available right after lrn_prepare_W (before any other hot-path call)");
                    GemmParams p;
                    p.A = B.LS.p(); p.B = B.T2.p(); p.C = B.T1.p(); p.M = B.m; p.N = B.m; p.K = B.m;
                    p.lda = B.ld; p.ldb = B.ld; p.ldc = B.ld; p.colscale = B.dm32.p;
                    gemm(p, st);
                    mat_transpose(st, B.m, B.Gi.p(), B.ld, B.T1.p(), B.ld);
                    M = &B.Gi;
                    break;
                }
                case LRN_ARR_SI: M = &B.Si; break;
                case LRN_ARR_RD: M = &B.Rd; break;
                case LRN_ARR_DELX: M = &B.dX; break;
                case LRN_ARR_DELS: M = &B.dS; break;
                case LRN_ARR_RNT: M = &B.RNT; break;
                case LRN_ARR_XN: M = &B.Xn; break;
                case LRN_ARR_SN: M = &B.Sn; break;
                case LRN_ARR_D: vec_out(B.D.p, B.m); break;
                case LRN_ARR_DDSI: vec_out(B.DDsi.p, B.m); break;
                default: LRN_REQUIRE(false, "unknown array id");
            }
            if (M) download_dense(h, M->p(), M->ld, B.m, B.m, out);
        }
        LRN_CUDA(cudaStreamSynchronize(st));
        return LRN_OK;
    });
}

int32_t lrn_timers(lrn_handle_t h, double* ms, int64_t* calls, int32_t reset) {
    if (h && h->group) return lrn_timers(static_cast<Group*>(h->group)->members[0], ms, calls, reset);
    return guarded(h, [&]() -> int32_t {
        flush_timers(h);
        for (int i = 0; i < LRN_T_COUNT; i++) {
            if (ms) ms[i] = h->t_ms[i];
            if (calls) calls[i] = h->t_calls[i];
            if (reset) { h->t_ms[i] = 0; h->t_calls[i] = 0; }
        }
        return LRN_OK;
    });
}

const char* lrn_timer_name(int32_t phase, int32_t rank1) {
    static const char* names[LRN_T_COUNT] = {"prep W", "residuals", "BBBBs", "RHS", "cholesky", "solve", "find_step", "prec",
                                             "CG", "check_convergence", "prep W SVD", "eigmin"};
    if (phase < 0 || phase >= LRN_T_COUNT) return nullptr;
    if (phase == LRN_T_ASSEMBLE && rank1) return "BBBB_rank1";
    return names[phase];
}

int32_t lrn_set_option(lrn_handle_t h, const char* name, double value) {
    LRN_GROUP(h, lrn_set_option(m_, name, value));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(name, "null name");
        std::string n(name);
        if (n == "aamat") h->opt.aamat = (int)value;
        else if (n == "erank") { LRN_REQUIRE(h->prec_ready == 0, "erank cannot change after a preconditioner was built"); h->opt.erank = (int)value; }
        else if (n == "svd_tol") h->opt.svd_tol = value;
        else if (n == "lanczos_tol") h->opt.lanczos_tol = value;
        else if (n == "lanczos_kmax") h->lanczos_kmax = std::max(4, (int)value);   // test hook: forces the bisection fallback
        else if (n == "chol_int8") h->chol_int8 = value != 0 ? 1 : 0;
        else if (n == "pair_kernel") h->use_staged_pairs = (int)value;   // 0: gather kernel (one thread per pair), 1: staged kernel, -1: auto
        else if (n == "sparse_op") {
            // 0: dense W M W operator, 1: sparse-aware operator wherever the data allows it, -1: automatic (density rule)
            for (auto& B : h->blk) {
                if (value > 0) B.sp.sparse_op = B.sp.sparse_ok;
                else if (value == 0) B.sp.sparse_op = false;
                else B.sp.sparse_op = B.sp.sparse_ok && (double)B.sp.npos <= 0.05 * (double)B.m * B.m;
            }
        }
        else LRN_REQUIRE(false, "unknown option name");
        return LRN_OK;
    });
}

int64_t lrn_kernel_launches(void) { return (int64_t)lrn::g_kernel_launches.load(); }

int32_t lrn_stats(lrn_handle_t h, int64_t* out3) {
    if (h && h->group) return lrn_stats(static_cast<Group*>(h->group)->members[0], out3);
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(out3, "null output");
        out3[0] = h->stat_svd_sweeps; out3[1] = h->stat_lanczos_iters; out3[2] = h->stat_lanczos_fail;
        // (the number of Cholesky bisection steps taken after non-converged Lanczos runs is folded into the failure count's
        // companion counter: see lrn_set_option("lanczos_kmax"))
        return LRN_OK;
    });
}

}  // extern "C"

// The CG / preconditioner entry points live in pcg.cu; they use apply_A through this hook.
namespace lrn {
void solver_apply_A(lrn_solver* h, const double* x, double* out) { apply_A(h, x, out); }
void solver_flush_timers(lrn_solver* h) { flush_timers(h); }
}  // namespace lrn
