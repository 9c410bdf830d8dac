// Model preparation behind the ABI (SURVEY 8(f) rows N1-N3): what MOI.copy_to + _prepare_A do on the Julia host
// (src/MOI_wrapper.jl:152-223, src/model.jl:120-229) and what examples/solve_sdpa.jl:14-34 does through MOI.FileFormats.SDPA,
// as one bulk pass over the triplets in C++:
//   * lrn_create_from_triplets : (k, block, i, j, v) triplets in SDPA convention -> per-block AA_i (n_var x m_i^2, math sign,
//     both triangles), C_i, rank-one factors B_i (datarank = -1, prep_B src/model.jl:176-197), C_lin / d_lin, b; then the same
//     device build as lrn_set_block_* + lrn_finalize (by-constraint CSR, by-position CSC, sigmaA order, F1/F3 split =
//     prep_sparse! src/model.jl:153-174).  No per-nonzero push!, no O(n_var) dense eigen calls on m x m matrices: the rank-one
//     test of a matrix works on its |idx| x |idx| nonzero sub-block only.
//   * lrn_load_sdpa            : .dat-s reader in front of it.
//   * lrn_initial_point        : src/initial_point.jl:17-81 from the norms kept at build time (a C / C++ host needs no model copy).
// SDPA problem:  min c'y  s.t.  sum_k F_k y_k - F_0 >= 0   ->   b = -c, C_i = -F_0, calA_k = -F_k, C_lin = -coeff', d_lin = -F_0[r,r]
// (src/MOI_wrapper.jl:186-217, src/model.jl:133).
#include "group.cuh"
#include <algorithm>
#include <cmath>
#include <fstream>
#include <sstream>

using namespace lrn;

namespace {

struct HostModel {
    int64_t n = 0;
    std::vector<int64_t> msizes;               // PSD blocks only
    std::vector<HostCSC> AA, Cm, Bm;           // 0-based CSC (AA: n x m^2 columns p + q m; C: m x m; B: n x m)
    HostCSC Clin;
    std::vector<double> d_lin, b;
    int64_t nlin = 0;
    bool rank1 = false;
};

// CSC from unsorted (row, col, val) triplets; duplicates are summed
void csc_from_triplets(HostCSC& M, int64_t ncol, std::vector<int64_t>& r, std::vector<int64_t>& c, std::vector<double>& v) {
    const size_t nz = r.size();
    std::vector<size_t> order(nz);
    for (size_t t = 0; t < nz; t++) order[t] = t;
    std::sort(order.begin(), order.end(), [&](size_t a, size_t b2) { return c[a] != c[b2] ? c[a] < c[b2] : r[a] < r[b2]; });
    M.colptr.assign(ncol + 1, 0);
    M.rowval.clear(); M.nzval.clear();
    M.rowval.reserve(nz); M.nzval.reserve(nz);
    std::vector<int64_t> colof;
    colof.reserve(nz);
    for (size_t t = 0; t < nz; t++) {
        const size_t e = order[t];
        if (!M.rowval.empty() && colof.back() == c[e] && M.rowval.back() == r[e]) { M.nzval.back() += v[e]; continue; }
        M.rowval.push_back(r[e]); M.nzval.push_back(v[e]); colof.push_back(c[e]);
    }
    for (int64_t cc : colof) M.colptr[cc + 1]++;
    for (int64_t cc = 0; cc < ncol; cc++) M.colptr[cc + 1] += M.colptr[cc];
    M.set = true;
}

// largest eigenpair of a small dense symmetric matrix (cyclic Jacobi); returns the eigenvector in `vec`
void top_eigvec(std::vector<double> A, int s, std::vector<double>& vec) {
    std::vector<double> V((size_t)s * s, 0.0);
    for (int i = 0; i < s; i++) V[(size_t)i * s + i] = 1.0;
    for (int sweep = 0; sweep < 60; sweep++) {
        double off = 0.0;
        for (int p = 0; p < s; p++) for (int q = p + 1; q < s; q++) off += A[(size_t)p * s + q] * A[(size_t)p * s + q];
        if (off < 1e-300) break;
        for (int p = 0; p < s; p++)
            for (int q = p + 1; q < s; q++) {
                const double apq = A[(size_t)p * s + q];
                if (std::fabs(apq) < 1e-300) continue;
                const double theta = (A[(size_t)q * s + q] - A[(size_t)p * s + p]) / (2.0 * apq);
                const double t = (theta >= 0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
                const double cs = 1.0 / std::sqrt(t * t + 1.0), sn = t * cs;
                for (int k = 0; k < s; k++) {
                    const double akp = A[(size_t)k * s + p], akq = A[(size_t)k * s + q];
                    A[(size_t)k * s + p] = cs * akp - sn * akq; A[(size_t)k * s + q] = sn * akp + cs * akq;
                }
                for (int k = 0; k < s; k++) {
                    const double apk = A[(size_t)p * s + k], aqk = A[(size_t)q * s + k];
                    A[(size_t)p * s + k] = cs * apk - sn * aqk; A[(size_t)q * s + k] = sn * apk + cs * aqk;
                }
                for (int k = 0; k < s; k++) {
                    const double vkp = V[(size_t)k * s + p], vkq = V[(size_t)k * s + q];
                    V[(size_t)k * s + p] = cs * vkp - sn * vkq; V[(size_t)k * s + q] = sn * vkp + cs * vkq;
                }
            }
    }
    int best = 0;
    for (int i = 1; i < s; i++) if (A[(size_t)i * s + i] > A[(size_t)best * s + best]) best = i;
    vec.resize(s);
    for (int k = 0; k < s; k++) vec[k] = V[(size_t)k * s + best];
}

// triplets (SDPA convention, 1-based block / i / j, one triangle stored) -> HostModel
void build_model(HostModel& M, int64_t n, int64_t nblocks, const int64_t* bs, int64_t nt, const int64_t* tk, const int64_t* tb,
                 const int64_t* ti, const int64_t* tj, const double* tv, const double* c, int datarank) {
    LRN_REQUIRE(n >= 1 && nblocks >= 1 && bs && c, "bad problem header");
    LRN_REQUIRE(nt == 0 || (tk && tb && ti && tj && tv), "null triplet arrays");
    M.n = n;
    std::vector<int> psd_of(nblocks, -1);
    std::vector<int64_t> lin_off(nblocks, -1);
    for (int64_t bl = 0; bl < nblocks; bl++) {
        if (bs[bl] > 0) { psd_of[bl] = (int)M.msizes.size(); M.msizes.push_back(bs[bl]); }
        else if (bs[bl] < 0) { lin_off[bl] = M.nlin; M.nlin += -bs[bl]; }
    }
    const int nlmi = (int)M.msizes.size();
    M.AA.resize(nlmi); M.Cm.resize(nlmi); M.Bm.resize(nlmi);
    struct Trip { std::vector<int64_t> r, c; std::vector<double> v; };
    std::vector<Trip> aa(nlmi), cc(nlmi);
    Trip lin;
    M.d_lin.assign(M.nlin, 0.0);
    for (int64_t t = 0; t < nt; t++) {
        const int64_t k = tk[t], bl = tb[t] - 1, i = ti[t] - 1, j = tj[t] - 1;
        LRN_REQUIRE(bl >= 0 && bl < nblocks && k >= 0 && k <= n, "triplet block / constraint index out of range");
        if (psd_of[bl] >= 0) {
            const int ib = psd_of[bl];
            const int64_t m = M.msizes[ib];
            LRN_REQUIRE(i >= 0 && i < m && j >= 0 && j < m, "triplet position out of range");
            Trip& T = (k == 0) ? cc[ib] : aa[ib];
            // both triangles are stored (src/MOI_wrapper.jl:186-196); math sign calA = -F_k, C = -F_0
            for (int rep = 0; rep < (i == j ? 1 : 2); rep++) {
                const int64_t p = rep ? j : i, q = rep ? i : j;
                if (k == 0) { T.r.push_back(p); T.c.push_back(q); }
                else { T.r.push_back(k - 1); T.c.push_back(p + q * m); }
                T.v.push_back(-tv[t]);
            }
        } else if (lin_off[bl] >= 0) {
            LRN_REQUIRE(i == j && i >= 0 && i < -bs[bl], "off-diagonal entry in a diagonal SDPA block");
            const int64_t r = lin_off[bl] + i;
            if (k == 0) M.d_lin[r] += -tv[t];
            else { lin.r.push_back(k - 1); lin.c.push_back(r); lin.v.push_back(-tv[t]); }
        }
    }
    for (int ib = 0; ib < nlmi; ib++) {
        const int64_t m = M.msizes[ib];
        csc_from_triplets(M.AA[ib], m * m, aa[ib].r, aa[ib].c, aa[ib].v);
        csc_from_triplets(M.Cm[ib], m, cc[ib].r, cc[ib].c, cc[ib].v);
    }
    if (M.nlin > 0) csc_from_triplets(M.Clin, M.nlin, lin.r, lin.c, lin.v);
    M.b.resize(n);
    for (int64_t j = 0; j < n; j++) M.b[j] = -c[j];
    // ---- rank-one factors (prep_B, src/model.jl:176-197): A[i,k+1] = F_k = b_k b_k' on its nonzero sub-block ------------------
    if (datarank == -1) {
        M.rank1 = true;
        for (int ib = 0; ib < nlmi && M.rank1; ib++) {
            const int64_t m = M.msizes[ib];
            const HostCSC& A = M.AA[ib];
            // by-constraint lists of (p, q, F value = -calA value)
            std::vector<int64_t> cnt(n + 1, 0);
            for (int64_t r : A.rowval) cnt[r + 1]++;
            for (int64_t j = 0; j < n; j++) cnt[j + 1] += cnt[j];
            std::vector<int64_t> fill(cnt.begin(), cnt.end() - 1), ep(A.rowval.size()), eq(A.rowval.size());
            std::vector<double> ev(A.rowval.size());
            for (int64_t col = 0; col < m * m; col++)
                for (int64_t e = A.colptr[col]; e < A.colptr[col + 1]; e++) {
                    const int64_t d = fill[A.rowval[e]]++;
                    ep[d] = col % m; eq[d] = col / m; ev[d] = -A.nzval[e];
                }
            std::vector<int64_t> br, bc;
            std::vector<double> bv;
            for (int64_t k = 0; k < n; k++) {
                const int64_t e0 = cnt[k], e1 = cnt[k + 1];
                if (e0 == e1) continue;
                std::vector<int64_t> idx(ep.begin() + e0, ep.begin() + e1);
                std::sort(idx.begin(), idx.end());
                idx.erase(std::unique(idx.begin(), idx.end()), idx.end());
                const int s = (int)idx.size();
                std::vector<double> T((size_t)s * s, 0.0);
                for (int64_t e = e0; e < e1; e++) {
                    const auto ip = std::lower_bound(idx.begin(), idx.end(), ep[e]) - idx.begin();
                    const auto iq = std::lower_bound(idx.begin(), idx.end(), eq[e]);
                    if (iq == idx.end() || *iq != eq[e]) continue;
                    T[(size_t)ip * s + (iq - idx.begin())] += ev[e];
                }
                std::vector<double> sym((size_t)s * s), vec;
                for (int a = 0; a < s; a++) for (int b2 = 0; b2 < s; b2++) sym[(size_t)a * s + b2] = 0.5 * (T[(size_t)a * s + b2] + T[(size_t)b2 * s + a]);
                top_eigvec(sym, s, vec);
                double err = 0.0;
                std::vector<double> bbb(s);
                bool ok = true;
                for (int a = 0; a < s; a++) {
                    const double d = T[(size_t)a * s + a];
                    if (d < 0) ok = false;
                    bbb[a] = (vec[a] > 0 ? 1.0 : (vec[a] < 0 ? -1.0 : 0.0)) * std::sqrt(std::fabs(d));
                }
                for (int a = 0; a < s; a++) for (int b2 = 0; b2 < s; b2++) {
                    const double d = T[(size_t)a * s + b2] - bbb[a] * bbb[b2];
                    err += d * d;
                }
                if (!ok || !(std::sqrt(err) <= 5.0e-6))
                    throw std::invalid_argument("a constraint matrix is not rank one within 5e-6; use datarank = 0 to disable the rank-1 conversion");
                for (int a = 0; a < s; a++) { br.push_back(k); bc.push_back(idx[a]); bv.push_back(bbb[a]); }
            }
            csc_from_triplets(M.Bm[ib], m, br, bc, bv);
        }
    }
}

// Frobenius norms / row norms that initial_point needs (src/initial_point.jl:28-71)
void stage_on(lrn_solver* h, const HostModel& M) {
    LRN_REQUIRE(!h->finalized, "already finalized");
    for (size_t ib = 0; ib < M.msizes.size(); ib++) {
        h->blk[ib].hAA = M.AA[ib];
        h->blk[ib].hC = M.Cm[ib];
        if (M.rank1) h->blk[ib].hB = M.Bm[ib];
    }
    if (M.nlin > 0) {
        h->hClin = M.Clin;
        h->d_lin.upload(M.d_lin.data(), M.nlin, h->st);
        double s = 0;
        for (double d : M.d_lin) s += d * d;
        h->normd = std::sqrt(s);
    }
    h->b.upload(M.b.data(), M.n, h->st);
    h->hb = M.b;
    double s = 0;
    for (double v : M.b) s += v * v;
    h->normb = std::sqrt(s);
    LRN_CUDA(cudaStreamSynchronize(h->st));
}

}  // namespace

namespace lrn {
// norms of the model data for lrn_initial_point; called by lrn_finalize while the host copies still exist
void record_model_norms(lrn_solver* h, const std::vector<double>& b_host) {
    h->ip_normAA.assign(h->nlmi, 0.0);
    for (int i = 0; i < h->nlmi; i++) {
        double s = 0;
        for (double v : h->blk[i].hAA.nzval) s += v * v;
        h->ip_normAA[i] = std::sqrt(s);
    }
    double s2 = 0;
    for (double v : b_host) s2 += (1 + std::fabs(v)) * (1 + std::fabs(v));
    h->ip_normb2 = std::sqrt(s2);
    h->ip_pmax = 0.0; h->ip_rownmax = 0.0;
    if (h->nlin > 0 && h->hClin.set) {
        std::vector<double> rown(h->n_var, 0.0);
        for (size_t e = 0; e < h->hClin.rowval.size(); e++) rown[h->hClin.rowval[e]] += h->hClin.nzval[e] * h->hClin.nzval[e];
        for (int j = 0; j < h->n_var; j++) {
            const double rn = std::sqrt(rown[j]);
            h->ip_rownmax = std::max(h->ip_rownmax, rn);
            h->ip_pmax = std::max(h->ip_pmax, (1 + std::fabs(b_host[j])) / (1 + rn));
        }
    }
    h->ip_ready = true;
}
}  // namespace lrn

extern "C" {

int32_t lrn_create_from_triplets(lrn_handle_t* out, int64_t n_var, int64_t nblocks, const int64_t* blocksizes, int64_t ntrip,
                                 const int64_t* tk, const int64_t* tblk, const int64_t* ti, const int64_t* tj, const double* tv,
                                 const double* c, const lrn_options_t* opt, int32_t ngpus) {
    if (!out) return LRN_ERR_ARG;
    *out = nullptr;
    HostModel M;
    lrn_options_t o;
    if (opt) o = *opt; else lrn_default_options(&o);
    try {
        build_model(M, n_var, nblocks, blocksizes, ntrip, tk, tblk, ti, tj, tv, c, o.datarank);
    } catch (const std::exception& e) {
        fprintf(stderr, "lrn_create_from_triplets: %s\n", e.what());
        return LRN_ERR_ARG;
    }
    lrn_handle_t h = nullptr;
    const int nlmi = (int)M.msizes.size();
    int32_t rc = (ngpus == 1) ? lrn_create(&h, M.n, nlmi, nlmi ? M.msizes.data() : nullptr, M.nlin, &o)
                              : lrn_create_multi(&h, M.n, nlmi, nlmi ? M.msizes.data() : nullptr, M.nlin, &o, ngpus, nullptr);
    *out = h;
    if (rc != LRN_OK) return rc;
    auto stage = [&](lrn_solver* m) -> int32_t {
        try {
            LRN_CUDA(cudaSetDevice(m->device));
            stage_on(m, M);
            return LRN_OK;
        } catch (const std::exception& e) {
            m->err = e.what();
            return LRN_ERR_CUDA;
        }
    };
    if (h->group) rc = group_call(h, [&](lrn_solver* m, int) -> int32_t { return stage(m); });
    else rc = stage(h);
    if (rc != LRN_OK) return rc;
    return lrn_finalize(h);
}

int32_t lrn_load_sdpa(lrn_handle_t* out, const char* path, const lrn_options_t* opt, int32_t ngpus) {
    if (!out || !path) return LRN_ERR_ARG;
    *out = nullptr;
    std::ifstream f(path);
    if (!f) { fprintf(stderr, "lrn_load_sdpa: cannot open %s\n", path); return LRN_ERR_ARG; }
    auto clean = [](std::string s) {
        for (char& ch : s) {
            if (ch == '{' || ch == '}' || ch == '(' || ch == ')' || ch == ',') ch = ' ';
            if (ch == 'D' || ch == 'd') ch = 'e';
        }
        return s;
    };
    std::vector<std::string> lines;
    std::string ln;
    while (std::getline(f, ln)) {
        size_t a = ln.find_first_not_of(" \t\r");
        if (a == std::string::npos) continue;
        if (ln[a] == '"' || ln[a] == '*') continue;
        lines.push_back(clean(ln.substr(a)));
    }
    size_t li = 0;
    auto next_numbers = [&](std::vector<double>& dst, size_t want) {
        while (dst.size() < want && li < lines.size()) {
            std::istringstream ss(lines[li++]);
            double v;
            while (ss >> v) dst.push_back(v);
        }
    };
    std::vector<double> head, bsd, cv;
    if (lines.size() < 4) return LRN_ERR_ARG;
    { std::istringstream ss(lines[li++]); double v; ss >> v; head.push_back(v); }
    { std::istringstream ss(lines[li++]); double v; ss >> v; head.push_back(v); }
    const int64_t n = (int64_t)head[0], nblocks = (int64_t)head[1];
    if (n < 1 || nblocks < 1) return LRN_ERR_ARG;
    next_numbers(bsd, (size_t)nblocks);
    next_numbers(cv, (size_t)n);
    if (bsd.size() < (size_t)nblocks || cv.size() < (size_t)n) return LRN_ERR_ARG;
    std::vector<int64_t> bs(nblocks), tk, tb, ti, tj;
    for (int64_t b2 = 0; b2 < nblocks; b2++) bs[b2] = (int64_t)bsd[b2];
    cv.resize(n);
    std::vector<double> tv;
    for (; li < lines.size(); li++) {
        std::istringstream ss(lines[li]);
        double a[5];
        int got = 0;
        while (got < 5 && (ss >> a[got])) got++;
        if (got < 5) continue;
        tk.push_back((int64_t)a[0]); tb.push_back((int64_t)a[1]); ti.push_back((int64_t)a[2]); tj.push_back((int64_t)a[3]);
        tv.push_back(a[4]);
    }
    return lrn_create_from_triplets(out, n, nblocks, bs.data(), (int64_t)tv.size(), tk.data(), tb.data(), ti.data(), tj.data(),
                                    tv.data(), cv.data(), opt, ngpus);
}

// test hook (no device needed): run the host-side model preparation and hand one prepared matrix back as 0-based CSC.
// which: 0 = AA_iblk (n x m^2), 1 = C_iblk (m x m), 2 = B_iblk (n x m, datarank = -1), 3 = C_lin (n x nlin); vec_out (optional)
// receives b (which 0..2) or d_lin (which 3).  Returns the number of stored entries, or < 0 (also when cap is too small).
int64_t lrn_dbg_model_block(int64_t n_var, int64_t nblocks, const int64_t* blocksizes, int64_t ntrip, const int64_t* tk,
                            const int64_t* tblk, const int64_t* ti, const int64_t* tj, const double* tv, const double* c,
                            int32_t datarank, int64_t iblk, int32_t which, int64_t cap, int64_t* colptr_out, int64_t* rowval_out,
                            double* nzval_out, double* vec_out) {
    try {
        HostModel M;
        build_model(M, n_var, nblocks, blocksizes, ntrip, tk, tblk, ti, tj, tv, c, datarank);
        const HostCSC* X = nullptr;
        if (which == 3) X = &M.Clin;
        else {
            if (iblk < 0 || iblk >= (int64_t)M.msizes.size()) return -1;
            X = which == 0 ? &M.AA[iblk] : (which == 1 ? &M.Cm[iblk] : &M.Bm[iblk]);
        }
        const int64_t nnz = (int64_t)X->rowval.size();
        if (nnz > cap) return -2;
        if (colptr_out) std::copy(X->colptr.begin(), X->colptr.end(), colptr_out);
        if (rowval_out) std::copy(X->rowval.begin(), X->rowval.end(), rowval_out);
        if (nzval_out) std::copy(X->nzval.begin(), X->nzval.end(), nzval_out);
        if (vec_out) {
            const std::vector<double>& v = (which == 3) ? M.d_lin : M.b;
            std::copy(v.begin(), v.end(), vec_out);
        }
        return nnz;
    } catch (const std::exception& e) {
        fprintf(stderr, "lrn_dbg_model_block: %s\n", e.what());
        return -3;
    }
}

// src/initial_point.jl:17-81: X_i = Eps_i I, S_i = Eta_i I, y = 0, x_lin = Epss, s_lin = Etaa
int32_t lrn_initial_point(lrn_handle_t h, int32_t initpoint) {
    LRN_GROUP(h, lrn_initial_point(m_, initpoint));
    if (!h) return LRN_ERR_ARG;
    try {
        LRN_CUDA(cudaSetDevice(h->device));
        LRN_REQUIRE(h->finalized && h->ip_ready, "lrn_finalize first");
        cudaStream_t st = h->st;
        for (int i = 0; i < h->nlmi; i++) {
            if (!h->owns(i)) continue;                 // blocks distributed over the ranks: the owner's
            Block& B = h->blk[i];
            const double sm = std::sqrt((double)B.m);
            double Eps = 1.0, Eta = (double)h->n_var;
            if (initpoint != 0) {
                const double f = h->ip_normb2 / (1 + h->ip_normAA[i]);
                Eps = sm * std::max(1.0, sm * f);
                double mf = std::max(f, B.normC);
                mf = (1 + mf) / sm;
                Eta = sm * std::max(1.0, mf);
            }
            mat_set_identity(st, B.m, B.X.p(), B.ld, Eps);
            mat_set_identity(st, B.m, B.S.p(), B.ld, Eta);
            B.chol_cached = false;
            B.rdb_valid = false;
        }
        LRN_CUDA(cudaMemsetAsync(h->y.p, 0, (size_t)h->n_var * sizeof(double), st));
        if (h->nlin > 0) {
            double Epss = 1.0, Etaa = 1.0;
            if (initpoint != 0) {
                Epss = std::max(1.0, h->ip_pmax);
                Etaa = std::max(1.0, std::max(h->ip_rownmax, h->normd) / std::sqrt((double)h->nlin));
            }
            vec_axpby(st, h->nlin, h->x_lin.p, Epss, h->ones.p, 0.0, nullptr);
            vec_axpby(st, h->nlin, h->s_lin.p, Etaa, h->ones.p, 0.0, nullptr);
            vec_op(st, h->nlin, VEC_RECIP, h->si_lin.p, h->s_lin.p, nullptr);
        }
        LRN_CUDA(cudaStreamSynchronize(st));
        h->have_factor = false;
        return LRN_OK;
    } catch (const std::invalid_argument& e) {
        h->err = e.what();
        return LRN_ERR_ARG;
    } catch (const std::exception& e) {
        h->err = e.what();
        return LRN_ERR_CUDA;
    }
}

}  // extern "C"
