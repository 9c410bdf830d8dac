// Test / benchmark hooks (include/loraine_b200_debug.h).
#include "../../include/loraine_b200.h"
#include "../../include/loraine_b200_debug.h"
#include "chol.cuh"
#include "eig.cuh"
#include "gemm.cuh"
#include "ops.cuh"
#include <memory>

using namespace lrn;

namespace {

struct HostMat {   // device copy of a host column-major matrix with padded ld (+ optional 8-byte misalignment)
    DevBuf<double> buf;
    double* p = nullptr;
    int rows = 0, cols = 0, ld = 0;
    HostMat(const double* h, int r, int c, bool misalign = false) : rows(r), cols(c) {
        ld = misalign ? r + 1 + (r % 2) : pad_ld(r);          // odd ld for the misaligned variant
        if (misalign && ld % 2 == 0) ld += 1;
        buf.alloc((size_t)ld * std::max(c, 1) + 2);
        p = buf.p + (misalign ? 1 : 0);
        if (h && r > 0 && c > 0)
            LRN_CUDA(cudaMemcpy2D(p, (size_t)ld * 8, h, (size_t)r * 8, (size_t)r * 8, c, cudaMemcpyHostToDevice));
    }
    void download(double* h) const {
        if (rows > 0 && cols > 0)
            LRN_CUDA(cudaMemcpy2D(h, (size_t)rows * 8, p, (size_t)ld * 8, (size_t)rows * 8, cols, cudaMemcpyDeviceToHost));
    }
};

template <typename F>
int32_t guard(F&& f) {
    try {
        return f();
    } catch (const std::exception& e) {
        fprintf(stderr, "loraine_b200 debug hook: %s\n", e.what());
        return LRN_ERR_CUDA;
    }
}

__global__ void k_dmma_peak(double* out, int iters) {
    double a = 1.0 + threadIdx.x * 1e-9, b = 1.0 - threadIdx.x * 1e-9;
    double c[16][2];
#pragma unroll
    for (int i = 0; i < 16; i++) c[i][0] = c[i][1] = 0.0;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int i = 0; i < 16; i++)
            asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                         : "+d"(c[i][0]), "+d"(c[i][1]) : "d"(a), "d"(b));
    }
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 16; i++) s += c[i][0] + c[i][1];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
__global__ void k_dfma_peak(double* out, int iters) {
    double a = 1.0 + threadIdx.x * 1e-9, b = 1.0 - threadIdx.x * 1e-12;
    double c[16];
#pragma unroll
    for (int i = 0; i < 16; i++) c[i] = i;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int i = 0; i < 16; i++) c[i] = fma(c[i], a, b);
    }
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 16; i++) s += c[i];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
__global__ void k_copy(const double4* __restrict__ a, double4* __restrict__ b, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) b[i] = a[i];
}

}  // namespace

extern "C" {

int32_t lrn_dbg_gemm(int32_t M, int32_t N, int32_t K, int32_t transA, int32_t transB, double alpha, const double* A,
                     const double* B, double beta, double* C, int32_t mode, int32_t lower, const double* colscale,
                     int32_t misalign, int32_t reps, double* ms_per_launch) {
    return guard([&]() -> int32_t {
        HostMat dA(A, transA ? K : M, transA ? M : K, misalign != 0);
        HostMat dB(B, transB ? N : K, transB ? K : N, misalign != 0);
        HostMat dC(C, M, N, false);
        DevBuf<double> cs;
        if (colscale) cs.upload(colscale, N);
        GemmParams p;
        p.A = dA.p; p.B = dB.p; p.C = dC.p; p.M = M; p.N = N; p.K = K; p.lda = dA.ld; p.ldb = dB.ld; p.ldc = dC.ld;
        p.transA = transA != 0; p.transB = transB != 0; p.alpha = alpha; p.beta = beta; p.mode = mode & 1; p.ktri = (mode & 2) ? 1 : 0; p.lower = lower;
        p.colscale = colscale ? cs.p : nullptr;
        cudaStream_t st = 0;
        gemm(p, st);
        LRN_CUDA(cudaDeviceSynchronize());
        dC.download(C);
        if (reps > 0 && ms_per_launch) {
            cudaEvent_t e0, e1;
            LRN_CUDA(cudaEventCreate(&e0)); LRN_CUDA(cudaEventCreate(&e1));
            GemmParams q = p;
            if (beta != 0.0 && (mode & 1) == 0) q.beta = 0.0;       // keep magnitudes bounded over repetitions
            for (int w = 0; w < 3; w++) gemm(q, st);
            LRN_CUDA(cudaEventRecord(e0, st));
            for (int r = 0; r < reps; r++) gemm(q, st);
            LRN_CUDA(cudaEventRecord(e1, st));
            LRN_CUDA(cudaEventSynchronize(e1));
            float ms = 0;
            LRN_CUDA(cudaEventElapsedTime(&ms, e0, e1));
            *ms_per_launch = ms / reps;
            cudaEventDestroy(e0); cudaEventDestroy(e1);
        }
        return LRN_OK;
    });
}

static int g_dbg_chol_int8 = 0;

int32_t lrn_dbg_chol_int8(int32_t mode) {
    if (mode < 0 || mode > 2) return LRN_ERR_ARG;
    g_dbg_chol_int8 = mode;
    return LRN_OK;
}

int32_t lrn_dbg_syrk_i8(int32_t rows, int32_t K, const double* P, int32_t a_row0, int32_t b_row0, int32_t M, int32_t N, int64_t row0,
                        int64_t col0, int32_t lower, double* C, double* sigma, int32_t reps, double* ms_per_launch) {
    return guard([&]() -> int32_t {
        HostMat dP(P, rows, K), dC(C, M, N);
        const int rows_pad = round_up(std::max(rows, std::max(a_row0 + round_up(M, 128), b_row0 + round_up(N, 64))), 8);
        DevBuf<int8_t> sl(i8_slice_bytes(rows_pad, K));
        DevBuf<double> sg(rows_pad);
        cudaStream_t st = 0;
        i8_slice(dP.p, dP.ld, rows, K, rows_pad, sl.p, sg.p, st);
        syrk_update_i8(sl.p, sg.p, rows_pad, K, a_row0, b_row0, M, N, dC.p, dC.ld, row0, col0, lower != 0, st);
        LRN_CUDA(cudaDeviceSynchronize());
        dC.download(C);
        if (sigma) LRN_CUDA(cudaMemcpy(sigma, sg.p, (size_t)rows * sizeof(double), cudaMemcpyDeviceToHost));
        if (reps > 0 && ms_per_launch) {
            cudaEvent_t e0, e1;
            LRN_CUDA(cudaEventCreate(&e0)); LRN_CUDA(cudaEventCreate(&e1));
            for (int r = 0; r < 2; r++) syrk_update_i8(sl.p, sg.p, rows_pad, K, a_row0, b_row0, M, N, dC.p, dC.ld, row0, col0, lower != 0, st);
            LRN_CUDA(cudaEventRecord(e0, st));
            for (int r = 0; r < reps; r++) syrk_update_i8(sl.p, sg.p, rows_pad, K, a_row0, b_row0, M, N, dC.p, dC.ld, row0, col0, lower != 0, st);
            LRN_CUDA(cudaEventRecord(e1, st));
            LRN_CUDA(cudaEventSynchronize(e1));
            float ms = 0;
            LRN_CUDA(cudaEventElapsedTime(&ms, e0, e1));
            *ms_per_launch = ms / reps;
            cudaEventDestroy(e0); cudaEventDestroy(e1);
        }
        return LRN_OK;
    });
}

int32_t lrn_dbg_cholesky(int32_t n, double* A, double* x, int32_t which, int32_t* info, int32_t reps, double* ms_factor) {
    return guard([&]() -> int32_t {
        HostMat dA(A, n, n), dA0(A, n, n);
        CholWork w;
        w.int8 = g_dbg_chol_int8;
        cudaStream_t st = 0;
        cholesky_lower(dA.p, n, dA.ld, w, st);
        int inf = 0;
        LRN_CUDA(cudaMemcpy(&inf, w.info_ptr(), sizeof(int), cudaMemcpyDeviceToHost));
        if (info) *info = inf;
        if (x && which && inf == 0) {
            DevBuf<double> dx, tmp(n);
            dx.upload(x, n);
            chol_solve(dA.p, n, dA.ld, w, dx.p, tmp.p, which, st);
            LRN_CUDA(cudaMemcpy(x, dx.p, n * sizeof(double), cudaMemcpyDeviceToHost));
        }
        zero_strict_upper(dA.p, n, dA.ld, st);
        LRN_CUDA(cudaDeviceSynchronize());
        dA.download(A);
        if (reps > 0 && ms_factor) {
            cudaEvent_t e0, e1;
            LRN_CUDA(cudaEventCreate(&e0)); LRN_CUDA(cudaEventCreate(&e1));
            float tot = 0;
            for (int r = 0; r < reps; r++) {
                LRN_CUDA(cudaMemcpyAsync(dA.p, dA0.p, (size_t)dA.ld * n * 8, cudaMemcpyDeviceToDevice, st));
                LRN_CUDA(cudaEventRecord(e0, st));
                cholesky_lower(dA.p, n, dA.ld, w, st);
                LRN_CUDA(cudaEventRecord(e1, st));
                LRN_CUDA(cudaEventSynchronize(e1));
                float ms = 0;
                LRN_CUDA(cudaEventElapsedTime(&ms, e0, e1));
                tot += ms;
            }
            *ms_factor = tot / reps;
            cudaEventDestroy(e0); cudaEventDestroy(e1);
        }
        return LRN_OK;
    });
}

int32_t lrn_dbg_eig_small(int32_t n, const double* A, double* evals, double* V, int32_t relative) {
    return guard([&]() -> int32_t {
        HostMat dA(A, n, n), dV(nullptr, n, n);
        DevBuf<double> ev(n);
        EigSmallParams e;
        e.A = dA.p; e.lda = dA.ld; e.n = n; e.evals = ev.p; e.V = dV.p; e.ldv = dV.ld; e.sort_desc = 1; e.relative = relative;
        jacobi_eig_small(e, 0);
        LRN_CUDA(cudaDeviceSynchronize());
        LRN_CUDA(cudaMemcpy(evals, ev.p, n * sizeof(double), cudaMemcpyDeviceToHost));
        dV.download(V);
        return LRN_OK;
    });
}

int32_t lrn_dbg_svd(int32_t m, const double* A, double* UD, double* V, double* sigma, double tol, int32_t* sweeps, double* ms) {
    return guard([&]() -> int32_t {
        HostMat dA(A, m, m), dU(nullptr, m, m), dV(nullptr, V ? m : 1, V ? m : 1);
        DevBuf<double> sg(m);
        SvdWork w;
        cudaStream_t st = 0;
        cudaEvent_t e0, e1;
        LRN_CUDA(cudaEventCreate(&e0)); LRN_CUDA(cudaEventCreate(&e1));
        w.ensure(m, V != nullptr);
        LRN_CUDA(cudaEventRecord(e0, st));
        int sw = svd_block_jacobi(dA.p, dA.ld, m, dU.p, dU.ld, V ? dV.p : nullptr, dV.ld, sg.p, w, tol > 0 ? tol : 1e-9, 30, st);
        LRN_CUDA(cudaEventRecord(e1, st));
        LRN_CUDA(cudaDeviceSynchronize());
        float t = 0;
        LRN_CUDA(cudaEventElapsedTime(&t, e0, e1));
        if (ms) *ms = t;
        if (sweeps) *sweeps = sw;
        dU.download(UD);
        if (V) dV.download(V);
        LRN_CUDA(cudaMemcpy(sigma, sg.p, m * sizeof(double), cudaMemcpyDeviceToHost));
        cudaEventDestroy(e0); cudaEventDestroy(e1);
        return LRN_OK;
    });
}

int32_t lrn_dbg_lanczos(int32_t m, const double* T, int32_t nev_top, double tol, double* lmin, double* lmax, double* top_vals,
                        double* top_vecs, int32_t* iters, int32_t* converged) {
    return guard([&]() -> int32_t {
        HostMat dT(T, m, m), dV(nullptr, m, std::max(nev_top, 1));
        LanczosWork w;
        std::vector<double> tv(std::max(nev_top, 1));
        LanczosResult r = lanczos_extreme(dT.p, m, dT.ld, nev_top > 0 ? 3 : 1, nev_top, tv.data(), dV.p, dV.ld, tol > 0 ? tol : 1e-10, w, 0);
        LRN_CUDA(cudaDeviceSynchronize());
        if (lmin) *lmin = r.lmin;
        if (lmax) *lmax = r.lmax;
        if (iters) *iters = r.iters;
        if (converged) *converged = r.converged ? 1 : 0;
        if (nev_top > 0) {
            for (int t = 0; t < nev_top; t++) top_vals[t] = tv[t];
            dV.download(top_vecs);
        }
        return LRN_OK;
    });
}

int32_t lrn_dbg_batched_lambda_min(int32_t count, int32_t m, const double* mats, double* out) {
    return guard([&]() -> int32_t {
        std::vector<std::unique_ptr<HostMat>> hm;
        std::vector<double*> ptrs; std::vector<int> ms, lds;
        for (int z = 0; z < count; z++) {
            hm.emplace_back(new HostMat(mats + (size_t)z * m * m, m, m));
            ptrs.push_back(hm.back()->p); ms.push_back(m); lds.push_back(hm.back()->ld);
        }
        DevBuf<double*> dp; DevBuf<int> dm, dl; DevBuf<double> dout(count);
        dp.upload(ptrs); dm.upload(ms); dl.upload(lds);
        LRN_CUDA(cudaDeviceSynchronize());
        batched_lambda_min(dp.p, dm.p, dl.p, count, dout.p, 0);
        LRN_CUDA(cudaDeviceSynchronize());
        LRN_CUDA(cudaMemcpy(out, dout.p, count * sizeof(double), cudaMemcpyDeviceToHost));
        return LRN_OK;
    });
}

int32_t lrn_dbg_gemm_profile(int32_t mode, double* ms, double* flops, int64_t* launches) {
    return guard([&]() -> int32_t {
        long long n = 0;
        gemm_profile(mode, ms, flops, &n);
        if (launches) *launches = n;
        return LRN_OK;
    });
}

int32_t lrn_dbg_peak(int32_t kind, double* value) {
    return guard([&]() -> int32_t {
        cudaEvent_t e0, e1;
        LRN_CUDA(cudaEventCreate(&e0)); LRN_CUDA(cudaEventCreate(&e1));
        float ms = 0;
        if (kind == 0 || kind == 1) {
            const int blocks = 148 * 8, threads = 256, iters = 4096;
            DevBuf<double> out((size_t)blocks * threads);
            for (int w = 0; w < 2; w++) {
                if (kind == 0) k_dmma_peak<<<blocks, threads>>>(out.p, iters); else k_dfma_peak<<<blocks, threads>>>(out.p, iters);
            }
            LRN_CUDA(cudaEventRecord(e0));
            if (kind == 0) k_dmma_peak<<<blocks, threads>>>(out.p, iters); else k_dfma_peak<<<blocks, threads>>>(out.p, iters);
            LRN_CUDA(cudaEventRecord(e1));
            LRN_CUDA(cudaEventSynchronize(e1));
            LRN_CUDA(cudaEventElapsedTime(&ms, e0, e1));
            double flops = (kind == 0) ? (double)blocks * (threads / 32) * iters * 16.0 * 512.0
                                       : (double)blocks * threads * iters * 16.0 * 2.0;
            *value = flops / (ms * 1e-3) / 1e12;      // TFLOP/s
        } else {
            const size_t n = (size_t)1 << 27;         // 128 Mi double4 = 4 GiB per buffer is too much: use 2^25 double4 = 1 GiB
            const size_t cnt = (size_t)1 << 25;
            (void)n;
            DevBuf<double> a(cnt * 4), b(cnt * 4);
            for (int w = 0; w < 2; w++) k_copy<<<148 * 16, 256>>>((const double4*)a.p, (double4*)b.p, cnt);
            LRN_CUDA(cudaEventRecord(e0));
            for (int r = 0; r < 5; r++) k_copy<<<148 * 16, 256>>>((const double4*)a.p, (double4*)b.p, cnt);
            LRN_CUDA(cudaEventRecord(e1));
            LRN_CUDA(cudaEventSynchronize(e1));
            LRN_CUDA(cudaEventElapsedTime(&ms, e0, e1));
            *value = 5.0 * 2.0 * cnt * 32.0 / (ms * 1e-3) / 1e9;   // GB/s (read + write)
        }
        cudaEventDestroy(e0); cudaEventDestroy(e1);
        return LRN_OK;
    });
}

}  // extern "C"
