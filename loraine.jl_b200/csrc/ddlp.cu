// Double-double ("Float64x2") interior-point hot path for models without semidefinite blocks (SURVEY.md section 8(f), row N4;
// C ABI in include/loraine_b200_dd.h).  The reference runs `Optimizer{Float64x2}` through its generic Julia code with
// MultiFloats.jl numbers (README.md:37-54, examples/k.jl:8); for nlmi = 0 the iteration consists of
//   residuals        src/predictor_corrector.jl:8-22        Schur matrix   :36-39        right-hand sides :43-50, :183-192
//   Cholesky + solve :57-90, :199                             find_step_lin  :329-364      sigma trace      :163-166
//   find_mu          src/Solvers.jl:480-494                   DIMACS errors  :496-523
// Everything below is plain CUDA-core arithmetic on (hi, lo) pairs (dd.cuh): a double-double multiply-add is 28 FP64
// instructions (24 DADD + 2 DMUL + 2 DFMA), most of them dependent, so these kernels are bound by FP64 issue (the trailing
// update runs the FP64 pipe at 89 %, profiles/r2_dd_syrk_ncu_full.csv) or by dependent-issue latency, not by memory.  Layout: vectors as arrays of dd (16 B per
// entry, one 128-bit access), H and L dense column-major with leading dimension n.
#include "ddlp.cuh"
#include "group.cuh"
#include "dist.cuh"

#include "../../include/loraine_b200_debug.h"

using namespace lrn;

namespace {

constexpr int TB = 256;
constexpr int TS = 32;          // Cholesky tile
inline unsigned nblk(long long n, int t = TB) { return (unsigned)std::max<long long>(1, cdiv(n, t)); }

// ------------------------------------------------------------------------------------------------------------------------
// sparse products: out[r] = in[r] + sign * sum_e val[e] v[idx[e]]   (one warp per row of the given compressed structure)
// ------------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(TB) k_dd_spmv(int rows, const int* __restrict__ ptr, const int* __restrict__ idx,
                                                 const dd* __restrict__ val, const dd* __restrict__ v, const dd* __restrict__ in,
                                                 dd* __restrict__ out, double sign) {
    const int r = (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (r >= rows) return;
    dd acc = dd_make(0.0);
    for (int e = ptr[r] + lane; e < ptr[r + 1]; e += 32) acc = dd_fma(val[e], v[idx[e]], acc);
    acc = dd_warp_sum(acc);
    if (lane == 0) {
        acc = dd_mul_d(acc, sign);
        out[r] = in ? dd_add(in[r], acc) : acc;
    }
}

// H(:, i) (rows j >= i) = sum_k C[i,k] w[k] C[j,k]: one CTA per multiplier row i; the LP columns k of that row one after the
// other (two of them may hit the same j), the entries j of column k in parallel.          src/predictor_corrector.jl:37
// SHARD: only the rows j of row blocks (height pw) g with g % world == rank are written, every other entry of the column is
// zero.  An owned entry receives the same dd_fma sequence as without sharding, so the shards of all ranks add up to the
// single-GPU matrix bit for bit.
template <bool SHARD>
__global__ void __launch_bounds__(TB) k_dd_lp_schur(int n, const int* __restrict__ rptr, const int* __restrict__ ridx,
                                                     const dd* __restrict__ rval, const int* __restrict__ cptr,
                                                     const int* __restrict__ cidx, const dd* __restrict__ cval,
                                                     const dd* __restrict__ w, dd* __restrict__ H, int rank, int world, int pw) {
    const int i = blockIdx.x;
    dd* col = H + (size_t)i * n;
    for (int j = threadIdx.x; j < n; j += blockDim.x) col[j] = dd_make(0.0);
    __syncthreads();
    for (int e = rptr[i]; e < rptr[i + 1]; e++) {
        const int k = ridx[e];
        const dd coef = dd_mul(rval[e], w[k]);
        for (int f = cptr[k] + threadIdx.x; f < cptr[k + 1]; f += blockDim.x) {
            const int j = cidx[f];
            if (j >= i && (!SHARD || (j / pw) % world == rank)) col[j] = dd_fma(coef, cval[f], col[j]);
        }
        __syncthreads();
    }
}

__global__ void k_dd_mirror_lower(int n, dd* __restrict__ H) {      // Hermitian(BBBB, :L): upper := lower'
    const int j = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && i > j) H[(size_t)i * n + j] = H[(size_t)j * n + i];
}

__global__ void k_dd_shift_diag(int n, dd* __restrict__ H, double delta) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) H[(size_t)i * n + i] = dd_add_d(H[(size_t)i * n + i], delta);
}
// sharded H: keep the rank's own rows of the lower triangle, zero everything else (what k_dd_lp_schur<true> leaves)
__global__ void k_dd_keep_own_lower(int n, dd* __restrict__ H, int rank, int world, int pw) {
    const int j = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && (i < j || (i / pw) % world != rank)) H[(size_t)j * n + i] = dd_make(0.0);
}
// sharded H: the diagonal entries of the rank's own row blocks only
__global__ void k_dd_shift_own_diag(int n, dd* __restrict__ H, double delta, int rank, int world, int pw) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && (i / pw) % world == rank) H[(size_t)i * n + i] = dd_add_d(H[(size_t)i * n + i], delta);
}

// ------------------------------------------------------------------------------------------------------------------------
// triangular solves with the dd factor, 32 unknowns per step.  One CTA of 1024 threads for n <= 64; k_dd_trsv_multi otherwise
// ------------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) k_dd_trsv_fwd(const dd* __restrict__ L, const dd* __restrict__ rdiag, int n, dd* __restrict__ x) {
    __shared__ dd xt[TS];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int k0 = 0; k0 < n; k0 += TS) {
        const int w = min(TS, n - k0);
        if (warp == 0) {
            dd v = (lane < w) ? x[k0 + lane] : dd_make(0.0);
            for (int c = 0; c < w; c++) {
                dd xc = dd_make(0.0);
                if (lane == c) xc = dd_mul(v, rdiag[k0 + c]);
                xc = dd_shfl(xc, c);
                if (lane == c) v = xc;
                else if (lane > c && lane < w) v = dd_fms(L[(size_t)(k0 + c) * n + k0 + lane], xc, v);
            }
            if (lane < w) { xt[lane] = v; x[k0 + lane] = v; }
        }
        __syncthreads();
        for (int i = k0 + w + tid; i < n; i += blockDim.x) {
            dd a0 = x[i], a1 = dd_make(0.0), a2 = dd_make(0.0), a3 = dd_make(0.0);
            int c = 0;
            for (; c + 4 <= w; c += 4) {
                a0 = dd_fms(L[(size_t)(k0 + c) * n + i], xt[c], a0);
                a1 = dd_fms(L[(size_t)(k0 + c + 1) * n + i], xt[c + 1], a1);
                a2 = dd_fms(L[(size_t)(k0 + c + 2) * n + i], xt[c + 2], a2);
                a3 = dd_fms(L[(size_t)(k0 + c + 3) * n + i], xt[c + 3], a3);
            }
            for (; c < w; c++) a0 = dd_fms(L[(size_t)(k0 + c) * n + i], xt[c], a0);
            x[i] = dd_add(dd_add(a0, a1), dd_add(a2, a3));
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(1024) k_dd_trsv_bwd(const dd* __restrict__ L, const dd* __restrict__ rdiag, int n, dd* __restrict__ x) {
    __shared__ dd tsum[TS];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int last = ((n - 1) / TS) * TS;
    for (int k0 = last; k0 >= 0; k0 -= TS) {
        const int w = min(TS, n - k0);
        // t[c] = sum_{i >= k0 + w} L[i, k0 + c] x[i]: warp c owns column k0 + c (contiguous in i)
        if (warp < w) {
            dd acc = dd_make(0.0);
            const dd* col = L + (size_t)(k0 + warp) * n;
            for (int i = k0 + w + lane; i < n; i += 32) acc = dd_fma(col[i], x[i], acc);
            acc = dd_warp_sum(acc);
            if (lane == 0) tsum[warp] = acc;
        }
        __syncthreads();
        if (warp == 0) {
            dd v = (lane < w) ? dd_sub(x[k0 + lane], tsum[lane]) : dd_make(0.0);
            for (int c = w - 1; c >= 0; c--) {
                dd xc = dd_make(0.0);
                if (lane == c) xc = dd_mul(v, rdiag[k0 + c]);
                xc = dd_shfl(xc, c);
                if (lane == c) v = xc;
                else if (lane < c) v = dd_fms(L[(size_t)(k0 + lane) * n + k0 + c], xc, v);    // L'[lane, c] = L[c, lane]
            }
            if (lane < w) x[k0 + lane] = v;
        }
        __syncthreads();
    }
}

// Multi-CTA variant for more than two tiles: row tile i (32 unknowns) belongs to CTA i mod G (backward: counted from the end);
// a CTA subtracts the products with the finished tiles as they are published (flag word per tile, value = epoch of this
// launch), then solves its diagonal tile and publishes.  The factor is streamed by all CTAs instead of one SM (the single-CTA
// kernel is bound by what one SM can pull from HBM).  Launched cooperatively: the wait needs every CTA resident.
constexpr int TRSV_T = 256;                // 8 warps
constexpr long long TRSV_SPIN_MAX = 1ll << 26;

__device__ __forceinline__ bool dd_wait_flag(const int* flag, int epoch, int* err) {
    long long spins = 0;
    while (true) {
        int v;
        asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
        if (v == epoch) return true;
        if (++spins > TRSV_SPIN_MAX || *(volatile int*)err != 0) { *(volatile int*)err = 1; return false; }
        __nanosleep(64);
    }
}
__device__ __forceinline__ dd dd_ldcg(const dd* p) {
    const double2 v = __ldcg(reinterpret_cast<const double2*>(p));
    return dd_make(v.x, v.y);
}

__global__ void __launch_bounds__(TRSV_T) k_dd_trsv_multi(const dd* __restrict__ L, const dd* __restrict__ rdiag, int n, dd* x,
                                                         int* flags, int epoch, int backward, int* err) {
    __shared__ dd part[TRSV_T / 32][TS];
    __shared__ dd dt[TS][TS + 1];
    __shared__ dd rds[TS];
    __shared__ int failed;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = TRSV_T / 32;
    const int nt = (n + TS - 1) / TS, G = gridDim.x;
    if (tid == 0) failed = 0;
    __syncthreads();
    for (int seq = blockIdx.x; seq < nt; seq += G) {
        const int i = backward ? nt - 1 - seq : seq;
        const int r0 = i * TS, w = min(TS, n - r0);
        // the diagonal tile and its pivot reciprocals go to shared memory now: the 32 dependent steps of the tile solve below
        // must not wait for global memory
        for (int idx = tid; idx < TS * TS; idx += TRSV_T) {
            const int r = idx & 31, c = idx >> 5;
            dt[r][c] = (r < w && c < w) ? L[(size_t)(r0 + c) * n + r0 + r] : dd_make(0.0);
        }
        if (tid < TS) rds[tid] = (tid < w) ? rdiag[r0 + tid] : dd_make(0.0);
        // ---- products with the tiles this one depends on: forward k < i (lane = row of tile i), backward k > i (lane = column) ----
        dd a0 = dd_make(0.0), a1 = dd_make(0.0), a2 = dd_make(0.0), a3 = dd_make(0.0);
        const int ndep = backward ? nt - 1 - i : i;
        for (int q = warp; q < ndep; q += nw) {
            const int k = backward ? nt - 1 - q : q;           // dependencies in the order they are published
            const int c0 = k * TS, wk = min(TS, n - c0);
            {
                bool ok = true;
                if (lane == 0) ok = dd_wait_flag(flags + k, epoch, err);
                ok = __shfl_sync(0xffffffffu, ok ? 1 : 0, 0) != 0;
                if (!ok) { failed = 1; break; }
                if (lane < w) {
                    const dd* Lp = backward ? L + (size_t)(r0 + lane) * n + c0 : L + (size_t)c0 * n + r0 + lane;
                    const size_t step = backward ? 1 : (size_t)n;
                    int c = 0;
                    for (; c + 4 <= wk; c += 4) {
                        a0 = dd_fma(Lp[(size_t)c * step], dd_ldcg(x + c0 + c), a0);
                        a1 = dd_fma(Lp[(size_t)(c + 1) * step], dd_ldcg(x + c0 + c + 1), a1);
                        a2 = dd_fma(Lp[(size_t)(c + 2) * step], dd_ldcg(x + c0 + c + 2), a2);
                        a3 = dd_fma(Lp[(size_t)(c + 3) * step], dd_ldcg(x + c0 + c + 3), a3);
                    }
                    for (; c < wk; c++) a0 = dd_fma(Lp[(size_t)c * step], dd_ldcg(x + c0 + c), a0);
                }
            }
        }
        part[warp][lane] = dd_add(dd_add(a0, a1), dd_add(a2, a3));
        __syncthreads();
        if (failed) return;                                     // time-out: reported through *err by the host
        // ---- diagonal tile: warp 0 ----
        if (warp == 0) {
            dd v = dd_make(0.0);
            if (lane < w) {
                dd sum = part[0][lane];
                for (int q = 1; q < nw; q++) sum = dd_add(sum, part[q][lane]);
                v = dd_sub(x[r0 + lane], sum);
            }
            if (!backward) {
                for (int c = 0; c < w; c++) {
                    dd xc = dd_make(0.0);
                    if (lane == c) xc = dd_mul(v, rds[c]);
                    xc = dd_shfl(xc, c);
                    if (lane == c) v = xc;
                    else if (lane > c && lane < w) v = dd_fms(dt[lane][c], xc, v);
                }
            } else {
                for (int c = w - 1; c >= 0; c--) {
                    dd xc = dd_make(0.0);
                    if (lane == c) xc = dd_mul(v, rds[c]);
                    xc = dd_shfl(xc, c);
                    if (lane == c) v = xc;
                    else if (lane < c) v = dd_fms(dt[c][lane], xc, v);          // L'[lane, c] = L[c, lane]
                }
            }
            if (lane < w) x[r0 + lane] = v;
            __threadfence();
            __syncwarp();
            if (lane == 0) asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(flags + i), "r"(epoch) : "memory");
        }
        __syncthreads();                                        // part[] is reused by the next tile of this CTA
    }
}

// ------------------------------------------------------------------------------------------------------------------------
// element-wise kernels
// ------------------------------------------------------------------------------------------------------------------------
__global__ void k_dd_recip(int n, const dd* __restrict__ s, dd* __restrict__ si) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) si[i] = dd_recip(s[i]);
}
__global__ void k_dd_mul2(int n, const dd* __restrict__ a, const dd* __restrict__ b, dd* __restrict__ o) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) o[i] = dd_mul(a[i], b[i]);
}
// Rd_lin = d - s - (C' y)                                                                  src/predictor_corrector.jl:20
__global__ void k_dd_rd(int n, const dd* __restrict__ d, const dd* __restrict__ s, const dd* __restrict__ cty, dd* __restrict__ rd) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) rd[i] = dd_sub(dd_sub(d[i], s[i]), cty[i]);
}
// t = (x .* si) .* rd + x [+ (dx .* ds) .* si - sigmamu .* si]                             src/predictor_corrector.jl:49, :190-191
__global__ void k_dd_rhs_inner(int n, int corr, dd sigmamu, const dd* __restrict__ x, const dd* __restrict__ si,
                               const dd* __restrict__ rd, const dd* __restrict__ dx, const dd* __restrict__ ds, dd* __restrict__ t) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    dd v = dd_add(dd_mul(dd_mul(x[i], si[i]), rd[i]), x[i]);
    if (corr) {
        const dd tmp = dd_sub(dd_mul(dd_mul(dx[i], ds[i]), si[i]), dd_mul(sigmamu, si[i]));
        v = dd_add(v, tmp);
    }
    t[i] = v;
}
// delX_lin = -x - x .* si .* ds [+ sigmamu .* si + rnt]                                    src/predictor_corrector.jl:332-334
__global__ void k_dd_delx(int n, int corr, dd sigmamu, const dd* __restrict__ x, const dd* __restrict__ si,
                          const dd* __restrict__ ds, const dd* __restrict__ rnt, dd* __restrict__ dx) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    dd v = dd_sub(dd_neg(x[i]), dd_mul(dd_mul(x[i], si[i]), ds[i]));
    if (corr) v = dd_add(dd_add(v, dd_mul(sigmamu, si[i])), rnt[i]);
    dx[i] = v;
}
// predictor: Xn = x + alpha dx, Sn = s + beta ds, RNT = -(dx .* ds) .* si                  src/predictor_corrector.jl:351-354
__global__ void k_dd_pred_update(int n, const dd* __restrict__ ab, const dd* __restrict__ x, const dd* __restrict__ s,
                                 const dd* __restrict__ si, const dd* __restrict__ dx, const dd* __restrict__ ds,
                                 dd* __restrict__ xn, dd* __restrict__ sn, dd* __restrict__ rnt) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    xn[i] = dd_fma(ab[0], dx[i], x[i]);
    sn[i] = dd_fma(ab[1], ds[i], s[i]);
    rnt[i] = dd_neg(dd_mul(dd_mul(dx[i], ds[i]), si[i]));
}
// corrector: x += alpha dx, s += beta ds, S_lin_inv = 1 ./ s                               src/predictor_corrector.jl:358-360
__global__ void k_dd_corr_update(int n, const dd* __restrict__ ab, dd* __restrict__ x, dd* __restrict__ s, dd* __restrict__ si,
                                 const dd* __restrict__ dx, const dd* __restrict__ ds) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    x[i] = dd_fma(ab[0], dx[i], x[i]);
    const dd sv = dd_fma(ab[1], ds[i], s[i]);
    s[i] = sv;
    si[i] = dd_recip(sv);
}
__global__ void k_dd_axpy_scalar(int n, const dd* __restrict__ a, const dd* __restrict__ v, dd* __restrict__ y) {   // y += a[0] v
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = dd_fma(a[0], v[i], y[i]);
}

// ------------------------------------------------------------------------------------------------------------------------
// reductions (one CTA; the vectors of this path are short next to the n^3 factorisation)
// ------------------------------------------------------------------------------------------------------------------------
__device__ dd block_sum_dd(dd v, dd* sh) {
    v = dd_warp_sum(v);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) sh[w] = v;
    __syncthreads();
    dd r = (threadIdx.x < (blockDim.x >> 5)) ? sh[threadIdx.x] : dd_make(0.0);
    if (w == 0) r = dd_warp_sum(r);
    if (threadIdx.x == 0) sh[0] = r;
    __syncthreads();
    return sh[0];
}
__device__ dd block_min_dd(dd v, dd* sh) {
    v = dd_warp_min(v);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) sh[w] = v;
    __syncthreads();
    dd r = (threadIdx.x < (blockDim.x >> 5)) ? sh[threadIdx.x] : dd_make(INFINITY);
    if (w == 0) r = dd_warp_min(r);
    if (threadIdx.x == 0) sh[0] = r;
    __syncthreads();
    return sh[0];
}
// out[slot] = sum a[i] b[i]
__global__ void __launch_bounds__(1024) k_dd_dot(int n, const dd* __restrict__ a, const dd* __restrict__ b, dd* __restrict__ out, int slot) {
    __shared__ dd sh[32];
    dd acc = dd_make(0.0);
    for (int i = threadIdx.x; i < n; i += blockDim.x) acc = dd_fma(a[i], b[i], acc);
    acc = block_sum_dd(acc, sh);
    if (threadIdx.x == 0) out[slot] = acc;
}
// out[slot] = min_i num[i] / den[i]   (den == nullptr: min_i num[i])
__global__ void __launch_bounds__(1024) k_dd_min_ratio(int n, const dd* __restrict__ num, const dd* __restrict__ den, dd* __restrict__ out, int slot) {
    __shared__ dd sh[32];
    dd m = dd_make(INFINITY);
    for (int i = threadIdx.x; i < n; i += blockDim.x) m = dd_min(m, den ? dd_div(num[i], den[i]) : num[i]);
    m = block_min_dd(m, sh);
    if (threadIdx.x == 0) out[slot] = m;
}
// step length from the minimal ratio: 0.99 when mimi > -1e-6, else min(1, -tau / mimi)      src/predictor_corrector.jl:336-347
__global__ void k_dd_steplen(dd* __restrict__ red, int slot_in, int slot_out, double tau) {
    const dd mimi = red[slot_in];
    dd a;
    if (dd_gt(mimi, dd_make(-1e-6))) a = dd_make(0.99);
    else a = dd_min(dd_make(1.0), dd_div(dd_make(-tau), mimi));
    red[slot_out] = a;
}
// red slots
enum { R_MU = 0, R_MIMIX = 1, R_MIMIS = 2, R_ALPHA = 3, R_BETA = 4, R_DOT = 5, R_NB = 6, R_ND = 7, R_BY = 8, R_DX = 9, R_RP2 = 10,
       R_RD2 = 11, R_MINX = 12, R_MINS = 13, R_SX = 14, R_ERR = 16 /* ..21 */, R_COUNT = 24 };

__global__ void k_dd_scale_slot(dd* __restrict__ red, int slot, double denom) { red[slot] = dd_div(red[slot], dd_make(denom)); }
// norm of Float64 model data: the reference evaluates norm(b), norm(d_lin) in Float64 (the model stays Float64 whatever T is),
// so the correctly rounded double is kept
__global__ void k_dd_norm_slot(dd* __restrict__ red, int slot) { red[slot] = dd_make(dd_sqrt(red[slot]).hi); }

// DIMACS errors for nlmi = 0                                                                   src/Solvers.jl:496-517
__global__ void k_dd_dimacs(dd* __restrict__ red) {
    const dd one = dd_make(1.0), zero = dd_make(0.0);
    const dd nb = red[R_NB], nd = red[R_ND], by = red[R_BY], dx = red[R_DX];
    const dd onb = dd_add(one, nb), ond = dd_add(one, nd);
    red[R_ERR + 0] = dd_div(dd_sqrt(red[R_RP2]), onb);
    red[R_ERR + 1] = dd_max(zero, dd_div(dd_neg(red[R_MINX]), onb));
    red[R_ERR + 2] = dd_div(dd_sqrt(red[R_RD2]), ond);
    red[R_ERR + 3] = dd_max(zero, dd_div(dd_neg(red[R_MINS]), ond));
    red[R_ERR + 4] = dd_div(dd_sub(dx, by), dd_add(one, dd_abs(by)));               // btrace(C, X) = 0 without PSD blocks
    red[R_ERR + 5] = dd_div(red[R_SX], dd_add(dd_add(one, dd_abs(dx)), dd_abs(by)));
}

// ------------------------------------------------------------------------------------------------------------------------
template <typename F>
int32_t guarded(lrn_dd_solver* h, F&& f) {
    if (!h) return LRN_ERR_ARG;
    try {
        LRN_CUDA(cudaSetDevice(h->device));
        return f();
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

struct Timed {                       // synchronous phase timer (this path is not latency-critical)
    lrn_dd_solver* h;
    int slot;
    Timed(lrn_dd_solver* h_, int slot_) : h(h_), slot(slot_) { cudaEventRecord(h->ev0, h->st); }
    ~Timed() {
        cudaEventRecord(h->ev1, h->st);
        if (cudaEventSynchronize(h->ev1) == cudaSuccess) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, h->ev0, h->ev1) == cudaSuccess) h->t_ms[slot] += ms;
        }
    }
};

std::vector<dd> pack(const double* hi, const double* lo, size_t n) {
    std::vector<dd> v(n);
    for (size_t i = 0; i < n; i++) { v[i].hi = hi[i]; v[i].lo = lo ? lo[i] : 0.0; }
    return v;
}
void upload_dd(lrn_dd_solver* h, DevBuf<dd>& dst, const double* hi, const double* lo, size_t n) {
    std::vector<dd> v = pack(hi, lo, n);
    LRN_CUDA(cudaMemcpyAsync(dst.p, v.data(), n * sizeof(dd), cudaMemcpyHostToDevice, h->st));
    LRN_CUDA(cudaStreamSynchronize(h->st));     // `v` is pageable and about to go out of scope
}
void download_dd(lrn_dd_solver* h, const dd* src, double* hi, double* lo, size_t n) {
    std::vector<dd> v(n);
    LRN_CUDA(cudaMemcpyAsync(v.data(), src, n * sizeof(dd), cudaMemcpyDeviceToHost, h->st));
    LRN_CUDA(cudaStreamSynchronize(h->st));
    for (size_t i = 0; i < n; i++) { if (hi) hi[i] = v[i].hi; if (lo) lo[i] = v[i].lo; }
}
dd read_slot(lrn_dd_solver* h, int slot) {
    dd v;
    LRN_CUDA(cudaMemcpyAsync(&v, h->red.p + slot, sizeof(dd), cudaMemcpyDeviceToHost, h->st));
    LRN_CUDA(cudaStreamSynchronize(h->st));
    return v;
}
void spmv(lrn_dd_solver* h, bool by_rows, const dd* v, const dd* in, dd* out, double sign) {
    const int rows = by_rows ? h->n : h->nlin;
    if (rows == 0) return;
    k_dd_spmv<<<nblk((long long)rows * 32), TB, 0, h->st>>>(rows, by_rows ? h->rptr.p : h->cptr.p, by_rows ? h->ridx.p : h->cidx.p,
                                                            by_rows ? h->rval.p : h->cval.p, v, in, out, sign);
    LRN_CHECK_LAUNCH();
}
void dot(lrn_dd_solver* h, int n, const dd* a, const dd* b, int slot) {
    k_dd_dot<<<1, 1024, 0, h->st>>>(n, a, b, h->red.p, slot);
    LRN_CHECK_LAUNCH();
}
void trsv(lrn_dd_solver* h, bool fwd, dd* x) {
    const int nt = (int)cdiv(h->n, TS);
    if (nt > 2 && h->trsv_ctas > 0) {
        const dd* Lp = h->L.p;
        const dd* rd = h->rdiag.p;
        int n = h->n, epoch = ++h->trsv_epoch, backward = fwd ? 0 : 1;
        int* flags = h->flags.p;
        int* err = h->info.p + 1;
        void* args[] = {&Lp, &rd, &n, &x, &flags, &epoch, &backward, &err};
        LRN_CUDA(cudaLaunchCooperativeKernel((const void*)k_dd_trsv_multi, dim3((unsigned)std::min(nt, h->trsv_ctas)), dim3(TRSV_T),
                                             args, 0, h->st));
        g_kernel_launches.fetch_add(1, std::memory_order_relaxed);
        return;
    }
    if (fwd) k_dd_trsv_fwd<<<1, 1024, 0, h->st>>>(h->L.p, h->rdiag.p, h->n, x);
    else k_dd_trsv_bwd<<<1, 1024, 0, h->st>>>(h->L.p, h->rdiag.p, h->n, x);
    LRN_CHECK_LAUNCH();
}

lrn_dd_solver* dd_member0(lrn_dd_solver* facade) { return static_cast<GroupOf<lrn_dd_solver>*>(facade->group)->members[0]; }

}  // namespace

extern "C" {

int32_t lrn_dd_create(lrn_dd_handle_t* out, int64_t n_var, int64_t nlin, int32_t device) {
    if (!out) return LRN_ERR_ARG;
    *out = nullptr;
    if (n_var < 1 || nlin < 1 || n_var > 20000 || nlin > (1 << 24)) return LRN_ERR_ARG;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return LRN_ERR_CUDA; }   // no CPU fallback
    lrn_dd_solver* h = new lrn_dd_solver();
    int32_t rc = guarded(h, [&]() -> int32_t {
        if (device < 0) LRN_CUDA(cudaGetDevice(&h->device)); else h->device = device;
        LRN_CUDA(cudaSetDevice(h->device));
        cudaDeviceProp prop;
        LRN_CUDA(cudaGetDeviceProperties(&prop, h->device));
        LRN_REQUIRE(prop.major == 10, "libloraine_b200 is built for sm_100a only");
        int prio_lo = 0, prio_hi = 0;
        LRN_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
        LRN_CUDA(cudaStreamCreateWithPriority(&h->st, cudaStreamNonBlocking, prio_hi));
        LRN_CUDA(cudaStreamCreateWithPriority(&h->st2, cudaStreamNonBlocking, prio_lo));
        LRN_CUDA(cudaEventCreateWithFlags(&h->evP, cudaEventDisableTiming));
        LRN_CUDA(cudaEventCreateWithFlags(&h->evR, cudaEventDisableTiming));
        LRN_CUDA(cudaEventCreate(&h->ev0));
        LRN_CUDA(cudaEventCreate(&h->ev1));
        h->n = (int)n_var;
        h->nlin = (int)nlin;
        const size_t n = (size_t)n_var, m = (size_t)nlin;
        for (DevBuf<dd>* v : {&h->d, &h->x, &h->s, &h->si, &h->rd, &h->dx, &h->ds, &h->xn, &h->sn, &h->rnt, &h->w, &h->tl}) v->alloc(m);
        for (DevBuf<dd>* v : {&h->b, &h->y, &h->rp, &h->rhs, &h->dely, &h->tn, &h->rdiag}) v->alloc(n);
        h->H.alloc(n * n);
        h->L.alloc(n * n);
        h->red.alloc(R_COUNT);
        h->info.alloc(2);
        h->flags.alloc((size_t)cdiv(n_var, TS));
        // every CTA of the multi-CTA triangular solve must be resident (it waits on flags published by the others)
        int per_sm = 0, coop = 0;
        LRN_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, h->device));
        LRN_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_dd_trsv_multi, TRSV_T, 0));
        h->trsv_ctas = h->trsv_ctas_max = (coop && per_sm > 0) ? std::min(prop.multiProcessorCount, 128) : 0;
        return LRN_OK;
    });
    if (rc != LRN_OK) {
        fprintf(stderr, "[loraine_b200] lrn_dd_create failed: %s\n", h->err.c_str());
        lrn_dd_destroy(h);
        return rc;
    }
    *out = h;
    return LRN_OK;
}

int32_t lrn_dd_destroy(lrn_dd_handle_t h) {
    if (!h) return LRN_OK;
    if (h->group) {
        auto* g = static_cast<GroupOf<lrn_dd_solver>*>(h->group);
        // the communicators of one ncclCommInitAll clique are destroyed from concurrent threads (ncclCommDestroy may wait for peers)
        std::vector<std::thread> th;
        for (auto* m : g->members) th.emplace_back([m] { lrn_dd_destroy(m); });
        for (auto& t : th) t.join();
        delete g;
        delete h;
        return LRN_OK;
    }
    cudaSetDevice(h->device);
    if (h->st) { cudaStreamSynchronize(h->st); cudaStreamDestroy(h->st); }
    if (h->st2) { cudaStreamSynchronize(h->st2); cudaStreamDestroy(h->st2); }
    if (h->evP) cudaEventDestroy(h->evP);
    if (h->evR) cudaEventDestroy(h->evR);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->nccl) { delete static_cast<DistCtx*>(h->nccl); h->nccl = nullptr; }
    delete h;
    return LRN_OK;
}

const char* lrn_dd_last_error(lrn_dd_handle_t h) {
    if (h && h->group && h->err.empty()) return dd_member0(h)->err.c_str();
    return h ? h->err.c_str() : "null handle";
}

int32_t lrn_dd_set_lin(lrn_dd_handle_t h, const int64_t* colptr, const int64_t* rowval, const double* nz_hi, const double* nz_lo,
                       const double* d_hi, const double* d_lo) {
    LRN_GROUP(h, lrn_dd_set_lin(m_, colptr, rowval, nz_hi, nz_lo, d_hi, d_lo));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(colptr && rowval && nz_hi && d_hi, "null argument");
        const int n = h->n, m = h->nlin;
        LRN_REQUIRE(colptr[0] == 1, "colptr must be 1-based");
        const long long nnz = colptr[m] - 1;
        LRN_REQUIRE(nnz >= 0 && nnz < (1ll << 31), "bad colptr");
        std::vector<int> cp(m + 1), ci((size_t)nnz), rp(n + 1, 0), ri((size_t)nnz);
        std::vector<dd> cv((size_t)nnz), rv((size_t)nnz);
        for (int k = 0; k <= m; k++) {
            LRN_REQUIRE(colptr[k] >= 1 && colptr[k] - 1 <= nnz && (k == 0 || colptr[k] >= colptr[k - 1]), "colptr not monotone");
            cp[k] = (int)(colptr[k] - 1);
        }
        for (int k = 0; k < m; k++)      // the Schur kernel updates the entries of one column in parallel: no duplicates allowed
            for (int e = cp[k] + 1; e < cp[k + 1]; e++)
                LRN_REQUIRE(rowval[e] > rowval[e - 1], "row indices of a column must be strictly increasing (sorted, no duplicates)");
        for (long long e = 0; e < nnz; e++) {
            LRN_REQUIRE(rowval[e] >= 1 && rowval[e] <= n, "row index out of range");
            ci[e] = (int)(rowval[e] - 1);
            cv[e].hi = nz_hi[e];
            cv[e].lo = nz_lo ? nz_lo[e] : 0.0;
            rp[ci[e] + 1]++;
        }
        for (int i = 0; i < n; i++) rp[i + 1] += rp[i];
        std::vector<int> fill(rp.begin(), rp.end() - 1);
        for (int k = 0; k < m; k++)                      // columns in increasing order: every CSR row ends up sorted by k
            for (int e = cp[k]; e < cp[k + 1]; e++) {
                const int pos = fill[ci[e]]++;
                ri[pos] = k;
                rv[pos] = cv[e];
            }
        h->nnz = nnz;
        h->cptr.upload(cp, h->st); h->cidx.upload(ci, h->st); h->rptr.upload(rp, h->st); h->ridx.upload(ri, h->st);
        h->cval.upload(cv, h->st); h->rval.upload(rv, h->st);
        LRN_CUDA(cudaStreamSynchronize(h->st));
        upload_dd(h, h->d, d_hi, d_lo, (size_t)m);
        h->have_lin = true;
        return LRN_OK;
    });
}

int32_t lrn_dd_set_b(lrn_dd_handle_t h, const double* b_hi, const double* b_lo) {
    LRN_GROUP(h, lrn_dd_set_b(m_, b_hi, b_lo));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(b_hi, "null argument");
        upload_dd(h, h->b, b_hi, b_lo, (size_t)h->n);
        h->have_b = true;
        return LRN_OK;
    });
}

int32_t lrn_dd_finalize(lrn_dd_handle_t h) {
    LRN_GROUP(h, lrn_dd_finalize(m_));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(h->have_lin && h->have_b, "lrn_dd_set_lin and lrn_dd_set_b first");
        // norm(b), norm(d_lin) for the DIMACS denominators (src/Solvers.jl:499, :514)
        dot(h, h->n, h->b.p, h->b.p, R_NB);
        dot(h, h->nlin, h->d.p, h->d.p, R_ND);
        k_dd_norm_slot<<<1, 1, 0, h->st>>>(h->red.p, R_NB); LRN_CHECK_LAUNCH();
        k_dd_norm_slot<<<1, 1, 0, h->st>>>(h->red.p, R_ND); LRN_CHECK_LAUNCH();
        LRN_CUDA(cudaStreamSynchronize(h->st));
        h->finalized = true;
        return LRN_OK;
    });
}

int32_t lrn_dd_set_iterate(lrn_dd_handle_t h, const double* y_hi, const double* y_lo, const double* x_hi, const double* x_lo,
                           const double* s_hi, const double* s_lo) {
    LRN_GROUP(h, lrn_dd_set_iterate(m_, y_hi, y_lo, x_hi, x_lo, s_hi, s_lo));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(h->finalized, "lrn_dd_finalize first");
        LRN_REQUIRE(y_hi && x_hi && s_hi, "null argument");
        upload_dd(h, h->y, y_hi, y_lo, (size_t)h->n);
        upload_dd(h, h->x, x_hi, x_lo, (size_t)h->nlin);
        upload_dd(h, h->s, s_hi, s_lo, (size_t)h->nlin);
        k_dd_recip<<<nblk(h->nlin), TB, 0, h->st>>>(h->nlin, h->s.p, h->si.p);      // S_lin_inv, src/initial_point.jl:71
        LRN_CHECK_LAUNCH();
        h->have_iterate = true;
        h->have_H = h->have_factor = false;
        return LRN_OK;
    });
}

int32_t lrn_dd_get_solution(lrn_dd_handle_t h, double* y_hi, double* y_lo, double* x_hi, double* x_lo, double* s_hi, double* s_lo) {
    if (h && h->group) return lrn_dd_get_solution(dd_member0(h), y_hi, y_lo, x_hi, x_lo, s_hi, s_lo);     // replicated
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(h->have_iterate, "no iterate");
        if (y_hi || y_lo) download_dd(h, h->y.p, y_hi, y_lo, (size_t)h->n);
        if (x_hi || x_lo) download_dd(h, h->x.p, x_hi, x_lo, (size_t)h->nlin);
        if (s_hi || s_lo) download_dd(h, h->s.p, s_hi, s_lo, (size_t)h->nlin);
        return LRN_OK;
    });
}

int32_t lrn_dd_find_mu(lrn_dd_handle_t h, double mu[2]) {
    LRN_GROUP(h, lrn_dd_find_mu(m_, r_ == 0 ? mu : group_scratch().d));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(h->have_iterate && mu, "no iterate");
        Timed t(h, 3);
        dot(h, h->nlin, h->x.p, h->s.p, R_MU);
        k_dd_scale_slot<<<1, 1, 0, h->st>>>(h->red.p, R_MU, (double)h->nlin); LRN_CHECK_LAUNCH();
        const dd v = read_slot(h, R_MU);
        mu[0] = v.hi; mu[1] = v.lo;
        return LRN_OK;
    });
}

int32_t lrn_dd_prepare_W(lrn_dd_handle_t h) {
    LRN_GROUP(h, lrn_dd_prepare_W(m_));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(h->have_iterate, "no iterate");
        Timed t(h, 3);
        k_dd_recip<<<nblk(h->nlin), TB, 0, h->st>>>(h->nlin, h->s.p, h->si.p);
        LRN_CHECK_LAUNCH();
        return LRN_OK;
    });
}

int32_t lrn_dd_residuals(lrn_dd_handle_t h) {
    LRN_GROUP(h, lrn_dd_residuals(m_));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(h->have_iterate, "no iterate");
        Timed t(h, 3);
        spmv(h, true, h->x.p, h->b.p, h->rp.p, -1.0);                                 // Rp = b - C x
        spmv(h, false, h->y.p, nullptr, h->tl.p, 1.0);                                // C' y
        k_dd_rd<<<nblk(h->nlin), TB, 0, h->st>>>(h->nlin, h->d.p, h->s.p, h->tl.p, h->rd.p);
        LRN_CHECK_LAUNCH();
        return LRN_OK;
    });
}

int32_t lrn_dd_schur_assemble(lrn_dd_handle_t h) {
    LRN_GROUP(h, lrn_dd_schur_assemble(m_));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(h->have_iterate, "no iterate");
        Timed t(h, 0);
        const int n = h->n;
        k_dd_mul2<<<nblk(h->nlin), TB, 0, h->st>>>(h->nlin, h->x.p, h->si.p, h->w.p);
        LRN_CHECK_LAUNCH();
        if (dd_sharded(h)) {
            // own rows of the lower triangle only (the upper mirror would mix the shards); lrn_dd_get_array(1) gathers them
            k_dd_lp_schur<true><<<n, TB, 0, h->st>>>(n, h->rptr.p, h->ridx.p, h->rval.p, h->cptr.p, h->cidx.p, h->cval.p, h->w.p,
                                                     h->H.p, h->rank, h->world, h->pw);
            LRN_CHECK_LAUNCH();
        } else {
            k_dd_lp_schur<false><<<n, TB, 0, h->st>>>(n, h->rptr.p, h->ridx.p, h->rval.p, h->cptr.p, h->cidx.p, h->cval.p, h->w.p,
                                                      h->H.p, 0, 1, 1);
            LRN_CHECK_LAUNCH();
            k_dd_mirror_lower<<<dim3(nblk(n), (unsigned)n), TB, 0, h->st>>>(n, h->H.p);
            LRN_CHECK_LAUNCH();
        }
        h->H_gathered = false;
        h->have_H = true;
        h->have_factor = false;
        return LRN_OK;
    });
}

int32_t lrn_dd_schur_shift(lrn_dd_handle_t h, double delta) {
    LRN_GROUP(h, lrn_dd_schur_shift(m_, delta));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(h->have_H, "lrn_dd_schur_assemble first");
        if (dd_sharded(h) && !h->H_gathered)
            k_dd_shift_own_diag<<<nblk(h->n), TB, 0, h->st>>>(h->n, h->H.p, delta, h->rank, h->world, h->pw);
        else
            k_dd_shift_diag<<<nblk(h->n), TB, 0, h->st>>>(h->n, h->H.p, delta);
        LRN_CHECK_LAUNCH();
        return LRN_OK;
    });
}

int32_t lrn_dd_schur_factor(lrn_dd_handle_t h) {
    LRN_GROUP(h, lrn_dd_schur_factor(m_));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(h->have_H, "lrn_dd_schur_assemble first");
        int info = 0;
        if (dd_sharded(h)) {
            // a handle sharded through lrn_dd_dbg_set_shard holds one shard of H: it must not factor it
            if (!h->nccl) throw std::runtime_error("the Schur rows are sharded but the handle has no NCCL communicator "
                                                   "(lrn_dd_dist_init / lrn_dd_create_multi)");
            Timed t(h, 1);
            info = dd_factor_dist(h);
        } else {
            Timed t(h, 1);
            const int n = h->n;
            // (replaying the factorisation as a CUDA graph was measured: 6.85 ms against 6.24 ms eager at n = 2000 -- the chain
            // of dependent tile kernels on the device is the limiter, not the ~10 host calls per step)
            auto enqueue = [&]() {
                LRN_CUDA(cudaMemcpyAsync(h->L.p, h->H.p, (size_t)n * n * sizeof(dd), cudaMemcpyDeviceToDevice, h->st));
                LRN_CUDA(cudaMemsetAsync(h->info.p, 0, sizeof(int), h->st));
                // One-step look-ahead on two streams: the panel chain (diagonal tile, tiles below it, update of the NEXT tile
                // column) runs on h->st (high priority), the update of the rest of the trailing matrix on h->st2.  Both update
                // kernels of consecutive steps touch the same tiles, so the chain waits for rest(k-1) before col(k).
                bool rest_pending = false;
                for (int k0 = 0; k0 < n; k0 += TS) {
                    const int w = std::min(TS, n - k0);
                    k_dd_potrf_tile<<<1, dim3(TS, TS), 0, h->st>>>(h->L.p, n, k0, w, h->info.p, h->rdiag.p);
                    LRN_CHECK_LAUNCH();
                    const int below = n - k0 - w;
                    if (below <= 0) break;
                    const unsigned nt = (unsigned)cdiv(below, TS);
                    k_dd_trsm_tile<<<nt, TS * TRSM_CB, 0, h->st>>>(h->L.p, n, k0, w, h->rdiag.p);
                    LRN_CHECK_LAUNCH();
                    if (rest_pending) LRN_CUDA(cudaStreamWaitEvent(h->st, h->evR, 0));       // rest(k-1) before col(k)
                    rest_pending = false;
                    if (nt > 1) {
                        LRN_CUDA(cudaEventRecord(h->evP, h->st));
                        LRN_CUDA(cudaStreamWaitEvent(h->st2, h->evP, 0));
                        k_dd_syrk_tile<<<dim3(nt, nt - 1), dim3(TS, TS), 0, h->st2>>>(h->L.p, n, k0, w, 1);
                        LRN_CHECK_LAUNCH();
                        LRN_CUDA(cudaEventRecord(h->evR, h->st2));
                        rest_pending = true;
                    }
                    k_dd_syrk_tile<<<dim3(nt, 1), dim3(TS, TS), 0, h->st>>>(h->L.p, n, k0, w, 0);
                    LRN_CHECK_LAUNCH();
                }
                if (rest_pending) LRN_CUDA(cudaStreamWaitEvent(h->st, h->evR, 0));
            };
            enqueue();
            LRN_CUDA(cudaMemcpyAsync(&info, h->info.p, sizeof(int), cudaMemcpyDeviceToHost, h->st));
            LRN_CUDA(cudaStreamSynchronize(h->st));
        }
        h->have_factor = (info == 0);
        return info;
    });
}

int32_t lrn_dd_rhs_predictor(lrn_dd_handle_t h) {
    LRN_GROUP(h, lrn_dd_rhs_predictor(m_));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(h->have_iterate, "no iterate");
        Timed t(h, 3);
        k_dd_rhs_inner<<<nblk(h->nlin), TB, 0, h->st>>>(h->nlin, 0, dd_make(0.0), h->x.p, h->si.p, h->rd.p, h->dx.p, h->ds.p, h->tl.p);
        LRN_CHECK_LAUNCH();
        spmv(h, true, h->tl.p, h->rp.p, h->rhs.p, 1.0);
        return LRN_OK;
    });
}

int32_t lrn_dd_rhs_corrector(lrn_dd_handle_t h, const double sigma[2], const double mu[2]) {
    LRN_GROUP(h, lrn_dd_rhs_corrector(m_, sigma, mu));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(h->have_iterate && sigma && mu, "no iterate");
        Timed t(h, 3);
        // sigma * mu on the host in double-double (same operation order as the reference: (sigma * mu) .* Si_lin)
        const dd sm = dd_mul(dd_make(sigma[0], sigma[1]), dd_make(mu[0], mu[1]));
        k_dd_rhs_inner<<<nblk(h->nlin), TB, 0, h->st>>>(h->nlin, 1, sm, h->x.p, h->si.p, h->rd.p, h->dx.p, h->ds.p, h->tl.p);
        LRN_CHECK_LAUNCH();
        spmv(h, true, h->tl.p, h->rp.p, h->rhs.p, 1.0);
        return LRN_OK;
    });
}

int32_t lrn_dd_schur_solve(lrn_dd_handle_t h, int32_t which) {
    LRN_GROUP(h, lrn_dd_schur_solve(m_, which));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(which == 3 || which == 6, "which must be 3 or 6");
        // a call-order error, not a bad argument: no factor, or the last factorisation failed
        if (!h->have_factor) throw std::runtime_error("no valid Cholesky factor (lrn_dd_schur_factor first, and it must return 0)");
        Timed t(h, 2);
        LRN_CUDA(cudaMemcpyAsync(h->dely.p, h->rhs.p, (size_t)h->n * sizeof(dd), cudaMemcpyDeviceToDevice, h->st));
        for (int rep = 0; rep < (which == 6 ? 2 : 1); rep++) {
            trsv(h, true, h->dely.p);
            trsv(h, false, h->dely.p);
        }
        int timed_out = 0;
        LRN_CUDA(cudaMemcpyAsync(&timed_out, h->info.p + 1, sizeof(int), cudaMemcpyDeviceToHost, h->st));
        LRN_CUDA(cudaStreamSynchronize(h->st));
        if (timed_out) {
            LRN_CUDA(cudaMemsetAsync(h->info.p + 1, 0, sizeof(int), h->st));
            throw std::runtime_error("double-double triangular solve: flag wait timed out");
        }
        return LRN_OK;
    });
}

int32_t lrn_dd_find_step(lrn_dd_handle_t h, int32_t predict, const double sigma[2], const double mu[2], double tau,
                         double alpha_lin[2], double beta_lin[2]) {
    LRN_GROUP(h, lrn_dd_find_step(m_, predict, sigma, mu, tau, r_ == 0 ? alpha_lin : group_scratch().d,
                                  r_ == 0 ? beta_lin : group_scratch().d + 2));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(h->have_iterate && sigma && mu && alpha_lin && beta_lin, "no iterate");
        Timed t(h, 3);
        const int m = h->nlin;
        const dd sm = dd_mul(dd_make(sigma[0], sigma[1]), dd_make(mu[0], mu[1]));
        spmv(h, false, h->dely.p, h->rd.p, h->ds.p, -1.0);                            // delS_lin = Rd_lin - C' dely
        k_dd_delx<<<nblk(m), TB, 0, h->st>>>(m, predict ? 0 : 1, sm, h->x.p, h->si.p, h->ds.p, h->rnt.p, h->dx.p);
        LRN_CHECK_LAUNCH();
        k_dd_min_ratio<<<1, 1024, 0, h->st>>>(m, h->dx.p, h->x.p, h->red.p, R_MIMIX); LRN_CHECK_LAUNCH();
        k_dd_min_ratio<<<1, 1024, 0, h->st>>>(m, h->ds.p, h->s.p, h->red.p, R_MIMIS); LRN_CHECK_LAUNCH();
        k_dd_steplen<<<1, 1, 0, h->st>>>(h->red.p, R_MIMIX, R_ALPHA, tau); LRN_CHECK_LAUNCH();
        k_dd_steplen<<<1, 1, 0, h->st>>>(h->red.p, R_MIMIS, R_BETA, tau); LRN_CHECK_LAUNCH();
        if (predict) {
            k_dd_pred_update<<<nblk(m), TB, 0, h->st>>>(m, h->red.p + R_ALPHA, h->x.p, h->s.p, h->si.p, h->dx.p, h->ds.p, h->xn.p,
                                                        h->sn.p, h->rnt.p);
            LRN_CHECK_LAUNCH();
        } else {
            // without PSD blocks minimum([alpha; alpha_lin]) = alpha_lin                       src/predictor_corrector.jl:314, :358-359
            k_dd_axpy_scalar<<<nblk(h->n), TB, 0, h->st>>>(h->n, h->red.p + R_BETA, h->dely.p, h->y.p);
            LRN_CHECK_LAUNCH();
            k_dd_corr_update<<<nblk(m), TB, 0, h->st>>>(m, h->red.p + R_ALPHA, h->x.p, h->s.p, h->si.p, h->dx.p, h->ds.p);
            LRN_CHECK_LAUNCH();
            h->have_H = h->have_factor = false;
        }
        const dd a = read_slot(h, R_ALPHA), b = read_slot(h, R_BETA);
        alpha_lin[0] = a.hi; alpha_lin[1] = a.lo; beta_lin[0] = b.hi; beta_lin[1] = b.lo;
        return LRN_OK;
    });
}

int32_t lrn_dd_sigma_trace(lrn_dd_handle_t h, double dot_lin[2]) {
    LRN_GROUP(h, lrn_dd_sigma_trace(m_, r_ == 0 ? dot_lin : group_scratch().d));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(h->have_iterate && dot_lin, "no iterate");
        Timed t(h, 3);
        dot(h, h->nlin, h->xn.p, h->sn.p, R_DOT);
        const dd v = read_slot(h, R_DOT);
        dot_lin[0] = v.hi; dot_lin[1] = v.lo;
        return LRN_OK;
    });
}

int32_t lrn_dd_dimacs(lrn_dd_handle_t h, double err6[12], double by[2], double dx[2]) {
    LRN_GROUP(h, r_ == 0 ? lrn_dd_dimacs(m_, err6, by, dx)
                       : lrn_dd_dimacs(m_, group_scratch().d, group_scratch().d + 12, group_scratch().d + 14));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(h->have_iterate && err6 && by && dx, "no iterate");
        Timed t(h, 3);
        dot(h, h->n, h->b.p, h->y.p, R_BY);
        dot(h, h->nlin, h->d.p, h->x.p, R_DX);
        dot(h, h->n, h->rp.p, h->rp.p, R_RP2);
        dot(h, h->nlin, h->rd.p, h->rd.p, R_RD2);
        dot(h, h->nlin, h->s.p, h->x.p, R_SX);
        k_dd_min_ratio<<<1, 1024, 0, h->st>>>(h->nlin, h->x.p, nullptr, h->red.p, R_MINX); LRN_CHECK_LAUNCH();
        k_dd_min_ratio<<<1, 1024, 0, h->st>>>(h->nlin, h->s.p, nullptr, h->red.p, R_MINS); LRN_CHECK_LAUNCH();
        k_dd_dimacs<<<1, 1, 0, h->st>>>(h->red.p); LRN_CHECK_LAUNCH();
        dd r[R_COUNT];
        LRN_CUDA(cudaMemcpyAsync(r, h->red.p, sizeof r, cudaMemcpyDeviceToHost, h->st));
        LRN_CUDA(cudaStreamSynchronize(h->st));
        for (int k = 0; k < 6; k++) { err6[2 * k] = r[R_ERR + k].hi; err6[2 * k + 1] = r[R_ERR + k].lo; }
        by[0] = r[R_BY].hi; by[1] = r[R_BY].lo; dx[0] = r[R_DX].hi; dx[1] = r[R_DX].lo;
        return LRN_OK;
    });
}

int32_t lrn_dd_get_array(lrn_dd_handle_t h, int32_t which, double* hi, double* lo) {
    // H is a collective on a facade (every member contributes its row shard); everything else is replicated -> member 0
    if (h && h->group && which != 1) return lrn_dd_get_array(dd_member0(h), which, hi, lo);
    LRN_GROUP(h, lrn_dd_get_array(m_, which, r_ == 0 ? hi : nullptr, r_ == 0 ? lo : nullptr));
    return guarded(h, [&]() -> int32_t {
        // (a null output is allowed for H on a sharded handle: ranks other than the caller's only take part in the gather)
        LRN_REQUIRE(hi || (which == 1 && dd_sharded(h)), "null argument");
        const size_t n = (size_t)h->n, m = (size_t)h->nlin;
        switch (which) {
            case 1:
                LRN_REQUIRE(h->have_H, "no Schur matrix");
                if (h->nccl && !h->H_gathered) {
                    // every rank holds its own rows of the lower triangle, zeros elsewhere: the sum is exact
                    dd_gather_H(h);
                    k_dd_mirror_lower<<<dim3(nblk((long long)n), (unsigned)n), TB, 0, h->st>>>((int)n, h->H.p);
                    LRN_CHECK_LAUNCH();
                    h->H_gathered = true;
                }
                if (hi) download_dd(h, h->H.p, hi, lo, n * n);
                break;
            case 2: LRN_REQUIRE(h->have_factor, "no factor"); download_dd(h, h->L.p, hi, lo, n * n); break;
            case 3: download_dd(h, h->rp.p, hi, lo, n); break;
            case 4: download_dd(h, h->rd.p, hi, lo, m); break;
            case 5: download_dd(h, h->rhs.p, hi, lo, n); break;
            case 6: download_dd(h, h->dely.p, hi, lo, n); break;
            case 7: download_dd(h, h->dx.p, hi, lo, m); break;
            case 8: download_dd(h, h->ds.p, hi, lo, m); break;
            case 9: download_dd(h, h->xn.p, hi, lo, m); break;
            case 10: download_dd(h, h->sn.p, hi, lo, m); break;
            case 11: download_dd(h, h->rnt.p, hi, lo, m); break;
            case 12: download_dd(h, h->si.p, hi, lo, m); break;
            default: LRN_REQUIRE(false, "unknown array id");
        }
        return LRN_OK;
    });
}

int32_t lrn_dd_timers(lrn_dd_handle_t h, double ms[4], int32_t reset) {
    // a facade reports member 0's device times; a reset resets every member
    if (h && h->group && !reset) return lrn_dd_timers(dd_member0(h), ms, 0);
    LRN_GROUP(h, lrn_dd_timers(m_, r_ == 0 ? ms : group_scratch().d, reset));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(ms, "null argument");
        for (int k = 0; k < 4; k++) { ms[k] = h->t_ms[k]; if (reset) h->t_ms[k] = 0.0; }
        return LRN_OK;
    });
}

// ---- test hooks (loraine_b200_debug.h) -----------------------------------------------------------------------------------
int32_t lrn_dd_dbg_set_array(lrn_dd_handle_t h, int32_t which, const double* hi, const double* lo) {
    if (which != 1 && which != 5) return LRN_ERR_ARG;
    LRN_GROUP(h, lrn_dd_dbg_set_array(m_, which, hi, lo));
    return guarded(h, [&]() -> int32_t {
        LRN_REQUIRE(hi, "null argument");
        const int n = h->n;
        if (which == 5) {
            upload_dd(h, h->rhs, hi, lo, (size_t)n);
            return LRN_OK;
        }
        upload_dd(h, h->H, hi, lo, (size_t)n * n);
        if (dd_sharded(h)) {
            k_dd_keep_own_lower<<<dim3(nblk(n), (unsigned)n), TB, 0, h->st>>>(n, h->H.p, h->rank, h->world, h->pw);
            LRN_CHECK_LAUNCH();
            LRN_CUDA(cudaStreamSynchronize(h->st));
        }
        h->H_gathered = false;
        h->have_H = true;
        h->have_factor = false;
        return LRN_OK;
    });
}

int32_t lrn_dd_dbg_set_trsv_ctas(lrn_dd_handle_t h, int32_t ctas) {
    if (ctas < -1) return LRN_ERR_ARG;
    LRN_GROUP(h, lrn_dd_dbg_set_trsv_ctas(m_, ctas));
    if (!h) return LRN_ERR_ARG;
    h->trsv_ctas = ctas < 0 ? h->trsv_ctas_max : std::min(ctas, h->trsv_ctas_max);
    return LRN_OK;
}

}  // extern "C"
