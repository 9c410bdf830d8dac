// Ozaki-split INT8 trailing update of the blocked Cholesky (tcgen05.mma kind::i8, accumulators in tensor memory).
//
// The solved panel P (rows x K, K <= 1024) is sliced once per panel (i8_slice_kernel):
//     sigma_i = 2^e_i with max_k |P_ik| / sigma_i in [1/2, 255/256)   (0 for a zero row, NaN for a row holding a NaN or an Inf)
//     x = P_ik / sigma_i,  r_0 = x,  d_t = rint(2^7 r_{t-1}),  r_t = 2^7 r_{t-1} - d_t      t = 1..8  (every step exact in FP64)
// so |d_1| <= 127, |d_t| <= 64 for t >= 2, and |x - sum_t d_t 2^-7t| <= 2^-57.  The update C -= P_rows P_cols^T is then
//     C_l = sum_{a+b=l} sum_k dA_a dB_b        l = 2..9   (36 INT8 products, exact in INT32: |C_l| <= 8 * 1024 * 127^2 < 2^31)
//     acc = C_9;  acc = C_l + acc 2^-7 (l = 8..2);  C_out = C_in - (acc 2^-14) (sigma_i sigma_j)
// in that fixed order (tests/chol_i8_model.py reproduces it bit for bit).  DESIGN.md "Cholesky" has the error argument.
//
// Update kernel: one CTA per 128 x 64 output tile (lower-only tiles enumerated band by band), 10 warps:
//   warp 8      producer: 16 cp.async.bulk copies per stage (8 digit planes of the 128 A rows + 8 of the 64 B rows, 32 B of K)
//   warp 9      one thread issues the 36 digit-plane products of a stage as 12 tcgen05.mma (M = 128, N = 64 x up to 4 planes,
//               K = 32, S8 x S8 -> S32); tcgen05.commit frees the stage
//   warps 0..7  epilogue (two warps per TMEM lane quadrant, 32 columns each): load their part of the C tile during the main
//               loop, then fold the 8 level accumulators (8 x 64 TMEM columns = all 512) into it and write it back
// The slicing kernel writes every (plane, 32-wide K block) as rows_pad rows of 32 bytes in the canonical no-swizzle K-major
// layout of the MMA (core matrices of 8 rows x 16 B, the two K halves of an 8-row group 128 B apart), so a tile of any plane is
// one contiguous bulk copy and the shared-memory descriptors need LBO = 128 B (K direction), SBO = 256 B (8-row groups).
#include "chol.cuh"
#include "gemm.cuh"
#include <algorithm>

namespace lrn {
namespace {

constexpr int PL = 8;                          // digit planes
constexpr int BM = 128, BN = 64, BK = 32;      // output tile, K per stage (one MMA K step)
constexpr int ST = 4;                          // pipeline stages
constexpr int A_BYTES = BM * BK, B_BYTES = BN * BK;
constexpr int STAGE_BYTES = PL * (A_BYTES + B_BYTES);      // 48 KB
constexpr int GN = 32;                         // tile columns per band (B rows of a band stay in L2 while A tiles stream)
constexpr size_t UPD_SMEM = (size_t)ST * STAGE_BYTES + 128 + BN * sizeof(double);   // stages, barriers, column scales
constexpr uint32_t TMEM_COLS = 512;

// ---- slicing ------------------------------------------------------------------------------------------------------------
// block = 32 rows x 8 K-parts; part p takes the 32-wide K blocks p, p + 8, ...
__global__ void __launch_bounds__(256)
    i8_slice_kernel(const double* __restrict__ P, int ldp, int rows, int K, int KB, int rows_pad, int8_t* __restrict__ slices,
                    double* __restrict__ sigma) {
    __shared__ double smax[8][32];
    __shared__ int sbad[8][32];
    const int r = threadIdx.x & 31, part = threadIdx.x >> 5;
    const int i = blockIdx.x * 32 + r;
    double m = 0.0;
    int bad = 0;
    if (i < rows) {
        for (int kb = part; kb < KB; kb += 8) {
            const int k0 = kb * BK, k1 = min(K, k0 + BK);
#pragma unroll 8
            for (int k = k0; k < k1; k++) {
                const double v = fabs(P[i + (size_t)k * ldp]);
                bad |= !(v <= 1.7976931348623157e308);
                m = fmax(m, v);
            }
        }
    }
    smax[part][r] = m;
    sbad[part][r] = bad;
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 8; q++) { m = fmax(m, smax[q][r]); bad |= sbad[q][r]; }
    double s;
    if (bad) s = __longlong_as_double(0x7ff8000000000000LL);
    else if (m == 0.0) s = 0.0;
    else {
        int e;
        const double f = frexp(m, &e);                 // m = f 2^e, f in [1/2, 1)
        s = ldexp(1.0, f < 0x1.fep-1 ? e : e + 1);     // keeps 2^7 max|x| below 127.5, so |d_1| <= 127
    }
    if (part == 0 && i < rows_pad) sigma[i] = s;
    const bool live = i < rows && s > 0.0;             // zero and NaN rows get zero digits
    for (int kb = part; kb < KB; kb += 8) {
#pragma unroll
        for (int kc = 0; kc < 2; kc++) {
            uint32_t w[PL][4];
#pragma unroll
            for (int t = 0; t < PL; t++)
#pragma unroll
                for (int q = 0; q < 4; q++) w[t][q] = 0u;
#pragma unroll
            for (int u = 0; u < 16; u++) {
                const int k = kb * BK + kc * 16 + u;
                const double v = (live && k < K) ? P[i + (size_t)k * ldp] : 0.0;
                double rr = v / s;
                if (!live) rr = 0.0;
#pragma unroll
                for (int t = 0; t < PL; t++) {
                    const double y = __dmul_rn(rr, 128.0);
                    const double d = rint(y);
                    rr = __dsub_rn(y, d);
                    w[t][u >> 2] |= ((uint32_t)(int)d & 0xffu) << (8 * (u & 3));
                }
            }
            if (i < rows_pad) {
#pragma unroll
                for (int t = 0; t < PL; t++) {
                    int8_t* dst = slices + (((size_t)t * KB + kb) * rows_pad + (i & ~7)) * BK + kc * 128 + (i & 7) * 16;
                    *reinterpret_cast<uint4*>(dst) = make_uint4(w[t][0], w[t][1], w[t][2], w[t][3]);
                }
            }
        }
    }
}

// ---- tcgen05 / mbarrier helpers --------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "LAB_WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra LAB_DONE_%=;\n"
        "bra LAB_WAIT_%=;\n"
        "LAB_DONE_%=:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// shared-memory matrix descriptor: no swizzle, K-major, LBO = 128 B (next 16 B of K), SBO = 256 B (next 8 rows), version 1
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr) {
    return (uint64_t)((addr & 0x3FFFFu) >> 4) | ((uint64_t)(128 >> 4) << 16) | ((uint64_t)(256 >> 4) << 32) | (1ull << 46);
}
// instruction descriptor: D S32, A and B signed 8-bit, both K-major, M = 128, N = 64 * nplanes
__host__ __device__ constexpr uint32_t idesc(int nplanes) {
    return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN * nplanes >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}

__device__ __forceinline__ void mma_i8(uint32_t d_tmem, uint64_t a, uint64_t b, uint32_t id, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(d_tmem), "l"(a), "l"(b), "r"(id), "r"(accumulate));
}
__device__ __forceinline__ void mma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&v)[8]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];\n"
        "tcgen05.wait::ld.sync.aligned;\n"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
        : "r"(taddr)
        : "memory");
}

struct UpdParams {
    const int8_t* slices;
    const double* sigma;
    double* C;
    long long ldc;
    int rows_pad, KB, a_row0, b_row0, M, N, Mt, Nt;
    long long row0, col0;
    int lower;
};

// t-th computed tile: bands of GN tile columns; inside a band the tile rows that lie wholly above the diagonal for every column
// of the band are left out, the rest are taken row by row (consecutive CTAs share the A tile, the band's B rows stay in L2)
__host__ __device__ __forceinline__ bool tile_of(long long t, const UpdParams& p, int& bm, int& bn) {
    for (int b0 = 0; b0 < p.Nt; b0 += GN) {
        const int gw = p.Nt - b0 < GN ? p.Nt - b0 : GN;
        int lo = 0;
        if (p.lower) {
            const long long need = p.col0 + (long long)b0 * BN - p.row0 - (BM - 1);
            if (need > 0) lo = (need + BM - 1) / BM < p.Mt ? (int)((need + BM - 1) / BM) : p.Mt;
        }
        const long long cnt = (long long)(p.Mt - lo) * gw;
        if (t < cnt) { bm = lo + (int)(t / gw); bn = b0 + (int)(t % gw); return true; }
        t -= cnt;
    }
    return false;
}

__global__ void __launch_bounds__(320, 1) i8_update_kernel(const UpdParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    int bm, bn;
    if (!tile_of(blockIdx.x, p, bm, bn)) return;
    const int m0 = bm * BM, n0 = bn * BN;
    if (p.lower && p.row0 + m0 + BM - 1 < p.col0 + n0) return;          // wholly above the diagonal
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(smem);
    const uint32_t bars = sbase + (uint32_t)(ST * STAGE_BYTES);            // full[ST], empty[ST], accum, tmem address slot
    const uint32_t accbar = bars + 16 * ST;
    uint32_t* tslot = reinterpret_cast<uint32_t*>(smem + ST * STAGE_BYTES + 16 * ST + 8);
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(sbase + (uint32_t)(ST * STAGE_BYTES + 16 * ST + 8)),
                     "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 32) {
        for (int s = 0; s < ST; s++) { mbar_init(bars + 8 * s, 1); mbar_init(bars + 8 * (ST + s), 1); }
        mbar_init(accbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tslot;
    const int KT = p.KB;

    if (warp == 8) {
        // ---- producer -------------------------------------------------------------------------------------------------------
        const size_t plane = (size_t)p.KB * p.rows_pad * BK;
        const int8_t* Ag = p.slices + (size_t)(p.a_row0 + m0) * BK;
        const int8_t* Bg = p.slices + (size_t)(p.b_row0 + n0) * BK;
        for (int kt = 0; kt < KT; kt++) {
            const int s = kt % ST;
            mbar_wait(bars + 8 * (ST + s), ((kt / ST) & 1) ^ 1);
            if (lane == 0) mbar_expect_tx(bars + 8 * s, (uint32_t)STAGE_BYTES);
            __syncwarp();
            const uint32_t st0 = sbase + (uint32_t)(s * STAGE_BYTES);
            const size_t koff = (size_t)kt * p.rows_pad * BK;
            if (lane < PL) bulk_g2s(st0 + lane * A_BYTES, Ag + lane * plane + koff, A_BYTES, bars + 8 * s);
            else if (lane < 2 * PL) bulk_g2s(st0 + PL * A_BYTES + (lane - PL) * B_BYTES, Bg + (lane - PL) * plane + koff, B_BYTES, bars + 8 * s);
        }
    } else if (warp == 9) {
        // ---- MMA issue: accumulator a + b (level a + b + 2) += plane a of the A rows x plane b of the B rows, a + b <= 7.  The B
        // planes of a stage and the accumulators are both contiguous, so planes b .. b + 3 stacked along N (N = 256) feed the
        // accumulators a + b .. a + b + 3 in one MMA: 12 MMAs per stage, each A tile read from shared memory once per 256 columns
        if (lane == 0) {
            for (int kt = 0; kt < KT; kt++) {
                const int s = kt % ST;
                mbar_wait(bars + 8 * s, (kt / ST) & 1);
                tc_fence_after();
                const uint32_t st0 = sbase + (uint32_t)(s * STAGE_BYTES);
#pragma unroll
                for (int a = 0; a < PL; a++) {
                    const uint64_t da = smem_desc(st0 + a * A_BYTES);
#pragma unroll
                    for (int b = 0; a + b < PL; b += 4) {
                        const int np = PL - a - b < 4 ? PL - a - b : 4;
                        mma_i8(tmem + (uint32_t)((a + b) * BN), da, smem_desc(st0 + PL * A_BYTES + b * B_BYTES), idesc(np),
                               (kt > 0 || a > 0) ? 1u : 0u);
                    }
                }
                mma_commit(bars + 8 * (ST + s));                             // stage s may be refilled once these MMAs are done
            }
            mma_commit(accbar);
        }
        __syncwarp();
    } else {
        // ---- epilogue: thread = one row of the tile (TMEM lane 32 (warp % 4) + lane) and one half of its 64 columns.  The C
        // values and the column scales are read while the MMAs run (no other launch writes this tile meanwhile), so the fold
        // waits on no global load -------------------------------------------------------------------------------------------------
        constexpr int EC = BN / 2;                                           // columns per epilogue thread
        const int q = warp & 3, h = warp >> 2, row = m0 + q * 32 + lane;
        double* sgj = reinterpret_cast<double*>(smem + ST * STAGE_BYTES + 128);
        if (tid < BN) sgj[tid] = n0 + tid < p.N ? p.sigma[p.b_row0 + n0 + tid] : 0.0;
        const double si = p.sigma[p.a_row0 + row];
        double cv[EC];
        double* crow = p.C + (size_t)(n0 + h * EC) * p.ldc + row;
        int ncol = p.N - n0 - h * EC;
        ncol = ncol < 0 ? 0 : (ncol < EC ? ncol : EC);
        const bool live = row < p.M;
#pragma unroll
        for (int j = 0; j < EC; j++) cv[j] = (live && j < ncol) ? crow[(size_t)j * p.ldc] : 0.0;
        asm volatile("bar.sync 1, 256;" ::: "memory");                    // the eight epilogue warps: sgj is complete
        mbar_wait(accbar, 0);
        tc_fence_after();
        const uint32_t trow = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(h * EC);
#pragma unroll
        for (int c = 0; c < EC / 8; c++) {
            double acc[8];
            uint32_t v[8];
            tmem_ld8(trow + (uint32_t)(7 * BN + c * 8), v);
#pragma unroll
            for (int j = 0; j < 8; j++) acc[j] = (double)(int)v[j];
#pragma unroll 1
            for (int l = 6; l >= 0; l--) {
                tmem_ld8(trow + (uint32_t)(l * BN + c * 8), v);
#pragma unroll
                for (int j = 0; j < 8; j++) acc[j] = __dadd_rn((double)(int)v[j], __dmul_rn(acc[j], 0x1p-7));
            }
#pragma unroll
            for (int j = 0; j < 8; j++)
                cv[c * 8 + j] = __dsub_rn(cv[c * 8 + j], __dmul_rn(__dmul_rn(acc[j], 0x1p-14), __dmul_rn(si, sgj[h * EC + c * 8 + j])));
        }
        if (live) {
#pragma unroll
            for (int j = 0; j < EC; j++)
                if (j < ncol) crow[(size_t)j * p.ldc] = cv[j];
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(TMEM_COLS) : "memory");
    }
}

}  // namespace

size_t i8_slice_bytes(int rows_pad, int K) { return (size_t)PL * cdiv(K, BK) * rows_pad * BK; }

void i8_slice(const double* P, int ldp, int rows, int K, int rows_pad, int8_t* slices, double* sigma, cudaStream_t st) {
    LRN_REQUIRE(K >= 1 && K <= 1024, "INT8 Ozaki slicing takes 1 <= K <= 1024 (the level sums are exact in INT32 up to K = 1024)");
    LRN_REQUIRE(rows >= 0 && rows_pad >= rows && rows_pad % 8 == 0, "slices: rows_pad");
    const int KB = (int)cdiv(K, BK);
    i8_slice_kernel<<<(unsigned)cdiv(rows_pad, 32), 256, 0, st>>>(P, ldp, rows, K, KB, rows_pad, slices, sigma);
    LRN_CHECK_LAUNCH();
}

void syrk_update_i8(const int8_t* slices, const double* sigma, int rows_pad, int K, int a_row0, int b_row0, int M, int N, double* C,
                    int ldc, long long row0, long long col0, bool lower, cudaStream_t st) {
    if (M <= 0 || N <= 0) return;
    LRN_REQUIRE(K >= 1 && K <= 1024, "INT8 Ozaki update takes 1 <= K <= 1024");
    LRN_REQUIRE(a_row0 % 8 == 0 && b_row0 % 8 == 0, "slice row offsets must be multiples of 8");
    LRN_REQUIRE(a_row0 + cdiv(M, BM) * BM <= rows_pad && b_row0 + cdiv(N, BN) * BN <= rows_pad, "slices have too few padded rows");
    static PerDeviceOnce once;
    once.run([&] { LRN_CUDA(cudaFuncSetAttribute(i8_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)UPD_SMEM)); });
    UpdParams p;
    p.slices = slices; p.sigma = sigma; p.C = C; p.ldc = ldc;
    p.rows_pad = rows_pad; p.KB = (int)cdiv(K, BK); p.a_row0 = a_row0; p.b_row0 = b_row0; p.M = M; p.N = N;
    p.Mt = (int)cdiv(M, BM); p.Nt = (int)cdiv(N, BN); p.row0 = row0; p.col0 = col0; p.lower = lower ? 1 : 0;
    long long tiles = 0;                                                   // the tiles tile_of enumerates
    for (int b0 = 0; b0 < p.Nt; b0 += GN) {
        int bm = 0, bn = 0;
        if (!tile_of(tiles, p, bm, bn)) break;
        tiles += (long long)(p.Mt - bm) * std::min(GN, p.Nt - b0);
    }
    if (tiles == 0) return;
    LRN_REQUIRE(tiles < (1LL << 31), "too many tiles");
    cudaEvent_t ev = nullptr;
    const bool prof = gemm_prof_begin(st, ev);
    i8_update_kernel<<<(unsigned)tiles, 320, UPD_SMEM, st>>>(p);
    LRN_CHECK_LAUNCH();
    if (prof) gemm_prof_end(ev, st, 2.0 * M * (double)N * K * (lower ? 0.5 : 1.0), 3);
}

}  // namespace lrn
