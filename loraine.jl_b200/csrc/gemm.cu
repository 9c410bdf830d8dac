// FP64 DMMA GEMM (mma.sync.m8n8k4.f64 -> SASS DMMA.8x8x4, the native FP64 tensor shape on sm_100a), cp.async multi-stage
// shared-memory pipeline with padded, bank-conflict-free operand tiles.
//
// Tile shapes:  L = 128x128x16, 8 warps (2x4, warp tile 64x32)   -- large problems, 1 CTA/SM
//               S =  64x 64x16, 4 warps (2x2, warp tile 32x32)   -- small/medium problems, several CTAs/SM
// Operand tiles in shared memory are stored along their global-memory contiguous dimension so that every copy is a
// 16-byte cp.async (8-byte when the caller's pointers/leading dimensions are not 16 B aligned):
//   "MN-major" tile  [BK][BMN+4]   (operand contiguous along M or N)   fragment read  [k][r] : (k*(BMN+4)+r)  mod 16 distinct
//   "K-major"  tile  [BMN][BK+4]   (operand contiguous along K)        fragment read  [r][k] : (r*20+k)       mod 16 distinct
// so each half-warp LDS.64 fragment load touches 16 distinct 8-byte bank pairs (no conflicts).
#include "gemm.cuh"
#include <atomic>

namespace lrn {

namespace {


__device__ __forceinline__ void cp_async16(void* smem, const void* gmem, int src_bytes) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async8(void* smem, const void* gmem, int src_bytes) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(s), "l"(gmem), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// Load one operand tile (BMN x BK of op(X)) into shared memory.
//   CONTIG_MN = true : global element (r,k) at X[r + k*ld]  -> smem [k][r] with row stride BMN+4
//   CONTIG_MN = false: global element (r,k) at X[k + r*ld]  -> smem [r][k] with row stride BK+4
template <int BMN, int BK, int NT, bool CONTIG_MN, bool ALIGN16>
__device__ __forceinline__ void load_tile(double* __restrict__ s, const double* __restrict__ X, int ld, int r0, int k0,
                                          int R, int K, int tid) {
    if (CONTIG_MN) {
        if (ALIGN16) {
            constexpr int CH = BMN / 2;              // 16 B chunks per k-line
            constexpr int TOT = BK * CH;
#pragma unroll
            for (int c = tid; c < TOT; c += NT) {
                int k = c / CH, rc = (c % CH) * 2;
                int gr = r0 + rc, gk = k0 + k;
                int bytes = (gk < K) ? min(max((R - gr) * 8, 0), 16) : 0;
                const double* g = bytes ? (X + (size_t)gk * ld + gr) : X;
                cp_async16(s + k * (BMN + 4) + rc, g, bytes);
            }
        } else {
            constexpr int TOT = BK * BMN;
#pragma unroll
            for (int c = tid; c < TOT; c += NT) {
                int k = c / BMN, rc = c % BMN;
                int gr = r0 + rc, gk = k0 + k;
                int bytes = (gk < K && gr < R) ? 8 : 0;
                const double* g = bytes ? (X + (size_t)gk * ld + gr) : X;
                cp_async8(s + k * (BMN + 4) + rc, g, bytes);
            }
        }
    } else {
        if (ALIGN16) {
            constexpr int CH = BK / 2;
            constexpr int TOT = BMN * CH;
#pragma unroll
            for (int c = tid; c < TOT; c += NT) {
                int r = c / CH, kc = (c % CH) * 2;
                int gr = r0 + r, gk = k0 + kc;
                int bytes = (gr < R) ? min(max((K - gk) * 8, 0), 16) : 0;
                const double* g = bytes ? (X + (size_t)gr * ld + gk) : X;
                cp_async16(s + r * (BK + 4) + kc, g, bytes);
            }
        } else {
            constexpr int TOT = BMN * BK;
#pragma unroll
            for (int c = tid; c < TOT; c += NT) {
                int r = c / BK, kc = c % BK;
                int gr = r0 + r, gk = k0 + kc;
                int bytes = (gr < R && gk < K) ? 8 : 0;
                const double* g = bytes ? (X + (size_t)gr * ld + gk) : X;
                cp_async8(s + r * (BK + 4) + kc, g, bytes);
            }
        }
    }
}

template <int BM, int BN, int BK, int STAGES>
struct TileSmem {
    static constexpr int cmax(int a, int b) { return a > b ? a : b; }
    static constexpr int A_ELEMS = cmax(BM * (BK + 4), BK * (BM + 4));
    static constexpr int B_ELEMS = cmax(BN * (BK + 4), BK * (BN + 4));
    static constexpr int STAGE_ELEMS = A_ELEMS + B_ELEMS;
    static constexpr size_t BYTES = (size_t)STAGES * STAGE_ELEMS * sizeof(double);
};

template <int BM, int BN, int BK, int STAGES, int WARPS_M, int WARPS_N, bool TA, bool TB, bool ALIGN16>
__global__ void __launch_bounds__(WARPS_M* WARPS_N * 32)
    dgemm_dmma_kernel(const GemmParams p) {
    constexpr int NT = WARPS_M * WARPS_N * 32;
    constexpr int WM = BM / WARPS_M, WN = BN / WARPS_N;
    constexpr int MI = WM / 8, NI = WN / 8;
    using SM = TileSmem<BM, BN, BK, STAGES>;
    extern __shared__ __align__(16) double smem[];

    const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
    const int z = blockIdx.z;
    const int z1 = z / p.batch2, z2 = z - z1 * p.batch2;
    if (p.lower && (p.row0 + (long long)z1 * p.row0z + m0 + BM - 1 < p.col0 + n0)) return;
    const double* __restrict__ A = p.A + (size_t)z1 * p.sA + (size_t)z2 * p.sA2;
    const double* __restrict__ B = p.B + (size_t)z1 * p.sB + (size_t)z2 * p.sB2;
    double* __restrict__ C = p.cblkmap ? p.C : p.C + (size_t)z1 * p.sC + (size_t)z2 * p.sC2;
    const int Kz = (p.K_last > 0 && z2 == p.batch2 - 1) ? p.K_last : p.K;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm0 = (warp / WARPS_N) * WM, wn0 = (warp % WARPS_N) * WN;
    const int lr = lane >> 2, lk = lane & 3;

    double acc[MI][NI][2];
#pragma unroll
    for (int i = 0; i < MI; i++)
#pragma unroll
        for (int j = 0; j < NI; j++) acc[i][j][0] = acc[i][j][1] = 0.0;

    const int KT = (Kz + BK - 1) / BK;
    const int kt0 = p.ktri ? max(m0, n0) / BK : 0;
    auto issue = [&](int kt) {
        double* sA = smem + (size_t)((kt - kt0) % STAGES) * SM::STAGE_ELEMS;
        double* sB = sA + SM::A_ELEMS;
        // op(A) is M x K: !TA -> contiguous along M; TA -> contiguous along K
        load_tile<BM, BK, NT, !TA, ALIGN16>(sA, A, p.lda, m0, kt * BK, p.M, Kz, tid);
        // op(B) is K x N: !TB -> contiguous along K; TB -> contiguous along N
        load_tile<BN, BK, NT, TB, ALIGN16>(sB, B, p.ldb, n0, kt * BK, p.N, Kz, tid);
    };

#pragma unroll
    for (int s = 0; s < STAGES - 1; s++) {
        if (kt0 + s < KT) issue(kt0 + s);
        cp_async_commit();
    }
    for (int kt = kt0; kt < KT; kt++) {
        cp_async_wait<STAGES - 2>();
        __syncthreads();
        if (kt + STAGES - 1 < KT) issue(kt + STAGES - 1);
        cp_async_commit();
        const double* sA = smem + (size_t)((kt - kt0) % STAGES) * SM::STAGE_ELEMS;
        const double* sB = sA + SM::A_ELEMS;
#pragma unroll
        for (int kk = 0; kk < BK; kk += 4) {
            double a[MI], b[NI];
#pragma unroll
            for (int i = 0; i < MI; i++) {
                int r = wm0 + i * 8 + lr;
                a[i] = TA ? sA[r * (BK + 4) + kk + lk] : sA[(kk + lk) * (BM + 4) + r];
            }
#pragma unroll
            for (int j = 0; j < NI; j++) {
                int c = wn0 + j * 8 + lr;
                b[j] = TB ? sB[(kk + lk) * (BN + 4) + c] : sB[c * (BK + 4) + kk + lk];
            }
#pragma unroll
            for (int i = 0; i < MI; i++)
#pragma unroll
                for (int j = 0; j < NI; j++) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
        }
    }
    cp_async_wait<0>();

    const double* cs = p.colscale ? p.colscale + (size_t)z1 * p.sScale : nullptr;
    const double alpha = p.alpha, beta = p.beta;
#pragma unroll
    for (int j = 0; j < NI; j++) {
#pragma unroll
        for (int t = 0; t < 2; t++) {
            int col = n0 + wn0 + j * 8 + lk * 2 + t;
            if (col >= p.N) continue;
            double sc = cs ? cs[col] : 1.0;
            int dcol = col;
            if (p.cblkmap) dcol = p.cblkmap[z1 * (p.N >> 5) + (col >> 5)] * 32 + (col & 31);
#pragma unroll
            for (int i = 0; i < MI; i++) {
                int row = m0 + wm0 + i * 8 + lr;
                if (row >= p.M) continue;
                double v = acc[i][j][t] * sc;
                double* cp = C + (size_t)dcol * p.ldc + row;
                if (p.mode == 1) v = v * v;
                v *= alpha;
                if (beta != 0.0) v += beta * (*cp);
                *cp = v;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// TMA-fed variant for the large products (Schur SYRK with squared epilogue, Cholesky trailing update, the m x m congruences):
// with an MN-major operand one k-line of a 128-wide tile is a contiguous 1 KB segment in global memory (a K-major B operand
// is moved as 128 segments of 256 B).
// A dedicated producer warp moves those segments with the bulk-copy engine (cp.async.bulk -> SASS UBLKCP) into the padded
// shared-memory rows and signals mbarriers; the 8 consumer warps never touch a load instruction or a block barrier in the
// main loop.  Full 128 x 128 tiles only (the host sends edge strips to the cp.async kernel), K % 32 == 0.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int BKB = 32, STB = 3, LDT = 128 + 4, LDK = BKB + 4;
constexpr int BULK_A_ELEMS = BKB * LDT;                      // A tile: [k][128 + 4]
constexpr int BULK_B_ELEMS = 128 * LDK;                      // B tile: [k][128 + 4] (A B^T) or [n][32 + 4] (A B); the larger one
constexpr int BULK_STAGE_ELEMS = BULK_A_ELEMS + BULK_B_ELEMS;
constexpr size_t BULK_SMEM = (size_t)STB * BULK_STAGE_ELEMS * sizeof(double) + 64;

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
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

// TB = true : C (+)= f(A B^T), B is N x K stored N-major (k-lines of 1 KB, like A)
// TB = false: C (+)= A B,       B is K x N column-major: one 256 B segment (32 k) per column of the tile, stored [n][32 + 4]
template <bool TB>
__global__ void __launch_bounds__(288, 1) dgemm_dmma_bulk_kernel(const GemmParams p) {
    extern __shared__ __align__(16) double smem[];
    const int m0 = blockIdx.x * 128, n0 = blockIdx.y * 128;
    const int z = blockIdx.z;                  // strided batch (row blocks of a block-cyclic distribution)
    if (p.lower && (p.row0 + (long long)z * p.row0z + m0 + 127 < p.col0 + n0)) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(smem);
    const uint32_t bars = sbase + (uint32_t)(STB * BULK_STAGE_ELEMS * sizeof(double));     // full[0..2], empty[0..2]
    if (tid == 0) {
        for (int s = 0; s < STB; s++) { mbar_init(bars + 8 * s, 1); mbar_init(bars + 8 * (STB + s), 8); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const int KT = p.K / BKB;
    if (warp == 8) {
        // ---- producer warp: lane l moves k-line l of the A tile and of the B tile -----------------------------------
        const double* Ag = p.A + (size_t)z * p.sA + m0;
        const double* Bg = (TB ? p.B + n0 : p.B + (size_t)n0 * p.ldb) + (size_t)z * p.sB;
        auto prefetch_c = [&]() {
            // pull the 128 x 128 tile of C (read-modify-write epilogue, beta != 0) towards L2 while the main loop runs, so that
            // the epilogue's reads do not wait on HBM: 128 columns x 8 lines of 128 B
            const char* Cg = reinterpret_cast<const char*>(p.C + (size_t)z * p.sC + (size_t)n0 * p.ldc + m0);
#pragma unroll 4
            for (int col = lane; col < 128; col += 32) {
                const char* cp = Cg + (size_t)col * p.ldc * sizeof(double);
#pragma unroll
                for (int q = 0; q < 8; q++) asm volatile("prefetch.global.L2 [%0];" ::"l"(cp + q * 128));
            }
        };
        for (int kt = 0; kt < KT; kt++) {
            if (p.beta != 0.0 && kt == (KT > STB ? STB : 0)) prefetch_c();   // after the pipeline is primed
            const int s = kt % STB;
            mbar_wait(bars + 8 * (STB + s), ((kt / STB) & 1) ^ 1);
            if (lane == 0) mbar_expect_tx(bars + 8 * s, 2u * BKB * 128u * 8u);
            __syncwarp();
            const uint32_t st0 = sbase + (uint32_t)(s * BULK_STAGE_ELEMS * sizeof(double));
            const uint32_t sa = st0 + (uint32_t)(lane * LDT * sizeof(double));
            const size_t k = (size_t)kt * BKB + lane;
            bulk_g2s(sa, Ag + k * p.lda, 128u * 8u, bars + 8 * s);
            if (TB) {
                const uint32_t sb = st0 + (uint32_t)((BULK_A_ELEMS + lane * LDT) * sizeof(double));
                bulk_g2s(sb, Bg + k * p.ldb, 128u * 8u, bars + 8 * s);
            } else {
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    const int n = lane + 32 * q;
                    const uint32_t sb = st0 + (uint32_t)((BULK_A_ELEMS + n * LDK) * sizeof(double));
                    bulk_g2s(sb, Bg + (size_t)n * p.ldb + (size_t)kt * BKB, BKB * 8u, bars + 8 * s);
                }
            }
        }
        return;
    }
    // ---- consumer warps: 2 x 4 layout, warp tile 64 x 32 (identical fragment code to the cp.async kernel) -------------
    const int wm0 = (warp / 4) * 64, wn0 = (warp % 4) * 32;
    const int lr = lane >> 2, lk = lane & 3;
    double acc[8][4][2];
#pragma unroll
    for (int i = 0; i < 8; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) acc[i][j][0] = acc[i][j][1] = 0.0;
    for (int kt = 0; kt < KT; kt++) {
        const int s = kt % STB;
        mbar_wait(bars + 8 * s, (kt / STB) & 1);
        const double* sA = smem + (size_t)s * BULK_STAGE_ELEMS;
        const double* sB = sA + BULK_A_ELEMS;
#pragma unroll
        for (int kk = 0; kk < BKB; kk += 4) {
            double a[8], b[4];
#pragma unroll
            for (int i = 0; i < 8; i++) a[i] = sA[(kk + lk) * LDT + wm0 + i * 8 + lr];
#pragma unroll
            for (int j = 0; j < 4; j++) b[j] = TB ? sB[(kk + lk) * LDT + wn0 + j * 8 + lr] : sB[(wn0 + j * 8 + lr) * LDK + kk + lk];
#pragma unroll
            for (int i = 0; i < 8; i++)
#pragma unroll
                for (int j = 0; j < 4; j++) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(bars + 8 * (STB + s));
    }
    const double alpha = p.alpha, beta = p.beta;
    double* __restrict__ Cz = p.C + (size_t)z * p.sC;
#pragma unroll
    for (int j = 0; j < 4; j++) {
#pragma unroll
        for (int t = 0; t < 2; t++) {
            const int col = n0 + wn0 + j * 8 + lk * 2 + t;
#pragma unroll
            for (int i = 0; i < 8; i++) {
                const int row = m0 + wm0 + i * 8 + lr;
                double v = acc[i][j][t];
                double* cp = Cz + (size_t)col * p.ldc + row;
                if (p.mode == 1) v = v * v;
                v *= alpha;
                if (beta != 0.0) v += beta * (*cp);
                *cp = v;
            }
        }
    }
}


// ---------------------------------------------------------------------------------------------------------------------
// Panel rotation of the block-Jacobi SVD:  nxt[:, slot(2z), slot(2z+1)] = cur[:, 64z .. 64z+63] * J_z  for every pair z.
// Persistent CTAs walk a flattened (pair, 128-row tile) list.  The 64 x 64 rotation J_z stays resident in shared memory
// while the producer warp streams the 128 x 64 panel tiles through a two-stage bulk-copy (TMA) ring; the eight consumer
// warps (4 x 2, warp tile 32 x 32) run 256 DMMAs per tile and scatter the rotated columns straight from registers to the
// slots the round-robin ordering assigns them in the next round.  Rows are padded to whole tiles (zero rows stay zero).
// ---------------------------------------------------------------------------------------------------------------------
constexpr int PR_LDA = 128 + 4, PR_LDJ = 64 + 4, PR_ST = 2;
constexpr int PR_A_ELEMS = 64 * PR_LDA, PR_J_ELEMS = 64 * PR_LDJ, PR_STAGE_ELEMS = PR_A_ELEMS + PR_J_ELEMS;
constexpr size_t PR_SMEM = (size_t)PR_ST * PR_STAGE_ELEMS * sizeof(double) + 64;

__global__ void __launch_bounds__(288) panel_rotate_kernel(const PanelRotateParams p) {
    extern __shared__ __align__(16) double smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(smem);
    const uint32_t bars = sbase + (uint32_t)(PR_ST * PR_STAGE_ELEMS * sizeof(double));   // full[s] = bars + 8 s, empty[s] after them
    if (tid == 0) {
        for (int s = 0; s < PR_ST; s++) { mbar_init(bars + 8 * s, 1); mbar_init(bars + 8 * (PR_ST + s), 8); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    // tasks are dealt round-robin (task t -> CTA t mod grid); every stage carries its own copy of the pair's rotation, so a
    // CTA may move from pair to pair freely (the 32 KB rotations come from L2).  Walking the pairs in opposite directions in
    // consecutive kernels to catch the tail of the 200 MB work matrix in L2 was measured: no gain (within 1 %).
    const long long G = gridDim.x;
    if (warp == 8) {
        int i = 0;
        for (long long t = blockIdx.x; t < p.total; t += G, i++) {
            const int z = (int)(t / p.tiles), tile = (int)(t - (long long)z * p.tiles);
            const int s = i % PR_ST;
            mbar_wait(bars + 8 * (PR_ST + s), ((i / PR_ST) & 1) ^ 1);
            if (lane == 0) mbar_expect_tx(bars + 8 * s, 64u * 128u * 8u + 64u * 64u * 8u);
            __syncwarp();
            const double* Ag = p.cur + (size_t)z * 64 * p.ldw + (size_t)tile * 128;
            const double* Jg = p.rot + (size_t)z * 4096;
            const uint32_t sa = sbase + (uint32_t)(s * PR_STAGE_ELEMS * sizeof(double));
            const uint32_t sj = sa + (uint32_t)(PR_A_ELEMS * sizeof(double));
            for (int l = lane; l < 64; l += 32) {
                bulk_g2s(sa + (uint32_t)(l * PR_LDA * sizeof(double)), Ag + (size_t)l * p.ldw, 128u * 8u, bars + 8 * s);
                bulk_g2s(sj + (uint32_t)(l * PR_LDJ * sizeof(double)), Jg + l * 64, 64u * 8u, bars + 8 * s);
            }
        }
        return;
    }
    const int wm0 = (warp >> 1) * 32, wn0 = (warp & 1) * 32;
    const int lr = lane >> 2, lk = lane & 3;
    int i = 0;
    for (long long t = blockIdx.x; t < p.total; t += G, i++) {
        const int z = (int)(t / p.tiles), tile = (int)(t - (long long)z * p.tiles);
        const int s = i % PR_ST;
        mbar_wait(bars + 8 * s, (i / PR_ST) & 1);
        const double* sA = smem + (size_t)s * PR_STAGE_ELEMS;
        const double* sJ = sA + PR_A_ELEMS;
        double acc[4][4][2];
#pragma unroll
        for (int a = 0; a < 4; a++)
#pragma unroll
            for (int b = 0; b < 4; b++) acc[a][b][0] = acc[a][b][1] = 0.0;
#pragma unroll 4
        for (int kk = 0; kk < 64; kk += 4) {
            double a[4], b[4];
#pragma unroll
            for (int q = 0; q < 4; q++) a[q] = sA[(kk + lk) * PR_LDA + wm0 + q * 8 + lr];
#pragma unroll
            for (int q = 0; q < 4; q++) b[q] = sJ[(wn0 + q * 8 + lr) * PR_LDJ + kk + lk];
#pragma unroll
            for (int a_ = 0; a_ < 4; a_++)
#pragma unroll
                for (int b_ = 0; b_ < 4; b_++) dmma884(acc[a_][b_][0], acc[a_][b_][1], a[a_], b[b_]);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(bars + 8 * (PR_ST + s));
        // both 32-column halves of the pair go to their own slot of the next arrangement
        const int slot = p.slotmap[2 * z + (warp & 1)];
        double* Cz = p.nxt + (size_t)slot * 32 * p.ldw + (size_t)tile * 128 + wm0 + lr;
#pragma unroll
        for (int b_ = 0; b_ < 4; b_++)
#pragma unroll
            for (int u = 0; u < 2; u++) {
                double* cc = Cz + (size_t)(b_ * 8 + lk * 2 + u) * p.ldw;
#pragma unroll
                for (int a_ = 0; a_ < 4; a_++) cc[a_ * 8] = acc[a_][b_][u];
            }
    }
}

std::atomic<long long> g_launches{0};

// optional per-launch profiling (bench roofline): CUDA events around every DMMA GEMM launch on its own stream
// fam: 0 cp.async kernel, 1 TMA-fed kernel, 2 panel rotation, 3 INT8 Ozaki update (chol_i8.cu; not a DMMA kernel)
struct ProfRec { cudaEvent_t a, b; double flops; int fam = 0; };
constexpr int NFAM = 4, NFAM_DMMA = 3;
double g_fam_ms[NFAM] = {}, g_fam_flops[NFAM] = {};
long long g_fam_n[NFAM] = {};
bool g_prof_on = false;
std::vector<ProfRec> g_prof;
constexpr size_t PROF_CAP = 60000;
}  // namespace
std::atomic<long long> g_kernel_launches{0};
namespace {

template <int BM, int BN, int BK, int STAGES, int WARPS_M, int WARPS_N, bool TA, bool TB, bool AL>
void launch_cfg(const GemmParams& p, cudaStream_t st) {
    auto kern = dgemm_dmma_kernel<BM, BN, BK, STAGES, WARPS_M, WARPS_N, TA, TB, AL>;
    static PerDeviceOnce once;               // the shared-memory opt-in is a per-device attribute
    constexpr size_t smem = TileSmem<BM, BN, BK, STAGES>::BYTES;
    once.run([&] { LRN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); });
    dim3 grid((unsigned)cdiv(p.M, BM), (unsigned)cdiv(p.N, BN), (unsigned)(p.batch * p.batch2));
    const bool prof = g_prof_on && g_prof.size() < PROF_CAP;
    ProfRec rec;
    if (prof) {
        LRN_CUDA(cudaEventCreate(&rec.a));
        LRN_CUDA(cudaEventCreate(&rec.b));
        double kk = (p.K_last > 0 && p.batch2 > 1) ? ((double)p.K * (p.batch2 - 1) + p.K_last) / p.batch2 : (double)p.K;
        rec.flops = 2.0 * p.M * (double)p.N * kk * p.batch * p.batch2 * (p.lower ? 0.5 : 1.0) * (p.ktri ? 1.0 / 3.0 : 1.0);
        LRN_CUDA(cudaEventRecord(rec.a, st));
    }
    kern<<<grid, WARPS_M * WARPS_N * 32, smem, st>>>(p);
    LRN_CHECK_LAUNCH();
    if (prof) {
        LRN_CUDA(cudaEventRecord(rec.b, st));
        g_prof.push_back(rec);
    }
    g_launches.fetch_add(1, std::memory_order_relaxed);
}

template <bool TA, bool TB, bool AL>
void launch_shape(const GemmParams& p, cudaStream_t st) {
    long long tilesL = cdiv(p.M, 128) * cdiv(p.N, 128) * (long long)p.batch * p.batch2;
    if (p.lower) tilesL = tilesL / 2 + cdiv(p.M, 128);
    if (tilesL >= 100 && p.M > 64 && p.N > 64) {
        launch_cfg<128, 128, 32, 3, 2, 4, TA, TB, AL>(p, st);
        return;
    }
    const long long ctasM = cdiv(p.M, 128) * cdiv(p.N, 64) * (long long)p.batch * p.batch2;
    if (p.N <= 64 && p.M >= 512 && ctasM >= 148 && !p.lower) {
        // tall-skinny products (block-Jacobi panel rotations, panel solves): 128 x 64 tiles, 8 warps of 32 x 32
        launch_cfg<128, 64, 16, 3, 4, 2, TA, TB, AL>(p, st);
        return;
    }
    if (p.M <= 32 && p.N <= 32 && p.K >= 256) {
        // 32 x 32 cross Gram blocks of the block-Jacobi SVD (split-K batches): the product streams its operands once
        launch_cfg<32, 32, 32, 4, 2, 2, TA, TB, AL>(p, st);
        return;
    }
    if (p.K >= 512) {
        // long-K small-output products (Gram matrices of the block-Jacobi panels): deeper K tiles, fewer barriers
        launch_cfg<64, 64, 32, 3, 2, 2, TA, TB, AL>(p, st);
        return;
    }
    launch_cfg<64, 64, 16, 4, 2, 2, TA, TB, AL>(p, st);
}

template <bool AL>
void launch_trans(const GemmParams& p, cudaStream_t st) {
    if (!p.transA && !p.transB) launch_shape<false, false, AL>(p, st);
    else if (!p.transA && p.transB) launch_shape<false, true, AL>(p, st);
    else if (p.transA && !p.transB) launch_shape<true, false, AL>(p, st);
    else launch_shape<true, true, AL>(p, st);
}

}  // namespace

namespace {
std::atomic<bool> g_bulk_enabled{true};
void launch_bulk(const GemmParams& p, cudaStream_t st) {
    static PerDeviceOnce once;
    once.run([&] {
        LRN_CUDA(cudaFuncSetAttribute(dgemm_dmma_bulk_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BULK_SMEM));
        LRN_CUDA(cudaFuncSetAttribute(dgemm_dmma_bulk_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BULK_SMEM));
    });
    dim3 grid((unsigned)(p.M / 128), (unsigned)(p.N / 128), (unsigned)p.batch);
    const bool prof = g_prof_on && g_prof.size() < PROF_CAP;
    ProfRec rec;
    if (prof) {
        LRN_CUDA(cudaEventCreate(&rec.a));
        LRN_CUDA(cudaEventCreate(&rec.b));
        rec.flops = 2.0 * p.M * (double)p.N * p.K * p.batch * (p.lower ? 0.5 : 1.0);
        LRN_CUDA(cudaEventRecord(rec.a, st));
    }
    if (p.transB) dgemm_dmma_bulk_kernel<true><<<grid, 288, BULK_SMEM, st>>>(p);
    else dgemm_dmma_bulk_kernel<false><<<grid, 288, BULK_SMEM, st>>>(p);
    LRN_CHECK_LAUNCH();
    if (prof) {
        LRN_CUDA(cudaEventRecord(rec.b, st));
        rec.fam = 1;
        g_prof.push_back(rec);
    }
    g_launches.fetch_add(1, std::memory_order_relaxed);
}
}  // namespace

void panel_rotate(const PanelRotateParams& p, cudaStream_t st) {
    static PerDeviceOnce once;
    once.run([&] { LRN_CUDA(cudaFuncSetAttribute(panel_rotate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PR_SMEM)); });
    const int sms = device_sm_count();
    LRN_REQUIRE(p.ldw % 2 == 0 && p.tiles * 128 <= p.ldw, "panel_rotate: rows must be padded to whole 128-row tiles");
    if (p.total <= 0) return;
    const bool prof = g_prof_on && g_prof.size() < PROF_CAP;
    ProfRec rec;
    if (prof) {
        LRN_CUDA(cudaEventCreate(&rec.a));
        LRN_CUDA(cudaEventCreate(&rec.b));
        rec.flops = 2.0 * 128.0 * 64.0 * 64.0 * (double)p.total;
        LRN_CUDA(cudaEventRecord(rec.a, st));
    }
    const unsigned grid = (unsigned)std::min<long long>(sms, p.total);
    panel_rotate_kernel<<<grid, 288, PR_SMEM, st>>>(p);
    LRN_CHECK_LAUNCH();
    if (prof) {
        LRN_CUDA(cudaEventRecord(rec.b, st));
        rec.fam = 2;
        g_prof.push_back(rec);
    }
    g_launches.fetch_add(1, std::memory_order_relaxed);
}

void gemm_set_bulk(bool on) { g_bulk_enabled.store(on); }

int device_sm_count() {
    static std::atomic<int> cached[64];
    int dev = 0;
    cudaGetDevice(&dev);
    int v = cached[dev & 63].load(std::memory_order_relaxed);
    if (v == 0) {
        LRN_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev));
        cached[dev & 63].store(v, std::memory_order_relaxed);
    }
    return v;
}

void gemm(const GemmParams& p, cudaStream_t stream) {
    if (p.M <= 0 || p.N <= 0 || p.batch <= 0) return;
    // TMA (bulk copy) path: large A B^T and A B products with 16-byte aligned operands.  The kernel takes whole 128 x 128
    // tiles and K in multiples of 32; the bottom / right edge strips and a K remainder (added with beta = 1, plain epilogue
    // only) go through the generic kernel.  A strided batch (row blocks of the block-cyclic distributed factorisation) is
    // taken when every problem consists of whole tiles.
    const int Kf = p.K / 32 * 32;
    const int Mf = p.M / 128 * 128, Nf = p.N / 128 * 128;
    long long tiles = (long long)(Mf / 128) * (Nf / 128) * p.batch;
    if (p.lower) tiles = tiles / 2 + Mf / 128;
    if (g_bulk_enabled.load(std::memory_order_relaxed) && !p.no_bulk && !p.ktri && !p.transA && p.batch2 == 1 && !p.colscale &&
        !p.cblkmap && Kf >= 64 && (Kf == p.K || p.mode == 0) && Mf >= 128 && Nf >= 128 && tiles >= 120 &&
        ((reinterpret_cast<uintptr_t>(p.A) | reinterpret_cast<uintptr_t>(p.B)) % 16 == 0) && p.lda % 2 == 0 && p.ldb % 2 == 0 &&
        p.sA % 2 == 0 && p.sB % 2 == 0) {
        GemmParams f = p;
        f.M = Mf; f.N = Nf; f.K = Kf;
        launch_bulk(f, stream);
        if (Kf < p.K) {                          // K remainder on the full-tile region
            GemmParams e = f;
            e.A = p.A + (size_t)Kf * p.lda;
            e.B = p.transB ? p.B + (size_t)Kf * p.ldb : p.B + Kf;
            e.K = p.K - Kf; e.beta = 1.0; e.no_bulk = true;
            gemm(e, stream);
        }
        if (Mf < p.M) {                          // bottom strip: rows [Mf, M), all columns
            GemmParams e = p;
            e.A = p.A + Mf; e.C = p.C + Mf; e.M = p.M - Mf; e.row0 = p.row0 + Mf; e.no_bulk = true;
            gemm(e, stream);
        }
        if (Nf < p.N) {                          // right strip: rows [0, Mf), columns [Nf, N)
            GemmParams e = p;
            e.B = p.transB ? p.B + Nf : p.B + (size_t)Nf * p.ldb;
            e.C = p.C + (size_t)Nf * p.ldc; e.M = Mf; e.N = p.N - Nf; e.col0 = p.col0 + Nf; e.no_bulk = true;
            gemm(e, stream);
        }
        return;
    }
    LRN_REQUIRE(p.A && p.B && p.C, "null operand");
    LRN_REQUIRE(p.K >= 0, "negative K");
    bool al = ((reinterpret_cast<uintptr_t>(p.A) | reinterpret_cast<uintptr_t>(p.B)) % 16 == 0) && (p.lda % 2 == 0) &&
              (p.ldb % 2 == 0) && (p.sA % 2 == 0) && (p.sB % 2 == 0) && (p.sA2 % 2 == 0) && (p.sB2 % 2 == 0);
    LRN_REQUIRE(p.batch2 >= 1, "batch2");
    LRN_REQUIRE(!p.cblkmap || (p.N % 32 == 0), "cblkmap needs N % 32 == 0");
    if (al) launch_trans<true>(p, stream);
    else launch_trans<false>(p, stream);
}

long long gemm_launch_count() { return g_launches.load(); }

bool gemm_profile_active() { return g_prof_on; }

bool gemm_prof_begin(cudaStream_t st, cudaEvent_t& start) {
    if (!g_prof_on || g_prof.size() >= PROF_CAP) return false;
    LRN_CUDA(cudaEventCreate(&start));
    LRN_CUDA(cudaEventRecord(start, st));
    return true;
}

void gemm_prof_end(cudaEvent_t start, cudaStream_t st, double flops, int fam) {
    ProfRec rec;
    rec.a = start;
    LRN_CUDA(cudaEventCreate(&rec.b));
    LRN_CUDA(cudaEventRecord(rec.b, st));
    rec.flops = flops;
    rec.fam = fam;
    g_prof.push_back(rec);
}

void gemm_profile(int mode, double* ms, double* flops, long long* launches) {
    if (mode == 1) {
        for (auto& r : g_prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
        g_prof.clear();
        g_prof_on = true;
        return;
    }
    if (mode >= 10 && mode < 10 + NFAM) {    // per-kernel totals of the last stopped profile
        const int f = mode - 10;
        if (ms) *ms = g_fam_ms[f];
        if (flops) *flops = g_fam_flops[f];
        if (launches) *launches = g_fam_n[f];
        return;
    }
    g_prof_on = false;
    LRN_CUDA(cudaDeviceSynchronize());
    double t = 0.0, f = 0.0;
    long long n = 0;
    for (int k = 0; k < NFAM; k++) { g_fam_ms[k] = 0.0; g_fam_flops[k] = 0.0; g_fam_n[k] = 0; }
    for (auto& r : g_prof) {
        float e = 0.f;
        if (cudaEventElapsedTime(&e, r.a, r.b) == cudaSuccess) {
            if (r.fam < NFAM_DMMA) { t += e; f += r.flops; }
            g_fam_ms[r.fam] += e; g_fam_flops[r.fam] += r.flops; g_fam_n[r.fam]++;
        }
        if (r.fam < NFAM_DMMA) n++;
        cudaEventDestroy(r.a); cudaEventDestroy(r.b);
    }
    if (ms) *ms = t;
    if (flops) *flops = f;
    if (launches) *launches = n;
    g_prof.clear();
}

}  // namespace lrn
