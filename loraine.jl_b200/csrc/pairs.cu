// Sparse-pair Schur assembly, F3 formula of makeBBBBsi (src/makeBBBB.jl:139-213, `_dot` :39-64), staged through shared memory:
//     H[j,k] = tr(calA_j W calA_k W) = sum_{(p,q) in calA_k} v_k[p,q] T_j[p,q],      T_j = W calA_j W  sampled at k's entries,
//     T_j[p,q] = W[p, I_j] A_j W[I_j, q]        (I_j = distinct indices of calA_j, A_j its |I_j| x |I_j| coefficient block).
// (H is symmetric: the roles of j and k are interchangeable; the kernel stages on the COLUMN side.)
// A CTA owns up to 8 CONSECUTIVE constraints k (columns of H) and stages the rows W[x, I_k], x = 0..m-1, of all of them in
// shared memory once ([x][S] layout: the |I_k| values a pair needs sit in one 16-byte aligned vector).  It then streams the
// lower-triangle entry lists of every constraint j >= k (symmetric storage: T_k is symmetric, so the strict upper entries are
// folded into doubled weights -- half the gathers of the reference loop), one thread per j; both gathers of an entry are two
// vector loads from shared memory instead of 2 |calA_k| scalar gathers from L2.  Consecutive threads handle consecutive rows j,
// so the read-modify-write of a column of H is coalesced.  Constraints j are bucketed by entry count (uniform work per warp)
// and sorted by index inside a bucket (the j >= k restriction is a suffix).  Multi-GPU: a thread skips the rows its rank does
// not own (row blocks are runs of consecutive j, so warps stay uniform).
// Bound: shared-memory bandwidth (random 16 B vector loads) -- algorithmic traffic 2 x 8 |I_j| bytes per (j, entry of k).
#include "ops.cuh"
#include <algorithm>

namespace lrn {
namespace {

constexpr int PT = 512;    // threads per CTA

template <int C>
__device__ __forceinline__ double bilinear(const double* __restrict__ Rp, const double* __restrict__ Rq, const double* __restrict__ A) {
    // sum_{a,b < C} Rp[a] A[a][b] Rq[b]; Rp / Rq 16-byte aligned, A in shared memory (broadcast reads), row stride PAIR_MAXC
    double rp[C], rq[C];
#pragma unroll
    for (int a = 0; a < C; a += 2) {
        const double2 u = *reinterpret_cast<const double2*>(Rp + a);
        const double2 v = *reinterpret_cast<const double2*>(Rq + a);
        rp[a] = u.x; rp[a + 1] = u.y; rq[a] = v.x; rq[a + 1] = v.y;
    }
    double t = 0.0;
#pragma unroll
    for (int a = 0; a < C; a++) {
        double s = 0.0;
#pragma unroll
        for (int b = 0; b < C; b++) s = fma(A[a * PAIR_MAXC + b], rq[b], s);
        t = fma(rp[a], s, t);
    }
    return t;
}

__global__ void __launch_bounds__(PT, 1)
    k_schur_pairs_staged(int m, const double* __restrict__ W, int ldw, double* __restrict__ H, int ldh, const int* __restrict__ g_r0,
                         const int* __restrict__ g_cnt, const int* __restrict__ g_S, const int* __restrict__ g_idx0,
                         const int* __restrict__ gidx, const int* __restrict__ row_off, const int* __restrict__ row_c,
                         const double* __restrict__ rowA, int nbuckets, const int* __restrict__ b_first,
                         const int* __restrict__ b_ids, const int* __restrict__ b_eptr, const int2* __restrict__ e_pq,
                         const double* __restrict__ e_w, RowOwner own, int accumulate) {
    extern __shared__ __align__(16) double smem[];
    __shared__ double sA[PAIR_ROWS * PAIR_MAXC * PAIR_MAXC];
    __shared__ int s_off[PAIR_ROWS], s_c[PAIR_ROWS];
    const int g = blockIdx.x;
    const int r0 = g_r0[g], cnt = g_cnt[g], S = g_S[g];      // columns r0 .. r0 + cnt - 1 of H
    const int tid = threadIdx.x;
    // ---- stage W[x, I] for the S indices of the group: Ws[x * S + ci] --------------------------------------------------
    {
        const int* idx = gidx + g_idx0[g];
        for (int ci = 0; ci < S; ci++) {
            const double* col = W + (size_t)idx[ci] * ldw;          // column = row of the symmetric W
            for (int x = tid; x < m; x += PT) smem[(size_t)x * S + ci] = col[x];
        }
        for (int t = tid; t < PAIR_ROWS * PAIR_MAXC * PAIR_MAXC; t += PT) sA[t] = rowA[(size_t)g * PAIR_ROWS * PAIR_MAXC * PAIR_MAXC + t];
        if (tid < PAIR_ROWS) { s_off[tid] = row_off[g * PAIR_ROWS + tid]; s_c[tid] = row_c[g * PAIR_ROWS + tid]; }
    }
    __syncthreads();
    for (int b = 0; b < nbuckets; b++) {
        const int m0 = b_first[b], m1 = b_first[b + 1];
        // members with id >= r0: ids ascending inside the bucket -> binary search for the start of the suffix
        int lo = m0, hi = m1;
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (b_ids[mid] < r0) lo = mid + 1; else hi = mid; }
        for (int t = lo + tid; t < m1; t += PT) {
            const int j = b_ids[t];
            if (!own.owns(j)) continue;
            const int f0 = b_eptr[t], f1 = b_eptr[t + 1];
            double* dst = H + (size_t)r0 * ldh + own.local(j);      // own-rows layout: j's local row
            // rows of the group one after the other (the branch on the size class is uniform over the CTA); the few entries
            // of k are re-read from L1 for every row
#pragma unroll 1
            for (int r = 0; r < cnt; r++) {
                const int c = s_c[r];
                if (c == 0 || j < r0 + r) continue;            // no matrix in this block / above the diagonal of H
                const int off = s_off[r];
                const double* A = sA + r * PAIR_MAXC * PAIR_MAXC;
                double acc = 0.0;
                if (c <= 2) {
                    for (int f = f0; f < f1; f++) {
                        const int2 pq = e_pq[f];
                        acc = fma(e_w[f], bilinear<2>(smem + (size_t)pq.x * S + off, smem + (size_t)pq.y * S + off, A), acc);
                    }
                } else if (c <= 4) {
                    for (int f = f0; f < f1; f++) {
                        const int2 pq = e_pq[f];
                        acc = fma(e_w[f], bilinear<4>(smem + (size_t)pq.x * S + off, smem + (size_t)pq.y * S + off, A), acc);
                    }
                } else {
                    for (int f = f0; f < f1; f++) {
                        const int2 pq = e_pq[f];
                        acc = fma(e_w[f], bilinear<8>(smem + (size_t)pq.x * S + off, smem + (size_t)pq.y * S + off, A), acc);
                    }
                }
                // every (j, k) of a block is produced exactly once: the first block of an assembly stores (H was cleared), later
                // blocks add -- a plain store keeps the HBM round trip of a read-modify-write out of the dependency chain
                if (accumulate) dst[(size_t)r * ldh] += acc;
                else dst[(size_t)r * ldh] = acc;
            }
        }
    }
}

}  // namespace

void sp_build_pair_plan(SparseBlock& sb, const std::vector<int>& rowptr, const std::vector<int>& ep, const std::vector<int>& eq,
                        const std::vector<double>& ev, cudaStream_t st) {
    PairPlan& P = sb.pairs;
    P.ok = false;
    const int n = sb.n_var, m = sb.m;
    if (!sb.sparse_ok || sb.nF1 != 0 || sb.npart == 0) return;
    // shared-memory budget: rows W[x, .] of S doubles for x < m
    const size_t budget = 200 * 1024;
    int smax = (int)std::min<size_t>(PAIR_ROWS * PAIR_MAXC, budget / ((size_t)m * sizeof(double)));
    smax &= ~1;
    if (smax < 2) return;
    // per constraint: distinct indices, dense coefficient block in local indices
    std::vector<std::vector<int>> I(n);
    int maxc = 0;
    for (int j = 0; j < n; j++) {
        auto& v = I[j];
        for (int e = rowptr[j]; e < rowptr[j + 1]; e++) { v.push_back(ep[e]); v.push_back(eq[e]); }
        std::sort(v.begin(), v.end());
        v.erase(std::unique(v.begin(), v.end()), v.end());
        maxc = std::max(maxc, (int)v.size());
    }
    if (maxc > PAIR_MAXC || ((maxc + 1) & ~1) > smax) return;
    auto padded = [](int c) { return c <= 2 ? (c == 0 ? 0 : 2) : (c <= 4 ? 4 : 8); };     // slot = what bilinear<C> reads
    // ---- groups: aligned chunks of 8 rows, halved until their staged width fits -------------------------------------------
    std::vector<int> g_r0, g_cnt, g_S, g_idx0, gidx, row_off, row_c;
    std::vector<double> rowA;
    std::vector<std::pair<int, int>> chunks;     // (r0, cnt)
    for (int r0 = 0; r0 < n; r0 += PAIR_ROWS) {
        std::vector<std::pair<int, int>> stack{{r0, std::min(PAIR_ROWS, n - r0)}};
        while (!stack.empty()) {
            auto [a, c] = stack.back();
            stack.pop_back();
            int S = 0;
            for (int j = a; j < a + c; j++) S += padded((int)I[j].size());
            if (S > smax && c > 1) {
                const int h = c / 2;
                stack.push_back({a + h, c - h});
                stack.push_back({a, h});
                continue;
            }
            if (S > smax) return;                 // a single constraint does not fit: keep the gather kernel
            chunks.push_back({a, c});
        }
    }
    std::sort(chunks.begin(), chunks.end(), [](auto& x, auto& y) { return x.first < y.first; });   // long columns first
    for (auto [a, c] : chunks) {
        int S = 0;
        bool any = false;
        for (int j = a; j < a + c; j++) any = any || !I[j].empty();
        if (!any) continue;                       // no participating constraint in this chunk: its rows of H stay zero
        g_r0.push_back(a); g_cnt.push_back(c); g_idx0.push_back((int)gidx.size());
        const size_t base = rowA.size();
        rowA.resize(base + (size_t)PAIR_ROWS * PAIR_MAXC * PAIR_MAXC, 0.0);
        for (int r = 0; r < PAIR_ROWS; r++) {
            if (r >= c) { row_off.push_back(0); row_c.push_back(0); continue; }
            const int j = a + r;
            const auto& v = I[j];
            row_off.push_back(S); row_c.push_back((int)v.size());
            const int pc = padded((int)v.size());
            for (int t = 0; t < pc; t++) gidx.push_back(t < (int)v.size() ? v[t] : v.back());
            double* A = rowA.data() + base + (size_t)r * PAIR_MAXC * PAIR_MAXC;
            for (int e = rowptr[j]; e < rowptr[j + 1]; e++) {
                const int la = (int)(std::lower_bound(v.begin(), v.end(), ep[e]) - v.begin());
                const int lb = (int)(std::lower_bound(v.begin(), v.end(), eq[e]) - v.begin());
                A[la * PAIR_MAXC + lb] += ev[e];
            }
            S += pc;
        }
        if (S == 0) { gidx.push_back(0); gidx.push_back(0); S = 2; }      // cannot happen (any == true), keeps S > 0
        g_S.push_back(S);
    }
    // ---- column side: lower-triangle entries with doubled off-diagonal weights, bucketed by entry count -----------------
    auto bucket_of = [](int c) { int b = 0; while ((1 << b) < c) b++; return b; };     // 1 | 2 | 3-4 | 5-8 | 9-16 | ...
    std::vector<std::vector<int>> members;
    std::vector<int> lcount(n, 0);
    for (int j = 0; j < n; j++) {
        int c = 0;
        for (int e = rowptr[j]; e < rowptr[j + 1]; e++) if (ep[e] >= eq[e]) c++;
        lcount[j] = c;
        if (c == 0) continue;
        const int b = bucket_of(c);
        if ((int)members.size() <= b) members.resize(b + 1);
        members[b].push_back(j);
    }
    std::vector<int> b_first{0}, b_ids, b_eptr{0};
    std::vector<int2> e_pq;
    std::vector<double> e_w;
    for (auto& mem : members) {
        if (mem.empty()) continue;
        for (int j : mem) {
            for (int e = rowptr[j]; e < rowptr[j + 1]; e++) {
                if (ep[e] < eq[e]) continue;
                e_pq.push_back(make_int2(ep[e], eq[e]));
                e_w.push_back(ep[e] == eq[e] ? ev[e] : 2.0 * ev[e]);
            }
            b_ids.push_back(j);
            b_eptr.push_back((int)e_pq.size());
        }
        b_first.push_back((int)b_ids.size());
    }
    if (g_r0.empty() || b_ids.empty()) return;
    P.ngroups = (int)g_r0.size();
    P.nbuckets = (int)b_first.size() - 1;
    P.smax = smax;
    P.smem = (size_t)m * smax * sizeof(double);
    P.g_r0.upload(g_r0, st); P.g_cnt.upload(g_cnt, st); P.g_S.upload(g_S, st); P.g_idx0.upload(g_idx0, st);
    P.gidx.upload(gidx, st); P.row_off.upload(row_off, st); P.row_c.upload(row_c, st); P.rowA.upload(rowA, st);
    P.b_first.upload(b_first, st); P.b_ids.upload(b_ids, st); P.b_eptr.upload(b_eptr, st);
    P.h_b_first = b_first;
    P.e_pq.upload(e_pq, st); P.e_w.upload(e_w, st);
    LRN_CUDA(cudaStreamSynchronize(st));
    P.ok = true;
}

void sp_schur_pairs_staged(cudaStream_t st, const SparseBlock& sb, const double* W, int ldw, double* H, int ldh, RowOwner own,
                           bool accumulate) {
    const PairPlan& P = sb.pairs;
    LRN_REQUIRE(P.ok, "no staged pair plan for this block");
    static PerDeviceOnce once;
    once.run([&] { LRN_CUDA(cudaFuncSetAttribute(k_schur_pairs_staged, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024)); });
    k_schur_pairs_staged<<<(unsigned)P.ngroups, PT, P.smem, st>>>(sb.m, W, ldw, H, ldh, P.g_r0.p, P.g_cnt.p, P.g_S.p, P.g_idx0.p,
                                                                 P.gidx.p, P.row_off.p, P.row_c.p, P.rowA.p, P.nbuckets,
                                                                 P.b_first.p, P.b_ids.p, P.b_eptr.p, P.e_pq.p, P.e_w.p, own,
                                                                 accumulate ? 1 : 0);
    LRN_CHECK_LAUNCH();
}

}  // namespace lrn
