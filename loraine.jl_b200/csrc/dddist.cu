// Multi-GPU double-double LP path: the Schur matrix H (n x n) is assembled and factored row-block-cyclically over the ranks of
// an NCCL communicator (row block g of height pw belongs to rank g % world); every other part of the iteration is replicated.
// Two forms, as for Float64 (dist.cu, group.cu): one process per GPU (lrn_dd_dist_init) and one host thread driving N devices
// (lrn_dd_create_multi, a facade over one ordinary handle per device).
//
// Factorisation (right-looking, on the 32 x 32 tile arithmetic of ddlp.cuh).  Step p, diagonal block p, owner p % world:
//   1. the owner factors the diagonal block: pw / 32 tile steps (k_dd_potrf_tile, k_dd_trsm_tile and k_dd_syrk_tile limited to
//      the block), which also produce the pivot reciprocals;
//   2. it broadcasts the factored block, its pivot reciprocals and the info word (first bad pivot) in one ncclBroadcast;
//   3. every rank solves its own row blocks of column panel p against that block, slice by slice as on one GPU: for each
//      32-column slice the tile solve, then the update of the remaining slices of the panel;
//   4. one ncclAllGather of the solved row blocks (each send padded to the largest count) gives every rank the full panel,
//      stored in place in its L;
//   5. every rank updates its own row blocks of the trailing lower triangle with the panel, one 32-column slice after the other.
// Every entry of L therefore sees the same sequence of double-double operations as in the single-GPU factorisation
// (lrn_dd_schur_factor without a communicator): the factor is the single-GPU factor bit for bit, and every rank ends with all
// of it (the triangular solves run replicated).  A dd travels as two ncclFloat64, which is exact.
//
// Failure protocol: every rank enqueues the same collectives in the same order whatever the pivots are; the info word travels
// with every diagonal block, so all ranks return the same LAPACK-style index, and the kernels of later steps return at once.
#include "ddlp.cuh"
#include "group.cuh"
#include "dist.cuh"

#include "../../include/loraine_b200_debug.h"

using namespace lrn;

namespace {

constexpr int TS = DD_TS;

// diagonal block p (w x w at (c0, c0)) + its pivot reciprocals + the info word -> xb (block with leading dimension pw)
__global__ void k_dd_pack_diag(const dd* __restrict__ L, int n, int c0, int w, int pw, const dd* __restrict__ rdiag,
                               const int* __restrict__ info, dd* __restrict__ xb) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
    if (i < w) xb[(size_t)j * pw + i] = L[(size_t)(c0 + j) * n + c0 + i];
    if (j == 0 && i < w) xb[(size_t)pw * pw + i] = rdiag[c0 + i];
    if (j == 0 && i == 0) xb[(size_t)pw * pw + pw] = dd_make((double)*info);
}
__global__ void k_dd_take_diag(const dd* __restrict__ xb, int n, int c0, int w, int pw, dd* __restrict__ L, dd* __restrict__ rdiag,
                               int* __restrict__ info) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
    if (i < w) L[(size_t)(c0 + j) * n + c0 + i] = xb[(size_t)j * pw + i];
    if (j == 0 && i < w) rdiag[c0 + i] = xb[(size_t)pw * pw + i];
    if (j == 0 && i == 0) *info = (int)xb[(size_t)pw * pw + pw].hi;
}

// the tile solve of k_dd_trsm_tile for the row tiles tiles[blockIdx.x] (my row tiles below the diagonal block)
__global__ void __launch_bounds__(DD_TS * TRSM_CB) k_dd_trsm_list(dd* __restrict__ A, int n, int k0, int w, const dd* __restrict__ rdiag,
                                                                   const int* __restrict__ tiles, const int* __restrict__ info) {
    if (*info != 0) return;                                 // an earlier diagonal block failed
    dd_trsm_tile_body(A, n, k0, w, rdiag, tiles[blockIdx.x] * DD_TS);
}
// the tile update of k_dd_syrk_tile for row tiles tiles[blockIdx.x], column tiles jt0 + blockIdx.y (lower triangle only)
__global__ void __launch_bounds__(DD_TS * DD_TS) k_dd_syrk_list(dd* __restrict__ A, int n, int k0, int w, const int* __restrict__ tiles,
                                                                 int jt0, const int* __restrict__ info) {
    const int it = tiles[blockIdx.x], jt = jt0 + blockIdx.y;
    if (jt > it || *info != 0) return;
    dd_syrk_tile_body(A, n, k0, w, it * DD_TS, jt * DD_TS);
}

// first row block >= p owned by `rank`, and how many of its blocks are >= p (as in dist.cu)
__host__ __device__ inline int first_block(int p, int rank, int world) { return p + ((rank - p % world + world) % world); }
inline int count_blocks(int p, int rank, int world, int nblk) {
    const int f = first_block(p, rank, world);
    return f >= nblk ? 0 : (nblk - 1 - f) / world + 1;
}

// my solved row blocks g = first + z * world of panel p (columns c0 .. c0 + w) -> send[z] (pw x w, ld pw)
__global__ void k_dd_pack_panel(const dd* __restrict__ L, int n, int c0, int w, int pw, int first, int world, int cnt, dd* __restrict__ send) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y, z = blockIdx.z;
    const int row = (first + z * world) * pw + i;
    if (i < pw && j < w && z < cnt && row < n) send[((size_t)z * w + j) * pw + i] = L[(size_t)(c0 + j) * n + row];
}
// recv[r][z] (rank r's slot z, maxcnt slots per rank) -> its place in L.  p1: first row block of the exchange
__global__ void k_dd_unpack_panel(const dd* __restrict__ recv, dd* __restrict__ L, int n, int c0, int w, int pw, int p1, int world,
                                  int maxcnt, int nblk) {
    const int slot = blockIdx.z, r = slot / maxcnt, z = slot - r * maxcnt;
    const int g = first_block(p1, r, world) + z * world;
    const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
    const int row = g * pw + i;
    if (g >= nblk || i >= pw || j >= w || row >= n) return;
    L[(size_t)(c0 + j) * n + row] = recv[((size_t)slot * w + j) * pw + i];
}

DistCtx& ctx_of(lrn_dd_solver* h) { return *static_cast<DistCtx*>(h->nccl); }

}  // namespace

namespace lrn {

void dd_gather_H(lrn_dd_solver* h) {
    LRN_NCCL(nccl_api().AllReduce(h->H.p, h->H.p, (size_t)h->n * h->n * 2, ncclDouble, ncclSum, ctx_of(h).comm, h->st));
}

int dd_factor_dist(lrn_dd_solver* h) {
    DistCtx& ctx = ctx_of(h);
    const int n = h->n, pw = h->pw, world = h->world, rank = h->rank;
    LRN_REQUIRE(pw % TS == 0, "row block height must be a multiple of 32");
    const int nblk = (int)cdiv(n, pw);
    cudaStream_t st = h->st;
    // my 32-row tiles in increasing order: the tiles below diagonal block p are a suffix of the list
    std::vector<int> tiles;
    for (int g = rank; g < nblk; g += world)
        for (int t = g * pw / TS; t < (int)cdiv(std::min(n, (g + 1) * pw), TS); t++) tiles.push_back(t);
    if (h->tiles.n < tiles.size() || h->tiles.n == 0) h->tiles.alloc(std::max<size_t>(1, tiles.size()));
    if (!tiles.empty()) {
        LRN_CUDA(cudaMemcpyAsync(h->tiles.p, tiles.data(), tiles.size() * sizeof(int), cudaMemcpyHostToDevice, st));
        LRN_CUDA(cudaStreamSynchronize(st));                // `tiles` is pageable and goes out of scope at the end
    }
    const size_t blk = (size_t)pw * pw;
    const int maxcnt0 = (int)std::max<long long>(1, cdiv(nblk - 1, world));
    if (h->xb.n < blk + pw + 1) h->xb.alloc(blk + pw + 1);
    if (h->sendbuf.n < (size_t)maxcnt0 * blk) h->sendbuf.alloc((size_t)maxcnt0 * blk);
    if (h->recvbuf.n < (size_t)maxcnt0 * blk * world) h->recvbuf.alloc((size_t)maxcnt0 * blk * world);
    dd* L = h->L.p;
    int* info = h->info.p;
    LRN_CUDA(cudaMemcpyAsync(L, h->H.p, (size_t)n * n * sizeof(dd), cudaMemcpyDeviceToDevice, st));
    LRN_CUDA(cudaMemsetAsync(info, 0, sizeof(int), st));
    size_t off = 0;                                         // first of my tiles below the current diagonal block
    for (int p = 0; p < nblk; p++) {
        const int c0 = p * pw, w = std::min(pw, n - c0), owner = p % world;
        // ---- 1-2. diagonal block: factored by its owner, broadcast with the pivot reciprocals and the info word --------------
        if (rank == owner) {
            for (int k0 = c0; k0 < c0 + w; k0 += TS) {
                const int tw = std::min(TS, c0 + w - k0);
                k_dd_potrf_tile<<<1, dim3(TS, TS), 0, st>>>(L, n, k0, tw, info, h->rdiag.p);
                LRN_CHECK_LAUNCH();
                const int below = c0 + w - k0 - tw;
                if (below <= 0) break;
                const unsigned nt = (unsigned)cdiv(below, TS);
                k_dd_trsm_tile<<<nt, TS * TRSM_CB, 0, st>>>(L, n, k0, tw, h->rdiag.p);
                LRN_CHECK_LAUNCH();
                k_dd_syrk_tile<<<dim3(nt, nt), dim3(TS, TS), 0, st>>>(L, n, k0, tw, 0);
                LRN_CHECK_LAUNCH();
            }
            k_dd_pack_diag<<<dim3((unsigned)cdiv(w, 128), (unsigned)w), 128, 0, st>>>(L, n, c0, w, pw, h->rdiag.p, info, h->xb.p);
            LRN_CHECK_LAUNCH();
        }
        LRN_NCCL(nccl_api().Broadcast(h->xb.p, h->xb.p, (blk + pw + 1) * 2, ncclDouble, owner, ctx.comm, st));
        if (rank != owner) {
            k_dd_take_diag<<<dim3((unsigned)cdiv(w, 128), (unsigned)w), 128, 0, st>>>(h->xb.p, n, c0, w, pw, L, h->rdiag.p, info);
            LRN_CHECK_LAUNCH();
        }
        if (p + 1 == nblk) break;                           // (w == pw from here on)
        while (off < tiles.size() && tiles[off] * TS < c0 + w) off++;
        const unsigned mine = (unsigned)(tiles.size() - off);
        const int* my_tiles = h->tiles.p + off;
        // ---- 3. my row blocks of the panel, in the single-GPU tile order -----------------------------------------------------
        if (mine > 0)
            for (int k0 = c0; k0 < c0 + w; k0 += TS) {
                k_dd_trsm_list<<<mine, TS * TRSM_CB, 0, st>>>(L, n, k0, TS, h->rdiag.p, my_tiles, info);
                LRN_CHECK_LAUNCH();
                const int rest = (c0 + w - k0 - TS) / TS;   // column tiles of the panel right of this slice
                if (rest > 0) {
                    k_dd_syrk_list<<<dim3(mine, (unsigned)rest), dim3(TS, TS), 0, st>>>(L, n, k0, TS, my_tiles, (k0 + TS) / TS, info);
                    LRN_CHECK_LAUNCH();
                }
            }
        // ---- 4. all-gather of the solved row blocks --------------------------------------------------------------------------
        const int f = first_block(p + 1, rank, world), cnt = count_blocks(p + 1, rank, world, nblk);
        const int maxcnt = (int)cdiv(nblk - p - 1, world);
        const size_t slot = (size_t)pw * w;
        if (cnt > 0) {
            k_dd_pack_panel<<<dim3((unsigned)cdiv(pw, 128), (unsigned)w, (unsigned)cnt), 128, 0, st>>>(L, n, c0, w, pw, f, world, cnt,
                                                                                                       h->sendbuf.p);
            LRN_CHECK_LAUNCH();
        }
        LRN_NCCL(nccl_api().AllGather(h->sendbuf.p, h->recvbuf.p, (size_t)maxcnt * slot * 2, ncclDouble, ctx.comm, st));
        k_dd_unpack_panel<<<dim3((unsigned)cdiv(pw, 128), (unsigned)w, (unsigned)(world * maxcnt)), 128, 0, st>>>(
            h->recvbuf.p, L, n, c0, w, pw, p + 1, world, maxcnt, nblk);
        LRN_CHECK_LAUNCH();
        // ---- 5. trailing update of my row blocks, one slice of the panel after the other -------------------------------------
        if (mine > 0) {
            const int jt0 = (c0 + w) / TS;
            const unsigned ncols = (unsigned)(cdiv(n, TS) - jt0);
            for (int k0 = c0; k0 < c0 + w; k0 += TS) {
                k_dd_syrk_list<<<dim3(mine, ncols), dim3(TS, TS), 0, st>>>(L, n, k0, TS, my_tiles, jt0, info);
                LRN_CHECK_LAUNCH();
            }
        }
    }
    int hinfo = 0;
    LRN_CUDA(cudaMemcpyAsync(&hinfo, info, sizeof(int), cudaMemcpyDeviceToHost, st));
    LRN_CUDA(cudaStreamSynchronize(st));
    return hinfo;
}

}  // namespace lrn

extern "C" {

int32_t lrn_dd_create_multi(lrn_dd_handle_t* out, int64_t n_var, int64_t nlin, int32_t ngpus, const int32_t* devices) {
    if (!out) return LRN_ERR_ARG;
    *out = nullptr;
    if (ngpus == 1) return lrn_dd_create(out, n_var, nlin, devices ? devices[0] : -1);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return LRN_ERR_NO_DEVICE; }   // no CPU fallback
    if (ngpus <= 0) ngpus = ndev;
    if (ngpus > ndev) return LRN_ERR_ARG;
    if (ngpus == 1) return lrn_dd_create(out, n_var, nlin, devices ? devices[0] : -1);
    lrn_dd_solver* facade = new lrn_dd_solver();
    auto* g = new GroupOf<lrn_dd_solver>();
    facade->group = g;
    facade->n = (int)n_var;
    facade->nlin = (int)nlin;
    std::vector<int> devs(ngpus);
    for (int r = 0; r < ngpus; r++) devs[r] = devices ? devices[r] : r;
    int32_t rc = LRN_OK;
    for (int r = 0; r < ngpus && rc == LRN_OK; r++) {
        lrn_dd_handle_t m = nullptr;
        rc = lrn_dd_create(&m, n_var, nlin, devs[r]);
        if (m) g->members.push_back(m);
    }
    if (rc == LRN_OK) {
        try {
            const NcclApi& api = nccl_api();
            if (!api.CommInitAll) throw std::runtime_error("ncclCommInitAll not found in libnccl");
            std::vector<ncclComm_t> comms(ngpus);
            LRN_NCCL(api.CommInitAll(comms.data(), ngpus, devs.data()));
            for (int r = 0; r < ngpus; r++) {
                auto* ctx = new DistCtx();
                ctx->rank = r; ctx->world = ngpus; ctx->comm = comms[r];
                lrn_dd_solver* m = g->members[r];
                m->nccl = ctx; m->rank = r; m->world = ngpus; m->pw = dd_block_rows(n_var);
            }
        } catch (const std::exception& e) {
            fprintf(stderr, "[loraine_b200] lrn_dd_create_multi failed: %s\n", e.what());
            rc = LRN_ERR_NCCL;
        }
    }
    if (rc != LRN_OK) {
        lrn_dd_destroy(facade);
        return rc;
    }
    *out = facade;
    return LRN_OK;
}

int32_t lrn_dd_dist_init(lrn_dd_handle_t h, int32_t rank, int32_t world, const void* unique_id128) {
    if (!h || !unique_id128 || world < 1 || rank < 0 || rank >= world) return LRN_ERR_ARG;
    if (h->group) { h->err = "lrn_dd_dist_init: the handle already drives several GPUs in-process (lrn_dd_create_multi)"; return LRN_ERR_STATE; }
    try {
        LRN_CUDA(cudaSetDevice(h->device));
        LRN_CUDA(cudaStreamSynchronize(h->st));
        ncclUniqueId id;
        std::memcpy(&id, unique_id128, sizeof id);
        auto* ctx = new DistCtx();
        ctx->rank = rank;
        ctx->world = world;
        try {
            LRN_NCCL(nccl_api().CommInitRank(&ctx->comm, world, id, rank));
        } catch (...) {
            delete ctx;
            throw;
        }
        if (h->nccl) delete static_cast<DistCtx*>(h->nccl);
        h->nccl = ctx;
        h->rank = rank;
        h->world = world;
        h->pw = dd_block_rows(h->n);
        h->have_H = h->have_factor = false;          // the Schur matrix is assembled again under the new ownership
        return LRN_OK;
    } catch (const std::exception& e) {
        h->err = e.what();
        return LRN_ERR_NCCL;
    }
}

int32_t lrn_dd_dbg_set_shard(lrn_dd_handle_t h, int32_t rank, int32_t world, int32_t block_rows) {
    if (!h || h->group || world < 1 || rank < 0 || rank >= world || block_rows < 0 || block_rows % 32 != 0) return LRN_ERR_ARG;
    if (h->nccl) return LRN_ERR_STATE;
    h->rank = rank;
    h->world = world;
    h->pw = block_rows > 0 ? block_rows : dd_block_rows(h->n);
    h->have_H = h->have_factor = false;
    return LRN_OK;
}

}  // extern "C"
