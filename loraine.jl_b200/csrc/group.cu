// lrn_create_multi: in-process multi-GPU group (see group.cuh) -- the form of the multi-GPU boundary SURVEY 8(b) asks for:
// one host thread, N devices, communicators made with ncclCommInitAll inside the library.
#include "group.cuh"
#include "dist.cuh"
#include <cmath>
#include <algorithm>

#include "../../include/loraine_b200_debug.h"

using namespace lrn;

namespace {
// acc[0] += sum (a - b)^2, acc[1] += sum b^2 over the lower triangle
__global__ void k_lower_diff(const double* __restrict__ A, int lda, const double* __restrict__ B, int ldb, int n, double* acc) {
    const int j = blockIdx.y + gridDim.y * blockIdx.z;
    if (j >= n) return;
    double d2 = 0.0, b2 = 0.0;
    for (int i = j + blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const double a = A[(size_t)j * lda + i], b = B[(size_t)j * ldb + i];
        d2 += (a - b) * (a - b);
        b2 += b * b;
    }
    d2 = warp_sum(d2);
    b2 = warp_sum(b2);
    if ((threadIdx.x & 31) == 0 && (d2 != 0.0 || b2 != 0.0)) {
        atomicAdd(acc, d2);
        atomicAdd(acc + 1, b2);
    }
}
}  // namespace

extern "C" {

int32_t lrn_create_multi(lrn_handle_t* out, int64_t n_var, int64_t nlmi, const int64_t* msizes, int64_t nlin,
                         const lrn_options_t* opt, int32_t ngpus, const int32_t* devices) {
    if (!out) return LRN_ERR_ARG;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return LRN_ERR_NO_DEVICE;
    if (ngpus <= 0) ngpus = ndev;
    if (ngpus > ndev) return LRN_ERR_ARG;
    if (ngpus == 1) {
        lrn_options_t o;
        if (opt) o = *opt; else lrn_default_options(&o);
        if (devices) o.device = devices[0];
        return lrn_create(out, n_var, nlmi, msizes, nlin, &o);
    }
    lrn_solver* facade = new lrn_solver();
    Group* g = new Group();
    facade->group = g;
    facade->n_var = (int)n_var; facade->nlmi = (int)nlmi; facade->nlin = (int)nlin;
    *out = facade;
    std::vector<int> devs(ngpus);
    for (int r = 0; r < ngpus; r++) devs[r] = devices ? devices[r] : r;
    for (int r = 0; r < ngpus; r++) {
        lrn_options_t o;
        if (opt) o = *opt; else lrn_default_options(&o);
        o.device = devs[r];
        lrn_handle_t m = nullptr;
        int32_t rc = lrn_create(&m, n_var, nlmi, msizes, nlin, &o);
        if (m) g->members.push_back(m);
        if (rc != LRN_OK) {
            facade->err = m ? m->err : "lrn_create failed for a group member";
            return rc;
        }
    }
    try {
        const NcclApi& api = nccl_api();
        if (!api.CommInitAll) throw std::runtime_error("ncclCommInitAll not found in libnccl");
        std::vector<ncclComm_t> comms(ngpus);
        LRN_NCCL(api.CommInitAll(comms.data(), ngpus, devs.data()));
        for (int r = 0; r < ngpus; r++) {
            auto* ctx = new DistCtx();
            ctx->rank = r; ctx->world = ngpus; ctx->comm = comms[r];
            lrn_solver* m = g->members[r];
            m->nccl = ctx; m->rank = r; m->world = ngpus;
            m->dist_pw = (m->n_var >= 16384) ? 512 : (m->n_var >= 4096 ? 256 : 128);
        }
    } catch (const std::exception& e) {
        facade->err = e.what();
        return LRN_ERR_NCCL;
    }
    return LRN_OK;
}

// test hook: give a single-GPU handle the Schur-row ownership of `rank` out of `world` WITHOUT a communicator, so that the
// sharded assembly can be checked on one GPU (the shards of all ranks must add up to the full matrix)
int32_t lrn_dbg_set_shard(lrn_handle_t h, int32_t rank, int32_t world, int32_t block_rows) {
    if (!h || h->group || world < 1 || rank < 0 || rank >= world) return LRN_ERR_ARG;
    if (h->nccl && static_cast<DistCtx*>(h->nccl)->active()) return LRN_ERR_STATE;
    if (h->finalized && h->rows_local) return LRN_ERR_STATE;      // the own-rows arrays are already sized for one rank
    h->rank = rank;
    h->world = world;
    h->dist_pw = block_rows > 0 ? block_rows : ((h->n_var >= 16384) ? 512 : (h->n_var >= 4096 ? 256 : 128));
    return LRN_OK;
}

int32_t lrn_dbg_schur_layout(lrn_handle_t h, int32_t force, int32_t* layout) {
    if (!h || force < -2 || force > 1) return LRN_ERR_ARG;
    if (h->group) {
        for (auto* m : static_cast<Group*>(h->group)->members) {
            const int32_t rc = lrn_dbg_schur_layout(m, force, nullptr);
            if (rc != LRN_OK) return rc;
        }
        return lrn_dbg_schur_layout(static_cast<Group*>(h->group)->members[0], -2, layout);
    }
    if (force != -2) {
        if (h->finalized) { h->err = "lrn_dbg_schur_layout: the layout is chosen by lrn_finalize"; return LRN_ERR_STATE; }
        h->layout_force = force;
    }
    if (layout) *layout = h->finalized && h->opt.kit == 0 ? (h->rows_local ? 1 : 0) : -1;
    return LRN_OK;
}

int32_t lrn_dbg_block_layout(lrn_handle_t h, int32_t force, int32_t* layout) {
    if (!h || force < -2 || force > 1) return LRN_ERR_ARG;
    if (h->group) {
        for (auto* m : static_cast<Group*>(h->group)->members) {
            const int32_t rc = lrn_dbg_block_layout(m, force, nullptr);
            if (rc != LRN_OK) return rc;
        }
        return lrn_dbg_block_layout(static_cast<Group*>(h->group)->members[0], -2, layout);
    }
    if (force != -2) {
        if (h->finalized) { h->err = "lrn_dbg_block_layout: the layout is chosen by lrn_finalize"; return LRN_ERR_STATE; }
        h->blk_force = force;
    }
    if (layout) *layout = h->finalized ? (h->blk_sharded ? 1 : 0) : -1;
    return LRN_OK;
}

int32_t lrn_dbg_create_loopback(lrn_handle_t* out, int64_t n_var, int64_t nlmi, const int64_t* msizes, int64_t nlin,
                                const lrn_options_t* opt, int32_t world, int32_t block_rows) {
    if (!out) return LRN_ERR_ARG;
    *out = nullptr;
    if (world < 1 || world > 8 || block_rows < 0 || block_rows % 64 != 0 || block_rows > 512) return LRN_ERR_ARG;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return LRN_ERR_NO_DEVICE;
    lrn_solver* facade = new lrn_solver();
    Group* g = new Group();
    facade->group = g;
    facade->n_var = (int)n_var; facade->nlmi = (int)nlmi; facade->nlin = (int)nlin;
    *out = facade;
    for (int r = 0; r < world; r++) {
        lrn_options_t o;
        if (opt) o = *opt; else lrn_default_options(&o);
        o.device = dev;
        lrn_handle_t m = nullptr;
        int32_t rc = lrn_create(&m, n_var, nlmi, msizes, nlin, &o);
        if (m) g->members.push_back(m);
        if (rc != LRN_OK) {
            facade->err = m ? m->err : "lrn_create failed for a group member";
            return rc;
        }
    }
    try {
        LRN_CUDA(cudaSetDevice(dev));
        std::vector<DistCtx*> ctx = make_loopback(world);
        for (int r = 0; r < world; r++) {
            lrn_solver* m = g->members[r];
            m->nccl = ctx[r]; m->rank = r; m->world = world;
            m->dist_pw = block_rows > 0 ? block_rows : ((m->n_var >= 16384) ? 512 : (m->n_var >= 4096 ? 256 : 128));
        }
    } catch (const std::exception& e) {
        facade->err = e.what();
        return LRN_ERR_CUDA;
    }
    return LRN_OK;
}

int32_t lrn_dbg_compare(lrn_handle_t a, lrn_handle_t b, int32_t which, double* relerr) {
    if (!a || !b || !relerr || a->group || b->group || a->n_var != b->n_var || a->device != b->device) return LRN_ERR_ARG;
    if (which != LRN_ARR_H && which != LRN_ARR_L) return LRN_ERR_ARG;
    if ((a->rows_local && a->world > 1) || (b->rows_local && b->world > 1)) {
        a->err = "lrn_dbg_compare: a handle keeps only its own Schur rows (own-rows layout)";
        return LRN_ERR_STATE;
    }
    try {
        LRN_CUDA(cudaSetDevice(a->device));
        const DMat& Ma = (which == LRN_ARR_H) ? a->H : a->L;
        const DMat& Mb = (which == LRN_ARR_H) ? b->H : b->L;
        LRN_REQUIRE(Ma.p() && Mb.p(), "Schur matrix is only allocated for kit = 0");
        LRN_CUDA(cudaStreamSynchronize(a->st));
        LRN_CUDA(cudaStreamSynchronize(b->st));
        DevBuf<double> acc(2);
        const int n = a->n_var;
        const unsigned gy = (unsigned)std::min(n, 32768);
        dim3 grid(8, gy, (unsigned)cdiv(n, gy));
        k_lower_diff<<<grid, 256, 0, a->st>>>(Ma.p(), Ma.ld, Mb.p(), Mb.ld, n, acc.p);
        LRN_CHECK_LAUNCH();
        double hst[2] = {0, 0};
        LRN_CUDA(cudaMemcpyAsync(hst, acc.p, sizeof hst, cudaMemcpyDeviceToHost, a->st));
        LRN_CUDA(cudaStreamSynchronize(a->st));
        *relerr = std::sqrt(hst[0]) / std::sqrt(hst[1] > 0 ? hst[1] : 1e-300);
        return LRN_OK;
    } catch (const std::exception& e) {
        a->err = e.what();
        return LRN_ERR_CUDA;
    }
}

int32_t lrn_dbg_gather_H(lrn_handle_t h) {
    LRN_GROUP(h, lrn_dbg_gather_H(m_));
    if (!h) return LRN_ERR_ARG;
    try {
        LRN_CUDA(cudaSetDevice(h->device));
        LRN_REQUIRE(h->H.p(), "Schur matrix is only allocated for kit = 0");
        if (h->rows_local && h->world > 1) {
            h->err = "lrn_dbg_gather_H: the handle keeps only its own Schur rows (own-rows layout)";
            return LRN_ERR_STATE;
        }
        if (h->world > 1 && h->nccl && static_cast<DistCtx*>(h->nccl)->active() && !h->H_gathered) {
            dist_allreduce_sum(h->H.p(), (size_t)h->H.ld * h->n_var, *static_cast<DistCtx*>(h->nccl), h->st);
            LRN_CUDA(cudaStreamSynchronize(h->st));
            h->H_gathered = true;
        }
        return LRN_OK;
    } catch (const std::exception& e) {
        h->err = e.what();
        return LRN_ERR_NCCL;
    }
}

}  // extern "C"
