// NCCL plumbing (one process per GPU).  libnccl is resolved at run time with dlopen so that the library has no
// link-time dependency on a particular NCCL build (torch bundles 2.28.9, the system has 2.27.3).
#pragma once
#include "common.cuh"
#include <nccl.h>
#include <vector>
#include <memory>

namespace lrn {

struct NcclApi {
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    bool ok = false;
};
const NcclApi& nccl_api();   // throws std::runtime_error when libnccl cannot be loaded

struct LoopGroup;                      // in-process loopback transport (tests): see dist.cu

struct DistCtx {
    ncclComm_t comm = nullptr;
    std::shared_ptr<LoopGroup> loop;   // loopback members share one rendezvous (no NCCL; every member on the same device)
    int rank = 0, world = 1;
    bool emulated = false;             // test hook: (rank, world) set without a communicator (assembly ownership only)
    DevBuf<double> xb;                 // broadcast buffer: inverse of the current diagonal block + its 64 x 64 inverse blocks
    DevBuf<double> sendbuf, recvbuf;   // solved row blocks of the current panel: mine / everybody's (ncclAllGather)
    DevBuf<int> infos;                 // world pivot flags
    // ---- peer-memory exchange (NVLink P2P through CUDA IPC or in-process peer access) ------------------------------------
    // Every rank maps the other ranks' xb (diagonal-block inverse), factor matrix L and flag words.  The owner of a diagonal
    // block PUSHES its inverse into every peer's xb and every rank PUSHES its solved row blocks of the panel straight to their
    // final place in every peer's L (no staging, no unpack pass), each followed by a flag store that the receivers poll on.
    int p2p = -1;                      // -1 not tried, 0 unavailable (NCCL broadcast / all-gather are used), 1 active
    std::vector<double*> peer_xb, peer_L;
    std::vector<int*> peer_flags;
    size_t flags_off = 0;              // offset (doubles) of the flag words inside xb
    std::vector<void*> ipc_opened;     // mappings to close
    const double* L_mapped = nullptr;  // the factor matrix the peers mapped (a different matrix needs a new exchange)
    int* flags = nullptr;              // lives at the end of xb (one mapping): [0] X arrived (step stamp); [1 + r] blocks of rank r
                                       // arrived; [63] time-out marker; [64], [65] completion counters of the push kernels
    DevBuf<double*> d_peer_xb, d_peer_L;
    DevBuf<int*> d_peer_flags;
    long long epoch = 0;               // factorisations so far (stamps are epoch * (nblk + 1) + step + 1: never reset)
    // ---- own-rows layout: the factor lives only in the ranks' own row blocks --------------------------------------------
    DevBuf<double> panels;             // solved panels p (all rows, global row index, ld pad_ld(n)), 4 column slots: p & 3
    DevBuf<double> xinv;               // inverse X(p) of every diagonal block (pw x pw each, replicated): the triangular solves
    DevBuf<double> svec;               // pw-long partial sums of the backward solve
    cudaStream_t solve_side = nullptr; // forward solve: updates of the rows below the look-ahead block
    cudaEvent_t solve_ev[2] = {nullptr, nullptr};
    ~DistCtx();
    bool active() const { return comm != nullptr || loop != nullptr; }
    // collectives (NCCL, or the loopback rendezvous); stream-ordered on `st`
    void bcast(double* buf, size_t count, int root, cudaStream_t st);
    void allgather(const void* send, void* recv, size_t bytes_per_rank, cudaStream_t st);
    void allreduce_sum(double* buf, size_t count, cudaStream_t st);
    void allreduce_max(int* buf, size_t count, cudaStream_t st);
};
// `world` loopback members of one in-process group, all on the current device (tests: several ranks on one GPU)
std::vector<DistCtx*> make_loopback(int world);

struct CholWork;
// Distributed right-looking Cholesky, 1-D block-cyclic by ROW blocks of height pw (row block g -> rank g % world).
// On entry every rank holds its OWN row blocks of the lower triangle of A (other rows: don't care).  Step p: the owner of
// diagonal block p factors it and broadcasts the inverse of the factor (<= 2 MB); every rank solves its own rows of column
// panel p with one batched DMMA GEMM; the solved row blocks are exchanged with ONE ncclAllGather (each rank sends 1/world of
// the panel) and stored in place, so every rank ends with the complete factor L (triangular solves run replicated; in the
// own-rows layout below, the panel goes to a panel slot instead and the solves are distributed); every
// rank then updates its own row blocks of the trailing matrix (strided-batch lower-staircase GEMM on the TMA-fed kernel).
// The panel chain of step p+1 runs on a high-priority stream while the main stream still applies the update of step p.
// rows_local: A holds only the rank's own row blocks stacked (local_rows(...) x n, ld lda, ops.cuh); every solved panel is
// gathered into ctx.panels instead of into A, and the trailing updates read it from there.  The inverses X(p) are kept in
// ctx.xinv for chol_solve_dist.  The peer-memory panel push (exchange mode 2) falls back to mode 1.
void cholesky_dist(double* A, int n, int lda, CholWork& work, DistCtx& ctx, int pw, cudaStream_t st, bool rows_local = false);
// Triangular solves with an own-rows factor (after cholesky_dist(..., rows_local = true)); x (n, replicated on entry and on
// exit): which & 1 forward L y = x (fan-out: owner of block p applies X(p), broadcasts y_p, every rank updates its own rows),
// which & 2 backward L' x = y (fan-in: per-rank partial sums of block p, one all-reduce of pw doubles, X(p)').  Collective.
void chol_solve_dist(const double* A, int n, int lda, DistCtx& ctx, int pw, double* x, int which, cudaStream_t st);
// device bytes of the own-rows extras (panel slots, stored inverses, partial sums)
size_t dist_rows_local_bytes(int n, int pw);
// device bytes of the exchange buffers cholesky_dist keeps in its DistCtx
size_t dist_work_bytes(int n, int pw, int world);
// Schur assembly, rank-one path, for the row blocks of one rank:  H[rows g, 0:(g+1) pw] += ((BG)(BG)').^2 (lower staircase)
void syrk_sq_row_blocks(const double* BG, int ldbg, int n, int K, double* H, int ldh, int rank, int world, int pw, cudaStream_t st,
                        bool rows_local = false);
// in-place sum of a device buffer over all ranks
void dist_allreduce_sum(double* buf, size_t count, DistCtx& ctx, cudaStream_t st);

#define LRN_NCCL(call)                                                                         \
    do {                                                                                       \
        ncclResult_t r__ = (call);                                                             \
        if (r__ != ncclSuccess) {                                                              \
            char buf__[512];                                                                   \
            snprintf(buf__, sizeof buf__, "%s:%d: %s -> %s", __FILE__, __LINE__, #call,        \
                     lrn::nccl_api().GetErrorString ? lrn::nccl_api().GetErrorString(r__) : "nccl error"); \
            throw std::runtime_error(buf__);                                                   \
        }                                                                                      \
    } while (0)

}  // namespace lrn
