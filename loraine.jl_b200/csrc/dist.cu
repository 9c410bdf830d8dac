#include "dist.cuh"
#include "solver.cuh"
#include "chol.cuh"
#include "gemm.cuh"
#include <dlfcn.h>
#include <algorithm>
#include <vector>
#include <unistd.h>
#include <memory>
#include <mutex>
#include <condition_variable>
#include <chrono>

namespace lrn {

const NcclApi& nccl_api() {
    static NcclApi api;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* hnd = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!hnd) hnd = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (hnd) {
            auto sym = [&](const char* n) { return dlsym(hnd, n); };
            api.GetUniqueId = (decltype(api.GetUniqueId))sym("ncclGetUniqueId");
            api.CommInitRank = (decltype(api.CommInitRank))sym("ncclCommInitRank");
            api.CommInitAll = (decltype(api.CommInitAll))sym("ncclCommInitAll");
            api.CommDestroy = (decltype(api.CommDestroy))sym("ncclCommDestroy");
            api.Broadcast = (decltype(api.Broadcast))sym("ncclBroadcast");
            api.AllReduce = (decltype(api.AllReduce))sym("ncclAllReduce");
            api.AllGather = (decltype(api.AllGather))sym("ncclAllGather");
            api.GroupStart = (decltype(api.GroupStart))sym("ncclGroupStart");
            api.GroupEnd = (decltype(api.GroupEnd))sym("ncclGroupEnd");
            api.GetErrorString = (decltype(api.GetErrorString))sym("ncclGetErrorString");
            api.ok = api.GetUniqueId && api.CommInitRank && api.Broadcast && api.AllReduce && api.AllGather;
        }
    }
    if (!api.ok) throw std::runtime_error("libnccl.so.2 could not be loaded (needed for multi-GPU runs)");
    return api;
}

// ---- loopback transport ----------------------------------------------------------------------------------------------------
// The members of a loopback group are ordinary handles on ONE device, driven from their own host threads (group_call).  A
// collective is a host rendezvous: every member records a "ready" event on its stream and publishes its buffers; after the
// first barrier each member makes its stream wait for every ready event and enqueues device-to-device copies (or a summing
// kernel) that read the other members' buffers; a "done" event and a second barrier keep every buffer untouched until all
// members have read it.  A member that does not arrive within LOOP_WAIT_S turns into an error instead of a hang.
constexpr int LOOP_WAIT_S = 120;
constexpr int LOOP_MAX_WORLD = 8;
struct LoopGroup {
    int world = 0;
    std::mutex mu;
    std::condition_variable cv;
    int arrived = 0;
    long long gen = 0;
    struct Slot { const void* send = nullptr; void* recv = nullptr; };
    std::vector<Slot> slot;
    std::vector<cudaEvent_t> ready, done;
    std::vector<DevBuf<char>> scratch;          // per member: result of an all-reduce before it is copied in place
    ~LoopGroup() {
        for (auto e : ready) cudaEventDestroy(e);
        for (auto e : done) cudaEventDestroy(e);
    }
    void barrier() {
        std::unique_lock<std::mutex> lk(mu);
        const long long g = gen;
        if (++arrived == world) { arrived = 0; gen++; cv.notify_all(); return; }
        if (!cv.wait_for(lk, std::chrono::seconds(LOOP_WAIT_S), [&] { return gen != g; }))
            throw std::runtime_error("loopback collective: a group member did not arrive within " + std::to_string(LOOP_WAIT_S) + " s");
    }
};

std::vector<DistCtx*> make_loopback(int world) {
    LRN_REQUIRE(world >= 1 && world <= LOOP_MAX_WORLD, "loopback world must be 1..8");
    auto g = std::make_shared<LoopGroup>();
    g->world = world;
    g->slot.resize(world);
    g->ready.resize(world); g->done.resize(world);
    g->scratch.resize(world);
    for (int r = 0; r < world; r++) {
        LRN_CUDA(cudaEventCreateWithFlags(&g->ready[r], cudaEventDisableTiming));
        LRN_CUDA(cudaEventCreateWithFlags(&g->done[r], cudaEventDisableTiming));
    }
    std::vector<DistCtx*> out;
    for (int r = 0; r < world; r++) {
        auto* c = new DistCtx();
        c->rank = r; c->world = world; c->loop = g;
        c->p2p = 0;                               // no peer-memory exchange: nothing spins on a flag
        out.push_back(c);
    }
    return out;
}

namespace {
template <typename T> struct PtrSet { const T* p[LOOP_MAX_WORLD]; };
template <typename T, bool MAX>
__global__ void k_loop_reduce(T* __restrict__ out, PtrSet<T> in, int world, size_t count) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x) {
        T a = in.p[0][i];                         // rank order: every member gets the same bits
        for (int r = 1; r < world; r++) a = MAX ? (in.p[r][i] > a ? in.p[r][i] : a) : a + in.p[r][i];
        out[i] = a;
    }
}
template <typename F>
void loop_collective(DistCtx& c, const void* send, void* recv, cudaStream_t st, F&& body) {
    LoopGroup& g = *c.loop;
    const int r = c.rank;
    LRN_CUDA(cudaEventRecord(g.ready[r], st));
    g.slot[r].send = send; g.slot[r].recv = recv;
    g.barrier();
    for (int s = 0; s < g.world; s++) if (s != r) LRN_CUDA(cudaStreamWaitEvent(st, g.ready[s], 0));
    body(g);
    LRN_CUDA(cudaEventRecord(g.done[r], st));
    g.barrier();
    for (int s = 0; s < g.world; s++) if (s != r) LRN_CUDA(cudaStreamWaitEvent(st, g.done[s], 0));
}
template <typename T, bool MAX>
void loop_allreduce(DistCtx& c, T* buf, size_t count, cudaStream_t st) {
    if (c.world <= 1 || count == 0) return;
    DevBuf<char>& scr = c.loop->scratch[c.rank];
    if (scr.n < count * sizeof(T)) scr.alloc(count * sizeof(T));
    T* tmp = reinterpret_cast<T*>(scr.p);
    loop_collective(c, buf, buf, st, [&](LoopGroup& g) {
        PtrSet<T> ps;
        for (int s = 0; s < g.world; s++) ps.p[s] = static_cast<const T*>(g.slot[s].send);
        k_loop_reduce<T, MAX><<<(unsigned)std::min<long long>(cdiv((long long)count, 256), 4096), 256, 0, st>>>(tmp, ps, g.world, count);
        LRN_CHECK_LAUNCH();
    });
    LRN_CUDA(cudaMemcpyAsync(buf, tmp, count * sizeof(T), cudaMemcpyDeviceToDevice, st));
}
}  // namespace

void DistCtx::bcast(double* buf, size_t count, int root, cudaStream_t st) {
    if (world <= 1 || count == 0) return;
    if (!loop) { LRN_NCCL(nccl_api().Broadcast(buf, buf, count, ncclDouble, root, comm, st)); return; }
    loop_collective(*this, buf, buf, st, [&](LoopGroup& g) {
        if (rank != root)
            LRN_CUDA(cudaMemcpyAsync(buf, g.slot[root].send, count * sizeof(double), cudaMemcpyDeviceToDevice, st));
    });
}
void DistCtx::allgather(const void* send, void* recv, size_t bytes, cudaStream_t st) {
    if (!loop) { LRN_NCCL(nccl_api().AllGather(send, recv, bytes, ncclChar, comm, st)); return; }
    loop_collective(*this, send, recv, st, [&](LoopGroup& g) {
        for (int s = 0; s < g.world; s++)
            LRN_CUDA(cudaMemcpyAsync(static_cast<char*>(recv) + (size_t)s * bytes, g.slot[s].send, bytes, cudaMemcpyDeviceToDevice, st));
    });
}
void DistCtx::allreduce_sum(double* buf, size_t count, cudaStream_t st) {
    if (!loop) { LRN_NCCL(nccl_api().AllReduce(buf, buf, count, ncclDouble, ncclSum, comm, st)); return; }
    loop_allreduce<double, false>(*this, buf, count, st);
}
void DistCtx::allreduce_max(int* buf, size_t count, cudaStream_t st) {
    if (!loop) { LRN_NCCL(nccl_api().AllReduce(buf, buf, count, ncclInt32, ncclMax, comm, st)); return; }
    loop_allreduce<int, true>(*this, buf, count, st);
}

DistCtx::~DistCtx() {
    for (void* m : ipc_opened) cudaIpcCloseMemHandle(m);
    ipc_opened.clear();
    if (solve_side) { cudaStreamSynchronize(solve_side); cudaStreamDestroy(solve_side); solve_side = nullptr; }
    for (auto& e : solve_ev) if (e) { cudaEventDestroy(e); e = nullptr; }
    if (comm && nccl_api().CommDestroy) nccl_api().CommDestroy(comm);
    comm = nullptr;
}

namespace {
// recv[r][z] (pw x pw, ld pw) holds row block g = first_r + z * world of column panel p as solved by rank r; store every
// block at its place in L.  grid = (row chunks, w columns, world * maxcnt slots)
__global__ void k_unpack_blocks(const double* __restrict__ recv, double* __restrict__ L, int lda, int n, int c0, int w, int pw, int p,
                                int world, int maxcnt, int nblk) {
    const int slot = blockIdx.z, r = slot / maxcnt, z = slot - r * maxcnt;
    const int first = p + ((r - p % world + world) % world);
    const int g = first + z * world;
    if (g >= nblk) return;
    const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
    const int row = g * pw + i;
    if (i >= pw || row >= n || j >= w) return;
    L[(size_t)(c0 + j) * lda + row] = recv[((size_t)slot * pw + j) * pw + i];
}
// own-rows layout: the same blocks go to the panel slot P (global rows, ld ldp); the rank's own blocks also to its local rows
// of A (column c0 + j, local row (g / world) pw + i)
__global__ void k_unpack_panel(const double* __restrict__ recv, double* __restrict__ P, int ldp, double* __restrict__ A, int lda,
                               int n, int c0, int w, int pw, int p, int world, int self, int maxcnt, int nblk) {
    const int slot = blockIdx.z, r = slot / maxcnt, z = slot - r * maxcnt;
    const int first = p + ((r - p % world + world) % world);
    const int g = first + z * world;
    if (g >= nblk) return;
    const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
    const int row = g * pw + i;
    if (i >= pw || row >= n || j >= w) return;
    const double v = recv[((size_t)slot * pw + j) * pw + i];
    P[(size_t)j * ldp + row] = v;
    if (r == self) A[(size_t)(c0 + j) * lda + (g / world) * pw + i] = v;
}
__global__ void k_min_nonzero(int* a, const int* b, int cnt) {
    int best = 0;
    for (int r = 0; r < cnt; r++) if (b[r] != 0 && (best == 0 || b[r] < best)) best = b[r];
    *a = best;
}
__global__ void k_copy_block(const double* __restrict__ src, int lds, double* __restrict__ dst, int ldd, int rows, int cols) {
    int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
    if (i < rows && j < cols) dst[(size_t)j * ldd + i] = src[(size_t)j * lds + i];
}

// ---- peer-memory exchange kernels ------------------------------------------------------------------------------------------
constexpr long long P2P_SPIN_LIMIT = 4000000000LL;     // ~2 s of SM clocks: a lost peer must not hang the GPU

// copy `count` doubles (multiple of 2) from src to the same offset of every peer buffer, then publish `stamp` in every peer's
// flag word `slot` (the last CTA to finish does it, after a system-wide fence)
__global__ void k_push_vec(const double* src, double* const* __restrict__ peers, int world, int self, size_t dst_off, size_t count,
                           int* const* __restrict__ peer_flags, int slot, int stamp, unsigned int* __restrict__ done_ctr) {
    const size_t n2 = count / 2;
    const double2* s2 = reinterpret_cast<const double2*>(src);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += (size_t)gridDim.x * blockDim.x) {
        const double2 v = s2[i];
        for (int r = 0; r < world; r++)
            if (r != self) reinterpret_cast<double2*>(peers[r] + dst_off)[i] = v;
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int prev = atomicAdd(done_ctr, 1u);
        if (prev == gridDim.x - 1) {
            *done_ctr = 0;
            __threadfence_system();
            for (int r = 0; r < world; r++) *reinterpret_cast<volatile int*>(peer_flags[r] + slot) = stamp;
        }
    }
}
// my solved row blocks of panel p (send[z], pw x w, ld pw; block g = first + z * world) -> every peer's L at their final place
__global__ void k_push_blocks(const double* __restrict__ send, double* const* __restrict__ peers, int world, int lda, int n, int c0,
                              int w, int pw, int first, int cnt, int* const* __restrict__ peer_flags, int slot, int stamp,
                              unsigned int* __restrict__ done_ctr) {
    // grid: (row pairs of a block, column, slot z)
    const int z = blockIdx.z, j = blockIdx.y;
    const int g = first + z * world;
    const int i = 2 * (blockIdx.x * blockDim.x + threadIdx.x);
    const int row = g * pw + i;
    if (z < cnt && j < w && i < pw && row < n) {
        const double* sp_ = send + ((size_t)z * pw + j) * pw + i;
        const size_t off = (size_t)(c0 + j) * lda + row;
        if (row + 1 < n && i + 1 < pw) {
            const double2 v = *reinterpret_cast<const double2*>(sp_);
            for (int r = 0; r < world; r++) *reinterpret_cast<double2*>(peers[r] + off) = v;
        } else {
            const double v = *sp_;
            for (int r = 0; r < world; r++) peers[r][off] = v;
        }
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int total = gridDim.x * gridDim.y * gridDim.z;
        const unsigned int prev = atomicAdd(done_ctr, 1u);
        if (prev == total - 1) {
            *done_ctr = 0;
            __threadfence_system();
            for (int r = 0; r < world; r++) *reinterpret_cast<volatile int*>(peer_flags[r] + slot) = stamp;
        }
    }
}
// wait until flags[slot0 .. slot0 + nslots) have all reached `stamp` (written by the peers over NVLink)
__global__ void k_wait_flags(volatile int* flags, int slot0, int nslots, int stamp) {
    const int t = threadIdx.x;
    if (t < nslots) {
        const long long t0 = clock64();
        while (flags[slot0 + t] < stamp) {
            if (clock64() - t0 > P2P_SPIN_LIMIT) { flags[63] = 1; break; }
        }
    }
    __threadfence_system();
}

__global__ void k_check_timeout(int* flags, int* info) {
    if (flags[63] != 0) { *info = -77; flags[63] = 0; }
}

struct IpcPacket {
    cudaIpcMemHandle_t hx, hl;
    unsigned long long px, pl;          // raw pointers (same-process peers)
    unsigned long long ox, ol;          // byte offsets of the buffers inside their underlying allocations (IPC maps the base)
    long long pid;
    int dev, pad;
};

// offset of a device pointer inside the allocation cudaIpcGetMemHandle exports (cuMemGetAddressRange, resolved at run time)
size_t alloc_offset(const void* ptr) {
    typedef int (*fn_t)(unsigned long long*, size_t*, unsigned long long);
    static fn_t fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* hnd = dlopen("libcuda.so.1", RTLD_NOW | RTLD_GLOBAL);
        if (hnd) fn = (fn_t)dlsym(hnd, "cuMemGetAddressRange_v2");
    });
    unsigned long long base = 0;
    size_t size = 0;
    if (fn && fn(&base, &size, (unsigned long long)ptr) == 0 && base) return (size_t)((unsigned long long)ptr - base);
    return 0;
}

// One-time (per factor matrix) exchange of the buffer mappings.  Collective.  Leaves ctx.p2p = 1 on success on ALL ranks,
// 0 otherwise (agreed with a max-reduction so that no rank takes the peer path alone).
void setup_p2p(DistCtx& ctx, double* L, cudaStream_t st) {
    const int world = ctx.world;
    ctx.flags = reinterpret_cast<int*>(ctx.xb.p + ctx.flags_off);
    if (ctx.loop) { ctx.p2p = 0; ctx.L_mapped = L; return; }      // loopback: copies only, no peer mapping, no spin-waits
    const char* env = getenv("LRN_DIST_P2P");
    int ok = (env && atoi(env) == 0) ? 0 : 1;
    if (world < 2) ok = 0;
    for (void* m : ctx.ipc_opened) cudaIpcCloseMemHandle(m);
    ctx.ipc_opened.clear();
    IpcPacket mine;
    std::memset(&mine, 0, sizeof mine);
    int dev = 0;
    cudaGetDevice(&dev);
    mine.dev = dev;
    mine.pid = (long long)getpid();
    mine.px = (unsigned long long)ctx.xb.p; mine.pl = (unsigned long long)L;
    mine.ox = alloc_offset(ctx.xb.p); mine.ol = alloc_offset(L);
    if (ok) {
        if (cudaIpcGetMemHandle(&mine.hx, ctx.xb.p) != cudaSuccess || cudaIpcGetMemHandle(&mine.hl, L) != cudaSuccess) {
            cudaGetLastError();
            mine.pid = -1;                       // this rank cannot export: everybody falls back
        }
    }
    static_assert(sizeof(IpcPacket) <= 256, "IpcPacket must fit the exchange slot");
    DevBuf<char> sb(256), rb((size_t)256 * world);
    LRN_CUDA(cudaMemcpyAsync(sb.p, &mine, sizeof mine, cudaMemcpyHostToDevice, st));
    ctx.allgather(sb.p, rb.p, 256, st);
    std::vector<char> all((size_t)256 * world);
    LRN_CUDA(cudaMemcpyAsync(all.data(), rb.p, all.size(), cudaMemcpyDeviceToHost, st));
    LRN_CUDA(cudaStreamSynchronize(st));
    ctx.peer_xb.assign(world, nullptr); ctx.peer_L.assign(world, nullptr); ctx.peer_flags.assign(world, nullptr);
    for (int r = 0; r < world && ok; r++) {
        IpcPacket pk;
        std::memcpy(&pk, all.data() + (size_t)256 * r, sizeof pk);
        if (pk.pid < 0) { ok = 0; break; }
        if (r == ctx.rank) {
            ctx.peer_xb[r] = ctx.xb.p; ctx.peer_L[r] = L;
        } else if (pk.pid == mine.pid) {         // same process (lrn_create_multi): plain peer access
            int can = 0;
            cudaDeviceCanAccessPeer(&can, dev, pk.dev);
            if (!can) { ok = 0; break; }
            cudaError_t e = cudaDeviceEnablePeerAccess(pk.dev, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); ok = 0; break; }
            cudaGetLastError();
            ctx.peer_xb[r] = (double*)pk.px; ctx.peer_L[r] = (double*)pk.pl;
        } else {
            void *mx = nullptr, *ml = nullptr;
            if (cudaIpcOpenMemHandle(&mx, pk.hx, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess ||
                cudaIpcOpenMemHandle(&ml, pk.hl, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
                cudaGetLastError();
                for (void* m : {mx, ml}) if (m) cudaIpcCloseMemHandle(m);
                ok = 0;
                break;
            }
            ctx.ipc_opened.push_back(mx); ctx.ipc_opened.push_back(ml);
            ctx.peer_xb[r] = (double*)((char*)mx + pk.ox); ctx.peer_L[r] = (double*)((char*)ml + pk.ol);
        }
        ctx.peer_flags[r] = reinterpret_cast<int*>(ctx.peer_xb[r] + ctx.flags_off);
    }
    // agree: every rank must have succeeded
    int* dflag = ctx.infos.p;
    const int bad = ok ? 0 : 1;
    LRN_CUDA(cudaMemcpyAsync(dflag, &bad, sizeof(int), cudaMemcpyHostToDevice, st));
    ctx.allreduce_max(dflag, 1, st);
    int anybad = 1;
    LRN_CUDA(cudaMemcpyAsync(&anybad, dflag, sizeof(int), cudaMemcpyDeviceToHost, st));
    LRN_CUDA(cudaStreamSynchronize(st));
    ctx.p2p = anybad ? 0 : ((env && atoi(env) >= 2) ? 2 : 1);
    ctx.L_mapped = L;
    if (ctx.p2p) {
        ctx.d_peer_xb.upload(ctx.peer_xb, st); ctx.d_peer_L.upload(ctx.peer_L, st); ctx.d_peer_flags.upload(ctx.peer_flags, st);
        LRN_CUDA(cudaMemsetAsync(ctx.flags, 0, 66 * sizeof(int), st));
        LRN_CUDA(cudaStreamSynchronize(st));
        // nobody may push before everybody has cleared its flags
        ctx.allreduce_max(dflag, 1, st);
        LRN_CUDA(cudaStreamSynchronize(st));
        ctx.epoch = 0;
    }
    if (getenv("LRN_DIST_TRACE") && ctx.rank == 0)
        fprintf(stderr, "[lrn dist] exchange mode %d: %s\n", ctx.p2p,
                ctx.p2p == 2 ? "inverse and solved panel pushed over peer memory" :
                ctx.p2p == 1 ? "inverse pushed over peer memory, solved panel through ncclAllGather" : "NCCL broadcast / all-gather");
}

// first row block >= p owned by `rank`, and how many of its blocks are >= p
inline int first_block(int p, int rank, int world) { return p + ((rank - p % world + world) % world); }
inline int count_blocks(int p, int rank, int world, int nblk) {
    const int f = first_block(p, rank, world);
    return f >= nblk ? 0 : (nblk - 1 - f) / world + 1;
}

// C[rows of my blocks g >= gmin, cols [cbeg, cend)] (+)= alpha * f(A[rows, 0:K] * Bm[cbeg:cend, 0:K]^T); `lower` clips every row
// block at its own diagonal block (staircase).  Whole blocks go through one strided-batch launch, a partial last block through
// a second one.
// c_local: C holds the rank's own row blocks stacked (own-rows layout): block g sits at local row (g / world) pw, the batch
// stride is pw; the lower-tile test keeps the global rows.
void row_block_gemm(cudaStream_t st, int n, int pw, int rank, int world, int gmin, const double* A, int lda, const double* Bm,
                    int ldb, double* C, int ldc, int cbeg, int cend, int K, double alpha, double beta, int mode, bool lower,
                    bool c_local = false) {
    const int nblk = (int)cdiv(n, pw);
    const int f = first_block(gmin, rank, world);
    if (f >= nblk || cend <= cbeg) return;
    const int cnt = (nblk - 1 - f) / world + 1;
    const int glast = f + (cnt - 1) * world;
    const bool last_partial = (glast == nblk - 1) && (n - glast * pw < pw);
    const int nfull = last_partial ? cnt - 1 : cnt;
    auto crow = [&](int g) { return (size_t)(c_local ? (g / world) * pw : g * pw); };
    auto base = [&](GemmParams& g) {
        g.B = Bm + cbeg; g.ldb = ldb; g.lda = lda; g.ldc = ldc; g.K = K; g.transB = true;
        g.alpha = alpha; g.beta = beta; g.mode = mode; g.lower = lower ? 1 : 0; g.col0 = cbeg;
    };
    if (nfull > 0) {
        GemmParams g;
        base(g);
        const int gl = f + (nfull - 1) * world;
        g.A = A + (size_t)f * pw; g.C = C + (size_t)cbeg * ldc + crow(f);
        g.M = pw; g.N = (lower ? std::min(cend, (gl + 1) * pw) : cend) - cbeg;
        g.batch = nfull; g.sA = (long long)world * pw; g.sC = c_local ? (long long)pw : (long long)world * pw; g.sB = 0;
        g.row0 = f * pw; g.row0z = (long long)world * pw;
        if (g.N > 0) gemm(g, st);
    }
    if (last_partial) {
        GemmParams g;
        base(g);
        g.A = A + (size_t)glast * pw; g.C = C + (size_t)cbeg * ldc + crow(glast);
        g.M = n - glast * pw; g.N = cend - cbeg; g.row0 = glast * pw;
        gemm(g, st);
    }
}
}  // namespace

void dist_allreduce_sum(double* buf, size_t count, DistCtx& ctx, cudaStream_t st) { ctx.allreduce_sum(buf, count, st); }

void syrk_sq_row_blocks(const double* BG, int ldbg, int n, int K, double* H, int ldh, int rank, int world, int pw, cudaStream_t st,
                        bool rows_local) {
    row_block_gemm(st, n, pw, rank, world, 0, BG, ldbg, BG, ldbg, H, ldh, 0, n, K, 1.0, 1.0, 1, true, rows_local);
}

namespace {
// buffer sizes (doubles) of cholesky_dist
struct DistBufs {
    size_t xb, send, recv;
    DistBufs(int n, int pw, int world) {
        const size_t blk = (size_t)pw * pw, ndmax = (size_t)(pw / CHOL_DB) * CHOL_DB * CHOL_DB;
        const size_t maxcnt0 = (size_t)cdiv(cdiv(n, pw), world);
        // two inverse buffers of X | 64 x 64 inverse blocks | scratch of the inversion (step parity: X(p+1) is produced while
        // X(p) is still being used) + flag words of the peer exchange
        xb = 2 * (2 * blk + ndmax) + 64;
        send = maxcnt0 * blk;
        recv = send * world;
    }
};
}  // namespace

size_t dist_rows_local_bytes(int n, int pw) {
    const size_t nblk = (size_t)cdiv(n, pw);
    return ((size_t)4 * pad_ld(n) * pw + nblk * pw * pw + pw) * sizeof(double);
}

size_t dist_work_bytes(int n, int pw, int world) {
    const DistBufs b(n, pw, world);
    return (b.xb + b.send + b.recv) * sizeof(double) + (size_t)world * sizeof(int);
}

void cholesky_dist(double* A, int n, int lda, CholWork& work, DistCtx& ctx, int pw, cudaStream_t st, bool rows_local) {
    work.tinv_for = nullptr;   // the triangular solves rebuild their diagonal-block inverses from the new factor
    work.ensure(n);
    LRN_REQUIRE(pw % CHOL_DB == 0 && pw <= 512, "row block height must be a multiple of 64, at most 512");
    LRN_REQUIRE(ctx.active(), "no NCCL communicator (lrn_dist_init)");
    const int world = ctx.world, rank = ctx.rank;
    const int nblk = (int)cdiv(n, pw);
    const size_t blk = (size_t)pw * pw, ndmax = (size_t)(pw / CHOL_DB) * CHOL_DB * CHOL_DB;
    const size_t xhalf = 2 * blk + ndmax;            // one inverse buffer: X | 64 x 64 inverse blocks | scratch of the inversion
    const DistBufs bufs(n, pw, world);
    if (ctx.xb.n < bufs.xb) { ctx.xb.alloc(bufs.xb); ctx.flags_off = 2 * xhalf; ctx.p2p = -1; }
    if (ctx.sendbuf.n < bufs.send) ctx.sendbuf.alloc(bufs.send);
    if (ctx.recvbuf.n < bufs.recv) ctx.recvbuf.alloc(bufs.recv);
    if (ctx.infos.n < (size_t)world) ctx.infos.alloc(world);
    if (ctx.p2p < 0 || (ctx.p2p >= 1 && ctx.L_mapped != A)) setup_p2p(ctx, A, st);     // collective, once per factor matrix
    // exchange mode: 0 NCCL only; 1 (default) the 2 MB inverse travels over peer memory (latency-bound), the solved panel through
    // ncclAllGather (bandwidth-bound: NCCL replicates inside the NVSwitch, a peer push sends world-1 copies); 2 everything pushed
    // (not in the own-rows layout: the peers hold no place for a whole panel in their factor, mode 1 is used instead)
    const int mode = (rows_local && ctx.p2p >= 2) ? 1 : ctx.p2p;
    const bool push_x = mode >= 1, push_panel = mode >= 2;
    // own-rows layout: local row of a global row, panel slots (p & 3: the pair p-1, p of an odd step is side by side, and the
    // slot that panel p+1 lands in is never read by the update of step p), stored inverses
    auto loc = [&](int row) { return rows_local ? (size_t)((row / pw) / world) * pw + row % pw : (size_t)row; };
    const int ldp = pad_ld(n);
    if (rows_local) {
        if (ctx.panels.n < (size_t)4 * ldp * pw) ctx.panels.alloc((size_t)4 * ldp * pw);
        if (ctx.xinv.n < (size_t)nblk * blk) ctx.xinv.alloc((size_t)nblk * blk);
    }
    auto panel = [&](int p) { return ctx.panels.p + (size_t)(p & 3) * pw * ldp; };
    const int stamp0 = (int)(ctx.epoch * (nblk + 1));
    unsigned int* ctr0 = reinterpret_cast<unsigned int*>(ctx.flags ? ctx.flags + 64 : nullptr);
    unsigned int* ctr1 = reinterpret_cast<unsigned int*>(ctx.flags ? ctx.flags + 65 : nullptr);
    ensure_aux(work);
    cudaStream_t sp = work.aux;    // panel stream: X arrival, row solves, exchange of the solved panel
    cudaStream_t sq = work.aux2;   // diagonal stream: early update + factorisation + inversion of the NEXT diagonal block
    cudaEvent_t evStart = work.ev[0], evU = work.ev[1], evB = work.ev[2], evS = work.ev[3], evD = work.ev[4], evU2 = work.ev[5];
    int* info = work.info_ptr();
    LRN_CUDA(cudaMemsetAsync(info, 0, sizeof(int), st));
    LRN_CUDA(cudaEventRecord(evStart, st));
    LRN_CUDA(cudaStreamWaitEvent(sp, evStart, 0));
    LRN_CUDA(cudaStreamWaitEvent(sq, evStart, 0));
    // optional timeline (LRN_DIST_TRACE=1): CUDA events around every stage of the panel chain and of the update, summed per stage
    static const bool trace = getenv("LRN_DIST_TRACE") != nullptr;
    struct Ev { cudaEvent_t e; int stage; };
    std::vector<Ev> tev;
    auto mark = [&](cudaStream_t s_, int stage) {
        if (!trace) return;
        Ev v; v.stage = stage;
        LRN_CUDA(cudaEventCreate(&v.e));
        LRN_CUDA(cudaEventRecord(v.e, s_));
        tev.push_back(v);
    };
    auto xbuf = [&](int p) { return ctx.xb.p + (size_t)(p & 1) * xhalf; };
    // factor diagonal block q (already fully updated), build the inverse of its factor and hand it to the other ranks
    auto factor_and_publish = [&](int q) {
        const int c0 = q * pw, w = std::min(pw, n - c0);
        double* X = xbuf(q);
        double* dk = work.dinv.p + (size_t)(c0 / CHOL_DB) * CHOL_DB * CHOL_DB;
        const int nd = (int)cdiv(w, CHOL_DB) * CHOL_DB * CHOL_DB;
        chol_diag_block(A + (size_t)c0 * lda + loc(c0), lda, w, dk, X, pw, X + blk + ndmax, info, c0, sq);
        LRN_CUDA(cudaMemcpyAsync(X + blk, dk, (size_t)nd * sizeof(double), cudaMemcpyDeviceToDevice, sq));
        if (push_x) {
            k_push_vec<<<96, 256, 0, sq>>>(X, ctx.d_peer_xb.p, world, rank, (size_t)(q & 1) * xhalf, blk + ndmax, ctx.d_peer_flags.p, 0,
                                           stamp0 + q + 1, ctr0);
            LRN_CHECK_LAUNCH();
        }
        LRN_CUDA(cudaEventRecord(evD, sq));
    };
    if (rank == 0 % world) factor_and_publish(0);
    for (int p = 0; p < nblk; p++) {
        const int c0 = p * pw, w = std::min(pw, n - c0), owner = p % world;
        double* X = xbuf(p);
        double* xd = X + blk;
        double* dk = work.dinv.p + (size_t)(c0 / CHOL_DB) * CHOL_DB * CHOL_DB;
        const int nd = (int)cdiv(w, CHOL_DB) * CHOL_DB * CHOL_DB;
        const int stamp = stamp0 + p + 1;
        // ---- panel chain of step p ------------------------------------------------------------------------------------
        if (p > 0) LRN_CUDA(cudaStreamWaitEvent(sp, evU, 0));             // my rows of column block p have the update of step p-1
        mark(sp, 0);
        if (rank == owner) LRN_CUDA(cudaStreamWaitEvent(sp, evD, 0));     // (my own factorisation of block p, on the diagonal stream)
        mark(sp, 1);
        if (push_x) {
            if (rank != owner) {                                          // the owner pushed X(p) into xbuf(p) and raised flag 0
                k_wait_flags<<<1, 32, 0, sp>>>(ctx.flags, 0, 1, stamp);
                LRN_CHECK_LAUNCH();
            }
        } else if (world > 1) {
            ctx.bcast(X, blk + ndmax, owner, sp);
        }
        if (rows_local) LRN_CUDA(cudaMemcpyAsync(ctx.xinv.p + (size_t)p * blk, X, blk * sizeof(double), cudaMemcpyDeviceToDevice, sp));
        if (rank != owner) LRN_CUDA(cudaMemcpyAsync(dk, xd, (size_t)nd * sizeof(double), cudaMemcpyDeviceToDevice, sp));
        mark(sp, 2);
        const int maxcnt = (int)cdiv(nblk - p, world);
        const int f = first_block(p, rank, world), cnt = count_blocks(p, rank, world, nblk);
        if (p + 1 < nblk || world > 1) {
            // my row blocks g > p of the panel:  send[z] = A[g rows, panel p] * X^T ; the owner's slot 0 is the diagonal block itself
            const int z0 = (rank == owner) ? 1 : 0;
            if (rank == owner) {
                dim3 grid((unsigned)cdiv(w, 256), (unsigned)w);
                k_copy_block<<<grid, 256, 0, sp>>>(A + (size_t)c0 * lda + loc(c0), lda, ctx.sendbuf.p, pw, w, w);
                LRN_CHECK_LAUNCH();
            }
            if (cnt > z0) {
                const int glast = f + (cnt - 1) * world;
                const bool last_partial = (glast == nblk - 1) && (n - glast * pw < pw);
                const int nfull = (last_partial ? cnt - 1 : cnt) - z0;
                if (nfull > 0) {
                    GemmParams g;
                    g.A = A + (size_t)c0 * lda + loc((f + z0 * world) * pw); g.lda = lda;
                    g.sA = rows_local ? (long long)pw : (long long)world * pw;
                    g.B = X; g.ldb = pw; g.transB = true;
                    g.C = ctx.sendbuf.p + (size_t)z0 * blk; g.ldc = pw; g.sC = (long long)blk;
                    g.M = pw; g.N = w; g.K = w; g.batch = nfull;
                    gemm(g, sp);
                }
                if (last_partial && glast > p) {
                    GemmParams g;
                    g.A = A + (size_t)c0 * lda + loc(glast * pw); g.lda = lda;
                    g.B = X; g.ldb = pw; g.transB = true;
                    g.C = ctx.sendbuf.p + (size_t)(cnt - 1) * blk; g.ldc = pw;
                    g.M = n - glast * pw; g.N = w; g.K = w;
                    gemm(g, sp);
                }
            }
        }
        LRN_CUDA(cudaEventRecord(evS, sp));
        mark(sp, 3);
        // ---- diagonal stream: the owner of block p+1 has just solved ITS OWN rows of panel p, which is all the update of its
        //      diagonal block needs: update, factor, invert and publish X(p+1) while the panel of step p is still being exchanged
        if (p + 1 < nblk && rank == (p + 1) % world) {
            const int c1 = c0 + pw, hb1 = std::min(pw, n - c1);
            LRN_CUDA(cudaStreamWaitEvent(sq, evS, 0));
            if (p > 0) LRN_CUDA(cudaStreamWaitEvent(sq, evU2, 0));        // column block p+1 has the update of step p-1
            const double* Srow = ctx.sendbuf.p + (size_t)((p + 1 - f) / world) * blk;     // my solved block g = p+1
            GemmParams g;
            g.A = Srow; g.B = Srow; g.C = A + (size_t)c1 * lda + loc(c1);
            g.M = hb1; g.N = hb1; g.K = w; g.lda = pw; g.ldb = pw; g.ldc = lda;
            g.transB = true; g.alpha = -1.0; g.beta = 1.0; g.lower = 1;
            gemm(g, sq);
            factor_and_publish(p + 1);
        }
        // ---- exchange of the solved panel -----------------------------------------------------------------------------------
        if (p + 1 < nblk || world > 1) {
            if (push_panel) {
                // every rank stores its solved blocks at their final place in EVERY rank's L (its own included) over NVLink,
                // raises flag 1 + rank everywhere, then waits until the blocks of all ranks have landed here
                dim3 grid((unsigned)cdiv(pw / 2, 128), (unsigned)w, (unsigned)std::max(cnt, 1));
                k_push_blocks<<<grid, 128, 0, sp>>>(ctx.sendbuf.p, ctx.d_peer_L.p, world, lda, n, c0, w, pw, f, cnt, ctx.d_peer_flags.p,
                                                    1 + rank, stamp, ctr1);
                LRN_CHECK_LAUNCH();
                mark(sp, 4);
                k_wait_flags<<<1, 64, 0, sp>>>(ctx.flags, 1, world, stamp);
                LRN_CHECK_LAUNCH();
            } else {
                const double* src = ctx.sendbuf.p;
                if (world > 1) {
                    ctx.allgather(ctx.sendbuf.p, ctx.recvbuf.p, (size_t)maxcnt * blk * sizeof(double), sp);
                    src = ctx.recvbuf.p;
                }
                mark(sp, 4);
                dim3 grid((unsigned)cdiv(pw, 256), (unsigned)w, (unsigned)(world * maxcnt));
                if (rows_local) k_unpack_panel<<<grid, 256, 0, sp>>>(src, panel(p), ldp, A, lda, n, c0, w, pw, p, world, rank, maxcnt, nblk);
                else k_unpack_blocks<<<grid, 256, 0, sp>>>(src, A, lda, n, c0, w, pw, p, world, maxcnt, nblk);
                LRN_CHECK_LAUNCH();
            }
            mark(sp, 5);
        }
        LRN_CUDA(cudaEventRecord(evB, sp));
        LRN_CUDA(cudaStreamWaitEvent(st, evB, 0));
        if (p + 1 >= nblk) break;
        // ---- trailing update on the main stream.  Two column blocks ahead first: column block p+1 (my rows are solved next; its
        //      diagonal block was already updated on the diagonal stream) and column block p+2 (its diagonal block is factored
        //      during step p+1).  The REST of the trailing matrix is updated every second step only, with the two panels p-1, p at
        //      once (K = 2 pw: half as many C-tile read-modify-write epilogues and pipeline fills per flop on the TMA-fed kernel):
        //        even step p : columns p+1, p+2 with panel p                                         (rest deferred)
        //        odd step p  : column p+1 with panel p, column p+2 with panels p-1..p, rest (>= p+3) with panels p-1..p
        const double* P = rows_local ? panel(p) : A + (size_t)c0 * lda;   // column panel p: rows are global
        const int lp = rows_local ? ldp : lda;
        const bool cl = rows_local;
        const int c1 = c0 + pw, c2 = std::min(n, c1 + pw), c3 = std::min(n, c2 + pw);
        const bool pair_rest = (pw % 32 == 0);                             // (always: pw is 128, 256 or 512)
        mark(st, 10);
        if (!(p & 1) || !pair_rest) {
            // (one launch for both look-ahead column blocks: N = 2 pw keeps the strided-batch product on the TMA-fed kernel)
            row_block_gemm(st, n, pw, rank, world, p + 2, P, lp, P, lp, A, lda, c1, c3, w, -1.0, 1.0, 0, true, cl);
            LRN_CUDA(cudaEventRecord(evU, st));
            LRN_CUDA(cudaEventRecord(evU2, st));
            mark(st, 11);
            const bool last_even_with_rest = pair_rest && (p + 2 >= nblk);   // no odd step follows that could take the rest
            if ((!pair_rest || last_even_with_rest) && c3 < n)
                row_block_gemm(st, n, pw, rank, world, p + 3, P, lp, P, lp, A, lda, c3, n, w, -1.0, 1.0, 0, true, cl);
        } else {
            const double* P2 = P - (size_t)pw * lp;                        // panels p-1 and p side by side: K = 2 pw
            row_block_gemm(st, n, pw, rank, world, p + 2, P, lp, P, lp, A, lda, c1, c2, w, -1.0, 1.0, 0, true, cl);
            LRN_CUDA(cudaEventRecord(evU, st));
            if (c2 < n) row_block_gemm(st, n, pw, rank, world, p + 2, P2, lp, P2, lp, A, lda, c2, c3, pw + w, -1.0, 1.0, 0, true, cl);
            LRN_CUDA(cudaEventRecord(evU2, st));
            mark(st, 11);
            if (c3 < n) row_block_gemm(st, n, pw, rank, world, p + 3, P2, lp, P2, lp, A, lda, c3, n, pw + w, -1.0, 1.0, 0, true, cl);
        }
        mark(st, 12);
    }
    LRN_CUDA(cudaEventRecord(evD, sq));
    LRN_CUDA(cudaStreamWaitEvent(st, evD, 0));
    if (trace) {
        LRN_CUDA(cudaStreamSynchronize(sp));
        LRN_CUDA(cudaStreamSynchronize(sq));
        LRN_CUDA(cudaStreamSynchronize(st));
        // stage sums on the panel stream: 0->1 wait for my own diagonal block, 1->2 X arrival, 2->3 row solves, 3->4 exchange,
        // 4->5 unpack / flag wait, 5->next 0 wait for the update of the main stream
        double sum[16] = {0};
        for (size_t i = 0; i + 1 < tev.size(); i++) {
            const int a = tev[i].stage, b2 = tev[i + 1].stage;
            float ms = 0.f;
            if (b2 == a + 1 && a != 5) { cudaEventElapsedTime(&ms, tev[i].e, tev[i + 1].e); sum[a] += ms; }
        }
        const Ev* last5 = nullptr;
        for (auto& v : tev) {
            if (v.stage == 5) last5 = &v;
            if (v.stage == 0 && last5) { float ms = 0.f; cudaEventElapsedTime(&ms, last5->e, v.e); sum[6] += ms; last5 = nullptr; }
        }
        float total = 0.f;
        if (!tev.empty()) cudaEventElapsedTime(&total, tev.front().e, tev.back().e);
        if (rank == 0)
            fprintf(stderr, "[lrn dist trace] world %d n %d mode %d: own-diag wait %.2f  X arrival %.2f  solve %.2f  exchange %.2f  unpack/flags %.2f  "
                            "panel-stream wait %.2f | 2 look-ahead column blocks %.2f  rest update %.2f | first-to-last event %.2f ms\n",
                    world, n, mode, sum[0], sum[1], sum[2], sum[3], sum[4], sum[6], sum[10], sum[11], total);
        for (auto& v : tev) cudaEventDestroy(v.e);
    }
    ctx.epoch++;
    if (push_x) {                                  // a peer that never answered: report instead of returning a wrong factor
        k_check_timeout<<<1, 1, 0, st>>>(ctx.flags, info);
        LRN_CHECK_LAUNCH();
    }
    // the first failing pivot index is known to the owner of that block only: take the smallest non-zero over ranks
    if (world > 1) {
        ctx.allgather(info, ctx.infos.p, sizeof(int), st);
        k_min_nonzero<<<1, 1, 0, st>>>(info, ctx.infos.p, world);
        LRN_CHECK_LAUNCH();
    }
}

// ---- triangular solves with an own-rows factor --------------------------------------------------------------------------
namespace {
constexpr int TS_THREADS = 512;
// x[0:w] <- X x[0:w]  (X = inverse of the lower diagonal block, ld pw; one CTA)
__global__ void __launch_bounds__(TS_THREADS) k_ts_fwd_diag(const double* __restrict__ X, int w, int pw, double* __restrict__ x) {
    __shared__ double r[512];
    for (int i = threadIdx.x; i < w; i += blockDim.x) r[i] = x[i];
    __syncthreads();
    for (int i = threadIdx.x; i < w; i += blockDim.x) {
        double a = 0.0;
        for (int j = 0; j <= i; j++) a = fma(X[(size_t)j * pw + i], r[j], a);
        x[i] = a;
    }
}
// x[0:w] <- X' (x[0:w] - s[0:w])  (one warp per output: lanes read a column of X)
__global__ void __launch_bounds__(TS_THREADS) k_ts_bwd_diag(const double* __restrict__ X, int w, int pw, double* __restrict__ x,
                                                           const double* __restrict__ s) {
    __shared__ double t[512];
    for (int i = threadIdx.x; i < w; i += blockDim.x) t[i] = x[i] - s[i];
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    for (int i = warp; i < w; i += nw) {
        double a = 0.0;
        for (int j = i + lane; j < w; j += 32) a = fma(X[(size_t)i * pw + j], t[j], a);
        a = warp_sum(a);
        if (lane == 0) x[i] = a;
    }
}
// global row of local row l of `rank`
__device__ __forceinline__ int ts_global_row(int l, int pw, int rank, int world) { return ((l / pw) * world + rank) * pw + l % pw; }
// x[grow(l)] -= L[l, c0:c0+w] y  for local rows l in [lo, hi): 64 rows x 4 column quarters per CTA, quarters summed in order
__global__ void __launch_bounds__(256) k_ts_fwd_update(const double* __restrict__ L, int ld, int lo, int hi, int c0, int w,
                                                      const double* __restrict__ y, double* __restrict__ x, int pw, int rank, int world) {
    __shared__ double ys[512];
    __shared__ double part[4][64];
    for (int i = threadIdx.y * 64 + threadIdx.x; i < w; i += 256) ys[i] = y[i];
    __syncthreads();
    const int l = lo + blockIdx.x * 64 + threadIdx.x;
    const int q = (w + 3) / 4, j0 = threadIdx.y * q, j1 = min(w, j0 + q);
    double a = 0.0;
    if (l < hi)
        for (int j = j0; j < j1; j++) a = fma(L[(size_t)(c0 + j) * ld + l], ys[j], a);
    part[threadIdx.y][threadIdx.x] = a;
    __syncthreads();
    if (threadIdx.y == 0 && l < hi) {
        const double t = ((part[0][threadIdx.x] + part[1][threadIdx.x]) + part[2][threadIdx.x]) + part[3][threadIdx.x];
        x[ts_global_row(l, pw, rank, world)] -= t;
    }
}
// s[j] = sum_{l in [lo, hi)} L[l, c0 + j] x[grow(l)]   (one CTA per column, fixed reduction order)
__global__ void __launch_bounds__(256) k_ts_bwd_partial(const double* __restrict__ L, int ld, int lo, int hi, int c0,
                                                       const double* __restrict__ x, double* __restrict__ s, int pw, int rank, int world) {
    __shared__ double sh[32];
    const int j = blockIdx.x;
    const double* col = L + (size_t)(c0 + j) * ld;
    double a = 0.0;
    for (int l = lo + threadIdx.x; l < hi; l += blockDim.x) a = fma(col[l], x[ts_global_row(l, pw, rank, world)], a);
    a = block_sum(a, sh);
    if (threadIdx.x == 0) s[j] = a;
}
}  // namespace

void chol_solve_dist(const double* A, int n, int lda, DistCtx& ctx, int pw, double* x, int which, cudaStream_t st) {
    const int world = ctx.world, rank = ctx.rank, nblk = (int)cdiv(n, pw);
    const size_t blk = (size_t)pw * pw;
    LRN_REQUIRE(ctx.xinv.n >= (size_t)nblk * blk, "no own-rows factor (cholesky_dist with rows_local)");
    if (ctx.svec.n < (size_t)pw) ctx.svec.alloc(pw);
    const int nloc = local_rows(n, pw, rank, world);
    // local rows of my blocks g > p start at the local row of my first such block
    auto lo_after = [&](int p) {
        const int f = first_block(p + 1, rank, world);
        return f >= nblk ? nloc : (f / world) * pw;
    };
    if (which & 1) {
        // Look-ahead: the main stream carries the critical chain -- apply X(p), broadcast y_p, and (owner of block p+1 only)
        // update the rows of block p+1 -- while the update of my rows in blocks >= p+2 runs on the side stream.  Every row
        // still receives its updates in step order: the update of block p+1 at step p waits for the side-stream update of
        // step p-1 (which also covered block p+1), so the result is the same as without look-ahead.
        if (!ctx.solve_side) {
            LRN_CUDA(cudaStreamCreateWithFlags(&ctx.solve_side, cudaStreamNonBlocking));
            for (auto& e : ctx.solve_ev) LRN_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        }
        cudaStream_t ss = ctx.solve_side;
        cudaEvent_t evY = ctx.solve_ev[0], evRest = ctx.solve_ev[1];
        LRN_CUDA(cudaEventRecord(evY, st));
        LRN_CUDA(cudaStreamWaitEvent(ss, evY, 0));                 // x is ready on the side stream
        auto update = [&](int lo, int hi, int c0, int w, cudaStream_t s_) {
            if (lo >= hi) return;
            k_ts_fwd_update<<<(unsigned)cdiv(hi - lo, 64), dim3(64, 4), 0, s_>>>(A, lda, lo, hi, c0, w, x + c0, x, pw, rank, world);
            LRN_CHECK_LAUNCH();
        };
        for (int p = 0; p < nblk; p++) {
            const int c0 = p * pw, w = std::min(pw, n - c0), owner = p % world;
            if (rank == owner) {
                k_ts_fwd_diag<<<1, TS_THREADS, 0, st>>>(ctx.xinv.p + (size_t)p * blk, w, pw, x + c0);
                LRN_CHECK_LAUNCH();
            }
            ctx.bcast(x + c0, (size_t)w, owner, st);          // y_p on every rank
            LRN_CUDA(cudaEventRecord(evY, st));
            // rows of block p+1 on its owner: after the side-stream update of step p-1, which wrote them last
            if (p + 1 < nblk && rank == (p + 1) % world) {
                if (p > 0) LRN_CUDA(cudaStreamWaitEvent(st, evRest, 0));
                const int l0 = ((p + 1) / world) * pw;
                update(l0, l0 + std::min(pw, n - (p + 1) * pw), c0, w, st);
            }
            // my rows in blocks >= p+2 on the side stream, once y_p is there
            LRN_CUDA(cudaStreamWaitEvent(ss, evY, 0));
            update(lo_after(p + 1), nloc, c0, w, ss);
            LRN_CUDA(cudaEventRecord(evRest, ss));
        }
        LRN_CUDA(cudaStreamWaitEvent(st, evRest, 0));
    }
    if (which & 2) {
        for (int p = nblk - 1; p >= 0; p--) {
            const int c0 = p * pw, w = std::min(pw, n - c0);
            k_ts_bwd_partial<<<(unsigned)w, 256, 0, st>>>(A, lda, lo_after(p), nloc, c0, x, ctx.svec.p, pw, rank, world);
            LRN_CHECK_LAUNCH();
            ctx.allreduce_sum(ctx.svec.p, (size_t)w, st);    // sum over the ranks of L[rows > block p, block p]' x
            k_ts_bwd_diag<<<1, TS_THREADS, 0, st>>>(ctx.xinv.p + (size_t)p * blk, w, pw, x + c0, ctx.svec.p);
            LRN_CHECK_LAUNCH();
        }
    }
}

}  // namespace lrn

using namespace lrn;

extern "C" {

int32_t lrn_dist_unique_id(void* out128) {
    if (!out128) return LRN_ERR_ARG;
    try {
        static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is expected to be 128 bytes");
        ncclUniqueId id;
        if (nccl_api().GetUniqueId(&id) != ncclSuccess) return LRN_ERR_NCCL;
        std::memcpy(out128, &id, sizeof id);
        return LRN_OK;
    } catch (...) {
        return LRN_ERR_NCCL;
    }
}

int32_t lrn_dist_init(lrn_handle_t h, int32_t rank, int32_t world, const void* unique_id128) {
    if (!h || !unique_id128 || world < 1 || rank < 0 || rank >= world) return LRN_ERR_ARG;
    if (h->group) { h->err = "lrn_dist_init: the handle already drives several GPUs in-process (lrn_create_multi)"; return LRN_ERR_STATE; }
    try {
        LRN_CUDA(cudaSetDevice(h->device));
        ncclUniqueId id;
        std::memcpy(&id, unique_id128, sizeof id);
        std::unique_ptr<DistCtx> ctx(new DistCtx());
        ctx->rank = rank;
        ctx->world = world;
        LRN_NCCL(nccl_api().CommInitRank(&ctx->comm, world, id, rank));
        const int pw = (h->n_var >= 16384) ? 512 : (h->n_var >= 4096 ? 256 : 128);
        if (h->finalized && h->H.p()) {
            // lrn_finalize counted no exchange buffers (it ran without a communicator): refuse now if the buffers the
            // distributed factorisation will allocate do not fit, with the same decision on every rank
            size_t free_b = 0, total_b = 0;
            LRN_CUDA(cudaMemGetInfo(&free_b, &total_b));
            const size_t need = dist_work_bytes(h->n_var, pw, world);
            const int mine = need > free_b ? 1 : 0;
            DevBuf<int> flag(1);
            LRN_CUDA(cudaMemcpyAsync(flag.p, &mine, sizeof(int), cudaMemcpyHostToDevice, h->st));
            ctx->allreduce_max(flag.p, 1, h->st);
            int any = 0;
            LRN_CUDA(cudaMemcpyAsync(&any, flag.p, sizeof(int), cudaMemcpyDeviceToHost, h->st));
            LRN_CUDA(cudaStreamSynchronize(h->st));
            if (any) {
                h->err = "lrn_dist_init: the exchange buffers of the distributed factorisation need " + std::to_string(need) +
                         " bytes of device memory on this rank, " + std::to_string(free_b) + " bytes are free" +
                         (mine ? "" : " (another rank is short of memory)");
                return LRN_ERR_ARG;
            }
        }
        if (h->nccl) delete static_cast<DistCtx*>(h->nccl);
        h->nccl = ctx.release();
        h->rank = rank;
        h->world = world;
        h->dist_pw = pw;
        return LRN_OK;
    } catch (const std::exception& e) {
        h->err = e.what();
        return LRN_ERR_NCCL;
    }
}

}  // extern "C"
