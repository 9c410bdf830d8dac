// Device-resident solver state behind the opaque C handle (mirrors MySolver / MyModel / Halpha of the reference,
// src/Solvers.jl:18-162, src/model.jl:34-87, but as typed, pre-allocated device buffers).
#pragma once
#include "../../include/loraine_b200.h"
#include "chol.cuh"
#include "common.cuh"
#include "eig.cuh"
#include "gemm.cuh"
#include "ops.cuh"
#include <memory>
#include <string>
#include <vector>

namespace lrn {

struct HostCSC {                       // staging copy of a Julia SparseMatrixCSC (converted to 0-based)
    std::vector<int64_t> colptr;
    std::vector<int64_t> rowval;
    std::vector<double> nzval;
    bool set = false;
};

struct Block {
    int m = 0, ld = 0;
    HostCSC hAA, hB, hC;               // released after finalize
    SparseBlock sp;
    DMat C;
    double normC = 0.0;
    DMat X, S, dX, dS, Xn, Sn, G, Gi, W, Si, Rd, RNT, LX, LS, T1, T2, T3, T4;
    DMat RdB;                          // G' Rd G of the current iteration (sparse data: shared by both find_steps and the corrector RHS)
    bool rdb_valid = false;
    DevBuf<double> D, DDsi, dm12, dm32, vtmp;
    CholWork cholX, cholS;
    SvdWork svd;
    bool chol_cached = false;
    bool ud_valid = false;             // T2 holds U*D of the last prepare_W and LS its factor (Gi parity hook)
    // H_alpha preconditioner pieces (src/Solvers.jl:149-162 Halpha)
    DMat U, Zf, MU, ZY;                // U m x erank ; Z = chol(2 W0 + U U') lower ; work m x erank
    double tau = 0.0;
};

struct SvdGroup {                       // PSD blocks of equal size share one batched block-Jacobi SVD
    int m = 0;
    std::vector<int> blocks;
    SvdBatchWork w;
    DevBuf<const double*> A;
    DevBuf<double*> UD, sig;
};

struct PhaseEvt {
    cudaEvent_t a, b;
    int phase;
};

// Largest n_var lrn_create admits for the direct (kit = 0) path.  In the replicated layout every rank holds the dense
// n_var x n_var FP64 Schur matrix and its factor (16 n_var^2 bytes) plus about 19 KB per row of Cholesky workspace
// (chol_work_bytes), so on a 180 GB B200 the path ends near n_var = 105 000 (178 GB); 140 000 (314 GB) fits no single GPU.
// With several GPUs lrn_finalize falls back to the own-rows layout (rows_local: 16 n_var^2 / world bytes per rank).  lrn_finalize refuses any kit = 0 model whose state does not fit the free device memory (direct_footprint in
// solver.cu).  The CG path (kit = 1) forms neither matrix.
constexpr int64_t KIT0_MAX_NVAR = 140000;
// Row-slab height of the H_alpha build (pcg.cu): n_var when the whole T (n_var x kS) and A_j u_r (n_var x maxm) fit the slab
// budget, otherwise the largest multiple of 8 that does; force > 0 is used as given (clamped to n_var).
int prec_slab_rows(int n_var, int kS, int maxm, int64_t force);
// device bytes of one slab pair (T and A_j u_r) of height `rows`
size_t prec_slab_bytes(int rows, int kS, int maxm);

}  // namespace lrn

struct lrn_solver {
    lrn_options_t opt;
    int device = 0;
    int n_var = 0, nlmi = 0, nlin = 0;
    long long sum_m = 0;
    bool finalized = false;
    std::vector<lrn::Block> blk;
    lrn::HostCSC hClin;
    lrn::SparseLin lin;
    lrn::DevBuf<double> b, d_lin, y, dely, rhs, Rp, tn1, tn2, ones;
    lrn::DevBuf<double> x_lin, s_lin, si_lin, dx_lin, ds_lin, xn_lin, sn_lin, rnt_lin, rd_lin, tl1, tl2;
    double normb = 0.0, normd = 0.0;
    // model norms kept for lrn_initial_point (src/initial_point.jl:28-71): ||AA_i||_F, ||1 + |b|||, max_j (1+|b_j|)/(1+||C_lin[j,:]||),
    // max_j ||C_lin[j,:]||
    std::vector<double> hb, ip_normAA;
    double ip_normb2 = 0.0, ip_pmax = 0.0, ip_rownmax = 0.0;
    bool ip_ready = false;
    lrn::DMat H, L, BG;
    lrn::CholWork cholH;
    bool have_factor = false;
    lrn::DevBuf<int> blk_info;         // 2 per block (chol X, chol S)
    // batched lambda_min of the small blocks (m <= EIG_BATCH_MAXM): matrices T3_i (X part) and T1_i (S part)
    std::vector<std::unique_ptr<lrn::SvdGroup>> svd_groups;
    std::vector<int> svd_group_of;     // per block: group index or -1
    std::vector<int> eig_small;        // block indices handled by the batched kernel
    lrn::DevBuf<double*> eig_ptrs;
    lrn::DevBuf<int> eig_ms, eig_lds;
    lrn::DevBuf<double> eig_out;
    lrn::Reducer red;
    lrn::LanczosWork lan, lan2;        // lan2 + st2: the second of two independent lambda_min runs (corrector) on its own stream
    cudaStream_t st2 = nullptr;
    cudaEvent_t ev2 = nullptr;
    int lanczos_kmax = 500;            // Krylov dimension cap (test hook: small values force the bisection fallback)
    lrn::DMat eig_scratch;             // shifted copy of the matrix for the Cholesky bisection fallback of lambda_min
    lrn::CholWork eig_chol;
    long long stat_bisect = 0;
    cudaStream_t st = nullptr;
    // side streams for independent per-block work of multi-block problems (fork / join around the loop with events)
    static constexpr int NSIDE = 4;
    cudaStream_t side[NSIDE] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t evFork = nullptr, evJoin[NSIDE] = {nullptr, nullptr, nullptr, nullptr};
    std::string err;
    // timers
    std::vector<lrn::PhaseEvt> pending;
    std::vector<cudaEvent_t> evpool;
    double t_ms[LRN_T_COUNT] = {0};
    long long t_calls[LRN_T_COUNT] = {0};
    long long stat_svd_sweeps = 0, stat_lanczos_iters = 0, stat_lanczos_fail = 0;
    // CG / preconditioner state
    lrn::DevBuf<double> cg_r, cg_z, cg_p, cg_Ap, cg_scal;
    lrn::DevBuf<double> pDiag, pDsq, pT, pS, pY, pYw, pAU;
    lrn::DMat pDd;                     // dense AAAATtau when nlin > 0
    lrn::CholWork cholS, cholD;
    bool pDense = false;
    int kS = 0;
    // H_alpha build in row slabs: pT (pad_ld(slab_rows) x kS) and pAU (pad_ld(slab_rows) x max m) hold slab_rows rows of T
    // and of A_j u_r
    int slab_rows = 0;
    int64_t slab_force = 0;            // debug hook: forced slab height (0 = automatic)
    int prec_ready = 0;                // kind prepared (0 none)
    // distributed
    int rank = 0, world = 1;
    void* nccl = nullptr;              // lrn::DistCtx*
    int dist_pw = 512;                 // row block height of the block-cyclic Schur distribution
    int use_staged_pairs = -1;         // sparse-pair Schur term: 1 staged kernel (pairs.cu) when the block has a plan, 0 gather kernel,
                                       // -1 automatic (staged from 1024 participating constraints per block on)
    int chol_int8 = 1;                 // Schur factor: trailing updates as Ozaki INT8 products for n_var >= 16384 (CholWork::int8;
                                       // lrn_set_option("chol_int8", 0) keeps them on DMMA)
    bool H_gathered = false;           // the row-block shards of H have already been summed over the ranks (parity hooks)
    bool rows_local = false;           // kit = 0 storage: H and L hold only this rank's own row blocks (RowOwner::local, ops.cuh)
    int layout_force = -1;             // test hook lrn_dbg_schur_layout: -1 lrn_finalize decides, 0 replicated, 1 own rows
    // PSD blocks distributed over the ranks (lrn_finalize: kit = 0, nlmi >= 2, a communicator with world > 1): block i lives
    // on rank blk_owner[i] (lrn::block_owner, ops.cuh); the other ranks keep its sparse data and the gathered W_i (G_i when
    // datarank = -1), which is all their Schur rows need
    bool blk_sharded = false;
    int blk_force = -1;                // test hook lrn_dbg_block_layout: -1 lrn_finalize decides, 0 replicated, 1 sharded
    std::vector<int> blk_owner;
    lrn::DevBuf<double> gbuf;          // W / G all-gather: chunk 0 this rank's packed blocks, chunk 1 + r rank r's (gchunk doubles
                                       // each, the last one a status flag); between two prepare_W calls the F1 scratch
    size_t gchunk = 0;
    lrn::DevBuf<double> vpart, vparts; // residual / RHS partial n_var vectors: this rank's, every rank's (rank order)
    lrn::DevBuf<double> vshare;        // per-block values (mu, step lengths, DIMACS terms) filled in by the owners, then summed
    bool owns(int i) const { return !blk_sharded || blk_owner[i] == rank; }
    void* group = nullptr;             // lrn::Group*: this handle is the facade of an in-process multi-GPU group (group.cuh)
};
