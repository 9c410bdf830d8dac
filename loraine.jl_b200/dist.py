"""Multi-GPU plumbing on the host: one process per GPU (torchrun), NCCL communicator inside the library.

`torch.distributed` is only used to hand the 128-byte NCCL unique id from rank 0 to the other ranks (any backend: nccl on
the GPU box, gloo in the CPU tests); the data path (panel broadcasts of the distributed Cholesky) runs inside the library.
"""
from __future__ import annotations

import ctypes as C


def row_owner(row: int, pw: int, world: int) -> int:
    """1-D block-cyclic ownership of Schur-matrix ROWS (mirrors lrn::RowOwner::owns in csrc/ops.cuh): entry (r, c), c <= r, of
    the lower triangle is assembled and factored by the owner of row r."""
    return (row // pw) % world if world > 1 else 0


def block_rows(n_var: int) -> int:
    """height of a row block; mirrors lrn_dist_init / lrn_create_multi (csrc/dist.cu, csrc/group.cu)"""
    return 512 if n_var >= 16384 else (256 if n_var >= 4096 else 128)


def dd_block_rows(n_var: int) -> int:
    """height of a row block of the double-double LP path (mirrors lrn::dd_block_rows in csrc/ddlp.cuh)"""
    return 256 if n_var >= 4096 else (128 if n_var >= 1024 else 64)


def first_block(p: int, rank: int, world: int) -> int:
    """first row block >= p owned by `rank` (mirrors first_block in csrc/dist.cu)"""
    return p + ((rank - p % world + world) % world)


def count_blocks(p: int, rank: int, world: int, nblk: int) -> int:
    """number of row blocks >= p owned by `rank` (mirrors count_blocks in csrc/dist.cu)"""
    f = first_block(p, rank, world)
    return 0 if f >= nblk else (nblk - 1 - f) // world + 1


def exchange_unique_id(make_id, rank: int, world: int) -> bytes:
    """rank 0 calls make_id() -> 128 bytes; every rank returns the same bytes."""
    import torch.distributed as dist
    obj = [make_id() if rank == 0 else None]
    if world > 1:
        dist.broadcast_object_list(obj, src=0)
    if not isinstance(obj[0], (bytes, bytearray)) or len(obj[0]) != 128:
        raise RuntimeError("NCCL unique id exchange failed")
    return bytes(obj[0])


def init_distributed(solver) -> bool:
    """Attach the solver's device handle to the job's NCCL communicator (call after setup_solver).  Returns True when the
    Schur assembly / factorisation is sharded over more than one rank."""
    import torch.distributed as dist
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size() <= 1:
        return False
    rank, world = dist.get_rank(), dist.get_world_size()
    lib = solver.lib

    def make_id():
        buf = C.create_string_buffer(128)
        rc = lib.lrn_dist_unique_id(buf)
        if rc != 0:
            raise RuntimeError(f"lrn_dist_unique_id failed ({rc})")
        return buf.raw
    uid = exchange_unique_id(make_id, rank, world)
    buf = C.create_string_buffer(uid, 128)
    solver._call("lrn_dist_init", rank, world, buf)
    solver.dist_rank, solver.dist_world = rank, world
    return True


def init_distributed_dd(solver) -> bool:
    """The double-double counterpart of init_distributed for a dd_lp.DDSolver (call after dd_lp.setup_solver, before the first
    iteration): attaches the handle to the job's NCCL communicator with lrn_dd_dist_init.  Every rank then runs the whole
    solve; the Schur assembly and factorisation are sharded, everything else is replicated.  Returns True when the job has
    more than one rank."""
    import torch.distributed as dist
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size() <= 1:
        return False
    rank, world = dist.get_rank(), dist.get_world_size()
    lib = solver.lib

    def make_id():
        buf = C.create_string_buffer(128)
        rc = lib.lrn_dist_unique_id(buf)
        if rc != 0:
            raise RuntimeError(f"lrn_dist_unique_id failed ({rc})")
        return buf.raw
    uid = exchange_unique_id(make_id, rank, world)
    solver._call("lrn_dd_dist_init", rank, world, C.create_string_buffer(uid, 128))
    solver.dist_rank, solver.dist_world = rank, world
    return True


def dist_parity(sd, make_single, rank: int, iters: int = 2) -> dict | None:
    """Run `iters` interior-point iterations on the sharded solver `sd` (collective: every rank calls) and, on rank 0, the
    same iterations on a single-GPU solver made by `make_single()` on the same device, restarted from the sharded solver's
    iterate at the top of every iteration.  Returns on rank 0 the largest relative Frobenius distances of the assembled Schur
    matrix (row-block shards summed over the ranks), of the Cholesky factor and of dely -- all compared on the device, so it
    works at n_var = 40000 -- and None elsewhere."""
    import numpy as np
    from . import solver as S
    lib = sd.lib
    s1 = make_single() if rank == 0 else None
    S.initial_point(sd)
    if s1 is not None:
        S.initial_point(s1)
    md = sd.model
    PD = C.POINTER(C.c_double)
    worst = dict(H=0.0, L=0.0, dely=0.0)
    pair = [sd] + ([s1] if s1 is not None else [])
    for it in range(iters):
        if s1 is not None and it > 0:                      # same iterate on both sides
            y, X, xl = S.get_solution(sd)
            Sm = [np.zeros((m, m), order="F") for m in md.msizes]
            sl = np.zeros(md.nlin)
            Sp = (PD * max(1, md.nlmi))(*[x.ctypes.data_as(PD) for x in Sm])
            sd._call("lrn_get_slack", Sp, sl.ctypes.data_as(PD) if md.nlin else None)
            S.set_iterate(s1, X, Sm, y, xl, sl)
        for s in pair:
            s.iter += 1
            s.cg_iter_pre = s.cg_iter_cor = 0
            S.find_mu(s)
            S.prepare_W(s)
            s._call("lrn_residuals")
            s._call("lrn_schur_assemble")
        rc = lib.lrn_dbg_gather_H(sd.h)
        if rc != 0:
            raise RuntimeError(f"lrn_dbg_gather_H failed ({rc}): {sd._err()}")
        err = C.c_double()
        if s1 is not None:
            assert lib.lrn_dbg_compare(sd.h, s1.h, 1, C.byref(err)) == 0, sd._err()
            worst["H"] = max(worst["H"], err.value)
        for s in pair:
            s._call("lrn_rhs_predictor")
            s._call("lrn_schur_factor")
            s.cholBBBB = S._DeviceFactor(s, False)
            s.cholBBBB.solve_reference_expression()
        if s1 is not None:
            assert lib.lrn_dbg_compare(sd.h, s1.h, 2, C.byref(err)) == 0, sd._err()
            worst["L"] = max(worst["L"], err.value)
            dd, d1 = sd.get_array("DELY"), s1.get_array("DELY")
            worst["dely"] = max(worst["dely"], float(np.linalg.norm(dd - d1) / max(np.linalg.norm(d1), 1e-300)))
        for s in pair:
            s.predict = True
            S.find_step(s)
            S.sigma_update(s)
            S.corrector(s, None)
            S.check_convergence(s)
    if s1 is None:
        return None
    out = dict(worst, iterations=iters, dimacs_sharded=float(sd.DIMACS_error), dimacs_single=float(s1.DIMACS_error),
               objective_sharded=float(sd.primal_obj), objective_single=float(s1.primal_obj))
    s1.close()
    return out
