"""The own-rows layout of the kit = 0 Schur matrix H and its factor L (every rank stores only its own row blocks), checked on
ONE GPU: the sharded assembly through the test hook lrn_dbg_set_shard, and the distributed factorisation and triangular
solves at world 1, 2 and 3 through the in-process loopback transport (lrn_dbg_create_loopback: every member on the same
device), against the replicated layout on the same world.  The multi-GPU checks at n_var = 120 000 skip below two GPUs."""
import ctypes as C

import numpy as np
import pytest

from test_gpu_solver import OPTS_SDPA, golden, relerr

pytestmark = pytest.mark.gpu


class _LoopLib:
    """the library, except that the in-process multi-GPU facade is the loopback group on the current device"""

    def __init__(self, lib, world, block_rows=0):
        self._lib, self._world, self._br = lib, world, block_rows

    def __getattr__(self, name):
        return getattr(self._lib, name)

    def lrn_create_multi(self, out, n, nlmi, ms, nlin, opt, ngpus, devices):
        return self._lib.lrn_dbg_create_loopback(out, n, nlmi, ms, nlin, opt, self._world, self._br)


def _solver(pkg, arrays, opts, world=None, layout=None, shard=None, block_rows=0):
    """a set-up solver: `world` loopback members (None: a plain single-GPU handle), the Schur layout forced before
    lrn_finalize (None: automatic), `shard` = (rank, world, block_rows) ownership without a communicator"""
    from loraine_jl_b200 import solver as S
    opt = pkg.Optimizer()
    for k, v in opts.items():
        opt.set_attribute(k, v)
    opt.copy_to(pkg.raw_from_sdpa_arrays(*arrays))
    g = opt.solver
    if world is not None:
        g.extra["ngpus"] = 0                   # anything but 1 takes the lrn_create_multi branch, which _LoopLib replaces
        g.lib = _LoopLib(g.lib, world, block_rows)

    def before_finalize(s):
        if shard is not None:
            assert s.lib.lrn_dbg_set_shard(s.h, *shard) == 0
        if layout is not None:
            assert s.lib.lrn_dbg_schur_layout(s.h, layout, None) == 0
    S.setup_solver(g, opt.halpha, before_finalize=before_finalize)
    return opt, g


def _layout(g):
    out = C.c_int32(-9)
    assert g.lib.lrn_dbg_schur_layout(g.h, -2, C.byref(out)) == 0
    return out.value


def _prepare(S, g, steps=0, halpha=None):
    """initial point, `steps` IP iterations, then the Schur matrix and the predictor right-hand side of the next one"""
    S.initial_point(g)
    for _ in range(steps):
        S.myIPstep(g, halpha); g.itertime = 0.0; S.check_convergence(g)
    g.iter += 1
    S.find_mu(g); S.prepare_W(g)
    g._call("lrn_residuals"); g._call("lrn_schur_assemble"); g._call("lrn_rhs_predictor")


# ---- assembly ------------------------------------------------------------------------------------------------------------
def _assembly_case(pkg, golden_dir, case):
    if case == "maxcut-rank1":                                     # rank-one SYRK
        return pkg.problems.maxcut_torus(8, 12, 96), dict(OPTS_SDPA, datarank=-1), {}
    if case == "staged":                                           # staged pair kernel (pairs.cu)
        return pkg.problems.large_schur(30, 200, 40000), dict(OPTS_SDPA), {"pair_kernel": 1}
    if case == "gather":                                           # gather pair kernel
        return pkg.problems.large_schur(30, 200, 40000), dict(OPTS_SDPA), {"pair_kernel": 0}
    if case == "lp":                                               # LP row kernel
        return pkg.problems.multiblock_lp(3, 12, 10, 7), dict(OPTS_SDPA), {}
    return golden(golden_dir, case)[1], dict(OPTS_SDPA), {}        # control1: F1 columns + pairs


@pytest.mark.parametrize("case", ["control1", "maxcut-rank1", "staged", "gather", "lp"])
def test_own_rows_assembly_equals_the_replicated_shard(pkg, golden_dir, case):
    """Every assembly path writes each rank's rows to their local places: the own-rows shard of every rank equals the rows
    the same rank assembles in the replicated layout, bit for bit, at world 2 and 3, with a ragged last block and (for the
    block heights that leave it so) a rank without rows.  Rows of other ranks stay zero."""
    from loraine_jl_b200 import solver as S
    arrays, opts, options = _assembly_case(pkg, golden_dir, case)
    opt0, g0 = _solver(pkg, arrays, opts)
    S.initial_point(g0)
    S.myIPstep(g0, opt0.halpha)
    from test_gpu_round2 import _iterate
    it = _iterate(S, g0)
    n = g0.model.n
    g0.close()
    seen_empty = seen_ragged = False
    for world in (2, 3):
        for br in (8, 32, 64):
            nblk = -(-n // br)
            seen_ragged |= n % br != 0
            for rank in range(world):
                mats = []
                for layout in (0, 1):
                    _, g = _solver(pkg, arrays, opts, layout=layout, shard=(rank, world, br))
                    for k, v in options.items():
                        g._call("lrn_set_option", k.encode(), float(v))
                    S.initial_point(g)
                    S.set_iterate(g, *it)
                    g.iter += 1
                    S.find_mu(g); S.prepare_W(g)
                    g._call("lrn_residuals"); g._call("lrn_schur_assemble")
                    assert _layout(g) == layout
                    mats.append(np.tril(g.get_array("H")))
                    g.close()
                mine = np.array([pkg.dist.row_owner(r, br, world) == rank for r in range(n)])
                seen_empty |= not mine.any()
                assert np.array_equal(mats[1][mine], mats[0][mine]), (case, world, br, rank)
                assert not mats[1][~mine].any()
                assert mine.sum() == pkg.dist.local_rows(n, br, rank, world) and nblk >= 1
    assert seen_ragged
    if n <= 64 * 2:
        assert seen_empty


def test_own_rows_shift_and_get_array_on_a_shard(pkg, golden_dir):
    """lrn_schur_shift moves the own diagonal entries at their local places; a shard handle without a communicator returns its
    own rows of H at their global places and zeros elsewhere"""
    from loraine_jl_b200 import solver as S
    arrays = golden(golden_dir, "control1")[1]
    n = int(arrays[0])
    for layout in (0, 1):
        _, g = _solver(pkg, arrays, OPTS_SDPA, layout=layout, shard=(1, 2, 8))
        S.initial_point(g)
        g.iter += 1
        S.find_mu(g); S.prepare_W(g)
        g._call("lrn_residuals"); g._call("lrn_schur_assemble")
        H0 = np.tril(g.get_array("H"))
        g._call("lrn_schur_shift", 3.0)
        H1 = np.tril(g.get_array("H"))
        mine = np.array([pkg.dist.row_owner(r, 8, 2) == 1 for r in range(n)])
        d0, d1 = np.diag(H0), np.diag(H1)
        assert np.allclose(d1[mine] - d0[mine], 3.0, rtol=0, atol=1e-12 * (1 + np.abs(d0).max())), layout
        assert not d1[~mine].any() and not d0[~mine].any()
        g.close()


# ---- factorisation and solves through the loopback transport --------------------------------------------------------------
def _pair(pkg, arrays, opts, world, block_rows=0, steps=0):
    """replicated and own-rows loopback handles on the same world, at the same Schur matrix"""
    from loraine_jl_b200 import solver as S
    out = []
    for layout in (0, 1):
        opt, g = _solver(pkg, arrays, opts, world=world, layout=layout, block_rows=block_rows)
        assert _layout(g) == layout
        _prepare(S, g, steps, opt.halpha)
        out.append(g)
    return out


def _backward_errors(H, L, r, x):
    """which -> normwise backward error of the solve result x[which] for the right-hand side r"""
    nH, nL = np.linalg.norm(H), np.linalg.norm(L)            # Frobenius: cheap at n_var = 17 001
    e = {1: np.linalg.norm(L @ x[1] - r) / (nL * np.linalg.norm(x[1]) + np.linalg.norm(r)),
         2: np.linalg.norm(L.T @ x[2] - r) / (nL * np.linalg.norm(x[2]) + np.linalg.norm(r)),
         3: np.linalg.norm(H @ x[3] - r) / (nH * np.linalg.norm(x[3]) + np.linalg.norm(r)),
         6: np.linalg.norm(H @ (H @ x[6]) - r) / (nH * nH * np.linalg.norm(x[6]) + np.linalg.norm(r))}
    return e


SIZES = [(300, 40, 128), (1100, 60, 128), (5000, 120, 256), (17001, 300, 512)]


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("n,m,pw", SIZES)
def test_loopback_own_rows_factor_and_solves(pkg, world, n, m, pw):
    """At world 2 and 3 (loopback on one GPU), n_var = 300 / 1100 / 5000 / 17001 (block heights 128 / 128 / 256 / 512, every
    last block ragged): the own-rows factor equals the replicated distributed factor on the same world bit for bit, the
    fan-out / fan-in solves (which = 1, 2, 3, 6) have a backward error within 10x of the replicated solves, and a pivot failure
    is reported at the same LAPACK-style index -- in this rank's blocks, in another rank's and in the last block -- after
    which a shift and a new factorisation recover."""
    arrays = pkg.problems.large_schur(m, n, 40000 + n)
    opts = dict(kit=0, datarank=0, initpoint=1, verb=0, eDIMACS=1e-6)
    g0, g1 = _pair(pkg, arrays, opts, world)
    assert g0._call("lrn_schur_factor") == 0 and g1._call("lrn_schur_factor") == 0
    H = g0.get_array("H")
    L0, L1 = np.tril(g0.get_array("L")), np.tril(g1.get_array("L"))
    assert np.array_equal(L1, L0), relerr(L1, L0)
    r = g0.get_array("RHS")
    assert np.array_equal(g1.get_array("RHS"), r)
    x0, x1 = {}, {}
    for which in (1, 2, 3, 6):
        for g, x in ((g0, x0), (g1, x1)):
            g._call("lrn_schur_solve", which)
            x[which] = g.get_array("DELY")
    e0, e1 = _backward_errors(H, L0, r, x0), _backward_errors(H, L0, r, x1)
    for which in (1, 2, 3, 6):
        assert e1[which] <= 10 * max(e0[which], 1e-17), (which, e0[which], e1[which])
        assert relerr(x1[which], x0[which]) <= 1e-8, which
    # a matrix that is negative definite fails at the first pivot on both layouts; shift back and refactor
    for g in (g0, g1):
        g._call("lrn_schur_shift", -2.0 * float(np.max(np.diag(H))))
    i0 = g0._call("lrn_schur_factor", allow_positive=True)
    assert i0 == 1 and g1._call("lrn_schur_factor", allow_positive=True) == i0
    for g in (g0, g1):
        g._call("lrn_schur_shift", 2.0 * float(np.max(np.diag(H))))
        assert g._call("lrn_schur_factor") == 0
    assert np.array_equal(np.tril(g1.get_array("L")), np.tril(g0.get_array("L")))
    g0.close(); g1.close()


@pytest.mark.parametrize("world", [2, 3])
def test_loopback_pivot_index_in_every_kind_of_block(pkg, world):
    """The first failing pivot is found by the owner of its block; every rank returns the same LAPACK-style index in both
    layouts, and it is the right one: H = L D L' (unit lower L, D = 1 except D[k] = -1) has its first non-positive pivot at
    k + 1, for k in rank 0's first block, rank 1's first block and the ragged last block (n_var = 1100, 128-row blocks).
    With D = 1 the same handles factor again, and both layouts give the same factor."""
    n, m, pw = 1100, 60, 128
    arrays = pkg.problems.large_schur(m, n, 40000 + n)
    g0, g1 = _pair(pkg, arrays, dict(kit=0, datarank=0, initpoint=1, verb=0, eDIMACS=1e-6), world)
    rng = np.random.default_rng(7)
    Lu = np.tril(rng.standard_normal((n, n)), -1) * (0.3 / np.sqrt(n)) + np.eye(n)
    nblk = -(-n // pw)
    PD = C.POINTER(C.c_double)
    for k in (pw // 2 + 3, pw + 17, (nblk - 1) * pw + 5):
        D = np.ones(n)
        D[k] = -1.0
        H = np.asfortranarray((Lu * D) @ Lu.T)
        for g in (g0, g1):
            assert g.lib.lrn_dbg_set_H(g.h, H.ctypes.data_as(PD)) == 0
        i0 = g0._call("lrn_schur_factor", allow_positive=True)
        i1 = g1._call("lrn_schur_factor", allow_positive=True)
        assert i0 == i1 == k + 1, (k, i0, i1)
    H = np.asfortranarray(Lu @ Lu.T)
    for g in (g0, g1):
        assert g.lib.lrn_dbg_set_H(g.h, H.ctypes.data_as(PD)) == 0
        assert g._call("lrn_schur_factor") == 0
    L0, L1 = np.tril(g0.get_array("L")), np.tril(g1.get_array("L"))
    assert np.array_equal(L1, L0)
    assert relerr(L0, np.linalg.cholesky(H)) <= 1e-12
    g0.close(); g1.close()


def test_footprint_hook_matches_the_python_mirror(pkg, golden_dir):
    """lrn_finalize's footprint (direct_footprint in solver.cu) differs between the layouts by exactly what
    dist.schur_bytes mirrors: H and L of either size, and the own-rows panel slots, stored inverses and partial sums"""
    arrays = golden(golden_dir, "theta1")[1]
    n = int(arrays[0])
    for rank, world, br in ((0, 1, 64), (0, 2, 64), (1, 2, 64), (2, 3, 64), (1, 3, 128)):
        _, g = _solver(pkg, arrays, dict(OPTS_SDPA), shard=(rank, world, br))
        b = [C.c_int64(), C.c_int64()]
        for k in (0, 1):
            assert g.lib.lrn_dbg_schur_footprint(g.h, k, C.byref(b[k])) == 0
        want = pkg.dist.schur_bytes(n, br, rank, world, True) - pkg.dist.schur_bytes(n, br, rank, world, False)
        assert b[1].value - b[0].value == want, (rank, world, br)
        g.close()


def test_world1_own_rows_against_replicated(pkg, golden_dir):
    """A one-member loopback group (a world-1 communicator): the own-rows layout is the identity there, so H and L equal the
    replicated layout's bit for bit, and dely and two IP iterations agree"""
    from loraine_jl_b200 import solver as S
    arrays = golden(golden_dir, "theta1")[1]
    g0, g1 = _pair(pkg, arrays, dict(OPTS_SDPA), 1, block_rows=64)
    assert np.array_equal(g1.get_array("H"), g0.get_array("H"))
    for g in (g0, g1):
        assert g._call("lrn_schur_factor") == 0
        g._call("lrn_schur_solve", 3)
    assert np.array_equal(np.tril(g1.get_array("L")), np.tril(g0.get_array("L")))
    assert relerr(g1.get_array("DELY"), g0.get_array("DELY")) <= 1e-12
    g0.close(); g1.close()
    objs = []
    for layout in (0, 1):
        opt, g = _solver(pkg, arrays, dict(OPTS_SDPA), world=1, layout=layout, block_rows=64)
        S.initial_point(g)
        for _ in range(2):
            S.myIPstep(g, opt.halpha); g.itertime = 0.0; S.check_convergence(g)
        objs.append((g.primal_obj, g.dual_obj))
        g.close()
    assert abs(objs[1][0] - objs[0][0]) <= 1e-10 * (1 + abs(objs[0][0]))
    assert abs(objs[1][1] - objs[0][1]) <= 1e-10 * (1 + abs(objs[0][1]))


@pytest.mark.parametrize("name,want", [("theta1", 23.0), ("control1", 17.78463)])
@pytest.mark.parametrize("block_rows", [0, 64])
def test_loopback_world2_own_rows_solves_to_the_known_optimum(pkg, golden_dir, name, want, block_rows):
    """A whole solve in the own-rows layout at world 2 (loopback): theta1 (n_var = 104) and control1 (n_var = 21) reach their
    known objectives.  At the default block height one rank owns no rows; with 64-row blocks theta1 has rows on both ranks."""
    from loraine_jl_b200 import solver as S
    arrays = golden(golden_dir, name)[1]
    opt, g = _solver(pkg, arrays, dict(OPTS_SDPA), world=2, layout=1, block_rows=block_rows)
    assert _layout(g) == 1
    S.solve(g, opt.halpha, setup=False)
    assert g.status == 1
    assert abs(abs(g.primal_obj) - want) <= 1e-5 * (1 + abs(want)), g.primal_obj
    g.close()


def test_own_rows_handles_refuse_full_matrix_hooks(pkg, golden_dir):
    """lrn_dbg_gather_H and lrn_dbg_compare need full matrices: LRN_ERR_STATE on an own-rows handle with world > 1"""
    arrays = golden(golden_dir, "theta1")[1]
    _, g = _solver(pkg, arrays, dict(OPTS_SDPA), world=2, layout=1, block_rows=64)
    assert g.lib.lrn_dbg_gather_H(g.h) == -4
    g.close()
    shards = [_solver(pkg, arrays, dict(OPTS_SDPA), layout=1, shard=(r, 2, 64))[1] for r in range(2)]
    err = C.c_double()
    assert shards[0].lib.lrn_dbg_compare(shards[0].h, shards[1].h, 1, C.byref(err)) == -4
    for g in shards:
        g.close()


# ---- several GPUs ----------------------------------------------------------------------------------------------------------
def _two_gpus():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")


def _used_bytes(devices):
    import torch
    return [torch.cuda.mem_get_info(d) for d in devices]


def test_two_gpus_admit_and_solve_a_model_one_gpu_refuses(pkg):
    """n_var = 120 000 kit = 0 matrix completion: one GPU refuses it; ngpus = 2 admits it in the own-rows layout (the default
    peer-memory exchange of the inverses), each GPU's device memory after the solve is within 4 GB of the footprint
    lrn_finalize computed, and the solve reaches the known optimum -||M||_* at eDIMACS 1e-6"""
    _two_gpus()
    import mc_instances as mc
    from loraine_jl_b200 import solver as S
    inst = mc.matrix_completion(500, 500, 3, 120000, seed=5)
    opts = dict(OPTS_SDPA, eDIMACS=1e-6)
    with pytest.raises(Exception, match="bytes of device memory"):
        _solver(pkg, inst.arrays, opts)
    free0 = _used_bytes((0, 1))
    opt, g = _solver(pkg, inst.arrays, dict(opts, ngpus=2))
    assert _layout(g) == 1
    S.solve(g, opt.halpha, setup=False)
    assert g.status == 1
    assert abs(g.primal_obj - inst.optimum) <= 1e-5 * abs(inst.optimum), (g.primal_obj, inst.optimum)
    fp = C.c_int64()
    assert g.lib.lrn_dbg_schur_footprint(g.h, 1, C.byref(fp)) == 0
    free1 = _used_bytes((0, 1))
    for d in (0, 1):
        used = free0[d][0] - free1[d][0]
        assert abs(used - fp.value) <= 4e9, (d, used, fp.value)
    g.close()


def test_two_gpus_forced_own_rows_against_replicated(pkg):
    """n_var = 20 000 on two GPUs (NCCL, default exchange mode): the forced own-rows layout takes the same number of IP
    iterations as the replicated layout and reaches the same objectives to 1e-8"""
    _two_gpus()
    import mc_instances as mc
    from loraine_jl_b200 import solver as S
    inst = mc.matrix_completion(200, 200, 2, 20000, seed=3)
    res = []
    for layout in (0, 1):
        opt, g = _solver(pkg, inst.arrays, dict(OPTS_SDPA, ngpus=2), layout=layout)
        assert _layout(g) == layout
        S.solve(g, opt.halpha, setup=False)
        assert g.status == 1
        res.append((g.iter, g.primal_obj, g.dual_obj))
        g.close()
    assert res[1][0] == res[0][0]
    for k in (1, 2):
        assert abs(res[1][k] - res[0][k]) <= 1e-8 * (1 + abs(res[0][k])), (k, res)


_TWO_RANKS = """
import ctypes as C, os, sys
import torch, torch.distributed as dist
sys.path.insert(0, {root!r}); sys.path.insert(0, os.path.join({root!r}, "tests"))
import __graft_entry__ as g
pkg = g.load_package()
import mc_instances as mc
from loraine_jl_b200 import solver as S
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dist.init_process_group("gloo")
inst = mc.matrix_completion(500, 500, 3, 120000, seed=5)
opt = pkg.Optimizer()
for k, v in dict(kit=0, tol_cg=1e-2, tol_cg_min=1e-6, eDIMACS=1e-6, preconditioner=1, erank=1, aamat=2, verb=0, datarank=0,
                 initpoint=1, maxit=100, datasparsity=8, device=rank).items():
    opt.set_attribute(k, v)
opt.copy_to(pkg.raw_from_sdpa_arrays(*inst.arrays))
s = opt.solver
S.setup_solver(s, opt.halpha, before_finalize=pkg.dist.attach_before_finalize)
lay = C.c_int32(-9)
assert s.lib.lrn_dbg_schur_layout(s.h, -2, C.byref(lay)) == 0 and lay.value == 1, lay.value
S.solve(s, opt.halpha, setup=False)
assert s.status == 1
assert abs(s.primal_obj - inst.optimum) <= 1e-5 * abs(inst.optimum), (s.primal_obj, inst.optimum)
s.close()
dist.barrier()
open(os.path.join({out!r}, "ok%d" % rank), "w").write("ok")
dist.destroy_process_group()
"""


def test_two_processes_attach_before_finalize(pkg, tmp_path):
    """The n_var = 120 000 model through two torchrun ranks (one process per GPU) that attach to the communicator between
    lrn_set_b and lrn_finalize (setup_solver(..., before_finalize=dist.attach_before_finalize)): lrn_finalize chooses the
    own-rows layout on both ranks and the solve reaches -||M||_*.  The launcher runs in its own process group, joined with a
    time-out; on a time-out the whole group is killed, so that no process is left behind."""
    _two_gpus()
    import os
    import signal
    import socket
    import subprocess
    import sys
    import textwrap
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = tmp_path / "two_ranks.py"
    script.write_text(textwrap.dedent(_TWO_RANKS.format(root=root, out=str(tmp_path))))
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), str(script)]
    p = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, start_new_session=True,
                         env=dict(os.environ, OMP_NUM_THREADS="1"))
    try:
        out, _ = p.communicate(timeout=1800)
    except subprocess.TimeoutExpired:
        os.killpg(p.pid, signal.SIGKILL)
        p.communicate()
        pytest.fail("two-process run timed out")
    assert p.returncode == 0, out[-4000:]
    assert (tmp_path / "ok0").exists() and (tmp_path / "ok1").exists()
