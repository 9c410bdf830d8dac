"""PSD blocks distributed over the ranks (kit = 0, several blocks, a communicator with world > 1): every block has one owner
(dist.block_owner) that runs its m x m work; prepare_W all-gathers W_i (G_i for datarank = -1); the residual and right-hand
side terms are combined from per-rank partial vectors; step lengths, mu and the DIMACS terms are shared per block.

Checked on ONE GPU through the loopback transport (lrn_dbg_create_loopback, world 2 and 3) against a single-GPU handle and
against the replicated block layout forced at the same world (lrn_dbg_block_layout).  In the first two iterations every
compared quantity (mu, W_i / G_i, the Schur matrix H summed over the shards, the residual and both right-hand sides, both
dely, every alpha_i and beta_i, sigma, the DIMACS errors and objectives) agrees to RTOL = 1e-12 relative: only the order of
the block sums differs.  Whole solves end where the condition of H amplifies that difference: the primal objective agrees to
1e-9, the dual one to 1e-7 (both relative to 1 + |value|)."""
import ctypes as C

import numpy as np
import pytest

from test_gpu_schur_rows_local import _LoopLib
from test_gpu_solver import OPTS_SDPA, golden, relerr

pytestmark = pytest.mark.gpu

RTOL = 1e-12
PD = C.POINTER(C.c_double)


# ---- models --------------------------------------------------------------------------------------------------------------
def _mixed_blocks(sizes=(40, 200, 500), seed=7):
    """Diag(y_b) >= R_b for blocks of the given sides (the layout of problems.multiblock_lp without the LP block): 40 takes
    the unbatched small-block eigmin, 200 the batched kernel, 500 the Lanczos path of large blocks"""
    body, off = [], 0
    for b, m in enumerate(sizes):
        rng = np.random.default_rng(seed + b)
        Nn = rng.standard_normal((m, m))
        R = 0.5 * (Nn + Nn.T) / np.sqrt(m)
        iu, ju = np.triu_indices(m)
        body.append(np.column_stack([np.zeros(iu.size), (b + 1) * np.ones(iu.size), iu + 1, ju + 1, R[iu, ju]]))
        p = np.arange(1, m + 1)
        body.append(np.column_stack([off + p, (b + 1) * np.ones(m), p, p, np.ones(m)]))
        off += m
    return off, list(sizes), np.ones(off), np.concatenate(body)


def _two_maxcuts(pkg):
    """block-diagonal max-cut relaxation of two torus graphs (rank-one constraints: datarank = -1)"""
    n1, _, c1, b1 = pkg.problems.maxcut_torus(4, 6, 11)
    n2, _, c2, b2 = pkg.problems.maxcut_torus(5, 6, 12)
    b2 = b2.copy()
    b2[:, 1] = 2
    b2[b2[:, 0] > 0, 0] += n1
    return n1 + n2, [n1, n2], np.concatenate([c1, c2]), np.concatenate([b1, b2])


def _model(pkg, golden_dir, name):
    if name == "vib3":
        return golden(golden_dir, "vib3")[1], dict(OPTS_SDPA)
    if name == "control1":
        return golden(golden_dir, "control1")[1], dict(OPTS_SDPA)
    if name == "multiblock_lp":
        return pkg.problems.multiblock_lp(3, 12, 10, 7), dict(OPTS_SDPA)
    if name == "maxcut2":
        return _two_maxcuts(pkg), dict(OPTS_SDPA, datarank=-1)
    return _mixed_blocks(), dict(OPTS_SDPA)


MODELS = ["vib3", "control1", "multiblock_lp", "maxcut2", "mixed"]


def _solver(pkg, arrays, opts, world=None, blocks=None):
    """a set-up solver: `world` loopback members (None: a plain single-GPU handle), the block layout forced before lrn_finalize
    (None: automatic)"""
    from loraine_jl_b200 import solver as S
    opt = pkg.Optimizer()
    for k, v in opts.items():
        opt.set_attribute(k, v)
    opt.copy_to(pkg.raw_from_sdpa_arrays(*arrays))
    g = opt.solver
    if world is not None:
        g.extra["ngpus"] = 0
        g.lib = _LoopLib(g.lib, world)

    def before_finalize(s):
        if blocks is not None:
            assert s.lib.lrn_dbg_block_layout(s.h, blocks, None) == 0
    S.setup_solver(g, opt.halpha, before_finalize=before_finalize)
    return opt, g


def _blocks(g):
    out = C.c_int32(-9)
    assert g.lib.lrn_dbg_block_layout(g.h, -2, C.byref(out)) == 0
    return out.value


def _iterations(S, g, iters=2):
    """`iters` IP iterations phase by phase from the initial point; returns what each phase produced"""
    md = g.model
    rec = []
    S.initial_point(g)
    for it in range(iters):
        r = {}
        g.iter += 1
        g.cg_iter_pre = g.cg_iter_cor = 0
        r["mu"] = S.find_mu(g)
        S.prepare_W(g)
        r["W"] = [g.get_array("G" if g.datarank == -1 else "W", i) for i in range(md.nlmi)]
        g._call("lrn_residuals")
        r["RP"] = g.get_array("RP")
        g._call("lrn_schur_assemble")
        r["H"] = g.get_array("H")
        g._call("lrn_rhs_predictor")
        r["RHS"] = g.get_array("RHS")
        assert g._call("lrn_schur_factor") == 0
        g.cholBBBB = S._DeviceFactor(g, False)
        g.cholBBBB.solve_reference_expression()
        r["DELY"] = g.get_array("DELY")
        g.predict = True
        S.find_step(g)
        r["alpha_p"], r["beta_p"] = g.alpha.copy(), g.beta.copy()
        S.sigma_update(g)
        r["sigma"] = g.sigma
        S.corrector(g, None)
        r["alpha_c"], r["beta_c"] = g.alpha.copy(), g.beta.copy()
        r["DELY_c"] = g.get_array("DELY")
        S.check_convergence(g)
        r["err"] = np.array([g.err1, g.err2, g.err3, g.err4, g.err5, g.err6])
        r["obj"] = (g.primal_obj, g.dual_obj)
        rec.append(r)
    return rec


def _close(a, b, tol):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    return np.linalg.norm(a - b) <= tol * max(np.linalg.norm(b), 1e-300)


def _compare(got, want, label):
    worst = 0.0
    for it, (rg, rw) in enumerate(zip(got, want)):
        for k, vw in rw.items():
            vg = rg[k]
            pairs = zip(vg, vw) if k == "W" else [(vg, vw)]
            for a, b in pairs:
                assert _close(a, b, RTOL), (label, it, k, relerr(np.asarray(a, dtype=float), np.asarray(b, dtype=float)))
                worst = max(worst, relerr(np.asarray(a, dtype=float), np.asarray(b, dtype=float)))
    return worst


def _member_copies(g, world, iblk, which):
    out = []
    m = g.model.msizes[iblk]
    for r in range(world):
        a = np.zeros((m, m), order="F")
        assert g.lib.lrn_dbg_member_block(g.h, r, iblk, which, a.ctypes.data_as(PD)) == 0, g._err()
        out.append(a)
    return out


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("name", MODELS)
def test_two_iterations_phase_by_phase(pkg, golden_dir, name, world):
    """Two IP iterations phase by phase with the blocks distributed at world 2 and 3 (loopback) agree with one GPU and with
    the replicated block layout at the same world; every member's gathered W_i (G_i) equals the owner's bit for bit.  Two
    blocks at world 3 leave one rank without a block."""
    from loraine_jl_b200 import solver as S
    arrays, opts = _model(pkg, golden_dir, name)
    _, g1 = _solver(pkg, arrays, opts)
    ref = _iterations(S, g1)
    g1.close()
    _, gr = _solver(pkg, arrays, opts, world=world, blocks=0)
    assert _blocks(gr) == 0
    rep = _iterations(S, gr)
    gr.close()
    _, gs = _solver(pkg, arrays, opts, world=world)
    assert _blocks(gs) == 1                                          # the default for kit = 0 with several blocks
    got = _iterations(S, gs)
    msizes = gs.model.msizes
    owner = pkg.dist.block_owner(msizes, world)
    which = 11 if gs.datarank == -1 else 10
    for i in range(len(msizes)):
        copies = _member_copies(gs, world, i, which)
        for r in range(world):
            assert np.array_equal(copies[r], copies[owner[i]]), (i, r)
        assert np.array_equal(copies[owner[i]], got[-1]["W"][i])
    if world > len(msizes):
        assert set(owner) != set(range(world))
    gs.close()
    w1 = _compare(got, ref, "vs one GPU")
    w2 = _compare(got, rep, "vs replicated")
    print(f"{name} world {world}: largest relative difference {w1:.2e} (one GPU), {w2:.2e} (replicated blocks)")


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("name,want", [("vib3", 0.10271028), ("control1", 17.78462702), ("multiblock_lp", None),
                                       ("maxcut2", None), ("mixed", None)])
def test_whole_solves_match_one_gpu(pkg, golden_dir, name, want, world):
    """Whole solves with distributed blocks take the iteration count of one GPU, end with its status and reach its objective
    within 1e-9 (the dual one within 1e-7; and the known optima of vib3 and control1); the gathered X_i and S_i equal the
    single-GPU ones to the accuracy of the solve"""
    from loraine_jl_b200 import solver as S
    arrays, opts = _model(pkg, golden_dir, name)
    res = []
    for w in (None, world):
        opt, g = _solver(pkg, arrays, opts, world=w)
        S.solve(g, opt.halpha, setup=False)
        y, X, _ = S.get_solution(g)
        md = g.model
        Sm = [np.zeros((m, m), order="F") for m in md.msizes]
        sl = np.zeros(max(md.nlin, 1))
        Sp = (PD * max(1, md.nlmi))(*[x.ctypes.data_as(PD) for x in Sm])
        g._call("lrn_get_slack", Sp, sl.ctypes.data_as(PD) if md.nlin else None)
        res.append((g.iter, g.status, g.primal_obj, g.dual_obj, y.copy(), [x.copy() for x in X], Sm))
        g.close()
    (i1, s1, p1, d1, y1, X1, S1), (i2, s2, p2, d2, y2, X2, S2) = res
    assert s1 == 1 and s2 == s1 and i2 == i1, (i1, i2, s1, s2)
    assert abs(p2 - p1) <= 1e-9 * (1 + abs(p1)) and abs(d2 - d1) <= 1e-7 * (1 + abs(d1)), (p1, p2, d1, d2)
    if want is not None:
        assert abs(p2 - want) <= 1e-6 * (1 + abs(want)), (p2, want)
    assert relerr(y2, y1) <= 1e-6
    for a, b in zip(X2 + S2, X1 + S1):
        assert a.any() and relerr(a, b) <= 1e-6


def test_distributed_runs_are_bit_identical(pkg, golden_dir):
    """Two runs with the blocks distributed (world 3, loopback, mixed block sides with an LP block) give the same bits: the
    partial vectors are combined in rank order and the shared per-block values have one nonzero contribution each"""
    from loraine_jl_b200 import solver as S
    arrays, opts = _model(pkg, golden_dir, "multiblock_lp")
    outs = []
    for _ in range(2):
        opt, g = _solver(pkg, arrays, opts, world=3)
        S.initial_point(g)
        for _ in range(4):
            S.myIPstep(g, opt.halpha); g.itertime = 0.0; S.check_convergence(g)
        y, X, xl = S.get_solution(g)
        outs.append((y.copy(), [x.copy() for x in X], xl.copy(), g.DIMACS_error, g.get_array("RHS"), g.alpha.copy()))
        g.close()
    a, b = outs
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[2], b[2]) and a[3] == b[3]
    assert all(np.array_equal(x, z) for x, z in zip(a[1], b[1]))
    assert np.array_equal(a[4], b[4]) and np.array_equal(a[5], b[5])


@pytest.mark.parametrize("world", [2, 3])
def test_footprint_and_block_state_per_member(pkg, world):
    """Per member, the footprint lrn_finalize counts with distributed blocks differs from the replicated one by exactly
    dist.block_shard_bytes; a member keeps the whole state of the blocks it owns and only one m x m array (W) of the others --
    no X, S, SVD or scratch state"""
    arrays = _mixed_blocks((40, 200, 500, 120))
    _, g = _solver(pkg, arrays, dict(OPTS_SDPA), world=world)
    assert _blocks(g) == 1
    md = g.model
    n = md.n
    owner = pkg.dist.block_owner(md.msizes, world)
    for r in range(world):
        b = [C.c_int64(), C.c_int64()]
        held = (C.c_int64 * md.nlmi)()
        assert g.lib.lrn_dbg_block_footprint(g.h, r, 0, C.byref(b[0]), None) == 0
        assert g.lib.lrn_dbg_block_footprint(g.h, r, 1, C.byref(b[1]), held) == 0
        assert b[1].value - b[0].value == pkg.dist.block_shard_bytes(md.msizes, n, r, world), r
        for i, m in enumerate(md.msizes):
            mm = pkg.dist.pad_ld(m) * m * 8
            if owner[i] == r:
                assert held[i] >= 19 * mm, (r, i, held[i])
            else:
                assert held[i] == mm, (r, i, held[i])
    g.close()
    _, g = _solver(pkg, arrays, dict(OPTS_SDPA), world=world, blocks=0)
    held = (C.c_int64 * md.nlmi)()
    for r in range(world):
        assert g.lib.lrn_dbg_block_footprint(g.h, r, 0, None, held) == 0
        assert all(held[i] >= 19 * pkg.dist.pad_ld(m) * m * 8 for i, m in enumerate(md.msizes))
    g.close()


def test_kit1_and_single_block_models_stay_replicated(pkg, golden_dir):
    """kit = 1 and single-block models keep every block on every rank; forcing the distributed layout on a handle without a
    communicator fails at lrn_finalize"""
    arrays = golden(golden_dir, "vib3")[1]
    _, g = _solver(pkg, arrays, dict(OPTS_SDPA, kit=1), world=2)
    assert _blocks(g) == 0
    g.close()
    _, g = _solver(pkg, golden(golden_dir, "theta1")[1], dict(OPTS_SDPA), world=2)
    assert _blocks(g) == 0
    g.close()
    _, g = _solver(pkg, arrays, dict(OPTS_SDPA))
    assert _blocks(g) == 0
    g.close()
    with pytest.raises(Exception, match="sharded block layout"):
        _solver(pkg, arrays, dict(OPTS_SDPA), blocks=1)


# ---- two processes on two GPUs -------------------------------------------------------------------------------------------
_TWO_RANKS = """
import ctypes as C, os, sys
import numpy as np
import torch, torch.distributed as dist
sys.path.insert(0, {root!r}); sys.path.insert(0, os.path.join({root!r}, "tests"))
import __graft_entry__ as g
pkg = g.load_package()
from loraine_jl_b200 import solver as S
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dist.init_process_group("gloo")
opt = pkg.Optimizer()
for k, v in dict(kit=0, eDIMACS=1e-7, verb=0, datarank=0, initpoint=1, maxit=100, device=rank).items():
    opt.set_attribute(k, v)
opt.copy_to(pkg.raw_from_sdpa_arrays(*pkg.problems.multiblock_lp(5, 60, 40, 9)))
s = opt.solver
S.setup_solver(s, opt.halpha, before_finalize=pkg.dist.attach_before_finalize)
lay = C.c_int32(-9)
assert s.lib.lrn_dbg_block_layout(s.h, -2, C.byref(lay)) == 0 and lay.value == 1, lay.value
S.solve(s, opt.halpha, setup=False)
y, X, xl = S.get_solution(s)                     # collective: every block from its owner on both ranks
W = s.get_array("W", 3)
np.savez(os.path.join({out!r}, "rank%d.npz" % rank), y=y, W=W, iters=s.iter, status=s.status, obj=s.primal_obj,
         **{{"X%d" % i: x for i, x in enumerate(X)}})
s.close()
dist.barrier()
dist.destroy_process_group()
"""


def test_two_processes_distribute_the_blocks(pkg, tmp_path):
    """Two torchrun ranks (one process per GPU) that attach before lrn_finalize distribute five blocks; the solve matches one
    GPU, and the collective getters give both ranks the same X_i and W_i"""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import os
    import signal
    import socket
    import subprocess
    import sys
    import textwrap
    from loraine_jl_b200 import solver as S
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
        out, _ = p.communicate(timeout=900)
    except subprocess.TimeoutExpired:
        os.killpg(p.pid, signal.SIGKILL)
        p.communicate()
        pytest.fail("two-process run timed out")
    assert p.returncode == 0, out[-4000:]
    r0, r1 = (np.load(tmp_path / f"rank{r}.npz") for r in (0, 1))
    opt, g = _solver(pkg, pkg.problems.multiblock_lp(5, 60, 40, 9), dict(kit=0, eDIMACS=1e-7, verb=0, datarank=0, initpoint=1,
                                                                            maxit=100))
    S.solve(g, opt.halpha, setup=False)
    y1, X1, _ = S.get_solution(g)
    for r in (r0, r1):
        assert int(r["status"]) == g.status == 1 and int(r["iters"]) == g.iter
        assert abs(float(r["obj"]) - g.primal_obj) <= 1e-9 * (1 + abs(g.primal_obj))
    assert np.array_equal(r0["y"], r1["y"]) and np.array_equal(r0["W"], r1["W"])
    for i, x in enumerate(X1):
        assert np.array_equal(r0[f"X{i}"], r1[f"X{i}"])
        assert relerr(r0[f"X{i}"], x) <= 1e-6
    g.close()
