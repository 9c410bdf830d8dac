"""GPU tests of the multi-GPU double-double LP path (lrn_dd_create_multi, lrn_dd_dist_init, csrc/dddist.cu): the sharded Schur
assembly checked shard by shard on ONE GPU, the distributed Cholesky run with a world-1 NCCL communicator against the
single-GPU handle (the factorisation follows the single-GPU tile order, so the results agree to the last bit), the pivot
failure protocol, the in-process handle through Optimizer(T="Float64x2"), and two processes on two GPUs."""
import ctypes as C
import os
import signal
import subprocess
import sys
import textwrap
from fractions import Fraction

import mpmath as mp
import numpy as np
import pytest

import jump_examples as je
import test_gpu_dd
from dd_common import random_lp
from test_gpu_dd import _mp_vec, _rel, _setup

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PD = C.POINTER(C.c_double)


def _world1(s):
    """attach a dd handle to a one-rank NCCL communicator: the whole distributed code path on one GPU"""
    import torch  # noqa: F401  (loads the bundled libnccl into the process)
    buf = C.create_string_buffer(128)
    assert s.lib.lrn_dist_unique_id(buf) == 0
    s._call("lrn_dd_dist_init", 0, 1, buf)


def _iterate(s):
    hi = {k: np.zeros(s.model.n if k[0] == "y" else s.model.nlin) for k in ("yh", "yl", "xh", "xl", "sh", "sl")}
    s._call("lrn_dd_get_solution", *[hi[k].ctypes.data_as(PD) for k in ("yh", "yl", "xh", "xl", "sh", "sl")])
    return hi


def _set_iterate(s, it):
    s._call("lrn_dd_set_iterate", *[it[k].ctypes.data_as(PD) for k in ("yh", "yl", "xh", "xl", "sh", "sl")])


def _ddrel(a, b):
    """relative Frobenius distance of two double-double arrays (hi, lo); exact 0 for identical arrays"""
    d = (a[0] - b[0]) + (a[1] - b[1])
    den = np.linalg.norm(b[0])
    return float(np.linalg.norm(d) / den) if den else float(np.linalg.norm(d))


def _same(a, b):
    return np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


@pytest.mark.parametrize("world", [2, 3])
def test_dd_row_shards_add_up_to_the_single_gpu_schur_matrix(pkg, world):
    """lrn_dd_dbg_set_shard (no communicator): every rank's lrn_dd_schur_assemble writes exactly its own 32-row blocks of the
    lower triangle, the shards are disjoint, their sum is the single-GPU lower triangle bit for bit, and a hooked handle
    refuses to factor its shard (LRN_ERR_STATE)."""
    spec = random_lp(300, 700, 9, density=0.1)
    dd_lp, s0, _ = _setup(pkg, spec)
    dd_lp.myIPstep(s0)
    s0.itertime = 0.0
    dd_lp.check_convergence(s0)
    it = _iterate(s0)
    dd_lp.find_mu(s0); dd_lp.prepare_W(s0)
    s0._call("lrn_dd_residuals"); s0._call("lrn_dd_schur_assemble")
    H0 = tuple(np.tril(a) for a in s0.get_array("H"))
    n, br = 300, 32
    rows = np.arange(n)
    total = [np.zeros((n, n)), np.zeros((n, n))]
    filled = np.zeros((n, n), dtype=np.int32)
    for rank in range(world):
        _, s, _ = _setup(pkg, spec)
        _set_iterate(s, it)
        assert s.lib.lrn_dd_dbg_set_shard(s.h, rank, world, br) == 0
        dd_lp.find_mu(s); dd_lp.prepare_W(s)
        s._call("lrn_dd_residuals"); s._call("lrn_dd_schur_assemble")
        Hh, Hl = s.get_array("H")
        mine = (rows // br) % world == rank
        assert not Hh[~mine].any() and not Hl[~mine].any(), (world, rank)        # nothing outside my rows, no upper mirror
        assert not np.triu(Hh, 1).any()
        assert np.abs(np.diag(Hh)[mine]).min() > 0
        assert s.lib.lrn_dd_schur_factor(s.h) == -4                              # LRN_ERR_STATE: must not factor a shard
        total[0] += Hh
        total[1] += Hl
        filled += (Hh != 0) | (Hl != 0)
        s.close()
    assert filled.max() <= 1
    assert _same(total, H0), world
    s0.close()


def _phases(dd_lp, s):
    """one IP iteration call by call; returns what the parity checks compare"""
    out = {}
    s.iter += 1
    dd_lp.find_mu(s); dd_lp.prepare_W(s)
    s.predict = True
    for name in ("lrn_dd_residuals", "lrn_dd_schur_assemble", "lrn_dd_rhs_predictor"):
        s._call(name)
    assert s._call("lrn_dd_schur_factor", allow_positive=True) == 0
    s.chol_is_factor_object = False
    out["H"] = s.get_array("H")
    out["L"] = tuple(np.tril(a) for a in s.get_array("L"))
    out["rhs_pred"] = s.get_array("RHS")
    s._call("lrn_dd_schur_solve", 3)
    out["dely_pred"] = s.get_array("DELY")
    dd_lp._find_step(s, True)
    out["ab_pred"] = (tuple(s.alpha_lin), tuple(s.beta_lin))
    out["sigma"] = dd_lp.sigma_update(s)
    dd_lp.corrector(s)
    out["rhs_corr"] = s.get_array("RHS")
    out["dely"] = s.get_array("DELY")
    out["ab"] = (tuple(s.alpha_lin), tuple(s.beta_lin))
    dd_lp.get_solution(s)
    out["y"], out["x"], out["s"] = s.y_dd, s.X_lin_dd, s.S_lin_dd
    return out


@pytest.mark.parametrize("n,nlin,density", [(300, 700, 0.1), (1100, 2200, 0.02)])
def test_dd_distributed_cholesky_with_a_world1_communicator(pkg, n, nlin, density):
    """the whole distributed path (sharded assembly, diagonal-block broadcast, row solves, all-gather, trailing update, H
    gather) with a one-rank communicator: n = 300 -> 5 row blocks of 64 (ragged last one), n = 1100 -> 9 blocks of 128.
    Two full IP iterations against a plain handle on the same device."""
    spec = random_lp(n, nlin, 21 + n, density=density)
    dd_lp, s1, _ = _setup(pkg, spec)
    _, s2, _ = _setup(pkg, spec)
    _world1(s2)
    assert pkg.dist.dd_block_rows(n) == (64 if n < 1024 else 128)
    tol = mp.mpf(1e-28)
    for _ in range(2):
        a, b = _phases(dd_lp, s1), _phases(dd_lp, s2)
        assert _same(b["H"], a["H"])
        assert _ddrel(b["L"], a["L"]) <= 1e-28
        for k in ("rhs_pred", "dely_pred", "rhs_corr", "dely", "y", "x", "s"):
            assert _rel(_mp_vec(*b[k]), _mp_vec(*a[k])) <= tol, k
        assert b["ab_pred"] == a["ab_pred"] and b["ab"] == a["ab"] and b["sigma"] == a["sigma"]
    s1.close(); s2.close()


def test_dd_phase_parity_with_a_world1_communicator(pkg, monkeypatch):
    """test_phase_parity_two_iterations (every phase against the 160-bit oracle at 1e-26) on a world-1 distributed handle;
    n = 70 gives 2 row blocks of 64."""
    def setup_world1(pkg_, spec, eD=1e-25):
        dd_lp, s, omd = _setup(pkg_, spec, eD)
        _world1(s)
        return dd_lp, s, omd
    monkeypatch.setattr(test_gpu_dd, "_setup", setup_world1)
    test_gpu_dd.test_phase_parity_two_iterations(pkg, 70, 160)


def test_dd_pivot_failure_world1(pkg):
    """a non-positive pivot: the world-1 distributed factorisation reports the single-GPU LAPACK-style index; shifting back
    factors again, to the single-GPU factor"""
    spec = random_lp(300, 700, 9, density=0.1)
    dd_lp, s1, _ = _setup(pkg, spec)
    _, s2, _ = _setup(pkg, spec)
    _world1(s2)
    for s in (s1, s2):
        dd_lp.find_mu(s); dd_lp.prepare_W(s)
        s._call("lrn_dd_residuals"); s._call("lrn_dd_schur_assemble"); s._call("lrn_dd_rhs_predictor")
        assert s._call("lrn_dd_schur_factor", allow_positive=True) == 0
    L0 = tuple(np.tril(a) for a in s1.get_array("L"))
    for s in (s1, s2):
        s._call("lrn_dd_schur_shift", -1e6)
    i1 = s1._call("lrn_dd_schur_factor", allow_positive=True)
    i2 = s2._call("lrn_dd_schur_factor", allow_positive=True)
    assert i1 > 0 and i2 == i1
    for s in (s1, s2):
        s._call("lrn_dd_schur_shift", 1e6)
        assert s._call("lrn_dd_schur_factor", allow_positive=True) == 0
    L1 = tuple(np.tril(a) for a in s1.get_array("L"))
    L2 = tuple(np.tril(a) for a in s2.get_array("L"))
    assert _ddrel(L2, L1) <= 1e-28
    assert _ddrel(L1, L0) <= 1e-24                     # (the diagonal went through -1e6 and back: a few ulps of 1e6 in dd)
    s1.close(); s2.close()


@pytest.mark.parametrize("case", ["k.jl", "random_lp"])
def test_dd_in_process_multi_gpu_optimizer(pkg, case):
    """Optimizer(T="Float64x2") with ngpus = 1, 2 and all visible GPUs (lrn_dd_create_multi).  examples/k.jl has a single
    multiplier: every rank but 0 owns no row.  With one visible GPU this checks the fallback to a single-device handle."""
    import torch
    ndev = torch.cuda.device_count()
    spec = je.ex_k_lp() if case == "k.jl" else random_lp(300, 700, 5)
    res = []
    for ngpus in sorted({1, min(2, ndev), ndev}):
        opt = pkg.Optimizer(T="Float64x2")
        opt.set_attribute("verb", 0)
        opt.set_attribute("eDIMACS", 1e-24)
        opt.set_attribute("ngpus", ngpus)
        opt.copy_to(pkg.RawProblem(**je.fields(spec)), max_sense=(case == "k.jl"))
        opt.optimize()
        s = opt.solver
        assert opt.termination_status() == "OPTIMAL", ngpus
        res.append((ngpus, s.iter, opt.objective_value_dd(), _mp_vec(*s.y_dd)))
        s.close()
    _, it0, obj0, y0 = res[0]
    for ngpus, it, obj, y in res[1:]:
        assert it == it0, ngpus
        assert abs(obj - obj0) <= Fraction(1, 10 ** 24) * abs(obj0), ngpus
        assert _rel(y, y0) <= mp.mpf(1e-20), ngpus
    if case == "k.jl":
        assert abs(obj0 - 4) <= Fraction(1, 10 ** 24)


_TWO_RANKS = """
import ctypes as C, os, sys
import numpy as np
import torch, torch.distributed as dist
sys.path.insert(0, {root!r}); sys.path.insert(0, os.path.join({root!r}, "tests"))
import __graft_entry__ as g
pkg = g.load_package()
from loraine_jl_b200 import dd_lp
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dist.init_process_group("gloo")
spec = pkg.problems.random_lp(1100, 2200, 7, density=0.02)
o = dict(pkg.DEFAULT_OPTIONS, eDIMACS=1e-24, verb=0, device=rank)

def run(sharded):
    s = dd_lp.DDSolver(pkg.prepare_model(pkg.RawProblem(**spec)), o)
    dd_lp.setup_solver(s)
    if sharded:
        assert pkg.dist.init_distributed_dd(s)
    dd_lp.initial_point(s)
    out = []
    for _ in range(2):
        dd_lp.myIPstep(s)
        out.append(s.get_array("DELY"))
        s.itertime = 0.0
        dd_lp.check_convergence(s)
    s.close()
    return out

got = run(True)
if rank == 0:
    want = run(False)
    for a, b in zip(got, want):
        d = (a[0] - b[0]) + (a[1] - b[1])
        rel = np.linalg.norm(d) / np.linalg.norm(b[0])
        assert rel <= 1e-28, rel
dist.barrier()
open(os.path.join({out!r}, "ok%d" % rank), "w").write("ok")
dist.destroy_process_group()
"""


def test_dd_two_processes_two_gpus(pkg, tmp_path):
    """lrn_dd_dist_init with two processes on two GPUs (torch.distributed.run, gloo only for the unique-id exchange): the
    same dely as one GPU in both iterations.  The launcher runs in its own process group, joined with a time-out; on a
    time-out the whole group is killed, so that no process is left behind."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "two_ranks.py"
    script.write_text(textwrap.dedent(_TWO_RANKS.format(root=ROOT, out=str(tmp_path))))
    import socket
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
    assert (tmp_path / "ok0").exists() and (tmp_path / "ok1").exists()
