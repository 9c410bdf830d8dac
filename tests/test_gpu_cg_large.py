"""kit = 1 (CG) beyond the size of the direct path: the row-slab build of the H_alpha preconditioner, admission above
n_var = 140 000, the device-memory check of lrn_finalize, and nuclear-norm matrix completion solved to its known optimum.

On this model class the reference's H_alpha preconditioner does not reach eDIMACS = 1e-6: with erank >= 2 the Cholesky
factorisation of S = T'T + I fails once mu is about 1e-7 (T has k(k-1)/2 null directions, antisymmetric combinations of
the columns of U, while its other singular values grow as 1/tau), and with erank = 1 the NumPy oracle needs about 100 IP
iterations on a 60 x 60 instance.  H_beta (preconditioner 2) solves it in 16-17.  So the solves to the optimum use
H_beta; the H_alpha tests check the slab build and a few IP iterations against the one-slab build.
"""
import ctypes as C

import numpy as np
import pytest

import mc_instances as mc

pytestmark = pytest.mark.gpu

CG = dict(kit=1, aamat=2, initpoint=1, verb=0, eDIMACS=1e-6)


def _error():
    from loraine_jl_b200.solver import LoraineB200Error
    return LoraineB200Error


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def relerr(a, b):
    return np.linalg.norm(np.asarray(a) - np.asarray(b)) / max(np.linalg.norm(np.asarray(b)), 1e-300)


def _optimizer(pkg, inst, **opts):
    opt = pkg.Optimizer()
    for k, v in dict(CG, **opts).items():
        opt.set_attribute(k, v)
    opt.load_sdpa(*inst.arrays)
    return opt


def _slab(s, rows):
    used = C.c_int64(-1)
    assert s.lib.lrn_dbg_prec_slab(s.h, rows, C.byref(used)) == 0
    return used.value


def _check_optimum(s, inst, rel_obj=1e-5, rel_y=1e-4):
    assert s.status == 1, s.status
    assert abs(s.primal_obj - inst.optimum) <= rel_obj * abs(inst.optimum), (s.primal_obj, inst.optimum)
    r = inst.M.shape[0]
    assert relerr(s.X[0][:r, r:], inst.M) <= rel_y


def _prepare_alpha(S, s):
    """one predictor's worth of state, then the H_alpha build"""
    S.find_mu(s)
    S.prepare_W(s)
    s._call("lrn_residuals")
    s._call("lrn_rhs_predictor")
    s._call("lrn_prec_prepare", 1)


@pytest.fixture(scope="module")
def inst20k():
    return mc.matrix_completion(200, 200, 2, 20000, seed=21)


@pytest.fixture(scope="module")
def inst162k():
    return mc.matrix_completion(600, 600, 2, 162000, seed=22)


def test_slab_parity_operator(pkg, inst20k):
    """The H_alpha apply after slab builds of height 1, 777, 1000 and n_var - 1 equals the one-slab build."""
    from loraine_jl_b200 import solver as S
    opt = _optimizer(pkg, inst20k, preconditioner=1, erank=2)
    s = opt.solver
    S.setup_solver(s, opt.halpha)
    S.initial_point(s)
    for _ in range(3):
        S.myIPstep(s, opt.halpha)
    n = inst20k.n
    _prepare_alpha(S, s)
    assert _slab(s, 0) == n                                # 20000 x (800 + 400) doubles fit one slab
    x = np.random.default_rng(5).standard_normal(n)
    ref = np.zeros(n)
    s._call("lrn_apply_operator", 1, _dp(x), _dp(ref))
    for R in (1, 777, 1000, n - 1):
        _slab(s, R)
        s._call("lrn_prec_prepare", 1)
        assert _slab(s, R) == R
        out = np.zeros(n)
        s._call("lrn_apply_operator", 1, _dp(x), _dp(out))
        assert relerr(out, ref) <= 1e-11, R
    _slab(s, 0)
    s._call("lrn_prec_prepare", 1)
    out = np.zeros(n)
    s._call("lrn_apply_operator", 1, _dp(x), _dp(out))
    np.testing.assert_array_equal(out, ref)               # back to one slab: the same launches, the same bits
    s.close()


def test_slab_parity_ip_iterations(pkg, inst20k):
    """Five IP iterations with slab builds of height 1, 777, 1000 and n_var - 1 follow the one-slab run: the same
    iterations, CG totals within 2 %, objectives within 1e-8."""
    from loraine_jl_b200 import solver as S

    def run(R):
        opt = _optimizer(pkg, inst20k, preconditioner=1, erank=2)
        s = opt.solver
        S.setup_solver(s, opt.halpha)
        _slab(s, R)
        S.solve(s, opt.halpha, max_iters=5, setup=False)
        tr = [(t["iter"], t["obj"]) for t in s.trace]
        used = _slab(s, R)
        s.close()
        return tr, s.cg_iter_tot, used

    ref, cg0, used0 = run(0)
    assert used0 == inst20k.n and len(ref) == 5
    for R in (1, 777, 1000, inst20k.n - 1):
        tr, cg, used = run(R)
        assert used == R
        assert [t[0] for t in tr] == [t[0] for t in ref]
        assert abs(cg - cg0) <= 0.02 * cg0, (R, cg, cg0)
        for (_, a), (_, b) in zip(tr, ref):
            assert abs(a - b) <= 1e-8 * (1 + abs(b)), (R, a, b)


def test_above_old_limit_kit0_refused(pkg, inst162k):
    opt = _optimizer(pkg, inst162k, kit=0)
    with pytest.raises(_error(), match=r"n_var out of range \(1\.\.140000\)"):
        opt.optimize()


def test_above_old_limit_solves(pkg, inst162k):
    """600 x 600, rank 2, 162 000 observed entries (n_var above 140 000): kit = 1 reaches the known optimum -||M||_*, and
    the H_alpha build there runs in several slabs whose S gives the same apply as one whole-height slab."""
    from loraine_jl_b200 import solver as S
    opt = _optimizer(pkg, inst162k, preconditioner=2)
    opt.optimize()
    s = opt.solver
    _check_optimum(s, inst162k)
    assert abs(opt.objective_value() - inst162k.optimum) <= 1e-5 * abs(inst162k.optimum)
    s.close()

    opt = _optimizer(pkg, inst162k, preconditioner=1, erank=2)
    s = opt.solver
    S.setup_solver(s, opt.halpha)
    S.initial_point(s)
    for _ in range(2):
        S.myIPstep(s, opt.halpha)
        assert s.status == 0
    _prepare_alpha(S, s)
    n = inst162k.n
    used = _slab(s, 0)
    assert 8 <= used < n and used % 8 == 0
    x = np.random.default_rng(6).standard_normal(n)
    sl = np.zeros(n)
    s._call("lrn_apply_operator", 1, _dp(x), _dp(sl))
    _slab(s, n)
    s._call("lrn_prec_prepare", 1)
    whole = np.zeros(n)
    s._call("lrn_apply_operator", 1, _dp(x), _dp(whole))
    assert relerr(sl, whole) <= 1e-11
    with pytest.raises(_error(), match="exists only for kit = 0"):
        s.get_array("H")
    s.close()


def test_two_million_constraint_scale(pkg):
    """2000 x 2000, rank 1, 1.2 M observed entries (more than 2^20 constraints, one 4000 x 4000 block): the H_alpha state
    adds less than 10 GB across lrn_finalize and the first lrn_prec_prepare (whole T and A_j u_r would be 77 GB), its build
    runs in slabs, and the model solves to -||M||_*."""
    import torch
    from loraine_jl_b200 import solver as S
    inst = mc.matrix_completion(2000, 2000, 1, 1_200_000, seed=23)
    opt = _optimizer(pkg, inst, preconditioner=1, erank=1)
    s = opt.solver
    torch.cuda.init()
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info(0)[0]
    S.setup_solver(s, opt.halpha)
    S.initial_point(s)
    _prepare_alpha(S, s)
    torch.cuda.synchronize()
    drop = free0 - torch.cuda.mem_get_info(0)[0]
    assert drop < 10e9, drop
    used = _slab(s, 0)
    assert used < inst.n
    s.preconditioner = 2
    S.solve(s, opt.halpha, setup=False)
    _check_optimum(s, inst)
    s.close()


def test_lp_block_above_limit(pkg):
    """With an LP block H_alpha would form and factor the dense n_var x n_var AAAATtau: refused above 140 000; H_beta,
    which needs only its diagonal, runs."""
    from loraine_jl_b200 import solver as S
    inst = mc.matrix_completion(600, 600, 2, 162000, seed=22, lp_rows=10)
    opt = _optimizer(pkg, inst, preconditioner=1, erank=2)
    s = opt.solver
    S.setup_solver(s, opt.halpha)
    S.initial_point(s)
    S.find_mu(s)
    S.prepare_W(s)
    s._call("lrn_residuals")
    s._call("lrn_rhs_predictor")
    rc = s.lib.lrn_prec_prepare(s.h, 1)
    assert rc == -6, rc                                    # LRN_ERR_UNSUPPORTED
    assert "AAAATtau" in s._err() and "preconditioner 2" in s._err()
    s.close()
    opt = _optimizer(pkg, inst, preconditioner=2)
    opt.optimize(max_iters=2)
    assert opt.solver.iter == 2 and opt.solver.status == 0 and opt.solver.cg_iter_tot > 0
    opt.solver.close()


def test_finalize_refuses_state_larger_than_the_device(pkg, inst20k):
    """erank = 398 on the m = 400 block makes S (159 200^2 doubles, 203 GB) larger than any B200: lrn_finalize refuses it
    with both byte counts instead of failing partway through a solve."""
    opt = _optimizer(pkg, inst20k, preconditioner=1, erank=398)
    with pytest.raises(_error(), match=r"kit = 1 state needs \d+ bytes of device memory, \d+ bytes are free"):
        opt.optimize()


def test_two_gpus_replicate_single_gpu(pkg, inst162k):
    """ngpus = 2 runs the replicated kit = 1 path: the iterate equals the single-GPU one bit for bit."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")

    def run(ngpus):
        opt = _optimizer(pkg, inst162k, preconditioner=1, erank=2, ngpus=ngpus)
        opt.optimize(max_iters=3)
        s = opt.solver
        out = (s.y.copy(), s.X[0].copy(), s.cg_iter_tot)
        s.close()
        return out

    y1, X1, cg1 = run(1)
    y2, X2, cg2 = run(2)
    assert cg1 == cg2
    np.testing.assert_array_equal(y1, y2)
    np.testing.assert_array_equal(X1, X2)
