"""Host side of the double-double LP path (include/loraine_b200_dd.h): `Optimizer{Float64x2}` of the reference (README.md:37-54,
examples/k.jl:8) for models without semidefinite blocks.

Same split as solver.py: the control flow of src/Solvers.jl:304-361, :448-568 and src/predictor_corrector.jl stays on the host,
every array expression is one call into libloraine_b200.so (CUDA, double-double arithmetic); there is no CPU fallback.
A Float64x2 scalar travels as a (hi, lo) pair -- the two limbs of MultiFloats' Float64x2; the few scalar decisions the host
takes on such pairs (comparisons, the sum of the DIMACS errors, 3 * step^2) are done exactly with `fractions.Fraction`.
"""
from __future__ import annotations

import ctypes as C
import math
import time
from fractions import Fraction

import numpy as np
import scipy.sparse as sp

from . import _lib
from .model import MyModel


class LoraineB200DDError(RuntimeError):
    pass


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int64))


def frac(pair) -> Fraction:
    """exact value of a double-double (hi, lo)"""
    return Fraction(float(pair[0])) + Fraction(float(pair[1]))


def pair_of(x) -> np.ndarray:
    """nearest double-double of an exact / double value"""
    if isinstance(x, Fraction):
        hi = float(x)
        return np.array([hi, float(x - Fraction(hi))])
    if isinstance(x, (tuple, list, np.ndarray)):
        return np.array([float(x[0]), float(x[1])])
    return np.array([float(x), 0.0])


class DDSolver:
    """MySolver{Float64x2} for nlmi = 0 (src/Solvers.jl:18-147)."""

    def __init__(self, model: MyModel, o: dict):
        if model.nlmi != 0:
            raise TypeError("Optimizer{Float64x2}: the B200 double-double path covers models without PSD blocks only; "
                            "semidefinite models run in Float64 (no fallback)")
        if model.nlin == 0:
            raise ValueError("empty model")
        self.model = model
        self.eDIMACS = float(o["eDIMACS"])
        self.maxit = int(o["maxit"])
        self.initpoint = int(o["initpoint"])
        self.verb = int(o["verb"])
        self.device = int(o.get("device", -1))
        self.ngpus = int(o.get("ngpus", 1))        # 1: one device; otherwise lrn_dd_create_multi (<= 0: every visible device)
        self.lib = _lib.lib()
        self.h = C.c_void_p()
        self.status = 0
        self.iter = 0
        self.regcount = 0
        self.tottime = 0.0

    # ---- plumbing ------------------------------------------------------------------------------------------------------
    def _err(self):
        return (self.lib.lrn_dd_last_error(self.h) or b"").decode()

    def _call(self, name, *args, allow_positive=False):
        rc = getattr(self.lib, name)(self.h, *args)
        if rc < 0 or (rc > 0 and not allow_positive):
            raise LoraineB200DDError(f"{name} failed ({rc}): {self._err()}")
        return rc

    def close(self):
        if self.h:
            self.lib.lrn_dd_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def get_array(self, name):
        md = self.model
        which = _lib.DD_ARR[name]
        size = md.n * md.n if which in (1, 2) else (md.n if which in (3, 5, 6) else md.nlin)
        hi, lo = np.zeros(size), np.zeros(size)
        self._call("lrn_dd_get_array", which, _dp(hi), _dp(lo))
        if which in (1, 2):
            return hi.reshape(md.n, md.n, order="F"), lo.reshape(md.n, md.n, order="F")
        return hi, lo

    def timers(self, reset=False):
        ms = np.zeros(4)
        self._call("lrn_dd_timers", _dp(ms), 1 if reset else 0)
        return dict(schur_assemble=ms[0], schur_factor=ms[1], schur_solve=ms[2], other=ms[3])


def setup_solver(s: DDSolver):
    md = s.model
    if s.h:
        s.close()
    if s.ngpus != 1:                           # one host thread, N devices: the library owns the NCCL communicator
        rc = s.lib.lrn_dd_create_multi(C.byref(s.h), md.n, md.nlin, s.ngpus, None)
        if rc != 0:
            raise LoraineB200DDError(f"lrn_dd_create_multi(ngpus={s.ngpus}) failed ({rc}): not enough usable sm_100 CUDA devices "
                                     "or no NCCL; there is no CPU fallback")
    else:
        rc = s.lib.lrn_dd_create(C.byref(s.h), md.n, md.nlin, s.device)
        if rc != 0:
            raise LoraineB200DDError(f"lrn_dd_create failed ({rc}): no usable sm_100 CUDA device; there is no CPU fallback")
    M = sp.csc_matrix(md.C_lin)
    M.sum_duplicates()
    M.sort_indices()
    cp = M.indptr.astype(np.int64) + 1
    rv = M.indices.astype(np.int64) + 1
    nz = np.ascontiguousarray(M.data, dtype=np.float64)
    d = np.ascontiguousarray(md.d_lin, dtype=np.float64)
    b = np.ascontiguousarray(md.b, dtype=np.float64)
    s._call("lrn_dd_set_lin", _ip(cp), _ip(rv), _dp(nz), None, _dp(d), None)
    s._call("lrn_dd_set_b", _dp(b), None)
    s._call("lrn_dd_finalize")
    s.regcount = 0


def initial_point(s: DDSolver):
    """src/initial_point.jl:1-81 (Float64 norms of the model data on the host), then upload."""
    md = s.model
    n, dd = md.n, md.nlin
    b2 = 1 + np.abs(md.b)
    rown = np.sqrt(np.asarray(md.C_lin.multiply(md.C_lin).sum(axis=1)).ravel())
    if s.initpoint == 0:
        Epss, Etaa = 1.0, 1.0
    else:
        Epss = max(1.0, float((b2 / (1 + rown)).max()))
        mf = max(float(rown.max()), float(np.linalg.norm(md.d_lin))) / math.sqrt(dd)
        Etaa = max(1.0, mf)
    y = np.zeros(n)
    x = Epss * np.ones(dd)
    sl = Etaa * np.ones(dd)
    s._call("lrn_dd_set_iterate", _dp(y), None, _dp(x), None, _dp(sl), None)
    s.sigma = 3.0
    s.tau = 0.95
    s.expon = 3.0
    s.DIMACS_error = Fraction(1)
    s.iter = 0
    s.status = 0


def find_mu(s):
    mu = np.zeros(2)
    s._call("lrn_dd_find_mu", _dp(mu))
    s.mu = mu
    return mu


def prepare_W(s):
    s._call("lrn_dd_prepare_W")


def _find_step(s, predict):
    a, b = np.zeros(2), np.zeros(2)
    s._call("lrn_dd_find_step", 1 if predict else 0, _dp(pair_of(s.sigma)), _dp(s.mu), float(s.tau), _dp(a), _dp(b))
    s.alpha_lin, s.beta_lin = a, b


def predictor(s):
    """src/predictor_corrector.jl:5-146, kit = 0 branch."""
    s.predict = True
    s._call("lrn_dd_residuals")
    s._call("lrn_dd_schur_assemble")
    s._call("lrn_dd_rhs_predictor")
    rc = s._call("lrn_dd_schur_factor", allow_positive=True)
    s.chol_is_factor_object = False
    if rc > 0:
        if s.verb > 0:
            print("Matrix H not positive definite, trying to regularize")
        icount = 0
        s.regcount += 1
        if s.regcount > 5:
            if s.verb > 0:
                print("WARNING: too many regularizations of H, giving up")
            s.status = 3
            return
        while True:
            s._call("lrn_dd_schur_shift", 1e-4)
            icount += 1
            if s._call("lrn_dd_schur_factor", allow_positive=True) == 0:
                break
            if icount > 1000:
                if s.verb > 0:
                    print("WARNING: H cannot be made positive definite, giving up")
                s.status = 3
                return
        s.chol_is_factor_object = True
    s._call("lrn_dd_schur_solve", 6 if s.chol_is_factor_object else 3)
    _find_step(s, True)


def sigma_update(s):
    """src/predictor_corrector.jl:148-179: the exponent from the exact double-double step, the power in Float64 (:173-175)."""
    md = s.model
    step_pred = min(frac(s.alpha_lin), frac(s.beta_lin))
    mu = frac(s.mu)
    if mu > Fraction(1e-6):
        if step_pred < Fraction(1 / math.sqrt(3)):
            expon_used = 1.0
        else:
            expon_used = max(s.expon, float(3 * step_pred * step_pred))
    else:
        expon_used = max(1.0, min(s.expon, float(3 * step_pred * step_pred)))
    dl = np.zeros(2)
    s._call("lrn_dd_sigma_trace", _dp(dl))
    tmp12 = float(frac(dl) / md.nlin)
    s.sigma = min(1.0, (tmp12 / float(mu)) ** expon_used)
    return s.sigma


def corrector(s):
    """src/predictor_corrector.jl:181-246, kit = 0 branch."""
    s.predict = False
    s._call("lrn_dd_rhs_corrector", _dp(pair_of(s.sigma)), _dp(s.mu))
    s._call("lrn_dd_schur_solve", 6 if s.chol_is_factor_object else 3)
    _find_step(s, False)


def check_convergence(s):
    """src/Solvers.jl:496-568 for nlmi = 0."""
    md = s.model
    err = np.zeros(12)
    by, dx = np.zeros(2), np.zeros(2)
    s._call("lrn_dd_dimacs", _dp(err), _dp(by), _dp(dx))
    e = [frac(err[2 * k:2 * k + 2]) for k in range(6)]
    s.err1, s.err2, s.err3, s.err4, s.err5, s.err6 = e
    D = e[1] + e[2] + e[3] + abs(e[4]) + e[5]              # nlmi = 0: err1 is not part of the sum (src/Solvers.jl:521)
    s.DIMACS_error = D
    s.by, s.dx = by, dx
    s.primal_obj = -frac(by) + Fraction(md.b_const)
    s.dual_obj = -frac(dx)
    if s.verb > 0 and s.status == 0:
        print(f"{s.iter:3d} {float(s.primal_obj):16.8e} {float(D):9.2e} {s.itertime:8.2f}")
    if D < Fraction(s.eDIMACS):
        s.status = 1
        if s.verb > 0:
            print("Primal objective: ", float(s.primal_obj))
            print("Dual objective:   ", float(s.dual_obj))
    if D > Fraction(1e55):
        s.status = 2
    elif abs(frac(by)) > Fraction(1e55):
        s.status = 3


def myIPstep(s):
    """src/Solvers.jl:448-478"""
    s.iter += 1
    if s.iter > s.maxit:
        s.status = 4
        if s.verb > 0:
            print("WARNING: Stopped by iteration limit (stopping status = 4)")
    find_mu(s)
    prepare_W(s)
    predictor(s)
    if s.status == 3:
        return
    sigma_update(s)
    corrector(s)


def get_solution(s):
    md = s.model
    out = {k: np.zeros(md.n if k.startswith("y") else md.nlin) for k in ("y_hi", "y_lo", "x_hi", "x_lo", "s_hi", "s_lo")}
    s._call("lrn_dd_get_solution", *[_dp(out[k]) for k in ("y_hi", "y_lo", "x_hi", "x_lo", "s_hi", "s_lo")])
    s.y_dd = (out["y_hi"], out["y_lo"])
    s.X_lin_dd = (out["x_hi"], out["x_lo"])
    s.S_lin_dd = (out["s_hi"], out["s_lo"])
    s.y, s.X_lin, s.S_lin = out["y_hi"], out["x_hi"], out["s_hi"]
    return s


def solve(s: DDSolver, max_iters=None, setup=True):
    """src/Solvers.jl:304-361"""
    t1 = time.perf_counter()
    if setup:
        setup_solver(s)
        initial_point(s)
    while s.status == 0:
        t2 = time.perf_counter()
        myIPstep(s)
        s.itertime = time.perf_counter() - t2
        if s.status == 3:
            break
        check_convergence(s)
        if max_iters is not None and s.iter >= max_iters:
            break
    get_solution(s)
    s.tottime = time.perf_counter() - t1
    return s
