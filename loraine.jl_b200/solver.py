"""Host-side mirror of the reference's `Solvers` module (src/Solvers.jl, src/predictor_corrector.jl, src/prepare_W.jl,
src/initial_point.jl) with every array expression replaced by one call into the C-ABI CUDA library.

The control flow (predictor/corrector, regularisation retry loop, sigma update, convergence test, hybrid
preconditioner switch, option checks) is kept statement by statement so that this file reads like the reference
with `ccall`s in place of the linear algebra; julia/LoraineB200.jl is the same thing for a Julia host.
Function names, argument meaning and error behaviour follow the reference.
"""
from __future__ import annotations

import ctypes as C
import math
import time

import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from . import _lib
from .model import MyModel, RawProblem, prepare_model, raw_from_sdpa_arrays

# src/Solvers.jl:169-185
DEFAULT_OPTIONS = {
    "kit": 0, "tol_cg": 1.0e-2, "tol_cg_up": 0.5, "tol_cg_min": 1.0e-7, "eDIMACS": 1.0e-7, "preconditioner": 1,
    "erank": 1, "aamat": 1, "fig_ev": 0, "verb": 1, "datarank": 0, "initpoint": 0, "timing": 1, "maxit": 100,
    "datasparsity": 8,
}


class PosDefException(Exception):
    """Raised like LinearAlgebra.PosDefException(info) when a Cholesky factorisation meets a non-positive pivot."""

    def __init__(self, info):
        super().__init__(f"matrix is not positive definite; Cholesky factorization failed (info = {info}).")
        self.info = info


class LoraineB200Error(RuntimeError):
    pass


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int64))


class Halpha:
    """src/Solvers.jl:149-162 -- the factors live on the device; this object only records that they exist."""

    def __init__(self, kit):
        self.kit = kit
        self.prepared_kind = 0


class _DeviceFactor:
    """The `solver.cholBBBB` seam (src/predictor_corrector.jl:57,85,89-90,199).

    `is_cholesky_object = False`: plays the LowerTriangular factor L; the reference expression
    `cholBBBB' \\ (cholBBBB \\ h)` is L' \\ (L \\ h).  `True` (only after a regularised retry, :85): plays Julia's
    `Cholesky` object whose adjoint is itself, so the same expression evaluates H^-1 (H^-1 h) -- kept as is.
    """

    def __init__(self, solver, is_cholesky_object):
        self.solver = solver
        self.is_cholesky_object = is_cholesky_object

    def solve_reference_expression(self):
        self.solver._call("lrn_schur_solve", 6 if self.is_cholesky_object else 3)


class MySolver:
    """src/Solvers.jl:18-147.  Iterates and scalings are device resident (behind `self.h`)."""

    def __init__(self, model: MyModel, o: dict):
        for k in ("kit", "preconditioner", "erank", "aamat", "fig_ev", "verb", "datarank", "initpoint", "timing", "maxit",
                  "datasparsity"):
            setattr(self, k, int(o[k]))
        for k in ("tol_cg", "tol_cg_up", "tol_cg_min", "eDIMACS"):
            setattr(self, k, float(o[k]))
        self.model = model
        self.lib = _lib.lib()
        self.h = C.c_void_p()
        self.cg_iter_tot = 0
        self.trace = []
        self.status = 0
        self.extra = {k: o[k] for k in ("svd_tol", "lanczos_tol", "schur_split", "device", "ngpus") if k in o}

    # -- plumbing ---------------------------------------------------------------------------------------------------
    def _err(self):
        msg = self.lib.lrn_last_error(self.h)
        return msg.decode() if msg else ""

    def _call(self, name, *args, allow_positive=False):
        rc = getattr(self.lib, name)(self.h, *args)
        if rc < 0:
            raise LoraineB200Error(f"{name} failed ({rc}): {self._err()}")
        if rc > 0 and not allow_positive:
            raise PosDefException(rc)
        return rc

    def close(self):
        if self.h:
            self.lib.lrn_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def get_array(self, name, iblk=0):
        md = self.model
        which = _lib.ARR[name]
        if which in (1, 2) and self.kit != 0:      # before allocating an n x n host array: kit = 1 has no Schur matrix
            raise LoraineB200Error(f"{name} (the Schur matrix or its factor) exists only for kit = 0")
        if which < 10:
            shape = (md.n, md.n) if which in (1, 2) else (md.n,)
        elif which in (14, 15):
            shape = (md.msizes[iblk],)
        else:
            shape = (md.msizes[iblk], md.msizes[iblk])
        out = np.zeros(shape, dtype=np.float64, order="F")
        self._call("lrn_get_array", which, iblk, _dp(out))
        return out

    def timers(self, reset=False):
        ms = np.zeros(len(_lib.T_NAMES))
        calls = np.zeros(len(_lib.T_NAMES), dtype=np.int64)
        self._call("lrn_timers", _dp(ms), _ip(calls), 1 if reset else 0)
        return {n: (float(ms[i]), int(calls[i])) for i, n in enumerate(_lib.T_NAMES)}

    def stats(self):
        out = np.zeros(3, dtype=np.int64)
        self._call("lrn_stats", _ip(out))
        return dict(svd_sweeps=int(out[0]), lanczos_iters=int(out[1]), lanczos_not_converged=int(out[2]))


def _csc_args(M):
    M = sp.csc_matrix(M)
    M.sort_indices()
    colptr = (M.indptr.astype(np.int64) + 1)
    rowval = (M.indices.astype(np.int64) + 1)
    nzval = np.ascontiguousarray(M.data, dtype=np.float64)
    return colptr, rowval, nzval


def load(model: MyModel, options: dict, T=float):
    """src/Solvers.jl:187-302 (+ upload of the prepared model to the device)."""
    if T not in (float, np.float64):
        raise TypeError("loraine_b200: Float64 is the only supported element type on the GPU "
                        "(Optimizer{Float64xN} is rejected instead of falling back)")
    o = dict(DEFAULT_OPTIONS)
    o.update(options)
    s = MySolver(model, o)
    verb = s.verb
    if verb > 0:
        print("\n *** Loraine.jl v0.2.5 hot path on loraine_b200 (sm_100a) ***")
        print(" *** Initialisation STARTS")
        print(f" Number of variables: {model.n:5d}")
        print(f" LMI constraints    : {model.nlmi:5d}")
        if model.nlmi > 0:
            print(" Matrix size(s)     :" + "".join(f"{m:6d}" for m in model.msizes[:20]) + (" ..." if model.nlmi > 20 else ""))
        print(f" Linear constraints : {model.nlin:5d}")
        print(f" Preconditioner     : {s.preconditioner:5d}" if s.kit > 0 else " Preconditioner     :  none, using direct solver")
    # parameter checks, src/Solvers.jl:263-291
    if s.kit < 0 or s.kit > 1:
        s.kit = 0
        print(f" ---Parameter kit out of range, setting kit = {s.kit}")
    if s.tol_cg < s.tol_cg_min and s.kit == 1:
        s.tol_cg = s.tol_cg_min
        print(f" ---Parameter tol_cg smaller than tol_cg_min, setting tol_cg = {s.tol_cg:7.1e}")
    if s.tol_cg_min > s.eDIMACS and s.kit == 1:
        s.tol_cg_min = s.eDIMACS
        print(f" ---Parameter tol_cg_min switched to eDIMACS = {s.eDIMACS:7.1e}")
    if s.kit == 1 and (s.preconditioner < 0 or s.preconditioner > 4):
        s.preconditioner = 1
        print(f" ---Parameter preconditioner out of range, setting preconditioner = {s.preconditioner}")
    if s.erank < 0:
        s.erank = 1
        print(f" ---Parameter erank negative, setting erank = {s.erank}")
    if s.datarank < -1:
        s.datarank = 0
        print(f" ---Parameter datarank out of range, setting datarank = {s.datarank}")
    if s.initpoint < 0 or s.initpoint > 1:
        s.initpoint = 1
        print(f" ---Parameter kit out of range, setting initpoint = {s.initpoint}")
    return s, Halpha(s.kit)


def setup_solver(s: MySolver, halpha: Halpha, before_finalize=None):
    """src/Solvers.jl:363-446: kit / datarank fall-backs, then device allocation (instead of the per-block `zeros`).
    before_finalize (optional) is called with the solver after lrn_set_b and before lrn_finalize, e.g.
    dist.attach_before_finalize, which attaches a torchrun rank to its communicator so that lrn_finalize can shard H and L."""
    md = s.model
    s.alpha = np.zeros(md.nlmi)
    s.beta = np.zeros(md.nlmi)
    s.alpha_lin = 1.0
    s.beta_lin = 1.0
    s.regcount = 0
    if s.kit == 1:
        if md.nlmi == 0:
            if s.verb > 0:
                print("WARNING: Switching to a direct solver, no LMIs")
            s.kit = 0
        elif s.erank >= max(md.msizes) - 1:
            if s.verb > 0:
                print("WARNING: Switching to a direct solver, erank bigger than matrix size")
            s.kit = 0
    if len(md.B) > 0:
        for i in range(md.nlmi):
            if md.B[i].nnz == 0:
                s.datarank = 0
    if s.datarank == -1 and len(md.B) != md.nlmi:
        s.datarank = 0
    # ---- device handle -------------------------------------------------------------------------------------------
    lib = s.lib
    opt = _lib.lrn_options_t()
    lib.lrn_default_options(C.byref(opt))
    opt.kit, opt.datarank, opt.preconditioner = s.kit, s.datarank, s.preconditioner
    opt.erank, opt.aamat, opt.datasparsity = s.erank, s.aamat, s.datasparsity
    opt.schur_split = int(s.extra.get("schur_split", 0))
    opt.svd_tol = float(s.extra.get("svd_tol", 0.0))
    opt.lanczos_tol = float(s.extra.get("lanczos_tol", 0.0))
    opt.device = int(s.extra.get("device", -1))
    ms = np.array(md.msizes, dtype=np.int64)
    if getattr(s, "sdpa_arrays", None) is not None:
        _setup_native(s, opt)
        return
    if s.h:                                    # a second setup_solver on the same object (solve() after a manual set-up)
        s.close()
    ngpus = int(s.extra.get("ngpus", 1))
    if ngpus != 1:                             # one host thread, N devices: the library owns the NCCL communicators
        rc = lib.lrn_create_multi(C.byref(s.h), md.n, md.nlmi, _ip(ms) if md.nlmi else None, md.nlin, C.byref(opt), ngpus, None)
    else:
        rc = lib.lrn_create(C.byref(s.h), md.n, md.nlmi, _ip(ms) if md.nlmi else None, md.nlin, C.byref(opt))
    if rc != 0:
        msg = s._err() if s.h else "no usable sm_100 CUDA device"
        raise LoraineB200Error(f"lrn_create failed ({rc}): {msg}; there is no CPU fallback")
    for i in range(md.nlmi):
        _set_csc(s, "lrn_set_block_AA", i, md.AA[i])
        _set_csc(s, "lrn_set_block_C", i, md.C[i])
        if s.datarank == -1:
            _set_csc(s, "lrn_set_block_B", i, md.B[i])
    if md.nlin > 0:
        cp, rv, nz = _csc_args(md.C_lin)
        d = np.ascontiguousarray(md.d_lin, dtype=np.float64)
        s._call("lrn_set_lin", _ip(cp), _ip(rv), _dp(nz), _dp(d))
    b = np.ascontiguousarray(md.b, dtype=np.float64)
    s._call("lrn_set_b", _dp(b))
    if before_finalize is not None:
        before_finalize(s)
    s._call("lrn_finalize")


def _setup_native(s, opt):
    """Model preparation inside the library (lrn_create_from_triplets: the bulk replacement of MOI.copy_to's triplet builder
    and of _prepare_A, src/MOI_wrapper.jl:152-209, src/model.jl:120-229): the SDPA triplets go down as they are."""
    n, bs, c, body = s.sdpa_arrays
    body = np.asarray(body, dtype=np.float64).reshape(-1, 5)
    tk, tb, ti, tj = (np.ascontiguousarray(body[:, k], dtype=np.int64) for k in range(4))
    tv = np.ascontiguousarray(body[:, 4], dtype=np.float64)
    bsa = np.array(bs, dtype=np.int64)
    cc = np.ascontiguousarray(c, dtype=np.float64)
    if s.h:
        s.close()
    rc = s.lib.lrn_create_from_triplets(C.byref(s.h), int(n), len(bs), _ip(bsa), tv.shape[0], _ip(tk), _ip(tb), _ip(ti), _ip(tj),
                                        _dp(tv), _dp(cc), C.byref(opt), int(s.extra.get("ngpus", 1)))
    if rc != 0:
        msg = s._err() if s.h else "model preparation failed (see stderr)"
        raise LoraineB200Error(f"lrn_create_from_triplets failed ({rc}): {msg}; there is no CPU fallback")
    s.native_model = True


def _set_csc(s, fname, i, M):
    cp, rv, nz = _csc_args(M)    # locals keep the numpy buffers alive for the duration of the call
    s._call(fname, i, _ip(cp), _ip(rv), _dp(nz))


def initial_point(s: MySolver):
    """src/initial_point.jl:1-81 (host: a few norms of the model data), then upload."""
    md = s.model
    if getattr(s, "native_model", False):
        # find_initial! on the device from the norms recorded by lrn_finalize (no host copy of the model needed)
        s._call("lrn_initial_point", int(s.initpoint))
        s.sigma, s.tau, s.expon, s.DIMACS_error, s.iter, s.status = 3.0, 0.95, 3.0, 1.0, 0, 0
        return
    n = md.b.shape[0]
    y = np.zeros(n)
    b2 = 1 + np.abs(md.b)
    f = 0.0
    Xs, Ss = [], []
    for i in range(md.nlmi):
        m = md.msizes[i]
        if s.initpoint == 0:
            Eps = 1.0
        else:
            f = np.linalg.norm(b2) / (1 + spla.norm(md.AA[i]))
            Eps = math.sqrt(m) * max(1.0, math.sqrt(m) * f)
        if s.initpoint == 0:
            Eta = float(md.n)
        else:
            mf = max(f, spla.norm(md.C[i]))
            mf = (1 + mf) / math.sqrt(m)
            Eta = math.sqrt(m) * max(1.0, mf)
        Xs.append(Eps)
        Ss.append(Eta)
    if md.nlin > 0:
        dd = md.d_lin.shape[0]
        rown = np.sqrt(np.asarray(md.C_lin.multiply(md.C_lin).sum(axis=1)).ravel())
        if s.initpoint == 0:
            Epss, Etaa = 1.0, 1.0
        else:
            Epss = max(1.0, float((b2 / (1 + rown)).max()))
            mf = max(float(rown.max()), float(np.linalg.norm(md.d_lin))) / math.sqrt(dd)
            Etaa = max(1.0, mf)
        x_lin = Epss * np.ones(dd)
        s_lin = Etaa * np.ones(dd)
    else:
        x_lin = s_lin = np.zeros(0)
    set_iterate(s, [e * np.eye(m) for e, m in zip(Xs, md.msizes)], [e * np.eye(m) for e, m in zip(Ss, md.msizes)], y,
                x_lin, s_lin)
    s.sigma = 3.0
    s.tau = 0.95
    s.expon = 3.0
    s.DIMACS_error = 1.0
    s.iter = 0
    s.status = 0


def set_iterate(s, X, S, y, x_lin, s_lin):
    md = s.model
    Xc = [np.asfortranarray(x, dtype=np.float64) for x in X]
    Sc = [np.asfortranarray(x, dtype=np.float64) for x in S]
    PD = C.POINTER(C.c_double)
    Xp = (PD * max(1, md.nlmi))(*[_dp(x) for x in Xc])
    Sp = (PD * max(1, md.nlmi))(*[_dp(x) for x in Sc])
    y = np.ascontiguousarray(y, dtype=np.float64)
    xl = np.ascontiguousarray(x_lin, dtype=np.float64)
    sl = np.ascontiguousarray(s_lin, dtype=np.float64)
    s._call("lrn_set_iterate", Xp, Sp, _dp(y), _dp(xl) if md.nlin else None, _dp(sl) if md.nlin else None)


def get_solution(s, out=None):
    """download y, X, x_lin (src/MOI_wrapper.jl:315-354 read them from the solver); `out` = (y, [X_i], x_lin) lets the caller
    provide (e.g. pinned) Fortran-ordered destination buffers"""
    md = s.model
    PD = C.POINTER(C.c_double)
    if out is not None:
        y, X, xl = out
    else:
        y = np.zeros(md.n)
        X = [np.zeros((m, m), order="F") for m in md.msizes]
        xl = np.zeros(md.nlin)
    Xp = (PD * max(1, md.nlmi))(*[_dp(x) for x in X])
    s._call("lrn_get_solution", _dp(y), Xp, _dp(xl) if md.nlin else None)
    s.y, s.X, s.X_lin = y, X, xl
    return y, X, xl


def find_mu(s):
    """src/Solvers.jl:480-494."""
    mu = C.c_double()
    s._call("lrn_find_mu", C.byref(mu))
    s.mu = mu.value
    return s.mu


def prepare_W(s):
    """src/prepare_W.jl:28-94."""
    st4 = C.c_int32(0)
    s._call("lrn_prepare_W", C.byref(st4))
    if st4.value:
        if s.verb > 0:
            print("WARNING: X or S cannot be made positive definite, giving up")
        s.status = 4


def predictor(s, halpha):
    """src/predictor_corrector.jl:5-146."""
    md = s.model
    s.predict = True
    s._call("lrn_residuals")                                   # :8-22
    if s.kit == 0:
        s._call("lrn_schur_assemble")                          # :24-40
    s._call("lrn_rhs_predictor")                               # :43-50
    if s.kit == 0:                                             # :53-97
        try:
            s._call("lrn_schur_factor")
            s.cholBBBB = _DeviceFactor(s, False)
        except PosDefException:
            if s.verb > 0:
                print("Matrix H not positive definite, trying to regularize")
            icount = 0
            s.regcount += 1
            if s.regcount > 5:
                if s.verb > 0:
                    print("WARNING: too many regularizations of H, giving up")
                s.status = 3
                return
            while True:                                        # while isposdef(BBBB) == false
                s._call("lrn_schur_shift", 1e-4)
                icount += 1
                if s._call("lrn_schur_factor", allow_positive=True) == 0:
                    break
                if icount > 1000:
                    if s.verb > 0:
                        print("WARNING: H cannot be made positive definite, giving up")
                    s.status = 3
                    return
            s.cholBBBB = _DeviceFactor(s, True)
        s.cholBBBB.solve_reference_expression()                # :89-90
    else:                                                      # :118-140
        if s.preconditioner == 0:
            kind = 0
        elif s.preconditioner == 1:
            s._call("lrn_prec_prepare", 1)
            kind = 1
        elif s.preconditioner in (2, 4):
            s._call("lrn_prec_prepare", 2)
            kind = 2
        else:
            raise ValueError("preconditioner 3 is undefined in the reference (src/predictor_corrector.jl:120-128)")
        halpha.prepared_kind = kind
        num_iters = _cg(s, kind)
        s.cg_iter_pre += num_iters
        s.cg_iter_tot += num_iters
    find_step(s)


def _cg(s, kind):
    it = C.c_int64(0)
    code = C.c_int32(0)
    s._call("lrn_pcg", float(s.tol_cg), 10000, kind, C.byref(it), C.byref(code))
    s.cg_exit_code = code.value
    return it.value


def sigma_update(s):
    """src/predictor_corrector.jl:148-179."""
    md = s.model
    step_pred = min(min(list(s.alpha) + [s.alpha_lin]), min(list(s.beta) + [s.beta_lin]))
    if s.mu > 1e-6:
        expon_used = 1.0 if step_pred < 1 / math.sqrt(3) else max(s.expon, 3.0 * step_pred ** 2)
    else:
        expon_used = max(1.0, min(s.expon, 3.0 * step_pred ** 2))
    tr = C.c_double()
    dl = C.c_double()
    s._call("lrn_sigma_trace", C.byref(tr), C.byref(dl))
    if tr.value < 0:
        s.sigma = 0.8
    else:
        tmp1 = tr.value if md.nlmi > 0 else 0.0
        tmp2 = dl.value if md.nlin > 0 else 0.0
        tmp12 = (tmp1 + tmp2) / (sum(md.msizes) + md.nlin)
        s.sigma = min(1.0, (tmp12 / s.mu) ** expon_used)
    return s.sigma


def corrector(s, halpha):
    """src/predictor_corrector.jl:181-246."""
    s.predict = False
    s._call("lrn_rhs_corrector", float(s.sigma), float(s.mu))  # :183-192
    if s.kit == 0:
        s.cholBBBB.solve_reference_expression()                # :199
    else:
        kind = 0 if s.preconditioner == 0 else (1 if s.preconditioner == 1 else 2)
        num_iters = _cg(s, kind)
        s.cg_iter_cor += num_iters
        s.cg_iter_tot += num_iters
    find_step(s)


def find_step(s):
    """src/predictor_corrector.jl:248-364 (find_step + find_step_lin)."""
    md = s.model
    al = C.c_double(1.0)
    bl = C.c_double(1.0)
    alpha = np.zeros(max(1, md.nlmi))
    beta = np.zeros(max(1, md.nlmi))
    s._call("lrn_find_step", 1 if s.predict else 0, float(s.sigma), float(s.mu), float(s.tau), _dp(alpha), _dp(beta),
            C.byref(al), C.byref(bl))
    s.alpha, s.beta = alpha[:md.nlmi].copy(), beta[:md.nlmi].copy()
    s.alpha_lin, s.beta_lin = al.value, bl.value


def check_convergence(s):
    """src/Solvers.jl:496-568."""
    md = s.model
    err = np.zeros(6)
    by, trCX, dx = C.c_double(), C.c_double(), C.c_double()
    s._call("lrn_dimacs", _dp(err), C.byref(by), C.byref(trCX), C.byref(dx))
    s.err1, s.err2, s.err3, s.err4, s.err5, s.err6 = (float(e) for e in err)
    if md.nlmi > 0:
        D = s.err1 + s.err2 + s.err3 + s.err4 + abs(s.err5) + s.err6
    else:
        D = s.err2 + s.err3 + s.err4 + abs(s.err5) + s.err6
    s.DIMACS_error = D
    s.primal_obj = -by.value + md.b_const
    s.dual_obj = -trCX.value - dx.value
    if s.verb > 0 and s.status == 0:
        if s.verb > 1:
            tail = f"{s.cg_iter_pre:7d} {s.cg_iter_cor:7d} " if s.kit == 1 else ""
            print(f"{s.iter:3d} {s.primal_obj:16.8e} {D:9.2e} {s.err1:9.2e} {s.err2:9.2e} {s.err3:9.2e} {s.err4:9.2e} "
                  f"{s.err5:9.2e} {s.err6:9.2e} {tail}{s.itertime:8.2f}")
        elif s.kit == 0:
            print(f"{s.iter:3d} {s.primal_obj:16.8e} {D:9.2e} {s.itertime:8.2f}")
        else:
            print(f"{s.iter:3d} {s.primal_obj:16.8e} {D:9.2e} {s.cg_iter_pre + s.cg_iter_cor:9d} {s.itertime:8.2f}")
    if D < s.eDIMACS:
        s.status = 1
        if s.verb > 0:
            print("Primal objective: ", s.primal_obj)
            print("Dual objective:   ", s.dual_obj)
    if D > 1e55:
        s.status = 2
        if s.verb > 0:
            print("WARNING: Problem probably infeasible (stopping status = 2)")
    elif abs(by.value) > 1e55:
        s.status = 3
        if s.verb > 0:
            print("WARNING: Problem probably unbounded or infeasible (stopping status = 3)")
    return D


def myIPstep(s, halpha):
    """src/Solvers.jl:448-478."""
    s.iter += 1
    if s.iter > s.maxit:
        s.status = 4
        if s.verb > 0:
            print("WARNING: Stopped by iteration limit (stopping status = 4)")
    s.cg_iter_pre = 0
    s.cg_iter_cor = 0
    find_mu(s)
    prepare_W(s)
    predictor(s, halpha)
    if s.status == 3:
        # H could not be made positive definite (src/predictor_corrector.jl:66-70, :76-83): the reference carries on with
        # cholBBBB = I for the rest of this iteration and leaves the loop at src/Solvers.jl:336; there is no factor on the
        # device, so the iteration ends here with the same status (INFEASIBLE_OR_UNBOUNDED)
        return
    sigma_update(s)
    corrector(s, halpha)


def solve(s: MySolver, halpha: Halpha, max_iters=None, setup=True):
    """src/Solvers.jl:304-361.  setup=False keeps the device handle of an earlier setup_solver (e.g. one that was attached to
    an NCCL communicator with dist.init_distributed) and only restarts from the initial point."""
    t1 = time.perf_counter()
    if s.verb > 0:
        print(" *** IP STARTS")
        print(" it        obj         error     CPU/it" if s.kit == 0 else " it        obj         error     cg_iter   CPU/it")
    if setup or not s.h:
        setup_solver(s, halpha)
    initial_point(s)
    while s.status == 0:
        t2 = time.perf_counter()
        myIPstep(s, halpha)
        s.itertime = time.perf_counter() - t2
        s.tol_cg = max(s.tol_cg * s.tol_cg_up, s.tol_cg_min)
        if s.status == 3:
            break
        check_convergence(s)
        s.trace.append(dict(iter=s.iter, obj=s.primal_obj, dual_obj=s.dual_obj, dimacs=s.DIMACS_error, mu=s.mu,
                            sigma=s.sigma, alpha=min(list(s.alpha) + [s.alpha_lin]), beta=min(list(s.beta) + [s.beta_lin]),
                            err=[s.err1, s.err2, s.err3, s.err4, s.err5, s.err6], cg_pre=s.cg_iter_pre, cg_cor=s.cg_iter_cor,
                            itertime=s.itertime))
        if s.preconditioner == 4:
            if (s.cg_iter_cor / 2 > s.erank * s.model.nlmi * math.sqrt(s.model.n) / 20 and s.iter > math.sqrt(s.model.n) / 60) \
                    or s.cg_iter_cor > 100:
                s.preconditioner = 1
                s.aamat = 2
                if s.verb > 0:
                    print("Switching to preconditioner 1")
                s._call("lrn_set_option", b"aamat", 2.0)
        if max_iters is not None and s.iter >= max_iters:
            break
    s.tottime = time.perf_counter() - t1
    get_solution(s)
    if s.verb > 0:
        if s.kit == 1:
            print(f" *** Total CG iterations: {s.cg_iter_tot:8d} ")
        if s.status == 1:
            print(f" *** Optimal solution found in {s.tottime:8.2f} seconds")
    return s


class Optimizer:
    """Minimal stand-in for `Loraine.Optimizer{T}` (src/MOI_wrapper.jl:42-66, :86-103, :136-140, :241-354) so that tests and
    the benchmark read like the reference's examples.  T = Float64, or "Float64x2" for models without PSD blocks (the
    double-double LP path of dd_lp.py, examples/k.jl:8); every other element type is rejected -- there is no fallback."""

    def __init__(self, T=float):
        self.dd = T == "Float64x2"
        if not self.dd and T not in (float, np.float64):
            raise TypeError("Optimizer{T}: only T = Float64 (and Float64x2 for models without PSD blocks) is supported by "
                            "the B200 path (no Float64xN fallback)")
        self.options = dict(DEFAULT_OPTIONS)
        self.solver = None
        self.halpha = None
        self.max_sense = False
        self.silent = False

    def set_attribute(self, name, value):
        if name not in DEFAULT_OPTIONS and name not in ("svd_tol", "lanczos_tol", "schur_split", "device", "ngpus"):
            raise KeyError(f"UnsupportedAttribute: {name}")
        self.options[name] = value

    def get_attribute(self, name):
        return self.options[name]

    def copy_to(self, raw: RawProblem, max_sense=False):
        self.max_sense = max_sense
        model = prepare_model(raw, datarank=int(self.options["datarank"]), kappa=int(self.options["datasparsity"]))
        opts = dict(self.options)
        if self.silent:
            opts["verb"] = 0
        if self.dd:
            from . import dd_lp
            self.solver, self.halpha = dd_lp.DDSolver(model, opts), None       # raises TypeError when the model has PSD blocks
            return
        self.solver, self.halpha = load(model, opts)

    def load_sdpa(self, n, bs, c, body, max_sense=False):
        """SDPA arrays (what read_sdpa returns) with the model preparation done INSIDE the library (lrn_create_from_triplets
        and lrn_initial_point); the host keeps a MyModel only for the objective getters."""
        self.copy_to(raw_from_sdpa_arrays(n, bs, c, body), max_sense=max_sense)
        self.solver.sdpa_arrays = (int(n), [int(b) for b in bs], np.asarray(c, float), np.asarray(body, float))

    def optimize(self, max_iters=None):
        if self.dd:
            from . import dd_lp
            dd_lp.solve(self.solver, max_iters=max_iters)
            return
        solve(self.solver, self.halpha, max_iters=max_iters)

    def objective_value(self):
        s = self.solver
        val = float(s.model.b @ s.y) - s.model.b_const
        return val if self.max_sense else -val

    def objective_value_dd(self):
        """Float64x2 solves: the objective as an exact fraction of the (hi, lo) result (b'y - b_const, sense applied)."""
        from . import dd_lp
        s = self.solver
        val = dd_lp.frac(s.by) - dd_lp.Fraction(s.model.b_const)
        return val if self.max_sense else -val

    def dual_objective_value(self):
        s = self.solver
        val = sum(float(s.model.C[i].multiply(s.X[i]).sum()) for i in range(s.model.nlmi))
        if s.model.nlin:
            val += float(s.model.d_lin @ s.X_lin)
        val -= s.model.b_const
        return val if self.max_sense else -val

    def termination_status(self):
        st = 0 if self.solver is None else self.solver.status
        return {0: "OPTIMIZE_NOT_CALLED", 1: "OPTIMAL", 2: "INFEASIBLE", 3: "INFEASIBLE_OR_UNBOUNDED", 4: "ITERATION_LIMIT"}[st]

    def solve_time_sec(self):
        return self.solver.tottime
