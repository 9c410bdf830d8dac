"""ctypes binding of include/loraine_b200.h.  Fails loudly when the CUDA library is missing."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libloraine_b200.so")

T_NAMES = ["prepare_W", "residuals", "schur_assemble", "rhs", "schur_factor", "schur_solve", "find_step", "prec_prepare",
           "cg", "dimacs", "svd", "eigmin"]

ARR = dict(H=1, L=2, RHS=3, DELY=4, RP=5, W=10, G=11, GI=12, SI=13, D=14, DDSI=15, RD=16, DELX=17, DELS=18, RNT=19,
           XN=20, SN=21)


class lrn_options_t(C.Structure):
    _fields_ = [("kit", C.c_int32), ("datarank", C.c_int32), ("preconditioner", C.c_int32), ("erank", C.c_int32),
                ("aamat", C.c_int32), ("datasparsity", C.c_int32), ("schur_split", C.c_int32), ("rank1_mode", C.c_int32),
                ("svd_tol", C.c_double), ("lanczos_tol", C.c_double), ("device", C.c_int32), ("reserved", C.c_int32)]


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} not found: build it with loraine.jl_b200/csrc/build.sh "
                          "(python -c 'import __graft_entry__ as g; g.build()'). There is no CPU fallback.")
    L = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    i32, i64, dbl, vp = C.c_int32, C.c_int64, C.c_double, C.c_void_p
    pi64, pdbl, pi32 = C.POINTER(C.c_int64), C.POINTER(C.c_double), C.POINTER(C.c_int32)
    ppd = C.POINTER(C.POINTER(C.c_double))
    sig = {
        "lrn_default_options": (None, [C.POINTER(lrn_options_t)]),
        "lrn_create": (i32, [C.POINTER(vp), i64, i64, pi64, i64, C.POINTER(lrn_options_t)]),
        "lrn_set_block_AA": (i32, [vp, i64, pi64, pi64, pdbl]),
        "lrn_set_block_C": (i32, [vp, i64, pi64, pi64, pdbl]),
        "lrn_set_block_B": (i32, [vp, i64, pi64, pi64, pdbl]),
        "lrn_set_lin": (i32, [vp, pi64, pi64, pdbl, pdbl]),
        "lrn_set_b": (i32, [vp, pdbl]),
        "lrn_finalize": (i32, [vp]),
        "lrn_destroy": (i32, [vp]),
        "lrn_get_dims": (i32, [vp, pi64, pi64, pi64, pi64]),
        "lrn_last_error": (C.c_char_p, [vp]),
        "lrn_set_iterate": (i32, [vp, ppd, ppd, pdbl, pdbl, pdbl]),
        "lrn_get_solution": (i32, [vp, pdbl, ppd, pdbl]),
        "lrn_get_slack": (i32, [vp, ppd, pdbl]),
        "lrn_find_mu": (i32, [vp, pdbl]),
        "lrn_prepare_W": (i32, [vp, pi32]),
        "lrn_residuals": (i32, [vp]),
        "lrn_schur_assemble": (i32, [vp]),
        "lrn_rhs_predictor": (i32, [vp]),
        "lrn_rhs_corrector": (i32, [vp, dbl, dbl]),
        "lrn_schur_factor": (i32, [vp]),
        "lrn_schur_shift": (i32, [vp, dbl]),
        "lrn_schur_solve": (i32, [vp, i32]),
        "lrn_prec_prepare": (i32, [vp, i32]),
        "lrn_pcg": (i32, [vp, dbl, i64, i32, pi64, pi32]),
        "lrn_find_step": (i32, [vp, i32, dbl, dbl, dbl, pdbl, pdbl, pdbl, pdbl]),
        "lrn_sigma_trace": (i32, [vp, pdbl, pdbl]),
        "lrn_dimacs": (i32, [vp, pdbl, pdbl, pdbl, pdbl]),
        "lrn_get_array": (i32, [vp, i32, i64, pdbl]),
        "lrn_apply_operator": (i32, [vp, i32, pdbl, pdbl]),
        "lrn_timers": (i32, [vp, pdbl, pi64, i32]),
        "lrn_kernel_launches": (i64, []),
        "lrn_timer_name": (C.c_char_p, [i32, i32]),
        "lrn_stats": (i32, [vp, pi64]),
        "lrn_set_option": (i32, [vp, C.c_char_p, dbl]),
        "lrn_create_from_triplets": (i32, [C.POINTER(vp), i64, i64, pi64, i64, pi64, pi64, pi64, pi64, pdbl, pdbl,
                                           C.POINTER(lrn_options_t), i32]),
        "lrn_load_sdpa": (i32, [C.POINTER(vp), C.c_char_p, C.POINTER(lrn_options_t), i32]),
        "lrn_initial_point": (i32, [vp, i32]),
        "lrn_create_multi": (i32, [C.POINTER(vp), i64, i64, pi64, i64, C.POINTER(lrn_options_t), i32, pi32]),
        "lrn_dbg_set_shard": (i32, [vp, i32, i32, i32]),
        "lrn_dbg_prec_slab": (i32, [vp, i64, pi64]),
        "lrn_dbg_model_block": (i64, [i64, i64, pi64, i64, pi64, pi64, pi64, pi64, pdbl, pdbl, i32, i64, i32, i64, pi64, pi64, pdbl,
                                      pdbl]),
        "lrn_dbg_compare": (i32, [vp, vp, i32, pdbl]),
        "lrn_dbg_chol_int8": (i32, [i32]),
        "lrn_dbg_syrk_i8": (i32, [i32, i32, pdbl, i32, i32, i32, i32, i64, i64, i32, pdbl, pdbl, i32, pdbl]),
        "lrn_dbg_gather_H": (i32, [vp]),
        "lrn_dist_unique_id": (i32, [C.c_char_p]),
        "lrn_dist_init": (i32, [vp, i32, i32, C.c_char_p]),
        # include/loraine_b200_dd.h (double-double LP path)
        "lrn_dd_create": (i32, [C.POINTER(vp), i64, i64, i32]),
        "lrn_dd_create_multi": (i32, [C.POINTER(vp), i64, i64, i32, pi32]),
        "lrn_dd_dist_init": (i32, [vp, i32, i32, C.c_char_p]),
        "lrn_dd_dbg_set_shard": (i32, [vp, i32, i32, i32]),
        "lrn_dd_set_lin": (i32, [vp, pi64, pi64, pdbl, pdbl, pdbl, pdbl]),
        "lrn_dd_set_b": (i32, [vp, pdbl, pdbl]),
        "lrn_dd_finalize": (i32, [vp]),
        "lrn_dd_destroy": (i32, [vp]),
        "lrn_dd_last_error": (C.c_char_p, [vp]),
        "lrn_dd_set_iterate": (i32, [vp, pdbl, pdbl, pdbl, pdbl, pdbl, pdbl]),
        "lrn_dd_get_solution": (i32, [vp, pdbl, pdbl, pdbl, pdbl, pdbl, pdbl]),
        "lrn_dd_find_mu": (i32, [vp, pdbl]),
        "lrn_dd_prepare_W": (i32, [vp]),
        "lrn_dd_residuals": (i32, [vp]),
        "lrn_dd_schur_assemble": (i32, [vp]),
        "lrn_dd_rhs_predictor": (i32, [vp]),
        "lrn_dd_rhs_corrector": (i32, [vp, pdbl, pdbl]),
        "lrn_dd_schur_factor": (i32, [vp]),
        "lrn_dd_schur_shift": (i32, [vp, dbl]),
        "lrn_dd_schur_solve": (i32, [vp, i32]),
        "lrn_dd_find_step": (i32, [vp, i32, pdbl, pdbl, dbl, pdbl, pdbl]),
        "lrn_dd_sigma_trace": (i32, [vp, pdbl]),
        "lrn_dd_dimacs": (i32, [vp, pdbl, pdbl, pdbl]),
        "lrn_dd_get_array": (i32, [vp, i32, pdbl, pdbl]),
        "lrn_dd_timers": (i32, [vp, pdbl, i32]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


DECLARED_SYMBOLS = ["lrn_default_options", "lrn_create", "lrn_set_block_AA", "lrn_set_block_C", "lrn_set_block_B",
                    "lrn_set_lin", "lrn_set_b", "lrn_finalize", "lrn_destroy", "lrn_last_error", "lrn_set_iterate",
                    "lrn_get_solution", "lrn_get_slack", "lrn_find_mu", "lrn_prepare_W", "lrn_residuals",
                    "lrn_schur_assemble", "lrn_rhs_predictor", "lrn_rhs_corrector", "lrn_schur_factor", "lrn_schur_shift",
                    "lrn_schur_solve", "lrn_prec_prepare", "lrn_pcg", "lrn_find_step", "lrn_sigma_trace", "lrn_dimacs",
                    "lrn_get_array", "lrn_apply_operator", "lrn_timers", "lrn_kernel_launches", "lrn_stats", "lrn_set_option",
                    "lrn_dist_unique_id", "lrn_dist_init", "lrn_create_multi",
                    "lrn_create_from_triplets", "lrn_load_sdpa", "lrn_initial_point", "lrn_get_dims", "lrn_timer_name"]

DD_SYMBOLS = ["lrn_dd_create", "lrn_dd_set_lin", "lrn_dd_set_b", "lrn_dd_finalize", "lrn_dd_destroy", "lrn_dd_last_error",
              "lrn_dd_set_iterate", "lrn_dd_get_solution", "lrn_dd_find_mu", "lrn_dd_prepare_W", "lrn_dd_residuals",
              "lrn_dd_schur_assemble", "lrn_dd_rhs_predictor", "lrn_dd_rhs_corrector", "lrn_dd_schur_factor", "lrn_dd_schur_shift",
              "lrn_dd_schur_solve", "lrn_dd_find_step", "lrn_dd_sigma_trace", "lrn_dd_dimacs", "lrn_dd_get_array", "lrn_dd_timers",
              "lrn_dd_create_multi", "lrn_dd_dist_init"]
DD_ARR = dict(H=1, L=2, RP=3, RD=4, RHS=5, DELY=6, DELX=7, DELS=8, XN=9, SN=10, RNT=11, SI=12)

DEBUG_SYMBOLS = ["lrn_dbg_gemm", "lrn_dbg_cholesky", "lrn_dbg_eig_small", "lrn_dbg_svd", "lrn_dbg_lanczos",
                 "lrn_dbg_batched_lambda_min", "lrn_dbg_peak", "lrn_dbg_gemm_profile", "lrn_dbg_set_shard", "lrn_dbg_compare",
                 "lrn_dbg_gather_H", "lrn_dbg_model_block", "lrn_dd_dbg_set_shard", "lrn_dbg_prec_slab",
                 "lrn_dbg_chol_int8", "lrn_dbg_syrk_i8"]
