"""Dense Cholesky of SPD matrices with the trailing updates on DMMA (FP64 tensor cores) and as Ozaki INT8 products, alternated
in one process: time per factorisation (CUDA events), FP64-equivalent rate n^3/3 / time, the INT8 update kernel's own rate
against the data-sheet INT8 figure, and the backward error max |H - L L^T|_ij / sqrt(h_ii h_jj).

    python scripts/bench_chol_i8.py [--sizes 16384 20000 40000] [--reps 3] [--out profiles/chol_i8_b200.jsonl]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as g  # noqa: E402

INT8_DATASHEET_TOPS = 4500.0     # dense INT8, one B200 of an HGX B200 (1000 W)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[16384, 20000, 40000])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "chol_i8_b200.jsonl"))
    a = ap.parse_args()
    import torch
    g.load_package()
    from loraine_jl_b200 import _lib
    L = _lib.lib()
    pd, pi = C.POINTER(C.c_double), C.POINTER(C.c_int32)
    L.lrn_dbg_cholesky.argtypes = [C.c_int32, pd, pd, C.c_int32, pi, C.c_int32, pd]
    L.lrn_dbg_gemm_profile.argtypes = [C.c_int32, pd, pd, C.POINTER(C.c_int64)]
    name = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "a") as fo:
        for n in a.sizes:
            gen = torch.Generator(device="cuda").manual_seed(n)
            G = torch.randn(n, n, generator=gen, device="cuda", dtype=torch.float64) / n ** 0.5
            Ad = G @ G.T
            Ad.diagonal().add_(1.0)
            del G
            A = np.asfortranarray(Ad.cpu().numpy())
            d = torch.sqrt(torch.diagonal(Ad))
            rec = dict(n=n, card=name, reps=a.reps, ms={"dmma": [], "int8": []})
            for r in range(a.reps):
                for label, mode in (("dmma", 0), ("int8", 2)):
                    L.lrn_dbg_chol_int8(mode)
                    out = A.copy(order="F")
                    info, ms = C.c_int32(-1), C.c_double()
                    prof = r == 0 and mode == 2
                    if prof:
                        L.lrn_dbg_gemm_profile(1, None, None, None)
                    assert L.lrn_dbg_cholesky(n, out.ctypes.data_as(pd), None, 0, C.byref(info), 1, C.byref(ms)) == 0
                    if prof:
                        L.lrn_dbg_gemm_profile(0, None, None, None)
                        km, kf, kn = C.c_double(), C.c_double(), C.c_int64()
                        L.lrn_dbg_gemm_profile(13, C.byref(km), C.byref(kf), C.byref(kn))
                        # the profiled run is the untimed first factorisation plus the timed one: halve the totals
                        rec["int8_kernel"] = dict(ms=km.value / 2, launches=kn.value // 2,
                                                  fp64_equiv_tflops=kf.value / (km.value * 1e-3) / 1e12 if km.value else None,
                                                  int8_tops=36 * kf.value / (km.value * 1e-3) / 1e12 if km.value else None,
                                                  frac_of_datasheet=36 * kf.value / (km.value * 1e-3) / 1e12 / INT8_DATASHEET_TOPS
                                                  if km.value else None,
                                                  note="concurrent launches on the panel and main streams overlap")
                    assert info.value == 0, (label, info.value)
                    rec["ms"][label].append(ms.value)
                    if r == 0:
                        Lt = torch.from_numpy(out).to("cuda")
                        R = torch.tril(Ad - Lt @ Lt.T).abs_()
                        R /= d[:, None]
                        R /= d[None, :]
                        rec["backward_error_" + label] = float(R.max())
                        del Lt, R
                        torch.cuda.empty_cache()
            L.lrn_dbg_chol_int8(0)
            for label in ("dmma", "int8"):
                best = min(rec["ms"][label])
                rec[label + "_fp64_equiv_tflops"] = n ** 3 / 3 / (best * 1e-3) / 1e12
            rec["speedup_min_over_runs"] = min(rec["ms"]["dmma"]) / max(rec["ms"]["int8"])
            print(json.dumps(rec), flush=True)
            fo.write(json.dumps(rec) + "\n")
            del Ad, A
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
