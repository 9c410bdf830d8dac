"""kit = 1 (CG) on nuclear-norm matrix completion beyond the direct path's n_var limit (tests/mc_instances.py).

Per instance, one JSON line with
  - the H_alpha build (lrn_prec_prepare(h, 1)): slab height, wall time of the first build (includes the buffer allocation)
    and of a repeat, and its rate as 2 n_var kS^2 flop (the S = T'T product) over the repeat's time;
  - the device-memory drop across lrn_finalize and the first lrn_prec_prepare (cudaMemGetInfo through torch);
  - an H_alpha solve capped at --alpha-iters IP iterations and an H_beta (preconditioner 2) solve to eDIMACS = 1e-6:
    IP and CG iteration counts, seconds per IP iteration, status, and the objective error against -||M||_*;
  - the GPU name and power limit read in the same run.

    python scripts/bench_cg_large.py --out results.jsonl [--only mc600]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

INSTANCES = {
    "mc200": dict(shape=(200, 200, 2, 20000, 21), erank=2),
    "mc600": dict(shape=(600, 600, 2, 162000, 22), erank=2),
    "mc2000": dict(shape=(2000, 2000, 1, 1_200_000, 23), erank=1),
}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True)
    name, power, clock = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return dict(gpu=name, power_limit=power, max_sm_clock=clock)


def optimizer(pkg, inst, **opts):
    opt = pkg.Optimizer()
    for k, v in dict(kit=1, aamat=2, initpoint=1, verb=0, eDIMACS=1e-6, **opts).items():
        opt.set_attribute(k, v)
    opt.load_sdpa(*inst.arrays)
    return opt


def solve_stats(s, inst, t0, error=None):
    it = max(s.iter, 1)
    r = dict(ip_iters=s.iter, cg_iters=s.cg_iter_tot, s_per_ip_iter=(time.perf_counter() - t0) / it, status=s.status)
    if error is None and s.status == 1:
        r["obj_rel_err"] = abs(s.primal_obj - inst.optimum) / abs(inst.optimum)
    if error is not None:
        r["error"] = error
    return r


def run(pkg, name, spec, alpha_iters):
    import ctypes as C
    import torch
    import mc_instances as mc
    from loraine_jl_b200 import solver as S
    r, c, k, n_obs, seed = spec["shape"]
    inst = mc.matrix_completion(r, c, k, n_obs, seed=seed)
    erank = spec["erank"]
    kS = erank * (r + c)
    out = dict(instance=name, rows=r, cols=c, rank=k, n_var=n_obs, m=r + c, erank=erank, kS=kS)
    # H_alpha build: memory across lrn_finalize + first lrn_prec_prepare, first and repeated build time
    opt = optimizer(pkg, inst, preconditioner=1, erank=erank)
    s = opt.solver
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info(0)[0]
    S.setup_solver(s, opt.halpha)
    S.initial_point(s)
    S.find_mu(s)
    S.prepare_W(s)
    s._call("lrn_residuals")
    s._call("lrn_rhs_predictor")
    t = time.perf_counter()
    s._call("lrn_prec_prepare", 1)
    out["prec_first_ms"] = (time.perf_counter() - t) * 1e3
    torch.cuda.synchronize()
    out["mem_drop_bytes"] = free0 - torch.cuda.mem_get_info(0)[0]
    t = time.perf_counter()
    s._call("lrn_prec_prepare", 1)
    ms = (time.perf_counter() - t) * 1e3
    used = C.c_int64(0)
    s.lib.lrn_dbg_prec_slab(s.h, 0, C.byref(used))
    out.update(slab_rows=used.value, prec_ms=ms, prec_tflops=2.0 * n_obs * kS * kS / (ms * 1e-3) / 1e12)
    # H_alpha solve, capped
    t0 = time.perf_counter()
    err = None
    try:
        S.solve(s, opt.halpha, max_iters=alpha_iters, setup=False)
    except Exception as e:  # the reference's failure modes (PosDefException of chol(S)) are reported, not hidden
        err = f"{type(e).__name__}: {e}"
    out["h_alpha"] = solve_stats(s, inst, t0, err)
    s.close()
    # H_beta solve to the optimum
    opt = optimizer(pkg, inst, preconditioner=2)
    s = opt.solver
    t0 = time.perf_counter()
    S.setup_solver(s, opt.halpha)
    S.solve(s, opt.halpha, setup=False)
    out["h_beta"] = solve_stats(s, inst, t0)
    s.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", nargs="*", default=list(INSTANCES))
    ap.add_argument("--alpha-iters", type=int, default=8)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_cg_large.py measures on the GPU; no CUDA device is visible")
    import __graft_entry__ as g
    pkg = g.load_package()
    torch.cuda.init()
    info = gpu_info()
    for name in a.only:
        line = json.dumps(dict(run(pkg, name, INSTANCES[name], a.alpha_iters), **info))
        print(line, flush=True)
        if a.out:
            with open(a.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
