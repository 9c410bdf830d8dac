"""The own-rows layout of the kit = 0 Schur matrix on several GPUs (lrn_create_multi): seconds per IP iteration, the
factorisation, the forward and the backward triangular solve (fan-out / fan-in, one collective of at most pw doubles per
step), and the device bytes of every rank against the footprint lrn_finalize computed.

    python scripts/bench_rows_local.py [--iters 3] [--out profiles/rows_local_b200.jsonl]

Lines: n_var = 120 000 matrix completion on 2 / 4 / 8 GPUs (own rows: the replicated layout does not fit), and configs[4]
(C5, n_var = 40 000) on 2 GPUs in both layouts.  A configuration needing more GPUs than the machine has is written as
"not measured".  Every line carries the GPU name and power limit (nvidia-smi).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import __graft_entry__ as g  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else None


def run(pkg, arrays, opts, ngpus, layout, iters):
    import torch
    from loraine_jl_b200 import solver as S
    devs = list(range(ngpus))
    free0 = [torch.cuda.mem_get_info(d)[0] for d in devs]
    opt = pkg.Optimizer()
    for k, v in dict(opts, ngpus=ngpus, verb=0).items():
        opt.set_attribute(k, v)
    opt.copy_to(pkg.raw_from_sdpa_arrays(*arrays))
    s = opt.solver

    def force(h):
        if layout is not None:
            assert h.lib.lrn_dbg_schur_layout(h.h, layout, None) == 0
    S.setup_solver(s, opt.halpha, before_finalize=force)
    lay = C.c_int32(-9)
    s.lib.lrn_dbg_schur_layout(s.h, -2, C.byref(lay))
    S.initial_point(s)
    S.myIPstep(s, opt.halpha)                       # warm-up: first-use allocations of the factorisation and the solves
    s.itertime = 0.0
    S.check_convergence(s)
    s.timers(reset=True)
    t0 = time.perf_counter()
    for _ in range(iters):
        S.myIPstep(s, opt.halpha)
        s.itertime = 0.0
        S.check_convergence(s)
    t_it = (time.perf_counter() - t0) / iters
    ms, calls = s.timers()["schur_factor"]
    fac = ms / max(1, calls)
    solve = {}
    for which, key in ((1, "forward_ms"), (2, "backward_ms")):
        best = None
        for _ in range(3):
            t = time.perf_counter()
            s._call("lrn_schur_solve", which)
            s.get_array("DELY")                     # synchronises
            best = min(best or 1e30, (time.perf_counter() - t) * 1e3)
        solve[key] = best
    fp = C.c_int64()
    s.lib.lrn_dbg_schur_footprint(s.h, 1 if lay.value == 1 else 0, C.byref(fp))
    used = [free0[d] - torch.cuda.mem_get_info(d)[0] for d in devs]
    s.close()
    return dict(layout="own_rows" if lay.value == 1 else "replicated", s_per_iter=t_it, factor_ms=fac, **solve,
                device_bytes_per_rank=used, footprint_bytes_rank0=fp.value)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "rows_local_b200.jsonl"))
    a = ap.parse_args()
    import torch
    pkg = g.load_package()
    import mc_instances as mc
    ndev = torch.cuda.device_count()
    gpu = card()
    lines = []
    runs = [("mc120k", k, None) for k in (2, 4, 8)] + [("C5", 2, 0), ("C5", 2, 1)]
    for name, k, layout in runs:
        rec = dict(config=name, ngpus=k, forced_layout=layout, gpu=gpu)
        if name == "mc120k":
            rec["n_var"] = 120000
        else:
            rec["n_var"] = 40000
        if ndev < k:
            rec["result"] = "not measured"
            rec["reason"] = f"{ndev} GPU(s) on the machine"
        else:
            if name == "mc120k":
                inst = mc.matrix_completion(500, 500, 3, 120000, seed=5)
                arrays, opts = inst.arrays, dict(kit=0, datarank=0, eDIMACS=1e-6)
            else:
                cfg = pkg.problems.CONFIGS["C5"]
                arrays, opts = cfg["gen"](), dict(cfg["options"])
            rec.update(run(pkg, arrays, opts, k, layout, a.iters))
        lines.append(rec)
        print(json.dumps(rec), flush=True)
    with open(a.out, "w") as f:
        for r in lines:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
