"""Multi-GPU scaling of the double-double LP path (Optimizer{Float64x2} without PSD blocks, include/loraine_b200_dd.h).

Instance: problems.random_lp(n, 2 n, 1, density=0.02) -- the generator and density of bench.py's dd_lp sub-record, at larger n.
For every n and every GPU count the in-process handle (lrn_dd_create_multi; ngpus = 1 is the plain single-GPU handle) runs
--warmup IP iterations, then --iters timed ones, and prints ONE JSON line:
  sec_per_iter        host clock around the timed iterations (every entry point ends in a device synchronise)
  assemble/factor/solve_ms_per_iter   device times of member 0 from lrn_dd_timers (CUDA events)
  factor_dd_fma_per_s (n^3/6) dd multiply-adds per iteration over the factor time, against ngpus x 0.665e12 (the FP64-issue
                      bound of a B200 at 28 FP64 instructions per dd multiply-add, DESIGN.md section 3)
  rel_dely / rel_y    relative difference of the last dely and of y from the 1-GPU run on the same instance
  gpu / power_limit_w the card and its power limit, read with nvidia-smi in the same run
The 1-GPU run leaves its model, dely and y in --ref-dir; `--dist` runs the same measurement as one process per GPU under
torchrun (lrn_dd_dist_init) on that model:
  python scripts/bench_dd_multi.py --n 5000 20000 --ngpus 1 2 4 8 --ref-dir /tmp/ddref --out profiles/dd_multi.jsonl
  torchrun --nproc-per-node 8 scripts/bench_dd_multi.py --dist --n 20000 --ref-dir /tmp/ddref --out profiles/dd_multi.jsonl
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
DD_FMA_BOUND = 0.665e12          # dd multiply-adds per second and GPU at the FP64 issue rate (DESIGN.md section 3)


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"], capture_output=True,
                       text=True, check=True)
    name, watts = [x.strip() for x in r.stdout.splitlines()[0].split(",")]
    return name, float(watts)


def model_for(pkg, n, ref_dir):
    """the model of random_lp(n, 2 n, 1, density=0.02); cached as sparse arrays in ref_dir (the generator builds C_lin dense)"""
    path = os.path.join(ref_dir, f"model_{n}.npz")
    if os.path.exists(path):
        z = np.load(path)
        C_lin = sp.csc_matrix((z["data"], z["indices"], z["indptr"]), shape=tuple(z["shape"]))
        raw = pkg.RawProblem(n=n, msizes=[], A=[], b=z["b"], b_const=0.0, C_lin=C_lin, d_lin=z["d_lin"])
    else:
        spec = pkg.problems.random_lp(n, 2 * n, 1, density=0.02)
        raw = pkg.RawProblem(**spec)
        del spec
        C_lin = sp.csc_matrix(raw.C_lin)
        np.savez(path, data=C_lin.data, indices=C_lin.indices, indptr=C_lin.indptr, shape=np.array(C_lin.shape), b=raw.b,
                 d_lin=raw.d_lin)
    return pkg.prepare_model(raw)


def measure(pkg, md, ngpus, warmup, iters, dist_rank=None):
    from loraine_jl_b200 import dd_lp, dist
    o = dict(pkg.DEFAULT_OPTIONS, eDIMACS=1e-30, verb=0, maxit=10 ** 6, ngpus=1 if dist_rank is not None else ngpus)
    if dist_rank is not None:
        o["device"] = dist_rank
    s = dd_lp.DDSolver(md, o)
    dd_lp.setup_solver(s)
    if dist_rank is not None:
        assert dist.init_distributed_dd(s)
    dd_lp.initial_point(s)

    def step():
        dd_lp.myIPstep(s)
        s.itertime = 0.0
        dd_lp.check_convergence(s)
        if s.status != 0:
            raise RuntimeError(f"the solve stopped (status {s.status}) inside the measured window")
    for _ in range(warmup):
        step()
    s.timers(reset=True)
    t0 = time.perf_counter()
    for _ in range(iters):
        step()
    sec = (time.perf_counter() - t0) / iters
    t = s.timers()
    dely = s.get_array("DELY")
    dd_lp.get_solution(s)
    y = s.y_dd
    s.close()
    return sec, {k: v / iters for k, v in t.items()}, dely, y


def rel(a, b):
    d = (a[0] - b[0]) + (a[1] - b[1])
    return float(np.linalg.norm(d) / max(np.linalg.norm(b[0]), 1e-300))


def record(n, ngpus, mode, sec, t, dely, y, ref, args, name, watts):
    f_s = t["schur_factor"] / 1e3
    rate = (n ** 3 / 6) / f_s if f_s > 0 else float("nan")
    out = dict(bench="dd_multi", mode=mode, n=n, nlin=2 * n, density=0.02, ngpus=ngpus, warmup=args.warmup, iters=args.iters,
               sec_per_iter=round(sec, 4), assemble_ms_per_iter=round(t["schur_assemble"], 2),
               factor_ms_per_iter=round(t["schur_factor"], 2), solve_ms_per_iter=round(t["schur_solve"], 2),
               other_ms_per_iter=round(t["other"], 2), factor_dd_fma_per_s=float("%.4g" % rate),
               factor_share_of_bound=round(rate / (ngpus * DD_FMA_BOUND), 4),
               rel_dely=rel(dely, ref["dely"]) if ref else 0.0, rel_y=rel(y, ref["y"]) if ref else 0.0,
               gpu=name, power_limit_w=watts)
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        with open(args.out, "a") as f:
            f.write(line + "\n")


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--n", type=int, nargs="+", default=[5000, 20000])
    ap.add_argument("--ngpus", type=int, nargs="+", default=[1, 2, 4, 8])
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--ref-dir", required=True, help="model cache and 1-GPU reference results (not part of the output)")
    ap.add_argument("--out", default=None, help="append the JSON lines to this file as well")
    ap.add_argument("--dist", action="store_true", help="one process per GPU (run under torchrun)")
    args = ap.parse_args()
    if args.iters < 3:
        ap.error("--iters must be at least 3")
    import torch
    import __graft_entry__ as g
    pkg = g.load_package()
    if not torch.cuda.is_available():
        raise SystemExit("bench_dd_multi.py needs CUDA devices (there is no CPU fallback)")
    os.makedirs(args.ref_dir, exist_ok=True)
    name, watts = card()
    if args.dist:
        import torch.distributed as tdist
        rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
        tdist.init_process_group("gloo")
        for n in args.n:
            md = model_for(pkg, n, args.ref_dir) if rank == 0 else None
            tdist.barrier()                          # rank 0 writes the model cache if the in-process run did not
            if rank != 0:
                md = model_for(pkg, n, args.ref_dir)
            sec, t, dely, y = measure(pkg, md, world, args.warmup, args.iters, dist_rank=int(os.environ.get("LOCAL_RANK", rank)))
            if rank == 0:
                rp = os.path.join(args.ref_dir, f"ref_{n}_{args.warmup}_{args.iters}.npz")
                ref = None
                if os.path.exists(rp):
                    z = np.load(rp)
                    ref = dict(dely=(z["dh"], z["dl"]), y=(z["yh"], z["yl"]))
                record(n, world, "torchrun", sec, t, dely, y, ref, args, name, watts)
            tdist.barrier()
        tdist.destroy_process_group()
        return
    ndev = torch.cuda.device_count()
    for n in args.n:
        md = model_for(pkg, n, args.ref_dir)
        ref = None
        for ngpus in sorted(set(args.ngpus)):
            if ngpus > ndev:
                print(json.dumps(dict(bench="dd_multi", n=n, ngpus=ngpus, skipped=f"only {ndev} GPUs visible")), flush=True)
                continue
            sec, t, dely, y = measure(pkg, md, ngpus, args.warmup, args.iters)
            if ngpus == 1:
                ref = dict(dely=dely, y=y)
                np.savez(os.path.join(args.ref_dir, f"ref_{n}_{args.warmup}_{args.iters}.npz"), dh=dely[0], dl=dely[1], yh=y[0],
                         yl=y[1])
            record(n, ngpus, "in-process", sec, t, dely, y, ref if ngpus > 1 else None, args, name, watts)


if __name__ == "__main__":
    main()
