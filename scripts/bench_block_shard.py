"""PSD blocks distributed over the GPUs (lrn_create_multi, kit = 0) against the replicated block layout forced at the same
number of GPUs (lrn_dbg_block_layout): seconds per IP iteration, the prepare_W, right-hand side and find_step milliseconds
per iteration, and the device bytes of every rank against the footprint lrn_finalize computed for it.

    python scripts/bench_block_shard.py [--iters 3] [--reps 2] [--out profiles/block_shard_b200.jsonl]

Workloads: configs[3] (C4: 50 blocks of side 200 and 2000 LP rows, full size) and multiblock_lp with 8 blocks of side 2000
(and its 2000 LP rows), the case where each block's chain (Cholesky, SVD, congruences) is large.  Runs on 1 / 2 / 4 / 8 GPUs;
with more than one GPU the two arms alternate `reps` times.  One GPU has one arm (the blocks cannot be distributed over a
single rank).  A run needing more GPUs than the machine has is written as "not measured".  Every line carries the GPU name
and power limit (nvidia-smi).
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
import __graft_entry__ as g  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else None


def run(pkg, arrays, opts, ngpus, blocks, iters):
    import torch
    from loraine_jl_b200 import solver as S
    devs = list(range(ngpus))
    torch.cuda.synchronize()
    free0 = [torch.cuda.mem_get_info(d)[0] for d in devs]
    opt = pkg.Optimizer()
    for k, v in dict(opts, ngpus=ngpus, verb=0).items():
        opt.set_attribute(k, v)
    opt.copy_to(pkg.raw_from_sdpa_arrays(*arrays))
    s = opt.solver

    def force(h):
        if blocks is not None:
            assert h.lib.lrn_dbg_block_layout(h.h, blocks, None) == 0
    S.setup_solver(s, opt.halpha, before_finalize=force)
    lay = C.c_int32(-9)
    s.lib.lrn_dbg_block_layout(s.h, -2, C.byref(lay))
    S.initial_point(s)
    S.myIPstep(s, opt.halpha)                       # warm-up: first-use allocations of every phase
    s.itertime = 0.0
    S.check_convergence(s)
    s.timers(reset=True)
    t0 = time.perf_counter()
    for _ in range(iters):
        S.myIPstep(s, opt.halpha)
        s.itertime = 0.0
        S.check_convergence(s)
    t_it = (time.perf_counter() - t0) / iters
    tm = s.timers()
    fp = []
    for r in range(ngpus):
        b = C.c_int64()
        s.lib.lrn_dbg_block_footprint(s.h, r, 1 if lay.value == 1 else 0, C.byref(b), None)
        fp.append(b.value)
    used = [free0[d] - torch.cuda.mem_get_info(d)[0] for d in devs]
    s.close()
    return dict(blocks="distributed" if lay.value == 1 else "replicated", s_per_iter=t_it,
                prepare_W_ms=tm["prepare_W"][0] / iters, rhs_ms=tm["rhs"][0] / iters, find_step_ms=tm["find_step"][0] / iters,
                device_bytes_per_rank=used, footprint_bytes_per_rank=fp)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "block_shard_b200.jsonl"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU")
    pkg = g.load_package()
    ndev = torch.cuda.device_count()
    gpu = card()
    work = {"C4": (lambda: pkg.problems.CONFIGS["C4"]["gen"](), dict(pkg.problems.CONFIGS["C4"]["options"])),
            "8x2000": (lambda: pkg.problems.multiblock_lp(8, 2000, 2000, 50), dict(kit=0, datarank=0, initpoint=1, eDIMACS=1e-6))}
    lines = []
    for name, (gen, opts) in work.items():
        arrays = gen()
        for k in (1, 2, 4, 8):
            arms = [None] if k == 1 else [None, 0] * a.reps
            for blocks in arms:
                rec = dict(config=name, ngpus=k, forced_blocks=blocks, gpu=gpu)
                if ndev < k:
                    rec["result"] = "not measured"
                    rec["reason"] = f"{ndev} GPU(s) on the machine"
                else:
                    rec.update(run(pkg, arrays, opts, k, blocks, a.iters))
                lines.append(rec)
                print(json.dumps(rec), flush=True)
                if ndev < k:
                    break                                   # one "not measured" line per configuration
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for r in lines:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
