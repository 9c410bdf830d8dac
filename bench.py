#!/usr/bin/env python
"""Benchmark of the Loraine.jl per-iteration interior-point hot path on B200.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload C5|C2|C3|C4|...-mini] [--dump-outputs DIR]

A "step" is ONE interior-point iteration (find_mu, prepare_W, predictor, sigma_update, corrector, check_convergence).
The workload is the configuration BASELINE.json's metric ("... at 1/2/4/8 B200") is quoted on: configs[4], the synthetic
large-Schur SDP with n_var = 40000 constraints and one PSD block of side 1000 (kit = 0).  It fits one GPU, so it is the
workload for EVERY N, 1 included: `--gpus N` (under torchrun) runs ONE solve whose Schur assembly and Cholesky
factorisation are sharded over the N ranks (row-block-cyclic, NCCL) -- strong scaling; `value` = seconds per iteration of
that one solve, max over ranks.  At N = 1 the line also carries the single-GPU configs[1..3] as `sub_records`.
`--dump-outputs DIR` writes the iterate left by the last timed step (see dump_outputs) so that two builds can be compared
output for output: the instance comes from a seeded generator, so the same arguments give the same inputs on every run.

`value`  : seconds per IP iteration with the problem and the iterate resident in HBM.
`e2e`    : the same iteration driven through the C ABI with the iterate in HOST (pinned) memory: X, S, y uploaded before and
           downloaded after every iteration inside the timed region.
`cpu_baseline` / `--impl reference`: the reference's CPU algorithm on the SAME full-size instance on the box's host cores.
           Julia is not in the image, so this is the NumPy/LAPACK oracle ("port"; sparse Schur assembly through the plain-C
           restatement oracle/schur_pairs.c, dpotrf in place).  One CPU iteration of configs[4] takes tens of seconds, so
           the arm measures at most 1 warm-up + 2 timed iterations and says so (`steps`, `steps_requested`).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "sec/IP-iteration"
UNIT = "s"

# stdout carries exactly ONE line (the JSON record): every other writer to file descriptor 1 (NCCL's version banner, library
# messages of any rank) is sent to stderr; the record itself goes to a private duplicate of the original stdout
_RECORD_OUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(line):
    _RECORD_OUT.write(json.dumps(line) + "\n")
    _RECORD_OUT.flush()


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4,
                    help="timed IP iterations of the workload; the --impl reference arm times at most --cpu-max-steps of them "
                         "and the N = 1 sub-records at most 4, each record states the count it timed")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C5")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-solve", action="store_true", help="skip the end-to-end solve to convergence reported under `solve`")
    ap.add_argument("--no-sub", action="store_true", help="N = 1: skip the configs[1..3] sub-records")
    ap.add_argument("--no-parity", action="store_true", help="N > 1: skip the sharded-vs-single-GPU parity check")
    ap.add_argument("--cpu-max-steps", type=int, default=2, help="reference arm: timed CPU iterations are capped at this number")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the iterate of the last timed step as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 implementation")
    return args


# ----------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """samples nvidia-smi clocks / throttle reasons DURING the timed region (profiling recipe's clocks line)"""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append([t.strip() for t in ln.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        reasons = []
        for name, col in (("hw_slowdown", 3), ("hw_thermal_slowdown", 4), ("sw_thermal_slowdown", 5), ("sw_power_cap", 6)):
            if any(len(r) >= 7 and r[col].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=reasons,
                    samples=len(sm))


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def algorithmic_flops(md, datarank):
    """SURVEY 8(d).  Rank-one assembly: sum_i n_var^2 m_i (lower SYRK, 2 flop/MAC) + 2 nnz(B_i) m_i + n_var^2/2.
    General assembly: sum_i sum_j min(F1_j, F3_j), F1_j = 2 m nnz_j + 2 m^3 + 2 sum_{k>=j} nnz_k, F3_j = 4 nnz_j sum_{k>=j} nnz_k
    (k over the matrices present in block i in sigmaA order).  Cholesky: n_var^3 / 3."""
    n = float(md.n)
    asm = 0.0
    for i, m in enumerate(md.msizes):
        if datarank == -1 and md.B:
            asm += n * n * m + 2.0 * md.B[i].nnz * m + 0.5 * n * n
        else:
            nz = np.sort(md.nzA[:, i][md.nzA[:, i] > 0])[::-1].astype(np.float64)
            suf = np.cumsum(nz[::-1])[::-1]
            f1 = 2.0 * m * nz + 2.0 * float(m) ** 3 + 2.0 * suf
            f3 = 4.0 * nz * suf
            asm += float(np.minimum(f1, f3).sum())
    if md.nlin:
        asm += 2.0 * float((np.diff(md.C_lin.tocsc().indptr).astype(np.float64) ** 2).sum())
    return dict(assemble=asm, factor=n ** 3 / 3.0)


def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every host core.  Returns the BLAS thread count."""
    n = os.cpu_count() or 1
    try:
        from threadpoolctl import threadpool_limits, threadpool_info
        threadpool_limits(limits=n)
        got = [int(p.get("num_threads", 0)) for p in threadpool_info() if p.get("user_api") == "blas"]
        return max(got) if got else n
    except Exception:
        return int(os.environ.get("OMP_NUM_THREADS", n))


DUMP_BYTES = 64 << 20


def iterate_arrays(S, s):
    """what a caller of the iteration receives: the blocks X_i and S_i, y, x_lin and s_lin (when there is an LP block), and
    (primal objective, dual objective, DIMACS error)"""
    md = s.model
    y, X, xl = S.get_solution(s)
    Sm = [np.zeros((m, m), order="F") for m in md.msizes]
    sl = np.zeros(md.nlin)
    PD = C.POINTER(C.c_double)
    s._call("lrn_get_slack", (PD * max(1, md.nlmi))(*[x.ctypes.data_as(PD) for x in Sm]), sl.ctypes.data_as(PD) if md.nlin else None)
    out = {f"X_{i}": x for i, x in enumerate(X)}
    out.update({f"S_{i}": x for i, x in enumerate(Sm)})
    out["y"] = y
    if md.nlin:
        out.update(x_lin=xl, s_lin=sl)
    out["objectives"] = np.array([s.primal_obj, s.dual_obj, s.DIMACS_error])
    return out


def dump_outputs(out_dir, arrays):
    """writes every array as out_dir/<name>.npy in float64.  When they would take more than DUMP_BYTES together, each array
    larger than an even share of that budget is replaced by a sample of its entries (column-major flat indices drawn with
    seed 0, sorted), which is the same on every run for the same shapes."""
    os.makedirs(out_dir, exist_ok=True)
    budget = DUMP_BYTES - 256 * len(arrays)                        # 256 bytes per file cover the .npy header
    share = budget // (8 * len(arrays))
    sample = 8 * sum(np.size(a) for a in arrays.values()) > budget
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64)
        if sample and a.size > share:
            a = a.ravel(order="F")[np.sort(np.random.default_rng(0).choice(a.size, share, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def workload_name(w):
    return {"C5": "configs[4]: synthetic large-Schur SDP n_var=40000 constraints, 1 PSD block m=1000, kit=0, datarank=0 (seed 40000)",
            "C4": "configs[3]: synthetic multi-block SDP, 50 PSD blocks of size 200 + LP block of 2000 rows, n_var=10000, kit=0",
            "C3": "configs[2]: synthetic Lovasz-theta SDP (thetaG11 layout) m=801, n_var=2401, kit=1 CG, preconditioner=1",
            "C2": "configs[1]: synthetic Max-Cut SDP (ex_maxcut.jl / maxG11 layout) n=5000, 1 PSD block m=5000, datarank=-1 rank-one "
                  "Schur path, kit=0 (torus 50x100, +-1 weights, seed 5000)"}.get(w, w)


# ----------------------------------------------------------------------------------------------------------------------
#  CPU arm: the oracle ("port") on the SAME full-size instance
# ----------------------------------------------------------------------------------------------------------------------
def cpu_iterations(pkg, workload, warmup, steps):
    """runs warmup + steps interior-point iterations of the oracle on the full-size instance of `workload` with all host
    threads; returns (seconds per timed iteration, description, threads, per-phase seconds of the timed iterations)"""
    from oracle import loraine_oracle as lo, sdpa_io, c_oracle
    blas_threads = use_all_host_threads()
    cfg = pkg.problems.CONFIGS[workload]
    arrays = cfg["gen"]()
    o = dict(cfg["options"], verb=0)
    md = lo.prepare_model(sdpa_io.raw_from_sdpa_arrays(*arrays), datarank=int(o.get("datarank", 0)), kappa=int(o.get("datasparsity", 8)))
    s, ha = lo.load(md, o)
    # large general-path instances: sparse Schur assembly through oracle/schur_pairs.c (the NumPy form needs minutes at
    # n_var = 40000), Cholesky in place; same arithmetic (pinned in tests/test_oracle_golden.py)
    s.lean = bool(md.n >= 4000 and int(o.get("datarank", 0)) != -1 and int(o.get("kit", 0)) == 0)
    threads = blas_threads
    if s.lean:
        threads = max(threads, c_oracle.max_threads())
    lo.setup_solver(s, ha)
    lo.initial_point(s)

    def step():
        lo.myIPstep(s, ha)
        s.tol_cg = max(s.tol_cg * s.tol_cg_up, s.tol_cg_min)
        lo.check_convergence(s)
        if s.status != 0:
            lo.initial_point(s)
    for _ in range(warmup):
        step()
    s.phase_time = {}
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    raw = (time.perf_counter() - t0) / max(1, steps)
    note = (f"full-size instance (same generator, seed and options as the GPU arm), {warmup} warm-up + {steps} timed IP iteration(s) of "
            f"the NumPy/LAPACK oracle" + (" with the plain-C sparse Schur assembly (oracle/schur_pairs.c) and in-place dpotrf" if s.lean else ""))
    return raw, note, threads, {k: v / max(1, steps) for k, v in s.phase_time.items()}


def run_reference(args):
    """The reference's CPU implementation of the path on the host cores.  Julia is not installed in this image, so the
    arm executes the NumPy/LAPACK oracle (oracle/, kind = "port") with all host threads on the full-size instance."""
    rank, world, local = dist_env()
    if rank != 0:
        return
    import __graft_entry__ as g
    pkg = g.load_package()
    warm = min(args.warmup, 1)
    steps = max(1, min(args.steps, args.cpu_max_steps))
    raw, note, cores, phases = cpu_iterations(pkg, args.workload, warm, steps)
    line = dict(metric=METRIC, value=raw, unit=UNIT, n_gpus=args.gpus, steps=steps, warmup=warm, steps_requested=args.steps,
                warmup_requested=args.warmup, ms_per_step=raw * 1e3, higher_is_better=False, scaling="strong", vs_baseline=None,
                dtype="f64", data="synthetic", impl="reference",
                config=dict(workload=workload_name(args.workload), sample=note, same_config=True),
                cpu_baseline=dict(value=raw, unit=UNIT, cores=cores, kind="port", sample=note, phases_s_per_iteration=phases),
                e2e=dict(value=raw, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    emit(line)


# ----------------------------------------------------------------------------------------------------------------------
#  GPU arm
# ----------------------------------------------------------------------------------------------------------------------
class Runner:
    """one workload on this rank's GPU (sharded over the job's ranks when the workload is configs[4] and world > 1)"""

    def __init__(self, pkg, workload, local, sharded):
        from loraine_jl_b200 import solver as S
        self.S, self.pkg, self.workload, self.local = S, pkg, workload, local
        self.cfg = pkg.problems.CONFIGS[workload]
        self.arrays = self.cfg["gen"]()
        self.opt = self._optimizer()
        self.s, self.ha = self.opt.solver, self.opt.halpha
        S.setup_solver(self.s, self.ha)
        self.sharded = bool(sharded and pkg.dist.init_distributed(self.s))
        S.initial_point(self.s)
        self.restart = False

    def _optimizer(self):
        opt = self.pkg.Optimizer()
        for k, v in dict(self.cfg["options"], verb=0, device=self.local).items():
            opt.set_attribute(k, v)
        opt.copy_to(self.pkg.raw_from_sdpa_arrays(*self.arrays))
        return opt

    def make_single(self):
        """a second, single-GPU solver of the same instance on the same device (parity reference of the sharded path)"""
        opt = self._optimizer()
        self.S.setup_solver(opt.solver, opt.halpha)
        return opt.solver

    def step(self, sync_status=None):
        S, s = self.S, self.s
        if self.restart:          # the last step converged (or failed): restart the same solve so that every step is a real iteration
            S.initial_point(s)
        S.myIPstep(s, self.ha)
        s.itertime = 0.0
        s.tol_cg = max(s.tol_cg * s.tol_cg_up, s.tol_cg_min)
        S.check_convergence(s)
        # restarting at the start of the next step keeps this step's iterate on the device until then (--dump-outputs)
        self.restart = (s.status if sync_status is None else sync_status(s.status)) != 0


def measure(run, args, world, rank, barrier, sync_status, L, want_solve, dump_dir=None):
    """timed device-resident steps, e2e steps, per-launch DMMA profile, optional full solve -> dict of raw results;
    dump_dir: rank 0 writes the iterate of the last timed step there"""
    import torch
    S, s, md = run.S, run.s, run.s.model
    warm = max(args.warmup, 3)
    tol_cg0 = s.tol_cg
    for _ in range(warm):
        run.step(sync_status)
    sampler = ClockSampler(run.local)
    if rank == 0:
        sampler.start()
    s.timers(reset=True)
    launches0 = L.lrn_kernel_launches()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        run.step(sync_status)
    barrier()
    t_dev = time.perf_counter() - t0
    launches = L.lrn_kernel_launches() - launches0
    phase = s.timers(reset=True)
    clocks = sampler.stop() if rank == 0 else None
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, iterate_arrays(S, s))
    # ---- e2e: the iterate lives in HOST memory; upload before / download after every iteration ------------------------
    S.initial_point(s)
    run.restart = False
    s.tol_cg = tol_cg0
    y, X, xl = S.get_solution(s)
    PD = C.POINTER(C.c_double)
    Sm = [np.zeros((m, m), order="F") for m in md.msizes]
    sl = np.zeros(md.nlin)
    Sp = (PD * max(1, md.nlmi))(*[x.ctypes.data_as(PD) for x in Sm])
    s._call("lrn_get_slack", Sp, sl.ctypes.data_as(PD) if md.nlin else None)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()
    Xh = [np.asfortranarray(pin(x.T).T) for x in X]
    Sh = [np.asfortranarray(pin(x.T).T) for x in Sm]
    yh, xlh, slh = pin(y), pin(xl), pin(sl)
    Shp = (PD * max(1, md.nlmi))(*[x.ctypes.data_as(PD) for x in Sh])
    h2d = sum(x.nbytes for x in Xh) + sum(x.nbytes for x in Sh) + yh.nbytes + xlh.nbytes + slh.nbytes

    def e2e_step():
        S.set_iterate(s, Xh, Sh, yh, xlh, slh)                      # H2D from the pinned buffers
        S.myIPstep(s, run.ha)
        s.itertime = 0.0
        s.tol_cg = max(s.tol_cg * s.tol_cg_up, s.tol_cg_min)
        S.check_convergence(s)
        st = s.status if sync_status is None else sync_status(s.status)
        if st != 0:
            S.initial_point(s)
        S.get_solution(s, out=(yh, Xh, xlh))                        # D2H straight into the pinned buffers
        s._call("lrn_get_slack", Shp, slh.ctypes.data_as(PD) if md.nlin else None)

    for _ in range(warm):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    barrier()
    t_e2e = time.perf_counter() - t0
    # ---- roofline pass: per-launch CUDA events around every DMMA GEMM launch (on the launching stream) ----------------
    ms, fl, nl = C.c_double(), C.c_double(), C.c_int64()
    L.lrn_dbg_gemm_profile(1, None, None, None)
    run.step(sync_status)
    L.lrn_dbg_gemm_profile(0, C.byref(ms), C.byref(fl), C.byref(nl))
    fams = []
    for code, kname in ((10, "dgemm_dmma_kernel (cp.async-fed DMMA GEMM: congruences, Gram products, TRSM, edge strips)"),
                        (11, "dgemm_dmma_bulk_kernel (TMA-fed DMMA GEMM: Schur SYRK, Cholesky trailing updates, panel solves, large congruences)"),
                        (12, "panel_rotate_kernel (TMA-fed DMMA panel rotation of the block-Jacobi SVD)")):
        fm, ff, fn = C.c_double(), C.c_double(), C.c_int64()
        L.lrn_dbg_gemm_profile(code, C.byref(fm), C.byref(ff), C.byref(fn))
        if fn.value > 0 and fm.value > 0:
            fams.append(dict(kernel=kname, launches=int(fn.value), kernel_ms_per_step=fm.value,
                             algorithmic_flops_per_launch=ff.value / fn.value,
                             avg_launch_us=1e3 * fm.value / fn.value, achieved=ff.value / (fm.value * 1e-3) / 1e12))
    # ---- end-to-end solve to the reference's stopping rule (outside the timed regions) -------------------------------
    solve_info = None
    if want_solve:
        barrier()
        t0 = time.perf_counter()
        if sync_status is None:
            S.solve(s, run.ha, setup=False)
        else:                                   # sharded: same loop, the termination test is agreed between the ranks
            S.initial_point(s)
            while True:
                S.myIPstep(s, run.ha)
                s.tol_cg = max(s.tol_cg * s.tol_cg_up, s.tol_cg_min)
                S.check_convergence(s)
                if sync_status(s.status) != 0 or s.iter > s.maxit:
                    break
        barrier()
        solve_info = dict(seconds=time.perf_counter() - t0, iterations=int(s.iter), status=int(s.status),
                          dimacs_error=float(s.DIMACS_error), primal_obj=float(s.primal_obj), dual_obj=float(s.dual_obj),
                          cg_iterations=int(s.cg_iter_tot) if s.kit == 1 else None)
    alg = algorithmic_flops(md, int(s.datarank))
    asm_ms = phase["schur_assemble"][0] / max(1, phase["schur_assemble"][1])
    fac_ms = phase["schur_factor"][0] / max(1, phase["schur_factor"][1])
    schur = dict(assemble_ms=asm_ms, assemble_tflops=alg["assemble"] / (asm_ms * 1e-3) / 1e12 if asm_ms > 0 else None,
                 factor_ms=fac_ms, factor_tflops=alg["factor"] / (fac_ms * 1e-3) / 1e12 if fac_ms > 0 else None,
                 assemble_plus_factor_tflops=(alg["assemble"] + alg["factor"]) / ((asm_ms + fac_ms) * 1e-3) / 1e12
                 if asm_ms + fac_ms > 0 else None,
                 note="algorithmic flops of the WHOLE matrix (SURVEY 8(d)) over this rank's phase time: aggregate rate of the job")
    return dict(t_dev=t_dev, t_e2e=t_e2e, launches=int(launches), phase=phase, clocks=clocks, h2d=int(h2d), fams=fams,
                all_dmma=dict(ms=ms.value, flops=fl.value, launches=int(nl.value)), solve=solve_info, schur=schur,
                stats=s.stats(), warm=warm)


def run_b200(args):
    rank, world, local = dist_env()
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        # keep stdout for the one JSON line: NCCL's own messages (version banner, INFO) go to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import __graft_entry__ as g
    pkg = g.load_package()
    from loraine_jl_b200 import _lib
    L = _lib.lib()
    L.lrn_dbg_peak.argtypes = [C.c_int32, C.POINTER(C.c_double)]
    L.lrn_dbg_gemm_profile.argtypes = [C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int64)]

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    shardable = args.workload.startswith("C5") or args.workload.startswith("C2")
    run = Runner(pkg, args.workload, local, sharded=(world > 1 and shardable))
    sync_status = None
    if world > 1 and run.sharded:
        flag = torch.zeros(1, device="cuda", dtype=torch.int32)

        def sync_status(st):                     # every rank takes the same restart / stop decision (collectives must line up)
            flag[0] = int(st)
            dist.all_reduce(flag, op=dist.ReduceOp.MAX)
            return int(flag.item())
    s, md = run.s, run.s.model
    res = measure(run, args, world, rank, barrier, sync_status, L, want_solve=not args.no_solve, dump_dir=args.dump_outputs)
    # ---- sharded path against the single-GPU path on the same inputs (outside the timed regions) ---------------------
    parity = None
    if run.sharded and not args.no_parity:
        parity = pkg.dist.dist_parity(s, run.make_single, rank, iters=2)
    tmax = torch.tensor([res["t_dev"], res["t_e2e"]], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    t_dev, t_e2e = float(tmax[0]), float(tmax[1])
    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    peak = C.c_double()
    L.lrn_dbg_peak(0, C.byref(peak))
    # sharded: all ranks advance ONE solve together; replicas (a workload that does not shard): `world` independent solves
    units = 1 if (run.sharded or world == 1) else world
    sec_per_iter = t_dev / (args.steps * units)
    e2e_val = t_e2e / (args.steps * units)
    fams = res["fams"]
    dom = max(fams, key=lambda d: d["kernel_ms_per_step"]) if fams else None
    phase = res["phase"]
    line = dict(
        metric=METRIC, value=sec_per_iter, unit=UNIT, n_gpus=world, steps=args.steps, warmup=res["warm"],
        ms_per_step=1e3 * t_dev / args.steps, higher_is_better=False, scaling="strong" if (run.sharded or world == 1) else "weak",
        vs_baseline=None, dtype="f64", data="synthetic",
        config=dict(workload=workload_name(args.workload), n_var=md.n, msizes=md.msizes[:4], nlin=md.nlin,
                    options=run.cfg["options"],
                    l2="inputs larger than L2 (Schur matrix and factor: 12.8 GB each; the dense m x m operands are re-read from HBM "
                       "between kernels)" if md.n >= 20000 else "inputs larger than L2 (every dense operand of the iteration exceeds 126 MB "
                       "in total; 19+ resident m x m matrices per block)",
                    parallelism=("Schur assembly + Cholesky sharded row-block-cyclic over %d GPUs (diagonal-block inverse broadcast, "
                                 "ncclAllGather of the solved panel, NCCL over NVLink), m x m work replicated" % world)
                    if run.sharded else ("replicas only" if world > 1 else "single GPU")),
        e2e=dict(value=e2e_val, unit=UNIT, h2d_bytes_per_step=res["h2d"], d2h_bytes_per_step=res["h2d"], steps=args.steps),
        gpu_launches=res["launches"], clocks=res["clocks"], solve=res["solve"],
        phases_ms_per_iteration={k: v[0] / args.steps for k, v in phase.items()},
        # CUDA-event time of the ABI calls of one step on the library stream (nested phases svd / eigmin not double counted)
        device_event_ms_per_step=sum(v[0] for k, v in phase.items() if k not in ("svd", "eigmin")) / args.steps,
        schur=res["schur"],
        roofline=dict(bound="tensor", kernel=dom["kernel"] if dom else None,
                      achieved=dom["achieved"] if dom else None, peak=peak.value, unit="TFLOP/s",
                      frac=dom["achieved"] / peak.value if dom and peak.value else None,
                      traffic=None,   # no dram__bytes capture of this launch mix is kept for this round; see profiles/ for per-kernel ncu
                      launches_profiled=dom["launches"] if dom else 0, kernel_ms_per_step=dom["kernel_ms_per_step"] if dom else None,
                      avg_launch_us=dom["avg_launch_us"] if dom else None,
                      algorithmic_flops_per_launch=dom["algorithmic_flops_per_launch"] if dom else None,
                      all_dmma_kernels=dict(achieved=res["all_dmma"]["flops"] / (res["all_dmma"]["ms"] * 1e-3) / 1e12
                                            if res["all_dmma"]["ms"] > 0 else None,
                                            launches=res["all_dmma"]["launches"], kernel_ms_per_step=res["all_dmma"]["ms"]),
                      by_kernel=fams,
                      note="per-launch CUDA events on the launching stream; the panel stream and the main stream run this kernel "
                           "concurrently during the factorisation (look-ahead), so launch durations overlap and share SMs: the sum "
                           "understates the rate of the phase as a whole, which is schur.factor_tflops",
                      peak_source="measured in this run: register-resident mma.sync.m8n8k4.f64 loop on all SMs "
                                  "(MEASURED_PEAKS.json has no FP64 entry; cuBLAS DGEMM 8192^3 on this pool: 35.4 TFLOP/s)"),
        stats=res["stats"], dist_parity=parity,
    )
    # ---- single-GPU sub-records of the other named configs (N = 1 only) ----------------------------------------------
    if world == 1 and not args.no_sub and args.workload == "C5":
        run.s.close()
        del run
        subs = {}
        sub_args = argparse.Namespace(**vars(args))
        sub_args.steps = min(args.steps, 4)
        for w in ("C2", "C3", "C4"):
            r = Runner(pkg, w, local, sharded=False)
            m = measure(r, sub_args, 1, 0, barrier, None, L, want_solve=not args.no_solve)
            f2 = max(m["fams"], key=lambda d: d["kernel_ms_per_step"]) if m["fams"] else None
            subs[w] = dict(workload=workload_name(w), value=m["t_dev"] / sub_args.steps, unit=UNIT, steps=sub_args.steps, warmup=m["warm"],
                           e2e=m["t_e2e"] / sub_args.steps, gpu_launches=m["launches"], solve=m["solve"], schur=m["schur"],
                           phases_ms_per_iteration={k: v[0] / sub_args.steps for k, v in m["phase"].items()},
                           dominant_dmma_kernel=dict(kernel=f2["kernel"], achieved_tflops=f2["achieved"],
                                                     frac=f2["achieved"] / peak.value if peak.value else None,
                                                     kernel_ms_per_step=f2["kernel_ms_per_step"]) if f2 else None,
                           stats=m["stats"])
            r.s.close()
            del r
        subs["dd_lp"] = dd_lp_record(pkg, sub_args)
        line["sub_records"] = subs
    if world == 1 and not args.no_cpu_baseline:
        raw, note, cores, phases = cpu_iterations(pkg, args.workload, 0, 1)
        line["cpu_baseline"] = dict(value=raw, unit=UNIT, cores=cores, kind="port", sample=note, same_config=True,
                                    phases_s_per_iteration=phases)
    emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def dd_lp_record(pkg, args):
    """Double-double (Float64x2) LP path (include/loraine_b200_dd.h, SURVEY 8(f) N4): sec / IP iteration on a synthetic LP with
    2000 multipliers and 5000 LP rows (2 % dense), the rate of the double-double Cholesky against the FP64 issue bound, and a full
    solve to DIMACS error 1e-24."""
    import time
    import torch
    from loraine_jl_b200 import dd_lp
    n, nlin = 2000, 5000
    spec = pkg.problems.random_lp(n, nlin, 1, density=0.02)
    md = pkg.prepare_model(pkg.RawProblem(**spec))
    s = dd_lp.DDSolver(md, dict(pkg.DEFAULT_OPTIONS, eDIMACS=1e-24, verb=0))
    dd_lp.setup_solver(s)
    dd_lp.initial_point(s)
    for _ in range(3):                                     # warm-up iterations (the iterate stays well inside the cone)
        dd_lp.myIPstep(s)
    s.timers(reset=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        dd_lp.myIPstep(s)
    torch.cuda.synchronize()
    sec = (time.perf_counter() - t0) / args.steps
    t = s.timers()
    s.itertime = 0.0
    dd_lp.check_convergence(s)
    t1 = time.perf_counter()
    dd_lp.solve(s, setup=False)
    solve_s = time.perf_counter() - t1
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    # one double-double multiply-add = 28 FP64 instructions in the SASS of k_dd_syrk_tile (24 DADD + 2 DMUL + 2 DFMA);
    # 64 FP64 instructions / clk / SM; a Cholesky factorisation is n^3/6 multiply-adds
    bound = 64.0 * sm * 1.965e9 / 28.0
    fma = n ** 3 / 6.0
    rate = fma / (t["schur_factor"] / args.steps * 1e-3)
    rec = dict(workload="synthetic LP without PSD blocks, Optimizer{Float64x2}: 2000 multipliers, 5000 LP rows, 2 % dense",
               value=sec, unit=UNIT, steps=args.steps, warmup=3, dtype="f64x2 (double-double)",
               phases_ms_per_iteration={k: v / args.steps for k, v in t.items()},
               cholesky=dict(dd_fma_per_s=rate, bound_dd_fma_per_s=bound, frac=rate / bound,
                             note="n^3/6 double-double multiply-adds; bound = FP64 issue rate (64 / clk / SM at 1965 MHz) / 28 "
                                  "instructions per double-double multiply-add; n = 2000 is 63 dependent tile steps: chain-bound, "
                                  "n = 5000 reaches 0.75 of the bound (scripts/prof_ddlp.py)"),
               solve=dict(status=int(s.status), iterations=int(s.iter), dimacs_error=float(s.DIMACS_error), seconds_after_warmup=solve_s))
    s.close()
    return rec


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
