"""Admission of the direct path (kit = 0) by device memory: lrn_finalize adds up the bytes of the dense Schur matrix, its
factor, the Cholesky workspace and the model before allocating anything, and refuses a model that does not fit with both
byte counts instead of a bare CUDA out-of-memory error."""
import re

import pytest

import mc_instances as mc

pytestmark = pytest.mark.gpu

KIT0 = dict(kit=0, initpoint=1, verb=0, eDIMACS=1e-6)


def _error():
    from loraine_jl_b200.solver import LoraineB200Error
    return LoraineB200Error


def _optimizer(pkg, inst):
    opt = pkg.Optimizer()
    for k, v in KIT0.items():
        opt.set_attribute(k, v)
    opt.load_sdpa(*inst.arrays)
    return opt


def _free_bytes():
    import torch
    torch.cuda.empty_cache()
    torch.cuda.synchronize()
    return torch.cuda.mem_get_info(0)[0]


def test_kit0_larger_than_one_gpu_refused_with_byte_counts(pkg):
    """n_var = 110 000 is below the lrn_create limit of 140 000, but H and L alone take 16 n_var^2 = 194 GB: lrn_finalize
    refuses the model, naming the bytes it needs and the bytes that are free, and allocates nothing."""
    n = 110000
    inst = mc.matrix_completion(600, 600, 2, n, seed=23)
    free0 = _free_bytes()
    opt = _optimizer(pkg, inst)
    with pytest.raises(_error(), match=r"kit = 0 state needs \d+ bytes of device memory, \d+ bytes are free") as ei:
        opt.optimize()
    need, free = (int(v) for v in re.search(r"needs (\d+) bytes of device memory, (\d+) bytes are free", str(ei.value)).groups())
    assert need > free
    assert need >= 16 * n * n
    opt.solver.close()
    assert free0 - _free_bytes() < 2 ** 30


def test_kit0_below_one_gpu_ceiling_admitted(pkg):
    """n_var = 96 000 fits a B200: lrn_finalize admits it and allocates the dense H and L (16 n_var^2 = 147 GB)."""
    from loraine_jl_b200 import solver as S
    n = 96000
    inst = mc.matrix_completion(600, 600, 2, n, seed=24)
    free0 = _free_bytes()
    opt = _optimizer(pkg, inst)
    s = opt.solver
    S.setup_solver(s, opt.halpha)
    used = free0 - _free_bytes()
    assert 16 * n * n <= used <= 16 * n * n + 4 * 2 ** 30, used
    s.close()
