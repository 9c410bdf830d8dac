"""CPU tests of the multi-GPU double-double LP path: the row ownership of the sharded Schur matrix, and the in-process
multi-GPU constructor refusing to run without a GPU."""
import ctypes as C

import pytest


@pytest.mark.parametrize("n", [64, 300, 1100, 5000, 20000])
def test_dd_row_ownership_is_a_partition(pkg, n):
    d = pkg.dist
    pw = d.dd_block_rows(n)
    assert pw == (256 if n >= 4096 else (128 if n >= 1024 else 64)) and pw % 32 == 0
    nblk = -(-n // pw)
    for world in range(1, 9):
        owners = [d.row_owner(r, pw, world) for r in range(n)]
        assert set(owners) <= set(range(world))
        for r in range(0, n, pw):                       # constant inside a row block, rotating between consecutive blocks
            assert len(set(owners[r:r + pw])) == 1
            assert owners[r] == (r // pw) % world
        counts = [owners.count(r) for r in range(world)]
        assert sum(counts) == n and max(counts) - min(counts) <= pw
        for p in range(nblk - 1):
            # the all-gather of step p carries every row block below the diagonal block exactly once
            blocks = []
            for r in range(world):
                f, c = d.first_block(p + 1, r, world), d.count_blocks(p + 1, r, world, nblk)
                blocks += [f + z * world for z in range(c)]
                assert c <= -(-(nblk - p - 1) // world)
            assert sorted(blocks) == list(range(p + 1, nblk))


def test_dd_create_multi_without_gpu_fails(pkg):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from loraine_jl_b200 import _lib
    L = _lib.lib()
    for ngpus in (1, 2, 0, -1, 8):
        h = C.c_void_p()
        assert L.lrn_dd_create_multi(C.byref(h), 10, 20, ngpus, None) < 0, ngpus
        assert not h.value
    # the Python host surfaces the error instead of falling back
    spec = pkg.problems.random_lp(8, 20, 3)
    opt = pkg.Optimizer(T="Float64x2")
    opt.set_attribute("verb", 0)
    opt.set_attribute("ngpus", 2)
    opt.copy_to(pkg.RawProblem(**spec))
    with pytest.raises(Exception) as ei:
        opt.optimize()
    assert "no CPU fallback" in str(ei.value)
