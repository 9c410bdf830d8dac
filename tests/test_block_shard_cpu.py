"""Ownership of the PSD blocks when they are distributed over the ranks (loraine_jl_b200.dist.block_owner, mirroring
lrn::block_owner in csrc/ops.cuh) against an independent greedy restatement and brute-force optima, and the footprint the
distributed block layout adds or saves (dist.block_shard_bytes, mirroring direct_footprint in csrc/solver.cu)."""
import heapq
import itertools

import numpy as np
import pytest


@pytest.fixture(scope="module")
def dist(pkg):
    return pkg.dist


def _greedy(msizes, world):
    """the longest-processing-time rule with a heap keyed (load, rank)"""
    heap = [(0, r) for r in range(world)]
    owner = [None] * len(msizes)
    for i in sorted(range(len(msizes)), key=lambda i: (-msizes[i] ** 3, i)):
        load, r = heapq.heappop(heap)
        owner[i] = r
        heapq.heappush(heap, (load + msizes[i] ** 3, r))
    return owner


def _cases():
    rng = np.random.default_rng(11)
    out = [[13, 12], [10, 5], [40, 200, 500], [200] * 50, [2000] * 8, [7], [5, 5, 5, 5, 5], [1, 46000, 3, 46000],
           [30, 30, 20, 20, 20, 10, 10, 10, 10]]
    for _ in range(20):
        out.append([int(x) for x in rng.integers(1, 600, size=int(rng.integers(1, 13)))])
    return out


@pytest.mark.parametrize("world", range(1, 9))
@pytest.mark.parametrize("msizes", _cases(), ids=lambda m: "x".join(map(str, m[:6])) + ("" if len(m) <= 6 else "..."))
def test_block_owner_is_the_deterministic_greedy_balance(dist, world, msizes):
    owner = dist.block_owner(msizes, world)
    assert len(owner) == len(msizes)                                   # every block owned exactly once
    assert all(0 <= r < world for r in owner)
    assert owner == dist.block_owner(list(msizes), world)              # deterministic
    assert owner == _greedy(msizes, world)
    # each block went to a least-loaded rank, the lowest of them on a tie
    load = [0] * world
    for i in sorted(range(len(msizes)), key=lambda i: (-msizes[i] ** 3, i)):
        assert owner[i] == min(range(world), key=lambda r: (load[r], r))
        load[owner[i]] += msizes[i] ** 3
    if world == 1:
        assert set(owner) <= {0}
    if len(msizes) < world:                                            # ranks without a block
        assert len(set(owner)) == len(msizes)


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("seed", range(12))
def test_block_owner_meets_the_lpt_bound_of_the_brute_force_optimum(dist, world, seed):
    """Graham's bound: the largest per-rank load is at most (4/3 - 1/(3 world)) times the optimum, found by enumerating
    every assignment"""
    rng = np.random.default_rng(seed)
    msizes = [int(x) for x in rng.integers(1, 60, size=int(rng.integers(2, 8)))]
    w = [m ** 3 for m in msizes]
    owner = dist.block_owner(msizes, world)
    span = max(sum(w[i] for i in range(len(w)) if owner[i] == r) for r in range(world))
    best = min(max(sum(w[i] for i in range(len(w)) if a[i] == r) for r in range(world))
               for a in itertools.product(range(world), repeat=len(w)))
    assert span * 3 * world <= (4 * world - 1) * best


def test_block_shard_bytes_formula(dist):
    """vib3's blocks (13, 12) at world 2: rank 0 owns block 0 (13^3 > 12^3), rank 1 block 1.  Rank 0 saves 23 of the 24
    m x m arrays of block 1 (ld 16) and adds the all-gather buffer (3 chunks of 16 * 13 + 1 doubles), three n_var vectors and
    ten shared values"""
    n = 544
    assert dist.block_owner([13, 12], 2) == [0, 1]
    want0 = (3 * (16 * 13 + 1 + n) + 10) * 8 - 23 * 16 * 12 * 8
    want1 = (3 * (16 * 13 + 1 + n) + 10) * 8 - 23 * 16 * 13 * 8
    assert dist.block_shard_bytes([13, 12], n, 0, 2) == want0
    assert dist.block_shard_bytes([13, 12], n, 1, 2) == want1
    # world 3 with two blocks: rank 2 owns nothing and saves both blocks' state
    want2 = (4 * (16 * 13 + 1 + n) + 10) * 8 - 23 * (16 * 13 + 16 * 12) * 8
    assert dist.block_shard_bytes([13, 12], n, 2, 3) == want2
    # 8 blocks of side 2000 on 4 ranks: two blocks each; every rank keeps 2 of 8 blocks' full state
    mm = 2000 * 2000
    assert dist.block_shard_bytes([2000] * 8, 10000, 1, 4) == (5 * (2 * mm + 1 + 10000) + 40) * 8 - 6 * 23 * mm * 8
    # the saving outgrows the buffers as soon as a rank owns less than all blocks of a large model
    assert dist.block_shard_bytes([2000] * 8, 10000, 0, 2) < 0
