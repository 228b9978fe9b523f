"""CPU, gloo: the partitions and the reduce-scatter layout of the sharded CC_Matrix_Multiplication
(parallel.sharded_cc_matrix_multiplication).  The grouped mod-q sum runs as a numpy stand-in here (the CUDA kernel
ckks_add_many_grouped needs a GPU; tests/test_gpu_sharded_matmul.py covers it)."""
import importlib
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = "seal-fyp-logistic-regression_b200"
Q = [(1 << 60) - 93, (1 << 40) - 87]       # two moduli of the sizes the chains use (any value below 2^61 works)


def _grouped_sum_mod(x, groups, q):
    """numpy stand-in for ckks_add_many_grouped: out[m] = sum_g x[g * M + m] mod q (exact, Python integers)"""
    M = x.shape[0] // groups
    out = np.zeros((M,) + x.shape[1:], dtype=object)
    for g in range(groups):
        out = out + x[g * M:(g + 1) * M].astype(object)
    return (out % q).astype(np.uint64)


def _worker(rank, world, port, ret):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        par = importlib.import_module(PKG + ".parallel")
        ex = par.TorchExchange()
        assert (ex.rank, ex.world) == (rank, world)
        ok = []
        for d in (8, 12, 64):
            K, words = d - 1, 16
            counts = [len(par.owned_block(K, q, world)) for q in range(world)]
            own = par.owned_block(K, rank, world)
            for q in Q:
                rng = np.random.default_rng(d * 7 + q % 1000)        # same stream on every rank
                parts = rng.integers(0, q, size=(world, K, 2, words), dtype=np.uint64)   # rank g's partial of every k
                mine = torch.from_numpy(parts[rank].view(np.int64).copy())
                recv = ex.all_to_all(mine, counts, [len(own)] * world).numpy().view(np.uint64)
                assert recv.shape[0] == world * len(own)
                got = _grouped_sum_mod(recv, world, q)
                want = (parts.astype(object).sum(axis=0) % q).astype(np.uint64)[own.start:own.stop]
                ok.append(bool(np.array_equal(got, want)))
                # the all-gather of the other two exchanges: rank-major
                g = ex.all_gather(torch.from_numpy(parts[rank, :1].view(np.int64).copy())).numpy().view(np.uint64)
                ok.append(bool(np.array_equal(g, parts[:, 0])))
        ret[rank] = all(ok)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_reduce_scatter_layout_gloo(world):
    """all-to-all of the stacked per-k partials + grouped mod-q sum = the per-k sums over all ranks, for even and uneven
    splits of the d-1 products (d - 1 = 7, 11, 63 over 2 and 3 ranks)"""
    mgr = mp.Manager()
    ret = mgr.dict()
    port = 31500 + (os.getpid() % 2000) + 10 * world
    mp.spawn(_worker, args=(world, port, ret), nprocs=world, join=True)
    assert len(ret) == world and all(ret[r] for r in range(world))


@pytest.mark.parametrize("world", [1, 2, 3, 4, 8])
def test_rotation_shares_partition_the_d_squared_rotations(world):
    par = importlib.import_module(PKG + ".parallel")
    for d in (8, 16, 64):
        dd = d * d
        parts = [par.shard_rotations_shared(list(range(dd)), r, world) for r in range(world)]
        owners = np.zeros(dd, dtype=int)
        for p in parts:
            owners[p] += 1
        assert (owners == 1).all(), (d, world)
        assert all(p == sorted(p) for p in parts)


@pytest.mark.parametrize("world", [1, 2, 3, 4, 8])
def test_owned_blocks_partition_the_products(world):
    """K_r: contiguous blocks of k = 1..d-1, sizes differing by at most one, in rank order"""
    par = importlib.import_module(PKG + ".parallel")
    for d in (2, 5, 8, 16, 64):
        blocks = [par.owned_block(d - 1, r, world) for r in range(world)]
        ks = [k + 1 for b in blocks for k in b]
        assert ks == list(range(1, d)), (d, world)
        sizes = [len(b) for b in blocks]
        assert max(sizes) - min(sizes) <= 1 and sizes == sorted(sizes, reverse=True)

