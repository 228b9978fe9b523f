"""CPU, gloo: the partition of the sharded config-1 training iteration (parallel.config1_shards) and the broadcast that
hands rank 0's pred - labels and refreshed weights to the other ranks (TorchExchange.broadcast).  The iteration itself
needs a GPU; tests/test_gpu_sharded_lr.py covers it."""
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
SHAPES = [(2000, 8), (16, 4), (3, 8), (1, 1), (7, 2)]


def _covered_once(blocks, n):
    owners = np.zeros(n, dtype=int)
    for b in blocks:
        owners[list(b)] += 1
    return bool((owners == 1).all())


def _worker(rank, world, port, ret):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        par = importlib.import_module(PKG + ".parallel")
        ex = par.TorchExchange()
        ok = [(ex.rank, ex.world) == (rank, world)]
        for R, C in SHAPES:
            mine = [(b.start, b.stop) for b in par.config1_shards(R, C, rank, world)]
            everyone = [None] * world
            dist.all_gather_object(everyone, mine)          # what every rank computed for itself
            rows = [range(*e[0]) for e in everyone]
            feats = [range(*e[1]) for e in everyone]
            ok.append(_covered_once(rows, R) and _covered_once(feats, C))
            ok.append(all(e == [(b.start, b.stop) for b in par.config1_shards(R, C, q, world)]
                          for q, e in enumerate(everyone)))
        for shape, dtype in (((1, 2, 3, 16), torch.int64), ((4,), torch.float64)):
            want = torch.arange(int(np.prod(shape)), dtype=dtype).reshape(shape) * 7 + 1
            t = want.clone() if rank == 0 else torch.zeros(shape, dtype=dtype)
            got = ex.broadcast(t)
            ok.append(torch.equal(got, want))
        ret[rank] = ok
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_partition_and_broadcast_gloo(world):
    """every rank computes the same blocks for every rank, they cover each row and feature once, and the broadcast
    delivers rank 0's tensor (ciphertext words and the float64 header) everywhere"""
    mgr = mp.Manager()
    ret = mgr.dict()
    port = 32500 + (os.getpid() % 2000) + 10 * world
    mp.spawn(_worker, args=(world, port, ret), nprocs=world, join=True)
    assert len(ret) == world
    for r in range(world):
        assert all(ret[r]), (r, ret[r])


@pytest.mark.parametrize("world", [1, 2, 3, 4, 8, 9, 16])
def test_config1_shards_cover_rows_and_features_once(world):
    par = importlib.import_module(PKG + ".parallel")
    for R, C in SHAPES:
        blocks = [par.config1_shards(R, C, r, world) for r in range(world)]
        rows, feats = [b[0] for b in blocks], [b[1] for b in blocks]
        assert _covered_once(rows, R) and _covered_once(feats, C), (R, C, world)
        for part, n in ((rows, R), (feats, C)):
            sizes = [len(b) for b in part]
            assert [i for b in part for i in b] == list(range(n))            # contiguous, in rank order
            assert max(sizes) - min(sizes) <= 1 and sizes == sorted(sizes, reverse=True)
        assert blocks == [par.config1_shards(R, C, r, world) for r in range(world)]    # deterministic


def test_config1_shards_more_ranks_than_features_or_rows():
    par = importlib.import_module(PKG + ".parallel")
    feats = [len(par.config1_shards(2000, 8, r, 16)[1]) for r in range(16)]
    assert feats == [1] * 8 + [0] * 8                                        # ranks 8..15 add a zero gradient partial
    rows = [len(par.config1_shards(3, 8, r, 4)[0]) for r in range(4)]
    assert rows == [1, 1, 1, 0]                                              # rank 3 adds a zero prediction partial


def test_config1_keyswitches_add_up_to_one_gpu():
    """per-rank key switches summed over the ranks equal the one-GPU count at every world size: 2000 x 9 row key
    switches, 8 x (1 + 3 + 1999) feature key switches (rotating by -2000 = NAF -2048 + 64 - 16 costs 3) and the 3
    relinearisations of the Horner polynomial"""
    par = importlib.import_module(PKG + ".parallel")
    one = par.config1_keyswitches(2000, 8, 0, 1)
    assert one == 2000 * 9 + 8 * 2003 + 3 == 34027
    for world in (2, 3, 4, 8, 16):
        assert sum(par.config1_keyswitches(2000, 8, r, world) for r in range(world)) == one
    assert [par.config1_keyswitches(2000, 8, r, 8) for r in range(8)] == [4256] + [4253] * 7
