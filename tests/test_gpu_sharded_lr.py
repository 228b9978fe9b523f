"""GPU: the sharded config-1 training iteration (parallel.sharded_update_weights) and training loop
(parallel.sharded_train_cipher), bit-identical to the one-GPU lr.update_weights / lr.train_cipher.

World sizes 1, 2, 3, 4 and 8 are emulated in one process with the exchange of test_gpu_sharded_matmul.py (ranks run
one after the other on one GPU, each up to its next collective), extended by a broadcast.  A real NCCL run covers 2
ranks (4 and 8 where that many GPUs are visible)."""
import importlib
import json
import os
import sys

import numpy as np
import pytest
import torch

from test_gpu_sharded_matmul import EmulatedExchange, _same

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = "seal-fyp-logistic-regression_b200"
CHAIN = [60] + [40] * 8 + [60]
POW2 = [s for i in range(13) for s in (1 << i, -(1 << i))]
SCALE, LR = 2.0 ** 40, 0.1


def _mods():
    return tuple(importlib.import_module(PKG + m) for m in (".lr", ".parallel", ".client", ".params"))


class BroadcastingExchange(EmulatedExchange):
    """the emulated collectives plus broadcast: every rank gets its own copy of rank src's tensor"""

    def for_rank(self, rank):
        view, ex = super().for_rank(rank), self
        view.broadcast = lambda t, src=0: ex._collective(rank, t, lambda s: [s[src].clone() for _ in range(ex.world)])
        return view


@pytest.fixture(scope="module")
def he(eng):
    """N = 2^15, {60, 40 x 8, 60}: one Horner degree-3 iteration uses every level; power-of-two Galois keys"""
    lr, par, client, params = _mods()
    ctx = eng.Context(15, params.coeff_modulus_create(15, CHAIN))
    kg = client.KeyGenerator(ctx, seed=31)
    return dict(ctx=ctx, ev=eng.Evaluator(ctx), enc=client.CKKSEncoder(ctx), keys=kg.keyset(steps=POW2), pk=kg.public_key(),
                decr=client.Decryptor(ctx, kg.secret_key()))


def _encrypt(he, X, y, w0, seed):
    lr, _, client, _ = _mods()
    R, C = X.shape
    lay = lr.RowLayout(R, C, he["ctx"].n // 2)
    enc, encr = he["enc"], client.Encryptor(he["ctx"], he["pk"], seed=seed)
    return lay, [encr.encrypt(enc.encode(v, SCALE)) for v in (lay.rows(X), lay.columns(X), lay.labels(y), lay.weights(w0))]


def _data(R, C, seed):
    rng = np.random.default_rng(seed)
    return rng.normal(0, 1, (R, C)), (rng.uniform(0, 1, R) > 0.5).astype(float), rng.uniform(-1, 1, C)


def _run_sharded(he, cts, R, C, world, poly_seed, train=None):
    """every emulated rank gets its own row / feature blocks only; rank 0 alone holds an encryptor (and the decryptor)"""
    _, par, client, _ = _mods()
    rows, cols, labs, wct = cts

    def fn(r, ex):
        rb, fb = par.config1_shards(R, C, r, world)
        encr = client.Encryptor(he["ctx"], he["pk"], seed=poly_seed) if r == 0 else None
        args = (he["ev"], rows[rb.start:rb.stop], list(rb), cols[fb.start:fb.stop], list(fb), labs, wct, LR)
        if train is None:
            return par.sharded_update_weights(*args, R, C, SCALE, he["keys"], he["enc"], encr, r, world, ex)
        lay, iters = train
        return par.sharded_train_cipher(*args, iters, lay, SCALE, he["keys"], he["enc"], encr, he["decr"] if r == 0 else None,
                                        r, world, ex)
    return BroadcastingExchange(world).run(fn)


@pytest.mark.parametrize("R,C,worlds", [(12, 4, (1, 2, 3, 4, 8)), (32, 8, (1, 2, 3, 4, 8)), (6, 4, (8,))])
def test_emulated_sharded_update_weights_is_bit_identical(he, R, C, worlds):
    """world 8 > C = 4: four ranks own no feature; world 8 > R = 6: two ranks own no row (zero partials)"""
    lr, _, client, _ = _mods()
    X, y, w0 = _data(R, C, seed=R + C)
    _, cts = _encrypt(he, X, y, w0, seed=40 + R)
    want = lr.update_weights(he["ev"], *cts, LR, SCALE, he["keys"], he["enc"],
                             client.Encryptor(he["ctx"], he["pk"], seed=41 + R))
    dec = he["enc"].decode(he["decr"].decrypt(want))[0, :C]
    assert np.abs(dec - lr.plain_epoch(X, y, w0, LR, 3)).max() < 1e-3
    for world in worlds:
        got = _run_sharded(he, cts, R, C, world, poly_seed=41 + R)
        for r in range(world):
            assert _same(got[r], want), (R, C, world, r)


@pytest.mark.parametrize("world", [2, 3])
def test_emulated_sharded_train_cipher_is_bit_identical(he, world):
    """two iterations with rank 0 refreshing the weights in between, against lr.train_cipher with the same seeds, and
    against two plaintext steps (as test_train_cipher_two_iterations)"""
    lr, _, client, _ = _mods()
    R, C = 8, 4
    X, y, w0 = _data(R, C, seed=23)
    lay, cts = _encrypt(he, X, y, w0, seed=50)
    want = lr.train_cipher(he["ev"], *cts, LR, 2, lay, SCALE, he["keys"], he["enc"],
                           client.Encryptor(he["ctx"], he["pk"], seed=51), he["decr"])
    got = _run_sharded(he, cts, R, C, world, poly_seed=51, train=(lay, 2))
    for r in range(world):
        assert got[r].limbs == he["ctx"].top_limbs and _same(got[r], want), (world, r)
    plain = w0
    for _ in range(2):
        plain = lr.plain_epoch(X, y, plain, LR, 3)
    assert np.abs(he["enc"].decode(he["decr"].decrypt(got[0]))[0, :C] - plain).max() < 1e-3


def test_emulated_sharded_pulsar_real_data(he):
    """config 1 itself: the 2000 x 8 pulsar rows, the reference program's initial weights, emulated world size 2"""
    lr, _, client, _ = _mods()
    pulsar = importlib.import_module(PKG + ".pulsar")
    with open(os.path.join(ROOT, "tests", "golden", "pulsar_plain_lr.json")) as fh:
        w0 = np.array(json.load(fh)["initial_weights"])
    X, y = pulsar.load_csv()
    X, y = pulsar.standard_scaler(X).astype(np.float64), y.astype(np.float64)
    R, C = X.shape
    _, cts = _encrypt(he, X, y, w0, seed=72)
    want = lr.update_weights(he["ev"], *cts, LR, SCALE, he["keys"], he["enc"], client.Encryptor(he["ctx"], he["pk"], seed=73))
    got = _run_sharded(he, cts, R, C, 2, poly_seed=73)
    assert _same(got[0], want) and _same(got[1], want)
    dec = he["enc"].decode(he["decr"].decrypt(got[1]))[0, :C]
    assert np.abs(dec - lr.plain_epoch(X, y, w0, LR, 3)).max() < 1e-3


def _nccl_worker(rank, world, port, ret):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        eng = importlib.import_module(PKG).load_engine()
        lr, par, client, params = _mods()
        R, C = 16, 4
        ctx = eng.Context(15, params.coeff_modulus_create(15, CHAIN), device=rank)
        kg = client.KeyGenerator(ctx, seed=61)                   # same keys and inputs on every rank
        he = dict(ctx=ctx, ev=eng.Evaluator(ctx), enc=client.CKKSEncoder(ctx), keys=kg.keyset(steps=POW2[:12]),
                  pk=kg.public_key())
        X, y, w0 = _data(R, C, seed=62)
        _, (rows, cols, labs, wct) = _encrypt(he, X, y, w0, seed=63)
        rb, fb = par.config1_shards(R, C, rank, world)
        encr = client.Encryptor(ctx, he["pk"], seed=64) if rank == 0 else None
        got = par.sharded_update_weights(he["ev"], rows[rb.start:rb.stop], list(rb), cols[fb.start:fb.stop], list(fb), labs,
                                         wct, LR, R, C, SCALE, he["keys"], he["enc"], encr, rank, world, par.TorchExchange())
        want = lr.update_weights(he["ev"], rows, cols, labs, wct, LR, SCALE, he["keys"], he["enc"],
                                 client.Encryptor(ctx, he["pk"], seed=64))
        dec = he["enc"].decode(client.Decryptor(ctx, kg.secret_key()).decrypt(got))[0, :C]
        ret[rank] = (_same(got, want), float(np.abs(dec - lr.plain_epoch(X, y, w0, LR, 3)).max()))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4, 8])
def test_nccl_sharded_update_weights_is_bit_identical(eng, world):
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs, %d visible" % (world, torch.cuda.device_count()))
    mgr = mp.Manager()
    ret = mgr.dict()
    port = 35500 + (os.getpid() % 2000) + 10 * world
    mp.spawn(_nccl_worker, args=(world, port, ret), nprocs=world, join=True)
    assert len(ret) == world
    for r in range(world):
        same, err = ret[r]
        assert same, r
        assert err < 1e-3, (r, err)
