"""GPU: the grouped fused product-sum (ckks_multiply_sum_grouped / Evaluator.multiply_sum_grouped) and column-layout
encrypted LR with the Chebyshev sigmoid (lr.column_epoch_gradient(method="chebyshev"), lr.train_columns,
parallel.sharded_train_columns).

The kernel is bit-identical to SEAL's multiply + add_many per group; the column epoch is bit-identical to a sequential
restatement on the CPU oracle; the pulsar steps and the training loop are checked against plaintext Chebyshev LR and the
reference program's weights; the sharded loop is compared with torch.equal against the one-GPU loop, with world sizes
emulated in one process and, where 2 or more GPUs are visible, over NCCL."""
import ctypes
import importlib
import json
import os
import sys

import numpy as np
import pytest
import torch

import ref_workloads as rw
from test_gpu_chebyshev import _oracle_chebyshev
from test_gpu_sharded_lr import BroadcastingExchange
from test_gpu_sharded_matmul import _same
from test_gpu_workloads import Bridge, _enc

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = "seal-fyp-logistic-regression_b200"
CHAIN12 = [60] + [40] * 11 + [60]                 # column layout with the degree-63 Chebyshev sigmoid: 11 rescales
POW2 = [s for i in range(13) for s in (1 << i, -(1 << i))]
SCALE, LR = 2.0 ** 40, 0.1


def _mods():
    return tuple(importlib.import_module(PKG + m) for m in (".workloads", ".lr", ".parallel", ".client", ".params", ".capi"))


# ------------------------------------------------------------------ the kernel
KERNEL_CASES = [(12, [50, 40, 40, 50]), (15, [60, 40, 40, 40, 60])]    # 50 / 60-bit primes: 128-bit path, 40-bit: FP64


@pytest.mark.parametrize("log_n,bits", KERNEL_CASES)
@pytest.mark.parametrize("T,G", [(1, 1), (8, 1), (8, 16), (3, 5)])
def test_multiply_sum_grouped_bit_identical_to_seal_sequence(make_fixture, log_n, bits, T, G):
    fx = make_fixture(log_n, bits)
    ev = fx.ev
    rng = np.random.default_rng(log_n * 100 + T * 10 + G)
    for limbs in range(1, len(bits)):
        a = fx.ctx.upload(fx.random_ct(rng, G * T, 2, limbs))
        b = fx.ctx.upload(fx.random_ct(rng, T, 2, limbs))
        got = ev.multiply_sum_grouped(a, b, G)
        assert got.batch == G and got.size == 3 and got.limbs == limbs
        want = np.stack([ev.add_many(ev.multiply(a[g * T:(g + 1) * T], b)).numpy()[0] for g in range(G)])
        assert np.array_equal(got.numpy(), want), limbs
        if G == 1:
            assert np.array_equal(got.numpy(), ev.multiply_sum(a, b).numpy()), limbs


def test_multiply_sum_grouped_rejections(make_fixture):
    fx = make_fixture(*KERNEL_CASES[0])
    _, _, _, _, _, capi = _mods()
    ev, ctx = fx.ev, fx.ctx
    rng = np.random.default_rng(3)
    a = ctx.upload(fx.random_ct(rng, 6, 2, 3))
    b = ctx.upload(fx.random_ct(rng, 3, 2, 3))

    def raw(a, b, groups, out=None, vo=None):
        vo = (ctx.empty(max(groups, 1), 3, a.limbs) if out is None else out).view() if vo is None else vo
        va, vb = a.view(), b.view()
        return ctx.lib.ckks_multiply_sum_grouped(ev.h, ctypes.byref(va), ctypes.byref(vb), groups, ctypes.byref(vo), None)
    assert raw(a, b, 2) == capi.CKKS_OK
    assert raw(a, b, 0) == capi.CKKS_ERR_INVALID                                             # groups < 1
    assert raw(a, b, -1) == capi.CKKS_ERR_INVALID
    assert raw(a, b, 3) == capi.CKKS_ERR_INVALID                                             # 6 != 3 x 3
    assert raw(a, b[0:2], 2) == capi.CKKS_ERR_INVALID                                        # 6 != 2 x 2
    assert raw(a, ctx.upload(fx.random_ct(rng, 3, 2, 2)), 2) == capi.CKKS_ERR_INVALID       # limbs
    assert raw(a, b, 2, out=ctx.empty(2, 3, 2)) == capi.CKKS_ERR_INVALID                    # out limbs
    assert raw(a, b, 2, out=ctx.empty(3, 3, 3)) == capi.CKKS_ERR_INVALID                    # out batch
    assert raw(a, b, 2, out=ctx.empty(2, 2, 3)) == capi.CKKS_ERR_INVALID                    # out size
    assert raw(ctx.upload(fx.random_ct(rng, 6, 3, 3)), b, 2) == capi.CKKS_ERR_INVALID       # a size
    assert raw(a, ctx.upload(fx.random_ct(rng, 3, 3, 3)), 2) == capi.CKKS_ERR_INVALID       # b size
    a1, b1 = a[0:3], b

    def alias(ct):
        v = ct.view()
        v.batch, v.size = 1, 3
        return v
    assert raw(a1, b1, 1) == capi.CKKS_OK
    assert raw(a1, b1, 1, vo=alias(a1)) == capi.CKKS_ERR_INVALID                             # out aliases a
    assert raw(a1, b1, 1, vo=alias(b1)) == capi.CKKS_ERR_INVALID                             # out aliases b
    with pytest.raises(capi.CkksInvalidArgument):
        ev.multiply_sum_grouped(a, b, 4)
    with pytest.raises(capi.CkksInvalidArgument):
        ev.multiply_sum_grouped(a, b, 0)
    big = ctx.upload(fx.random_ct(rng, 6, 2, 3), scale=2.0 ** 100)
    with pytest.raises(capi.CkksInvalidArgument, match="scale out of bounds"):
        ev.multiply_sum_grouped(big, ctx.upload(fx.random_ct(rng, 3, 2, 3), scale=2.0 ** 100), 2)


# ------------------------------------------------------------------ the column epoch vs the CPU oracle
def _oracle_column_epoch(fx, wl, E, cols, labs, wb, C, B, coeffs, scale, encode):
    """column_epoch_gradient(method="chebyshev") restated one oracle op at a time: ref_workloads.column_epoch_gradient
    with the prediction's scale kept as it is and the sigmoid replaced by the oracle restatement of chebyshev_cipher"""
    grads = []
    for m in range(len(labs)):
        z = E.rescale(E.relinearize(E.add_many([E.multiply(cols[m * C + j], wb[j]) for j in range(C)])))
        data, sc = _oracle_chebyshev(wl, fx.orc, fx.rlk, z.data, z.scale, coeffs, scale)
        pred = rw.OCt(data, sc)
        lab = E.mod_switch_to(labs[m], pred.limbs)
        pred.scale = lab.scale
        pl = E.sub(pred, lab)
        for j in range(C):
            g = rw.cipher_dot_product(E, E.mod_switch_to(cols[m * C + j], pl.limbs), pl, B)
            mask = np.zeros(C)
            mask[j] = 1.0
            grads.append(E.multiply_plain(g, encode(mask, scale, g.limbs)))
    gradient = E.rescale(E.add_many(grads))
    gradient.scale = rw.pow2(gradient.scale)
    return gradient


def test_column_chebyshev_epoch_bit_exact_vs_oracle(make_fixture):
    """N = 2^14, R = 64, C = 4, B = 16 (M = 4), degree-15 Chebyshev sigmoid on [-8, 8]: 1 + 5 + 3 levels"""
    wl, lr = _mods()[:2]
    sig = lr.ChebyshevSigmoid(15, 8.0)
    fx = make_fixture(14, [50] + [40] * 9 + [50], steps=(1, -16))
    assert fx.L == lr.column_rescales("chebyshev", sigmoid=sig) + 1
    E, br = rw.OEval(fx.orc, fx.rlk, fx.gks), Bridge(fx)
    rng = np.random.default_rng(64)
    R, C, B = 64, 4, 16
    X, y, w0 = rng.normal(0, 1, (R, C)), (rng.uniform(0, 1, R) > 0.5).astype(float), rng.uniform(-1, 1, C)
    lay = lr.ColumnLayout(R, C, B, fx.n // 2)
    cols = np.stack([_enc(fx, 700 + i, v, SCALE) for i, v in enumerate(lay.columns(X))])
    labs = np.stack([_enc(fx, 770 + i, v, SCALE) for i, v in enumerate(lay.labels(y))])
    wb = np.stack([_enc(fx, 780 + j, v, SCALE) for j, v in enumerate(lay.weight_broadcasts(w0, "chebyshev", sig))])
    wct = _enc(fx, 790, lay.weights(w0), SCALE)
    up = lambda a: fx.ctx.upload(a, scale=SCALE)                               # noqa: E731

    grad = lr.column_epoch_gradient(fx.ev, up(cols), up(labs), up(wb), C, B, SCALE, fx.keys, br, None, method="chebyshev",
                                    sigmoid=sig)
    neww = lr.apply_gradient(fx.ev, grad, up(wct), LR, R, SCALE, br)
    ograd = _oracle_column_epoch(fx, wl, E, [rw.OCt(c, SCALE) for c in cols], [rw.OCt(c, SCALE) for c in labs],
                                 [rw.OCt(c, SCALE) for c in wb], C, B, sig.coeffs, SCALE, br.o_encode)
    oneww = rw.apply_gradient(E, ograd, rw.OCt(wct, SCALE), LR, R, SCALE, br.o_encode)
    assert (grad.limbs, grad.scale) == (ograd.limbs, ograd.scale)
    assert np.array_equal(grad.numpy()[0], ograd.data)
    assert (neww.limbs, neww.scale) == (oneww.limbs, oneww.scale) and neww.limbs == 1
    assert np.array_equal(neww.numpy()[0], oneww.data)
    got = fx.orc.decode(fx.orc.decrypt(fx.sk, neww.numpy()[0]), neww.scale)[:C]
    assert np.abs(got - lr.plain_epoch(X, y, w0, LR, method="chebyshev", sigmoid=sig)).max() < 1e-4


# ------------------------------------------------------------------ pulsar on N = 2^15, {60, 40 x 11, 60}
@pytest.fixture(scope="module")
def he12(eng):
    _, _, _, client, params, _ = _mods()
    ctx = eng.Context(15, params.coeff_modulus_create(15, CHAIN12))
    kg = client.KeyGenerator(ctx, seed=121)
    return dict(ctx=ctx, ev=eng.Evaluator(ctx), enc=client.CKKSEncoder(ctx), keys=kg.keyset(steps=POW2), pk=kg.public_key(),
                decr=client.Decryptor(ctx, kg.secret_key()), client=client)


def _pulsar():
    pulsar = importlib.import_module(PKG + ".pulsar")
    with open(os.path.join(ROOT, "tests", "golden", "pulsar_plain_lr.json")) as fh:
        gold = json.load(fh)
    X, y = pulsar.load_csv()
    return gold, pulsar.standard_scaler(X).astype(np.float64), y.astype(np.float64)


def _encrypt(he, X, y, w0, B, seed):
    """-> layout, [cols, labels, packed weights, weight broadcasts] (Chebyshev broadcasts), one encryptor"""
    lr = _mods()[1]
    lay = lr.ColumnLayout(X.shape[0], X.shape[1], B, he["ctx"].n // 2)
    enc, encr = he["enc"], he["client"].Encryptor(he["ctx"], he["pk"], seed=seed)
    vals = (lay.columns(X), lay.labels(y), lay.weights(w0), lay.weight_broadcasts(w0, "chebyshev"))
    return lay, [encr.encrypt(enc.encode(v, SCALE)) for v in vals]


def _decode_w(he, ct, C):
    return he["enc"].decode(he["decr"].decrypt(ct))[0, :C]


@pytest.mark.parametrize("B", [2000, 250])
def test_pulsar_column_chebyshev_one_step(he12, B):
    """one encrypted step from the reference's initial weights: within 1e-4 of the plaintext Chebyshev step and 1e-3 of
    the reference program's weights_after_iteration_0; the iteration ends at one limb"""
    lr = _mods()[1]
    gold, X, y = _pulsar()
    w0 = np.array(gold["initial_weights"])
    lay, (cols, labs, wct, wb) = _encrypt(he12, X, y, w0, B, seed=200 + B)
    grad = lr.column_epoch_gradient(he12["ev"], cols, labs, wb, lay.C, B, SCALE, he12["keys"], he12["enc"], None,
                                    method="chebyshev")
    neww = lr.apply_gradient(he12["ev"], grad, wct, LR, lay.R, SCALE, he12["enc"])
    assert neww.limbs == 1
    dec = _decode_w(he12, neww, lay.C)
    assert np.abs(dec - lr.plain_epoch(X, y, w0, LR, method="chebyshev")).max() < 1e-4
    assert np.abs(dec - np.array(gold["weights_after_iteration_0"])).max() < 1e-3


def test_pulsar_train_columns_three_iterations(he12):
    lr = _mods()[1]
    gold, X, y = _pulsar()
    w0 = np.array(gold["initial_weights"])
    lay, (cols, labs, wct, wb) = _encrypt(he12, X, y, w0, 250, seed=300)
    encr = he12["client"].Encryptor(he12["ctx"], he12["pk"], seed=301)
    wct, wb = lr.train_columns(he12["ev"], cols, labs, wct, wb, LR, 3, lay, SCALE, he12["keys"], he12["enc"], encr,
                               he12["decr"], method="chebyshev")
    top = he12["ctx"].top_limbs
    assert wct.limbs == top and wb.limbs == top and wb.batch == lay.C
    plain = w0
    for _ in range(3):
        plain = lr.plain_epoch(X, y, plain, LR, method="chebyshev")
    assert np.abs(_decode_w(he12, wct, lay.C) - plain).max() < 1e-4
    bc = he12["enc"].decode(he12["decr"].decrypt(wb))[:, :8]
    assert np.abs(bc - plain[:, None] / lr.SIGMOID_CHEBYSHEV.bound).max() < 1e-6


# ------------------------------------------------------------------ the sharded loop
def _shard(cols, labs, units, C):
    """the column and label ciphertexts of the mini-batches `units` touch (contiguous), and their indices"""
    ids = sorted({m for m, _ in units})
    lo, hi = (ids[0], ids[-1] + 1) if ids else (0, 0)
    return cols[lo * C:hi * C], labs[lo:hi], ids


def test_emulated_sharded_train_columns_is_bit_identical(he12):
    """R = 64, C = 4, B = 16 (M * C = 16 units), two iterations: world sizes 2, 3, 8 and 17 (one rank without units)
    against lr.train_columns with the same seeds, on every rank"""
    lr, par = _mods()[1:3]
    R, C, B = 64, 4, 16
    rng = np.random.default_rng(17)
    X, y, w0 = rng.normal(0, 1, (R, C)), (rng.uniform(0, 1, R) > 0.5).astype(float), rng.uniform(-1, 1, C)
    lay, (cols, labs, wct, wb) = _encrypt(he12, X, y, w0, B, seed=400)
    client = he12["client"]
    want = lr.train_columns(he12["ev"], cols, labs, wct, wb, LR, 2, lay, SCALE, he12["keys"], he12["enc"],
                            client.Encryptor(he12["ctx"], he12["pk"], seed=401), he12["decr"], method="chebyshev")
    plain = w0
    for _ in range(2):
        plain = lr.plain_epoch(X, y, plain, LR, method="chebyshev")
    assert np.abs(_decode_w(he12, want[0], C) - plain).max() < 1e-4
    for world in (2, 3, 8, lay.M * C + 1):
        def fn(r, ex):
            units = par.column_units(lay.M, C, r, world)
            c, l, ids = _shard(cols, labs, units, C)
            encr = client.Encryptor(he12["ctx"], he12["pk"], seed=401) if r == 0 else None
            return par.sharded_train_columns(he12["ev"], c, l, ids, units, wct, wb, LR, 2, lay, SCALE, he12["keys"],
                                             he12["enc"], encr, he12["decr"] if r == 0 else None, r, world, ex)
        got = BroadcastingExchange(world).run(fn)
        for r in range(world):
            assert _same(got[r][0], want[0]) and _same(got[r][1], want[1]), (world, r)


def _nccl_worker(rank, world, port, ret):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        eng = importlib.import_module(PKG).load_engine()
        _, lr, par, client, params, _ = _mods()
        ctx = eng.Context(15, params.coeff_modulus_create(15, CHAIN12), device=rank)
        kg = client.KeyGenerator(ctx, seed=131)                  # same keys and inputs on every rank
        he = dict(ctx=ctx, ev=eng.Evaluator(ctx), enc=client.CKKSEncoder(ctx), keys=kg.keyset(steps=POW2), pk=kg.public_key(),
                  decr=client.Decryptor(ctx, kg.secret_key()), client=client)
        R, C, B = 32, 4, 8
        rng = np.random.default_rng(32)
        X, y, w0 = rng.normal(0, 1, (R, C)), (rng.uniform(0, 1, R) > 0.5).astype(float), rng.uniform(-1, 1, C)
        lay, (cols, labs, wct, wb) = _encrypt(he, X, y, w0, B, seed=500)
        units = par.column_units(lay.M, C, rank, world)
        c, l, ids = _shard(cols, labs, units, C)
        encr = client.Encryptor(ctx, he["pk"], seed=501) if rank == 0 else None
        got = par.sharded_train_columns(he["ev"], c, l, ids, units, wct, wb, LR, 2, lay, SCALE, he["keys"], he["enc"], encr,
                                        he["decr"] if rank == 0 else None, rank, world, par.TorchExchange())
        want = lr.train_columns(he["ev"], cols, labs, wct, wb, LR, 2, lay, SCALE, he["keys"], he["enc"],
                                client.Encryptor(ctx, he["pk"], seed=501), he["decr"], method="chebyshev")
        plain = w0
        for _ in range(2):
            plain = lr.plain_epoch(X, y, plain, LR, method="chebyshev")
        ret[rank] = (_same(got[0], want[0]) and _same(got[1], want[1]),
                     float(np.abs(_decode_w(he, got[0], C) - plain).max()))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4, 8])
def test_nccl_sharded_train_columns_is_bit_identical(eng, world):
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs, %d visible" % (world, torch.cuda.device_count()))
    mgr = mp.Manager()
    ret = mgr.dict()
    port = 37500 + (os.getpid() % 2000) + 10 * world
    mp.spawn(_nccl_worker, args=(world, port, ret), nprocs=world, join=True)
    assert len(ret) == world
    for r in range(world):
        same, err = ret[r]
        assert same, r
        assert err < 1e-4, (r, err)
