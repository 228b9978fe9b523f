"""GPU: the ciphertext matrix product (ckks_multiply_sum_matrix / Evaluator.multiply_sum_matrix) and the blocked encrypted
matrix product (workloads.cc_matrix_multiplication_blocked, parallel.sharded_cc_matrix_multiplication_blocked).

The kernel equals multiply + add_many word for word.  Every output tile of the blocked product equals word for word the
sum over l of the per-tile products (cc_matrix_multiplication_sparse for method="reference",
cc_matrix_multiplication_nonzero_hoisted for method="hoisted"), and decrypts to A B.  The sharded form is compared with
the one-GPU call on every rank, with world sizes emulated in one process and, where that many GPUs are visible, NCCL."""
import ctypes
import importlib
import os
import sys

import numpy as np
import pytest
import torch

from test_gpu_sharded_matmul import POW2_14, EmulatedExchange

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = "seal-fyp-logistic-regression_b200"
SCALE, EPS = 2.0 ** 40, 1e-8
CHAIN4 = [60, 40, 40, 40, 40, 60]


def _mods():
    return tuple(importlib.import_module(PKG + m) for m in (".workloads", ".parallel", ".client", ".params", ".capi"))


def _same(a, b):
    return (a.batch, a.size, a.limbs, a.scale) == (b.batch, b.size, b.limbs, b.scale) and torch.equal(
        a.data[:, :, :a.limbs], b.data[:, :, :b.limbs])


# ------------------------------------------------------------------ the kernel
def _restated(ev, a, b, rows, inner, cols):
    """multiply + add_many per output"""
    outs = []
    for i in range(rows):
        for j in range(cols):
            bj = type(b)(b.ctx, b.data[j::cols].contiguous(), b.limbs, b.scale)
            outs.append(ev.add_many(ev.multiply(a[i * inner:(i + 1) * inner], bj)).data[:, :, :a.limbs])
    return torch.cat(outs)


# data limbs with 50- and 60-bit primes (128-bit path) and 40-bit primes (FP64 path)
KERNEL_CASES = [(12, [50, 40, 40, 50]), (13, [60, 40, 60])]


@pytest.mark.parametrize("log_n,bits", KERNEL_CASES)
@pytest.mark.parametrize("rows,inner,cols", [(1, 1, 2), (1, 5, 7), (3, 1, 4), (2, 3, 5), (4, 9, 4), (3, 130, 6), (2, 4, 1),
                                             (1, 1, 1)])
def test_multiply_sum_matrix_equals_multiply_add_many(make_fixture, log_n, bits, rows, inner, cols):
    fx = make_fixture(log_n, bits)
    ev = fx.ev
    rng = np.random.default_rng(log_n + 7 * rows + 11 * inner + 13 * cols)
    for limbs in sorted({1, len(bits) - 1}):
        a = fx.ctx.upload(fx.random_ct(rng, rows * inner, 2, limbs))
        b = fx.ctx.upload(fx.random_ct(rng, inner * cols, 2, limbs))
        got = ev.multiply_sum_matrix(a, b, rows, cols)
        assert (got.batch, got.size, got.limbs, got.scale) == (rows * cols, 3, limbs, a.scale * b.scale)
        assert torch.equal(got.data[:, :, :limbs], _restated(ev, a, b, rows, inner, cols)), limbs
        if cols == 1:
            assert torch.equal(got.data[:, :, :limbs], ev.multiply_sum_grouped(a, b, rows).data[:, :, :limbs])


def test_long_sums_at_a_60_bit_prime(make_fixture):
    """inner >= 4096: many reductions of the lazy sums, every residue at p - 1 (the largest products) on limb 0 (60 bits,
    128-bit path) and limb 1 (40 bits, FP64 path)"""
    fx = make_fixture(12, [60, 40, 60])
    ev, ctx = fx.ev, fx.ctx
    rows, inner, cols = 1, 4100, 3
    rng = np.random.default_rng(4100)
    x = fx.random_ct(rng, rows * inner, 2, 2)
    y = fx.random_ct(rng, inner * cols, 2, 2)
    for j in range(2):
        x[:, :, j, :256] = fx.primes[j] - 1
        y[:, :, j, :256] = fx.primes[j] - 1
    a, b = ctx.upload(x), ctx.upload(y)
    got = ev.multiply_sum_matrix(a, b, rows, cols)
    assert torch.equal(got.data[:, :, :2], _restated(ev, a, b, rows, inner, cols))
    # the words at p - 1: sum of inner products (p-1)^2 = inner (mod p) for poly 0 and 2, 2 inner for poly 1
    for j in range(2):
        p = fx.primes[j]
        w = got.numpy()[:, :, j, :256]
        assert (w[:, 0] == inner % p).all() and (w[:, 1] == 2 * inner % p).all() and (w[:, 2] == inner % p).all()


def test_multiply_sum_matrix_rejections(make_fixture):
    fx = make_fixture(*KERNEL_CASES[0])
    capi = _mods()[4]
    ev, ctx = fx.ev, fx.ctx
    rng = np.random.default_rng(5)
    rows, inner, cols, L = 2, 3, 4, 3
    a = ctx.upload(fx.random_ct(rng, rows * inner, 2, L))
    b = ctx.upload(fx.random_ct(rng, inner * cols, 2, L))

    def raw(a, b, r, i, c, out=None, vo=None):
        vo = (ctx.empty(max(r * c, 1), 3, a.limbs) if out is None else out).view() if vo is None else vo
        va, vb = a.view(), b.view()
        return ctx.lib.ckks_multiply_sum_matrix(ev.h, ctypes.byref(va), ctypes.byref(vb), r, i, c, ctypes.byref(vo), None)
    OK, INV = capi.CKKS_OK, capi.CKKS_ERR_INVALID
    assert raw(a, b, rows, inner, cols) == OK
    for r, i, c in ((0, 3, 4), (2, 0, 4), (2, 3, 0), (-1, 3, 4), (2, -3, 4), (2, 3, -4)):
        assert raw(a, b, r, i, c) == INV, (r, i, c)                                          # below 1
    assert raw(a, b, 3, 2, 4) == INV                                                         # a: 6 = rows x inner, b not
    assert raw(a, b, 2, 3, 3) == INV                                                         # b batch != inner x cols
    assert raw(a, b[0:8], 2, 3, 4) == INV
    assert raw(a, b, 2, 3, 4, out=ctx.empty(7, 3, L)) == INV                                 # out batch != rows x cols
    assert raw(a, b, 2, 3, 4, out=ctx.empty(9, 3, L)) == INV
    assert raw(a, ctx.upload(fx.random_ct(rng, 12, 2, 2)), 2, 3, 4) == INV                   # limbs
    assert raw(a, b, 2, 3, 4, out=ctx.empty(8, 3, 2)) == INV                                 # out limbs
    assert raw(a, b, 2, 3, 4, out=ctx.empty(8, 2, L)) == INV                                 # out size
    assert raw(ctx.upload(fx.random_ct(rng, 6, 3, L)), b, 2, 3, 4) == INV                    # a size
    assert raw(a, ctx.upload(fx.random_ct(rng, 12, 3, L)), 2, 3, 4) == INV                   # b size

    def inside(ct, batch_off):
        """an out view of 8 size-3 entries (24 entries of ct's size 2) from entry batch_off of ct's storage"""
        n = ctx.n
        return capi.View(ct.data[batch_off:].data_ptr(), 3 * ct.cap * n, ct.cap * n, 8, 3, L, 0)
    big_a = ctx.upload(fx.random_ct(rng, 60, 2, L))
    big_b = ctx.upload(fx.random_ct(rng, 60, 2, L))
    assert raw(big_a[0:6], b, 2, 3, 4, vo=inside(big_a, 10)) == OK                          # disjoint storage
    assert raw(big_a[0:6], b, 2, 3, 4, vo=inside(big_a, 3)) == INV                          # out overlaps a (not at a's start)
    assert raw(a, big_b[0:12], 2, 3, 4, vo=inside(big_b, 5)) == INV                         # out overlaps b
    assert raw(a, b, 2, 3, 4, vo=inside(a, 0)) == INV
    null = capi.View(0, 0, 0, 8, 3, L, 0)
    assert raw(a, b, 2, 3, 4, vo=null) == INV
    torch.cuda.synchronize()
    with pytest.raises(capi.CkksInvalidArgument):
        ev.multiply_sum_matrix(a, b, 4, cols)
    with pytest.raises(capi.CkksInvalidArgument):
        ev.multiply_sum_matrix(a, b, rows, 3)
    with pytest.raises(capi.CkksInvalidArgument):
        ev.multiply_sum_matrix(a, b, 0, cols)
    with pytest.raises(capi.CkksInvalidArgument, match="scale out of bounds"):
        ev.multiply_sum_matrix(ctx.upload(fx.random_ct(rng, 6, 2, L), scale=2.0 ** 100),
                               ctx.upload(fx.random_ct(rng, 12, 2, L), scale=2.0 ** 100), rows, cols)


# ------------------------------------------------------------------ the workload
class Problem:
    """config-4 chain {60, 40 x 4, 60} at N = 16384: DiagonalSets for both methods and the keys of each"""

    def __init__(self, eng, d, seed):
        wl, _, client, params, _ = _mods()
        ctx = eng.Context(14, params.coeff_modulus_create(14, CHAIN4))
        self.ctx, self.ev, self.enc, self.d = ctx, eng.Evaluator(ctx), client.CKKSEncoder(ctx), d
        kg = client.KeyGenerator(ctx, seed=seed)
        self.encr = client.Encryptor(ctx, kg.public_key(), seed=seed + 1)
        self.decr = client.Decryptor(ctx, kg.secret_key())
        both = lambda U: (wl.DiagonalSet.from_matrix(U, EPS, SCALE, self.enc),
                          wl.DiagonalSet.from_matrix(U, EPS, SCALE, self.enc, limbs=ctx.K))
        m = [both(wl.u_sigma(d)), both(wl.u_tau(d)), [both(wl.v_k(d, k)) for k in range(1, d)],
             [both(wl.w_k(d, k)) for k in range(1, d)]]
        self.mats = {}
        for i, method in enumerate(("reference", "hoisted")):
            self.mats[method] = (m[0][i], m[1][i], [v[i] for v in m[2]], [w[i] for w in m[3]])
        self.keys = {"reference": kg.keyset(steps=POW2_14),
                     "hoisted": kg.keyset(steps=wl.matmul_nonzero_hoisted_steps(d))}
        self.plans = {k: wl.PlanCache(ctx, v) for k, v in self.keys.items()}

    def encrypt_tiles(self, M):
        wl = _mods()[0]
        t, grid = wl.matrix_tiles(M, self.d)
        return self.encr.encrypt(self.enc.encode(t, SCALE)), grid

    def decrypt(self, C, shape):
        wl = _mods()[0]
        return wl.matrix_from_tiles(self.enc.decode(self.decr.decrypt(C)), shape, self.d)

    def args(self, method):
        return (*self.mats[method], self.keys[method], self.plans[method])


@pytest.fixture(scope="module")
def prob8(eng):
    return Problem(eng, 8, seed=501)


def _per_tile_sum(wl, ev, P, At, Bt, tiles, method):
    """the sum over l of the existing per-tile products, added with Evaluator.add"""
    tn, tm, tp = tiles
    fn = wl.cc_matrix_multiplication_sparse if method == "reference" else wl.cc_matrix_multiplication_nonzero_hoisted
    outs = []
    for i in range(tn):
        for j in range(tp):
            acc = None
            for l in range(tm):
                p = fn(ev, At[i * tm + l], Bt[l * tp + j], P.d, *P.args(method))
                acc = p if acc is None else ev.add(acc, p)
            outs.append(acc)
    return outs


@pytest.mark.parametrize("method", ["reference", "hoisted"])
@pytest.mark.parametrize("n,m,p", [(16, 24, 16), (20, 13, 9)])
def test_blocked_equals_the_per_tile_sum(prob8, method, n, m, p):
    wl = _mods()[0]
    P, ev, d = prob8, prob8.ev, 8
    rng = np.random.default_rng(n * 100 + m * 10 + p)
    A, B = rng.uniform(-1, 1, (n, m)), rng.uniform(-1, 1, (m, p))
    At, (tn, tm) = P.encrypt_tiles(A)
    Bt, (_, tp) = P.encrypt_tiles(B)
    got = wl.cc_matrix_multiplication_blocked(ev, At, Bt, (tn, tm, tp), d, *P.args(method), method=method)
    assert (got.batch, got.size, got.limbs) == (tn * tp, 3, At.limbs - 1)
    want = _per_tile_sum(wl, ev, P, At, Bt, (tn, tm, tp), method)
    for o, w in enumerate(want):
        assert _same(got[o], w), o
    assert np.abs(P.decrypt(got, (n, p)) - A @ B).max() < 1e-3


def test_blocked_rejects_bad_grids(prob8):
    wl, _, _, _, capi = _mods()
    P = prob8
    At, _ = P.encrypt_tiles(np.ones((16, 16)))
    with pytest.raises(ValueError):
        wl.cc_matrix_multiplication_blocked(P.ev, At, At, (2, 2, 1), 8, *P.args("hoisted"), method="hoisted")
    with pytest.raises(ValueError):
        wl.cc_matrix_multiplication_blocked(P.ev, At, At, (2, 2, 2), 8, *P.args("hoisted"), method="other")


def test_blocked_d64_hoisted_128(eng):
    """d = 64 tiles (d^2 = N/4), 128 x 128: 2 x 2 x 2 tiles"""
    wl = _mods()[0]
    P = Problem(eng, 64, seed=641)
    rng = np.random.default_rng(128)
    A, B = rng.uniform(0, 1, (128, 128)), rng.uniform(0, 1, (128, 128))
    At, _ = P.encrypt_tiles(A)
    Bt, _ = P.encrypt_tiles(B)
    got = wl.cc_matrix_multiplication_blocked(P.ev, At, Bt, (2, 2, 2), 64, *P.args("hoisted"), method="hoisted")
    want = _per_tile_sum(wl, P.ev, P, At, Bt, (2, 2, 2), "hoisted")
    for o, w in enumerate(want):
        assert _same(got[o], w), o
    assert np.abs(P.decrypt(got, (128, 128)) - A @ B).max() < 1e-3


# ------------------------------------------------------------------ sharding
@pytest.mark.parametrize("method", ["reference", "hoisted"])
def test_emulated_sharding_is_bit_identical(prob8, method):
    wl, par, _, _, _ = _mods()
    P, ev, d = prob8, prob8.ev, 8
    rng = np.random.default_rng(77)
    A, B = rng.uniform(-1, 1, (20, 13)), rng.uniform(-1, 1, (13, 9))
    At, (tn, tm) = P.encrypt_tiles(A)
    Bt, (_, tp) = P.encrypt_tiles(B)
    tiles = (tn, tm, tp)                                   # 3 x 2 x 2: 10 transforms, 6 outputs
    want = wl.cc_matrix_multiplication_blocked(ev, At, Bt, tiles, d, *P.args(method), method=method)
    n_tr = tn * tm + tm * tp
    for world in sorted({1, 2, 3, 4, 8, n_tr + 1}):
        got = EmulatedExchange(world).run(lambda r, ex: par.sharded_cc_matrix_multiplication_blocked(
            ev, At, Bt, tiles, d, *P.args(method), r, world, ex, method=method))
        for r in range(world):
            assert _same(got[r], want), (method, world, r)
    assert np.abs(P.decrypt(got[-1], (20, 9)) - A @ B).max() < 1e-3


def _nccl_worker(rank, world, port, ret):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        eng = importlib.import_module(PKG).load_engine()
        wl, par, client, params, _ = _mods()
        d = 4
        ctx = eng.Context(14, params.coeff_modulus_create(14, CHAIN4), device=rank)
        ev, enc = eng.Evaluator(ctx), client.CKKSEncoder(ctx)
        kg = client.KeyGenerator(ctx, seed=91)                       # same keys and inputs on every rank
        keys = kg.keyset(steps=wl.matmul_nonzero_hoisted_steps(d))
        encr = client.Encryptor(ctx, kg.public_key(), seed=92)
        rng = np.random.default_rng(93)
        A, B = rng.uniform(0, 1, (10, 7)), rng.uniform(0, 1, (7, 6))
        At, Bt = (encr.encrypt(enc.encode(wl.matrix_tiles(M, d)[0], SCALE)) for M in (A, B))
        sp = lambda M: wl.DiagonalSet.from_matrix(M, EPS, SCALE, enc, limbs=ctx.K)
        mats = (sp(wl.u_sigma(d)), sp(wl.u_tau(d)), [sp(wl.v_k(d, k)) for k in range(1, d)],
                [sp(wl.w_k(d, k)) for k in range(1, d)])
        plans = wl.PlanCache(ctx, keys)
        tiles = (3, 2, 2)
        got = par.sharded_cc_matrix_multiplication_blocked(ev, At, Bt, tiles, d, *mats, keys, plans, rank, world,
                                                           par.TorchExchange(), method="hoisted")
        want = wl.cc_matrix_multiplication_blocked(ev, At, Bt, tiles, d, *mats, keys, plans, method="hoisted")
        ret[rank] = bool(_same(got, want))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4, 8])
def test_nccl_sharding_is_bit_identical(eng, world):
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs, %d visible" % (world, torch.cuda.device_count()))
    ret = mp.Manager().dict()
    port = 37500 + (os.getpid() % 2000) + 10 * world
    mp.spawn(_nccl_worker, args=(world, port, ret), nprocs=world, join=True)
    assert len(ret) == world and all(ret[r] for r in range(world)), dict(ret)


def test_cpp_blocked_product_is_the_per_tile_sum(pkg, tmp_path):
    """tests/cpp/matmul_blocked_driver.cpp, compiled here against seal/seal.h and ckks_b200_helper.h: at d = 4 every output
    tile of b200::CC_Matrix_Multiplication_blocked is bit-identical to the sum of b200::CC_Matrix_Multiplication over l"""
    import subprocess
    import test_shim
    exe = str(tmp_path / "matmul_blocked_driver")
    res = subprocess.run(["g++", "-std=c++17", "-O2"] + test_shim.INC +
                         [os.path.join(test_shim.ROOT, "tests", "cpp", "matmul_blocked_driver.cpp"), "-o", exe, test_shim.LIB,
                          "-Wl,-rpath," + os.path.dirname(test_shim.LIB)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert res.returncode == 0, res.stdout[-3000:]
    run = subprocess.run([exe], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert run.returncode == 0 and "MATMUL BLOCKED OK" in run.stdout, run.stdout[-3000:]
