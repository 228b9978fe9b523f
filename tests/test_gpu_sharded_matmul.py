"""GPU: the grouped mod-q sum (ckks_add_many_grouped) and the sharded CC_Matrix_Multiplication
(parallel.sharded_cc_matrix_multiplication), bit-identical to the one-GPU cc_matrix_multiplication_sparse.

World sizes 2, 4 and 8 are emulated in one process: the ranks run one after the other on one GPU, each up to its next
collective, and the emulated exchange hands the stacked partials back.  A real NCCL run covers 2 ranks (4 and 8 where
that many GPUs are visible)."""
import ctypes
import importlib
import os
import sys
import threading

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = "seal-fyp-logistic-regression_b200"
POW2_14 = tuple(s for i in range(13) for s in (1 << i, -(1 << i)))
SCALE, EPS = 2.0 ** 40, 1e-8


def _mods():
    return tuple(importlib.import_module(PKG + m) for m in (".workloads", ".parallel", ".client", ".params"))


# ------------------------------------------------------------------ ckks_add_many_grouped
_CTX = {}


def _ctx(eng, log_n):
    if log_n not in _CTX:
        params = importlib.import_module(PKG + ".params")
        ctx = eng.Context(log_n, params.coeff_modulus_create(log_n, [60, 40, 60]))
        _CTX[log_n] = (ctx, eng.Evaluator(ctx))
    return _CTX[log_n]


def _random_cts(ctx, batch, size, seed):
    """uniform residues below each prime, with the first 64 words of every limb at p - 1 (the lazy sum's worst case)"""
    L = ctx.top_limbs
    g = torch.Generator(device=ctx.device).manual_seed(seed)
    ct = ctx.empty(batch, size, L)
    for j in range(L):
        p = ctx.primes[j]
        ct.data[:, :, j].random_(0, p, generator=g)
        ct.data[:, :, j, :64] = p - 1
    return ct


@pytest.mark.parametrize("log_n", [14, 15])
@pytest.mark.parametrize("size", [2, 3])
@pytest.mark.parametrize("groups,M", [(1, 1), (2, 1), (3, 1), (8, 1), (1, 63), (2, 63), (3, 63), (8, 63), (17, 1), (17, 5)])
def test_add_many_grouped_matches_add_many_and_exact_sums(eng, log_n, size, groups, M):
    ctx, ev = _ctx(eng, log_n)
    cts = _random_cts(ctx, groups * M, size, seed=1000 * log_n + 10 * size + groups + M)
    got = ev.add_many_grouped(cts, groups)
    assert (got.batch, got.size, got.limbs, got.scale) == (M, size, cts.limbs, cts.scale)
    for m in range(M):   # add_many of group m = entries m, M + m, ...
        grp = eng.Ciphertext(ctx, cts.data[m::M].contiguous(), cts.limbs, cts.scale)
        assert torch.equal(got.data[m], ev.add_many(grp).data[0]), m
    x = cts.numpy()
    x = x.reshape((groups, M) + x.shape[1:])
    want = np.empty_like(x[0])
    for j in range(cts.limbs):
        p = np.uint64(ctx.primes[j])
        acc = np.zeros_like(x[0, :, :, j])
        for g in range(groups):                       # both operands < p < 2^61: a + b never wraps
            acc = (acc + x[g, :, :, j]) % p
        want[:, :, j] = acc
    assert np.array_equal(got.numpy(), want)


def test_add_many_grouped_rejects_bad_shapes(eng):
    capi = importlib.import_module(PKG + ".capi")
    ctx, ev = _ctx(eng, 14)
    cts = _random_cts(ctx, 6, 2, seed=5)
    with pytest.raises(capi.CkksInvalidArgument):
        ev.add_many_grouped(cts, 0)
    with pytest.raises(capi.CkksInvalidArgument):
        ev.add_many_grouped(cts, 4)                                 # 6 is not 4 x M
    with pytest.raises(capi.CkksInvalidArgument):
        ev.add_many_grouped(cts, 2, out=ctx.empty(2, 2, cts.limbs))  # in batch 6 != 2 x 2 (the C entry point checks)
    with pytest.raises(capi.CkksInvalidArgument):
        ev.add_many_grouped(cts, 2, out=ctx.empty(3, 3, cts.limbs))  # size
    with pytest.raises(capi.CkksInvalidArgument):
        ev.add_many_grouped(cts, 6, out=cts[0:1])                  # out aliases in
    vi, vo = cts.view(), ctx.empty(3, 2, cts.limbs).view()       # limbs: the evaluator always passes equal ones
    vo.limbs = cts.limbs - 1
    assert ctx.lib.ckks_add_many_grouped(ev.h, ctypes.byref(vi), 2, ctypes.byref(vo), None) == capi.CKKS_ERR_INVALID
    vo.limbs = cts.limbs
    assert ctx.lib.ckks_add_many_grouped(ev.h, ctypes.byref(vi), -1, ctypes.byref(vo), None) == capi.CKKS_ERR_INVALID
    assert ctx.lib.ckks_add_many_grouped(ev.h, ctypes.byref(vi), 2, ctypes.byref(vo), None) == capi.CKKS_OK
    torch.cuda.synchronize()


# ------------------------------------------------------------------ the sharded product
class EmulatedExchange:
    """the collectives of `world` ranks that run as threads of one process, one at a time: a rank runs until its next
    collective, leaves its contribution and passes the turn on; the last rank to arrive forms every rank's result and
    the turn starts again at rank 0.  Only one thread issues GPU work at any time."""

    def __init__(self, world):
        self.world, self.turn, self.epoch, self.error = world, 0, 0, None
        self.cond = threading.Condition()
        self.slots, self.results = [None] * world, None

    def _wait(self, rank, epoch):
        while not (self.turn == rank and self.epoch >= epoch) and self.error is None:
            self.cond.wait(timeout=1.0)
        if self.error is not None:
            raise RuntimeError("another rank failed")

    def _collective(self, rank, payload, form):
        with self.cond:
            self.slots[rank] = payload
            epoch = self.epoch + 1
            if rank == self.world - 1:
                self.results = form(self.slots)
                self.slots = [None] * self.world
                self.epoch, self.turn = epoch, 0
            else:
                self.turn = rank + 1
            self.cond.notify_all()
            self._wait(rank, epoch)
            return self.results[rank]

    def for_rank(self, rank):
        ex = self

        class View:
            def all_gather(self, t):
                return ex._collective(rank, t, lambda s: [torch.cat(s, 0)] * ex.world)

            def all_to_all(self, t, send_counts, recv_counts):
                def form(slots):
                    starts = np.concatenate([[0], np.cumsum(send_counts)])
                    return [torch.cat([sl[starts[q]:starts[q + 1]] for sl in slots], 0) for q in range(ex.world)]
                return ex._collective(rank, t, form)
        return View()

    def run(self, fn):
        """fn(rank, exchange) on every rank; returns the per-rank results"""
        out = [None] * self.world

        def body(r):
            try:
                with self.cond:
                    self._wait(r, 0)
                out[r] = fn(r, self.for_rank(r))
                torch.cuda.synchronize()
                with self.cond:
                    self.turn = r + 1
                    self.cond.notify_all()
            except BaseException as exc:   # wake the others, report the first failure below
                with self.cond:
                    self.error = self.error or exc
                    self.cond.notify_all()

        threads = [threading.Thread(target=body, args=(r,)) for r in range(self.world)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        if self.error is not None:
            raise self.error
        return out


def _problem(eng, d, seed):
    wl, _, client, params = _mods()
    ctx = eng.Context(14, params.coeff_modulus_create(14, [60, 40, 40, 40, 40, 60]))
    ev = eng.Evaluator(ctx)
    enc = client.CKKSEncoder(ctx)
    kg = client.KeyGenerator(ctx, seed=seed)
    keys = kg.keyset(steps=POW2_14)
    encr = client.Encryptor(ctx, kg.public_key(), seed=seed + 1)
    rng = np.random.default_rng(seed + 2)
    A, B = rng.uniform(0, 1, (d, d)), rng.uniform(0, 1, (d, d))
    sp = lambda U: wl.DiagonalSet.from_matrix(U, EPS, SCALE, enc)
    mats = (sp(wl.u_sigma(d)), sp(wl.u_tau(d)), [sp(wl.v_k(d, k)) for k in range(1, d)], [sp(wl.w_k(d, k)) for k in range(1, d)])
    ctA = encr.encrypt(enc.encode(A.reshape(-1), SCALE))
    ctB = encr.encrypt(enc.encode(B.reshape(-1), SCALE))
    return dict(ctx=ctx, ev=ev, keys=keys, plans=wl.PlanCache(ctx, keys), ctA=ctA, ctB=ctB, mats=mats,
                dec=client.Decryptor(ctx, kg.secret_key()), enc=enc, AB=A @ B)


def _same(a, b):
    return (a.size, a.limbs, a.scale) == (b.size, b.limbs, b.scale) and torch.equal(a.data[:, :, :a.limbs], b.data[:, :, :b.limbs])


@pytest.mark.parametrize("d", [8, 64])
def test_emulated_sharding_is_bit_identical(eng, d):
    wl, par, _, _ = _mods()
    P = _problem(eng, d, seed=80 + d)
    ev, ctA, ctB, keys, plans = P["ev"], P["ctA"], P["ctB"], P["keys"], P["plans"]
    sigma, tau, V, W = P["mats"]
    want = wl.cc_matrix_multiplication_sparse(ev, ctA, ctB, d, sigma, tau, V, W, keys, plans)
    dd = d * d
    dec = P["enc"].decode(P["dec"].decrypt(want))[0, :dd].reshape(d, d)
    assert np.abs(dec - P["AB"]).max() < 1e-2
    for world in (1, 2, 4, 8):
        got = EmulatedExchange(world).run(
            lambda r, ex: par.sharded_cc_matrix_multiplication(ev, ctA, ctB, d, sigma, tau, V, W, keys, plans, r, world, ex))
        for r in range(world):
            assert _same(got[r], want), (d, world, r)


def _nccl_worker(rank, world, port, ret):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        eng = importlib.import_module(PKG).load_engine()
        wl, par, client, params = _mods()
        d = 16
        ctx = eng.Context(14, params.coeff_modulus_create(14, [60, 40, 40, 40, 40, 60]), device=rank)
        ev = eng.Evaluator(ctx)
        enc = client.CKKSEncoder(ctx)
        kg = client.KeyGenerator(ctx, seed=16)                   # same keys and inputs on every rank
        keys = kg.keyset(steps=POW2_14)
        encr = client.Encryptor(ctx, kg.public_key(), seed=17)
        rng = np.random.default_rng(18)
        A, B = rng.uniform(0, 1, (d, d)), rng.uniform(0, 1, (d, d))
        sp = lambda U: wl.DiagonalSet.from_matrix(U, EPS, SCALE, enc)
        sigma, tau = sp(wl.u_sigma(d)), sp(wl.u_tau(d))
        V, W = [sp(wl.v_k(d, k)) for k in range(1, d)], [sp(wl.w_k(d, k)) for k in range(1, d)]
        ctA = encr.encrypt(enc.encode(A.reshape(-1), SCALE))
        ctB = encr.encrypt(enc.encode(B.reshape(-1), SCALE))
        plans = wl.PlanCache(ctx, keys)
        got = par.sharded_cc_matrix_multiplication(ev, ctA, ctB, d, sigma, tau, V, W, keys, plans, rank, world,
                                                   par.TorchExchange())
        want = wl.cc_matrix_multiplication_sparse(ev, ctA, ctB, d, sigma, tau, V, W, keys, plans)
        dec = enc.decode(client.Decryptor(ctx, kg.secret_key()).decrypt(got))[0, :d * d].reshape(d, d)
        ret[rank] = (_same(got, want), float(np.abs(dec - A @ B).max()))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4, 8])
def test_nccl_sharding_is_bit_identical(eng, world):
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs, %d visible" % (world, torch.cuda.device_count()))
    mgr = mp.Manager()
    ret = mgr.dict()
    port = 33500 + (os.getpid() % 2000) + 10 * world
    mp.spawn(_nccl_worker, args=(world, port, ret), nprocs=world, join=True)
    assert len(ret) == world
    for r in range(world):
        same, err = ret[r]
        assert same, r
        assert err < 1e-2, (r, err)
