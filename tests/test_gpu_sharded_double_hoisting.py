"""GPU: double hoisting split at its mod-down (ckks_rotate_multiply_sum_hoisted_partial, ckks_rms_mod_down) and the sharded
double-hoisted workloads (parallel.sharded_linear_transform_plain_double_hoisted, the BSGS variant and
sharded_cc_matrix_multiplication_nonzero_hoisted), word for word against one GPU.

The full call itself is checked against an oracle restatement in test_gpu_double_hoisting; here every result is compared
with it.  World sizes are emulated in one process (the ranks run one after the other on one GPU, test_gpu_sharded_matmul's
EmulatedExchange); an NCCL run covers 2, 4 and 8 ranks where that many GPUs are visible."""
import ctypes as C
import importlib
import os
import sys

import numpy as np
import pytest
import torch

import test_gpu_double_hoisting as dh
from test_gpu_sharded_matmul import EmulatedExchange

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = "seal-fyp-logistic-regression_b200"
SCALE, EPS = 2.0 ** 40, 1e-8


def _mods():
    return tuple(importlib.import_module(PKG + m) for m in (".workloads", ".parallel", ".client", ".params", ".capi"))


def _table(rng, n_in, n_pt):
    """test_gpu_double_hoisting's table (outputs of 1, 2 and 49 terms, step 0, repeated and negative steps, weight-1
    terms, two inputs, an output of step-0 terms only) plus outputs without terms"""
    t = dh._table(rng, n_in, n_pt)
    return [[]] + t[:3] + [[]] + t[3:] + [[(0, 0, 2)]]


def _full(fx, eng, ct, pt, outputs):
    plan = eng.RotMulSumPlan(fx.ctx, fx.keys, ct.batch, pt.batch, outputs)
    return fx.ev.rotate_multiply_sum_hoisted(ct, pt, plan)


def _partial(fx, eng, ct, pt, outputs):
    plan = eng.RotMulSumPlan(fx.ctx, fx.keys, ct.batch, pt.batch, outputs)
    return fx.ev.rotate_multiply_sum_hoisted_partial(ct, pt, plan)


def _same(a, b):
    return (a.batch, a.limbs, a.scale) == (b.batch, b.limbs, b.scale) and torch.equal(a.data[:, :, :a.limbs],
                                                                                     b.data[:, :, :b.limbs])


@pytest.mark.parametrize("bits", dh.CHAINS, ids=lambda b: "-".join(map(str, b)))
def test_mod_down_of_partial_is_the_full_call(make_fixture, eng, bits):
    """top level, one level down (limb L != K - 1) and L = 1; mixed FP64 / integer primes and a small special prime"""
    fx, rng, n_in, pts = dh._case(make_fixture, bits, sum(bits) + 1)
    outputs = _table(rng, n_in, pts.shape[0])
    pt = fx.ctx.upload_plain(pts, scale=1.0)
    for L in sorted({fx.L, fx.L - 1, 1} - {0}, reverse=True):
        ct = fx.ctx.upload(fx.random_ct(rng, n_in, 2, L), cap=fx.L, scale=1.0)
        part = _partial(fx, eng, ct, pt, outputs)
        assert part.data.shape == (len(outputs), 2, L + 1, fx.n) and part.limbs == L
        x = part.data.cpu().numpy().view(np.uint64)
        K = len(fx.primes)
        for j, p in enumerate(list(fx.primes[:L]) + [fx.primes[K - 1]]):
            assert (x[:, :, j] < np.uint64(p)).all(), j                     # canonical residues
        assert not x[0].any() and not x[4].any()                            # outputs without terms: zeros
        assert not x[5, :, L].any()                                         # step-0 terms only: nothing mod P
        assert _same(fx.ev.rms_mod_down(part, 1), _full(fx, eng, ct, pt, outputs)), L


def test_rounding_modes_and_chunked_workspace(make_fixture, eng):
    fx, rng, n_in, pts = dh._case(make_fixture, dh.CHAINS[0], 78)
    outputs = _table(rng, n_in, pts.shape[0])
    L = fx.L
    ct = fx.ctx.upload(fx.random_ct(rng, n_in, 2, L), scale=1.0)
    pt = fx.ctx.upload_plain(pts, scale=1.0)
    try:
        for mode in (0, 1, 2, 3):
            fx.ctx.set_rounding(mode)
            assert _same(fx.ev.rms_mod_down(_partial(fx, eng, ct, pt, outputs), 1), _full(fx, eng, ct, pt, outputs)), mode
    finally:
        fx.ctx.set_rounding(1)
    full = _full(fx, eng, ct, pt, outputs)
    part = _partial(fx, eng, ct, pt, outputs)
    fixed = n_in * fx.n * (L + L * (L + 1)) * 8
    try:   # about one unit's partial at a time in the partial, one output at a time in the mod-down
        fx.ctx.set_workspace_cap(fixed + fx.n * 2 * (L + 1) * 8)
        small = _partial(fx, eng, ct, pt, outputs)
        fx.ctx.set_workspace_cap(fx.n * (4 * L + 2) * 8)
        down = fx.ev.rms_mod_down(small, 1)
    finally:
        fx.ctx.set_workspace_cap(1 << 30)
    assert torch.equal(small.data, part.data)
    assert _same(down, full)


def _random_partition(rng, outputs, G):
    """each term to a random group, every group keeping the order of its terms; at G = 2 every term goes to group 0, so
    group 1 is a plan without terms (as are groups that draw nothing at G = 8)"""
    owner = [[int(rng.integers(G)) if G > 2 else int(rng.integers(G - 1)) for _ in terms] for terms in outputs]
    return [[[t for t, w in zip(terms, own) if w == g] for terms, own in zip(outputs, owner)] for g in range(G)]


@pytest.mark.parametrize("G", [2, 3, 8])
def test_random_partitions_sum_to_the_full_call(make_fixture, eng, G):
    fx, rng, n_in, pts = dh._case(make_fixture, dh.CHAINS[0], 90 + G)
    outputs = _table(rng, n_in, pts.shape[0])
    pt = fx.ctx.upload_plain(pts, scale=1.0)
    eng_mod = importlib.import_module(PKG + ".engine")
    for L in (fx.L, 1):
        ct = fx.ctx.upload(fx.random_ct(rng, n_in, 2, L), cap=fx.L, scale=1.0)
        full = _full(fx, eng, ct, pt, outputs)
        groups = _random_partition(rng, outputs, G)
        parts = [_partial(fx, eng, ct, pt, grp) for grp in groups]
        order = rng.permutation(G)
        got = fx.ev.rms_mod_down([parts[g] for g in order], G)               # a list of G partials, permuted
        assert _same(got, full), (G, L)
        stacked = eng_mod.ExtendedPartial(fx.ctx, torch.cat([parts[g].data for g in order[::-1]]), L, 1.0)
        assert _same(fx.ev.rms_mod_down(stacked, G), full), (G, L)        # one stacked partial


def test_sub_plan_outputs_equal_the_full_plans(make_fixture, eng):
    """a plan of a subset of the outputs (its own work split) gives those outputs of the full plan word for word"""
    fx, rng, n_in, pts = dh._case(make_fixture, dh.CHAINS[1], 55)
    outputs = _table(rng, n_in, pts.shape[0])
    pt = fx.ctx.upload_plain(pts, scale=1.0)
    ct = fx.ctx.upload(fx.random_ct(rng, n_in, 2, fx.L), scale=1.0)
    full = _full(fx, eng, ct, pt, outputs)
    for sub in ([3], [2, 3], [1, 3, 6, 7], list(range(len(outputs)))[::2]):
        got = _full(fx, eng, ct, pt, [outputs[o] for o in sub])
        assert torch.equal(got.data[:, :, :fx.L], full.data[sub][:, :, :fx.L]), sub


def test_rejections(make_fixture, eng):
    _, _, _, _, capi = _mods()
    fx, rng, n_in, pts = dh._case(make_fixture, dh.CHAINS[0], 6)
    Inv = capi.CkksInvalidArgument
    L, K, n = fx.L, len(fx.primes), fx.n
    ev, lib = fx.ev, fx.ctx.lib
    plan = eng.RotMulSumPlan(fx.ctx, fx.keys, 2, 2, [[(0, 1, 0)], [(1, -1, 1)]])
    ct = fx.ctx.upload(fx.random_ct(rng, 2, 2, L), scale=1.0)
    pt = fx.ctx.upload_plain(pts[:2], scale=1.0)
    part = ev.rotate_multiply_sum_hoisted_partial(ct, pt, plan)
    # the partial: the full call's checks, out at L + 1 limbs
    with pytest.raises(Inv, match="key level"):
        ev.rotate_multiply_sum_hoisted_partial(ct, fx.ctx.upload_plain(pts[:2, :L], scale=1.0), plan)
    with pytest.raises(Inv, match="in batch"):
        ev.rotate_multiply_sum_hoisted_partial(ct[0], pt, plan)
    with pytest.raises(Inv, match="scale out of bounds"):
        ev.rotate_multiply_sum_hoisted_partial(fx.ctx.upload(fx.random_ct(rng, 2, 2, L), scale=2.0 ** 100),
                                               fx.ctx.upload_plain(pts[:2], scale=2.0 ** 100), plan)
    view = lambda data, batch, limbs: capi.View(data.data_ptr(), 2 * data.shape[2] * n, data.shape[2] * n, batch, 2, limbs, 0)
    vi, vp = ct.view(), pt.view()
    buf = torch.zeros((3, 2, L + 1, n), dtype=torch.int64, device=ct.data.device)

    def partial_rc(vo, vin=vi):
        return lib.ckks_rotate_multiply_sum_hoisted_partial(ev.h, plan._h, C.byref(vin), C.byref(vp), C.byref(vo), None)
    assert partial_rc(view(buf, 2, L + 1)) == capi.CKKS_OK
    assert partial_rc(view(buf, 2, L)) == capi.CKKS_ERR_INVALID                # out not at L + 1 limbs
    assert partial_rc(view(buf, 3, L + 1)) == capi.CKKS_ERR_INVALID            # out batch
    alias = capi.View(ct.data.data_ptr(), 2 * (L + 1) * n, (L + 1) * n, 2, 2, L + 1, 0)
    assert partial_rc(alias) == capi.CKKS_ERR_INVALID                          # out overlaps in
    alias_pt = capi.View(pt.data.data_ptr(), 2 * (L + 1) * n, (L + 1) * n, 2, 2, L + 1, 0)
    assert partial_rc(alias_pt) == capi.CKKS_ERR_INVALID                       # out overlaps pts
    assert lib.ckks_rotate_multiply_sum_hoisted_partial(ev.h, None, C.byref(vi), C.byref(vp), C.byref(view(buf, 2, L + 1)),
                                                        None) == capi.CKKS_ERR_INVALID
    # the mod-down
    parts4 = torch.cat([part.data, part.data])                                 # 2 groups x 2 outputs
    out = torch.zeros((4, 2, L, n), dtype=torch.int64, device=ct.data.device)
    ovw = lambda batch, limbs, size=2, data=out: capi.View(data.data_ptr(), 2 * data.shape[2] * n, data.shape[2] * n,
                                                           batch, size, limbs, 0)

    def md(vparts, groups, vo):
        return lib.ckks_rms_mod_down(ev.h, C.byref(vparts), groups, C.byref(vo), None)
    vparts = view(parts4, 4, L + 1)
    assert md(vparts, 2, ovw(2, L)) == capi.CKKS_OK
    assert md(vparts, 1, ovw(4, L)) == capi.CKKS_OK
    assert md(vparts, 0, ovw(2, L)) == capi.CKKS_ERR_INVALID                   # groups < 1
    assert md(vparts, -2, ovw(2, L)) == capi.CKKS_ERR_INVALID
    assert md(vparts, 3, ovw(2, L)) == capi.CKKS_ERR_INVALID                   # batch != groups x out batch
    assert md(vparts, 2, ovw(1, L)) == capi.CKKS_ERR_INVALID
    assert md(vparts, 2, ovw(2, L - 1)) == capi.CKKS_ERR_INVALID               # limbs != out limbs + 1
    assert md(view(parts4, 4, L), 2, ovw(2, L)) == capi.CKKS_ERR_INVALID
    big = torch.zeros((2, 2, K + 1, n), dtype=torch.int64, device=ct.data.device)
    wide = torch.zeros((2, 2, K, n), dtype=torch.int64, device=ct.data.device)
    assert md(view(wide, 2, K), 1, ovw(2, K, data=big)) == capi.CKKS_ERR_INVALID   # out limbs > K - 1 (parts at K)
    assert md(capi.View(parts4.data_ptr(), 3 * (L + 1) * n, (L + 1) * n, 4, 3, L + 1, 0), 2,
              ovw(2, L)) == capi.CKKS_ERR_INVALID                              # parts size 3
    assert md(vparts, 2, ovw(2, L, size=3)) == capi.CKKS_ERR_INVALID           # out size 3
    in_parts = capi.View(parts4.data_ptr(), 2 * L * n, L * n, 2, 2, L, 0)
    assert md(vparts, 2, in_parts) == capi.CKKS_ERR_INVALID                    # out overlaps parts
    torch.cuda.synchronize()
    with pytest.raises(Inv, match="scale mismatch"):
        other = importlib.import_module(PKG + ".engine").ExtendedPartial(fx.ctx, part.data, L, 2.0)
        ev.rms_mod_down([part, other], 2)
    with pytest.raises(Inv):
        ev.rms_mod_down(part, 3)


# ---------------------------------------------------------------------------------------------- workloads
@pytest.fixture(scope="module")
def config3(eng):
    """N = 16384, {60, 40, 40, 60}: the one-GPU keys of the d = 16 / 64 / 128 transforms (every rank's keys are a subset)"""
    wl, _, client, params, _ = _mods()
    ctx = eng.Context(14, params.coeff_modulus_create(14, [60, 40, 40, 60]))
    kg = client.KeyGenerator(ctx, seed=61)
    steps = set()
    for d in (16, 64, 128):
        steps |= set(wl.linear_transform_double_hoisted_steps(d))
        steps |= set(wl.bsgs_double_hoisted_steps(d, max(1, int(round(d ** 0.5)))))
    keys = kg.keyset(steps=sorted(steps), relin=False)
    return dict(ctx=ctx, ev=eng.Evaluator(ctx), enc=client.CKKSEncoder(ctx), keys=keys, plans=wl.PlanCache(ctx, keys),
                encr=client.Encryptor(ctx, kg.public_key(), seed=62), decr=client.Decryptor(ctx, kg.secret_key()))


def _worlds(extra):
    return sorted({1, 2, 3, 4, 8, extra})


@pytest.mark.parametrize("d", [16, 64, 128])
def test_emulated_sharded_transforms(config3, d):
    wl, par, _, _, _ = _mods()
    c = config3
    ctx, ev, enc, keys, plans = c["ctx"], c["ev"], c["enc"], c["keys"], c["plans"]
    rng = np.random.default_rng(d + 1)
    U, v = rng.uniform(0, 1, (d, d)), rng.uniform(0, 1, d)
    ct = c["encr"].encrypt(enc.encode(v, SCALE))
    dec = lambda x: enc.decode(c["decr"].decrypt(x))[0, :d]
    diags = enc.encode(wl.all_diagonals(U), SCALE, limbs=ctx.K)
    bd = wl.BsgsDiagonals(U, SCALE, enc, limbs=ctx.K)
    want = wl.linear_transform_plain_double_hoisted(ev, ct, diags, keys, plans)
    want_bsgs = wl.linear_transform_plain_bsgs_double_hoisted(ev, ct, bd, keys, plans)
    assert np.abs(dec(want) - U @ v).max() < 1e-4 and np.abs(dec(want_bsgs) - U @ v).max() < 1e-4
    for world in _worlds(bd.G + 1):
        got = EmulatedExchange(world).run(lambda r, ex: par.sharded_linear_transform_plain_double_hoisted(
            ev, ct, diags, keys, plans, r, world, ex))
        got_bsgs = EmulatedExchange(world).run(lambda r, ex: par.sharded_linear_transform_plain_bsgs_double_hoisted(
            ev, ct, bd, keys, plans, r, world, ex))
        for r in range(world):
            assert _same(got[r], want), (d, world, r)
            assert _same(got_bsgs[r], want_bsgs), (d, world, r)
        assert np.abs(dec(got[0]) - U @ v).max() < 1e-4 and np.abs(dec(got_bsgs[-1]) - U @ v).max() < 1e-4


@pytest.mark.parametrize("d", [8, 64])
def test_emulated_sharded_matmul(eng, d):
    """config-4 chain {60, 40 x 4, 60} at N = 16384"""
    wl, par, client, params, _ = _mods()
    ctx = eng.Context(14, params.coeff_modulus_create(14, [60, 40, 40, 40, 40, 60]))
    ev, enc = eng.Evaluator(ctx), client.CKKSEncoder(ctx)
    kg = client.KeyGenerator(ctx, seed=47)
    keys = kg.keyset(steps=wl.matmul_nonzero_hoisted_steps(d))
    encr, decr = client.Encryptor(ctx, kg.public_key(), seed=48), client.Decryptor(ctx, kg.secret_key())
    plans = wl.PlanCache(ctx, keys)
    rng = np.random.default_rng(d + 3)
    dd = d * d
    A, B = rng.uniform(0, 1, (d, d)), rng.uniform(0, 1, (d, d))
    ctA = encr.encrypt(enc.encode(A.reshape(-1), SCALE))
    ctB = encr.encrypt(enc.encode(B.reshape(-1), SCALE))
    sp = lambda U: wl.DiagonalSet.from_matrix(U, EPS, SCALE, enc, limbs=ctx.K)
    sig, tau = sp(wl.u_sigma(d)), sp(wl.u_tau(d))
    V = [sp(wl.v_k(d, k)) for k in range(1, d)]
    W = [sp(wl.w_k(d, k)) for k in range(1, d)]
    want = wl.cc_matrix_multiplication_nonzero_hoisted(ev, ctA, ctB, d, sig, tau, V, W, keys, plans)
    dec = lambda x: enc.decode(decr.decrypt(x))[0, :dd].reshape(d, d)
    assert np.abs(dec(want) - A @ B).max() < 1e-3
    for world in _worlds(d):   # d > d - 1 products: a rank without k
        got = EmulatedExchange(world).run(lambda r, ex: par.sharded_cc_matrix_multiplication_nonzero_hoisted(
            ev, ctA, ctB, d, sig, tau, V, W, keys, plans, r, world, ex))
        for r in range(world):
            assert got[r].size == 3 and _same(got[r], want), (d, world, r)
        assert np.abs(dec(got[-1]) - A @ B).max() < 1e-3


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
        d = 16
        ctx = eng.Context(14, params.coeff_modulus_create(14, [60, 40, 40, 40, 40, 60]), device=rank)
        ev, enc = eng.Evaluator(ctx), client.CKKSEncoder(ctx)
        kg = client.KeyGenerator(ctx, seed=71)                       # same keys and inputs on every rank
        keys = kg.keyset(steps=sorted(set(wl.matmul_nonzero_hoisted_steps(4)) | set(wl.linear_transform_double_hoisted_steps(d))
                                      | set(wl.bsgs_double_hoisted_steps(d, 4))))
        encr = client.Encryptor(ctx, kg.public_key(), seed=72)
        rng = np.random.default_rng(73)
        U, v = rng.uniform(0, 1, (d, d)), rng.uniform(0, 1, d)
        A, B = rng.uniform(0, 1, (4, 4)), rng.uniform(0, 1, (4, 4))
        ct = encr.encrypt(enc.encode(v, SCALE))
        diags = enc.encode(wl.all_diagonals(U), SCALE, limbs=ctx.K)
        bd = wl.BsgsDiagonals(U, SCALE, enc, baby=4, limbs=ctx.K)
        ctA, ctB = encr.encrypt(enc.encode(A.reshape(-1), SCALE)), encr.encrypt(enc.encode(B.reshape(-1), SCALE))
        sp = lambda M: wl.DiagonalSet.from_matrix(M, EPS, SCALE, enc, limbs=ctx.K)
        mats = (sp(wl.u_sigma(4)), sp(wl.u_tau(4)), [sp(wl.v_k(4, k)) for k in range(1, 4)], [sp(wl.w_k(4, k)) for k in range(1, 4)])
        plans, ex = wl.PlanCache(ctx, keys), par.TorchExchange()
        pairs = [
            (par.sharded_linear_transform_plain_double_hoisted(ev, ct, diags, keys, plans, rank, world, ex),
             wl.linear_transform_plain_double_hoisted(ev, ct, diags, keys, plans)),
            (par.sharded_linear_transform_plain_bsgs_double_hoisted(ev, ct, bd, keys, plans, rank, world, ex),
             wl.linear_transform_plain_bsgs_double_hoisted(ev, ct, bd, keys, plans)),
            (par.sharded_cc_matrix_multiplication_nonzero_hoisted(ev, ctA, ctB, 4, *mats, keys, plans, rank, world, ex),
             wl.cc_matrix_multiplication_nonzero_hoisted(ev, ctA, ctB, 4, *mats, keys, plans)),
        ]
        ret[rank] = [bool(_same(g, w)) for g, w in pairs]
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4, 8])
def test_nccl_sharding_is_bit_identical(eng, world):
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs, %d visible" % (world, torch.cuda.device_count()))
    ret = mp.Manager().dict()
    port = 35500 + (os.getpid() % 2000) + 10 * world
    mp.spawn(_nccl_worker, args=(world, port, ret), nprocs=world, join=True)
    assert len(ret) == world
    for r in range(world):
        assert all(ret[r]), (r, ret[r])
