"""GPU: constant-coefficient sums (ckks_multiply_const_sum / Evaluator.multiply_const_sum), the Chebyshev polynomial
evaluator (workloads.chebyshev_cipher) and encrypted LR with the Chebyshev sigmoid (method="chebyshev") on config 1.

The kernel is bit-identical to SEAL's multiply_plain by encode(double) plaintexts + add_many + add_plain;
chebyshev_cipher is bit-identical to a sequential restatement of its op sequence on the CPU oracle; the decrypted values
and the LR steps are checked against numpy within stated tolerances."""
import ctypes
import importlib
import json
import os

import numpy as np
import pytest
import torch
from numpy.polynomial import chebyshev as Ch

from test_gpu_sharded_lr import BroadcastingExchange

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = "seal-fyp-logistic-regression_b200"
CHAIN13 = [60] + [40] * 12 + [60]                 # config 1 with the degree-63 Chebyshev sigmoid
POW2 = [s for i in range(13) for s in (1 << i, -(1 << i))]
SCALE, LR = 2.0 ** 40, 0.1


def _mods():
    return tuple(importlib.import_module(PKG + m) for m in (".workloads", ".lr", ".parallel", ".client", ".params", ".capi"))


# ------------------------------------------------------------------ the kernel
def _raw(fx, src, T, G, coeffs, scales, c0=None, s0=None, out=None):
    """ckks_multiply_const_sum straight through the C ABI (no Python-side scale checks)"""
    M = src.batch // max(T, 1)
    out = fx.ctx.empty(max(G, 1) * M, src.size, src.limbs) if out is None else out
    cf, sc = np.ascontiguousarray(coeffs, dtype=np.float64), np.ascontiguousarray(scales, dtype=np.float64)
    k0 = None if c0 is None else np.ascontiguousarray(c0, dtype=np.float64)
    k1 = None if s0 is None else np.ascontiguousarray(s0, dtype=np.float64)
    vi, vo = src.view(), out.view()
    rc = fx.ctx.lib.ckks_multiply_const_sum(fx.ev.h, ctypes.byref(vi), T, G, cf.ctypes.data, sc.ctypes.data,
                                            None if k0 is None else k0.ctypes.data, None if k1 is None else k1.ctypes.data,
                                            ctypes.byref(vo), None)
    return rc, out


def _reference(fx, src, T, G, coeffs, scales, c0, s0):
    """SEAL's sequence: multiply_plain by encode(c, s) per term, add_many, add_plain(encode(c0, s0))"""
    ev, M, L = fx.ev, src.batch // T, src.limbs
    outs = []
    for g in range(G):
        for m in range(M):
            prods = [ev.multiply_plain(src[i * M + m], ev.encode_scalar(coeffs[g * T + i], scales[g * T + i], limbs=L))
                     for i in range(T)]
            acc = ev.add_many(type(src)(fx.ctx, torch.cat([p.data for p in prods]), L, 1.0))
            if c0 is not None:
                acc.scale = s0[g]
                acc = ev.add_plain(acc, ev.encode_scalar(c0[g], s0[g], limbs=L))
            outs.append(acc.numpy()[0])
    return np.stack(outs)


KERNEL_CASES = [(12, [50, 40, 40, 50]), (15, [60, 40, 40, 40, 60])]


@pytest.mark.parametrize("log_n,bits", KERNEL_CASES)
@pytest.mark.parametrize("T,G,M,size", [(1, 1, 1, 2), (5, 1, 2, 2), (1, 3, 1, 2), (7, 8, 1, 2), (4, 11, 2, 3)])
def test_const_sum_bit_identical_to_seal_sequence(make_fixture, log_n, bits, T, G, M, size):
    fx = make_fixture(log_n, bits)
    rng = np.random.default_rng(T * 100 + G * 10 + M + log_n)
    kinds = [lambda: rng.uniform(-1, 1), lambda: 0.0, lambda: -rng.uniform(0, 3), lambda: rng.uniform(-1, 1) * 1e-9,
             lambda: rng.uniform(-1, 1) * 1e6]
    coeffs = np.array([kinds[k % len(kinds)]() for k in range(G * T)])
    coeffs[rng.integers(0, G * T)] = 0.0
    scales = 2.0 ** rng.uniform(10, 40, G * T)
    c0 = rng.uniform(-2, 2, G)
    s0 = 2.0 ** rng.uniform(20, 40, G)
    for limbs in range(1, len(bits)):
        src = fx.ctx.upload(fx.random_ct(rng, T * M, size, limbs))
        for k0, k1 in ((c0, s0), (None, None)):
            rc, got = _raw(fx, src, T, G, coeffs, scales, k0, k1)
            assert rc == 0
            assert np.array_equal(got.numpy(), _reference(fx, src, T, G, coeffs, scales, k0, k1)), (limbs, k0 is None)


def test_const_sum_all_zero_group_and_rejections(make_fixture):
    fx = make_fixture(*KERNEL_CASES[0])
    _, _, _, _, _, capi = _mods()
    rng = np.random.default_rng(5)
    src = fx.ctx.upload(fx.random_ct(rng, 6, 2, 3))
    rc, got = _raw(fx, src, 3, 2, [0.0, 0.0, 0.0, 1.0, 0.0, 2.0], [2.0 ** 30] * 6, [0.25, 0.0], [2.0 ** 30] * 2)
    assert rc == 0
    g0 = got.numpy()[:2]                                     # group 0: no term, the constant 0.25 * 2^30 alone
    assert not g0[:, 1].any() and (g0[:, 0] == 2 ** 28).all()
    ok = dict(coeffs=[1.0] * 6, scales=[2.0 ** 30] * 6)
    assert _raw(fx, src, 4, 2, **ok)[0] == capi.CKKS_ERR_INVALID                                   # 6 % 4
    assert _raw(fx, src, 0, 2, **ok)[0] == capi.CKKS_ERR_INVALID                                   # T < 1
    assert _raw(fx, src, 3, 0, **ok)[0] == capi.CKKS_ERR_INVALID                                   # G < 1
    assert _raw(fx, src, 3, 2, out=fx.ctx.empty(3, 2, 3), **ok)[0] == capi.CKKS_ERR_INVALID        # out batch
    assert _raw(fx, src, 3, 2, out=fx.ctx.empty(4, 3, 3), **ok)[0] == capi.CKKS_ERR_INVALID        # out size
    assert _raw(fx, src, 3, 2, out=src[2:6], **ok)[0] == capi.CKKS_ERR_INVALID                     # aliases in
    assert _raw(fx, src, 3, 2, [1.0] * 6, [0.0] + [2.0 ** 30] * 5)[0] == capi.CKKS_ERR_INVALID    # scale <= 0
    assert _raw(fx, src, 3, 2, [1e300] * 6, [1e300] * 6)[0] == capi.CKKS_ERR_INVALID              # c * s not finite
    assert _raw(fx, src, 3, 2, [1.0] * 6, [2.0 ** 30] * 6, [1.0, 1.0], [2.0 ** 30, float("nan")])[0] == capi.CKKS_ERR_INVALID
    big = fx.ctx.upload(fx.random_ct(rng, 700, 2, 3))
    assert _raw(fx, big, 700, 1, [1.0] * 700, [1.0] * 700)[0] == capi.CKKS_ERR_INVALID            # 701 x 3 > 2048


def test_evaluator_multiply_const_sum_scales(make_fixture):
    fx = make_fixture(*KERNEL_CASES[0])
    _, _, _, _, _, capi = _mods()
    ev, rng = fx.ev, np.random.default_rng(9)
    a = fx.ctx.upload(fx.random_ct(rng, 2, 2, 3), scale=2.0 ** 20)
    b = fx.ctx.upload(fx.random_ct(rng, 2, 2, 3), scale=2.0 ** 25)
    out = ev.multiply_const_sum([a, b], [[0.5, -1.5], [2.0, 0.0]], [2.0 ** 20, 2.0 ** 15], constant=[0.1, -0.2], groups=2)
    assert out.batch == 4 and out.scale == 2.0 ** 40 and out.limbs == 3
    src = type(a)(fx.ctx, torch.cat([a.data, b.data]), 3, 1.0)
    want = _reference(fx, src, 2, 2, [0.5, -1.5, 2.0, 0.0], [2.0 ** 20, 2.0 ** 15] * 2, [0.1, -0.2], [2.0 ** 40] * 2)
    assert np.array_equal(out.numpy(), want)
    with pytest.raises(capi.CkksInvalidArgument, match="scale mismatch"):
        ev.multiply_const_sum([a, b], [1.0, 1.0], [2.0 ** 20, 2.0 ** 20])
    with pytest.raises(capi.CkksInvalidArgument, match="scale out of bounds"):
        ev.multiply_const_sum(a, [1.0], 2.0 ** 200)
    with pytest.raises(capi.CkksInvalidArgument):
        ev.multiply_const_sum([a, b[0:1]], [1.0, 1.0], [2.0 ** 20, 2.0 ** 15])


# ------------------------------------------------------------------ chebyshev_cipher vs the CPU oracle
def _pt_const(orc, c, s, L):
    """encode(double): residues of nearbyint(c * s) in every NTT position"""
    v = round(c * s)
    return np.stack([np.full(orc.n, v % p, dtype=np.uint64) for p in orc.primes[:L]])


def _oracle_const_sum(orc, terms, coeffs, pts, konst=None):
    """sum_i multiply_plain(terms[i], encode(coeffs[i], pts[i])) (+ add_plain(encode(konst, scale))) term by term"""
    L = terms[0].shape[1]
    acc = None
    for x, c, s in zip(terms, coeffs, pts):
        y = orc.multiply_plain(x, _pt_const(orc, c, s, L))
        acc = y if acc is None else orc.add(acc, y)
    if konst is not None:
        acc = orc.add_plain(acc, _pt_const(orc, konst[0], konst[1], L))
    return acc


def _oracle_chebyshev(wl, orc, rlk, t, t_scale, coeffs, target):
    """chebyshev_cipher restated for ONE ciphertext, one oracle op at a time"""
    degree = len(coeffs) - 1
    m, l = wl._bsgs_shape(degree)
    K, b = wl._basis_doublings(m, l), 1 << l

    def mul(x, y):
        return orc.relinearize(orc.multiply(x, y), rlk)

    def lim(x, L):
        return np.ascontiguousarray(x[:, :L])

    def q(x):
        return orc.primes[x.shape[1] - 1]
    T, s = {1: t}, t_scale
    for k in range(K):
        h = 1 << k
        P = {j: mul(T[j], T[h]) for j in range(1, h + 1)}
        new = {}
        for j in range(1, h + 1):
            new[j] = _oracle_const_sum(orc, [T[j]], [1.0], [s])
            if j < h:
                new[h + j] = _oracle_const_sum(orc, [P[j], T[h - j]], [2.0, -1.0], [1.0, s])
            else:
                new[h + j] = _oracle_const_sum(orc, [P[j]], [2.0], [1.0], konst=(-1.0, s * s))
        s2 = s * s
        T = {}
        for j, x in new.items():
            T[j] = orc.rescale(x)
        s = s2 / float(q(new[1]))
    giants, gs = {}, {}
    if m > l:
        giants[l], gs[l] = T[b], s
        for k in range(l, m - 1):
            g = giants[k]
            sq = _oracle_const_sum(orc, [mul(g, g)], [2.0], [1.0], konst=(-1.0, gs[k] * gs[k]))
            gs[k + 1] = gs[k] * gs[k] / float(q(sq))
            giants[k + 1] = orc.rescale(sq)
    L = T[1].shape[1]
    drops = [orc.primes[L - 1 - i] for i in range(m - l + 1)]
    gscales = [gs[k] for k in range(l, m)]

    def result_scale(rho):
        sc = s * rho / float(drops[0])
        for qq, g in zip(drops[1:], gscales):
            sc = sc * g / float(qq)
        return sc
    guess = target / s
    for qq in drops:
        guess *= float(qq)
    for g in gscales:
        guess /= g
    rho = wl._solve_scale(result_scale, target, guess)
    Y = []
    for leaf in wl.chebyshev_split(coeffs, 1 << m, l):
        Y.append(orc.rescale(_oracle_const_sum(orc, [T[i] for i in range(1, b)], leaf[1:b], [rho] * (b - 1),
                                               konst=(leaf[0], s * rho))))
    sc = s * rho / float(drops[0])
    for k in range(l, m):
        g = lim(giants[k], Y[0].shape[1])
        nxt = []
        for j in range(len(Y) // 2):
            P = mul(Y[2 * j + 1], g)
            nxt.append(orc.rescale(_oracle_const_sum(orc, [P, Y[2 * j]], [1.0, 1.0], [1.0, gs[k]])))
        sc = sc * gs[k] / float(orc.primes[Y[0].shape[1] - 1])
        Y = nxt
    return Y[0], sc


@pytest.mark.parametrize("degree", [15, 63])
def test_chebyshev_cipher_bit_exact_vs_oracle(make_fixture, degree):
    wl = _mods()[0]
    fx = make_fixture(14, [50] + [40] * 8 + [50])
    rng = np.random.default_rng(degree)
    coeffs = rng.uniform(-1, 1, degree + 1)
    L = fx.L
    t_np = fx.random_ct(rng, 2, 2, L)
    t = fx.ctx.upload(t_np, scale=2.0 ** 40)
    got = wl.chebyshev_cipher(fx.ev, t, coeffs, fx.keys)
    assert got.limbs == L - wl.chebyshev_depth(degree) and got.batch == 2
    for m in range(2):
        want, want_scale = _oracle_chebyshev(wl, fx.orc, fx.rlk, t_np[m], 2.0 ** 40, coeffs, 2.0 ** 40)
        assert got.scale == want_scale
        assert np.array_equal(got.numpy()[m], want), m


# ------------------------------------------------------------------ decrypted accuracy and config 1 on pulsar
@pytest.fixture(scope="module")
def he13(eng):
    """N = 2^15, {60, 40 x 12, 60}: one Chebyshev iteration of config 1 uses every level; power-of-two Galois keys"""
    _, _, _, client, params, _ = _mods()
    ctx = eng.Context(15, params.coeff_modulus_create(15, CHAIN13))
    kg = client.KeyGenerator(ctx, seed=131)
    return dict(ctx=ctx, ev=eng.Evaluator(ctx), enc=client.CKKSEncoder(ctx), keys=kg.keyset(steps=POW2), pk=kg.public_key(),
                decr=client.Decryptor(ctx, kg.secret_key()), client=client)


def test_chebyshev_cipher_accuracy_degree_63(he13):
    """random coefficients scaled to sum |c_i| = 2 (the sigmoid's 1.99) and the sigmoid itself, on 32768 random t: the
    error grows with sum |c_i| (T_n amplifies the input's noise up to n^2-fold near +-1)"""
    wl, lr = _mods()[:2]
    rng = np.random.default_rng(63)
    vals = rng.uniform(-1, 1, (2, he13["ctx"].n // 2))
    encr = he13["client"].Encryptor(he13["ctx"], he13["pk"], seed=7)
    t = encr.encrypt(he13["enc"].encode(vals, SCALE))
    rand = rng.uniform(-1, 1, 64)
    for coeffs in (2.0 * rand / np.abs(rand).sum(), lr.SIGMOID_CHEBYSHEV.coeffs):
        out = wl.chebyshev_cipher(he13["ev"], t, coeffs, he13["keys"])
        assert out.scale == SCALE and out.limbs == t.limbs - 7
        err = np.abs(he13["enc"].decode(he13["decr"].decrypt(out)) - Ch.chebval(vals, coeffs)).max()
        print("max error", err)
        assert err < 1e-5


def _pulsar():
    pulsar = importlib.import_module(PKG + ".pulsar")
    with open(os.path.join(ROOT, "tests", "golden", "pulsar_plain_lr.json")) as fh:
        gold = json.load(fh)
    X, y = pulsar.load_csv()
    return gold, pulsar.standard_scaler(X).astype(np.float64), y.astype(np.float64)


def _encrypt(he, X, y, w0, seed):
    lr = _mods()[1]
    R, C = X.shape
    lay = lr.RowLayout(R, C, he["ctx"].n // 2)
    enc, encr = he["enc"], he["client"].Encryptor(he["ctx"], he["pk"], seed=seed)
    return lay, [encr.encrypt(enc.encode(v, SCALE)) for v in (lay.rows(X), lay.columns(X), lay.labels(y), lay.weights(w0))]


def test_config1_pulsar_chebyshev_update_weights(he13):
    """one encrypted step from the reference's initial weights: within 1e-4 of the plaintext Chebyshev step, within 1e-3
    of the reference program's weights_after_iteration_0"""
    lr = _mods()[1]
    gold, X, y = _pulsar()
    w0 = np.array(gold["initial_weights"])
    _, cts = _encrypt(he13, X, y, w0, seed=140)
    got = lr.update_weights(he13["ev"], *cts, LR, SCALE, he13["keys"], he13["enc"], None, method="chebyshev")
    dec = he13["enc"].decode(he13["decr"].decrypt(got))[0, :X.shape[1]]
    assert np.abs(dec - lr.plain_epoch(X, y, w0, LR, method="chebyshev")).max() < 1e-4
    assert np.abs(dec - np.array(gold["weights_after_iteration_0"])).max() < 1e-3


def test_config1_pulsar_chebyshev_train_three_iterations(he13):
    lr = _mods()[1]
    gold, X, y = _pulsar()
    w0 = np.array(gold["initial_weights"])
    lay, cts = _encrypt(he13, X, y, w0, seed=150)
    encr = he13["client"].Encryptor(he13["ctx"], he13["pk"], seed=151)
    got = lr.train_cipher(he13["ev"], *cts, LR, 3, lay, SCALE, he13["keys"], he13["enc"], encr, he13["decr"],
                          method="chebyshev")
    assert got.limbs == he13["ctx"].top_limbs
    plain = w0
    for _ in range(3):
        plain = lr.plain_epoch(X, y, plain, LR, method="chebyshev")
    assert np.abs(he13["enc"].decode(he13["decr"].decrypt(got))[0, :X.shape[1]] - plain).max() < 1e-4


def test_emulated_sharded_chebyshev_update_weights_is_bit_identical(he13):
    """emulated world sizes 2, 3 and 8 (8 > C = 4: ranks without features) against the one-GPU Chebyshev step"""
    lr, par = _mods()[1:3]
    R, C = 24, 4
    rng = np.random.default_rng(24)
    X, y, w0 = rng.normal(0, 1, (R, C)), (rng.uniform(0, 1, R) > 0.5).astype(float), rng.uniform(-1, 1, C)
    _, (rows, cols, labs, wct) = _encrypt(he13, X, y, w0, seed=160)
    want = lr.update_weights(he13["ev"], rows, cols, labs, wct, LR, SCALE, he13["keys"], he13["enc"], None,
                             method="chebyshev")
    dec = he13["enc"].decode(he13["decr"].decrypt(want))[0, :C]
    assert np.abs(dec - lr.plain_epoch(X, y, w0, LR, method="chebyshev")).max() < 1e-4
    for world in (2, 3, 8):
        def fn(r, ex):
            rb, fb = par.config1_shards(R, C, r, world)
            return par.sharded_update_weights(he13["ev"], rows[rb.start:rb.stop], list(rb), cols[fb.start:fb.stop], list(fb),
                                              labs, wct, LR, R, C, SCALE, he13["keys"], he13["enc"], None, r, world, ex,
                                              method="chebyshev")
        got = BroadcastingExchange(world).run(fn)
        for r in range(world):
            assert got[r].limbs == want.limbs and got[r].scale == want.scale and torch.equal(
                got[r].data[:, :, :want.limbs], want.data[:, :, :want.limbs]), (world, r)
