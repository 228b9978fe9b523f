"""The Chebyshev sigmoid of encrypted LR on the host (CPU-only): the interpolant, the baby-step / giant-step split and its
depth, the plaintext Chebyshev LR against the reference program's pulsar cost history, and chebyshev_cipher's op
sequence and exact-scale bookkeeping run through a stand-in evaluator that carries slot values instead of ciphertexts."""
import importlib
import json
import os

import numpy as np
import pytest
import torch
from numpy.polynomial import chebyshev as Ch

PKG = "seal-fyp-logistic-regression_b200"
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _mods():
    return tuple(importlib.import_module(PKG + m) for m in (".workloads", ".lr", ".pulsar", ".parallel"))


def test_interpolant_degree_63_on_48():
    wl, lr, _, _ = _mods()
    c = wl.chebyshev_interpolant(lambda x: 1.0 / (1.0 + np.exp(-x)), 48.0, 63)
    x = np.linspace(-48.0, 48.0, 40001)
    assert np.abs(Ch.chebval(x / 48.0, c) - 1.0 / (1.0 + np.exp(-x))).max() < 1e-2     # 9.3e-3, at the steep centre
    assert c[0] == pytest.approx(0.5, abs=1e-15) and np.abs(c[2::2]).max() < 3e-15     # sigmoid - 1/2 is odd
    assert np.abs(c).sum() < 2.0
    assert np.abs(c - Ch.chebinterpolate(lambda t: 1.0 / (1.0 + np.exp(-48.0 * t)), 63)).max() < 1e-13
    assert np.array_equal(lr.SIGMOID_CHEBYSHEV.coeffs, c)


def test_depth_and_keyswitches():
    wl, _, _, par = _mods()
    assert wl.chebyshev_depth(63) == 7
    assert wl.chebyshev_keyswitches(63) == 16                 # basis 1 + 2 + 4, T_16 and T_32, giant steps 4 + 2 + 1
    for d in range(1, 130):
        assert wl.chebyshev_depth(d) <= int(d).bit_length() + 1
    R, C = 2000, 8
    assert (par.config1_keyswitches(R, C, 0, 1, method="chebyshev") - par.config1_keyswitches(R, C, 0, 1)
            == 16 - 3)
    assert par.config1_keyswitches(R, C, 1, 2, method="chebyshev") == par.config1_keyswitches(R, C, 1, 2)


@pytest.mark.parametrize("degree", [1, 2, 5, 15, 31, 63, 100])
def test_split_reassembles_the_polynomial(degree):
    """leaves combined bottom-up as chebyshev_cipher does: u_j = Y_{2j+1} T_{2^k} + Y_{2j}"""
    wl, _, _, _ = _mods()
    c = np.random.default_rng(degree).normal(size=degree + 1)
    m, l = wl._bsgs_shape(degree)
    t = np.linspace(-1, 1, 257)
    Y = [Ch.chebval(t, leaf) for leaf in wl.chebyshev_split(c, 1 << m, l)]
    assert all(len(leaf) == 1 << l for leaf in wl.chebyshev_split(c, 1 << m, l))
    k = l
    while len(Y) > 1:
        Tk = Ch.chebval(t, [0.0] * (1 << k) + [1.0])
        Y = [Y[2 * j + 1] * Tk + Y[2 * j] for j in range(len(Y) // 2)]
        k += 1
    assert k == m and np.abs(Y[0] - Ch.chebval(t, c)).max() < 1e-12


def _pulsar():
    _, lr, pulsar, _ = _mods()
    with open(os.path.join(GOLD, "pulsar_plain_lr.json")) as fh:
        gold = json.load(fh)
    X, y = pulsar.load_csv()
    Xs = pulsar.standard_scaler(X)
    return lr, pulsar, gold, Xs, Xs.astype(np.float64), y.astype(np.float64)


def test_plain_chebyshev_lr_follows_the_reference_cost_history():
    """the reference program's 100 iterations (true sigmoid) from its initial weights, lr 0.1: the degree-63 Chebyshev
    sigmoid stays within 1e-3 of every printed cost (observed 1.6e-4); the degree-3 polynomial diverges"""
    lr, pulsar, gold, Xs, X, y = _pulsar()
    w = np.array(gold["initial_weights"])
    w1 = lr.plain_epoch(X, y, w, gold["learning_rate"], method="chebyshev")
    assert np.abs(w1 - np.array(gold["weights_after_iteration_0"])).max() < 2e-4                 # observed 9.3e-5
    costs = []
    for _ in range(gold["iterations"]):
        w = lr.plain_epoch(X, y, w, gold["learning_rate"], method="chebyshev")
        costs.append(pulsar.cost_function(Xs, y, w))
    assert np.abs(np.array(costs) - np.array(gold["cost_history"])).max() < 1e-3
    assert np.abs(w - np.array(gold["final_weights"])).max() < 1e-2
    w3 = lr.plain_epoch(X, y, np.array(gold["initial_weights"]), gold["learning_rate"], 3)
    assert np.abs(w3 - np.array(gold["weights_after_iteration_0"])).max() > 1e-2                 # today's polynomial


# ------------------------------------------------------------------ chebyshev_cipher through a stand-in evaluator
class _Ct:
    """slot values [B][1][1][slots] (float64) with SEAL's metadata; getitem gives views as Ciphertext does"""

    def __init__(self, ctx, data, limbs, scale=1.0, size=2):
        self.ctx, self.data, self.limbs, self.scale, self.size = ctx, data, int(limbs), float(scale), size

    batch = property(lambda self: self.data.shape[0])

    def __getitem__(self, idx):
        return _Ct(self.ctx, self.data[idx], self.limbs, self.scale, self.size)


class _Ctx:
    def __init__(self, primes):
        self.primes = primes


class _Ev:
    """the Evaluator's scale and level arithmetic with SEAL's exact scale checks; counts relinearisations"""

    def __init__(self, ctx):
        self.ctx, self.relins = ctx, 0

    def mod_switch_to(self, x, limbs):
        assert limbs <= x.limbs
        return _Ct(x.ctx, x.data, limbs, x.scale, x.size)

    def multiply(self, a, b):
        assert a.limbs == b.limbs and (b.batch in (1, a.batch)) and a.size == b.size == 2
        return _Ct(a.ctx, a.data * b.data, a.limbs, a.scale * b.scale, 3)

    def relinearize(self, ct, keys):
        assert ct.size == 3
        self.relins += ct.batch
        return _Ct(ct.ctx, ct.data, ct.limbs, ct.scale, 2)

    def rescale_to_next_inplace(self, ct):
        ct.scale = ct.scale / float(self.ctx.primes[ct.limbs - 1])
        ct.limbs -= 1
        return ct

    def multiply_const_sum(self, cts, coeffs, pt_scales, constant=None, groups=1):
        cts = [cts] if isinstance(cts, _Ct) else list(cts)
        coeffs = np.asarray(coeffs, dtype=np.float64).reshape(groups, -1)
        T = coeffs.shape[1]
        if len(cts) == 1:
            M = cts[0].batch // T
            terms = [cts[0][i * M:(i + 1) * M] for i in range(T)]
        else:
            terms = cts
        assert len(terms) == T and len({(c.limbs, c.batch, c.size) for c in terms}) == 1
        pt = np.broadcast_to(np.asarray(pt_scales, dtype=np.float64), (groups, T))
        scale = terms[0].scale * float(pt[0, 0])
        assert all(terms[i].scale * float(pt[g, i]) == scale for g in range(groups) for i in range(T)), "scale mismatch"
        out = []
        for g in range(groups):
            acc = sum(terms[i].data * coeffs[g, i] for i in range(T))
            out.append(acc + (constant[g] if constant is not None else 0.0))
        return _Ct(terms[0].ctx, torch.cat(out, dim=0), terms[0].limbs, scale)


@pytest.mark.parametrize("degree,M", [(1, 1), (3, 1), (15, 1), (15, 3), (63, 1), (63, 2)])
def test_chebyshev_cipher_sequence_and_exact_scale(monkeypatch, degree, M):
    """values follow chebval, every sum adds equal scales, the result carries the requested scale (to the last bits),
    the levels and relinearisations are chebyshev_depth / chebyshev_keyswitches"""
    wl, _, _, _ = _mods()
    monkeypatch.setattr(wl, "Ciphertext", lambda ctx, data, limbs, scale: _Ct(ctx, data, limbs, scale))
    rng = np.random.default_rng(degree + M)
    primes = [2 ** 60 - 2 ** 26 + 1] + [int(p) for p in rng.integers(2 ** 39 + 2 ** 38, 2 ** 40 + 2 ** 38, 14) | 1] + [2 ** 60 - 93]
    ctx = _Ctx(primes)
    ev = _Ev(ctx)
    c = rng.uniform(-1, 1, degree + 1)
    t = torch.tensor(rng.uniform(-1, 1, (M, 1, 1, 64)))
    limbs = 13
    x = _Ct(ctx, t.clone(), limbs, 2.0 ** 40 * 1.37)
    out = wl.chebyshev_cipher(ev, x, c, None, scale=2.0 ** 40)
    assert abs(out.scale / 2.0 ** 40 - 1.0) < 1e-15                    # exact when a float leaf scale gets there
    assert out.limbs == limbs - wl.chebyshev_depth(degree) and out.batch == M and out.size == 2
    assert ev.relins == M * wl.chebyshev_keyswitches(degree)
    assert np.abs(out.data.numpy() - Ch.chebval(t.numpy(), c)).max() < 1e-9
