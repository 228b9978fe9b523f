"""Column-layout encrypted LR with the Chebyshev sigmoid on the host (CPU-only): the weight packing with the 1/bound
folded into the broadcasts, a slot-level numpy restatement of column_epoch_gradient against plaintext Chebyshev LR, the
(mini-batch, feature) unit partition, the key-switch and level counts, and the sigmoids the sharded loop refuses."""
import importlib
import json
import os

import numpy as np
import pytest
from numpy.polynomial import chebyshev as Ch

PKG = "seal-fyp-logistic-regression_b200"
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _mods():
    return tuple(importlib.import_module(PKG + m) for m in (".workloads", ".lr", ".pulsar", ".parallel"))


def _pulsar():
    _, _, pulsar, _ = _mods()
    with open(os.path.join(GOLD, "pulsar_plain_lr.json")) as fh:
        gold = json.load(fh)
    X, y = pulsar.load_csv()
    return gold, pulsar.standard_scaler(X).astype(np.float64), y.astype(np.float64)


def test_weight_packing():
    _, lr, _, _ = _mods()
    lay = lr.ColumnLayout(64, 4, 16, 128)
    w = np.array([0.5, -1.25, 3.0, 2.0])
    packed = lay.weights(w)
    assert packed.shape == (128,) and np.array_equal(packed[:4], w) and not packed[4:].any()
    for method in ("tree", "horner"):
        wb = lay.weight_broadcasts(w, method)
        assert wb.shape == (4, 128) and np.array_equal(wb, np.repeat(w[:, None], 128, axis=1))
    wb = lay.weight_broadcasts(w, "chebyshev")
    assert np.array_equal(wb, np.repeat(w[:, None] / lr.SIGMOID_CHEBYSHEV.bound, 128, axis=1))
    sig = lr.ChebyshevSigmoid(15, 8.0)
    assert np.array_equal(lay.weight_broadcasts(w, "chebyshev", sig)[:, 0], w / 8.0)


def _rotate(v, steps):
    """SEAL rotate_vector on the slot vector: slot i of the result is slot i + steps of v"""
    return np.roll(v, -steps)


def _slot_epoch(lay, X, y, w, sig):
    """column_epoch_gradient(method="chebyshev") restated on slot vectors: prediction sum_j col_j * wb_j, the
    polynomial, minus the labels, then per (m, j) the reference's cipher_dot_product (duplicate by rotate(-B), B - 1
    unit rotations summed), the one-hot mask e_j, and the sum over every unit"""
    cols, labs = lay.columns(X), lay.labels(y)
    wb = lay.weight_broadcasts(w, "chebyshev", sig)
    C, B = lay.C, lay.B
    grad = np.zeros(lay.slots)
    for m in range(lay.M):
        z = sum(cols[m * C + j] * wb[j] for j in range(C))
        pl = Ch.chebval(z, sig.coeffs) - labs[m]
        for j in range(C):
            mult = cols[m * C + j] * pl
            dup = mult + _rotate(mult, -B)
            for _ in range(B - 1):
                dup = _rotate(dup, 1)
                mult = mult + dup
            mask = np.zeros(lay.slots)
            mask[j] = 1.0
            grad += mult * mask
    return grad


@pytest.mark.parametrize("div", [1, 2, 8])
def test_slot_restatement_equals_plaintext_chebyshev_lr(div):
    _, lr, _, _ = _mods()
    rng = np.random.default_rng(div)
    R, C = 64, 4
    X, y, w = rng.normal(0, 2, (R, C)), (rng.uniform(0, 1, R) > 0.5).astype(float), rng.uniform(-3, 3, C)
    lay = lr.ColumnLayout(R, C, R // div, 256)
    sig = lr.SIGMOID_CHEBYSHEV
    grad = _slot_epoch(lay, X, y, w, sig)
    assert not grad[C:].any()
    new = w - (0.1 / R) * grad[:C]                                   # apply_gradient
    assert np.abs(new - lr.plain_epoch(X, y, w, 0.1, method="chebyshev")).max() < 1e-12


def test_slot_restatement_on_pulsar():
    _, lr, _, _ = _mods()
    gold, X, y = _pulsar()
    w0 = np.array(gold["initial_weights"])
    R = X.shape[0]
    lay = lr.ColumnLayout(R, X.shape[1], R // 8, 16384)
    # one unit's chain is B - 1 = 249 rotations of a 16384-slot vector: check the units of mini-batch 0 against numpy
    Xm, ym = X[:lay.B], y[:lay.B]
    sub = lr.ColumnLayout(lay.B, lay.C, lay.B, lay.slots)
    grad = _slot_epoch(sub, Xm, ym, w0, lr.SIGMOID_CHEBYSHEV)[:lay.C]
    assert np.abs(grad - Xm.T @ (lr.SIGMOID_CHEBYSHEV(Xm @ w0) - ym)).max() < 1e-9


@pytest.mark.parametrize("M,C", [(1, 8), (8, 8), (16, 8), (3, 5)])
def test_column_units_cover_every_unit_once(M, C):
    par = _mods()[3]
    everything = [(m, j) for m in range(M) for j in range(C)]
    for world in range(1, M * C + 2):
        got = [par.column_units(M, C, r, world) for r in range(world)]
        assert [u for part in got for u in part] == everything, world     # contiguous, in (m, j) order
        sizes = [len(part) for part in got]
        assert max(sizes) - min(sizes) <= 1
    assert par.column_units(M, C, M * C, M * C + 1) == []


def test_column_keyswitches():
    wl, _, _, par = _mods()
    R, C, deg = 2000, 8, wl.chebyshev_keyswitches(63)

    def formula(B):
        M = R // B
        return M * (1 + deg) + M * C * (1 + par.naf_weight(-B) + B - 1)
    assert par.naf_weight(-2000) == par.naf_weight(-250) == 3
    assert par.column_keyswitches(R, C, 2000, 0, 1, "chebyshev") == formula(2000) == 16041
    assert par.column_keyswitches(R, C, 250, 0, 1, "chebyshev") == formula(250) == 16328
    for B, busiest in ((250, (8164, 4082, 2041)), (2000, (8029, 4023, 2020))):
        for world, want in zip((2, 4, 8), busiest):
            assert max(par.column_keyswitches(R, C, B, r, world, "chebyshev") for r in range(world)) == want, (B, world)
    # the bench.py epoch (tree degree 7, 32768 x 8 in mini-batches of 8192): 6 relinearisations per mini-batch
    assert par.column_keyswitches(32768, 8, 8192, 0, 1, "tree") == 4 * 7 + 32 * (1 + 1 + 8191)
    assert par.column_keyswitches(R, C, 250, 64, 65, "chebyshev") == 0


def test_column_level_count():
    wl, lr, _, _ = _mods()
    assert wl.chebyshev_depth(lr.SIGMOID_CHEBYSHEV.degree) == 7
    assert lr.column_rescales("chebyshev") == 11                   # 1 + 7 + 1 + 1 + 1: {60, 40 x 11, 60}
    assert lr.column_rescales("tree", 7) == 8                      # bench.py's {60, 40 x 8, 60}
    assert lr.column_rescales("horner", 3) == 7
    assert lr.column_rescales("chebyshev", sigmoid=lr.ChebyshevSigmoid(15, 8.0)) == 4 + wl.chebyshev_depth(15)


@pytest.mark.parametrize("method", ["tree", "horner"])
def test_sharded_train_columns_rejects_reference_polynomials(method):
    par = _mods()[3]
    with pytest.raises(ValueError, match="encrypt a coefficient"):
        par.sharded_train_columns(None, None, None, [], [], None, None, 0.1, 1, None, 2.0 ** 40, None, None, None, None,
                                  0, 1, None, method=method)
