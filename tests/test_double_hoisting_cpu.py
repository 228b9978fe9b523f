"""CPU: the term tables of the double-hoisted workloads (workloads.linear_transform_plain_double_hoisted, the BSGS variant and
cc_matrix_multiplication_nonzero_hoisted), applied as slot rotations and products in numpy, reproduce U v, the BSGS sum and
A B; and their Galois step sets are complete and minimal.  The GPU entry point itself is covered by
tests/test_gpu_double_hoisting.py."""
import importlib

import numpy as np
import pytest

PKG = "seal-fyp-logistic-regression_b200"


def _wl():
    return importlib.import_module(PKG + ".workloads")


class SlotEncoder:
    """stands in for CKKSEncoder: a 'plaintext' is its slot vector"""

    def __init__(self, slots):
        self.slots = slots

    def encode(self, values, scale, limbs=None):
        v = np.atleast_2d(np.asarray(values, dtype=np.float64))
        out = np.zeros((v.shape[0], self.slots))
        out[:, :v.shape[1]] = v
        return out


def rot(x, s):
    """rotate_vector on slot vectors: rot(x, s)[i] = x[(i + s) mod n]"""
    return np.roll(x, -s)


def apply_terms(outputs, inputs, pts):
    """out[o] = sum_{(a, s, p) in outputs[o]} pts[p] (.) rot(inputs[a], s)   (p = -1: weight 1)"""
    outs = []
    for terms in outputs:
        acc = np.zeros(inputs.shape[1])
        for a, s, p in terms:
            r = rot(inputs[a], s)
            acc += r if p < 0 else pts[p] * r
        outs.append(acc)
    return np.array(outs)


def dup(x, d):
    """duplicate_fill: x + rot(x, -d)"""
    return x + rot(x, -d)


def _used(*tables):
    return {s for outputs in tables for terms in outputs for _, s, _ in terms}


@pytest.mark.parametrize("d", [16, 64, 128])
def test_linear_transform_terms(d):
    wl = _wl()
    rng = np.random.default_rng(d)
    n = 4 * d
    U, v = rng.uniform(-1, 1, (d, d)), rng.uniform(-1, 1, d)
    x = np.zeros(n)
    x[:d] = v
    diags = SlotEncoder(n).encode(wl.all_diagonals(U), 1.0)
    table = wl.diagonal_terms([range(d)], [0])
    assert len(table) == 1 and len(table[0]) == d                      # one output of d terms
    out = apply_terms(table, dup(x, d)[None], diags)
    assert np.allclose(out[0, :d], U @ v)
    steps = wl.linear_transform_double_hoisted_steps(d)
    assert set(steps) == {-d} | set(range(1, d))
    assert set(steps) == ({-d} | _used(table)) - {0}                   # complete and minimal


@pytest.mark.parametrize("d,b", [(16, None), (64, 16), (128, None), (128, 16), (100, 7)])
def test_bsgs_terms(d, b):
    wl = _wl()
    rng = np.random.default_rng(d + 1)
    n = 4 * d
    U, v = rng.uniform(-1, 1, (d, d)), rng.uniform(-1, 1, d)
    x = np.zeros(n)
    x[:d] = v
    bd = wl.BsgsDiagonals(U, 1.0, SlotEncoder(n), baby=b, limbs=4)   # key-level encoding is accepted
    baby, giant = wl.bsgs_terms(bd.d, bd.b)
    assert len(baby) == bd.G and sum(len(t) for t in baby) == d
    assert len(giant) == 1 and len(giant[0]) == bd.G and all(p == -1 for _, _, p in giant[0])
    inner = apply_terms(baby, dup(x, d)[None], bd.plain)
    out = apply_terms(giant, inner, None)
    assert np.allclose(out[0, :d], U @ v)
    steps = wl.bsgs_double_hoisted_steps(d, bd.b)
    assert set(steps) == {-d} | set(range(1, bd.b)) | {g * bd.b for g in range(1, bd.G)}
    assert set(steps) == ({-d} | _used(baby, giant)) - {0}


@pytest.mark.parametrize("d", [4, 8])
def test_matmul_terms(d):
    wl = _wl()
    rng = np.random.default_rng(d + 2)
    dd = d * d
    n = 4 * dd
    enc = SlotEncoder(n)
    A, B = rng.uniform(-1, 1, (d, d)), rng.uniform(-1, 1, (d, d))
    sig = wl.DiagonalSet.from_matrix(wl.u_sigma(d), 0.0, 1.0, enc, limbs=4)
    tau = wl.DiagonalSet.from_matrix(wl.u_tau(d), 0.0, 1.0, enc, limbs=4)
    V = [wl.DiagonalSet.from_matrix(wl.v_k(d, k), 0.0, 1.0, enc, limbs=4) for k in range(1, d)]
    W = [wl.DiagonalSet.from_matrix(wl.w_k(d, k), 0.0, 1.0, enc, limbs=4) for k in range(1, d)]
    # the closed-form diagonal indices are those of the dense matrices
    ci = wl.matmul_diagonal_indices(d)
    assert ci[0] == sig.index and ci[1] == tau.index
    assert ci[2] == [s.index for s in V] and ci[3] == [s.index for s in W]
    first, second = wl.matmul_nonzero_hoisted_terms(sig.index, tau.index, [s.index for s in V], [s.index for s in W])
    assert len(first) == 2 and len(second) == 2 * (d - 1)
    assert [len(t) for t in second] == [2] * (d - 1) + [1] * (d - 1)   # V_k: 2 non-empty diagonals, W_k: 1
    a, b = np.zeros(n), np.zeros(n)
    a[:dd], b[:dd] = A.ravel(), B.ravel()
    AB0 = apply_terms(first, np.array([dup(a, dd), dup(b, dd)]), np.concatenate([sig.special, tau.special]))
    pts2 = np.concatenate([s.special for s in V + W])
    step2 = apply_terms(second, np.array([dup(AB0[0], dd), dup(AB0[1], dd)]), pts2)
    C = AB0[0] * AB0[1] + sum(step2[k] * step2[d - 1 + k] for k in range(d - 1))
    assert np.allclose(C[:dd], (A @ B).ravel())
    steps = wl.matmul_nonzero_hoisted_steps(d)
    assert set(steps) == ({-dd} | _used(first, second)) - {0}
    assert set(steps) == ({-dd} | set(sig.index) | set(tau.index) | {l for s in V + W for l in s.index}) - {0}


def test_matmul_steps_at_64():
    """the d = 64 step set: U_sigma has 127 non-empty diagonals, U_tau 64, V_k 2 and W_k 1 each"""
    wl = _wl()
    sig, tau, V, W = wl.matmul_diagonal_indices(64)
    assert len(sig) == 127 and len(tau) == 64
    assert all(len(v) == 2 for v in V) and all(len(w) == 1 for w in W)
    steps = wl.matmul_nonzero_hoisted_steps(64)
    assert -4096 in steps and 0 not in steps
    assert len(steps) == len(set(steps))
