"""CPU: the host side of the blocked encrypted matrix product (workloads.cc_matrix_multiplication_blocked): the tile
helpers, the decomposition C_ij = sum_l sum_k X_{il,k} (.) Y_{lj,k} restated on slot vectors, and the partition of the
sharded form (parallel.blocked_shards).  The GPU side is tests/test_gpu_matmul_blocked.py."""
import importlib

import numpy as np
import pytest

PKG = "seal-fyp-logistic-regression_b200"


def _mods():
    return importlib.import_module(PKG + ".workloads"), importlib.import_module(PKG + ".parallel")


@pytest.mark.parametrize("shape,d", [((20, 13), 8), ((8, 8), 8), ((1, 1), 4), ((64, 130), 64), ((7, 3), 2), ((5, 17), 4)])
def test_tiles_round_trip(shape, d):
    wl, _ = _mods()
    M = np.random.default_rng(sum(shape) + d).normal(size=shape)
    tiles, grid = wl.matrix_tiles(M, d)
    assert grid == (-(-shape[0] // d), -(-shape[1] // d))
    assert tiles.shape == (grid[0] * grid[1], d * d)
    assert np.array_equal(wl.matrix_from_tiles(tiles, shape, d), M)
    # row-major tile order, row-major d^2-slot layout, zero padding
    for tr in range(grid[0]):
        for tc in range(grid[1]):
            T = tiles[tr * grid[1] + tc].reshape(d, d)
            blk = M[tr * d:(tr + 1) * d, tc * d:(tc + 1) * d]
            assert np.array_equal(T[:blk.shape[0], :blk.shape[1]], blk)
            assert not T[blk.shape[0]:].any() and not T[:, blk.shape[1]:].any()
    # decoded tiles carry more slots than d^2 (the duplicate half): ignored
    wide = np.concatenate([tiles, np.ones_like(tiles)], axis=1)
    assert np.array_equal(wl.matrix_from_tiles(wide, shape, d), M)


def _sigma(x, d):
    X = x.reshape(d, d)
    i, j = np.meshgrid(np.arange(d), np.arange(d), indexing="ij")
    return X[i, (i + j) % d].reshape(-1)


def _tau(x, d):
    X = x.reshape(d, d)
    i, j = np.meshgrid(np.arange(d), np.arange(d), indexing="ij")
    return X[(i + j) % d, j].reshape(-1)


def _v(x, d, k):
    X = x.reshape(d, d)
    return np.roll(X, -k, axis=1).reshape(-1)       # V_k: entry (i, j) <- (i, j + k)


def _w(x, d, k):
    X = x.reshape(d, d)
    return np.roll(X, -k, axis=0).reshape(-1)       # W_k: entry (i, j) <- (i + k, j)


def test_closed_forms_match_the_permutation_matrices():
    wl, _ = _mods()
    d = 5
    x = np.random.default_rng(1).normal(size=d * d)
    assert np.array_equal(wl.u_sigma(d) @ x, _sigma(x, d))
    assert np.array_equal(wl.u_tau(d) @ x, _tau(x, d))
    for k in range(1, d):
        assert np.array_equal(wl.v_k(d, k) @ x, _v(x, d, k))
        assert np.array_equal(wl.w_k(d, k) @ x, _w(x, d, k))


def _entries(tiles, d, side):
    """the d slot vectors of each tile: k = 0 is sigma (tau), k >= 1 V_k sigma (W_k tau)"""
    out = []
    for t in tiles:
        x0 = _sigma(t, d) if side == 0 else _tau(t, d)
        out.append([x0] + [(_v if side == 0 else _w)(x0, d, k) for k in range(1, d)])
    return np.array(out)                              # [tiles, d, d*d]


@pytest.mark.parametrize("n,m,p,d", [(20, 13, 9, 8), (8, 8, 8, 8), (3, 17, 5, 4), (16, 4, 1, 4), (1, 9, 12, 8)])
def test_decomposition_is_the_matrix_product(n, m, p, d):
    wl, _ = _mods()
    rng = np.random.default_rng(n * m * p)
    A, B = rng.uniform(-1, 1, (n, m)), rng.uniform(-1, 1, (m, p))
    At, (tn, tm) = wl.matrix_tiles(A, d)
    Bt, (tm2, tp) = wl.matrix_tiles(B, d)
    assert tm == tm2
    X, Y = _entries(At, d, 0), _entries(Bt, d, 1)
    # the contraction: (t_n x t_m d) by (t_m d x t_p) with slot-wise products
    Xm = X.reshape(tn, tm * d, d * d)
    Ym = Y.reshape(tm, tp, d, d * d).transpose(0, 2, 1, 3).reshape(tm * d, tp, d * d)
    C = np.einsum("irs,rjs->ijs", Xm, Ym).reshape(tn * tp, d * d)
    assert np.allclose(wl.matrix_from_tiles(C, (n, p), d), A @ B, atol=1e-12)
    # ... which is the sum over l of the per-tile products
    for i in range(tn):
        for j in range(tp):
            per = sum((X[i * tm + l] * Y[l * tp + j]).sum(0) for l in range(tm))
            assert np.allclose(per, C[i * tp + j], atol=1e-12)


@pytest.mark.parametrize("tiles", [(2, 3, 2), (1, 1, 1), (4, 4, 4), (3, 1, 5), (1, 7, 1)])
def test_shard_partition_covers_everything_once(tiles):
    _, par = _mods()
    tn, tm, tp = tiles
    n_tr, n_out = tn * tm + tm * tp, tn * tp
    for G in list(range(1, 10)) + [n_tr + 1, n_out + 1, 2 * n_tr + 3]:
        shards = [par.blocked_shards(tiles, r, G) for r in range(G)]
        tr = [list(s[0]) for s in shards]
        out = [list(s[1]) for s in shards]
        assert sum(tr, []) == list(range(n_tr)), G                 # contiguous runs, in order, each once
        assert sum(out, []) == list(range(n_out)), G
        for parts, total in ((tr, n_tr), (out, n_out)):
            sizes = [len(x) for x in parts]
            assert max(sizes) - min(sizes) <= 1 and max(sizes) == -(-total // G), G   # balanced
            if G > total:
                assert sizes.count(0) == G - total
