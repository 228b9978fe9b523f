"""CPU: the term partition of the sharded double-hoisted workloads (parallel.shard_terms) and the Galois step sets of each
rank.  The GPU side, bit-identity with one GPU, is tests/test_gpu_sharded_double_hoisting.py."""
import importlib

import numpy as np
import pytest

PKG = "seal-fyp-logistic-regression_b200"


def _mods():
    return importlib.import_module(PKG + ".workloads"), importlib.import_module(PKG + ".parallel")


def _tables():
    wl, _ = _mods()
    rng = np.random.default_rng(3)
    rand = [[(int(rng.integers(2)), int(rng.choice([0, 0, 1, -3, 7])), int(rng.integers(-1, 4)))
             for _ in range(int(rng.integers(0, 9)))] for _ in range(11)]
    yield "random", rand
    yield "one-output", wl.diagonal_terms([range(64)], [0])
    baby, giant = wl.bsgs_terms(128, 11)
    yield "bsgs-baby", baby
    yield "bsgs-giant", giant
    yield "matmul-8", wl.matmul_nonzero_hoisted_terms(*wl.matmul_diagonal_indices(8))[0]
    yield "step0-only", [[(0, 0, 0), (0, 0, -1)], [], [(0, 0, 1)]]
    yield "empty", [[], []]


@pytest.mark.parametrize("G", range(1, 18))
def test_shard_terms_covers_once_in_order_and_balanced(G):
    _, par = _mods()
    for name, outputs in _tables():
        shares = [par.shard_terms(outputs, r, G) for r in range(G)]
        assert shares == [par.shard_terms(outputs, r, G) for r in range(G)], name      # deterministic
        total = sum(1 for terms in outputs for t in terms if t[1] != 0)
        loads = []
        for r, share in enumerate(shares):
            assert len(share) == len(outputs), name
            loads.append(sum(1 for terms in share for t in terms if t[1] != 0))
        for o, terms in enumerate(outputs):
            # every term exactly once: the ranks' runs, in rank order, concatenate to the output's term list
            assert [t for share in shares for t in share[o]] == list(terms), (name, o)
            # each rank's run is contiguous in the output's list
            pos = 0
            for share in shares:
                run = share[o]
                assert list(terms[pos:pos + len(run)]) == run, (name, o)
                pos += len(run)
        assert sum(loads) == total
        assert max(loads) <= -(-total // G) + len(outputs), (name, loads)
        assert max(loads) - min(loads) <= 1, (name, loads)


@pytest.mark.parametrize("G", [1, 2, 3, 4, 8, 17])
def test_rank_steps_complete_minimal_and_cover_one_gpu(G):
    wl, par = _mods()
    for d in (16, 64, 128):
        lt = wl.diagonal_terms([range(d)], [0])
        shares = {r: par.shard_terms(lt, r, G) for r in range(G)}
        for r in range(G):   # complete and minimal: the steps of the rank's terms, plus the fill when it has any term
            has = any(shares[r])
            assert par.linear_transform_double_hoisted_rank_steps(d, r, G) == sorted(
                wl.term_steps(shares[r]) | ({-d} if has else set()))
        assert set().union(*(par.linear_transform_double_hoisted_rank_steps(d, r, G) for r in range(G))) == set(
            wl.linear_transform_double_hoisted_steps(d))

        b = max(1, int(round(d ** 0.5)))
        baby, _ = wl.bsgs_terms(d, b)
        for r in range(G):
            own = list(par.owned_block(len(baby), r, G))
            want = {s for g in own for _, s, _ in baby[g] if s != 0} | {g * b for g in own if g} | ({-d} if own else set())
            assert par.bsgs_double_hoisted_rank_steps(d, b, r, G) == sorted(want), (d, G, r)
        assert set().union(*(par.bsgs_double_hoisted_rank_steps(d, b, r, G) for r in range(G))) == set(
            wl.bsgs_double_hoisted_steps(d, b))
    for d in (8, 16):
        sig, tau, V, W = wl.matmul_diagonal_indices(d)
        first, second = wl.matmul_nonzero_hoisted_terms(sig, tau, V, W)
        for r in range(G):
            mine = par.shard_terms(first, r, G)
            own = list(par.owned_block(d - 1, r, G))
            want = wl.term_steps(mine) | {l for k in own for l in list(V[k]) + list(W[k]) if l != 0}
            want |= {-d * d} if any(mine) or own else set()
            assert par.matmul_nonzero_hoisted_rank_steps(d, r, G) == sorted(want), (d, G, r)
        assert set().union(*(par.matmul_nonzero_hoisted_rank_steps(d, r, G) for r in range(G))) == set(
            wl.matmul_nonzero_hoisted_steps(d))


def test_rank_tables_apply_to_the_one_gpu_sums():
    """numpy slot restatement: summing the ranks' shares of a term table gives the one-GPU sums, and the BSGS ranks'
    giant terms over their own baby outputs add up to the BSGS transform"""
    wl, par = _mods()
    rng = np.random.default_rng(9)
    n, d = 256, 16
    x = rng.uniform(-1, 1, (2, n))
    pts = rng.uniform(-1, 1, (40, n))

    def apply(outputs, ins, pts):
        return np.array([sum(((pts[p] if p >= 0 else 1.0) * np.roll(ins[a], -s) for a, s, p in terms),
                             np.zeros(n)) for terms in outputs])
    lt = wl.diagonal_terms([range(d)], [0])
    for G in (1, 2, 3, 8, 17):
        got = sum(apply(par.shard_terms(lt, r, G), x, pts) for r in range(G))
        assert np.allclose(got, apply(lt, x, pts))
    b = 4
    baby, giant = wl.bsgs_terms(d, b)
    want = apply(giant, apply(baby, x, pts), None)
    for G in (1, 2, 3, 5, 8):
        total = np.zeros((1, n))
        for r in range(G):
            own, rb, rg = par._bsgs_rank_tables(d, b, r, G)
            if own:
                total += apply(rg, apply(rb, x, pts), None)
        assert np.allclose(total, want), G
