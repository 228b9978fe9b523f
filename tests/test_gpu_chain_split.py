"""The rotate-and-sum chain with c0 carried split (ckks_rotate_sum_chain on its graph-replayed steps, count >= 4).

Inside the chain c0 of dup and of acc is kept as an NTT-form part plus ONE signed integer polynomial of mod-down
remainders in coefficient order, and folded back after the last replayed step (DESIGN.md section 4).  Every returned
ciphertext must still be bit-identical to the sequential apply_galois + add of the oracle (SEAL's op sequence), across
batch sizes and lane layouts, odd tails, every rounding mode, mixed FP64 / integer prime chains, a small special prime,
a single data prime, a chunked workspace, the bench chain at N = 32768, and a second call that replays cached graphs.
"""
import numpy as np
import pytest

from test_gpu_parity import CHAINS, _random_chains

pytestmark = pytest.mark.gpu

BENCH_CHAIN = [60] + [40] * 8 + [60]


def _oracle_chain(fx, ct, count, g, keep=()):
    """sequential oracle steps of one entry: {step: (dup, acc)} for every step in keep (and the last)"""
    d, a = ct
    out = {}
    for k in range(1, count + 1):
        d = fx.orc.apply_galois(d, g, fx.gks[g])
        a = fx.orc.add(a, d)
        if k in keep or k == count:
            out[k] = (d, a)
    return out


def _run_chain(fx, dup0, acc0, count, cap=None, rounds=1):
    """the engine's chain on fresh copies of dup0 / acc0; rounds > 1 repeats the call on the same storage (cached graphs)"""
    dup, acc = fx.ctx.upload(dup0, cap=cap), fx.ctx.upload(acc0, cap=cap)
    scratch = dup.like()
    res = []
    for _ in range(rounds):
        dup.data.copy_(fx.ctx.upload(dup0, cap=cap).data)
        acc.data.copy_(fx.ctx.upload(acc0, cap=cap).data)
        last = fx.ev.rotate_sum_chain(dup, acc, 1, count, fx.keys, scratch=scratch)
        res.append((last.numpy(), acc.numpy()))
    return res


COUNTS = (4, 5, 16, 17, 35)
BATCHES = (1, 2, 4, 6, 8, 16, 17, 33)


@pytest.fixture(scope="module")
def small_case(make_fixture):
    """N = 4096, L = 2: 33 random entries and their oracle chains up to 35 steps (batch b uses the first b entries)"""
    fx = make_fixture(12, CHAINS[12])
    rng = np.random.default_rng(4242)
    dup0 = fx.random_ct(rng, max(BATCHES), 2, fx.L)
    acc0 = fx.random_ct(rng, max(BATCHES), 2, fx.L)
    g = fx.orc.galois_elt(1)
    want = [_oracle_chain(fx, (dup0[b], acc0[b]), max(COUNTS), g, keep=COUNTS) for b in range(max(BATCHES))]
    return fx, dup0, acc0, want


@pytest.mark.parametrize("batch", BATCHES)
def test_chain_split_batches_and_counts(small_case, batch):
    """graphs of 8 pairs, of 1 pair and an eager odd tail; one lane (batch 1, 2), lanes of two (4, 6, 8), two lanes
    of eight or more (16, 17, 33); the second call of each count replays the cached graphs"""
    fx, dup0, acc0, want = small_case
    for count in COUNTS:
        for r, (got_d, got_a) in enumerate(_run_chain(fx, dup0[:batch], acc0[:batch], count, rounds=2)):
            for b in range(batch):
                assert np.array_equal(got_d[b], want[b][count][0]), ("dup", count, b, r)
                assert np.array_equal(got_a[b], want[b][count][1]), ("acc", count, b, r)


@pytest.mark.parametrize("mode", [0, 1, 2, 3])
def test_chain_split_rounding_modes(make_fixture, mode):
    """the remainder w = ((t + P/2) mod P) - P/2 in rounding modes, w = t in floor modes (set_rounding 0..3)"""
    fx = make_fixture(12, CHAINS[12])
    rng = np.random.default_rng(60 + mode)
    dup0, acc0 = fx.random_ct(rng, 3, 2, fx.L), fx.random_ct(rng, 3, 2, fx.L)
    g = fx.orc.galois_elt(1)
    try:
        fx.ctx.set_rounding(mode)
        fx.orc.set_rounding(mode)
        (got_d, got_a), = _run_chain(fx, dup0, acc0, 7)
        for b in range(3):
            d, a = _oracle_chain(fx, (dup0[b], acc0[b]), 7, g)[7]
            assert np.array_equal(got_d[b], d), ("dup", mode, b)
            assert np.array_equal(got_a[b], a), ("acc", mode, b)
    finally:
        fx.ctx.set_rounding(1)
        fx.orc.set_rounding(1)


def _check_chain(fx, L, batch, count, seed, entries=None):
    rng = np.random.default_rng(seed)
    dup0, acc0 = fx.random_ct(rng, batch, 2, L), fx.random_ct(rng, batch, 2, L)
    g = fx.orc.galois_elt(1)
    (got_d, got_a), = _run_chain(fx, dup0, acc0, count, cap=fx.L)
    for b in (range(batch) if entries is None else entries):
        d, a = _oracle_chain(fx, (dup0[b], acc0[b]), count, g)[count]
        assert np.array_equal(got_d[b], d), ("dup", L, b)
        assert np.array_equal(got_a[b], a), ("acc", L, b)


@pytest.mark.parametrize("bits", _random_chains(10), ids=lambda b: "-".join(map(str, b)))
def test_chain_split_mixed_prime_chains(make_fixture, bits):
    """every placement of FP64 (below 2^41) and integer primes, the special prime included, at N = 8192"""
    fx = make_fixture(13, bits, steps=(1,))
    _check_chain(fx, fx.L, 3, 5, sum(bits))


@pytest.mark.parametrize("log_n,bits", [
    (13, [50, 30, 30, 30, 30, 40]),          # small special prime: its limb comes from the FP64 inner product
    (13, [40, 60, 40]),                      # a large prime between small ones, small special prime
    (12, [36, 36]),                          # L = 1
])
def test_chain_split_extreme_chains(make_fixture, log_n, bits):
    fx = make_fixture(log_n, bits, steps=(1,))
    for L in sorted({fx.L, 1}, reverse=True):
        _check_chain(fx, L, 4, 6, len(bits) + L)


def test_chain_split_single_limb_of_longer_chain(make_fixture):
    """L = 1 at the bottom of a longer chain (the special prime is not the next prime)"""
    _check_chain(make_fixture(12, CHAINS[12]), 1, 5, 9, 81)


def test_chain_split_chunked_workspace(make_fixture, small_case):
    """a workspace cap that splits every step into chunks of about two ciphertexts: the remainder arrays are indexed by
    the global batch entry in every chunk and lane"""
    fx, dup0, acc0, want = small_case
    fx.ctx.set_workspace_cap(3 * 8 * fx.n * 40)
    try:
        for batch in (6, 17):
            (got_d, got_a), = _run_chain(fx, dup0[:batch], acc0[:batch], 17)
            for b in range(batch):
                assert np.array_equal(got_d[b], want[b][17][0]), ("dup", batch, b)
                assert np.array_equal(got_a[b], want[b][17][1]), ("acc", batch, b)
    finally:
        fx.ctx.set_workspace_cap(1 << 30)


@pytest.fixture(scope="module")
def fx_bench(make_fixture):
    return make_fixture(15, BENCH_CHAIN, steps=(1, -16))


@pytest.mark.parametrize("batch", [32, 8, 4])
def test_chain_split_bench_chain(fx_bench, batch):
    """N = 32768, L = 3 of the bench chain, 40 steps: every entry against the GPU's own apply_galois + add, and three
    entries against the oracle"""
    fx = fx_bench
    L, count = 3, 40
    rng = np.random.default_rng(3200)
    dup0, acc0 = fx.random_ct(rng, 32, 2, L)[:batch], fx.random_ct(rng, 32, 2, L)[:batch]
    g = fx.orc.galois_elt(1)
    (got_d, got_a), = _run_chain(fx, dup0, acc0, count, cap=fx.L)
    d, a = fx.ctx.upload(dup0, cap=fx.L), fx.ctx.upload(acc0, cap=fx.L)
    for _ in range(count):
        d = fx.ev.apply_galois(d, g, fx.keys)
        a = fx.ev.add(a, d)
    assert np.array_equal(got_d, d.numpy())
    assert np.array_equal(got_a, a.numpy())
    for b in (0, 1, batch - 1):
        od, oa = _oracle_chain(fx, (dup0[b], acc0[b]), count, g)[count]
        assert np.array_equal(got_d[b], od), ("dup", b)
        assert np.array_equal(got_a[b], oa), ("acc", b)


def test_chain_unfused_pipeline_matches_oracle():
    """the unfused key-switch pipeline (CKKS_FUSE=0) has no split mode: its chains keep c0 whole and must still match the
    oracle -- the chain tests above re-run in a child process with that pipeline selected"""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, CKKS_FUSE="0")
    res = subprocess.run([sys.executable, "-m", "pytest", os.path.join(root, "tests", "test_gpu_chain_split.py"), "-m", "gpu", "-q", "-x",
                          "-k", "test_chain_split_batches_and_counts or test_chain_split_extreme_chains or test_chain_split_rounding_modes"],
                         env=env, cwd=root, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1200)
    assert res.returncode == 0 and "passed" in res.stdout, res.stdout[-2000:]
