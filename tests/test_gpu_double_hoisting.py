"""Double-hoisted rotate-multiply-sum (ckks_rotate_multiply_sum_hoisted, Evaluator.rotate_multiply_sum_hoisted).

The exact gate: the entry point's output equals, word for word, a numpy restatement of its definition built from the
oracle's per-limb ntt / intt / galois_permute and exact modular products:
    D:    digit i of c1 = INTT_i(c1[i]) lifted to [0, q_i), reduced into every prime of Q_L u {P} and NTT'd
    U:    u_z[k] = sum_i sigma_z(D_i) (.) ksk_z[i][k]                      over Q_L u {P}
    ACC:  ACC_o[k] = sum_{z in o, step != 0} w_z (.) u_z[k]                w_z = pt limbs 0..L-1 and K-1, or 1
    out:  out_o[k] = ModDown_P(ACC_o[k]) + [k = 0] sum_{step != 0} w_z (.) sigma_z(c0) + sum_{step = 0} w_z (.) c_k
Then the workloads built on it decrypt to U v and A B, within noise of the hoisted and non-empty-diagonal modes.
"""
import ctypes as C
import importlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
PKG = "seal-fyp-logistic-regression_b200"

# N = 4096: 60-bit (integer path) and 40-bit (FP64 path) data primes, a 30-bit special prime (FP64 inner product);
# and a chain whose special prime is a 60-bit integer-path prime
CHAINS = [[60, 40, 60, 40, 30], [40, 60, 60]]
STEPS = (1, -1, 2, 3, -5, 7, -16, 100, -1000, 1500)


def _obj(x):
    return np.asarray(x, dtype=np.uint64).astype(object)


def _u64(x):
    return np.asarray(x, dtype=object).astype(np.uint64)


def restate(fx, ins, pts, outputs, L, round_half):
    """numpy / oracle restatement of the entry point (module docstring); ins [A][2][L][N], pts [P][K][N]"""
    orc, primes = fx.orc, fx.primes
    K = len(primes)
    P = primes[K - 1]
    ext = list(range(L)) + [K - 1]
    digits, inner = {}, {}

    def D(a):
        if a not in digits:
            c1 = ins[a][1]
            rows = []
            for i in range(L):
                di = orc.intt(i, c1[i])
                rows.append({pj: (c1[i] if pj == i else orc.ntt(pj, di % np.uint64(primes[pj]))) for pj in ext})
            digits[a] = rows
        return digits[a]

    def u(a, step):
        if (a, step) not in inner:
            g = orc.galois_elt(step)
            key = fx.gks[g]
            res = [{}, {}]
            for k in (0, 1):
                for pj in ext:
                    acc = np.zeros(fx.n, dtype=object)
                    for i in range(L):
                        acc = (acc + _obj(orc.galois_permute(g, D(a)[i][pj])) * _obj(key[i][k][pj])) % primes[pj]
                    res[k][pj] = acc
            inner[(a, step)] = res
        return inner[(a, step)]

    out = np.zeros((len(outputs), 2, L, fx.n), dtype=np.uint64)
    half = P >> 1 if round_half else 0
    for o, terms in enumerate(outputs):
        acc = [{pj: np.zeros(fx.n, dtype=object) for pj in ext} for _ in (0, 1)]
        base = [[np.zeros(fx.n, dtype=object) for _ in range(L)] for _ in (0, 1)]
        keyswitched = False
        for a, step, p in terms:
            w = lambda pj: 1 if p < 0 else _obj(pts[p][pj])
            if step == 0:
                for k in (0, 1):
                    for j in range(L):
                        base[k][j] = (base[k][j] + w(j) * _obj(ins[a][k][j])) % primes[j]
                continue
            keyswitched = True
            g = orc.galois_elt(step)
            uz = u(a, step)
            for k in (0, 1):
                for pj in ext:
                    acc[k][pj] = (acc[k][pj] + w(pj) * uz[k][pj]) % primes[pj]
            for j in range(L):
                base[0][j] = (base[0][j] + w(j) * _obj(orc.galois_permute(g, ins[a][0][j]))) % primes[j]
        for k in (0, 1):
            if keyswitched:
                r = (_obj(orc.intt(K - 1, _u64(acc[k][K - 1]))) + half) % P
            for j in range(L):
                q = primes[j]
                v = base[k][j]
                if keyswitched:
                    t = _obj(orc.ntt(j, _u64((r - half) % q)))
                    v = (v + (acc[k][j] - t) * pow(P, -1, q)) % q
                out[o, k, j] = _u64(v)
    return out


def _table(rng, n_in, n_pt):
    """outputs of 1, 2 and >= 37 terms; step 0, repeated and negative steps, weight-1 terms, two inputs; an output of
    step-0 terms only (no key switch) and one with a single weight-1 term"""
    big = [(int(rng.integers(n_in)), int(rng.choice(STEPS + (0,))), int(rng.integers(-1, n_pt))) for _ in range(45)]
    big += [(0, 3, 0), (0, 3, 1), (1, -5, -1), (1, -5, -1)]
    return [
        [(0, 7, 2)],
        [(1, -1, 1), (0, 0, 3)],
        big,
        [(1, 0, 0), (0, 0, -1)],
        [(1, 1500, -1)],
        [(int(rng.integers(n_in)), s, int(rng.integers(n_pt))) for s in STEPS],
    ]


def _run(fx, eng, ins, pts, outputs, L, cap=None):
    ct = fx.ctx.upload(ins, cap=cap, scale=1.0)
    pt = fx.ctx.upload_plain(pts, scale=1.0)
    plan = eng.RotMulSumPlan(fx.ctx, fx.keys, ins.shape[0], pts.shape[0], outputs)
    got = fx.ev.rotate_multiply_sum_hoisted(ct, pt, plan)
    assert got.limbs == L and got.batch == len(outputs)
    return got.numpy(), plan


def _case(make_fixture, bits, seed):
    fx = make_fixture(12, bits, steps=STEPS)
    rng = np.random.default_rng(seed)
    n_in, n_pt = 2, 5
    pts = np.stack([np.stack([rng.integers(0, p, fx.n, dtype=np.uint64) for p in fx.primes]) for _ in range(n_pt)])
    return fx, rng, n_in, pts


@pytest.mark.parametrize("bits", CHAINS, ids=lambda b: "-".join(map(str, b)))
def test_exact_against_restatement(make_fixture, eng, bits):
    """top level, one level down and L = 1"""
    fx, rng, n_in, pts = _case(make_fixture, bits, sum(bits))
    outputs = _table(rng, n_in, pts.shape[0])
    for L in sorted({fx.L, fx.L - 1, 1} - {0}, reverse=True):
        ins = fx.random_ct(rng, n_in, 2, L)
        got, plan = _run(fx, eng, ins, pts, outputs, L, cap=fx.L)
        assert np.array_equal(got, restate(fx, ins, pts, outputs, L, True)), L
    nz = [[t for t in terms if t[1] != 0] for terms in outputs]
    assert plan.inner_products == sum(len(t) for t in nz) and plan.mod_downs == sum(1 for t in nz if t)


def test_rounding_modes_and_chunked_workspace(make_fixture, eng):
    fx, rng, n_in, pts = _case(make_fixture, CHAINS[0], 77)
    outputs = _table(rng, n_in, pts.shape[0])
    L = fx.L
    ins = fx.random_ct(rng, n_in, 2, L)
    try:
        for mode in (0, 1, 2, 3):
            fx.ctx.set_rounding(mode)
            got, _ = _run(fx, eng, ins, pts, outputs, L)
            assert np.array_equal(got, restate(fx, ins, pts, outputs, L, mode in (1, 2))), mode
    finally:
        fx.ctx.set_rounding(1)
    full, _ = _run(fx, eng, ins, pts, outputs, L)
    # room for the decomposition and about one output at a time: every output is a chunk of its own
    fixed = n_in * fx.n * (L + L * (L + 1)) * 8
    try:
        fx.ctx.set_workspace_cap(fixed + fx.n * (4 * L + 2) * 8 * 2)
        small, _ = _run(fx, eng, ins, pts, outputs, L)
    finally:
        fx.ctx.set_workspace_cap(1 << 30)
    assert np.array_equal(small, full)


def test_rejections(make_fixture, eng):
    capi = importlib.import_module(PKG + ".capi")
    fx, rng, n_in, pts = _case(make_fixture, CHAINS[0], 5)
    Inv = capi.CkksInvalidArgument
    L, K = fx.L, len(fx.primes)
    with pytest.raises(Inv, match="key"):                         # a step without its own key
        eng.RotMulSumPlan(fx.ctx, fx.keys, 1, 1, [[(0, 5, 0)]])
    for s in (fx.n // 2, -fx.n // 2):                             # |step| >= N/2
        with pytest.raises(Inv, match="step"):
            eng.RotMulSumPlan(fx.ctx, fx.keys, 1, 1, [[(0, s, 0)]])
    with pytest.raises(Inv, match="input index"):
        eng.RotMulSumPlan(fx.ctx, fx.keys, 1, 1, [[(1, 1, 0)]])
    with pytest.raises(Inv, match="plaintext index"):
        eng.RotMulSumPlan(fx.ctx, fx.keys, 1, 1, [[(0, 1, 1)]])
    with pytest.raises(Inv, match="plaintext index"):
        eng.RotMulSumPlan(fx.ctx, fx.keys, 1, 1, [[(0, 1, -2)]])
    lib = capi.load()
    ints = lambda xs: (C.c_int * len(xs))(*xs)
    h = C.c_void_p()
    for first in ([0, 2, 1], [1, 1, 2], [0, 1, 1], [0, 1, 3]):  # not monotone / not from 0 / not covering the 2 terms
        rc = lib.ckks_rmsplan_create(fx.ctx._h, fx.keys._h, 1, 1, 2, ints(first), 2, ints([0, 0]), ints([1, 2]),
                                     ints([0, 0]), C.byref(h))
        assert rc == capi.CKKS_ERR_INVALID, first
    assert lib.ckks_rmsplan_create(fx.ctx._h, fx.keys._h, 1, 1, 2, ints([0, 1, 2]), 2, ints([0, 0]), ints([1, 2]),
                                   ints([0, 0]), C.byref(h)) == 0
    lib.ckks_rmsplan_destroy(h)
    plan = eng.RotMulSumPlan(fx.ctx, fx.keys, 2, 2, [[(0, 1, 0)], [(1, -1, 1)]])
    ct = fx.ctx.upload(fx.random_ct(rng, 2, 2, L), scale=1.0)
    pt = fx.ctx.upload_plain(pts[:2], scale=1.0)
    ev = fx.ev
    with pytest.raises(Inv, match="key level"):                   # pts not at K limbs
        ev.rotate_multiply_sum_hoisted(ct, fx.ctx.upload_plain(pts[:2, :L], scale=1.0), plan)
    with pytest.raises(Inv, match="size"):                        # in.size != 2
        ev.rotate_multiply_sum_hoisted(fx.ctx.upload(fx.random_ct(rng, 2, 3, L), scale=1.0), pt, plan)
    with pytest.raises(Inv, match="not valid"):                   # in.limbs > K - 1
        ev.rotate_multiply_sum_hoisted(fx.ctx.upload(fx.random_ct(rng, 2, 2, K), scale=1.0), pt, plan)
    with pytest.raises(Inv, match="in batch"):
        ev.rotate_multiply_sum_hoisted(ct[0], pt, plan)
    with pytest.raises(Inv, match="out batch"):
        ev.rotate_multiply_sum_hoisted(ct, pt, plan, out=fx.ctx.upload(fx.random_ct(rng, 3, 2, L), scale=1.0))
    with pytest.raises(Inv, match="alias in"):
        ev.rotate_multiply_sum_hoisted(ct, pt, plan, out=ct)
    store = fx.ctx.upload(fx.random_ct(rng, 2, 2, K), scale=1.0)  # out in the plaintexts' storage
    pts_in_store = eng.Ciphertext(fx.ctx, store.data.view(4, 1, K, fx.n), K, 1.0)
    with pytest.raises(Inv, match="alias pts"):
        ev.rotate_multiply_sum_hoisted(ct, pts_in_store[2:4], plan, out=eng.Ciphertext(fx.ctx, store.data, L, 1.0))
    with pytest.raises(Inv, match="scale mismatch"):              # weighted and unweighted terms of one output
        mixed = eng.RotMulSumPlan(fx.ctx, fx.keys, 2, 2, [[(0, 1, 0), (1, -1, -1)], [(1, 2, 1)]])
        ev.rotate_multiply_sum_hoisted(ct, fx.ctx.upload_plain(pts[:2], scale=2.0), mixed)
    with pytest.raises(Inv, match="scale out of bounds"):
        ev.rotate_multiply_sum_hoisted(fx.ctx.upload(fx.random_ct(rng, 2, 2, L), scale=2.0 ** 100),
                                       fx.ctx.upload_plain(pts[:2], scale=2.0 ** 100), plan)


# ---------------------------------------------------------------------------------------------- workloads
def _mods():
    return (importlib.import_module(PKG + ".workloads"), importlib.import_module(PKG + ".client"),
            importlib.import_module(PKG + ".params"))


@pytest.fixture(scope="module")
def config3(eng):
    """N = 16384, {60, 40, 40, 60}: keys for every step of the d = 16 / 64 / 128 transforms, direct"""
    wl, client, params = _mods()
    ctx = eng.Context(14, params.coeff_modulus_create(14, [60, 40, 40, 60]))
    kg = client.KeyGenerator(ctx, seed=31)
    steps = set()
    for d in (16, 64, 128):
        steps |= set(wl.linear_transform_double_hoisted_steps(d))
        steps |= set(wl.bsgs_double_hoisted_steps(d, max(1, int(round(d ** 0.5)))))
    keys = kg.keyset(steps=sorted(steps), relin=False)
    return dict(ctx=ctx, ev=eng.Evaluator(ctx), enc=client.CKKSEncoder(ctx), keys=keys, plans=wl.PlanCache(ctx, keys),
                encr=client.Encryptor(ctx, kg.public_key(), seed=32), decr=client.Decryptor(ctx, kg.secret_key()))


@pytest.mark.parametrize("d", [16, 64, 128])
def test_linear_transforms_decrypt_to_Uv(config3, d):
    wl, _, _ = _mods()
    c = config3
    ctx, ev, enc = c["ctx"], c["ev"], c["enc"]
    rng = np.random.default_rng(d)
    scale = 2.0 ** 40
    U, v = rng.uniform(0, 1, (d, d)), rng.uniform(0, 1, d)
    ct = c["encr"].encrypt(enc.encode(v, scale))
    dec = lambda x: enc.decode(c["decr"].decrypt(x))[0, :d]
    ref = wl.linear_transform_plain_hoisted(ev, ct, enc.encode(wl.all_diagonals(U), scale), c["keys"], c["plans"])
    diags = enc.encode(wl.all_diagonals(U), scale, limbs=ctx.K)                       # key-level encoding
    got = wl.linear_transform_plain_double_hoisted(ev, ct, diags, c["keys"], c["plans"])
    assert got.limbs == ref.limbs and got.scale == ref.scale and got.batch == 1
    plan = c["plans"].rms(1, d, wl.diagonal_terms([range(d)], [0]))
    assert plan.mod_downs == 1 and plan.inner_products == d - 1
    assert np.abs(dec(got) - U @ v).max() < 1e-4
    assert np.abs(dec(got) - dec(ref)).max() < 1e-4
    bd = wl.BsgsDiagonals(U, scale, enc, limbs=ctx.K)
    got = wl.linear_transform_plain_bsgs_double_hoisted(ev, ct, bd, c["keys"], c["plans"])
    assert got.limbs == ref.limbs and got.scale == ref.scale
    assert np.abs(dec(got) - U @ v).max() < 1e-4
    assert np.abs(dec(got) - dec(ref)).max() < 1e-4


@pytest.mark.parametrize("d", [8, 64])
def test_matmul_nonzero_hoisted_decrypts_to_product(eng, d):
    """config-4 chain {60, 40 x 4, 60} at N = 16384"""
    wl, client, params = _mods()
    ctx = eng.Context(14, params.coeff_modulus_create(14, [60, 40, 40, 40, 40, 60]))
    ev, enc = eng.Evaluator(ctx), client.CKKSEncoder(ctx)
    kg = client.KeyGenerator(ctx, seed=43)
    keys = kg.keyset(steps=wl.matmul_nonzero_hoisted_steps(d))
    encr, decr = client.Encryptor(ctx, kg.public_key(), seed=44), client.Decryptor(ctx, kg.secret_key())
    plans = wl.PlanCache(ctx, keys)
    rng = np.random.default_rng(d)
    scale, eps, dd = 2.0 ** 40, 1e-8, d * d
    A, B = rng.uniform(0, 1, (d, d)), rng.uniform(0, 1, (d, d))
    ctA = encr.encrypt(enc.encode(A.reshape(-1), scale))
    ctB = encr.encrypt(enc.encode(B.reshape(-1), scale))
    both = lambda U: (wl.DiagonalSet.from_matrix(U, eps, scale, enc), wl.DiagonalSet.from_matrix(U, eps, scale, enc, limbs=ctx.K))
    sig, tau = both(wl.u_sigma(d)), both(wl.u_tau(d))      # one dense d^2 x d^2 matrix alive at a time
    V = [both(wl.v_k(d, k)) for k in range(1, d)]
    W = [both(wl.w_k(d, k)) for k in range(1, d)]
    ref = wl.cc_matrix_multiplication_nonzero(ev, ctA, ctB, d, sig[0], tau[0], [v[0] for v in V], [w[0] for w in W], keys, plans)
    got = wl.cc_matrix_multiplication_nonzero_hoisted(ev, ctA, ctB, d, sig[1], tau[1], [v[1] for v in V], [w[1] for w in W],
                                                      keys, plans)
    assert got.size == 3 and got.limbs == ref.limbs and got.scale == ref.scale
    dec = lambda x: enc.decode(decr.decrypt(x))[0, :dd].reshape(d, d)
    assert np.abs(dec(got) - A @ B).max() < 1e-3
    assert np.abs(dec(got) - dec(ref)).max() < 1e-3


def test_cpp_linear_transform_double_hoisted(pkg, tmp_path):
    """tests/cpp/double_hoisting_driver.cpp, compiled here against seal/seal.h and ckks_b200_helper.h: the C++ transform
    decrypts to U v within 1e-4"""
    import os
    import subprocess
    import test_shim
    exe = str(tmp_path / "double_hoisting_driver")
    res = subprocess.run(["g++", "-std=c++17", "-O2"] + test_shim.INC +
                         [os.path.join(test_shim.ROOT, "tests", "cpp", "double_hoisting_driver.cpp"), "-o", exe, test_shim.LIB,
                          "-Wl,-rpath," + os.path.dirname(test_shim.LIB)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert res.returncode == 0, res.stdout[-3000:]
    run = subprocess.run([exe], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert run.returncode == 0 and "DOUBLE HOISTED OK" in run.stdout, run.stdout[-3000:]
