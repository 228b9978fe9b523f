"""The reference's layer-2 HE algorithms, re-expressed over the batched GPU Evaluator.

Every function names the reference function it mirrors (file:line) and issues the SAME evaluator
op sequence per ciphertext; what changes is only the grouping: independent ciphertexts are
batched into single kernel launches (rotation plans, fused multiply+add_many), and identical
sub-computations the reference repeats (the rotations of one ciphertext shared by many linear
transforms) are computed once.  Both transformations keep every evaluated ciphertext polynomial
bit-identical to the sequential reference (modular sums are order-independent).
"""
import math

import numpy as np
import torch

from . import capi
from .engine import Ciphertext, RotPlan


def force_scale_pow2(ct):
    """`x.scale() = pow(2, (int)log2(x.scale()))` -- the reference's "manual rescale"
    (helper.h:489, matrix_multiplication.cpp:119-120, logistic_regression_ckks.cpp:241)"""
    ct.scale = float(2.0 ** int(math.log2(ct.scale)))
    return ct


class PlanCache:
    """rotation plans keyed by their step list (plans hold device-side schedules)"""

    def __init__(self, ctx, keys):
        self.ctx, self.keys, self._plans = ctx, keys, {}

    def get(self, steps):
        key = tuple(int(s) for s in steps)
        if key not in self._plans:
            self._plans[key] = RotPlan(self.ctx, self.keys, key)
        return self._plans[key]


# ------------------------------------------------------------------ linear transforms
def duplicate_fill(ev, ct, d, keys):
    """"Fill ct with duplicate": ct + rotate_vector(ct, -d)   (helper.h:241-247)"""
    return ev.add(ct, ev.rotate_vector(ct, -d, keys))


def rotations_of(ev, ct_new, d, plans):
    """all d rotations rot(ct_new, l), l = 0..d-1, of the hot loop helper.h:252-257, batched"""
    return ev.rotate_plan(ct_new, plans.get(range(d)))


def linear_transform_plain(ev, ct, diags, keys, plans, rots=None):
    """Linear_Transform_Plain (helper.h:237-262; linear_transformation.cpp:149-174):
    sum_l diag_l (.) rot(ct + rot(ct,-d), l).  `diags`: Plaintext batch of d diagonals."""
    d = diags.batch
    if rots is None:
        rots = rotations_of(ev, duplicate_fill(ev, ct, d, keys), d, plans)
    return ev.multiply_plain_sum(rots, diags)


def linear_transform_cipher(ev, ct, diag_cts, keys, plans):
    """Linear_Transform_Cipher (helper.h:212-234): ciphertext diagonals, size-3 result"""
    d = diag_cts.batch
    rots = rotations_of(ev, duplicate_fill(ev, ct, d, keys), d, plans)
    return ev.multiply_sum(rots, diag_cts)


class BsgsDiagonals:
    """the d diagonals of a transform, pre-rotated for the baby-step / giant-step evaluation
    (SURVEY 8(f4)): diagonal l = g*b + s is encoded with its entries moved to slots [g*b, g*b + d)."""

    def __init__(self, U, scale, encoder, baby=None, limbs=None):
        d = U.shape[0]
        self.d = d
        self.b = int(baby) if baby else max(1, int(round(math.sqrt(d))))
        self.G = (d + self.b - 1) // self.b
        diags = all_diagonals(U)
        vals = np.zeros((d, 2 * d))
        for l in range(d):
            off = (l // self.b) * self.b
            vals[l, off:off + d] = diags[l]
        self.plain = encoder.encode(vals, scale, limbs=limbs)      # batch d, entry l


def linear_transform_plain_bsgs(ev, ct, bd, keys, plans):
    """Linear_Transform_Plain by baby steps and giant steps (SURVEY 8(f4)) -- an explicit,
    tolerance-checked alternative to linear_transform_plain, never the default:
        sum_g rot( sum_s rot(diag_{gb+s}, -gb) (.) rot(ct + rot(ct,-d), s), gb )
    b + G - 2 composite rotations instead of d - 1; the decrypted result equals the reference
    sequence within noise, the ciphertext polynomials do not."""
    d, b, G = bd.d, bd.b, bd.G
    dup = duplicate_fill(ev, ct, d, keys)
    baby = ev.rotate_plan(dup, plans.get(range(b)))                # batch b: rot(dup, s)
    inner = []
    for g in range(G):
        lo, hi = g * b, min(d, (g + 1) * b)
        pts = Ciphertext(bd.plain.ctx, bd.plain.data[lo:hi], bd.plain.limbs, bd.plain.scale)
        inner.append(ev.multiply_plain_sum(baby[0:hi - lo], pts))
    giant = ev.rotate_plan(_stack(inner), plans.get([g * b for g in range(G)]))
    return ev.add_many(giant)


def linear_transform_plain_hoisted(ev, ct, diags, keys, plans):
    """Linear_Transform_Plain (helper.h:237-262) with HOISTED rotations (SURVEY 8(f4)): all d-1 rotations of the hot loop
    act on the same ct_new (helper.h:252-257), so its digit decomposition is computed once and every rotation only permutes
    the extended digits, multiplies by its own key and mods down.  `keys` must hold a Galois key for every step 1..d-1 and
    for -d (KeyGenerator.keyset(steps=[-d] + list(range(1, d)))).  d key-switch inner products instead of sum_l NAF(l) full
    key switches (d = 128: 128 instead of 356, each ~45 % of the NTT work).  Same decrypted vector as the reference sequence
    within noise; ciphertext polynomials differ -- a tolerance-checked mode, never the default."""
    d = diags.batch
    rots = ev.rotate_plan_hoisted(duplicate_fill(ev, ct, d, keys), plans.get(range(d)))
    return ev.multiply_plain_sum(rots, diags)


def linear_transform_plain_bsgs_hoisted(ev, ct, bd, keys, plans):
    """baby-step / giant-step evaluation with the b baby rotations hoisted (they share ct_new); the G giant rotations act on
    different ciphertexts and stay ordinary rotations.  `keys`: steps -d, 1..b-1 and g*b for g = 1..G-1."""
    d, b, G = bd.d, bd.b, bd.G
    dup = duplicate_fill(ev, ct, d, keys)
    baby = ev.rotate_plan_hoisted(dup, plans.get(range(b)))
    inner = []
    for g in range(G):
        lo, hi = g * b, min(d, (g + 1) * b)
        pts = Ciphertext(bd.plain.ctx, bd.plain.data[lo:hi], bd.plain.limbs, bd.plain.scale)
        inner.append(ev.multiply_plain_sum(baby[0:hi - lo], pts))
    giant = ev.rotate_plan(_stack(inner), plans.get([g * b for g in range(G)]))
    return ev.add_many(giant)


def linear_transform_ciphermatrix_plainvector(ev, pt_rotations, ct_diags):
    """Linear_Transform_CipherMatrix_PlainVector (helper.h:265-278)"""
    return ev.multiply_plain_sum(ct_diags, pt_rotations)


def c_matrix_encode(ev, rows, keys, plans):
    """C_Matrix_Encode (helper.h:307-322): pack d row ciphertexts into one, row i rotated by -i*d"""
    d = rows.batch
    rot = ev.rotate_plan(rows, plans.get([-(i * d) for i in range(d)]))
    return ev.add_many(rot)


def c_matrix_decode(ev, matrix, d, scale, keys, encoder, plans):
    """C_Matrix_Decode (helper.h:325-360): mask row i with ones, rotate it back by i*d"""
    masks = np.zeros((d, d * d))
    for i in range(d):
        masks[i, i * d:(i + 1) * d] = 1.0
    mask_pt = encoder.encode(masks, scale, limbs=matrix.limbs)
    bcast = Ciphertext(matrix.ctx, matrix.data.expand(d, -1, -1, -1).contiguous(), matrix.limbs, matrix.scale)
    rows = ev.multiply_plain(bcast, mask_pt)
    return ev.rotate_plan(rows, plans.get([i * d for i in range(d)]))


# ------------------------------------------------------------------ permutation matrices (host)
def u_sigma(d):
    """get_U_sigma (helper.h:700-742), closed form (SURVEY.md 3.2)"""
    U = np.zeros((d * d, d * d))
    for i in range(d):
        for j in range(d):
            U[d * i + j, d * i + (i + j) % d] = 1.0
    return U


def u_tau(d):
    """get_U_tau (helper.h:745-785)"""
    U = np.zeros((d * d, d * d))
    for i in range(d):
        for j in range(d):
            U[d * i + j, d * ((i + j) % d) + j] = 1.0
    return U


def v_k(d, k):
    """get_V_k (helper.h:788-818)"""
    U = np.zeros((d * d, d * d))
    for i in range(d):
        for j in range(d):
            U[d * i + j, d * i + (j + k) % d] = 1.0
    return U


def w_k(d, k):
    """get_W_k (helper.h:821-851)"""
    U = np.zeros((d * d, d * d))
    for i in range(d):
        for j in range(d):
            U[d * i + j, d * ((i + k) % d) + j] = 1.0
    return U


def u_transpose(d):
    """get_U_transpose (helper.h:386-413)"""
    U = np.zeros((d * d, d * d))
    for i in range(d):
        for o in range(d):
            U[d * i + o, d * o + i] = 1.0
    return U


def all_diagonals(U):
    """get_all_diagonals (helper.h:197-209): diag_l[k] = U[k][(k+l) mod n]"""
    n = U.shape[0]
    k = np.arange(n)
    return np.stack([U[k, (k + l) % n] for l in range(n)])


# ------------------------------------------------------------------ matrix multiplication
def cc_matrix_multiplication(ev, ctA, ctB, d, sigma_diags, tau_diags, V_diags, W_diags, keys, plans):
    """CC_Matrix_Multiplication (matrix_multiplication.cpp:11-132; matrix_mult_benchmark.cpp:13-71).
    V_diags / W_diags: lists of d-1 Plaintext batches (d*d diagonals each).
    The rotations of ctA[0] (resp. ctB[0]) are shared by all V_k (W_k) transforms."""
    dd = d * d
    A0 = linear_transform_plain(ev, ctA, sigma_diags, keys, plans)          # Step 1-1
    B0 = linear_transform_plain(ev, ctB, tau_diags, keys, plans)            # Step 1-2
    rotA = rotations_of(ev, duplicate_fill(ev, A0, dd, keys), dd, plans)    # Step 2 (shared)
    rotB = rotations_of(ev, duplicate_fill(ev, B0, dd, keys), dd, plans)
    A = [ev.multiply_plain_sum(rotA, V_diags[k]) for k in range(d - 1)]
    B = [ev.multiply_plain_sum(rotB, W_diags[k]) for k in range(d - 1)]
    # Step 3: rescale the step-2 outputs, multiply, accumulate
    Ak = _stack(A)
    Bk = _stack(B)
    ev.rescale_to_next_inplace(Ak)
    ev.rescale_to_next_inplace(Bk)
    ctAB = ev.multiply(A0, B0)
    ev.mod_switch_to_next_inplace(ctAB)
    force_scale_pow2(Ak)
    force_scale_pow2(Bk)
    rest = ev.multiply_sum(Ak, Bk)
    if rest.scale != ctAB.scale:
        raise capi.CkksInvalidArgument("scale mismatch")
    return ev.add(ctAB, rest)


def _stack(cts):
    """list of batch-1 ciphertexts -> one batch"""
    data = torch.cat([c.data for c in cts], dim=0)
    return Ciphertext(cts[0].ctx, data, cts[0].limbs, cts[0].scale)


# ------------------------------------------------------------------ dot product
def cipher_dot_product(ev, ctA, ctB, size, keys, method="reference"):
    """cipher_dot_product (helper.h:416-502), batched over independent (ctA[b], ctB[b]) pairs:
    multiply, relinearize, rescale, rotate-and-sum over `size` slots, force the scale.

    method="reference" runs the reference's own sequence (size-1 dependent unit rotations; every
    ciphertext polynomial bit-identical to SEAL's).  method="doubling" is the SURVEY 8(f4) upgrade:
    the same cyclic sums from log2(size) rotations by 1, 2, 4, ... -- equal decrypted values within
    noise, different polynomials, so it is a separate tolerance-checked mode and never the default."""
    mult = ev.multiply(ctA, ctB)
    mult = ev.relinearize(mult, keys)
    ev.rescale_to_next_inplace(mult)
    dup = ev.add(mult, ev.rotate_vector(mult, -size, keys))      # "vector has duplicate now"
    if method == "doubling":
        if size & (size - 1):
            raise ValueError("the doubling rotate-and-sum needs a power-of-two size")
        step = 1
        while step < size:
            dup = ev.add(dup, ev.rotate_vector(dup, step, keys))
            step *= 2
        return force_scale_pow2(dup)
    if method != "reference":
        raise ValueError("unknown rotate-and-sum method")
    # for i in 1..size-1: rotate_vector_inplace(dup, 1); add_inplace(mult, dup)   (helper.h:472-476)
    ev.rotate_sum_chain(dup, mult, 1, size - 1, keys)
    return force_scale_pow2(mult)


# ------------------------------------------------------------------ polynomial evaluation
def compute_all_powers(ev, ctx_ct, degree, keys):
    """compute_all_powers (helper.h:505-547; polynomial.cpp:56-96): x^2..x^degree by the split
    that minimises multiplicative depth; returns list indexed by power (index 0 unused)"""
    powers = [None] * (degree + 1)
    powers[1] = ctx_ct
    levels = [0] * (degree + 1)
    for i in range(2, degree + 1):
        minlevel, cand = i, -1
        for j in range(1, i // 2 + 1):
            k = i - j
            newlevel = max(levels[j], levels[k]) + 1
            if newlevel < minlevel:
                cand, minlevel = j, newlevel
        levels[i] = minlevel
        if cand < 0:
            raise RuntimeError("error")
        temp = ev.mod_switch_to(powers[cand], powers[i - cand].limbs)
        prod = ev.multiply(temp, powers[i - cand])
        prod = ev.relinearize(prod, keys)
        powers[i] = ev.rescale_to_next_inplace(prod)
    return powers


def horner_cipher(ev, x, coeffs, scale, keys, encoder, encryptor):
    """Horner_cipher (logistic_regression_ckks.cpp:139-205; polynomial.cpp:99-230)"""
    degree = len(coeffs) - 1
    temp = encryptor.encrypt(encoder.encode(float(coeffs[degree]), scale))
    if x.batch > 1:
        temp = Ciphertext(temp.ctx, temp.data.expand(x.batch, -1, -1, -1).contiguous(), temp.limbs, temp.scale)
    x = ev.mod_switch_to(x, x.limbs)
    for i in range(degree - 1, -1, -1):
        if x.limbs > temp.limbs:
            ev.mod_switch_to_inplace(x, temp.limbs)
        elif x.limbs < temp.limbs:
            ev.mod_switch_to_inplace(temp, x.limbs)
        temp = ev.multiply(temp, x)
        temp = ev.relinearize(temp, keys)
        ev.rescale_to_next_inplace(temp)
        temp.scale = float(2.0 ** 40)                                  # "Manual rescale" (:195)
        ev.add_plain_inplace(temp, encoder.encode(float(coeffs[i]), scale, limbs=temp.limbs))
    return temp


def tree_cipher(ev, x, coeffs, scale, keys, encoder, encryptor):
    """Tree_cipher (logistic_regression_ckks.cpp:55-137; polynomial.cpp:233-359)"""
    degree = len(coeffs) - 1
    powers = compute_all_powers(ev, x, degree, keys)
    enc_result = encryptor.encrypt(encoder.encode(float(coeffs[0]), scale))
    if x.batch > 1:
        enc_result = Ciphertext(enc_result.ctx, enc_result.data.expand(x.batch, -1, -1, -1).contiguous(),
                                enc_result.limbs, enc_result.scale)
    for i in range(1, degree + 1):
        pt = encoder.encode(float(coeffs[i]), scale, limbs=powers[i].limbs)
        temp = ev.multiply_plain(powers[i], pt)
        ev.rescale_to_next_inplace(temp)
        ev.mod_switch_to_inplace(enc_result, temp.limbs)
        force_scale_pow2(enc_result)
        temp.scale = float(2.0 ** int(math.log2(enc_result.scale)))
        ev.add_inplace(enc_result, temp)
    return enc_result


# ------------------------------------------------------------------ polynomials in the Chebyshev basis
def chebyshev_interpolant(f, B, degree):
    """coefficients c_0..c_degree of the Chebyshev interpolant of f on [-B, B]: f(x) ~ sum c_i T_i(x / B)
    (interpolation at the degree + 1 Chebyshev points of the first kind)"""
    k = np.arange(degree + 1)
    t = np.cos(np.pi * (k + 0.5) / (degree + 1))
    v = np.asarray(f(B * t), dtype=np.float64)
    c = 2.0 / (degree + 1) * np.cos(np.outer(k, np.pi * (k + 0.5) / (degree + 1))) @ v
    c[0] /= 2.0
    return c


def _bsgs_shape(degree):
    """(m, l): the polynomial is padded to 2^m coefficients, the baby steps are T_1..T_{2^l - 1}, the giant steps
    T_{2^l}, ..., T_{2^(m-1)}"""
    if degree < 1:
        raise ValueError("chebyshev: degree must be at least 1")
    m = max(1, int(degree).bit_length())   # 2^m > degree
    return m, (m + 1) // 2


def _basis_doublings(m, l):
    """the power basis T_1..T_{2^K} is built by K doublings: up to the first giant step T_{2^l} when there are giant
    steps, else up to the last baby step T_{2^l - 1}"""
    top = (1 << l) if m > l else (1 << l) - 1
    return max(0, (top - 1).bit_length())


def chebyshev_depth(degree):
    """levels chebyshev_cipher consumes for a polynomial of this degree: the doublings of the power basis, one for the
    baby-step sums and one per giant step (m + 1 = ceil(log2(degree + 1)) + 1 when there are giant steps)"""
    m, l = _bsgs_shape(degree)
    return _basis_doublings(m, l) + 1 + (m - l)


def chebyshev_keyswitches(degree):
    """relinearisations of one chebyshev_cipher per input ciphertext: 2^k products in doubling k of the power basis, one
    square per further giant step, 2^(m-1-k) products at the giant step T_{2^k}"""
    m, l = _bsgs_shape(degree)
    K = _basis_doublings(m, l)
    return (1 << K) - 1 + max(0, m - 1 - K) + ((1 << (m - l)) - 1)


def chebyshev_split(coeffs, degree_pow2, l):
    """the baby-step polynomials ("leaves") of sum c_i T_i padded to 2^m coefficients: p = q T_{2^(m-1)} + r, recursively
    down to 2^l coefficients; leaf g collects the divisions by T_{2^k} whose quotient it is part of in bit k - l of g.
    Division by T_n (c of length 2n): q_0 = c_n, q_j = 2 c_{n+j}, r_i = c_i - c_{2n-i} (r_0 = c_0)."""
    c = np.zeros(degree_pow2)
    c[:len(coeffs)] = coeffs

    def rec(c):
        if len(c) <= (1 << l):
            return [c]
        n = len(c) // 2
        q = np.empty(n)
        q[0] = c[n]
        q[1:] = 2.0 * c[n + 1:]
        r = c[:n].copy()
        r[1:] -= c[2 * n - 1:n:-1]
        return rec(r) + rec(q)
    return rec(c)


def _repeat(ct, times):
    """`times` copies of a batch (a batch of 1 is broadcast by multiply as it is)"""
    if times == 1 or ct.batch == 1:
        return ct
    return Ciphertext(ct.ctx, ct.data[:, :, :ct.limbs].repeat(times, 1, 1, 1), ct.limbs, ct.scale)


def chebyshev_cipher(ev, t, coeffs, keys, scale=None):
    """sum_i coeffs[i] T_i(t) for a batch of M ciphertexts holding t in [-1, 1], by baby steps and giant steps
    (T_{a+b} = 2 T_a T_b - T_{|a-b|}); consumes chebyshev_depth(degree) levels and needs only the relinearisation key.

    1. Power basis, one depth level at a time: [T_1..T_{2^k}] (uniform scale s_k) times T_{2^k} is one batched multiply +
       relinearize; one grouped multiply_const_sum forms T_{2^k + j} = 2 T_j T_{2^k} - T_{2^k - j} (and - 1 for j = 2^k)
       and carries T_1..T_{2^k} over (times 1 encoded at s_k), all at scale s_k^2; one batched rescale.  Giant steps
       beyond the basis: T_{2n} = 2 T_n^2 - 1.
    2. Baby-step sums: the 2^(m-l) leaves of chebyshev_split, sum_{i < 2^l} c_i T_i, in ONE multiply_const_sum over
       T_1..T_{2^l - 1} with every constant encoded at the leaf scale rho; rescale.
    3. Giant steps T_{2^k}, k = l..m-1: u_j = Y_{2j+1} T_{2^k} + Y_{2j}; the products are relinearized and one
       multiply_const_sum adds them to the Y_{2j} lifted by a constant 1 encoded at the giant step's scale, so both
       terms carry exactly the product's scale before the rescale.

    Scales are exact: every sum adds terms whose scales are the same float (constants are encoded at the scale that
    makes them so) and nothing is reassigned.  The leaf scale rho is the one free parameter; it is chosen by replaying
    the evaluator's scale arithmetic so that the result carries `scale` (default t.scale): exactly when some float rho
    gets there, else the nearest float reachable (a few 1e-16 relative).  This avoids the up to 1e-5 relative error per
    rescale of forcing power-of-two scales when the primes are only near 2^40."""
    ctx = t.ctx
    coeffs = np.asarray(coeffs, dtype=np.float64)
    degree = len(coeffs) - 1
    m, l = _bsgs_shape(degree)
    K, b, M = _basis_doublings(m, l), 1 << l, t.batch
    target = float(t.scale if scale is None else scale)
    if t.limbs <= chebyshev_depth(degree):
        raise capi.CkksInvalidArgument("chebyshev: %d levels needed, the input has %d limbs"
                                       % (chebyshev_depth(degree), t.limbs))
    # 1. power basis [T_1..T_{2^k}], entry (j-1)*M + m
    basis = ev.mod_switch_to(t, t.limbs)
    for k in range(K):
        h = 1 << k
        top = basis[(h - 1) * M:h * M]
        prods = ev.relinearize(ev.multiply(basis, _repeat(top, h)), keys)       # T_j T_h, scale s_k^2
        cf = np.zeros((2 * h, 2 * h))
        konst = np.zeros(2 * h)
        for j in range(1, h + 1):
            cf[j - 1, h + j - 1] = 1.0                                          # carry T_j
            cf[h + j - 1, j - 1] = 2.0                                          # T_{h+j} = 2 T_j T_h - T_{h-j}
            if j < h:
                cf[h + j - 1, h + (h - j) - 1] = -1.0
            else:
                konst[h + j - 1] = -1.0
        pts = [1.0] * h + [basis.scale] * h
        cs = ev.multiply_const_sum(_split_terms(prods, h) + _split_terms(basis, h), cf, pts, constant=konst, groups=2 * h)
        basis = ev.rescale_to_next_inplace(cs)
    giants = {}
    if m > l:
        giants[l] = basis[(b - 1) * M:b * M]
        for k in range(l, m - 1):
            g = giants[k]
            sq = ev.relinearize(ev.multiply(g, g), keys)
            giants[k + 1] = ev.rescale_to_next_inplace(ev.multiply_const_sum(sq, [2.0], 1.0, constant=[-1.0]))
    # the leaf scale rho that makes the result's scale exactly `target`
    L = basis.limbs
    drops = [ctx.primes[L - 1 - i] for i in range(m - l + 1)]
    gscales = [giants[k].scale for k in range(l, m)]

    def result_scale(rho):
        sc = basis.scale * rho / float(drops[0])
        for q, gs in zip(drops[1:], gscales):
            sc = sc * gs / float(q)
        return sc
    guess = target / basis.scale
    for q in drops:
        guess *= float(q)
    for gs in gscales:
        guess /= gs
    rho = _solve_scale(result_scale, target, guess)
    # 2. every baby-step sum in one launch
    leaves = chebyshev_split(coeffs, 1 << m, l)
    G = len(leaves)
    cf = np.stack([leaf[1:b] for leaf in leaves])
    Y = ev.multiply_const_sum(basis[0:(b - 1) * M], cf, rho, constant=[leaf[0] for leaf in leaves], groups=G)
    ev.rescale_to_next_inplace(Y)
    # 3. giant steps: u_j = Y_{2j+1} T_{2^k} + Y_{2j}
    for k in range(l, m):
        n = Y.batch // (2 * M)
        odd = Ciphertext(ctx, torch.cat([Y.data[(2 * j + 1) * M:(2 * j + 2) * M, :, :Y.limbs] for j in range(n)], dim=0),
                         Y.limbs, Y.scale)
        g = ev.mod_switch_to(giants[k], Y.limbs)
        prods = ev.relinearize(ev.multiply(odd, _repeat(g, n)), keys)
        cf = np.zeros((n, 3 * n))
        for j in range(n):
            cf[j, j] = 1.0                                                      # Y_{2j+1} T_{2^k}
            cf[j, n + 2 * j] = 1.0                                              # Y_{2j}, times 1 encoded at T_{2^k}'s scale
        pts = [1.0] * n + [g.scale] * (2 * n)
        Y = ev.multiply_const_sum(_split_terms(prods, n) + _split_terms(Y, 2 * n), cf, pts, groups=n)
        ev.rescale_to_next_inplace(Y)
    return Y


def _split_terms(ct, T):
    """a batch of T*M ciphertexts -> T views of M entries"""
    M = ct.batch // T
    return [ct[i * M:(i + 1) * M] for i in range(T)]


def _solve_scale(fn, target, x):
    """x with fn(x) == target for a non-decreasing float function fn close to proportional, else the closest x found"""
    for _ in range(8):                                       # proportional corrections
        y = fn(x)
        if y == target:
            return x
        x = x * (target / y)
    best, gap = x, abs(fn(x) - target)
    up = fn(x) < target
    for _ in range(4096):                                    # then float steps towards the target
        x = math.nextafter(x, math.inf if up else 0.0)
        y = fn(x)
        if y == target:
            return x
        if abs(y - target) < gap:
            best, gap = x, abs(y - target)
        if (y > target) == up:
            break
    return best


# ------------------------------------------------------------------ diagonal sets with a shared default
class DiagonalSet:
    """The plaintext diagonals of one matrix in de-duplicated form: `default` is the plaintext shared
    by most diagonals (the drivers add epsilon = 1e-8 to every entry, so the diagonals of a
    permutation matrix that would be zero all encode the same all-epsilon vector,
    matrix_multiplication.cpp:239-246), `index`/`special` list the diagonals that differ.
    sum_l diag_l (.) rot_l  =  default (.) (sum_all rot - sum_special rot) + sum_special diag_l (.) rot_l
    holds exactly modulo every prime, so the result is bit-identical to the dense evaluation while
    the d^2 x (d^2 plaintexts) of CC_Matrix_Multiplication at d = 64 (344 GB dense) never exist."""

    def __init__(self, n, default, index, special):
        self.n, self.default, self.index, self.special = n, default, list(index), special

    @staticmethod
    def from_matrix(U, eps, scale, encoder, limbs=None):
        n = U.shape[0]
        # only the non-empty diagonals are materialised: entry (r, c) lies on diagonal (c - r) mod n at
        # position r  (diag_l[k] = U[k][(k+l) mod n], helper.h:175-209) -- O(nnz) instead of O(n^2)
        r, c = np.nonzero(U)
        l = (c - r) % n
        idx = np.unique(l)
        pos = np.searchsorted(idx, l)
        vals = np.zeros((len(idx), n))
        vals[pos, r] = U[r, c]
        default = encoder.encode(np.full(n, eps), scale, limbs=limbs)
        special = encoder.encode(vals + eps, scale, limbs=limbs)
        return DiagonalSet(n, default, [int(x) for x in idx], special)


def linear_transform_plain_sparse(ev, ct, dset, keys, plans, rots=None, s_all=None):
    """Linear_Transform_Plain (helper.h:237-262) for a DiagonalSet; bit-identical to the dense form"""
    d = dset.n
    if rots is None:
        rots = rotations_of(ev, duplicate_fill(ev, ct, d, keys), d, plans)
    if s_all is None:
        s_all = ev.add_many(rots)
    sel_idx = torch.tensor(dset.index, device=rots.data.device)
    sel = Ciphertext(rots.ctx, rots.data.index_select(0, sel_idx), rots.limbs, rots.scale)
    rest = ev.sub(s_all, ev.add_many(sel))
    out = ev.multiply_plain(rest, dset.default)
    return ev.add(out, ev.multiply_plain_sum(sel, dset.special))


def cc_matrix_multiplication_sparse(ev, ctA, ctB, d, sigma, tau, V, W, keys, plans):
    """CC_Matrix_Multiplication with DiagonalSets (sigma, tau, V[k], W[k]); same op sequence and
    bit-identical result as cc_matrix_multiplication, feasible at d = 64 (d^2 = 4096 = N/4)"""
    dd = d * d
    A0 = linear_transform_plain_sparse(ev, ctA, sigma, keys, plans)
    B0 = linear_transform_plain_sparse(ev, ctB, tau, keys, plans)
    rotA = rotations_of(ev, duplicate_fill(ev, A0, dd, keys), dd, plans)
    sA = ev.add_many(rotA)
    A = [linear_transform_plain_sparse(ev, None, V[k], keys, plans, rots=rotA, s_all=sA) for k in range(d - 1)]
    del rotA
    rotB = rotations_of(ev, duplicate_fill(ev, B0, dd, keys), dd, plans)
    sB = ev.add_many(rotB)
    B = [linear_transform_plain_sparse(ev, None, W[k], keys, plans, rots=rotB, s_all=sB) for k in range(d - 1)]
    del rotB
    Ak, Bk = _stack(A), _stack(B)
    ev.rescale_to_next_inplace(Ak)
    ev.rescale_to_next_inplace(Bk)
    ctAB = ev.multiply(A0, B0)
    ev.mod_switch_to_next_inplace(ctAB)
    force_scale_pow2(Ak)
    force_scale_pow2(Bk)
    rest = ev.multiply_sum(Ak, Bk)
    if rest.scale != ctAB.scale:
        raise capi.CkksInvalidArgument("scale mismatch")
    return ev.add(ctAB, rest)


# ------------------------------------------------------------------ tolerance mode: only the non-empty diagonals
def linear_transform_plain_nonzero(ev, ct, dset, keys, plans, dup=None):
    """SURVEY 8(f4) "skipping all-epsilon diagonals": Linear_Transform_Plain restricted to the diagonals of the matrix that
    are not identically zero.  The reference adds epsilon = 1e-8 to every diagonal entry only because SEAL refuses to
    multiply by an all-zero plaintext (matrix_multiplication.cpp:239-246); its all-epsilon diagonals contribute
    1e-8 * (sum of the rotated slots) -- an error term of the reference, not part of A @ B.  Dropping them removes d^2 minus
    a few hundred rotations per transform (U_sigma at d = 64: 127 of 4096 diagonals are non-empty, V_k / W_k: 2 / 1).  The
    result decrypts to the reference's within 1e-8 * d^2 * max|slot|; ciphertext polynomials differ -- a tolerance-checked
    mode, never the default."""
    d = dset.n
    if dup is None:
        dup = duplicate_fill(ev, ct, d, keys)
    rots = ev.rotate_plan(dup, plans.get(dset.index))
    return ev.multiply_plain_sum(rots, dset.special)


def cc_matrix_multiplication_nonzero(ev, ctA, ctB, d, sigma, tau, V, W, keys, plans):
    """CC_Matrix_Multiplication (matrix_mult_benchmark.cpp:13-71) evaluating only the non-empty diagonals of the 2 + 2(d-1)
    permutation matrices (DiagonalSets): at d = 64 about 1.5 thousand key switches instead of the reference's 2.33 million
    (72 820 with the shared rotations of cc_matrix_multiplication_sparse).  Same op sequence otherwise (rescale of the step-2
    outputs, forced scales, size-3 accumulation).  The rotations of ctA[0] / ctB[0] needed by the V_k / W_k are computed once
    as one plan over the union of their steps."""
    dd = d * d
    A0 = linear_transform_plain_nonzero(ev, ctA, sigma, keys, plans)
    B0 = linear_transform_plain_nonzero(ev, ctB, tau, keys, plans)

    def step2(X0, sets):
        steps = sorted({l for s in sets for l in s.index})
        pos = {l: i for i, l in enumerate(steps)}
        rots = ev.rotate_plan(duplicate_fill(ev, X0, dd, keys), plans.get(steps))
        outs = []
        for s in sets:
            idx = torch.tensor([pos[l] for l in s.index], device=rots.data.device)
            sel = Ciphertext(rots.ctx, rots.data.index_select(0, idx), rots.limbs, rots.scale)
            outs.append(ev.multiply_plain_sum(sel, s.special))
        return _stack(outs)

    Ak, Bk = step2(A0, V), step2(B0, W)
    ev.rescale_to_next_inplace(Ak)
    ev.rescale_to_next_inplace(Bk)
    ctAB = ev.multiply(A0, B0)
    ev.mod_switch_to_next_inplace(ctAB)
    force_scale_pow2(Ak)
    force_scale_pow2(Bk)
    rest = ev.multiply_sum(Ak, Bk)
    if rest.scale != ctAB.scale:
        raise capi.CkksInvalidArgument("scale mismatch")
    return ev.add(ctAB, rest)
