"""Encrypted logistic-regression training: the reference's gradient loop on the GPU evaluator.

Mirrors logistic_regression_ckks.cpp: predict_cipher_weights (:208-266), update_weights (:269-345),
train_cipher (:348-385) over cipher_dot_product (helper.h:416-502) and the Horner / tree sigmoid
polynomial (:139-205, :55-137).  The committed program cannot finish an iteration (SURVEY.md 3.4);
the repairs applied here are the minimal ones listed there and touch only client-side layout and
level bookkeeping, never the evaluator op sequence of an individual ciphertext:

  R1  row i is encoded cyclically at slots i..i+C-1 and the weights periodically (slot s holds
      w[s mod C]), so the rotate-and-sum of row i leaves its full dot product at slot i where the
      reference's one-hot mask e_i picks it up (:222-229 vs helper.h:472-476);
  R2  the modulus chain has enough primes ({60, 40 x 8, 60}, N = 32768 for the full sequence);
  R3  after the learning-rate multiply the gradient is rescaled and the weights are brought to
      its level and scale before `sub` (:336-342);
  R4  the refresh re-encodes the decoded weights at the top level (:362-381);
  R5  standardised features are the ones encrypted (:570 vs :582-590);
  R6  the 1/8 input scaling of the sigmoid approximation is folded into the coefficients.

method="chebyshev" (opt-in, not the reference's) replaces the degree-3 polynomial, which is fitted on [-8, 8] while the
pulsar data reach |x.w| = 38, by the Chebyshev interpolant of the sigmoid on [-B, B] (ChebyshevSigmoid, default degree 63,
B = 48) evaluated by workloads.chebyshev_cipher with exact scales.  The 1/B input scaling is folded into the one-hot
prediction masks (e_i / B), so it costs no level; the polynomial takes chebyshev_depth(63) = 7 levels, so config 1 needs
{60, 40 x 12, 60}.  The column layout accepts it too: there the 1/B is folded into the weight broadcasts (the key
holder encrypts w_j / B), and an iteration takes 1 + 7 + 1 + 1 + 1 = 11 levels ({60, 40 x 11, 60}).

Two layouts:
  * `RowLayout`     -- the reference's: one ciphertext per sample row for the prediction and one per
                       feature column for the gradient (config 1, R + C <= N/2 slots).
  * `ColumnLayout`  -- mini-batches of B samples held as C column ciphertexts (config 5, where one
                       ciphertext per row cannot express R = 32768 samples): the prediction is
                       sum_j col_j * w_j with the weights supplied as C broadcast ciphertexts; the
                       gradient is the reference's per-feature cipher_dot_product over B slots.
                       Mini-batches are the sharding unit across GPUs.
"""
import math

import numpy as np
import torch

from .engine import Ciphertext
from .workloads import (chebyshev_cipher, chebyshev_depth, chebyshev_interpolant, cipher_dot_product, force_scale_pow2,
                        horner_cipher, tree_cipher)

# logistic_regression_ckks.cpp:247,251,255 (zero coefficients are written 0.00001 there because
# Tree_cipher dereferences every coefficient plaintext)
SIGMOID_COEFFS = {
    3: [0.5, 1.20069, 0.00001, -0.81562],
    5: [0.5, 1.53048, 0.00001, -2.3533056, 0.00001, 1.3511295],
    7: [0.5, 1.73496, 0.00001, -4.19407, 0.00001, 5.43402, 0.00001, -2.50739],
}


def folded_coeffs(degree):
    """R6: sigmoid(x) ~ sum a_i (x/8)^i  ->  coefficients a_i / 8^i applied to x directly"""
    return [a / 8.0 ** i for i, a in enumerate(SIGMOID_COEFFS[degree])]


def sigmoid_approx(x, degree):
    """sigmoid_approx (logistic_regression_ckks.cpp:388-412), with the x^7 term repaired"""
    return sum(c * x ** i for i, c in enumerate(folded_coeffs(degree)))


class ChebyshevSigmoid:
    """the sigmoid as sum c_i T_i(x / bound): its Chebyshev interpolant of `degree` on [-bound, bound].  Degree 63 on
    [-48, 48] is within 1e-2 of the sigmoid there (largest at the steep centre) and its coefficients are bounded
    (sum |c_i| < 2): monomial coefficients of the same fit would be ~48^-63 and vanish at scale 2^40."""

    def __init__(self, degree=63, bound=48.0):
        self.degree, self.bound = int(degree), float(bound)
        self.coeffs = chebyshev_interpolant(lambda x: 1.0 / (1.0 + np.exp(-x)), self.bound, self.degree)

    def __call__(self, x):
        return np.polynomial.chebyshev.chebval(np.asarray(x) / self.bound, self.coeffs)


SIGMOID_CHEBYSHEV = ChebyshevSigmoid()


def plain_epoch(X, y, w, lr, degree=3, method="horner", sigmoid=None):
    """plaintext semantics of one update_weights (logistic_regression.cpp:136-178 with the
    polynomial sigmoid): w - lr/R * X^T (sigma(Xw) - y).  method="chebyshev": sigma is `sigmoid`
    (a ChebyshevSigmoid, default SIGMOID_CHEBYSHEV) and `degree` is not used."""
    R = X.shape[0]
    if method == "chebyshev":
        p = (sigmoid or SIGMOID_CHEBYSHEV)(X @ w)
    else:
        p = sigmoid_approx(X @ w, degree)
    return w - (lr / R) * (X.T @ (p - y))


def _bcast(ct, batch):
    if ct.batch == batch:
        return ct
    return Ciphertext(ct.ctx, ct.data.expand(batch, -1, -1, -1).contiguous(), ct.limbs, ct.scale)


def _poly(method):
    return tree_cipher if method == "tree" else horner_cipher


def prediction_masks(masks, method, sigmoid):
    """the one-hot prediction masks, divided by the sigmoid's bound for method="chebyshev" (the polynomial's input is
    x.w / B; folding 1/B into the mask costs no level)"""
    return masks / (sigmoid or SIGMOID_CHEBYSHEV).bound if method == "chebyshev" else masks


def sigmoid_cipher(ev, lin, scale, keys, encoder, encryptor, degree, method, sigmoid):
    """the sigmoid polynomial of the prediction: the reference's (forced power-of-two scale on its input, then
    Horner_cipher / Tree_cipher) or, for method="chebyshev", chebyshev_cipher with exact scales, landing on `scale`"""
    if method == "chebyshev":
        return chebyshev_cipher(ev, lin, (sigmoid or SIGMOID_CHEBYSHEV).coeffs, keys, scale=scale)
    force_scale_pow2(lin)
    return _poly(method)(ev, lin, folded_coeffs(degree), scale, keys, encoder, encryptor)


class RowLayout:
    """the reference's data layout (repairs R1, R5): client-side packing helpers"""

    def __init__(self, R, C, slots):
        if R + C > slots or 2 * R > slots:
            raise ValueError("R + C and 2R must fit in N/2 slots")
        self.R, self.C, self.slots = R, C, slots

    def rows(self, X):
        out = np.zeros((self.R, self.slots))
        for i in range(self.R):
            s = np.arange(i, i + self.C)
            out[i, s] = X[i, s % self.C]
        return out

    def columns(self, X):
        out = np.zeros((self.C, self.slots))
        out[:, : self.R] = X.T
        return out

    def weights(self, w):
        out = np.zeros(self.slots)
        s = np.arange(self.R + self.C)
        out[s] = w[s % self.C]
        return out

    def labels(self, y):
        out = np.zeros(self.slots)
        out[: self.R] = y
        return out


def predict_cipher_weights(ev, features, weights, C, scale, keys, encoder, encryptor, degree=3, method="horner",
                           sigmoid=None):
    """predict_cipher_weights (logistic_regression_ckks.cpp:208-266): per-row dot product with the
    weights, one-hot mask at slot i, add_many, rescale, sigmoid polynomial.  `features`: batch of R
    row ciphertexts; `weights`: one ciphertext.  method="chebyshev": masks e_i / B and the
    ChebyshevSigmoid `sigmoid` (no encryptor needed)."""
    R = features.batch
    results = cipher_dot_product(ev, features, weights, C, keys)          # hot loop 1, batched over rows
    masks = np.zeros((R, R))
    masks[np.arange(R), np.arange(R)] = 1.0
    mask_pt = encoder.encode(prediction_masks(masks, method, sigmoid), scale)
    ev.mod_switch_to_next_inplace(mask_pt)                                # :227
    ev.multiply_plain_inplace(results, mask_pt)
    lin = ev.add_many(results)
    lin = ev.relinearize(lin, keys)                                       # no-op on size 2 (:236)
    ev.rescale_to_next_inplace(lin)
    return sigmoid_cipher(ev, lin, scale, keys, encoder, encryptor, degree, method, sigmoid)


def update_weights(ev, features, features_T, labels, weights, lr, scale, keys, encoder, encryptor,
                   degree=3, method="horner", sigmoid=None):
    """update_weights (logistic_regression_ckks.cpp:269-345) with repairs R3"""
    R, C = features.batch, features_T.batch
    pred = predict_cipher_weights(ev, features, weights, C, scale, keys, encoder, encryptor, degree, method, sigmoid)
    lab = ev.mod_switch_to(labels, pred.limbs)                            # :286
    if lab.scale != pred.scale:
        pred.scale = lab.scale                                            # both are 2^40 after the forced scales
    pred_labels = ev.sub(pred, lab)
    cols = ev.mod_switch_to(features_T, pred_labels.limbs)                # :295
    grads = cipher_dot_product(ev, cols, pred_labels, R, keys)            # hot loop 2, batched over features
    masks = np.zeros((C, C))
    masks[np.arange(C), np.arange(C)] = 1.0
    mask_pt = encoder.encode(masks, scale, limbs=grads.limbs)             # :305-308
    ev.multiply_plain_inplace(grads, mask_pt)
    gradient = ev.add_many(grads)
    gradient = ev.relinearize(gradient, keys)
    ev.rescale_to_next_inplace(gradient)
    force_scale_pow2(gradient)
    n_pt = encoder.encode(float(lr / R), scale, limbs=gradient.limbs)     # :330-333
    ev.multiply_plain_inplace(gradient, n_pt)
    ev.rescale_to_next_inplace(gradient)                                  # R3
    force_scale_pow2(gradient)
    w_low = ev.mod_switch_to(weights, gradient.limbs)                     # R3
    w_low.scale = gradient.scale
    new_weights = ev.sub(gradient, w_low)                                 # :341
    return ev.negate_inplace(new_weights)                                 # :342


def train_cipher(ev, features, features_T, labels, weights, lr, iters, layout, scale, keys, encoder, encryptor, decryptor,
                 degree=3, method="horner", sigmoid=None):
    """train_cipher (logistic_regression_ckks.cpp:348-385): `iters` x (update_weights, then the key holder
    decrypts, decodes and re-encrypts the weights).  Repair R4: the decoded weights are re-packed
    (RowLayout.weights) and encoded at the top level -- the reference re-encrypts the exhausted low-level
    plaintext, which leaves the next iteration without levels (:376-381)."""
    new_weights = weights
    for _ in range(iters):
        new_weights = update_weights(ev, features, features_T, labels, new_weights, lr, scale, keys, encoder, encryptor,
                                     degree=degree, method=method, sigmoid=sigmoid)
        decoded = encoder.decode(decryptor.decrypt(new_weights))[0, : layout.C]
        new_weights = encryptor.encrypt(encoder.encode(layout.weights(decoded), scale))
    return new_weights


class ColumnLayout:
    """config 5 packing: mini-batch m holds samples [m*B, (m+1)*B) as C column ciphertexts"""

    def __init__(self, R, C, B, slots):
        if R % B or 2 * B > slots:
            raise ValueError("B must divide R and 2B must fit in N/2 slots")
        self.R, self.C, self.B, self.slots, self.M = R, C, B, slots, R // B

    def columns(self, X):
        """-> [M*C][slots]: entry m*C + j = feature j of mini-batch m"""
        out = np.zeros((self.M * self.C, self.slots))
        for m in range(self.M):
            out[m * self.C:(m + 1) * self.C, : self.B] = X[m * self.B:(m + 1) * self.B].T
        return out

    def labels(self, y):
        out = np.zeros((self.M, self.slots))
        out[:, : self.B] = y.reshape(self.M, self.B)
        return out

    def weights(self, w):
        """the packed weights apply_gradient updates: slot j holds w_j for j < C"""
        out = np.zeros(self.slots)
        out[: self.C] = w
        return out

    def weight_broadcasts(self, w, method="tree", sigmoid=None):
        """-> [C][slots]: row j holds w_j in every slot, divided by the sigmoid's bound for method="chebyshev" (the
        polynomial's input is x.w / bound; folding 1/bound into the broadcasts costs no level)"""
        w = np.asarray(w, dtype=np.float64)
        if method == "chebyshev":
            w = w / (sigmoid or SIGMOID_CHEBYSHEV).bound
        return np.repeat(w[:, None], self.slots, axis=1)


def column_rescales(method="tree", degree=7, sigmoid=None):
    """levels one column-layout iteration (column_epoch_gradient + apply_gradient) consumes: the prediction, the
    sigmoid polynomial, the dot product, the mask and the learning rate, one rescale each except the polynomial's
    ceil(log2 degree) + 1 (Tree_cipher), degree (Horner_cipher) or chebyshev_depth (chebyshev_cipher)"""
    if method == "chebyshev":
        poly = chebyshev_depth((sigmoid or SIGMOID_CHEBYSHEV).degree)
    elif method == "tree":
        poly = (degree - 1).bit_length() + 1
    else:
        poly = degree
    return 1 + poly + 1 + 1 + 1


def column_epoch_gradient(ev, cols, labels, w_bcast, C, B, scale, keys, encoder, encryptor, degree=7,
                          method="tree", dot_method="reference", units=None, combine=None, sigmoid=None, mark=None):
    """One pass of the gradient loop over the mini-batches held by this GPU (column layout).

    cols    : batch M*C of column ciphertexts (entry m*C + j)
    labels  : batch M of label ciphertexts
    w_bcast : batch C of ciphertexts, entry j = Enc(w_j in every slot)
    returns : one gradient ciphertext, slot j = sum_m sum_i x_ij (sigma(x_i.w) - y_i), plus its level

    Per mini-batch the evaluator sequence is: z = sum_j multiply(col_j, w_j); relinearize; rescale;
    sigmoid polynomial (Tree_cipher / Horner_cipher; for method="chebyshev" chebyshev_cipher on z as it is, with
    w_bcast holding w_j / bound, see ColumnLayout.weight_broadcasts); sub labels; then, per feature j, the reference's
    cipher_dot_product(col_j, pred - y, B) and the one-hot mask e_j (update_weights :295-311);
    add_many; rescale.  The M sums z are one grouped multiply_sum against the shared broadcasts.

    `units` (optional) restricts the gradient dot products to a list of (mini-batch, feature) pairs -- the
    sharding unit when ONE problem is split over several GPUs (SURVEY 8(e): "shard features j and
    mini-batches"); the prediction is still evaluated for every mini-batch held here, the result is the
    partial gradient sum over `units`.  `combine` (optional) is applied to the partial sum BEFORE the final rescale --
    pass parallel.combine_partials there (all-gather + mod-q add): summing first and rescaling once keeps the
    sharded result bit-identical to the unsharded one (rescale rounds, so it does not commute with the sum).
    `mark(name)` (optional) is called as each phase ends: prediction, polynomial, gradient, combine."""
    mark = mark or (lambda name: None)
    M = labels.batch
    z = ev.multiply_sum_grouped(cols, w_bcast, M)                         # M size-3 sums of C products
    z = ev.relinearize(z, keys)
    ev.rescale_to_next_inplace(z)
    mark("prediction")
    pred = sigmoid_cipher(ev, z, scale, keys, encoder, encryptor, degree, method, sigmoid)
    lab = ev.mod_switch_to(labels, pred.limbs)
    pred.scale = lab.scale
    pred_labels = ev.sub(pred, lab)                                       # batch M
    mark("polynomial")
    colv = ev.mod_switch_to(cols, pred_labels.limbs)
    masks = np.zeros((C, C))
    masks[np.arange(C), np.arange(C)] = 1.0
    if units is None:
        pl = Ciphertext(cols.ctx, pred_labels.data.repeat_interleave(C, dim=0), pred_labels.limbs, pred_labels.scale)
        grads = cipher_dot_product(ev, colv, pl, B, keys, method=dot_method)  # M*C chains in lock-step
        mask_pt = encoder.encode(masks, scale, limbs=grads.limbs)
        mp = Ciphertext(cols.ctx, mask_pt.data.repeat(M, 1, 1, 1), mask_pt.limbs, mask_pt.scale)
    else:
        dev = cols.data.device
        ci = torch.tensor([m * C + j for m, j in units], device=dev)
        mi = torch.tensor([m for m, _ in units], device=dev)
        ji = torch.tensor([j for _, j in units], device=dev)
        csel = Ciphertext(cols.ctx, colv.data.index_select(0, ci), colv.limbs, colv.scale)
        pl = Ciphertext(cols.ctx, pred_labels.data.index_select(0, mi), pred_labels.limbs, pred_labels.scale)
        grads = cipher_dot_product(ev, csel, pl, B, keys, method=dot_method)  # len(units) chains in lock-step
        mask_pt = encoder.encode(masks, scale, limbs=grads.limbs)
        mp = Ciphertext(cols.ctx, mask_pt.data.index_select(0, ji), mask_pt.limbs, mask_pt.scale)
    ev.multiply_plain_inplace(grads, mp)
    gradient = ev.add_many(grads)                                         # over features and mini-batches
    mark("gradient")
    if combine is not None:
        gradient = combine(gradient)                                      # ... and over GPUs
    mark("combine")
    ev.rescale_to_next_inplace(gradient)
    return force_scale_pow2(gradient)


def apply_gradient(ev, gradient, weights, lr, R, scale, encoder):
    """the tail of update_weights (:326-342, repair R3): weights - lr/R * gradient"""
    n_pt = encoder.encode(float(lr / R), scale, limbs=gradient.limbs)
    g = ev.multiply_plain(gradient, n_pt)
    ev.rescale_to_next_inplace(g)
    force_scale_pow2(g)
    w_low = ev.mod_switch_to(weights, g.limbs)
    w_low.scale = g.scale
    return ev.negate_inplace(ev.sub(g, w_low))


def refresh_columns(new_weights, layout, scale, encoder, encryptor, decryptor, method="tree", sigmoid=None):
    """the key holder's refresh of the column layout (repair R4): decrypt the updated weights, decode slots [0, C),
    re-encode the packed weights and the C broadcasts at the top level and re-encrypt them (in this order)"""
    decoded = encoder.decode(decryptor.decrypt(new_weights))[0, : layout.C]
    weights = encryptor.encrypt(encoder.encode(layout.weights(decoded), scale))
    w_bcast = encryptor.encrypt(encoder.encode(layout.weight_broadcasts(decoded, method, sigmoid), scale))
    return weights, w_bcast


def train_columns(ev, cols, labels, weights, w_bcast, lr, iters, layout, scale, keys, encoder, encryptor, decryptor,
                  degree=7, method="tree", sigmoid=None):
    """full-batch gradient descent in the column layout: `iters` x (column_epoch_gradient over every mini-batch,
    apply_gradient, refresh_columns), the loop of train_cipher (logistic_regression_ckks.cpp:348-385).
    `weights`: the packed weights (ColumnLayout.weights), `w_bcast`: the C broadcasts (ColumnLayout.weight_broadcasts
    with the same method and sigmoid).  Returns the refreshed (weights, w_bcast), both at the top level."""
    for _ in range(iters):
        grad = column_epoch_gradient(ev, cols, labels, w_bcast, layout.C, layout.B, scale, keys, encoder, encryptor,
                                     degree=degree, method=method, sigmoid=sigmoid)
        new_weights = apply_gradient(ev, grad, weights, lr, layout.R, scale, encoder)
        weights, w_bcast = refresh_columns(new_weights, layout, scale, encoder, encryptor, decryptor, method, sigmoid)
    return weights, w_bcast
