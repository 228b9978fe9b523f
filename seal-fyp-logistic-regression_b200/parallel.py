"""Multi-GPU sharding of the hot path (SURVEY.md 8(e)): independent ciphertexts are partitioned
across ranks (one process per GPU, torch.distributed), every rank computes its partial result
with no collective in the data path, and the partial ciphertexts are combined with one
all-gather followed by the mod-q add kernel (NCCL's sum is not modular).  Modular addition is
associative and commutative, so the combined ciphertext is bit-identical to the sequential
add_many of the reference (helper.h:259, logistic_regression_ckks.cpp:316)."""
import math

import numpy as np
import torch
import torch.distributed as dist

from . import capi
from .engine import Ciphertext, ExtendedPartial
from .lr import (SIGMOID_CHEBYSHEV, apply_gradient, column_epoch_gradient, prediction_masks, refresh_columns,
                 sigmoid_cipher)
from .workloads import (MatmulEntries, _column_major_rows, _stack, bsgs_terms, chebyshev_depth, chebyshev_keyswitches,
                        cipher_dot_product, diagonal_terms, duplicate_fill, force_scale_pow2, matmul_diagonal_indices,
                        matmul_nonzero_hoisted_terms, matmul_operands, term_steps)


def world():
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def shard_units(n_units, rank, world_size):
    """interleaved partition: unit u belongs to rank u mod G.  For the diagonals of a linear
    transform this balances the NAF weight (key switches) of the rotations far better than
    contiguous blocks (SURVEY.md 8(e))."""
    return list(range(rank, n_units, world_size))


def naf_weight(steps):
    """number of key switches SEAL's rotate_vector spends on `steps` with the default power-of-two Galois
    keys: the number of non-zero digits of its non-adjacent form (util::naf; SURVEY.md A.6)"""
    v, w = abs(int(steps)), 0
    while v:
        if v & 1:
            z = 2 - (v & 3)
            v -= z
            w += 1
        v >>= 1
    return w


def shard_units_weighted(weights, rank, world_size):
    """partition units by COST instead of index: longest-processing-time greedy (heaviest unit first, always
    onto the least-loaded rank; ties broken by rank index so every rank computes the same assignment).
    For the diagonals of a linear transform the cost of diagonal l is naf_weight(l) key switches: `l mod G`
    gives rank 0 all even diagonals (157 key switches at d = 128, G = 2) and rank 1 all odd ones (199);
    this split is 178 / 178.  Returns this rank's unit indices in increasing order."""
    order = sorted(range(len(weights)), key=lambda u: (-weights[u], u))
    load = [0] * world_size
    mine = []
    for u in order:
        r = min(range(world_size), key=lambda k: (load[k], k))
        load[r] += weights[u]
        if r == rank:
            mine.append(u)
    return sorted(mine)


def naf_terms(steps):
    """the signed power-of-two terms SEAL's rotate_vector applies for `steps`, in its order (least significant
    first; util::naf, SURVEY.md A.6)"""
    v, i, out = abs(int(steps)), 0, []
    sign = 1 if steps >= 0 else -1
    while v:
        if v & 1:
            z = 2 - (v & 3)
            v -= z
            out.append(sign * z * (1 << i))
        v >>= 1
        i += 1
    return out


def shard_rotations_shared(steps, rank, world_size):
    """partition the rotations of ONE ciphertext for rotation plans that share common NAF prefixes
    (ckks_rotplan_keyswitches_shared): rotations are ordered by their term sequences, so that rotations with a common
    prefix are neighbours, and the order is cut into world_size contiguous runs of equal cost, where a rotation costs the
    terms it does not share with its predecessor in the run (= the key switches the run's prefix tree adds for it).
    d = 128: 169 key switches on 1 GPU, 85 / 85 on 2, 4 x 43 on 4, 8 x 22 on 8 (cost-balanced without regard to prefixes: 90 / 51 / 31).
    Returns this rank's indices into `steps`, increasing."""
    seqs = [tuple(naf_terms(st)) for st in steps]
    order = sorted(range(len(steps)), key=lambda u: (seqs[u], u))

    def lcp(a, b):
        n = 0
        while n < len(a) and n < len(b) and a[n] == b[n]:
            n += 1
        return n

    def cuts(limit):
        """greedy: fewest runs with cost <= limit each; returns the list of runs"""
        runs, cur, cost = [], [], 0
        for u in order:
            add = len(seqs[u]) - (lcp(seqs[cur[-1]], seqs[u]) if cur else 0)
            if cur and cost + add > limit:
                runs.append(cur)
                cur, cost = [], 0
                add = len(seqs[u])
            cur.append(u)
            cost += add
        if cur:
            runs.append(cur)
        return runs

    lo, hi = max([len(q) for q in seqs] + [1]), sum(len(q) for q in seqs) + 1
    while lo < hi:                       # smallest per-run cost that needs at most world_size runs
        mid = (lo + hi) // 2
        if len(cuts(mid)) <= world_size:
            hi = mid
        else:
            lo = mid + 1
    runs = cuts(lo)
    runs += [[] for _ in range(world_size - len(runs))]
    return sorted(runs[rank])


def gather_partials(t):
    """all-gather one tensor per rank -> [G, ...] on every rank (any backend)"""
    rank, G = world()
    if G == 1:
        return t.unsqueeze(0) if t.dim() == 3 else t
    flat = t.reshape((1,) + tuple(t.shape[-3:])) if t.dim() == 3 else t
    out = torch.empty((G * flat.shape[0],) + tuple(flat.shape[1:]), dtype=flat.dtype, device=flat.device)
    dist.all_gather_into_tensor(out, flat.contiguous())
    return out


def combine_partials(ev, partial):
    """partial: batch-1 Ciphertext held by every rank -> sum over ranks (mod q) on every rank"""
    rank, G = world()
    if G == 1:
        return partial
    gathered = gather_partials(partial.data)
    return ev.add_many(Ciphertext(partial.ctx, gathered, partial.limbs, partial.scale))


def sharded_linear_transform_plain(ev, ct_new_rots_fn, diags_local, d, plans_steps):
    """helper for a sharded Linear_Transform_Plain: this rank owns the diagonals `plans_steps`
    (a subset of range(d)); returns the combined ciphertext"""
    rots = ct_new_rots_fn(plans_steps)
    part = ev.multiply_plain_sum(rots, diags_local)
    return combine_partials(ev, part)


# ------------------------------------------------------------------ sharded CC_Matrix_Multiplication
class TorchExchange:
    """the collectives of the sharded workloads over the default torch.distributed group (NCCL on GPUs).  Tests substitute
    an emulation with the same methods; every tensor is [batch, ...] and splits count batch entries."""

    def __init__(self):
        self.rank, self.world = world()

    def all_gather(self, t):
        """[b, ...] on every rank -> [world * b, ...], rank-major"""
        if self.world == 1:
            return t
        out = torch.empty((self.world * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        dist.all_gather_into_tensor(out, t.contiguous())
        return out

    def all_to_all(self, t, send_counts, recv_counts):
        """block q of `t` (send_counts[q] entries) goes to rank q; the result holds recv_counts[g] entries from each rank g,
        rank-major"""
        if self.world == 1:
            return t
        out = torch.empty((sum(recv_counts),) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        dist.all_to_all_single(out, t.contiguous(), output_split_sizes=list(recv_counts), input_split_sizes=list(send_counts))
        return out

    def broadcast(self, t, src=0):
        """rank src's `t` on every rank; the other ranks pass a contiguous tensor of the same shape and dtype to receive into"""
        if self.world == 1:
            return t
        dist.broadcast(t, src)
        return t


def owned_block(n_units, rank, world_size):
    """contiguous partition of range(n_units): the first n_units mod G ranks own one unit more.  Contiguous blocks let the
    reduce-scatter send one slice of the stacked partials to each rank."""
    base, extra = divmod(n_units, world_size)
    start = rank * base + min(rank, extra)
    return range(start, start + base + (1 if rank < extra else 0))


def _zeros(ct, size, batch, scale):
    return Ciphertext(ct.ctx, torch.zeros((batch, size, ct.cap, ct.ctx.n), dtype=torch.int64, device=ct.data.device),
                      ct.limbs, scale)


def _combine(ev, part, exchange):
    """sum of one batch-1 partial ciphertext over the ranks (mod q), on every rank"""
    gathered = exchange.all_gather(part.data)
    return ev.add_many(Ciphertext(part.ctx, gathered, part.limbs, part.scale))


def _partial_sparse_transform(ev, rots, s_mine, pos, dset):
    """this rank's share of linear_transform_plain_sparse: `rots` are the rotations by this rank's steps (`pos`: step ->
    batch index), `s_mine` their sum.  default (.) (sum_mine rot - sum_{mine & index} rot) + sum_{mine & index} special (.) rot;
    modular products and sums distribute exactly, so the ranks' partials add up to the unsharded transform word for word."""
    hit = [i for i, l in enumerate(dset.index) if l in pos]
    if not hit:
        return ev.multiply_plain(s_mine, dset.default)
    dev = rots.data.device
    sel = Ciphertext(rots.ctx, rots.data.index_select(0, torch.tensor([pos[dset.index[i]] for i in hit], device=dev)),
                     rots.limbs, rots.scale)
    sp = dset.special
    special = Ciphertext(sp.ctx, sp.data.index_select(0, torch.tensor(hit, device=dev)), sp.limbs, sp.scale)
    rest = ev.sub(s_mine, ev.add_many(sel))
    return ev.add(ev.multiply_plain(rest, dset.default), ev.multiply_plain_sum(sel, special))


def _partial_transforms(ev, X, dsets, mine, keys, plans):
    """this rank's partials of the transforms `dsets` of X (all sharing the rotations of X + rot(X, -n)) -> one batch"""
    n = dsets[0].n
    scale = X.scale * dsets[0].default.scale
    if not mine:
        return _zeros(X, 2, len(dsets), scale)
    rots = ev.rotate_plan(duplicate_fill(ev, X, n, keys), plans.get(mine))
    s_mine = ev.add_many(rots)
    pos = {l: i for i, l in enumerate(mine)}
    return _stack([_partial_sparse_transform(ev, rots, s_mine, pos, ds) for ds in dsets])


def _rescaled_pow2_scale(ctx, scale, limbs):
    """the scale rescale_to_next + force_scale_pow2 give a ciphertext at `limbs` limbs with `scale`"""
    return float(2.0 ** int(math.log2(scale / float(ctx.primes[limbs - 1]))))


def sharded_cc_matrix_multiplication(ev, ctA, ctB, d, sigma, tau, V, W, keys, plans, rank, world_size, exchange):
    """cc_matrix_multiplication_sparse (CC_Matrix_Multiplication, matrix_mult_benchmark.cpp:13-71) with its d^2 rotations
    of each transformed ciphertext sharded over `world_size` ranks (SURVEY 8(e)); every rank returns the product,
    bit-identical to the one-GPU function.  `exchange`: TorchExchange, or a test emulation with its two methods.

    Step 1: each rank rotates dup(ctA) / dup(ctB) by its prefix-aware share of range(d^2) and computes its partial of the
    sigma / tau transform; all-gather + mod-q add gives A0 and B0 on every rank.
    Step 2: the same share of the rotations of dup(A0) / dup(B0) gives every rank a partial A_k / B_k for all d-1 k.  Rank r
    owns the contiguous block K_r of k: one all-to-all sends each block to its owner, ckks_add_many_grouped sums the
    world_size contributions of every owned k.  The sum is taken before the rescale, which rounds and does not commute
    with it.
    Step 3: each rank rescales its A_k / B_k, forces the scales and accumulates sum_{k in K_r} A_k x B_k; all-gather +
    mod-q add of these size-3 partials, then + mod_switch(A0 x B0)."""
    dd = d * d
    mine = shard_rotations_shared(list(range(dd)), rank, world_size)
    X0 = []
    for ct, ds in ((ctA, sigma), (ctB, tau)):
        X0.append(_combine(ev, _partial_transforms(ev, ct, [ds], mine, keys, plans), exchange))
    A0, B0 = X0

    counts = [len(owned_block(d - 1, q, world_size)) for q in range(world_size)]
    own = counts[rank]
    XK = []
    for X, dsets in ((A0, V), (B0, W)):
        part = _partial_transforms(ev, X, dsets, mine, keys, plans)
        recv = exchange.all_to_all(part.data, counts, [own] * world_size)
        XK.append(ev.add_many_grouped(Ciphertext(part.ctx, recv, part.limbs, part.scale), world_size) if own else part)
    Ak, Bk = XK

    ctAB = ev.multiply(A0, B0)
    ev.mod_switch_to_next_inplace(ctAB)
    if own:
        for X in (Ak, Bk):
            ev.rescale_to_next_inplace(X)
            force_scale_pow2(X)
        rest = ev.multiply_sum(Ak, Bk)
    else:                                   # more ranks than products: this rank adds zero
        scale = (_rescaled_pow2_scale(A0.ctx, Ak.scale, Ak.limbs) * _rescaled_pow2_scale(B0.ctx, Bk.scale, Bk.limbs))
        rest = _zeros(Ak, 3, 1, scale)
        rest.limbs = Ak.limbs - 1
    rest = _combine(ev, rest, exchange)
    if rest.scale != ctAB.scale:
        raise capi.CkksInvalidArgument("scale mismatch")
    return ev.add(ctAB, rest)


# ------------------------------------------------------------------ sharded config-1 training iteration
def config1_shards(R, C, rank, world_size):
    """this rank's contiguous block of the R sample rows (prediction) and of the C feature columns (gradient).  Every row
    and every feature belongs to exactly one rank; with more ranks than features (or rows) the last ranks own none."""
    return owned_block(R, rank, world_size), owned_block(C, rank, world_size)


def config1_keyswitches(R, C, rank, world_size, degree=3, method="horner", sigmoid=None):
    """key switches of this rank in one sharded_update_weights with the Horner polynomial (rank 0 evaluates it): per own
    row 1 relinearisation + rotate_vector(-C) + C - 1 chain steps, per own feature 1 + rotate_vector(-R) + R - 1; a
    rotation by a step without its own Galois key costs the NAF weight of the step (power-of-two keys).  With
    method="chebyshev" rank 0's polynomial costs chebyshev_keyswitches(sigmoid degree) relinearisations."""
    rows, feats = config1_shards(R, C, rank, world_size)
    poly = chebyshev_keyswitches((sigmoid or SIGMOID_CHEBYSHEV).degree) if method == "chebyshev" else degree
    return (len(rows) * (1 + naf_weight(C) + C - 1) + (poly if rank == 0 else 0)
            + len(feats) * (1 + naf_weight(R) + R - 1))


def _one_hot(ids, width):
    m = np.zeros((len(ids), width))
    m[np.arange(len(ids)), list(ids)] = 1.0
    return m


def _active(ct):
    """`ct` with its buffer cut to the active limbs: what an exchange has to move"""
    if ct.cap == ct.limbs:
        return ct
    return Ciphertext(ct.ctx, ct.data[:, :, : ct.limbs].contiguous(), ct.limbs, ct.scale)


def _zero_partial(ctx, limbs, scale):
    return Ciphertext(ctx, torch.zeros((1, 2, limbs, ctx.n), dtype=torch.int64, device=ctx.device), limbs, scale)


def _broadcast_ct(ctx, ct, rank, exchange):
    """rank 0's ciphertext `ct` on every rank (the other ranks pass None): shape, level and scale first (exact in
    float64), then the active limbs"""
    head = torch.zeros(4, dtype=torch.float64, device=ctx.device)
    if rank == 0:
        ct = _active(ct)
        head = torch.tensor([ct.batch, ct.size, ct.limbs, ct.scale], dtype=torch.float64, device=ctx.device)
    batch, size, limbs, scale = exchange.broadcast(head).tolist()
    batch, size, limbs = int(batch), int(size), int(limbs)
    data = ct.data if rank == 0 else torch.empty((batch, size, limbs, ctx.n), dtype=torch.int64, device=ctx.device)
    return Ciphertext(ctx, exchange.broadcast(data), limbs, scale)


def sharded_update_weights(ev, rows_local, row_ids, cols_local, feature_ids, labels, weights, lr, R, C, scale, keys,
                           encoder, encryptor, rank, world_size, exchange, degree=3, method="horner", mark=None,
                           sigmoid=None):
    """lr.update_weights (logistic_regression_ckks.cpp:269-345, config 1) with its R row dot products and its C feature
    dot products sharded over `world_size` ranks; every rank returns the new-weights ciphertext, bit-identical to the
    one-GPU function on the full inputs.

    rows_local / row_ids: this rank's row ciphertexts and their row indices, cols_local / feature_ids: its feature-column
    ciphertexts and their feature indices (config1_shards; either may be an empty batch, which still carries level and
    scale).  labels and weights are replicated.  `exchange`: TorchExchange, or a test emulation with its all_gather and
    broadcast.  `encryptor`: rank 0's, which makes exactly the calls of the one-GPU function (the polynomial encrypts its
    top coefficient); the other ranks pass None.  `mark(name)`, when given, is called as each phase ends.

    Prediction: cipher_dot_product of the own rows with the weights, the one-hot masks e_i of the own rows only, fused
    multiply_plain_sum; all-gather + mod-q add of the partials BEFORE relinearize / rescale (the rescale rounds and does
    not commute with the sum).  Rank 0 rescales, evaluates the sigmoid polynomial, subtracts the labels and broadcasts
    pred - labels.  Gradient: cipher_dot_product of the own feature columns with pred - labels (R - 1 dependent unit
    rotations each; a chain cannot be split without changing the ciphertext, so this phase shards at most C ways), masks
    e_j, multiply_plain_sum, all-gather + mod-q add before the rescale; the learning-rate tail runs on every rank."""
    if not 0 <= rank < world_size or rows_local.batch != len(row_ids) or cols_local.batch != len(feature_ids):
        raise ValueError("sharded_update_weights: rank or shard sizes do not match")
    mark = mark or (lambda name: None)
    ctx = weights.ctx
    if rows_local.batch:
        results = cipher_dot_product(ev, rows_local, weights, C, keys)
        mask_pt = encoder.encode(prediction_masks(_one_hot(row_ids, R), method, sigmoid), scale)
        ev.mod_switch_to_next_inplace(mask_pt)
        part = ev.multiply_plain_sum(results, mask_pt)
    else:
        part = _zero_partial(ctx, weights.limbs - 1,
                             _rescaled_pow2_scale(ctx, rows_local.scale * weights.scale, weights.limbs) * scale)
    mark("prediction")
    lin = _combine(ev, _active(part), exchange)
    mark("combine_prediction")
    pred_labels = None
    if rank == 0:
        lin = ev.relinearize(lin, keys)
        ev.rescale_to_next_inplace(lin)
        pred = sigmoid_cipher(ev, lin, scale, keys, encoder, encryptor, degree, method, sigmoid)
        lab = ev.mod_switch_to(labels, pred.limbs)
        if lab.scale != pred.scale:
            pred.scale = lab.scale
        pred_labels = ev.sub(pred, lab)
    pred_labels = _broadcast_ct(ctx, pred_labels, rank, exchange)
    mark("polynomial_broadcast")
    cols = ev.mod_switch_to(cols_local, pred_labels.limbs)
    if cols.batch:
        grads = cipher_dot_product(ev, cols, pred_labels, R, keys)
        mask_pt = encoder.encode(_one_hot(feature_ids, C), scale, limbs=grads.limbs)
        part = ev.multiply_plain_sum(grads, mask_pt)
    else:
        part = _zero_partial(ctx, pred_labels.limbs - 1,
                             _rescaled_pow2_scale(ctx, cols.scale * pred_labels.scale, pred_labels.limbs) * scale)
    mark("gradient")
    gradient = _combine(ev, _active(part), exchange)
    mark("combine_gradient")
    gradient = ev.relinearize(gradient, keys)
    ev.rescale_to_next_inplace(gradient)
    force_scale_pow2(gradient)
    new_weights = apply_gradient(ev, gradient, weights, lr, R, scale, encoder)
    mark("tail")
    return new_weights


def sharded_train_cipher(ev, rows_local, row_ids, cols_local, feature_ids, labels, weights, lr, iters, layout, scale, keys,
                         encoder, encryptor, decryptor, rank, world_size, exchange, degree=3, method="horner", sigmoid=None):
    """lr.train_cipher (logistic_regression_ckks.cpp:348-385, repair R4) over sharded_update_weights: after every
    iteration rank 0, the key holder (only it has a `decryptor` and an `encryptor`), decrypts and decodes the weights,
    re-packs them (RowLayout.weights), encodes them at the top level, re-encrypts them and broadcasts the ciphertext.
    Rank 0's encryptor sees the calls of the one-GPU train_cipher in the same order, so with the same seeds every rank
    returns a ciphertext bit-identical to it."""
    new_weights = weights
    for _ in range(iters):
        new_weights = sharded_update_weights(ev, rows_local, row_ids, cols_local, feature_ids, labels, new_weights, lr,
                                             layout.R, layout.C, scale, keys, encoder, encryptor, rank, world_size, exchange,
                                             degree=degree, method=method, sigmoid=sigmoid)
        fresh = None
        if rank == 0:
            decoded = encoder.decode(decryptor.decrypt(new_weights))[0, : layout.C]
            fresh = encryptor.encrypt(encoder.encode(layout.weights(decoded), scale))
        new_weights = _broadcast_ct(weights.ctx, fresh, rank, exchange)
    return new_weights


# ------------------------------------------------------------------ sharded column-layout training
def column_units(M, C, rank, world_size):
    """this rank's (mini-batch, feature) gradient units of the column layout: a contiguous block of the M*C units in
    (m, j) order, so that a rank touches as few mini-batches as possible.  The first M*C mod G ranks own one unit more;
    with more ranks than units the last ranks own none."""
    return [(u // C, u % C) for u in owned_block(M * C, rank, world_size)]


def column_keyswitches(R, C, B, rank, world_size, method, degree=7, sigmoid=None):
    """key switches of this rank in one sharded_train_columns iteration with the power-of-two Galois keys: per
    mini-batch its units touch, 1 prediction relinearisation + the polynomial's relinearisations (chebyshev_keyswitches
    of the sigmoid's degree, degree - 1 for Tree_cipher, degree for Horner_cipher; repeated on every rank that shares
    the mini-batch); per own unit 1 relinearisation + rotate_vector(-B) (its NAF weight) + B - 1 chain steps"""
    units = column_units(R // B, C, rank, world_size)
    if method == "chebyshev":
        poly = chebyshev_keyswitches((sigmoid or SIGMOID_CHEBYSHEV).degree)
    else:
        poly = degree - 1 if method == "tree" else degree
    return len({m for m, _ in units}) * (1 + poly) + len(units) * (1 + naf_weight(B) + B - 1)


def sharded_train_columns(ev, cols_local, labels_local, minibatch_ids, units, weights, w_bcast, lr, iters, layout, scale,
                          keys, encoder, encryptor, decryptor, rank, world_size, exchange, method="chebyshev",
                          sigmoid=None, mark=None):
    """lr.train_columns with the M*C (mini-batch, feature) gradient units sharded over `world_size` ranks; after every
    iteration every rank holds (weights, w_bcast) bit-identical to the one-GPU loop.

    cols_local / labels_local: the column (entry k*C + j) and label ciphertexts of the mini-batches `minibatch_ids`
    (increasing) that this rank's `units` (column_units, global (m, j) pairs) touch; both may be empty batches, which
    still carry level and scale.  weights / w_bcast: replicated.  `encryptor` and `decryptor`: rank 0's, the key
    holder's; the other ranks pass None.  `exchange`: TorchExchange, or a test emulation with all_gather and broadcast.

    Each rank evaluates the prediction and the polynomial of its own mini-batches (repeated where ranks share one) and
    the gradient chains of its own units; the partial gradients are summed by all-gather + mod-q add before the rescale
    (a rank without units adds zero), and the learning-rate tail runs on every rank.  Rank 0 then refreshes the weights
    (lr.refresh_columns) and broadcasts the packed weights and the C broadcasts.  Only method="chebyshev" is accepted:
    Tree_cipher and Horner_cipher encrypt a coefficient on every call, so ranks evaluating the same mini-batch would
    disagree.  `mark(name)`, when given, is called as each phase ends: prediction, polynomial, gradient, combine,
    tail, refresh."""
    if method != "chebyshev":
        raise ValueError("sharded_train_columns: only method='chebyshev' is deterministic; the reference polynomials "
                         "encrypt a coefficient, so ranks sharing a mini-batch would disagree")
    C = layout.C
    if (not 0 <= rank < world_size or cols_local.batch != len(minibatch_ids) * C or labels_local.batch != len(minibatch_ids)
            or any(m not in minibatch_ids for m, _ in units)):
        raise ValueError("sharded_train_columns: rank, shard sizes or units do not match")
    mark = mark or (lambda name: None)
    ctx = weights.ctx
    pos = {m: k for k, m in enumerate(minibatch_ids)}
    local = [(pos[m], j) for m, j in units]

    def combine(part):
        return _combine(ev, _active(part), exchange)
    for _ in range(iters):
        if local:
            grad = column_epoch_gradient(ev, cols_local, labels_local, w_bcast, C, layout.B, scale, keys, encoder, encryptor,
                                         method=method, units=local, combine=combine, sigmoid=sigmoid, mark=mark)
        else:                               # no unit here: the prediction's level and scale give the zero partial
            Lp = cols_local.limbs - 1 - chebyshev_depth((sigmoid or SIGMOID_CHEBYSHEV).degree)
            part = _zero_partial(ctx, Lp - 1, _rescaled_pow2_scale(ctx, cols_local.scale * labels_local.scale, Lp) * scale)
            for name in ("prediction", "polynomial", "gradient"):
                mark(name)
            grad = combine(part)
            mark("combine")
            ev.rescale_to_next_inplace(grad)
            force_scale_pow2(grad)
        new_weights = apply_gradient(ev, grad, weights, lr, layout.R, scale, encoder)
        mark("tail")
        fresh = (None, None)
        if rank == 0:
            fresh = refresh_columns(new_weights, layout, scale, encoder, encryptor, decryptor, method, sigmoid)
        weights, w_bcast = [_broadcast_ct(ctx, ct, rank, exchange) for ct in fresh]
        mark("refresh")
    return weights, w_bcast


# ------------------------------------------------------------------ sharded double hoisting
# An output of rotate_multiply_sum_hoisted is ModDown_P(sum_z w_z (.) IP_z) + base.  The sum is taken in Q_L u {P}, exact
# modulo every prime and indifferent to how its terms are grouped, so ranks split the terms of one output, exchange their
# extended-basis partials (rotate_multiply_sum_hoisted_partial, which folds P * base in) and each runs the one mod-down
# (rms_mod_down) on the sum: one mod-down per output at every world size, word for word the one-GPU ciphertext.  A rank
# needs the Galois keys of its own terms' steps only.
def shard_terms(outputs, rank, world_size):
    """this rank's share of a term table (one list of (input, step, plaintext) terms per output): the terms of all
    outputs, in order, are cut into world_size contiguous runs with equal numbers of non-zero-step terms (key inner
    products; owned_block of their count); a step-0 term goes with the next non-zero-step term (the last one when none
    follows).  Returns one list per output, each a contiguous run of that output's terms in their order; ranks beyond
    the number of non-zero-step terms get nothing."""
    total = sum(1 for terms in outputs for _, s, _ in terms if s != 0)
    block = owned_block(total, rank, world_size)
    mine, k = [], 0
    for terms in outputs:
        run = []
        for t in terms:
            if (k in block) if total else rank == 0:
                run.append(t)
            if t[1] != 0:
                k += 1
            k = min(k, total - 1)
        mine.append(run)
    return mine


def _rank_steps(fill, *tables):
    """Galois steps of a rank's term tables, plus the duplicate-fill step when it runs any term"""
    used = any(terms for outputs in tables for terms in outputs)
    return sorted(term_steps(*tables) | ({fill} if used else set()))


def linear_transform_double_hoisted_rank_steps(d, rank, world_size):
    """Galois steps of this rank in sharded_linear_transform_plain_double_hoisted"""
    return _rank_steps(-d, shard_terms(diagonal_terms([range(d)], [0]), rank, world_size))


def _bsgs_rank_tables(d, b, rank, world_size):
    """this rank's baby outputs (owned_block of the G outputs), their baby term table and its giant terms (inputs: the
    owned baby outputs in order)"""
    baby, _ = bsgs_terms(d, b)
    own = list(owned_block(len(baby), rank, world_size))
    return own, [baby[g] for g in own], [[(i, g * b, -1) for i, g in enumerate(own)]] if own else []


def bsgs_double_hoisted_rank_steps(d, b, rank, world_size):
    """Galois steps of this rank in sharded_linear_transform_plain_bsgs_double_hoisted"""
    _, baby, giant = _bsgs_rank_tables(d, b, rank, world_size)
    return _rank_steps(-d, baby, giant)


def _matmul_rank_tables(sig, tau, V, W, rank, world_size):
    """this rank's share of cc_matrix_multiplication_nonzero_hoisted: its sigma / tau terms (shard_terms), its block of
    k (owned_block of d - 1) and the V_k / W_k term table of those k (plaintexts numbered V_k of own, then W_k of own)"""
    first, _ = matmul_nonzero_hoisted_terms(sig, tau, V, W)
    own = list(owned_block(len(V), rank, world_size))
    second = diagonal_terms([V[k] for k in own] + [W[k] for k in own], [0] * len(own) + [1] * len(own))
    return shard_terms(first, rank, world_size), own, second


def matmul_nonzero_hoisted_rank_steps(d, rank, world_size):
    """Galois steps of this rank in sharded_cc_matrix_multiplication_nonzero_hoisted"""
    first, _, second = _matmul_rank_tables(*matmul_diagonal_indices(d), rank, world_size)
    return _rank_steps(-d * d, first, second)


def _zero_extended(ct, n):
    """the extended-basis partial of a rank without terms: zeros"""
    data = torch.zeros((n, 2, ct.limbs + 1, ct.ctx.n), dtype=torch.int64, device=ct.data.device)
    return ExtendedPartial(ct.ctx, data, ct.limbs, ct.scale)


def _mod_down_sum(ev, part, scale, world_size, exchange, mark):
    """all-gather of every rank's partial, then the one mod-down of their sum.  `scale`: the one-GPU output scale (a
    rank without terms holds zeros, whose scale is immaterial)"""
    mark("partial")
    gathered = exchange.all_gather(part.data)
    mark("exchange")
    out = ev.rms_mod_down(ExtendedPartial(part.ctx, gathered, part.limbs, scale), world_size)
    mark("mod_down")
    return out


def sharded_linear_transform_plain_double_hoisted(ev, ct, diags, keys, plans, rank, world_size, exchange, mark=None):
    """linear_transform_plain_double_hoisted with the terms of its one output sharded (shard_terms); every rank with
    terms runs the duplicate fill, one all-gather of one partial, one mod-down.  Every rank returns the one-GPU
    ciphertext.  `keys`: linear_transform_double_hoisted_rank_steps(d, rank, world_size).  `mark(name)`: optional
    phase callback."""
    mark = mark or (lambda name: None)
    d = diags.batch
    mine = shard_terms(diagonal_terms([range(d)], [0]), rank, world_size)
    if mine[0]:
        part = ev.rotate_multiply_sum_hoisted_partial(duplicate_fill(ev, ct, d, keys), diags, plans.rms(1, d, mine))
    else:
        part = _zero_extended(ct, 1)
    return _mod_down_sum(ev, part, ct.scale * diags.scale, world_size, exchange, mark)


def sharded_linear_transform_plain_bsgs_double_hoisted(ev, ct, bd, keys, plans, rank, world_size, exchange, mark=None):
    """linear_transform_plain_bsgs_double_hoisted with whole baby outputs sharded by owned_block: a rank computes its
    baby outputs (no exchange: a sub-plan's outputs equal the full plan's) and the partial of the giant terms over them;
    one all-gather of one partial and one mod-down give every rank the one-GPU ciphertext.
    `keys`: bsgs_double_hoisted_rank_steps(d, b, rank, world_size)."""
    mark = mark or (lambda name: None)
    d, b = bd.d, bd.b
    own, baby, giant = _bsgs_rank_tables(d, b, rank, world_size)
    if own:
        inner = ev.rotate_multiply_sum_hoisted(duplicate_fill(ev, ct, d, keys), bd.plain, plans.rms(1, d, baby))
        part = ev.rotate_multiply_sum_hoisted_partial(inner, None, plans.rms(len(own), 0, giant))
    else:
        part = _zero_extended(ct, 1)
    return _mod_down_sum(ev, part, ct.scale * bd.plain.scale, world_size, exchange, mark)


def sharded_cc_matrix_multiplication_nonzero_hoisted(ev, ctA, ctB, d, sigma, tau, V, W, keys, plans, rank, world_size,
                                                     exchange, mark=None):
    """cc_matrix_multiplication_nonzero_hoisted over world_size ranks; every rank returns the one-GPU product word for word.
    1. sigma(A) / tau(B) with sharded terms: all-gather of the partials and one mod-down, A0 and B0 on every rank.
    2. V_k / W_k for this rank's block of k (owned_block(d - 1)), whole outputs, no exchange.
    3. The tail of sharded_cc_matrix_multiplication: rescale, forced scales, multiply_sum over the owned k, all-gather +
       mod-q add of the size-3 partials, + mod_switch(A0 x B0).
    `keys`: matmul_nonzero_hoisted_rank_steps(d, rank, world_size)."""
    mark = mark or (lambda name: None)
    dd = d * d
    first, own, second = _matmul_rank_tables(sigma.index, tau.index, [s.index for s in V], [s.index for s in W], rank,
                                             world_size)
    pts = _stack([sigma.special, tau.special])
    if any(first):
        X = _stack([duplicate_fill(ev, ctA, dd, keys), duplicate_fill(ev, ctB, dd, keys)])
        part = ev.rotate_multiply_sum_hoisted_partial(X, pts, plans.rms(2, pts.batch, first))
    else:
        part = _zero_extended(ctA, 2)
    AB0 = _mod_down_sum(ev, part, ctA.scale * pts.scale, world_size, exchange, mark)
    A0, B0 = AB0[0], AB0[1]

    ctAB = ev.multiply(A0, B0)
    ev.mod_switch_to_next_inplace(ctAB)
    pt_scale = V[0].special.scale
    if own:
        Y = _stack([duplicate_fill(ev, A0, dd, keys), duplicate_fill(ev, B0, dd, keys)])
        pts = _stack([V[k].special for k in own] + [W[k].special for k in own])
        XK = ev.rotate_multiply_sum_hoisted(Y, pts, plans.rms(2, pts.batch, second))
        mark("step2")
        Ak, Bk = XK[0:len(own)], XK[len(own):]
        for X in (Ak, Bk):
            ev.rescale_to_next_inplace(X)
            force_scale_pow2(X)
        rest = ev.multiply_sum(Ak, Bk)
    else:                                   # more ranks than products: this rank adds zero
        mark("step2")
        scale = (_rescaled_pow2_scale(A0.ctx, A0.scale * pt_scale, A0.limbs)
                 * _rescaled_pow2_scale(B0.ctx, B0.scale * pt_scale, B0.limbs))
        rest = _zeros(A0, 3, 1, scale)
        rest.limbs = A0.limbs - 1
    rest = _combine(ev, rest, exchange)
    if rest.scale != ctAB.scale:
        raise capi.CkksInvalidArgument("scale mismatch")
    out = ev.add(ctAB, rest)
    mark("tail")
    return out


# ------------------------------------------------------------------ sharded blocked matrix product
def blocked_shards(tiles, rank, world_size):
    """this rank's share of cc_matrix_multiplication_blocked at tile grid (t_n, t_m, t_p): a contiguous run of the
    t_n t_m + t_m t_p operand transforms (A's tiles, then B's, row-major) and a contiguous block of the t_n t_p output
    tiles (owned_block of each count; ranks beyond a count get an empty range)"""
    tn, tm, tp = tiles
    return owned_block(tn * tm + tm * tp, rank, world_size), owned_block(tn * tp, rank, world_size)


def _operand_scales(ctx, ct, first, sets, limbs):
    """(scale of the entries k >= 1, scale0) of matmul_operands for tiles like `ct`, from the scale arithmetic alone (a
    rank that transforms no tile of this operand still needs them)"""
    s0 = ct.scale * first.special.scale
    return _rescaled_pow2_scale(ctx, s0 * sets[0].special.scale, limbs), s0


def sharded_cc_matrix_multiplication_blocked(ev, A_tiles, B_tiles, tiles, d, sigma, tau, V, W, keys, plans, rank,
                                             world_size, exchange, method="reference"):
    """cc_matrix_multiplication_blocked over world_size ranks; every rank returns the t_n t_p output tiles of the one-GPU
    call word for word.  Every rank holds all input tiles and needs the one-GPU call's Galois keys.

    1. The rank transforms its contiguous run of the t_n t_m + t_m t_p tiles (blocked_shards; matmul_operands, A's and
       B's tiles of the run in one call each).  One all-gather of the entries, padded to the longest run: d size-2
       ciphertexts per transformed tile at the product's level L - 1, so (t_n t_m + t_m t_p) d * 2 (L - 1) N words in
       all (plus padding).  A rank with no tile sends zeros.
    2. It contracts its owned_block of the output tiles (row-major), one multiply_sum_matrix per touched tile row.
    3. A second all-gather of the t_n t_p size-3 outputs (3 (L - 1) N words each, padded; zeros from ranks that own
       none) gives every rank all of them."""
    tn, tm, tp = (int(x) for x in tiles)
    if min(tn, tm, tp) < 1 or A_tiles.batch != tn * tm or B_tiles.batch != tm * tp:
        raise ValueError("sharded_cc_matrix_multiplication_blocked: tile batches do not match the tile grid")
    ctx, nA = A_tiles.ctx, tn * tm
    mine, outs = blocked_shards((tn, tm, tp), rank, world_size)
    L = A_tiles.limbs - 1
    sX, sX0 = _operand_scales(ctx, A_tiles, sigma, V, A_tiles.limbs)
    sY, sY0 = _operand_scales(ctx, B_tiles, tau, W, B_tiles.limbs)
    # 1. this rank's transforms, padded to the longest run, all-gathered
    per = -(-(nA + tm * tp) // world_size)
    send = torch.zeros((per * d, 2, L, ctx.n), dtype=torch.int64, device=A_tiles.data.device)
    pos = 0
    for src, lo, hi, side in ((A_tiles, mine.start, min(mine.stop, nA), 0),
                              (B_tiles, max(mine.start, nA) - nA, mine.stop - nA, 1)):
        if hi > lo:
            ent = matmul_operands(ev, src[lo:hi], [side] * (hi - lo), d, sigma, tau, V, W, keys, plans, method)
            send[pos:pos + ent.data.batch] = ent.data.data[:, :, :L]
            pos += ent.data.batch
    got = exchange.all_gather(send)
    order = []
    for q in range(world_size):
        blk = owned_block(nA + tm * tp, q, world_size)
        order += range(q * per * d, q * per * d + len(blk) * d)
    got = got.index_select(0, torch.as_tensor(order, device=got.device))
    X = MatmulEntries(Ciphertext(ctx, got[:nA * d].contiguous(), L, sX), d, sX0)
    Y = MatmulEntries(Ciphertext(ctx, got[nA * d:].contiguous(), L, sY), d, sY0)
    del got
    if X.scale0 * Y.scale0 != X.data.scale * Y.data.scale:
        raise capi.CkksInvalidArgument("scale mismatch")
    # 2. the owned output tiles, one contraction per touched tile row
    per_out = -(-(tn * tp) // world_size)
    part = torch.zeros((per_out, 3, L, ctx.n), dtype=torch.int64, device=send.device)
    del send
    if len(outs):
        Yc = _column_major_rows(Y, tp)
        inner = tm * d
        o = outs.start
        while o < outs.stop:
            i, j0 = divmod(o, tp)
            j1 = min(tp, j0 + outs.stop - o)
            if j1 - j0 == tp:
                b = Yc
            else:
                cols = torch.arange(j0, j1, device=part.device)
                idx = (torch.arange(inner, device=part.device)[:, None] * tp + cols[None, :]).reshape(-1)
                b = Ciphertext(ctx, Yc.data.index_select(0, idx), L, Yc.scale)
            a = X.data[i * inner:(i + 1) * inner]
            r = ev.multiply_sum_matrix(a, b, 1, j1 - j0)
            part[o - outs.start:o - outs.start + j1 - j0] = r.data[:, :, :L]
            o += j1 - j0
    # 3. every rank's outputs
    got = exchange.all_gather(part)
    order = []
    for q in range(world_size):
        blk = owned_block(tn * tp, q, world_size)
        order += range(q * per_out, q * per_out + len(blk))
    got = got.index_select(0, torch.as_tensor(order, device=got.device))
    return Ciphertext(ctx, got, L, sX * sY)
