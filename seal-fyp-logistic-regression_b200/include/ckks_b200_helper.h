// ckks_b200_helper.h -- batched drop-ins for the rotation-heavy functions of the reference's helper.h.
//
// Same names, argument order and results as the reference's functions, in namespace b200, built on the
// batched entry points of include/ckks_b200.h (rotation plans, fused multiply + add_many, the fused
// rotate-and-sum chain) instead of one evaluator call per ciphertext.  Every function issues, per
// ciphertext, exactly the reference's evaluator sequence, so the returned ciphertext polynomials are
// bit-identical to what the reference's own function returns through seal/seal.h (checked by
// tests/cpp/helper_driver.cpp); what changes is that independent ciphertexts share kernel launches.
//
//   reference (helper.h)                               here
//   Linear_Transform_Plain            :237-262         b200::Linear_Transform_Plain
//   Linear_Transform_Cipher           :212-234         b200::Linear_Transform_Cipher
//   Linear_Transform_CipherMatrix_PlainVector :265-278 b200::Linear_Transform_CipherMatrix_PlainVector
//   C_Matrix_Encode                   :307-322         b200::C_Matrix_Encode
//   C_Matrix_Decode                   :325-360         b200::C_Matrix_Decode
//   cipher_dot_product                :416-502         b200::cipher_dot_product
//   CC_Matrix_Multiplication (matrix_mult_benchmark.cpp:13-71)  b200::CC_Matrix_Multiplication
//   (no counterpart: per tile, summed over l)                   b200::CC_Matrix_Multiplication_blocked
//
// A maintainer switches a call site by prefixing it with b200:: (or `using b200::Linear_Transform_Plain;`).
// Differences from the reference, all deliberate: arguments are taken by const reference (the reference
// copies them by value, which is only cheaper here); a zero plaintext diagonal does not raise SEAL's
// "result ciphertext is transparent" (the reference's drivers add an epsilon to avoid it).
#pragma once
#include <cmath>
#include <memory>
#include <stdexcept>
#include <vector>

#include "seal/seal.h"

namespace b200 {
namespace detail {

using seal::detail::BufPtr;
using seal::detail::check;
using seal::detail::DevBuf;
using seal::detail::Engine;
using seal::detail::Poly;

// B objects of `size` polynomials with `limbs` limbs each, contiguous: [B][size][limbs][N]
struct Batch {
    std::shared_ptr<Engine> e;
    BufPtr buf;
    int batch = 0, size = 0, limbs = 0;
    double scale = 1.0;
    Batch(std::shared_ptr<Engine> eng, int batch_, int size_, int limbs_, double scale_)
        : e(std::move(eng)), batch(batch_), size(size_), limbs(limbs_), scale(scale_) {
        buf = std::make_shared<DevBuf>(e, (std::size_t)batch * size * limbs * e->n);
    }
    std::size_t entry_words() const { return (std::size_t)size * limbs * e->n; }
    ckks_view view() const {
        ckks_view v;
        v.data = buf->p;
        v.batch_stride = entry_words();
        v.poly_stride = (std::uint64_t)limbs * e->n;
        v.batch = batch;
        v.size = size;
        v.limbs = limbs;
        v.reserved = 0;
        return v;
    }
    // copy one shim object into / out of entry b (limb capacity of the object may exceed its level)
    void put(int b, const Poly &p) {
        if (!p.buf || p.size != size || p.limbs != limbs) throw std::invalid_argument("encrypted1 and encrypted2 parameter mismatch");
        for (int k = 0; k < size; k++)
            check(ckks_copy(e->ctx, buf->p + b * entry_words() + (std::size_t)k * limbs * e->n,
                            p.buf->p + (std::size_t)k * p.cap * e->n, (std::size_t)limbs * e->n * 8, nullptr));
    }
    void get(int b, Poly &p) const {
        p.allocate(e, size, limbs);
        p.scale = scale;
        check(ckks_copy(e->ctx, p.buf->p, buf->p + b * entry_words(), entry_words() * 8, nullptr));
    }
};

template <class T>
inline Batch gather(const std::vector<T> &objs) {
    if (objs.empty()) throw std::invalid_argument("encrypteds cannot be empty");
    const Poly &p0 = objs[0].poly();
    if (!p0.buf) throw std::invalid_argument("encrypted is not valid for encryption parameters");
    Batch b(p0.eng, (int)objs.size(), p0.size, p0.limbs, p0.scale);
    for (std::size_t i = 0; i < objs.size(); i++) {
        if (objs[i].poly().scale != p0.scale) throw std::invalid_argument("scale mismatch");
        b.put((int)i, objs[i].poly());
    }
    return b;
}

struct Plan {   // RAII around ckks_rotplan
    ckks_rotplan *p = nullptr;
    Plan(const std::shared_ptr<Engine> &e, const seal::GaloisKeys &gk, const std::vector<int> &steps) {
        if (!gk.s || !gk.s->ks) throw std::invalid_argument("galois_keys is not valid for encryption parameters");
        check(ckks_rotplan_create(e->ctx, gk.s->ks, steps.data(), (int)steps.size(), &p));
    }
    ~Plan() {
        if (p) ckks_rotplan_destroy(p);
    }
    Plan(const Plan &) = delete;
};

// rot(ct, steps[b]) for every b as one batched call; `in` is one ciphertext (batch 1) or a batch
inline Batch rotate_all(const ckks_view &in, const std::shared_ptr<Engine> &e, double scale, const seal::GaloisKeys &gk,
                        const std::vector<int> &steps) {
    Plan plan(e, gk, steps);
    Batch out(e, (int)steps.size(), 2, in.limbs, scale), scratch(e, (int)steps.size(), 2, in.limbs, scale);
    ckks_view vo = out.view(), vs = scratch.view();
    check(ckks_rotate_plan(e->ctx, plan.p, &in, &vo, &vs, nullptr));
    return out;
}

inline void scale_ok(const Engine &e, double scale, int limbs) {
    long double lg = 0;
    for (int j = 0; j < limbs; j++) lg += std::log2((long double)e.primes[j]);
    if (scale <= 0 || (int)std::log2(scale) >= (int)std::floor(lg) + 1) throw std::invalid_argument("scale out of bounds");
}

// ct + rotate_vector(ct, -d): "Fill ct with duplicate" (helper.h:241-247)
inline seal::Ciphertext duplicate(const seal::Ciphertext &ct, int d, const seal::GaloisKeys &gk, seal::Evaluator &ev) {
    seal::Ciphertext rot, out;
    ev.rotate_vector(ct, -d, gk, rot);
    ev.add(ct, rot, out);
    return out;
}

// The V_k (W_k) step of CC_Matrix_Multiplication for k = 1..K1 on the sigma (tau) transform `base`: the d*d rotations of
// base + rotate_vector(base, -d*d) are computed once and shared by the K1 transforms, which are rescaled and given the
// reference's "manual rescale" power-of-two scale.  Returns the K1 results as one batch at base's level - 1.
inline Batch shifted(const seal::Ciphertext &base, const std::vector<std::vector<seal::Plaintext>> &sets, int K1,
                     const seal::GaloisKeys &gal_keys, seal::Evaluator &evaluator) {
    const int dd = (int)sets[0].size();
    std::vector<int> steps(dd);
    for (int l = 0; l < dd; l++) steps[l] = l;
    seal::Ciphertext dup = duplicate(base, dd, gal_keys, evaluator);
    const Poly &pn = dup.poly();
    Batch rots = rotate_all(pn.view(), pn.eng, pn.scale, gal_keys, steps);
    double pscale = sets[0][0].poly().scale;
    scale_ok(*pn.eng, pn.scale * pscale, pn.limbs);
    Batch out(pn.eng, K1, 2, pn.limbs, pn.scale * pscale);
    for (int k = 0; k < K1; k++) {
        if ((int)sets[k].size() != dd) throw std::invalid_argument("encrypted and plain parameter mismatch");
        Batch diags = gather(sets[k]);
        if (diags.limbs != pn.limbs || diags.scale != pscale) throw std::invalid_argument("encrypted and plain parameter mismatch");
        ckks_view vr = rots.view(), vd = diags.view(), vo = out.view();
        vo.data += (std::size_t)k * out.entry_words();
        vo.batch = 1;
        check(ckks_multiply_plain_sum(pn.eng->ctx, &vr, &vd, &vo, nullptr));
    }
    // rescale_to_next_inplace on every A_k / B_k, then the reference's "manual rescale" of the scale
    Batch low(pn.eng, K1, 2, pn.limbs - 1, 0.0);
    if (pn.limbs < 2) throw std::invalid_argument("end of modulus switching chain reached");
    ckks_view vi = out.view(), vl = low.view();
    check(ckks_rescale(pn.eng->ctx, &vi, &vl, nullptr));
    low.scale = std::pow(2.0, (int)std::log2(out.scale / (double)pn.eng->primes[pn.limbs - 1]));
    return low;
}

}  // namespace detail

// helper.h:237-262 -- sum_l U_diagonals[l] (.) rotate_vector(ct + rotate_vector(ct, -d), l)
inline seal::Ciphertext Linear_Transform_Plain(const seal::Ciphertext &ct, const std::vector<seal::Plaintext> &U_diagonals,
                                               const seal::GaloisKeys &gal_keys, const seal::EncryptionParameters &params) {
    auto context = seal::SEALContext::Create(params);
    seal::Evaluator evaluator(context);
    const int d = (int)U_diagonals.size();
    detail::Batch diags = detail::gather(U_diagonals);
    seal::Ciphertext ct_new = detail::duplicate(ct, d, gal_keys, evaluator);
    const detail::Poly &pn = ct_new.poly();
    if (pn.limbs != diags.limbs) throw std::invalid_argument("encrypted and plain parameter mismatch");
    detail::scale_ok(*pn.eng, pn.scale * diags.scale, pn.limbs);
    std::vector<int> steps(d);
    for (int l = 0; l < d; l++) steps[l] = l;
    detail::Batch rots = detail::rotate_all(pn.view(), pn.eng, pn.scale, gal_keys, steps);
    seal::Ciphertext out;
    out.poly().allocate(pn.eng, 2, pn.limbs);
    out.poly().scale = pn.scale * diags.scale;
    ckks_view vr = rots.view(), vd = diags.view(), vo = out.poly().view();
    detail::check(ckks_multiply_plain_sum(pn.eng->ctx, &vr, &vd, &vo, nullptr));
    return out;
}

// SURVEY 8(f4), opt-in: Linear_Transform_Plain with HOISTED rotations -- the d-1 rotations of the hot loop (helper.h:252-257)
// all act on the same ct_new, so its digit decomposition is shared (ckks_rotate_plan_hoisted).  gal_keys must hold a key for
// every step 1..d-1 themselves and for -d (keygen.galois_keys(steps)).  The result decrypts like Linear_Transform_Plain's within
// key-switch noise; its polynomials are NOT SEAL's (SEAL permutes before lifting digits), hence a separate function.
inline seal::Ciphertext Linear_Transform_Plain_hoisted(const seal::Ciphertext &ct, const std::vector<seal::Plaintext> &U_diagonals,
                                                       const seal::GaloisKeys &gal_keys, const seal::EncryptionParameters &params) {
    auto context = seal::SEALContext::Create(params);
    seal::Evaluator evaluator(context);
    const int d = (int)U_diagonals.size();
    detail::Batch diags = detail::gather(U_diagonals);
    seal::Ciphertext ct_new = detail::duplicate(ct, d, gal_keys, evaluator);
    const detail::Poly &pn = ct_new.poly();
    if (pn.limbs != diags.limbs) throw std::invalid_argument("encrypted and plain parameter mismatch");
    detail::scale_ok(*pn.eng, pn.scale * diags.scale, pn.limbs);
    std::vector<int> steps(d);
    for (int l = 0; l < d; l++) steps[l] = l;
    detail::Plan plan(pn.eng, gal_keys, steps);
    detail::Batch rots(pn.eng, d, 2, pn.limbs, pn.scale);
    ckks_view vi = pn.view(), vr = rots.view();
    detail::check(ckks_rotate_plan_hoisted(pn.eng->ctx, plan.p, &vi, &vr, nullptr));
    seal::Ciphertext out;
    out.poly().allocate(pn.eng, 2, pn.limbs);
    out.poly().scale = pn.scale * diags.scale;
    ckks_view vd = diags.view(), vo = out.poly().view();
    detail::check(ckks_multiply_plain_sum(pn.eng->ctx, &vr, &vd, &vo, nullptr));
    return out;
}

// Opt-in: Linear_Transform_Plain with DOUBLE hoisting -- one digit decomposition of ct_new, the d-1 key inner products
// weighted by their diagonals and summed in the extended basis, ONE mod-down (ckks_rotate_multiply_sum_hoisted).
// U_diagonals are encoded at the key level: encoder.encode(diag, context->key_parms_id(), scale, pt).  gal_keys: a key for
// every step 1..d-1 and for -d.  Decrypts like Linear_Transform_Plain within key-switch noise; different polynomials.
inline seal::Ciphertext Linear_Transform_Plain_double_hoisted(const seal::Ciphertext &ct, const std::vector<seal::Plaintext> &U_diagonals,
                                                              const seal::GaloisKeys &gal_keys, const seal::EncryptionParameters &params) {
    auto context = seal::SEALContext::Create(params);
    seal::Evaluator evaluator(context);
    const int d = (int)U_diagonals.size();
    detail::Batch diags = detail::gather(U_diagonals);
    seal::Ciphertext ct_new = detail::duplicate(ct, d, gal_keys, evaluator);
    const detail::Poly &pn = ct_new.poly();
    if (diags.limbs != pn.eng->K) throw std::invalid_argument("U_diagonals must be encoded at the key level (key_parms_id)");
    detail::scale_ok(*pn.eng, pn.scale * diags.scale, pn.limbs);
    if (!gal_keys.s || !gal_keys.s->ks) throw std::invalid_argument("galois_keys is not valid for encryption parameters");
    std::vector<int> first{0, d}, in_idx(d, 0), steps(d), pt_idx(d);
    for (int l = 0; l < d; l++) steps[l] = pt_idx[l] = l;
    ckks_rmsplan *plan = nullptr;
    detail::check(ckks_rmsplan_create(pn.eng->ctx, gal_keys.s->ks, 1, d, 1, first.data(), d, in_idx.data(), steps.data(),
                                      pt_idx.data(), &plan));
    seal::Ciphertext out;
    out.poly().allocate(pn.eng, 2, pn.limbs);
    out.poly().scale = pn.scale * diags.scale;
    ckks_view vi = pn.view(), vd = diags.view(), vo = out.poly().view();
    const int rc = ckks_rotate_multiply_sum_hoisted(pn.eng->ctx, plan, &vi, &vd, &vo, nullptr);
    ckks_rmsplan_destroy(plan);
    detail::check(rc);
    return out;
}

// helper.h:212-234 -- the same with ciphertext diagonals; the result has size 3 (no relinearisation)
inline seal::Ciphertext Linear_Transform_Cipher(const seal::Ciphertext &ct, const std::vector<seal::Ciphertext> &U_diagonals,
                                                const seal::GaloisKeys &gal_keys, seal::Evaluator &evaluator) {
    const int d = (int)U_diagonals.size();
    detail::Batch diags = detail::gather(U_diagonals);
    if (diags.size != 2) throw std::invalid_argument("encrypted size must be 2");
    seal::Ciphertext ct_new = detail::duplicate(ct, d, gal_keys, evaluator);
    const detail::Poly &pn = ct_new.poly();
    if (pn.limbs != diags.limbs) throw std::invalid_argument("encrypted1 and encrypted2 parameter mismatch");
    detail::scale_ok(*pn.eng, pn.scale * diags.scale, pn.limbs);
    std::vector<int> steps(d);
    for (int l = 0; l < d; l++) steps[l] = l;
    detail::Batch rots = detail::rotate_all(pn.view(), pn.eng, pn.scale, gal_keys, steps);
    seal::Ciphertext out;
    out.poly().allocate(pn.eng, 3, pn.limbs);
    out.poly().scale = pn.scale * diags.scale;
    ckks_view vr = rots.view(), vd = diags.view(), vo = out.poly().view();
    detail::check(ckks_multiply_sum(pn.eng->ctx, &vr, &vd, &vo, nullptr));
    return out;
}

// helper.h:265-278 -- sum_i U_diagonals[i] (.) pt_rotations[i] (no rotations: the vector is in the clear)
inline seal::Ciphertext Linear_Transform_CipherMatrix_PlainVector(const std::vector<seal::Plaintext> &pt_rotations,
                                                                  const std::vector<seal::Ciphertext> &U_diagonals,
                                                                  const seal::GaloisKeys &, seal::Evaluator &) {
    if (pt_rotations.size() != U_diagonals.size()) throw std::invalid_argument("encrypted and plain parameter mismatch");
    detail::Batch cts = detail::gather(U_diagonals), pts = detail::gather(pt_rotations);
    if (cts.limbs != pts.limbs) throw std::invalid_argument("encrypted and plain parameter mismatch");
    detail::scale_ok(*cts.e, cts.scale * pts.scale, cts.limbs);
    seal::Ciphertext out;
    out.poly().allocate(cts.e, cts.size, cts.limbs);
    out.poly().scale = cts.scale * pts.scale;
    ckks_view vc = cts.view(), vp = pts.view(), vo = out.poly().view();
    detail::check(ckks_multiply_plain_sum(cts.e->ctx, &vc, &vp, &vo, nullptr));
    return out;
}

// helper.h:307-322 -- pack the d row ciphertexts of a matrix into one: sum_i rotate_vector(matrix[i], -i*d)
inline seal::Ciphertext C_Matrix_Encode(const std::vector<seal::Ciphertext> &matrix, const seal::GaloisKeys &gal_keys,
                                        seal::Evaluator &) {
    const int d = (int)matrix.size();
    detail::Batch rows = detail::gather(matrix);
    if (rows.size != 2) throw std::invalid_argument("encrypted size must be 2");
    std::vector<int> steps(d);
    for (int i = 0; i < d; i++) steps[i] = -(i * d);
    detail::Batch rot = detail::rotate_all(rows.view(), rows.e, rows.scale, gal_keys, steps);
    seal::Ciphertext out;
    out.poly().allocate(rows.e, 2, rows.limbs);
    out.poly().scale = rows.scale;
    ckks_view vr = rot.view(), vo = out.poly().view();
    detail::check(ckks_add_many(rows.e->ctx, &vr, &vo, nullptr));
    return out;
}

// helper.h:325-360 -- split a packed matrix back into its d row ciphertexts: mask row i with ones (the d
// masks are encoded as one batch on the device), then rotate_vector by i*d (one rotation plan)
inline std::vector<seal::Ciphertext> C_Matrix_Decode(const seal::Ciphertext &matrix, int dimension, double scale,
                                                     const seal::GaloisKeys &gal_keys, seal::CKKSEncoder &ckks_encoder,
                                                     seal::Evaluator &) {
    const detail::Poly &pm = matrix.poly();
    if (!pm.buf) throw std::invalid_argument("encrypted is not valid for encryption parameters");
    if (pm.size != 2) throw std::invalid_argument("encrypted size must be 2");
    const int d = dimension, dd = d * d;
    if (d < 1 || (std::size_t)dd > ckks_encoder.slot_count()) throw std::invalid_argument("values has invalid size");
    if (pm.limbs != pm.eng->K - 1) throw std::invalid_argument("encrypted and plain parameter mismatch");   // masks are encoded at the top level
    detail::scale_ok(*pm.eng, pm.scale * scale, pm.limbs);
    std::vector<double> masks((std::size_t)d * dd, 0.0);
    for (int i = 0; i < d; i++)
        for (int j = 0; j < d; j++) masks[(std::size_t)i * dd + j + i * d] = 1.0;
    detail::DevBuf vals(pm.eng, masks.size());
    detail::check(ckks_upload(pm.eng->ctx, vals.p, masks.data(), masks.size() * 8, nullptr));
    detail::check(ckks_stream_sync(pm.eng->ctx, nullptr));   // `masks` is pageable host memory about to go out of scope
    detail::Batch pts(pm.eng, d, 1, pm.limbs, scale);
    ckks_view vp = pts.view();
    detail::check(ckks_encode(pm.eng->ctx, reinterpret_cast<const double *>(vals.p), dd, scale, &vp, nullptr));
    detail::Batch rows(pm.eng, d, 2, pm.limbs, pm.scale * scale);
    ckks_view vm = pm.view(), vr = rows.view();
    vm.batch = d;            // the same ciphertext for every mask
    vm.batch_stride = 0;
    detail::check(ckks_multiply_plain(pm.eng->ctx, &vm, &vp, &vr, nullptr));
    std::vector<int> steps(d);
    for (int i = 0; i < d; i++) steps[i] = i * d;
    detail::Batch rot = detail::rotate_all(vr, pm.eng, rows.scale, gal_keys, steps);
    std::vector<seal::Ciphertext> out(d);
    for (int i = 0; i < d; i++) rot.get(i, out[i].poly());
    return out;
}

// helper.h:416-502 -- multiply, relinearize, rescale, then the rotate-and-sum loop over `size` slots
// (size-1 dependent unit rotations, each fused with its add and replayed from a CUDA graph), scale forced
// to a power of two as the reference does
inline seal::Ciphertext cipher_dot_product(const seal::Ciphertext &ctA, const seal::Ciphertext &ctB, int size,
                                           const seal::RelinKeys &relin_keys, const seal::GaloisKeys &gal_keys,
                                           seal::Evaluator &evaluator) {
    seal::Ciphertext mult;
    evaluator.multiply(ctA, ctB, mult);
    evaluator.relinearize_inplace(mult, relin_keys);
    evaluator.rescale_to_next_inplace(mult);
    seal::Ciphertext zero_filled, dup;
    evaluator.rotate_vector(mult, -size, gal_keys, zero_filled);
    evaluator.add(mult, zero_filled, dup);
    if (size > 1) {
        if (!gal_keys.s || !gal_keys.s->ks) throw std::invalid_argument("galois_keys is not valid for encryption parameters");
        mult.poly().make_unique();
        dup.poly().make_unique();
        detail::Poly &pm = mult.poly(), &pd = dup.poly();
        detail::Poly scratch;
        scratch.allocate(pm.eng, 2, pd.limbs);
        ckks_view va = pd.view(), vb = scratch.view(), vc = pm.view();
        vb.limbs = va.limbs;
        int final_in_b = 0;
        detail::check(ckks_rotate_sum_chain(pm.eng->ctx, gal_keys.s->ks, &va, &vb, &vc, 1, size - 1, &final_in_b, nullptr));
    }
    mult.scale() = std::pow(2.0, (int)std::log2(mult.scale()));
    return mult;
}

// matrix_multiplication.cpp:11-132 / matrix_mult_benchmark.cpp:13-71 -- encrypted d x d matrix product of
// eprint 2018/1041: sigma(A), tau(B), the d-1 column / row shifts V_k, W_k of them, and sum_k A_k (.) B_k.
// Every V_k (W_k) transform of the reference rotates the same ciphertext by the same d*d steps; here those
// rotations are computed once and shared, which leaves every ciphertext polynomial unchanged.
inline seal::Ciphertext CC_Matrix_Multiplication(const seal::Ciphertext &ctA, const seal::Ciphertext &ctB, int dimension,
                                                 const std::vector<seal::Plaintext> &U_sigma_diagonals,
                                                 const std::vector<seal::Plaintext> &U_tau_diagonals,
                                                 const std::vector<std::vector<seal::Plaintext>> &V_diagonals,
                                                 const std::vector<std::vector<seal::Plaintext>> &W_diagonals,
                                                 const seal::GaloisKeys &gal_keys, const seal::EncryptionParameters &params) {
    auto context = seal::SEALContext::Create(params);
    seal::Evaluator evaluator(context);
    if (dimension < 1 || (int)V_diagonals.size() < dimension - 1 || (int)W_diagonals.size() < dimension - 1)
        throw std::invalid_argument("dimension does not match the diagonal sets");
    seal::Ciphertext A0 = Linear_Transform_Plain(ctA, U_sigma_diagonals, gal_keys, params);
    seal::Ciphertext B0 = Linear_Transform_Plain(ctB, U_tau_diagonals, gal_keys, params);
    seal::Ciphertext ctAB;
    evaluator.multiply(A0, B0, ctAB);
    evaluator.mod_switch_to_next_inplace(ctAB);
    if (dimension == 1) return ctAB;
    const int K1 = dimension - 1;
    detail::Batch Ak = detail::shifted(A0, V_diagonals, K1, gal_keys, evaluator),
                  Bk = detail::shifted(B0, W_diagonals, K1, gal_keys, evaluator);
    detail::scale_ok(*Ak.e, Ak.scale * Bk.scale, Ak.limbs);
    seal::Ciphertext rest;
    rest.poly().allocate(Ak.e, 3, Ak.limbs);
    rest.poly().scale = Ak.scale * Bk.scale;
    ckks_view va = Ak.view(), vb = Bk.view(), vo = rest.poly().view();
    detail::check(ckks_multiply_sum(Ak.e->ctx, &va, &vb, &vo, nullptr));
    seal::Ciphertext out;
    evaluator.add(ctAB, rest, out);
    return out;
}

// Blocked encrypted matrix product of any shape (eprint 2018/1041 per d x d tile): A is tn x tm tiles, B tm x tp, each
// tile a ciphertext in the reference's row-major d*d-slot layout, both vectors in row-major tile order.  Returns the
// tn*tp size-3 tiles of A B (row-major, not relinearised), output (i, j) bit-identical to adding
// CC_Matrix_Multiplication(A_il, B_lj) over l with Evaluator::add.  One tile product is
//     ModSwitch(A0 x B0) + sum_{k>=1} A_k x B_k = sum_{k=0}^{d-1} X_k x Y_k,  X_0 = ModSwitch(A0), X_k = A_k (Y for B),
// since the mod switch drops a limb and the tensor product works limb by limb; so every tile is transformed once
// (tn*tm + tm*tp transforms instead of 2 tn*tm*tp) and the sums over l and k are one ckks_multiply_sum_matrix.
// dimension must be at least 2: 1 x 1 tiles, which CC_Matrix_Multiplication accepts, throw std::invalid_argument.
inline std::vector<seal::Ciphertext> CC_Matrix_Multiplication_blocked(
    const std::vector<seal::Ciphertext> &A_tiles, const std::vector<seal::Ciphertext> &B_tiles, int tn, int tm, int tp,
    int dimension, const std::vector<seal::Plaintext> &U_sigma_diagonals, const std::vector<seal::Plaintext> &U_tau_diagonals,
    const std::vector<std::vector<seal::Plaintext>> &V_diagonals, const std::vector<std::vector<seal::Plaintext>> &W_diagonals,
    const seal::GaloisKeys &gal_keys, const seal::EncryptionParameters &params) {
    auto context = seal::SEALContext::Create(params);
    seal::Evaluator evaluator(context);
    if (tn < 1 || tm < 1 || tp < 1 || (long long)A_tiles.size() != (long long)tn * tm || (long long)B_tiles.size() != (long long)tm * tp)
        throw std::invalid_argument("tile vectors do not match the tile counts");
    if (dimension < 2 || (int)V_diagonals.size() < dimension - 1 || (int)W_diagonals.size() < dimension - 1)
        throw std::invalid_argument("dimension does not match the diagonal sets");
    const int d = dimension, K1 = d - 1;
    // the d entries of every tile; X in row-major tile order (entry (i*tm + l)*d + k = i*(tm d) + l d + k), Y in the
    // contraction's row order (entry (l d + k)*tp + j)
    std::unique_ptr<detail::Batch> X, Y;
    double s0[2] = {0, 0};
    auto operand = [&](const seal::Ciphertext &tile, const std::vector<seal::Plaintext> &first,
                       const std::vector<std::vector<seal::Plaintext>> &sets, std::unique_ptr<detail::Batch> &dst, int n,
                       int side, auto index) {
        seal::Ciphertext x0 = Linear_Transform_Plain(tile, first, gal_keys, params);
        detail::Batch xk = detail::shifted(x0, sets, K1, gal_keys, evaluator);
        evaluator.mod_switch_to_next_inplace(x0);
        if (!dst) {
            dst.reset(new detail::Batch(xk.e, n * d, 2, xk.limbs, xk.scale));
            s0[side] = x0.poly().scale;
        }
        if (xk.scale != dst->scale || x0.poly().scale != s0[side] || xk.limbs != dst->limbs)
            throw std::invalid_argument("scale mismatch");
        dst->put(index(0), x0.poly());
        for (int k = 1; k < d; k++)
            detail::check(ckks_copy(xk.e->ctx, dst->buf->p + (std::size_t)index(k) * dst->entry_words(),
                                    xk.buf->p + (std::size_t)(k - 1) * xk.entry_words(), xk.entry_words() * 8, nullptr));
    };
    for (int t = 0; t < tn * tm; t++)
        operand(A_tiles[t], U_sigma_diagonals, V_diagonals, X, tn * tm, 0, [&](int k) { return t * d + k; });
    for (int t = 0; t < tm * tp; t++) {
        const int l = t / tp, j = t % tp;
        operand(B_tiles[t], U_tau_diagonals, W_diagonals, Y, tm * tp, 1, [&](int k) { return (l * d + k) * tp + j; });
    }
    if (s0[0] * s0[1] != X->scale * Y->scale) throw std::invalid_argument("scale mismatch");
    detail::scale_ok(*X->e, X->scale * Y->scale, X->limbs);
    detail::Batch C(X->e, tn * tp, 3, X->limbs, X->scale * Y->scale);
    ckks_view va = X->view(), vb = Y->view(), vo = C.view();
    detail::check(ckks_multiply_sum_matrix(X->e->ctx, &va, &vb, tn, tm * d, tp, &vo, nullptr));
    std::vector<seal::Ciphertext> out(tn * tp);
    for (int o = 0; o < tn * tp; o++) C.get(o, out[o].poly());
    return out;
}

}  // namespace b200
