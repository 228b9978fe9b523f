/*
 * ckks_b200.h -- C ABI of the B200-native CKKS evaluation engine (libckks_b200.so).
 *
 * This is the drop-in boundary for the reference's hot path: the Microsoft SEAL
 * `Evaluator` surface that MarwanNour/SEAL-FYP-Logistic-Regression calls from its matrix /
 * vector helpers and its logistic-regression loop.  The reference reaches SEAL through
 * `#include "seal/seal.h"` (helper.h:4) and `target_link_libraries(<exe> SEAL::seal)`
 * (CMakeLists.txt:25-40); the C++ shim in
 * seal-fyp-logistic-regression_b200/include/seal/seal.h forwards every Evaluator member to
 * one of the entry points below.  Each entry point names the SEAL member it stands in for
 * and a reference call site.
 *
 * Conventions
 *   - plain C: opaque handles, raw device/host pointers, sizes, int status codes
 *     (0 = CKKS_OK); no C++ or torch types.  ckks_last_error() gives the message.
 *   - all polynomial data are uint64 words in device memory, always in NTT form
 *     (bit-reversed evaluation order) exactly as SEAL stores CKKS data.
 *   - a ckks_view describes a batch of ciphertexts (or plaintexts, size == 1):
 *       word address of (b, poly s, limb j, coeff c)
 *           = data + b*batch_stride + s*poly_stride + j*N + c
 *     limb j is modulo prime j of the context; the special prime is prime K-1.
 *     Keeping poly_stride fixed at the top level's L*N makes mod-switch a metadata change.
 *   - every call is asynchronous on the given CUDA stream (a cudaStream_t passed as
 *     void*; NULL = the legacy default stream) and never synchronises the device.
 *   - there is no CPU fallback: without a CUDA device every compute call fails.
 */
#ifndef CKKS_B200_H
#define CKKS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CKKS_OK 0
#define CKKS_ERR_INVALID 1   /* std::invalid_argument in SEAL */
#define CKKS_ERR_CUDA 2
#define CKKS_ERR_NOMEM 3
#define CKKS_ERR_LOGIC 4     /* std::logic_error in SEAL */

typedef struct ckks_ctx ckks_ctx;
typedef struct ckks_keyset ckks_keyset;
typedef void *ckks_stream;

typedef struct ckks_view {
    uint64_t *data;        /* device pointer */
    uint64_t batch_stride; /* words between consecutive ciphertexts */
    uint64_t poly_stride;  /* words between consecutive polynomials */
    int32_t batch;         /* number of ciphertexts */
    int32_t size;          /* polynomials per ciphertext (1 for a plaintext) */
    int32_t limbs;         /* active RNS limbs L (primes 0..L-1) */
    int32_t reserved;
} ckks_view;

const char *ckks_last_error(void);
const char *ckks_version(void);

/* ---- context: SEAL EncryptionParameters + SEALContext (logistic_regression_ckks.cpp:418-427,
 * linear_transformation2.cpp:229-239).  primes[K-1] is the special prime. */
int ckks_ctx_create(int log_n, int n_primes, const uint64_t *primes, int device, ckks_ctx **out);
void ckks_ctx_destroy(ckks_ctx *ctx);
int ckks_ctx_log_n(const ckks_ctx *ctx);
int ckks_ctx_n_primes(const ckks_ctx *ctx);
uint64_t ckks_ctx_prime(const ckks_ctx *ctx, int j);
/* the two divide-by-last-prime steps (SURVEY.md A.7 key-switch mod-down, A.8 rescale; both marked unconfirmed against a real
 * SEAL 3.4.5 build there): mode 0 = floor in both, 1 = round to nearest in both (default), 2 = key switch rounds / rescale
 * floors, 3 = key switch floors / rescale rounds.  tools/seal_replay.py on files written by real SEAL decides. */
int ckks_ctx_set_rounding(ckks_ctx *ctx, int mode);
/* cap (bytes) on the internal key-switch workspace; larger batches are processed in chunks */
int ckks_ctx_set_workspace_cap(ckks_ctx *ctx, size_t bytes);
/* number of concurrent half-/quarter-batch pipelines a rotate-and-sum chain is split into (1..4, default 2) */
int ckks_ctx_set_chain_lanes(ckks_ctx *ctx, int lanes);
/* pre-allocate the workspace for key switching `batch` ciphertexts at `limbs` (needed before
 * CUDA-graph capture, which forbids allocation) */
int ckks_ctx_reserve(ckks_ctx *ctx, int batch, int limbs);
/* number of kernels this context has launched since creation / since the last reset */
uint64_t ckks_ctx_launch_count(const ckks_ctx *ctx);
void ckks_ctx_reset_launch_count(ckks_ctx *ctx);

/* ---- memory / stream helpers for hosts that do not bring their own allocator.  Device buffers come
 * from the stream-ordered memory pool of the device (cudaMallocAsync / cudaFreeAsync, freed memory kept
 * for reuse).  The _async forms are ordered on the caller's stream `s`: use them (with the stream the buffer is
 * computed on) when that stream is a non-blocking one; the plain forms are the same calls on the default stream
 * (what the seal/seal.h shim does -- it issues every call on the default stream). */
int ckks_dev_alloc_async(ckks_ctx *ctx, size_t bytes, void **out, ckks_stream s);
int ckks_dev_free_async(ckks_ctx *ctx, void *p, ckks_stream s);
int ckks_dev_alloc(ckks_ctx *ctx, size_t bytes, void **out);
int ckks_dev_free(ckks_ctx *ctx, void *p);
int ckks_host_alloc(size_t bytes, void **out);   /* pinned */
int ckks_host_free(void *p);
int ckks_upload(ckks_ctx *ctx, void *dst_dev, const void *src_host, size_t bytes, ckks_stream s);
int ckks_download(ckks_ctx *ctx, void *dst_host, const void *src_dev, size_t bytes, ckks_stream s);
int ckks_copy(ckks_ctx *ctx, void *dst_dev, const void *src_dev, size_t bytes, ckks_stream s);   /* device to device */
int ckks_stream_sync(ckks_ctx *ctx, ckks_stream s);

/* ---- negacyclic NTT (SEAL util::ntt_negacyclic_harvey / inverse_...): n_polys x limbs limbs in
 * place, limb l uses prime first_prime + l; canonical output in [0,p). */
int ckks_ntt_forward(ckks_ctx *ctx, uint64_t *data, int n_polys, int limbs, int first_prime,
                     uint64_t poly_stride, ckks_stream s);
int ckks_ntt_inverse(ckks_ctx *ctx, uint64_t *data, int n_polys, int limbs, int first_prime,
                     uint64_t poly_stride, ckks_stream s);

/* ---- element-wise evaluator ops (out may alias an input when strides are identical) */
/* Evaluator::add / add_inplace (helper.h:247,484; logistic_regression_ckks.cpp:131) */
int ckks_add(ckks_ctx *ctx, const ckks_view *a, const ckks_view *b, const ckks_view *out, ckks_stream s);
/* Evaluator::sub (logistic_regression_ckks.cpp:288,341) */
int ckks_sub(ckks_ctx *ctx, const ckks_view *a, const ckks_view *b, const ckks_view *out, ckks_stream s);
/* Evaluator::negate_inplace (logistic_regression_ckks.cpp:342) */
int ckks_negate(ckks_ctx *ctx, const ckks_view *a, const ckks_view *out, ckks_stream s);
/* Evaluator::multiply / multiply_inplace, sizes (Sa,Sb) -> Sa+Sb-1 (helper.h:222,432;
 * matrix_multiplication.cpp:105,126; logistic_regression_ckks.cpp:184) */
int ckks_multiply(ckks_ctx *ctx, const ckks_view *a, const ckks_view *b, const ckks_view *out, ckks_stream s);
/* Evaluator::multiply_plain (helper.h:250,256,271).  pt->size == 1; pt->batch is 1 (broadcast)
 * or ct->batch */
int ckks_multiply_plain(ckks_ctx *ctx, const ckks_view *ct, const ckks_view *pt, const ckks_view *out,
                        ckks_stream s);
/* Evaluator::add_plain_inplace (logistic_regression_ckks.cpp:198) */
int ckks_add_plain(ckks_ctx *ctx, const ckks_view *ct, const ckks_view *pt, const ckks_view *out,
                   ckks_stream s);
/* Evaluator::add_many (helper.h:233,259,276,320): out (batch 1) = sum over the batch of `in`;
 * also the mod-q add that combines all-gathered partial ciphertexts across GPUs */
int ckks_add_many(ckks_ctx *ctx, const ckks_view *in, const ckks_view *out, ckks_stream s);
/* out[m] = sum_{g < groups} in[g * out->batch + m]  (mod q_j), for m < out->batch.
 * in->batch == groups * out->batch; same size / limbs; out must not alias in.  Bit-identical to
 * ckks_add_many applied to each group.  The reduce-scatter step of sharded workloads (NCCL's sum
 * is not modular). */
int ckks_add_many_grouped(ckks_ctx *ctx, const ckks_view *in, int groups, const ckks_view *out,
                          ckks_stream s);
/* Constant-coefficient sums, e.g. the baby-step sums of a polynomial in the Chebyshev basis:
 *   out[g * M + m] = sum_{i < terms} in[i * M + m] (.) const(coeffs[g * terms + i], scales[g * terms + i])
 *                    (+ const(const_coeffs[g], const_scales[g]) added to poly 0)
 * for g < groups, m < M = in->batch / terms; out->batch == groups * M.  const(c, s) is the constant
 * plaintext ckks_encode_scalar(c, s) writes (residues of nearbyint(c * s)), so the result is
 * bit-identical to multiply_plain by each such plaintext, add_many, add_plain.  Terms whose residues
 * are zero are skipped; every input word is read once for all groups.  const_coeffs / const_scales
 * may both be NULL (no constant).  CKKS_ERR_INVALID: bad shapes, terms or groups < 1,
 * (terms + 1) * limbs > 2048, out overlapping in, a scale <= 0 or a non-finite c * s. */
int ckks_multiply_const_sum(ckks_ctx *ctx, const ckks_view *in, int terms, int groups,
                            const double *coeffs, const double *scales, const double *const_coeffs,
                            const double *const_scales, const ckks_view *out, ckks_stream s);
/* SEAL's "result ciphertext is transparent" test: *flag_dev (device int32, one per batch entry)
 * is set to 1 when polys 1.. of the entry are all zero */
int ckks_is_transparent(ckks_ctx *ctx, const ckks_view *ct, int32_t *flag_dev, ckks_stream s);

/* ---- key switching.  Key layout (device): [digit i < K-1][component k < 2][limb j < K][N],
 * NTT form at the key level, as produced by SEAL KeyGenerator::generate_one_kswitch_key. */
size_t ckks_ksk_words(const ckks_ctx *ctx);
/* Evaluator::relinearize_inplace for size 3 -> 2 (helper.h:440,541;
 * logistic_regression_ckks.cpp:187).  out may alias in. */
int ckks_relinearize(ckks_ctx *ctx, const ckks_view *in, const uint64_t *rlk, const ckks_view *out,
                     ckks_stream s);
/* Evaluator::apply_galois: one Galois step of rotate_vector (permutation + key switch).
 * out must not alias in. */
int ckks_apply_galois(ckks_ctx *ctx, const ckks_view *in, uint64_t galois_elt, const uint64_t *gk,
                      const ckks_view *out, ckks_stream s);
/* util::steps_to_galois_elt; returns 0 for |steps| >= N/2 ("step count too large") */
uint64_t ckks_galois_elt_from_step(const ckks_ctx *ctx, int steps);

/* key registry = SEAL RelinKeys + GaloisKeys.  Registering a key captures its contents: the engine keeps a private
 * copy in the tile layout its inner-product kernels read fastest, and every entry point that is later given the
 * same pointer (ckks_relinearize, ckks_apply_galois, the keyset-based calls) uses that copy.  The caller's buffer
 * must stay allocated and unchanged while a keyset references it; register it again after changing it.
 * ckks_keyset_set_relin / _set_galois are set-up calls and SYNCHRONOUS with respect to every stream of the device (the
 * device is drained before the key is captured and the capture is complete on return): the key may have been produced on
 * any stream and may be used on any stream afterwards.  Rotation plans compiled before a key was replaced pick up the
 * new copy at their next ckks_rotate_plan. */
int ckks_keyset_create(ckks_ctx *ctx, ckks_keyset **out);
void ckks_keyset_destroy(ckks_keyset *ks);
int ckks_keyset_set_relin(ckks_keyset *ks, const uint64_t *rlk);
int ckks_keyset_set_galois(ckks_keyset *ks, uint64_t galois_elt, const uint64_t *gk);
int ckks_keyset_has_galois(const ckks_keyset *ks, uint64_t galois_elt);
/* Evaluator::rotate_vector (helper.h:222,244,255,318,350,471,475) including SEAL's NAF fallback
 * when the key for `steps` itself is absent.  out must not alias in.  `scratch` is a view like
 * `out` (distinct storage) used to ping-pong composite rotations; may be NULL when the step
 * maps to a single key. */
int ckks_rotate(ckks_ctx *ctx, const ckks_keyset *ks, const ckks_view *in, int steps, const ckks_view *out,
                const ckks_view *scratch, ckks_stream s);

/* Rotation plan: a fixed list of step counts, one per batch entry, compiled once into rounds so
 * that the d-1 different rotations of a Halevi-Shoup linear transform (helper.h:252-257) run as a
 * few batched key switches instead of d-1 dependent calls.  Each entry follows exactly SEAL's
 * rotate_vector for its step (direct key, else NAF terms least-significant first). */
typedef struct ckks_rotplan ckks_rotplan;
int ckks_rotplan_create(ckks_ctx *ctx, ckks_keyset *ks, const int *steps, int batch, ckks_rotplan **out);
void ckks_rotplan_destroy(ckks_rotplan *plan);
uint64_t ckks_rotplan_keyswitches(const ckks_rotplan *plan); /* total Galois key switches per run */
/* key switches per run when every entry rotates the same input ciphertext (ckks_rotate_plan with in->batch == 1): rotations
 * whose NAF chains begin with the same terms share those key switches; every output is still bit-identical to its own
 * rotate_vector call (Evaluator::rotate_vector, helper.h:252-257) */
uint64_t ckks_rotplan_keyswitches_shared(const ckks_rotplan *plan);
int ckks_rotplan_rounds(const ckks_rotplan *plan);
/* in->batch is the plan's batch, or 1 to rotate one ciphertext by every step of the plan;
 * out and scratch (needed when some entry has more than one NAF term) are plan-batch views */
int ckks_rotate_plan(ckks_ctx *ctx, const ckks_rotplan *plan, const ckks_view *in, const ckks_view *out,
                     const ckks_view *scratch, ckks_stream s);

/* SURVEY 8(f4), opt-in: every rotation of the plan applied to ONE ciphertext (in->batch == 1) with a SHARED digit
 * decomposition ("hoisting", Halevi-Shoup): the hot loop of Linear_Transform_Plain / _Cipher (helper.h:252-257) rotates the same
 * ct_new d-1 times.  Every non-zero step needs its own Galois key (KeyGenerator::galois_keys(steps); no NAF chains).  The
 * result decrypts to the same values as ckks_rotate_plan within key-switch noise but its polynomials are NOT bit-identical
 * to SEAL's (SEAL permutes before lifting the digits), so the reference-parity path never calls this. */
int ckks_rotate_plan_hoisted(ckks_ctx *ctx, const ckks_rotplan *plan, const ckks_view *in, const ckks_view *out, ckks_stream s);

/* The rotate-and-sum loop of cipher_dot_product (helper.h:472-476), `count` times:
 *     dup = rotate_vector(dup, steps);  acc = acc + dup
 * on a batch of independent ciphertexts.  `a` holds dup on entry; the rotation ping-pongs between
 * a and b (distinct storage, same shape), the add is fused into the key switch, and pairs of steps
 * are replayed from a cached CUDA graph.  *final_in_b tells where dup ended up.  The key for
 * `steps` itself must be present (the loop uses step 1). */
int ckks_rotate_sum_chain(ckks_ctx *ctx, const ckks_keyset *ks, const ckks_view *a, const ckks_view *b,
                          const ckks_view *acc, int steps, int count, int *final_in_b, ckks_stream s);

/* ---- fused multiply + add_many (bit-identical to the sequential ops: sums are modulo q)
 * out (batch 1) = sum_b cts[b] (.) pts[b]        -- multiply_plain + add_many, helper.h:250-259 */
int ckks_multiply_plain_sum(ckks_ctx *ctx, const ckks_view *cts, const ckks_view *pts, const ckks_view *out,
                            ckks_stream s);
/* out (batch 1, size 3) = sum_b a[b] x b[b] for size-2 inputs -- multiply + add_many,
 * helper.h:222-233, matrix_multiplication.cpp:123-129 */
int ckks_multiply_sum(ckks_ctx *ctx, const ckks_view *a, const ckks_view *b, const ckks_view *out, ckks_stream s);

/* ---- rescale / mod switch */
/* Evaluator::rescale_to_next_inplace (helper.h:441,543; matrix_multiplication.cpp:71-72):
 * out->limbs == in->limbs - 1.  out may alias in when strides are identical. */
int ckks_rescale(ckks_ctx *ctx, const ckks_view *in, const ckks_view *out, ckks_stream s);
/* Evaluator::mod_switch_to_next_inplace on ciphertexts / NTT-form plaintexts
 * (logistic_regression_ckks.cpp:177-182,227,286,295): copies limbs 0..out->limbs-1.  When in and
 * out share storage and strides this is a no-op (the caller only lowers `limbs`). */
int ckks_mod_switch_drop(ckks_ctx *ctx, const ckks_view *in, const ckks_view *out, ckks_stream s);

/* ---- CKKSEncoder on the device (tolerance-compared, see DESIGN.md) --------------------------------
 * CKKSEncoder::encode(const vector<double>&, double scale, Plaintext&)
 * (linear_transformation2.cpp:328-330, logistic_regression_ckks.cpp:225,305,590-611), batched: `values` is a
 * DEVICE array [out->batch][count] of doubles, count <= N/2 (the remaining slots are zero, as in
 * SEAL); `out` is a size-1 view (plaintext) with out->limbs limbs and receives NTT form. */
int ckks_encode(ckks_ctx *ctx, const double *values, int count, double scale, const ckks_view *out,
                ckks_stream s);
/* CKKSEncoder::encode(double value, double scale, Plaintext&) (logistic_regression_ckks.cpp:78,157,331):
 * the same constant in every slot, every batch entry of `out`. */
int ckks_encode_scalar(ckks_ctx *ctx, double value, double scale, const ckks_view *out, ckks_stream s);
/* CKKSEncoder::decode(const Plaintext&, vector<double>&) (linear_transformation2.cpp:384,
 * logistic_regression_ckks.cpp:365,499): `in` is a size-1 view at any level, `values` a DEVICE array
 * [in->batch][N/2] receiving the real parts of the slots.  `in` is not modified. */
int ckks_decode(ckks_ctx *ctx, const ckks_view *in, double scale, double *values, ckks_stream s);

/* ---- KeyGenerator / Encryptor randomness on the device (tolerance-compared paths only) ------------
 * util::sample_poly_ternary / sample_poly_normal (sigma 3.2, clipped at 6 sigma) / sample_poly_uniform as
 * used by KeyGenerator (keygen.secret_key(), public_key(), relin_keys(), galois_keys():
 * linear_transformation2.cpp:236-239) and Encryptor::encrypt (:347-349).  `out` is a size-1 view of
 * out->batch polynomials over limbs [0, out->limbs); ternary and normal polynomials hold the same small
 * integer in every limb and are returned in NTT form, uniform polynomials are independent per limb.
 * The generator is ChaCha20 (RFC 8439 block function) in counter mode under a 256-bit key: a CSPRNG like SEAL 3.4.5's
 * own (Blake2-based) default generator.  (`key`, `stream_id`) must not repeat between calls.
 *   ckks_sample_keyed  -- `key` = 32 bytes from a cryptographic source (the seal/seal.h shim and client.py read the
 *                         operating system's CSPRNG): the entry point for real keys and encryptions.
 *   ckks_sample        -- reproducible variant for tests and benchmarks: the 64-bit `seed` is expanded into the key, so
 *                         the stream has at most 64 bits of entropy.  NOT for real keys. */
#define CKKS_SAMPLE_TERNARY 0
#define CKKS_SAMPLE_NORMAL 1
#define CKKS_SAMPLE_UNIFORM 2
int ckks_sample_keyed(ckks_ctx *ctx, int kind, const uint8_t key[32], uint64_t stream_id, const ckks_view *out, ckks_stream s);
int ckks_sample(ckks_ctx *ctx, int kind, uint64_t seed, uint64_t stream_id, const ckks_view *out, ckks_stream s);

#ifdef __cplusplus
}
#endif
#endif
