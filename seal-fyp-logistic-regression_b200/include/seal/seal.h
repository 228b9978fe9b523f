// seal/seal.h -- source-compatible shim of the Microsoft SEAL surface that
// MarwanNour/SEAL-FYP-Logistic-Regression uses on its CKKS hot path, backed by the B200 engine
// (libckks_b200.so, include/ckks_b200.h).  The reference reaches SEAL through
// `#include "seal/seal.h"` + `using namespace seal;` (helper.h:4-7); put this directory on the
// include path and link libckks_b200.so instead of SEAL::seal (INTEGRATION.md).
//
// It accepts the UNION of the two API spellings found in the reference (SURVEY.md 2.3):
//   3.4/3.5: scheme_type::CKKS, SEALContext::Create(parms) -> shared_ptr, keygen.public_key(),
//            keygen.relin_keys(), keygen.galois_keys()
//   3.6    : scheme_type::ckks, SEALContext context(parms), keygen.create_public_key(pk), ...
//
// Ownership / semantics follow SEAL: value types, inputs by const&, destination overwritten,
// std::invalid_argument / std::logic_error on misuse.  Ciphertext / Plaintext / key data live in
// device memory (copy-on-write, so the reference's by-value parameter passing stays cheap); every
// Evaluator member enqueues kernels on one CUDA stream and returns; decrypt / decode synchronise.
// Ring arithmetic is always done by the GPU engine: there is no CPU fallback in this shim.  The
// host only samples randomness and does the floating-point canonical embedding.
//
// Not provided (outside the reference's CKKS path): BFV evaluation, IntegerEncoder, BatchEncoder,
// serialization, ciphertext sizes above 3.
#pragma once

#include <algorithm>
#include <array>
#include <cmath>
#include <complex>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <istream>
#include <map>
#include <memory>
#include <mutex>
#include <ostream>
#include <random>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <vector>

#include "ckks_b200.h"

namespace seal {

using parms_id_type = std::array<std::uint64_t, 4>;
static const parms_id_type parms_id_zero = {0, 0, 0, 0};

enum class scheme_type : std::uint8_t { none = 0, BFV = 1, bfv = 1, CKKS = 2, ckks = 2 };
enum class sec_level_type : int { none = 0, tc128 = 128, tc192 = 192, tc256 = 256 };

class MemoryPoolHandle {};
struct MemoryManager {
    static MemoryPoolHandle GetPool() { return MemoryPoolHandle(); }
};

namespace detail {

inline void check(int rc) {
    if (rc == CKKS_OK) return;
    std::string msg = ckks_last_error();
    if (rc == CKKS_ERR_INVALID) throw std::invalid_argument(msg);
    if (rc == CKKS_ERR_LOGIC) throw std::logic_error(msg);
    if (rc == CKKS_ERR_NOMEM) throw std::bad_alloc();
    throw std::runtime_error(msg);
}

typedef unsigned __int128 u128;
inline std::uint64_t mulmod(std::uint64_t a, std::uint64_t b, std::uint64_t p) { return (std::uint64_t)((u128)a * b % p); }
inline std::uint64_t powmod(std::uint64_t a, std::uint64_t e, std::uint64_t p) {
    std::uint64_t r = 1;
    a %= p;
    for (; e; e >>= 1, a = mulmod(a, a, p))
        if (e & 1) r = mulmod(r, a, p);
    return r;
}
inline bool is_prime(std::uint64_t n) {
    if (n < 2) return false;
    for (std::uint64_t w : {2ull, 3ull, 5ull, 7ull, 11ull, 13ull, 17ull, 19ull, 23ull, 29ull, 31ull, 37ull}) {
        if (n % w == 0) return n == w;
    }
    std::uint64_t d = n - 1;
    int r = 0;
    while (!(d & 1)) d >>= 1, ++r;
    for (std::uint64_t w : {2ull, 3ull, 5ull, 7ull, 11ull, 13ull, 17ull, 19ull, 23ull, 29ull, 31ull, 37ull}) {
        std::uint64_t x = powmod(w, d, n);
        if (x == 1 || x == n - 1) continue;
        bool comp = true;
        for (int i = 1; i < r && comp; ++i) {
            x = mulmod(x, x, n);
            if (x == n - 1) comp = false;
        }
        if (comp) return false;
    }
    return true;
}
inline int bit_length(std::uint64_t v) {
    int b = 0;
    while (v) ++b, v >>= 1;
    return b;
}
inline std::uint32_t bitrev(std::uint32_t v, int bits) {
    std::uint32_t r = 0;
    for (int i = 0; i < bits; ++i, v >>= 1) r = (r << 1) | (v & 1);
    return r;
}

}  // namespace detail

// ------------------------------------------------------------------------------------ moduli
class SmallModulus {
public:
    SmallModulus(std::uint64_t v = 0) : value_(v) {}
    std::uint64_t value() const { return value_; }
    int bit_count() const { return detail::bit_length(value_); }
    bool is_zero() const { return value_ == 0; }
    bool operator==(const SmallModulus &o) const { return value_ == o.value_; }

private:
    std::uint64_t value_;
};
using Modulus = SmallModulus;

class CoeffModulus {
public:
    // SEAL CoeffModulus::MaxBitCount (128-bit classical security)
    static int MaxBitCount(std::size_t n, sec_level_type = sec_level_type::tc128) {
        switch (n) {
        case 1024: return 27;
        case 2048: return 54;
        case 4096: return 109;
        case 8192: return 218;
        case 16384: return 438;
        case 32768: return 881;
        default: return 0;
        }
    }
    // SEAL CoeffModulus::Create: per bit size the c largest primes = 1 mod 2N below 2^bits; the
    // request is served in order from the smallest of each size (SURVEY.md A.1)
    static std::vector<SmallModulus> Create(std::size_t n, std::vector<int> bits) {
        std::map<int, std::vector<std::uint64_t>> pool;
        for (int b : bits) {
            if (b < 2 || b > 60) throw std::invalid_argument("bit_sizes is invalid");
            pool[b];
        }
        for (auto &kv : pool) {
            std::size_t need = (std::size_t)std::count(bits.begin(), bits.end(), kv.first);
            std::uint64_t step = 2 * (std::uint64_t)n, v = (1ull << kv.first) - step + 1;
            while (kv.second.size() < need && v > (1ull << (kv.first - 1))) {
                if (detail::is_prime(v)) kv.second.push_back(v);
                v -= step;
            }
            if (kv.second.size() < need) throw std::logic_error("failed to find enough qualifying primes");
        }
        std::vector<SmallModulus> out;
        for (int b : bits) {
            out.emplace_back(pool[b].back());
            pool[b].pop_back();
        }
        return out;
    }
    // SEAL default_coeff_modulus_128
    static std::vector<SmallModulus> BFVDefault(std::size_t n, sec_level_type = sec_level_type::tc128) {
        static const std::map<std::size_t, std::vector<std::uint64_t>> t = {
            {4096, {0xffffee001, 0xffffc4001, 0x1ffffe0001}},
            {8192, {0x7fffffd8001, 0x7fffffc8001, 0xfffffffc001, 0xffffff6c001, 0xfffffebc001}},
            {16384, {0xfffffffd8001, 0xfffffffa0001, 0xfffffff00001, 0x1fffffff68001, 0x1fffffff50001, 0x1ffffffee8001,
                     0x1ffffffea0001, 0x1ffffffe88001, 0x1ffffffe48001}},
            {32768, {0x7fffffffe90001, 0x7fffffffbf0001, 0x7fffffffbd0001, 0x7fffffffba0001, 0x7fffffffaa0001,
                     0x7fffffffa50001, 0x7fffffff9f0001, 0x7fffffff7e0001, 0x7fffffff770001, 0x7fffffff380001,
                     0x7fffffff330001, 0x7fffffff2d0001, 0x7fffffff170001, 0x7fffffff150001, 0x7ffffffef00001,
                     0xfffffffff70001}}};
        auto it = t.find(n);
        if (it == t.end()) throw std::invalid_argument("poly_modulus_degree is invalid");
        return std::vector<SmallModulus>(it->second.begin(), it->second.end());
    }
};

class EncryptionParameters {
public:
    EncryptionParameters(scheme_type s = scheme_type::none) : scheme_(s) {}
    void set_poly_modulus_degree(std::size_t n) { n_ = n; }
    void set_coeff_modulus(const std::vector<SmallModulus> &m) { coeff_ = m; }
    void set_plain_modulus(const SmallModulus &m) { plain_ = m; }
    void set_plain_modulus(std::uint64_t m) { plain_ = SmallModulus(m); }
    scheme_type scheme() const { return scheme_; }
    std::size_t poly_modulus_degree() const { return n_; }
    const std::vector<SmallModulus> &coeff_modulus() const { return coeff_; }
    const SmallModulus &plain_modulus() const { return plain_; }
    // SEAL 3.4.x binary stream (uncompressed): see the serialization block at the end of this header
    inline std::streamoff save(std::ostream &stream) const;
    inline void load(std::istream &stream);

private:
    scheme_type scheme_;
    std::size_t n_ = 0;
    std::vector<SmallModulus> coeff_;
    SmallModulus plain_;
};

// ------------------------------------------------------------------------------------ engine glue
namespace detail {

// one GPU engine context per distinct parameter set, shared by every SEALContext built from it
// (the reference rebuilds SEALContext inside helpers on every call, helper.h:239-240)
struct Engine {
    ckks_ctx *ctx = nullptr;
    int log_n = 0, K = 0;
    std::size_t n = 0;
    std::vector<std::uint64_t> primes;
    std::map<std::size_t, std::vector<std::uint64_t *>> pool;   // free device buffers by word count
    std::mutex mu;
    // SEAL is synchronous: a caller timing evaluator calls with a host clock (benchmark.cpp) sees only the
    // enqueue cost of this asynchronous engine.  CKKS_SHIM_SYNC=1 makes every evaluator call wait for its
    // result, so such timings measure completed work.
    bool sync_each = std::getenv("CKKS_SHIM_SYNC") != nullptr;
    void settle() {
        if (sync_each) ckks_stream_sync(ctx, nullptr);
    }
    ~Engine() {
        for (auto &kv : pool)
            for (auto p : kv.second) ckks_dev_free(ctx, p);
        if (ctx) ckks_ctx_destroy(ctx);
    }
    std::uint64_t *alloc(std::size_t words) {
        {
            std::lock_guard<std::mutex> g(mu);
            auto &v = pool[words];
            if (!v.empty()) {
                auto p = v.back();
                v.pop_back();
                return p;
            }
        }
        void *p = nullptr;
        check(ckks_dev_alloc(ctx, words * 8, &p));
        return (std::uint64_t *)p;
    }
    void release(std::uint64_t *p, std::size_t words) {
        std::lock_guard<std::mutex> g(mu);
        pool[words].push_back(p);   // all work is ordered on one stream, so reuse is safe
    }
    static std::shared_ptr<Engine> get(std::size_t n, const std::vector<std::uint64_t> &primes) {
        static std::mutex m;
        static std::map<std::pair<std::size_t, std::vector<std::uint64_t>>, std::weak_ptr<Engine>> reg;
        std::lock_guard<std::mutex> g(m);
        auto key = std::make_pair(n, primes);
        if (auto sp = reg[key].lock()) return sp;
        auto e = std::make_shared<Engine>();
        e->n = n;
        e->log_n = bit_length(n) - 1;
        e->K = (int)primes.size();
        e->primes = primes;
        check(ckks_ctx_create(e->log_n, e->K, primes.data(), 0, &e->ctx));
        reg[key] = e;
        return e;
    }
};

struct DevBuf {
    std::shared_ptr<Engine> eng;
    std::uint64_t *p = nullptr;
    std::size_t words = 0;
    DevBuf(std::shared_ptr<Engine> e, std::size_t w) : eng(std::move(e)), p(eng->alloc(w)), words(w) {}
    ~DevBuf() { eng->release(p, words); }
    DevBuf(const DevBuf &) = delete;
};
using BufPtr = std::shared_ptr<DevBuf>;

inline parms_id_type make_id(const Engine &e, int limbs) {
    std::uint64_t h = 1469598103934665603ull;
    for (int j = 0; j < limbs; j++) h = (h ^ e.primes[j]) * 1099511628211ull;
    return {(std::uint64_t)limbs, (std::uint64_t)e.n, h, 0x434b4b53ull};
}

// polynomial container shared by Plaintext and Ciphertext: [size][cap][N] device words
struct Poly {
    std::shared_ptr<Engine> eng;
    BufPtr buf;
    int size = 0, limbs = 0, cap = 0;
    double scale = 1.0;
    void allocate(std::shared_ptr<Engine> e, int size_, int limbs_) {
        eng = std::move(e);
        size = size_;
        limbs = cap = limbs_;
        buf = std::make_shared<DevBuf>(eng, (std::size_t)size * cap * eng->n);
    }
    ckks_view view() const {
        ckks_view v;
        v.data = buf->p;
        v.batch_stride = (std::uint64_t)size * cap * eng->n;
        v.poly_stride = (std::uint64_t)cap * eng->n;
        v.batch = 1;
        v.size = size;
        v.limbs = limbs;
        v.reserved = 0;
        return v;
    }
    void make_unique() {   // copy-on-write before an in-place update
        if (buf && buf.use_count() > 1) {
            auto nb = std::make_shared<DevBuf>(eng, buf->words);
            check(ckks_copy(eng->ctx, nb->p, buf->p, buf->words * 8, nullptr));
            buf = nb;
        }
    }
    parms_id_type parms_id() const { return eng ? make_id(*eng, limbs) : parms_id_zero; }
};

}  // namespace detail

// ------------------------------------------------------------------------------------ context
class SEALContext {
public:
    class ContextData {
    public:
        const EncryptionParameters &parms() const { return parms_; }
        const parms_id_type &parms_id() const { return id_; }
        std::size_t chain_index() const { return chain_index_; }
        int total_coeff_modulus_bit_count() const { return total_bits_; }
        std::shared_ptr<const ContextData> next_context_data() const { return next_; }
        std::shared_ptr<const ContextData> prev_context_data() const { return prev_.lock(); }

    private:
        friend class SEALContext;
        EncryptionParameters parms_;
        parms_id_type id_;
        std::size_t chain_index_ = 0;
        int total_bits_ = 0;
        std::shared_ptr<const ContextData> next_;
        std::weak_ptr<const ContextData> prev_;
    };

    explicit SEALContext(const EncryptionParameters &parms, bool = true, sec_level_type = sec_level_type::tc128) {
        if (parms.scheme() != scheme_type::CKKS)
            throw std::invalid_argument("this engine implements the CKKS path only");
        std::vector<std::uint64_t> primes;
        for (auto &m : parms.coeff_modulus()) primes.push_back(m.value());
        eng_ = detail::Engine::get(parms.poly_modulus_degree(), primes);
        int K = eng_->K;
        std::shared_ptr<ContextData> prev;
        for (int limbs = K; limbs >= 1; --limbs) {   // key level, then the data levels
            auto cd = std::make_shared<ContextData>();
            EncryptionParameters p(parms.scheme());
            p.set_poly_modulus_degree(parms.poly_modulus_degree());
            p.set_coeff_modulus(std::vector<SmallModulus>(parms.coeff_modulus().begin(), parms.coeff_modulus().begin() + limbs));
            cd->parms_ = p;
            cd->id_ = detail::make_id(*eng_, limbs);
            cd->chain_index_ = (std::size_t)(limbs == K ? K - 1 : limbs - 1);
            int bits = 0;
            // bit count of the product of the primes (SEAL: total_coeff_modulus_bit_count)
            long double lg = 0;
            for (int j = 0; j < limbs; j++) lg += std::log2((long double)eng_->primes[j]);
            bits = (int)std::floor(lg) + 1;
            cd->total_bits_ = bits;
            if (prev) {
                prev->next_ = cd;
                cd->prev_ = prev;
            }
            data_[limbs] = cd;
            prev = cd;
        }
    }
    static std::shared_ptr<SEALContext> Create(const EncryptionParameters &parms, bool expand = true,
                                               sec_level_type sec = sec_level_type::tc128) {
        return std::make_shared<SEALContext>(parms, expand, sec);
    }
    std::shared_ptr<const ContextData> get_context_data(const parms_id_type &id) const {
        auto it = data_.find((int)id[0]);
        if (it == data_.end() || it->second->id_ != id) return nullptr;
        return it->second;
    }
    std::shared_ptr<const ContextData> key_context_data() const { return data_.at(eng_->K); }
    std::shared_ptr<const ContextData> first_context_data() const { return data_.at(eng_->K - 1); }
    std::shared_ptr<const ContextData> last_context_data() const { return data_.at(1); }
    const parms_id_type &key_parms_id() const { return key_context_data()->parms_id(); }
    const parms_id_type &first_parms_id() const { return first_context_data()->parms_id(); }
    const parms_id_type &last_parms_id() const { return last_context_data()->parms_id(); }
    bool parameters_set() const { return true; }
    const std::shared_ptr<detail::Engine> &engine() const { return eng_; }

private:
    std::shared_ptr<detail::Engine> eng_;
    std::map<int, std::shared_ptr<ContextData>> data_;
};

namespace detail {
inline std::shared_ptr<Engine> engine_of(const std::shared_ptr<SEALContext> &c) {
    if (!c) throw std::invalid_argument("invalid context");
    return c->engine();
}
inline std::shared_ptr<Engine> engine_of(const SEALContext &c) { return c.engine(); }
}  // namespace detail

// ------------------------------------------------------------------------------------ data objects
class Plaintext {
public:
    Plaintext() = default;
    double &scale() { return p_.scale; }
    const double &scale() const { return p_.scale; }
    parms_id_type parms_id() const { return p_.parms_id(); }
    bool is_ntt_form() const { return true; }
    std::size_t coeff_count() const { return p_.eng ? (std::size_t)p_.limbs * p_.eng->n : 0; }
    inline std::streamoff save(std::ostream &stream) const;
    template <class Ctx>
    inline void load(const Ctx &context, std::istream &stream);
    detail::Poly &poly() { return p_; }
    const detail::Poly &poly() const { return p_; }

private:
    detail::Poly p_;
};

class Ciphertext {
public:
    Ciphertext() = default;
    double &scale() { return p_.scale; }
    const double &scale() const { return p_.scale; }
    parms_id_type parms_id() const { return p_.parms_id(); }
    std::size_t size() const { return (std::size_t)p_.size; }
    std::size_t coeff_mod_count() const { return (std::size_t)p_.limbs; }
    std::size_t poly_modulus_degree() const { return p_.eng ? p_.eng->n : 0; }
    bool is_ntt_form() const { return true; }
    inline std::streamoff save(std::ostream &stream) const;
    template <class Ctx>
    inline void load(const Ctx &context, std::istream &stream);
    detail::Poly &poly() { return p_; }
    const detail::Poly &poly() const { return p_; }

private:
    detail::Poly p_;
};

class SecretKey {
public:
    detail::BufPtr buf;   // [K][N], NTT form
    inline std::streamoff save(std::ostream &stream) const;
};
class PublicKey {
public:
    detail::BufPtr buf;   // [2][K][N]
    inline std::streamoff save(std::ostream &stream) const;
};

class KSwitchKeys {
public:
    struct Shared {
        std::shared_ptr<detail::Engine> eng;
        ckks_keyset *ks = nullptr;
        std::map<std::uint64_t, detail::BufPtr> keys;   // Galois element (or 0 for relin) -> key
        ~Shared() {
            if (ks) ckks_keyset_destroy(ks);
        }
    };
    std::shared_ptr<Shared> s;   // copies of RelinKeys / GaloisKeys share device storage
    std::size_t size() const { return s ? s->keys.size() : 0; }

protected:
    inline std::streamoff save_impl(std::ostream &stream, bool galois) const;
    inline void load_impl(std::shared_ptr<detail::Engine> eng, std::istream &stream, bool galois);
};
class RelinKeys : public KSwitchKeys {
public:
    std::streamoff save(std::ostream &stream) const { return save_impl(stream, false); }
    template <class Ctx>
    inline void load(const Ctx &context, std::istream &stream);
};
class GaloisKeys : public KSwitchKeys {
public:
    std::streamoff save(std::ostream &stream) const { return save_impl(stream, true); }
    template <class Ctx>
    inline void load(const Ctx &context, std::istream &stream);
    bool has_key(std::uint64_t galois_elt) const { return s && s->keys.count(galois_elt); }
    static std::size_t get_index(std::uint64_t galois_elt) { return (std::size_t)((galois_elt - 1) >> 1); }
};

// ------------------------------------------------------------------------------------ host-side ring helpers
namespace detail {

// thin wrappers: every ring operation goes through the GPU engine
// 256-bit generator key from the operating system's entropy source (std::random_device reads getrandom / /dev/urandom /
// RDRAND on the supported platforms): the device-side sampler is ChaCha20 in counter mode under this key
// (ckks_sample_keyed), i.e. a CSPRNG like SEAL 3.4.5's own default generator.
struct SampleKey256 {
    std::uint8_t b[32];
};
inline SampleKey256 fresh_key() {
    std::random_device rd;
    SampleKey256 k;
    for (int i = 0; i < 8; i++) {
        const std::uint32_t w = rd();
        std::memcpy(k.b + 4 * i, &w, 4);
    }
    return k;
}
inline void secure_zero(void *p, std::size_t bytes) {
    volatile unsigned char *q = static_cast<volatile unsigned char *>(p);
    while (bytes--) *q++ = 0;
}

struct Ring {
    std::shared_ptr<Engine> e;
    SampleKey256 key_;
    std::uint64_t stream_ = 0;
    explicit Ring(std::shared_ptr<Engine> eng, const SampleKey256 &key) : e(std::move(eng)), key_(key) {}
    ~Ring() { secure_zero(key_.b, sizeof(key_.b)); }

    ckks_view view(std::uint64_t *p, int batch, int size, int limbs) const {
        ckks_view v;
        v.data = p;
        v.poly_stride = (std::uint64_t)limbs * e->n;
        v.batch_stride = (std::uint64_t)size * limbs * e->n;
        v.batch = batch;
        v.size = size;
        v.limbs = limbs;
        v.reserved = 0;
        return v;
    }
    // Sampling runs on the device (ckks_sample_keyed): ChaCha20 in counter mode keyed by this object's
    // 256-bit key, one stream id (nonce) per call.  count polynomials over primes [0, limbs): device [count][limbs][N];
    // ternary and normal polynomials hold the same small integer in every limb and come back in NTT form.
    BufPtr draw(int kind, int count, int limbs) {
        auto b = std::make_shared<DevBuf>(e, (std::size_t)count * limbs * e->n);
        ckks_view v = view(b->p, count, 1, limbs);
        check(ckks_sample_keyed(e->ctx, kind, key_.b, ++stream_, &v, nullptr));
        return b;
    }
    BufPtr ternary_ntt(int count, int limbs) { return draw(CKKS_SAMPLE_TERNARY, count, limbs); }
    BufPtr errors_ntt(int count, int limbs) { return draw(CKKS_SAMPLE_NORMAL, count, limbs); }   // sigma 3.2, clipped at 6 sigma
    BufPtr uniform(int count, int limbs) { return draw(CKKS_SAMPLE_UNIFORM, count, limbs); }
    // count x (-(a s + e), a) over primes [0, limbs): device [count][2][limbs][N]
    BufPtr enc_zero_sym(int count, const std::uint64_t *sk, int limbs) {
        std::size_t n = e->n, pw = (std::size_t)limbs * n;
        auto a = uniform(count, limbs);
        auto err = errors_ntt(count, limbs);
        auto out = std::make_shared<DevBuf>(e, (std::size_t)count * 2 * pw);
        auto tmp = std::make_shared<DevBuf>(e, (std::size_t)count * pw);
        ckks_view va = view(a->p, count, 1, limbs), vs = view(const_cast<std::uint64_t *>(sk), 1, 1, limbs);
        vs.poly_stride = vs.batch_stride = (std::uint64_t)e->K * n;   // secret key rows are K limbs apart
        ckks_view vt = view(tmp->p, count, 1, limbs), ve = view(err->p, count, 1, limbs);
        check(ckks_multiply_plain(e->ctx, &va, &vs, &vt, nullptr));
        check(ckks_add(e->ctx, &vt, &ve, &vt, nullptr));
        check(ckks_negate(e->ctx, &vt, &vt, nullptr));
        for (int c = 0; c < count; c++) {
            check(ckks_copy(e->ctx, out->p + ((std::size_t)c * 2) * pw, tmp->p + (std::size_t)c * pw, pw * 8, nullptr));
            check(ckks_copy(e->ctx, out->p + ((std::size_t)c * 2 + 1) * pw, a->p + (std::size_t)c * pw, pw * 8, nullptr));
        }
        return out;
    }
};

}  // namespace detail

// ------------------------------------------------------------------------------------ KeyGenerator
class KeyGenerator {
public:
    template <class Ctx>
    explicit KeyGenerator(const Ctx &context) : ring_(detail::engine_of(context), detail::fresh_key()) {
        auto &e = ring_.e;
        sk_.buf = ring_.ternary_ntt(1, e->K);
    }
    const SecretKey &secret_key() const { return sk_; }
    PublicKey public_key() {
        PublicKey pk;
        pk.buf = ring_.enc_zero_sym(1, sk_.buf->p, ring_.e->K);
        return pk;
    }
    void create_public_key(PublicKey &pk) { pk = public_key(); }

    RelinKeys relin_keys() {
        auto &e = ring_.e;
        std::size_t kw = (std::size_t)e->K * e->n;
        auto s2 = std::make_shared<detail::DevBuf>(e, kw);
        ckks_view vs = ring_.view(sk_.buf->p, 1, 1, e->K), vo = ring_.view(s2->p, 1, 1, e->K);
        detail::check(ckks_multiply_plain(e->ctx, &vs, &vs, &vo, nullptr));
        RelinKeys rk;
        rk.s = make_shared_keys();
        rk.s->keys[0] = kswitch_key(s2->p);
        detail::check(ckks_keyset_set_relin(rk.s->ks, rk.s->keys[0]->p));
        return rk;
    }
    RelinKeys relin_keys_local() { return relin_keys(); }
    void create_relin_keys(RelinKeys &rk) { rk = relin_keys(); }

    // default: steps +-2^i and the conjugation (SEAL KeyGenerator::galois_keys())
    GaloisKeys galois_keys() {
        auto &e = ring_.e;
        std::vector<std::uint64_t> elts = {2 * (std::uint64_t)e->n - 1};
        for (int i = 0; i < e->log_n - 1; i++) {
            elts.push_back(ckks_galois_elt_from_step(e->ctx, 1 << i));
            elts.push_back(ckks_galois_elt_from_step(e->ctx, -(1 << i)));
        }
        return galois_keys(elts);
    }
    GaloisKeys galois_keys(const std::vector<int> &steps) {
        std::vector<std::uint64_t> elts;
        for (int s : steps) {
            std::uint64_t g = ckks_galois_elt_from_step(ring_.e->ctx, s);
            if (!g) throw std::invalid_argument("step count too large");
            elts.push_back(g);
        }
        return galois_keys(elts);
    }
    GaloisKeys galois_keys(const std::vector<std::uint64_t> &elts) {
        auto &e = ring_.e;
        GaloisKeys gk;
        gk.s = make_shared_keys();
        std::size_t n = e->n;
        std::vector<std::uint64_t> hsk((std::size_t)e->K * n), perm_sk(hsk.size());
        // the host copies of the secret key are wiped on every exit path
        struct Wipe {
            std::vector<std::uint64_t> &a, &b;
            ~Wipe() {
                detail::secure_zero(a.data(), a.size() * 8);
                detail::secure_zero(b.data(), b.size() * 8);
            }
        } wipe{hsk, perm_sk};
        detail::check(ckks_download(e->ctx, hsk.data(), sk_.buf->p, hsk.size() * 8, nullptr));
        detail::check(ckks_stream_sync(e->ctx, nullptr));
        for (std::uint64_t g : elts) {
            if (gk.s->keys.count(g)) continue;
            // sigma_g(s) in NTT form is a permutation of s (SEAL apply_galois_ntt)
            for (std::size_t i = 0; i < n; i++) {
                std::uint64_t ex = (g * (2ull * detail::bitrev((std::uint32_t)i, e->log_n) + 1)) & (2 * n - 1);
                std::size_t src = detail::bitrev((std::uint32_t)((ex - 1) >> 1), e->log_n);
                for (int j = 0; j < e->K; j++) perm_sk[(std::size_t)j * n + i] = hsk[(std::size_t)j * n + src];
            }
            auto d = std::make_shared<detail::DevBuf>(e, perm_sk.size());
            detail::check(ckks_upload(e->ctx, d->p, perm_sk.data(), perm_sk.size() * 8, nullptr));
            detail::check(ckks_stream_sync(e->ctx, nullptr));
            gk.s->keys[g] = kswitch_key(d->p);
            detail::check(ckks_keyset_set_galois(gk.s->ks, g, gk.s->keys[g]->p));
        }
        return gk;
    }
    void create_galois_keys(GaloisKeys &gk) { gk = galois_keys(); }
    void create_galois_keys(const std::vector<int> &steps, GaloisKeys &gk) { gk = galois_keys(steps); }

private:
    std::shared_ptr<KSwitchKeys::Shared> make_shared_keys() {
        auto s = std::make_shared<KSwitchKeys::Shared>();
        s->eng = ring_.e;
        detail::check(ckks_keyset_create(ring_.e->ctx, &s->ks));
        return s;
    }
    // SEAL generate_one_kswitch_key (SURVEY.md A.5): digit i = Enc(0) with (P mod q_i) new_key in limb i
    detail::BufPtr kswitch_key(const std::uint64_t *new_key) {
        auto &e = ring_.e;
        int K = e->K;
        std::size_t n = e->n, kw = (std::size_t)K * n;
        auto key = ring_.enc_zero_sym(K - 1, sk_.buf->p, K);   // [K-1][2][K][N]
        std::vector<std::uint64_t> fac(kw);
        for (int j = 0; j < K; j++)
            for (std::size_t q = 0; q < n; q++) fac[(std::size_t)j * n + q] = e->primes[K - 1] % e->primes[j];
        auto dfac = std::make_shared<detail::DevBuf>(e, kw), scaled = std::make_shared<detail::DevBuf>(e, kw);
        detail::check(ckks_upload(e->ctx, dfac->p, fac.data(), kw * 8, nullptr));
        detail::check(ckks_stream_sync(e->ctx, nullptr));
        ckks_view vn = ring_.view(const_cast<std::uint64_t *>(new_key), 1, 1, K), vf = ring_.view(dfac->p, 1, 1, K),
                  vsc = ring_.view(scaled->p, 1, 1, K);
        detail::check(ckks_multiply_plain(e->ctx, &vn, &vf, &vsc, nullptr));
        // add limb i of `scaled` into limb i of component 0 of digit i: done as a full-width add of a
        // one-hot limb selection, i.e. K-1 single-limb adds expressed through per-limb views
        for (int i = 0; i < K - 1; i++) {
            // a (i+1)-limb view whose only touched limb is i would still add limbs < i, so use the NTT-free
            // route: copy limb i of scaled into a zeroed K-limb poly and add it
            auto z = std::make_shared<detail::DevBuf>(e, kw);
            std::vector<std::uint64_t> zeros(kw, 0);
            detail::check(ckks_upload(e->ctx, z->p, zeros.data(), kw * 8, nullptr));
            detail::check(ckks_stream_sync(e->ctx, nullptr));
            detail::check(ckks_copy(e->ctx, z->p + (std::size_t)i * n, scaled->p + (std::size_t)i * n, n * 8, nullptr));
            std::uint64_t *c0 = key->p + ((std::size_t)i * 2) * kw;
            ckks_view vc = ring_.view(c0, 1, 1, K), vz = ring_.view(z->p, 1, 1, K);
            detail::check(ckks_add(e->ctx, &vc, &vz, &vc, nullptr));
        }
        return key;
    }
    detail::Ring ring_;
    SecretKey sk_;
};

// ------------------------------------------------------------------------------------ CKKSEncoder
class CKKSEncoder {
public:
    template <class Ctx>
    explicit CKKSEncoder(const Ctx &context) : e_(detail::engine_of(context)) {}
    std::size_t slot_count() const { return e_->n / 2; }

    void encode(const std::vector<double> &values, parms_id_type id, double scale, Plaintext &dst, MemoryPoolHandle = {}) {
        encode_impl(values, (int)id[0], scale, dst);
    }
    void encode(const std::vector<double> &values, double scale, Plaintext &dst, MemoryPoolHandle = {}) {
        encode_impl(values, e_->K - 1, scale, dst);
    }
    void encode(double value, parms_id_type id, double scale, Plaintext &dst, MemoryPoolHandle = {}) {
        encode_const(value, (int)id[0], scale, dst);
    }
    void encode(double value, double scale, Plaintext &dst, MemoryPoolHandle = {}) { encode_const(value, e_->K - 1, scale, dst); }

    // inverse NTT, CRT composition, embedding DFT and slot gather all run on the device (ckks_decode)
    void decode(const Plaintext &plain, std::vector<double> &out, MemoryPoolHandle = {}) {
        const detail::Poly &p = plain.poly();
        if (!p.buf) throw std::invalid_argument("plain is not valid for encryption parameters");
        std::size_t slots = e_->n / 2;
        detail::DevBuf vals(e_, slots);
        ckks_view v = p.view();
        detail::check(ckks_decode(e_->ctx, &v, p.scale, reinterpret_cast<double *>(vals.p), nullptr));
        out.resize(slots);
        detail::check(ckks_download(e_->ctx, out.data(), vals.p, slots * 8, nullptr));
        detail::check(ckks_stream_sync(e_->ctx, nullptr));
    }

private:
    void check_target(double largest, int limbs, double scale) const {
        // as in SEAL, any level of the context may be targeted, the key level (all K primes) included: the double-hoisted
        // transforms multiply plaintexts into the extended basis Q_L u {P}
        if (limbs < 1 || limbs > e_->K) throw std::invalid_argument("parms_id is not valid for encryption parameters");
        if (!(scale > 0)) throw std::invalid_argument("scale out of bounds");
        int bits = 0;
        for (int j = 0; j < limbs; j++) bits += 64 - __builtin_clzll(e_->primes[j]);
        if (std::log2(scale) >= bits) throw std::invalid_argument("scale out of bounds");
        if (largest > 0 && std::log2(largest) + std::log2(scale) + 1 >= bits) throw std::invalid_argument("encoded values are too large");
    }
    // embedding DFT, rounding, RNS reduction and forward NTT on the device (ckks_encode)
    void encode_impl(const std::vector<double> &values, int limbs, double scale, Plaintext &dst) {
        std::size_t slots = e_->n / 2;
        if (values.size() > slots) throw std::invalid_argument("values has invalid size");
        double largest = 0;
        for (double x : values) largest = std::max(largest, std::fabs(x));
        check_target(largest, limbs, scale);
        detail::Poly &p = dst.poly();
        p.allocate(e_, 1, limbs);
        p.scale = scale;
        ckks_view v = p.view();
        if (values.empty()) {
            detail::check(ckks_encode(e_->ctx, nullptr, 0, scale, &v, nullptr));
            return;
        }
        detail::DevBuf vals(e_, values.size());
        detail::check(ckks_upload(e_->ctx, vals.p, values.data(), values.size() * 8, nullptr));
        detail::check(ckks_encode(e_->ctx, reinterpret_cast<const double *>(vals.p), (int)values.size(), scale, &v, nullptr));
    }
    void encode_const(double value, int limbs, double scale, Plaintext &dst) {
        check_target(std::fabs(value), limbs, scale);
        detail::Poly &p = dst.poly();
        p.allocate(e_, 1, limbs);
        p.scale = scale;
        ckks_view v = p.view();
        detail::check(ckks_encode_scalar(e_->ctx, value, scale, &v, nullptr));
    }
    std::shared_ptr<detail::Engine> e_;
};

// ------------------------------------------------------------------------------------ Encryptor / Decryptor
class Encryptor {
public:
    template <class Ctx>
    Encryptor(const Ctx &context, const PublicKey &pk) : ring_(detail::engine_of(context), detail::fresh_key()), pk_(pk) {}

    // (u pk + e) one level above the plaintext's level, divided-and-rounded by the extra prime
    // (the rescale kernels), plus the plaintext in c0 (SURVEY.md A.9)
    void encrypt(const Plaintext &plain, Ciphertext &dst, MemoryPoolHandle = {}) {
        auto &e = ring_.e;
        const detail::Poly &pt = plain.poly();
        if (!pt.buf) throw std::invalid_argument("plain is not valid for encryption parameters");
        std::size_t n = e->n;
        int L = pt.limbs, W = L + 1, K = e->K;
        auto u = ring_.ternary_ntt(1, W);
        auto big = std::make_shared<detail::DevBuf>(e, (std::size_t)2 * W * n);
        for (int k = 0; k < 2; k++) {
            auto err = ring_.errors_ntt(1, W);
            ckks_view vu = ring_.view(u->p, 1, 1, W), ve = ring_.view(err->p, 1, 1, W);
            ckks_view vpk = ring_.view(pk_.buf->p + (std::size_t)k * K * n, 1, 1, W);
            ckks_view vo = ring_.view(big->p + (std::size_t)k * W * n, 1, 1, W);
            detail::check(ckks_multiply_plain(e->ctx, &vu, &vpk, &vo, nullptr));
            detail::check(ckks_add(e->ctx, &vo, &ve, &vo, nullptr));
        }
        detail::Poly out;
        out.allocate(e, 2, L);
        out.scale = pt.scale;
        ckks_view vin = ring_.view(big->p, 1, 2, W), vout = out.view(), vpt = pt.view();
        detail::check(ckks_rescale(e->ctx, &vin, &vout, nullptr));
        detail::check(ckks_add_plain(e->ctx, &vout, &vpt, &vout, nullptr));
        dst.poly() = out;
    }

private:
    detail::Ring ring_;
    PublicKey pk_;
};

class Decryptor {
public:
    template <class Ctx>
    Decryptor(const Ctx &context, const SecretKey &sk) : ring_(detail::engine_of(context), detail::SampleKey256{}), sk_(sk) {}   // draws nothing

    void decrypt(const Ciphertext &encrypted, Plaintext &dst) {
        auto &e = ring_.e;
        const detail::Poly &ct = encrypted.poly();
        if (!ct.buf) throw std::invalid_argument("encrypted is not valid for encryption parameters");
        std::size_t n = e->n;
        int L = ct.limbs, S = ct.size;
        detail::Poly out;
        out.allocate(e, 1, L);
        out.scale = ct.scale;
        ckks_view vs = ring_.view(sk_.buf->p, 1, 1, L);
        vs.poly_stride = vs.batch_stride = (std::uint64_t)e->K * n;
        ckks_view vo = out.view();
        auto poly_view = [&](int k) {
            ckks_view v = ct.view();
            v.data += (std::uint64_t)k * v.poly_stride;
            v.size = 1;
            return v;
        };
        ckks_view top = poly_view(S - 1);
        // Horner in s: acc = c_{S-1}; acc = acc * s + c_k
        ckks_view vt = top;
        for (int k = S - 2; k >= 0; k--) {
            detail::check(ckks_multiply_plain(e->ctx, &vt, &vs, &vo, nullptr));
            ckks_view vk = poly_view(k);
            detail::check(ckks_add(e->ctx, &vo, &vk, &vo, nullptr));
            vt = vo;
        }
        if (S == 1) detail::check(ckks_copy(e->ctx, vo.data, top.data, (std::size_t)L * n * 8, nullptr));
        dst.poly() = out;
    }

private:
    detail::Ring ring_;
    SecretKey sk_;
};

// ------------------------------------------------------------------------------------ Evaluator
class Evaluator {
public:
    template <class Ctx>
    explicit Evaluator(const Ctx &context) : e_(detail::engine_of(context)) {}

    // ---- add / sub / negate (helper.h:247,259,484; logistic_regression_ckks.cpp:288,341-342)
    void add_inplace(Ciphertext &a, const Ciphertext &b) { binary(a, b, a, 0); }
    void add(const Ciphertext &a, const Ciphertext &b, Ciphertext &dst) { binary(a, b, dst, 0); }
    void sub_inplace(Ciphertext &a, const Ciphertext &b) { binary(a, b, a, 1); }
    void sub(const Ciphertext &a, const Ciphertext &b, Ciphertext &dst) { binary(a, b, dst, 1); }
    void negate_inplace(Ciphertext &a) {
        a.poly().make_unique();
        ckks_view v = a.poly().view();
        detail::check(ckks_negate(e_->ctx, &v, &v, nullptr));
    }
    void negate(const Ciphertext &a, Ciphertext &dst) {
        dst = a;
        negate_inplace(dst);
    }
    void add_many(const std::vector<Ciphertext> &cts, Ciphertext &dst) {
        if (cts.empty()) throw std::invalid_argument("encrypteds cannot be empty");
        Ciphertext acc = cts[0];
        for (std::size_t i = 1; i < cts.size(); i++) add_inplace(acc, cts[i]);
        dst = acc;
    }

    // ---- multiply (helper.h:222,432; matrix_multiplication.cpp:105,126)
    void multiply(const Ciphertext &a, const Ciphertext &b, Ciphertext &dst, MemoryPoolHandle = {}) {
        const detail::Poly &pa = a.poly(), &pb = b.poly();
        need(pa), need(pb);
        if (pa.limbs != pb.limbs) throw std::invalid_argument("encrypted1 and encrypted2 parameter mismatch");
        double scale = pa.scale * pb.scale;
        scale_ok(scale, pa.limbs);
        detail::Poly out;
        out.allocate(e_, pa.size + pb.size - 1, pa.limbs);
        out.scale = scale;
        ckks_view va = pa.view(), vb = pb.view(), vo = out.view();
        detail::check(ckks_multiply(e_->ctx, &va, &vb, &vo, nullptr));
        dst.poly() = out;
        e_->settle();
    }
    void multiply_inplace(Ciphertext &a, const Ciphertext &b, MemoryPoolHandle = {}) { multiply(a, b, a); }
    void square(const Ciphertext &a, Ciphertext &dst, MemoryPoolHandle = {}) { multiply(a, a, dst); }
    void square_inplace(Ciphertext &a, MemoryPoolHandle = {}) { multiply(a, a, a); }

    // ---- plaintext ops (helper.h:250,256,271; logistic_regression_ckks.cpp:198)
    void multiply_plain(const Ciphertext &a, const Plaintext &p, Ciphertext &dst, MemoryPoolHandle = {}) {
        const detail::Poly &pa = a.poly(), &pp = p.poly();
        need(pa), need(pp);
        if (pa.limbs != pp.limbs) throw std::invalid_argument("encrypted and plain parameter mismatch");
        double scale = pa.scale * pp.scale;
        scale_ok(scale, pa.limbs);
        detail::Poly out;
        out.allocate(e_, pa.size, pa.limbs);
        out.scale = scale;
        ckks_view va = pa.view(), vp = pp.view(), vo = out.view();
        detail::check(ckks_multiply_plain(e_->ctx, &va, &vp, &vo, nullptr));
        transparent_check(out);
        dst.poly() = out;
        e_->settle();
    }
    void multiply_plain_inplace(Ciphertext &a, const Plaintext &p, MemoryPoolHandle = {}) { multiply_plain(a, p, a); }
    void add_plain(const Ciphertext &a, const Plaintext &p, Ciphertext &dst) {
        const detail::Poly &pa = a.poly(), &pp = p.poly();
        need(pa), need(pp);
        if (pa.limbs != pp.limbs) throw std::invalid_argument("encrypted and plain parameter mismatch");
        if (pa.scale != pp.scale) throw std::invalid_argument("scale mismatch");
        detail::Poly out;
        out.allocate(e_, pa.size, pa.limbs);
        out.scale = pa.scale;
        ckks_view va = pa.view(), vp = pp.view(), vo = out.view();
        detail::check(ckks_add_plain(e_->ctx, &va, &vp, &vo, nullptr));
        dst.poly() = out;
        e_->settle();
    }
    void add_plain_inplace(Ciphertext &a, const Plaintext &p) { add_plain(a, p, a); }

    // ---- key switching (helper.h:440,541; every rotate_vector call)
    void relinearize_inplace(Ciphertext &a, const RelinKeys &rk, MemoryPoolHandle = {}) { relinearize(a, rk, a); }
    void relinearize(const Ciphertext &a, const RelinKeys &rk, Ciphertext &dst, MemoryPoolHandle = {}) {
        const detail::Poly &pa = a.poly();
        need(pa);
        if (pa.size == 2) {   // SEAL: nothing to do
            dst = a;
            return;
        }
        if (!rk.s || !rk.s->keys.count(0)) throw std::invalid_argument("relin_keys is not valid for encryption parameters");
        detail::Poly out;
        out.allocate(e_, 2, pa.limbs);
        out.scale = pa.scale;
        ckks_view va = pa.view(), vo = out.view();
        detail::check(ckks_relinearize(e_->ctx, &va, rk.s->keys.at(0)->p, &vo, nullptr));
        dst.poly() = out;
        e_->settle();
    }
    void rotate_vector(const Ciphertext &a, int steps, const GaloisKeys &gk, Ciphertext &dst, MemoryPoolHandle = {}) {
        const detail::Poly &pa = a.poly();
        need(pa);
        if (!gk.s) throw std::invalid_argument("galois_keys is not valid for encryption parameters");
        if (pa.size > 2) throw std::invalid_argument("encrypted size must be 2");
        detail::Poly out, scratch;
        out.allocate(e_, 2, pa.limbs);
        scratch.allocate(e_, 2, pa.limbs);
        out.scale = pa.scale;
        ckks_view va = pa.view(), vo = out.view(), vs = scratch.view();
        detail::check(ckks_rotate(e_->ctx, gk.s->ks, &va, steps, &vo, &vs, nullptr));
        dst.poly() = out;
        e_->settle();
    }
    void rotate_vector_inplace(Ciphertext &a, int steps, const GaloisKeys &gk, MemoryPoolHandle = {}) {
        rotate_vector(a, steps, gk, a);
    }
    void apply_galois(const Ciphertext &a, std::uint64_t galois_elt, const GaloisKeys &gk, Ciphertext &dst, MemoryPoolHandle = {}) {
        const detail::Poly &pa = a.poly();
        need(pa);
        if (!gk.has_key(galois_elt)) throw std::invalid_argument("Galois key not present");
        detail::Poly out;
        out.allocate(e_, 2, pa.limbs);
        out.scale = pa.scale;
        ckks_view va = pa.view(), vo = out.view();
        detail::check(ckks_apply_galois(e_->ctx, &va, galois_elt, gk.s->keys.at(galois_elt)->p, &vo, nullptr));
        dst.poly() = out;
        e_->settle();
    }
    void apply_galois_inplace(Ciphertext &a, std::uint64_t galois_elt, const GaloisKeys &gk, MemoryPoolHandle = {}) {
        apply_galois(a, galois_elt, gk, a);
    }

    // ---- rescale / mod switch (helper.h:441,536,543; matrix_multiplication.cpp:71-72,112)
    void rescale_to_next(const Ciphertext &a, Ciphertext &dst, MemoryPoolHandle = {}) {
        const detail::Poly &pa = a.poly();
        need(pa);
        if (pa.limbs < 2) throw std::invalid_argument("end of modulus switching chain reached");
        detail::Poly out;
        out.allocate(e_, pa.size, pa.limbs - 1);
        out.scale = pa.scale / (double)e_->primes[pa.limbs - 1];
        ckks_view va = pa.view(), vo = out.view();
        detail::check(ckks_rescale(e_->ctx, &va, &vo, nullptr));
        dst.poly() = out;
        e_->settle();
    }
    void rescale_to_next_inplace(Ciphertext &a, MemoryPoolHandle = {}) { rescale_to_next(a, a); }
    void mod_switch_to_next_inplace(Ciphertext &a, MemoryPoolHandle = {}) { drop(a.poly(), a.poly().limbs - 1); }
    void mod_switch_to_next_inplace(Plaintext &p) { drop(p.poly(), p.poly().limbs - 1); }
    void mod_switch_to_next(const Ciphertext &a, Ciphertext &dst, MemoryPoolHandle = {}) {
        dst = a;
        mod_switch_to_next_inplace(dst);
    }
    void mod_switch_to_next(const Plaintext &a, Plaintext &dst) {
        dst = a;
        mod_switch_to_next_inplace(dst);
    }
    void mod_switch_to_inplace(Ciphertext &a, parms_id_type id, MemoryPoolHandle = {}) { drop(a.poly(), (int)id[0]); }
    void mod_switch_to_inplace(Plaintext &p, parms_id_type id) { drop(p.poly(), (int)id[0]); }
    void mod_switch_to(const Ciphertext &a, parms_id_type id, Ciphertext &dst, MemoryPoolHandle = {}) {
        dst = a;
        mod_switch_to_inplace(dst, id);
    }

private:
    static void need(const detail::Poly &p) {
        if (!p.buf) throw std::invalid_argument("encrypted is not valid for encryption parameters");
    }
    void scale_ok(double scale, int limbs) const {
        long double lg = 0;
        for (int j = 0; j < limbs; j++) lg += std::log2((long double)e_->primes[j]);
        int bits = (int)std::floor(lg) + 1;
        if (scale <= 0 || (int)std::log2(scale) >= bits) throw std::invalid_argument("scale out of bounds");
    }
    void transparent_check(const detail::Poly &p) {
        auto flag = std::make_shared<detail::DevBuf>(e_, 2);
        ckks_view v = p.view();
        detail::check(ckks_is_transparent(e_->ctx, &v, (std::int32_t *)flag->p, nullptr));
        std::int32_t h = 0;
        detail::check(ckks_download(e_->ctx, &h, flag->p, 4, nullptr));
        detail::check(ckks_stream_sync(e_->ctx, nullptr));
        if (h) throw std::logic_error("result ciphertext is transparent");
    }
    // CKKS mod-switch: the last limbs are simply dropped; with a fixed limb capacity this is metadata
    void drop(detail::Poly &p, int limbs) {
        need(p);
        if (limbs == p.limbs) return;
        if (limbs > p.limbs || limbs < 1) {
            if (p.limbs < 2 && limbs < 1) throw std::invalid_argument("end of modulus switching chain reached");
            throw std::invalid_argument("cannot switch to higher level modulus");
        }
        p.limbs = limbs;
    }
    void binary(const Ciphertext &a, const Ciphertext &b, Ciphertext &dst, int op) {
        const detail::Poly &pa = a.poly(), &pb = b.poly();
        need(pa), need(pb);
        if (pa.limbs != pb.limbs) throw std::invalid_argument("encrypted1 and encrypted2 parameter mismatch");
        if (pa.scale != pb.scale) throw std::invalid_argument("scale mismatch");
        int S = std::max(pa.size, pb.size);
        detail::Poly out;
        out.allocate(e_, S, pa.limbs);
        out.scale = pa.scale;
        // SEAL allows different sizes: the common polys are combined, the rest copied (negated for sub)
        int common = std::min(pa.size, pb.size);
        ckks_view va = pa.view(), vb = pb.view(), vo = out.view();
        va.size = vb.size = vo.size = common;
        detail::check(op == 0 ? ckks_add(e_->ctx, &va, &vb, &vo, nullptr) : ckks_sub(e_->ctx, &va, &vb, &vo, nullptr));
        if (S > common) {
            const detail::Poly &big = pa.size > pb.size ? pa : pb;
            ckks_view vbg = big.view(), vt = out.view();
            vbg.data += (std::uint64_t)common * vbg.poly_stride;
            vt.data += (std::uint64_t)common * vt.poly_stride;
            vbg.size = vt.size = S - common;
            if (op == 1 && pb.size > pa.size) detail::check(ckks_negate(e_->ctx, &vbg, &vt, nullptr));
            else detail::check(copy_polys(e_->ctx, &vbg, &vt));
        }
        dst.poly() = out;
        e_->settle();
    }
    static int copy_polys(ckks_ctx *ctx, const ckks_view *src, const ckks_view *dst) {
        std::size_t n = (std::size_t)1 << ckks_ctx_log_n(ctx);
        for (int s = 0; s < src->size; s++) {
            int rc = ckks_copy(ctx, dst->data + (std::uint64_t)s * dst->poly_stride, src->data + (std::uint64_t)s * src->poly_stride,
                               (std::size_t)src->limbs * n * 8, nullptr);
            if (rc) return rc;
        }
        return CKKS_OK;
    }
    std::shared_ptr<detail::Engine> e_;
};

// ------------------------------------------------------------------------------------ serialization (SURVEY 8 row f2)
// SEAL 3.4.x binary streams, uncompressed (compr_mode none; SEAL reads those whatever its own default is):
//   object = { uint16 magic 0xA15E, uint8 0, uint8 compr_mode, uint32 size } + body, nested objects carry their own header.
// Layouts per class: seal-fyp-logistic-regression_b200/sealio.py (the Python reader/writer of the same format; tools/seal_replay.py
// replays files written by a real SEAL build on this engine).  Data is SEAL's in-memory layout, which is also the
// engine's, so save/load are a header plus one device <-> host copy.
namespace detail {
inline void io_write(std::ostream &o, const void *p, std::size_t n) {
    o.write(static_cast<const char *>(p), (std::streamsize)n);
    if (!o) throw std::runtime_error("I/O error");
}
template <class T>
inline void io_pod(std::string &b, T v) { b.append(reinterpret_cast<const char *>(&v), sizeof(T)); }
inline std::string io_object(const std::string &body) {
    std::string out;
    io_pod<std::uint16_t>(out, 0xA15E);
    io_pod<std::uint8_t>(out, 0);
    io_pod<std::uint8_t>(out, 0);   // compr_mode_type::none
    io_pod<std::uint32_t>(out, (std::uint32_t)(8 + body.size()));
    out += body;
    return out;
}
// reads one object (3.4 header, or the 16-byte header of 3.5+) -> body; compressed streams are refused (no zlib here)
inline std::string io_read_object(std::istream &in) {
    unsigned char h[16];
    in.read(reinterpret_cast<char *>(h), 4);
    if (!in || h[0] != 0x5E || h[1] != 0xA1) throw std::logic_error("loaded SEALHeader is invalid");
    std::uint64_t size, hdr;
    std::uint8_t compr;
    if (h[2] == 0x00) {
        compr = h[3];
        std::uint32_t s32;
        in.read(reinterpret_cast<char *>(&s32), 4);
        size = s32;
        hdr = 8;
    } else if (h[2] == 0x10) {
        in.read(reinterpret_cast<char *>(h + 4), 12);
        compr = h[5];
        std::memcpy(&size, h + 8, 8);
        hdr = 16;
    } else {
        throw std::logic_error("loaded SEALHeader is invalid");
    }
    if (!in || size < hdr) throw std::logic_error("loaded SEALHeader is invalid");
    if (compr != 0) throw std::logic_error("unsupported compression mode (save with compr_mode_type::none)");
    std::string body((std::size_t)(size - hdr), '\0');
    in.read(&body[0], (std::streamsize)body.size());
    if (!in) throw std::runtime_error("I/O error");
    return body;
}
struct IoCursor {
    const std::string &b;
    std::size_t off = 0;
    template <class T>
    T pod() {
        if (off + sizeof(T) > b.size()) throw std::logic_error("loaded data is invalid");
        T v;
        std::memcpy(&v, b.data() + off, sizeof(T));
        off += sizeof(T);
        return v;
    }
    std::string object() {   // nested object
        struct View : std::streambuf {
            View(const char *p, std::size_t n) { setg(const_cast<char *>(p), const_cast<char *>(p), const_cast<char *>(p) + n); }
            std::size_t used() const { return (std::size_t)(gptr() - eback()); }
        } sb(b.data() + off, b.size() - off);
        std::istream in(&sb);
        std::string body = io_read_object(in);
        off += sb.used();
        return body;
    }
};
// SHA3-256 (FIPS 202): SEAL 3.4.x hashes the parameter words with it to form parms_id
inline void sha3_256(const std::uint8_t *msg, std::size_t len, std::uint8_t out[32]) {
    static const std::uint64_t RC[24] = {
        0x0000000000000001ull, 0x0000000000008082ull, 0x800000000000808aull, 0x8000000080008000ull, 0x000000000000808bull,
        0x0000000080000001ull, 0x8000000080008081ull, 0x8000000000008009ull, 0x000000000000008aull, 0x0000000000000088ull,
        0x0000000080008009ull, 0x000000008000000aull, 0x000000008000808bull, 0x800000000000008bull, 0x8000000000008089ull,
        0x8000000000008003ull, 0x8000000000008002ull, 0x8000000000000080ull, 0x000000000000800aull, 0x800000008000000aull,
        0x8000000080008081ull, 0x8000000000008080ull, 0x0000000080000001ull, 0x8000000080008008ull};
    static const int ROT[24] = {1, 3, 6, 10, 15, 21, 28, 36, 45, 55, 2, 14, 27, 41, 56, 8, 25, 43, 62, 18, 39, 61, 20, 44};
    static const int PIL[24] = {10, 7, 11, 17, 18, 3, 5, 16, 8, 21, 24, 4, 15, 23, 19, 13, 12, 2, 20, 14, 22, 9, 6, 1};
    std::uint64_t st[25] = {0};
    auto permute = [&]() {
        for (int r = 0; r < 24; r++) {
            std::uint64_t bc[5];
            for (int i = 0; i < 5; i++) bc[i] = st[i] ^ st[i + 5] ^ st[i + 10] ^ st[i + 15] ^ st[i + 20];
            for (int i = 0; i < 5; i++) {
                std::uint64_t t = bc[(i + 4) % 5] ^ ((bc[(i + 1) % 5] << 1) | (bc[(i + 1) % 5] >> 63));
                for (int j = 0; j < 25; j += 5) st[j + i] ^= t;
            }
            std::uint64_t t = st[1];
            for (int i = 0; i < 24; i++) {
                int j = PIL[i];
                std::uint64_t b = st[j];
                st[j] = (t << ROT[i]) | (t >> (64 - ROT[i]));
                t = b;
            }
            for (int j = 0; j < 25; j += 5) {
                std::uint64_t row[5];
                for (int i = 0; i < 5; i++) row[i] = st[j + i];
                for (int i = 0; i < 5; i++) st[j + i] ^= (~row[(i + 1) % 5]) & row[(i + 2) % 5];
            }
            st[0] ^= RC[r];
        }
    };
    const std::size_t rate = 136;
    std::vector<std::uint8_t> buf(msg, msg + len);
    buf.push_back(0x06);
    while (buf.size() % rate) buf.push_back(0);
    buf.back() |= 0x80;
    for (std::size_t off = 0; off < buf.size(); off += rate) {
        for (std::size_t i = 0; i < rate / 8; i++) {
            std::uint64_t w;
            std::memcpy(&w, buf.data() + off + 8 * i, 8);
            st[i] ^= w;
        }
        permute();
    }
    std::memcpy(out, st, 32);
}
// SEAL's parms_id of the level with `limbs` primes: SHA3-256 over {scheme, N, q_0 .. q_{limbs-1}, plain_modulus = 0}
inline parms_id_type seal_parms_id(const Engine &e, int limbs) {
    std::vector<std::uint64_t> w{(std::uint64_t)scheme_type::CKKS, (std::uint64_t)e.n};
    for (int j = 0; j < limbs; j++) w.push_back(e.primes[j]);
    w.push_back(0);
    std::uint8_t dig[32];
    sha3_256(reinterpret_cast<const std::uint8_t *>(w.data()), w.size() * 8, dig);
    parms_id_type id;
    std::memcpy(id.data(), dig, 32);
    return id;
}
// body of a Ciphertext object over device words [size][cap][N] (active limbs only)
inline std::string io_ct_body(const std::shared_ptr<Engine> &e, const std::uint64_t *dev, int size, int limbs, int cap, double scale) {
    const std::size_t n = e->n;
    std::vector<std::uint64_t> host((std::size_t)size * limbs * n);
    for (int s = 0; s < size; s++)
        check(ckks_download(e->ctx, host.data() + (std::size_t)s * limbs * n, dev + (std::size_t)s * cap * n, (std::size_t)limbs * n * 8, nullptr));
    check(ckks_stream_sync(e->ctx, nullptr));
    std::string b;
    const parms_id_type id = seal_parms_id(*e, limbs);
    b.append(reinterpret_cast<const char *>(id.data()), 32);
    io_pod<std::uint8_t>(b, 1);   // is_ntt_form
    io_pod<std::uint64_t>(b, (std::uint64_t)size);
    io_pod<std::uint64_t>(b, (std::uint64_t)n);
    io_pod<std::uint64_t>(b, (std::uint64_t)limbs);
    io_pod<double>(b, scale);
    std::string arr;
    io_pod<std::uint64_t>(arr, (std::uint64_t)host.size());
    arr.append(reinterpret_cast<const char *>(host.data()), host.size() * 8);
    b += io_object(arr);
    return b;
}
// parses a Ciphertext body into host words; returns {size, limbs, scale}
struct IoCt {
    int size = 0, limbs = 0;
    double scale = 1.0;
    std::vector<std::uint64_t> words;
};
inline IoCt io_parse_ct(const std::string &body, const Engine &e) {
    IoCursor c{body};
    c.off = 32;   // parms_id: the level is taken from coeff_mod_count (ids are hashes of the same information)
    IoCt r;
    (void)c.pod<std::uint8_t>();
    r.size = (int)c.pod<std::uint64_t>();
    const std::uint64_t n = c.pod<std::uint64_t>();
    r.limbs = (int)c.pod<std::uint64_t>();
    r.scale = c.pod<double>();
    if (n != e.n || r.limbs < 1 || r.limbs > e.K || r.size < 1 || r.size > 3) throw std::logic_error("ciphertext data is invalid");
    std::string arr = c.object();
    IoCursor a{arr};
    const std::uint64_t cnt = a.pod<std::uint64_t>();
    if (cnt != (std::uint64_t)r.size * r.limbs * n || arr.size() != 8 + cnt * 8) throw std::logic_error("ciphertext data is invalid");
    r.words.resize(cnt);
    std::memcpy(r.words.data(), arr.data() + 8, cnt * 8);
    for (int s = 0; s < r.size; s++)
        for (int j = 0; j < r.limbs; j++)
            for (std::uint64_t i = 0; i < n; i++)
                if (r.words[((std::size_t)s * r.limbs + j) * n + i] >= e.primes[j]) throw std::logic_error("ciphertext data is invalid");
    return r;
}
}  // namespace detail

inline std::streamoff EncryptionParameters::save(std::ostream &stream) const {
    std::string b;
    detail::io_pod<std::uint8_t>(b, (std::uint8_t)scheme_);
    detail::io_pod<std::uint64_t>(b, (std::uint64_t)n_);
    detail::io_pod<std::uint64_t>(b, (std::uint64_t)coeff_.size());
    auto mod = [](std::uint64_t v) {
        std::string m;
        detail::io_pod<std::uint64_t>(m, v);
        return detail::io_object(m);
    };
    for (const auto &q : coeff_) b += mod(q.value());
    b += mod(plain_.value());
    const std::string out = detail::io_object(b);
    detail::io_write(stream, out.data(), out.size());
    return (std::streamoff)out.size();
}
inline void EncryptionParameters::load(std::istream &stream) {
    const std::string body = detail::io_read_object(stream);
    detail::IoCursor c{body};
    scheme_ = (scheme_type)c.pod<std::uint8_t>();
    n_ = (std::size_t)c.pod<std::uint64_t>();
    const std::uint64_t cnt = c.pod<std::uint64_t>();
    if (cnt > 64) throw std::logic_error("coeff_modulus is invalid");
    coeff_.clear();
    for (std::uint64_t i = 0; i <= cnt; i++) {
        const std::string m = c.object();
        if (m.size() != 8) throw std::logic_error("SmallModulus is invalid");
        std::uint64_t v;
        std::memcpy(&v, m.data(), 8);
        if (i < cnt) coeff_.push_back(SmallModulus(v));
        else plain_ = SmallModulus(v);
    }
}

inline std::streamoff Ciphertext::save(std::ostream &stream) const {
    if (!p_.buf) throw std::logic_error("cannot save an empty ciphertext");
    const std::string out = detail::io_object(detail::io_ct_body(p_.eng, p_.buf->p, p_.size, p_.limbs, p_.cap, p_.scale));
    detail::io_write(stream, out.data(), out.size());
    return (std::streamoff)out.size();
}
template <class Ctx>
inline void Ciphertext::load(const Ctx &context, std::istream &stream) {
    auto e = detail::engine_of(context);
    const detail::IoCt r = detail::io_parse_ct(detail::io_read_object(stream), *e);
    if (r.limbs > e->K - 1) throw std::logic_error("ciphertext data is invalid");
    p_.allocate(e, r.size, r.limbs);
    p_.scale = r.scale;
    detail::check(ckks_upload(e->ctx, p_.buf->p, r.words.data(), r.words.size() * 8, nullptr));
    detail::check(ckks_stream_sync(e->ctx, nullptr));
}

inline std::streamoff Plaintext::save(std::ostream &stream) const {
    if (!p_.buf) throw std::logic_error("cannot save an empty plaintext");
    auto &e = p_.eng;
    const std::size_t n = e->n;
    std::vector<std::uint64_t> host((std::size_t)p_.limbs * n);
    detail::check(ckks_download(e->ctx, host.data(), p_.buf->p, host.size() * 8, nullptr));
    detail::check(ckks_stream_sync(e->ctx, nullptr));
    std::string b;
    const parms_id_type id = detail::seal_parms_id(*e, p_.limbs);
    b.append(reinterpret_cast<const char *>(id.data()), 32);
    detail::io_pod<double>(b, p_.scale);
    std::string arr;
    detail::io_pod<std::uint64_t>(arr, (std::uint64_t)host.size());
    arr.append(reinterpret_cast<const char *>(host.data()), host.size() * 8);
    b += detail::io_object(arr);
    const std::string out = detail::io_object(b);
    detail::io_write(stream, out.data(), out.size());
    return (std::streamoff)out.size();
}
template <class Ctx>
inline void Plaintext::load(const Ctx &context, std::istream &stream) {
    auto e = detail::engine_of(context);
    const std::string body = detail::io_read_object(stream);
    detail::IoCursor c{body};
    c.off = 32;
    const double scale = c.pod<double>();
    const std::string arr = c.object();
    detail::IoCursor a{arr};
    const std::uint64_t cnt = a.pod<std::uint64_t>();
    if (cnt == 0 || cnt % e->n || cnt / e->n > (std::uint64_t)e->K || arr.size() != 8 + cnt * 8) throw std::logic_error("plaintext data is invalid");
    p_.allocate(e, 1, (int)(cnt / e->n));
    p_.scale = scale;
    detail::check(ckks_upload(e->ctx, p_.buf->p, arr.data() + 8, cnt * 8, nullptr));
    detail::check(ckks_stream_sync(e->ctx, nullptr));
}

inline std::streamoff PublicKey::save(std::ostream &stream) const {
    if (!buf) throw std::logic_error("cannot save an empty key");
    auto &e = buf->eng;
    const std::string out = detail::io_object(detail::io_object(detail::io_ct_body(e, buf->p, 2, e->K, e->K, 1.0)));
    detail::io_write(stream, out.data(), out.size());
    return (std::streamoff)out.size();
}
inline std::streamoff SecretKey::save(std::ostream &stream) const {
    if (!buf) throw std::logic_error("cannot save an empty key");
    auto &e = buf->eng;
    std::vector<std::uint64_t> host((std::size_t)e->K * e->n);
    detail::check(ckks_download(e->ctx, host.data(), buf->p, host.size() * 8, nullptr));
    detail::check(ckks_stream_sync(e->ctx, nullptr));
    std::string b;
    const parms_id_type id = detail::seal_parms_id(*e, e->K);
    b.append(reinterpret_cast<const char *>(id.data()), 32);
    detail::io_pod<double>(b, 1.0);
    std::string arr;
    detail::io_pod<std::uint64_t>(arr, (std::uint64_t)host.size());
    arr.append(reinterpret_cast<const char *>(host.data()), host.size() * 8);
    detail::secure_zero(host.data(), host.size() * 8);
    b += detail::io_object(arr);
    const std::string out = detail::io_object(detail::io_object(b));   // SecretKey wraps a Plaintext
    detail::io_write(stream, out.data(), out.size());
    return (std::streamoff)out.size();
}

inline std::streamoff KSwitchKeys::save_impl(std::ostream &stream, bool galois) const {
    if (!s || s->keys.empty()) throw std::logic_error("cannot save empty keys");
    auto &e = s->eng;
    const int K = e->K;
    const std::size_t kw = (std::size_t)2 * K * e->n;   // words of one decomposition digit
    std::string b;
    const parms_id_type id = detail::seal_parms_id(*e, K);
    b.append(reinterpret_cast<const char *>(id.data()), 32);
    const std::uint64_t dim1 = galois ? (std::uint64_t)e->n : 1;   // SEAL sizes GaloisKeys::keys_ to coeff_count
    detail::io_pod<std::uint64_t>(b, dim1);
    std::map<std::uint64_t, detail::BufPtr> by_index;
    for (auto &kv : s->keys) by_index[galois ? (kv.first - 1) >> 1 : 0] = kv.second;
    for (std::uint64_t idx = 0; idx < dim1; idx++) {
        auto it = by_index.find(idx);
        if (it == by_index.end()) {
            detail::io_pod<std::uint64_t>(b, 0);
            continue;
        }
        detail::io_pod<std::uint64_t>(b, (std::uint64_t)(K - 1));
        for (int d = 0; d < K - 1; d++)   // each digit: a PublicKey object wrapping a size-2 ciphertext at the key level
            b += detail::io_object(detail::io_object(detail::io_ct_body(e, it->second->p + (std::size_t)d * kw, 2, K, K, 1.0)));
    }
    const std::string out = detail::io_object(b);
    detail::io_write(stream, out.data(), out.size());
    return (std::streamoff)out.size();
}
inline void KSwitchKeys::load_impl(std::shared_ptr<detail::Engine> e, std::istream &stream, bool galois) {
    const std::string body = detail::io_read_object(stream);
    detail::IoCursor c{body};
    c.off = 32;
    const std::uint64_t dim1 = c.pod<std::uint64_t>();
    const int K = e->K;
    const std::size_t kw = (std::size_t)2 * K * e->n;
    s = std::make_shared<Shared>();
    s->eng = e;
    detail::check(ckks_keyset_create(e->ctx, &s->ks));
    for (std::uint64_t idx = 0; idx < dim1; idx++) {
        const std::uint64_t dim2 = c.pod<std::uint64_t>();
        if (dim2 == 0) continue;
        if (dim2 != (std::uint64_t)(K - 1)) throw std::logic_error("key-switching key data is invalid");
        auto d = std::make_shared<detail::DevBuf>(e, (std::size_t)(K - 1) * kw);
        for (int j = 0; j < K - 1; j++) {
            const std::string pk = c.object();
            detail::IoCursor pc{pk};
            const detail::IoCt ct = detail::io_parse_ct(pc.object(), *e);
            if (ct.size != 2 || ct.limbs != K) throw std::logic_error("key-switching key data is invalid");
            detail::check(ckks_upload(e->ctx, d->p + (std::size_t)j * kw, ct.words.data(), kw * 8, nullptr));
            detail::check(ckks_stream_sync(e->ctx, nullptr));
        }
        const std::uint64_t g = galois ? 2 * idx + 1 : 0;
        s->keys[g] = d;
        if (galois) detail::check(ckks_keyset_set_galois(s->ks, g, d->p));
        else detail::check(ckks_keyset_set_relin(s->ks, d->p));
    }
}
template <class Ctx>
inline void RelinKeys::load(const Ctx &context, std::istream &stream) { load_impl(detail::engine_of(context), stream, false); }
template <class Ctx>
inline void GaloisKeys::load(const Ctx &context, std::istream &stream) { load_impl(detail::engine_of(context), stream, true); }

}  // namespace seal

