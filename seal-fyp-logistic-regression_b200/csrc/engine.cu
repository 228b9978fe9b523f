// engine.cu -- context, launch logic and the extern "C" surface declared in include/ckks_b200.h.
//
// One context = one CKKS parameter set on one device.  Every entry point validates its views,
// enqueues kernels on the caller's stream and returns; nothing here synchronises the device
// and nothing falls back to the CPU.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <map>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/ckks_b200.h"
#include "kernels.cuh"
#include "encoder.cuh"
#include "tables.h"

// ------------------------------------------------------------------------------------ errors
static thread_local std::string g_err;
static int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}
#define CU(call)                                                                              \
    do {                                                                                      \
        cudaError_t e__ = (call);                                                             \
        if (e__ != cudaSuccess)                                                               \
            return fail(CKKS_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));  \
    } while (0)
#define LAUNCH_CHECK(ctx)                                                                  \
    do {                                                                                   \
        (ctx)->launches++;                                                                 \
        cudaError_t e__ = cudaPeekAtLastError();                                           \
        if (e__ != cudaSuccess)                                                            \
            return fail(CKKS_ERR_CUDA, std::string("kernel launch: ") + cudaGetErrorString(e__)); \
    } while (0)

// Programmatic dependent launch: the next kernel of a pipeline may become resident while the previous one drains; it runs
// its prologue (constants, index tables) and blocks at griddepcontrol.wait until the predecessor's memory is visible.  The
// kernels release their successor late (PDL_LATE in kernels.cuh), so only the immediate successor gets the head start.
// -1 = automatic (on for launches that carry >= 8 ciphertexts), 0 = never, 1 = always (CKKS_PDL)
static int g_pdl_mode = getenv("CKKS_PDL") ? atoi(getenv("CKKS_PDL")) : -1;
static thread_local bool g_pdl_now = false;   // decided per batched key switch (keyswitch()), read by launch_pdl
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(NTT_THREADS);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    // Measured on the fused pipeline with the late trigger (N = 32768, L = 3): -6 % at batch 16, -5 % at 8, -2 % at 32 and at 2,
    // but +7 % at batch 4 -- hence on from 8 ciphertexts per launch.
    cfg.numAttrs = g_pdl_now ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// thread-block-cluster launch (cluster = grid.x CTAs: the digits of one output tile), dynamic shared memory opted in once
template <typename... KArgs, typename... Args>
static cudaError_t launch_cluster(void (*kernel)(KArgs...), dim3 grid, size_t smem, cudaStream_t st, Args... args) {
    static thread_local std::map<std::pair<int, const void *>, bool> ready;   // the attribute is per device
    int dev = 0;
    cudaGetDevice(&dev);
    if (!ready[{dev, (const void *)kernel}]) {
        cudaError_t e = cudaFuncSetAttribute((const void *)kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        ready[{dev, (const void *)kernel}] = true;
    }
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(NTT_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = grid.x;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// ------------------------------------------------------------------------------------ context
struct ckks_ctx {
    int log_n = 0, n = 0, K = 0, device = 0;
    std::vector<uint64_t> primes;
    Tables t{};
    void *d_mod = nullptr, *d_twf = nullptr, *d_twi = nullptr, *d_inv = nullptr, *d_invs = nullptr, *d_half = nullptr;
    void *d_fp = nullptr, *d_twfd = nullptr, *d_twid = nullptr;
    std::unordered_map<uint64_t, uint32_t *> perms;
    bool pool_ready = false;
    struct TiledKey {
        u64 *copy = nullptr;
        int refs = 0;
    };
    std::vector<struct ckks_keyset *> keysets;                   // live key registries (orphaned when the context goes first)
    std::unordered_map<const uint64_t *, TiledKey> tiled_keys;   // registered key (caller's pointer) -> engine-owned tiled copy
    uint32_t *d_kidx = nullptr;                 // encoder: slot i -> DFT position (3^i mod 2N - 1)/2
    std::vector<HalfDigits> half_digits;        // decoder: mixed-radix digits of (Q_L - 1)/2, index L
    u64 *ws = nullptr;
    size_t ws_bytes = 0;
    size_t ws_cap = size_t(1) << 30;
    uint64_t launches = 0;
    // rotate-and-sum chains: private streams + cached CUDA graphs of 1 and of 8 ping-pong pairs of steps
    cudaStream_t chain_stream = nullptr;
    cudaEvent_t ev_in = nullptr, ev_out = nullptr;
    // lane 0 is the normal path; lane 1 has its own workspace, side stream and events so that a chain can
    // run two half-batches as concurrent pipelines (each lane's FP64 inner-product kernel runs on its side
    // stream beside the integer one)
    struct Lane {
        u64 *ws = nullptr;
        size_t ws_bytes = 0;
        cudaStream_t side = nullptr, main = nullptr;
        cudaEvent_t fork = nullptr, join = nullptr, begin = nullptr, end = nullptr;
    } lane[4];
    int chain_lanes = 2;
    int round_rescale = 1;     // divide-and-round (1) or floor (0) in rescale; t.round_half is the key switch's switch
    int fuse = 1;              // fused column passes / INTT-in-MAC (CKKS_FUSE=0 selects the unfused round-1 pipeline)
    int split1 = 0, split3 = 0; // forced nsplit of the fused column kernels (0 = heuristic)
    struct ChainGraph {
        cudaGraphExec_t exec;
        uint64_t launches;
    };
    std::map<std::vector<uint64_t>, ChainGraph> chain_graphs;
};

struct ckks_keyset {
    ckks_ctx *ctx;
    const uint64_t *relin = nullptr;
    std::unordered_map<uint64_t, const uint64_t *> galois;
    // slot tables for per-entry key selection inside one launch (rotation plans)
    std::vector<uint64_t> slot_elt;
    std::unordered_map<uint64_t, int> slot_of;
    const uint32_t **d_perm_tab = nullptr;
    const u64 **d_key_tab = nullptr;
    int tab_cap = 0;
    bool tab_dirty = true;
};

// A fixed set of rotations (one step count per batch entry) compiled into rounds: round r applies
// the r-th NAF term of every entry that still has one, all in a single batched key switch.
struct ckks_rotplan {
    ckks_ctx *ctx;
    ckks_keyset *ks;
    int batch = 0;
    std::vector<int> round_off, round_cnt;
    std::vector<int> zero_entries;
    KsSel *d_sel = nullptr;
    uint64_t keyswitches = 0;
    // shared-prefix form, used when every entry rotates the SAME input ciphertext (in->batch == 1): rotations whose NAF
    // chains start with the same terms share those key switches -- the intermediate ciphertext is a deterministic function
    // of the input and the keys, so every output stays bit-identical to its own rotate_vector call (helper.h:252-257:
    // d = 128 needs 169 instead of 355 key switches).  Node storage: the output entry of the rotation that ends at the
    // node, else a scratch entry.
    std::vector<int> sh_round_off, sh_round_cnt;
    std::vector<std::pair<int, int>> sh_copies;   // (from entry, to entry) for repeated steps
    KsSel *d_sel_sh = nullptr;
    uint64_t keyswitches_shared = 0;
};

static int upload_vec(void **dst, const void *src, size_t bytes) {
    CU(cudaMalloc(dst, bytes));
    CU(cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice));
    return CKKS_OK;
}

extern "C" const char *ckks_last_error(void) { return g_err.c_str(); }
extern "C" const char *ckks_version(void) { return "ckks_b200 0.1 (sm_100a)"; }

extern "C" int ckks_ctx_create(int log_n, int n_primes, const uint64_t *primes, int device, ckks_ctx **out) {
    if (!out || !primes) return fail(CKKS_ERR_INVALID, "null argument");
    if (log_n < 12 || log_n > 15) return fail(CKKS_ERR_INVALID, "poly_modulus_degree must be 4096..32768");
    if (n_primes < 2 || n_primes > 32) return fail(CKKS_ERR_INVALID, "coeff_modulus needs 2..32 primes");
    ckks::HostTables ht;
    std::vector<uint64_t> pv(primes, primes + n_primes);
    try {
        ckks::build_tables(log_n, pv, ht);
    } catch (const std::exception &e) {
        return fail(CKKS_ERR_INVALID, e.what());
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(CKKS_ERR_CUDA, "no CUDA device: this engine has no CPU fallback");
    CU(cudaSetDevice(device));
    ckks_ctx *c = new ckks_ctx;
    c->log_n = log_n;
    c->n = 1 << log_n;
    c->K = n_primes;
    c->device = device;
    c->primes = pv;
    int rc;
    if ((rc = upload_vec(&c->d_mod, ht.mod.data(), ht.mod.size() * 8)) ||
        (rc = upload_vec(&c->d_twf, ht.twf.data(), ht.twf.size() * 8)) ||
        (rc = upload_vec(&c->d_twi, ht.twi.data(), ht.twi.size() * 8)) ||
        (rc = upload_vec(&c->d_inv, ht.inv.data(), ht.inv.size() * 8)) ||
        (rc = upload_vec(&c->d_invs, ht.invs.data(), ht.invs.size() * 8)) ||
        (rc = upload_vec(&c->d_half, ht.halfmod.data(), ht.halfmod.size() * 8)) ||
        (rc = upload_vec(&c->d_fp, ht.fpc.data(), ht.fpc.size() * 8)) ||
        (rc = upload_vec(&c->d_twfd, ht.twfd.data(), ht.twfd.size() * 8)) ||
        (rc = upload_vec(&c->d_twid, ht.twid.data(), ht.twid.size() * 8))) {
        ckks_ctx_destroy(c);
        return rc;
    }
    c->t.mod = (const ModConst *)c->d_mod;
    c->t.twf = (const tw_t *)c->d_twf;
    c->t.twi = (const tw_t *)c->d_twi;
    c->t.inv = (const u64 *)c->d_inv;
    c->t.invs = (const u64 *)c->d_invs;
    c->t.halfmod = (const u64 *)c->d_half;
    c->t.fp = (const FpConst *)c->d_fp;
    c->t.twfd = (const double *)c->d_twfd;
    c->t.twid = (const double *)c->d_twid;
    c->t.K = n_primes;
    c->t.round_half = 1;
    if (const char *e = getenv("CKKS_FUSE")) c->fuse = atoi(e);
    if (const char *e = getenv("CKKS_SPLIT1")) c->split1 = atoi(e);
    if (const char *e = getenv("CKKS_SPLIT3")) c->split3 = atoi(e);
    if (const char *e = getenv("CKKS_WS_CAP_MB")) c->ws_cap = (size_t)atol(e) << 20;
    if (const char *e = getenv("CKKS_LANES")) c->chain_lanes = atoi(e) < 1 ? 1 : (atoi(e) > 4 ? 4 : atoi(e));
    *out = c;
    return CKKS_OK;
}

extern "C" void ckks_ctx_destroy(ckks_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    for (auto &kv : c->perms) cudaFree(kv.second);
    for (auto &kv : c->tiled_keys) cudaFree(kv.second.copy);
    for (ckks_keyset *ks : c->keysets) ks->ctx = nullptr;
    cudaFree(c->d_kidx);
    for (auto &kv : c->chain_graphs) cudaGraphExecDestroy(kv.second.exec);
    if (c->chain_stream) cudaStreamDestroy(c->chain_stream);
    for (auto &ln : c->lane) {
        if (ln.side) cudaStreamDestroy(ln.side);
        if (ln.main) cudaStreamDestroy(ln.main);
        for (cudaEvent_t e : {ln.fork, ln.join, ln.begin, ln.end})
            if (e) cudaEventDestroy(e);
        if (&ln != &c->lane[0]) cudaFree(ln.ws);
    }
    if (c->ev_in) cudaEventDestroy(c->ev_in);
    if (c->ev_out) cudaEventDestroy(c->ev_out);
    cudaFree(c->d_mod); cudaFree(c->d_twf); cudaFree(c->d_twi);
    cudaFree(c->d_inv); cudaFree(c->d_invs); cudaFree(c->d_half);
    cudaFree(c->d_fp); cudaFree(c->d_twfd); cudaFree(c->d_twid);
    cudaFree(c->ws);
    delete c;
}

extern "C" int ckks_ctx_log_n(const ckks_ctx *c) { return c->log_n; }
extern "C" int ckks_ctx_n_primes(const ckks_ctx *c) { return c->K; }
extern "C" uint64_t ckks_ctx_prime(const ckks_ctx *c, int j) { return (j >= 0 && j < c->K) ? c->primes[j] : 0; }
extern "C" int ckks_ctx_set_rounding(ckks_ctx *c, int mode) {
    if (mode < 0 || mode > 3) return fail(CKKS_ERR_INVALID, "rounding mode must be 0..3");
    c->t.round_half = (mode == 1 || mode == 2) ? 1 : 0;     // key-switch mod-down
    c->round_rescale = (mode == 1 || mode == 3) ? 1 : 0;    // rescale
    for (auto &kv : c->chain_graphs) cudaGraphExecDestroy(kv.second.exec);   // captured kernels carry the flag by value
    c->chain_graphs.clear();
    return CKKS_OK;
}
extern "C" int ckks_ctx_set_chain_lanes(ckks_ctx *c, int lanes) {
    if (lanes < 1 || lanes > 4) return fail(CKKS_ERR_INVALID, "chain lanes must be 1..4");
    c->chain_lanes = lanes;
    return CKKS_OK;
}
extern "C" int ckks_ctx_set_workspace_cap(ckks_ctx *c, size_t bytes) {
    c->ws_cap = bytes;
    return CKKS_OK;
}
extern "C" uint64_t ckks_ctx_launch_count(const ckks_ctx *c) { return c->launches; }
extern "C" void ckks_ctx_reset_launch_count(ckks_ctx *c) { c->launches = 0; }

static int ensure_ws(ckks_ctx *c, size_t bytes) {
    if (bytes <= c->ws_bytes) return CKKS_OK;
    CU(cudaSetDevice(c->device));
    if (c->ws) {
        CU(cudaDeviceSynchronize());  // growing mid-stream: let in-flight users of the old buffer finish
        CU(cudaFree(c->ws));
        c->ws = nullptr;
        c->ws_bytes = 0;
    }
    cudaError_t e = cudaMalloc((void **)&c->ws, bytes);
    if (e != cudaSuccess) return fail(CKKS_ERR_NOMEM, "workspace allocation failed");
    c->ws_bytes = bytes;
    return CKKS_OK;
}

static int ensure_lane(ckks_ctx *c, int li, size_t bytes) {
    ckks_ctx::Lane &ln = c->lane[li];
    if (!ln.side) {
        CU(cudaStreamCreateWithFlags(&ln.side, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&ln.main, cudaStreamNonBlocking));
        for (cudaEvent_t *e : {&ln.fork, &ln.join, &ln.begin, &ln.end}) CU(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
    }
    if (li == 0) {
        int rc = ensure_ws(c, bytes);
        ln.ws = c->ws;
        ln.ws_bytes = c->ws_bytes;
        return rc;
    }
    if (bytes <= ln.ws_bytes) return CKKS_OK;
    if (ln.ws) {
        CU(cudaDeviceSynchronize());
        CU(cudaFree(ln.ws));
        ln.ws = nullptr;
        ln.ws_bytes = 0;
    }
    if (cudaMalloc((void **)&ln.ws, bytes) != cudaSuccess) return fail(CKKS_ERR_NOMEM, "workspace allocation failed");
    ln.ws_bytes = bytes;
    return CKKS_OK;
}

// words of workspace one key switch needs per ciphertext at L limbs
static size_t ks_words_per_ct(const ckks_ctx *c, int L) {
    return (size_t)c->n * ((size_t)L + (size_t)L * (L + 1) + 2 * (size_t)(L + 1) + 2 * (size_t)L);
}
static int ks_chunk(const ckks_ctx *c, int B, int L) {
    size_t per = ks_words_per_ct(c, L) * 8;
    size_t fit = c->ws_cap / per;
    if (fit < 1) fit = 1;
    if (fit > 16384) fit = 16384;
    return (int)(fit < (size_t)B ? fit : (size_t)B);
}

extern "C" int ckks_ctx_reserve(ckks_ctx *c, int batch, int limbs) {
    if (batch < 1 || limbs < 1 || limbs >= c->K + 1) return fail(CKKS_ERR_INVALID, "bad reserve request");
    int bc = ks_chunk(c, batch, limbs);
    return ensure_ws(c, ks_words_per_ct(c, limbs) * 8 * (size_t)bc);
}

// ------------------------------------------------------------------------------------ helpers
// Device buffers for callers without their own allocator (the seal.h shim allocates one per
// Plaintext / Ciphertext): served from the device's stream-ordered memory pool on the default
// stream, with the pool told to keep freed memory -- a plain cudaMalloc costs ~2 ms on this part
// and cudaFree synchronises the device, which dominated the reference's programs.
extern "C" int ckks_dev_alloc_async(ckks_ctx *c, size_t bytes, void **out, ckks_stream s) {
    CU(cudaSetDevice(c->device));
    if (!c->pool_ready) {
        cudaMemPool_t pool;
        CU(cudaDeviceGetDefaultMemPool(&pool, c->device));
        uint64_t keep = ~0ull;
        CU(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
        c->pool_ready = true;
    }
    if (cudaMallocAsync(out, bytes, (cudaStream_t)s) != cudaSuccess) {
        cudaGetLastError();
        return fail(CKKS_ERR_NOMEM, "device allocation failed");
    }
    return CKKS_OK;
}
extern "C" int ckks_dev_free_async(ckks_ctx *c, void *p, ckks_stream s) {
    CU(cudaSetDevice(c->device));
    CU(cudaFreeAsync(p, (cudaStream_t)s));
    return CKKS_OK;
}
// default-stream forms (what the seal/seal.h shim uses: it runs every call on the default stream)
extern "C" int ckks_dev_alloc(ckks_ctx *c, size_t bytes, void **out) { return ckks_dev_alloc_async(c, bytes, out, nullptr); }
extern "C" int ckks_dev_free(ckks_ctx *c, void *p) { return ckks_dev_free_async(c, p, nullptr); }
extern "C" int ckks_host_alloc(size_t bytes, void **out) {
    if (cudaMallocHost(out, bytes) != cudaSuccess) return fail(CKKS_ERR_NOMEM, "pinned allocation failed");
    return CKKS_OK;
}
extern "C" int ckks_host_free(void *p) {
    CU(cudaFreeHost(p));
    return CKKS_OK;
}
extern "C" int ckks_upload(ckks_ctx *, void *dst, const void *src, size_t bytes, ckks_stream s) {
    CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, (cudaStream_t)s));
    return CKKS_OK;
}
extern "C" int ckks_download(ckks_ctx *, void *dst, const void *src, size_t bytes, ckks_stream s) {
    CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, (cudaStream_t)s));
    return CKKS_OK;
}
extern "C" int ckks_copy(ckks_ctx *, void *dst, const void *src, size_t bytes, ckks_stream s) {
    CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)s));
    return CKKS_OK;
}
extern "C" int ckks_stream_sync(ckks_ctx *, ckks_stream s) {
    CU(cudaStreamSynchronize((cudaStream_t)s));
    return CKKS_OK;
}

static inline DView dv(const ckks_view *v) { return DView{(u64 *)v->data, v->batch_stride, v->poly_stride}; }

static int check_view(const ckks_ctx *c, const ckks_view *v, const char *name) {
    if (!v || !v->data) return fail(CKKS_ERR_INVALID, std::string(name) + ": null view");
    if (v->batch < 1 || v->size < 1) return fail(CKKS_ERR_INVALID, std::string(name) + ": empty view");
    if (v->limbs < 1 || v->limbs > c->K)   // K limbs = key level (element-wise ops and rescale only)
        return fail(CKKS_ERR_INVALID, std::string(name) + ": limbs outside the modulus chain of this context");
    if ((size_t)v->poly_stride < (size_t)v->limbs * c->n) return fail(CKKS_ERR_INVALID, std::string(name) + ": poly_stride too small");
    if (v->batch > 1 && (size_t)v->batch_stride < (size_t)v->size * v->poly_stride && v->batch_stride != 0)
        return fail(CKKS_ERR_INVALID, std::string(name) + ": batch_stride too small");
    if (((uintptr_t)v->data & 15) || (v->poly_stride & 1) || (v->batch_stride & 1))
        return fail(CKKS_ERR_INVALID, std::string(name) + ": data must be 16-byte aligned");
    if (v->batch > 65535) return fail(CKKS_ERR_INVALID, std::string(name) + ": batch > 65535");
    return CKKS_OK;
}
static int same_shape(const ckks_view *a, const ckks_view *b, const char *what) {
    if (a->batch != b->batch || a->size != b->size || a->limbs != b->limbs)
        return fail(CKKS_ERR_INVALID, std::string(what) + " parameter mismatch");
    return CKKS_OK;
}

#define DISPATCH_LOGN(c, MACRO)                                                   \
    switch ((c)->log_n) {                                                         \
    case 12: MACRO(12); break;                                                    \
    case 13: MACRO(13); break;                                                    \
    case 14: MACRO(14); break;                                                    \
    case 15: MACRO(15); break;                                                    \
    default: return fail(CKKS_ERR_INVALID, "unsupported degree");                 \
    }

// ------------------------------------------------------------------------------------ NTT API
static int ntt_api(ckks_ctx *c, uint64_t *data, int n_polys, int limbs, int first_prime, uint64_t ps, bool inverse, cudaStream_t st) {
    if (!data || n_polys < 1 || limbs < 1 || first_prime < 0 || first_prime + limbs > c->K)
        return fail(CKKS_ERR_INVALID, "ntt: bad arguments");
    if (ps < (uint64_t)limbs * c->n) return fail(CKKS_ERR_INVALID, "ntt: poly_stride too small");
    if (n_polys > 65535) return fail(CKKS_ERR_INVALID, "ntt: more than 65535 polys");
    CU(cudaSetDevice(c->device));
    DView v{(u64 *)data, ps, 0};
    // north-star variant: one limb per CTA, limb resident in shared memory (N <= 16384); opt-in, see kernels.cuh
    static const bool limb_per_cta = getenv("CKKS_NTT_LIMB") && atoi(getenv("CKKS_NTT_LIMB"));
    if (limb_per_cta && c->log_n <= 14) {
        const size_t smem = ((size_t)c->n + 4 * NTT_TILE) * 8;
        const unsigned grid = (unsigned)n_polys * (unsigned)limbs;
#define RUNL(LN)                                                                                                          \
    {                                                                                                                     \
        if (inverse) {                                                                                                    \
            CU(cudaFuncSetAttribute(k_ntt_limb<LN, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));       \
            k_ntt_limb<LN, true><<<grid, 1024, smem, st>>>(v, limbs, first_prime, c->t);                                  \
        } else {                                                                                                          \
            CU(cudaFuncSetAttribute(k_ntt_limb<LN, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));      \
            k_ntt_limb<LN, false><<<grid, 1024, smem, st>>>(v, limbs, first_prime, c->t);                                 \
        }                                                                                                                 \
        LAUNCH_CHECK(c);                                                                                                  \
    }
        switch (c->log_n) {
        case 12: RUNL(12); break;
        case 13: RUNL(13); break;
        default: RUNL(14); break;
        }
#undef RUNL
        return CKKS_OK;
    }
#define RUN(LN)                                                                                             \
    {                                                                                                       \
        dim3 gc(NttGeo<LN>::COL_TILES, limbs, n_polys), gr(NttGeo<LN>::ROW_TILES, limbs, n_polys);          \
        if (!inverse) {                                                                                     \
            k_fwd_col<LN><<<gc, NTT_THREADS, 0, st>>>(v, v, limbs, first_prime, c->t); LAUNCH_CHECK(c);     \
            k_fwd_row<LN><<<gr, NTT_THREADS, 0, st>>>(v, v, limbs, first_prime, c->t); LAUNCH_CHECK(c);     \
        } else {                                                                                            \
            k_inv_row<LN><<<gr, NTT_THREADS, 0, st>>>(v, v, limbs, first_prime, c->t); LAUNCH_CHECK(c);     \
            k_inv_col<LN, false><<<gc, NTT_THREADS, 0, st>>>(v, v, limbs, first_prime, c->t); LAUNCH_CHECK(c); \
        }                                                                                                   \
    }
    DISPATCH_LOGN(c, RUN)
#undef RUN
    return CKKS_OK;
}
extern "C" int ckks_ntt_forward(ckks_ctx *c, uint64_t *d, int np, int l, int fp, uint64_t ps, ckks_stream s) {
    return ntt_api(c, d, np, l, fp, ps, false, (cudaStream_t)s);
}
extern "C" int ckks_ntt_inverse(ckks_ctx *c, uint64_t *d, int np, int l, int fp, uint64_t ps, ckks_stream s) {
    return ntt_api(c, d, np, l, fp, ps, true, (cudaStream_t)s);
}

// ------------------------------------------------------------------------------------ element-wise
static inline dim3 ew_grid(const ckks_ctx *c, int y, int z) { return dim3((c->n / 2 + 255) / 256, y, z); }

static int addsub(ckks_ctx *c, int op, const ckks_view *a, const ckks_view *b, const ckks_view *o, cudaStream_t st) {
    int rc;
    if ((rc = check_view(c, a, "a")) || (rc = check_view(c, o, "out")) || (rc = same_shape(a, o, "destination"))) return rc;
    if (op != 2 && ((rc = check_view(c, b, "b")) || (rc = same_shape(a, b, "encrypted1 and encrypted2")))) return rc;
    CU(cudaSetDevice(c->device));
    dim3 g = ew_grid(c, a->size * a->limbs, a->batch);
    DView vb = op != 2 ? dv(b) : dv(a);
    if (op == 0) k_ew_addsub<0><<<g, 256, 0, st>>>(dv(a), vb, dv(o), a->limbs, c->n, c->t);
    if (op == 1) k_ew_addsub<1><<<g, 256, 0, st>>>(dv(a), vb, dv(o), a->limbs, c->n, c->t);
    if (op == 2) k_ew_addsub<2><<<g, 256, 0, st>>>(dv(a), vb, dv(o), a->limbs, c->n, c->t);
    LAUNCH_CHECK(c);
    return CKKS_OK;
}
extern "C" int ckks_add(ckks_ctx *c, const ckks_view *a, const ckks_view *b, const ckks_view *o, ckks_stream s) {
    return addsub(c, 0, a, b, o, (cudaStream_t)s);
}
extern "C" int ckks_sub(ckks_ctx *c, const ckks_view *a, const ckks_view *b, const ckks_view *o, ckks_stream s) {
    return addsub(c, 1, a, b, o, (cudaStream_t)s);
}
extern "C" int ckks_negate(ckks_ctx *c, const ckks_view *a, const ckks_view *o, ckks_stream s) {
    return addsub(c, 2, a, nullptr, o, (cudaStream_t)s);
}

extern "C" int ckks_multiply(ckks_ctx *c, const ckks_view *a, const ckks_view *b, const ckks_view *o, ckks_stream s) {
    int rc;
    if ((rc = check_view(c, a, "a")) || (rc = check_view(c, b, "b")) || (rc = check_view(c, o, "out"))) return rc;
    if ((a->batch != b->batch && b->batch != 1) || a->limbs != b->limbs)
        return fail(CKKS_ERR_INVALID, "encrypted1 and encrypted2 parameter mismatch");
    if (o->batch != a->batch || o->limbs != a->limbs || o->size != a->size + b->size - 1)
        return fail(CKKS_ERR_INVALID, "destination parameter mismatch");
    if (o->data == a->data || o->data == b->data) return fail(CKKS_ERR_INVALID, "multiply: out must not alias an input");
    CU(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)s;
    dim3 g = ew_grid(c, a->limbs, a->batch);
    DView vb = dv(b);
    if (b->batch == 1) vb.bs = 0;   // one ciphertext multiplied into every batch entry
#define MUL(SA, SB) k_ew_multiply<SA, SB><<<g, 256, 0, st>>>(dv(a), vb, dv(o), a->limbs, c->n, c->t)
    if (a->size == 2 && b->size == 2) MUL(2, 2);
    else if (a->size == 3 && b->size == 2) MUL(3, 2);
    else if (a->size == 2 && b->size == 3) MUL(2, 3);
    else if (a->size == 3 && b->size == 3) MUL(3, 3);
    else if (a->size == 2 && b->size == 1) MUL(2, 1);
    else if (a->size == 1 && b->size == 2) MUL(1, 2);
    else return fail(CKKS_ERR_INVALID, "multiply: ciphertext sizes above 3 are not supported");
#undef MUL
    LAUNCH_CHECK(c);
    return CKKS_OK;
}

static int plain_op(ckks_ctx *c, bool mul, const ckks_view *ct, const ckks_view *pt, const ckks_view *o, cudaStream_t st) {
    int rc;
    if ((rc = check_view(c, ct, "encrypted")) || (rc = check_view(c, pt, "plain")) || (rc = check_view(c, o, "out")) ||
        (rc = same_shape(ct, o, "destination")))
        return rc;
    if (pt->size != 1 || pt->limbs != ct->limbs || (pt->batch != 1 && pt->batch != ct->batch))
        return fail(CKKS_ERR_INVALID, "encrypted and plain parameter mismatch");
    CU(cudaSetDevice(c->device));
    DView p = dv(pt);
    if (pt->batch == 1) p.bs = 0;
    dim3 g = ew_grid(c, ct->size * ct->limbs, ct->batch);
    if (mul) k_ew_mul_plain<<<g, 256, 0, st>>>(dv(ct), p, dv(o), ct->limbs, c->n, c->t);
    else k_ew_add_plain<<<g, 256, 0, st>>>(dv(ct), p, dv(o), ct->limbs, c->n, c->t);
    LAUNCH_CHECK(c);
    return CKKS_OK;
}
extern "C" int ckks_multiply_plain(ckks_ctx *c, const ckks_view *ct, const ckks_view *pt, const ckks_view *o, ckks_stream s) {
    return plain_op(c, true, ct, pt, o, (cudaStream_t)s);
}
extern "C" int ckks_add_plain(ckks_ctx *c, const ckks_view *ct, const ckks_view *pt, const ckks_view *o, ckks_stream s) {
    return plain_op(c, false, ct, pt, o, (cudaStream_t)s);
}

extern "C" int ckks_add_many(ckks_ctx *c, const ckks_view *in, const ckks_view *o, ckks_stream s) {
    int rc;
    if ((rc = check_view(c, in, "in")) || (rc = check_view(c, o, "out"))) return rc;
    if (o->batch != 1 || o->size != in->size || o->limbs != in->limbs) return fail(CKKS_ERR_INVALID, "destination parameter mismatch");
    CU(cudaSetDevice(c->device));
    k_ew_add_many<<<ew_grid(c, in->size * in->limbs, 1), 256, 0, (cudaStream_t)s>>>(dv(in), dv(o), in->batch, in->limbs, c->n, c->t);
    LAUNCH_CHECK(c);
    return CKKS_OK;
}

extern "C" int ckks_add_many_grouped(ckks_ctx *c, const ckks_view *in, int groups, const ckks_view *o, ckks_stream s) {
    int rc;
    if ((rc = check_view(c, in, "in")) || (rc = check_view(c, o, "out"))) return rc;
    if (groups < 1) return fail(CKKS_ERR_INVALID, "add_many_grouped: groups must be at least 1");
    if ((long long)groups * o->batch != in->batch)
        return fail(CKKS_ERR_INVALID, "add_many_grouped: in batch must be groups x out batch");
    if (o->size != in->size || o->limbs != in->limbs) return fail(CKKS_ERR_INVALID, "destination parameter mismatch");
    if (o->data == in->data) return fail(CKKS_ERR_INVALID, "add_many_grouped: out must not alias in");
    CU(cudaSetDevice(c->device));
    k_ew_add_many_grouped<<<ew_grid(c, in->size * in->limbs, o->batch), 256, 0, (cudaStream_t)s>>>(
        dv(in), dv(o), groups, o->batch, in->limbs, c->n, c->t);
    LAUNCH_CHECK(c);
    return CKKS_OK;
}

extern "C" int ckks_is_transparent(ckks_ctx *c, const ckks_view *ct, int32_t *flags, ckks_stream s) {
    int rc;
    if ((rc = check_view(c, ct, "encrypted"))) return rc;
    if (!flags) return fail(CKKS_ERR_INVALID, "null flags");
    CU(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)s;
    k_fill_i32<<<(ct->batch + 255) / 256, 256, 0, st>>>(flags, ct->batch, 1);
    LAUNCH_CHECK(c);
    if (ct->size > 1) {
        k_transparent<<<ew_grid(c, (ct->size - 1) * ct->limbs, ct->batch), 256, 0, st>>>(dv(ct), flags, ct->limbs, c->n);
        LAUNCH_CHECK(c);
    }
    return CKKS_OK;
}

extern "C" int ckks_mod_switch_drop(ckks_ctx *c, const ckks_view *in, const ckks_view *o, ckks_stream s) {
    int rc;
    if ((rc = check_view(c, in, "in")) || (rc = check_view(c, o, "out"))) return rc;
    if (o->batch != in->batch || o->size != in->size || o->limbs >= in->limbs)
        return fail(CKKS_ERR_INVALID, "mod_switch: destination must sit lower in the modulus chain");
    if (o->data == in->data) {
        if (o->poly_stride == in->poly_stride && o->batch_stride == in->batch_stride) return CKKS_OK;  // metadata only
        return fail(CKKS_ERR_INVALID, "mod_switch: in-place only with identical strides");
    }
    CU(cudaSetDevice(c->device));
    k_ew_copy<<<ew_grid(c, o->size * o->limbs, o->batch), 256, 0, (cudaStream_t)s>>>(dv(in), dv(o), o->limbs, c->n);
    LAUNCH_CHECK(c);
    return CKKS_OK;
}

// ------------------------------------------------------------------------------------ key switching
extern "C" size_t ckks_ksk_words(const ckks_ctx *c) { return (size_t)(c->K - 1) * 2 * c->K * c->n; }
extern "C" uint64_t ckks_galois_elt_from_step(const ckks_ctx *c, int steps) { return ckks::galois_elt_from_step(c->log_n, steps); }

static int get_perm(ckks_ctx *c, uint64_t g, const uint32_t **out) {
    if (!(g & 1) || g >= 2ull * c->n) return fail(CKKS_ERR_INVALID, "Galois element is not valid");
    auto it = c->perms.find(g);
    if (it == c->perms.end()) {
        std::vector<uint32_t> h;
        ckks::build_galois_perm(c->log_n, g, h);
        uint32_t *d = nullptr;
        CU(cudaSetDevice(c->device));
        CU(cudaMalloc((void **)&d, h.size() * 4));
        CU(cudaMemcpy(d, h.data(), h.size() * 4, cudaMemcpyHostToDevice));
        it = c->perms.emplace(g, d).first;
    }
    *out = it->second;
    return CKKS_OK;
}

// nsplit of the fused column kernels: one CTA per tile does every target prime when the launch already fills the
// GPU (148 SMs x 4 resident CTAs); a small batch splits the targets over up to `maxsplit` CTAs per tile instead
static int pick_split(int forced, int tiles, int maxsplit) {
    (void)tiles;   // measured (profiles/r02_keyswitch_experiments.md): splitting never wins, not even at batch 4
    int ns = forced > 0 ? forced : 1;
    if (ns > maxsplit) ns = maxsplit;
    return ns < 1 ? 1 : ns;
}

// Batched key switch over `nslots` launch slots.
// mode 1: relinearize (target = poly 2 of the source, base = polys 0,1)
// mode 2: Galois      (target = permuted poly 1, base = permuted poly 0)
static int keyswitch(ckks_ctx *c, int mode, int L, int nslots, KsRoute rt, cudaStream_t st, bool chained = false, int li = 0, int slot0 = 0) {
    const int K = c->K;
    const size_t N = c->n;
    const int Bc = ks_chunk(c, nslots, L);
    int rc;
    if ((rc = ensure_lane(c, li, ks_words_per_ct(c, L) * 8 * (size_t)Bc))) return rc;
    ckks_ctx::Lane &ln = c->lane[li];
    u64 *D = ln.ws;
    u64 *T1 = D + (size_t)Bc * L * N;
    u64 *ACC = T1 + (size_t)Bc * L * (L + 1) * N;
    u64 *T2 = ACC + (size_t)Bc * 2 * (L + 1) * N;
    rt.tgt_poly = mode == 1 ? 2 : 1;
    // output limbs by prime size: integer kernel for large primes, FP64 kernel for small ones
    JjList big{}, small{};
    const int fuse = c->fuse;
    for (int jj = L; jj >= 0; jj--) {   // special-prime limb first: with the fused INTT its CTAs are the longest
        const int pj = jj == L ? K - 1 : jj;
        JjList &dst = (c->primes[pj] >> 41) == 0 ? small : big;
        dst.jj[dst.n++] = (signed char)jj;
    }
    const bool special_small = (c->primes[K - 1] >> 41) == 0;
    static const int ksplit_below = getenv("CKKS_KSPLIT_BELOW") ? atoi(getenv("CKKS_KSPLIT_BELOW")) : 3;
    // ciphertexts per launch below which the inner product runs as thread-block clusters over the digits (k_ks_mac_cl).
    // Measured (profiles/r02_keyswitch_experiments.md): for a single ciphertext (the reference's own sequential programs on
    // the shim) -10 % latency at N = 16384, L = 3 (-4 % at L = 2, N = 8192; -3 % at N = 4096), equal at N = 32768, +18 % with a
    // single digit, slower from two ciphertexts on -- hence the default below; CKKS_CLUSTER_BELOW=n forces it for every
    // launch of fewer than n ciphertexts at any degree and level.
    static const int cluster_env = getenv("CKKS_CLUSTER_BELOW") ? atoi(getenv("CKKS_CLUSTER_BELOW")) : -1;
    const int cluster_below = cluster_env >= 0 ? cluster_env : (c->log_n <= 14 && L >= 2 ? 2 : 0);
    for (int b0 = slot0; b0 < slot0 + nslots; b0 += Bc) {
        const int bc = (slot0 + nslots - b0) < Bc ? (slot0 + nslots - b0) : Bc;
        g_pdl_now = g_pdl_mode < 0 ? bc >= 8 : g_pdl_mode != 0;
        // one or two ciphertexts (the GPU is mostly empty, latency is what counts -- e.g. the reference's own sequential
        // programs on the shim): the special-prime limb's CTAs are the longest of the pipeline (L transforms + 2 INTT row
        // passes); split them by key component over two CTAs (-9 % at batch 2).  From batch 4 on every kernel already has
        // about one CTA per SM and extra CTAs only make the critical ones share an SM (+7 % at batch 4, measured).
        JjList bigl = big;
        if (fuse && !special_small && bc < ksplit_below && big.n > 0 && big.n < 35 && big.jj[0] == L) {
            for (int q = bigl.n; q > 0; q--) {
                bigl.jj[q] = bigl.jj[q - 1];
                bigl.kh[q] = bigl.kh[q - 1];
            }
            bigl.n++;
            bigl.kh[0] = 1;
            bigl.kh[1] = 2;
        }
        rt.b0 = b0;
        DView dD{D, (u64)L * N, 0};
        DView spec{ACC + (size_t)L * N, (u64)(L + 1) * N, 0};             // special-prime limb of every (b,k)
        DView minu{ACC, 2 * (u64)(L + 1) * N, (u64)(L + 1) * N};
#define RUN(LN)                                                                                                         \
    {                                                                                                                   \
        typedef NttGeo<LN> G;                                                                                           \
        /* the first kernel follows arbitrary stream work (copies, foreign kernels): ordinary launch unless  \
           the caller chains key switches back to back */                                                      \
        if (chained && mode == 2) launch_pdl(k_ks_intt_row<LN, true>, dim3(G::ROW_TILES, L, bc), st, rt, D, L, c->t); \
        else if (mode == 2) k_ks_intt_row<LN, true><<<dim3(G::ROW_TILES, L, bc), NTT_THREADS, 0, st>>>(rt, D, L, c->t); \
        else k_ks_intt_row<LN, false><<<dim3(G::ROW_TILES, L, bc), NTT_THREADS, 0, st>>>(rt, D, L, c->t);       \
        LAUNCH_CHECK(c);                                                                                                \
        if (fuse) {                                                                                                     \
            const int ns1 = pick_split(c->split1, G::COL_TILES * L * bc, L);                                            \
            launch_pdl(k_ks_invcol_modup<LN>, dim3(G::COL_TILES, L * ns1, bc), st, D, T1, L, ns1, c->t);                \
            LAUNCH_CHECK(c);                                                                                            \
        } else {                                                                                                        \
            launch_pdl(k_inv_col<LN, false>, dim3(G::COL_TILES, L, bc), st, dD, dD, L, 0, c->t);                \
            LAUNCH_CHECK(c);                                                                                            \
            launch_pdl(k_ks_modup_col<LN>, dim3(G::COL_TILES, L *(L + 1), bc), st, D, T1, L, c->t);             \
            LAUNCH_CHECK(c);                                                                                            \
        }                                                                                                               \
        /* the FP64 inner product (small-prime limbs) is independent of the integer one and of the special-prime  \
           INTT that follows: fork it onto the side stream, join before the last kernel reads its output */       \
        const bool use_cl = fuse && bc < cluster_below && L <= 8 && (long)(L + 1) * bc <= 65535;                       \
        cudaStream_t sfp = (big.n && small.n && !use_cl) ? ln.side : st;                                               \
        if (use_cl) {                                                                                                   \
            /* small batch: one cluster of L CTAs per output tile (k_ks_mac_cl), integer and FP64 limbs in one launch */ \
            if (mode == 2) CU(launch_cluster(k_ks_mac_cl<LN, true>, dim3(L, G::ROW_TILES, (L + 1) * bc), 65536, st, T1, rt, ACC, L, fuse, c->t)); \
            else CU(launch_cluster(k_ks_mac_cl<LN, false>, dim3(L, G::ROW_TILES, (L + 1) * bc), 65536, st, T1, rt, ACC, L, fuse, c->t)); \
            LAUNCH_CHECK(c);                                                                                            \
        }                                                                                                               \
        if (small.n && !use_cl) {                                                                                                  \
            if (sfp != st) {                                                                                            \
                CU(cudaEventRecord(ln.fork, st));                                                                       \
                CU(cudaStreamWaitEvent(sfp, ln.fork, 0));                                                               \
            }                                                                                                           \
            if (mode == 2) k_ks_mac_fp<LN, true><<<dim3(G::ROW_TILES, small.n, bc), NTT_THREADS, 0, sfp>>>(T1, rt, ACC, L, small, fuse, c->t); \
            else k_ks_mac_fp<LN, false><<<dim3(G::ROW_TILES, small.n, bc), NTT_THREADS, 0, sfp>>>(T1, rt, ACC, L, small, fuse, c->t); \
            LAUNCH_CHECK(c);                                                                                            \
            if (sfp != st) CU(cudaEventRecord(ln.join, sfp));                                                           \
        }                                                                                                               \
        if (big.n && !use_cl) {                                                                                         \
            if (mode == 2) launch_pdl(k_ks_mac<LN, true>, dim3(G::ROW_TILES, bigl.n, bc), st, T1, rt, ACC, L, bigl, fuse, c->t); \
            else launch_pdl(k_ks_mac<LN, false>, dim3(G::ROW_TILES, bigl.n, bc), st, T1, rt, ACC, L, bigl, fuse, c->t);   \
            LAUNCH_CHECK(c);                                                                                            \
        }                                                                                                               \
        /* a small special prime puts its limb on the side stream: the INTT below must wait for it */            \
        if (sfp != st && special_small) CU(cudaStreamWaitEvent(st, ln.join, 0));                                        \
        if (fuse) {                                                                                                     \
            const int ns3 = pick_split(c->split3, G::COL_TILES * 2 * bc, L);                                            \
            launch_pdl(k_md_invcol_fwdcol<LN>, dim3(G::COL_TILES, ns3, 2 * bc), st, spec, T2, L, K - 1, ns3, c->t);     \
            LAUNCH_CHECK(c);                                                                                            \
        } else {                                                                                                        \
            launch_pdl(k_inv_row<LN>, dim3(G::ROW_TILES, 1, 2 * bc), st, spec, spec, 1, K - 1, c->t);           \
            LAUNCH_CHECK(c);                                                                                            \
            launch_pdl(k_inv_col<LN, true>, dim3(G::COL_TILES, 1, 2 * bc), st, spec, spec, 1, K - 1, c->t);     \
            LAUNCH_CHECK(c);                                                                                            \
            launch_pdl(k_md_fwd_col<LN>, dim3(G::COL_TILES, L, 2 * bc), st, spec, T2, L, K - 1, c->t);          \
            LAUNCH_CHECK(c);                                                                                            \
        }                                                                                                               \
        if (sfp != st && !special_small) CU(cudaStreamWaitEvent(st, ln.join, 0));                                       \
        if (mode == 2) launch_pdl(k_md_fwd_row<LN, 2>, dim3(G::ROW_TILES, L, 2 * bc), st, T2, minu, rt, 2, L, K - 1, c->t); \
        else launch_pdl(k_md_fwd_row<LN, 1>, dim3(G::ROW_TILES, L, 2 * bc), st, T2, minu, rt, 2, L, K - 1, c->t); \
        LAUNCH_CHECK(c);                                                                                                \
    }
        DISPATCH_LOGN(c, RUN)
#undef RUN
    }
    return CKKS_OK;
}

// the engine-owned tiled copy of a registered key, or the caller's buffer (standard layout) for an unregistered one
static const u64 *resolve_key(const ckks_ctx *c, const uint64_t *key, int *tiled) {
    auto it = c->tiled_keys.find(key);
    if (it == c->tiled_keys.end()) {
        *tiled = 0;
        return (const u64 *)key;
    }
    *tiled = 1;
    return it->second.copy;
}

static KsRoute uniform_route(const ckks_ctx *c, const ckks_view *in, const ckks_view *out, const uint32_t *perm, const uint64_t *key) {
    KsRoute rt{};
    rt.v[0] = dv(in);
    rt.v[1] = dv(out);
    rt.v[2] = dv(out);
    rt.perm0 = perm;
    rt.key0 = resolve_key(c, key, &rt.key_tiled);
    return rt;
}

// A batch of 16 or more key switches is split into two halves that run as concurrent pipelines on the
// lanes' streams (fork/join with events on the caller's stream): the short kernels of one half overlap
// the long kernels of the other.
static int keyswitch_lanes(ckks_ctx *c, int mode, int L, int nslots, const KsRoute &rt, cudaStream_t st) {
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(st, &cap);
    if (nslots < 16 || c->chain_lanes < 2 || cap != cudaStreamCaptureStatusNone) return keyswitch(c, mode, L, nslots, rt, st);
    int rc;
    const int half = nslots / 2;
    for (int li = 0; li < 2; li++) {
        const int cnt = li == 0 ? half : nslots - half;
        if ((rc = ensure_lane(c, li, ks_words_per_ct(c, L) * 8 * (size_t)ks_chunk(c, cnt, L)))) return rc;
    }
    if (!c->ev_in) {
        CU(cudaEventCreateWithFlags(&c->ev_in, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&c->ev_out, cudaEventDisableTiming));
    }
    CU(cudaEventRecord(c->ev_in, st));
    for (int li = 0; li < 2; li++) {
        ckks_ctx::Lane &ln = c->lane[li];
        CU(cudaStreamWaitEvent(ln.main, c->ev_in, 0));
        if ((rc = keyswitch(c, mode, L, li == 0 ? half : nslots - half, rt, ln.main, false, li, li == 0 ? 0 : half))) return rc;
        CU(cudaEventRecord(ln.end, ln.main));
        CU(cudaStreamWaitEvent(st, ln.end, 0));
    }
    return CKKS_OK;
}

extern "C" int ckks_relinearize(ckks_ctx *c, const ckks_view *in, const uint64_t *rlk, const ckks_view *out, ckks_stream s) {
    int rc;
    if ((rc = check_view(c, in, "encrypted")) || (rc = check_view(c, out, "out"))) return rc;
    if (!rlk) return fail(CKKS_ERR_INVALID, "relin_keys is not valid for encryption parameters");
    if (in->limbs > c->K - 1) return fail(CKKS_ERR_INVALID, "encrypted is not valid for encryption parameters");
    if (in->size != 3) return fail(CKKS_ERR_INVALID, "relinearize: only size-3 ciphertexts are supported");
    if (out->size != 2 || out->batch != in->batch || out->limbs != in->limbs) return fail(CKKS_ERR_INVALID, "destination parameter mismatch");
    if (out->data == in->data && (out->poly_stride != in->poly_stride || out->batch_stride != in->batch_stride))
        return fail(CKKS_ERR_INVALID, "relinearize: in-place only with identical strides");
    CU(cudaSetDevice(c->device));
    return keyswitch_lanes(c, 1, in->limbs, in->batch, uniform_route(c, in, out, nullptr, rlk), (cudaStream_t)s);
}

extern "C" int ckks_apply_galois(ckks_ctx *c, const ckks_view *in, uint64_t g, const uint64_t *gk, const ckks_view *out, ckks_stream s) {
    int rc;
    if ((rc = check_view(c, in, "encrypted")) || (rc = check_view(c, out, "out"))) return rc;
    if (!gk) return fail(CKKS_ERR_INVALID, "Galois key not present");
    if (in->limbs > c->K - 1) return fail(CKKS_ERR_INVALID, "encrypted is not valid for encryption parameters");
    if (in->size != 2) return fail(CKKS_ERR_INVALID, "encrypted size must be 2");
    if ((rc = same_shape(in, out, "destination"))) return rc;
    if (out->data == in->data) return fail(CKKS_ERR_INVALID, "apply_galois: out must not alias in");
    const uint32_t *perm = nullptr;
    if ((rc = get_perm(c, g, &perm))) return rc;
    CU(cudaSetDevice(c->device));
    return keyswitch_lanes(c, 2, in->limbs, in->batch, uniform_route(c, in, out, perm, gk), (cudaStream_t)s);
}

extern "C" int ckks_keyset_create(ckks_ctx *c, ckks_keyset **out) {
    if (!c || !out) return fail(CKKS_ERR_INVALID, "null argument");
    *out = new ckks_keyset{c};
    c->keysets.push_back(*out);
    return CKKS_OK;
}
// Registration captures the key: a private copy in the tiled layout the inner-product kernels read fastest
// (k_retile_key).  The copy lives while some keyset references the caller's pointer; entry points that receive
// that pointer directly (ckks_relinearize, ckks_apply_galois) find it through the context's registry.
static int register_key(ckks_ctx *c, const uint64_t *key) {
    if (!key) return fail(CKKS_ERR_INVALID, "null key");
    if ((uintptr_t)key & 15) return fail(CKKS_ERR_INVALID, "key must be 16-byte aligned");
    CU(cudaSetDevice(c->device));
    ckks_ctx::TiledKey &t = c->tiled_keys[key];
    const size_t words = ckks_ksk_words(c);
    if (!t.copy && cudaMalloc((void **)&t.copy, words * 8) != cudaSuccess) {
        cudaGetLastError();
        c->tiled_keys.erase(key);
        return fail(CKKS_ERR_NOMEM, "device allocation failed");
    }
    t.refs++;
    // Registration is a set-up step, not a hot-path call, and it is SYNCHRONOUS with respect to every stream: the caller's
    // key buffer may have been produced on any (non-blocking) stream and the first key switch may run on any other, so
    // the device is drained before the capture and the capture is complete on return.
    CU(cudaDeviceSynchronize());
    k_retile_key<<<(unsigned)(words / NTT_TILE), NTT_THREADS>>>((const u64 *)key, t.copy, c->log_n, c->t);   // (re)capture the contents
    LAUNCH_CHECK(c);
    CU(cudaDeviceSynchronize());
    return CKKS_OK;
}
static void unregister_key(ckks_ctx *c, const uint64_t *key) {
    auto it = c->tiled_keys.find(key);
    if (it == c->tiled_keys.end() || --it->second.refs > 0) return;
    cudaSetDevice(c->device);
    cudaFree(it->second.copy);   // synchronises: no kernel still reads the copy
    c->tiled_keys.erase(it);
    for (auto &kv : c->chain_graphs) cudaGraphExecDestroy(kv.second.exec);   // cached graphs may hold the freed address
    c->chain_graphs.clear();
}

extern "C" void ckks_keyset_destroy(ckks_keyset *ks) {
    if (!ks) return;
    if (ks->ctx) {   // (a context destroyed before its keysets has already released the copies)
        if (ks->relin) unregister_key(ks->ctx, ks->relin);
        for (auto &kv : ks->galois) unregister_key(ks->ctx, kv.second);
        auto &v = ks->ctx->keysets;
        for (size_t i = 0; i < v.size(); i++)
            if (v[i] == ks) {
                v.erase(v.begin() + i);
                break;
            }
    }
    cudaFree((void *)ks->d_perm_tab);
    cudaFree((void *)ks->d_key_tab);
    delete ks;
}
extern "C" int ckks_keyset_set_relin(ckks_keyset *ks, const uint64_t *rlk) {
    int rc = register_key(ks->ctx, rlk);
    if (rc) return rc;
    if (ks->relin) unregister_key(ks->ctx, ks->relin);
    ks->relin = rlk;
    return CKKS_OK;
}
extern "C" int ckks_keyset_set_galois(ckks_keyset *ks, uint64_t g, const uint64_t *gk) {
    const uint32_t *perm = nullptr;
    int rc = get_perm(ks->ctx, g, &perm);  // build the permutation table now (not capturable later)
    if (rc) return rc;
    if ((rc = register_key(ks->ctx, gk))) return rc;
    auto old = ks->galois.find(g);
    if (old != ks->galois.end()) unregister_key(ks->ctx, old->second);
    ks->galois[g] = gk;
    if (!ks->slot_of.count(g)) {
        ks->slot_of[g] = (int)ks->slot_elt.size();
        ks->slot_elt.push_back(g);
    }
    ks->tab_dirty = true;
    return CKKS_OK;
}
extern "C" int ckks_keyset_has_galois(const ckks_keyset *ks, uint64_t g) { return ks->galois.count(g) ? 1 : 0; }

extern "C" int ckks_rotate(ckks_ctx *c, const ckks_keyset *ks, const ckks_view *in, int steps, const ckks_view *out,
                           const ckks_view *scratch, ckks_stream s) {
    int rc;
    if (!ks) return fail(CKKS_ERR_INVALID, "null keyset");
    if ((rc = check_view(c, in, "encrypted")) || (rc = check_view(c, out, "out")) || (rc = same_shape(in, out, "destination"))) return rc;
    if (steps == 0) {  // SEAL: rotate by 0 returns the input unchanged
        CU(cudaSetDevice(c->device));
        k_ew_copy<<<ew_grid(c, in->size * in->limbs, in->batch), 256, 0, (cudaStream_t)s>>>(dv(in), dv(out), in->limbs, c->n);
        LAUNCH_CHECK(c);
        return CKKS_OK;
    }
    uint64_t g = ckks::galois_elt_from_step(c->log_n, steps);
    if (!g) return fail(CKKS_ERR_INVALID, "step count too large");
    auto it = ks->galois.find(g);
    if (it != ks->galois.end()) return ckks_apply_galois(c, in, g, it->second, out, s);
    // SEAL Evaluator::rotate_internal: NAF decomposition, terms applied least-significant first
    std::vector<int> terms = ckks::naf_terms(steps), eff;
    if (terms.size() == 1) return fail(CKKS_ERR_INVALID, "Galois key not present");
    for (int tstep : terms)
        if ((tstep < 0 ? -tstep : tstep) != c->n / 2) eff.push_back(tstep);
    for (int tstep : eff) {
        uint64_t gt = ckks::galois_elt_from_step(c->log_n, tstep);
        if (!gt || !ks->galois.count(gt)) return fail(CKKS_ERR_INVALID, "Galois key not present");
    }
    if (eff.size() > 1) {
        if ((rc = check_view(c, scratch, "scratch")) || (rc = same_shape(in, scratch, "scratch"))) return rc;
        if (scratch->data == in->data || scratch->data == out->data) return fail(CKKS_ERR_INVALID, "scratch must be distinct storage");
    }
    const ckks_view *cur = in;
    for (size_t i = 0; i < eff.size(); i++) {
        const ckks_view *dstv = ((eff.size() - 1 - i) % 2 == 0) ? out : scratch;
        uint64_t gt = ckks::galois_elt_from_step(c->log_n, eff[i]);
        if ((rc = ckks_apply_galois(c, cur, gt, ks->galois.at(gt), dstv, s))) return rc;
        cur = dstv;
    }
    return CKKS_OK;
}

// ------------------------------------------------------------------------------------ rotate-and-sum chain
// `count` iterations of   dup = rotate_vector(dup, steps);  acc += dup   (cipher_dot_product's loop,
// helper.h:472-476) on a batch of independent ciphertexts.  The rotation ping-pongs between the
// views a and b (a holds dup on entry); the add is fused into the key switch's last kernel; two
// steps (a->b, b->a) are captured once into a CUDA graph and replayed, so the dependent chain costs
// one graph launch per two key switches instead of 18 kernel launches.
extern "C" int ckks_rotate_sum_chain(ckks_ctx *c, const ckks_keyset *ks, const ckks_view *a, const ckks_view *b,
                                     const ckks_view *acc, int steps, int count, int *final_in_b, ckks_stream s) {
    int rc;
    if (!ks) return fail(CKKS_ERR_INVALID, "null keyset");
    if ((rc = check_view(c, a, "a")) || (rc = check_view(c, b, "b")) || (rc = check_view(c, acc, "acc"))) return rc;
    if ((rc = same_shape(a, b, "b")) || (rc = same_shape(a, acc, "acc"))) return rc;
    if (a->size != 2) return fail(CKKS_ERR_INVALID, "encrypted size must be 2");
    if (a->limbs > c->K - 1) return fail(CKKS_ERR_INVALID, "encrypted is not valid for encryption parameters");
    if (a->data == b->data || a->data == acc->data || b->data == acc->data) return fail(CKKS_ERR_INVALID, "a, b and acc must be distinct storage");
    if (count < 0) return fail(CKKS_ERR_INVALID, "negative count");
    uint64_t g = ckks::galois_elt_from_step(c->log_n, steps);
    if (!g) return fail(CKKS_ERR_INVALID, "step count too large");
    auto it = ks->galois.find(g);
    if (it == ks->galois.end()) return fail(CKKS_ERR_INVALID, "Galois key not present");
    const uint32_t *perm = nullptr;
    if ((rc = get_perm(c, g, &perm))) return rc;
    CU(cudaSetDevice(c->device));
    const int L = a->limbs, B = a->batch;
    if ((rc = ensure_ws(c, ks_words_per_ct(c, L) * 8 * (size_t)ks_chunk(c, B, L)))) return rc;
    cudaStream_t user = (cudaStream_t)s;
    // one step on the batch entries [off, off+cnt) through lane `li`
    auto one = [&](const ckks_view *src, const ckks_view *dst, cudaStream_t st, bool chained, int li, int off, int cnt) -> int {
        ckks_view vs = *src, vd = *dst, va = *acc;
        vs.data += (uint64_t)off * vs.batch_stride;
        vd.data += (uint64_t)off * vd.batch_stride;
        va.data += (uint64_t)off * va.batch_stride;
        vs.batch = vd.batch = va.batch = cnt;
        KsRoute rt = uniform_route(c, &vs, &vd, perm, it->second);
        rt.accv = dv(&va);
        rt.has_acc = 1;
        return keyswitch(c, 2, L, cnt, rt, st, chained, li);
    };
    int done = 0;
    if (count >= 4) {
        // two half-batches run as independent pipelines (lanes) on their own streams: the short kernels of
        // one lane (special-prime INTT: 1-2 waves) overlap the long ones of the other.  Each lane replays a
        // cached CUDA graph of ping-pong steps; the lanes only meet again at the end of the chain.
        int nl = c->chain_lanes;
        static const int lane_min = getenv("CKKS_LANE_MIN") ? atoi(getenv("CKKS_LANE_MIN")) : 0;   // ciphertexts per lane (0 = rule below)
        while (nl > 1 && B / nl < (lane_min > 0 ? lane_min : 8)) nl--;
        // small batches (the strong-scaling regime: 4 / 8 chains per GPU): lanes of TWO ciphertexts -- each lane's launches then
        // take the split special-prime inner product and the lanes fill the GPU side by side.  Measured per chain step at
        // N = 32768, L = 3: batch 4: 58.9 us (2 x 2) against 63.6 (one lane) and 62.3 (4 x 1); batch 8: 86.6 us (4 x 2) against
        // 92.6 (one lane) and 95.9 (2 x 4); batch 16: 133.8 (2 x 8) against 137.5 (4 x 4); batch 2: one lane.
        if (lane_min == 0 && c->chain_lanes >= 2 && B >= 4 && B <= 8 && B % 2 == 0) nl = B / 2;
        int split[5];
        for (int li = 0; li <= nl; li++) split[li] = (int)((long)B * li / nl);
        if (!c->ev_in) {
            CU(cudaEventCreateWithFlags(&c->ev_in, cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&c->ev_out, cudaEventDisableTiming));
        }
        // graphs of 1 and of CHAIN_GRAPH_PAIRS ping-pong pairs per lane: a long chain replays the big one (one graph launch
        // per 2 * CHAIN_GRAPH_PAIRS dependent steps -- fewer launch gaps between graphs, less host work), the remainder
        // the small one
        const int pairs = count / 2;
        static const int big_pairs = getenv("CKKS_CHAIN_GRAPH_PAIRS") ? atoi(getenv("CKKS_CHAIN_GRAPH_PAIRS")) : 8;
        cudaGraphExec_t execs[2][4] = {{nullptr, nullptr, nullptr, nullptr}, {nullptr, nullptr, nullptr, nullptr}};
        uint64_t per_graph[2] = {0, 0};
        const int gp[2] = {1, big_pairs > 1 && pairs >= big_pairs ? big_pairs : 0};
        for (int which = 0; which < 2; which++) {
            if (!gp[which]) continue;
            for (int li = 0; li < nl; li++) {
                const int off = split[li], cnt = split[li + 1] - split[li];
                if ((rc = ensure_lane(c, li, ks_words_per_ct(c, L) * 8 * (size_t)ks_chunk(c, cnt, L)))) return rc;
                ckks_ctx::Lane &ln = c->lane[li];
                int key_tiled = 0;
                std::vector<uint64_t> key = {(uint64_t)a->data, (uint64_t)b->data, (uint64_t)acc->data, (uint64_t)resolve_key(c, it->second, &key_tiled), g,
                                             (uint64_t)L, (uint64_t)off, (uint64_t)cnt, a->batch_stride, a->poly_stride, b->batch_stride,
                                             b->poly_stride, acc->batch_stride, acc->poly_stride, (uint64_t)ln.ws, (uint64_t)c->t.round_half,
                                             (uint64_t)gp[which]};
                auto gi = c->chain_graphs.find(key);
                if (gi == c->chain_graphs.end()) {
                    cudaGraph_t graph = nullptr;
                    uint64_t before = c->launches;
                    CU(cudaStreamBeginCapture(ln.main, cudaStreamCaptureModeThreadLocal));
                    for (int q = 0; q < gp[which] && !rc; q++) {
                        rc = one(a, b, ln.main, q > 0, li, off, cnt);
                        if (!rc) rc = one(b, a, ln.main, true, li, off, cnt);
                    }
                    cudaError_t ce = cudaStreamEndCapture(ln.main, &graph);
                    uint64_t per = c->launches - before;
                    c->launches = before;
                    if (rc) return rc;
                    if (ce != cudaSuccess) return fail(CKKS_ERR_CUDA, std::string("graph capture: ") + cudaGetErrorString(ce));
                    ckks_ctx::ChainGraph cg{};
                    cg.launches = per;
                    ce = cudaGraphInstantiate(&cg.exec, graph, 0);
                    cudaGraphDestroy(graph);
                    if (ce != cudaSuccess) return fail(CKKS_ERR_CUDA, std::string("graph instantiate: ") + cudaGetErrorString(ce));
                    if (c->chain_graphs.size() > 64) {   // bounded cache (graphs of this call are re-created on demand)
                        for (auto &kv : c->chain_graphs) cudaGraphExecDestroy(kv.second.exec);
                        c->chain_graphs.clear();
                        for (auto &row : execs)
                            for (auto &e : row) e = nullptr;
                        which = -1;                   // start over: earlier handles of this call were just destroyed
                        per_graph[0] = per_graph[1] = 0;
                        cudaGraphExecDestroy(cg.exec);
                        break;
                    }
                    gi = c->chain_graphs.emplace(key, cg).first;
                }
                execs[which][li] = gi->second.exec;
                per_graph[which] += gi->second.launches;
            }
        }
        CU(cudaEventRecord(c->ev_in, user));
        for (int li = 0; li < nl; li++) CU(cudaStreamWaitEvent(c->lane[li].main, c->ev_in, 0));
        int left = pairs;
        if (gp[1])
            for (; left >= gp[1]; left -= gp[1]) {
                for (int li = 0; li < nl; li++) CU(cudaGraphLaunch(execs[1][li], c->lane[li].main));
                c->launches += per_graph[1];
            }
        for (; left > 0; left--) {
            for (int li = 0; li < nl; li++) CU(cudaGraphLaunch(execs[0][li], c->lane[li].main));
            c->launches += per_graph[0];
        }
        for (int li = 0; li < nl; li++) {
            CU(cudaEventRecord(c->lane[li].end, c->lane[li].main));
            CU(cudaStreamWaitEvent(user, c->lane[li].end, 0));
        }
        done = pairs * 2;
    }
    const ckks_view *src = a, *dst = b;
    for (; done < count; done++) {
        if ((rc = one(src, dst, user, false, 0, 0, B))) return rc;
        const ckks_view *t = src;
        src = dst;
        dst = t;
    }
    if (final_in_b) *final_in_b = (src == b) ? 1 : 0;
    return CKKS_OK;
}

// ------------------------------------------------------------------------------------ rotation plans
static int sync_key_tables(ckks_keyset *ks) {
    if (!ks->tab_dirty) return CKKS_OK;
    ckks_ctx *c = ks->ctx;
    CU(cudaSetDevice(c->device));
    const int n = (int)ks->slot_elt.size();
    if (n > ks->tab_cap) {
        CU(cudaDeviceSynchronize());
        cudaFree((void *)ks->d_perm_tab);
        cudaFree((void *)ks->d_key_tab);
        ks->tab_cap = n + 32;
        CU(cudaMalloc((void **)&ks->d_perm_tab, sizeof(void *) * ks->tab_cap));
        CU(cudaMalloc((void **)&ks->d_key_tab, sizeof(void *) * ks->tab_cap));
    }
    std::vector<const uint32_t *> hp(n);
    std::vector<const u64 *> hk(n);
    for (int i = 0; i < n; i++) {
        int rc = get_perm(c, ks->slot_elt[i], &hp[i]);
        if (rc) return rc;
        int tiled = 0;
        hk[i] = resolve_key(c, ks->galois.at(ks->slot_elt[i]), &tiled);   // registered keys: always the tiled copy
    }
    if (n) {
        CU(cudaMemcpy((void *)ks->d_perm_tab, hp.data(), sizeof(void *) * n, cudaMemcpyHostToDevice));
        CU(cudaMemcpy((void *)ks->d_key_tab, hk.data(), sizeof(void *) * n, cudaMemcpyHostToDevice));
    }
    ks->tab_dirty = false;
    return CKKS_OK;
}

// SEAL Evaluator::rotate_internal: the key for `steps` itself if present, else the NAF terms
static int rotation_terms(const ckks_ctx *c, const ckks_keyset *ks, int steps, std::vector<int> &terms) {
    terms.clear();
    if (steps == 0) return CKKS_OK;
    uint64_t g = ckks::galois_elt_from_step(c->log_n, steps);
    if (!g) return fail(CKKS_ERR_INVALID, "step count too large");
    if (ks->galois.count(g)) {
        terms.push_back(steps);
        return CKKS_OK;
    }
    std::vector<int> naf = ckks::naf_terms(steps);
    if (naf.size() == 1) return fail(CKKS_ERR_INVALID, "Galois key not present");
    for (int tstep : naf) {
        if ((tstep < 0 ? -tstep : tstep) == c->n / 2) continue;
        uint64_t gt = ckks::galois_elt_from_step(c->log_n, tstep);
        if (!gt || !ks->galois.count(gt)) return fail(CKKS_ERR_INVALID, "Galois key not present");
        terms.push_back(tstep);
    }
    return CKKS_OK;
}

extern "C" int ckks_rotplan_create(ckks_ctx *c, ckks_keyset *ks, const int *steps, int batch, ckks_rotplan **out) {
    if (!c || !ks || !steps || !out || batch < 1) return fail(CKKS_ERR_INVALID, "rotplan: bad arguments");
    int rc;
    if ((rc = sync_key_tables(ks))) return rc;
    std::vector<std::vector<int>> terms(batch);
    size_t rounds = 0;
    ckks_rotplan *p = new ckks_rotplan;
    p->ctx = c;
    p->ks = ks;
    p->batch = batch;
    for (int b = 0; b < batch; b++) {
        if ((rc = rotation_terms(c, ks, steps[b], terms[b]))) {
            delete p;
            return rc;
        }
        if (terms[b].empty()) p->zero_entries.push_back(b);
        if (terms[b].size() > rounds) rounds = terms[b].size();
        p->keyswitches += terms[b].size();
    }
    std::vector<KsSel> sel;
    for (size_t r = 0; r < rounds; r++) {
        p->round_off.push_back((int)sel.size());
        for (int b = 0; b < batch; b++) {
            const int m = (int)terms[b].size();
            if ((size_t)m <= r) continue;
            KsSel e;
            e.entry = e.sentry = b;
            e.slot = ks->slot_of.at(ckks::galois_elt_from_step(c->log_n, terms[b][r]));
            e.src = (short)(r == 0 ? 0 : (((m - (int)r) % 2 == 0) ? 1 : 2));
            e.dst = (short)(((m - 1 - (int)r) % 2 == 0) ? 1 : 2);
            sel.push_back(e);
        }
        p->round_cnt.push_back((int)sel.size() - p->round_off.back());
    }
    // shared-prefix form: a trie over the NAF term sequences
    struct Node {
        int parent, term, depth, view, entry;
        std::map<int, int> kids;
    };
    std::vector<Node> nodes(1, Node{-1, 0, 0, 0, 0, {}});
    std::vector<KsSel> sh;
    int next_tmp = 0;
    bool shared_ok = batch > 1 && rounds > 1;
    for (int b = 0; b < batch && shared_ok; b++) {
        int cur = 0;
        for (size_t r = 0; r < terms[b].size(); r++) {
            auto it = nodes[cur].kids.find(terms[b][r]);
            if (it == nodes[cur].kids.end()) {
                nodes.push_back(Node{cur, terms[b][r], (int)r + 1, -1, -1, {}});
                nodes[cur].kids[terms[b][r]] = (int)nodes.size() - 1;
                cur = (int)nodes.size() - 1;
            } else {
                cur = it->second;
            }
        }
        if (cur == 0) continue;                       // rotate by 0: copied from the input
        if (nodes[cur].view == 1) p->sh_copies.push_back({nodes[cur].entry, b});   // the same step twice
        else nodes[cur].view = 1, nodes[cur].entry = b;
    }
    for (size_t q = 1; q < nodes.size() && shared_ok; q++)
        if (nodes[q].view < 0) {
            nodes[q].view = 2;
            nodes[q].entry = next_tmp++;
            if (next_tmp > batch) shared_ok = false;  // more pure intermediates than scratch entries: keep the plain form
        }
    if (shared_ok && nodes.size() - 1 < p->keyswitches) {
        for (size_t r = 1; r <= rounds; r++) {
            p->sh_round_off.push_back((int)sh.size());
            for (size_t q = 1; q < nodes.size(); q++) {
                if ((size_t)nodes[q].depth != r) continue;
                const Node &par = nodes[nodes[q].parent];
                KsSel e;
                e.entry = nodes[q].entry;
                e.slot = ks->slot_of.at(ckks::galois_elt_from_step(c->log_n, nodes[q].term));
                e.src = (short)(nodes[q].parent == 0 ? 0 : par.view);
                e.dst = (short)nodes[q].view;
                e.sentry = nodes[q].parent == 0 ? 0 : par.entry;
                sh.push_back(e);
            }
            p->sh_round_cnt.push_back((int)sh.size() - p->sh_round_off.back());
        }
        p->keyswitches_shared = sh.size();
    } else {
        p->sh_copies.clear();
        p->keyswitches_shared = p->keyswitches;
    }
    if (!sel.empty()) {
        if (cudaSetDevice(c->device) != cudaSuccess || cudaMalloc((void **)&p->d_sel, sel.size() * sizeof(KsSel)) != cudaSuccess ||
            cudaMemcpy(p->d_sel, sel.data(), sel.size() * sizeof(KsSel), cudaMemcpyHostToDevice) != cudaSuccess ||
            (!sh.empty() && (cudaMalloc((void **)&p->d_sel_sh, sh.size() * sizeof(KsSel)) != cudaSuccess ||
                             cudaMemcpy(p->d_sel_sh, sh.data(), sh.size() * sizeof(KsSel), cudaMemcpyHostToDevice) != cudaSuccess))) {
            ckks_rotplan_destroy(p);
            return fail(CKKS_ERR_CUDA, "rotplan: device allocation failed");
        }
    }
    *out = p;
    return CKKS_OK;
}
extern "C" void ckks_rotplan_destroy(ckks_rotplan *p) {
    if (!p) return;
    cudaFree(p->d_sel);
    cudaFree(p->d_sel_sh);
    delete p;
}
extern "C" uint64_t ckks_rotplan_keyswitches(const ckks_rotplan *p) { return p->keyswitches; }
extern "C" uint64_t ckks_rotplan_keyswitches_shared(const ckks_rotplan *p) { return p->keyswitches_shared; }
extern "C" int ckks_rotplan_rounds(const ckks_rotplan *p) { return (int)p->round_cnt.size(); }

extern "C" int ckks_rotate_plan(ckks_ctx *c, const ckks_rotplan *p, const ckks_view *in, const ckks_view *out,
                                const ckks_view *scratch, ckks_stream s) {
    int rc;
    if (!p) return fail(CKKS_ERR_INVALID, "null plan");
    if ((rc = check_view(c, in, "encrypted")) || (rc = check_view(c, out, "out"))) return rc;
    if (in->size != 2 || out->size != 2) return fail(CKKS_ERR_INVALID, "encrypted size must be 2");
    if (in->limbs > c->K - 1) return fail(CKKS_ERR_INVALID, "encrypted is not valid for encryption parameters");
    if (out->batch != p->batch || out->limbs != in->limbs || (in->batch != p->batch && in->batch != 1))
        return fail(CKKS_ERR_INVALID, "rotate_plan: batch/level mismatch");
    if (out->data == in->data) return fail(CKKS_ERR_INVALID, "rotate_plan: out must not alias in");
    const bool need_scratch = p->round_cnt.size() > 1;
    if (need_scratch) {
        if ((rc = check_view(c, scratch, "scratch")) || (rc = same_shape(out, scratch, "scratch"))) return rc;
        if (scratch->data == in->data || scratch->data == out->data) return fail(CKKS_ERR_INVALID, "scratch must be distinct storage");
    }
    CU(cudaSetDevice(c->device));
    // a Galois key replaced after the plan was compiled has a new engine-owned copy: refresh the device-side key table
    // (no-op unless the keyset changed) and make sure every key the plan selects is still registered
    if ((rc = sync_key_tables(p->ks))) return rc;
    cudaStream_t st = (cudaStream_t)s;
    KsRoute rt{};
    rt.v[0] = dv(in);
    if (in->batch == 1) rt.v[0].bs = 0;   // one input ciphertext shared by every rotation
    rt.v[1] = dv(out);
    rt.v[2] = need_scratch ? dv(scratch) : dv(out);
    rt.perm_tab = p->ks->d_perm_tab;
    rt.key_tab = p->ks->d_key_tab;
    rt.key_tiled = 1;
    for (int b : p->zero_entries) {   // rotate by 0: SEAL returns the input unchanged
        DView src = rt.v[0], dst = rt.v[1];
        src.data += (u64)b * src.bs;
        dst.data += (u64)b * dst.bs;
        k_ew_copy<<<ew_grid(c, 2 * in->limbs, 1), 256, 0, st>>>(src, dst, in->limbs, c->n);
        LAUNCH_CHECK(c);
    }
    static const bool share = !(getenv("CKKS_ROT_SHARE") && atoi(getenv("CKKS_ROT_SHARE")) == 0);
    if (share && in->batch == 1 && p->d_sel_sh) {   // one input ciphertext: rotations share their common NAF prefixes
        for (size_t r = 0; r < p->sh_round_cnt.size(); r++) {
            rt.sel = p->d_sel_sh + p->sh_round_off[r];
            if ((rc = keyswitch_lanes(c, 2, in->limbs, p->sh_round_cnt[r], rt, st))) return rc;
        }
        for (const auto &cp : p->sh_copies) {
            DView src = rt.v[1], dst = rt.v[1];
            src.data += (u64)cp.first * src.bs;
            dst.data += (u64)cp.second * dst.bs;
            k_ew_copy<<<ew_grid(c, 2 * in->limbs, 1), 256, 0, st>>>(src, dst, in->limbs, c->n);
            LAUNCH_CHECK(c);
        }
        return CKKS_OK;
    }
    for (size_t r = 0; r < p->round_cnt.size(); r++) {
        rt.sel = p->d_sel + p->round_off[r];
        if ((rc = keyswitch_lanes(c, 2, in->limbs, p->round_cnt[r], rt, st))) return rc;
    }
    return CKKS_OK;
}

// ------------------------------------------------------------------------------------ hoisted rotations (SURVEY 8 f4)
// All rotations of a plan applied to ONE ciphertext with a shared digit decomposition (kernels.cuh, "hoisted rotations").
// Every non-zero step of the plan must have its own Galois key (no NAF chains: a chained step acts on a different input).
// NOT bit-identical to SEAL's rotate_vector (same decrypted values within key-switch noise): an explicit opt-in mode.
extern "C" int ckks_rotate_plan_hoisted(ckks_ctx *c, const ckks_rotplan *p, const ckks_view *in, const ckks_view *out, ckks_stream s) {
    int rc;
    if (!p) return fail(CKKS_ERR_INVALID, "null plan");
    if ((rc = check_view(c, in, "encrypted")) || (rc = check_view(c, out, "out"))) return rc;
    if (in->size != 2 || out->size != 2) return fail(CKKS_ERR_INVALID, "encrypted size must be 2");
    if (in->batch != 1) return fail(CKKS_ERR_INVALID, "hoisted rotations share the decomposition of ONE input ciphertext");
    if (in->limbs > c->K - 1) return fail(CKKS_ERR_INVALID, "encrypted is not valid for encryption parameters");
    if (out->batch != p->batch || out->limbs != in->limbs) return fail(CKKS_ERR_INVALID, "rotate_plan: batch/level mismatch");
    if (out->data == in->data) return fail(CKKS_ERR_INVALID, "rotate_plan: out must not alias in");
    if (p->round_cnt.size() > 1) return fail(CKKS_ERR_INVALID, "Galois key not present (hoisting needs a key for every step itself)");
    CU(cudaSetDevice(c->device));
    if ((rc = sync_key_tables(p->ks))) return rc;
    cudaStream_t st = (cudaStream_t)s;
    const int L = in->limbs, K = c->K;
    const size_t N = c->n;
    KsRoute rt{};
    rt.v[0] = dv(in);
    rt.v[0].bs = 0;
    rt.v[1] = dv(out);
    rt.v[2] = dv(out);
    for (int b : p->zero_entries) {   // rotate by 0: the input unchanged
        DView dst = rt.v[1];
        dst.data += (u64)b * dst.bs;
        k_ew_copy<<<ew_grid(c, 2 * L, 1), 256, 0, st>>>(rt.v[0], dst, L, c->n);
        LAUNCH_CHECK(c);
    }
    if (p->round_cnt.empty()) return CKKS_OK;
    const int R = p->round_cnt[0];
    const size_t shared_words = N * ((size_t)L + (size_t)L * (L + 1));
    const size_t per_rot = N * (2 * (size_t)(L + 1) + 2 * (size_t)L);
    size_t fit = c->ws_cap > shared_words * 8 ? (c->ws_cap - shared_words * 8) / (per_rot * 8) : 1;
    if (fit < 1) fit = 1;
    if (fit > 16384) fit = 16384;
    const int Bc = (int)(fit < (size_t)R ? fit : (size_t)R);
    if ((rc = ensure_ws(c, (shared_words + per_rot * Bc) * 8))) return rc;
    u64 *D = c->ws, *T1 = D + (size_t)L * N, *ACC = T1 + (size_t)L * (L + 1) * N, *T2 = ACC + (size_t)Bc * 2 * (L + 1) * N;
    KsRoute r0 = rt;       // decomposition of the input: no permutation, no per-entry routing
    r0.tgt_poly = 1;
    rt.tgt_poly = 1;
    rt.perm_tab = p->ks->d_perm_tab;
    rt.key_tab = p->ks->d_key_tab;
    rt.key_tiled = 1;
#define RUN(LN)                                                                                                     \
    {                                                                                                               \
        typedef NttGeo<LN> G;                                                                                       \
        k_ks_intt_row<LN, false><<<dim3(G::ROW_TILES, L, 1), NTT_THREADS, 0, st>>>(r0, D, L, c->t);                 \
        LAUNCH_CHECK(c);                                                                                            \
        k_ks_invcol_modup<LN><<<dim3(G::COL_TILES, L, 1), NTT_THREADS, 0, st>>>(D, T1, L, 1, c->t);                 \
        LAUNCH_CHECK(c);                                                                                            \
        k_hoist_finish<LN><<<dim3(G::ROW_TILES, L *(L + 1), 1), NTT_THREADS, 0, st>>>(T1, rt.v[0], L, c->t);        \
        LAUNCH_CHECK(c);                                                                                            \
        for (int b0 = 0; b0 < R; b0 += Bc) {                                                                        \
            const int bc = (R - b0) < Bc ? (R - b0) : Bc;                                                           \
            rt.sel = p->d_sel + p->round_off[0];                                                                    \
            rt.b0 = b0;                                                                                             \
            DView spec{ACC + (size_t)L * N, (u64)(L + 1) * N, 0};                                                   \
            DView minu{ACC, 2 * (u64)(L + 1) * N, (u64)(L + 1) * N};                                                \
            k_hoist_mac<LN><<<dim3(G::ROW_TILES, L + 1, bc), NTT_THREADS, 0, st>>>(T1, rt, ACC, L, c->t);           \
            LAUNCH_CHECK(c);                                                                                        \
            k_md_invcol_fwdcol<LN><<<dim3(G::COL_TILES, 1, 2 * bc), NTT_THREADS, 0, st>>>(spec, T2, L, K - 1, 1, c->t); \
            LAUNCH_CHECK(c);                                                                                        \
            k_md_fwd_row<LN, 2><<<dim3(G::ROW_TILES, L, 2 * bc), NTT_THREADS, 0, st>>>(T2, minu, rt, 2, L, K - 1, c->t); \
            LAUNCH_CHECK(c);                                                                                        \
        }                                                                                                           \
    }
    DISPATCH_LOGN(c, RUN)
#undef RUN
    return CKKS_OK;
}

// ------------------------------------------------------------------------------------ fused products
static int mul_sum(ckks_ctx *c, bool plain, const ckks_view *a, const ckks_view *b, const ckks_view *o, cudaStream_t st) {
    int rc;
    if ((rc = check_view(c, a, "a")) || (rc = check_view(c, b, "b")) || (rc = check_view(c, o, "out"))) return rc;
    if (a->batch != b->batch || a->limbs != b->limbs || o->limbs != a->limbs || o->batch != 1)
        return fail(CKKS_ERR_INVALID, "multiply_sum: parameter mismatch");
    if (plain ? (b->size != 1 || o->size != a->size) : (a->size != 2 || b->size != 2 || o->size != 3))
        return fail(CKKS_ERR_INVALID, "multiply_sum: size mismatch");
    if (o->data == a->data || o->data == b->data) return fail(CKKS_ERR_INVALID, "multiply_sum: out must not alias an input");
    CU(cudaSetDevice(c->device));
    if (plain) k_ew_mul_sum<true><<<ew_grid(c, a->size * a->limbs, 1), 256, 0, st>>>(dv(a), dv(b), dv(o), a->batch, a->limbs, c->n, c->t);
    else k_ew_mul_sum<false><<<ew_grid(c, a->limbs, 1), 256, 0, st>>>(dv(a), dv(b), dv(o), a->batch, a->limbs, c->n, c->t);
    LAUNCH_CHECK(c);
    return CKKS_OK;
}
extern "C" int ckks_multiply_plain_sum(ckks_ctx *c, const ckks_view *cts, const ckks_view *pts, const ckks_view *o, ckks_stream s) {
    return mul_sum(c, true, cts, pts, o, (cudaStream_t)s);
}
extern "C" int ckks_multiply_sum(ckks_ctx *c, const ckks_view *a, const ckks_view *b, const ckks_view *o, ckks_stream s) {
    return mul_sum(c, false, a, b, o, (cudaStream_t)s);
}

// ------------------------------------------------------------------------------------ rescale
extern "C" int ckks_rescale(ckks_ctx *c, const ckks_view *in, const ckks_view *out, ckks_stream s) {
    int rc;
    if ((rc = check_view(c, in, "encrypted")) || (rc = check_view(c, out, "out"))) return rc;
    if (in->limbs < 2) return fail(CKKS_ERR_INVALID, "end of modulus switching chain reached");
    if (out->batch != in->batch || out->size != in->size || out->limbs != in->limbs - 1)
        return fail(CKKS_ERR_INVALID, "destination parameter mismatch");
    if (out->data == in->data && (out->poly_stride != in->poly_stride || out->batch_stride != in->batch_stride))
        return fail(CKKS_ERR_INVALID, "rescale: in-place only with identical strides");
    CU(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)s;
    const int L = in->limbs, S = in->size, B = in->batch, Lo = L - 1;
    const size_t N = c->n;
    const size_t per = (size_t)S * N * (1 + Lo);
    size_t fit = c->ws_cap / (per * 8);
    if (fit < 1) fit = 1;
    int Bc = (int)(fit < (size_t)B ? fit : (size_t)B);
    while ((long)Bc * S > 65535) Bc--;
    if ((rc = ensure_ws(c, per * 8 * Bc))) return rc;
    u64 *R = c->ws, *T2 = R + (size_t)Bc * S * N;
    Tables tr = c->t;
    tr.round_half = c->round_rescale;
    for (int b0 = 0; b0 < B; b0 += Bc) {
        const int bc = (B - b0) < Bc ? (B - b0) : Bc;
        g_pdl_now = g_pdl_mode < 0 ? bc * S >= 16 : g_pdl_mode != 0;
        DView src{(u64 *)in->data + (u64)b0 * in->batch_stride, in->batch_stride, in->poly_stride};
        DView last{src.data + (size_t)Lo * N, src.bs, src.ps};
        DView dR{R, (u64)S * N, (u64)N};
        DView Rz{R, (u64)N, 0};
        DView dst{(u64 *)out->data + (u64)b0 * out->batch_stride, out->batch_stride, out->poly_stride};
        KsRoute rrt{};
        rrt.v[0] = src; rrt.v[1] = dst; rrt.v[2] = dst;
#define RUN(LN)                                                                                                   \
    {                                                                                                             \
        typedef NttGeo<LN> G;                                                                                     \
        k_inv_row<LN><<<dim3(G::ROW_TILES, S, bc), NTT_THREADS, 0, st>>>(last, dR, 1, Lo, tr);                  \
        LAUNCH_CHECK(c);                                                                                          \
        if (c->fuse) {                                                                                            \
            const int ns3 = pick_split(c->split3, G::COL_TILES * S * bc, Lo);                                     \
            launch_pdl(k_md_invcol_fwdcol<LN>, dim3(G::COL_TILES, ns3, bc * S), st, Rz, T2, Lo, Lo, ns3, tr);   \
            LAUNCH_CHECK(c);                                                                                      \
        } else {                                                                                                  \
            launch_pdl(k_inv_col<LN, true>, dim3(G::COL_TILES, S, bc), st, dR, dR, 1, Lo, tr);          \
            LAUNCH_CHECK(c);                                                                                      \
            launch_pdl(k_md_fwd_col<LN>, dim3(G::COL_TILES, Lo, bc * S), st, Rz, T2, Lo, Lo, tr);       \
            LAUNCH_CHECK(c);                                                                                      \
        }                                                                                                         \
        launch_pdl(k_md_fwd_row<LN, 0>, dim3(G::ROW_TILES, Lo, bc * S), st, T2, src, rrt, S, Lo, Lo, tr); \
        LAUNCH_CHECK(c);                                                                                          \
    }
        DISPATCH_LOGN(c, RUN)
#undef RUN
    }
    return CKKS_OK;
}

// ------------------------------------------------------------------------------------ encoder (SURVEY 8 f1)
static int ensure_encoder_tables(ckks_ctx *c) {
    if (c->d_kidx) return CKKS_OK;
    const uint32_t n = (uint32_t)c->n, m = 2 * n;
    std::vector<uint32_t> k(n / 2);
    uint64_t pos = 1;
    for (uint32_t i = 0; i < n / 2; i++) {
        k[i] = (uint32_t)((pos - 1) >> 1);
        pos = pos * 3 % m;
    }
    int rc = upload_vec((void **)&c->d_kidx, k.data(), k.size() * sizeof(uint32_t));
    if (rc) return rc;
    // (Q_L - 1)/2 in the mixed radix q_0, q_1, ...: little-endian multi-word arithmetic on the host
    c->half_digits.assign(c->K + 1, HalfDigits{});
    for (int L = 1; L <= c->K; L++) {
        std::vector<uint64_t> big{1};
        for (int i = 0; i < L; i++) {   // big *= q_i
            unsigned __int128 carry = 0;
            for (auto &w : big) {
                unsigned __int128 v = (unsigned __int128)w * c->primes[i] + carry;
                w = (uint64_t)v;
                carry = v >> 64;
            }
            if (carry) big.push_back((uint64_t)carry);
        }
        big[0] -= 1;                     // Q is odd
        for (size_t w = 0; w < big.size(); w++)   // >>= 1
            big[w] = (big[w] >> 1) | (w + 1 < big.size() ? big[w + 1] << 63 : 0);
        for (int i = 0; i < L; i++) {   // digit = big mod q_i; big /= q_i
            unsigned __int128 rem = 0;
            for (size_t w = big.size(); w-- > 0;) {
                unsigned __int128 cur = (rem << 64) | big[w];
                big[w] = (uint64_t)(cur / c->primes[i]);
                rem = cur % c->primes[i];
            }
            c->half_digits[L].d[i] = (uint64_t)rem;
        }
    }
    return CKKS_OK;
}

template <int SGN>
static int run_fft(ckks_ctx *c, double2 *v, int batch, cudaStream_t st) {
#define RUN(LN)                                                                                          \
    {                                                                                                    \
        k_fft_top<LN, SGN><<<dim3(FFT_TILE / 256, batch), 256, 0, st>>>(v); LAUNCH_CHECK(c);             \
        k_fft_tile<SGN><<<dim3((1 << LN) / FFT_TILE, batch), 256, 0, st>>>(v, 1 << LN); LAUNCH_CHECK(c); \
    }
    DISPATCH_LOGN(c, RUN)
#undef RUN
    return CKKS_OK;
}

static int encoder_chunk(const ckks_ctx *c, int batch, size_t bytes_per_entry) {
    size_t fit = c->ws_cap / bytes_per_entry;
    if (fit < 1) fit = 1;
    if (fit > 65535) fit = 65535;
    return (int)(fit < (size_t)batch ? fit : (size_t)batch);
}

extern "C" int ckks_encode(ckks_ctx *c, const double *values, int count, double scale, const ckks_view *out, ckks_stream s) {
    int rc;
    if ((rc = check_view(c, out, "plain"))) return rc;
    if (out->size != 1) return fail(CKKS_ERR_INVALID, "encode: destination must be a plaintext (size 1)");
    if (count < 0 || count > c->n / 2) return fail(CKKS_ERR_INVALID, "values has invalid size");
    if (count > 0 && !values) return fail(CKKS_ERR_INVALID, "encode: null values");
    if (!(scale > 0.0)) return fail(CKKS_ERR_INVALID, "scale out of bounds");
    if (out->batch > 1 && out->batch_stride == 0) return fail(CKKS_ERR_INVALID, "encode: destination entries must be distinct");
    CU(cudaSetDevice(c->device));
    if ((rc = ensure_encoder_tables(c))) return rc;
    cudaStream_t st = (cudaStream_t)s;
    const size_t N = c->n;
    const int B = out->batch, Bc = encoder_chunk(c, B, N * sizeof(double2));
    if ((rc = ensure_ws(c, (size_t)Bc * N * sizeof(double2)))) return rc;
    double2 *v = (double2 *)c->ws;
    for (int b0 = 0; b0 < B; b0 += Bc) {
        const int bc = (B - b0) < Bc ? (B - b0) : Bc;
        k_enc_scatter<<<dim3((unsigned)(N / 2 + 255) / 256, bc), 256, 0, st>>>(values + (size_t)b0 * count, count, c->d_kidx, v, (int)N);
        LAUNCH_CHECK(c);
        if ((rc = run_fft<-1>(c, v, bc, st))) return rc;
        DView dst{(u64 *)out->data + (u64)b0 * out->batch_stride, out->batch_stride, out->poly_stride};
#define RUN(LN) k_enc_round<LN><<<dim3((1 << LN) / 256, bc), 256, 0, st>>>(v, scale / (double)N, dst, out->limbs, c->t); LAUNCH_CHECK(c);
        DISPATCH_LOGN(c, RUN)
#undef RUN
        // plaintexts live in NTT form: transform the bc x limbs coefficient limbs in place
        if ((rc = ntt_api(c, (uint64_t *)dst.data, bc, out->limbs, 0, B > 1 ? out->batch_stride : out->poly_stride, false, st))) return rc;
    }
    return CKKS_OK;
}

static uint64_t host_residue(double r, uint64_t p) {
    const bool neg = r < 0.0;
    double a = neg ? -r : r;
    uint64_t res;
    if (a < 4611686018427387904.0) {
        res = (uint64_t)a % p;
    } else {
        int e;
        const double fr = frexp(a, &e);
        const uint64_t mant = (uint64_t)ldexp(fr, 53);
        e -= 53;
        unsigned __int128 pw = 1, base = 2;
        for (; e > 0; e >>= 1) {
            if (e & 1) pw = pw * base % p;
            base = base * base % p;
        }
        res = (uint64_t)((unsigned __int128)(mant % p) * pw % p);
    }
    return (neg && res) ? p - res : res;
}

extern "C" int ckks_encode_scalar(ckks_ctx *c, double value, double scale, const ckks_view *out, ckks_stream s) {
    int rc;
    if ((rc = check_view(c, out, "plain"))) return rc;
    if (out->size != 1) return fail(CKKS_ERR_INVALID, "encode: destination must be a plaintext (size 1)");
    if (!(scale > 0.0)) return fail(CKKS_ERR_INVALID, "scale out of bounds");
    if (out->limbs > 32) return fail(CKKS_ERR_INVALID, "encode: more than 32 limbs");
    CU(cudaSetDevice(c->device));
    ConstResidues cr{};
    const double r = nearbyint(value * scale);
    for (int l = 0; l < out->limbs; l++) cr.r[l] = host_residue(r, c->primes[l]);
    k_enc_fill<<<dim3((c->n + 255) / 256, out->limbs, out->batch), 256, 0, (cudaStream_t)s>>>(dv(out), cr, c->n);
    LAUNCH_CHECK(c);
    return CKKS_OK;
}

// ------------------------------------------------------------------------------------ constant-coefficient sums
// words from the first to one past the last active word of a view
static size_t view_words(const ckks_view *v, int n) {
    return (size_t)(v->batch - 1) * v->batch_stride + (size_t)(v->size - 1) * v->poly_stride + (size_t)v->limbs * n;
}

extern "C" int ckks_multiply_const_sum(ckks_ctx *c, const ckks_view *in, int terms, int groups, const double *coeffs,
                                       const double *scales, const double *const_coeffs, const double *const_scales,
                                       const ckks_view *out, ckks_stream s) {
    int rc;
    if ((rc = check_view(c, in, "in")) || (rc = check_view(c, out, "out"))) return rc;
    if (terms < 1 || groups < 1) return fail(CKKS_ERR_INVALID, "multiply_const_sum: terms and groups must be at least 1");
    if (in->batch % terms) return fail(CKKS_ERR_INVALID, "multiply_const_sum: in batch must be terms x out batch / groups");
    const int M = in->batch / terms;
    if ((long long)groups * M != out->batch)
        return fail(CKKS_ERR_INVALID, "multiply_const_sum: out batch must be groups x in batch / terms");
    if (out->size != in->size || out->limbs != in->limbs) return fail(CKKS_ERR_INVALID, "destination parameter mismatch");
    if (in->batch > 1 && in->batch_stride == 0) return fail(CKKS_ERR_INVALID, "multiply_const_sum: in entries must be distinct");
    if (out->batch > 1 && out->batch_stride == 0) return fail(CKKS_ERR_INVALID, "multiply_const_sum: out entries must be distinct");
    const uint64_t *ib = (const uint64_t *)in->data, *ob = (const uint64_t *)out->data;
    if (ob < ib + view_words(in, c->n) && ib < ob + view_words(out, c->n))
        return fail(CKKS_ERR_INVALID, "multiply_const_sum: out must not alias in");
    if (!coeffs || !scales) return fail(CKKS_ERR_INVALID, "multiply_const_sum: null coefficients");
    if (!const_coeffs != !const_scales) return fail(CKKS_ERR_INVALID, "multiply_const_sum: constant values and scales go together");
    const int L = in->limbs;
    // the same checks and residues as ckks_encode_scalar(value, scale) for every constant
    auto residues = [&](double value, double scale, u64 *r) {
        if (!(scale > 0.0)) return fail(CKKS_ERR_INVALID, "scale out of bounds");
        const double v = nearbyint(value * scale);
        if (!std::isfinite(v)) return fail(CKKS_ERR_INVALID, "multiply_const_sum: constant times scale is not finite");
        for (int l = 0; l < L; l++) r[l] = host_residue(v, c->primes[l]);
        return (int)CKKS_OK;
    };
    const size_t per_group = (size_t)(terms + 1) * L;
    if (per_group > CONST_SUM_WORDS) return fail(CKKS_ERR_INVALID, "multiply_const_sum: (terms + 1) x limbs exceeds 2048");
    const int chunk = (int)std::min<size_t>(CONST_SUM_GROUPS, CONST_SUM_WORDS / per_group);
    std::vector<ConstSumTable> tabs((groups + chunk - 1) / chunk);
    for (int g0 = 0, k = 0; g0 < groups; g0 += chunk, k++) {
        const int G = std::min(chunk, groups - g0);
        u64 *r = tabs[k].r, *r0 = r + (size_t)G * terms * L;
        for (int g = 0; g < G; g++) {
            for (int i = 0; i < terms; i++) {
                const size_t q = (size_t)(g0 + g) * terms + i;
                if ((rc = residues(coeffs[q], scales[q], r + ((size_t)g * terms + i) * L))) return rc;
            }
            if (const_coeffs) {
                if ((rc = residues(const_coeffs[g0 + g], const_scales[g0 + g], r0 + (size_t)g * L))) return rc;
            } else {
                for (int l = 0; l < L; l++) r0[(size_t)g * L + l] = 0;
            }
        }
    }
    CU(cudaSetDevice(c->device));
    for (int g0 = 0, k = 0; g0 < groups; g0 += chunk, k++) {
        const int G = std::min(chunk, groups - g0);
        DView o = dv(out);
        o.data += (size_t)g0 * M * out->batch_stride;
        k_ew_const_sum<<<ew_grid(c, in->size * L, M), 256, 0, (cudaStream_t)s>>>(dv(in), o, tabs[k], G, terms, M, L, c->n, c->t);
        LAUNCH_CHECK(c);
    }
    return CKKS_OK;
}

extern "C" int ckks_decode(ckks_ctx *c, const ckks_view *in, double scale, double *values, ckks_stream s) {
    int rc;
    if ((rc = check_view(c, in, "plain"))) return rc;
    if (in->size != 1) return fail(CKKS_ERR_INVALID, "decode: source must be a plaintext (size 1)");
    if (!values) return fail(CKKS_ERR_INVALID, "decode: null destination");
    if (!(scale > 0.0)) return fail(CKKS_ERR_INVALID, "scale out of bounds");
    if (in->limbs > 32) return fail(CKKS_ERR_INVALID, "decode: more than 32 limbs");
    if (in->batch > 1 && in->batch_stride == 0) return fail(CKKS_ERR_INVALID, "decode: broadcast views are not supported");
    CU(cudaSetDevice(c->device));
    if ((rc = ensure_encoder_tables(c))) return rc;
    cudaStream_t st = (cudaStream_t)s;
    const size_t N = c->n;
    const int B = in->batch, L = in->limbs;
    const size_t per = N * sizeof(double2) + (size_t)L * N * 8;
    const int Bc = encoder_chunk(c, B, per);
    if ((rc = ensure_ws(c, per * Bc))) return rc;
    double2 *v = (double2 *)c->ws;
    u64 *res = c->ws + (size_t)Bc * N * 2;
    for (int b0 = 0; b0 < B; b0 += Bc) {
        const int bc = (B - b0) < Bc ? (B - b0) : Bc;
        // the inverse transform runs in place: work on a copy of the plaintext limbs
        CU(cudaMemcpy2DAsync(res, (size_t)L * N * 8, (const u64 *)in->data + (u64)b0 * in->batch_stride,
                             (size_t)(B > 1 ? in->batch_stride : in->poly_stride) * 8, (size_t)L * N * 8, bc,
                             cudaMemcpyDeviceToDevice, st));
        if ((rc = ntt_api(c, (uint64_t *)res, bc, L, 0, (uint64_t)L * N, true, st))) return rc;
#define RUN(LN) k_dec_compose<LN><<<dim3((1 << LN) / 256, bc), 256, 0, st>>>(res, L, c->half_digits[L], 1.0 / scale, v, c->t); LAUNCH_CHECK(c);
        DISPATCH_LOGN(c, RUN)
#undef RUN
        if ((rc = run_fft<1>(c, v, bc, st))) return rc;
#define RUN(LN) k_dec_gather<LN><<<dim3((1 << LN) / 512, bc), 256, 0, st>>>(v, c->d_kidx, values + (size_t)b0 * (N / 2)); LAUNCH_CHECK(c);
        DISPATCH_LOGN(c, RUN)
#undef RUN
    }
    return CKKS_OK;
}

// ------------------------------------------------------------------------------------ sampling (SURVEY 8 f3)
static int sample_impl(ckks_ctx *c, int kind, const SampleKey &key, uint64_t stream_id, const ckks_view *out, ckks_stream s) {
    int rc;
    if ((rc = check_view(c, out, "destination"))) return rc;
    if (out->size != 1) return fail(CKKS_ERR_INVALID, "sample: destination must have size 1");
    if (kind < 0 || kind > 2) return fail(CKKS_ERR_INVALID, "sample: unknown distribution");
    if (out->batch > 1 && out->batch_stride == 0) return fail(CKKS_ERR_INVALID, "sample: destination entries must be distinct");
    if (out->batch >= (1 << 20)) return fail(CKKS_ERR_INVALID, "sample: batch too large");
    CU(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)s;
    const dim3 grid((c->n + 255) / 256, out->batch);
    if (kind == 2) {
        k_sample_uniform<<<grid, 256, 0, st>>>(dv(out), out->limbs, c->n, key, stream_id, c->t);
        LAUNCH_CHECK(c);
        return CKKS_OK;   // uniform in the NTT domain is uniform
    }
    k_sample_small<<<grid, 256, 0, st>>>(dv(out), out->limbs, c->n, kind, key, stream_id, c->t);
    LAUNCH_CHECK(c);
    return ntt_api(c, (uint64_t *)out->data, out->batch, out->limbs, 0, out->batch > 1 ? out->batch_stride : out->poly_stride, false, st);
}

// ChaCha20 under the caller's 256-bit key (32 bytes from a CSPRNG): the entry point KeyGenerator / Encryptor use
extern "C" int ckks_sample_keyed(ckks_ctx *c, int kind, const uint8_t key[32], uint64_t stream_id, const ckks_view *out, ckks_stream s) {
    if (!key) return fail(CKKS_ERR_INVALID, "sample: null key");
    SampleKey k;
    memcpy(k.k, key, 32);
    return sample_impl(c, kind, k, stream_id, out, s);
}
// Reproducible sampling for tests and benchmarks: the 64-bit seed is expanded into the ChaCha20 key, so the output
// has at most 64 bits of entropy -- NOT for real keys (use ckks_sample_keyed)
extern "C" int ckks_sample(ckks_ctx *c, int kind, uint64_t seed, uint64_t stream_id, const ckks_view *out, ckks_stream s) {
    SampleKey k;
    uint64_t w[4] = {seed, ~seed, seed * 0x9E3779B97F4A7C15ull + 1, (seed ^ 0xD1B54A32D192ED03ull) * 0xBF58476D1CE4E5B9ull};
    memcpy(k.k, w, 32);
    return sample_impl(c, kind, k, stream_id, out, s);
}
