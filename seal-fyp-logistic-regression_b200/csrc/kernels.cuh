// kernels.cuh -- sm_100a kernels of the CKKS evaluation engine.
//
// Families (SURVEY.md section 2.2):
//   * plain batched NTT / INTT (column + row pass per transform)
//   * element-wise dyadic ops (add, sub, negate, multiply, multiply_plain, add_plain, add_many)
//   * key switching: digit INTT (with the Galois gather fused into its load), mod-up base
//     conversion fused into the column pass of the NTT, key inner product fused into the row
//     pass, mod-down fused into the NTT passes of the special-prime limb
//   * rescale: same mod-down machinery with the last data prime
//
// Grid conventions: blockIdx.x = tile inside a limb, blockIdx.y = limb / (digit,limb) pair,
// blockIdx.z = ciphertext (or ciphertext*poly) index.  All CTAs are NTT_THREADS threads.
#pragma once
#include <cooperative_groups.h>
#include "ntt_passes.cuh"

struct Tables {
    const ModConst *mod;  // [K]
    const tw_t *twf;      // [K][N] forward twiddles
    const tw_t *twi;      // [K][N] inverse twiddles
    const u64 *inv;       // [K][K]  inv[a*K+j]  = q_a^-1 mod q_j
    const u64 *invs;      // [K][K]  Shoup companion
    const u64 *halfmod;   // [K][K]  (q_a >> 1) mod q_j
    const FpConst *fp;    // [K]     FP64-path constants (ok != 0 for primes below 2^41)
    const double *twfd;   // [K][N]  forward twiddles as doubles
    const double *twid;   // [K][N]  inverse twiddles as doubles
    int K;
    int round_half;
};

struct DView {
    u64 *data;
    u64 bs;  // batch stride (words)
    u64 ps;  // poly stride (words)
};

__device__ __forceinline__ ModConst load_mod(const Tables &t, int j) { return t.mod[j]; }
__device__ __forceinline__ double *as_fp(u64 *smem) { return reinterpret_cast<double *>(smem); }
__device__ __forceinline__ double bits_fp(u64 v) { return __longlong_as_double((long long)v); }
__device__ __forceinline__ u64 fp_bits(double v) { return (u64)__double_as_longlong(v); }

// eight contiguous words of a thread (64 bytes) as four 16-byte accesses
__device__ __forceinline__ void load8(u64 (&x)[8], const u64 *p) {
    const ulonglong2 *q = reinterpret_cast<const ulonglong2 *>(p);
#pragma unroll
    for (int v = 0; v < 4; v++) {
        ulonglong2 a = q[v];
        x[2 * v] = a.x;
        x[2 * v + 1] = a.y;
    }
}
__device__ __forceinline__ void store8(u64 *p, const u64 (&x)[8]) {
    ulonglong2 *q = reinterpret_cast<ulonglong2 *>(p);
#pragma unroll
    for (int v = 0; v < 4; v++) q[v] = make_ulonglong2(x[2 * v], x[2 * v + 1]);
}
// the thread's eight source indices of a Galois gather (32 contiguous bytes of the table)
__device__ __forceinline__ void load_perm8(unsigned (&ix)[8], const uint32_t *perm) {
    const uint4 *q = reinterpret_cast<const uint4 *>(perm);
    uint4 a = __ldg(q), b = __ldg(q + 1);
    ix[0] = a.x; ix[1] = a.y; ix[2] = a.z; ix[3] = a.w;
    ix[4] = b.x; ix[5] = b.y; ix[6] = b.z; ix[7] = b.w;
}
// programmatic dependent launch (sm_90+): let the successor start its prologue / wait for the
// predecessor's results
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
// A pipeline kernel lets its successor start (programmatic dependent launch) only once its own inputs are in registers
// and its main work is under way -- PDL_LATE() sits after the loads / the first transform, before the final stores -- so
// that just the immediate successor gets a head start for its prologue (round 1 triggered at the top of every kernel,
// which cascades the whole pipeline into residency: slower at small batches, profiles/r02_keyswitch_experiments.md).
#define PDL_LATE() pdl_launch_dependents()
// ---- TMA 1-D bulk copy global -> shared with mbarrier completion (SASS: UBLKCP), used to stage the
// next digit's 16 KB tile while the current digit is transformed
__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(u64 *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void tma_load_tile(void *dst, const void *src, unsigned bytes, u64 *bar) {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(u64 *bar, unsigned parity) {
    unsigned done;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done)
                     : "r"(smem_u32(bar)), "r"(parity)
                     : "memory");
    } while (!done);
}
__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// Per-entry routing of a batched key switch: which ciphertext of the views a launch slot works
// on, which key/permutation it uses, and which of the three views (0 = in, 1 = out, 2 = scratch)
// it reads from and writes to.  With sel == nullptr slot z works on entry z with key 0,
// reading view 0 and writing view 1.
struct KsSel {
    int entry;    // batch entry written (view dst)
    int slot;     // key slot
    short src;    // view read
    short dst;    // view written
    int sentry;   // batch entry read (view src); differs from `entry` only in shared-prefix rotation plans
};
struct KsRoute {
    DView v[3];                        // in, out, scratch
    const KsSel *sel;                  // [launch slots] or nullptr
    const uint32_t *const *perm_tab;   // [key slots] (device) or nullptr
    const u64 *const *key_tab;         // [key slots] (device) or nullptr
    const uint32_t *perm0;             // used when sel == nullptr
    const u64 *key0;
    int b0;                            // first launch slot of this chunk
    int tgt_poly;                      // polynomial that is key-switched (2 relin, 1 Galois)
    DView accv;                        // optional: accv[entry] += result (rotate-and-sum chains)
    int has_acc;
    int key_tiled;                     // keys are engine-owned copies in the thread-major tile layout (k_retile_key)
};
__device__ __forceinline__ KsSel route_sel(const KsRoute &r, int z) {
    if (r.sel) return r.sel[r.b0 + z];
    KsSel s;
    s.entry = s.sentry = r.b0 + z; s.slot = 0; s.src = 0; s.dst = 1;
    return s;
}
__device__ __forceinline__ const uint32_t *route_perm(const KsRoute &r, const KsSel &s) {
    return r.sel ? r.perm_tab[s.slot] : r.perm0;
}
__device__ __forceinline__ const u64 *route_key(const KsRoute &r, const KsSel &s) {
    return r.sel ? r.key_tab[s.slot] : r.key0;
}

// =============================================================================== plain NTT
// limb instance y = s*limbs + l of batch entry z; prime = first_prime + l
template <int LOGN>
__global__ void __launch_bounds__(NTT_THREADS) k_fwd_col(DView src, DView dst, int limbs, int first_prime, Tables t) {
    typedef NttGeo<LOGN> G;
    __shared__ u64 smem[NTT_TILE];
    const int s = blockIdx.y / limbs, l = blockIdx.y % limbs, pj = first_prime + l;
    const u64 *in = src.data + blockIdx.z * src.bs + s * src.ps + (u64)l * G::N;
    u64 *out = dst.data + blockIdx.z * dst.bs + s * dst.ps + (u64)l * G::N;
    const ModConst m = load_mod(t, pj);
    const int c0 = blockIdx.x * 32;
    const FpConst f = t.fp[pj];
    if (f.ok != 0.0) {   // small prime: FP64 butterflies; the intermediate limb holds doubles
        double xd[8];
#pragma unroll
        for (int e = 0; e < 8; e++) xd[e] = fp_from_u64(in[col_coarse_idx<LOGN>(c0, e)]);
        fwd_col_pass_fp<LOGN>(xd, t.twfd + (size_t)pj * G::N, f, as_fp(smem));
#pragma unroll
        for (int e = 0; e < 8; e++) out[col_fine_idx<LOGN>(c0, e)] = fp_bits(xd[e]);
        return;
    }
    u64 x[8];
#pragma unroll
    for (int e = 0; e < 8; e++) x[e] = in[col_coarse_idx<LOGN>(c0, e)];
    fwd_col_pass<LOGN>(x, t.twf + (size_t)pj * G::N, m, smem);
#pragma unroll
    for (int e = 0; e < 8; e++) out[col_fine_idx<LOGN>(c0, e)] = x[e];  // lazy
}

template <int LOGN>
__global__ void __launch_bounds__(NTT_THREADS) k_fwd_row(DView src, DView dst, int limbs, int first_prime, Tables t) {
    typedef NttGeo<LOGN> G;
    __shared__ u64 smem[NTT_TILE];
    const int s = blockIdx.y / limbs, l = blockIdx.y % limbs, pj = first_prime + l;
    const u64 *in = src.data + blockIdx.z * src.bs + s * src.ps + (u64)l * G::N;
    u64 *out = dst.data + blockIdx.z * dst.bs + s * dst.ps + (u64)l * G::N;
    const ModConst m = load_mod(t, pj);
    const int t0 = blockIdx.x * NTT_TILE;
    u64 x[8];
    const FpConst f = t.fp[pj];
    if (f.ok != 0.0) {
        double xd[8];
#pragma unroll
        for (int e = 0; e < 8; e++) xd[e] = bits_fp(in[t0 + row_strided_li<LOGN>(e)]);
        fwd_row_pass_fp<LOGN>(xd, t.twfd + (size_t)pj * G::N, f, t0, as_fp(smem));
#pragma unroll
        for (int e = 0; e < 8; e++) x[e] = fp_to_canonical(xd[e], f);
        store8(out + t0 + 8 * threadIdx.x, x);
        return;
    }
#pragma unroll
    for (int e = 0; e < 8; e++) x[e] = in[t0 + row_strided_li<LOGN>(e)];
    fwd_row_pass<LOGN>(x, t.twf + (size_t)pj * G::N, m, t0, smem);
#pragma unroll
    for (int e = 0; e < 8; e++) x[e] = reduce64(x[e], m);
    store8(out + t0 + 8 * threadIdx.x, x);
}

template <int LOGN>
__global__ void __launch_bounds__(NTT_THREADS, 5) k_inv_row(DView src, DView dst, int limbs, int first_prime, Tables t) {
    typedef NttGeo<LOGN> G;
    __shared__ u64 smem[NTT_TILE];
    const int s = blockIdx.y / limbs, l = blockIdx.y % limbs, pj = first_prime + l;
    const u64 *in = src.data + blockIdx.z * src.bs + s * src.ps + (u64)l * G::N;
    u64 *out = dst.data + blockIdx.z * dst.bs + s * dst.ps + (u64)l * G::N;
    const ModConst m = load_mod(t, pj);
    const int t0 = blockIdx.x * NTT_TILE;
    u64 x[8];
    const FpConst f = t.fp[pj];
    pdl_wait();
    load8(x, in + t0 + 8 * threadIdx.x);
    if (f.ok != 0.0) {
        double xd[8];
#pragma unroll
        for (int e = 0; e < 8; e++) xd[e] = fp_from_u64(x[e]);
        inv_row_pass_fp<LOGN>(xd, t.twid + (size_t)pj * G::N, f, t0, as_fp(smem));
#pragma unroll
        for (int e = 0; e < 8; e++) out[t0 + row_strided_li<LOGN>(e)] = fp_bits(xd[e]);
        return;
    }
    inv_row_pass<LOGN>(x, t.twi + (size_t)pj * G::N, m, t0, smem);
#pragma unroll
    for (int e = 0; e < 8; e++) out[t0 + row_strided_li<LOGN>(e)] = x[e];  // lazy
}

// ADD_HALF: store (v + (p >> 1)) mod p instead of v -- the "flooring to rounding" step of SEAL's
// divide-by-last-prime (SURVEY A.7/A.8), fused into the last pass of the inverse transform
template <int LOGN, bool ADD_HALF>
__global__ void __launch_bounds__(NTT_THREADS) k_inv_col(DView src, DView dst, int limbs, int first_prime, Tables t) {
    typedef NttGeo<LOGN> G;
    __shared__ u64 smem[NTT_TILE];
    const int s = blockIdx.y / limbs, l = blockIdx.y % limbs, pj = first_prime + l;
    const u64 *in = src.data + blockIdx.z * src.bs + s * src.ps + (u64)l * G::N;
    u64 *out = dst.data + blockIdx.z * dst.bs + s * dst.ps + (u64)l * G::N;
    const ModConst m = load_mod(t, pj);
    const int c0 = blockIdx.x * 32;
    u64 x[8];
    const FpConst f = t.fp[pj];
    const u64 half = (ADD_HALF && t.round_half) ? (m.p >> 1) : 0;
    pdl_wait();
#pragma unroll
    for (int e = 0; e < 8; e++) x[e] = in[col_fine_idx<LOGN>(c0, e)];
    if (f.ok != 0.0) {
        double xd[8];
#pragma unroll
        for (int e = 0; e < 8; e++) xd[e] = bits_fp(x[e]);
        inv_col_pass_fp<LOGN>(xd, t.twid + (size_t)pj * G::N, f, as_fp(smem));
#pragma unroll
        for (int e = 0; e < 8; e++) {
            u64 v = fp_to_canonical(xd[e], f);
            if (ADD_HALF) v = csub(v + half, m.p);
            out[col_coarse_idx<LOGN>(c0, e)] = v;
        }
        return;
    }
    inv_col_pass<LOGN>(x, t.twi + (size_t)pj * G::N, m, smem);
#pragma unroll
    for (int e = 0; e < 8; e++) {
        u64 v = csub(csub(x[e], m.p2), m.p);
        if (ADD_HALF) v = csub(v + half, m.p);
        out[col_coarse_idx<LOGN>(c0, e)] = v;
    }
}

// ---- north-star variant (a): ONE RNS LIMB PER CTA, the limb resident in shared memory between the two passes (N <= 16384:
// a limb is at most 128 KB; N = 32768 would need a 2-CTA cluster, see DESIGN.md section 4).  1024 threads = four groups of
// 256 that run the same tile passes as the two-kernel transform, each group on its own tiles and exchange buffer, with the
// 64 x N2 limb matrix in shared memory instead of HBM/L2 in between: one global read and one global write per limb.
// Selected for the plain NTT entry points by CKKS_NTT_LIMB=1 (measured against the two-pass kernels in
// profiles/r02_keyswitch_experiments.md).
template <int LOGN, bool INVERSE>
__global__ void __launch_bounds__(1024, 1) k_ntt_limb(DView v, int limbs, int first_prime, Tables t) {
    typedef NttGeo<LOGN> G;
    extern __shared__ __align__(16) u64 sm_limb[];            // [N] limb, then 4 x [NTT_TILE] exchange buffers
    u64 *limb = sm_limb;
    const int grp = threadIdx.x >> 8;
    u64 *exch = sm_limb + G::N + grp * NTT_TILE;
    const int l = blockIdx.x % limbs, pj = first_prime + l;
    u64 *data = v.data + (u64)(blockIdx.x / limbs) * v.bs + (u64)l * G::N;
    const ModConst m = load_mod(t, pj);
    const FpConst f = t.fp[pj];
    const bool fp = f.ok != 0.0;
    u64 x[8];
    double xd[8];
    // every group runs the same number of passes (they share the CTA-wide barriers inside the pass functions): a group
    // without a tile of its own in the last round repeats another tile and discards the result
    constexpr int CROUNDS = (G::COL_TILES + 3) / 4, RROUNDS = (G::ROW_TILES + 3) / 4;
    const unsigned tid = threadIdx.x & 255;
    if (!INVERSE) {
        for (int r = 0; r < CROUNDS; r++) {
            const int tile = 4 * r + grp;
            const bool active = tile < G::COL_TILES;
            const int c0 = (active ? tile : tile % G::COL_TILES) * 32;
#pragma unroll
            for (int e = 0; e < 8; e++) x[e] = data[col_coarse_idx<LOGN>(c0, e)];
            if (fp) {
#pragma unroll
                for (int e = 0; e < 8; e++) xd[e] = fp_from_u64(x[e]);
                fwd_col_pass_fp<LOGN>(xd, t.twfd + (size_t)pj * G::N, f, as_fp(exch));
#pragma unroll
                for (int e = 0; e < 8; e++) x[e] = fp_bits(xd[e]);
            } else {
                fwd_col_pass<LOGN>(x, t.twf + (size_t)pj * G::N, m, exch);
            }
            if (active) {
#pragma unroll
                for (int e = 0; e < 8; e++) limb[col_fine_idx<LOGN>(c0, e)] = x[e];
            }
            __syncthreads();   // exchange buffer reuse by this group's next tile; after the last round: limb complete
        }
        for (int r = 0; r < RROUNDS; r++) {
            const int tile = 4 * r + grp;
            const bool active = tile < G::ROW_TILES;
            const int t0 = (active ? tile : tile % G::ROW_TILES) * NTT_TILE;
            if (fp) {
#pragma unroll
                for (int e = 0; e < 8; e++) xd[e] = bits_fp(limb[t0 + row_strided_li<LOGN>(e)]);
                fwd_row_pass_fp<LOGN>(xd, t.twfd + (size_t)pj * G::N, f, t0, as_fp(exch));
#pragma unroll
                for (int e = 0; e < 8; e++) x[e] = fp_to_canonical(xd[e], f);
            } else {
#pragma unroll
                for (int e = 0; e < 8; e++) x[e] = limb[t0 + row_strided_li<LOGN>(e)];
                fwd_row_pass<LOGN>(x, t.twf + (size_t)pj * G::N, m, t0, exch);
#pragma unroll
                for (int e = 0; e < 8; e++) x[e] = reduce64(x[e], m);
            }
            if (active) store8(data + t0 + 8 * tid, x);
            __syncthreads();
        }
    } else {
        for (int r = 0; r < RROUNDS; r++) {
            const int tile = 4 * r + grp;
            const bool active = tile < G::ROW_TILES;
            const int t0 = (active ? tile : tile % G::ROW_TILES) * NTT_TILE;
            load8(x, data + t0 + 8 * tid);
            if (fp) {
#pragma unroll
                for (int e = 0; e < 8; e++) xd[e] = fp_from_u64(x[e]);
                inv_row_pass_fp<LOGN>(xd, t.twid + (size_t)pj * G::N, f, t0, as_fp(exch));
#pragma unroll
                for (int e = 0; e < 8; e++) x[e] = fp_bits(xd[e]);
            } else {
                inv_row_pass<LOGN>(x, t.twi + (size_t)pj * G::N, m, t0, exch);
            }
            if (active) {
#pragma unroll
                for (int e = 0; e < 8; e++) limb[t0 + row_strided_li<LOGN>(e)] = x[e];
            }
            __syncthreads();
        }
        for (int r = 0; r < CROUNDS; r++) {
            const int tile = 4 * r + grp;
            const bool active = tile < G::COL_TILES;
            const int c0 = (active ? tile : tile % G::COL_TILES) * 32;
#pragma unroll
            for (int e = 0; e < 8; e++) x[e] = limb[col_fine_idx<LOGN>(c0, e)];
            if (fp) {
#pragma unroll
                for (int e = 0; e < 8; e++) xd[e] = bits_fp(x[e]);
                inv_col_pass_fp<LOGN>(xd, t.twid + (size_t)pj * G::N, f, as_fp(exch));
#pragma unroll
                for (int e = 0; e < 8; e++) x[e] = fp_to_canonical(xd[e], f);
            } else {
                inv_col_pass<LOGN>(x, t.twi + (size_t)pj * G::N, m, exch);
#pragma unroll
                for (int e = 0; e < 8; e++) x[e] = csub(csub(x[e], m.p2), m.p);
            }
            if (active) {
#pragma unroll
                for (int e = 0; e < 8; e++) data[col_coarse_idx<LOGN>(c0, e)] = x[e];
            }
            __syncthreads();
        }
    }
}

// =============================================================================== key switching
// (1) digit INTT, row pass.  target limb i of ciphertext b: tgt.data + b*tgt.bs + i*N.
// With GALOIS the Galois automorphism is applied while loading: in NTT form it is the pure
// permutation out[g] = in[perm[g]] (SEAL util::apply_galois_ntt); perm maps each row of the
// limb matrix into a single source row, so the gather stays inside one 0.5-4 KB segment.
#ifdef V_NOLOAD   // experiment only: input words synthesised instead of loaded = upper bound of any prefetch / staging scheme
#define VLOAD(e, expr) ((u64)(threadIdx.x * 8u + (e) + blockIdx.x) & 0xffffffffull)
#else
#define VLOAD(e, expr) (expr)
#endif
#ifndef V_OCC_INTT
#define V_OCC_INTT 5
#endif
#ifndef V_OCC_COL
#define V_OCC_COL 4
#endif
template <int LOGN, bool GALOIS>
__global__ void __launch_bounds__(NTT_THREADS, V_OCC_INTT) k_ks_intt_row(KsRoute rt, u64 *D, int L, Tables t) {
    typedef NttGeo<LOGN> G;
    __shared__ u64 smem[NTT_TILE];
    const int i = blockIdx.y, b = blockIdx.z;
    const KsSel sl = route_sel(rt, b);
    const DView tgt = rt.v[sl.src];
    const uint32_t *__restrict__ perm = GALOIS ? route_perm(rt, sl) : nullptr;
    const u64 *in = tgt.data + sl.sentry * tgt.bs + rt.tgt_poly * tgt.ps + (u64)i * G::N;
    u64 *out = D + ((u64)b * L + i) * G::N;
    const ModConst m = load_mod(t, i);
    const int t0 = blockIdx.x * NTT_TILE;
    u64 x[8];
    if (GALOIS) {
        unsigned ix[8];
        load_perm8(ix, perm + t0 + 8 * threadIdx.x);   // static table: before the dependency wait
        pdl_wait();
#pragma unroll
        for (int e = 0; e < 8; e++) x[e] = VLOAD(e, in[ix[e]]);
    } else {
        pdl_wait();
        load8(x, in + t0 + 8 * threadIdx.x);
    }
    const FpConst f = t.fp[i];
    PDL_LATE();   // (inputs are in registers)
    if (f.ok != 0.0) {
        double xd[8];
#pragma unroll
        for (int e = 0; e < 8; e++) xd[e] = fp_from_u64(x[e]);
        inv_row_pass_fp<LOGN>(xd, t.twid + (size_t)i * G::N, f, t0, as_fp(smem));
#pragma unroll
        for (int e = 0; e < 8; e++) out[t0 + row_strided_li<LOGN>(e)] = fp_bits(xd[e]);
        return;
    }
    inv_row_pass<LOGN>(x, t.twi + (size_t)i * G::N, m, t0, smem);
#pragma unroll
    for (int e = 0; e < 8; e++) out[t0 + row_strided_li<LOGN>(e)] = x[e];
}

// (3) mod-up, column pass: digit i (coefficient form, canonical) reduced into prime pj and pushed
// through the first six NTT stages.  y = i*(L+1) + jj; jj == L is the special prime.
template <int LOGN>
__global__ void __launch_bounds__(NTT_THREADS, 5) k_ks_modup_col(const u64 *D, u64 *T1, int L, Tables t) {
    typedef NttGeo<LOGN> G;
    __shared__ u64 smem[NTT_TILE];
    const int i = blockIdx.y / (L + 1), jj = blockIdx.y % (L + 1), b = blockIdx.z;
    const int pj = jj == L ? t.K - 1 : jj;
    if (pj == i) return;  // that limb is taken directly from the NTT-form target
    const u64 *in = D + ((u64)b * L + i) * G::N;
    u64 *out = T1 + (((u64)b * L + i) * (L + 1) + jj) * G::N;
    const ModConst m = load_mod(t, pj);
    const int c0 = blockIdx.x * 32;
    u64 x[8];
    // SEAL reduces the digit modulo q_j only when q_i > q_j; the transform itself accepts any value
    // below 8 q_j, so the Barrett reduction is needed only for a much larger source prime
    const bool need_reduce = t.mod[i].p >= m.p4;
    const FpConst f = t.fp[pj];
    pdl_wait();
#pragma unroll
    for (int e = 0; e < 8; e++) {
        u64 v = in[col_coarse_idx<LOGN>(c0, e)];
        x[e] = need_reduce ? reduce64(v, m) : v;
    }
    if (f.ok != 0.0) {   // x < 4 q_j < 2^43: exact as doubles
        double xd[8];
#pragma unroll
        for (int e = 0; e < 8; e++) xd[e] = fp_from_u64(x[e]);
        fwd_col_pass_fp<LOGN>(xd, t.twfd + (size_t)pj * G::N, f, as_fp(smem));
#pragma unroll
        for (int e = 0; e < 8; e++) out[col_fine_idx<LOGN>(c0, e)] = fp_bits(xd[e]);
        return;
    }
    fwd_col_pass<LOGN>(x, t.twf + (size_t)pj * G::N, m, smem);
#pragma unroll
    for (int e = 0; e < 8; e++) out[col_fine_idx<LOGN>(c0, e)] = x[e];
}

// (2+3) fused: inverse column pass of digit i (its row pass is in D) and, on the same 64 x 32 tile and
// register layout, the mod-up column pass into every other prime -- the digit never returns to memory in
// coefficient form (one launch and one D round trip less than k_inv_col + k_ks_modup_col).
// grid: (COL_TILES, L * nsplit, batch); part p of a digit handles its targets p, p + nsplit, ...
// (nsplit > 1 trades a repeated inverse pass for more CTAs when the batch is too small to fill the GPU).
template <int LOGN>
__global__ void __launch_bounds__(NTT_THREADS, V_OCC_COL) k_ks_invcol_modup(const u64 *D, u64 *T1, int L, int nsplit, Tables t) {
    typedef NttGeo<LOGN> G;
    __shared__ u64 smem[2][NTT_TILE];   // alternating exchange buffers: no barrier needed between passes
    const int i = blockIdx.y / nsplit, part = blockIdx.y % nsplit, b = blockIdx.z;
    const u64 *in = D + ((u64)b * L + i) * G::N;
    const ModConst mi = load_mod(t, i);
    const FpConst fi = t.fp[i];
    const int c0 = blockIdx.x * 32;
    u64 v[8];
    pdl_wait();
#pragma unroll
    for (int e = 0; e < 8; e++) v[e] = VLOAD(e, in[col_fine_idx<LOGN>(c0, e)]);
    if (fi.ok != 0.0) {
        double xd[8];
#pragma unroll
        for (int e = 0; e < 8; e++) xd[e] = bits_fp(v[e]);
        inv_col_pass_fp<LOGN>(xd, t.twid + (size_t)i * G::N, fi, as_fp(smem[0]));
#pragma unroll
        for (int e = 0; e < 8; e++) v[e] = fp_to_canonical(xd[e], fi);
    } else {
        inv_col_pass<LOGN>(v, t.twi + (size_t)i * G::N, mi, smem[0]);
#pragma unroll
        for (int e = 0; e < 8; e++) v[e] = csub(csub(v[e], mi.p2), mi.p);
    }
    PDL_LATE();
    int buf = 1, cnt = 0;
    for (int jj = 0; jj <= L; jj++) {
        const int pj = jj == L ? t.K - 1 : jj;
        if (pj == i) continue;   // that limb is taken directly from the NTT-form target
        if ((cnt++ % nsplit) != part) continue;
        const ModConst m = load_mod(t, pj);
        const FpConst f = t.fp[pj];
        // SEAL reduces the digit modulo q_j only when q_i > q_j; the transform itself accepts any value
        // below 8 q_j, so the Barrett reduction is needed only for a much larger source prime
        const bool need_reduce = mi.p >= m.p4;
        u64 *out = T1 + (((u64)b * L + i) * (L + 1) + jj) * G::N;
        if (f.ok != 0.0) {   // a congruent double below 2^43 in magnitude: the reduction of a large source prime stays on the FP64 pipe
            double xd[8];
#pragma unroll
            for (int e = 0; e < 8; e++) xd[e] = need_reduce ? fp_reduce_big(v[e], f) : fp_from_u64(v[e]);
            fwd_col_pass_fp<LOGN>(xd, t.twfd + (size_t)pj * G::N, f, as_fp(smem[buf]));
#pragma unroll
            for (int e = 0; e < 8; e++) out[col_fine_idx<LOGN>(c0, e)] = fp_bits(xd[e]);
        } else {
            u64 x[8];
#pragma unroll
            for (int e = 0; e < 8; e++) x[e] = need_reduce ? reduce64(v[e], m) : v[e];
            fwd_col_pass<LOGN>(x, t.twf + (size_t)pj * G::N, m, smem[buf]);
#pragma unroll
            for (int e = 0; e < 8; e++) out[col_fine_idx<LOGN>(c0, e)] = x[e];
        }
        buf ^= 1;
    }
}

// (4) mod-up row pass fused with the key inner product: for output limb jj of ciphertext b,
//     acc_k = sum_i NTT_pj(digit_i) (.) ksk[i][k][pj]     (k = 0,1), 128-bit lazy sums,
// one Barrett reduction at the end.  Key limbs stream once from HBM, fully coalesced.
// The output limbs are split by prime size into two launches (JjList): large primes take the
// integer path below, small primes the FP64 kernel k_ks_mac_fp.
struct JjList {
    int n;
    signed char jj[36];
    signed char kh[36];   // 0 = both key components in this CTA; 1 / 2 = only component 0 / 1 (the special-prime limb of a
                          // small batch is split over two CTAs: each repeats the transforms but runs one INTT instead of two)
};
template <int LOGN, bool GALOIS>
__global__ void __launch_bounds__(NTT_THREADS, 2) k_ks_mac(const u64 *T1, KsRoute rt, u64 *ACC, int L, JjList list, int fuse_inv, Tables t) {
    typedef NttGeo<LOGN> G;
    // TMA-staged input tiles of the current / next digit; the current one doubles as the exchange buffer
    __shared__ __align__(128) u64 stage[2][NTT_TILE];
    __shared__ u64 bars[2];
    const int jj = list.jj[blockIdx.y], kh = list.kh[blockIdx.y], b = blockIdx.z;
    const KsSel sl = route_sel(rt, b);
    const DView tgt = rt.v[sl.src];
    const uint32_t *__restrict__ perm = GALOIS ? route_perm(rt, sl) : nullptr;
    const u64 *__restrict__ ksk = route_key(rt, sl);
    const int K = t.K, pj = jj == L ? K - 1 : jj;
    const ModConst m = load_mod(t, pj);
    const tw_t *tw = t.twf + (size_t)pj * G::N;
    const int t0 = blockIdx.x * NTT_TILE;
    u64 lo0[8], hi0[8], lo1[8], hi1[8];
#pragma unroll
    for (int e = 0; e < 8; e++) lo0[e] = hi0[e] = lo1[e] = hi1[e] = 0;
    if (threadIdx.x == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
    }
    __syncthreads();
    pdl_wait();
    // digits that need a transform, in order; their tiles are fetched one ahead by TMA
    auto tile_of = [&](int i) { return T1 + (((u64)b * L + i) * (L + 1) + jj) * G::N + t0; };
    int nxt = 0;                       // next digit whose tile has not been requested yet
    while (nxt < L && nxt == pj) nxt++;
    unsigned ph[2] = {0, 0};
    int slot = 0;
    if (threadIdx.x == 0 && nxt < L) tma_load_tile(stage[0], tile_of(nxt), NTT_TILE * 8, &bars[0]);
    for (int i = 0; i < L; i++) {
        u64 x[8];
        // the key stream comes from HBM: start it before the transform of this digit
        prefetch_l2(ksk + (((u64)i * 2 + 0) * K + pj) * G::N + t0 + 8 * threadIdx.x);
        prefetch_l2(ksk + (((u64)i * 2 + 1) * K + pj) * G::N + t0 + 8 * threadIdx.x);
        if (i == pj) {
            const u64 *in = tgt.data + sl.sentry * tgt.bs + rt.tgt_poly * tgt.ps + (u64)i * G::N;
            if (GALOIS) {
                unsigned ix[8];
                load_perm8(ix, perm + t0 + 8 * threadIdx.x);
#pragma unroll
                for (int e = 0; e < 8; e++) x[e] = in[ix[e]];
            } else {
                load8(x, in + t0 + 8 * threadIdx.x);
            }
        } else {
            // this digit's tile was requested one iteration ago; request the following one now
            int after = i + 1;
            while (after < L && after == pj) after++;
            __syncthreads();  // every thread is done with the other stage buffer (previous digit's exchanges)
            if (threadIdx.x == 0 && after < L) tma_load_tile(stage[slot ^ 1], tile_of(after), NTT_TILE * 8, &bars[slot ^ 1]);
            mbar_wait(&bars[slot], ph[slot]);
            ph[slot] ^= 1;
#pragma unroll
            for (int e = 0; e < 8; e++) x[e] = stage[slot][row_strided_li<LOGN>(e)];
            __syncthreads();  // tile consumed: the buffer now serves as the exchange buffer of the transform
            fwd_row_pass<LOGN>(x, tw, m, t0, stage[slot]);
            slot ^= 1;
        }
        // standard layout: the thread's 8 words are contiguous (4 x 16 B, 64 B apart between threads: every warp
        // load touches 16 lines); tiled layout: word pair v of thread t sits at 512 v + 2 t (4 lines per warp load)
        const int koff = rt.key_tiled ? 2 * threadIdx.x : 8 * threadIdx.x, kstep = rt.key_tiled ? 256 : 1;
        const ulonglong2 *k0 = reinterpret_cast<const ulonglong2 *>(ksk + (((u64)i * 2 + 0) * K + pj) * G::N + t0 + koff);
        const ulonglong2 *k1 = reinterpret_cast<const ulonglong2 *>(ksk + (((u64)i * 2 + 1) * K + pj) * G::N + t0 + koff);
#pragma unroll
        if (kh != 2) {
#pragma unroll
            for (int v = 0; v < 4; v++) {
                ulonglong2 a = __ldg(k0 + kstep * v);
                mac128(lo0[2 * v], hi0[2 * v], x[2 * v], a.x);
                mac128(lo0[2 * v + 1], hi0[2 * v + 1], x[2 * v + 1], a.y);
            }
        }
        if (kh != 1) {
#pragma unroll
            for (int v = 0; v < 4; v++) {
                ulonglong2 c = __ldg(k1 + kstep * v);
                mac128(lo1[2 * v], hi1[2 * v], x[2 * v], c.x);
                mac128(lo1[2 * v + 1], hi1[2 * v + 1], x[2 * v + 1], c.y);
            }
        }
    }
    PDL_LATE();
    if (fuse_inv && jj == L) {
        // special-prime limb: the accumulated tile is exactly the input tile of the mod-down INTT's row pass --
        // run it here (k_inv_row fused), writing the strided-side result over the limb's slot in ACC
        u64 *b0 = ACC + (((u64)b * 2 + 0) * (L + 1) + jj) * G::N + t0;
        u64 *b1 = ACC + (((u64)b * 2 + 1) * (L + 1) + jj) * G::N + t0;
        const tw_t *twi = t.twi + (size_t)pj * G::N;
        u64 r[8];
        __syncthreads();   // every thread is done with the exchange buffers of the last digit
        if (kh != 2) {
#pragma unroll
            for (int e = 0; e < 8; e++) r[e] = barrett128(lo0[e], hi0[e], m);
            inv_row_pass<LOGN>(r, twi, m, t0, stage[0]);
#pragma unroll
            for (int e = 0; e < 8; e++) b0[row_strided_li<LOGN>(e)] = r[e];
        }
        if (kh != 1) {
#pragma unroll
            for (int e = 0; e < 8; e++) r[e] = barrett128(lo1[e], hi1[e], m);
            inv_row_pass<LOGN>(r, twi, m, t0, stage[1]);
#pragma unroll
            for (int e = 0; e < 8; e++) b1[row_strided_li<LOGN>(e)] = r[e];
        }
        return;
    }
    u64 *o0 = ACC + (((u64)b * 2 + 0) * (L + 1) + jj) * G::N + t0 + 8 * threadIdx.x;
    u64 *o1 = ACC + (((u64)b * 2 + 1) * (L + 1) + jj) * G::N + t0 + 8 * threadIdx.x;
#pragma unroll
    for (int v = 0; v < 4; v++) {
        ulonglong2 r0, r1;
        r0.x = barrett128(lo0[2 * v], hi0[2 * v], m);
        r0.y = barrett128(lo0[2 * v + 1], hi0[2 * v + 1], m);
        r1.x = barrett128(lo1[2 * v], hi1[2 * v], m);
        r1.y = barrett128(lo1[2 * v + 1], hi1[2 * v + 1], m);
        reinterpret_cast<ulonglong2 *>(o0)[v] = r0;
        reinterpret_cast<ulonglong2 *>(o1)[v] = r1;
    }
}

// FP64 variant for output limbs with a small prime: transform, products and the running sums all
// stay on the FP64 pipe (|sum| < 2p per term, at most 32 terms: exact), one canonicalisation at the end
#ifndef V_MACFP_OCC
#define V_MACFP_OCC 3
#endif
template <int LOGN, bool GALOIS>
__global__ void __launch_bounds__(NTT_THREADS, V_MACFP_OCC) k_ks_mac_fp(const u64 *T1, KsRoute rt, u64 *ACC, int L, JjList list, int fuse_inv, Tables t) {
    typedef NttGeo<LOGN> G;
    __shared__ __align__(128) u64 stage[2][NTT_TILE];   // TMA-staged tiles; the current one is also the exchange buffer
    __shared__ u64 bars[2];
    const int jj = list.jj[blockIdx.y], b = blockIdx.z;
    const KsSel sl = route_sel(rt, b);
    const DView tgt = rt.v[sl.src];
    const uint32_t *__restrict__ perm = GALOIS ? route_perm(rt, sl) : nullptr;
    const u64 *__restrict__ ksk = route_key(rt, sl);
    const int K = t.K, pj = jj == L ? K - 1 : jj;
    const FpConst f = t.fp[pj];
    const double *tw = t.twfd + (size_t)pj * G::N;
    const int t0 = blockIdx.x * NTT_TILE;
    double a0[8], a1[8];
#pragma unroll
    for (int e = 0; e < 8; e++) a0[e] = a1[e] = 0.0;
    if (threadIdx.x == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
    }
    __syncthreads();
    pdl_wait();
    auto tile_of = [&](int i) { return T1 + (((u64)b * L + i) * (L + 1) + jj) * G::N + t0; };
    int nxt = 0;
    while (nxt < L && nxt == pj) nxt++;
    unsigned ph[2] = {0, 0};
    int slot = 0;
    if (threadIdx.x == 0 && nxt < L) tma_load_tile(stage[0], tile_of(nxt), NTT_TILE * 8, &bars[0]);
    for (int i = 0; i < L; i++) {
        double x[8];
#ifdef V_MACFP_EARLYKEY
        // the digit's key words are requested before its transform: ~300 cycles of L2 latency hidden behind the row pass
        ulonglong2 ka[4], kc[4];
        {
            const int koff = rt.key_tiled ? 2 * threadIdx.x : 8 * threadIdx.x, kstep = rt.key_tiled ? 256 : 1;
            const ulonglong2 *k0 = reinterpret_cast<const ulonglong2 *>(ksk + (((u64)i * 2 + 0) * K + pj) * G::N + t0 + koff);
            const ulonglong2 *k1 = reinterpret_cast<const ulonglong2 *>(ksk + (((u64)i * 2 + 1) * K + pj) * G::N + t0 + koff);
#pragma unroll
            for (int v = 0; v < 4; v++) {
                ka[v] = __ldg(k0 + kstep * v);
                kc[v] = __ldg(k1 + kstep * v);
            }
        }
#else
        prefetch_l2(ksk + (((u64)i * 2 + 0) * K + pj) * G::N + t0 + 8 * threadIdx.x);
        prefetch_l2(ksk + (((u64)i * 2 + 1) * K + pj) * G::N + t0 + 8 * threadIdx.x);
#endif
        if (i == pj) {
            const u64 *in = tgt.data + sl.sentry * tgt.bs + rt.tgt_poly * tgt.ps + (u64)i * G::N;
            u64 xi[8];
            if (GALOIS) {
                unsigned ix[8];
                load_perm8(ix, perm + t0 + 8 * threadIdx.x);
#pragma unroll
                for (int e = 0; e < 8; e++) xi[e] = in[ix[e]];
            } else {
                load8(xi, in + t0 + 8 * threadIdx.x);
            }
#pragma unroll
            for (int e = 0; e < 8; e++) x[e] = fp_from_u64(xi[e]);
        } else {
            int after = i + 1;
            while (after < L && after == pj) after++;
            __syncthreads();
            if (threadIdx.x == 0 && after < L) tma_load_tile(stage[slot ^ 1], tile_of(after), NTT_TILE * 8, &bars[slot ^ 1]);
            mbar_wait(&bars[slot], ph[slot]);
            ph[slot] ^= 1;
#pragma unroll
            for (int e = 0; e < 8; e++) x[e] = bits_fp(stage[slot][row_strided_li<LOGN>(e)]);
            __syncthreads();
            fwd_row_pass_fp<LOGN>(x, tw, f, t0, as_fp(stage[slot]));   // lazy, |x| < 32p
            slot ^= 1;
        }
#ifdef V_MACFP_EARLYKEY
#pragma unroll
        for (int v = 0; v < 4; v++) {
            ulonglong2 a = ka[v], c = kc[v];
#else
        // standard layout: the thread's 8 words are contiguous (4 x 16 B, 64 B apart between threads: every warp
        // load touches 16 lines); tiled layout: word pair v of thread t sits at 512 v + 2 t (4 lines per warp load)
        const int koff = rt.key_tiled ? 2 * threadIdx.x : 8 * threadIdx.x, kstep = rt.key_tiled ? 256 : 1;
        const ulonglong2 *k0 = reinterpret_cast<const ulonglong2 *>(ksk + (((u64)i * 2 + 0) * K + pj) * G::N + t0 + koff);
        const ulonglong2 *k1 = reinterpret_cast<const ulonglong2 *>(ksk + (((u64)i * 2 + 1) * K + pj) * G::N + t0 + koff);
#pragma unroll
        for (int v = 0; v < 4; v++) {
            ulonglong2 a = __ldg(k0 + kstep * v), c = __ldg(k1 + kstep * v);
#endif
            // engine-owned (tiled) key copies hold small-prime limbs as doubles already (k_retile_key)
            const double kax = rt.key_tiled ? bits_fp(a.x) : fp_from_u64(a.x), kay = rt.key_tiled ? bits_fp(a.y) : fp_from_u64(a.y);
            const double kcx = rt.key_tiled ? bits_fp(c.x) : fp_from_u64(c.x), kcy = rt.key_tiled ? bits_fp(c.y) : fp_from_u64(c.y);
            a0[2 * v] = __dadd_rn(a0[2 * v], fp_mulmod(x[2 * v], kax, f));
            a0[2 * v + 1] = __dadd_rn(a0[2 * v + 1], fp_mulmod(x[2 * v + 1], kay, f));
            a1[2 * v] = __dadd_rn(a1[2 * v], fp_mulmod(x[2 * v], kcx, f));
            a1[2 * v + 1] = __dadd_rn(a1[2 * v + 1], fp_mulmod(x[2 * v + 1], kcy, f));
        }
    }
    PDL_LATE();
    if (fuse_inv && jj == L) {   // small special prime: mod-down INTT row pass fused, as in k_ks_mac
        u64 *b0 = ACC + (((u64)b * 2 + 0) * (L + 1) + jj) * G::N + t0;
        u64 *b1 = ACC + (((u64)b * 2 + 1) * (L + 1) + jj) * G::N + t0;
        const double *twi = t.twid + (size_t)pj * G::N;
        __syncthreads();
#pragma unroll
        for (int e = 0; e < 8; e++) a0[e] = fp_reduce(a0[e], f);
        inv_row_pass_fp<LOGN>(a0, twi, f, t0, as_fp(stage[0]));
#pragma unroll
        for (int e = 0; e < 8; e++) b0[row_strided_li<LOGN>(e)] = fp_bits(a0[e]);
#pragma unroll
        for (int e = 0; e < 8; e++) a1[e] = fp_reduce(a1[e], f);
        inv_row_pass_fp<LOGN>(a1, twi, f, t0, as_fp(stage[1]));
#pragma unroll
        for (int e = 0; e < 8; e++) b1[row_strided_li<LOGN>(e)] = fp_bits(a1[e]);
        return;
    }
    u64 r0[8], r1[8];
#pragma unroll
    for (int e = 0; e < 8; e++) {
        r0[e] = fp_to_canonical(a0[e], f);
        r1[e] = fp_to_canonical(a1[e], f);
    }
    store8(ACC + (((u64)b * 2 + 0) * (L + 1) + jj) * G::N + t0 + 8 * threadIdx.x, r0);
    store8(ACC + (((u64)b * 2 + 1) * (L + 1) + jj) * G::N + t0 + 8 * threadIdx.x, r1);
}

// (4c) small-batch variant of the inner product on a thread-block cluster: the L digits of one output tile go to the L
// CTAs of a cluster (blockIdx.x = digit = cluster rank) instead of one CTA looping over them.  Each CTA transforms its digit,
// multiplies it with its two key words and parks the 16 products per thread in its own shared memory; after a cluster
// barrier rank k (k = 0, 1) sums component k over all ranks through distributed shared memory, reduces, and -- for the
// special-prime limb -- continues into the mod-down INTT's row pass.  The critical path of the pipeline's longest kernel
// drops from L transforms + 2 inverse passes to 1 + 1.  Same sums (exact integer / integer-valued FP64 arithmetic), so the
// result is bit-identical to k_ks_mac / k_ks_mac_fp.  Dynamic shared memory: 64 KB ([2][8][256] x (lo, hi); the first
// 16 KB double as the exchange buffer of the forward pass, the component-k block as that of rank k's inverse pass).
template <int LOGN, bool GALOIS>
__global__ void __launch_bounds__(NTT_THREADS, 3) k_ks_mac_cl(const u64 *T1, KsRoute rt, u64 *ACC, int L, int fuse_inv, Tables t) {
    typedef NttGeo<LOGN> G;
    extern __shared__ __align__(128) u64 dsm[];
    cooperative_groups::cluster_group cl = cooperative_groups::this_cluster();
    const int i = blockIdx.x, jj = blockIdx.z % (L + 1), b = blockIdx.z / (L + 1), tid = threadIdx.x;
    const KsSel sl = route_sel(rt, b);
    const DView tgt = rt.v[sl.src];
    const uint32_t *__restrict__ perm = GALOIS ? route_perm(rt, sl) : nullptr;
    const u64 *__restrict__ ksk = route_key(rt, sl);
    const int K = t.K, pj = jj == L ? K - 1 : jj;
    const ModConst m = load_mod(t, pj);
    const FpConst f = t.fp[pj];
    const bool fp = f.ok != 0.0;
    const int t0 = blockIdx.y * NTT_TILE;
    const int koff = rt.key_tiled ? 2 * tid : 8 * tid, kstep = rt.key_tiled ? 256 : 1;
    const ulonglong2 *k0 = reinterpret_cast<const ulonglong2 *>(ksk + (((u64)i * 2 + 0) * K + pj) * G::N + t0 + koff);
    const ulonglong2 *k1 = reinterpret_cast<const ulonglong2 *>(ksk + (((u64)i * 2 + 1) * K + pj) * G::N + t0 + koff);
    prefetch_l2(ksk + (((u64)i * 2 + 0) * K + pj) * G::N + t0 + 8 * tid);
    prefetch_l2(ksk + (((u64)i * 2 + 1) * K + pj) * G::N + t0 + 8 * tid);
    pdl_wait();
    u64 x[8];
    double xd[8];
    if (i == pj) {   // the digit's own prime: the NTT-form limb of the target itself
        const u64 *in = tgt.data + sl.sentry * tgt.bs + rt.tgt_poly * tgt.ps + (u64)i * G::N;
        if (GALOIS) {
            unsigned ix[8];
            load_perm8(ix, perm + t0 + 8 * tid);
#pragma unroll
            for (int e = 0; e < 8; e++) x[e] = in[ix[e]];
        } else {
            load8(x, in + t0 + 8 * tid);
        }
        if (fp) {
#pragma unroll
            for (int e = 0; e < 8; e++) xd[e] = fp_from_u64(x[e]);
        }
    } else {
        const u64 *tile = T1 + (((u64)b * L + i) * (L + 1) + jj) * G::N + t0;
#pragma unroll
        for (int e = 0; e < 8; e++) x[e] = tile[row_strided_li<LOGN>(e)];
        if (fp) {
#pragma unroll
            for (int e = 0; e < 8; e++) xd[e] = bits_fp(x[e]);
            fwd_row_pass_fp<LOGN>(xd, t.twfd + (size_t)pj * G::N, f, t0, as_fp(dsm));
        } else {
            fwd_row_pass<LOGN>(x, t.twf + (size_t)pj * G::N, m, t0, dsm);
        }
        __syncthreads();   // the exchange buffer is about to receive products
    }
    PDL_LATE();
    const int n_k = L < 2 ? 2 : 1;   // components this rank finishes (a single-digit key switch: rank 0 does both)
    if (fp) {
        double *pr = as_fp(dsm);     // [2][8][256]
#pragma unroll
        for (int v = 0; v < 4; v++) {
            ulonglong2 a = __ldg(k0 + kstep * v), c = __ldg(k1 + kstep * v);
            const double kax = rt.key_tiled ? bits_fp(a.x) : fp_from_u64(a.x), kay = rt.key_tiled ? bits_fp(a.y) : fp_from_u64(a.y);
            const double kcx = rt.key_tiled ? bits_fp(c.x) : fp_from_u64(c.x), kcy = rt.key_tiled ? bits_fp(c.y) : fp_from_u64(c.y);
            pr[(2 * v) * 256 + tid] = fp_mulmod(xd[2 * v], kax, f);
            pr[(2 * v + 1) * 256 + tid] = fp_mulmod(xd[2 * v + 1], kay, f);
            pr[(8 + 2 * v) * 256 + tid] = fp_mulmod(xd[2 * v], kcx, f);
            pr[(8 + 2 * v + 1) * 256 + tid] = fp_mulmod(xd[2 * v + 1], kcy, f);
        }
        cl.sync();
        if (i < 2) {
            for (int kk = 0; kk < n_k; kk++) {
                const int k = i + kk;
                double s[8];
#pragma unroll
                for (int e = 0; e < 8; e++) s[e] = 0.0;
                for (int r = 0; r < L; r++) {
                    const double *rp = cl.map_shared_rank(pr, r) + k * 2048 + tid;
#pragma unroll
                    for (int e = 0; e < 8; e++) s[e] = __dadd_rn(s[e], rp[e * 256]);
                }
                u64 *dst = ACC + (((u64)b * 2 + k) * (L + 1) + jj) * G::N + t0;
                if (fuse_inv && jj == L) {
#pragma unroll
                    for (int e = 0; e < 8; e++) s[e] = fp_reduce(s[e], f);
                    __syncthreads();   // own component-k block fully read: it becomes the exchange buffer
                    inv_row_pass_fp<LOGN>(s, t.twid + (size_t)pj * G::N, f, t0, pr + k * 2048);
#pragma unroll
                    for (int e = 0; e < 8; e++) dst[row_strided_li<LOGN>(e)] = fp_bits(s[e]);
                } else {
                    u64 r8[8];
#pragma unroll
                    for (int e = 0; e < 8; e++) r8[e] = fp_to_canonical(s[e], f);
                    store8(dst + 8 * tid, r8);
                }
            }
        }
    } else {
        u64 *plo = dsm, *phi = dsm + 4096;   // [2][8][256] each
#pragma unroll
        for (int v = 0; v < 4; v++) {
            ulonglong2 a = __ldg(k0 + kstep * v), c = __ldg(k1 + kstep * v);
            plo[(2 * v) * 256 + tid] = x[2 * v] * a.x;
            phi[(2 * v) * 256 + tid] = __umul64hi(x[2 * v], a.x);
            plo[(2 * v + 1) * 256 + tid] = x[2 * v + 1] * a.y;
            phi[(2 * v + 1) * 256 + tid] = __umul64hi(x[2 * v + 1], a.y);
            plo[(8 + 2 * v) * 256 + tid] = x[2 * v] * c.x;
            phi[(8 + 2 * v) * 256 + tid] = __umul64hi(x[2 * v], c.x);
            plo[(8 + 2 * v + 1) * 256 + tid] = x[2 * v + 1] * c.y;
            phi[(8 + 2 * v + 1) * 256 + tid] = __umul64hi(x[2 * v + 1], c.y);
        }
        cl.sync();
        if (i < 2) {
            for (int kk = 0; kk < n_k; kk++) {
                const int k = i + kk;
                u64 lo[8], hi[8];
#pragma unroll
                for (int e = 0; e < 8; e++) lo[e] = hi[e] = 0;
                for (int r = 0; r < L; r++) {
                    const u64 *rl = cl.map_shared_rank(plo, r) + k * 2048 + tid;
                    const u64 *rh = cl.map_shared_rank(phi, r) + k * 2048 + tid;
#pragma unroll
                    for (int e = 0; e < 8; e++) {
                        const u64 al = rl[e * 256], ah = rh[e * 256];
                        lo[e] += al;
                        hi[e] += ah + (lo[e] < al);
                    }
                }
                u64 r8[8];
#pragma unroll
                for (int e = 0; e < 8; e++) r8[e] = barrett128(lo[e], hi[e], m);
                u64 *dst = ACC + (((u64)b * 2 + k) * (L + 1) + jj) * G::N + t0;
                if (fuse_inv && jj == L) {
                    __syncthreads();   // own component-k block fully read: it becomes the exchange buffer
                    inv_row_pass<LOGN>(r8, t.twi + (size_t)pj * G::N, m, t0, plo + k * 2048);
#pragma unroll
                    for (int e = 0; e < 8; e++) dst[row_strided_li<LOGN>(e)] = r8[e];
                } else {
                    store8(dst + 8 * tid, r8);
                }
            }
        }
    }
    cl.sync();   // peers may still be reading this CTA's products
}

// (7) mod-down / rescale, column pass: R holds r' = (INTT(last limb) + half) mod q_a for poly
// instance z; the value is carried into prime j as (r' mod q_j) - (half mod q_j) and pushed
// through the first six NTT stages.  R limb of instance z: R.data + z*R.bs.
template <int LOGN>
__global__ void __launch_bounds__(NTT_THREADS, 5) k_md_fwd_col(DView R, u64 *T2, int Lout, int a, Tables t) {
    typedef NttGeo<LOGN> G;
    __shared__ u64 smem[NTT_TILE];
    const int j = blockIdx.y, z = blockIdx.z;
    const u64 *in = R.data + z * R.bs;
    u64 *out = T2 + ((u64)z * Lout + j) * G::N;
    const ModConst m = load_mod(t, j);
    const u64 hm = t.round_half ? t.halfmod[a * t.K + j] : 0;
    const int c0 = blockIdx.x * 32;
    u64 x[8];
    const bool need_reduce = t.mod[a].p >= m.p4;   // else r' + q_j - hm < 8 q_j is already a valid lazy input
    const FpConst f = t.fp[j];
    pdl_wait();
#pragma unroll
    for (int e = 0; e < 8; e++) {
        u64 v = in[col_coarse_idx<LOGN>(c0, e)];
        x[e] = need_reduce ? submod(reduce64(v, m), hm, m.p) : v + m.p - hm;
    }
    if (f.ok != 0.0) {   // x < 5 q_j: exact as doubles
        double xd[8];
#pragma unroll
        for (int e = 0; e < 8; e++) xd[e] = fp_from_u64(x[e]);
        fwd_col_pass_fp<LOGN>(xd, t.twfd + (size_t)j * G::N, f, as_fp(smem));
#pragma unroll
        for (int e = 0; e < 8; e++) out[col_fine_idx<LOGN>(c0, e)] = fp_bits(xd[e]);
        return;
    }
    fwd_col_pass<LOGN>(x, t.twf + (size_t)j * G::N, m, smem);
#pragma unroll
    for (int e = 0; e < 8; e++) out[col_fine_idx<LOGN>(c0, e)] = x[e];
}

// (6+7) fused: inverse column pass of the divisor-prime limb (special prime P for a key switch, last data
// prime for a rescale; its row pass is in R), the "+ half" of SEAL's rounding, and on the same tile the
// column pass of (r' mod q_j) - (half mod q_j) for every remaining prime j.
// grid: (COL_TILES, nsplit, instances); part p handles j = p, p + nsplit, ...
template <int LOGN>
__global__ void __launch_bounds__(NTT_THREADS, V_OCC_COL) k_md_invcol_fwdcol(DView R, u64 *T2, int Lout, int a, int nsplit, Tables t) {
    typedef NttGeo<LOGN> G;
    __shared__ u64 smem[2][NTT_TILE];
    const int part = blockIdx.y, z = blockIdx.z;
    const u64 *in = R.data + z * R.bs;
    const ModConst ma = load_mod(t, a);
    const FpConst fa = t.fp[a];
    const u64 half = t.round_half ? (ma.p >> 1) : 0;
    const int c0 = blockIdx.x * 32;
    u64 v[8];
    pdl_wait();
#pragma unroll
    for (int e = 0; e < 8; e++) v[e] = VLOAD(e, in[col_fine_idx<LOGN>(c0, e)]);
    if (fa.ok != 0.0) {
        double xd[8];
#pragma unroll
        for (int e = 0; e < 8; e++) xd[e] = bits_fp(v[e]);
        inv_col_pass_fp<LOGN>(xd, t.twid + (size_t)a * G::N, fa, as_fp(smem[0]));
#pragma unroll
        for (int e = 0; e < 8; e++) v[e] = csub(fp_to_canonical(xd[e], fa) + half, ma.p);
    } else {
        inv_col_pass<LOGN>(v, t.twi + (size_t)a * G::N, ma, smem[0]);
#pragma unroll
        for (int e = 0; e < 8; e++) v[e] = csub(csub(csub(v[e], ma.p2), ma.p) + half, ma.p);
    }
    PDL_LATE();
    int buf = 1;
    for (int j = part; j < Lout; j += nsplit) {
        const ModConst m = load_mod(t, j);
        const FpConst f = t.fp[j];
        const u64 hm = t.round_half ? t.halfmod[a * t.K + j] : 0;
        const bool need_reduce = ma.p >= m.p4;   // else r' + q_j - hm < 8 q_j is already a valid lazy input
        u64 *out = T2 + ((u64)z * Lout + j) * G::N;
        if (f.ok != 0.0) {   // a congruent double below 2^43 in magnitude (the row pass canonicalises)
            double xd[8];
            const double hmd = fp_from_u64(hm);
#pragma unroll
            for (int e = 0; e < 8; e++)
                xd[e] = need_reduce ? __dadd_rn(fp_reduce_big(v[e], f), -hmd) : fp_from_u64(v[e] + m.p - hm);
            fwd_col_pass_fp<LOGN>(xd, t.twfd + (size_t)j * G::N, f, as_fp(smem[buf]));
#pragma unroll
            for (int e = 0; e < 8; e++) out[col_fine_idx<LOGN>(c0, e)] = fp_bits(xd[e]);
        } else {
            u64 x[8];
#pragma unroll
            for (int e = 0; e < 8; e++) x[e] = need_reduce ? submod(reduce64(v[e], m), hm, m.p) : v[e] + m.p - hm;
            fwd_col_pass<LOGN>(x, t.twf + (size_t)j * G::N, m, smem[buf]);
#pragma unroll
            for (int e = 0; e < 8; e++) out[col_fine_idx<LOGN>(c0, e)] = x[e];
        }
        buf ^= 1;
    }
}

// (8) mod-down / rescale, row pass with the epilogue
//     out = (minuend - NTT(u)) * q_a^-1  [+ base]          mod q_j
// MODE 0 (rescale): no base.  MODE 1 (relinearize): base = in[b][k].  MODE 2 (Galois):
// base = permuted in[b][0] for k == 0 and nothing for k == 1 (SEAL wipes c1 before switching).
// z = b*S + s enumerates (ciphertext, poly).
#ifndef V_MDROW_OCC
#define V_MDROW_OCC 4
#endif
template <int LOGN, int MODE>
__global__ void __launch_bounds__(NTT_THREADS, V_MDROW_OCC) k_md_fwd_row(const u64 *T2, DView minuend, KsRoute rt, int S, int Lout, int a, Tables t) {
    typedef NttGeo<LOGN> G;
    __shared__ u64 smem[NTT_TILE];
    const int j = blockIdx.y, z = blockIdx.z, b = z / S, s = z % S;
    const KsSel sl = route_sel(rt, b);
    const DView base = rt.v[sl.src], dst = rt.v[sl.dst];
    const uint32_t *__restrict__ perm = MODE == 2 ? route_perm(rt, sl) : nullptr;
    const u64 *in = T2 + ((u64)z * Lout + j) * G::N;
    const ModConst m = load_mod(t, j);
    const u64 qi = t.inv[a * t.K + j], qis = t.invs[a * t.K + j];
    const int t0 = blockIdx.x * NTT_TILE;
    u64 x[8];
    const FpConst f = t.fp[j];
    pdl_wait();
#pragma unroll
    for (int e = 0; e < 8; e++) x[e] = VLOAD(e, in[t0 + row_strided_li<LOGN>(e)]);
    const u64 *mi = minuend.data + b * minuend.bs + s * minuend.ps + (u64)j * G::N + t0 + 8 * threadIdx.x;
    u64 *out = dst.data + sl.entry * dst.bs + s * dst.ps + (u64)j * G::N + t0 + 8 * threadIdx.x;
    u64 mv[8], bv[8];
#ifdef V_MDROW_EARLY
    load8(mv, mi);   // the accumulator limb is requested before the transform instead of after it
#endif
    double xd[8];
    const bool fp = f.ok != 0.0;
    if (fp) {
#pragma unroll
        for (int e = 0; e < 8; e++) xd[e] = bits_fp(x[e]);
        fwd_row_pass_fp<LOGN>(xd, t.twfd + (size_t)j * G::N, f, t0, as_fp(smem));   // lazy, |xd| < 32p
    } else {
        fwd_row_pass<LOGN>(x, t.twf + (size_t)j * G::N, m, t0, smem);
    }
    // all epilogue loads are issued before the first store (out may alias base, so the compiler
    // would otherwise serialise load -> store -> load ...)
#ifdef V_NOLOAD
#pragma unroll
    for (int e = 0; e < 8; e++) mv[e] = VLOAD(e, 0) + 5, bv[e] = VLOAD(e, 0) + 9;
    if (false)
#endif
    {
#ifndef V_MDROW_EARLY
        load8(mv, mi);
#endif
        if (MODE == 1) {
            load8(bv, base.data + sl.sentry * base.bs + s * base.ps + (u64)j * G::N + t0 + 8 * threadIdx.x);
        } else if (MODE == 2) {
            if (s == 0) {
                unsigned ix[8];
                load_perm8(ix, perm + t0 + 8 * threadIdx.x);
                const u64 *bp = base.data + sl.sentry * base.bs + (u64)j * G::N;
#pragma unroll
                for (int e = 0; e < 8; e++) bv[e] = bp[ix[e]];
            }
        }
    }
    PDL_LATE();
    // (minuend - NTT(u)) * q_a^-1 without canonicalising the transform output first: the lazy value
    // (< 8p + 2^32) is subtracted from minuend + 9p (a multiple of p, no underflow), one truncated
    // Shoup multiply brings the product to [0,4p), two conditional subtractions make it canonical
    const u64 p9 = m.p4 + m.p4 + m.p;
    if (fp) {   // small prime: the whole epilogue on the FP64 pipe
        const double qd = fp_from_u64(qi);
#pragma unroll
        for (int e = 0; e < 8; e++) {
            double r = fp_mulmod(__dadd_rn(fp_from_u64(mv[e]), -xd[e]), qd, f);
            if (MODE == 1 || (MODE == 2 && s == 0)) r = __dadd_rn(r, fp_from_u64(bv[e]));
            x[e] = fp_to_canonical(r, f);
        }
    } else {
#pragma unroll
        for (int e = 0; e < 8; e++) {
            u64 r = shoup_lazy(mv[e] + p9 - x[e], qi, qis, m.negp);
            r = csub(csub(r, m.p2), m.p);
            if (MODE == 1 || (MODE == 2 && s == 0)) r = addmod(r, bv[e], m.p);
            x[e] = r;
        }
    }
    store8(out, x);
    if (MODE == 2 && rt.has_acc) {
        // add_inplace(acc, rotated) of the rotate-and-sum loop (helper.h:472-476), fused
        u64 *ap = rt.accv.data + sl.entry * rt.accv.bs + s * rt.accv.ps + (u64)j * G::N + t0 + 8 * threadIdx.x;
        u64 av[8];
        load8(av, ap);
#pragma unroll
        for (int e = 0; e < 8; e++) av[e] = addmod(av[e], x[e], m.p);
        store8(ap, av);
    }
}

// =============================================================================== hoisted rotations (SURVEY 8 f4)
// Many rotations of ONE ciphertext (the hot loop of Linear_Transform_*, helper.h:252-257: every rotation acts on the same
// ct_new) can share the digit decomposition: decompose c1 once (digit INTT + mod-up NTT into every prime), then per rotation
// only permute the extended digits (the Galois automorphism is a permutation in NTT form), take the inner product with
// that rotation's key and mod-down.  SEAL permutes BEFORE it lifts the digits to non-negative residues, so the hoisted
// digits differ from SEAL's by multiples of q_i on the negated coefficients: the result decrypts to the same values within
// key-switch noise but is NOT bit-identical -- a separate, tolerance-checked mode, never the default (SURVEY section 7).
//
// (h1) finish the mod-up transform: T1[i][jj] holds the column pass (k_ks_invcol_modup); run the row pass and store the
// canonical NTT values in place; the slot of the digit's own prime receives the NTT-form limb of c1 itself.
template <int LOGN>
__global__ void __launch_bounds__(NTT_THREADS, 4) k_hoist_finish(u64 *T1, DView ct, int L, Tables t) {
    typedef NttGeo<LOGN> G;
    __shared__ u64 smem[NTT_TILE];
    const int i = blockIdx.y / (L + 1), jj = blockIdx.y % (L + 1);
    const int pj = jj == L ? t.K - 1 : jj;
    u64 *tile = T1 + ((u64)i * (L + 1) + jj) * G::N + (u64)blockIdx.x * NTT_TILE;
    const int t0 = blockIdx.x * NTT_TILE;
    u64 x[8];
    if (pj == i) {
        load8(x, ct.data + ct.ps + (u64)i * G::N + t0 + 8 * threadIdx.x);   // poly 1, limb i
        store8(tile + 8 * threadIdx.x, x);
        return;
    }
    const ModConst m = load_mod(t, pj);
    const FpConst f = t.fp[pj];
#pragma unroll
    for (int e = 0; e < 8; e++) x[e] = tile[row_strided_li<LOGN>(e)];
    if (f.ok != 0.0) {
        double xd[8];
#pragma unroll
        for (int e = 0; e < 8; e++) xd[e] = bits_fp(x[e]);
        fwd_row_pass_fp<LOGN>(xd, t.twfd + (size_t)pj * G::N, f, t0, as_fp(smem));
#pragma unroll
        for (int e = 0; e < 8; e++) x[e] = fp_to_canonical(xd[e], f);
    } else {
        fwd_row_pass<LOGN>(x, t.twf + (size_t)pj * G::N, m, t0, smem);
#pragma unroll
        for (int e = 0; e < 8; e++) x[e] = reduce64(x[e], m);
    }
    __syncthreads();   // every thread has read its inputs long ago; the outputs overwrite the same tile
    store8(tile + 8 * threadIdx.x, x);
}

// (h2) per rotation z: acc_k[jj][g] = sum_i T1F[i][jj][perm_z[g]] * ksk_z[i][k][jj][g]; the special-prime limb continues
// into the mod-down INTT's row pass like k_ks_mac.  grid (ROW_TILES, L + 1, rotations).
template <int LOGN>
__global__ void __launch_bounds__(NTT_THREADS, 2) k_hoist_mac(const u64 *T1F, KsRoute rt, u64 *ACC, int L, Tables t) {
    typedef NttGeo<LOGN> G;
    __shared__ u64 smem[NTT_TILE];
    const int jj = L - (int)blockIdx.y, b = blockIdx.z;   // special-prime limb first
    const KsSel sl = route_sel(rt, b);
    const uint32_t *__restrict__ perm = route_perm(rt, sl);
    const u64 *__restrict__ ksk = route_key(rt, sl);
    const int K = t.K, pj = jj == L ? K - 1 : jj;
    const ModConst m = load_mod(t, pj);
    const FpConst f = t.fp[pj];
    const int t0 = blockIdx.x * NTT_TILE;
    unsigned ix[8];
    load_perm8(ix, perm + t0 + 8 * threadIdx.x);
    const int koff = rt.key_tiled ? 2 * threadIdx.x : 8 * threadIdx.x, kstep = rt.key_tiled ? 256 : 1;
    u64 *o0 = ACC + (((u64)b * 2 + 0) * (L + 1) + jj) * G::N + t0;
    u64 *o1 = ACC + (((u64)b * 2 + 1) * (L + 1) + jj) * G::N + t0;
    u64 r0[8], r1[8];
    if (f.ok != 0.0) {
        double a0[8], a1[8];
#pragma unroll
        for (int e = 0; e < 8; e++) a0[e] = a1[e] = 0.0;
        for (int i = 0; i < L; i++) {
            const u64 *src = T1F + ((u64)i * (L + 1) + jj) * G::N;
            const ulonglong2 *k0 = reinterpret_cast<const ulonglong2 *>(ksk + (((u64)i * 2 + 0) * K + pj) * G::N + t0 + koff);
            const ulonglong2 *k1 = reinterpret_cast<const ulonglong2 *>(ksk + (((u64)i * 2 + 1) * K + pj) * G::N + t0 + koff);
#pragma unroll
            for (int v = 0; v < 4; v++) {
                const ulonglong2 a = __ldg(k0 + kstep * v), c = __ldg(k1 + kstep * v);
                const double x0 = fp_from_u64(src[ix[2 * v]]), x1 = fp_from_u64(src[ix[2 * v + 1]]);
                const double kax = rt.key_tiled ? bits_fp(a.x) : fp_from_u64(a.x), kay = rt.key_tiled ? bits_fp(a.y) : fp_from_u64(a.y);
                const double kcx = rt.key_tiled ? bits_fp(c.x) : fp_from_u64(c.x), kcy = rt.key_tiled ? bits_fp(c.y) : fp_from_u64(c.y);
                a0[2 * v] = __dadd_rn(a0[2 * v], fp_mulmod(x0, kax, f));
                a0[2 * v + 1] = __dadd_rn(a0[2 * v + 1], fp_mulmod(x1, kay, f));
                a1[2 * v] = __dadd_rn(a1[2 * v], fp_mulmod(x0, kcx, f));
                a1[2 * v + 1] = __dadd_rn(a1[2 * v + 1], fp_mulmod(x1, kcy, f));
            }
        }
#pragma unroll
        for (int e = 0; e < 8; e++) {
            r0[e] = fp_to_canonical(a0[e], f);
            r1[e] = fp_to_canonical(a1[e], f);
        }
    } else {
        u64 lo0[8], hi0[8], lo1[8], hi1[8];
#pragma unroll
        for (int e = 0; e < 8; e++) lo0[e] = hi0[e] = lo1[e] = hi1[e] = 0;
        for (int i = 0; i < L; i++) {
            const u64 *src = T1F + ((u64)i * (L + 1) + jj) * G::N;
            const ulonglong2 *k0 = reinterpret_cast<const ulonglong2 *>(ksk + (((u64)i * 2 + 0) * K + pj) * G::N + t0 + koff);
            const ulonglong2 *k1 = reinterpret_cast<const ulonglong2 *>(ksk + (((u64)i * 2 + 1) * K + pj) * G::N + t0 + koff);
#pragma unroll
            for (int v = 0; v < 4; v++) {
                const ulonglong2 a = __ldg(k0 + kstep * v), c = __ldg(k1 + kstep * v);
                const u64 x0 = src[ix[2 * v]], x1 = src[ix[2 * v + 1]];
                mac128(lo0[2 * v], hi0[2 * v], x0, a.x);
                mac128(lo0[2 * v + 1], hi0[2 * v + 1], x1, a.y);
                mac128(lo1[2 * v], hi1[2 * v], x0, c.x);
                mac128(lo1[2 * v + 1], hi1[2 * v + 1], x1, c.y);
            }
        }
#pragma unroll
        for (int e = 0; e < 8; e++) {
            r0[e] = barrett128(lo0[e], hi0[e], m);
            r1[e] = barrett128(lo1[e], hi1[e], m);
        }
    }
    if (jj == L) {   // special-prime limb: mod-down INTT row pass fused (its column pass follows in k_md_invcol_fwdcol)
        if (f.ok != 0.0) {
            double xd[8];
#pragma unroll
            for (int e = 0; e < 8; e++) xd[e] = fp_from_u64(r0[e]);
            inv_row_pass_fp<LOGN>(xd, t.twid + (size_t)pj * G::N, f, t0, as_fp(smem));
#pragma unroll
            for (int e = 0; e < 8; e++) o0[row_strided_li<LOGN>(e)] = fp_bits(xd[e]);
            __syncthreads();
#pragma unroll
            for (int e = 0; e < 8; e++) xd[e] = fp_from_u64(r1[e]);
            inv_row_pass_fp<LOGN>(xd, t.twid + (size_t)pj * G::N, f, t0, as_fp(smem));
#pragma unroll
            for (int e = 0; e < 8; e++) o1[row_strided_li<LOGN>(e)] = fp_bits(xd[e]);
        } else {
            inv_row_pass<LOGN>(r0, t.twi + (size_t)pj * G::N, m, t0, smem);
#pragma unroll
            for (int e = 0; e < 8; e++) o0[row_strided_li<LOGN>(e)] = r0[e];
            __syncthreads();
            inv_row_pass<LOGN>(r1, t.twi + (size_t)pj * G::N, m, t0, smem);
#pragma unroll
            for (int e = 0; e < 8; e++) o1[row_strided_li<LOGN>(e)] = r1[e];
        }
        return;
    }
    store8(o0 + 8 * threadIdx.x, r0);
    store8(o1 + 8 * threadIdx.x, r1);
}

// Key-switch keys are static: at registration the engine makes a private copy in which, inside every 2048-word
// tile, word pair v (0..3) of thread t (0..255) is stored at 512 v + 2 t instead of 8 t + 2 v, so that the
// inner-product kernels' 16-byte key loads are contiguous across a warp.
__global__ void k_retile_key(const u64 *src, u64 *dst, int log_n, Tables t) {
    const size_t base = (size_t)blockIdx.x * NTT_TILE;
    // limb of this tile: layout [digit][k][limb j < K][N]; small-prime limbs are stored as doubles so that the
    // FP64 inner-product kernel needs no integer -> double conversion per key word (values < 2^41: exact)
    const bool as_double = t.fp[(int)((base >> log_n) % (size_t)t.K)].ok != 0.0;
    const ulonglong2 *s = reinterpret_cast<const ulonglong2 *>(src + base + 8 * threadIdx.x);
#pragma unroll
    for (int v = 0; v < 4; v++) {
        ulonglong2 w = s[v];
        if (as_double) {
            w.x = fp_bits(fp_from_u64(w.x));
            w.y = fp_bits(fp_from_u64(w.y));
        }
        *reinterpret_cast<ulonglong2 *>(dst + base + 512 * v + 2 * threadIdx.x) = w;
    }
}

// =============================================================================== element-wise
// one thread = two adjacent coefficients of limb instance (z = batch, y = s*L + j)
#define EW_PROLOGUE(LIMBS)                                                      \
    const int s = blockIdx.y / (LIMBS), j = blockIdx.y % (LIMBS);               \
    const u64 c = ((u64)blockIdx.x * blockDim.x + threadIdx.x) * 2;             \
    if (c >= (u64)n) return;                                                    \
    const ModConst m = t.mod[j];

__device__ __forceinline__ const ulonglong2 *vp(const DView &v, int b, int s, int j, int n, u64 c) {
    return reinterpret_cast<const ulonglong2 *>(v.data + b * v.bs + s * v.ps + (u64)j * n + c);
}
__device__ __forceinline__ ulonglong2 *vpw(const DView &v, int b, int s, int j, int n, u64 c) {
    return reinterpret_cast<ulonglong2 *>(v.data + b * v.bs + s * v.ps + (u64)j * n + c);
}

// x * y mod p for canonical operands of a prime below 2^41, on the FP64 pipe (6 exact operations instead of the ~10 wide
// integer multiplies of a 128-bit product + Barrett reduction): keeps the element-wise products memory-bound
__device__ __forceinline__ u64 fp_mulmod_u64(u64 x, u64 y, const FpConst &f) {
    return fp_to_canonical(fp_mulmod(fp_from_u64(x), fp_from_u64(y), f), f);
}

// OP 0 add, 1 sub, 2 negate (b unused)
template <int OP>
__global__ void __launch_bounds__(256) k_ew_addsub(DView a, DView b, DView o, int L, int n, Tables t) {
    EW_PROLOGUE(L)
    ulonglong2 x = *vp(a, blockIdx.z, s, j, n, c), y, r;
    if (OP != 2) y = *vp(b, blockIdx.z, s, j, n, c);
    if (OP == 0) { r.x = addmod(x.x, y.x, m.p); r.y = addmod(x.y, y.y, m.p); }
    if (OP == 1) { r.x = submod(x.x, y.x, m.p); r.y = submod(x.y, y.y, m.p); }
    if (OP == 2) { r.x = x.x ? m.p - x.x : 0; r.y = x.y ? m.p - x.y : 0; }
    *vpw(o, blockIdx.z, s, j, n, c) = r;
}

// every poly of ct times the plaintext (pt batch stride 0 = broadcast)
__global__ void __launch_bounds__(256) k_ew_mul_plain(DView ct, DView pt, DView o, int L, int n, Tables t) {
    EW_PROLOGUE(L)
    ulonglong2 x = *vp(ct, blockIdx.z, s, j, n, c), y = *vp(pt, blockIdx.z, 0, j, n, c), r;
    const FpConst f = t.fp[j];
    if (f.ok != 0.0) {
        r.x = fp_mulmod_u64(x.x, y.x, f);
        r.y = fp_mulmod_u64(x.y, y.y, f);
    } else {
        r.x = mulmod(x.x, y.x, m);
        r.y = mulmod(x.y, y.y, m);
    }
    *vpw(o, blockIdx.z, s, j, n, c) = r;
}

// plain added to poly 0, other polys copied
__global__ void __launch_bounds__(256) k_ew_add_plain(DView ct, DView pt, DView o, int L, int n, Tables t) {
    EW_PROLOGUE(L)
    ulonglong2 x = *vp(ct, blockIdx.z, s, j, n, c), r = x;
    if (s == 0) {
        ulonglong2 y = *vp(pt, blockIdx.z, 0, j, n, c);
        r.x = addmod(x.x, y.x, m.p);
        r.y = addmod(x.y, y.y, m.p);
    }
    *vpw(o, blockIdx.z, s, j, n, c) = r;
}

// ct x ct: out_k = sum_{i+l=k} a_i (.) b_l; sums kept in 128 bits, one reduction per output
template <int SA, int SB>
__global__ void __launch_bounds__(256) k_ew_multiply(DView a, DView b, DView o, int L, int n, Tables t) {
    const int j = blockIdx.y;
    const u64 c = ((u64)blockIdx.x * blockDim.x + threadIdx.x) * 2;
    if (c >= (u64)n) return;
    const ModConst m = t.mod[j];
    ulonglong2 xa[SA], xb[SB];
#pragma unroll
    for (int i = 0; i < SA; i++) xa[i] = *vp(a, blockIdx.z, i, j, n, c);
#pragma unroll
    for (int i = 0; i < SB; i++) xb[i] = *vp(b, blockIdx.z, i, j, n, c);
    const FpConst f = t.fp[j];
    if (f.ok != 0.0) {   // small prime: products and their sums as exact doubles (at most 3 terms of magnitude < 2p each)
        double ax[SA], ay[SA], bx[SB], by[SB];
#pragma unroll
        for (int i = 0; i < SA; i++) { ax[i] = fp_from_u64(xa[i].x); ay[i] = fp_from_u64(xa[i].y); }
#pragma unroll
        for (int i = 0; i < SB; i++) { bx[i] = fp_from_u64(xb[i].x); by[i] = fp_from_u64(xb[i].y); }
#pragma unroll
        for (int k = 0; k < SA + SB - 1; k++) {
            double s0 = 0.0, s1 = 0.0;
#pragma unroll
            for (int i = 0; i < SA; i++) {
                const int l = k - i;
                if (l >= 0 && l < SB) {
                    s0 = __dadd_rn(s0, fp_mulmod(ax[i], bx[l], f));
                    s1 = __dadd_rn(s1, fp_mulmod(ay[i], by[l], f));
                }
            }
            ulonglong2 r;
            r.x = fp_to_canonical(s0, f);
            r.y = fp_to_canonical(s1, f);
            *vpw(o, blockIdx.z, k, j, n, c) = r;
        }
        return;
    }
#pragma unroll
    for (int k = 0; k < SA + SB - 1; k++) {
        u64 l0 = 0, h0 = 0, l1 = 0, h1 = 0;
#pragma unroll
        for (int i = 0; i < SA; i++) {
            const int l = k - i;
            if (l >= 0 && l < SB) {
                mac128(l0, h0, xa[i].x, xb[l].x);
                mac128(l1, h1, xa[i].y, xb[l].y);
            }
        }
        ulonglong2 r;
        r.x = barrett128(l0, h0, m);
        r.y = barrett128(l1, h1, m);
        *vpw(o, blockIdx.z, k, j, n, c) = r;
    }
}

// out = in[0] + in[1] + ... + in[B-1]  (sequential modular adds, SEAL add_many order)
__global__ void __launch_bounds__(256) k_ew_add_many(DView in, DView o, int B, int L, int n, Tables t) {
    EW_PROLOGUE(L)
    ulonglong2 acc = *vp(in, 0, s, j, n, c);
    for (int b = 1; b < B; b++) {
        ulonglong2 y = *vp(in, b, s, j, n, c);
        acc.x = addmod(acc.x, y.x, m.p);
        acc.y = addmod(acc.y, y.y, m.p);
    }
    *vpw(o, 0, s, j, n, c) = acc;
}

// out[m] = in[m] + in[M + m] + ... + in[(G-1) M + m] for m = blockIdx.z: G independent add_many over strided groups
// (the reduce-scatter sum of sharded workloads).  Lazy 64-bit sum: 8 canonical words of a prime below 2^61 fit, so
// the running sum is brought back below p after every 7 further terms; one reduction at the end gives the same
// canonical residue as add_many's sequential modular adds.
__global__ void __launch_bounds__(256) k_ew_add_many_grouped(DView in, DView o, int G, int M, int L, int n, Tables t) {
    EW_PROLOGUE(L)
    const int b = blockIdx.z;
    ulonglong2 acc = *vp(in, b, s, j, n, c);
    for (int g = 1; g < G; g++) {
        ulonglong2 y = *vp(in, g * M + b, s, j, n, c);
        acc.x += y.x;
        acc.y += y.y;
        if (g % 7 == 0) { acc.x = reduce64(acc.x, m); acc.y = reduce64(acc.y, m); }
    }
    acc.x = reduce64(acc.x, m);
    acc.y = reduce64(acc.y, m);
    *vpw(o, b, s, j, n, c) = acc;
}

// fused multiply + add_many: out = sum_b a[b] (.) b[b]
//   PLAIN: b is a plaintext batch (every poly of a[b] times pt[b]), output size = size of a
//   else : size-2 x size-2 ciphertext products, output size 3 (Linear_Transform_Cipher)
// 128-bit lazy sums with a reduction every 16 terms; identical to SEAL's sequential
// multiply + add_inplace because the sum is taken modulo q either way.
template <bool PLAIN>
__global__ void __launch_bounds__(256) k_ew_mul_sum(DView a, DView b, DView o, int B, int L, int n, Tables t) {
    const int s = PLAIN ? blockIdx.y / L : 0, j = blockIdx.y % L;
    const u64 c = ((u64)blockIdx.x * blockDim.x + threadIdx.x) * 2;
    if (c >= (u64)n) return;
    const ModConst m = t.mod[j];
    const FpConst f = t.fp[j];
    if (f.ok != 0.0) {
        // small prime: every product reduced on the FP64 pipe (|term| < 2p), running sums exact in doubles, brought back
        // below p every 256 terms (256 * 2p < 2^50)
        if (PLAIN) {
            double s0 = 0.0, s1 = 0.0;
            for (int q = 0; q < B; q++) {
                ulonglong2 x = *vp(a, q, s, j, n, c), y = *vp(b, q, 0, j, n, c);
                s0 = __dadd_rn(s0, fp_mulmod(fp_from_u64(x.x), fp_from_u64(y.x), f));
                s1 = __dadd_rn(s1, fp_mulmod(fp_from_u64(x.y), fp_from_u64(y.y), f));
                if ((q & 255) == 255) { s0 = fp_reduce(s0, f); s1 = fp_reduce(s1, f); }
            }
            ulonglong2 r;
            r.x = fp_to_canonical(s0, f);
            r.y = fp_to_canonical(s1, f);
            *vpw(o, 0, s, j, n, c) = r;
        } else {
            double sx[3] = {0.0, 0.0, 0.0}, sy[3] = {0.0, 0.0, 0.0};
            for (int q = 0; q < B; q++) {
                ulonglong2 a0 = *vp(a, q, 0, j, n, c), a1 = *vp(a, q, 1, j, n, c);
                ulonglong2 b0 = *vp(b, q, 0, j, n, c), b1 = *vp(b, q, 1, j, n, c);
                const double a0x = fp_from_u64(a0.x), a0y = fp_from_u64(a0.y), a1x = fp_from_u64(a1.x), a1y = fp_from_u64(a1.y);
                const double b0x = fp_from_u64(b0.x), b0y = fp_from_u64(b0.y), b1x = fp_from_u64(b1.x), b1y = fp_from_u64(b1.y);
                sx[0] = __dadd_rn(sx[0], fp_mulmod(a0x, b0x, f)); sy[0] = __dadd_rn(sy[0], fp_mulmod(a0y, b0y, f));
                sx[1] = __dadd_rn(sx[1], __dadd_rn(fp_mulmod(a0x, b1x, f), fp_mulmod(a1x, b0x, f)));
                sy[1] = __dadd_rn(sy[1], __dadd_rn(fp_mulmod(a0y, b1y, f), fp_mulmod(a1y, b0y, f)));
                sx[2] = __dadd_rn(sx[2], fp_mulmod(a1x, b1x, f)); sy[2] = __dadd_rn(sy[2], fp_mulmod(a1y, b1y, f));
                if ((q & 127) == 127) {
#pragma unroll
                    for (int k = 0; k < 3; k++) { sx[k] = fp_reduce(sx[k], f); sy[k] = fp_reduce(sy[k], f); }
                }
            }
#pragma unroll
            for (int k = 0; k < 3; k++) {
                ulonglong2 r;
                r.x = fp_to_canonical(sx[k], f);
                r.y = fp_to_canonical(sy[k], f);
                *vpw(o, 0, k, j, n, c) = r;
            }
        }
        return;
    }
    if (PLAIN) {
        u64 l0 = 0, h0 = 0, l1 = 0, h1 = 0;
        for (int q = 0; q < B; q++) {
            ulonglong2 x = *vp(a, q, s, j, n, c), y = *vp(b, q, 0, j, n, c);
            mac128(l0, h0, x.x, y.x);
            mac128(l1, h1, x.y, y.y);
            if ((q & 15) == 15) {
                l0 = barrett128(l0, h0, m); h0 = 0;
                l1 = barrett128(l1, h1, m); h1 = 0;
            }
        }
        ulonglong2 r;
        r.x = barrett128(l0, h0, m);
        r.y = barrett128(l1, h1, m);
        *vpw(o, 0, s, j, n, c) = r;
    } else {
        u64 lo[3][2], hi[3][2];
#pragma unroll
        for (int k = 0; k < 3; k++) lo[k][0] = lo[k][1] = hi[k][0] = hi[k][1] = 0;
        for (int q = 0; q < B; q++) {
            ulonglong2 a0 = *vp(a, q, 0, j, n, c), a1 = *vp(a, q, 1, j, n, c);
            ulonglong2 b0 = *vp(b, q, 0, j, n, c), b1 = *vp(b, q, 1, j, n, c);
            mac128(lo[0][0], hi[0][0], a0.x, b0.x); mac128(lo[0][1], hi[0][1], a0.y, b0.y);
            mac128(lo[1][0], hi[1][0], a0.x, b1.x); mac128(lo[1][1], hi[1][1], a0.y, b1.y);
            mac128(lo[1][0], hi[1][0], a1.x, b0.x); mac128(lo[1][1], hi[1][1], a1.y, b0.y);
            mac128(lo[2][0], hi[2][0], a1.x, b1.x); mac128(lo[2][1], hi[2][1], a1.y, b1.y);
            if ((q & 7) == 7) {
#pragma unroll
                for (int k = 0; k < 3; k++) {
                    lo[k][0] = barrett128(lo[k][0], hi[k][0], m); hi[k][0] = 0;
                    lo[k][1] = barrett128(lo[k][1], hi[k][1], m); hi[k][1] = 0;
                }
            }
        }
#pragma unroll
        for (int k = 0; k < 3; k++) {
            ulonglong2 r;
            r.x = barrett128(lo[k][0], hi[k][0], m);
            r.y = barrett128(lo[k][1], hi[k][1], m);
            *vpw(o, 0, k, j, n, c) = r;
        }
    }
}

// constant-coefficient sums (ckks_multiply_const_sum).  The residues of the encoded constants are computed on the host
// (as ckks_encode_scalar does) and travel in the kernel parameters: words [g][i][j] of the G x T term constants of the
// launch, then [g][j] of the G constants added to poly 0.
#define CONST_SUM_WORDS 2048
#define CONST_SUM_GROUPS 8
struct ConstSumTable {
    u64 r[CONST_SUM_WORDS];
};
// out[g * M + m] = sum_{i < T} in[i * M + m] (.) r[g][i]  (+ r0[g] on poly 0), for g < G <= CONST_SUM_GROUPS, m = blockIdx.z.
// Every input word is read once for all G outputs; a term whose residue is zero on this limb is not read.  The products
// are summed lazily (FP64 below 2^41, 128-bit otherwise, as k_ew_mul_sum) and reduced once: the canonical result equals
// SEAL's multiply_plain by each constant plaintext, add_many, add_plain.
__global__ void __launch_bounds__(256) k_ew_const_sum(DView in, DView o, const __grid_constant__ ConstSumTable tab, int G,
                                                      int T, int M, int L, int n, Tables t) {
    EW_PROLOGUE(L)
    const int b = blockIdx.z;
    const u64 *r = tab.r, *r0 = tab.r + (size_t)G * T * L;
    const FpConst f = t.fp[j];
    if (f.ok != 0.0) {
        double s0[CONST_SUM_GROUPS], s1[CONST_SUM_GROUPS];
#pragma unroll
        for (int g = 0; g < CONST_SUM_GROUPS; g++) s0[g] = s1[g] = 0.0;
        for (int i = 0; i < T; i++) {
            bool any = false;
            for (int g = 0; g < G; g++) any |= r[(g * T + i) * L + j] != 0;
            if (!any) continue;
            const ulonglong2 x = *vp(in, i * M + b, s, j, n, c);
            const double xx = fp_from_u64(x.x), xy = fp_from_u64(x.y);
#pragma unroll
            for (int g = 0; g < CONST_SUM_GROUPS; g++) {
                if (g >= G) break;
                const u64 w = r[(g * T + i) * L + j];
                if (!w) continue;
                const double wd = fp_from_u64(w);
                s0[g] = __dadd_rn(s0[g], fp_mulmod(xx, wd, f));
                s1[g] = __dadd_rn(s1[g], fp_mulmod(xy, wd, f));
            }
            if ((i & 255) == 255) {   // |term| < 2p: 256 of them stay below 2^50
#pragma unroll
                for (int g = 0; g < CONST_SUM_GROUPS; g++) { s0[g] = fp_reduce(s0[g], f); s1[g] = fp_reduce(s1[g], f); }
            }
        }
#pragma unroll
        for (int g = 0; g < CONST_SUM_GROUPS; g++) {
            if (g >= G) break;
            ulonglong2 v;
            v.x = fp_to_canonical(s0[g], f);
            v.y = fp_to_canonical(s1[g], f);
            if (s == 0) { v.x = addmod(v.x, r0[g * L + j], m.p); v.y = addmod(v.y, r0[g * L + j], m.p); }
            *vpw(o, g * M + b, s, j, n, c) = v;
        }
        return;
    }
    u64 lo0[CONST_SUM_GROUPS], hi0[CONST_SUM_GROUPS], lo1[CONST_SUM_GROUPS], hi1[CONST_SUM_GROUPS];
#pragma unroll
    for (int g = 0; g < CONST_SUM_GROUPS; g++) lo0[g] = hi0[g] = lo1[g] = hi1[g] = 0;
    for (int i = 0; i < T; i++) {
        bool any = false;
        for (int g = 0; g < G; g++) any |= r[(g * T + i) * L + j] != 0;
        if (!any) continue;
        const ulonglong2 x = *vp(in, i * M + b, s, j, n, c);
#pragma unroll
        for (int g = 0; g < CONST_SUM_GROUPS; g++) {
            if (g >= G) break;
            const u64 w = r[(g * T + i) * L + j];
            if (!w) continue;
            mac128(lo0[g], hi0[g], x.x, w);
            mac128(lo1[g], hi1[g], x.y, w);
        }
        if ((i & 15) == 15) {   // 16 products of residues below 2^61 fit in 128 bits
#pragma unroll
            for (int g = 0; g < CONST_SUM_GROUPS; g++) {
                lo0[g] = barrett128(lo0[g], hi0[g], m); hi0[g] = 0;
                lo1[g] = barrett128(lo1[g], hi1[g], m); hi1[g] = 0;
            }
        }
    }
#pragma unroll
    for (int g = 0; g < CONST_SUM_GROUPS; g++) {
        if (g >= G) break;
        ulonglong2 v;
        v.x = barrett128(lo0[g], hi0[g], m);
        v.y = barrett128(lo1[g], hi1[g], m);
        if (s == 0) { v.x = addmod(v.x, r0[g * L + j], m.p); v.y = addmod(v.y, r0[g * L + j], m.p); }
        *vpw(o, g * M + b, s, j, n, c) = v;
    }
}

// strided limb copy (mod-switch drop into a differently laid out view)
__global__ void __launch_bounds__(256) k_ew_copy(DView a, DView o, int L, int n) {
    const int s = blockIdx.y / L, j = blockIdx.y % L;
    const u64 c = ((u64)blockIdx.x * blockDim.x + threadIdx.x) * 2;
    if (c >= (u64)n) return;
    *vpw(o, blockIdx.z, s, j, n, c) = *vp(a, blockIdx.z, s, j, n, c);
}

__global__ void k_fill_i32(int32_t *p, int n, int32_t v) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}
// flags[b] cleared when any word of polys 1.. of entry b is non-zero
__global__ void __launch_bounds__(256) k_transparent(DView ct, int32_t *flags, int L, int n) {
    const int s = 1 + blockIdx.y / L, j = blockIdx.y % L;
    const u64 c = ((u64)blockIdx.x * blockDim.x + threadIdx.x) * 2;
    if (c >= (u64)n) return;
    ulonglong2 x = *vp(ct, blockIdx.z, s, j, n, c);
    if (x.x | x.y) flags[blockIdx.z] = 0;
}
