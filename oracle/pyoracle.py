"""ctypes binding of the CPU oracle (oracle/ckks_oracle.c).

TEST INFRASTRUCTURE ONLY -- see oracle/ckks_oracle.h.  Imported by tests/, by
__graft_entry__.smoke() and by bench.py's cpu_baseline / --impl reference legs, never by
the product package.  PARITY UNPINNED: the reference has no golden vectors for this path
and SEAL itself is not available here.

All polynomial data are numpy uint64 arrays shaped [S][L][N] (ciphertexts), [L][N]
(plaintexts), [K][N] (secret key), [2][K][N] (public key), [K-1][2][K][N] (key-switch keys).
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libckks_oracle.so")

_u64p = C.POINTER(C.c_uint64)
_f64p = C.POINTER(C.c_double)
_intp = C.POINTER(C.c_int)


def _host_stamp():
    """content hash of the oracle sources + the host CPU's feature flags: the library is compiled
    -march=native, so a copy built on another machine (this repository travels to the GPU box with its
    built artefacts) must be rebuilt rather than trusted by modification time"""
    import hashlib
    h = hashlib.sha256()
    for f in ("ckks_oracle.c", "ckks_oracle.h", "Makefile"):
        with open(os.path.join(_HERE, f), "rb") as fh:
            h.update(fh.read())
    try:
        with open("/proc/cpuinfo") as fh:
            for line in fh:
                if line.startswith("flags") or line.startswith("model name"):
                    h.update(line.encode())
                    if line.startswith("flags"):
                        break
    except OSError:
        pass
    return h.hexdigest()


def build(force=False):
    global _LIB_PATH
    stamp_path = _LIB_PATH + ".hoststamp"
    stamp = _host_stamp()
    if not force and os.path.exists(_LIB_PATH) and os.path.exists(stamp_path):
        with open(stamp_path) as fh:
            if fh.read().strip() == stamp:
                return _LIB_PATH
    src_dir = os.path.dirname(_LIB_PATH)
    if not os.access(src_dir, os.W_OK):
        # a read-only tree built on another host: compile a private copy in a temporary directory instead
        import atexit
        import shutil
        import tempfile
        src_dir = tempfile.mkdtemp(prefix="ckks_oracle_")
        atexit.register(shutil.rmtree, src_dir, True)
        for f in ("ckks_oracle.c", "ckks_oracle.h", "Makefile"):
            shutil.copy(os.path.join(_HERE, f), src_dir)
        _LIB_PATH = os.path.join(src_dir, "libckks_oracle.so")
        stamp_path = _LIB_PATH + ".hoststamp"
    import fcntl
    with open(_LIB_PATH + ".lock", "w") as lock:          # one builder at a time (torchrun ranks, xdist workers)
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and os.path.exists(_LIB_PATH) and os.path.exists(stamp_path) and open(stamp_path).read().strip() == stamp:
                return _LIB_PATH
            subprocess.check_call(["make", "-C", src_dir, "-s", "-B", "libckks_oracle.so"])
            with open(stamp_path, "w") as fh:
                fh.write(stamp + "\n")
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return _LIB_PATH


def _load():
    build()
    lib = C.CDLL(_LIB_PATH)
    sig = {
        "orc_coeff_modulus_create": (C.c_int, [C.c_int, _intp, C.c_int, _u64p]),
        "orc_bfv_default": (C.c_int, [C.c_int, _u64p, C.c_int]),
        "orc_max_bit_count": (C.c_int, [C.c_int]),
        "orc_is_prime": (C.c_int, [C.c_uint64]),
        "orc_create": (C.c_void_p, [C.c_int, C.c_int, _u64p]),
        "orc_destroy": (None, [C.c_void_p]),
        "orc_set_rounding": (None, [C.c_void_p, C.c_int]),
        "orc_prime": (C.c_uint64, [C.c_void_p, C.c_int]),
        "orc_psi": (C.c_uint64, [C.c_void_p, C.c_int]),
        "orc_ntt": (None, [C.c_void_p, C.c_int, _u64p]),
        "orc_intt": (None, [C.c_void_p, C.c_int, _u64p]),
        "orc_ntt_naive": (None, [C.c_void_p, C.c_int, _u64p, _u64p]),
        "orc_add": (None, [C.c_void_p, C.c_int, C.c_int, _u64p, _u64p, _u64p]),
        "orc_sub": (None, [C.c_void_p, C.c_int, C.c_int, _u64p, _u64p, _u64p]),
        "orc_negate": (None, [C.c_void_p, C.c_int, C.c_int, _u64p, _u64p]),
        "orc_multiply": (None, [C.c_void_p, C.c_int, C.c_int, C.c_int, _u64p, _u64p, _u64p]),
        "orc_multiply_plain": (None, [C.c_void_p, C.c_int, C.c_int, _u64p, _u64p, _u64p]),
        "orc_add_plain": (None, [C.c_void_p, C.c_int, C.c_int, _u64p, _u64p, _u64p]),
        "orc_is_transparent": (C.c_int, [C.c_void_p, C.c_int, C.c_int, _u64p]),
        "orc_ksk_words": (C.c_size_t, [C.c_void_p]),
        "orc_switch_key": (None, [C.c_void_p, C.c_int, _u64p, _u64p, _u64p]),
        "orc_relinearize": (None, [C.c_void_p, C.c_int, _u64p, _u64p, _u64p]),
        "orc_apply_galois": (None, [C.c_void_p, C.c_int, _u64p, C.c_uint64, _u64p, _u64p]),
        "orc_galois_permute_limb": (None, [C.c_void_p, C.c_uint64, _u64p, _u64p]),
        "orc_galois_elt_from_step": (C.c_uint64, [C.c_void_p, C.c_int]),
        "orc_naf": (C.c_int, [C.c_int, _intp, C.c_int]),
        "orc_rescale": (None, [C.c_void_p, C.c_int, C.c_int, _u64p, _u64p]),
        "orc_mod_switch_drop": (None, [C.c_void_p, C.c_int, C.c_int, _u64p, _u64p]),
        "orc_gen_secret": (None, [C.c_void_p, C.c_uint64, _u64p]),
        "orc_gen_public": (None, [C.c_void_p, C.c_uint64, _u64p, _u64p]),
        "orc_gen_ksk": (None, [C.c_void_p, C.c_uint64, _u64p, _u64p, _u64p]),
        "orc_gen_relin_key": (None, [C.c_void_p, C.c_uint64, _u64p, _u64p]),
        "orc_gen_galois_key": (None, [C.c_void_p, C.c_uint64, _u64p, C.c_uint64, _u64p]),
        "orc_encrypt": (None, [C.c_void_p, C.c_uint64, C.c_int, _u64p, _u64p, _u64p]),
        "orc_encrypt_symmetric": (None, [C.c_void_p, C.c_uint64, C.c_int, _u64p, _u64p, _u64p]),
        "orc_decrypt": (None, [C.c_void_p, C.c_int, C.c_int, _u64p, _u64p, _u64p]),
        "orc_encode": (None, [C.c_void_p, C.c_int, _f64p, C.c_int, C.c_double, _u64p]),
        "orc_encode_const": (None, [C.c_void_p, C.c_int, C.c_double, C.c_double, _u64p]),
        "orc_decode": (None, [C.c_void_p, C.c_int, _u64p, C.c_double, _f64p]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = _load()
    return _lib


def _p(a):
    assert a.dtype == np.uint64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_u64p)


def _c(a):
    return np.ascontiguousarray(a, dtype=np.uint64)


def coeff_modulus_create(log_n, bit_sizes):
    bits = (C.c_int * len(bit_sizes))(*bit_sizes)
    out = np.zeros(len(bit_sizes), dtype=np.uint64)
    rc = lib().orc_coeff_modulus_create(log_n, bits, len(bit_sizes), _p(out))
    if rc != 0:
        raise ValueError("failed to find enough qualifying primes")
    return [int(x) for x in out]


def bfv_default(log_n):
    out = np.zeros(32, dtype=np.uint64)
    cnt = lib().orc_bfv_default(log_n, _p(out), 32)
    if cnt < 0:
        raise ValueError("no default modulus for this degree")
    return [int(x) for x in out[:cnt]]


def max_bit_count(log_n):
    return lib().orc_max_bit_count(log_n)


def is_prime(v):
    return bool(lib().orc_is_prime(v))


def naf(steps):
    out = (C.c_int * 40)()
    cnt = lib().orc_naf(steps, out, 40)
    return [out[i] for i in range(cnt)]


class Oracle:
    """One CKKS parameter set (degree N = 2**log_n, K primes, last one special)."""

    def __init__(self, log_n, primes):
        self.log_n = log_n
        self.n = 1 << log_n
        self.primes = [int(p) for p in primes]
        self.K = len(self.primes)
        arr = np.array(self.primes, dtype=np.uint64)
        self._h = lib().orc_create(log_n, self.K, _p(arr))
        if not self._h:
            raise ValueError("invalid CKKS parameters")

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.orc_destroy(self._h)
            self._h = None

    def set_rounding(self, on):
        lib().orc_set_rounding(self._h, int(on))   # 0 floor, 1/True round, 2 round key switch only, 3 round rescale only

    def psi(self, j):
        return int(lib().orc_psi(self._h, j))

    # ---- NTT
    def ntt(self, j, a):
        a = _c(a).copy()
        lib().orc_ntt(self._h, j, _p(a))
        return a

    def intt(self, j, a):
        a = _c(a).copy()
        lib().orc_intt(self._h, j, _p(a))
        return a

    def ntt_naive(self, j, a):
        a = _c(a)
        out = np.empty_like(a)
        lib().orc_ntt_naive(self._h, j, _p(a), _p(out))
        return out

    # ---- element-wise
    def _sl(self, ct):
        assert ct.ndim == 3 and ct.shape[2] == self.n
        return ct.shape[0], ct.shape[1]

    def add(self, a, b):
        a, b = _c(a), _c(b)
        S, L = self._sl(a)
        out = np.empty_like(a)
        lib().orc_add(self._h, S, L, _p(a), _p(b), _p(out))
        return out

    def sub(self, a, b):
        a, b = _c(a), _c(b)
        S, L = self._sl(a)
        out = np.empty_like(a)
        lib().orc_sub(self._h, S, L, _p(a), _p(b), _p(out))
        return out

    def negate(self, a):
        a = _c(a)
        S, L = self._sl(a)
        out = np.empty_like(a)
        lib().orc_negate(self._h, S, L, _p(a), _p(out))
        return out

    def multiply(self, a, b):
        a, b = _c(a), _c(b)
        Sa, L = self._sl(a)
        Sb, _ = self._sl(b)
        out = np.empty((Sa + Sb - 1, L, self.n), dtype=np.uint64)
        lib().orc_multiply(self._h, Sa, Sb, L, _p(a), _p(b), _p(out))
        return out

    def multiply_plain(self, ct, pt):
        ct, pt = _c(ct), _c(pt)
        S, L = self._sl(ct)
        out = np.empty_like(ct)
        lib().orc_multiply_plain(self._h, S, L, _p(ct), _p(pt), _p(out))
        return out

    def add_plain(self, ct, pt):
        ct, pt = _c(ct), _c(pt)
        S, L = self._sl(ct)
        out = np.empty_like(ct)
        lib().orc_add_plain(self._h, S, L, _p(ct), _p(pt), _p(out))
        return out

    def is_transparent(self, ct):
        ct = _c(ct)
        S, L = self._sl(ct)
        return bool(lib().orc_is_transparent(self._h, S, L, _p(ct)))

    # ---- key switching
    def ksk_shape(self):
        return (self.K - 1, 2, self.K, self.n)

    def relinearize(self, ct3, rlk):
        ct3, rlk = _c(ct3), _c(rlk)
        S, L = self._sl(ct3)
        assert S == 3
        out = np.empty((2, L, self.n), dtype=np.uint64)
        lib().orc_relinearize(self._h, L, _p(ct3), _p(rlk), _p(out))
        return out

    def galois_elt(self, steps):
        g = int(lib().orc_galois_elt_from_step(self._h, steps))
        if g == 0:
            raise ValueError("step count too large")
        return g

    def galois_permute(self, g, limb):
        limb = _c(limb)
        out = np.empty_like(limb)
        lib().orc_galois_permute_limb(self._h, g, _p(limb), _p(out))
        return out

    def apply_galois(self, ct, g, gk):
        ct, gk = _c(ct), _c(gk)
        S, L = self._sl(ct)
        assert S == 2
        out = np.empty_like(ct)
        lib().orc_apply_galois(self._h, L, _p(ct), g, _p(gk), _p(out))
        return out

    def rotate(self, ct, steps, gkeys):
        """SEAL Evaluator::rotate_vector with SEAL's NAF fallback (SURVEY A.6).
        gkeys: dict galois_elt -> key array."""
        if steps == 0:
            return _c(ct).copy()
        g = self.galois_elt(steps)
        if g in gkeys:
            return self.apply_galois(ct, g, gkeys[g])
        parts = naf(steps)
        if len(parts) == 1:
            raise KeyError("Galois key not present")
        out = _c(ct)
        for s in parts:
            if abs(s) == self.n // 2:
                continue
            out = self.rotate(out, s, gkeys)
        return out

    # ---- rescale / mod switch
    def rescale(self, ct):
        ct = _c(ct)
        S, L = self._sl(ct)
        out = np.empty((S, L - 1, self.n), dtype=np.uint64)
        lib().orc_rescale(self._h, S, L, _p(ct), _p(out))
        return out

    def mod_switch(self, x):
        """drop the last limb of a ciphertext [S][L][N] or plaintext [L][N]"""
        x = _c(x)
        return np.ascontiguousarray(x[..., :-1, :])

    # ---- keys / encryption / encoding
    def gen_secret(self, seed):
        sk = np.empty((self.K, self.n), dtype=np.uint64)
        lib().orc_gen_secret(self._h, seed, _p(sk))
        return sk

    def gen_public(self, seed, sk):
        pk = np.empty((2, self.K, self.n), dtype=np.uint64)
        lib().orc_gen_public(self._h, seed, _p(_c(sk)), _p(pk))
        return pk

    def gen_relin_key(self, seed, sk):
        k = np.empty(self.ksk_shape(), dtype=np.uint64)
        lib().orc_gen_relin_key(self._h, seed, _p(_c(sk)), _p(k))
        return k

    def gen_galois_key(self, seed, sk, g):
        k = np.empty(self.ksk_shape(), dtype=np.uint64)
        lib().orc_gen_galois_key(self._h, seed, _p(_c(sk)), g, _p(k))
        return k

    def default_galois_elts(self):
        """SEAL KeyGenerator::galois_keys() default set: steps +-2^i and conjugation."""
        elts = [2 * self.n - 1]
        for i in range(self.log_n - 1):
            elts.append(self.galois_elt(1 << i))
            elts.append(self.galois_elt(-(1 << i)))
        return sorted(set(elts))

    def gen_galois_keys(self, seed, sk, elts=None, steps=None):
        if elts is None:
            elts = self.default_galois_elts() if steps is None else [self.galois_elt(s) for s in steps]
        return {g: self.gen_galois_key(seed + 7919 * i + 1, sk, g) for i, g in enumerate(elts)}

    def encrypt(self, seed, pk, pt):
        pt = _c(pt)
        L = pt.shape[0]
        ct = np.empty((2, L, self.n), dtype=np.uint64)
        lib().orc_encrypt(self._h, seed, L, _p(_c(pk)), _p(pt), _p(ct))
        return ct

    def encrypt_symmetric(self, seed, sk, pt):
        pt = _c(pt)
        L = pt.shape[0]
        ct = np.empty((2, L, self.n), dtype=np.uint64)
        lib().orc_encrypt_symmetric(self._h, seed, L, _p(_c(sk)), _p(pt), _p(ct))
        return ct

    def decrypt(self, sk, ct):
        ct = _c(ct)
        S, L = self._sl(ct)
        pt = np.empty((L, self.n), dtype=np.uint64)
        lib().orc_decrypt(self._h, S, L, _p(_c(sk)), _p(ct), _p(pt))
        return pt

    def encode(self, values, scale, L=None):
        L = self.K - 1 if L is None else L
        pt = np.empty((L, self.n), dtype=np.uint64)
        if np.isscalar(values):
            lib().orc_encode_const(self._h, L, float(values), float(scale), _p(pt))
        else:
            v = np.ascontiguousarray(values, dtype=np.float64)
            lib().orc_encode(self._h, L, v.ctypes.data_as(_f64p), len(v), float(scale), _p(pt))
        return pt

    def decode(self, pt, scale):
        pt = _c(pt)
        out = np.empty(self.n // 2, dtype=np.float64)
        lib().orc_decode(self._h, pt.shape[0], _p(pt), float(scale), out.ctypes.data_as(_f64p))
        return out
