"""Host-side mirror of the SEAL `Evaluator` surface the reference calls, over the C ABI.

Python is only plumbing here: torch supplies device memory and streams, ctypes forwards to
libckks_b200.so (hand-written sm_100a kernels).  There is no eager / CPU fallback -- every
method ends in a C-ABI call and raises if the library or a CUDA device is missing.

Objects mirror SEAL's (reference: helper.h, logistic_regression_ckks.cpp) but are *batched*:
a `Ciphertext` holds B independent ciphertexts of the same size, level and scale in one
[B][S][cap][N] device tensor so that one call fills the GPU (SURVEY.md section 7, "Occupancy").
`limbs` plays the role of SEAL's parms_id (level with L RNS limbs); `cap` is the limb capacity
of the buffer so that mod-switching is a metadata change.
"""
import ctypes as C
import math

import numpy as np
import torch

from . import capi
from .capi import View, check


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class Context:
    """SEAL EncryptionParameters + SEALContext for CKKS (N = 2**log_n, primes[-1] special)."""

    def __init__(self, log_n, primes, device=0):
        self.lib = capi.load()
        self.log_n = int(log_n)
        self.n = 1 << self.log_n
        self.primes = [int(p) for p in primes]
        self.K = len(self.primes)
        self.device = torch.device("cuda", device)
        arr = (C.c_uint64 * self.K)(*self.primes)
        h = C.c_void_p()
        check(self.lib.ckks_ctx_create(self.log_n, self.K, arr, device, C.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            self.lib.ckks_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def top_limbs(self):
        return self.K - 1

    def total_bits(self, limbs):
        """ContextData::total_coeff_modulus_bit_count at the level with `limbs` primes"""
        q = 1
        for p in self.primes[:limbs]:
            q *= p
        return q.bit_length()

    def set_rounding(self, mode):
        """0 / False floor, 1 / True round (default), 2 round in key switching only, 3 round in rescale only"""
        check(self.lib.ckks_ctx_set_rounding(self._h, int(mode)))

    def set_workspace_cap(self, nbytes):
        check(self.lib.ckks_ctx_set_workspace_cap(self._h, int(nbytes)))

    def set_chain_lanes(self, lanes):
        check(self.lib.ckks_ctx_set_chain_lanes(self._h, int(lanes)))

    def reserve(self, batch, limbs):
        check(self.lib.ckks_ctx_reserve(self._h, batch, limbs))

    def launch_count(self):
        return int(self.lib.ckks_ctx_launch_count(self._h))

    def reset_launch_count(self):
        self.lib.ckks_ctx_reset_launch_count(self._h)

    def galois_elt(self, steps):
        g = int(self.lib.ckks_galois_elt_from_step(self._h, steps))
        if g == 0:
            raise capi.CkksInvalidArgument("step count too large")
        return g

    def ksk_shape(self):
        return (self.K - 1, 2, self.K, self.n)

    # ---- buffers
    def empty(self, batch, size, limbs, cap=None, scale=1.0):
        cap = limbs if cap is None else cap
        data = torch.empty((batch, size, cap, self.n), dtype=torch.int64, device=self.device)
        return Ciphertext(self, data, limbs, scale)

    def upload(self, arr, cap=None, scale=1.0):
        """numpy uint64 [B][S][L][N] (or [S][L][N]) -> device Ciphertext"""
        a = np.ascontiguousarray(arr, dtype=np.uint64)
        if a.ndim == 3:
            a = a[None]
        B, S, L, N = a.shape
        assert N == self.n
        out = self.empty(B, S, L, cap, scale)
        out.data[:, :, :L, :].copy_(torch.from_numpy(a.view(np.int64)))
        return out

    def upload_plain(self, arr, cap=None, scale=1.0):
        """numpy uint64 [L][N] or [B][L][N] -> Plaintext (size-1 view)"""
        a = np.ascontiguousarray(arr, dtype=np.uint64)
        if a.ndim == 2:
            a = a[None]
        return self.upload(a[:, None], cap, scale)

    def upload_key(self, arr):
        a = np.ascontiguousarray(arr, dtype=np.uint64)
        assert a.shape == self.ksk_shape()
        return torch.from_numpy(a.view(np.int64)).to(self.device)


class Ciphertext:
    """B ciphertexts (or plaintexts when size == 1) at one level, in device memory."""

    __slots__ = ("ctx", "data", "limbs", "scale")

    def __init__(self, ctx, data, limbs, scale=1.0):
        assert data.dim() == 4 and data.dtype == torch.int64 and data.is_contiguous()
        self.ctx, self.data, self.limbs, self.scale = ctx, data, int(limbs), float(scale)

    batch = property(lambda self: self.data.shape[0])
    size = property(lambda self: self.data.shape[1])
    cap = property(lambda self: self.data.shape[2])

    def view(self):
        n = self.ctx.n
        return View(self.data.data_ptr(), self.size * self.cap * n, self.cap * n, self.batch, self.size, self.limbs, 0)

    def numpy(self):
        """active limbs as numpy uint64 [B][S][L][N]"""
        return self.data[:, :, : self.limbs, :].contiguous().cpu().numpy().view(np.uint64)

    def clone(self):
        return Ciphertext(self.ctx, self.data.clone(), self.limbs, self.scale)

    def like(self, size=None, limbs=None, scale=None):
        size = self.size if size is None else size
        data = torch.empty((self.batch, size, self.cap, self.ctx.n), dtype=torch.int64, device=self.data.device)
        return Ciphertext(self.ctx, data, self.limbs if limbs is None else limbs, self.scale if scale is None else scale)

    def __getitem__(self, idx):
        """sub-batch (a view, no copy)"""
        if isinstance(idx, int):
            idx = slice(idx, idx + 1)
        return Ciphertext(self.ctx, self.data[idx], self.limbs, self.scale)


Plaintext = Ciphertext  # a plaintext is a size-1 batch entry


class KeySet:
    """SEAL RelinKeys + GaloisKeys: device-resident key-switching keys."""

    def __init__(self, ctx):
        self.ctx = ctx
        h = C.c_void_p()
        check(ctx.lib.ckks_keyset_create(ctx._h, C.byref(h)))
        self._h = h
        self._keep = []
        self.relin = None
        self.galois = {}

    def set_relin(self, key_tensor):
        self._keep.append(key_tensor)
        self.relin = key_tensor
        check(self.ctx.lib.ckks_keyset_set_relin(self._h, key_tensor.data_ptr()))

    def set_galois(self, galois_elt, key_tensor):
        self._keep.append(key_tensor)
        self.galois[int(galois_elt)] = key_tensor
        check(self.ctx.lib.ckks_keyset_set_galois(self._h, int(galois_elt), key_tensor.data_ptr()))

    def has_galois(self, galois_elt):
        return bool(self.ctx.lib.ckks_keyset_has_galois(self._h, int(galois_elt)))

    def __del__(self):
        try:
            if self._h:
                self.ctx.lib.ckks_keyset_destroy(self._h)
                self._h = None
        except Exception:
            pass


class Evaluator:
    """SEAL 3.4.5 Evaluator member names and error behaviour, batched, on the GPU."""

    def __init__(self, ctx):
        self.ctx = ctx
        self.lib = ctx.lib
        self.h = ctx._h

    # ---- SEAL-side checks (SURVEY.md 8(b) "Error convention")
    @staticmethod
    def _same(a, b):
        if a.limbs != b.limbs or a.batch != b.batch:
            raise capi.CkksInvalidArgument("encrypted1 and encrypted2 parameter mismatch")

    @staticmethod
    def _same_scale(a, b):
        if a.scale != b.scale:
            raise capi.CkksInvalidArgument("scale mismatch")

    def _scale_ok(self, scale, limbs):
        if scale <= 0 or int(math.log2(scale)) >= self.ctx.total_bits(limbs):
            raise capi.CkksInvalidArgument("scale out of bounds")

    def _check_transparent(self, ct):
        flags = torch.empty(ct.batch, dtype=torch.int32, device=ct.data.device)
        v = ct.view()
        check(self.lib.ckks_is_transparent(self.h, C.byref(v), flags.data_ptr(), _stream()))
        if bool(flags.any().item()):
            raise capi.CkksLogicError("result ciphertext is transparent")

    # ---- element-wise
    def add(self, a, b, out=None):
        self._same(a, b)
        self._same_scale(a, b)
        if a.size != b.size:
            raise capi.CkksInvalidArgument("add: ciphertext sizes differ")  # engine keeps sizes equal
        out = a.like() if out is None else out
        out.limbs = a.limbs
        va, vb, vo = a.view(), b.view(), out.view()
        check(self.lib.ckks_add(self.h, C.byref(va), C.byref(vb), C.byref(vo), _stream()))
        out.limbs, out.scale = a.limbs, a.scale
        return out

    def add_inplace(self, a, b):
        return self.add(a, b, out=a)

    def sub(self, a, b, out=None):
        self._same(a, b)
        self._same_scale(a, b)
        out = a.like() if out is None else out
        out.limbs = a.limbs
        va, vb, vo = a.view(), b.view(), out.view()
        check(self.lib.ckks_sub(self.h, C.byref(va), C.byref(vb), C.byref(vo), _stream()))
        out.limbs, out.scale = a.limbs, a.scale
        return out

    def negate_inplace(self, a):
        va = a.view()
        check(self.lib.ckks_negate(self.h, C.byref(va), C.byref(va), _stream()))
        return a

    def add_many(self, cts, out=None):
        """sum over the batch dimension of one Ciphertext -> batch-1 Ciphertext"""
        out = cts[0:1].like() if out is None else out
        out.limbs = cts.limbs
        vi, vo = cts.view(), out.view()
        check(self.lib.ckks_add_many(self.h, C.byref(vi), C.byref(vo), _stream()))
        out.limbs, out.scale = cts.limbs, cts.scale
        return out

    def add_many_grouped(self, cts, groups, out=None):
        """batch G*M -> batch M: out[m] = sum_g cts[g*M + m] (mod q), add_many of every strided group in one kernel"""
        if groups < 1 or cts.batch % groups:
            raise capi.CkksInvalidArgument("add_many_grouped: in batch must be groups x out batch")
        out = cts[0:cts.batch // groups].like() if out is None else out
        out.limbs = cts.limbs
        vi, vo = cts.view(), out.view()
        check(self.lib.ckks_add_many_grouped(self.h, C.byref(vi), int(groups), C.byref(vo), _stream()))
        out.limbs, out.scale = cts.limbs, cts.scale
        return out

    def multiply_const_sum(self, cts, coeffs, pt_scales, constant=None, groups=1, out=None):
        """Constant-coefficient sums of T terms for `groups` sets of coefficients, in one kernel:
            out[g*M + m] = sum_i cts_i[m] * coeffs[g][i]  (+ constant[g])
        bit-identical to SEAL's multiply_plain(cts_i, encode(coeffs[g][i], pt_scales[g][i])), add_many and
        add_plain(encode(constant[g], result scale)).

        cts       : a list of T Ciphertexts of batch M (each with its own scale), or one Ciphertext whose batch is T*M
                    (entry i*M + m is term i of sum m)
        coeffs    : [groups][T] (or [T] when groups == 1)
        pt_scales : the scale each coefficient is encoded at: a number, [T] (every group) or [groups][T]
        constant  : None or [groups] values added to poly 0, encoded at the result scale
        As SEAL's add requires, every term's ct.scale * pt_scale must be the same number, which is the result's scale
        ("scale mismatch" otherwise); "scale out of bounds" as multiply_plain.  Returns a Ciphertext of batch groups * M."""
        if isinstance(cts, Ciphertext):
            cts = [cts]
        cts = list(cts)
        coeffs = np.asarray(coeffs, dtype=np.float64).reshape(groups, -1)
        T = coeffs.shape[1] if len(cts) == 1 else len(cts)
        if len(cts) == 1 and cts[0].batch % T:
            raise capi.CkksInvalidArgument("multiply_const_sum: in batch must be terms x out batch / groups")
        if coeffs.shape[1] != T:
            raise capi.CkksInvalidArgument("multiply_const_sum: coeffs must have groups x terms entries")
        first = cts[0]
        for c in cts[1:]:
            if c.limbs != first.limbs or c.batch != first.batch or c.size != first.size:
                raise capi.CkksInvalidArgument("encrypted1 and encrypted2 parameter mismatch")
        pt = np.broadcast_to(np.asarray(pt_scales, dtype=np.float64), (groups, T))
        ct_scales = [c.scale for c in cts] if len(cts) == T else [first.scale] * T
        scale = ct_scales[0] * float(pt[0, 0])
        for g in range(groups):
            for i in range(T):
                if ct_scales[i] * float(pt[g, i]) != scale:
                    raise capi.CkksInvalidArgument("scale mismatch")
        self._scale_ok(scale, first.limbs)
        if len(cts) == 1:
            src = first
        else:   # one [T*M] input: the terms side by side (active limbs only)
            L = first.limbs
            src = Ciphertext(first.ctx, torch.cat([c.data[:, :, :L] for c in cts], dim=0), L, first.scale)
        M = src.batch // T
        if out is None:
            out = Ciphertext(self.ctx, torch.empty((groups * M, src.size, src.cap, self.ctx.n), dtype=torch.int64,
                                                   device=src.data.device), src.limbs, scale)
        out.limbs = src.limbs
        cf = np.ascontiguousarray(coeffs)
        ps = np.ascontiguousarray(pt)
        if constant is not None:
            k0 = np.ascontiguousarray(np.asarray(constant, dtype=np.float64).reshape(groups))
            s0 = np.full(groups, scale)
            k0p, s0p = k0.ctypes.data, s0.ctypes.data
        else:
            k0p = s0p = None
        vi, vo = src.view(), out.view()
        check(self.lib.ckks_multiply_const_sum(self.h, C.byref(vi), int(T), int(groups), cf.ctypes.data, ps.ctypes.data,
                                               k0p, s0p, C.byref(vo), _stream()))
        out.scale = scale
        return out

    def multiply(self, a, b, out=None):
        """ct x ct; b may be a single ciphertext multiplied into every entry of a"""
        if a.limbs != b.limbs or (a.batch != b.batch and b.batch != 1):
            raise capi.CkksInvalidArgument("encrypted1 and encrypted2 parameter mismatch")
        scale = a.scale * b.scale
        self._scale_ok(scale, a.limbs)
        out = a.like(size=a.size + b.size - 1) if out is None else out
        out.limbs = a.limbs
        va, vb, vo = a.view(), b.view(), out.view()
        check(self.lib.ckks_multiply(self.h, C.byref(va), C.byref(vb), C.byref(vo), _stream()))
        out.limbs, out.scale = a.limbs, scale
        return out

    def multiply_plain(self, ct, pt, out=None, check_transparent=False):
        if ct.limbs != pt.limbs:
            raise capi.CkksInvalidArgument("encrypted and plain parameter mismatch")
        scale = ct.scale * pt.scale
        self._scale_ok(scale, ct.limbs)
        out = ct.like() if out is None else out
        out.limbs = ct.limbs
        vc, vp, vo = ct.view(), pt.view(), out.view()
        check(self.lib.ckks_multiply_plain(self.h, C.byref(vc), C.byref(vp), C.byref(vo), _stream()))
        out.limbs, out.scale = ct.limbs, scale
        if check_transparent:
            self._check_transparent(out)
        return out

    def multiply_plain_inplace(self, ct, pt):
        return self.multiply_plain(ct, pt, out=ct)

    def add_plain(self, ct, pt, out=None):
        if ct.limbs != pt.limbs:
            raise capi.CkksInvalidArgument("encrypted and plain parameter mismatch")
        self._same_scale(ct, pt)
        out = ct.like() if out is None else out
        out.limbs = ct.limbs
        vc, vp, vo = ct.view(), pt.view(), out.view()
        check(self.lib.ckks_add_plain(self.h, C.byref(vc), C.byref(vp), C.byref(vo), _stream()))
        out.limbs, out.scale = ct.limbs, ct.scale
        return out

    def add_plain_inplace(self, ct, pt):
        return self.add_plain(ct, pt, out=ct)

    # ---- key switching
    def relinearize(self, ct, keys, out=None):
        if ct.size == 2:   # SEAL: nothing to do
            return ct
        if keys.relin is None:
            raise capi.CkksInvalidArgument("relin_keys is not valid for encryption parameters")
        out = ct.like(size=2) if out is None else out
        out.limbs = ct.limbs
        vi, vo = ct.view(), out.view()
        check(self.lib.ckks_relinearize(self.h, C.byref(vi), keys.relin.data_ptr(), C.byref(vo), _stream()))
        out.limbs, out.scale = ct.limbs, ct.scale
        return out

    def apply_galois(self, ct, galois_elt, keys, out=None):
        if not keys.has_galois(galois_elt):
            raise capi.CkksInvalidArgument("Galois key not present")
        out = ct.like() if out is None else out
        out.limbs = ct.limbs
        vi, vo = ct.view(), out.view()
        check(self.lib.ckks_apply_galois(self.h, C.byref(vi), int(galois_elt), keys.galois[int(galois_elt)].data_ptr(),
                                         C.byref(vo), _stream()))
        out.limbs, out.scale = ct.limbs, ct.scale
        return out

    def rotate_vector(self, ct, steps, keys, out=None, scratch=None):
        out = ct.like() if out is None else out
        out.limbs = ct.limbs
        vi, vo = ct.view(), out.view()
        vs = None
        if steps != 0 and not keys.has_galois(self.ctx.galois_elt(steps)):
            scratch = ct.like() if scratch is None else scratch   # composite step: NAF ping-pong
            scratch.limbs = ct.limbs
            vs = scratch.view()
        check(self.lib.ckks_rotate(self.h, keys._h, C.byref(vi), int(steps), C.byref(vo),
                                   C.byref(vs) if vs is not None else None, _stream()))
        out.scale = ct.scale
        return out

    # ---- rescale / mod switch
    def rescale_to_next(self, ct, out=None):
        if ct.limbs < 2:
            raise capi.CkksInvalidArgument("end of modulus switching chain reached")
        out = ct.like() if out is None else out
        vi, vo = ct.view(), out.view()
        vo.limbs = ct.limbs - 1
        check(self.lib.ckks_rescale(self.h, C.byref(vi), C.byref(vo), _stream()))
        out.scale = ct.scale / float(self.ctx.primes[ct.limbs - 1])
        out.limbs = ct.limbs - 1
        return out

    def rescale_to_next_inplace(self, ct):
        return self.rescale_to_next(ct, out=ct)

    def mod_switch_to_next_inplace(self, x):
        if x.limbs < 2:
            raise capi.CkksInvalidArgument("end of modulus switching chain reached")
        x.limbs -= 1   # limb capacity stays: dropping the last limb is metadata only
        return x

    def mod_switch_to_inplace(self, x, limbs):
        if limbs > x.limbs:
            raise capi.CkksInvalidArgument("cannot switch to higher level modulus")
        x.limbs = limbs
        return x

    def mod_switch_to(self, x, limbs):
        """non-destructive: a new object at the lower level that SHARES STORAGE with `x` (mod-switching is a metadata
        change here; SEAL's mod_switch_to returns a copy).  Treat the result as read-only or .clone() it: an in-place op
        on either object (add_inplace, multiply_plain_inplace, rescale with out=...) writes through to the other.  The
        workloads in this package only read such views."""
        if limbs > x.limbs:
            raise capi.CkksInvalidArgument("cannot switch to higher level modulus")
        return Ciphertext(x.ctx, x.data, limbs, x.scale)

    # ---- CKKSEncoder on the device (include/ckks_b200.h: ckks_encode / ckks_encode_scalar / ckks_decode)
    def encode(self, values, scale, limbs=None, cap=None):
        """CKKSEncoder::encode(vector<double>, scale, plain), batched: `values` is a float64 CUDA
        tensor [B][count] (count <= N/2); returns a batch of B plaintexts in NTT form."""
        ctx = self.ctx
        limbs = ctx.top_limbs if limbs is None else limbs
        if values.dim() == 1:
            values = values[None]
        values = values.to(device=ctx.device, dtype=torch.float64).contiguous()
        if values.shape[1] > ctx.n // 2:
            raise capi.CkksInvalidArgument("values has invalid size")
        out = ctx.empty(values.shape[0], 1, limbs, cap=cap, scale=scale)
        vo = out.view()
        check(self.lib.ckks_encode(self.h, values.data_ptr(), values.shape[1], float(scale), C.byref(vo), _stream()))
        return out

    def encode_scalar(self, value, scale, limbs=None, batch=1, cap=None):
        """CKKSEncoder::encode(double, scale, plain): the same constant in every slot"""
        limbs = self.ctx.top_limbs if limbs is None else limbs
        out = self.ctx.empty(batch, 1, limbs, cap=cap, scale=scale)
        vo = out.view()
        check(self.lib.ckks_encode_scalar(self.h, float(value), float(scale), C.byref(vo), _stream()))
        return out

    def decode(self, pt):
        """CKKSEncoder::decode(plain, vector<double>&) -> float64 CUDA tensor [B][N/2]"""
        if pt.data.shape[1] != 1:
            raise capi.CkksInvalidArgument("decode expects plaintexts (size 1)")
        out = torch.empty((pt.batch, self.ctx.n // 2), dtype=torch.float64, device=self.ctx.device)
        vi = pt.view()
        check(self.lib.ckks_decode(self.h, C.byref(vi), float(pt.scale), out.data_ptr(), _stream()))
        return out

    # ---- KeyGenerator / Encryptor randomness on the device (ckks_sample)
    TERNARY, NORMAL, UNIFORM = 0, 1, 2

    def sample(self, kind, seed, stream_id, count, limbs):
        """count polynomials over primes [0, limbs) -> int64 CUDA tensor [count][limbs][N]; ternary and
        normal (sigma 3.2, clipped) polynomials come back in NTT form.  `seed`: 32 bytes from a CSPRNG (ChaCha20 key,
        ckks_sample_keyed) or an int (reproducible test stream with at most 64 bits of entropy, ckks_sample)."""
        out = self.ctx.empty(count, 1, limbs)
        vo = out.view()
        if isinstance(seed, (bytes, bytearray)):
            if len(seed) != 32:
                raise capi.CkksInvalidArgument("sample: the key must be 32 bytes")
            check(self.lib.ckks_sample_keyed(self.h, int(kind), bytes(seed), int(stream_id), C.byref(vo), _stream()))
        else:
            check(self.lib.ckks_sample(self.h, int(kind), int(seed) & (2 ** 64 - 1), int(stream_id), C.byref(vo), _stream()))
        return out.data[:, 0]

    # ---- raw NTT (tests / encoder)
    def ntt_forward(self, tensor, first_prime=0):
        """tensor: [P][L][N] int64, limb l uses prime first_prime + l; in place"""
        P, L, N = tensor.shape
        check(self.lib.ckks_ntt_forward(self.h, tensor.data_ptr(), P, L, first_prime, L * N, _stream()))
        return tensor

    def ntt_inverse(self, tensor, first_prime=0):
        P, L, N = tensor.shape
        check(self.lib.ckks_ntt_inverse(self.h, tensor.data_ptr(), P, L, first_prime, L * N, _stream()))
        return tensor

    # ---- batched rotations with per-entry steps, fused products
    def rotate_plan(self, ct, plan, out=None, scratch=None):
        """entry b of the result = rotate_vector(ct[b] or the single ct, plan.steps[b])"""
        if out is None:
            out = Ciphertext(self.ctx, torch.empty((plan.batch, 2, ct.cap, self.ctx.n), dtype=torch.int64,
                                                   device=ct.data.device), ct.limbs, ct.scale)
        if scratch is None and plan.rounds > 1:
            scratch = out.like()
        out.limbs = ct.limbs
        vi, vo = ct.view(), out.view()
        vs = None
        if scratch is not None:
            scratch.limbs = ct.limbs
            vs = scratch.view()
        check(self.lib.ckks_rotate_plan(self.h, plan._h, C.byref(vi), C.byref(vo),
                                        C.byref(vs) if vs is not None else None, _stream()))
        out.scale = ct.scale
        return out

    def rotate_plan_hoisted(self, ct, plan, out=None):
        """SURVEY 8(f4), opt-in: all rotations of `plan` applied to the single ciphertext `ct` with one shared digit
        decomposition.  Needs a Galois key for every step itself; same decrypted values as rotate_plan within
        key-switch noise, NOT bit-identical polynomials."""
        if ct.batch != 1:
            raise capi.CkksInvalidArgument("hoisted rotations act on one ciphertext")
        if out is None:
            out = Ciphertext(self.ctx, torch.empty((plan.batch, 2, ct.cap, self.ctx.n), dtype=torch.int64,
                                                   device=ct.data.device), ct.limbs, ct.scale)
        out.limbs = ct.limbs
        vi, vo = ct.view(), out.view()
        check(self.lib.ckks_rotate_plan_hoisted(self.h, plan._h, C.byref(vi), C.byref(vo), _stream()))
        out.scale = ct.scale
        return out

    def rotate_sum_chain(self, dup, acc, steps, count, keys, scratch=None):
        """`count` times: dup = rotate_vector(dup, steps); acc += dup (fused, CUDA-graph replayed).
        Returns the Ciphertext that holds dup afterwards (dup's or scratch's storage)."""
        if dup.limbs != acc.limbs or dup.batch != acc.batch:
            raise capi.CkksInvalidArgument("encrypted1 and encrypted2 parameter mismatch")
        if dup.scale != acc.scale:
            raise capi.CkksInvalidArgument("scale mismatch")
        scratch = dup.like() if scratch is None else scratch
        scratch.limbs, scratch.scale = dup.limbs, dup.scale
        va, vb, vc = dup.view(), scratch.view(), acc.view()
        where = C.c_int(0)
        check(self.lib.ckks_rotate_sum_chain(self.h, keys._h, C.byref(va), C.byref(vb), C.byref(vc), int(steps), int(count),
                                             C.byref(where), _stream()))
        return scratch if where.value else dup

    def multiply_plain_sum(self, cts, pts, out=None):
        """multiply_plain of every batch entry with its plaintext, then add_many, in one kernel.  (SEAL's per-product
        "result ciphertext is transparent" check is not applied to the fused partial products; use multiply_plain(...,
        check_transparent=True) where that error behaviour is wanted -- the reference's drivers avoid it with epsilon.)"""
        if cts.limbs != pts.limbs or cts.batch != pts.batch:
            raise capi.CkksInvalidArgument("encrypted and plain parameter mismatch")
        scale = cts.scale * pts.scale
        self._scale_ok(scale, cts.limbs)
        out = cts[0:1].like() if out is None else out
        out.limbs = cts.limbs
        vc, vp, vo = cts.view(), pts.view(), out.view()
        check(self.lib.ckks_multiply_plain_sum(self.h, C.byref(vc), C.byref(vp), C.byref(vo), _stream()))
        out.scale = scale
        return out

    def multiply_sum(self, a, b, out=None):
        """multiply (2x2 -> 3) of every batch entry pair, then add_many, in one kernel"""
        self._same(a, b)
        scale = a.scale * b.scale
        self._scale_ok(scale, a.limbs)
        out = a[0:1].like(size=3) if out is None else out
        out.limbs = a.limbs
        va, vb, vo = a.view(), b.view(), out.view()
        check(self.lib.ckks_multiply_sum(self.h, C.byref(va), C.byref(vb), C.byref(vo), _stream()))
        out.scale = scale
        return out


class RotPlan:
    """a fixed list of rotation steps (one per batch entry) compiled into batched rounds"""

    def __init__(self, ctx, keys, steps):
        self.ctx, self.keys = ctx, keys
        self.steps = [int(s) for s in steps]
        self.batch = len(self.steps)
        arr = (C.c_int * self.batch)(*self.steps)
        h = C.c_void_p()
        check(ctx.lib.ckks_rotplan_create(ctx._h, keys._h, arr, self.batch, C.byref(h)))
        self._h = h
        self.keyswitches = int(ctx.lib.ckks_rotplan_keyswitches(h))
        # with ONE input ciphertext the rotations share common NAF prefixes (bit-identical outputs, fewer key switches)
        self.keyswitches_shared = int(ctx.lib.ckks_rotplan_keyswitches_shared(h))
        self.rounds = int(ctx.lib.ckks_rotplan_rounds(h))

    def __del__(self):
        try:
            if self._h:
                self.ctx.lib.ckks_rotplan_destroy(self._h)
                self._h = None
        except Exception:
            pass
