"""ctypes declarations for include/ckks_b200.h (the C ABI of libckks_b200.so).

Loading never falls back to anything else: if the shared object is missing the import of the
engine fails with instructions to build it.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libckks_b200.so")

CKKS_OK = 0
CKKS_ERR_INVALID = 1
CKKS_ERR_CUDA = 2
CKKS_ERR_NOMEM = 3
CKKS_ERR_LOGIC = 4


class View(C.Structure):
    """struct ckks_view"""
    _fields_ = [
        ("data", C.c_void_p),
        ("batch_stride", C.c_uint64),
        ("poly_stride", C.c_uint64),
        ("batch", C.c_int32),
        ("size", C.c_int32),
        ("limbs", C.c_int32),
        ("reserved", C.c_int32),
    ]


_VP = C.POINTER(View)
_u64p = C.POINTER(C.c_uint64)
_vpp = C.POINTER(C.c_void_p)

# name -> (restype, argtypes); must list every function include/ckks_b200.h declares
SIGNATURES = {
    "ckks_last_error": (C.c_char_p, []),
    "ckks_version": (C.c_char_p, []),
    "ckks_ctx_create": (C.c_int, [C.c_int, C.c_int, _u64p, C.c_int, _vpp]),
    "ckks_ctx_destroy": (None, [C.c_void_p]),
    "ckks_ctx_log_n": (C.c_int, [C.c_void_p]),
    "ckks_ctx_n_primes": (C.c_int, [C.c_void_p]),
    "ckks_ctx_prime": (C.c_uint64, [C.c_void_p, C.c_int]),
    "ckks_ctx_set_rounding": (C.c_int, [C.c_void_p, C.c_int]),
    "ckks_ctx_set_workspace_cap": (C.c_int, [C.c_void_p, C.c_size_t]),
    "ckks_ctx_set_chain_lanes": (C.c_int, [C.c_void_p, C.c_int]),
    "ckks_ctx_reserve": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "ckks_ctx_launch_count": (C.c_uint64, [C.c_void_p]),
    "ckks_ctx_reset_launch_count": (None, [C.c_void_p]),
    "ckks_dev_alloc": (C.c_int, [C.c_void_p, C.c_size_t, _vpp]),
    "ckks_dev_free": (C.c_int, [C.c_void_p, C.c_void_p]),
    "ckks_dev_alloc_async": (C.c_int, [C.c_void_p, C.c_size_t, _vpp, C.c_void_p]),
    "ckks_dev_free_async": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "ckks_host_alloc": (C.c_int, [C.c_size_t, _vpp]),
    "ckks_host_free": (C.c_int, [C.c_void_p]),
    "ckks_upload": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "ckks_download": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "ckks_copy": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "ckks_stream_sync": (C.c_int, [C.c_void_p, C.c_void_p]),
    "ckks_ntt_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_void_p]),
    "ckks_ntt_inverse": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_void_p]),
    "ckks_add": (C.c_int, [C.c_void_p, _VP, _VP, _VP, C.c_void_p]),
    "ckks_sub": (C.c_int, [C.c_void_p, _VP, _VP, _VP, C.c_void_p]),
    "ckks_negate": (C.c_int, [C.c_void_p, _VP, _VP, C.c_void_p]),
    "ckks_multiply": (C.c_int, [C.c_void_p, _VP, _VP, _VP, C.c_void_p]),
    "ckks_multiply_plain": (C.c_int, [C.c_void_p, _VP, _VP, _VP, C.c_void_p]),
    "ckks_add_plain": (C.c_int, [C.c_void_p, _VP, _VP, _VP, C.c_void_p]),
    "ckks_add_many": (C.c_int, [C.c_void_p, _VP, _VP, C.c_void_p]),
    "ckks_add_many_grouped": (C.c_int, [C.c_void_p, _VP, C.c_int, _VP, C.c_void_p]),
    "ckks_multiply_const_sum": (C.c_int, [C.c_void_p, _VP, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          _VP, C.c_void_p]),
    "ckks_is_transparent": (C.c_int, [C.c_void_p, _VP, C.c_void_p, C.c_void_p]),
    "ckks_ksk_words": (C.c_size_t, [C.c_void_p]),
    "ckks_relinearize": (C.c_int, [C.c_void_p, _VP, C.c_void_p, _VP, C.c_void_p]),
    "ckks_apply_galois": (C.c_int, [C.c_void_p, _VP, C.c_uint64, C.c_void_p, _VP, C.c_void_p]),
    "ckks_galois_elt_from_step": (C.c_uint64, [C.c_void_p, C.c_int]),
    "ckks_keyset_create": (C.c_int, [C.c_void_p, _vpp]),
    "ckks_keyset_destroy": (None, [C.c_void_p]),
    "ckks_keyset_set_relin": (C.c_int, [C.c_void_p, C.c_void_p]),
    "ckks_keyset_set_galois": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p]),
    "ckks_keyset_has_galois": (C.c_int, [C.c_void_p, C.c_uint64]),
    "ckks_rotate": (C.c_int, [C.c_void_p, C.c_void_p, _VP, C.c_int, _VP, _VP, C.c_void_p]),
    "ckks_rotplan_create": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_int), C.c_int, _vpp]),
    "ckks_rotplan_destroy": (None, [C.c_void_p]),
    "ckks_rotplan_keyswitches": (C.c_uint64, [C.c_void_p]),
    "ckks_rotplan_keyswitches_shared": (C.c_uint64, [C.c_void_p]),
    "ckks_rotplan_rounds": (C.c_int, [C.c_void_p]),
    "ckks_rotate_plan": (C.c_int, [C.c_void_p, C.c_void_p, _VP, _VP, _VP, C.c_void_p]),
    "ckks_rotate_plan_hoisted": (C.c_int, [C.c_void_p, C.c_void_p, _VP, _VP, C.c_void_p]),
    "ckks_rmsplan_create": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.c_int,
                                      C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), _vpp]),
    "ckks_rmsplan_destroy": (None, [C.c_void_p]),
    "ckks_rmsplan_inner_products": (C.c_uint64, [C.c_void_p]),
    "ckks_rmsplan_mod_downs": (C.c_uint64, [C.c_void_p]),
    "ckks_rotate_multiply_sum_hoisted": (C.c_int, [C.c_void_p, C.c_void_p, _VP, _VP, _VP, C.c_void_p]),
    "ckks_rotate_multiply_sum_hoisted_partial": (C.c_int, [C.c_void_p, C.c_void_p, _VP, _VP, _VP, C.c_void_p]),
    "ckks_rms_mod_down": (C.c_int, [C.c_void_p, _VP, C.c_int, _VP, C.c_void_p]),
    "ckks_rotate_sum_chain": (C.c_int, [C.c_void_p, C.c_void_p, _VP, _VP, _VP, C.c_int, C.c_int, C.POINTER(C.c_int), C.c_void_p]),
    "ckks_multiply_plain_sum": (C.c_int, [C.c_void_p, _VP, _VP, _VP, C.c_void_p]),
    "ckks_multiply_sum": (C.c_int, [C.c_void_p, _VP, _VP, _VP, C.c_void_p]),
    "ckks_multiply_sum_grouped": (C.c_int, [C.c_void_p, _VP, _VP, C.c_int, _VP, C.c_void_p]),
    "ckks_multiply_sum_matrix": (C.c_int, [C.c_void_p, _VP, _VP, C.c_int, C.c_int, C.c_int, _VP, C.c_void_p]),
    "ckks_rescale": (C.c_int, [C.c_void_p, _VP, _VP, C.c_void_p]),
    "ckks_mod_switch_drop": (C.c_int, [C.c_void_p, _VP, _VP, C.c_void_p]),
    "ckks_encode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_double, _VP, C.c_void_p]),
    "ckks_encode_scalar": (C.c_int, [C.c_void_p, C.c_double, C.c_double, _VP, C.c_void_p]),
    "ckks_decode": (C.c_int, [C.c_void_p, _VP, C.c_double, C.c_void_p, C.c_void_p]),
    "ckks_sample": (C.c_int, [C.c_void_p, C.c_int, C.c_uint64, C.c_uint64, _VP, C.c_void_p]),
    "ckks_sample_keyed": (C.c_int, [C.c_void_p, C.c_int, C.c_char_p, C.c_uint64, _VP, C.c_void_p]),
}

_lib = None


def load():
    """dlopen libckks_b200.so and bind every entry point; raises if the library is absent."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("CKKS_B200_LIB", LIB_PATH)   # profiling aid: A/B an experimental build (profiles/build_variant.sh)
    if not os.path.exists(path):
        raise ImportError(
            "libckks_b200.so is not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU or PyTorch fallback for the CKKS engine)")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class CkksError(RuntimeError):
    pass


class CkksInvalidArgument(CkksError, ValueError):
    """SEAL's std::invalid_argument"""


class CkksLogicError(CkksError):
    """SEAL's std::logic_error"""


def check(rc):
    if rc == CKKS_OK:
        return
    msg = load().ckks_last_error().decode()
    if rc == CKKS_ERR_INVALID:
        raise CkksInvalidArgument(msg)
    if rc == CKKS_ERR_LOGIC:
        raise CkksLogicError(msg)
    if rc == CKKS_ERR_NOMEM:
        raise MemoryError(msg)
    raise CkksError(msg)
