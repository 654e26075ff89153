"""ctypes binding of libbjj_cuda.so (include/bjj_cuda.h).  Fails loudly: there is no CPU fallback."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbjj_cuda.so")

_u8p = ctypes.c_void_p
_sz = ctypes.c_size_t
_ctx = ctypes.c_void_p
_int = ctypes.c_int
_base = ctypes.c_void_p     # bjj_base*: a fixed-base table (NULL selects B8)
_keyset = ctypes.c_void_p   # bjj_keyset*: keys with compact comb tables

# symbol -> (restype, argtypes); the single source the ABI test checks against include/bjj_cuda.h
SIGNATURES = {
    "bjj_device_count": (_int, []),
    "bjj_init": (_int, [_int, ctypes.POINTER(_ctx)]),
    "bjj_destroy": (None, [_ctx]),
    "bjj_sync": (_int, [_ctx]),
    "bjj_error_string": (ctypes.c_char_p, [_int]),
    "bjj_status_string": (ctypes.c_char_p, [_int]),
    "bjj_last_cuda_error": (ctypes.c_char_p, [_ctx]),
    "bjj_stream": (ctypes.c_void_p, [_ctx]),
    "bjj_device": (_int, [_ctx]),
    "bjj_kernel_launches": (ctypes.c_ulonglong, [_ctx]),
    "bjj_host_alloc": (ctypes.c_void_p, [_sz]),
    "bjj_host_free": (None, [ctypes.c_void_p]),
    "bjj_dev_alloc": (ctypes.c_void_p, [_ctx, _sz]),
    "bjj_dev_free": (None, [_ctx, ctypes.c_void_p]),
    "bjj_memcpy_h2d": (_int, [_ctx, ctypes.c_void_p, ctypes.c_void_p, _sz]),
    "bjj_memcpy_d2h": (_int, [_ctx, ctypes.c_void_p, ctypes.c_void_p, _sz]),
    "bjj_fr_op_batch": (_int, [_ctx, _int, _sz, _u8p, _u8p, _u8p]),
    "bjj_split_scalars_batch": (_int, [_ctx, _sz] + [_u8p] * 5),
    "bjj_add_batch": (_int, [_ctx, _sz] + [_u8p] * 9),
    "bjj_affine_batch": (_int, [_ctx, _sz] + [_u8p] * 5),
    "bjj_mul_scalar_batch": (_int, [_ctx, _sz] + [_u8p] * 5),
    "bjj_fixed_base_batch": (_int, [_ctx, _sz] + [_u8p] * 3),
    "bjj_public_batch": (_int, [_ctx, _sz] + [_u8p] * 3),
    "bjj_public_compressed_batch": (_int, [_ctx, _sz] + [_u8p] * 2),
    "bjj_scalar_key_batch": (_int, [_ctx, _sz] + [_u8p] * 2),
    "bjj_sign_batch": (_int, [_ctx, _sz] + [_u8p] * 6),
    "bjj_sign_compressed_batch": (_int, [_ctx, _sz] + [_u8p] * 4),
    "bjj_compress_batch": (_int, [_ctx, _sz] + [_u8p] * 3),
    "bjj_decompress_batch": (_int, [_ctx, _sz] + [_u8p] * 4),
    "bjj_poseidon_batch": (_int, [_ctx, _int, _sz, ctypes.POINTER(_u8p), _u8p]),
    "bjj_verify_batch": (_int, [_ctx, _sz] + [_u8p] * 7),
    "bjj_verify_compressed_batch": (_int, [_ctx, _sz] + [_u8p] * 5),
    "bjj_verify_schnorr_batch": (_int, [_ctx, _sz] + [_u8p] * 8),
    "bjj_base_create": (_int, [_ctx, _u8p, _u8p, ctypes.POINTER(_base)]),
    "bjj_base_destroy": (None, [_ctx, _base]),
    "bjj_base_mul_batch": (_int, [_ctx, _base, _sz] + [_u8p] * 3),
    "bjj_base_mul2_batch": (_int, [_ctx, _base, _base, _sz] + [_u8p] * 4),
    "bjj_msm_batch": (_int, [_ctx, _sz] + [_u8p] * 6),
    "bjj_verify_base_batch": (_int, [_ctx, _base, _sz] + [_u8p] * 5),
    "bjj_verify_base_compressed_batch": (_int, [_ctx, _base, _sz] + [_u8p] * 4),
    "bjj_keyset_create": (_int, [_ctx, _sz, _u8p, _u8p, _u8p, ctypes.POINTER(_keyset)]),
    "bjj_keyset_destroy": (None, [_ctx, _keyset]),
    "bjj_keyset_append": (_int, [_ctx, _keyset, _sz, _u8p, _u8p, _u8p]),
    "bjj_keyset_replace": (_int, [_ctx, _keyset, _sz, _sz, _u8p, _u8p, _u8p]),
    "bjj_verify_keyset_batch": (_int, [_ctx, _keyset, _sz] + [_u8p] * 6),
    "bjj_verify_keyset_compressed_batch": (_int, [_ctx, _keyset, _sz] + [_u8p] * 5),
    "bjj_keyset_mul_batch": (_int, [_ctx, _keyset, _sz] + [_u8p] * 4),
    "bjj_keyset_lookup_batch": (_int, [_ctx, _keyset, _sz] + [_u8p] * 2),
    "bjj_verify_keyset_lookup_compressed_batch": (_int, [_ctx, _keyset, _sz] + [_u8p] * 6),
}
# every batch op also has a device-pointer flavour with a trailing `void* stream`
for _name in [k for k in SIGNATURES if k.endswith("_batch")]:
    _res, _args = SIGNATURES[_name]
    SIGNATURES[_name + "_dev"] = (_res, list(_args) + [ctypes.c_void_p])

SIGNATURES["bjj_mul_scalar_wide_batch"] = (_int, [_ctx, _sz, _u8p, _u8p, _u8p, _int, _u8p, _u8p])
SIGNATURES["bjj_mul_scalar_wide_batch_dev"] = (_int, [_ctx, _sz, _u8p, _u8p, _u8p, _int, _u8p, _u8p, ctypes.c_void_p])
SIGNATURES["bjj_sign_schnorr_batch"] = (_int, [_ctx, _sz, _u8p, _u8p, _u8p, _int] + [_u8p] * 4)
SIGNATURES["bjj_sign_schnorr_batch_dev"] = (_int, [_ctx, _sz, _u8p, _u8p, _u8p, _int] + [_u8p] * 4 + [ctypes.c_void_p])
# verify_schnorr with s at the signer's width (s_words words per lane)
for _name, _head in (("bjj_verify_schnorr_base_batch", [_ctx, _base, _sz] + [_u8p] * 4),
                     ("bjj_verify_schnorr_keyset_batch", [_ctx, _keyset, _sz] + [_u8p] * 5),
                     ("bjj_verify_schnorr_wide_batch", [_ctx, _sz] + [_u8p] * 6)):
    SIGNATURES[_name] = (_int, _head + [_int, _u8p, _u8p])
    SIGNATURES[_name + "_dev"] = (_int, _head + [_int, _u8p, _u8p, ctypes.c_void_p])

# multi-device layer (one caller, one host batch, N devices); host pointers only
_multi = ctypes.c_void_p
SIGNATURES.update({
    "bjj_multi_init": (_int, [_int, ctypes.POINTER(_int), ctypes.POINTER(_multi)]),
    "bjj_multi_destroy": (None, [_multi]),
    "bjj_multi_devices": (_int, [_multi]),
    "bjj_multi_ctx": (_ctx, [_multi, _int]),
    "bjj_multi_set_host_register": (None, [_multi, _int]),
    "bjj_multi_kernel_launches": (ctypes.c_ulonglong, [_multi]),
    "bjj_multi_verify_batch": (_int, [_multi, _sz] + [_u8p] * 7),
    "bjj_multi_verify_compressed_batch": (_int, [_multi, _sz] + [_u8p] * 5),
    "bjj_multi_mul_scalar_batch": (_int, [_multi, _sz] + [_u8p] * 5),
    "bjj_multi_msm_batch": (_int, [_multi, _sz] + [_u8p] * 6),
    "bjj_multi_public_batch": (_int, [_multi, _sz] + [_u8p] * 3),
    "bjj_multi_public_compressed_batch": (_int, [_multi, _sz] + [_u8p] * 2),
    "bjj_multi_sign_compressed_batch": (_int, [_multi, _sz] + [_u8p] * 4),
    "bjj_multi_sign_schnorr_batch": (_int, [_multi, _sz, _u8p, _u8p, _u8p, _int] + [_u8p] * 4),
    "bjj_multi_fixed_base_batch": (_int, [_multi, _sz] + [_u8p] * 3),
    "bjj_multi_decompress_batch": (_int, [_multi, _sz] + [_u8p] * 4),
})

_lib = None


class BjjError(RuntimeError):
    def __init__(self, code, what, detail=""):
        self.code = code
        super().__init__("%s failed: code %d%s" % (what, code, (" (" + detail + ")") if detail else ""))


def load():
    """dlopen the CUDA library; raises if it has not been built (no silent fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "libbjj_cuda.so is missing at %s -- run `python -c 'import __graft_entry__ as g; g.build()'`. "
            "This package has no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)      # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
