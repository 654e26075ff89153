"""babyjubjub-rs_b200: B200-native batch engine for babyjubjub-rs's hot path (host-side mirror).

The reference is a Rust crate and there is no Rust toolchain in this image, so the host side above
the C ABI (include/bjj_cuda.h, libbjj_cuda.so) is mirrored twice: `host/bjj.hpp` (C++, header-only)
and this Python module, which the parity tests drive.  Names, argument meaning and error behaviour
follow the reference's public API (paths into the reference tree):

    Point{x,y}.projective/mul_scalar/compress/equals      src/lib.rs:134-186
    PointProjective{x,y,z}.affine/add                      src/lib.rs:62-132
    decompress_point, decompress_signature                 src/lib.rs:192-224, 260-268
    Signature{r_b8,s}.compress                             src/lib.rs:239-258
    PrivateKey{key}.scalar_key/public                      src/lib.rs:270-306
    verify(pk, sig, msg)                                   src/lib.rs:395-412
    + the batch entry points the north star adds: mul_scalar_batch, public_batch,
      decompress_batch, verify_batch (and add/compress/poseidon/fixed-base batches).
    + FixedBase / mul_fixed_base_batch / mul2_fixed_base_batch: k*P and k*P + l*Q on a
      precomputed table of a caller-chosen point P (the comb path B8 uses).
    + public_compressed_batch / sign_compressed_batch: PrivateKey::public().compress() and
      PrivateKey::sign(msg).compress() with the compression done on the device.
    + verify_base_batch: verify for many signatures of ONE key, with the key's FixedBase table
      (two comb walks per signature instead of verify_batch's per-lane ladder).
    + KeySet / verify_keyset_batch: verify for batches that mix many known keys, each key with a compact
      comb table (4,130 entries, 396 KB) and a key index per signature.
    + KeySet.lookup / verify_keyset_lookup_batch: the same keys found by their 32-byte compressed form on the device,
      so that a key-set verify takes verify_compressed's arrays; a key outside the set is a per-lane None.
    + sign_schnorr_batch: PrivateKey::sign_schnorr over a batch, with caller-supplied (or random 1024-bit)
      nonces and the unreduced s of the reference.
    + verify_schnorr_batch / verify_schnorr_base_batch / verify_schnorr_keyset_batch: verify_schnorr over a batch,
      taking sign_schnorr_batch's unreduced s as it is (any key; one key's FixedBase; a KeySet and a key per lane).

Every call runs on the GPU through libbjj_cuda.so; there is no CPU fallback -- importing works
without a GPU (so the ABI can be inspected), creating an Engine does not.
"""
import ctypes
import weakref

import numpy as np

from . import _lib
from ._lib import BjjError
from .sharding import MultiGpu, max_over_ranks, shard_range  # noqa: F401

Q = 21888242871839275222246405745257275088548364400416034343698204186575808495617
ORDER = 21888242871839275222246405745257275088614511777268538073601725287587578984328
SUBORDER = ORDER >> 3
B8 = (5299619240641551281634865583518297030282874472190772894086521144482721001553,
      16950150798460657717958625567821834550301663161624707787222815936182638968203)

FR_MUL, FR_ADD, FR_SUB, FR_INV, FR_SQR, FR_SQR_LAZY = 0, 1, 2, 3, 4, 5
STATUS_STRINGS = {
    0: "",
    1: "y outside the Finite Field over R",
    2: "no mod inv of Zero",
    3: "not a mod p square",
    4: "msg outside the Finite Field",
}
ERR_NONCANONICAL = 3
KEY_NONE = 0xFFFFFFFF       # key index of the lookup calls for a key outside the set


# ---- conversions ---------------------------------------------------------------------------------
def ints_to_le32(values):
    """list of non-negative ints < 2^256 -> uint8 array (n, 32), little-endian."""
    buf = b"".join(int(v).to_bytes(32, "little") for v in values)
    return np.frombuffer(buf, dtype=np.uint8).reshape(-1, 32).copy()


def le32_to_ints(arr):
    raw = np.ascontiguousarray(arr, dtype=np.uint8).tobytes()
    return [int.from_bytes(raw[i:i + 32], "little") for i in range(0, len(raw), 32)]


def _as_u8(a, width):
    a = np.ascontiguousarray(a, dtype=np.uint8)
    if a.ndim == 1:
        a = a.reshape(-1, width)
    if a.ndim != 2 or a.shape[1] != width:
        raise ValueError("expected uint8 array of shape (n, %d), got %r" % (width, a.shape))
    return a


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


class Engine:
    """One bjj_ctx on one device (one host thread, one stream; no NCCL -- nothing is exchanged)."""

    def __init__(self, device=0):
        self.lib = _lib.load()
        if self.lib.bjj_device_count() < 1:
            raise RuntimeError("babyjubjub-rs_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        ctx = ctypes.c_void_p()
        rc = self.lib.bjj_init(int(device), ctypes.byref(ctx))
        if rc != 0:
            raise BjjError(rc, "bjj_init", self.lib.bjj_error_string(rc).decode())
        self.ctx = ctx
        self.device = int(device)
        self._bases = weakref.WeakSet()     # FixedBase tables and KeySets of this context: freed before the context

    def close(self):
        if getattr(self, "ctx", None):
            for b in list(self._bases):
                b.close()
            self.lib.bjj_destroy(self.ctx)
            self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- plumbing
    def _check(self, rc, what, allow_noncanonical=False):
        if rc == 0 or (allow_noncanonical and rc == ERR_NONCANONICAL):
            return rc
        detail = self.lib.bjj_error_string(rc).decode()
        if rc == 1:
            detail += ": " + self.lib.bjj_last_cuda_error(self.ctx).decode()
        raise BjjError(rc, what, detail)

    @property
    def kernel_launches(self):
        return int(self.lib.bjj_kernel_launches(self.ctx))

    @property
    def stream(self):
        return self.lib.bjj_stream(self.ctx)

    def sync(self):
        return self._check(self.lib.bjj_sync(self.ctx), "bjj_sync")

    # -- batch ops on (n, 32) uint8 arrays (host memory)
    def fr_op_batch(self, op, a, b=None):
        a = _as_u8(a, 32)
        b = a if b is None else _as_u8(b, 32)
        out = np.empty_like(a)
        self._check(self.lib.bjj_fr_op_batch(self.ctx, op, len(a), _ptr(a), _ptr(b), _ptr(out)), "bjj_fr_op_batch")
        return out

    def split_scalars_batch(self, h, s):
        """test hook: verify's half-size scalars; returns (u, |v|, v_is_negative, w) -- see include/bjj_cuda.h"""
        h, s = _as_u8(h, 32), _as_u8(s, 32)
        u, v, w = np.empty_like(h), np.empty_like(h), np.empty_like(h)
        self._check(self.lib.bjj_split_scalars_batch(self.ctx, len(h), _ptr(h), _ptr(s), _ptr(u), _ptr(v), _ptr(w)),
                    "bjj_split_scalars_batch")
        neg = (v[:, 31] >> 7).astype(np.uint8)
        v = v.copy()
        v[:, 31] &= 0x7F
        return u, v, neg, w

    def add_batch(self, px, py, pz, qx, qy, qz):
        ins = [_as_u8(v, 32) for v in (px, py, pz, qx, qy, qz)]
        outs = [np.empty_like(ins[0]) for _ in range(3)]
        self._check(self.lib.bjj_add_batch(self.ctx, len(ins[0]), *[_ptr(v) for v in ins + outs]), "bjj_add_batch")
        return tuple(outs)

    def affine_batch(self, px, py, pz):
        ins = [_as_u8(v, 32) for v in (px, py, pz)]
        outs = [np.empty_like(ins[0]) for _ in range(2)]
        self._check(self.lib.bjj_affine_batch(self.ctx, len(ins[0]), *[_ptr(v) for v in ins + outs]), "bjj_affine_batch")
        return tuple(outs)

    def mul_scalar_batch(self, px, py, scalars):
        ins = [_as_u8(v, 32) for v in (px, py, scalars)]
        outs = [np.empty_like(ins[0]) for _ in range(2)]
        self._check(self.lib.bjj_mul_scalar_batch(self.ctx, len(ins[0]), *[_ptr(v) for v in ins + outs]),
                    "bjj_mul_scalar_batch")
        return tuple(outs)

    def mul_scalar_wide_batch(self, px, py, scalars, words):
        """scalars: uint8 array (n, 4 * words), little-endian; words a multiple of 8 in [8, 64] (src/lib.rs:149-164
        takes a BigInt of any size)"""
        px, py = _as_u8(px, 32), _as_u8(py, 32)
        k = _as_u8(scalars, 4 * int(words))
        rx, ry = np.empty_like(px), np.empty_like(px)
        self._check(self.lib.bjj_mul_scalar_wide_batch(self.ctx, len(px), _ptr(px), _ptr(py), _ptr(k), int(words), _ptr(rx), _ptr(ry)),
                    "bjj_mul_scalar_wide_batch")
        return rx, ry

    def fixed_base_batch(self, scalars):
        k = _as_u8(scalars, 32)
        outs = [np.empty_like(k) for _ in range(2)]
        self._check(self.lib.bjj_fixed_base_batch(self.ctx, len(k), _ptr(k), _ptr(outs[0]), _ptr(outs[1])),
                    "bjj_fixed_base_batch")
        return tuple(outs)

    def base_mul_batch(self, base, scalars):
        """k*P for every 256-bit scalar k (raw, unreduced); base: a FixedBase of this engine, or None for B8"""
        k = _as_u8(scalars, 32)
        rx, ry = np.empty_like(k), np.empty_like(k)
        self._check(self.lib.bjj_base_mul_batch(self.ctx, _handle(base), len(k), _ptr(k), _ptr(rx), _ptr(ry)),
                    "bjj_base_mul_batch")
        return rx, ry

    def base_mul2_batch(self, p, ks, q, ls):
        """k*P + l*Q lane by lane; p, q: FixedBase tables of this engine, or None for B8"""
        k, l = _as_u8(ks, 32), _as_u8(ls, 32)
        if len(k) != len(l):
            raise ValueError("k and l differ in length")
        rx, ry = np.empty_like(k), np.empty_like(k)
        self._check(self.lib.bjj_base_mul2_batch(self.ctx, _handle(p), _handle(q), len(k), _ptr(k), _ptr(l), _ptr(rx),
                                                 _ptr(ry)), "bjj_base_mul2_batch")
        return rx, ry

    def msm_batch(self, px, py, scalars):
        """R = sum_i k_i * P_i (include/bjj_cuda.h, bjj_msm_batch): 256-bit scalars, raw.  Returns (rx, ry, status): R's
        coordinates as (1, 32) arrays and one BJJ_KEY_* code per point.  Raises BjjError with code 2 (BJJ_ERR_ARG) when a
        point is off the curve or code 3 (BJJ_ERR_NONCANONICAL) for a coordinate >= Q, the status on the exception."""
        px, py, k = _as_u8(px, 32), _as_u8(py, 32), _as_u8(scalars, 32)
        if not len(px) == len(py) == len(k):
            raise ValueError("px, py and scalars differ in length")
        rx, ry = np.zeros((1, 32), np.uint8), np.zeros((1, 32), np.uint8)
        st = np.zeros(len(px), np.uint8)
        rc = self.lib.bjj_msm_batch(self.ctx, len(px), _ptr(px), _ptr(py), _ptr(k), _ptr(rx), _ptr(ry), _ptr(st))
        try:
            self._check(rc, "bjj_msm_batch")
        except BjjError as e:
            e.point_status = st
            raise
        return rx, ry, st

    def public_batch(self, keys):
        k = _as_u8(keys, 32)
        outs = [np.empty_like(k) for _ in range(2)]
        self._check(self.lib.bjj_public_batch(self.ctx, len(k), _ptr(k), _ptr(outs[0]), _ptr(outs[1])), "bjj_public_batch")
        return tuple(outs)

    def public_compressed_batch(self, keys):
        """compress(PrivateKey::public(key)) for every key -> (n, 32) uint8"""
        k = _as_u8(keys, 32)
        out = np.empty_like(k)
        self._check(self.lib.bjj_public_compressed_batch(self.ctx, len(k), _ptr(k), _ptr(out)), "bjj_public_compressed_batch")
        return out

    def scalar_key_batch(self, keys):
        k = _as_u8(keys, 32)
        out = np.empty_like(k)
        self._check(self.lib.bjj_scalar_key_batch(self.ctx, len(k), _ptr(k), _ptr(out)), "bjj_scalar_key_batch")
        return out

    def sign_batch(self, keys, msgs):
        k, m = _as_u8(keys, 32), _as_u8(msgs, 32)
        rx, ry, s = (np.empty_like(k) for _ in range(3))
        status = np.empty(len(k), dtype=np.uint8)
        self._check(self.lib.bjj_sign_batch(self.ctx, len(k), _ptr(k), _ptr(m), _ptr(rx), _ptr(ry), _ptr(s), _ptr(status)),
                    "bjj_sign_batch")
        return rx, ry, s, status

    def sign_compressed_batch(self, keys, msgs):
        """PrivateKey::sign(msg).compress() for every lane -> (sig (n, 64) uint8, status (n,) uint8); a lane with
        status 4 (msg > Q) has 64 zero bytes"""
        k, m = _as_u8(keys, 32), _as_u8(msgs, 32)
        sig = np.empty((len(k), 64), dtype=np.uint8)
        status = np.empty(len(k), dtype=np.uint8)
        self._check(self.lib.bjj_sign_compressed_batch(self.ctx, len(k), _ptr(k), _ptr(m), _ptr(sig), _ptr(status)),
                    "bjj_sign_compressed_batch")
        return sig, status

    def sign_schnorr_batch(self, keys, msgs, nonces, words):
        """PrivateKey::sign_schnorr with caller nonces: nonces is a uint8 array (n, 4 * words), little-endian, words a
        multiple of 8 in [8, 64] -> (rx, ry, s (n, 4 * (words + 8)) unreduced, status (n,)); a lane with status 4
        (msg > Q) has zero r and s"""
        k, m = _as_u8(keys, 32), _as_u8(msgs, 32)
        kn = _as_u8(nonces, 4 * int(words))
        if not len(k) == len(m) == len(kn):
            raise ValueError("keys, msgs and nonces differ in length")
        rx, ry = np.empty_like(k), np.empty_like(k)
        s = np.empty((len(k), 4 * (int(words) + 8)), dtype=np.uint8)
        status = np.empty(len(k), dtype=np.uint8)
        self._check(self.lib.bjj_sign_schnorr_batch(self.ctx, len(k), _ptr(k), _ptr(m), _ptr(kn), int(words), _ptr(rx), _ptr(ry),
                                                    _ptr(s), _ptr(status)), "bjj_sign_schnorr_batch")
        return rx, ry, s, status

    def compress_batch(self, px, py):
        x, y = _as_u8(px, 32), _as_u8(py, 32)
        out = np.empty_like(x)
        self._check(self.lib.bjj_compress_batch(self.ctx, len(x), _ptr(x), _ptr(y), _ptr(out)), "bjj_compress_batch")
        return out

    def decompress_batch(self, comp):
        c = _as_u8(comp, 32)
        rx, ry = np.empty_like(c), np.empty_like(c)
        status = np.empty(len(c), dtype=np.uint8)
        self._check(self.lib.bjj_decompress_batch(self.ctx, len(c), _ptr(c), _ptr(rx), _ptr(ry), _ptr(status)),
                    "bjj_decompress_batch")
        return rx, ry, status

    def poseidon_batch(self, inputs):
        ins = [_as_u8(v, 32) for v in inputs]
        if not 1 <= len(ins) <= 6:
            raise ValueError("Wrong inputs length")         # poseidon-rs 0.0.8: Err on 0 or more than 6 inputs
        arr = (ctypes.c_void_p * len(ins))(*[v.ctypes.data for v in ins])
        out = np.empty_like(ins[0])
        self._check(self.lib.bjj_poseidon_batch(self.ctx, len(ins), len(ins[0]), arr, _ptr(out)), "bjj_poseidon_batch")
        return out

    def verify_batch(self, r8x, r8y, s, ax, ay, msg):
        ins = [_as_u8(v, 32) for v in (r8x, r8y, s, ax, ay, msg)]
        ok = np.empty(len(ins[0]), dtype=np.uint8)
        self._check(self.lib.bjj_verify_batch(self.ctx, len(ins[0]), *[_ptr(v) for v in ins], _ptr(ok)), "bjj_verify_batch")
        return ok

    def verify_schnorr_batch(self, pkx, pky, msg, rx, ry, s):
        ins = [_as_u8(v, 32) for v in (pkx, pky, msg, rx, ry, s)]
        ok = np.empty(len(ins[0]), dtype=np.uint8)
        status = np.empty(len(ins[0]), dtype=np.uint8)
        self._check(self.lib.bjj_verify_schnorr_batch(self.ctx, len(ins[0]), *[_ptr(v) for v in ins], _ptr(ok), _ptr(status)),
                    "bjj_verify_schnorr_batch")
        return ok, status

    def verify_compressed_batch(self, sig64, pk32, msg):
        sg, pk, m = _as_u8(sig64, 64), _as_u8(pk32, 32), _as_u8(msg, 32)
        ok = np.empty(len(sg), dtype=np.uint8)
        status = np.empty(len(sg), dtype=np.uint8)
        self._check(self.lib.bjj_verify_compressed_batch(self.ctx, len(sg), _ptr(sg), _ptr(pk), _ptr(m), _ptr(ok), _ptr(status)),
                    "bjj_verify_compressed_batch")
        return ok, status

    def verify_base_batch(self, base, r8x, r8y, s, msg):
        """verify for every lane against the one key of `base` (a FixedBase of this engine) -> ok (n,) uint8"""
        ins = [_as_u8(v, 32) for v in (r8x, r8y, s, msg)]
        ok = np.empty(len(ins[0]), dtype=np.uint8)
        self._check(self.lib.bjj_verify_base_batch(self.ctx, _key_handle(base), len(ins[0]), *[_ptr(v) for v in ins], _ptr(ok)),
                    "bjj_verify_base_batch")
        return ok

    def verify_base_compressed_batch(self, base, sig64, msg):
        """verify of 64-byte compressed signatures against the one key of `base` -> (ok, status), both (n,) uint8;
        status is R8's decompression error"""
        sg, m = _as_u8(sig64, 64), _as_u8(msg, 32)
        ok = np.empty(len(sg), dtype=np.uint8)
        status = np.empty(len(sg), dtype=np.uint8)
        self._check(self.lib.bjj_verify_base_compressed_batch(self.ctx, _key_handle(base), len(sg), _ptr(sg), _ptr(m), _ptr(ok),
                                                              _ptr(status)), "bjj_verify_base_compressed_batch")
        return ok, status

    def verify_keyset_batch(self, keyset, key_index, r8x, r8y, s, msg):
        """verify for every lane against key key_index[i] of `keyset` (a KeySet of this engine) -> ok (n,) uint8"""
        ins = [_as_u8(v, 32) for v in (r8x, r8y, s, msg)]
        ki = _key_index(key_index, len(ins[0]))
        ok = np.empty(len(ins[0]), dtype=np.uint8)
        self._check(self.lib.bjj_verify_keyset_batch(self.ctx, _keyset_handle(keyset), len(ki), _ptr(ki), *[_ptr(v) for v in ins],
                                                     _ptr(ok)), "bjj_verify_keyset_batch")
        return ok

    def verify_keyset_compressed_batch(self, keyset, key_index, sig64, msg):
        """verify of 64-byte compressed signatures against key key_index[i] of `keyset` -> (ok, status), both (n,) uint8;
        status is R8's decompression error"""
        sg, m = _as_u8(sig64, 64), _as_u8(msg, 32)
        ki = _key_index(key_index, len(sg))
        ok = np.empty(len(sg), dtype=np.uint8)
        status = np.empty(len(sg), dtype=np.uint8)
        self._check(self.lib.bjj_verify_keyset_compressed_batch(self.ctx, _keyset_handle(keyset), len(ki), _ptr(ki), _ptr(sg), _ptr(m),
                                                                _ptr(ok), _ptr(status)), "bjj_verify_keyset_compressed_batch")
        return ok, status

    def keyset_mul_batch(self, keyset, key_index, scalars):
        """P_{key_index[i]} * k_i for every 256-bit scalar k_i (raw, unreduced) -> (rx, ry), (n, 32) uint8 each"""
        k = _as_u8(scalars, 32)
        ki = _key_index(key_index, len(k))
        rx, ry = np.empty_like(k), np.empty_like(k)
        self._check(self.lib.bjj_keyset_mul_batch(self.ctx, _keyset_handle(keyset), len(ki), _ptr(ki), _ptr(k), _ptr(rx), _ptr(ry)),
                    "bjj_keyset_mul_batch")
        return rx, ry

    def keyset_lookup_batch(self, keyset, pk32):
        """the index of the key of `keyset` whose compressed bytes are pk32[i], or KEY_NONE -> (n,) uint32"""
        pk = _as_u8(pk32, 32)
        ki = np.empty(len(pk), dtype="<u4")
        self._check(self.lib.bjj_keyset_lookup_batch(self.ctx, _keyset_handle(keyset), len(pk), _ptr(pk), _ptr(ki)),
                    "bjj_keyset_lookup_batch")
        return ki

    def verify_keyset_lookup_compressed_batch(self, keyset, sig64, pk32, msg):
        """verify_compressed_batch's arrays, for keys of `keyset` found by their compressed bytes -> (ok, status,
        key_index): (n,) uint8, uint8 and uint32.  A key outside the set gives ok 0, R8's status and KEY_NONE."""
        sg, pk, m = _as_u8(sig64, 64), _as_u8(pk32, 32), _as_u8(msg, 32)
        if len(pk) != len(sg) or len(m) != len(sg):
            raise ValueError("sig64, pk32 and msg differ in length")
        ok = np.empty(len(sg), dtype=np.uint8)
        status = np.empty(len(sg), dtype=np.uint8)
        ki = np.empty(len(sg), dtype="<u4")
        self._check(self.lib.bjj_verify_keyset_lookup_compressed_batch(self.ctx, _keyset_handle(keyset), len(sg), _ptr(sg), _ptr(pk),
                                                                       _ptr(m), _ptr(ok), _ptr(status), _ptr(ki)),
                    "bjj_verify_keyset_lookup_compressed_batch")
        return ok, status, ki

    # verify_schnorr with s as sign_schnorr_batch writes it: a uint8 array (n, 4 * words), little-endian and unreduced,
    # words a multiple of 8 in [8, 72]; each returns (ok, status), both (n,) uint8, status 4 where msg > Q
    def _schnorr_call(self, name, head, msg, rx, ry, s, words):
        ins = [_as_u8(v, 32) for v in (msg, rx, ry)] + [_as_u8(s, 4 * int(words))]
        n = len(ins[0])
        if any(len(v) != n for v in ins):
            raise ValueError("msg, r and s differ in length")
        ok = np.empty(n, dtype=np.uint8)
        status = np.empty(n, dtype=np.uint8)
        self._check(getattr(self.lib, name)(self.ctx, *head(n), *[_ptr(v) for v in ins], int(words), _ptr(ok), _ptr(status)), name)
        return ok, status

    def verify_schnorr_base_batch(self, base, msg, rx, ry, s, words):
        """verify_schnorr for every lane against the one key of `base` (a FixedBase of this engine)"""
        return self._schnorr_call("bjj_verify_schnorr_base_batch", lambda n: (_key_handle(base), n), msg, rx, ry, s, words)

    def verify_schnorr_keyset_batch(self, keyset, key_index, msg, rx, ry, s, words):
        """verify_schnorr for every lane against key key_index[i] of `keyset` (a KeySet of this engine)"""
        ki = _key_index(key_index, len(_as_u8(msg, 32)))
        return self._schnorr_call("bjj_verify_schnorr_keyset_batch", lambda n: (_keyset_handle(keyset), n, _ptr(ki)), msg, rx, ry, s,
                                  words)

    def verify_schnorr_wide_batch(self, pkx, pky, msg, rx, ry, s, words):
        """verify_schnorr for every lane against its own key (pkx, pky)"""
        pk = [_as_u8(v, 32) for v in (pkx, pky)]
        if len(pk[0]) != len(pk[1]) or len(pk[0]) != len(_as_u8(msg, 32)):
            raise ValueError("pk, msg, r and s differ in length")
        return self._schnorr_call("bjj_verify_schnorr_wide_batch", lambda n: (n, _ptr(pk[0]), _ptr(pk[1])), msg, rx, ry, s, words)



_default_engine = None


def default_engine():
    global _default_engine
    if _default_engine is None:
        _default_engine = Engine(0)
    return _default_engine


class FixedBase:
    """The comb table of one on-curve point P on one Engine (50 MB of device memory): P.mul_scalar(k) for many k at the
    rate of B8's fixed-base path.  Raises BjjError with code 2 (BJJ_ERR_ARG) for an off-curve P -- whose reference
    result depends on mul_scalar's exact double-and-add order, so it stays on mul_scalar_batch -- and with code 3
    (BJJ_ERR_NONCANONICAL) for a coordinate >= Q.  Free it with close() (or let it be collected)."""

    def __init__(self, point, engine=None):
        self.engine = engine or default_engine()
        x, y = (point.x, point.y) if isinstance(point, Point) else point
        self.point = Point(x, y)
        px, py = ints_to_le32([x]), ints_to_le32([y])
        handle = ctypes.c_void_p()
        rc = self.engine.lib.bjj_base_create(self.engine.ctx, _ptr(px), _ptr(py), ctypes.byref(handle))
        if rc != 0:
            self.engine._check(rc, "bjj_base_create")
        self.handle = handle
        self.engine._bases.add(self)

    def close(self):
        if getattr(self, "handle", None):
            self.engine.lib.bjj_base_destroy(self.engine.ctx, self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def mul_batch(self, scalars):
        """[P.mul_scalar(k) for k in scalars] (src/lib.rs:149-164) for Python ints of any size and sign"""
        rx, ry = self.engine.base_mul_batch(self, ints_to_le32([_base_scalar(k) for k in scalars]))
        return [Point(x, y) for x, y in zip(le32_to_ints(rx), le32_to_ints(ry))]


class KeySet:
    """N on-curve public keys on one Engine, each with a compact comb table (396,480 B of device memory per key):
    verify and k*P for batches that name a key per lane.  Raises BjjError with code 3 (BJJ_ERR_NONCANONICAL) when a
    coordinate is >= Q and with code 2 (BJJ_ERR_ARG) when a key is off the curve (or the list is empty); `status` then
    holds one code per key (0 ok, 1 off the curve, 2 non-canonical).  Free it with close() (or let it be collected)."""

    def __init__(self, points, engine=None):
        self.engine = engine or default_engine()
        pts = [(p.x, p.y) if isinstance(p, Point) else tuple(p) for p in points]
        self.points = [Point(x, y) for x, y in pts]
        self.handle = None
        ax, ay = ints_to_le32([p[0] for p in pts]), ints_to_le32([p[1] for p in pts])
        self.status = np.zeros(len(pts), dtype=np.uint8)
        handle = ctypes.c_void_p()
        rc = self.engine.lib.bjj_keyset_create(self.engine.ctx, len(pts), _ptr(ax), _ptr(ay), _ptr(self.status), ctypes.byref(handle))
        if rc != 0:
            self.engine._check(rc, "bjj_keyset_create")
        self.handle = handle
        self.engine._bases.add(self)

    def __len__(self):
        return len(self.points)

    def _edit(self, fn, name, head, points):
        pts = [(p.x, p.y) if isinstance(p, Point) else tuple(p) for p in points]
        ax, ay = ints_to_le32([p[0] for p in pts]), ints_to_le32([p[1] for p in pts])
        status = np.zeros(len(pts), dtype=np.uint8)
        rc = fn(self.engine.ctx, _keyset_handle(self), *head, len(pts), _ptr(ax), _ptr(ay), _ptr(status))
        if rc != 0:
            try:
                self.engine._check(rc, name)
            except BjjError as e:
                e.key_status = status
                raise
        return [Point(x, y) for x, y in pts], status

    def append(self, points):
        """adds keys under the indices len(self) ..; existing indices keep their keys, and `points` and `status` grow
        with the new keys.  Raises BjjError with create's codes and `key_status` (one code per new key) on the
        exception; the set, `points` and `status` then stay as they were."""
        new, st = self._edit(self.engine.lib.bjj_keyset_append, "bjj_keyset_append", (), points)
        self.points += new
        self.status = np.concatenate([self.status, st])

    def replace(self, first, points):
        """gives keys first .. first + len(points) - 1 new coordinates (key rotation), in `points` and `status` too.
        Raises BjjError with create's codes and `key_status` on the exception, or code 2 (BJJ_ERR_ARG) when the range
        runs past the set; the set, `points` and `status` then stay as they were."""
        first = int(first)
        if first < 0:
            raise ValueError("first must be >= 0")
        new, st = self._edit(self.engine.lib.bjj_keyset_replace, "bjj_keyset_replace", (first,), points)
        self.points[first:first + len(new)] = new
        self.status[first:first + len(new)] = st

    def close(self):
        if getattr(self, "handle", None):
            self.engine.lib.bjj_keyset_destroy(self.engine.ctx, self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def mul_batch(self, key_index, scalars):
        """[points[j].mul_scalar(k) for j, k in zip(key_index, scalars)] (src/lib.rs:149-164), Python ints of any size
        and sign"""
        rx, ry = self.engine.keyset_mul_batch(self, key_index, ints_to_le32([_base_scalar(k) for k in scalars]))
        return [Point(x, y) for x, y in zip(le32_to_ints(rx), le32_to_ints(ry))]

    def lookup(self, pks):
        """the index of each key (a Point or its 32 compressed bytes) in the set, the smallest if the set holds it twice,
        or None.  Keys with x = 0 are never found: decompress_point rejects their compressed forms."""
        ki = self.engine.keyset_lookup_batch(self, _pk32s(pks))
        return [None if k == KEY_NONE else int(k) for k in ki]


def _pk32s(pks):
    """Points or 32-byte compressed keys -> uint8 array (n, 32); a Point is compressed on the host (Point::compress)"""
    out = []
    for p in pks:
        if isinstance(p, Point):
            b = bytearray(p.y.to_bytes(32, "little"))
            if p.x > Q >> 1:
                b[31] |= 0x80
            out.append(bytes(b))
        else:
            b = bytes(p)
            if len(b) != 32:
                raise ValueError("a compressed key is 32 bytes, got %d" % len(b))
            out.append(b)
    return np.frombuffer(b"".join(out), dtype=np.uint8).reshape(-1, 32).copy()


def _keyset_handle(keyset):
    if keyset is None:
        raise ValueError("a keyset call needs a KeySet")
    if not keyset.handle:
        raise ValueError("KeySet is closed")
    return keyset.handle


def _key_index(key_index, n):
    """key indices as the ABI's little-endian uint32 per lane; an index outside [0, 2^32) cannot name a key"""
    ki = np.asarray(key_index)
    if ki.ndim != 1 or len(ki) != n:
        raise ValueError("expected %d key indices, got shape %r" % (n, ki.shape))
    if ki.dtype != np.uint32:
        if len(ki) and (ki.min() < 0 or ki.max() > 0xFFFFFFFF):
            raise ValueError("key index outside [0, 2^32)")
        ki = ki.astype(np.uint32)
    return np.ascontiguousarray(ki, dtype="<u4")


def _handle(base):
    if base is None:
        return None
    if not base.handle:
        raise ValueError("FixedBase is closed")
    return base.handle


def _key_handle(base):
    """the handle of a verify_base call, which must name its key (None does not select B8 there)"""
    if base is None:
        raise ValueError("verify_base_batch needs a FixedBase of the public key")
    return _handle(base)


def _base_scalar(k):
    """k as it crosses the 256-bit ABI of the fixed-base tables.  The reference multiplies by |k| (the sign is dropped,
    src/lib.rs:156); every on-curve point has an order dividing ORDER, so a wider |k| is reduced mod ORDER -- the same
    point.  Values below 2^256 go through unreduced."""
    k = abs(int(k))
    return k if k < (1 << 256) else k % ORDER


# ---- the reference's public API, as batches of one -------------------------------------------------
class PointProjective:
    """src/lib.rs:62-132"""

    def __init__(self, x, y, z):
        self.x, self.y, self.z = int(x), int(y), int(z)

    def affine(self):
        rx, ry = default_engine().affine_batch(*[ints_to_le32([v]) for v in (self.x, self.y, self.z)])
        return Point(le32_to_ints(rx)[0], le32_to_ints(ry)[0])

    def add(self, q):
        outs = default_engine().add_batch(*[ints_to_le32([v]) for v in (self.x, self.y, self.z, q.x, q.y, q.z)])
        return PointProjective(*[le32_to_ints(o)[0] for o in outs])


class Point:
    """src/lib.rs:134-186"""

    def __init__(self, x, y):
        self.x, self.y = int(x), int(y)

    def projective(self):
        return PointProjective(self.x, self.y, 1)

    def mul_scalar(self, n):
        return mul_scalar_batch([self], [n])[0]

    def compress(self):
        return default_engine().compress_batch(ints_to_le32([self.x]), ints_to_le32([self.y])).tobytes()

    def equals(self, p):
        return self.x == p.x and self.y == p.y

    def __eq__(self, other):
        return isinstance(other, Point) and self.equals(other)

    def __repr__(self):
        return "Point(x=Fr(0x%064x), y=Fr(0x%064x))" % (self.x, self.y)


def decompress_point(bb):
    """src/lib.rs:192-224; raises ValueError(<the reference's Err string>)."""
    if len(bb) != 32:
        raise ValueError("expected 32 bytes")
    rx, ry, st = default_engine().decompress_batch(np.frombuffer(bytes(bb), dtype=np.uint8).reshape(1, 32))
    if st[0]:
        raise ValueError(STATUS_STRINGS[int(st[0])])
    return Point(le32_to_ints(rx)[0], le32_to_ints(ry)[0])


class Signature:
    """src/lib.rs:239-258"""

    def __init__(self, r_b8, s):
        self.r_b8, self.s = r_b8, int(s)

    def compress(self):
        return self.r_b8.compress() + (self.s & ((1 << 256) - 1)).to_bytes(32, "little")


def decompress_signature(b):
    """src/lib.rs:260-268"""
    if len(b) != 64:
        raise ValueError("expected 64 bytes")
    return Signature(decompress_point(b[:32]), int.from_bytes(b[32:], "little"))


class PrivateKey:
    """src/lib.rs:270-342 (import, scalar_key, public, sign)."""

    def __init__(self, key):
        self.key = bytes(key)

    @staticmethod
    def import_(b):
        if len(b) != 32:
            raise ValueError("imported key can not be bigger than 32 bytes")       # src/lib.rs:277
        return PrivateKey(b)

    def scalar_key(self):
        out = default_engine().scalar_key_batch(np.frombuffer(self.key, dtype=np.uint8).reshape(1, 32))
        return le32_to_ints(out)[0]

    def public(self):
        rx, ry = default_engine().public_batch(np.frombuffer(self.key, dtype=np.uint8).reshape(1, 32))
        return Point(le32_to_ints(rx)[0], le32_to_ints(ry)[0])


def _sign(self, msg):
    """PrivateKey::sign, src/lib.rs:308-342; raises ValueError("msg outside the Finite Field")."""
    msg = int(msg)
    if msg > Q:
        raise ValueError(STATUS_STRINGS[4])
    rx, ry, s, st = default_engine().sign_batch(np.frombuffer(self.key, dtype=np.uint8).reshape(1, 32), ints_to_le32([msg]))
    if st[0]:
        raise ValueError(STATUS_STRINGS[int(st[0])])
    return Signature(Point(le32_to_ints(rx)[0], le32_to_ints(ry)[0]), le32_to_ints(s)[0])


PrivateKey.sign = _sign


def _sign_schnorr(self, m, k=None):
    """PrivateKey::sign_schnorr, src/lib.rs:345-362: k = 1024 random bits, r = B8*k, h = schnorr_hash(pk, m, r),
    s = k + scalar_key*h (NOT reduced, like the reference).  Host glue around one fixed-base multiplication and
    one Poseidon hash; B8 has order SUBORDER, so k crosses the 256-bit ABI reduced.  `k` may be supplied for
    reproducible tests."""
    import secrets
    k = secrets.randbits(1024) if k is None else int(k)
    rx, ry = default_engine().fixed_base_batch(ints_to_le32([k % SUBORDER]))
    r = Point(le32_to_ints(rx)[0], le32_to_ints(ry)[0])
    h = schnorr_hash(self.public(), m, r)
    return r, k + self.scalar_key() * h


PrivateKey.sign_schnorr = _sign_schnorr


def new_key():
    """src/lib.rs:387-393: a private key from 32 random bytes (the reference draws a 1024-bit integer and keeps its
    first 32 big-endian bytes)"""
    import secrets
    return PrivateKey(secrets.token_bytes(32))


def verify(pk, sig, msg):
    """src/lib.rs:395-412"""
    msg = int(msg)
    if msg > Q:
        return False
    if msg < 0:
        raise ValueError("negative msg (the reference panics in Fr::from_str)")
    eng = default_engine()
    ok = eng.verify_batch(*[ints_to_le32([v]) for v in (sig.r_b8.x, sig.r_b8.y, _verify_scalar(sig.s), pk.x, pk.y, msg)])
    return bool(ok[0])


def _verify_scalar(s):
    """S as it crosses the 256-bit ABI.  The reference evaluates B8.mul_scalar(S) on the BigInt as given (sign dropped,
    src/lib.rs:156, :405); B8 has order SUBORDER, so a wider S is reduced mod SUBORDER -- the same group element.
    Scalars below 2^256 go through unreduced (the device handles them, S + SUBORDER included)."""
    s = abs(int(s))
    return s if s < (1 << 256) else s % SUBORDER


def schnorr_hash(pk, msg, c):
    """src/lib.rs:364-373; raises ValueError("msg outside the Finite Field")."""
    msg = int(msg)
    if msg > Q:
        raise ValueError(STATUS_STRINGS[4])
    out = default_engine().poseidon_batch([ints_to_le32([v]) for v in (pk.x, pk.y, c.x, c.y, msg % Q)])
    return le32_to_ints(out)[0]


def verify_schnorr(pk, m, r, s):
    """src/lib.rs:375-385.  `s` may be the reference's unreduced k + x*h: B8 has order SUBORDER, so it is
    reduced on the host before crossing the 256-bit ABI."""
    m = int(m)
    ok, st = default_engine().verify_schnorr_batch(*[ints_to_le32([v]) for v in
                                                    (pk.x, pk.y, m if m <= Q else (1 << 256) - 1, r.x, r.y, abs(int(s)) % SUBORDER)])
    if st[0]:
        raise ValueError(STATUS_STRINGS[int(st[0])])
    return bool(ok[0])


# ---- batch entry points named by the north star ------------------------------------------------------
def mul_scalar_batch(points, scalars, engine=None):
    """Point::mul_scalar over a batch (src/lib.rs:149-164): scalars are BigInts of any size, the sign is dropped (:156).
    Up to 256 bits they cross the ABI as they are; wider ones use the wide entry point (on-curve points: reduced mod
    ORDER on the device; off-curve points: every bit replayed), up to 2048 bits."""
    eng = engine or default_engine()
    ks = [abs(int(k)) for k in scalars]
    px, py = ints_to_le32([p.x for p in points]), ints_to_le32([p.y for p in points])
    bits = max([k.bit_length() for k in ks] + [1])
    if bits <= 256:
        rx, ry = eng.mul_scalar_batch(px, py, ints_to_le32(ks))
    else:
        words = 8 * ((bits + 255) // 256)
        if words > 64:
            raise ValueError("scalars wider than 2048 bits are not supported by the device ABI")
        buf = np.frombuffer(b"".join(k.to_bytes(4 * words, "little") for k in ks), dtype=np.uint8).reshape(-1, 4 * words)
        rx, ry = eng.mul_scalar_wide_batch(px, py, buf, words)
    return [Point(x, y) for x, y in zip(le32_to_ints(rx), le32_to_ints(ry))]


def mul_fixed_base_batch(point, scalars, engine=None):
    """[point.mul_scalar(k) for k in scalars] on a table of the on-curve `point` (built for this call, then freed).
    Keep a FixedBase to reuse the table across calls."""
    base = FixedBase(point, engine)
    try:
        return base.mul_batch(scalars)
    finally:
        base.close()


def mul2_fixed_base_batch(p, ks, q, ls, engine=None):
    """[(k*p).projective().add((l*q).projective()).affine() for k, l in zip(ks, ls)] (src/lib.rs:70-131, 149-164) for
    on-curve p, q.  Each of p, q is a Point (its table is built for this call), a FixedBase, or None for B8."""
    eng = engine or default_engine()
    built = []
    try:
        def table(b):
            if b is None or isinstance(b, FixedBase):
                return b
            built.append(FixedBase(b, eng))
            return built[-1]
        tp, tq = table(p), table(q)
        rx, ry = eng.base_mul2_batch(tp, ints_to_le32([_base_scalar(k) for k in ks]), tq,
                                     ints_to_le32([_base_scalar(l) for l in ls]))
    finally:
        for b in built:
            b.close()
    return [Point(x, y) for x, y in zip(le32_to_ints(rx), le32_to_ints(ry))]


def msm(points, scalars, engine=None):
    """sum_i points[i].mul_scalar(scalars[i]) as the reference's fold computes it, acc.add(P_i.mul_scalar(k_i).projective())
    from (0 : 1 : 1), then affine() (src/lib.rs:70-131, 149-164), for on-curve points and BigInts of any size and sign:
    the sign is dropped and wider values are reduced mod ORDER, as _base_scalar maps them.  Raises BjjError with code 2
    (BJJ_ERR_ARG) when a point is off the curve, `point_status` on the exception naming it."""
    eng = engine or default_engine()
    if len(points) != len(scalars):
        raise ValueError("points and scalars differ in length")
    rx, ry, _ = eng.msm_batch(ints_to_le32([p.x for p in points]), ints_to_le32([p.y for p in points]),
                              ints_to_le32([_base_scalar(k) for k in scalars]))
    return Point(le32_to_ints(rx)[0], le32_to_ints(ry)[0])


def public_batch(keys, engine=None):
    eng = engine or default_engine()
    rx, ry = eng.public_batch(np.frombuffer(b"".join(bytes(k.key if isinstance(k, PrivateKey) else k) for k in keys),
                                            dtype=np.uint8).reshape(-1, 32))
    return [Point(x, y) for x, y in zip(le32_to_ints(rx), le32_to_ints(ry))]


def _keys_u8(keys):
    return np.frombuffer(b"".join(bytes(k.key if isinstance(k, PrivateKey) else k) for k in keys),
                         dtype=np.uint8).reshape(-1, 32)


def public_compressed_batch(keys, engine=None):
    """[k.public().compress() for k in keys] (src/lib.rs:304-306, 166-178) as 32-byte strings"""
    out = (engine or default_engine()).public_compressed_batch(_keys_u8(keys))
    return [bytes(r) for r in out]


def _sign_msgs(msgs):
    """messages of sign_compressed_batch as 32-byte words: a negative msg raises like verify; msg > Q, whose lane
    fails with the reference's Err, is clamped to an all-ones word (still > Q) so that it fits, as in verify_batch"""
    mm = [int(m) for m in msgs]
    if any(m < 0 for m in mm):
        raise ValueError("negative msg (the reference panics in Fr::from_str)")
    return ints_to_le32([m if m <= Q else (1 << 256) - 1 for m in mm])


def sign_compressed_batch(keys, msgs, engine=None):
    """[k.sign(m).compress() for k, m in zip(keys, msgs)] (src/lib.rs:308-342, 245-257) -> list of 64-byte strings, or
    ValueError("msg outside the Finite Field") instances for msg > Q (the reference returns Result)"""
    m = _sign_msgs(msgs)
    sig, st = (engine or default_engine()).sign_compressed_batch(_keys_u8(keys), m)
    return [bytes(r) if s == 0 else ValueError(STATUS_STRINGS[int(s)]) for r, s in zip(sig, st)]


def _schnorr_nonces(nonces):
    """nonces of sign_schnorr_batch as one uint8 array (n, 4 * words) and its word count: the smallest multiple of 8 words
    (256 bits) that holds the widest nonce, up to 64 words (2048 bits)"""
    ks = [int(k) for k in nonces]
    if any(k < 0 for k in ks):
        raise ValueError("negative nonce")
    bits = max([k.bit_length() for k in ks] + [1])
    if bits > 2048:
        raise ValueError("nonces wider than 2048 bits are not supported by the device ABI")
    words = 8 * ((bits + 255) // 256)
    buf = b"".join(k.to_bytes(4 * words, "little") for k in ks)
    return np.frombuffer(buf, dtype=np.uint8).reshape(-1, 4 * words).copy(), words


def sign_schnorr_batch(keys, msgs, nonces=None, engine=None):
    """[k.sign_schnorr(m) for k, m in zip(keys, msgs)] (src/lib.rs:344-362) -> list of (r: Point, s: int), s = k + x*h
    unreduced.  nonces: one non-negative int per lane (at most 2048 bits); None draws 1024 random bits per lane, as the
    reference does.  Raises ValueError("msg outside the Finite Field") if any msg > Q, and ValueError for a negative msg
    or nonce."""
    mm = [int(m) for m in msgs]
    if any(m > Q for m in mm):
        raise ValueError(STATUS_STRINGS[4])
    m = _sign_msgs(mm)
    if nonces is None:
        import secrets
        nonces = [secrets.randbits(1024) for _ in mm]
    kn, words = _schnorr_nonces(nonces)
    rx, ry, s, st = (engine or default_engine()).sign_schnorr_batch(_keys_u8(keys), m, kn, words)
    sw = 4 * (words + 8)
    raw = s.tobytes()
    return [(Point(x, y), int.from_bytes(raw[sw * i:sw * (i + 1)], "little"))
            for i, (x, y) in enumerate(zip(le32_to_ints(rx), le32_to_ints(ry)))]


def decompress_batch(blobs, engine=None):
    """-> list of Point or ValueError instances (the reference returns Result<Point, String>)."""
    eng = engine or default_engine()
    rx, ry, st = eng.decompress_batch(np.frombuffer(b"".join(bytes(b) for b in blobs), dtype=np.uint8).reshape(-1, 32))
    xs, ys = le32_to_ints(rx), le32_to_ints(ry)
    return [Point(x, y) if s == 0 else ValueError(STATUS_STRINGS[int(s)]) for x, y, s in zip(xs, ys, st)]


def verify_batch(pks, sigs, msgs, engine=None):
    eng = engine or default_engine()
    ok = eng.verify_batch(ints_to_le32([s.r_b8.x for s in sigs]), ints_to_le32([s.r_b8.y for s in sigs]),
                          ints_to_le32([_verify_scalar(s.s) for s in sigs]), ints_to_le32([p.x for p in pks]),
                          ints_to_le32([p.y for p in pks]), _verify_msgs(msgs))
    return [bool(v) for v in ok]


def _verify_msgs(msgs):
    """messages of verify_batch / verify_base_batch as 32-byte words: msg > Q is `false` in the reference, so such
    messages are clamped to an all-ones word (still > Q) to fit"""
    return ints_to_le32([int(m) if int(m) <= Q else (1 << 256) - 1 for m in msgs])


def verify_base_batch(base, sigs, msgs, engine=None):
    """[verify(base.point, sig, msg) for sig, msg in zip(sigs, msgs)] (src/lib.rs:395-412) for signatures of ONE key,
    whose FixedBase table `base` serves every lane; the same results as verify_batch with the key in every lane"""
    eng = engine or base.engine
    ok = eng.verify_base_batch(base, ints_to_le32([s.r_b8.x for s in sigs]), ints_to_le32([s.r_b8.y for s in sigs]),
                               ints_to_le32([_verify_scalar(s.s) for s in sigs]), _verify_msgs(msgs))
    return [bool(v) for v in ok]


def verify_keyset_batch(keyset, key_index, sigs, msgs, engine=None):
    """[verify(keyset.points[j], sig, msg) for j, sig, msg in zip(key_index, sigs, msgs)] (src/lib.rs:395-412) for
    signatures of many known keys; the same results as verify_batch with those keys.  An index outside the set raises
    BjjError (BJJ_ERR_ARG)."""
    eng = engine or keyset.engine
    ok = eng.verify_keyset_batch(keyset, np.asarray(key_index, dtype=np.int64).reshape(-1), ints_to_le32([s.r_b8.x for s in sigs]),
                                 ints_to_le32([s.r_b8.y for s in sigs]), ints_to_le32([_verify_scalar(s.s) for s in sigs]),
                                 _verify_msgs(msgs))
    return [bool(v) for v in ok]


def verify_keyset_lookup_batch(keyset, pk32s, sig64s, msgs, engine=None):
    """decompress_signature + decompress_point + verify (src/lib.rs:260-268, 192-224, 395-412) for 32-byte compressed
    keys of `keyset`, found by their bytes on the device -> per lane True / False, ValueError(<the reference's Err
    string>) when R8 does not decompress, else None when the key is not in the set"""
    if not (len(pk32s) == len(sig64s) == len(msgs)):
        raise ValueError("pk32s, sig64s and msgs differ in length")
    if any(len(bytes(s)) != 64 for s in sig64s):
        raise ValueError("a compressed signature is 64 bytes")
    eng = engine or keyset.engine
    sg = np.frombuffer(b"".join(bytes(s) for s in sig64s), dtype=np.uint8).reshape(-1, 64)
    ok, st, ki = eng.verify_keyset_lookup_compressed_batch(keyset, sg, _pk32s(pk32s), _verify_msgs(msgs))
    return [ValueError(STATUS_STRINGS[int(s)]) if s else None if k == KEY_NONE else bool(o) for o, s, k in zip(ok, st, ki)]


def _schnorr_sigs(msgs, sigs):
    """messages and (r, s) pairs of the verify_schnorr batches -> (msg, rx, ry, s, words): s (sign dropped, as
    B8.mul_scalar does) in the smallest multiple of 8 words (256 bits) that holds the widest, up to 72 words (2304 bits,
    sign_schnorr_batch's widest s).  A negative msg raises; msg > Q is clamped to an all-ones word (still > Q)."""
    if len(msgs) != len(sigs):
        raise ValueError("msgs and sigs differ in length")
    ss = [abs(int(s)) for _, s in sigs]
    bits = max([s.bit_length() for s in ss] + [1])
    if bits > 72 * 32:
        raise ValueError("s wider than 2304 bits is not supported by the device ABI")
    words = 8 * ((bits + 255) // 256)
    rs = [(r.x, r.y) if isinstance(r, Point) else tuple(r) for r, _ in sigs]
    sb = np.frombuffer(b"".join(s.to_bytes(4 * words, "little") for s in ss), dtype=np.uint8).reshape(-1, 4 * words)
    return _sign_msgs(msgs), ints_to_le32([r[0] for r in rs]), ints_to_le32([r[1] for r in rs]), sb, words


def _schnorr_results(ok, st):
    return [bool(o) if s == 0 else ValueError(STATUS_STRINGS[int(s)]) for o, s in zip(ok, st)]


def verify_schnorr_batch(pks, msgs, sigs, engine=None):
    """[verify_schnorr(pk, m, r, s) for pk, m, (r, s) in zip(pks, msgs, sigs)] (src/lib.rs:364-385), sigs as
    sign_schnorr_batch returns them, s unreduced and reduced mod SUBORDER on the device -> list of bool, or
    ValueError("msg outside the Finite Field") instances for msg > Q (the reference returns Result)"""
    eng = engine or default_engine()
    ok, st = eng.verify_schnorr_wide_batch(ints_to_le32([p.x for p in pks]), ints_to_le32([p.y for p in pks]), *_schnorr_sigs(msgs, sigs))
    return _schnorr_results(ok, st)


def verify_schnorr_base_batch(base, msgs, sigs, engine=None):
    """verify_schnorr_batch for signatures of ONE key, whose FixedBase table `base` serves every lane (two comb walks
    per signature)"""
    eng = engine or base.engine
    return _schnorr_results(*eng.verify_schnorr_base_batch(base, *_schnorr_sigs(msgs, sigs)))


def verify_schnorr_keyset_batch(keyset, key_index, msgs, sigs, engine=None):
    """verify_schnorr_batch with pk = keyset.points[key_index[i]] (two comb walks per signature).  An index outside the
    set raises BjjError (BJJ_ERR_ARG)."""
    eng = engine or keyset.engine
    ki = np.asarray(key_index, dtype=np.int64).reshape(-1)
    return _schnorr_results(*eng.verify_schnorr_keyset_batch(keyset, ki, *_schnorr_sigs(msgs, sigs)))


def multi_gpu(devices=None):
    """One Engine per device (all visible devices by default); see sharding.MultiGpu.run_sharded"""
    lib = _lib.load()
    if devices is None:
        devices = list(range(lib.bjj_device_count()))
    if not devices:
        raise RuntimeError("babyjubjub-rs_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return MultiGpu(Engine, devices)


def verify_batch_multi(mg, r8x, r8y, s, ax, ay, msg):
    """verify_batch sharded over every device of `mg` (contiguous slices, one host thread per device)"""
    ins = [_as_u8(v, 32) for v in (r8x, r8y, s, ax, ay, msg)]
    ok = np.empty(len(ins[0]), dtype=np.uint8)

    def work(eng, lo, hi):
        ok[lo:hi] = eng.verify_batch(*[v[lo:hi] for v in ins])
    mg.run_sharded(len(ok), work)
    return ok


class MultiEngine:
    """bjj_multi (include/bjj_cuda.h): ONE caller, ONE host batch, every device of the box -- config 4 as written.

    The library owns one context and one persistent host thread per device; a call cuts the arrays into
    contiguous shards and returns when all are done.  No NCCL: lanes never exchange anything.  `out=` lets a
    caller supply pinned result buffers (bjj_host_alloc); inputs may be pageable or pinned numpy arrays."""

    def __init__(self, devices=None, host_register=False):
        self.lib = _lib.load()
        if self.lib.bjj_device_count() < 1:
            raise RuntimeError("babyjubjub-rs_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        handle = ctypes.c_void_p()
        if devices is None:
            rc = self.lib.bjj_multi_init(0, None, ctypes.byref(handle))
        else:
            arr = (ctypes.c_int * len(devices))(*[int(d) for d in devices])
            rc = self.lib.bjj_multi_init(len(devices), arr, ctypes.byref(handle))
        if rc != 0:
            raise BjjError(rc, "bjj_multi_init", self.lib.bjj_error_string(rc).decode())
        self.handle = handle
        self.lib.bjj_multi_set_host_register(self.handle, 1 if host_register else 0)

    def close(self):
        if getattr(self, "handle", None):
            self.lib.bjj_multi_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def devices(self):
        return int(self.lib.bjj_multi_devices(self.handle))

    @property
    def kernel_launches(self):
        return int(self.lib.bjj_multi_kernel_launches(self.handle))

    def set_host_register(self, on):
        self.lib.bjj_multi_set_host_register(self.handle, 1 if on else 0)

    def _check(self, rc, what):
        if rc != 0:
            raise BjjError(rc, what, self.lib.bjj_error_string(rc).decode())

    def verify_batch(self, r8x, r8y, s, ax, ay, msg, out=None):
        ins = [_as_u8(v, 32) for v in (r8x, r8y, s, ax, ay, msg)]
        ok = np.empty(len(ins[0]), dtype=np.uint8) if out is None else out
        self._check(self.lib.bjj_multi_verify_batch(self.handle, len(ins[0]), *[_ptr(v) for v in ins], _ptr(ok)),
                    "bjj_multi_verify_batch")
        return ok

    def verify_compressed_batch(self, sig64, pk32, msg, out=None):
        sig64, pk32, msg = _as_u8(sig64, 64), _as_u8(pk32, 32), _as_u8(msg, 32)
        n = len(sig64)
        ok, st = (np.empty(n, dtype=np.uint8), np.empty(n, dtype=np.uint8)) if out is None else out
        self._check(self.lib.bjj_multi_verify_compressed_batch(self.handle, n, _ptr(sig64), _ptr(pk32), _ptr(msg), _ptr(ok),
                                                               _ptr(st)), "bjj_multi_verify_compressed_batch")
        return ok, st

    def mul_scalar_batch(self, px, py, scalars, out=None):
        px, py, k = _as_u8(px, 32), _as_u8(py, 32), _as_u8(scalars, 32)
        rx, ry = (np.empty_like(px), np.empty_like(px)) if out is None else out
        self._check(self.lib.bjj_multi_mul_scalar_batch(self.handle, len(px), _ptr(px), _ptr(py), _ptr(k), _ptr(rx), _ptr(ry)),
                    "bjj_multi_mul_scalar_batch")
        return rx, ry

    def msm_batch(self, px, py, scalars):
        """Engine.msm_batch over the devices: each sums its shard, device slot 0 sums the partial sums"""
        px, py, k = _as_u8(px, 32), _as_u8(py, 32), _as_u8(scalars, 32)
        if not len(px) == len(py) == len(k):
            raise ValueError("px, py and scalars differ in length")
        rx, ry = np.zeros((1, 32), np.uint8), np.zeros((1, 32), np.uint8)
        st = np.zeros(len(px), np.uint8)
        rc = self.lib.bjj_multi_msm_batch(self.handle, len(px), _ptr(px), _ptr(py), _ptr(k), _ptr(rx), _ptr(ry), _ptr(st))
        try:
            self._check(rc, "bjj_multi_msm_batch")
        except BjjError as e:
            e.point_status = st
            raise
        return rx, ry, st

    def public_batch(self, keys, out=None):
        keys = _as_u8(keys, 32)
        rx, ry = (np.empty_like(keys), np.empty_like(keys)) if out is None else out
        self._check(self.lib.bjj_multi_public_batch(self.handle, len(keys), _ptr(keys), _ptr(rx), _ptr(ry)),
                    "bjj_multi_public_batch")
        return rx, ry

    def public_compressed_batch(self, keys, out=None):
        keys = _as_u8(keys, 32)
        out = np.empty_like(keys) if out is None else out
        self._check(self.lib.bjj_multi_public_compressed_batch(self.handle, len(keys), _ptr(keys), _ptr(out)),
                    "bjj_multi_public_compressed_batch")
        return out

    def sign_compressed_batch(self, keys, msgs, out=None):
        keys, msgs = _as_u8(keys, 32), _as_u8(msgs, 32)
        n = len(keys)
        sig, st = (np.empty((n, 64), dtype=np.uint8), np.empty(n, dtype=np.uint8)) if out is None else out
        self._check(self.lib.bjj_multi_sign_compressed_batch(self.handle, n, _ptr(keys), _ptr(msgs), _ptr(sig), _ptr(st)),
                    "bjj_multi_sign_compressed_batch")
        return sig, st

    def sign_schnorr_batch(self, keys, msgs, nonces, words, out=None):
        keys, msgs = _as_u8(keys, 32), _as_u8(msgs, 32)
        kn = _as_u8(nonces, 4 * int(words))
        n = len(keys)
        if not n == len(msgs) == len(kn):
            raise ValueError("keys, msgs and nonces differ in length")
        rx, ry, s, st = ((np.empty_like(keys), np.empty_like(keys), np.empty((n, 4 * (int(words) + 8)), dtype=np.uint8),
                          np.empty(n, dtype=np.uint8)) if out is None else out)
        self._check(self.lib.bjj_multi_sign_schnorr_batch(self.handle, n, _ptr(keys), _ptr(msgs), _ptr(kn), int(words), _ptr(rx),
                                                          _ptr(ry), _ptr(s), _ptr(st)), "bjj_multi_sign_schnorr_batch")
        return rx, ry, s, st

    def fixed_base_batch(self, scalars, out=None):
        k = _as_u8(scalars, 32)
        rx, ry = (np.empty_like(k), np.empty_like(k)) if out is None else out
        self._check(self.lib.bjj_multi_fixed_base_batch(self.handle, len(k), _ptr(k), _ptr(rx), _ptr(ry)),
                    "bjj_multi_fixed_base_batch")
        return rx, ry

    def decompress_batch(self, comp, out=None):
        comp = _as_u8(comp, 32)
        n = len(comp)
        rx, ry, st = (np.empty_like(comp), np.empty_like(comp), np.empty(n, dtype=np.uint8)) if out is None else out
        self._check(self.lib.bjj_multi_decompress_batch(self.handle, n, _ptr(comp), _ptr(rx), _ptr(ry), _ptr(st)),
                    "bjj_multi_decompress_batch")
        return rx, ry, st
