"""Kernel launches per call (bjj_kernel_launches) of every entry point, host and _dev flavour, with the default
settings.  The count pins the sub-batch loop and the chunking of the host flavour: a call that splits its lanes
differently, or skips or repeats a kernel, changes it."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

# op: (launches of one call of 1,000 lanes in either flavour, arguments after the context).  Z: zeros, O: the point
# (0, 1) in every lane, R[i]: outputs.
CALLS = {
    "fr_op": (1, lambda n, Z, O, R: (0, n, Z, Z, R[0])),
    "split_scalars": (1, lambda n, Z, O, R: (n, Z, Z, R[0], R[1], R[2])),
    "add": (1, lambda n, Z, O, R: (n, Z, O, O, Z, O, O, R[0], R[1], R[2])),
    "affine": (1, lambda n, Z, O, R: (n, Z, O, O, R[0], R[1])),
    "mul_scalar": (3, lambda n, Z, O, R: (n, Z, O, Z, R[0], R[1])),                 # + exact ladder, batched affine
    "mul_scalar_wide": (4, lambda n, Z, O, R: (n, Z, O, Z, 16, R[0], R[1])),        # + scalar reduction
    "fixed_base": (2, lambda n, Z, O, R: (n, Z, R[0], R[1])),                       # comb kernel + batched affine
    "public": (3, lambda n, Z, O, R: (n, Z, R[0], R[1])),                           # + BLAKE-512 scalar
    "scalar_key": (1, lambda n, Z, O, R: (n, Z, R[0])),
    "sign": (7, lambda n, Z, O, R: (n, Z, Z, R[0], R[1], R[2], R[3])),
    "compress": (1, lambda n, Z, O, R: (n, Z, O, R[0])),
    "decompress": (3, lambda n, Z, O, R: (n, Z, R[0], R[1], R[2])),
    "poseidon": (1, lambda n, Z, O, R: (2, n, (ctypes.c_void_p * 2)(Z, Z), R[0])),
    "verify": (4, lambda n, Z, O, R: (n, Z, O, Z, Z, O, Z, R[0])),
    "verify_schnorr": (3, lambda n, Z, O, R: (n, Z, O, Z, Z, O, Z, R[0], R[1])),
    "verify_compressed": (8, lambda n, Z, O, R: (n, Z, Z, Z, R[0], R[1])),
}
# 2^21 + 5 lanes: the host flavour runs three chunks (2^18, 2^19, the rest), the _dev flavour two sub-batches
BIG = (1 << 21) + 5
BIG_CALLS = {("verify", False): 12, ("verify", True): 8, ("public", False): 9, ("public", True): 6}


def test_kernel_launches_per_call(gpu):
    lib, ctx = gpu.eng.lib, gpu.eng.ctx
    zeros = np.zeros((BIG, 64), dtype=np.uint8)
    ones = zeros.copy()
    ones.reshape(-1, 32)[:, 0] = 1
    outs = [np.empty((BIG, 64), dtype=np.uint8) for _ in range(4)]
    host = [a.ctypes.data_as(ctypes.c_void_p) for a in (zeros, ones)] + [[a.ctypes.data_as(ctypes.c_void_p) for a in outs]]
    dptrs = [ctypes.c_void_p(lib.bjj_dev_alloc(ctx, zeros.nbytes)) for _ in range(6)]
    try:
        assert all(p.value for p in dptrs)
        for p, a in zip(dptrs, (zeros, ones)):
            assert lib.bjj_memcpy_h2d(ctx, p, a.ctypes.data_as(ctypes.c_void_p), a.nbytes) == 0
        dev = dptrs[:2] + [dptrs[2:]]
        small = {(op, d): count for op, (count, _) in CALLS.items() for d in (False, True)}
        got, want = {}, {}
        for n, table in ((1000, small), (BIG, BIG_CALLS)):
            for (op, d), count in table.items():
                fn = getattr(lib, "bjj_%s_batch%s" % (op, "_dev" if d else ""))
                before = lib.bjj_kernel_launches(ctx)
                rc = fn(ctx, *CALLS[op][1](n, *(dev if d else host)), *((None,) if d else ()))
                assert rc == 0, (op, d, n, rc)
                got[op, d, n], want[op, d, n] = lib.bjj_kernel_launches(ctx) - before, count
        assert lib.bjj_sync(ctx) == 0
        assert got == want
    finally:
        for p in dptrs:
            lib.bjj_dev_free(ctx, p)
