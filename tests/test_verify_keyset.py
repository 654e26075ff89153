"""key sets (bjj_keyset_create, bjj_verify_keyset_batch, bjj_verify_keyset_compressed_batch, bjj_keyset_mul_batch): the
8-bit recoding, the compact tables and the lane bodies compiled for the host against the oracle; on the GPU both
flavours against the oracle and byte for byte against bjj_verify_batch with the keys gathered per lane (and against
bjj_verify_base_batch / bjj_base_mul_batch for one key), chunk and sub-batch boundaries, out-of-range key indices, a
non-canonical R8, creation errors, launch counts, a workspace shared with verify_batch's deferred exact lanes, and the
Python / C++ mirrors."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

from common import KEY_KAT, MSG_KAT, ROOT, pack, unpack
from oracle import bjj_oracle as O
from test_verify_base import case_arrays, compressed_cases, edge_cases, keys_with_secrets, oracle_ok

Q, ORDER, SUBORDER = O.Q, O.ORDER, O.SUBORDER
ERR_ARG, ERR_NONCANONICAL = 2, 3
BIG = (1 << 21) + 5
MASK = (1 << 256) - 1
BUILD_SUBBATCH = (1 << 21) // 4097          # keys per build sub-batch of bjj_keyset_create

CPP_SRC = os.path.join(ROOT, "tests", "cpp", "test_keyset.cpp")
PKG = os.path.join(ROOT, "babyjubjub-rs_b200")


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def u32(a):
    return np.ascontiguousarray(a, dtype="<u4")


def key_arrays(keys):
    return pack([k[0] for k in keys]), pack([k[1] for k in keys])


def interleaved_cases(rnd, kinds, make):
    """every key kind's cases (make(rnd, A, a)), interleaved across lanes -> key index per lane, cases"""
    per = [[(j, c) for c in make(rnd, A, a)] for j, (_, A, a) in enumerate(kinds)]
    lanes = [x for group in per for x in group]
    rnd.shuffle(lanes)
    return np.array([j for j, _ in lanes], np.uint32), [c for _, c in lanes]


# ---- CPU ----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def keyset_emu(tmp_path_factory):
    """tests/hostemu/keyset_emu.cpp (the key-set lane bodies compiled for the host), built into a temporary directory"""
    from common import build_hostemu
    build_hostemu()                     # generates the constants header the device sources include
    so = str(tmp_path_factory.mktemp("keyset_emu") / "libbjj_keyset_emu.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so,
                           os.path.join(ROOT, "tests", "hostemu", "keyset_emu.cpp")])
    lib = ctypes.CDLL(so)
    for f in ("emu_keyset_create", "emu_keyset_entry", "emu_keyset_mul", "emu_verify_keyset", "emu_verify_keyset_compressed"):
        getattr(lib, f).restype = ctypes.c_uint32
    return lib


def emu_create(emu, keys):
    ax, ay = key_arrays(keys)
    st = np.full(len(keys), 0xEE, np.uint8)
    rc = emu.emu_keyset_create(ctypes.c_size_t(len(keys)), _p(ax), _p(ay), _p(st))
    return rc, st


def test_hostemu_recode8(keyset_emu):
    """the 32 signed digits in [-128, 127] and the carry recombine to k"""
    rnd = random.Random(60)
    ks = [0, 1, ORDER - 1, ORDER, MASK, int.from_bytes(b"\x7f" * 32, "little"), int.from_bytes(b"\x80" * 32, "little"),
          int.from_bytes(b"\xff" * 32, "little"), int.from_bytes(b"\x7f\x80" * 16, "little"), Q, SUBORDER]
    ks += [rnd.getrandbits(256) for _ in range(300)]
    digits = np.zeros((len(ks), 33), np.int32)
    keyset_emu.emu_recode8(ctypes.c_size_t(len(ks)), _p(pack(ks)), _p(digits))
    for k, d in zip(ks, digits.tolist()):
        assert all(-128 <= v <= 127 for v in d[:32]) and d[32] in (0, 1), k
        assert sum(v << (8 * i) for i, v in enumerate(d)) == k, k


def test_hostemu_table_entries(keyset_emu):
    """entries j * 256^w * P of every key of a small set against the oracle: w in {0, 1, 31, 32}, j in {0, 1, 127, 128}
    (j <= 1 in the carry window) and random (w, j)"""
    kinds = keys_with_secrets()
    rc, st = emu_create(keyset_emu, [A for _, A, _ in kinds])
    assert rc == 0 and not st.any()
    rnd = random.Random(61)
    x, y = np.zeros(32, np.uint8), np.zeros(32, np.uint8)
    for key, (name, A, _) in enumerate(kinds):
        spots = [(w, j) for w in (0, 1, 31) for j in (0, 1, 127, 128)] + [(32, 0), (32, 1)]
        spots += [(rnd.randrange(32), rnd.randrange(129)) for _ in range(6)]
        for w, j in spots:
            assert keyset_emu.emu_keyset_entry(ctypes.c_size_t(key), w, j, _p(x), _p(y)) == 1, (name, w, j)
            want = O.mul_scalar(A, j << (8 * w))
            assert (unpack(x)[0], unpack(y)[0]) == want, (name, w, j)


def test_hostemu_create_rejects(keyset_emu):
    """key status codes: off the curve 1, a coordinate >= Q 2"""
    good = O.public(KEY_KAT)
    rc, st = emu_create(keyset_emu, [good, (good[0], (good[1] + 1) % Q), (good[0] + Q, good[1]) if good[0] + Q <= MASK else (Q, 1)])
    assert rc == 1 and list(st) == [0, 1, 2]


def test_hostemu_mul_against_oracle(keyset_emu):
    """the walk over the compact tables equals mul_scalar for every key kind, on scalar edges and random scalars; an
    index outside the set gives (0, 0) and the KEY_INDEX flag"""
    kinds = keys_with_secrets()
    rc, _ = emu_create(keyset_emu, [A for _, A, _ in kinds])
    assert rc == 0
    rnd = random.Random(62)
    scalars = [0, 1, 2, 7, 8, SUBORDER - 1, SUBORDER, ORDER - 1, ORDER, ORDER + 1, MASK, int.from_bytes(b"\x80" * 32, "little")]
    lanes = [(j, k) for j in range(len(kinds)) for k in scalars + [rnd.getrandbits(256) for _ in range(4)]]
    idx = np.array([j for j, _ in lanes] + [len(kinds)], np.uint32)
    ks = pack([k for _, k in lanes] + [5])
    rx, ry = np.zeros((len(idx), 32), np.uint8), np.zeros((len(idx), 32), np.uint8)
    flags = keyset_emu.emu_keyset_mul(ctypes.c_size_t(len(idx)), _p(u32(idx)), _p(ks), _p(rx), _p(ry))
    assert flags == 2
    got = list(zip(unpack(rx), unpack(ry)))
    for i, (j, k) in enumerate(lanes):
        assert got[i] == O.mul_scalar(kinds[j][1], k), (kinds[j][0], k)
    assert got[-1] == (0, 0)


def test_hostemu_verify_against_oracle(keyset_emu):
    """the two lane bodies against the oracle's verify on the edge cases of every key kind, all kinds in one set and
    interleaved across lanes; an index outside the set rejects its lane only and sets the KEY_INDEX flag"""
    kinds = keys_with_secrets()
    rc, _ = emu_create(keyset_emu, [A for _, A, _ in kinds])
    assert rc == 0
    idx, cases = interleaved_cases(random.Random(63), kinds, edge_cases)
    want = np.array([oracle_ok(kinds[j][1], [c])[0] for j, c in zip(idx, cases)], np.uint8)
    assert want.sum() >= 4 * len(kinds)
    ins = case_arrays(cases)
    ok = np.full(len(cases), 0xEE, np.uint8)
    assert keyset_emu.emu_verify_keyset(ctypes.c_size_t(len(cases)), _p(u32(idx)), *[_p(v) for v in ins], _p(ok)) == 0
    assert list(ok) == list(want), [i for i in range(len(cases)) if ok[i] != want[i]]
    bad = idx.copy()
    bad[0], bad[5] = len(kinds), 0xFFFFFFFF
    ok = np.full(len(cases), 0xEE, np.uint8)
    assert keyset_emu.emu_verify_keyset(ctypes.c_size_t(len(cases)), _p(u32(bad)), *[_p(v) for v in ins], _p(ok)) == 2
    w2 = want.copy()
    w2[[0, 5]] = 0
    assert list(ok) == list(w2)


def test_hostemu_compressed_against_oracle(keyset_emu):
    """R8's decompression phases and the two lane bodies against decompress_signature + verify, per key kind"""
    kinds = keys_with_secrets()
    rc, _ = emu_create(keyset_emu, [A for _, A, _ in kinds])
    assert rc == 0
    for j, (name, A, a) in enumerate(kinds):
        sig64, msgs, want_ok, want_st = compressed_cases(random.Random(64 + j), A, a)
        idx = np.full(len(sig64), j, np.uint32)
        ok, st = np.full(len(sig64), 0xEE, np.uint8), np.full(len(sig64), 0xEE, np.uint8)
        assert keyset_emu.emu_verify_keyset_compressed(ctypes.c_size_t(len(sig64)), _p(idx), _p(sig64), _p(msgs), _p(ok), _p(st)) == 0
        assert list(st) == list(want_st), name
        assert list(ok) == list(want_ok), name


def test_python_key_index_handling():
    import babyjubjub_rs_b200 as bjj
    ki = bjj._key_index([0, 5, 0xFFFFFFFF], 3)
    assert ki.dtype == np.dtype("<u4") and list(ki) == [0, 5, 0xFFFFFFFF]
    for bad in ([-1, 0], [1 << 32, 0]):
        with pytest.raises(ValueError):
            bjj._key_index(bad, 2)
    with pytest.raises(ValueError):
        bjj._key_index([0, 1, 2], 2)
    with pytest.raises(ValueError):
        bjj._keyset_handle(None)


def build_cpp(out_dir):
    exe = os.path.join(str(out_dir), "test_keyset")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-pthread", "-o", exe, CPP_SRC, "-L" + PKG, "-lbjj_cuda",
                           "-Wl,-rpath," + PKG])
    return exe


def test_cpp_keyset_builds_and_links(tmp_path):
    assert os.path.exists(build_cpp(tmp_path))


# ---- GPU ----------------------------------------------------------------------------------------------
def keyset(lib, ctx, keys_xy):
    """a key set of (n, 32) coordinate arrays -> (handle, rc, key_status)"""
    ax, ay = keys_xy
    st = np.full(len(ax), 0xEE, np.uint8)
    h = ctypes.c_void_p()
    rc = lib.bjj_keyset_create(ctx, len(ax), _p(ax), _p(ay), _p(st), ctypes.byref(h))
    return h, rc, st


def call(lib, ctx, name, ks, idx, ins, outs, dev, sync_rc=0):
    """bjj_<name>_batch (host or _dev flavour) over key set ks with key indices idx and host arrays `ins`; fills `outs`,
    returns the rc"""
    n = len(idx)
    fn = getattr(lib, "bjj_%s_batch%s" % (name, "_dev" if dev else ""))
    idx = u32(idx)
    if not dev:
        return fn(ctx, ks, n, *[_p(a) for a in [idx] + ins + outs])
    arrs = [idx] + ins + outs
    bufs = [lib.bjj_dev_alloc(ctx, max(a.nbytes, 1)) for a in arrs]
    try:
        assert all(bufs)
        for b, a in zip(bufs, arrs[:1 + len(ins)]):
            assert lib.bjj_memcpy_h2d(ctx, b, _p(a), a.nbytes) == 0
        rc = fn(ctx, ks, n, *bufs, None)
        for b, a in zip(bufs[1 + len(ins):], outs):
            assert lib.bjj_memcpy_d2h(ctx, _p(a), b, a.nbytes) == 0
        assert lib.bjj_sync(ctx) == sync_rc
    finally:
        for b in bufs:
            lib.bjj_dev_free(ctx, b)
    return rc


def verify_plain(lib, ctx, ks, idx, ins, dev, rc=0, sync_rc=0):
    ok = np.full(len(idx), 0xEE, np.uint8)
    assert call(lib, ctx, "verify_keyset", ks, idx, ins, [ok], dev, sync_rc) == rc
    return ok


def verify_packed(lib, ctx, ks, idx, sig64, msgs, dev, rc=0, sync_rc=0):
    ok, st = np.full(len(idx), 0xEE, np.uint8), np.full(len(idx), 0xEE, np.uint8)
    assert call(lib, ctx, "verify_keyset_compressed", ks, idx, [sig64, msgs], [ok, st], dev, sync_rc) == rc
    return ok, st


def signed_lanes(eng, n, n_keys, seed, corrupt=0.1, off_curve=0.01):
    """n signatures made on the device by n_keys keys (a seeded random key per lane), about `corrupt` of them corrupted
    (S, R8 or msg) and about `off_curve` given an off-curve R8 -> idx, [r8x, r8y, s, msg], (ax, ay) of the keys"""
    rng = np.random.default_rng(seed)
    priv = rng.integers(0, 256, size=(n_keys, 32), dtype=np.uint8)
    ax, ay = eng.public_batch(priv)
    idx = rng.integers(0, n_keys, size=n).astype(np.uint32)
    msgs = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    msgs[:, 31] &= 0x2F                                    # < Q
    r8x, r8y, s, st = eng.sign_batch(priv[idx], msgs)
    assert not st.any()
    lanes = rng.permutation(n)
    nc = int(n * corrupt)

    def flip_x(i, bit):
        x = int.from_bytes(r8x[i].tobytes(), "little") ^ (1 << bit)
        r8x[i] = np.frombuffer((x if x < Q else x - Q).to_bytes(32, "little"), np.uint8)
    for j, i in enumerate(lanes[:nc]):
        if j % 3 == 1:
            flip_x(i, int(rng.integers(0, 248)))
        else:
            [s, msgs][j % 3 // 2][i, rng.integers(0, 31)] ^= 1 << int(rng.integers(0, 8))
    for i in lanes[nc:nc + int(n * off_curve)]:
        flip_x(i, 0)
    return idx, [r8x, r8y, s, msgs], (ax, ay)


@pytest.mark.gpu
def test_against_oracle_both_flavours(gpu):
    """every key kind in one set, interleaved across lanes: both flavours of the plain and the compressed form against
    the oracle, status codes included"""
    eng = gpu.eng
    lib, ctx = eng.lib, eng.ctx
    kinds = keys_with_secrets()
    h, rc, st = keyset(lib, ctx, key_arrays([A for _, A, _ in kinds]))
    assert rc == 0 and not st.any()
    try:
        idx, cases = interleaved_cases(random.Random(70), kinds, edge_cases)
        want = np.array([oracle_ok(kinds[j][1], [c])[0] for j, c in zip(idx, cases)], np.uint8)
        for dev in (False, True):
            assert np.array_equal(verify_plain(lib, ctx, h, idx, case_arrays(cases), dev), want), dev
        parts = [compressed_cases(random.Random(71 + j), A, a) for j, (_, A, a) in enumerate(kinds)]
        cidx = np.concatenate([np.full(len(p[0]), j, np.uint32) for j, p in enumerate(parts)])
        perm = np.random.default_rng(71).permutation(len(cidx))
        sig64, msgs, want_ok, want_st = [np.concatenate([p[k] for p in parts])[perm] for k in range(4)]
        for dev in (False, True):
            ok, st = verify_packed(lib, ctx, h, cidx[perm], sig64, msgs, dev)
            assert np.array_equal(st, want_st) and np.array_equal(ok, want_ok), dev
    finally:
        lib.bjj_keyset_destroy(ctx, h)


@pytest.mark.gpu
def test_equal_to_verify_batch(gpu):
    """2^16 lanes of 1,000 keys made on the device, 10 % corrupted: ok byte-equal to bjj_verify_batch with A gathered per
    lane (and the compressed form to bjj_verify_compressed_batch); with one key also to bjj_verify_base_batch"""
    bjj, eng = gpu.bjj, gpu.eng
    n = 1 << 16
    idx, ins, (ax, ay) = signed_lanes(eng, n, 1000, 72, off_curve=0.02)
    want = eng.verify_batch(*ins[:3], ax[idx], ay[idx], ins[3])
    assert 0.85 * n < want.sum() < 0.95 * n
    ks = bjj.KeySet(list(zip(unpack(ax), unpack(ay))), eng)
    try:
        assert np.array_equal(eng.verify_keyset_batch(ks, idx, *ins), want)
        sig64 = np.concatenate([eng.compress_batch(ins[0], ins[1]), ins[2]], axis=1)
        rng = np.random.default_rng(72)
        bad = rng.choice(n, n // 50, replace=False)
        sig64[bad[: len(bad) // 2], 31] |= 0x7F            # y >= Q
        sig64[bad[len(bad) // 2:], 0] ^= 0x5A              # mostly not a square
        pk32 = eng.compress_batch(ax, ay)[idx]
        want_ok, want_st = eng.verify_compressed_batch(sig64, pk32, ins[3])
        assert set(np.unique(want_st)) >= {0, 1, 3}
        ok, st = eng.verify_keyset_compressed_batch(ks, idx, sig64, ins[3])
        assert np.array_equal(st, want_st) and np.array_equal(ok, want_ok)
    finally:
        ks.close()
    idx1, ins1, (ax1, ay1) = signed_lanes(eng, n, 1, 73)
    one = bjj.KeySet([(unpack(ax1)[0], unpack(ay1)[0])], eng)
    base = bjj.FixedBase((unpack(ax1)[0], unpack(ay1)[0]), eng)
    try:
        want = eng.verify_batch(*ins1[:3], ax1[idx1], ay1[idx1], ins1[3])
        assert np.array_equal(eng.verify_base_batch(base, *ins1), want)
        assert np.array_equal(eng.verify_keyset_batch(one, idx1, *ins1), want)
    finally:
        one.close()
        base.close()


@pytest.mark.gpu
def test_chunk_and_subbatch_boundaries(gpu, oracle_c):
    """2^21 + 5 lanes of 300 keys: the host flavour runs three chunks, _dev two sub-batches, both equal to verify_batch;
    launches per sub-batch 2 (plain) and 5 (compressed), also at 1,000 lanes; mul 2 per sub-batch; sampled lanes
    against the oracle"""
    eng = gpu.eng
    lib, ctx = eng.lib, eng.ctx
    idx, ins, (ax, ay) = signed_lanes(eng, BIG, 300, 74)
    sig64 = np.concatenate([eng.compress_batch(ins[0], ins[1]), ins[2]], axis=1)
    sig64[7::97, 31] |= 0x7F                               # y >= Q
    want = eng.verify_batch(*ins[:3], ax[idx], ay[idx], ins[3])
    want_ok, want_st = eng.verify_compressed_batch(sig64, eng.compress_batch(ax, ay)[idx], ins[3])
    h, rc, _ = keyset(lib, ctx, (ax, ay))
    assert rc == 0

    def launches(fn):
        before = lib.bjj_kernel_launches(ctx)
        r = fn()
        return r, lib.bjj_kernel_launches(ctx) - before
    try:
        for dev in (False, True):
            small = [a[:1000] for a in ins]
            _, k = launches(lambda: verify_plain(lib, ctx, h, idx[:1000], small, dev))
            assert k == 2, (dev, k)
            _, k = launches(lambda: verify_packed(lib, ctx, h, idx[:1000], sig64[:1000], ins[3][:1000], dev))
            assert k == 5, (dev, k)
            rx, ry = np.zeros((1000, 32), np.uint8), np.zeros((1000, 32), np.uint8)
            _, k = launches(lambda: call(lib, ctx, "keyset_mul", h, idx[:1000], [ins[2][:1000]], [rx, ry], dev))
            assert k == 2, (dev, k)
            ok, k = launches(lambda: verify_plain(lib, ctx, h, idx, ins, dev))
            assert k == (6 if not dev else 4), (dev, k)
            assert np.array_equal(ok, want), dev
            (cok, cst), k = launches(lambda: verify_packed(lib, ctx, h, idx, sig64, ins[3], dev))
            assert k == (15 if not dev else 10), (dev, k)
            assert np.array_equal(cok, want_ok) and np.array_equal(cst, want_st), dev
    finally:
        lib.bjj_keyset_destroy(ctx, h)
    sample = sorted(set(random.Random(74).sample(range(BIG), 2000)) | {0, (1 << 18) - 1, 1 << 18, (1 << 21) - 1, 1 << 21, BIG - 1})
    s_ins = [a[sample] for a in ins]
    assert np.array_equal(want[sample], oracle_c.verify(*s_ins[:3], ax[idx[sample]], ay[idx[sample]], s_ins[3]))


@pytest.mark.gpu
def test_key_index_out_of_range(gpu):
    """key_index >= n_keys: ok = 0 on that lane only (status 0 in the compressed form, (0, 0) from mul), BJJ_ERR_ARG
    from the host flavour and from bjj_sync after a _dev call, and the next call is clean; ARG outranks NONCANONICAL"""
    eng = gpu.eng
    lib, ctx = eng.lib, eng.ctx
    n = 4096
    idx, ins, (ax, ay) = signed_lanes(eng, n, 17, 75)
    want = eng.verify_batch(*ins[:3], ax[idx], ay[idx], ins[3])
    sig64 = np.concatenate([eng.compress_batch(ins[0], ins[1]), ins[2]], axis=1)
    # the compressed form decompresses R8 from its y and sign bit, so an off-curve R8 of `ins` does not survive: its
    # reference is verify_compressed_batch on the same 64-byte signatures
    want_c, want_st = eng.verify_compressed_batch(sig64, eng.compress_batch(ax, ay)[idx], ins[3])
    h, rc, _ = keyset(lib, ctx, (ax, ay))
    assert rc == 0
    bad = idx.copy()
    bad[[3, 100, n - 1]] = [17, 0xFFFFFFFF, 1000]
    w2, w2_c = want.copy(), want_c.copy()
    w2[[3, 100, n - 1]] = 0
    w2_c[[3, 100, n - 1]] = 0
    try:
        for dev in (False, True):
            rc_call, rc_sync = (0, ERR_ARG) if dev else (ERR_ARG, 0)
            assert np.array_equal(verify_plain(lib, ctx, h, bad, ins, dev, rc_call, rc_sync), w2), dev
            ok, st = verify_packed(lib, ctx, h, bad, sig64, ins[3], dev, rc_call, rc_sync)
            assert np.array_equal(ok, w2_c) and np.array_equal(st, want_st), dev      # status: R8's alone
            rx, ry = np.full((n, 32), 0xEE, np.uint8), np.full((n, 32), 0xEE, np.uint8)
            assert call(lib, ctx, "keyset_mul", h, bad, [ins[2]], [rx, ry], dev, rc_sync) == rc_call
            assert not rx[[3, 100, n - 1]].any() and not ry[[3, 100, n - 1]].any()
            assert np.array_equal(verify_plain(lib, ctx, h, idx, ins, dev), want), dev      # the next call is clean
        nc = [a.copy() for a in ins]
        nc[0][5] = pack([unpack(nc[0][5:6])[0] + Q if unpack(nc[0][5:6])[0] + Q <= MASK else Q])[0]
        verify_plain(lib, ctx, h, bad, nc, False, ERR_ARG)
        verify_plain(lib, ctx, h, idx, nc, False, ERR_NONCANONICAL)
    finally:
        lib.bjj_keyset_destroy(ctx, h)


@pytest.mark.gpu
def test_noncanonical_r8(gpu):
    """a coordinate of R8 >= Q: BJJ_ERR_NONCANONICAL and the ok[] of bjj_verify_batch (the batch computed mod Q)"""
    eng = gpu.eng
    lib, ctx = eng.lib, eng.ctx
    n = 256
    idx, ins, (ax, ay) = signed_lanes(eng, n, 5, 76)
    xs = unpack(ins[0])
    for i in (3, 4):
        ins[0][i] = pack([xs[i] + Q])[0] if xs[i] + Q <= MASK else ins[0][i]
    assert any(unpack(ins[0])[i] >= Q for i in (3, 4))
    want = np.zeros(n, np.uint8)
    assert lib.bjj_verify_batch(ctx, n, *[_p(a) for a in ins[:3]], _p(ax[idx]), _p(ay[idx]), _p(ins[3]), _p(want)) == ERR_NONCANONICAL
    h, rc, _ = keyset(lib, ctx, (ax, ay))
    assert rc == 0
    try:
        assert np.array_equal(verify_plain(lib, ctx, h, idx, ins, False, ERR_NONCANONICAL), want)
        assert np.array_equal(verify_plain(lib, ctx, h, idx, ins, True, 0, ERR_NONCANONICAL), want)
    finally:
        lib.bjj_keyset_destroy(ctx, h)


@pytest.mark.gpu
def test_create_errors_and_arguments(gpu):
    """an off-curve key, a coordinate >= Q, n_keys = 0, NULL pointers, a handle of another context, destroy(NULL)"""
    bjj, eng = gpu.bjj, gpu.eng
    lib, ctx = eng.lib, eng.ctx
    good = [O.public(KEY_KAT), O.B8, (0, 1), (0, Q - 1)]
    off = list(good)
    off[2] = (5, 7)
    h, rc, st = keyset(lib, ctx, key_arrays(off))
    assert rc == ERR_ARG and not h.value and list(st) == [0, 0, 1, 0]
    nc = list(off)
    nc[1] = (O.B8[0] + Q, O.B8[1])
    h, rc, st = keyset(lib, ctx, key_arrays(nc))
    assert rc == ERR_NONCANONICAL and not h.value and list(st) == [0, 2, 1, 0]
    ax, ay = key_arrays(good)
    hh = ctypes.c_void_p()
    assert lib.bjj_keyset_create(ctx, 0, _p(ax), _p(ay), None, ctypes.byref(hh)) == ERR_ARG
    assert lib.bjj_keyset_create(ctx, 4, None, _p(ay), None, ctypes.byref(hh)) == ERR_ARG
    assert lib.bjj_keyset_create(ctx, 4, _p(ax), None, None, ctypes.byref(hh)) == ERR_ARG
    assert lib.bjj_keyset_create(None, 4, _p(ax), _p(ay), None, ctypes.byref(hh)) == ERR_ARG
    assert lib.bjj_keyset_create(ctx, 4, _p(ax), _p(ay), None, None) == ERR_ARG
    assert lib.bjj_keyset_create(ctx, 1 << 32, _p(ax), _p(ay), None, ctypes.byref(hh)) == ERR_ARG
    lib.bjj_keyset_destroy(ctx, None)
    with pytest.raises(bjj.BjjError) as e:
        bjj.KeySet(off, eng)
    assert e.value.code == ERR_ARG
    other = bjj.Engine(0)
    mine = bjj.KeySet(good, eng)
    foreign = bjj.KeySet(good, other)
    try:
        i4, a32, m = np.zeros(4, np.uint32), pack([1] * 4), pack([2] * 4)
        o, s64 = np.zeros(4, np.uint8), np.zeros((4, 64), np.uint8)
        for dev in (False, True):
            sfx, tail = ("_dev", (None,)) if dev else ("", ())
            plain = getattr(lib, "bjj_verify_keyset_batch" + sfx)
            packed = getattr(lib, "bjj_verify_keyset_compressed_batch" + sfx)
            mul = getattr(lib, "bjj_keyset_mul_batch" + sfx)
            for hnd in (None, foreign.handle):
                assert plain(ctx, hnd, 4, _p(i4), _p(a32), _p(a32), _p(a32), _p(m), _p(o), *tail) == ERR_ARG
                assert packed(ctx, hnd, 4, _p(i4), _p(s64), _p(m), _p(o), _p(o), *tail) == ERR_ARG
                assert mul(ctx, hnd, 4, _p(i4), _p(a32), _p(a32), _p(a32), *tail) == ERR_ARG
            assert plain(ctx, mine.handle, 0, _p(i4), _p(a32), _p(a32), _p(a32), _p(m), _p(o), *tail) == 0
            assert plain(ctx, mine.handle, 4, None, _p(a32), _p(a32), _p(a32), _p(m), _p(o), *tail) == ERR_ARG
            assert mul(ctx, mine.handle, 4, None, _p(a32), _p(a32), _p(a32), *tail) == ERR_ARG
        lib.bjj_keyset_destroy(ctx, foreign.handle)           # a handle of another context: not freed by this one
        assert foreign.handle
    finally:
        mine.close()
        foreign.close()
        other.close()


@pytest.mark.gpu
def test_mul_against_oracle_and_base_mul(gpu):
    """keyset_mul equals mul_scalar on scalar edges for every key kind, and bjj_base_mul_batch for the same point"""
    bjj, eng = gpu.bjj, gpu.eng
    kinds = keys_with_secrets()
    ks = bjj.KeySet([A for _, A, _ in kinds], eng)
    try:
        rnd = random.Random(77)
        scalars = [0, 1, 2, 8, SUBORDER - 1, SUBORDER, ORDER - 1, ORDER, ORDER + 1, MASK, int.from_bytes(b"\x80" * 32, "little")]
        scalars += [rnd.getrandbits(256) for _ in range(5)]
        lanes = [(j, k) for j in range(len(kinds)) for k in scalars]
        rnd.shuffle(lanes)
        got = ks.mul_batch([j for j, _ in lanes], [k for _, k in lanes])
        for (j, k), p in zip(lanes, got):
            assert (p.x, p.y) == O.mul_scalar(kinds[j][1], k), (kinds[j][0], k)
        rng = np.random.default_rng(77)
        n = 50000
        kk = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
        for j, (name, A, _) in enumerate(kinds):
            base = bjj.FixedBase(A, eng)
            try:
                want = eng.base_mul_batch(base, kk)
            finally:
                base.close()
            got = eng.keyset_mul_batch(ks, np.full(n, j, np.uint32), kk)
            assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), name
    finally:
        ks.close()


@pytest.mark.gpu
def test_create_launches_and_build_subbatches(gpu):
    """bjj_keyset_create launches 1 check kernel + 2 per sub-batch of 511 keys; a set of 1,200 keys (three build
    sub-batches) serves keys of every sub-batch like FixedBase tables do"""
    bjj, eng = gpu.bjj, gpu.eng
    lib, ctx = eng.lib, eng.ctx
    rng = np.random.default_rng(78)
    priv = rng.integers(0, 256, size=(1200, 32), dtype=np.uint8)
    ax, ay = eng.public_batch(priv)
    for n_keys in (6, 1200):
        before = lib.bjj_kernel_launches(ctx)
        h, rc, st = keyset(lib, ctx, (ax[:n_keys], ay[:n_keys]))
        assert rc == 0 and not st.any()
        try:
            assert lib.bjj_kernel_launches(ctx) - before == 1 + 2 * (-(-n_keys // BUILD_SUBBATCH)), n_keys
            if n_keys == 1200:
                pick = [0, 1, 510, 511, 512, 1021, 1022, 1023, 1199]
                kk = rng.integers(0, 256, size=(len(pick), 32), dtype=np.uint8)
                rx, ry = np.zeros_like(kk), np.zeros_like(kk)
                assert call(lib, ctx, "keyset_mul", h, np.array(pick, np.uint32), [kk], [rx, ry], False) == 0
                for i, j in enumerate(pick):
                    assert O.mul_scalar((unpack(ax[j:j + 1])[0], unpack(ay[j:j + 1])[0]), unpack(kk[i:i + 1])[0]) == \
                        (unpack(rx[i:i + 1])[0], unpack(ry[i:i + 1])[0]), j
        finally:
            lib.bjj_keyset_destroy(ctx, h)


@pytest.mark.gpu
def test_after_verify_batch_with_exact_lanes(gpu):
    """verify_batch with many off-curve lanes (its exact kernel runs deferred on the workspace's side stream), then at
    once verify_keyset_batch on the same context: both correct, in both flavours"""
    bjj, eng = gpu.bjj, gpu.eng
    lib, ctx = eng.lib, eng.ctx
    n = (1 << 20) + 3
    idx, ins, (ax, ay) = signed_lanes(eng, n, 64, 79, off_curve=0.05)
    axn, ayn = ax[idx], ay[idx]
    ks = bjj.KeySet(list(zip(unpack(ax), unpack(ay))), eng)
    try:
        first = eng.verify_batch(*ins[:3], axn, ayn, ins[3])
        second = eng.verify_keyset_batch(ks, idx, *ins)
        assert np.array_equal(first, second)
        arrs = ins + [axn, ayn, u32(idx)]
        bufs = [lib.bjj_dev_alloc(ctx, a.nbytes) for a in arrs]
        okv, okk = lib.bjj_dev_alloc(ctx, n), lib.bjj_dev_alloc(ctx, n)
        try:
            for b, a in zip(bufs, arrs):
                assert lib.bjj_memcpy_h2d(ctx, b, _p(a), a.nbytes) == 0
            r8x, r8y, s, msg, dax, day, didx = bufs
            assert lib.bjj_verify_batch_dev(ctx, n, r8x, r8y, s, dax, day, msg, okv, None) == 0
            assert lib.bjj_verify_keyset_batch_dev(ctx, ks.handle, n, didx, r8x, r8y, s, msg, okk, None) == 0
            got_v, got_k = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
            assert lib.bjj_memcpy_d2h(ctx, _p(got_v), okv, n) == 0
            assert lib.bjj_memcpy_d2h(ctx, _p(got_k), okk, n) == 0
            assert lib.bjj_sync(ctx) == 0
        finally:
            for b in bufs + [okv, okk]:
                lib.bjj_dev_free(ctx, b)
        assert np.array_equal(got_v, first) and np.array_equal(got_k, first)
    finally:
        ks.close()


@pytest.mark.gpu
def test_python_and_cpp_mirrors(gpu, tmp_path):
    bjj, eng = gpu.bjj, gpu.eng
    keys = [KEY_KAT, bytes(range(32)), bytes(range(1, 33))]
    pks = [bjj.Point(*O.public(k)) for k in keys]
    msgs = [MSG_KAT, 0, Q, Q + 1, 1 << 256, 12345, 99]
    idx = [0, 1, 2, 0, 1, 2, 1]
    sigs = []
    for j, msg in zip(idx, msgs):
        r8, s = O.sign(keys[j], msg if msg <= Q else MSG_KAT)
        sigs.append(bjj.Signature(bjj.Point(*r8), s))
    sigs[5] = bjj.Signature(sigs[5].r_b8, sigs[5].s ^ 1)
    sigs[6] = bjj.Signature(sigs[6].r_b8, sigs[6].s + (SUBORDER << 300))      # wider S: reduced mod SUBORDER
    ks = bjj.KeySet(pks, eng)
    try:
        assert len(ks) == 3
        got = bjj.verify_keyset_batch(ks, idx, sigs, msgs)
        assert got == [True, True, True, False, False, False, True]
        assert got == bjj.verify_batch([pks[j] for j in idx], sigs, msgs, engine=eng)
        assert bjj.verify_keyset_batch(ks, [], [], []) == []
        with pytest.raises(bjj.BjjError) as e:
            bjj.verify_keyset_batch(ks, [0, 3], sigs[:2], msgs[:2])
        assert e.value.code == ERR_ARG
        pts = ks.mul_batch([2, 0, 1], [5, -7, ORDER + (1 << 300)])
        assert [(p.x, p.y) for p in pts] == [O.mul_scalar(O.public(keys[2]), 5), O.mul_scalar(O.public(keys[0]), 7),
                                             O.mul_scalar(O.public(keys[1]), (ORDER + (1 << 300)) % ORDER)]
    finally:
        ks.close()
    out = subprocess.run([build_cpp(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "keyset ok" in out.stdout
