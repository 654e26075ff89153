"""verify against one key with a comb table (bjj_verify_base_batch, bjj_verify_base_compressed_batch): the lane bodies
compiled for the host against the oracle, both flavours on the GPU against the oracle and byte for byte against
bjj_verify_batch / bjj_verify_compressed_batch with the key in every lane, chunk and sub-batch boundaries, launch
counts, a non-canonical R8, argument errors, a workspace shared with verify_batch's deferred exact lanes, and the
Python / C++ mirrors."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

from common import KEY_KAT, MSG_KAT, ROOT, pack, unpack
from oracle import bjj_oracle as O

Q, ORDER, SUBORDER = O.Q, O.ORDER, O.SUBORDER
ERR_ARG, ERR_NONCANONICAL = 2, 3
STATUS = {O.ERR_Y_RANGE: 1, O.ERR_NO_INV: 2, O.ERR_NOT_SQUARE: 3}
LANES = 4096
BIG = (1 << 21) + 5
IDENTITY = (0, 1)

CPP_SRC = os.path.join(ROOT, "tests", "cpp", "test_verify_base.cpp")
PKG = os.path.join(ROOT, "babyjubjub-rs_b200")


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def add(p, q):
    return O.proj_affine(O.proj_add(p + (1,), q + (1,)))


def torsion_points():
    """points of order 2, 4 and 8: SUBORDER * P for on-curve P outside the prime-order subgroup"""
    t2 = (0, Q - 1)
    x4 = O.modsqrt(pow(O.A, Q - 2, Q), Q)
    t4 = (x4, 0)
    y = 2
    while True:
        y += 1
        try:
            p = O.decompress_point(y.to_bytes(32, "little"))
        except ValueError:
            continue
        t = O.mul_scalar(p, SUBORDER)
        if O.mul_scalar(t, 4) != IDENTITY:
            return t2, t4, t


def keys_with_secrets():
    """(name, A, a) with A = a*B8 + (torsion): the key kinds verify_base must serve"""
    t2, t4, t8 = torsion_points()
    a = O.scalar_key(KEY_KAT)
    b = 0x1234567890ABCDEF1234567890ABCDEF
    return [("identity", IDENTITY, 0), ("order2", t2, 0), ("order8", t8, 0), ("full_order", add(O.mul_scalar(O.B8, b), t8), b),
            ("b8", O.B8, 1), ("public", O.public(KEY_KAT), a)]


def make_sig(A, a, r, msg):
    """(R8, S) with R8 = r*B8 and S = r + 8*hm*a mod SUBORDER: valid for A = a*B8 + T (8*T = O)"""
    r8 = O.mul_scalar(O.B8, r)
    hm = O.poseidon([r8[0], r8[1], A[0], A[1], msg % Q])
    return r8, (r + 8 * hm * a) % SUBORDER, msg


def edge_cases(rnd, A, a):
    """list of (R8, S, msg) for key A: valid signatures, corruptions, message, S and R8 edges"""
    t2, t4, t8 = torsion_points()
    cases = [make_sig(A, a, rnd.randrange(1, SUBORDER), rnd.randrange(Q)) for _ in range(3)]
    r8, s, m = cases[0]
    other = make_sig(A, a, rnd.randrange(1, SUBORDER), m)[0]
    cases += [(r8, s ^ 1, m), (r8, (s + SUBORDER) & ((1 << 256) - 1), m), (r8, s + 37 * SUBORDER, m), (other, s, m),
              (r8, s, m ^ 2)]
    cases += [make_sig(A, a, 5, Q), make_sig(A, a, 6, 0)]               # msg == Q is hashed as 0
    cases += [(r8, s, Q + 1), (r8, s, (1 << 256) - 1)]                  # msg > Q: false
    for sv in (0, SUBORDER, ORDER, (1 << 256) - 1):                     # S edges, R8 = S*B8 (valid for small-order A)
        cases.append((O.mul_scalar(O.B8, sv), sv, rnd.randrange(Q)))
    cases.append((IDENTITY, 0, 77))
    for off in ((0, 0), (1, 1), (Q - 1, Q - 1), ((r8[0] + 1) % Q, r8[1]), (r8[0], (r8[1] + 1) % Q), (5, 7)):
        cases.append((off, s, m))                                       # R8 off the curve
        cases.append((off, 0, m))
    for t in (t2, t4, t8):                                              # R8 with a torsion component
        rt = add(r8, t)
        cases.append((rt, s, m))
        hm = O.poseidon([rt[0], rt[1], A[0], A[1], m])
        cases.append((rt, (rnd.randrange(1, SUBORDER) + 8 * hm * a) % SUBORDER, m))
    return cases


def oracle_ok(A, cases):
    return np.array([int(O.verify(A, (r8, s), m)) for r8, s, m in cases], np.uint8)


def case_arrays(cases):
    mask = (1 << 256) - 1
    return [pack([c[0][0] for c in cases]), pack([c[0][1] for c in cases]), pack([c[1] & mask for c in cases]),
            pack([min(c[2], mask) for c in cases])]


def compressed_cases(rnd, A, a):
    """64-byte signatures (from the on-curve cases) plus undecompressable R8, and the oracle's (ok, status)"""
    sigs, msgs, want_ok, want_st = [], [], [], []
    for r8, s, m in edge_cases(rnd, A, a):
        if not O.on_curve(r8):
            continue
        sigs.append(O.compress_signature((r8, s)))
        msgs.append(m)
    good = sigs[0]
    ys = [b"\xff" * 31 + b"\x7f", (Q).to_bytes(32, "little")]           # y >= Q
    y = 3
    while len(ys) < 5:                                                  # not a square
        y += 1
        try:
            O.decompress_point(y.to_bytes(32, "little"))
        except ValueError as e:
            if str(e) == O.ERR_NOT_SQUARE:
                ys.append(y.to_bytes(32, "little"))
    for yb in ys:
        sigs.append(yb + good[32:])
        msgs.append(msgs[0])
    for sig, m in zip(sigs, msgs):
        try:
            r8, s = O.decompress_signature(sig)
        except ValueError as e:
            want_ok.append(0)
            want_st.append(STATUS[str(e)])
            continue
        want_ok.append(int(O.verify(A, (r8, s), m)))
        want_st.append(0)
    sig64 = np.frombuffer(b"".join(sigs), np.uint8).reshape(-1, 64).copy()
    return sig64, pack([min(m, (1 << 256) - 1) for m in msgs]), np.array(want_ok, np.uint8), np.array(want_st, np.uint8)


# ---- CPU ----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def verify_base_emu(tmp_path_factory):
    """tests/hostemu/verify_base_emu.cpp (the verify_base lane bodies compiled for the host), built into a temporary
    directory"""
    from common import build_hostemu
    build_hostemu()                     # generates the constants header the device sources include
    so = str(tmp_path_factory.mktemp("verify_base_emu") / "libbjj_verify_base_emu.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so,
                           os.path.join(ROOT, "tests", "hostemu", "verify_base_emu.cpp")])
    lib = ctypes.CDLL(so)
    lib.emu_verify_base.restype = ctypes.c_uint32
    return lib


def test_hostemu_scalar_reduction(verify_base_emu):
    """k = 8*hm mod ORDER for hm across [0, Q)"""
    rnd = random.Random(40)
    hms = [0, 1, 2, SUBORDER - 1, SUBORDER, SUBORDER + 1, ORDER // 8 * 7, Q - 1, Q - 2, (1 << 253) - 1, 1 << 253]
    hms += [rnd.randrange(Q) for _ in range(200)]
    out = np.zeros((len(hms), 32), np.uint8)
    verify_base_emu.emu_verify_base_scalar(ctypes.c_size_t(len(hms)), _p(pack(hms)), _p(out))
    assert unpack(out) == [8 * h % ORDER for h in hms]


@pytest.mark.parametrize("key", [k[0] for k in keys_with_secrets()])
def test_hostemu_against_oracle(verify_base_emu, key):
    """the two lane bodies (device source compiled for the host) against the oracle's verify, for every key kind"""
    name, A, a = next(k for k in keys_with_secrets() if k[0] == key)
    rnd = random.Random(sum(name.encode()))
    cases = edge_cases(rnd, A, a)
    want = oracle_ok(A, cases)
    assert want[:3].all() and want.sum() >= 4          # the valid signatures verify
    ins = case_arrays(cases)
    ok = np.full(len(cases), 0xEE, np.uint8)
    flags = verify_base_emu.emu_verify_base(ctypes.c_size_t(len(cases)), _p(pack([A[0]])), _p(pack([A[1]])), *[_p(v) for v in ins],
                                            _p(ok))
    assert flags == 0
    assert list(ok) == list(want), [i for i in range(len(cases)) if ok[i] != want[i]]


@pytest.mark.parametrize("key", ["order8", "public"])
def test_hostemu_compressed_against_oracle(verify_base_emu, key):
    """R8's decompression phases and the two lane bodies against decompress_signature + verify"""
    name, A, a = next(k for k in keys_with_secrets() if k[0] == key)
    sig64, msgs, want_ok, want_st = compressed_cases(random.Random(41), A, a)
    assert set(want_st) == {0, 1, 3}
    ok, st = np.full(len(sig64), 0xEE, np.uint8), np.full(len(sig64), 0xEE, np.uint8)
    verify_base_emu.emu_verify_base_compressed(ctypes.c_size_t(len(sig64)), _p(pack([A[0]])), _p(pack([A[1]])), _p(sig64), _p(msgs),
                                               _p(ok), _p(st))
    assert list(st) == list(want_st)
    assert list(ok) == list(want_ok)


def test_python_message_handling():
    import babyjubjub_rs_b200 as bjj
    assert unpack(bjj._verify_msgs([0, 5, Q, Q + 1, (1 << 256) - 1, 1 << 256, 7 << 300])) == [0, 5, Q] + [(1 << 256) - 1] * 4
    with pytest.raises(ValueError, match="FixedBase"):
        bjj._key_handle(None)                           # a verify names its key: None does not select B8


def build_cpp(out_dir):
    exe = os.path.join(str(out_dir), "test_verify_base")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-pthread", "-o", exe, CPP_SRC, "-L" + PKG, "-lbjj_cuda",
                           "-Wl,-rpath," + PKG])
    return exe


def test_cpp_verify_base_builds_and_links(tmp_path):
    assert os.path.exists(build_cpp(tmp_path))


# ---- GPU ----------------------------------------------------------------------------------------------
def call(lib, ctx, name, base, ins, outs, dev, sync_rc=0):
    """bjj_<name>_batch (host or _dev flavour) against `base` with host arrays `ins`; fills `outs`, returns the rc"""
    n = len(ins[0])
    fn = getattr(lib, "bjj_%s_batch%s" % (name, "_dev" if dev else ""))
    if not dev:
        return fn(ctx, base, n, *[_p(a) for a in ins + outs])
    bufs = [lib.bjj_dev_alloc(ctx, max(a.nbytes, 1)) for a in ins + outs]
    try:
        assert all(bufs)
        for b, a in zip(bufs, ins):
            assert lib.bjj_memcpy_h2d(ctx, b, _p(a), a.nbytes) == 0
        rc = fn(ctx, base, n, *bufs, None)
        for b, a in zip(bufs[len(ins):], outs):
            assert lib.bjj_memcpy_d2h(ctx, _p(a), b, a.nbytes) == 0
        assert lib.bjj_sync(ctx) == sync_rc
    finally:
        for b in bufs:
            lib.bjj_dev_free(ctx, b)
    return rc


def verify_plain(lib, ctx, base, ins, dev):
    ok = np.full(len(ins[0]), 0xEE, np.uint8)
    assert call(lib, ctx, "verify_base", base, ins, [ok], dev) == 0
    return ok


def verify_packed(lib, ctx, base, sig64, msgs, dev):
    ok, st = np.full(len(sig64), 0xEE, np.uint8), np.full(len(sig64), 0xEE, np.uint8)
    assert call(lib, ctx, "verify_base_compressed", base, [sig64, msgs], [ok, st], dev) == 0
    return ok, st


def signed_batch(eng, n, seed, corrupt=0.1, off_curve=0.01):
    """n signatures of one key made on the device, with about `corrupt` of the lanes corrupted (S, R8 or msg) and about
    `off_curve` of them given an off-curve R8; -> key, (r8x, r8y, s, msg), pk (ax, ay)"""
    rng = np.random.default_rng(seed)
    key = rng.integers(0, 256, size=32, dtype=np.uint8)
    keys = np.tile(key, (n, 1))
    msgs = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    msgs[:, 31] &= 0x2F                                    # < Q
    r8x, r8y, s, st = eng.sign_batch(keys, msgs)
    assert not st.any()
    ax, ay = eng.public_batch(keys[:1])
    lanes = rng.permutation(n)
    nc = int(n * corrupt)

    def flip_x(i, bit):
        """R8.x of lane i with one bit flipped, kept below Q: the inputs stay canonical (x >= Q is its own case, see
        test_noncanonical_r8)"""
        x = int.from_bytes(r8x[i].tobytes(), "little") ^ (1 << bit)
        r8x[i] = np.frombuffer((x if x < Q else x - Q).to_bytes(32, "little"), np.uint8)
    for j, i in enumerate(lanes[:nc]):
        if j % 3 == 1:
            flip_x(i, int(rng.integers(0, 248)))
        else:                                              # S: any 256-bit value; msg: byte 31 untouched, stays < Q
            [s, msgs][j % 3 // 2][i, rng.integers(0, 31)] ^= 1 << int(rng.integers(0, 8))
    for i in lanes[nc:nc + int(n * off_curve)]:
        flip_x(i, 0)                                       # off the curve (almost surely)
    assert all(v < Q for v in unpack(r8x)) and all(v < Q for v in unpack(msgs))
    return key, [r8x, r8y, s, msgs], (ax, ay)


def fixed_base(bjj, eng, ax, ay):
    return bjj.FixedBase((unpack(ax)[0], unpack(ay)[0]), eng)


@pytest.mark.gpu
def test_against_oracle_both_flavours(gpu, oracle_c):
    """4,096 lanes of one key (10 % corrupted, some off-curve R8) plus the edge cases, both flavours"""
    bjj, eng = gpu.bjj, gpu.eng
    lib, ctx = eng.lib, eng.ctx
    _, ins, (ax, ay) = signed_batch(eng, LANES, 42)
    want = oracle_c.verify(*ins[:3], np.repeat(ax, LANES, 0), np.repeat(ay, LANES, 0), ins[3])
    assert 0.85 * LANES < want.sum() < 0.95 * LANES
    base = fixed_base(bjj, eng, ax, ay)
    try:
        for dev in (False, True):
            assert np.array_equal(verify_plain(lib, ctx, base.handle, ins, dev), want), dev
    finally:
        base.close()
    # every key kind with its edge cases, both flavours, against the Python oracle
    for name, A, a in keys_with_secrets():
        cases = edge_cases(random.Random(43), A, a)
        want = oracle_ok(A, cases)
        base = bjj.FixedBase(A, eng)
        try:
            for dev in (False, True):
                assert np.array_equal(verify_plain(lib, ctx, base.handle, case_arrays(cases), dev), want), (name, dev)
            sig64, msgs, want_ok, want_st = compressed_cases(random.Random(44), A, a)
            for dev in (False, True):
                ok, st = verify_packed(lib, ctx, base.handle, sig64, msgs, dev)
                assert np.array_equal(st, want_st) and np.array_equal(ok, want_ok), (name, dev)
        finally:
            base.close()


@pytest.mark.gpu
def test_equal_to_verify_batch(gpu):
    """2^16 mixed lanes: ok byte-equal to bjj_verify_batch with A broadcast, and the compressed form byte-equal (ok and
    status) to bjj_verify_compressed_batch with pk32 broadcast, undecompressable R8 included"""
    bjj, eng = gpu.bjj, gpu.eng
    n = 1 << 16
    _, ins, (ax, ay) = signed_batch(eng, n, 45, off_curve=0.02)
    want = eng.verify_batch(*ins[:3], np.repeat(ax, n, 0), np.repeat(ay, n, 0), ins[3])
    assert 0 < want.sum() < n
    base = fixed_base(bjj, eng, ax, ay)
    try:
        assert np.array_equal(eng.verify_base_batch(base, *ins), want)
        sig64 = np.concatenate([eng.compress_batch(ins[0], ins[1]), ins[2]], axis=1)
        rng = np.random.default_rng(45)
        bad = rng.choice(n, n // 50, replace=False)
        sig64[bad[: len(bad) // 2], 31] |= 0x7F            # y >= Q
        sig64[bad[len(bad) // 2:], 0] ^= 0x5A              # mostly not a square
        pk32 = np.repeat(eng.compress_batch(ax, ay), n, 0)
        want_ok, want_st = eng.verify_compressed_batch(sig64, pk32, ins[3])
        assert set(np.unique(want_st)) >= {0, 1, 3}
        ok, st = eng.verify_base_compressed_batch(base, sig64, ins[3])
        assert np.array_equal(st, want_st) and np.array_equal(ok, want_ok)
    finally:
        base.close()


@pytest.mark.gpu
def test_chunk_and_subbatch_boundaries(gpu, oracle_c):
    """2^21 + 5 lanes: the host flavour runs three chunks, _dev two sub-batches; host arrays pageable, page-locked and
    mixed; launches per sub-batch 2 (plain) and 5 (compressed), also at 1,000 lanes; sampled lanes against the oracle"""
    bjj, eng = gpu.bjj, gpu.eng
    lib, ctx = eng.lib, eng.ctx
    _, ins, (ax, ay) = signed_batch(eng, BIG, 46)
    sig64 = np.concatenate([eng.compress_batch(ins[0], ins[1]), ins[2]], axis=1)
    sig64[7::97, 31] |= 0x7F                               # y >= Q
    rnd = random.Random(46)
    sample = sorted(set(rnd.sample(range(BIG), 3000)) | {0, 1, 2, 5, (1 << 18) - 1, 1 << 18, (1 << 21) - 1, 1 << 21, BIG - 1})
    pinned = []

    def pinned_like(a):
        ptr = lib.bjj_host_alloc(a.nbytes)
        assert ptr
        pinned.append(ptr)
        v = np.frombuffer((ctypes.c_uint8 * a.nbytes).from_address(ptr), dtype=np.uint8).reshape(a.shape)
        v[...] = a
        return v

    def launches(fn):
        before = lib.bjj_kernel_launches(ctx)
        r = fn()
        return r, lib.bjj_kernel_launches(ctx) - before

    base = fixed_base(bjj, eng, ax, ay)
    h = base.handle
    try:
        for dev in (False, True):
            small = [a[:1000] for a in ins]
            _, k = launches(lambda: verify_plain(lib, ctx, h, small, dev))
            assert k == 2, (dev, k)
            _, k = launches(lambda: verify_packed(lib, ctx, h, sig64[:1000], ins[3][:1000], dev))
            assert k == 5, (dev, k)
            ok, k = launches(lambda: verify_plain(lib, ctx, h, ins, dev))
            assert k == (6 if not dev else 4), (dev, k)
            (cok, cst), k = launches(lambda: verify_packed(lib, ctx, h, sig64, ins[3], dev))
            assert k == (15 if not dev else 10), (dev, k)
            if dev:
                assert np.array_equal(ok, ok_host) and np.array_equal(cok, cok_host) and np.array_equal(cst, cst_host)
            else:
                ok_host, cok_host, cst_host = ok, cok, cst
        pins = [pinned_like(a) for a in ins]
        psig = pinned_like(sig64)
        for mix in ((True,) * 4, (True, False, True, False), (False, True, False, True)):
            src = [p if m else a for p, a, m in zip(pins, ins, mix)]
            ok = pinned_like(np.zeros(BIG, np.uint8)) if mix[0] else np.zeros(BIG, np.uint8)
            assert call(lib, ctx, "verify_base", h, src, [ok], False) == 0
            assert np.array_equal(ok, ok_host), mix
            ok, st = np.zeros(BIG, np.uint8), (pinned_like(np.zeros(BIG, np.uint8)) if mix[1] else np.zeros(BIG, np.uint8))
            assert call(lib, ctx, "verify_base_compressed", h, [psig if mix[0] else sig64, src[3]], [ok, st], False) == 0
            assert np.array_equal(ok, cok_host) and np.array_equal(st, cst_host), mix
    finally:
        base.close()
        for ptr in pinned:
            lib.bjj_host_free(ptr)
    s_ins = [a[sample] for a in ins]
    want = oracle_c.verify(*s_ins[:3], np.repeat(ax, len(sample), 0), np.repeat(ay, len(sample), 0), s_ins[3])
    assert np.array_equal(ok_host[sample], want)
    want_ok, want_st = oracle_c.verify_compressed(sig64[sample], np.repeat(eng.compress_batch(ax, ay), len(sample), 0), s_ins[3])
    assert np.array_equal(cst_host[sample], want_st) and np.array_equal(cok_host[sample], want_ok)
    assert cst_host[7] == 1


@pytest.mark.gpu
def test_noncanonical_r8(gpu):
    """a coordinate of R8 >= Q: BJJ_ERR_NONCANONICAL and the ok[] of bjj_verify_batch (the batch computed mod Q)"""
    bjj, eng = gpu.bjj, gpu.eng
    lib, ctx = eng.lib, eng.ctx
    n = 256
    _, ins, (ax, ay) = signed_batch(eng, n, 47)
    xs = unpack(ins[0])
    for i in (3, 4):
        ins[0][i] = pack([xs[i] + Q])[0] if xs[i] + Q < (1 << 256) else ins[0][i]
    assert any(unpack(ins[0])[i] >= Q for i in (3, 4))
    want = np.zeros(n, np.uint8)
    assert lib.bjj_verify_batch(ctx, n, *[_p(a) for a in ins[:3]], _p(np.repeat(ax, n, 0)), _p(np.repeat(ay, n, 0)), _p(ins[3]),
                                _p(want)) == ERR_NONCANONICAL
    base = fixed_base(bjj, eng, ax, ay)
    try:
        ok = np.zeros(n, np.uint8)
        assert call(lib, ctx, "verify_base", base.handle, ins, [ok], False) == ERR_NONCANONICAL
        assert np.array_equal(ok, want)
        ok = np.zeros(n, np.uint8)
        assert call(lib, ctx, "verify_base", base.handle, ins, [ok], True, sync_rc=ERR_NONCANONICAL) == 0
        assert np.array_equal(ok, want)
    finally:
        base.close()


@pytest.mark.gpu
def test_arguments(gpu):
    """a NULL base, a base of another context, NULL arrays and n = 0"""
    bjj, eng = gpu.bjj, gpu.eng
    lib, ctx = eng.lib, eng.ctx
    a32, m, o = pack([1] * 64), pack([2] * 64), np.zeros(64, np.uint8)
    s64 = np.zeros((64, 64), np.uint8)
    base = bjj.FixedBase(O.B8, eng)
    other = bjj.Engine(0)
    foreign = bjj.FixedBase(O.B8, other)
    try:
        for dev in (False, True):
            sfx = "_dev" if dev else ""
            plain, packed = getattr(lib, "bjj_verify_base_batch" + sfx), getattr(lib, "bjj_verify_base_compressed_batch" + sfx)
            tail = (None,) if dev else ()
            args_p = [_p(a32), _p(a32), _p(a32), _p(m), _p(o)]
            args_c = [_p(s64), _p(m), _p(o), _p(o)]
            assert plain(ctx, base.handle, 0, *args_p, *tail) == 0
            assert packed(ctx, base.handle, 0, *args_c, *tail) == 0
            for h in (None, foreign.handle):
                assert plain(ctx, h, 64, *args_p, *tail) == ERR_ARG
                assert packed(ctx, h, 64, *args_c, *tail) == ERR_ARG
                assert plain(ctx, h, 0, *args_p, *tail) == ERR_ARG
            assert plain(None, base.handle, 64, *args_p, *tail) == ERR_ARG
            for i in range(5):
                args = list(args_p)
                args[i] = None
                assert plain(ctx, base.handle, 64, *args, *tail) == ERR_ARG, (dev, i)
            for i in range(4):
                args = list(args_c)
                args[i] = None
                assert packed(ctx, base.handle, 64, *args, *tail) == ERR_ARG, (dev, i)
        with pytest.raises(ValueError):
            eng.verify_base_batch(None, a32, a32, a32, m)
    finally:
        base.close()
        foreign.close()
        other.close()


@pytest.mark.gpu
def test_after_verify_batch_with_exact_lanes(gpu):
    """verify_batch with many off-curve lanes (its exact kernel runs deferred on the workspace's side stream), then at
    once verify_base_batch on the same context: both correct, in both flavours"""
    bjj, eng = gpu.bjj, gpu.eng
    lib, ctx = eng.lib, eng.ctx
    n = (1 << 20) + 3
    _, ins, (ax, ay) = signed_batch(eng, n, 48, off_curve=0.05)
    axn, ayn = np.repeat(ax, n, 0), np.repeat(ay, n, 0)
    base = fixed_base(bjj, eng, ax, ay)
    try:
        first = eng.verify_batch(*ins[:3], axn, ayn, ins[3])
        second = eng.verify_base_batch(base, *ins)
        assert np.array_equal(first, second)
        want = eng.verify_base_batch(base, *ins)
        # _dev: both calls enqueued on the context stream without a synchronisation between them
        bufs = [lib.bjj_dev_alloc(ctx, a.nbytes) for a in ins + [axn, ayn]]
        okv, okb = lib.bjj_dev_alloc(ctx, n), lib.bjj_dev_alloc(ctx, n)
        try:
            for b, a in zip(bufs, ins + [axn, ayn]):
                assert lib.bjj_memcpy_h2d(ctx, b, _p(a), a.nbytes) == 0
            r8x, r8y, s, msg, dax, day = bufs
            assert lib.bjj_verify_batch_dev(ctx, n, r8x, r8y, s, dax, day, msg, okv, None) == 0
            assert lib.bjj_verify_base_batch_dev(ctx, base.handle, n, r8x, r8y, s, msg, okb, None) == 0
            got_v, got_b = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
            assert lib.bjj_memcpy_d2h(ctx, _p(got_v), okv, n) == 0
            assert lib.bjj_memcpy_d2h(ctx, _p(got_b), okb, n) == 0
            assert lib.bjj_sync(ctx) == 0
        finally:
            for b in bufs + [okv, okb]:
                lib.bjj_dev_free(ctx, b)
        assert np.array_equal(got_v, want) and np.array_equal(got_b, want)
    finally:
        base.close()


@pytest.mark.gpu
def test_python_and_cpp_mirrors(gpu, tmp_path):
    bjj, eng = gpu.bjj, gpu.eng
    pk = bjj.Point(*O.public(KEY_KAT))
    msgs = [MSG_KAT, 0, Q, Q + 1, 1 << 256, 12345]
    sigs = []
    for msg in msgs:
        r8, s = O.sign(KEY_KAT, msg if msg <= Q else MSG_KAT)
        sigs.append(bjj.Signature(bjj.Point(*r8), s))
    sigs[5] = bjj.Signature(sigs[5].r_b8, sigs[5].s ^ 1)
    base = bjj.FixedBase(pk, eng)
    try:
        got = bjj.verify_base_batch(base, sigs, msgs)
        assert got == [True, True, True, False, False, False]
        assert got == bjj.verify_batch([pk] * len(sigs), sigs, msgs, engine=eng)
        assert bjj.verify_base_batch(base, [], []) == []
    finally:
        base.close()
    out = subprocess.run([build_cpp(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "verify base ok" in out.stdout
