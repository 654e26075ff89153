"""Schnorr signing with caller nonces (bjj_sign_schnorr_batch{,_dev}, bjj_multi_sign_schnorr_batch): the lane bodies on
the host and both flavours on the device against the oracle's sign_schnorr on the nonce, message and width edges;
consistency with fixed_base / public / scalar_key; round trips through verify_schnorr; chunk and sub-batch boundaries;
launch counts; argument errors and the Python / C++ mirrors."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

from common import KEY_KAT, MSG_KAT, ROOT, pack, unpack
from oracle import bjj_oracle as O

Q, L = O.Q, O.SUBORDER
ERR_ARG = 2
STATUS_MSG_RANGE = 4
WIDTHS = (8, 16, 32, 64)
LANES = 4096
BIG = (1 << 21) + 5

CPP_SRC = os.path.join(ROOT, "tests", "cpp", "test_sign_schnorr.cpp")
PKG = os.path.join(ROOT, "babyjubjub-rs_b200")


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def key_array(keys):
    return np.frombuffer(b"".join(keys), dtype=np.uint8).reshape(-1, 32).copy()


def nonce_array(ks, words):
    return np.frombuffer(b"".join(int(k).to_bytes(4 * words, "little") for k in ks), dtype=np.uint8).reshape(-1, 4 * words).copy()


def wide_ints(arr):
    raw = np.ascontiguousarray(arr, dtype=np.uint8)
    return [int.from_bytes(r.tobytes(), "little") for r in raw]


def edge_nonces(words):
    """0, 1, the SUBORDER and ORDER edges, test_gpu_parity's 2^1023 + 0xDEADBEEF, the all-ones nonce of the width and
    multiples of SUBORDER above 2^768 -- those that fit `words` words"""
    top = (1 << (32 * words)) - 1
    ks = [0, 1, L - 1, L, L + 1, O.ORDER, (1 << 1023) + 0xDEADBEEF, top,
          L * ((1 << 768) // L + 1), L * ((1 << 1000) // L + 12345), L * (top // L)]
    return [k for k in ks if k <= top]


EDGE_MSGS = [MSG_KAT, 0, Q - 1, Q, Q + 1, (1 << 256) - 1]


def edge_lanes(words, rnd):
    """(key, msg, nonce) lanes: every edge nonce with every edge message, the KAT key and random keys"""
    lanes = []
    for j, k in enumerate(edge_nonces(words)):
        for m in EDGE_MSGS:
            lanes.append((KEY_KAT if (j + len(lanes)) % 3 == 0 else rnd.randbytes(32), m, k))
    return lanes


def oracle_schnorr(lanes, words):
    """O.sign_schnorr lane by lane (the reference restated in Python) -> rx, ry, s (n, 4 * (words + 8)), status; a lane
    with msg > Q (the reference's Err) is all zeros with status 4"""
    rx, ry, s, st = [], [], [], []
    for key, m, k in lanes:
        if m > Q:
            with pytest.raises(ValueError, match="msg outside the Finite Field"):
                O.sign_schnorr(key, m, k)
            rx.append(0), ry.append(0), s.append(0), st.append(STATUS_MSG_RANGE)
            continue
        r, sv = O.sign_schnorr(key, m, k)
        rx.append(r[0]), ry.append(r[1]), s.append(sv), st.append(0)
    return pack(rx), pack(ry), nonce_array(s, words + 8), np.array(st, np.uint8)


def oracle_c_schnorr(oc, keys, msgs, nonces, words):
    """the same from the C oracle's fixed_base, public, scalar_key and Poseidon (r = (k mod SUBORDER) * B8: B8 has order
    SUBORDER; oracle_schnorr checks that reading on the edges) -- fast enough for thousands of lanes"""
    bad = [m > Q for m in msgs]
    rx, ry = oc.fixed_base(pack([0 if b else k % L for k, b in zip(nonces, bad)]))
    pkx, pky = oc.public(keys)
    sk = unpack(oc.scalar_key(keys))
    h = unpack(oc.poseidon([pkx, pky, rx, ry, pack([0 if b else m % Q for m, b in zip(msgs, bad)])]))
    s = [0 if b else k + x * hh for k, x, hh, b in zip(nonces, sk, h, bad)]
    badm = np.array(bad)
    rx[badm] = 0
    ry[badm] = 0
    return rx, ry, nonce_array(s, words + 8), np.where(badm, STATUS_MSG_RANGE, 0).astype(np.uint8)


def lanes_arrays(lanes, words):
    keys = key_array([k for k, _, _ in lanes])
    msgs = pack([min(m, (1 << 256) - 1) for _, m, _ in lanes])
    return keys, msgs, nonce_array([k for _, _, k in lanes], words)


# ---- CPU ----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def schnorr_emu(tmp_path_factory):
    """tests/hostemu/schnorr_emu.cpp (the Schnorr lane bodies compiled for the host), built into a temporary directory"""
    from common import build_hostemu
    build_hostemu()                     # generates the constants header the device sources include
    so = str(tmp_path_factory.mktemp("schnorr_emu") / "libbjj_schnorr_emu.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so,
                           os.path.join(ROOT, "tests", "hostemu", "schnorr_emu.cpp")])
    return ctypes.CDLL(so)


def emu_sign(emu, keys, msgs, nonces, words):
    n = len(keys)
    rx, ry = np.zeros((n, 32), np.uint8), np.zeros((n, 32), np.uint8)
    s = np.full((n, 4 * (words + 8)), 0xEE, np.uint8)
    st = np.full(n, 0xEE, np.uint8)
    emu.emu_sign_schnorr(ctypes.c_size_t(n), _p(keys), _p(msgs), _p(nonces), ctypes.c_int(words), _p(rx), _p(ry), _p(s), _p(st))
    return rx, ry, s, st


@pytest.mark.parametrize("words", WIDTHS)
def test_hostemu_nonce_reduction(schnorr_emu, words):
    """lane_mod_suborder_wide (Horner over 256-bit blocks with Montgomery products) is k mod SUBORDER"""
    rnd = random.Random(100 + words)
    ks = edge_nonces(words) + [rnd.getrandbits(32 * words) for _ in range(200)]
    out = np.zeros((len(ks), 32), np.uint8)
    schnorr_emu.emu_mod_suborder_wide(ctypes.c_size_t(len(ks)), _p(nonce_array(ks, words)), ctypes.c_int(words), _p(out))
    assert unpack(out) == [k % L for k in ks]


@pytest.mark.parametrize("words", WIDTHS)
def test_hostemu_sign_schnorr_edges(schnorr_emu, words):
    """the lane bodies in kernel order against O.sign_schnorr, byte for byte, s at full width"""
    rnd = random.Random(110 + words)
    lanes = edge_lanes(words, rnd) + [(rnd.randbytes(32), rnd.randrange(Q), rnd.getrandbits(32 * words)) for _ in range(8)]
    got = emu_sign(schnorr_emu, *lanes_arrays(lanes, words), words)
    want = oracle_schnorr(lanes, words)
    for g, w, what in zip(got, want, ("rx", "ry", "s", "status")):
        assert np.array_equal(g, w), (words, what, [i for i in range(len(lanes)) if not np.array_equal(g[i], w[i])][:5])
    assert STATUS_MSG_RANGE in want[3] and 0 in want[3]


def test_python_argument_handling():
    import babyjubjub_rs_b200 as bjj
    no_engine = object()                # every check below raises before any device work
    with pytest.raises(ValueError, match="negative nonce"):
        bjj.sign_schnorr_batch([KEY_KAT, KEY_KAT], [1, 2], [5, -5], engine=no_engine)
    with pytest.raises(ValueError, match="2048 bits"):
        bjj.sign_schnorr_batch([KEY_KAT], [1], [1 << 2048], engine=no_engine)
    with pytest.raises(ValueError, match="msg outside the Finite Field"):
        bjj.sign_schnorr_batch([KEY_KAT, KEY_KAT], [1, Q + 1], [5, 6], engine=no_engine)
    with pytest.raises(ValueError, match="negative msg"):
        bjj.sign_schnorr_batch([KEY_KAT], [-1], [5], engine=no_engine)
    with pytest.raises(ValueError, match="differ in length"):       # checked before the library is called
        bjj.Engine.sign_schnorr_batch(None, pack([1, 2]), pack([1]), nonce_array([1, 2], 8), 8)
    # the word count: the smallest multiple of 8 that holds the widest nonce
    for ks, words in (([0], 8), ([(1 << 256) - 1], 8), ([1 << 256], 16), ([3, (1 << 1023) + 0xDEADBEEF], 32),
                      ([(1 << 2048) - 1], 64)):
        arr, w = bjj._schnorr_nonces(ks)
        assert w == words and arr.shape == (len(ks), 4 * words) and wide_ints(arr) == ks


def build_cpp(out_dir):
    exe = os.path.join(str(out_dir), "test_sign_schnorr")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-pthread", "-o", exe, CPP_SRC, "-L" + PKG, "-lbjj_cuda",
                           "-Wl,-rpath," + PKG])
    return exe


def test_cpp_sign_schnorr_builds_and_links(tmp_path):
    assert os.path.exists(build_cpp(tmp_path))


# ---- GPU ----------------------------------------------------------------------------------------------
def call(lib, ctx, ins, words, outs, dev):
    """bjj_sign_schnorr_batch (host or _dev flavour) with host arrays ins = [keys, msgs, nonces]; fills outs = [rx, ry, s,
    status] and returns the return code"""
    n = len(ins[0])
    if not dev:
        return lib.bjj_sign_schnorr_batch(ctx, n, _p(ins[0]), _p(ins[1]), _p(ins[2]), words, *[_p(a) for a in outs])
    bufs = [lib.bjj_dev_alloc(ctx, max(a.nbytes, 1)) for a in ins + outs]
    try:
        assert all(bufs)
        for b, a in zip(bufs, ins):
            assert lib.bjj_memcpy_h2d(ctx, b, _p(a), a.nbytes) == 0
        rc = lib.bjj_sign_schnorr_batch_dev(ctx, n, bufs[0], bufs[1], bufs[2], words, *bufs[3:], None)
        for b, a in zip(bufs[len(ins):], outs):
            assert lib.bjj_memcpy_d2h(ctx, _p(a), b, a.nbytes) == 0
        assert lib.bjj_sync(ctx) == 0
    finally:
        for b in bufs:
            lib.bjj_dev_free(ctx, b)
    return rc


def sign(lib, ctx, keys, msgs, nonces, words, dev):
    n = len(keys)
    outs = [np.full((n, 32), 0xEE, np.uint8), np.full((n, 32), 0xEE, np.uint8), np.full((n, 4 * (words + 8)), 0xEE, np.uint8),
            np.full(n, 0xEE, np.uint8)]
    assert call(lib, ctx, [keys, msgs, nonces], words, outs, dev) == 0
    return outs


def random_lanes(rnd, n, words):
    keys = key_array([KEY_KAT] + [rnd.randbytes(32) for _ in range(n - 1)])
    ms = [rnd.randrange(Q) for _ in range(n)]
    for i in range(5, n, 16):
        ms[i] = rnd.randrange(Q + 1, 1 << 256)
    ms[0], ms[1] = MSG_KAT, Q
    ks = [rnd.getrandbits(32 * words) for _ in range(n)]
    return keys, ms, ks


@pytest.mark.gpu
def test_cpp_sign_schnorr_runs(tmp_path):
    out = subprocess.run([build_cpp(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "sign_schnorr ok" in out.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("words", WIDTHS)
def test_edges_against_oracle_both_flavours(gpu, words):
    lib, ctx = gpu.eng.lib, gpu.eng.ctx
    lanes = edge_lanes(words, random.Random(120 + words))
    arrs = lanes_arrays(lanes, words)
    want = oracle_schnorr(lanes, words)
    for dev in (False, True):
        got = sign(lib, ctx, *arrs, words, dev)
        for g, w, what in zip(got, want, ("rx", "ry", "s", "status")):
            assert np.array_equal(g, w), (dev, words, what)


@pytest.mark.gpu
def test_random_lanes_against_oracle_both_flavours(gpu, oracle_c):
    """4,096 lanes at nonce_words = 32 (the reference's 1024-bit nonce): all against the C oracle's composition, a sample
    against O.sign_schnorr; r equals fixed_base_batch on the reduced nonces, and s - k is scalar_key * h with pk from
    public_batch"""
    eng = gpu.eng
    lib, ctx = eng.lib, eng.ctx
    rnd = random.Random(130)
    keys, ms, ks = random_lanes(rnd, LANES, 32)
    msgs, nonces = pack(ms), nonce_array(ks, 32)
    want = oracle_c_schnorr(oracle_c, keys, ms, ks, 32)
    sample = [0, 1, 5] + rnd.sample(range(LANES), 40)
    ref = oracle_schnorr([(bytes(keys[i]), ms[i], ks[i]) for i in sample], 32)
    for w, r in zip(want, ref):
        assert np.array_equal(w[sample], r)
    for dev in (False, True):
        got = sign(lib, ctx, keys, msgs, nonces, 32, dev)
        for g, w, what in zip(got, want, ("rx", "ry", "s", "status")):
            assert np.array_equal(g, w), (dev, what)
    rx, ry, s, st = got
    good = st == 0
    assert (~good).sum() >= LANES // 20 and st[1] == 0
    fx, fy = eng.fixed_base_batch(pack([k % L for k in ks]))
    assert np.array_equal(rx[good], fx[good]) and np.array_equal(ry[good], fy[good])
    pkx, pky = eng.public_batch(keys)
    sk = unpack(eng.scalar_key_batch(keys))
    h = unpack(eng.poseidon_batch([pkx, pky, rx, ry, pack([m % Q if m <= Q else 0 for m in ms])]))
    sv = wide_ints(s)
    for i in np.flatnonzero(good):
        assert sv[i] == ks[i] + sk[i] * h[i], i


@pytest.mark.gpu
def test_round_trip_through_verify_schnorr(gpu):
    eng = gpu.eng
    rnd = random.Random(140)
    keys, ms, ks = random_lanes(rnd, LANES, 32)
    msgs = pack(ms)
    rx, ry, s, st = eng.sign_schnorr_batch(keys, msgs, nonce_array(ks, 32), 32)
    good = st == 0
    pkx, pky = eng.public_batch(keys)
    s_red = pack([v % L for v in wide_ints(s)])
    ok, vst = eng.verify_schnorr_batch(pkx[good], pky[good], msgs[good], rx[good], ry[good], s_red[good])
    assert ok.all() and not vst.any()
    msgs_bad = msgs[good].copy()
    msgs_bad[:, 0] ^= 1                                    # still below Q: a different message
    ok, vst = eng.verify_schnorr_batch(pkx[good], pky[good], msgs_bad, rx[good], ry[good], s_red[good])
    assert not ok.any() and not vst.any()
    s_bad = s.copy()
    s_bad[:, 1] ^= 0x10                                    # s + or - 2^12: a different group element
    s_bad = pack([v % L for v in wide_ints(s_bad)])
    ok, _ = eng.verify_schnorr_batch(pkx[good], pky[good], msgs[good], rx[good], ry[good], s_bad[good])
    assert not ok.any()


@pytest.mark.gpu
def test_chunk_and_subbatch_boundaries(gpu, oracle_c):
    """2^21 + 5 lanes at nonce_words = 32: the host flavour runs three chunks, _dev two sub-batches; host arrays
    pageable, page-locked and mixed; 7 launches per sub-batch, as sign_batch"""
    lib, ctx = gpu.eng.lib, gpu.eng.ctx
    words = 32
    rng = np.random.default_rng(150)
    keys = rng.integers(0, 256, size=(BIG, 32), dtype=np.uint8)
    keys[0] = key_array([KEY_KAT])[0]
    msgs = rng.integers(0, 256, size=(BIG, 32), dtype=np.uint8)
    msgs[:, 31] &= 0x2F                                    # < 0x30 * 2^248 < Q
    msgs[5::16, 31] = 0xFF                                 # > Q
    msgs[1] = pack([Q])[0]
    nonces = rng.integers(0, 256, size=(BIG, 4 * words), dtype=np.uint8)
    nonces[2] = 0
    nonces[3] = nonce_array([L], words)[0]
    rnd = random.Random(150)
    sample = sorted(set(rnd.sample(range(BIG), 2000)) |
                    {0, 1, 2, 3, 5, (1 << 18) - 1, 1 << 18, (1 << 20) - 1, 1 << 20, (1 << 21) - 1, 1 << 21, BIG - 1})
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

    try:
        for dev in (False, True):
            z = [np.zeros_like(keys) for _ in range(3)] + [np.zeros(BIG, np.uint8)]
            rc, n_sign = launches(lambda: call_sign(lib, ctx, keys, msgs, z, dev))
            assert rc == 0
            outs, n_schnorr = launches(lambda: sign(lib, ctx, keys, msgs, nonces, words, dev))
            assert n_schnorr == n_sign == (21 if not dev else 14), (dev, n_sign, n_schnorr)
            if dev:
                for a, b in zip(outs, host):
                    assert np.array_equal(a, b)
            else:
                host = outs
        # the host flavour from page-locked arrays, and from mixes of page-locked and pageable ones
        pk, pm, pn = pinned_like(keys), pinned_like(msgs), pinned_like(nonces)
        for k_in, m_in, n_in, pinned_out in ((pk, pm, pn, True), (pk, msgs, pn, False), (keys, pm, nonces, True)):
            outs = [np.zeros_like(a) for a in host]
            if pinned_out:
                outs[0], outs[2] = pinned_like(outs[0]), pinned_like(outs[2])
            assert call(lib, ctx, [k_in, m_in, n_in], words, outs, False) == 0
            for a, b in zip(outs, host):
                assert np.array_equal(a, b)
    finally:
        for ptr in pinned:
            lib.bjj_host_free(ptr)
    ms = unpack(msgs[sample])
    ks = wide_ints(nonces[sample])
    want = oracle_c_schnorr(oracle_c, keys[sample], ms, ks, words)
    for g, w in zip(host, want):
        assert np.array_equal(g[sample], w)
    edge = [0, 1, 2, 3, 5, (1 << 21) - 1, 1 << 21, BIG - 1]
    ref = oracle_schnorr([(bytes(keys[i]), unpack(msgs[i:i + 1])[0], wide_ints(nonces[i:i + 1])[0]) for i in edge], words)
    for g, r in zip(host, ref):
        assert np.array_equal(g[edge], r)
    assert host[3][1] == 0 and host[3][5] == STATUS_MSG_RANGE
    assert unpack(host[0][2:4]) == [0, 0] and unpack(host[1][2:4]) == [1, 1]        # k = 0 and k = SUBORDER: r = (0, 1)


def call_sign(lib, ctx, keys, msgs, outs, dev):
    """bjj_sign_batch (host or _dev flavour), the yardstick of the launch count"""
    if not dev:
        return lib.bjj_sign_batch(ctx, len(keys), _p(keys), _p(msgs), *[_p(a) for a in outs])
    ins = [keys, msgs]
    bufs = [lib.bjj_dev_alloc(ctx, max(a.nbytes, 1)) for a in ins + outs]
    try:
        assert all(bufs)
        for b, a in zip(bufs, ins):
            assert lib.bjj_memcpy_h2d(ctx, b, _p(a), a.nbytes) == 0
        rc = lib.bjj_sign_batch_dev(ctx, len(keys), *bufs, None)
        assert lib.bjj_sync(ctx) == 0
    finally:
        for b in bufs:
            lib.bjj_dev_free(ctx, b)
    return rc


@pytest.mark.gpu
def test_multi_engine_matches_single_engine(gpu):
    import babyjubjub_rs_b200 as bjj
    eng = gpu.eng
    ndev = eng.lib.bjj_device_count()
    rnd = random.Random(160)
    n = 3 * 4096 + 7                                       # not divisible by 2, 4, 8 devices
    keys, ms, ks = random_lanes(rnd, n, 32)
    msgs, nonces = pack(ms), nonce_array(ks, 32)
    want = eng.sign_schnorr_batch(keys, msgs, nonces, 32)
    for devices in sorted({(0,), tuple(range(ndev))}):
        me = bjj.MultiEngine(list(devices))
        try:
            got = me.sign_schnorr_batch(keys, msgs, nonces, 32)
            for g, w in zip(got, want):
                assert np.array_equal(g, w), devices
            out = tuple(np.zeros_like(w) for w in want)
            assert me.sign_schnorr_batch(keys, msgs, nonces, 32, out=out)[2] is out[2]
            for g, w in zip(out, want):
                assert np.array_equal(g, w), devices
            me.set_host_register(True)
            got = me.sign_schnorr_batch(keys[:4097], msgs[:4097], nonces[:4097], 32)
            for g, w in zip(got, want):
                assert np.array_equal(g, w[:4097]), devices
        finally:
            me.close()


@pytest.mark.gpu
def test_arguments(gpu):
    import babyjubjub_rs_b200 as bjj
    lib, ctx = gpu.eng.lib, gpu.eng.ctx
    k, m, kn = pack([1] * 64), pack([2] * 64), nonce_array([3] * 64, 64)
    rx, ry, s, st = np.zeros((64, 32), np.uint8), np.zeros((64, 32), np.uint8), np.zeros((64, 4 * 72), np.uint8), np.zeros(64, np.uint8)

    def args(words, null=None):
        a = [_p(k), _p(m), _p(kn), words, _p(rx), _p(ry), _p(s), _p(st)]
        if null is not None:
            a[null] = None
        return a
    me = bjj.MultiEngine([0])
    try:
        fns = [(lambda *a: lib.bjj_sign_schnorr_batch(ctx, 64, *a)), (lambda *a: lib.bjj_sign_schnorr_batch_dev(ctx, 64, *a, None)),
               (lambda *a: lib.bjj_multi_sign_schnorr_batch(me.handle, 64, *a))]
        for fn in fns:
            for words in (0, 7, 72, -8):
                assert fn(*args(words)) == ERR_ARG, words
            for null in (0, 1, 2, 4, 5, 6, 7):
                assert fn(*args(8, null)) == ERR_ARG, null
        assert lib.bjj_sign_schnorr_batch(None, 64, *args(8)) == ERR_ARG
        assert lib.bjj_sign_schnorr_batch_dev(None, 64, *args(8), None) == ERR_ARG
        assert lib.bjj_multi_sign_schnorr_batch(None, 64, *args(8)) == ERR_ARG
        assert lib.bjj_sign_schnorr_batch(ctx, 0, *args(8)) == 0
        assert lib.bjj_sign_schnorr_batch_dev(ctx, 0, *args(8), None) == 0
        assert lib.bjj_multi_sign_schnorr_batch(me.handle, 0, *args(8)) == 0
    finally:
        me.close()


@pytest.mark.gpu
def test_python_mirror(gpu):
    import babyjubjub_rs_b200 as bjj
    rnd = random.Random(170)
    keys = [KEY_KAT, bytes(32), b"\xff" * 32] + [rnd.randbytes(32) for _ in range(5)]
    msgs = [MSG_KAT, Q, 0, Q - 1, 5, rnd.randrange(Q), rnd.randrange(Q), 12345]
    nonces = [0, L, (1 << 1023) + 0xDEADBEEF, 1 << 1500, 7, rnd.getrandbits(1024), rnd.getrandbits(300), L * (1 << 800)]
    got = bjj.sign_schnorr_batch(keys, msgs, nonces, engine=gpu.eng)
    for key, msg, k, (r, s) in zip(keys, msgs, nonces, got):
        want_r, want_s = O.sign_schnorr(key, msg, k)
        assert (r.x, r.y) == want_r and s == want_s
    got = bjj.sign_schnorr_batch([bjj.PrivateKey(KEY_KAT)] * 3, [1, 2, 3], engine=gpu.eng)      # random 1024-bit nonces
    pk = O.public(KEY_KAT)
    for msg, (r, s) in zip([1, 2, 3], got):
        assert O.verify_schnorr(pk, msg, (r.x, r.y), s)
        k = s - O.scalar_key(KEY_KAT) * O.schnorr_hash(pk, msg, (r.x, r.y))
        assert 0 <= k < (1 << 1024) and O.sign_schnorr(KEY_KAT, msg, k) == ((r.x, r.y), s)
    assert bjj.sign_schnorr_batch([], [], [], engine=gpu.eng) == []
