"""Compressed outputs of key generation and signing (bjj_public_compressed_batch, bjj_sign_compressed_batch and their
bjj_multi wrappers): both flavours against the oracle, against the composition of the uncompressed calls with
compress, round trips through decompress / verify_compressed, chunk and sub-batch boundaries, launch counts, the
environment switches, argument errors and the Python / C++ mirrors."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

from common import KEY_KAT, MSG_KAT, ROOT, pack, unpack
from oracle import bjj_oracle as O

Q = O.Q
ERR_ARG = 2
STATUS_MSG_RANGE = 4
LANES = 4096
BIG = (1 << 21) + 5

CPP_SRC = os.path.join(ROOT, "tests", "cpp", "test_compressed.cpp")
CPP_EXE = os.path.join(ROOT, "tests", "cpp", "test_compressed")
PKG = os.path.join(ROOT, "babyjubjub-rs_b200")


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def key_array(keys):
    return np.frombuffer(b"".join(keys), dtype=np.uint8).reshape(-1, 32).copy()


def edge_keys(rnd, n):
    """the circomlib key of the reference's test vectors, all-zero, all-0xff, then random keys"""
    return key_array([KEY_KAT, bytes(32), b"\xff" * 32] + [rnd.randbytes(32) for _ in range(n - 3)])


def sign_msgs(rnd, n):
    """random messages below Q; about one lane in 16 above Q (rejected), one lane exactly Q (accepted, hashes as 0)"""
    ms = [rnd.randrange(Q) for _ in range(n)]
    for i in range(5, n, 16):
        ms[i] = rnd.randrange(Q + 1, 1 << 256)
    ms[1] = Q
    ms[2] = (1 << 256) - 1
    ms[0] = MSG_KAT
    return ms


def oracle_public_compressed(oracle_c, keys):
    x, y = oracle_c.public(keys)
    return oracle_c.compress(x, y)


def oracle_sign_compressed(oracle_c, keys, msgs):
    """compress(R8) || S per lane and the status; rejected lanes are 64 zero bytes (compress((0, 0)) is zero)"""
    rx, ry, s, st = oracle_c.sign(keys, msgs)
    return np.concatenate([oracle_c.compress(rx, ry), s], axis=1), st


def call(lib, ctx, name, ins, outs, dev):
    """bjj_<name>_batch (host or _dev flavour) with host arrays `ins`; fills `outs` and returns the return code"""
    n = len(ins[0])
    fn = getattr(lib, "bjj_%s_batch%s" % (name, "_dev" if dev else ""))
    if not dev:
        return fn(ctx, n, *[_p(a) for a in ins + outs])
    bufs = [lib.bjj_dev_alloc(ctx, max(a.nbytes, 1)) for a in ins + outs]
    try:
        assert all(bufs)
        for b, a in zip(bufs, ins):
            assert lib.bjj_memcpy_h2d(ctx, b, _p(a), a.nbytes) == 0
        rc = fn(ctx, n, *bufs, None)
        for b, a in zip(bufs[len(ins):], outs):
            assert lib.bjj_memcpy_d2h(ctx, _p(a), b, a.nbytes) == 0
        assert lib.bjj_sync(ctx) == 0
    finally:
        for b in bufs:
            lib.bjj_dev_free(ctx, b)
    return rc


def public_compressed(lib, ctx, keys, dev):
    out = np.zeros((len(keys), 32), np.uint8)
    assert call(lib, ctx, "public_compressed", [keys], [out], dev) == 0
    return out


def sign_compressed(lib, ctx, keys, msgs, dev):
    sig, st = np.zeros((len(keys), 64), np.uint8), np.full(len(keys), 0xEE, np.uint8)
    assert call(lib, ctx, "sign_compressed", [keys, msgs], [sig, st], dev) == 0
    return sig, st


# ---- CPU ----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def compressed_emu(tmp_path_factory):
    """tests/hostemu/compressed_emu.cpp (the compressed output forms of the device code, compiled for the host), built
    into a temporary directory"""
    from common import build_hostemu
    build_hostemu()                     # generates the constants header the device sources include
    so = str(tmp_path_factory.mktemp("compressed_emu") / "libbjj_compressed_emu.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so,
                           os.path.join(ROOT, "tests", "hostemu", "compressed_emu.cpp")])
    return ctypes.CDLL(so)


def test_hostemu_public_compressed(compressed_emu):
    """the batched affine pass in its compressed form (device source compiled for the host) against the oracle"""
    rnd = random.Random(21)
    keys = edge_keys(rnd, 64)
    out = np.zeros((64, 32), np.uint8)
    compressed_emu.emu_public_compressed(ctypes.c_size_t(64), _p(keys), _p(out))
    want = [O.compress(O.public(bytes(k))) for k in keys]
    assert [bytes(r) for r in out] == want


def test_hostemu_sign_compressed(compressed_emu):
    """the signing pipeline with the compressed finish against the oracle, msg > Q and msg == Q included"""
    rnd = random.Random(22)
    keys = edge_keys(rnd, 6)
    msgs = [MSG_KAT, Q, Q + 1, (1 << 256) - 1, 0, rnd.randrange(Q)]
    sig = np.zeros((6, 64), np.uint8)
    st = np.full(6, 0xEE, np.uint8)
    compressed_emu.emu_sign_compressed(ctypes.c_size_t(6), _p(keys), _p(pack(msgs)), _p(sig), _p(st))
    for i, m in enumerate(msgs):
        if m > Q:
            assert st[i] == STATUS_MSG_RANGE and not sig[i].any(), i
        else:
            assert st[i] == 0 and bytes(sig[i]) == O.compress_signature(O.sign(bytes(keys[i]), m)), i


def test_python_sign_message_clamping():
    import babyjubjub_rs_b200 as bjj
    words = unpack(bjj._sign_msgs([0, 5, Q, Q + 1, (1 << 256) - 1, 1 << 256, 7 << 300]))
    assert words == [0, 5, Q] + [(1 << 256) - 1] * 4
    with pytest.raises(ValueError, match="negative msg"):
        bjj._sign_msgs([1, -1])
    with pytest.raises(ValueError, match="negative msg"):
        bjj.sign_compressed_batch([KEY_KAT], [-5], engine=object())     # raises before any device work


def build_cpp():
    deps = [CPP_SRC, os.path.join(ROOT, "host", "bjj.hpp"), os.path.join(ROOT, "include", "bjj_cuda.h")]
    if not os.path.exists(CPP_EXE) or any(os.path.getmtime(d) > os.path.getmtime(CPP_EXE) for d in deps):
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-pthread", "-o", CPP_EXE, CPP_SRC, "-L" + PKG, "-lbjj_cuda",
                               "-Wl,-rpath," + PKG])
    return CPP_EXE


def test_cpp_compressed_builds_and_links():
    assert os.path.exists(build_cpp())


# ---- GPU ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_cpp_compressed_runs():
    out = subprocess.run([build_cpp()], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "compressed outputs ok" in out.stdout


@pytest.mark.gpu
def test_against_oracle_both_flavours(gpu, oracle_c):
    lib, ctx = gpu.eng.lib, gpu.eng.ctx
    rnd = random.Random(23)
    keys = edge_keys(rnd, LANES)
    ms = sign_msgs(rnd, LANES)
    msgs = pack(ms)
    want_pub = oracle_public_compressed(oracle_c, keys)
    want_sig, want_st = oracle_sign_compressed(oracle_c, keys, msgs)
    assert list(want_st[:3]) == [0, 0, STATUS_MSG_RANGE] and (want_st == STATUS_MSG_RANGE).sum() > LANES // 20
    for dev in (False, True):
        assert np.array_equal(public_compressed(lib, ctx, keys, dev), want_pub), dev
        sig, st = sign_compressed(lib, ctx, keys, msgs, dev)
        assert np.array_equal(st, want_st), dev
        assert np.array_equal(sig, want_sig), dev
        assert not sig[st == STATUS_MSG_RANGE].any()
    # the C++ checker against the Python restatement of the reference on the named lanes
    for i in (0, 1, 2):
        assert bytes(want_pub[i]) == O.compress(O.public(bytes(keys[i])))
    assert bytes(want_sig[0]) == O.compress_signature(O.sign(KEY_KAT, MSG_KAT))
    assert bytes(want_sig[1]) == O.compress_signature(O.sign(bytes(keys[1]), Q))


@pytest.mark.gpu
def test_composition_with_uncompressed_calls(gpu):
    eng = gpu.eng
    rnd = random.Random(24)
    keys = edge_keys(rnd, LANES)
    msgs = pack(sign_msgs(rnd, LANES))
    assert np.array_equal(eng.public_compressed_batch(keys), eng.compress_batch(*eng.public_batch(keys)))
    rx, ry, s, st = eng.sign_batch(keys, msgs)
    sig, st2 = eng.sign_compressed_batch(keys, msgs)
    assert np.array_equal(st, st2)
    assert np.array_equal(sig, np.concatenate([eng.compress_batch(rx, ry), s], axis=1))


@pytest.mark.gpu
def test_round_trip(gpu):
    eng = gpu.eng
    rnd = random.Random(25)
    keys = edge_keys(rnd, LANES)
    msgs = pack(sign_msgs(rnd, LANES))
    pub = eng.public_compressed_batch(keys)
    sig, st = eng.sign_compressed_batch(keys, msgs)
    good = st == 0
    ok, vst = eng.verify_compressed_batch(sig[good], pub[good], msgs[good])
    assert ok.all() and not vst.any()
    x, y, dst = eng.decompress_batch(pub)
    px, py = eng.public_batch(keys)
    assert not dst.any() and np.array_equal(x, px) and np.array_equal(y, py)


@pytest.mark.gpu
def test_chunk_and_subbatch_boundaries(gpu, oracle_c):
    """2^21 + 5 lanes: the host flavour runs three chunks, _dev two sub-batches; host arrays pageable, page-locked and
    mixed; the same launches as the uncompressed calls"""
    lib, ctx = gpu.eng.lib, gpu.eng.ctx
    rng = np.random.default_rng(26)
    keys = rng.integers(0, 256, size=(BIG, 32), dtype=np.uint8)
    keys[:3] = edge_keys(random.Random(26), 3)
    msgs = rng.integers(0, 256, size=(BIG, 32), dtype=np.uint8)
    msgs[:, 31] &= 0x2F                                    # < 0x30 * 2^248 < Q
    msgs[5::16, 31] = 0xFF                                 # > Q
    msgs[1] = pack([Q])[0]
    rnd = random.Random(26)
    sample = sorted(set(rnd.sample(range(BIG), 3000)) |
                    {0, 1, 2, 5, (1 << 18) - 1, 1 << 18, (1 << 21) - 1, 1 << 21, BIG - 1})
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
            _, n_pub = launches(lambda: call(lib, ctx, "public", [keys], [np.zeros_like(keys), np.zeros_like(keys)], dev))
            pub, n_pubc = launches(lambda: public_compressed(lib, ctx, keys, dev))
            assert n_pubc == n_pub == (9 if not dev else 6), (dev, n_pub, n_pubc)
            z = [np.zeros_like(keys) for _ in range(3)] + [np.zeros(BIG, np.uint8)]
            _, n_sign = launches(lambda: call(lib, ctx, "sign", [keys, msgs], z, dev))
            (sig, st), n_signc = launches(lambda: sign_compressed(lib, ctx, keys, msgs, dev))
            assert n_signc == n_sign == (21 if not dev else 14), (dev, n_sign, n_signc)
            if dev:
                assert np.array_equal(pub, pub_host) and np.array_equal(sig, sig_host) and np.array_equal(st, st_host)
            else:
                pub_host, sig_host, st_host = pub, sig, st
        # the host flavour from page-locked arrays, and from a mix of page-locked and pageable ones
        pk, pm = pinned_like(keys), pinned_like(msgs)
        for k_in, m_in, pinned_out in ((pk, pm, True), (pk, msgs, False), (keys, pm, True)):
            pub = pinned_like(np.zeros_like(keys)) if pinned_out else np.zeros_like(keys)
            assert call(lib, ctx, "public_compressed", [k_in], [pub], False) == 0
            assert np.array_equal(pub, pub_host)
            sig = pinned_like(np.zeros((BIG, 64), np.uint8)) if pinned_out else np.zeros((BIG, 64), np.uint8)
            st = np.zeros(BIG, np.uint8)
            assert call(lib, ctx, "sign_compressed", [k_in, m_in], [sig, st], False) == 0
            assert np.array_equal(sig, sig_host) and np.array_equal(st, st_host)
    finally:
        for ptr in pinned:
            lib.bjj_host_free(ptr)
    want_pub = oracle_public_compressed(oracle_c, keys[sample])
    want_sig, want_st = oracle_sign_compressed(oracle_c, keys[sample], msgs[sample])
    assert np.array_equal(pub_host[sample], want_pub)
    assert np.array_equal(st_host[sample], want_st) and np.array_equal(sig_host[sample], want_sig)
    assert st_host[1] == 0 and st_host[5] == STATUS_MSG_RANGE


@pytest.mark.gpu
def test_environment_switches(oracle_c):
    """BJJ_PUBLIC_FUSED=1 (k_public) and BJJ_SIGN_FUSED=1 (which leaves the compressed signing pipeline alone) give the
    same bytes"""
    from common import Gpu
    old = {k: os.environ.get(k) for k in ("BJJ_SIGN_FUSED", "BJJ_PUBLIC_FUSED")}
    os.environ["BJJ_SIGN_FUSED"] = "1"
    os.environ["BJJ_PUBLIC_FUSED"] = "1"
    try:
        alt = Gpu(0)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    try:
        lib, ctx = alt.eng.lib, alt.eng.ctx
        rnd = random.Random(27)
        keys = edge_keys(rnd, LANES)
        msgs = pack(sign_msgs(rnd, LANES))
        want_pub = oracle_public_compressed(oracle_c, keys)
        want_sig, want_st = oracle_sign_compressed(oracle_c, keys, msgs)
        for dev in (False, True):
            assert np.array_equal(public_compressed(lib, ctx, keys, dev), want_pub), dev
            sig, st = sign_compressed(lib, ctx, keys, msgs, dev)
            assert np.array_equal(st, want_st) and np.array_equal(sig, want_sig), dev
    finally:
        alt.eng.close()


@pytest.mark.gpu
def test_multi_engine_matches_single_engine(gpu):
    import babyjubjub_rs_b200 as bjj
    eng = gpu.eng
    ndev = eng.lib.bjj_device_count()
    rnd = random.Random(28)
    n = 3 * 4096 + 7                                       # not divisible by 2, 4, 8 devices
    keys = edge_keys(rnd, n)
    msgs = pack(sign_msgs(rnd, n))
    want_pub = eng.public_compressed_batch(keys)
    want_sig, want_st = eng.sign_compressed_batch(keys, msgs)
    for devices in sorted({(0,), tuple(range(ndev))}):
        me = bjj.MultiEngine(list(devices))
        try:
            assert me.devices == len(devices)
            assert np.array_equal(me.public_compressed_batch(keys), want_pub), devices
            sig, st = me.sign_compressed_batch(keys, msgs)
            assert np.array_equal(sig, want_sig) and np.array_equal(st, want_st), devices
            out = (np.zeros((n, 64), np.uint8), np.zeros(n, np.uint8))
            assert me.sign_compressed_batch(keys, msgs, out=out)[0] is out[0]
            assert np.array_equal(out[0], want_sig) and np.array_equal(out[1], want_st)
            pub = np.zeros_like(keys)
            assert me.public_compressed_batch(keys, out=pub) is pub and np.array_equal(pub, want_pub)
            me.set_host_register(True)
            assert np.array_equal(me.public_compressed_batch(keys[:4097]), want_pub[:4097])
        finally:
            me.close()


@pytest.mark.gpu
def test_arguments_and_python_mirror(gpu):
    import babyjubjub_rs_b200 as bjj
    lib, ctx = gpu.eng.lib, gpu.eng.ctx
    k, m = pack([1] * 64), pack([2] * 64)
    o32, o64, st = np.zeros((64, 32), np.uint8), np.zeros((64, 64), np.uint8), np.zeros(64, np.uint8)
    for dev in (False, True):
        sfx = "_dev" if dev else ""
        pub, sign = getattr(lib, "bjj_public_compressed_batch" + sfx), getattr(lib, "bjj_sign_compressed_batch" + sfx)
        tail = (None,) if dev else ()
        assert pub(ctx, 0, _p(k), _p(o32), *tail) == 0
        assert sign(ctx, 0, _p(k), _p(m), _p(o64), _p(st), *tail) == 0
        assert pub(None, 64, _p(k), _p(o32), *tail) == ERR_ARG
        assert pub(ctx, 64, None, _p(o32), *tail) == ERR_ARG
        assert pub(ctx, 64, _p(k), None, *tail) == ERR_ARG
        assert sign(None, 64, _p(k), _p(m), _p(o64), _p(st), *tail) == ERR_ARG
        for i in range(4):
            args = [_p(k), _p(m), _p(o64), _p(st)]
            args[i] = None
            assert sign(ctx, 64, *args, *tail) == ERR_ARG, (dev, i)
    me = bjj.MultiEngine([0])
    try:
        h = me.handle
        assert lib.bjj_multi_public_compressed_batch(h, 0, _p(k), _p(o32)) == 0
        assert lib.bjj_multi_sign_compressed_batch(h, 0, _p(k), _p(m), _p(o64), _p(st)) == 0
        assert lib.bjj_multi_public_compressed_batch(None, 64, _p(k), _p(o32)) == ERR_ARG
        assert lib.bjj_multi_public_compressed_batch(h, 64, None, _p(o32)) == ERR_ARG
        assert lib.bjj_multi_public_compressed_batch(h, 64, _p(k), None) == ERR_ARG
        for i in range(4):
            args = [_p(k), _p(m), _p(o64), _p(st)]
            args[i] = None
            assert lib.bjj_multi_sign_compressed_batch(h, 64, *args) == ERR_ARG, i
    finally:
        me.close()
    # module-level mirrors against the Python oracle
    rnd = random.Random(29)
    keys = [KEY_KAT, bytes(32), b"\xff" * 32] + [rnd.randbytes(32) for _ in range(5)]
    assert bjj.public_compressed_batch(keys, engine=gpu.eng) == [O.compress(O.public(key)) for key in keys]
    assert bjj.public_compressed_batch([bjj.PrivateKey(KEY_KAT)], engine=gpu.eng) == [O.compress(O.public(KEY_KAT))]
    msgs = [MSG_KAT, Q, Q + 1, 1 << 256, 0, rnd.randrange(Q), (1 << 256) - 1, 12345]
    got = bjj.sign_compressed_batch(keys, msgs, engine=gpu.eng)
    for key, msg, g in zip(keys, msgs, got):
        if msg > Q:
            assert isinstance(g, ValueError) and str(g) == "msg outside the Finite Field"
        else:
            assert g == O.compress_signature(O.sign(key, msg))
    assert bjj.public_compressed_batch([], engine=gpu.eng) == [] and bjj.sign_compressed_batch([], [], engine=gpu.eng) == []
