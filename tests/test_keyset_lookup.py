"""key-set keys by their compressed bytes (bjj_keyset_lookup_batch, bjj_verify_keyset_lookup_compressed_batch): the host
index builder and the lookup lane body compiled for the host against a dict over the oracle's compress, with crafted
probe chains under a fixed seed; on the GPU both flavours against the dict and byte for byte against
bjj_verify_compressed_batch, unknown keys without an error, launch counts, argument errors and the Python / C++
mirrors."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

from common import ROOT, pack
from oracle import bjj_oracle as O

Q = O.Q
NONE = 0xFFFFFFFF
ERR_ARG = 2
BIG = (1 << 21) + 5
BUILD_SUBBATCH = (1 << 21) // 4097          # keys per build sub-batch of bjj_keyset_create

CPP_SRC = os.path.join(ROOT, "tests", "cpp", "test_keyset_lookup.cpp")
PKG = os.path.join(ROOT, "babyjubjub-rs_b200")


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def blobs(arr):
    a = np.ascontiguousarray(arr, dtype=np.uint8).reshape(-1, 32)
    return [a[i].tobytes() for i in range(len(a))]


def dict_index(keys):
    """{compress(P_j): smallest j} over the keys with x != 0 -- what the lookup must find"""
    d = {}
    for j, k in enumerate(keys):
        if k[0] != 0:
            d.setdefault(O.compress(k), j)
    return d


def random_points(rnd, n):
    """n on-curve points from random compressed bytes (decompress_point of a random y and sign)"""
    out = []
    while len(out) < n:
        try:
            out.append(O.decompress_point(rnd.getrandbits(254).to_bytes(32, "little")[:31] + bytes([rnd.getrandbits(8) & 0x9F])))
        except ValueError:
            pass
    return out


def neg(p):
    return ((Q - p[0]) % Q, p[1])


# ---- CPU ----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lookup_emu(tmp_path_factory):
    """tests/hostemu/keyset_lookup_emu.cpp (the index builder and lane_keyset_lookup compiled for the host)"""
    from common import build_hostemu
    build_hostemu()                     # generates the constants header the device sources include
    so = str(tmp_path_factory.mktemp("keyset_lookup_emu") / "libbjj_keyset_lookup_emu.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so,
                           os.path.join(ROOT, "tests", "hostemu", "keyset_lookup_emu.cpp")])
    lib = ctypes.CDLL(so)
    lib.emu_lookup_build.restype = ctypes.c_size_t
    lib.emu_lookup_build.argtypes = [ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64]
    lib.emu_lookup_hash.argtypes = [ctypes.c_size_t, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_void_p]
    return lib


def emu_build(emu, keys, seed):
    ax, ay = pack([k[0] for k in keys]), pack([k[1] for k in keys])
    slots = emu.emu_lookup_build(len(keys), _p(ax), _p(ay), seed)
    table, comp = np.zeros(slots, np.uint32), np.zeros((len(keys), 32), np.uint8)
    emu.emu_lookup_table(_p(table), _p(comp))
    assert blobs(comp) == [O.compress(k) for k in keys]
    return table


def emu_lookup(emu, lanes):
    pk = np.frombuffer(b"".join(lanes), np.uint8).reshape(-1, 32).copy()
    out = np.full(len(lanes), 0xEEEEEEEE, np.uint32)
    emu.emu_lookup(ctypes.c_size_t(len(lanes)), _p(pk), _p(out))
    return [int(v) for v in out]


def emu_hash(emu, lanes, seed):
    pk = np.frombuffer(b"".join(lanes), np.uint8).reshape(-1, 32).copy()
    out = np.zeros(len(lanes), np.uint64)
    emu.emu_lookup_hash(len(lanes), _p(pk), seed, _p(out))
    return [int(v) for v in out]


def variants(rnd, c):
    """bytes that differ from a compressed key only in bit 255 or in one byte of y"""
    out = [c[:31] + bytes([c[31] ^ 0x80])]
    for _ in range(3):
        b = bytearray(c)
        b[rnd.randrange(32)] ^= 1 << rnd.randrange(8)
        out.append(bytes(b))
    return out


def check_lookup(emu, keys, lanes):
    want = dict_index(keys)
    got = emu_lookup(emu, lanes)
    assert got == [want.get(c, NONE) for c in lanes]
    return got


def test_hostemu_random_sets_with_duplicates(lookup_emu):
    """random sets in which some points appear two or three times: every key's bytes find its smallest index, whatever
    the seed; near misses (bit 255, one byte of y) and non-keys miss"""
    rnd = random.Random(80)
    for n, seed in ((1, 0), (2, 1), (7, 0xDEADBEEF), (100, 12345), (1000, (1 << 64) - 1)):
        pts = random_points(rnd, n)
        keys = pts + [pts[rnd.randrange(n)] for _ in range(n // 3)]
        rnd.shuffle(keys)
        table = emu_build(lookup_emu, keys, seed)
        assert len(table) >= 2 * len(keys) and len(table) & (len(table) - 1) == 0 and len(table) < 4 * len(keys) + 2
        assert sorted(int(t) for t in table if t != NONE) == sorted(set(dict_index(keys).values()))
        lanes = [O.compress(k) for k in keys]
        lanes += [v for c in lanes[:50] for v in variants(rnd, c)]
        lanes += [O.compress(p) for p in random_points(rnd, 20)]
        got = check_lookup(lookup_emu, keys, lanes)
        assert all(keys[got[j]] == keys[j] and got[j] <= j for j in range(len(keys)))
        for s2 in (seed ^ 1, seed + 77):       # another seed moves slots, never results
            emu_build(lookup_emu, keys, s2 & ((1 << 64) - 1))
            assert emu_lookup(lookup_emu, lanes) == got


def test_hostemu_negation_and_x_zero(lookup_emu):
    """P and -P (same y, bit 255 apart) are found under their own indices; (0, 1) and (0, Q-1) are not indexed"""
    rnd = random.Random(81)
    pts = random_points(rnd, 6)
    keys = [pts[0], neg(pts[0]), (0, 1), pts[1], (0, Q - 1), neg(pts[2]), pts[2], (0, 1)]
    emu_build(lookup_emu, keys, 99)
    lanes = [O.compress(k) for k in keys] + [O.compress(neg(pts[1]))]
    got = check_lookup(lookup_emu, keys, lanes)
    assert got == [0, 1, NONE, 3, NONE, 5, 6, NONE, NONE]
    assert O.compress(pts[0])[:31] == O.compress(neg(pts[0]))[:31]


def test_hostemu_edge_bytes(lookup_emu):
    """all-zero and all-ones lanes, y >= Q with either sign bit, and Q - 1, miss"""
    keys = random_points(random.Random(82), 40) + [(0, 1)]
    emu_build(lookup_emu, keys, 5)
    lanes = [bytes(32), b"\xff" * 32, b"\xff" * 31 + b"\x7f", Q.to_bytes(32, "little"),
             Q.to_bytes(32, "little")[:31] + bytes([Q.to_bytes(32, "little")[31] | 0x80]), (Q - 1).to_bytes(32, "little"),
             (1).to_bytes(32, "little")]
    assert check_lookup(lookup_emu, keys, lanes) == [NONE] * len(lanes)


def test_hostemu_crafted_probe_chain(lookup_emu):
    """a fixed seed and keys crafted to hash to one slot near the end of the table: they form one chain that wraps
    round to slot 0; hits at its end and misses that hash into it walk the whole chain, and a miss ends at the empty
    slot after it"""
    seed = 0x0123456789ABCDEF
    n_chain, n = 12, 16                     # 32 slots
    rnd = random.Random(83)
    target = 27
    chain, others = [], []
    while len(chain) < n_chain or len(others) < n - n_chain:
        p = random_points(rnd, 1)[0]
        s = emu_hash(lookup_emu, [O.compress(p)], seed)[0] & 31
        if s == target and len(chain) < n_chain:
            chain.append(p)
        elif 14 <= s <= 20 and len(others) < n - n_chain:       # well clear of the chain's run 27..31, 0..6
            others.append(p)
    keys = chain + others
    table = emu_build(lookup_emu, keys, seed)
    assert len(table) == 32
    run = [(target + k) % 32 for k in range(n_chain)]
    assert [int(table[s]) for s in run] == list(range(n_chain))          # slots 27..31, 0..6 in insertion order
    assert int(table[(target + n_chain) % 32]) == NONE
    misses = []
    while len(misses) < 8:
        b = rnd.getrandbits(256).to_bytes(32, "little")
        if emu_hash(lookup_emu, [b], seed)[0] & 31 == target:
            misses.append(b)
    lanes = [O.compress(k) for k in reversed(keys)] + misses + [v for c in [O.compress(chain[-1])] for v in variants(rnd, c)]
    got = check_lookup(lookup_emu, keys, lanes)
    assert got[:n] == list(reversed(range(n))) and got[n:n + 8] == [NONE] * 8


def test_python_argument_handling():
    import babyjubjub_rs_b200 as bjj
    p = bjj.Point(*random_points(random.Random(84), 1)[0])
    pk = bjj._pk32s([p, O.compress((p.x, p.y)), bytearray(32)])
    assert pk.shape == (3, 32) and pk[0].tobytes() == O.compress((p.x, p.y)) == pk[1].tobytes() and not pk[2].any()
    assert bjj._pk32s([]).shape == (0, 32)
    with pytest.raises(ValueError):
        bjj._pk32s([b"\x00" * 31])
    with pytest.raises(ValueError):
        bjj.verify_keyset_lookup_batch(None, [b"\x00" * 32], [], [1])
    with pytest.raises(ValueError):
        bjj.verify_keyset_lookup_batch(None, [b"\x00" * 32], [b"\x00" * 63], [1])
    with pytest.raises(ValueError):
        bjj._keyset_handle(None)
    assert bjj.KEY_NONE == NONE


def build_cpp(out_dir):
    exe = os.path.join(str(out_dir), "test_keyset_lookup")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-pthread", "-o", exe, CPP_SRC, "-L" + PKG, "-lbjj_cuda",
                           "-Wl,-rpath," + PKG])
    return exe


def test_cpp_keyset_lookup_builds_and_links(tmp_path):
    assert os.path.exists(build_cpp(tmp_path))


# ---- GPU ----------------------------------------------------------------------------------------------
def create(lib, ctx, ax, ay):
    h = ctypes.c_void_p()
    assert lib.bjj_keyset_create(ctx, len(ax), _p(ax), _p(ay), None, ctypes.byref(h)) == 0
    return h


def run(lib, ctx, name, ks, ins, outs, dev, rc=0):
    """bjj_<name>_batch over key set ks with host arrays `ins`, in either flavour; fills `outs`"""
    n = len(ins[0])
    fn = getattr(lib, "bjj_%s_batch%s" % (name, "_dev" if dev else ""))
    if not dev:
        assert fn(ctx, ks, n, *[_p(a) for a in ins + outs]) == rc
        return
    bufs = [lib.bjj_dev_alloc(ctx, max(a.nbytes, 1)) for a in ins + outs]
    try:
        assert all(bufs)
        for b, a in zip(bufs, ins):
            assert lib.bjj_memcpy_h2d(ctx, b, _p(a), a.nbytes) == 0
        assert fn(ctx, ks, n, *bufs, None) == rc
        for b, a in zip(bufs[len(ins):], outs):
            assert lib.bjj_memcpy_d2h(ctx, _p(a), b, a.nbytes) == 0
        assert lib.bjj_sync(ctx) == 0           # an unknown key is data: no sticky error either
    finally:
        for b in bufs:
            lib.bjj_dev_free(ctx, b)


def lookup(lib, ctx, ks, pk32, dev):
    ki = np.full(len(pk32), 0xEEEEEEEE, np.uint32)
    run(lib, ctx, "keyset_lookup", ks, [pk32], [ki], dev)
    return ki


def verify_lookup(lib, ctx, ks, sig64, pk32, msgs, dev):
    n = len(sig64)
    ok, st, ki = np.full(n, 0xEE, np.uint8), np.full(n, 0xEE, np.uint8), np.full(n, 0xEEEEEEEE, np.uint32)
    run(lib, ctx, "verify_keyset_lookup_compressed", ks, [sig64, pk32, msgs], [ok, st, ki], dev)
    return ok, st, ki


def launches(lib, ctx, fn):
    before = lib.bjj_kernel_launches(ctx)
    r = fn()
    return r, lib.bjj_kernel_launches(ctx) - before


def device_keys(eng, n, seed):
    """n key pairs made on the device -> private keys, (ax, ay), compressed public keys"""
    priv = np.random.default_rng(seed).integers(0, 256, size=(n, 32), dtype=np.uint8)
    ax, ay = eng.public_batch(priv)
    return priv, (ax, ay), eng.compress_batch(ax, ay)


def signed_lanes(eng, n, n_keys, n_outside, seed):
    """n compressed signatures by n_keys + n_outside device keys (the last n_outside not in the set), 10 % corrupted:
    S or msg bits, msg > Q, R8 with y >= Q and R8 that is mostly not a square -> key set (ax, ay), sig64, pk32, msgs"""
    rng = np.random.default_rng(seed)
    priv, (ax, ay), comp = device_keys(eng, n_keys + n_outside, seed)
    who = rng.integers(0, n_keys + n_outside, size=n)
    msgs = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    msgs[:, 31] &= 0x2F                                     # < Q
    sig64, st = eng.sign_compressed_batch(priv[who], msgs)
    assert not st.any()
    lanes = rng.permutation(n)[: n // 10]
    for j, i in enumerate(lanes):
        kind = j % 5
        if kind == 0:
            sig64[i, 32 + rng.integers(0, 31)] ^= 1 << int(rng.integers(0, 8))
        elif kind == 1:
            msgs[i, rng.integers(0, 31)] ^= 1 << int(rng.integers(0, 8))
        elif kind == 2:
            msgs[i] = 0xFF                                  # msg > Q
        elif kind == 3:
            sig64[i, 31] |= 0x7F                            # y >= Q
        else:
            sig64[i, 0] ^= 0x5A                             # mostly not a square
    return (ax[:n_keys], ay[:n_keys]), sig64, comp[who], msgs


@pytest.mark.gpu
def test_lookup_against_dict_big(gpu):
    """2^21 + 5 lanes over a set of 65,536 device keys (a few held twice, (0, 1) among them): hits, keys outside the
    set, near misses and random bytes, both flavours against the dict; 1 launch per sub-batch"""
    eng = gpu.eng
    lib, ctx = eng.lib, eng.ctx
    n_keys = 1 << 16
    _, (ax, ay), comp = device_keys(eng, n_keys + 4096, 90)
    ax, ay = ax[:n_keys].copy(), ay[:n_keys].copy()
    rng = np.random.default_rng(90)
    dup = rng.integers(0, n_keys, size=64)
    ax[n_keys - 64:], ay[n_keys - 64:] = ax[dup], ay[dup]
    ax[100], ay[100] = 0, pack([1])[0]                      # (0, 1): never found
    keys_comp = eng.compress_batch(ax, ay)
    want_d = {}
    for j, c in enumerate(blobs(keys_comp)):
        if j != 100:
            want_d.setdefault(c, j)
    src = rng.integers(0, 5, size=BIG)
    pk32 = keys_comp[rng.integers(0, n_keys, size=BIG)]
    out = comp[n_keys:][rng.integers(0, 4096, size=BIG)]
    pk32[src == 1] = out[src == 1]
    near = src == 2
    pk32[near, 31] ^= 0x80
    pk32[src == 3, rng.integers(0, 32)] ^= 1
    pk32[src == 4] = rng.integers(0, 256, size=(int((src == 4).sum()), 32), dtype=np.uint8)
    want = np.array([want_d.get(c, NONE) for c in blobs(pk32)], np.uint32)
    assert (want != NONE).mean() > 0.2 and (want == NONE).mean() > 0.5
    h = create(lib, ctx, ax, ay)
    try:
        for dev in (False, True):
            got, k = launches(lib, ctx, lambda: lookup(lib, ctx, h, pk32, dev))
            assert np.array_equal(got, want), dev
            assert k == (2 if dev else 3), (dev, k)          # _dev: two sub-batches; host: three chunks
            _, k = launches(lib, ctx, lambda: lookup(lib, ctx, h, pk32[:1000], dev))
            assert k == 1, (dev, k)
    finally:
        lib.bjj_keyset_destroy(ctx, h)


@pytest.mark.gpu
def test_verify_equals_verify_compressed(gpu):
    """2^16 compressed signatures by 1,100 device keys, 1,000 of them in the set (plus (0, 1)), 10 % corrupted: on
    found lanes ok and status byte-equal to bjj_verify_compressed_batch; other lanes ok 0, R8's status and KEY_NONE;
    the same as bjj_keyset_lookup followed by bjj_verify_keyset_compressed_batch on the found lanes"""
    eng = gpu.eng
    lib, ctx = eng.lib, eng.ctx
    n = 1 << 16
    (ax, ay), sig64, pk32, msgs = signed_lanes(eng, n, 1000, 100, 91)
    ax, ay = np.concatenate([ax, pack([0])]), np.concatenate([ay, pack([1])])
    pk32[5::997] = pack([1])[0]                             # compress((0, 1)): in the set, never found
    want_ok, want_st = eng.verify_compressed_batch(sig64, pk32, msgs)
    _, _, r8_st = eng.decompress_batch(np.ascontiguousarray(sig64[:, :32]))
    assert set(np.unique(r8_st)) >= {0, 1, 3}
    h = create(lib, ctx, ax, ay)
    try:
        ki = lookup(lib, ctx, h, pk32, False)
        found = ki != NONE
        assert 0.85 * n < found.sum() < 0.95 * n
        for dev in (False, True):
            ok, st, kid = verify_lookup(lib, ctx, h, sig64, pk32, msgs, dev)
            assert np.array_equal(kid, ki), dev
            assert np.array_equal(ok[found], want_ok[found]) and np.array_equal(st[found], want_st[found]), dev
            assert not ok[~found].any() and np.array_equal(st[~found], r8_st[~found]), dev
            assert 0.75 * n < ok.sum() < 0.9 * n
        fi = np.flatnonzero(found)
        ok2, st2 = np.zeros(len(fi), np.uint8), np.zeros(len(fi), np.uint8)
        assert lib.bjj_verify_keyset_compressed_batch(ctx, h, len(fi), _p(ki[fi].copy()), _p(sig64[fi].copy()),
                                                      _p(msgs[fi].copy()), _p(ok2), _p(st2)) == 0
        assert np.array_equal(ok2, ok[fi]) and np.array_equal(st2, st[fi])
    finally:
        lib.bjj_keyset_destroy(ctx, h)


@pytest.mark.gpu
def test_big_launches_and_unknown_keys_without_error(gpu):
    """2^21 + 5 lanes: 6 launches per sub-batch (also at 1,000 lanes), results equal to verify_compressed on found
    lanes; unknown keys raise nothing, in the call or at the next bjj_sync, and afterwards an index outside the set
    still gives BJJ_ERR_ARG from bjj_verify_keyset_compressed_batch; create launches as before"""
    eng = gpu.eng
    lib, ctx = eng.lib, eng.ctx
    (ax, ay), sig64, pk32, msgs = signed_lanes(eng, BIG, 300, 30, 92)
    want_ok, want_st = eng.verify_compressed_batch(sig64, pk32, msgs)
    h, k = launches(lib, ctx, lambda: create(lib, ctx, ax, ay))
    assert k == 1 + 2 * (-(-300 // BUILD_SUBBATCH))
    try:
        for dev in (False, True):
            (ok, st, ki), k = launches(lib, ctx, lambda: verify_lookup(lib, ctx, h, sig64, pk32, msgs, dev))
            assert k == (12 if dev else 18), (dev, k)
            found = ki != NONE
            assert (~found).sum() > BIG // 20
            assert np.array_equal(ok[found], want_ok[found]) and np.array_equal(st[found], want_st[found]), dev
            assert not ok[~found].any()
            _, k = launches(lib, ctx, lambda: verify_lookup(lib, ctx, h, sig64[:1000], pk32[:1000], msgs[:1000], dev))
            assert k == 6, (dev, k)
        assert lib.bjj_sync(ctx) == 0
        bad = np.zeros(4, np.uint32)
        bad[2] = 300
        o, s = np.zeros(4, np.uint8), np.zeros(4, np.uint8)
        assert lib.bjj_verify_keyset_compressed_batch(ctx, h, 4, _p(bad), _p(sig64[:4].copy()), _p(msgs[:4].copy()), _p(o), _p(s)) == ERR_ARG
    finally:
        lib.bjj_keyset_destroy(ctx, h)


@pytest.mark.gpu
def test_argument_errors(gpu):
    """NULL pointers, a NULL or foreign handle, n == 0; a closed KeySet in Python"""
    bjj, eng = gpu.bjj, gpu.eng
    lib, ctx = eng.lib, eng.ctx
    keys = [O.public(bytes(range(32))), O.B8]
    other = bjj.Engine(0)
    mine, foreign = bjj.KeySet(keys, eng), bjj.KeySet(keys, other)
    try:
        pk, s64, m = np.zeros((4, 32), np.uint8), np.zeros((4, 64), np.uint8), np.zeros((4, 32), np.uint8)
        o, ki = np.zeros(4, np.uint8), np.zeros(4, np.uint32)
        for dev in (False, True):
            sfx, tail = ("_dev", (None,)) if dev else ("", ())
            lk = getattr(lib, "bjj_keyset_lookup_batch" + sfx)
            vf = getattr(lib, "bjj_verify_keyset_lookup_compressed_batch" + sfx)
            for hnd in (None, foreign.handle):
                assert lk(ctx, hnd, 4, _p(pk), _p(ki), *tail) == ERR_ARG
                assert vf(ctx, hnd, 4, _p(s64), _p(pk), _p(m), _p(o), _p(o), _p(ki), *tail) == ERR_ARG
            assert lk(None, mine.handle, 4, _p(pk), _p(ki), *tail) == ERR_ARG
            assert lk(ctx, mine.handle, 4, None, _p(ki), *tail) == ERR_ARG
            assert lk(ctx, mine.handle, 4, _p(pk), None, *tail) == ERR_ARG
            assert lk(ctx, mine.handle, 0, _p(pk), _p(ki), *tail) == 0
            full = [_p(s64), _p(pk), _p(m), _p(o), _p(o), _p(ki)]
            for j in range(6):
                args = list(full)
                args[j] = None
                assert vf(ctx, mine.handle, 4, *args, *tail) == ERR_ARG, (dev, j)
            assert vf(ctx, mine.handle, 0, *full, *tail) == 0
        assert lib.bjj_sync(ctx) == 0
    finally:
        mine.close()
        foreign.close()
        other.close()
    with pytest.raises(ValueError):
        mine.lookup([O.compress(keys[0])])
    with pytest.raises(ValueError):
        bjj.verify_keyset_lookup_batch(mine, [b"\x00" * 32], [b"\x00" * 64], [1])


@pytest.mark.gpu
def test_python_and_cpp_mirrors(gpu, tmp_path):
    bjj, eng = gpu.bjj, gpu.eng
    keys = [bytes(range(32)), bytes(range(1, 33)), bytes(range(2, 34)), bytes(range(3, 35))]
    pts = [O.public(k) for k in keys]
    ks = bjj.KeySet([bjj.Point(*pts[0]), pts[1], pts[2], pts[1], (0, 1)], eng)
    try:
        comp = [O.compress(p) for p in pts]
        assert ks.lookup([bjj.Point(*pts[2]), comp[1], comp[3], O.compress(neg(pts[0])), O.compress((0, 1)), comp[0]]) == \
            [2, 1, None, None, None, 0]
        assert ks.lookup([]) == []
        msgs = [11, 12, 13, 14, 15, Q + 1]
        who = [0, 1, 3, 2, 2, 0]
        sigs = [O.compress_signature(O.sign(keys[j], m if m <= Q else 5)) for j, m in zip(who, msgs)]
        sigs[4] = b"\xff" * 31 + b"\x7f" + sigs[4][32:]     # R8 y >= Q
        got = bjj.verify_keyset_lookup_batch(ks, [comp[j] for j in who], sigs, msgs)
        assert got[:4] == [True, True, None, True] and got[5] is False
        assert isinstance(got[4], ValueError) and str(got[4]) == O.ERR_Y_RANGE
        assert bjj.verify_keyset_lookup_batch(ks, [], [], []) == []
    finally:
        ks.close()
    out = subprocess.run([build_cpp(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "keyset lookup ok" in out.stdout
