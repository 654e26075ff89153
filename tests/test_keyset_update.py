"""editing key sets in place (bjj_keyset_append, bjj_keyset_replace): the host index rebuild compiled for the host against
a dict over the oracle's compress; on the GPU every key-set call on an edited set byte-equal to a set created from the
current key list, lookups after edits, errors that leave the set unchanged, NOMEM, growth without a second copy of the
tables, in-flight work, launch counts and the Python / C++ mirrors."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

from common import ROOT, pack, unpack
from oracle import bjj_oracle as O

Q = O.Q
NONE = 0xFFFFFFFF
ERR_ARG, ERR_NONCANONICAL, ERR_NOMEM = 2, 3, 4
BIG = (1 << 21) + 5
BUILD_SUBBATCH = (1 << 21) // 4097          # keys per build sub-batch
TABLE_BYTES = 4130 * 96                     # one key's comb table
SCHNORR_WORDS = 16                          # s of sign_schnorr_batch with 256-bit nonces

CPP_SRC = os.path.join(ROOT, "tests", "cpp", "test_keyset_update.cpp")
PKG = os.path.join(ROOT, "babyjubjub-rs_b200")


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def dict_index(keys):
    """{compress(P_j): smallest j} over the keys with x != 0 -- what the lookup must find"""
    d = {}
    for j, k in enumerate(keys):
        if k[0] != 0:
            d.setdefault(O.compress(k), j)
    return d


def random_points(rnd, n):
    """n on-curve points from random compressed bytes"""
    out = []
    while len(out) < n:
        try:
            out.append(O.decompress_point(rnd.getrandbits(254).to_bytes(32, "little")[:31] + bytes([rnd.getrandbits(8) & 0x9F])))
        except ValueError:
            pass
    return out


def neg(p):
    return ((Q - p[0]) % Q, p[1])


def build_launches(n):
    return 1 + 2 * (-(-n // BUILD_SUBBATCH))


# ---- CPU ----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def update_emu(tmp_path_factory):
    """tests/hostemu/keyset_update_emu.cpp (keyset_compress, keyset_index_fill and lane_keyset_lookup for the host)"""
    from common import build_hostemu
    build_hostemu()                     # generates the constants header the device sources include
    so = str(tmp_path_factory.mktemp("keyset_update_emu") / "libbjj_keyset_update_emu.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so,
                           os.path.join(ROOT, "tests", "hostemu", "keyset_update_emu.cpp")])
    lib = ctypes.CDLL(so)
    lib.emu_update_reset.argtypes = [ctypes.c_uint64]
    lib.emu_update_edit.restype = ctypes.c_size_t
    lib.emu_update_edit.argtypes = [ctypes.c_size_t, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p]
    lib.emu_update_table.restype = ctypes.c_size_t
    lib.emu_update_table.argtypes = [ctypes.c_void_p]
    lib.emu_update_lookup.argtypes = [ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p]
    lib.emu_update_indexed.argtypes = [ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p]
    return lib


class EmuSet:
    """a key list mirrored by the host index of keyset_update_emu.cpp"""

    def __init__(self, emu, seed):
        self.emu, self.keys = emu, []
        emu.emu_update_reset(seed)

    def edit(self, first, pts):
        ax, ay = pack([p[0] for p in pts]), pack([p[1] for p in pts])
        n1 = self.emu.emu_update_edit(first, len(pts), _p(ax), _p(ay))
        self.keys[first:first + len(pts)] = pts
        assert n1 == len(self.keys)
        comp = np.zeros((n1, 32), np.uint8)
        slots = self.emu.emu_update_table(_p(comp))
        assert [comp[j].tobytes() for j in range(n1)] == [O.compress(k) for k in self.keys]
        assert slots >= 2 * n1 and slots & (slots - 1) == 0

    def append(self, pts):
        self.edit(len(self.keys), pts)

    def check(self, extra=()):
        """every key's bytes, their negations and `extra` against dict_index of the current list"""
        lanes = [O.compress(k) for k in self.keys] + [O.compress(neg(k)) for k in self.keys] + list(extra)
        pk = np.frombuffer(b"".join(lanes), np.uint8).reshape(-1, 32).copy()
        out = np.full(len(lanes), 0xEEEEEEEE, np.uint32)
        self.emu.emu_update_lookup(len(lanes), _p(pk), _p(out))
        want = dict_index(self.keys)
        assert [int(v) for v in out] == [want.get(c, NONE) for c in lanes]
        return [int(v) for v in out]


def test_hostemu_append_duplicates_across_old_and_new(update_emu):
    """appends that repeat old keys and each other: every key is found at its smallest index, old or new"""
    rnd = random.Random(90)
    pts = random_points(rnd, 300)
    s = EmuSet(update_emu, 0x5EED)
    s.append(pts[:100])
    s.check()
    for size in (1, 7, 50, 120):
        new = [pts[rnd.randrange(300)] for _ in range(size)]      # mostly new keys, some already in the set
        s.append(new)
        s.check()
    assert len(s.keys) == 278
    assert s.check()[:3] == [s.keys.index(s.keys[j]) for j in range(3)]


def test_hostemu_replace_duplicates_x_zero_and_negation(update_emu):
    """a replaced key's old bytes go to its duplicate, or nowhere; x = 0 keys are never indexed, in old or new keys;
    P and -P are found at their own indices"""
    rnd = random.Random(91)
    p = random_points(rnd, 8)
    s = EmuSet(update_emu, 17)
    s.append([p[0], p[1], p[2], p[3], (0, 1)])
    s.append([p[3], neg(p[1]), (0, Q - 1), p[4]])                 # p3 twice, -p1 next to p1
    got = s.check([O.compress((0, 1)), O.compress((0, Q - 1))])
    assert got[:9] == [0, 1, 2, 3, NONE, 3, 6, NONE, 8] and got[-2:] == [NONE, NONE]
    s.edit(3, [p[5]])                                             # p3's old bytes: found at its duplicate
    assert s.check([O.compress(p[3])])[-1] == 5
    s.edit(5, [p[6]])                                             # ... and now nowhere
    assert s.check([O.compress(p[3])])[-1] == NONE
    s.edit(0, [(0, 1), p[1]])                                     # x = 0 replaces a key; p1 at 1 twice
    got = s.check([O.compress(p[0])])
    assert got[0] == NONE and got[1] == 1 and got[-1] == NONE
    s.edit(8, [neg(p[6])])                                        # the last key
    assert s.check()[:9] == [NONE, 1, 2, 3, NONE, 5, 6, NONE, 8]


def test_hostemu_random_edit_sequences(update_emu):
    """random appends and replaces drawn from a small pool (so keys repeat), x = 0 keys and negations among them,
    against dict_index after every step"""
    rnd = random.Random(92)
    base = random_points(rnd, 40)
    pool = base + [neg(b) for b in base[:10]] + [(0, 1), (0, Q - 1)]
    for seed in (0, (1 << 64) - 1, 0xABCDEF):
        s = EmuSet(update_emu, seed)
        s.append([rnd.choice(pool) for _ in range(rnd.randrange(1, 30))])
        for _ in range(40):
            if rnd.random() < 0.4:
                s.append([rnd.choice(pool) for _ in range(rnd.randrange(1, 9))])
            else:
                first = rnd.randrange(len(s.keys))
                s.edit(first, [rnd.choice(pool) for _ in range(rnd.randrange(1, len(s.keys) - first + 1))])
            s.check()


def test_hostemu_indexed_bytes(update_emu):
    """only the compressed forms of (0, 1) and (0, Q-1) stay out of the index"""
    lanes = [(1).to_bytes(32, "little"), (Q - 1).to_bytes(32, "little"), bytes(32), (2).to_bytes(32, "little"),
             (1 | 1 << 255).to_bytes(32, "little"), (Q - 2).to_bytes(32, "little"), Q.to_bytes(32, "little"),
             (1 | 1 << 64).to_bytes(32, "little")]
    c = np.frombuffer(b"".join(lanes), np.uint8).copy()
    out = np.zeros(len(lanes), np.uint8)
    update_emu.emu_update_indexed(len(lanes), _p(c), _p(out))
    assert list(out) == [0, 0, 1, 1, 1, 1, 1, 1]


def test_python_replace_rejects_negative_first():
    import babyjubjub_rs_b200 as bjj
    ks = bjj.KeySet.__new__(bjj.KeySet)
    with pytest.raises(ValueError):
        ks.replace(-1, [])


def build_cpp(out_dir):
    exe = os.path.join(str(out_dir), "test_keyset_update")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-pthread", "-o", exe, CPP_SRC, "-L" + PKG, "-lbjj_cuda",
                           "-Wl,-rpath," + PKG])
    return exe


def test_cpp_keyset_update_builds_and_links(tmp_path):
    assert os.path.exists(build_cpp(tmp_path))


# ---- GPU ----------------------------------------------------------------------------------------------
def create(lib, ctx, ax, ay, rc=0):
    h = ctypes.c_void_p()
    st = np.full(len(ax), 0xEE, np.uint8)
    assert lib.bjj_keyset_create(ctx, len(ax), _p(ax), _p(ay), _p(st), ctypes.byref(h)) == rc
    return h


def append(lib, ctx, h, ax, ay, rc=0):
    st = np.full(len(ax), 0xEE, np.uint8)
    got = lib.bjj_keyset_append(ctx, h, len(ax), _p(ax), _p(ay), _p(st))
    assert got == rc, got
    return st


def replace(lib, ctx, h, first, ax, ay, rc=0):
    st = np.full(len(ax), 0xEE, np.uint8)
    got = lib.bjj_keyset_replace(ctx, h, first, len(ax), _p(ax), _p(ay), _p(st))
    assert got == rc, got
    return st


def launches(lib, ctx, fn):
    before = lib.bjj_kernel_launches(ctx)
    r = fn()
    return r, lib.bjj_kernel_launches(ctx) - before


def run(lib, ctx, name, ks, head, ins, outs, dev, tail=()):
    """bjj_<name>_batch over key set ks: `head` scalars after n, then the host arrays ins + outs (device copies for
    _dev), then `tail` scalars before the outputs; fills `outs`"""
    n = len(ins[0])
    fn = getattr(lib, "bjj_%s_batch%s" % (name, "_dev" if dev else ""))
    if not dev:
        assert fn(ctx, ks, n, *head, *[_p(a) for a in ins], *tail, *[_p(a) for a in outs]) == 0, name
        return
    bufs = [lib.bjj_dev_alloc(ctx, max(a.nbytes, 1)) for a in ins + outs]
    try:
        assert all(bufs)
        for b, a in zip(bufs, ins):
            assert lib.bjj_memcpy_h2d(ctx, b, _p(a), a.nbytes) == 0
        assert fn(ctx, ks, n, *head, *bufs[:len(ins)], *tail, *bufs[len(ins):], None) == 0, name
        for b, a in zip(bufs[len(ins):], outs):
            assert lib.bjj_memcpy_d2h(ctx, _p(a), b, a.nbytes) == 0
        assert lib.bjj_sync(ctx) == 0, name
    finally:
        for b in bufs:
            lib.bjj_dev_free(ctx, b)


def answers(lib, ctx, ks, lanes, dev):
    """the outputs of the five verify / lookup calls and keyset_mul over `lanes` -> {name: [arrays]}"""
    n = len(lanes["idx"])
    out = {}

    def go(name, ins, shapes, tail=()):
        outs = [np.full(s, 0xEE, d) for s, d in shapes]
        run(lib, ctx, name, ks, (), ins, outs, dev, tail)
        out[name] = outs
    b1, b4, b32 = ((n,), np.uint8), ((n,), np.uint32), ((n, 32), np.uint8)
    go("verify_keyset", [lanes["idx"], lanes["r8x"], lanes["r8y"], lanes["s"], lanes["msg"]], [b1])
    go("verify_keyset_compressed", [lanes["idx"], lanes["sig64"], lanes["msg"]], [b1, b1])
    go("verify_schnorr_keyset", [lanes["idx"], lanes["msg"], lanes["rx"], lanes["ry"], lanes["sw"]], [b1, b1],
       tail=(SCHNORR_WORDS,))
    go("keyset_mul", [lanes["idx"], lanes["k"]], [b32, b32])
    go("keyset_lookup", [lanes["pk32"]], [b4])
    go("verify_keyset_lookup_compressed", [lanes["sig64"], lanes["pk32"], lanes["msg"]], [b1, b1, b4])
    return out


def make_lanes(eng, priv, cur, old_priv, n, seed):
    """n lanes over the key list `cur` (indices into `priv`): signatures of three kinds by each lane's key, 10 %
    corrupted, 2 % signed by a replaced key's old private key; scalars; compressed keys of the list, of keys outside
    it and random bytes"""
    rng = np.random.default_rng(seed)
    idx = rng.integers(0, len(cur), size=n).astype(np.uint32)
    signer = np.asarray(cur)[idx]
    stale = rng.random(n) < 0.02
    signer[stale] = rng.choice(old_priv, size=int(stale.sum()))
    msg = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    msg[:, 31] &= 0x2F
    r8x, r8y, s, st = eng.sign_batch(priv[signer], msg)
    assert not st.any()
    sig64, st = eng.sign_compressed_batch(priv[signer], msg)
    assert not st.any()
    rx, ry, sw, st = eng.sign_schnorr_batch(priv[signer], msg, rng.integers(0, 256, size=(n, 32), dtype=np.uint8), 8)
    assert not st.any() and sw.shape == (n, 4 * SCHNORR_WORDS)
    bad = rng.random(n) < 0.1
    col = rng.integers(0, 31, size=n)
    for arr in (s, sig64[:, 32:], sw):
        arr[bad, col[bad]] ^= 1
    ax, ay = eng.public_batch(priv)
    comp = eng.compress_batch(ax, ay)
    pk32 = comp[signer].copy()
    kind = rng.integers(0, 4, size=n)
    pk32[kind == 1] = comp[rng.integers(0, len(priv), size=int((kind == 1).sum()))]
    pk32[kind == 2] = rng.integers(0, 256, size=(int((kind == 2).sum()), 32), dtype=np.uint8)
    k = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    return dict(idx=idx, r8x=r8x, r8y=r8y, s=s, msg=msg, sig64=sig64, rx=rx, ry=ry, sw=sw, k=k, pk32=pk32, signer=signer)


@pytest.mark.gpu
def test_edited_set_equals_created_set_big(gpu):
    """create(700 keys), appends of 1, 510, 511, 512 and 1,023 keys and twelve single keys, replaces in the middle and
    at both ends (launch counts checked on every edit): on 2^21 + 5 lanes both flavours of all six calls equal a set
    created from the current list byte for byte, and a sample of lanes of every kind equals the oracle"""
    eng = gpu.eng
    lib, ctx = eng.lib, eng.ctx
    rng = np.random.default_rng(93)
    n_priv = 4000
    priv = rng.integers(0, 256, size=(n_priv, 32), dtype=np.uint8)
    ax, ay = eng.public_batch(priv)
    cur = list(range(700))
    nxt = 700
    h, k = launches(lib, ctx, lambda: create(lib, ctx, ax[cur], ay[cur]))
    assert k == build_launches(700)
    try:
        for size in [1, 510, 511, 512, 1023] + [1] * 12:
            new = list(range(nxt, nxt + size))
            nxt += size
            st, k = launches(lib, ctx, lambda: append(lib, ctx, h, ax[new], ay[new]))
            assert not st.any() and k == build_launches(size), size
            cur += new
        old = []
        for first, count in ((1000, 600), (0, 3), (len(cur) - 5, 5), (len(cur) - 1, 1), (2000, 1)):
            new = list(range(nxt, nxt + count))
            nxt += count
            st, k = launches(lib, ctx, lambda: replace(lib, ctx, h, first, ax[new], ay[new]))
            assert not st.any() and k == build_launches(count), (first, count)
            old += cur[first:first + count]
            cur[first:first + count] = new
        assert nxt <= n_priv and len(cur) == 700 + 2569
        fresh = create(lib, ctx, ax[cur], ay[cur])
        try:
            lanes = make_lanes(eng, priv, cur, old, BIG, 94)
            for dev in (False, True):
                got, want = answers(lib, ctx, h, lanes, dev), answers(lib, ctx, fresh, lanes, dev)
                for name in want:
                    for g, w in zip(got[name], want[name]):
                        assert np.array_equal(g, w), (name, dev)
            ok = got["verify_keyset"][0]
            assert 0.8 * BIG < ok.sum() < 0.9 * BIG
            ki = got["keyset_lookup"][0]
            assert (ki == NONE).mean() > 0.2 and (ki != NONE).mean() > 0.5
        finally:
            lib.bjj_keyset_destroy(ctx, fresh)
        keys = list(zip(unpack(ax), unpack(ay)))
        want_d = dict_index([keys[j] for j in cur])
        stale = np.flatnonzero(~np.isin(lanes["signer"], cur))
        sample = list(np.random.default_rng(95).choice(BIG, 40, replace=False)) + list(stale[:5]) + [0, BIG - 1]
        for i in sample:
            A = keys[cur[lanes["idx"][i]]]
            m = unpack(lanes["msg"][i:i + 1])[0]
            sig = (unpack(lanes["r8x"][i:i + 1])[0], unpack(lanes["r8y"][i:i + 1])[0]), unpack(lanes["s"][i:i + 1])[0]
            assert got["verify_keyset"][0][i] == O.verify(A, sig, m), i
            assert got["keyset_lookup"][0][i] == want_d.get(lanes["pk32"][i].tobytes(), NONE), i
            kk = unpack(lanes["k"][i:i + 1])[0]
            assert O.mul_scalar(A, kk) == (unpack(got["keyset_mul"][0][i:i + 1])[0], unpack(got["keyset_mul"][1][i:i + 1])[0]), i
    finally:
        lib.bjj_keyset_destroy(ctx, h)


@pytest.mark.gpu
def test_lookup_after_edits(gpu):
    """a duplicate of key 3 appended is found at 3; replacing key 3 moves its old bytes to the duplicate; x = 0 keys
    appended are never found; -P is found at its own index; P and the replaced key as a fresh set would find them"""
    bjj, eng = gpu.bjj, gpu.eng
    pts = [O.public(bytes([j]) * 32) for j in range(1, 8)]
    ks = bjj.KeySet(pts[:5], eng)
    try:
        ks.append([pts[3]])
        assert ks.lookup([O.compress(pts[3])]) == [3] and len(ks) == 6
        ks.replace(3, [pts[5]])
        assert ks.lookup([O.compress(pts[3]), O.compress(pts[5])]) == [5, 3]
        ks.append([(0, 1), (0, Q - 1), neg(pts[1])])
        assert ks.lookup([O.compress(p) for p in ((0, 1), (0, Q - 1), neg(pts[1]), pts[1])]) == [None, None, 8, 1]
        want = bjj.KeySet([(p.x, p.y) for p in ks.points], eng)
        try:
            lanes = [O.compress(p) for p in pts] + [O.compress(neg(p)) for p in pts] + [O.compress((0, 1))]
            assert ks.lookup(lanes) == want.lookup(lanes)
            assert [(p.x, p.y) for p in ks.mul_batch(list(range(9)), [12345] * 9)] == \
                [(p.x, p.y) for p in want.mul_batch(list(range(9)), [12345] * 9)]
        finally:
            want.close()
    finally:
        ks.close()


def snapshot(lib, ctx, h, keys, extra):
    """lookups of every key, its negation and `extra`, and k * P_j for every key j (host flavour)"""
    comp = [O.compress(k) for k in keys] + [O.compress(neg(k)) for k in keys] + [O.compress(e) for e in extra]
    pk = np.frombuffer(b"".join(comp), np.uint8).reshape(-1, 32).copy()
    ki = np.zeros(len(comp), np.uint32)
    assert lib.bjj_keyset_lookup_batch(ctx, h, len(comp), _p(pk), _p(ki)) == 0
    kk = pack([7 + j for j in range(len(keys))])
    rx, ry = np.zeros_like(kk), np.zeros_like(kk)
    idx = np.arange(len(keys), dtype=np.uint32)
    assert lib.bjj_keyset_mul_batch(ctx, h, len(keys), _p(idx), _p(kk), _p(rx), _p(ry)) == 0
    # one index past the set is still outside it
    bad = np.array([len(keys)], np.uint32)
    assert lib.bjj_keyset_mul_batch(ctx, h, 1, _p(bad), _p(kk), _p(rx[:1].copy()), _p(ry[:1].copy())) == ERR_ARG
    return ki, rx, ry


@pytest.mark.gpu
def test_errors_leave_the_set_unchanged(gpu):
    """an off-curve key, a non-canonical key (which outranks it), NULL pointers, a NULL or foreign handle, n_new = 0,
    count = 0, replace past the end and n_keys + n_new > 2^32 - 1: each leaves lookups, k*P and the size as they were"""
    bjj, eng = gpu.bjj, gpu.eng
    lib, ctx = eng.lib, eng.ctx
    keys = [O.public(bytes([j]) * 32) for j in range(1, 6)]
    new = [O.public(bytes([j]) * 32) for j in range(6, 9)]
    ax, ay = pack([k[0] for k in keys]), pack([k[1] for k in keys])
    nx, ny = pack([k[0] for k in new]), pack([k[1] for k in new])
    h = create(lib, ctx, ax, ay)
    other = bjj.Engine(0)
    foreign = create(other.lib, other.ctx, ax, ay)
    try:
        before = snapshot(lib, ctx, h, keys, new)

        def same():
            after = snapshot(lib, ctx, h, keys, new)
            assert all(np.array_equal(a, b) for a, b in zip(before, after))
        off_x = nx.copy()
        off_x[1, 0] ^= 1                                  # key 1 off the curve
        assert list(append(lib, ctx, h, off_x, ny, ERR_ARG)) == [0, 1, 0]
        same()
        assert list(replace(lib, ctx, h, 1, off_x, ny, ERR_ARG)) == [0, 1, 0]
        same()
        nc = off_x.copy()
        nc[2] = pack([new[2][0] + Q])[0]                  # key 2's x >= Q: outranks key 1 off the curve
        assert list(append(lib, ctx, h, nc, ny, ERR_NONCANONICAL)) == [0, 1, 2]
        same()
        assert list(replace(lib, ctx, h, 2, nc, ny, ERR_NONCANONICAL)) == [0, 1, 2]
        same()
        st = np.zeros(3, np.uint8)
        for a, b in ((None, _p(ny)), (_p(nx), None)):
            assert lib.bjj_keyset_append(ctx, h, 3, a, b, _p(st)) == ERR_ARG
            assert lib.bjj_keyset_replace(ctx, h, 0, 3, a, b, _p(st)) == ERR_ARG
        for c, hnd in ((ctx, None), (ctx, foreign), (None, h)):
            assert lib.bjj_keyset_append(c, hnd, 3, _p(nx), _p(ny), _p(st)) == ERR_ARG
            assert lib.bjj_keyset_replace(c, hnd, 0, 3, _p(nx), _p(ny), _p(st)) == ERR_ARG
        assert lib.bjj_keyset_append(ctx, h, 0, _p(nx), _p(ny), _p(st)) == 0
        assert lib.bjj_keyset_replace(ctx, h, 2, 0, _p(nx), _p(ny), _p(st)) == 0
        assert lib.bjj_keyset_replace(ctx, h, 5, 0, _p(nx), _p(ny), _p(st)) == 0
        assert lib.bjj_keyset_replace(ctx, h, 6, 0, _p(nx), _p(ny), _p(st)) == ERR_ARG
        assert lib.bjj_keyset_replace(ctx, h, 3, 3, _p(nx), _p(ny), _p(st)) == ERR_ARG
        assert lib.bjj_keyset_replace(ctx, h, (1 << 64) - 1, 2, _p(nx), _p(ny), _p(st)) == ERR_ARG
        assert lib.bjj_keyset_replace(ctx, h, 1, (1 << 64) - 1, _p(nx), _p(ny), _p(st)) == ERR_ARG
        assert lib.bjj_keyset_append(ctx, h, (1 << 32) - 5, _p(nx), _p(ny), _p(st)) == ERR_ARG
        assert lib.bjj_keyset_append(ctx, h, (1 << 64) - 1, _p(nx), _p(ny), _p(st)) == ERR_ARG
        same()
        assert lib.bjj_sync(ctx) == 0
        # the Python mirror: BjjError with the codes above, points and the set unchanged
        ks = bjj.KeySet(keys, eng)
        try:
            with pytest.raises(bjj.BjjError) as e:
                ks.append([new[0], (new[1][0] ^ 1, new[1][1])])
            assert e.value.code == ERR_ARG and list(e.value.key_status) == [0, 1] and len(ks) == 5
            assert len(ks.status) == 5 and not ks.status.any()
            with pytest.raises(bjj.BjjError) as e:
                ks.replace(4, new[:2])
            assert e.value.code == ERR_ARG and [(p.x, p.y) for p in ks.points] == keys
            assert ks.lookup([O.compress(k) for k in new + keys]) == [None] * 3 + list(range(5))
        finally:
            ks.close()
    finally:
        lib.bjj_keyset_destroy(ctx, h)
        other.lib.bjj_keyset_destroy(other.ctx, foreign)
        other.close()


@pytest.mark.gpu
def test_nomem_for_the_build_scratch_leaves_the_set_unchanged(gpu):
    """a replace whose build needs more projective scratch than the context holds, with too little free memory to grow
    it: BJJ_ERR_NOMEM with the CUDA error cleared, planes, tables and lookups unchanged; with the memory back, the same
    replace succeeds"""
    import torch
    bjj = gpu.bjj
    eng = bjj.Engine(0)                           # a context of its own: its scratch only ever held one key's build
    lib, ctx = eng.lib, eng.ctx
    keys = [O.public(bytes([j]) * 32) for j in range(1, 65)]
    new = [O.public(bytes([j]) * 32) for j in range(65, 129)]
    h = create(lib, ctx, pack([keys[0][0]]), pack([keys[0][1]]))
    hog = []
    try:
        for k in keys[1:]:
            append(lib, ctx, h, pack([k[0]]), pack([k[1]]))
        before = snapshot(lib, ctx, h, keys, new)
        nx, ny = pack([k[0] for k in new]), pack([k[1] for k in new])
        # 64 keys need 64 x 4,097 x 128 B = 32 MiB of scratch; leave about 12 MiB free
        dev = torch.device("cuda", lib.bjj_device(ctx))
        want = mem_info()[0] - (12 << 20)
        while want > 0 and not hog:
            try:
                hog.append(torch.empty(want, dtype=torch.uint8, device=dev))
            except RuntimeError:
                want -= 2 << 20
        assert mem_info()[0] < 32 << 20
        assert lib.bjj_keyset_replace(ctx, h, 0, 64, _p(nx), _p(ny), None) == ERR_NOMEM
        hog.clear()
        torch.cuda.empty_cache()
        assert lib.bjj_sync(ctx) == 0
        after = snapshot(lib, ctx, h, keys, new)
        assert all(np.array_equal(a, b) for a, b in zip(before, after))
        replace(lib, ctx, h, 0, nx, ny)
        _, rx, ry = snapshot(lib, ctx, h, new, keys)
        for j in (0, 31, 63):
            assert (unpack(rx[j:j + 1])[0], unpack(ry[j:j + 1])[0]) == O.mul_scalar(new[j], 7 + j), j
        pk = np.frombuffer(b"".join(O.compress(k) for k in new + keys), np.uint8).reshape(-1, 32).copy()
        ki = np.zeros(128, np.uint32)
        assert lib.bjj_keyset_lookup_batch(ctx, h, 128, _p(pk), _p(ki)) == 0
        assert list(ki) == list(range(64)) + [NONE] * 64
    finally:
        hog.clear()
        lib.bjj_keyset_destroy(ctx, h)
        eng.close()


def mem_info():
    import torch
    free, total = torch.cuda.mem_get_info(0)
    return free, total


@pytest.mark.gpu
def test_nomem_leaves_the_set_unchanged(gpu):
    """appending more copies of B8 than free device memory holds (and more than the device holds at all) returns
    BJJ_ERR_NOMEM with the CUDA error cleared; the set answers as before and still grows afterwards"""
    eng = gpu.eng
    lib, ctx = eng.lib, eng.ctx
    keys = [O.public(bytes([j]) * 32) for j in range(1, 4)]
    h = create(lib, ctx, pack([k[0] for k in keys]), pack([k[1] for k in keys]))
    try:
        before = snapshot(lib, ctx, h, keys, [O.B8])
        free, total = mem_info()
        for n_new in (free // TABLE_BYTES + 64, total // TABLE_BYTES + 64):
            bx, by = np.tile(pack([O.B8[0]]), (n_new, 1)), np.tile(pack([O.B8[1]]), (n_new, 1))
            assert lib.bjj_keyset_append(ctx, h, n_new, _p(bx), _p(by), None) == ERR_NOMEM, n_new
            assert lib.bjj_sync(ctx) == 0
            after = snapshot(lib, ctx, h, keys, [O.B8])
            assert all(np.array_equal(a, b) for a, b in zip(before, after))
            del bx, by
        append(lib, ctx, h, pack([O.B8[0]]), pack([O.B8[1]]))
        ki = np.zeros(1, np.uint32)
        pk = np.frombuffer(O.compress(O.B8), np.uint8).reshape(1, 32).copy()
        assert lib.bjj_keyset_lookup_batch(ctx, h, 1, _p(pk), _p(ki)) == 0 and ki[0] == 3
    finally:
        lib.bjj_keyset_destroy(ctx, h)


@pytest.mark.gpu
def test_append_needs_no_second_copy(gpu):
    """a set of about 60 % of free device memory grows by another 10 %: the append succeeds (a reallocate-and-copy
    design would need 130 %), and free memory drops by the new tables rounded up to the 2 MB granularity, within 64 MB
    (the key planes, the index and the build's scratch)"""
    eng = gpu.eng
    lib, ctx = eng.lib, eng.ctx
    free, _ = mem_info()
    n0, n1 = int(0.6 * free) // TABLE_BYTES, int(0.1 * free) // TABLE_BYTES
    bx, by = np.tile(pack([O.B8[0]]), (n0 + n1, 1)), np.tile(pack([O.B8[1]]), (n0 + n1, 1))
    h = create(lib, ctx, bx[:n0], by[:n0])
    try:
        f0, _ = mem_info()
        append(lib, ctx, h, bx[n0:], by[n0:])
        f1, _ = mem_info()
        gran = 2 << 20
        want = -(-(n0 + n1) * TABLE_BYTES // gran) * gran - (-(-n0 * TABLE_BYTES // gran) * gran)
        assert abs((f0 - f1) - want) < 64 << 20, (f0 - f1, want)
        kk = pack([3, 5])
        idx = np.array([0, n0 + n1 - 1], np.uint32)
        rx, ry = np.zeros_like(kk), np.zeros_like(kk)
        assert lib.bjj_keyset_mul_batch(ctx, h, 2, _p(idx), _p(kk), _p(rx), _p(ry)) == 0
        assert [(a, b) for a, b in zip(unpack(rx), unpack(ry))] == [O.mul_scalar(O.B8, 3), O.mul_scalar(O.B8, 5)]
    finally:
        lib.bjj_keyset_destroy(ctx, h)


@pytest.mark.gpu
def test_in_flight_dev_call_sees_the_set_before_the_edit(gpu):
    """a _dev verify and a _dev lookup enqueued on a caller stream just before a replace (and an append) return what
    the set held before it"""
    import torch
    eng = gpu.eng
    lib, ctx = eng.lib, eng.ctx
    n = 1 << 18
    rng = np.random.default_rng(96)
    priv = rng.integers(0, 256, size=(64, 32), dtype=np.uint8)
    ax, ay = eng.public_batch(priv)
    comp = eng.compress_batch(ax, ay)
    idx = rng.integers(0, 32, size=n).astype(np.uint32)
    msg = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    msg[:, 31] &= 0x2F
    sig64, _ = eng.sign_compressed_batch(priv[idx], msg)
    pk32 = comp[idx]
    h = create(lib, ctx, ax[:32], ay[:32])
    try:
        dev = torch.device("cuda", lib.bjj_device(ctx))
        t = {k: torch.from_numpy(v.view(np.uint8).reshape(n, -1)).to(dev) for k, v in
             dict(idx=idx, sig64=sig64, msg=msg, pk32=pk32).items()}
        ok, st = torch.zeros(n, dtype=torch.uint8, device=dev), torch.zeros(n, dtype=torch.uint8, device=dev)
        ki = torch.zeros(n * 4, dtype=torch.uint8, device=dev)
        s = torch.cuda.Stream(device=dev)
        torch.cuda.synchronize(dev)
        with torch.cuda.stream(s):
            assert lib.bjj_verify_keyset_compressed_batch_dev(ctx, h, n, t["idx"].data_ptr(), t["sig64"].data_ptr(),
                                                              t["msg"].data_ptr(), ok.data_ptr(), st.data_ptr(),
                                                              ctypes.c_void_p(s.cuda_stream)) == 0
            assert lib.bjj_keyset_lookup_batch_dev(ctx, h, n, t["pk32"].data_ptr(), ki.data_ptr(),
                                                   ctypes.c_void_p(s.cuda_stream)) == 0
        replace(lib, ctx, h, 0, ax[32:64], ay[32:64])             # every key of the set changes
        append(lib, ctx, h, ax[:32], ay[:32])
        torch.cuda.synchronize(dev)
        assert lib.bjj_sync(ctx) == 0
        assert ok.cpu().numpy().all() and not st.cpu().numpy().any()
        assert np.array_equal(ki.cpu().numpy().view(np.uint32), idx)
        ok2, st2 = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
        assert lib.bjj_verify_keyset_compressed_batch(ctx, h, n, _p(idx), _p(sig64), _p(msg), _p(ok2), _p(st2)) == 0
        assert not ok2.any()                                       # indices 0..31 now hold other keys
    finally:
        lib.bjj_keyset_destroy(ctx, h)


@pytest.mark.gpu
def test_python_and_cpp_mirrors(gpu, tmp_path):
    """KeySet.append / replace equal the C calls on the same list (points and status follow), and the C++ program"""
    bjj, eng = gpu.bjj, gpu.eng
    lib, ctx = eng.lib, eng.ctx
    pts = [O.public(bytes([j]) * 32) for j in range(10, 20)]
    ks = bjj.KeySet(pts[:4], eng)
    try:
        ks.append([bjj.Point(*pts[4]), pts[5], pts[1]])
        ks.replace(2, [pts[6], pts[7]])
        ks.replace(6, [pts[8]])
        cur = [pts[0], pts[1], pts[6], pts[7], pts[4], pts[5], pts[8]]
        assert [(p.x, p.y) for p in ks.points] == cur and len(ks) == 7 and not ks.status.any() and len(ks.status) == 7
        h = create(lib, ctx, pack([p[0] for p in pts[:4]]), pack([p[1] for p in pts[:4]]))
        try:
            append(lib, ctx, h, pack([p[0] for p in (pts[4], pts[5], pts[1])]), pack([p[1] for p in (pts[4], pts[5], pts[1])]))
            replace(lib, ctx, h, 2, pack([pts[6][0], pts[7][0]]), pack([pts[6][1], pts[7][1]]))
            replace(lib, ctx, h, 6, pack([pts[8][0]]), pack([pts[8][1]]))
            lanes = [O.compress(p) for p in pts]
            pk = np.frombuffer(b"".join(lanes), np.uint8).reshape(-1, 32).copy()
            ki = np.zeros(len(lanes), np.uint32)
            assert lib.bjj_keyset_lookup_batch(ctx, h, len(lanes), _p(pk), _p(ki)) == 0
            assert ks.lookup(lanes) == [None if k == NONE else int(k) for k in ki] == [0, 1, None, None, 4, 5, 2, 3, 6, None]
            idx = list(range(7))
            assert [(p.x, p.y) for p in ks.mul_batch(idx, [99] * 7)] == [O.mul_scalar(p, 99) for p in cur]
        finally:
            lib.bjj_keyset_destroy(ctx, h)
    finally:
        ks.close()
    out = subprocess.run([build_cpp(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "keyset update ok" in out.stdout
