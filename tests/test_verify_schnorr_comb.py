"""verify_schnorr on the signer's unreduced s (bjj_verify_schnorr_base_batch, bjj_verify_schnorr_keyset_batch,
bjj_verify_schnorr_wide_batch): the comb lane bodies compiled for the host against the oracle, torsion keys and every
s width included; on the GPU every form in both flavours against the oracle, sign -> verify fully on the device, chunk
and sub-batch boundaries with launch counts, argument errors, a workspace shared with verify_batch's deferred exact
lanes, and the Python / C++ mirrors."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

from common import KEY_KAT, ROOT, pack, unpack
from oracle import bjj_oracle as O
from test_verify_base import IDENTITY, add, keys_with_secrets, torsion_points

Q, ORDER, SUBORDER = O.Q, O.ORDER, O.SUBORDER
ERR_ARG, ERR_NONCANONICAL = 2, 3
MSG_RANGE = 4
BIG = (1 << 21) + 5
MASK = (1 << 256) - 1
WIDTHS = list(range(8, 73, 8))

CPP_SRC = os.path.join(ROOT, "tests", "cpp", "test_verify_schnorr_comb.cpp")
PKG = os.path.join(ROOT, "babyjubjub-rs_b200")


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def u32(a):
    return np.ascontiguousarray(a, dtype="<u4")


def pack_wide(vals, words):
    return np.frombuffer(b"".join(int(v).to_bytes(4 * words, "little") for v in vals), np.uint8).reshape(-1, 4 * words).copy()


def schnorr_sig(pk, a, k, m):
    """(r, s, m) with r = k*B8 and s = k + a*h unreduced: the reference's signature for pk = a*B8 (+ torsion)"""
    r = O.mul_scalar(O.B8, k)
    return r, k + a * O.schnorr_hash(pk, m, r), m


def schnorr_cases(rnd, pk, a):
    """list of (r, s, msg) for key pk: valid signatures, corruptions, msg edges, r off the curve, r with a torsion
    component, s edges; every s below 2^1280 (fits 40 words)"""
    t2, t4, t8 = torsion_points()
    cases = [schnorr_sig(pk, a, rnd.getrandbits(1024), rnd.randrange(Q)) for _ in range(3)]
    r, s, m = cases[0]
    cases += [(r, s + 1, m), (r, s ^ (1 << 700), m), (r, s, (m + 1) % Q), (cases[1][0], s, m)]      # wrong s, msg, r
    cases += [(r, s + 37 * SUBORDER, m)]                                                          # s + multiple of l
    for _ in range(64):                         # a valid signature for a key with a torsion component T: h*T = O
        c = schnorr_sig(pk, a, rnd.getrandbits(64), m)
        if O.verify_schnorr(pk, m, c[0], c[1]):
            cases.append(c)
            break
    cases += [schnorr_sig(pk, a, rnd.getrandbits(1024), Q), schnorr_sig(pk, a, 5, 0)]             # msg == Q hashes as 0
    cases += [(r, s, Q + 1), (r, s, MASK)]                                                        # msg > Q: Err
    for off in ((0, 0), ((r[0] + 1) % Q, r[1]), (5, 7)):                                          # r off the curve
        cases += [(off, s, m), (off, 0, m)]
    for t in (t2, t4, t8):                                  # r with a torsion component, s = k + a*h(r + t)
        for _ in range(3):
            k = rnd.getrandbits(1024)
            rt = add(O.mul_scalar(O.B8, k), t)
            cases.append((rt, k + a * O.schnorr_hash(pk, m, rt), m))
    cases += [(IDENTITY, 0, 77), (IDENTITY, SUBORDER, 78), (IDENTITY, 12 * SUBORDER, 79), (O.B8, 1, 80), (O.B8, SUBORDER + 1, 81)]
    return cases


def oracle_case(pk, case):
    """(ok, status) of the reference's verify_schnorr"""
    r, s, m = case
    if m > Q:
        return 0, MSG_RANGE
    return int(O.verify_schnorr(pk, m, r, s)), 0


def case_arrays(cases, words):
    """msg, rx, ry, s (words words per lane) of (r, s, msg) cases"""
    return [pack([c[2] for c in cases]), pack([c[0][0] for c in cases]), pack([c[0][1] for c in cases]),
            pack_wide([c[1] for c in cases], words)]


def width_cases(rnd, pk, a, words):
    """cases whose s fills `words` words: a valid signature with the widest nonce that fits, and all-ones s"""
    kbits = 32 * words - 512
    cases = []
    if kbits > 0:
        cases.append(schnorr_sig(pk, a, rnd.getrandbits(kbits) | (1 << (kbits - 1)), rnd.randrange(Q)))
    ones = (1 << (32 * words)) - 1
    cases += [(O.mul_scalar(O.B8, ones), ones, 3), (IDENTITY, ones, 4)]
    return cases


# ---- CPU ----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    """tests/hostemu/schnorr_comb_emu.cpp (the comb lane bodies in Schnorr mode compiled for the host)"""
    from common import build_hostemu
    build_hostemu()                     # generates the constants header the device sources include
    so = str(tmp_path_factory.mktemp("schnorr_comb_emu") / "libbjj_schnorr_comb_emu.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so,
                           os.path.join(ROOT, "tests", "hostemu", "schnorr_comb_emu.cpp")])
    lib = ctypes.CDLL(so)
    for f in ("emu_keyset_create", "emu_verify_schnorr_base", "emu_verify_schnorr_keyset"):
        getattr(lib, f).restype = ctypes.c_uint32
    return lib


def check_emu_outputs(cases, want, ok, st, s_red, reached):
    assert list(st) == [w[1] for w in want]
    assert list(ok) == [w[0] for w in want], [i for i in range(len(cases)) if ok[i] != want[i][0]]
    red = unpack(s_red)
    for i, c in enumerate(cases):
        if reached[i]:
            assert red[i] == c[1] % SUBORDER, i


def emu_base(emu, pk, cases, words):
    n = len(cases)
    ins = case_arrays(cases, words)
    ok, st = np.full(n, 0xEE, np.uint8), np.full(n, 0xEE, np.uint8)
    s_red = np.zeros((n, 32), np.uint8)
    px, py = pack([pk[0]]), pack([pk[1]])
    flags = emu.emu_verify_schnorr_base(ctypes.c_size_t(n), _p(px), _p(py), *[_p(v) for v in ins], words, _p(ok), _p(st), _p(s_red))
    return flags, ok, st, s_red


def test_hostemu_base_against_oracle(emu):
    """the base lane bodies against verify_schnorr for every key kind (torsion keys included) at 40 words, and at every
    width 8..72 on width-filling s (all-ones words included); the reduced s equals s % SUBORDER"""
    for j, (name, pk, a) in enumerate(keys_with_secrets()):
        rnd = random.Random(90 + j)
        cases = schnorr_cases(rnd, pk, a)
        want = [oracle_case(pk, c) for c in cases]
        assert sum(w[0] for w in want) >= 2, name
        flags, ok, st, s_red = emu_base(emu, pk, cases, 40)
        assert flags == 0, name
        check_emu_outputs(cases, want, ok, st, s_red, [c[2] <= Q for c in cases])
        for words in WIDTHS:
            wc = width_cases(rnd, pk, a, words) + [cases[0], cases[-1]]
            wc = [c for c in wc if c[1] < 1 << (32 * words)]
            flags, ok, st, s_red = emu_base(emu, pk, wc, words)
            check_emu_outputs(wc, [oracle_case(pk, c) for c in wc], ok, st, s_red, [True] * len(wc))


def test_hostemu_keyset_against_oracle(emu):
    """the key-set lane bodies against verify_schnorr, all key kinds in one set and interleaved across lanes; an index
    outside the set rejects its lane only (its msg status still written) and sets the KEY_INDEX flag"""
    kinds = keys_with_secrets()
    ax, ay = pack([k[1][0] for k in kinds]), pack([k[1][1] for k in kinds])
    assert emu.emu_keyset_create(ctypes.c_size_t(len(kinds)), _p(ax), _p(ay)) == 0
    rnd = random.Random(99)
    lanes = [(j, c) for j, (_, pk, a) in enumerate(kinds) for c in schnorr_cases(rnd, pk, a)]
    rnd.shuffle(lanes)
    idx = np.array([j for j, _ in lanes], np.uint32)
    cases = [c for _, c in lanes]
    want = [oracle_case(kinds[j][1], c) for j, c in lanes]
    for bad in (False, True):
        ki = idx.copy()
        w = list(want)
        if bad:
            picks = [0, 5] + [i for i, c in enumerate(cases) if c[2] > Q][:1]
            ki[picks] = [len(kinds), 0xFFFFFFFF, len(kinds) + 3][:len(picks)]
            for i in picks:
                w[i] = (0, w[i][1])
        n = len(cases)
        ins = case_arrays(cases, 40)
        ok, st = np.full(n, 0xEE, np.uint8), np.full(n, 0xEE, np.uint8)
        s_red = np.zeros((n, 32), np.uint8)
        flags = emu.emu_verify_schnorr_keyset(ctypes.c_size_t(n), _p(u32(ki)), *[_p(v) for v in ins], 40, _p(ok), _p(st), _p(s_red))
        assert flags == (2 if bad else 0)
        check_emu_outputs(cases, w, ok, st, s_red, [c[2] <= Q and ki[i] < len(kinds) for i, c in enumerate(cases)])


def test_python_argument_handling():
    import babyjubjub_rs_b200 as bjj
    pt = bjj.Point(1, 2)
    m, rx, ry, s, words = bjj._schnorr_sigs([5, Q + 1], [(pt, 3), ((7, 8), (1 << 1100) + 1)])
    assert words == 40 and s.shape == (2, 160) and unpack(m) == [5, MASK] and unpack(rx) == [1, 7] and unpack(ry) == [2, 8]
    assert bjj._schnorr_sigs([0], [(pt, -(1 << 300))])[4] == 16           # the sign of s is dropped
    assert bjj._schnorr_sigs([0], [(pt, (1 << 2304) - 1)])[4] == 72
    for msgs, sigs in (([0], [(pt, 1 << 2304)]), ([-1], [(pt, 1)]), ([0, 1], [(pt, 1)])):
        with pytest.raises(ValueError):
            bjj._schnorr_sigs(msgs, sigs)
    got = bjj._schnorr_results(np.array([1, 0, 0], np.uint8), np.array([0, 0, 4], np.uint8))
    assert got[:2] == [True, False] and isinstance(got[2], ValueError) and str(got[2]) == "msg outside the Finite Field"


def build_cpp(out_dir):
    exe = os.path.join(str(out_dir), "test_verify_schnorr_comb")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-pthread", "-o", exe, CPP_SRC, "-L" + PKG, "-lbjj_cuda",
                           "-Wl,-rpath," + PKG])
    return exe


def test_cpp_builds_and_links(tmp_path):
    assert os.path.exists(build_cpp(tmp_path))


# ---- GPU ----------------------------------------------------------------------------------------------
class Forms:
    """the three forms over one set of keys: a FixedBase for `one` (or None), a key set of `keys` and the keys per lane"""

    def __init__(self, lib, ctx, keys_xy):
        self.lib, self.ctx = lib, ctx
        self.ax, self.ay = keys_xy
        st = np.zeros(len(self.ax), np.uint8)
        h = ctypes.c_void_p()
        assert lib.bjj_keyset_create(ctx, len(self.ax), _p(self.ax), _p(self.ay), _p(st), ctypes.byref(h)) == 0
        self.ks = h
        self.bases = {}

    def base(self, j):
        if j not in self.bases:
            h = ctypes.c_void_p()
            assert self.lib.bjj_base_create(self.ctx, _p(self.ax[j:j + 1]), _p(self.ay[j:j + 1]), ctypes.byref(h)) == 0
            self.bases[j] = h
        return self.bases[j]

    def close(self):
        self.lib.bjj_keyset_destroy(self.ctx, self.ks)
        for h in self.bases.values():
            self.lib.bjj_base_destroy(self.ctx, h)

    def run(self, form, idx, ins, words, dev, rc=0, sync_rc=0):
        """form in (base, keyset, wide); ins = [msg, rx, ry, s]; the base form needs one key index in idx -> ok, status"""
        lib, ctx = self.lib, self.ctx
        n = len(idx)
        ok, st = np.full(n, 0xEE, np.uint8), np.full(n, 0xEE, np.uint8)
        fn = getattr(lib, "bjj_verify_schnorr_%s_batch%s" % (form, "_dev" if dev else ""))
        if form == "base":
            assert n == 0 or len(set(idx.tolist())) == 1
            head_arrs, head = [], [self.base(int(idx[0]) if n else 0)]
        elif form == "keyset":
            head_arrs, head = [u32(idx)], [self.ks]
        else:
            head_arrs, head = [self.ax[idx], self.ay[idx]], []
        arrs = head_arrs + ins
        if not dev:
            got = fn(ctx, *head, n, *[_p(a) for a in arrs], words, _p(ok), _p(st))
        else:
            bufs = [lib.bjj_dev_alloc(ctx, max(a.nbytes, 1)) for a in arrs + [ok, st]]
            try:
                assert all(bufs)
                for b, a in zip(bufs, arrs):
                    assert lib.bjj_memcpy_h2d(ctx, b, _p(a), a.nbytes) == 0
                got = fn(ctx, *head, n, *bufs[:len(arrs)], words, bufs[-2], bufs[-1], None)
                assert lib.bjj_memcpy_d2h(ctx, _p(ok), bufs[-2], n) == 0
                assert lib.bjj_memcpy_d2h(ctx, _p(st), bufs[-1], n) == 0
                assert lib.bjj_sync(ctx) == sync_rc
            finally:
                for b in bufs:
                    lib.bjj_dev_free(ctx, b)
        assert got == rc, (form, dev, got)
        return ok, st


def reference_ok(eng, idx, ax, ay, ins, words):
    """bjj_verify_schnorr_batch with s reduced mod SUBORDER on the host"""
    raw = ins[3].tobytes()
    w = 4 * words
    s = pack([int.from_bytes(raw[w * i:w * (i + 1)], "little") % SUBORDER for i in range(len(idx))])
    return eng.verify_schnorr_batch(ax[idx], ay[idx], ins[0], ins[1], ins[2], s)


def signed_lanes(eng, n, n_keys, seed, corrupt=0.1):
    """n Schnorr signatures made by sign_schnorr_batch with seeded 1024-bit nonces (s: 40 words), a seeded random key per
    lane, about `corrupt` of them corrupted (s, r or msg) -> idx, [msg, rx, ry, s], (ax, ay)"""
    rng = np.random.default_rng(seed)
    priv = rng.integers(0, 256, size=(n_keys, 32), dtype=np.uint8)
    ax, ay = eng.public_batch(priv)
    idx = rng.integers(0, n_keys, size=n).astype(np.uint32)
    msgs = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    msgs[:, 31] &= 0x2F                                    # < Q
    nonces = rng.integers(0, 256, size=(n, 128), dtype=np.uint8)
    rx, ry, s, st = eng.sign_schnorr_batch(priv[idx], msgs, nonces, 32)
    assert not st.any() and s.shape == (n, 160)
    lanes = rng.permutation(n)[:int(n * corrupt)]
    for j, i in enumerate(lanes):
        if j % 3 == 0:
            s[i, rng.integers(0, 160)] ^= 1 << int(rng.integers(0, 8))
        elif j % 3 == 1:
            msgs[i, rng.integers(0, 31)] ^= 1 << int(rng.integers(0, 8))
        else:
            rx[i, 0] ^= 1                                  # r off the curve (mostly)
    return idx, [msgs, rx, ry, s], (ax, ay)


@pytest.mark.gpu
def test_against_oracle_every_form_and_width(gpu):
    """every key kind, torsion keys included: the three forms in both flavours against the oracle at s_words in
    {8, 16, 40, 72} (each case at every width that holds its s), status codes included"""
    eng = gpu.eng
    kinds = keys_with_secrets()
    forms = Forms(eng.lib, eng.ctx, (pack([k[1][0] for k in kinds]), pack([k[1][1] for k in kinds])))
    try:
        rnd = random.Random(100)
        per_kind = []
        for j, (_, pk, a) in enumerate(kinds):
            cases = schnorr_cases(rnd, pk, a) + [c for w in (8, 16, 40, 72) for c in width_cases(rnd, pk, a, w)]
            per_kind.append([(j, c, oracle_case(pk, c)) for c in cases])
        for words in (8, 16, 40, 72):
            fit = [[x for x in lanes if x[1][1] < 1 << (32 * words)] for lanes in per_kind]
            for dev in (False, True):
                for j, lanes in enumerate(fit):
                    idx = np.full(len(lanes), j, np.uint32)
                    ok, st = forms.run("base", idx, case_arrays([x[1] for x in lanes], words), words, dev)
                    assert list(ok) == [x[2][0] for x in lanes] and list(st) == [x[2][1] for x in lanes], (kinds[j][0], words, dev)
                allx = [x for lanes in fit for x in lanes]
                random.Random(words).shuffle(allx)
                idx = np.array([x[0] for x in allx], np.uint32)
                ins = case_arrays([x[1] for x in allx], words)
                for form in ("keyset", "wide"):
                    ok, st = forms.run(form, idx, ins, words, dev)
                    assert list(ok) == [x[2][0] for x in allx], (form, words, dev)
                    assert list(st) == [x[2][1] for x in allx], (form, words, dev)
    finally:
        forms.close()


@pytest.mark.gpu
def test_sign_then_verify_on_the_device(gpu):
    """bjj_sign_schnorr_batch_dev's output fed unchanged to the three _dev forms: ok = 1 on every lane; with 10 % of the
    lanes corrupted, ok equals bjj_verify_schnorr_batch on host-reduced s on every lane"""
    eng = gpu.eng
    lib, ctx = eng.lib, eng.ctx
    n, n_keys = 1 << 16, 1000
    rng = np.random.default_rng(101)
    priv = rng.integers(0, 256, size=(n_keys, 32), dtype=np.uint8)
    ax, ay = eng.public_batch(priv)
    idx = rng.integers(0, n_keys, size=n).astype(np.uint32)
    msgs = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    msgs[:, 31] &= 0x2F
    nonces = rng.integers(0, 256, size=(n, 128), dtype=np.uint8)
    forms = Forms(lib, ctx, (ax, ay))
    sizes = {"key": 32 * n, "msg": 32 * n, "nonce": 128 * n, "rx": 32 * n, "ry": 32 * n, "s": 160 * n, "st": n, "idx": 4 * n,
             "pkx": 32 * n, "pky": 32 * n, "ok": n, "vst": n}
    d = {k: lib.bjj_dev_alloc(ctx, v) for k, v in sizes.items()}
    try:
        assert all(d.values())
        for k, a in (("key", priv[idx]), ("msg", msgs), ("nonce", nonces), ("idx", u32(idx)), ("pkx", ax[idx]), ("pky", ay[idx])):
            a = np.ascontiguousarray(a)
            assert lib.bjj_memcpy_h2d(ctx, d[k], _p(a), a.nbytes) == 0
        assert lib.bjj_sign_schnorr_batch_dev(ctx, n, d["key"], d["msg"], d["nonce"], 32, d["rx"], d["ry"], d["s"], d["st"], None) == 0
        base = forms.base(0)
        sig_in = (d["msg"], d["rx"], d["ry"], d["s"])
        calls = {
            "keyset": lambda: lib.bjj_verify_schnorr_keyset_batch_dev(ctx, forms.ks, n, d["idx"], *sig_in, 40, d["ok"], d["vst"], None),
            "wide": lambda: lib.bjj_verify_schnorr_wide_batch_dev(ctx, n, d["pkx"], d["pky"], *sig_in, 40, d["ok"], d["vst"], None),
        }
        for name, call in calls.items():
            assert call() == 0
            ok, st = np.zeros(n, np.uint8), np.full(n, 0xEE, np.uint8)
            assert lib.bjj_memcpy_d2h(ctx, _p(ok), d["ok"], n) == 0
            assert lib.bjj_memcpy_d2h(ctx, _p(st), d["vst"], n) == 0
            assert lib.bjj_sync(ctx) == 0
            assert ok.all() and not st.any(), name
        # the base form on the lanes of key 0, gathered on the device by the keyset form's own inputs
        sel = np.flatnonzero(idx == 0)
        rx, ry, s = np.zeros((n, 32), np.uint8), np.zeros((n, 32), np.uint8), np.zeros((n, 160), np.uint8)
        for a, k in ((rx, "rx"), (ry, "ry"), (s, "s")):
            assert lib.bjj_memcpy_d2h(ctx, _p(a), d[k], a.nbytes) == 0
        assert lib.bjj_sync(ctx) == 0
        ok, st = forms.run("base", idx[sel], [msgs[sel], rx[sel], ry[sel], s[sel]], 40, True)
        assert ok.all() and not st.any()
    finally:
        for b in d.values():
            lib.bjj_dev_free(ctx, b)
    idx, ins, (ax, ay) = signed_lanes(eng, n, n_keys, 102)
    want = reference_ok(eng, idx, ax, ay, ins, 40)
    assert 0.85 * n < want[0].sum() < 0.95 * n
    forms2 = Forms(lib, ctx, (ax, ay))
    try:
        for form in ("keyset", "wide"):
            for dev in (False, True):
                ok, st = forms2.run(form, idx, ins, 40, dev)
                assert np.array_equal(ok, want[0]) and not st.any(), (form, dev)
        sel = np.flatnonzero(idx == 7)
        ok, st = forms2.run("base", idx[sel], [a[sel] for a in ins], 40, False)
        assert np.array_equal(ok, want[0][sel])
    finally:
        forms2.close()
        forms.close()


@pytest.mark.gpu
def test_chunk_and_subbatch_boundaries(gpu):
    """2^21 + 5 lanes of 300 keys: the host flavour runs three chunks, _dev two sub-batches, every form equal to
    bjj_verify_schnorr_batch on host-reduced s; launches per sub-batch (and per chunk) 2 (base), 2 (keyset) and
    1 + 3 (wide), also at 1,000 lanes"""
    eng = gpu.eng
    lib, ctx = eng.lib, eng.ctx
    idx, ins, (ax, ay) = signed_lanes(eng, BIG, 300, 103)
    want, _ = reference_ok(eng, idx, ax, ay, ins, 40)
    idx_one, ins_one, (ax1, ay1) = signed_lanes(eng, BIG, 1, 108)
    want1, _ = reference_ok(eng, idx_one, ax1, ay1, ins_one, 40)
    forms = Forms(lib, ctx, (ax, ay))
    one = Forms(lib, ctx, (ax1, ay1))
    one.base(0)                                            # the table is built before any launch is counted

    def launches(fn):
        before = lib.bjj_kernel_launches(ctx)
        r = fn()
        return r, lib.bjj_kernel_launches(ctx) - before
    try:
        for dev in (False, True):
            for form, per in (("base", 2), ("keyset", 2), ("wide", 4)):
                f = one if form == "base" else forms
                src_idx, src = (idx_one, ins_one) if form == "base" else (idx, ins)
                _, k = launches(lambda: f.run(form, src_idx[:1000], [a[:1000] for a in src], 40, dev))
                assert k == per, (form, dev, k)
                (ok, st), k = launches(lambda: f.run(form, src_idx, src, 40, dev))
                assert k == per * (2 if dev else 3), (form, dev, k)
                assert not st.any()
                assert np.array_equal(ok, want1 if form == "base" else want), (form, dev)
    finally:
        forms.close()
        one.close()


@pytest.mark.gpu
def test_argument_errors(gpu):
    """bad s_words (0, 4, 12, 80), NULL or foreign handles, NULL pointers and n = 0 in both flavours of every form"""
    bjj, eng = gpu.bjj, gpu.eng
    lib, ctx = eng.lib, eng.ctx
    good = [O.public(KEY_KAT), O.B8]
    ax, ay = pack([p[0] for p in good]), pack([p[1] for p in good])
    forms = Forms(lib, ctx, (ax, ay))
    other = bjj.Engine(0)
    foreign = Forms(other.lib, other.ctx, (ax, ay))
    try:
        fb = foreign.base(0)
        mine = forms.base(0)
        i4, a32, s = np.zeros(4, np.uint32), pack([1] * 4), np.zeros((4, 4 * 72), np.uint8)
        o = np.zeros(4, np.uint8)
        for dev in (False, True):
            sfx, tail = ("_dev", (None,)) if dev else ("", ())
            base = getattr(lib, "bjj_verify_schnorr_base_batch" + sfx)
            kset = getattr(lib, "bjj_verify_schnorr_keyset_batch" + sfx)
            wide = getattr(lib, "bjj_verify_schnorr_wide_batch" + sfx)
            for w in (0, 4, 12, 80, -8):
                assert base(ctx, mine, 4, _p(a32), _p(a32), _p(a32), _p(s), w, _p(o), _p(o), *tail) == ERR_ARG
                assert kset(ctx, forms.ks, 4, _p(i4), _p(a32), _p(a32), _p(a32), _p(s), w, _p(o), _p(o), *tail) == ERR_ARG
                assert wide(ctx, 4, _p(a32), _p(a32), _p(a32), _p(a32), _p(a32), _p(s), w, _p(o), _p(o), *tail) == ERR_ARG
            for h in (None, fb):
                assert base(ctx, h, 4, _p(a32), _p(a32), _p(a32), _p(s), 8, _p(o), _p(o), *tail) == ERR_ARG
            for h in (None, foreign.ks):
                assert kset(ctx, h, 4, _p(i4), _p(a32), _p(a32), _p(a32), _p(s), 8, _p(o), _p(o), *tail) == ERR_ARG
            assert base(ctx, mine, 4, _p(a32), _p(a32), _p(a32), _p(s), 8, _p(o), None, *tail) == ERR_ARG
            assert kset(ctx, forms.ks, 4, None, _p(a32), _p(a32), _p(a32), _p(s), 8, _p(o), _p(o), *tail) == ERR_ARG
            assert wide(ctx, 4, None, _p(a32), _p(a32), _p(a32), _p(a32), _p(s), 8, _p(o), _p(o), *tail) == ERR_ARG
            assert wide(None, 4, _p(a32), _p(a32), _p(a32), _p(a32), _p(a32), _p(s), 8, _p(o), _p(o), *tail) == ERR_ARG
            assert base(ctx, mine, 0, _p(a32), _p(a32), _p(a32), _p(s), 8, _p(o), _p(o), *tail) == 0
            assert kset(ctx, forms.ks, 0, _p(i4), _p(a32), _p(a32), _p(a32), _p(s), 8, _p(o), _p(o), *tail) == 0
            assert wide(ctx, 0, _p(a32), _p(a32), _p(a32), _p(a32), _p(a32), _p(s), 8, _p(o), _p(o), *tail) == 0
    finally:
        forms.close()
        foreign.close()
        other.close()


@pytest.mark.gpu
def test_key_index_and_noncanonical_r(gpu):
    """key_index >= n_keys: ok = 0 on that lane only (its msg status still written), BJJ_ERR_ARG from the host flavour
    and from bjj_sync after a _dev call, the next call clean; an r coordinate >= Q: BJJ_ERR_NONCANONICAL with the
    results of the batch computed mod Q, in every form"""
    eng = gpu.eng
    lib, ctx = eng.lib, eng.ctx
    n = 4096
    idx, ins, (ax, ay) = signed_lanes(eng, n, 17, 104)
    ins[0][9] = np.frombuffer((Q + 1).to_bytes(32, "little"), np.uint8)       # msg > Q
    want, want_st = reference_ok(eng, idx, ax, ay, ins, 40)
    assert want_st[9] == MSG_RANGE
    forms = Forms(lib, ctx, (ax, ay))
    try:
        bad = idx.copy()
        bad[[3, 9, 100, n - 1]] = [17, 5000, 0xFFFFFFFF, 1000]
        w2 = want.copy()
        w2[[3, 9, 100, n - 1]] = 0
        for dev in (False, True):
            rc_call, rc_sync = (0, ERR_ARG) if dev else (ERR_ARG, 0)
            ok, st = forms.run("keyset", bad, ins, 40, dev, rc_call, rc_sync)
            assert np.array_equal(ok, w2) and np.array_equal(st, want_st), dev
            ok, st = forms.run("keyset", idx, ins, 40, dev)
            assert np.array_equal(ok, want) and np.array_equal(st, want_st), dev
        nc = [a.copy() for a in ins]
        for i in (3, 4):
            x = unpack(nc[1][i:i + 1])[0]
            if x + Q <= MASK:
                nc[1][i] = pack([x + Q])[0]
        assert any(unpack(nc[1])[i] >= Q for i in (3, 4))
        sel = np.flatnonzero(idx == idx[3])
        for form, fi, fins, fw in (("keyset", idx, nc, want), ("wide", idx, nc, want),
                                   ("base", idx[sel], [a[sel] for a in nc], want[sel])):
            for dev in (False, True):
                rc_call, rc_sync = (0, ERR_NONCANONICAL) if dev else (ERR_NONCANONICAL, 0)
                ok, _ = forms.run(form, fi, fins, 40, dev, rc_call, rc_sync)
                assert np.array_equal(ok, fw), (form, dev)
    finally:
        forms.close()


@pytest.mark.gpu
def test_after_verify_batch_with_exact_lanes(gpu):
    """verify_batch with many off-curve lanes (its exact kernel runs deferred on the workspace's side stream), then at
    once each form on the same context: all correct, in both flavours"""
    eng = gpu.eng
    lib, ctx = eng.lib, eng.ctx
    n = (1 << 20) + 3
    rng = np.random.default_rng(105)
    priv = rng.integers(0, 256, size=(64, 32), dtype=np.uint8)
    vidx = rng.integers(0, 64, size=n)
    vmsg = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    vmsg[:, 31] &= 0x2F
    r8x, r8y, s32, _ = eng.sign_batch(priv[vidx], vmsg)
    r8x[::20, 0] ^= 1                                      # 5 % off the curve: exact lanes
    pax, pay = eng.public_batch(priv)
    vwant = eng.verify_batch(r8x, r8y, s32, pax[vidx], pay[vidx], vmsg)
    idx, ins, (ax, ay) = signed_lanes(eng, n, 64, 106)
    want, _ = reference_ok(eng, idx, ax, ay, ins, 40)
    forms = Forms(lib, ctx, (ax, ay))
    varrs = [r8x, r8y, s32, np.ascontiguousarray(pax[vidx]), np.ascontiguousarray(pay[vidx]), vmsg]
    vb = [lib.bjj_dev_alloc(ctx, a.nbytes) for a in varrs]
    okv = lib.bjj_dev_alloc(ctx, n)
    try:
        for b, a in zip(vb, varrs):
            assert lib.bjj_memcpy_h2d(ctx, b, _p(a), a.nbytes) == 0
        for form in ("keyset", "wide"):
            for dev in (False, True):
                assert lib.bjj_verify_batch_dev(ctx, n, *vb, okv, None) == 0
                ok, st = forms.run(form, idx, ins, 40, dev)
                got_v = np.zeros(n, np.uint8)
                assert lib.bjj_memcpy_d2h(ctx, _p(got_v), okv, n) == 0
                assert lib.bjj_sync(ctx) == 0
                assert np.array_equal(got_v, vwant) and np.array_equal(ok, want), (form, dev)
    finally:
        for b in vb + [okv]:
            lib.bjj_dev_free(ctx, b)
        forms.close()


@pytest.mark.gpu
def test_python_and_cpp_mirrors(gpu, tmp_path):
    bjj, eng = gpu.bjj, gpu.eng
    keys = [KEY_KAT, bytes(range(32)), bytes(range(1, 33))]
    pks = [bjj.Point(*O.public(k)) for k in keys]
    idx = [0, 1, 2, 0, 1, 2, 1, 0]
    msgs = [12345, 0, Q, 99, 7, 8, 9, 10]
    rnd = random.Random(107)
    sigs = bjj.sign_schnorr_batch([keys[j] for j in idx], msgs, [rnd.getrandbits(1024) for _ in idx], engine=eng)
    sigs[3] = (sigs[3][0], sigs[3][1] + 1)                         # wrong s
    sigs[4] = (sigs[4][0], sigs[4][1] + (SUBORDER << 1500))        # wider s, same group element
    sigs[5] = (sigs[5][0], sigs[5][1] % SUBORDER)                  # reduced s
    msgs[6] = Q + 1                                                # Err
    got = bjj.verify_schnorr_batch([pks[j] for j in idx], msgs, sigs, engine=eng)
    assert got[:6] + got[7:] == [True, True, True, False, True, True, True]
    assert isinstance(got[6], ValueError) and str(got[6]) == "msg outside the Finite Field"
    for i in (0, 3, 4):
        assert got[i] == bjj.verify_schnorr(pks[idx[i]], msgs[i], sigs[i][0], sigs[i][1])
    ks = bjj.KeySet(pks, eng)
    base = bjj.FixedBase(pks[0], eng)
    try:
        kgot = bjj.verify_schnorr_keyset_batch(ks, idx, msgs, sigs)
        assert [str(v) if isinstance(v, ValueError) else v for v in kgot] == [str(v) if isinstance(v, ValueError) else v for v in got]
        sel = [i for i, j in enumerate(idx) if j == 0]
        assert bjj.verify_schnorr_base_batch(base, [msgs[i] for i in sel], [sigs[i] for i in sel]) == [got[i] for i in sel]
        assert bjj.verify_schnorr_keyset_batch(ks, [], [], []) == []
        with pytest.raises(bjj.BjjError) as e:
            bjj.verify_schnorr_keyset_batch(ks, [0, 3], msgs[:2], sigs[:2])
        assert e.value.code == ERR_ARG
        with pytest.raises(ValueError):
            bjj.verify_schnorr_base_batch(None, msgs[:1], sigs[:1], engine=eng)
    finally:
        ks.close()
        base.close()
    out = subprocess.run([build_cpp(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "verify_schnorr comb ok" in out.stdout
