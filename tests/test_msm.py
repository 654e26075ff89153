"""bjj_msm_batch: R = sum_i k_i * P_i by bucket accumulation.  CPU: the lane bodies of msm.cuh compiled for the host
(digits of both window widths, runs split across threads and merged, the bucket reduction, the whole pipeline) against
the oracle's fold; the Python mirror's scalar mapping.  GPU: both flavours bit for bit against the fold on crafted
points and scalars, large n by linearity, extreme digit distributions, errors, launch counts, multi-device, C++."""
import ctypes
import os
import random
import subprocess
import time

import numpy as np
import pytest

from common import ROOT, pack, unpack
from oracle import bjj_oracle as O

Q, ORDER, SUBORDER = O.Q, O.ORDER, O.SUBORDER
IDENTITY = (0, 1)
ERR_ARG, ERR_NONCANONICAL = 2, 3
C16_POINTS = 1 << 20                  # bjj_cuda.cu: BJJ_MSM_C16_POINTS
DIGIT_EDGES = [0, 1, SUBORDER, ORDER - 1, ORDER, ORDER + 1, 1 << 255, (1 << 256) - 1, int("80" * 32, 16),
               int("8000" * 16, 16), int("7f" * 32, 16), int("7fff" * 16, 16), int("ff" * 31 + "7f", 16),
               int("7f" * 31 + "80", 16)]
CPP_SRC = os.path.join(ROOT, "tests", "cpp", "test_msm.cpp")
PKG = os.path.join(ROOT, "babyjubjub-rs_b200")


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def add(p, q):
    return O.proj_affine(O.proj_add(p + (1,), q + (1,)))


def neg(p):
    return ((Q - p[0]) % Q, p[1])


def fold(points, scalars):
    """the reference's composition: acc = (0 : 1 : 1); acc = acc.add(P_i.mul_scalar(k_i).projective()); acc.affine()"""
    acc = (0, 1, 1)
    for p, k in zip(points, scalars):
        acc = O.proj_add(acc, O.mul_scalar(p, k) + (1,))
    return O.proj_affine(acc)


def torsion_points():
    """points of order 2, 4 and 8"""
    t2 = (0, Q - 1)
    t4 = (O.modsqrt(pow(O.A, Q - 2, Q), Q), 0)
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


def crafted(rnd):
    """(points, scalars): torsion points, multiples of B8 with and without torsion, P next to -P, a point repeated, and
    the scalar edges"""
    t2, t4, t8 = torsion_points()
    b = [O.mul_scalar(O.B8, rnd.randrange(1, SUBORDER)) for _ in range(4)]
    pts = [IDENTITY, t2, t4, t8, O.B8, b[0], add(b[1], t8), add(b[2], t4), b[3], neg(b[3]), b[0], b[0]]
    ks = list(DIGIT_EDGES)
    while len(ks) < len(pts):
        ks.append(rnd.getrandbits(256))
    pts = (pts * ((len(ks) + len(pts) - 1) // len(pts)))[:max(len(pts), len(ks))]
    ks = (ks * ((len(pts) + len(ks) - 1) // len(ks)))[:len(pts)]
    return pts, ks


def arrays(points, scalars):
    return (pack([p[0] for p in points]), pack([p[1] for p in points]), pack(scalars))


# ---- CPU: msm.cuh on the host -------------------------------------------------------------------------------------

@pytest.fixture(scope="session")
def emu(tmp_path_factory):
    from common import build_hostemu
    build_hostemu()                     # generates the constants header the device sources include
    so = str(tmp_path_factory.mktemp("msm_emu") / "libbjj_msm_emu.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, os.path.join(ROOT, "tests", "hostemu", "msm_emu.cpp")])
    lib = ctypes.CDLL(so)
    lib.emu_msm_digits.restype = ctypes.c_int
    lib.emu_msm_digits.argtypes = [ctypes.c_int, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p]
    lib.emu_msm.restype = ctypes.c_uint32
    lib.emu_msm.argtypes = [ctypes.c_int, ctypes.c_size_t, ctypes.c_size_t] + [ctypes.c_void_p] * 7
    lib.emu_msm_bucket_reduce.argtypes = [ctypes.c_int] + [ctypes.c_void_p] * 4
    return lib


def emu_msm(emu, bits, points, scalars, chunk=0):
    px, py, k = arrays(points, scalars) if points else (np.zeros((1, 32), np.uint8),) * 3
    rx, ry = np.zeros((1, 32), np.uint8), np.zeros((1, 32), np.uint8)
    st = np.full(max(len(points), 1), 0xEE, np.uint8)
    levels = ctypes.c_int()
    flags = emu.emu_msm(bits, len(points), chunk, _p(px), _p(py), _p(k), _p(rx), _p(ry), _p(st), ctypes.byref(levels))
    return (unpack(rx)[0], unpack(ry)[0]), flags, st[:len(points)], levels.value


@pytest.mark.parametrize("bits", [8, 16])
def test_hostemu_digits_recompose(emu, bits):
    """the signed digits, carry window included, give k back: sum_w d_w 2^(c w) == k, |d_w| <= 2^(c-1)"""
    rnd = random.Random(bits)
    ks = DIGIT_EDGES + [rnd.getrandbits(256) for _ in range(200)]
    windows = 256 // bits + 1
    d = np.zeros((len(ks), windows), np.int32)
    assert emu.emu_msm_digits(bits, len(ks), _p(pack(ks)), _p(d)) == windows
    for k, row in zip(ks, d.tolist()):
        assert sum(v << (bits * w) for w, v in enumerate(row)) == k
        assert all(-(1 << (bits - 1)) <= v < (1 << (bits - 1)) for v in row[:-1]) and row[-1] in (0, 1)
    top = ks.index((1 << 256) - 1)
    assert d[top].tolist()[-1] == 1                     # 2^256 - 1 carries into the last window
    assert d[ks.index(0)].tolist() == [0] * windows


@pytest.mark.parametrize("bits", [8, 16])
def test_hostemu_crafted_against_fold(emu, bits):
    pts, ks = crafted(random.Random(5 + bits))
    r, flags, st, _ = emu_msm(emu, bits, pts, ks)
    assert flags == 0 and not st.any()
    assert r == fold(pts, ks)


@pytest.mark.parametrize("bits,n", [(8, 1), (8, 2), (8, 33), (16, 3), (8, 1000), (16, 1000)])
def test_hostemu_random_against_fold(emu, bits, n):
    rnd = random.Random(n * bits)
    base = [O.mul_scalar(O.B8, rnd.randrange(1, SUBORDER)) for _ in range(min(n, 40))]
    t8 = torsion_points()[2]
    pts = [add(base[i % len(base)], t8) if i % 3 == 0 else base[i % len(base)] for i in range(n)]
    ks = [rnd.getrandbits(256) for _ in range(n)]
    r, flags, _, _ = emu_msm(emu, bits, pts, ks)
    assert flags == 0
    want = fold(pts, ks)
    assert r == want
    assert emu_msm(emu, bits, pts, ks, chunk=97)[0] == want     # chunks into the same buckets


@pytest.mark.parametrize("bits", [8, 16])
def test_hostemu_one_bucket_split_across_runs_and_levels(emu, bits):
    """every scalar equal: each window's pairs fall into one bucket, which spans every run of the sorted list and is
    merged over several boundary levels"""
    rnd = random.Random(11)
    n = 1024
    pts = [O.mul_scalar(O.B8, rnd.randrange(1, SUBORDER)) for _ in range(8)] * (n // 8)
    k = rnd.getrandbits(256)
    r, flags, _, levels = emu_msm(emu, bits, pts, [k] * n)
    assert flags == 0 and levels >= 3
    acc = (0, 1, 1)
    for p in pts[:8]:
        acc = O.proj_add(acc, p + (1,))
    want = O.mul_scalar(O.proj_affine(acc), k * (n // 8))
    assert r == want
    # and the cancelling form: P and -P with equal scalars
    half = pts[:n // 2]
    assert emu_msm(emu, bits, half + [neg(p) for p in half], [k] * n)[0] == IDENTITY


def test_hostemu_empty_zero_and_errors(emu):
    assert emu_msm(emu, 8, [], [])[0] == IDENTITY
    pts, ks = crafted(random.Random(3))
    assert emu_msm(emu, 8, pts, [0] * len(pts))[0] == IDENTITY
    bad = list(pts)
    bad[5] = ((bad[5][0] + 1) % Q, bad[5][1])
    r, flags, st, _ = emu_msm(emu, 8, bad, ks)
    assert r == (0, 0) and flags & 4 and st.tolist() == [1 if i == 5 else 0 for i in range(len(pts))]
    # a coordinate >= Q: computed mod Q, status NONCANONICAL
    px, py, k = arrays(pts, ks)
    px[4] = pack([O.B8[0] + Q])[0]
    rx, ry = np.zeros((1, 32), np.uint8), np.zeros((1, 32), np.uint8)
    st = np.zeros(len(pts), np.uint8)
    lv = ctypes.c_int()
    flags = emu.emu_msm(8, len(pts), 0, _p(px), _p(py), _p(k), _p(rx), _p(ry), _p(st), ctypes.byref(lv))
    assert flags == 1 and st.tolist() == [2 if i == 4 else 0 for i in range(len(pts))]
    assert (unpack(rx)[0], unpack(ry)[0]) == fold(pts, ks)


def test_hostemu_bucket_reduction_against_direct_sum(emu):
    """W = sum_b b * B_b for one window of 2^7 buckets, computed directly by the oracle"""
    rnd = random.Random(19)
    t8 = torsion_points()[2]
    bk = [O.mul_scalar(O.B8, rnd.randrange(SUBORDER)) for _ in range(128)]
    bk[7] = add(bk[7], t8)
    bk[100] = IDENTITY
    rx, ry = np.zeros((1, 32), np.uint8), np.zeros((1, 32), np.uint8)
    emu.emu_msm_bucket_reduce(8, _p(pack([p[0] for p in bk])), _p(pack([p[1] for p in bk])), _p(rx), _p(ry))
    assert (unpack(rx)[0], unpack(ry)[0]) == fold(bk, range(1, 129))


def test_python_msm_scalar_mapping(monkeypatch):
    """msm drops the sign and reduces scalars of 256 bits and more mod ORDER only when they do not fit"""
    import babyjubjub_rs_b200 as bjj
    seen = {}

    class Fake:
        def msm_batch(self, px, py, k):
            seen["k"] = unpack(k)
            return np.zeros((1, 32), np.uint8), pack([1]), np.zeros(len(k), np.uint8)
    pts = [bjj.Point(*O.B8)] * 5
    ks = [-5, (1 << 256) - 1, 1 << 256, -(ORDER + 3), ORDER + 7 + (1 << 300)]
    r = bjj.msm(pts, ks, engine=Fake())
    assert (r.x, r.y) == IDENTITY
    assert seen["k"] == [5, (1 << 256) - 1, (1 << 256) % ORDER, ORDER + 3, (ORDER + 7 + (1 << 300)) % ORDER]
    with pytest.raises(ValueError):
        bjj.msm(pts, ks[:2], engine=Fake())


def build_cpp(out_dir):
    exe = os.path.join(str(out_dir), "test_msm")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-pthread", "-o", exe, CPP_SRC, "-L" + PKG, "-lbjj_cuda", "-Wl,-rpath," + PKG])
    return exe


def test_cpp_msm_builds_and_links(tmp_path):
    assert os.path.exists(build_cpp(tmp_path))


# ---- GPU ------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def eng():
    import babyjubjub_rs_b200 as bjj
    e = bjj.Engine(0)
    yield e
    e.close()


def call(eng, px, py, k, dev, status=True, rc=0):
    """bjj_msm_batch{,_dev}: ((x, y), status); `rc` the expected return (of bjj_sync for _dev)"""
    lib, ctx, n = eng.lib, eng.ctx, len(px)
    rx, ry = np.full((1, 32), 0xEE, np.uint8), np.full((1, 32), 0xEE, np.uint8)
    st = np.full(max(n, 1), 0xEE, np.uint8)
    if not dev:
        got = lib.bjj_msm_batch(ctx, n, _p(px), _p(py), _p(k), _p(rx), _p(ry), _p(st) if status else None)
        assert got == rc, got
    else:
        ins, outs = [px, py, k], [rx, ry] + ([st] if status else [])
        bufs = [lib.bjj_dev_alloc(ctx, max(a.nbytes, 1)) for a in ins + outs]
        try:
            assert all(bufs)
            for b, a in zip(bufs, ins):
                assert lib.bjj_memcpy_h2d(ctx, b, _p(a), a.nbytes) == 0
            assert lib.bjj_msm_batch_dev(ctx, n, *bufs[:3], bufs[3], bufs[4], bufs[5] if status else None, None) == 0
            for b, a in zip(bufs[3:], outs):
                assert lib.bjj_memcpy_d2h(ctx, _p(a), b, a.nbytes) == 0
            assert lib.bjj_sync(ctx) == rc
        finally:
            for b in bufs:
                lib.bjj_dev_free(ctx, b)
    return (unpack(rx)[0], unpack(ry)[0]), st[:n]


@pytest.mark.gpu
@pytest.mark.parametrize("dev", [False, True])
@pytest.mark.parametrize("n", [0, 1, 2, 3, 31, 32, 33, 1000])
def test_gpu_small_against_fold(eng, dev, n):
    rnd = random.Random(n)
    pts, ks = crafted(rnd)
    while len(pts) < n:
        more_p, more_k = crafted(rnd)
        pts, ks = pts + more_p, ks + more_k
    pts, ks = pts[:n], ks[:n]
    if n:
        r, st = call(eng, *arrays(pts, ks), dev)
        assert not st.any()
    else:
        z = np.zeros((0, 32), np.uint8)
        r, _ = call(eng, z, z, z, dev)
    assert r == fold(pts, ks)


def linear_inputs(eng, n, seed, same_scalar=False):
    """P_i = a_i * B8 + t_i * T8 made on the device; returns the arrays, and the expected sum
    (sum k_i a_i mod SUBORDER) * B8 + (sum k_i t_i mod 8) * T8"""
    import babyjubjub_rs_b200 as bjj
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    a[:, 31] &= 0x0F
    t = np.zeros((n, 32), np.uint8)
    t[:, 0] = rng.integers(0, 8, n, dtype=np.uint8)
    k = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    if same_scalar:
        k[:] = k[0]
    t8 = torsion_points()[2]
    tb = bjj.FixedBase(bjj.Point(*t8), eng)
    try:
        px, py = eng.base_mul2_batch(None, a, tb, t)
    finally:
        tb.close()
    ai, ti, ki = (unpack(v) for v in (a, t, k))
    sa = sum(x * y for x, y in zip(ki, ai)) % SUBORDER
    st = sum(x * y for x, y in zip(ki, ti)) % 8
    return (px, py, k), add(O.mul_scalar(O.B8, sa), O.mul_scalar(t8, st))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1 << 10, C16_POINTS - 1, C16_POINTS, C16_POINTS + 1, (1 << 21) + 1])
def test_gpu_large_by_linearity(eng, n):
    ins, want = linear_inputs(eng, n, n)
    assert call(eng, *ins, False, status=False)[0] == want
    assert call(eng, *ins, True, status=False)[0] == want


def timed(eng, ins):
    call(eng, *ins, True, status=False)
    t = time.perf_counter()
    r = call(eng, *ins, True, status=False)[0]
    return r, time.perf_counter() - t


@pytest.mark.gpu
def test_gpu_extreme_distributions(eng):
    """each checked for its result and for a time in line with random scalars"""
    n = 1 << 20
    ins, want = linear_inputs(eng, n, 1)
    r, t_rand = timed(eng, ins)
    assert r == want
    px, py, k = ins
    cases = []
    ins_eq, want_eq = linear_inputs(eng, n, 2, same_scalar=True)
    cases.append(("equal scalars", ins_eq, want_eq))
    cases.append(("zero scalars", (px, py, np.zeros_like(k)), IDENTITY))
    p0 = (unpack(px[:1])[0], unpack(py[:1])[0])
    kk = unpack(k)
    cases.append(("one point", (np.repeat(px[:1], n, 0), np.repeat(py[:1], n, 0), k), O.mul_scalar(p0, sum(kk) % ORDER)))
    ones = np.full_like(k, 0xFF)
    cases.append(("2^256 - 1", (px, py, ones), O.mul_scalar(fold_sum(eng, px, py), (1 << 256) - 1)))
    h = n // 2
    negx = pack([(Q - x) % Q for x in unpack(px[:h])])
    kh = np.concatenate([k[:h], k[:h]])
    cases.append(("P and -P", (np.concatenate([px[:h], negx]), np.concatenate([py[:h], py[:h]]), kh), IDENTITY))
    for name, c_ins, c_want in cases:
        r, t = timed(eng, c_ins)
        assert r == c_want, name
        assert t < 3 * t_rand + 0.05, (name, t, t_rand)


def fold_sum(eng, px, py):
    """sum of the points through msm with scalar 1 (checked against the fold at small n above)"""
    one = np.zeros_like(px)
    one[:, 0] = 1
    rx, ry, _ = eng.msm_batch(px, py, one)
    return (unpack(rx)[0], unpack(ry)[0])


@pytest.mark.gpu
@pytest.mark.parametrize("dev", [False, True])
def test_gpu_errors_and_recovery(eng, dev):
    n = 1 << 20
    ins, want = linear_inputs(eng, n, 3)
    px, py, k = (a.copy() for a in ins)
    px[12345, 0] ^= 1                                   # off the curve
    r, st = call(eng, px, py, k, dev, rc=ERR_ARG)
    assert r == (0, 0)
    assert st[12345] == 1 and np.count_nonzero(st) == 1
    assert call(eng, *ins, dev)[0] == want              # the next call is clean
    px, py, k = (a.copy() for a in ins)
    x = unpack(px[7:8])[0]
    px[7] = pack([x + Q])[0] if x + Q < (1 << 256) else px[7]
    r, st = call(eng, px, py, k, dev, rc=ERR_NONCANONICAL)
    assert r == want and st[7] == 2 and np.count_nonzero(st) == 1
    lib, z = eng.lib, np.zeros((1, 32), np.uint8)
    f = lib.bjj_msm_batch_dev if dev else lib.bjj_msm_batch
    tail = (None,) if dev else ()
    assert f(None, 1, _p(z), _p(z), _p(z), _p(z), _p(z), None, *tail) == ERR_ARG
    for i in range(5):
        args = [_p(z)] * 5
        args[i] = None
        assert f(eng.ctx, 1, *args, None, *tail) == ERR_ARG
    assert lib.bjj_sync(eng.ctx) == 0
    # verify_batch still gives its known answers
    from common import signature_cases, cases_to_arrays, oracle_verify
    cases = signature_cases(random.Random(4))
    ok = eng.verify_batch(*cases_to_arrays(cases))
    assert ok.tolist() == [1 if oracle_verify(c) else 0 for c in cases]


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1000, C16_POINTS + 1, (1 << 21) + 1])
def test_gpu_launch_counts_depend_on_n_only(eng, n):
    a, _ = linear_inputs(eng, n, 5)
    b = (a[0], a[1], np.zeros_like(a[2]))
    counts = []
    for ins in (a, b, a):
        before = eng.kernel_launches
        call(eng, *ins, False, status=False)
        counts.append(eng.kernel_launches - before)
    before = eng.kernel_launches
    call(eng, *a, True, status=False)
    d1 = eng.kernel_launches - before
    before = eng.kernel_launches
    call(eng, *b, True, status=False)
    assert counts[0] == counts[1] == counts[2] and d1 == eng.kernel_launches - before


@pytest.mark.gpu
def test_gpu_python_mirror(eng):
    import babyjubjub_rs_b200 as bjj
    pts, ks = crafted(random.Random(8))
    ks = ks + [-(ORDER + 5), 1 << 300]
    pts = pts + [O.B8, pts[5]]
    r = bjj.msm([bjj.Point(*p) for p in pts], ks, engine=eng)
    assert (r.x, r.y) == fold(pts, [abs(k) % ORDER if abs(k) >= (1 << 256) else abs(k) for k in ks])
    bad = [bjj.Point(1, 1)] + [bjj.Point(*p) for p in pts[1:]]
    with pytest.raises(bjj.BjjError) as e:
        bjj.msm(bad, ks, engine=eng)
    assert e.value.code == ERR_ARG and e.value.point_status[0] == 1


@pytest.mark.gpu
def test_gpu_multi_equals_single(eng):
    import babyjubjub_rs_b200 as bjj
    n = (1 << 20) + 3
    ins, want = linear_inputs(eng, n, 6)
    for g in range(1, eng.lib.bjj_device_count() + 1):
        m = bjj.MultiEngine(list(range(g)))
        try:
            rx, ry, st = m.msm_batch(*ins)
            assert (unpack(rx)[0], unpack(ry)[0]) == want, g
            assert not st.any()
            z = np.zeros((0, 32), np.uint8)
            rx, ry, _ = m.msm_batch(z, z, z)
            assert (unpack(rx)[0], unpack(ry)[0]) == IDENTITY
        finally:
            m.close()


@pytest.mark.gpu
def test_gpu_cpp_mirror(tmp_path):
    out = subprocess.run([build_cpp(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr
