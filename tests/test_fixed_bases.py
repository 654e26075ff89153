"""Fixed-base tables for caller-chosen points (bjj_base_*): k*P and k*P + l*Q on the comb path, both flavours, against
the oracle; error handling, handle lifetime, launch counts and the Python / C++ mirrors."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

from common import ROOT, pack, special_points, random_points, unpack
from oracle import bjj_oracle as O

ERR_ARG, ERR_NONCANONICAL = 2, 3
SCALAR_EDGES = [0, 1, O.SUBORDER - 1, O.SUBORDER, O.SUBORDER + 1, O.ORDER - 1, O.ORDER, 1 << 255, (1 << 256) - 1]
LANES = 4096
BIG = (1 << 21) + 5

CPP_SRC = os.path.join(ROOT, "tests", "cpp", "test_fixed_base.cpp")
CPP_EXE = os.path.join(ROOT, "tests", "cpp", "test_fixed_base")
PKG = os.path.join(ROOT, "babyjubjub-rs_b200")


def full_order_points(rnd, count):
    """on-curve points of order ORDER: decompressed from random y until SUBORDER*P has order 8"""
    out = []
    while len(out) < count:
        try:
            p = O.decompress_point(rnd.randrange(O.Q).to_bytes(32, "little"))
        except ValueError:
            continue
        t = O.mul_scalar(p, O.SUBORDER)
        if O.on_curve(p) and O.mul_scalar(t, 4) != (0, 1):
            out.append(p)
    return out


def scalars(rnd, n):
    return SCALAR_EDGES + [rnd.randrange(1 << 256) for _ in range(n - len(SCALAR_EDGES))]


def create(lib, ctx, p):
    h = ctypes.c_void_p()
    rc = lib.bjj_base_create(ctx, pack([p[0]]).ctypes.data_as(ctypes.c_void_p),
                             pack([p[1]]).ctypes.data_as(ctypes.c_void_p), ctypes.byref(h))
    return rc, h


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def run(lib, ctx, op, handles, ins, dev):
    """bjj_base_<op>_batch (host or _dev flavour) on (n, 32) input arrays -> (rc, rx, ry)"""
    n = len(ins[0])
    rx, ry = np.zeros((n, 32), np.uint8), np.zeros((n, 32), np.uint8)
    fn = getattr(lib, "bjj_base_%s_batch%s" % (op, "_dev" if dev else ""))
    if not dev:
        return fn(ctx, *handles, n, *[_p(a) for a in ins], _p(rx), _p(ry)), rx, ry
    bufs = [lib.bjj_dev_alloc(ctx, max(a.nbytes, 1)) for a in ins + [rx, ry]]
    try:
        assert all(bufs)
        for b, a in zip(bufs, ins):
            assert lib.bjj_memcpy_h2d(ctx, b, _p(a), a.nbytes) == 0
        rc = fn(ctx, *handles, n, *bufs, None)
        for b, a in zip(bufs[len(ins):], (rx, ry)):
            assert lib.bjj_memcpy_d2h(ctx, _p(a), b, a.nbytes) == 0
        assert lib.bjj_sync(ctx) == 0
    finally:
        for b in bufs:
            lib.bjj_dev_free(ctx, b)
    return rc, rx, ry


def oracle_mul(oracle_c, p, ks):
    n = len(ks)
    return oracle_c.mul_scalar(pack([p[0]] * n), pack([p[1]] * n), pack(ks))


def oracle_mul2(oracle_c, p, ks, q, ls):
    """(k*P).projective().add((l*Q).projective()).affine(), lane by lane"""
    a, b = oracle_mul(oracle_c, p, ks), oracle_mul(oracle_c, q, ls)
    out = [O.proj_affine(O.proj_add((x1, y1, 1), (x2, y2, 1)))
           for x1, y1, x2, y2 in zip(unpack(a[0]), unpack(a[1]), unpack(b[0]), unpack(b[1]))]
    return [pack([o[0] for o in out]), pack([o[1] for o in out])]


# ---- CPU ----------------------------------------------------------------------------------------------
def test_python_scalar_normalisation():
    import babyjubjub_rs_b200 as bjj
    f = bjj._base_scalar
    assert f(0) == 0 and f(-5) == 5 and f(O.ORDER + 3) == O.ORDER + 3
    assert f((1 << 256) - 1) == (1 << 256) - 1 and f(-((1 << 256) - 1)) == (1 << 256) - 1
    assert f(1 << 256) == (1 << 256) % O.ORDER
    assert f(-(3 << 300) - 7) == ((3 << 300) + 7) % O.ORDER


def build_cpp():
    deps = [CPP_SRC, os.path.join(ROOT, "host", "bjj.hpp"), os.path.join(ROOT, "include", "bjj_cuda.h")]
    if not os.path.exists(CPP_EXE) or any(os.path.getmtime(d) > os.path.getmtime(CPP_EXE) for d in deps):
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-pthread", "-o", CPP_EXE, CPP_SRC, "-L" + PKG, "-lbjj_cuda",
                               "-Wl,-rpath," + PKG])
    return CPP_EXE


def test_cpp_fixed_base_builds_and_links():
    assert os.path.exists(build_cpp())


# ---- GPU ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_cpp_fixed_base_runs():
    out = subprocess.run([build_cpp()], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "fixed base ok" in out.stdout


@pytest.mark.gpu
def test_base_mul_matches_oracle_both_flavours(gpu, oracle_c):
    lib, ctx = gpu.eng.lib, gpu.eng.ctx
    rnd = random.Random(11)
    on, _ = special_points()
    bases = on + random_points(rnd, 3) + full_order_points(rnd, 2)
    assert O.B8 in bases
    for p in bases:
        rc, h = create(lib, ctx, p)
        assert rc == 0 and h.value, p
        try:
            ks = scalars(rnd, LANES)
            want = oracle_mul(oracle_c, p, ks)
            for dev in (False, True):
                rc, rx, ry = run(lib, ctx, "mul", [h], [pack(ks)], dev)
                assert rc == 0
                assert np.array_equal(rx, want[0]) and np.array_equal(ry, want[1]), (p, dev)
        finally:
            lib.bjj_base_destroy(ctx, h)


@pytest.mark.gpu
def test_b8_anchor(gpu):
    lib, ctx = gpu.eng.lib, gpu.eng.ctx
    k = pack(scalars(random.Random(12), LANES))
    want = gpu.eng.fixed_base_batch(k)
    rc, h = create(lib, ctx, O.B8)
    assert rc == 0
    try:
        for handle in (None, h):
            for dev in (False, True):
                rc, rx, ry = run(lib, ctx, "mul", [handle], [k], dev)
                assert rc == 0 and np.array_equal(rx, want[0]) and np.array_equal(ry, want[1]), (handle, dev)
    finally:
        lib.bjj_base_destroy(ctx, h)


@pytest.mark.gpu
def test_base_mul2_matches_oracle(gpu, oracle_c):
    lib, ctx = gpu.eng.lib, gpu.eng.ctx
    rnd = random.Random(13)
    p, q = random_points(rnd, 2)
    t1, t2 = full_order_points(rnd, 2)
    x4 = special_points()[0][5]
    neg_p = ((O.Q - p[0]) % O.Q, p[1])
    pts = [p, q, neg_p, t1, t2, x4, O.B8]
    handles = {}
    try:
        for pt in pts:
            rc, handles[pt] = create(lib, ctx, pt)
            assert rc == 0
        handles[None] = None
        n = 512
        cases = [(p, q), (p, p), (p, None), (None, q), (None, None), (t1, t2), (t1, x4), (x4, None), (p, O.B8)]
        for a, b in cases:
            ks, ls = scalars(rnd, n), scalars(rnd, n)[::-1]
            want = oracle_mul2(oracle_c, a or O.B8, ks, b or O.B8, ls)
            for dev in (False, True):
                rc, rx, ry = run(lib, ctx, "mul2", [handles[a], handles[b]], [pack(ks), pack(ls)], dev)
                assert rc == 0
                assert np.array_equal(rx, want[0]) and np.array_equal(ry, want[1]), (a, b, dev)
        # Q = -P with k = l: the identity in every lane
        ks = scalars(rnd, n)
        for dev in (False, True):
            rc, rx, ry = run(lib, ctx, "mul2", [handles[p], handles[neg_p]], [pack(ks), pack(ks)], dev)
            assert rc == 0 and unpack(rx) == [0] * n and unpack(ry) == [1] * n
    finally:
        for h in handles.values():
            lib.bjj_base_destroy(ctx, h)


@pytest.mark.gpu
def test_errors_and_lifecycle(gpu, oracle_c):
    import babyjubjub_rs_b200 as bjj
    lib, ctx = gpu.eng.lib, gpu.eng.ctx
    rnd = random.Random(14)
    _, off = special_points()
    for p in off:
        rc, h = create(lib, ctx, p)
        assert rc == ERR_ARG and not h.value, p
    for p in ((O.B8[0] + O.Q, O.B8[1]), (0, 1 + O.Q), ((1 << 256) - 1, 1)):
        rc, h = create(lib, ctx, p)
        assert rc == ERR_NONCANONICAL and not h.value, p
    one = pack([1])
    h = ctypes.c_void_p()
    assert lib.bjj_base_create(None, _p(one), _p(one), ctypes.byref(h)) == ERR_ARG
    assert lib.bjj_base_create(ctx, None, _p(one), ctypes.byref(h)) == ERR_ARG
    assert lib.bjj_base_create(ctx, _p(one), _p(one), None) == ERR_ARG

    pts = random_points(rnd, 3)
    hs = [create(lib, ctx, p)[1] for p in pts]
    assert all(x.value for x in hs)
    k = pack(scalars(rnd, 64))
    out = np.zeros((64, 32), np.uint8)
    for dev in (False, True):
        sfx = "_dev" if dev else ""
        mul, mul2 = getattr(lib, "bjj_base_mul_batch" + sfx), getattr(lib, "bjj_base_mul2_batch" + sfx)
        tail = (None,) if dev else ()
        assert run(lib, ctx, "mul", [hs[0]], [k[:0]], dev)[0] == 0                   # n = 0
        assert run(lib, ctx, "mul2", [hs[0], None], [k[:0], k[:0]], dev)[0] == 0
        assert mul(None, hs[0], 64, _p(k), _p(out), _p(out), *tail) == ERR_ARG
        assert mul(ctx, hs[0], 64, None, _p(out), _p(out), *tail) == ERR_ARG
        assert mul(ctx, hs[0], 64, _p(k), _p(out), None, *tail) == ERR_ARG
        assert mul2(ctx, hs[0], None, 64, _p(k), None, _p(out), _p(out), *tail) == ERR_ARG
        assert mul2(ctx, None, hs[1], 64, _p(k), _p(k), None, _p(out), *tail) == ERR_ARG
    # a handle used with another context (both on device 0)
    other = bjj.Engine(0)
    try:
        for dev in (False, True):
            assert run(lib, other.ctx, "mul", [hs[0]], [k], dev)[0] == ERR_ARG
            assert run(lib, other.ctx, "mul2", [None, hs[1]], [k, k], dev)[0] == ERR_ARG
            assert run(lib, other.ctx, "mul2", [hs[1], None], [k, k], dev)[0] == ERR_ARG
        lib.bjj_base_destroy(other.ctx, hs[0])          # not its handle: left alone
    finally:
        other.close()
    # three handles coexist; destroying one leaves the others intact
    lib.bjj_base_destroy(ctx, hs[1])
    lib.bjj_base_destroy(ctx, None)
    ks = unpack(k)
    for p, h in ((pts[0], hs[0]), (pts[2], hs[2])):
        rc, rx, ry = run(lib, ctx, "mul", [h], [k], False)
        want = oracle_mul(oracle_c, p, ks)
        assert rc == 0 and np.array_equal(rx, want[0]) and np.array_equal(ry, want[1])
    lib.bjj_base_destroy(ctx, hs[0])
    lib.bjj_base_destroy(ctx, hs[2])


@pytest.mark.gpu
def test_boundaries_and_launch_counts(gpu, oracle_c):
    """2^21 + 5 lanes: the host flavour runs three chunks (2^18, 2^19, the rest), the _dev flavour two sub-batches"""
    lib, ctx = gpu.eng.lib, gpu.eng.ctx
    rnd = random.Random(15)
    p, q = random_points(rnd, 2)
    before = lib.bjj_kernel_launches(ctx)
    (rc1, hp), (rc2, hq) = create(lib, ctx, p), create(lib, ctx, q)
    assert rc1 == 0 and rc2 == 0 and lib.bjj_kernel_launches(ctx) - before == 2
    try:
        rng = np.random.default_rng(15)
        k = rng.integers(0, 256, size=(BIG, 32), dtype=np.uint8)
        l = rng.integers(0, 256, size=(BIG, 32), dtype=np.uint8)
        k[:len(SCALAR_EDGES)] = pack(SCALAR_EDGES)
        sample = sorted(set(rnd.sample(range(BIG), 4096)) | {0, 1, BIG - 1, (1 << 21) - 1, 1 << 21, (1 << 18) - 1, 1 << 18})
        for op, handles, ins in (("mul", [hp], [k]), ("mul2", [hp, hq], [k, l])):
            outs = {}
            for dev, want_launches in ((False, 6), (True, 4)):
                before = lib.bjj_kernel_launches(ctx)
                rc, rx, ry = run(lib, ctx, op, handles, ins, dev)
                assert rc == 0 and lib.bjj_kernel_launches(ctx) - before == want_launches, (op, dev)
                outs[dev] = (rx, ry)
                before = lib.bjj_kernel_launches(ctx)
                assert run(lib, ctx, op, handles, [a[:1000] for a in ins], dev)[0] == 0
                assert lib.bjj_kernel_launches(ctx) - before == 2, (op, dev)
            assert np.array_equal(outs[False][0], outs[True][0]) and np.array_equal(outs[False][1], outs[True][1]), op
            ks = unpack(k[sample])
            if op == "mul":
                want = oracle_mul(oracle_c, p, ks)
            else:
                want = oracle_mul2(oracle_c, p, ks, q, unpack(l[sample]))
            assert np.array_equal(outs[False][0][sample], want[0]) and np.array_equal(outs[False][1][sample], want[1]), op
    finally:
        lib.bjj_base_destroy(ctx, hp)
        lib.bjj_base_destroy(ctx, hq)


@pytest.mark.gpu
def test_python_mirror(gpu):
    import babyjubjub_rs_b200 as bjj
    rnd = random.Random(16)
    p, q = [bjj.Point(*pt) for pt in random_points(rnd, 1) + full_order_points(rnd, 1)]
    ks = [0, 1, -1, -O.ORDER, O.ORDER + 1, -(1 << 255), (1 << 256) - 1, 1 << 256, -(1 << 300) - 3, (5 << 1000) + 9]
    ks += [rnd.randrange(-(1 << 600), 1 << 600) for _ in range(40)]
    for pt in (p, q):
        want = bjj.mul_scalar_batch([pt] * len(ks), ks, engine=gpu.eng)
        base = bjj.FixedBase(pt, gpu.eng)
        try:
            assert base.mul_batch(ks) == want
        finally:
            base.close()
        assert bjj.mul_fixed_base_batch(pt, ks, engine=gpu.eng) == want
    ls = ks[::-1]
    got = bjj.mul2_fixed_base_batch(p, ks, q, ls, engine=gpu.eng)
    kp = bjj.mul_scalar_batch([p] * len(ks), ks, engine=gpu.eng)
    lq = bjj.mul_scalar_batch([q] * len(ls), ls, engine=gpu.eng)
    want = [O.proj_affine(O.proj_add((a.x, a.y, 1), (b.x, b.y, 1))) for a, b in zip(kp, lq)]
    assert [(r.x, r.y) for r in got] == want
    b8 = [bjj.Point(*O.B8)] * len(ls)
    assert bjj.mul2_fixed_base_batch(p, ks, None, ls, engine=gpu.eng) == \
        bjj.mul2_fixed_base_batch(p, ks, bjj.Point(*O.B8), ls, engine=gpu.eng)
    assert bjj.mul_fixed_base_batch(b8[0], ls, engine=gpu.eng) == bjj.mul_scalar_batch(b8, ls, engine=gpu.eng)
    with pytest.raises(bjj.BjjError) as e:
        bjj.FixedBase((1, 1), gpu.eng)
    assert e.value.code == ERR_ARG
    with pytest.raises(bjj.BjjError) as e:
        bjj.FixedBase((0, 1 + O.Q), gpu.eng)
    assert e.value.code == ERR_NONCANONICAL
