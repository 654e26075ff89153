"""Throughput of Schnorr signing with caller nonces (bjj_sign_schnorr_batch) on one GPU, against EdDSA signing and the
composed path it replaces, and of verify_schnorr on the valid signatures it makes.

    python babyjubjub-rs_b200/tools/bench_sign_schnorr.py [--out profiles/r5_sign_schnorr.json] [--log2-lanes 21]
                                                          [--steps 5] [--warmup 2] [--repeats 3] [--profile]

Measures, for 2^21 lanes of seeded random keys, messages below Q and nonces:
  - device-resident (CUDA events around `steps` back-to-back calls on one stream, closed by a synchronise):
    bjj_sign_schnorr_batch_dev at nonce_words = 32 (the reference's 1024-bit nonce) and at nonce_words = 8, and
    bjj_sign_batch_dev on the same keys and messages as the yardstick;
  - end to end from page-locked buffers (bjj_host_alloc; a host clock around `steps` host-flavour calls, each of which
    returns with its results in place): bjj_sign_schnorr_batch at nonce_words = 32, against the device calls of the
    composed path it replaces (bjj_scalar_key_batch, bjj_fixed_base_batch on nonces reduced mod SUBORDER,
    bjj_public_batch, bjj_poseidon_batch).  That path also needs the nonce reduction and s = k + sk * h on the host:
    their Python-integer cost is timed once on its own ("composed_host_arithmetic_s"), as it depends on the caller's
    language;
  - bjj_verify_schnorr_batch_dev on the valid signatures just made (s reduced mod SUBORDER on the host), to set beside
    bench.py's verify_schnorr figure, whose lanes are almost all rejections.
Every variant of a comparison is warmed up first; the variants then run alternately `repeats` times, and each rate is
reported per run with its mean and its spread (max - min over mean).  Every timed output is checked against the oracle
on a sample of lanes.  --profile adds per-kernel device times of one call each of sign_schnorr (nonce_words = 32) and
sign, from torch.profiler, in a phase after the timed runs.  The card's name and power limit are read in the same run.
"""
import argparse
import ctypes
import json
import os
import random
import subprocess
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SUBORDER = 21888242871839275222246405745257275088614511777268538073601725287587578984328 >> 3
Q = 21888242871839275222246405745257275088548364400416034343698204186575808495617


def card_info(index):
    out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True)
    if out.returncode != 0:
        return {"nvidia_smi": "failed: " + out.stderr.strip()}
    name, power = [f.strip() for f in out.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power}


def summary(rates):
    mean = sum(rates) / len(rates)
    return {"M_per_s_runs": [round(r, 2) for r in rates], "M_per_s_mean": round(mean, 2),
            "spread": round((max(rates) - min(rates)) / mean, 4)}


def alternate(variants, timed, warmup, repeats):
    """warms up every variant, then times them alternately `repeats` times; {name: summary}"""
    for fn in variants.values():
        for _ in range(warmup):
            fn()
    runs = {name: [] for name in variants}
    for _ in range(repeats):
        for name, fn in variants.items():
            runs[name].append(timed(fn))
    return {name: summary(r) for name, r in runs.items()}


def wide_ints(arr):
    return [int.from_bytes(r.tobytes(), "little") for r in np.ascontiguousarray(arr)]


def le32(vals):
    return np.frombuffer(b"".join(int(v).to_bytes(32, "little") for v in vals), dtype=np.uint8).reshape(-1, 32)


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r5_sign_schnorr.json"), help="JSON file to write")
    ap.add_argument("--log2-lanes", type=int, default=21)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--repeats", type=int, default=3, help="alternating runs of every variant (at least 2)")
    ap.add_argument("--sample", type=int, default=48, help="lanes of every timed output checked against the oracle")
    ap.add_argument("--profile", action="store_true", help="per-kernel times from torch.profiler, after the timed runs")
    args = ap.parse_args()
    if args.repeats < 2 or args.steps < 1:
        raise SystemExit("--repeats must be at least 2 and --steps at least 1")

    import torch
    import babyjubjub_rs_b200 as bjj
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import common                  # the checkers of the test suite, as bench.py uses them; the library never loads them
    O = common.O
    if not torch.cuda.is_available():
        raise SystemExit("bench_sign_schnorr.py needs a CUDA device: there is no CPU fallback")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    eng = bjj.Engine(0)
    lib, ctx = eng.lib, eng.ctx
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    sp = ctypes.c_void_p(stream.cuda_stream)
    n = 1 << args.log2_lanes
    steps = args.steps

    def check(rc, what):
        if rc != 0:
            raise RuntimeError("%s failed: %d (%s)" % (what, rc, lib.bjj_error_string(rc).decode()))

    def p(a):
        return ctypes.c_void_p(a.data_ptr()) if isinstance(a, torch.Tensor) else a.ctypes.data_as(ctypes.c_void_p)

    rng = np.random.default_rng(20261022)
    keys_np = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    msgs_np = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    msgs_np[:, 31] &= 0x2F                                 # < 0x30 * 2^248 < Q: every lane signs
    k32_np = rng.integers(0, 256, size=(n, 128), dtype=np.uint8)      # 1024-bit nonces
    k8_np = np.ascontiguousarray(k32_np[:, :32])                      # their low 256 bits
    sample = sorted(random.Random(5).sample(range(n), args.sample))
    mismatches = []

    def oracle_check(what, rx, ry, s, st, nonces, words):
        """sampled lanes of a sign_schnorr output against O.sign_schnorr"""
        ks = wide_ints(nonces[sample])
        ms = wide_ints(msgs_np[sample])
        for j, i in enumerate(sample):
            r, sv = O.sign_schnorr(bytes(keys_np[i]), ms[j], ks[j])
            got = (wide_ints(rx[i:i + 1])[0], wide_ints(ry[i:i + 1])[0], wide_ints(s[i:i + 1])[0], int(st[i]))
            if got != (r[0], r[1], sv, 0) or s.shape[1] != 4 * (words + 8):
                mismatches.append((what, i))

    # ---- device-resident: CUDA events ----------------------------------------------------------------------
    def dev_timed(fn):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        check(lib.bjj_sync(ctx), "bjj_sync")
        return n / (e0.elapsed_time(e1) / steps) / 1e3

    def t(shape):
        return torch.empty(shape, dtype=torch.uint8, device=dev)

    dk, dm = torch.from_numpy(keys_np).to(dev), torch.from_numpy(msgs_np).to(dev)
    dk32, dk8 = torch.from_numpy(k32_np).to(dev), torch.from_numpy(k8_np).to(dev)
    drx, dry, dst = t((n, 32)), t((n, 32)), t((n,))
    ds40, ds16 = t((n, 160)), t((n, 64))
    erx, ery, es, est = t((n, 32)), t((n, 32)), t((n, 32)), t((n,))

    def schnorr_dev(words):
        dkw, dsw = (dk32, ds40) if words == 32 else (dk8, ds16)
        return lambda: check(lib.bjj_sign_schnorr_batch_dev(ctx, n, p(dk), p(dm), p(dkw), words, p(drx), p(dry), p(dsw), p(dst), sp),
                             "sign_schnorr_dev")

    sign_dev = lambda: check(lib.bjj_sign_batch_dev(ctx, n, p(dk), p(dm), p(erx), p(ery), p(es), p(est), sp), "sign_dev")  # noqa: E731
    device_resident = alternate({"sign_schnorr_batch_dev_w32": schnorr_dev(32), "sign_schnorr_batch_dev_w8": schnorr_dev(8),
                                 "sign_batch_dev": sign_dev}, dev_timed, args.warmup, args.repeats)
    # the last timed call of each variant is checked: w8 (its r and status planes were overwritten by w32's)
    schnorr_dev(8)()
    torch.cuda.synchronize()
    oracle_check("sign_schnorr_batch_dev_w8", drx.cpu().numpy(), dry.cpu().numpy(), ds16.cpu().numpy(), dst.cpu().numpy(), k8_np, 8)
    schnorr_dev(32)()
    torch.cuda.synchronize()
    rx_d, ry_d, s_d, st_d = drx.cpu().numpy(), dry.cpu().numpy(), ds40.cpu().numpy(), dst.cpu().numpy()
    oracle_check("sign_schnorr_batch_dev_w32", rx_d, ry_d, s_d, st_d, k32_np, 32)
    e_rx, e_s = erx.cpu().numpy(), es.cpu().numpy()
    for i in sample[:8]:
        (r8x, _), sv = O.sign(bytes(keys_np[i]), wide_ints(msgs_np[i:i + 1])[0])
        if wide_ints(e_rx[i:i + 1])[0] != r8x or wide_ints(e_s[i:i + 1])[0] != sv:
            mismatches.append(("sign_batch_dev", i))

    # ---- verify_schnorr on the valid signatures just made ----------------------------------------------------
    pkx, pky = t((n, 32)), t((n, 32))
    check(lib.bjj_public_batch_dev(ctx, n, p(dk), p(pkx), p(pky), sp), "public_dev")
    t0 = time.perf_counter()
    s_red = le32([v % SUBORDER for v in wide_ints(s_d)])
    reduce_s_host = time.perf_counter() - t0
    dsr = torch.from_numpy(s_red.copy()).to(dev)
    vok, vst = t((n,)), t((n,))
    verify = alternate({"verify_schnorr_batch_dev_valid": lambda: check(
        lib.bjj_verify_schnorr_batch_dev(ctx, n, p(pkx), p(pky), p(dm), p(drx), p(dry), p(dsr), p(vok), p(vst), sp), "verify_schnorr")},
        dev_timed, args.warmup, args.repeats)
    torch.cuda.synchronize()
    verify_all_ok = bool((vok.cpu().numpy() == 1).all() and not vst.cpu().numpy().any())
    del dk, dm, dk32, dk8, drx, dry, dst, ds40, ds16, erx, ery, es, est, pkx, pky, dsr, vok, vst

    # ---- end to end from page-locked host buffers: host clock -------------------------------------------------
    pinned = []

    def host_array(shape):
        nbytes = int(np.prod(shape))
        ptr = lib.bjj_host_alloc(nbytes)
        if not ptr:
            raise RuntimeError("bjj_host_alloc(%d) failed" % nbytes)
        pinned.append(ptr)
        return np.frombuffer((ctypes.c_uint8 * nbytes).from_address(ptr), dtype=np.uint8).reshape(shape)

    def host_timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        return n / ((time.perf_counter() - t0) / steps) / 1e6

    try:
        hk, hm, hn = host_array((n, 32)), host_array((n, 32)), host_array((n, 128))
        hk[...], hm[...], hn[...] = keys_np, msgs_np, k32_np
        hrx, hry, hs, hst = host_array((n, 32)), host_array((n, 32)), host_array((n, 160)), host_array((n,))
        # the composed path: the nonces reduced on the host once (timed on its own below), then four device calls
        t0 = time.perf_counter()
        kred = le32([k % SUBORDER for k in wide_ints(k32_np)])
        reduce_k_host = time.perf_counter() - t0
        hkr = host_array((n, 32))
        hkr[...] = kred
        csk, crx, cry, cpx, cpy, ch = (host_array((n, 32)) for _ in range(6))
        pos = (ctypes.c_void_p * 5)(*[a.ctypes.data for a in (cpx, cpy, crx, cry, hm)])

        def composed():
            check(lib.bjj_scalar_key_batch(ctx, n, p(hk), p(csk)), "scalar_key")
            check(lib.bjj_fixed_base_batch(ctx, n, p(hkr), p(crx), p(cry)), "fixed_base")
            check(lib.bjj_public_batch(ctx, n, p(hk), p(cpx), p(cpy)), "public")
            check(lib.bjj_poseidon_batch(ctx, 5, n, pos, p(ch)), "poseidon")

        end_to_end = alternate({
            "sign_schnorr_batch_w32": lambda: check(lib.bjj_sign_schnorr_batch(ctx, n, p(hk), p(hm), p(hn), 32, p(hrx), p(hry), p(hs),
                                                                               p(hst)), "sign_schnorr"),
            "composed_device_calls": composed,
        }, host_timed, args.warmup, args.repeats)
        oracle_check("sign_schnorr_batch_w32", hrx, hry, hs, hst, k32_np, 32)
        t0 = time.perf_counter()
        s_host = [k + x * h for k, x, h in zip(wide_ints(k32_np), wide_ints(csk), wide_ints(ch))]
        s_host_time = time.perf_counter() - t0
        composed_same = bool(np.array_equal(crx, hrx) and np.array_equal(cry, hry) and
                             all(s_host[i] == wide_ints(hs[i:i + 1])[0] for i in sample))
        end_equals_dev = bool(np.array_equal(hrx, rx_d) and np.array_equal(hs, s_d) and np.array_equal(hst, st_d))
    finally:
        for ptr in pinned:
            lib.bjj_host_free(ptr)

    kernels = None
    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        dk, dm, dk32 = (torch.from_numpy(a).to(dev) for a in (keys_np, msgs_np, k32_np))
        drx, dry, dst, ds40, es = t((n, 32)), t((n, 32)), t((n,)), t((n, 160)), t((n, 32))
        kernels = {}
        for name, fn in (("sign_schnorr_batch_dev_w32", lambda: lib.bjj_sign_schnorr_batch_dev(
                ctx, n, p(dk), p(dm), p(dk32), 32, p(drx), p(dry), p(ds40), p(dst), sp)),
                         ("sign_batch_dev", lambda: lib.bjj_sign_batch_dev(ctx, n, p(dk), p(dm), p(drx), p(dry), p(es), p(dst), sp))):
            check(fn(), name)
            torch.cuda.synchronize()
            try:
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    check(fn(), name)
                    torch.cuda.synchronize()
                rows = {}
                for ev in prof.events():
                    us = getattr(ev, "device_time_total", 0) or 0
                    if us and "memset" not in ev.name.lower() and "memcpy" not in ev.name.lower():
                        rows.setdefault(ev.name, []).append(us / 1e3)
                kernels[name] = {k: {"launches": len(v), "ms": round(sum(v), 3)}
                                 for k, v in sorted(rows.items(), key=lambda kv: -sum(kv[1]))}
            except Exception as e:      # the timed results stand without the breakdown
                kernels[name] = {"error": repr(e)}
    eng.close()

    def ratio(a, b):
        return round(a["M_per_s_mean"] / b["M_per_s_mean"], 3)

    report = {
        "card": card_info(0),
        "torch_device_name": torch.cuda.get_device_name(0),
        "lanes": n,
        "steps": steps,
        "warmup": args.warmup,
        "repeats": args.repeats,
        "device_resident": device_resident,
        "verify_schnorr_valid_signatures": verify,
        "verify_schnorr_all_accepted": verify_all_ok,
        "end_to_end_pinned": end_to_end,
        "composed_host_arithmetic_s": {"nonce_mod_suborder": round(reduce_k_host, 3), "s_equals_k_plus_sk_h": round(s_host_time, 3),
                                       "note": "Python integers, once per batch of %d lanes; not in the rates above" % n},
        "verify_input_s_mod_suborder_host_s": round(reduce_s_host, 3),
        "ratios": {
            "schnorr_w32_dev_over_sign_dev": ratio(device_resident["sign_schnorr_batch_dev_w32"], device_resident["sign_batch_dev"]),
            "schnorr_w8_dev_over_sign_dev": ratio(device_resident["sign_schnorr_batch_dev_w8"], device_resident["sign_batch_dev"]),
            "schnorr_e2e_over_composed_device_calls": ratio(end_to_end["sign_schnorr_batch_w32"], end_to_end["composed_device_calls"]),
        },
        "oracle_sample_lanes": len(sample),
        "oracle_mismatches": mismatches,
        "composed_path_equals_sign_schnorr": composed_same,
        "host_flavour_equals_dev_flavour": end_equals_dev,
        "per_kernel_ms_one_call": kernels,
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(report, indent=1))
    if mismatches or not (composed_same and end_equals_dev and verify_all_ok):
        raise SystemExit("sign_schnorr outputs disagree with the oracle or the composed path")


if __name__ == "__main__":
    main()
