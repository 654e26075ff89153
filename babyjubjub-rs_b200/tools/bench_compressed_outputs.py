"""Throughput of the compressed outputs of key generation and signing against the uncompressed calls, on one GPU and,
when more than one is visible, on all of them.

    python babyjubjub-rs_b200/tools/bench_compressed_outputs.py --out DIR [--log2-keys 20] [--log2-sigs 21]
                                                                [--steps 10] [--warmup 3] [--repeats 3]

Measures, for 2^20 random keys and for 2^21 signatures over random messages below Q:
  - device-resident (CUDA events around `steps` back-to-back calls on one stream, closed by a synchronise):
    bjj_public_batch_dev against bjj_public_compressed_batch_dev, bjj_sign_batch_dev against
    bjj_sign_compressed_batch_dev;
  - end to end from page-locked buffers (bjj_host_alloc; a host clock around `steps` host-flavour calls, each of which
    returns with its results in place): bjj_public_batch, bjj_public_batch followed by bjj_compress_batch (what a caller
    who wants compressed keys does without the compressed entry point), bjj_public_compressed_batch; the same three for
    sign (bjj_sign_batch, + bjj_compress_batch of R8, bjj_sign_compressed_batch);
  - with more than one device: bjj_multi_public_batch against bjj_multi_public_compressed_batch on 2^20 keys per
    device, page-locked buffers, host clock.
Every variant of a comparison is warmed up first; the variants then run alternately `repeats` times, and each rate is
reported per run with its mean and its spread (max - min over mean).  Inputs come from a fixed seed; the key arrays
(32 MiB for 2^20 keys) fit the 126 MB L2, which matters little next to the arithmetic of these calls.  The
compressed outputs are checked byte for byte against the composed calls.  The card's name and power limit are read in
the same run.  Writes DIR/compressed_outputs.json and prints it.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def card_info(index):
    out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm",
                          "--format=csv,noheader"], capture_output=True, text=True)
    if out.returncode != 0:
        return {"nvidia_smi": "failed: " + out.stderr.strip()}
    name, power, clock = [f.strip() for f in out.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


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


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, help="directory for compressed_outputs.json")
    ap.add_argument("--log2-keys", type=int, default=20)
    ap.add_argument("--log2-sigs", type=int, default=21)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=3, help="alternating runs of every variant (at least 2)")
    args = ap.parse_args()
    if args.repeats < 2 or args.steps < 1:
        raise SystemExit("--repeats must be at least 2 and --steps at least 1")

    import torch
    import babyjubjub_rs_b200 as bjj
    if not torch.cuda.is_available():
        raise SystemExit("bench_compressed_outputs.py needs a CUDA device: there is no CPU fallback")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    eng = bjj.Engine(0)
    lib, ctx = eng.lib, eng.ctx
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    sp = ctypes.c_void_p(stream.cuda_stream)
    nk, ns = 1 << args.log2_keys, 1 << args.log2_sigs
    steps = args.steps

    def check(rc, what):
        if rc != 0:
            raise RuntimeError("%s failed: %d (%s)" % (what, rc, lib.bjj_error_string(rc).decode()))

    def p(a):
        return ctypes.c_void_p(a.data_ptr()) if isinstance(a, torch.Tensor) else a.ctypes.data_as(ctypes.c_void_p)

    rng = np.random.default_rng(20261021)
    keys_np = rng.integers(0, 256, size=(max(nk, ns), 32), dtype=np.uint8)
    msgs_np = rng.integers(0, 256, size=(ns, 32), dtype=np.uint8)
    msgs_np[:, 31] &= 0x2F                                 # < 0x30 * 2^248 < Q: every lane signs

    # ---- device-resident: CUDA events ----------------------------------------------------------------------
    def dev_timed(n):
        def timed(fn):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(steps):
                fn()
            e1.record(stream)
            torch.cuda.synchronize()
            check(lib.bjj_sync(ctx), "bjj_sync")
            return n / (e0.elapsed_time(e1) / steps) / 1e3
        return timed

    def t(shape):
        return torch.empty(shape, dtype=torch.uint8, device=dev)

    dk = torch.from_numpy(keys_np).to(dev)
    dm = torch.from_numpy(msgs_np).to(dev)
    drx, dry, ds, dout = t((ns, 32)), t((ns, 32)), t((ns, 32)), t((ns, 32))
    dsig, dst = t((ns, 64)), t((ns,))
    device_resident = {
        "public": alternate({
            "public_batch_dev": lambda: check(lib.bjj_public_batch_dev(ctx, nk, p(dk), p(drx), p(dry), sp), "public"),
            "public_compressed_batch_dev": lambda: check(lib.bjj_public_compressed_batch_dev(ctx, nk, p(dk), p(dout), sp),
                                                         "public_compressed"),
        }, dev_timed(nk), args.warmup, args.repeats),
        "sign": alternate({
            "sign_batch_dev": lambda: check(lib.bjj_sign_batch_dev(ctx, ns, p(dk), p(dm), p(drx), p(dry), p(ds), p(dst), sp),
                                            "sign"),
            "sign_compressed_batch_dev": lambda: check(lib.bjj_sign_compressed_batch_dev(ctx, ns, p(dk), p(dm), p(dsig), p(dst),
                                                                                         sp), "sign_compressed"),
        }, dev_timed(ns), args.warmup, args.repeats),
    }
    del dk, dm, drx, dry, ds, dout, dsig, dst

    # ---- end to end from page-locked host buffers: host clock -------------------------------------------------
    pinned = []

    def host_array(shape):
        nbytes = int(np.prod(shape))
        ptr = lib.bjj_host_alloc(nbytes)
        if not ptr:
            raise RuntimeError("bjj_host_alloc(%d) failed" % nbytes)
        pinned.append(ptr)
        return np.frombuffer((ctypes.c_uint8 * nbytes).from_address(ptr), dtype=np.uint8).reshape(shape)

    def host_timed(n):
        def timed(fn):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                fn()
            return n / ((time.perf_counter() - t0) / steps) / 1e6
        return timed

    try:
        hk, hm = host_array(keys_np.shape), host_array(msgs_np.shape)
        hk[...], hm[...] = keys_np, msgs_np
        hrx, hry, hs, hc = (host_array((ns, 32)) for _ in range(4))
        hout, hsig, hst = host_array((ns, 32)), host_array((ns, 64)), host_array((ns,))

        def public_then_compress():
            check(lib.bjj_public_batch(ctx, nk, p(hk), p(hrx), p(hry)), "public")
            check(lib.bjj_compress_batch(ctx, nk, p(hrx), p(hry), p(hc)), "compress")

        def sign_then_compress():
            check(lib.bjj_sign_batch(ctx, ns, p(hk), p(hm), p(hrx), p(hry), p(hs), p(hst)), "sign")
            check(lib.bjj_compress_batch(ctx, ns, p(hrx), p(hry), p(hc)), "compress")

        end_to_end = {
            "public": alternate({
                "public_batch": lambda: check(lib.bjj_public_batch(ctx, nk, p(hk), p(hrx), p(hry)), "public"),
                "public_batch_then_compress_batch": public_then_compress,
                "public_compressed_batch": lambda: check(lib.bjj_public_compressed_batch(ctx, nk, p(hk), p(hout)),
                                                         "public_compressed"),
            }, host_timed(nk), args.warmup, args.repeats),
        }
        public_same = bool(np.array_equal(hout[:nk], hc[:nk]))
        end_to_end["sign"] = alternate({
            "sign_batch": lambda: check(lib.bjj_sign_batch(ctx, ns, p(hk), p(hm), p(hrx), p(hry), p(hs), p(hst)), "sign"),
            "sign_batch_then_compress_batch": sign_then_compress,
            "sign_compressed_batch": lambda: check(lib.bjj_sign_compressed_batch(ctx, ns, p(hk), p(hm), p(hsig), p(hst)),
                                                   "sign_compressed"),
        }, host_timed(ns), args.warmup, args.repeats)
        sign_same = bool(np.array_equal(hsig[:, :32], hc) and np.array_equal(hsig[:, 32:], hs) and not hst.any())

        # ---- every visible device: bjj_multi ---------------------------------------------------------------------
        ndev = lib.bjj_device_count()
        multi = None
        if ndev > 1:
            me = bjj.MultiEngine()
            try:
                nm = nk * ndev
                mk = host_array((nm, 32))
                mk[...] = rng.integers(0, 256, size=(nm, 32), dtype=np.uint8)
                mrx, mry, mout, mc = (host_array((nm, 32)) for _ in range(4))

                def mcheck(rc, what):
                    if rc != 0:
                        raise RuntimeError("%s failed: %d" % (what, rc))
                multi = {"devices": ndev, "keys": nm, "results": alternate({
                    "multi_public_batch": lambda: mcheck(lib.bjj_multi_public_batch(me.handle, nm, p(mk), p(mrx), p(mry)),
                                                         "multi_public"),
                    "multi_public_compressed_batch": lambda: mcheck(
                        lib.bjj_multi_public_compressed_batch(me.handle, nm, p(mk), p(mout)), "multi_public_compressed"),
                }, host_timed(nm), args.warmup, args.repeats)}
                check(lib.bjj_compress_batch(ctx, nm, p(mrx), p(mry), p(mc)), "compress")
                multi["compressed_equals_composition"] = bool(np.array_equal(mout, mc))
            finally:
                me.close()
    finally:
        for ptr in pinned:
            lib.bjj_host_free(ptr)
    eng.close()

    def ratio(table, a, b):
        return round(table[a]["M_per_s_mean"] / table[b]["M_per_s_mean"], 3)

    report = {
        "card": card_info(0),
        "torch_device_name": torch.cuda.get_device_name(0),
        "keys": nk,
        "signatures": ns,
        "steps": steps,
        "warmup": args.warmup,
        "repeats": args.repeats,
        "device_resident": device_resident,
        "end_to_end_pinned": end_to_end,
        "multi_device": multi,
        "ratios": {
            "public_dev_compressed_over_affine": ratio(device_resident["public"], "public_compressed_batch_dev", "public_batch_dev"),
            "sign_dev_compressed_over_affine": ratio(device_resident["sign"], "sign_compressed_batch_dev", "sign_batch_dev"),
            "public_e2e_compressed_over_affine": ratio(end_to_end["public"], "public_compressed_batch", "public_batch"),
            "public_e2e_compressed_over_composed": ratio(end_to_end["public"], "public_compressed_batch",
                                                         "public_batch_then_compress_batch"),
            "sign_e2e_compressed_over_affine": ratio(end_to_end["sign"], "sign_compressed_batch", "sign_batch"),
            "sign_e2e_compressed_over_composed": ratio(end_to_end["sign"], "sign_compressed_batch",
                                                       "sign_batch_then_compress_batch"),
        },
        "public_compressed_equals_composition": public_same,
        "sign_compressed_equals_composition": sign_same,
    }
    if multi:
        report["ratios"]["multi_public_compressed_over_affine"] = ratio(multi["results"], "multi_public_compressed_batch",
                                                                        "multi_public_batch")
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "compressed_outputs.json"), "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(report, indent=1))
    if not (public_same and sign_same and (multi is None or multi["compressed_equals_composition"])):
        raise SystemExit("compressed outputs disagree with the composed calls")


if __name__ == "__main__":
    main()
