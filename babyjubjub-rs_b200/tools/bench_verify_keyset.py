"""Throughput of verify against a key set (bjj_verify_keyset_batch: a key index per lane, a compact comb per key) next to
bjj_verify_batch with the keys gathered per lane, on one GPU, for sets of 1, 256 and 65,536 keys.

    python babyjubjub-rs_b200/tools/bench_verify_keyset.py --out DIR [--log2-sigs 21] [--keys 1,256,65536]
                                                           [--steps 10] [--warmup 2] [--repeats 3]

Inputs, per key-set size K: K seeded private keys, a seeded random key index per lane, and 2^21 signatures made on the
device by bjj_sign_batch_dev (lane i signs with the key of its index) over random messages below Q; then about 10 % of
the lanes are corrupted on the host in the classes of bench_verify_base.py.  At K = 256 the tables (~100 MB) are close
to the size of L2, at K = 65,536 (~26 GB) they are read from HBM.  Measures:
  - bjj_keyset_create: a host clock around the synchronous call, per key;
  - device-resident (CUDA events around `steps` back-to-back calls on one stream, closed by a synchronise):
    bjj_verify_batch_dev (A gathered per lane) against bjj_verify_keyset_batch_dev, and at K = 1 also
    bjj_verify_base_batch_dev with a FixedBase of the key;
  - end to end from page-locked buffers (bjj_host_alloc; a host clock around `steps` host-flavour calls, each of which
    returns with its results in place): bjj_verify_batch against bjj_verify_keyset_batch.
Every variant is warmed up first; the variants then run alternately `repeats` times, and each rate is reported per run
with its mean and spread (max - min over mean).  The ok[] arrays of all variants are compared on every lane after every
timed round.  The card's name and power limit are read in the same run.  Writes DIR/verify_keyset.json and prints it.
"""
import argparse
import ctypes
import json
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for _p in (ROOT, HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from bench_verify_base import alternate, card_info, corrupt_one_key  # noqa: E402


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, help="directory for verify_keyset.json")
    ap.add_argument("--log2-sigs", type=int, default=21)
    ap.add_argument("--keys", default="1,256,65536", help="comma-separated key-set sizes")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--repeats", type=int, default=3, help="alternating runs of every variant (at least 2)")
    args = ap.parse_args()
    if args.repeats < 2 or args.steps < 1:
        raise SystemExit("--repeats must be at least 2 and --steps at least 1")

    import torch
    import babyjubjub_rs_b200 as bjj
    if not torch.cuda.is_available():
        raise SystemExit("bench_verify_keyset.py needs a CUDA device: there is no CPU fallback")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    eng = bjj.Engine(0)
    lib, ctx = eng.lib, eng.ctx
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    sp = ctypes.c_void_p(stream.cuda_stream)
    n, steps = 1 << args.log2_sigs, args.steps

    def check(rc, what):
        if rc != 0:
            raise RuntimeError("%s failed: %d (%s)" % (what, rc, lib.bjj_error_string(rc).decode()))

    def p(a):
        return ctypes.c_void_p(a.data_ptr()) if isinstance(a, torch.Tensor) else a.ctypes.data_as(ctypes.c_void_p)

    def t(shape):
        return torch.empty(shape, dtype=torch.uint8, device=dev)

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

    def host_timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        return n / ((time.perf_counter() - t0) / steps) / 1e6

    def ratio(table, a, b):
        return round(table[a]["M_per_s_mean"] / table[b]["M_per_s_mean"], 3)

    results = []
    mismatches = []
    for n_keys in [int(k) for k in args.keys.split(",")]:
        # ---- inputs: K keys, a random key per lane, n signatures made on the device, 10 % corrupted ----------------
        rng = np.random.default_rng(20261022 + n_keys)
        priv = rng.integers(0, 256, size=(n_keys, 32), dtype=np.uint8)
        idx = rng.integers(0, n_keys, size=n).astype("<u4")
        msgs_np = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
        msgs_np[:, 31] &= 0x2F                             # < Q: every lane signs
        dpriv = torch.from_numpy(priv).to(dev)
        didx = torch.from_numpy(idx.astype(np.int64)).to(dev)
        dk = dpriv[didx].contiguous()
        dm = torch.from_numpy(msgs_np).to(dev)
        drx, dry, ds, dst = t((n, 32)), t((n, 32)), t((n, 32)), t((n,))
        check(lib.bjj_sign_batch_dev(ctx, n, p(dk), p(dm), p(drx), p(dry), p(ds), p(dst), sp), "sign")
        dax, day = t((n_keys, 32)), t((n_keys, 32))
        check(lib.bjj_public_batch_dev(ctx, n_keys, p(dpriv), p(dax), p(day), sp), "public")
        torch.cuda.synchronize()
        check(lib.bjj_sync(ctx), "bjj_sync")
        assert not dst.any().item()
        r8x, r8y, s, ax, ay = (a.cpu().numpy() for a in (drx, dry, ds, dax, day))
        msg = msgs_np.copy()
        corrupted = corrupt_one_key(r8x, r8y, s, msg, 0xBA5E + n_keys)
        del dk, dm, drx, dry, ds, dst, dax, day, dpriv, didx
        axn, ayn = ax[idx], ay[idx]

        # ---- bjj_keyset_create ---------------------------------------------------------------------------------
        torch.cuda.synchronize()
        handle = ctypes.c_void_p()
        t0 = time.perf_counter()
        check(lib.bjj_keyset_create(ctx, n_keys, p(ax), p(ay), None, ctypes.byref(handle)), "keyset_create")
        create_s = time.perf_counter() - t0
        kh = handle
        base = bjj.FixedBase((int.from_bytes(ax[0].tobytes(), "little"), int.from_bytes(ay[0].tobytes(), "little")), eng) \
            if n_keys == 1 else None

        # ---- device-resident: CUDA events ----------------------------------------------------------------------
        d = [torch.from_numpy(c).to(dev) for c in (r8x, r8y, s, msg, axn, ayn)]
        d_idx = torch.from_numpy(idx.view(np.uint8).copy()).to(dev)
        oks = {"verify_batch_dev": t((n,)), "verify_keyset_batch_dev": t((n,))}
        variants = {
            "verify_batch_dev": lambda: check(lib.bjj_verify_batch_dev(ctx, n, p(d[0]), p(d[1]), p(d[2]), p(d[4]), p(d[5]), p(d[3]),
                                                                       p(oks["verify_batch_dev"]), sp), "verify"),
            "verify_keyset_batch_dev": lambda: check(lib.bjj_verify_keyset_batch_dev(ctx, kh, n, p(d_idx), p(d[0]), p(d[1]), p(d[2]),
                                                                                     p(d[3]), p(oks["verify_keyset_batch_dev"]), sp),
                                                     "verify_keyset"),
        }
        if base is not None:
            oks["verify_base_batch_dev"] = t((n,))
            variants["verify_base_batch_dev"] = lambda: check(lib.bjj_verify_base_batch_dev(ctx, base.handle, n, p(d[0]), p(d[1]), p(d[2]),
                                                                                             p(d[3]), p(oks["verify_base_batch_dev"]),
                                                                                             sp), "verify_base")
        for i, o in enumerate(oks.values()):
            o.fill_(0xE0 + i)

        def compare():
            torch.cuda.synchronize()
            ref = oks["verify_batch_dev"]
            mismatches.append(sum(int((o != ref).sum().item()) for o in oks.values()))
        device_resident = alternate(variants, dev_timed, args.warmup, args.repeats, compare)
        accepted = int(oks["verify_batch_dev"].sum().item())
        del d, d_idx, oks

        # ---- end to end from page-locked host buffers: host clock -------------------------------------------------
        pinned = []

        def host_array(shape):
            nbytes = int(np.prod(shape))
            ptr = lib.bjj_host_alloc(nbytes)
            if not ptr:
                raise RuntimeError("bjj_host_alloc(%d) failed" % nbytes)
            pinned.append(ptr)
            return np.frombuffer((ctypes.c_uint8 * nbytes).from_address(ptr), dtype=np.uint8).reshape(shape)

        try:
            h = [host_array((n, 32)) for _ in range(6)]
            for dst_, src in zip(h, (r8x, r8y, s, axn, ayn, msg)):
                dst_[...] = src
            hidx = host_array((n, 4))
            hidx[...] = idx.view(np.uint8).reshape(n, 4)
            hok_v, hok_k = host_array((n,)), host_array((n,))
            hok_v[...], hok_k[...] = 0xEE, 0xDD

            def compare_host():
                mismatches.append(int((hok_v != hok_k).sum()))
            end_to_end = alternate({
                "verify_batch": lambda: check(lib.bjj_verify_batch(ctx, n, *[p(a) for a in h], p(hok_v)), "verify"),
                "verify_keyset_batch": lambda: check(lib.bjj_verify_keyset_batch(ctx, kh, n, p(hidx), p(h[0]), p(h[1]), p(h[2]), p(h[5]),
                                                                                 p(hok_k)), "verify_keyset"),
            }, host_timed, args.warmup, args.repeats, compare_host)
        finally:
            for ptr in pinned:
                lib.bjj_host_free(ptr)
        if base is not None:
            base.close()
        lib.bjj_keyset_destroy(ctx, kh)

        entry = {
            "keys": n_keys,
            "table_bytes": n_keys * 4130 * 96,
            "keyset_create_s": round(create_s, 4),
            "keyset_create_us_per_key": round(create_s / n_keys * 1e6, 3),
            "corrupted_lanes": corrupted,
            "accepted_lanes": accepted,
            "device_resident": device_resident,
            "end_to_end_pinned": end_to_end,
            "ratios": {
                "dev_keyset_over_verify": ratio(device_resident, "verify_keyset_batch_dev", "verify_batch_dev"),
                "e2e_keyset_over_verify": ratio(end_to_end, "verify_keyset_batch", "verify_batch"),
            },
        }
        if n_keys == 1:
            entry["ratios"]["dev_keyset_over_base"] = ratio(device_resident, "verify_keyset_batch_dev", "verify_base_batch_dev")
        results.append(entry)
        print(json.dumps(entry), flush=True)
    eng.close()

    report = {
        "card": card_info(0),
        "torch_device_name": torch.cuda.get_device_name(0),
        "signatures": n,
        "steps": steps,
        "warmup": args.warmup,
        "repeats": args.repeats,
        "key_sets": results,
        "ok_mismatched_lanes_per_timed_round": mismatches,
    }
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "verify_keyset.json"), "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(report, indent=1))
    if any(mismatches):
        raise SystemExit("verify_keyset_batch and verify_batch disagree")


if __name__ == "__main__":
    main()
