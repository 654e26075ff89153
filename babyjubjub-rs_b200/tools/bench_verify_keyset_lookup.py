"""Throughput of verify against a key set with the keys named by their compressed bytes
(bjj_verify_keyset_lookup_compressed_batch) next to the calls it stands beside, on one GPU, for sets of 1, 256 and
65,536 keys.

    python babyjubjub-rs_b200/tools/bench_verify_keyset_lookup.py --out DIR [--log2-sigs 21] [--keys 1,256,65536]
                                                                  [--steps 10] [--warmup 2] [--repeats 3]

Inputs, per key-set size K: K seeded private keys in the set and K/19 + 1 more outside it; a seeded key per lane, 5 % of
lanes from the keys outside the set; 2^21 compressed signatures made on the device by bjj_sign_compressed_batch_dev over
random messages below Q, and the lanes' compressed public keys; then about 10 % of the lanes corrupted on the host (a
bit of S, a bit of msg, msg > Q, R8 with y >= Q, R8 that is mostly not a square).  The arms:
  1. bjj_verify_keyset_lookup_compressed_batch (the lookup on the device, then the key-set kernels);
  2. bjj_verify_keyset_compressed_batch with the key indices known in advance (index 0 for keys outside the set, whose
     signatures then fail): 1 against 2 is what the lookup costs;
  3. bjj_verify_compressed_batch, which decompresses every lane's key and verifies on the Straus path;
  4. bjj_keyset_lookup_batch alone.
Each arm runs device-resident (CUDA events around `steps` back-to-back _dev calls on one stream, closed by a
synchronise) and end to end from page-locked buffers (bjj_host_alloc; a host clock around `steps` host-flavour calls).
Every arm is warmed up first; the arms then run alternately `repeats` times, and each rate is reported per run with its
mean and spread (max - min over mean).  After every timed round: ok[] of arms 1 and 2 equal on every lane, ok[] of arm
3 equal to arm 1's on the lanes whose key is in the set (a signature by a key outside the set verifies there), and the
key indices of arms 1 and 4 equal to the indices known in advance.  The card's name and power limit are read in the
same run.  Writes DIR/verify_keyset_lookup.json and prints it.
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

from bench_verify_base import alternate, card_info  # noqa: E402

NONE = 0xFFFFFFFF


def corrupt(sig64, msg, seed):
    """about 1 lane in 10 corrupted in place, in five classes; returns the number of corrupted lanes"""
    n = len(sig64)
    rng = np.random.default_rng(seed)
    lanes = rng.permutation(n)[: n // 10]
    for k, part in enumerate(np.array_split(lanes, 5)):
        if k == 0:
            sig64[part, 32 + rng.integers(0, 31, size=len(part))] ^= (1 << rng.integers(0, 8, size=len(part))).astype(np.uint8)
        elif k == 1:
            msg[part, rng.integers(0, 31, size=len(part))] ^= (1 << rng.integers(0, 8, size=len(part))).astype(np.uint8)
        elif k == 2:
            msg[part] = 0xFF
        elif k == 3:
            sig64[part, 31] |= 0x7F
        else:
            sig64[part, 0] ^= 0x5A
    return len(lanes)


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, help="directory for verify_keyset_lookup.json")
    ap.add_argument("--log2-sigs", type=int, default=21)
    ap.add_argument("--keys", default="1,256,65536", help="comma-separated key-set sizes")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--repeats", type=int, default=3, help="alternating runs of every arm (at least 2)")
    args = ap.parse_args()
    if args.repeats < 2 or args.steps < 1:
        raise SystemExit("--repeats must be at least 2 and --steps at least 1")

    import torch
    import babyjubjub_rs_b200 as bjj
    if not torch.cuda.is_available():
        raise SystemExit("bench_verify_keyset_lookup.py needs a CUDA device: there is no CPU fallback")
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
        # ---- inputs ---------------------------------------------------------------------------------------------
        n_out = n_keys // 19 + 1
        rng = np.random.default_rng(20261023 + n_keys)
        priv = rng.integers(0, 256, size=(n_keys + n_out, 32), dtype=np.uint8)
        who = rng.integers(0, n_keys, size=n)
        outside = rng.random(n) < 0.05
        who[outside] = n_keys + rng.integers(0, n_out, size=int(outside.sum()))
        msgs_np = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
        msgs_np[:, 31] &= 0x2F                             # < Q: every lane signs
        dpriv = torch.from_numpy(priv).to(dev)
        dk = dpriv[torch.from_numpy(who).to(dev)].contiguous()
        dm = torch.from_numpy(msgs_np).to(dev)
        dsig, dst = t((n, 64)), t((n,))
        check(lib.bjj_sign_compressed_batch_dev(ctx, n, p(dk), p(dm), p(dsig), p(dst), sp), "sign_compressed")
        dax, day, dpk = t((n_keys + n_out, 32)), t((n_keys + n_out, 32)), t((n_keys + n_out, 32))
        check(lib.bjj_public_batch_dev(ctx, n_keys + n_out, p(dpriv), p(dax), p(day), sp), "public")
        check(lib.bjj_compress_batch_dev(ctx, n_keys + n_out, p(dax), p(day), p(dpk), sp), "compress")
        torch.cuda.synchronize()
        check(lib.bjj_sync(ctx), "bjj_sync")
        assert not dst.any().item()
        sig64, ax, ay, comp = (a.cpu().numpy() for a in (dsig, dax, day, dpk))
        ax, ay = ax[:n_keys].copy(), ay[:n_keys].copy()
        msg = msgs_np.copy()
        corrupted = corrupt(sig64, msg, 0x100C + n_keys)
        pk32 = comp[who]
        known = np.where(outside, NONE, who).astype("<u4")        # what the lookup must find
        known_ok = np.where(outside, 0, who).astype("<u4")        # arm 2's indices: a valid key for every lane
        found = ~outside
        del dk, dm, dsig, dst, dax, day, dpk, dpriv

        torch.cuda.synchronize()
        handle = ctypes.c_void_p()
        t0 = time.perf_counter()
        check(lib.bjj_keyset_create(ctx, n_keys, p(ax), p(ay), None, ctypes.byref(handle)), "keyset_create")
        create_s = time.perf_counter() - t0
        kh = handle

        # ---- device-resident: CUDA events ----------------------------------------------------------------------
        dsg, dpk, dmg = (torch.from_numpy(a).to(dev) for a in (sig64, pk32, msg))
        didx = torch.from_numpy(known_ok.view(np.uint8).reshape(n, 4).copy()).to(dev)
        ok1, ok2, ok3 = t((n,)), t((n,)), t((n,))
        st1, st2, st3 = t((n,)), t((n,)), t((n,))
        ki1, ki4 = t((n, 4)), t((n, 4))
        for i, o in enumerate((ok1, ok2, ok3, ki1, ki4)):
            o.fill_(0xE0 + i)
        variants = {
            "verify_keyset_lookup_compressed_batch_dev": lambda: check(lib.bjj_verify_keyset_lookup_compressed_batch_dev(
                ctx, kh, n, p(dsg), p(dpk), p(dmg), p(ok1), p(st1), p(ki1), sp), "verify_keyset_lookup"),
            "verify_keyset_compressed_batch_dev": lambda: check(lib.bjj_verify_keyset_compressed_batch_dev(
                ctx, kh, n, p(didx), p(dsg), p(dmg), p(ok2), p(st2), sp), "verify_keyset_compressed"),
            "verify_compressed_batch_dev": lambda: check(lib.bjj_verify_compressed_batch_dev(
                ctx, n, p(dsg), p(dpk), p(dmg), p(ok3), p(st3), sp), "verify_compressed"),
            "keyset_lookup_batch_dev": lambda: check(lib.bjj_keyset_lookup_batch_dev(ctx, kh, n, p(dpk), p(ki4), sp), "lookup"),
        }
        dfound = torch.from_numpy(found).to(dev)

        def compare():
            torch.cuda.synchronize()
            a, b, c = ok1.cpu().numpy(), ok2.cpu().numpy(), ok3.cpu().numpy()
            k1, k4 = ki1.cpu().numpy().view("<u4").ravel(), ki4.cpu().numpy().view("<u4").ravel()
            mismatches.append(int((a != b).sum()) + int((a[found] != c[found]).sum()) + int((k1 != known).sum())
                              + int((k4 != known).sum()))
        device_resident = alternate(variants, dev_timed, args.warmup, args.repeats, compare)
        accepted = int(ok1.sum().item())
        accepted_found_straus = int((ok3.bool() & dfound).sum().item())
        del dsg, dpk, dmg, didx, ok1, ok2, ok3, st1, st2, st3, ki1, ki4, dfound

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
            hsg, hpk, hmg, hidx = host_array((n, 64)), host_array((n, 32)), host_array((n, 32)), host_array((n, 4))
            hsg[...], hpk[...], hmg[...] = sig64, pk32, msg
            hidx[...] = known_ok.view(np.uint8).reshape(n, 4)
            h_ok = [host_array((n,)) for _ in range(3)]
            h_st = [host_array((n,)) for _ in range(3)]
            h_ki = [host_array((n, 4)) for _ in range(2)]
            for i, o in enumerate(h_ok + h_ki):
                o[...] = 0xE0 + i

            def compare_host():
                a, b, c = h_ok
                k1, k4 = (k.view("<u4").ravel() for k in h_ki)
                mismatches.append(int((a != b).sum()) + int((a[found] != c[found]).sum()) + int((k1 != known).sum())
                                  + int((k4 != known).sum()))
            end_to_end = alternate({
                "verify_keyset_lookup_compressed_batch": lambda: check(lib.bjj_verify_keyset_lookup_compressed_batch(
                    ctx, kh, n, p(hsg), p(hpk), p(hmg), p(h_ok[0]), p(h_st[0]), p(h_ki[0])), "verify_keyset_lookup"),
                "verify_keyset_compressed_batch": lambda: check(lib.bjj_verify_keyset_compressed_batch(
                    ctx, kh, n, p(hidx), p(hsg), p(hmg), p(h_ok[1]), p(h_st[1])), "verify_keyset_compressed"),
                "verify_compressed_batch": lambda: check(lib.bjj_verify_compressed_batch(
                    ctx, n, p(hsg), p(hpk), p(hmg), p(h_ok[2]), p(h_st[2])), "verify_compressed"),
                "keyset_lookup_batch": lambda: check(lib.bjj_keyset_lookup_batch(ctx, kh, n, p(hpk), p(h_ki[1])), "lookup"),
            }, host_timed, args.warmup, args.repeats, compare_host)
        finally:
            for ptr in pinned:
                lib.bjj_host_free(ptr)
        lib.bjj_keyset_destroy(ctx, kh)

        entry = {
            "keys": n_keys,
            "keys_outside_set": n_out,
            "lanes_outside_set": int(outside.sum()),
            "keyset_create_s": round(create_s, 4),
            "corrupted_lanes": corrupted,
            "accepted_lanes": accepted,
            "accepted_found_lanes_verify_compressed": accepted_found_straus,
            "device_resident": device_resident,
            "end_to_end_pinned": end_to_end,
            "ratios": {
                "dev_lookup_verify_over_known_index": ratio(device_resident, "verify_keyset_lookup_compressed_batch_dev",
                                                            "verify_keyset_compressed_batch_dev"),
                "dev_lookup_verify_over_verify_compressed": ratio(device_resident, "verify_keyset_lookup_compressed_batch_dev",
                                                                  "verify_compressed_batch_dev"),
                "e2e_lookup_verify_over_known_index": ratio(end_to_end, "verify_keyset_lookup_compressed_batch",
                                                            "verify_keyset_compressed_batch"),
                "e2e_lookup_verify_over_verify_compressed": ratio(end_to_end, "verify_keyset_lookup_compressed_batch",
                                                                  "verify_compressed_batch"),
            },
        }
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
        "mismatched_lanes_per_timed_round": mismatches,
    }
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "verify_keyset_lookup.json"), "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(report, indent=1))
    if any(mismatches):
        raise SystemExit("the arms disagree")


if __name__ == "__main__":
    main()
