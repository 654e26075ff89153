"""Throughput of verify_schnorr on the signer's unreduced s: bjj_verify_schnorr_base_batch (one key's comb table),
bjj_verify_schnorr_keyset_batch (a key index per lane, a compact comb per key) and bjj_verify_schnorr_wide_batch (any
key per lane, Straus path) next to bjj_verify_schnorr_batch on s reduced beforehand, on one GPU, for key sets of 1, 256
and 65,536 keys.

    python babyjubjub-rs_b200/tools/bench_verify_schnorr_comb.py --out DIR [--log2-sigs 21] [--keys 1,256,65536]
                                                                 [--steps 10] [--warmup 2] [--repeats 3]

Inputs, per key-set size K: K seeded private keys, a seeded random key index per lane, and 2^21 Schnorr signatures made
on the device by bjj_sign_schnorr_batch_dev with seeded 1024-bit nonces (so s is 40 words, as the reference's signer
makes it) over random messages below Q; then about 10 % of the lanes are corrupted on the host (a bit of s, a bit of
msg, or r replaced by the next lane's r).  The reference arm's s mod SUBORDER is computed on the host before timing.
Measures:
  - device-resident (CUDA events around `steps` back-to-back calls on one stream, closed by a synchronise): the keyset
    and wide forms and bjj_verify_schnorr_batch_dev, and at K = 1 also the base form with a FixedBase of the key;
  - end to end from page-locked buffers (bjj_host_alloc; a host clock around `steps` host-flavour calls, each of which
    returns with its results in place): the same arms.
Every arm is warmed up first; the arms then run alternately `repeats` times, and each rate is reported per run with its
mean and spread (max - min over mean).  The ok[] arrays of all arms are compared on every lane after every timed round.
The card's name and power limit are read in the same run.  Writes DIR/verify_schnorr_comb.json and prints it.
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

SUBORDER = 2736030358979909402780800718157159386076813972158567259200215660948447373041
NONCE_WORDS, S_WORDS = 32, 40


def corrupt(rx, ry, s, msg, seed):
    """about 1 lane in 10 corrupted in place: a bit of s, a bit of msg, or r taken from the next lane"""
    n = len(rx)
    rng = np.random.default_rng(seed)
    cls = np.where(rng.integers(0, 10, size=n) == 0, rng.integers(0, 3, size=n), -1)
    i = np.nonzero(cls == 0)[0]
    s[i, rng.integers(0, 4 * S_WORDS, size=len(i))] ^= (1 << rng.integers(0, 8, size=len(i))).astype(np.uint8)
    i = np.nonzero(cls == 1)[0]
    msg[i, rng.integers(0, 31, size=len(i))] ^= (1 << rng.integers(0, 8, size=len(i))).astype(np.uint8)
    i = np.nonzero(cls == 2)[0]
    rx[i], ry[i] = rx[(i + 1) % n].copy(), ry[(i + 1) % n].copy()
    return int((cls >= 0).sum())


def reduce_s(s):
    w = 4 * S_WORDS
    raw = s.tobytes()
    return np.frombuffer(b"".join((int.from_bytes(raw[w * i:w * (i + 1)], "little") % SUBORDER).to_bytes(32, "little")
                                  for i in range(len(s))), np.uint8).reshape(-1, 32).copy()


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, help="directory for verify_schnorr_comb.json")
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
        raise SystemExit("bench_verify_schnorr_comb.py needs a CUDA device: there is no CPU fallback")
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

    def ratios(table, ref):
        return {a: round(v["M_per_s_mean"] / table[ref]["M_per_s_mean"], 3) for a, v in table.items() if a != ref}

    results = []
    mismatches = []
    for n_keys in [int(k) for k in args.keys.split(",")]:
        # ---- inputs: K keys, a random key per lane, n signatures made on the device, 10 % corrupted ----------------
        rng = np.random.default_rng(20261023 + n_keys)
        priv = rng.integers(0, 256, size=(n_keys, 32), dtype=np.uint8)
        idx = rng.integers(0, n_keys, size=n).astype("<u4")
        msgs_np = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
        msgs_np[:, 31] &= 0x2F                             # < Q: every lane signs
        nonces = rng.integers(0, 256, size=(n, 4 * NONCE_WORDS), dtype=np.uint8)
        dpriv = torch.from_numpy(priv).to(dev)
        didx = torch.from_numpy(idx.astype(np.int64)).to(dev)
        dk = dpriv[didx].contiguous()
        dm, dn = torch.from_numpy(msgs_np).to(dev), torch.from_numpy(nonces).to(dev)
        drx, dry, ds, dst = t((n, 32)), t((n, 32)), t((n, 4 * S_WORDS)), t((n,))
        check(lib.bjj_sign_schnorr_batch_dev(ctx, n, p(dk), p(dm), p(dn), NONCE_WORDS, p(drx), p(dry), p(ds), p(dst), sp), "sign_schnorr")
        dax, day = t((n_keys, 32)), t((n_keys, 32))
        check(lib.bjj_public_batch_dev(ctx, n_keys, p(dpriv), p(dax), p(day), sp), "public")
        torch.cuda.synchronize()
        check(lib.bjj_sync(ctx), "bjj_sync")
        assert not dst.any().item()
        rx, ry, s, ax, ay = (a.cpu().numpy() for a in (drx, dry, ds, dax, day))
        msg = msgs_np.copy()
        corrupted = corrupt(rx, ry, s, msg, 0x5C40 + n_keys)
        del dk, dm, dn, drx, dry, ds, dst, dax, day, dpriv, didx
        axn, ayn = ax[idx], ay[idx]
        s_red = reduce_s(s)                                # the reference arm's input, prepared outside its time

        handle = ctypes.c_void_p()
        check(lib.bjj_keyset_create(ctx, n_keys, p(ax), p(ay), None, ctypes.byref(handle)), "keyset_create")
        kh = handle
        base = bjj.FixedBase((int.from_bytes(ax[0].tobytes(), "little"), int.from_bytes(ay[0].tobytes(), "little")), eng) \
            if n_keys == 1 else None

        # ---- device-resident: CUDA events ----------------------------------------------------------------------
        dmsg, drx, dry, ds, dsr, dax, day = (torch.from_numpy(np.ascontiguousarray(c)).to(dev) for c in (msg, rx, ry, s, s_red, axn, ayn))
        d_idx = torch.from_numpy(idx.view(np.uint8).copy()).to(dev)
        names = ["verify_schnorr_batch_dev", "verify_schnorr_keyset_batch_dev", "verify_schnorr_wide_batch_dev"]
        if base is not None:
            names.append("verify_schnorr_base_batch_dev")
        oks = {k: t((n,)) for k in names}
        sts = {k: t((n,)) for k in names}
        sig = (p(dmsg), p(drx), p(dry), p(ds), S_WORDS)
        variants = {
            "verify_schnorr_batch_dev": lambda: check(lib.bjj_verify_schnorr_batch_dev(
                ctx, n, p(dax), p(day), p(dmsg), p(drx), p(dry), p(dsr), p(oks["verify_schnorr_batch_dev"]),
                p(sts["verify_schnorr_batch_dev"]), sp), "verify_schnorr"),
            "verify_schnorr_keyset_batch_dev": lambda: check(lib.bjj_verify_schnorr_keyset_batch_dev(
                ctx, kh, n, p(d_idx), *sig, p(oks["verify_schnorr_keyset_batch_dev"]), p(sts["verify_schnorr_keyset_batch_dev"]), sp),
                "verify_schnorr_keyset"),
            "verify_schnorr_wide_batch_dev": lambda: check(lib.bjj_verify_schnorr_wide_batch_dev(
                ctx, n, p(dax), p(day), *sig, p(oks["verify_schnorr_wide_batch_dev"]), p(sts["verify_schnorr_wide_batch_dev"]), sp),
                "verify_schnorr_wide"),
        }
        if base is not None:
            variants["verify_schnorr_base_batch_dev"] = lambda: check(lib.bjj_verify_schnorr_base_batch_dev(
                ctx, base.handle, n, *sig, p(oks["verify_schnorr_base_batch_dev"]), p(sts["verify_schnorr_base_batch_dev"]), sp),
                "verify_schnorr_base")
        for i, o in enumerate(oks.values()):
            o.fill_(0xE0 + i)

        def compare():
            torch.cuda.synchronize()
            ref = oks["verify_schnorr_batch_dev"]
            mismatches.append(sum(int((o != ref).sum().item()) for o in oks.values()) +
                              sum(int(st_.any().item()) for st_ in sts.values()))
        device_resident = alternate(variants, dev_timed, args.warmup, args.repeats, compare)
        accepted = int(oks["verify_schnorr_batch_dev"].sum().item())
        del dmsg, drx, dry, ds, dsr, dax, day, d_idx, oks, sts

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
            hmsg, hrx, hry, hsr, hax, hay = (host_array((n, 32)) for _ in range(6))
            hs, hidx = host_array((n, 4 * S_WORDS)), host_array((n, 4))
            for dst_, src in zip((hmsg, hrx, hry, hsr, hax, hay, hs), (msg, rx, ry, s_red, axn, ayn, s)):
                dst_[...] = src
            hidx[...] = idx.view(np.uint8).reshape(n, 4)
            hok = {k[:-4]: host_array((n,)) for k in names}
            hst = host_array((n,))
            hsig = (p(hmsg), p(hrx), p(hry), p(hs), S_WORDS)
            host_variants = {
                "verify_schnorr_batch": lambda: check(lib.bjj_verify_schnorr_batch(
                    ctx, n, p(hax), p(hay), p(hmsg), p(hrx), p(hry), p(hsr), p(hok["verify_schnorr_batch"]), p(hst)), "verify_schnorr"),
                "verify_schnorr_keyset_batch": lambda: check(lib.bjj_verify_schnorr_keyset_batch(
                    ctx, kh, n, p(hidx), *hsig, p(hok["verify_schnorr_keyset_batch"]), p(hst)), "verify_schnorr_keyset"),
                "verify_schnorr_wide_batch": lambda: check(lib.bjj_verify_schnorr_wide_batch(
                    ctx, n, p(hax), p(hay), *hsig, p(hok["verify_schnorr_wide_batch"]), p(hst)), "verify_schnorr_wide"),
            }
            if base is not None:
                host_variants["verify_schnorr_base_batch"] = lambda: check(lib.bjj_verify_schnorr_base_batch(
                    ctx, base.handle, n, *hsig, p(hok["verify_schnorr_base_batch"]), p(hst)), "verify_schnorr_base")
            for i, o in enumerate(hok.values()):
                o[...] = 0xD0 + i

            def compare_host():
                ref = hok["verify_schnorr_batch"]
                mismatches.append(sum(int((o != ref).sum()) for o in hok.values()) + int(hst.any()))
            end_to_end = alternate(host_variants, host_timed, args.warmup, args.repeats, compare_host)
        finally:
            for ptr in pinned:
                lib.bjj_host_free(ptr)
        if base is not None:
            base.close()
        lib.bjj_keyset_destroy(ctx, kh)

        entry = {
            "keys": n_keys,
            "s_words": S_WORDS,
            "corrupted_lanes": corrupted,
            "accepted_lanes": accepted,
            "device_resident": device_resident,
            "end_to_end_pinned": end_to_end,
            "ratios_over_verify_schnorr": {"device_resident": ratios(device_resident, "verify_schnorr_batch_dev"),
                                           "end_to_end_pinned": ratios(end_to_end, "verify_schnorr_batch")},
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
        "ok_mismatched_lanes_per_timed_round": mismatches,
    }
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "verify_schnorr_comb.json"), "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(report, indent=1))
    if any(mismatches):
        raise SystemExit("the verify_schnorr forms disagree")


if __name__ == "__main__":
    main()
