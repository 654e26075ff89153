"""Throughput of verify against one key on the comb path (bjj_verify_base_batch) next to bjj_verify_batch with the key
in every lane, on one GPU.

    python babyjubjub-rs_b200/tools/bench_verify_base.py --out DIR [--log2-sigs 21] [--steps 10] [--warmup 3] [--repeats 3]

Inputs: one seeded key and 2^21 signatures of it over random messages below Q, made on the device by
bjj_sign_batch_dev, then about 10 % of the lanes corrupted on the host in the classes of bench.py that apply to one
key (flipped S bit, flipped msg bit, another lane's R8, S + SUBORDER (stays valid), msg > Q, R8 off the curve, R8 one
of (0, 0), (0, 1), (0, -1)).  Measures:
  - device-resident (CUDA events around `steps` back-to-back calls on one stream, closed by a synchronise):
    bjj_verify_batch_dev (A broadcast) against bjj_verify_base_batch_dev;
  - end to end from page-locked buffers (bjj_host_alloc; a host clock around `steps` host-flavour calls, each of which
    returns with its results in place): bjj_verify_batch against bjj_verify_base_batch;
  - the adversarial case: bjj_verify_base_batch_dev on the same signatures with every R8 moved off the curve
    (x + 1), so that every lane takes the literal replay of the reference's sum, next to bjj_verify_batch_dev on them.
Every variant of a comparison is warmed up first; the variants then run alternately `repeats` times, and each rate is
reported per run with its mean and its spread (max - min over mean).  The ok[] arrays of the two calls are compared on
every lane after every timed run.  The card's name and power limit are read in the same run.  Writes
DIR/verify_base.json and prints it.
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

Q = 21888242871839275222246405745257275088548364400416034343698204186575808495617
SUBORDER = 21888242871839275222246405745257275088614511777268538073601725287587578984328 >> 3


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


def alternate(variants, timed, warmup, repeats, after=None):
    """warms up every variant, then times them alternately `repeats` times (calling after() after each round);
    {name: summary}"""
    for fn in variants.values():
        for _ in range(warmup):
            fn()
    runs = {name: [] for name in variants}
    for _ in range(repeats):
        for name, fn in variants.items():
            runs[name].append(timed(fn))
        if after:
            after()
    return {name: summary(r) for name, r in runs.items()}


def _int(row):
    return int.from_bytes(row.tobytes(), "little")


def _row(v):
    return np.frombuffer(int(v).to_bytes(32, "little"), dtype=np.uint8)


def corrupt_one_key(r8x, r8y, s, msg, seed):
    """about 1 lane in 10 corrupted in place, by class; returns the number of corrupted lanes"""
    n = len(r8x)
    rng = np.random.default_rng(seed)
    cls = np.where(rng.integers(0, 10, size=n) == 0, rng.integers(0, 7, size=n), -1)
    orig = r8x.copy(), r8y.copy()
    idx = np.nonzero(cls == 0)[0]
    s[idx, rng.integers(0, 31, size=len(idx))] ^= (1 << rng.integers(0, 8, size=len(idx))).astype(np.uint8)
    idx = np.nonzero(cls == 1)[0]
    msg[idx, rng.integers(0, 31, size=len(idx))] ^= (1 << rng.integers(0, 8, size=len(idx))).astype(np.uint8)
    idx = np.nonzero(cls == 2)[0]
    r8x[idx], r8y[idx] = orig[0][(idx + 1) % n], orig[1][(idx + 1) % n]
    for i in np.nonzero(cls == 3)[0]:                      # stays valid: verify never range-checks S
        s[i] = _row(_int(s[i]) + SUBORDER)
    msg[cls == 4] = 0xFF
    for i in np.nonzero(cls == 5)[0]:
        r8x[i] = _row((_int(r8x[i]) + 1) % Q)
    specials = [(0, 0), (0, 1), (0, Q - 1)]
    for i in np.nonzero(cls == 6)[0]:
        x, y = specials[int(i) % 3]
        r8x[i], r8y[i] = _row(x), _row(y)
    return int((cls >= 0).sum())


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, help="directory for verify_base.json")
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
        raise SystemExit("bench_verify_base.py needs a CUDA device: there is no CPU fallback")
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

    # ---- inputs: one key, n signatures made on the device, 10 % corrupted ------------------------------------------
    rng = np.random.default_rng(20261021)
    key = rng.integers(0, 256, size=(1, 32), dtype=np.uint8)
    msgs_np = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    msgs_np[:, 31] &= 0x2F                                 # < 0x30 * 2^248 < Q: every lane signs
    dk = torch.from_numpy(np.repeat(key, n, 0)).to(dev)
    dm = torch.from_numpy(msgs_np).to(dev)
    drx, dry, ds, dst = t((n, 32)), t((n, 32)), t((n, 32)), t((n,))
    check(lib.bjj_sign_batch_dev(ctx, n, p(dk), p(dm), p(drx), p(dry), p(ds), p(dst), sp), "sign")
    dax, day = t((1, 32)), t((1, 32))
    check(lib.bjj_public_batch_dev(ctx, 1, p(dk), p(dax), p(day), sp), "public")
    torch.cuda.synchronize()
    check(lib.bjj_sync(ctx), "bjj_sync")
    assert not dst.any().item()
    r8x, r8y, s, ax, ay = (a.cpu().numpy() for a in (drx, dry, ds, dax, day))
    msg = msgs_np.copy()
    corrupted = corrupt_one_key(r8x, r8y, s, msg, 0xBA5E)
    del dk, dm, drx, dry, ds, dst, dax, day
    base = bjj.FixedBase((int.from_bytes(ax[0].tobytes(), "little"), int.from_bytes(ay[0].tobytes(), "little")), eng)
    bh = base.handle
    axn, ayn = np.repeat(ax, n, 0), np.repeat(ay, n, 0)
    mismatches = []

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

    def device_pair(cols):
        d = [torch.from_numpy(c).to(dev) for c in cols]
        d_ax, d_ay = torch.from_numpy(axn).to(dev), torch.from_numpy(ayn).to(dev)
        ok_v, ok_b = t((n,)), t((n,))
        ok_v.fill_(0xEE)
        ok_b.fill_(0xDD)

        def compare():
            torch.cuda.synchronize()
            mismatches.append(int((ok_v != ok_b).sum().item()))
        res = alternate({
            "verify_batch_dev": lambda: check(lib.bjj_verify_batch_dev(ctx, n, p(d[0]), p(d[1]), p(d[2]), p(d_ax), p(d_ay), p(d[3]),
                                                                       p(ok_v), sp), "verify"),
            "verify_base_batch_dev": lambda: check(lib.bjj_verify_base_batch_dev(ctx, bh, n, p(d[0]), p(d[1]), p(d[2]), p(d[3]),
                                                                                 p(ok_b), sp), "verify_base"),
        }, dev_timed, args.warmup, args.repeats, compare)
        accepted = int(ok_b.sum().item())
        return res, accepted

    device_resident, accepted = device_pair([r8x, r8y, s, msg])
    off_x = np.stack([_row((_int(x) + 1) % Q) for x in r8x])
    adversarial, adv_accepted = device_pair([off_x, r8y, s, msg])

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
        h = [host_array((n, 32)) for _ in range(6)]
        for dst_, src in zip(h, (r8x, r8y, s, axn, ayn, msg)):
            dst_[...] = src
        hok_v, hok_b = host_array((n,)), host_array((n,))
        hok_v[...], hok_b[...] = 0xEE, 0xDD

        def compare_host():
            mismatches.append(int((hok_v != hok_b).sum()))
        end_to_end = alternate({
            "verify_batch": lambda: check(lib.bjj_verify_batch(ctx, n, *[p(a) for a in h], p(hok_v)), "verify"),
            "verify_base_batch": lambda: check(lib.bjj_verify_base_batch(ctx, bh, n, p(h[0]), p(h[1]), p(h[2]), p(h[5]), p(hok_b)),
                                               "verify_base"),
        }, host_timed, args.warmup, args.repeats, compare_host)
    finally:
        for ptr in pinned:
            lib.bjj_host_free(ptr)
    base.close()
    eng.close()

    def ratio(table, a, b):
        return round(table[a]["M_per_s_mean"] / table[b]["M_per_s_mean"], 3)

    report = {
        "card": card_info(0),
        "torch_device_name": torch.cuda.get_device_name(0),
        "signatures": n,
        "corrupted_lanes": corrupted,
        "accepted_lanes": accepted,
        "steps": steps,
        "warmup": args.warmup,
        "repeats": args.repeats,
        "device_resident": device_resident,
        "end_to_end_pinned": end_to_end,
        "adversarial_all_r8_off_curve_device_resident": adversarial,
        "adversarial_accepted_lanes": adv_accepted,
        "ratios": {
            "dev_base_over_verify": ratio(device_resident, "verify_base_batch_dev", "verify_batch_dev"),
            "e2e_base_over_verify": ratio(end_to_end, "verify_base_batch", "verify_batch"),
            "adversarial_dev_base_over_verify": ratio(adversarial, "verify_base_batch_dev", "verify_batch_dev"),
        },
        "ok_mismatched_lanes_per_timed_round": mismatches,
    }
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "verify_base.json"), "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(report, indent=1))
    if any(mismatches):
        raise SystemExit("verify_base_batch and verify_batch disagree")


if __name__ == "__main__":
    main()
