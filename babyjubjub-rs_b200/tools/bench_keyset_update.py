"""Cost of editing a key set in place (bjj_keyset_append, bjj_keyset_replace) against creating it again, and verify
throughput on a set grown by appends against one created in a single call, on one GPU.

    python babyjubjub-rs_b200/tools/bench_keyset_update.py --out DIR [--base-keys 65536] [--edits 1,64,511,4096]
                                                           [--log2-sigs 21] [--steps 5] [--warmup 1] [--repeats 3]

1. Edits.  Per run and per k: bjj_keyset_create of base + k keys (what a change of k keys costs without these calls),
   then, on a fresh set of `base` keys, bjj_keyset_replace of k keys in the middle and bjj_keyset_append of k new keys.
   Each is one synchronous call timed with a host clock.  The runs alternate `repeats` times.
2. Verify on a grown set.  The same `base` keys once as bjj_keyset_create of half of them plus 32 appends of the rest,
   and once as one bjj_keyset_create.  2^21 signatures by seeded keys of the set (about 10 % corrupted), and their
   compressed keys: bjj_verify_keyset_batch_dev and bjj_verify_keyset_lookup_compressed_batch_dev on each set, CUDA
   events around `steps` back-to-back calls, the two sets alternating `repeats` times; ok[] equal on every lane.
3. Memory: the device bytes each of the two sets holds (the drop in free memory when it is built).
4. Sets per context: one-key sets created until bjj_keyset_create fails (or --max-sets): each reserves address space for
   total device memory / 396,480 B tables, so the address space, not device memory, bounds how many a process holds.
The card's name and power limit are read in the same run.  Writes DIR/keyset_update.json and prints it.
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


def p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, help="directory for keyset_update.json")
    ap.add_argument("--base-keys", type=int, default=65536)
    ap.add_argument("--edits", default="1,64,511,4096", help="comma-separated numbers of keys per edit")
    ap.add_argument("--log2-sigs", type=int, default=21)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--repeats", type=int, default=3, help="alternating runs (at least 2)")
    ap.add_argument("--max-sets", type=int, default=4096, help="one-key sets to create in part 4 before giving up")
    args = ap.parse_args()
    if args.repeats < 2 or args.steps < 1 or args.base_keys < 64:
        raise SystemExit("--repeats must be at least 2, --steps at least 1 and --base-keys at least 64")

    import torch
    import babyjubjub_rs_b200 as bjj
    if not torch.cuda.is_available():
        raise SystemExit("bench_keyset_update.py needs a CUDA device: there is no CPU fallback")
    dev = torch.device("cuda", 0)
    eng = bjj.Engine(0)
    lib, ctx = eng.lib, eng.ctx
    edits = [int(k) for k in args.edits.split(",")]
    base, kmax = args.base_keys, max(edits)

    def check(rc, what):
        if rc != 0:
            raise RuntimeError("%s failed: %d" % (what, rc))

    rng = np.random.default_rng(9)
    priv = rng.integers(0, 256, size=(base + 2 * kmax, 32), dtype=np.uint8)
    ax, ay = eng.public_batch(priv)

    def create(lo, hi):
        h = ctypes.c_void_p()
        t0 = time.perf_counter()
        check(lib.bjj_keyset_create(ctx, hi - lo, p(ax[lo:hi]), p(ay[lo:hi]), None, ctypes.byref(h)), "bjj_keyset_create")
        return h, time.perf_counter() - t0

    # ---- 1. edits ---------------------------------------------------------------------------------------
    t_create, t_append, t_replace = ({k: [] for k in edits} for _ in range(3))
    h, _ = create(0, base)                       # warm-up: modules, scratch
    lib.bjj_keyset_destroy(ctx, h)
    for _ in range(args.repeats):
        for k in edits:
            h, t = create(0, base + k)
            lib.bjj_keyset_destroy(ctx, h)
            t_create[k].append(t)
            h, _ = create(0, base)
            mid = base // 2 - k // 2
            new = slice(base + kmax, base + kmax + k)
            t0 = time.perf_counter()
            check(lib.bjj_keyset_replace(ctx, h, mid, k, p(ax[new]), p(ay[new]), None), "bjj_keyset_replace")
            t_replace[k].append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            check(lib.bjj_keyset_append(ctx, h, k, p(ax[base:base + k]), p(ay[base:base + k]), None), "bjj_keyset_append")
            t_append[k].append(time.perf_counter() - t0)
            lib.bjj_keyset_destroy(ctx, h)

    def ms(v):
        return {"ms_runs": [round(x * 1e3, 3) for x in v], "ms_mean": round(sum(v) / len(v) * 1e3, 3)}
    edit_rows = []
    for k in edits:
        c = sum(t_create[k]) / len(t_create[k])
        edit_rows.append({"k": k, "create_base_plus_k": ms(t_create[k]), "append": ms(t_append[k]), "replace": ms(t_replace[k]),
                          "create_over_append": round(c / (sum(t_append[k]) / len(t_append[k])), 1),
                          "create_over_replace": round(c / (sum(t_replace[k]) / len(t_replace[k])), 1)})
        print(json.dumps(edit_rows[-1]), flush=True)

    # ---- 2. verify on a grown set, 3. memory -------------------------------------------------------------------
    def free_bytes():
        torch.cuda.synchronize(dev)
        return torch.cuda.mem_get_info(dev)[0]
    f0 = free_bytes()
    half, step = base // 2, (base - base // 2) // 32
    grown, _ = create(0, half)
    for j in range(32):
        lo = half + j * step
        hi = base if j == 31 else lo + step
        check(lib.bjj_keyset_append(ctx, grown, hi - lo, p(ax[lo:hi]), p(ay[lo:hi]), None), "bjj_keyset_append")
    f1 = free_bytes()
    created, _ = create(0, base)
    f2 = free_bytes()

    n = 1 << args.log2_sigs
    idx = rng.integers(0, base, size=n).astype(np.uint32)
    msg = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    msg[:, 31] &= 0x2F
    r8x, r8y, s, st = eng.sign_batch(priv[idx], msg)
    sig64, st2 = eng.sign_compressed_batch(priv[idx], msg)
    assert not st.any() and not st2.any()
    bad = rng.random(n) < 0.1
    col = rng.integers(0, 31, size=n)
    s[bad, col[bad]] ^= 1
    sig64[bad, 32 + col[bad]] ^= 1
    pk32 = eng.compress_batch(ax[:base], ay[:base])[idx]
    d = {k: torch.from_numpy(np.ascontiguousarray(v).view(np.uint8).reshape(n, -1)).to(dev)
         for k, v in dict(idx=idx, r8x=r8x, r8y=r8y, s=s, msg=msg, sig64=sig64, pk32=pk32).items()}
    ok = {name: torch.zeros(n, dtype=torch.uint8, device=dev) for name in ("grown", "created")}
    st_d = torch.zeros(n, dtype=torch.uint8, device=dev)
    ki_d = torch.zeros(4 * n, dtype=torch.uint8, device=dev)
    stream = torch.cuda.Stream(dev)          # a stream of its own: NULL would select the context's stream, not the events'
    sp = ctypes.c_void_p(stream.cuda_stream)
    sets = {"grown": grown, "created": created}
    torch.cuda.synchronize(dev)

    def plain(name):
        check(lib.bjj_verify_keyset_batch_dev(ctx, sets[name], n, d["idx"].data_ptr(), d["r8x"].data_ptr(), d["r8y"].data_ptr(),
                                              d["s"].data_ptr(), d["msg"].data_ptr(), ok[name].data_ptr(), sp), "verify_keyset")

    def lookup(name):
        check(lib.bjj_verify_keyset_lookup_compressed_batch_dev(ctx, sets[name], n, d["sig64"].data_ptr(), d["pk32"].data_ptr(),
                                                                d["msg"].data_ptr(), ok[name].data_ptr(), st_d.data_ptr(),
                                                                ki_d.data_ptr(), sp), "verify_keyset_lookup_compressed")

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            fn()
        e1.record(stream)
        e1.synchronize()
        check(lib.bjj_sync(ctx), "bjj_sync")
        return n * args.steps / (e0.elapsed_time(e1) * 1e-3) / 1e6

    verify = {}
    for form, fn in (("verify_keyset_batch_dev", plain), ("verify_keyset_lookup_compressed_batch_dev", lookup)):
        equal = []

        def after():
            torch.cuda.synchronize(dev)
            equal.append(bool(torch.equal(ok["grown"], ok["created"])))
        res = alternate({"grown": lambda: fn("grown"), "created": lambda: fn("created")}, timed, args.warmup, args.repeats, after)
        frac = float(ok["created"].float().mean().item())
        assert all(equal), form
        verify[form] = {"grown": res["grown"], "created": res["created"], "ok_equal_every_round": all(equal),
                        "ok_fraction": round(frac, 4)}
        print(json.dumps({form: verify[form]}), flush=True)
    lib.bjj_keyset_destroy(ctx, grown)
    lib.bjj_keyset_destroy(ctx, created)

    # ---- 4. sets per context: every set reserves address space for a full device of tables ---------------------
    total = torch.cuda.mem_get_info(dev)[1]
    handles, rc, t0 = [], 0, time.perf_counter()
    while len(handles) < args.max_sets:
        h = ctypes.c_void_p()
        rc = lib.bjj_keyset_create(ctx, 1, p(ax[:1]), p(ay[:1]), None, ctypes.byref(h))
        if rc != 0:
            break
        handles.append(h)
    sets_s = time.perf_counter() - t0
    for h in handles:
        lib.bjj_keyset_destroy(ctx, h)
    check(lib.bjj_sync(ctx), "bjj_sync")
    after = ctypes.c_void_p()
    check(lib.bjj_keyset_create(ctx, 1, p(ax[:1]), p(ay[:1]), None, ctypes.byref(after)), "bjj_keyset_create after the limit")
    lib.bjj_keyset_destroy(ctx, after)
    per_set = -(-(total // (4130 * 96) * 4130 * 96) // (2 << 20)) * (2 << 20)
    sets = {"one_key_sets_created": len(handles), "stopped_by": "rc %d" % rc if rc else "--max-sets",
            "reserved_bytes_per_set": per_set, "reserved_bytes_total": per_set * len(handles),
            "create_ms_mean": round(sets_s / max(len(handles), 1) * 1e3, 3)}
    print(json.dumps({"sets_per_context": sets}), flush=True)

    report = {
        "tool": "babyjubjub-rs_b200/tools/bench_keyset_update.py",
        "card": card_info(0),
        "base_keys": base,
        "edits": edit_rows,
        "verify_on_grown_set": {"grown": "bjj_keyset_create(%d) + 32 x bjj_keyset_append(%d)" % (half, step),
                                "created": "bjj_keyset_create(%d)" % base, "lanes": n, "steps": args.steps, **verify},
        "device_bytes": {"grown": f0 - f1, "created": f1 - f2, "tables_alone": base * 4130 * 96},
        "sets_per_context": sets,
        "args": {k: v for k, v in vars(args).items() if k != "out"},
    }
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "keyset_update.json"), "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(report, indent=1))


if __name__ == "__main__":
    main()
