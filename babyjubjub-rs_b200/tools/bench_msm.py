"""Multi-scalar products R = sum_i k_i * P_i: bjj_msm_batch against the composed path on the same inputs, on one GPU.

    python babyjubjub-rs_b200/tools/bench_msm.py --out DIR [--log2-sizes 12,16,19,20,22,24] [--steps 3] [--warmup 1]
                                                 [--repeats 3] [--bits 0] [--profile-log2 20] [--multi]

Per size n (random on-curve points a_i * B8 made on the device, random 256-bit scalars):
  - msm_dev: bjj_msm_batch_dev on device arrays, CUDA events around `steps` back-to-back calls;
  - composed_dev: what a caller does without it, bjj_mul_scalar_batch_dev then bjj_add_batch_dev halving the list down
    to one point and bjj_affine_batch_dev, timed the same way;
  - msm_host: bjj_msm_batch from pinned host arrays (end to end, synchronous), host clock.
  The three alternate `repeats` times; the msm and composed results must be equal on every run.  Work: the algorithmic
  limb-MACs of the bucket method (DESIGN, "Multi-scalar products") over the 9.31 T/s IMAD.WIDE peak (DESIGN section 5).
--bits 8 / 16 forces the window width (BJJ_MSM_BITS, read once per process): run the tool once per width to measure
the crossover.  --profile-log2: one extra call under torch.profiler, per-kernel device times.  --multi: bjj_multi_msm_batch
at 1, 2, ... devices.  The card's name and power limit are read in the same run.  Writes DIR/msm.json and prints it.
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

IMAD_PEAK = 9.31e12          # IMAD.WIDE limb-MACs per second, DESIGN section 5
MUL_MACS = 128               # limb-MACs of one field multiplication (8 x 8 products + 8 x 8 reduction)


def work_macs(n, bits):
    """algorithmic limb-MACs of one call: per point 5M (prepare) and WINDOWS mixed additions (7M); per bucket the
    running sums (2 x 9M) and the final combination (c x 7M dbl + 9M per window)"""
    windows, half = 256 // bits + 1, 1 << (bits - 1)
    per_point = 5 + 7 * windows
    per_bucket = 18
    return MUL_MACS * (n * per_point + windows * half * per_bucket + windows * (bits * 7 + 9))


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True)
    ap.add_argument("--log2-sizes", default="12,16,19,20,22,24")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--bits", type=int, default=0, help="force the window width (8 or 16); 0 = chosen from n")
    ap.add_argument("--profile-log2", type=int, default=0)
    ap.add_argument("--multi", action="store_true")
    args = ap.parse_args()
    if args.bits:
        os.environ["BJJ_MSM_BITS"] = str(args.bits)

    import torch
    import babyjubjub_rs_b200 as bjj
    if not torch.cuda.is_available():
        raise SystemExit("bench_msm.py needs a CUDA device: there is no CPU fallback")
    dev = torch.device("cuda", 0)
    eng = bjj.Engine(0)
    lib, ctx = eng.lib, eng.ctx
    stream = torch.cuda.ExternalStream(eng.stream)
    out = {"card": card_info(0), "bits": args.bits or "auto (BJJ_MSM_C16_POINTS = 2^20)", "steps": args.steps,
           "repeats": args.repeats, "sizes": {}}

    def ptr(t):
        return ctypes.c_void_p(t.data_ptr())

    def ok(rc, what):
        if rc != 0:
            raise RuntimeError("%s returned %d" % (what, rc))

    rng = np.random.default_rng(1)
    for lg in [int(x) for x in args.log2_sizes.split(",")]:
        n = 1 << lg
        try:
            a = torch.from_numpy(rng.integers(0, 256, (n, 32), dtype=np.uint8)).to(dev)
            a[:, 31] &= 0x0F
            k = torch.from_numpy(rng.integers(0, 256, (n, 32), dtype=np.uint8)).to(dev)
            px, py = torch.empty_like(a), torch.empty_like(a)
            torch.cuda.synchronize()
            ok(lib.bjj_fixed_base_batch_dev(ctx, n, ptr(a), ptr(px), ptr(py), None), "fixed_base")
            ok(lib.bjj_sync(ctx), "sync")
            rx, ry = torch.empty((1, 32), dtype=torch.uint8, device=dev), torch.empty((1, 32), dtype=torch.uint8, device=dev)
            # composed-path buffers: products (x, y, z = 1) and two halving buffers
            cx, cy = torch.empty_like(a), torch.empty_like(a)
            cz = torch.zeros_like(a)
            cz[:, 0] = 1
            half = [tuple(torch.empty(((n + 1) // 2, 32), dtype=torch.uint8, device=dev) for _ in range(3)) for _ in range(2)]
            ax_, ay_ = torch.empty((1, 32), dtype=torch.uint8, device=dev), torch.empty((1, 32), dtype=torch.uint8, device=dev)
        except torch.cuda.OutOfMemoryError:
            out["sizes"][str(lg)] = {"skipped": "out of device memory"}
            continue
        torch.cuda.synchronize()

        def msm_dev():
            ok(lib.bjj_msm_batch_dev(ctx, n, ptr(px), ptr(py), ptr(k), ptr(rx), ptr(ry), None, None), "msm_dev")

        def composed_dev():
            ok(lib.bjj_mul_scalar_batch_dev(ctx, n, ptr(px), ptr(py), ptr(k), ptr(cx), ptr(cy), None), "mul_scalar_dev")
            # the products (x, y, 1), then halving between two buffers that never overwrite the constant z plane
            (sx, sy, sz), m, dst = (cx, cy, cz), n, 0
            while m > 1:
                h = m // 2
                dx, dy, dz = half[dst]
                ok(lib.bjj_add_batch_dev(ctx, h, ptr(sx), ptr(sy), ptr(sz), ptr(sx[h:]), ptr(sy[h:]), ptr(sz[h:]), ptr(dx), ptr(dy),
                                         ptr(dz), None), "add_dev")
                if m & 1:
                    ok(lib.bjj_add_batch_dev(ctx, 1, ptr(dx), ptr(dy), ptr(dz), ptr(sx[m - 1:]), ptr(sy[m - 1:]), ptr(sz[m - 1:]),
                                             ptr(dx), ptr(dy), ptr(dz), None), "add_dev")
                (sx, sy, sz), m, dst = half[dst], h, dst ^ 1
            ok(lib.bjj_affine_batch_dev(ctx, 1, ptr(sx), ptr(sy), ptr(sz), ptr(ax_), ptr(ay_), None), "affine_dev")

        hp = [torch.empty((n, 32), dtype=torch.uint8).pin_memory() for _ in range(3)]
        for h, d in zip(hp, (px, py, k)):
            h.copy_(d)
        hrx, hry = np.zeros((1, 32), np.uint8), np.zeros((1, 32), np.uint8)

        def msm_host():
            ok(lib.bjj_msm_batch(ctx, n, ptr(hp[0]), ptr(hp[1]), ptr(hp[2]), hrx.ctypes.data_as(ctypes.c_void_p),
                                 hry.ctypes.data_as(ctypes.c_void_p), None), "msm_host")

        def timed(fn):
            if fn is msm_host:
                t = time.perf_counter()
                for _ in range(args.steps):
                    fn()
                return n * args.steps / (time.perf_counter() - t) / 1e6
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(args.steps):
                fn()
            e1.record(stream)
            ok(lib.bjj_sync(ctx), "sync")
            e1.synchronize()
            return n * args.steps / (e0.elapsed_time(e1) / 1e3) / 1e6

        def check():
            ok(lib.bjj_sync(ctx), "sync")
            if not (torch.equal(rx, ax_) and torch.equal(ry, ay_) and np.array_equal(hrx, rx.cpu().numpy())
                    and np.array_equal(hry, ry.cpu().numpy())):
                raise RuntimeError("msm and the composed path differ at n = 2^%d" % lg)
            checks.append(True)

        checks = []
        res = alternate({"msm_dev": msm_dev, "composed_dev": composed_dev, "msm_host_pinned": msm_host}, timed, args.warmup,
                        args.repeats, after=check)
        bits = args.bits or (8 if n < (1 << 20) else 16)
        macs = work_macs(n, bits)
        t_msm = n / (res["msm_dev"]["M_per_s_mean"] * 1e6)
        res.update({"n": n, "bits": bits, "results_equal_runs": len(checks), "msm_dev_ms": round(1e3 * t_msm, 3),
                    "composed_dev_ms": round(1e3 * n / (res["composed_dev"]["M_per_s_mean"] * 1e6), 3),
                    "speedup_dev": round(res["msm_dev"]["M_per_s_mean"] / res["composed_dev"]["M_per_s_mean"], 2),
                    "limb_macs": macs, "limb_macs_per_term": round(macs / n), "imad_peak_fraction": round(macs / t_msm / IMAD_PEAK, 3)})
        out["sizes"][str(lg)] = res
        print(json.dumps({lg: res}), flush=True)
        if lg == args.profile_log2:
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                msm_dev()
                ok(lib.bjj_sync(ctx), "sync")
            kern = {}
            for ev in prof.key_averages():
                if ev.device_type.name == "CUDA" and ev.device_time_total > 0:
                    kern[ev.key[:80]] = round(ev.device_time_total / 1e3, 3)
            total = sum(kern.values())
            out["profile"] = {"log2_n": lg, "kernel_ms": kern, "total_ms": round(total, 3),
                              "sort_share": round(sum(v for key, v in kern.items() if "Radix" in key or "Onesweep" in key) / total, 3)}
        del a, k, px, py, cx, cy, cz, half, hp
        torch.cuda.empty_cache()

    if args.multi:
        n = 1 << 22
        pts = np.random.default_rng(2).integers(0, 256, (n, 32), dtype=np.uint8)
        pts[:, 31] &= 0x0F
        gx, gy = eng.fixed_base_batch(pts)
        kk = np.random.default_rng(3).integers(0, 256, (n, 32), dtype=np.uint8)
        want = eng.msm_batch(gx, gy, kk)[:2]
        multi = {}
        for g in range(1, lib.bjj_device_count() + 1):
            m = bjj.MultiEngine(list(range(g)))
            m.msm_batch(gx, gy, kk)
            t = time.perf_counter()
            r = m.msm_batch(gx, gy, kk)
            multi[g] = {"ms": round(1e3 * (time.perf_counter() - t), 3), "equal": bool(np.array_equal(r[0], want[0]) and
                                                                                          np.array_equal(r[1], want[1]))}
            m.close()
        out["multi_log2_n22"] = multi
    eng.close()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "msm.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
