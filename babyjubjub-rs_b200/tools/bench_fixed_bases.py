"""Throughput of the fixed-base tables for caller-chosen points (bjj_base_*), device-resident, on one GPU.

    python babyjubjub-rs_b200/tools/bench_fixed_bases.py --out DIR [--log2-lanes 22] [--steps 10] [--warmup 3]

Measures, for one random subgroup point P (and a second one, Q):
  - the table build of bjj_base_create (host clock around the call, which ends in a stream synchronise);
  - bjj_mul_scalar_batch_dev with P replicated into every lane: what a caller pays without a table;
  - bjj_base_mul_batch_dev on P's table;
  - bjj_fixed_base_batch_dev: B8's table, the same kernel over a table of the same size;
  - bjj_base_mul2_batch_dev with two caller tables (100 MB of tables against 126 MB of L2), and with B8 + P's table.
Every rate times `steps` back-to-back calls with CUDA events on one stream after `warmup` calls, closed by a
synchronise.  Scalars are uniform 256-bit values from a fixed seed.  The card's name and power limit are read in the
same run.  Writes DIR/fixed_bases.json and prints it.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

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


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, help="directory for fixed_bases.json")
    ap.add_argument("--log2-lanes", type=int, default=22)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--builds", type=int, default=5, help="timed table builds")
    args = ap.parse_args()

    import torch
    import babyjubjub_rs_b200 as bjj
    if not torch.cuda.is_available():
        raise SystemExit("bench_fixed_bases.py needs a CUDA device: there is no CPU fallback")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    eng = bjj.Engine(0)
    lib, ctx = eng.lib, eng.ctx
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    sp = ctypes.c_void_p(stream.cuda_stream)
    n = 1 << args.log2_lanes

    def ptr(t):
        return ctypes.c_void_p(t.data_ptr())

    def check(rc, what):
        if rc != 0:
            raise RuntimeError("%s failed: %d (%s)" % (what, rc, lib.bjj_error_string(rc).decode()))

    # P, Q: B8 times fixed 251-bit scalars (subgroup points), computed on the device
    pq = bjj.FixedBase(bjj.Point(*bjj.B8), eng).mul_batch([0x1234567 << 220, 0x7654321 << 220])
    p, q = pq

    # table build: host clock around bjj_base_create (synchronous on the context's stream)
    create_ms = []
    for i in range(1 + args.builds):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        base = bjj.FixedBase(p, eng)
        create_ms.append((time.perf_counter() - t0) * 1e3)
        base.close()
    create_ms = create_ms[1:]
    tp, tq = bjj.FixedBase(p, eng), bjj.FixedBase(q, eng)

    g = torch.Generator(device=dev)
    g.manual_seed(20261021)
    k = torch.randint(0, 256, (n, 32), dtype=torch.uint8, device=dev, generator=g)
    l = torch.randint(0, 256, (n, 32), dtype=torch.uint8, device=dev, generator=g)
    px = torch.tensor(list(bjj.ints_to_le32([p.x])[0]), dtype=torch.uint8, device=dev).repeat(n, 1)
    py = torch.tensor(list(bjj.ints_to_le32([p.y])[0]), dtype=torch.uint8, device=dev).repeat(n, 1)
    outs = {name: (torch.empty((n, 32), dtype=torch.uint8, device=dev), torch.empty((n, 32), dtype=torch.uint8, device=dev))
            for name in ("mul_scalar", "base_mul", "fixed_base", "mul2_two_tables", "mul2_b8_and_table")}
    calls = {
        "mul_scalar": lambda r: lib.bjj_mul_scalar_batch_dev(ctx, n, ptr(px), ptr(py), ptr(k), ptr(r[0]), ptr(r[1]), sp),
        "base_mul": lambda r: lib.bjj_base_mul_batch_dev(ctx, tp.handle, n, ptr(k), ptr(r[0]), ptr(r[1]), sp),
        "fixed_base": lambda r: lib.bjj_fixed_base_batch_dev(ctx, n, ptr(k), ptr(r[0]), ptr(r[1]), sp),
        "mul2_two_tables": lambda r: lib.bjj_base_mul2_batch_dev(ctx, tp.handle, tq.handle, n, ptr(k), ptr(l), ptr(r[0]),
                                                                 ptr(r[1]), sp),
        "mul2_b8_and_table": lambda r: lib.bjj_base_mul2_batch_dev(ctx, None, tp.handle, n, ptr(k), ptr(l), ptr(r[0]),
                                                                   ptr(r[1]), sp),
    }
    results = {}
    for name, fn in calls.items():
        r = outs[name]
        for _ in range(args.warmup):
            check(fn(r), name)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            check(fn(r), name)
        e1.record(stream)
        torch.cuda.synchronize()
        check(lib.bjj_sync(ctx), name)
        ms = e0.elapsed_time(e1) / args.steps
        results[name] = {"ms_per_call": round(ms, 4), "M_points_per_s": round(n / ms / 1e3, 2)}
    same = bool(torch.equal(outs["mul_scalar"][0], outs["base_mul"][0]) and torch.equal(outs["mul_scalar"][1], outs["base_mul"][1]))
    rate = {name: r["M_points_per_s"] for name, r in results.items()}
    report = {
        "card": card_info(0),
        "torch_device_name": torch.cuda.get_device_name(0),
        "lanes": n,
        "steps": args.steps,
        "warmup": args.warmup,
        "table_build_ms": {"mean": round(sum(create_ms) / len(create_ms), 3), "min": round(min(create_ms), 3),
                           "max": round(max(create_ms), 3), "runs": len(create_ms)},
        "results": results,
        "base_mul_over_replicated_mul_scalar": round(rate["base_mul"] / rate["mul_scalar"], 2),
        "base_mul_over_fixed_base": round(rate["base_mul"] / rate["fixed_base"], 3),
        "mul2_two_tables_over_base_mul": round(rate["mul2_two_tables"] / rate["base_mul"], 3),
        "mul2_b8_and_table_over_base_mul": round(rate["mul2_b8_and_table"] / rate["base_mul"], 3),
        "base_mul_equals_replicated_mul_scalar": same,
    }
    tp.close()
    tq.close()
    eng.close()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "fixed_bases.json"), "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(report, indent=1))
    if not same:
        raise SystemExit("base_mul and mul_scalar disagree")


if __name__ == "__main__":
    main()
